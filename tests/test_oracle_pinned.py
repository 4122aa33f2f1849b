"""CPU (-m "not gpu"): the oracle restatement against the golden fixtures generated from the UNMODIFIED
reference (oracle/make_golden.py)."""
import pytest
import torch

from util import load_golden, relerr
from oracle import ref_model as rm


def _inputs(rec):
    c = rec["case"]
    pe, pd = rm.init_params(c["V"], seed=c["pseed"])
    img, formula = rm.synthetic_batch(c["B"], c["H"], c["W"], c["V"], c["tmin"], c["tmax"], seed=c["dseed"])
    return c, pe, pd, img, formula


def _masks(seed, B, T):
    torch.manual_seed(seed)
    return torch.stack([torch.nn.functional.dropout(torch.ones(B, 512), 0.5, True) for _ in range(T)], dim=1)


@pytest.mark.parametrize("name", ["tiny_eval", "tiny_train", "tiny_nopos"])
def test_restatement_matches_golden(name):
    torch.set_num_threads(8)
    rec = load_golden(name)
    c, pe, pd, img, formula = _inputs(rec)
    T = formula.shape[1] - 1
    mask = _masks(rec["mask_seed"], c["B"], T) if c["train"] else None
    loss, aux = rm.get_loss(pe, pd, img, formula, dropout_mask=mask, positional=c["positional"])
    assert abs(loss.item() - rec["loss"]) <= 1e-6 * abs(rec["loss"])
    assert relerr(aux["scores"], rec["scores"]) < 1e-5
    assert relerr(aux["alphas"], rec["alphas"]) < 1e-5
    assert relerr(aux["enc"], rec["enc_out"]) < 1e-5
    # hoisting encoder_att out of the loop changes nothing beyond rounding (SURVEY quirk Q1)
    lh, _ = rm.get_loss(pe, pd, img, formula, dropout_mask=mask, hoist=True, positional=c["positional"])
    assert abs(lh.item() - rec["loss"]) <= 1e-5 * abs(rec["loss"])


def test_train_trajectory_matches_golden():
    rec = load_golden("tiny_train")
    c, pe, pd, img, formula = _inputs(rec)
    T = formula.shape[1] - 1
    st = {}
    traj = []
    for step in range(3):
        mask = _masks(rec["mask_seed"] + step, c["B"], T)
        neg, ge, gd, _ = rm.train_step(pe, pd, img, formula, st, dropout_mask=mask, positional=c["positional"])
        traj.append(neg)
        if step == 0:
            for k, want in rec["grad_dec"].items():
                if isinstance(want, dict):
                    assert abs(gd[k].double().sum().item() - want["sum"]) <= 1e-4 * (want["abssum"] + 1e-30)
                else:
                    assert relerr(gd[k], want) < 1e-4 or want.abs().max() < 1e-7
    for a, b in zip(traj, rec["get_loss_trajectory"]):
        assert abs(a - b) <= 1e-4 * abs(b)


def test_manual_backward_equals_autograd():
    """The hand-derived decoder backward (the algorithm lo_decoder.cu implements) == autograd, fp64."""
    V = 30
    pe, pd = rm.init_params(V, seed=3, dtype=torch.float64)
    img, formula = rm.synthetic_batch(3, 32, 64, V, 3, 6, seed=4)
    enc = rm.encoder_forward(pe, img.double()).reshape(3, -1, 512).detach().requires_grad_(True)
    T = formula.shape[1] - 1
    pdg = {k: v.clone().requires_grad_(True) for k, v in pd.items()}
    mask = (torch.rand(3, T, 512, generator=torch.Generator().manual_seed(1)) > 0.5).double() * 2
    s = rm.decoder_forward_saved(pdg, enc, formula, T, dropout_mask=mask)
    loss, _, _ = rm.loss_from_outputs(s["logits"], formula, [T] * 3, s["alphas"])
    loss.backward()
    with torch.no_grad():
        s2 = rm.decoder_forward_saved(pd, enc.detach(), formula, T, dropout_mask=mask)
        lm, g, denc = rm.decoder_backward_manual(pd, s2)
    assert abs(lm.item() - loss.item()) < 1e-12
    for k in pd:
        assert (pdg[k].grad - g[k]).abs().max().item() < 1e-12, k
    assert (enc.grad - denc).abs().max().item() < 1e-14


def test_restatement_matches_reference_outputs():
    """The reference's forward outputs stored in full (oracle/make_golden.py, where the restatement reproduced them bit for
    bit).  A CPU with another thread count or vector width may sum in another order, so floats are held to 1e-6."""
    torch.set_num_threads(8)
    rec = load_golden("reference_outputs")
    c = rec["case"]
    pe, pd = rm.init_params(c["V"], seed=c["pseed"])
    img, formula = rm.synthetic_batch(c["B"], c["H"], c["W"], c["V"], c["tmin"], c["tmax"], seed=c["dseed"])
    loss, aux = rm.get_loss(pe, pd, img, formula)
    assert abs(loss.item() - rec["loss"]) <= 1e-6 * abs(rec["loss"])
    assert aux["scores"].shape == rec["scores"].shape and relerr(aux["scores"], rec["scores"]) < 1e-6
    assert aux["alphas"].shape == rec["alphas"].shape and relerr(aux["alphas"], rec["alphas"]) < 1e-6
    # ragged lengths (shrinking batch) through DecoderWithAttention.forward
    out = rm.decoder_forward(pd, rm.encoder_forward(pe, img), formula, torch.tensor(c["lengths"]))
    assert out[2] == rec["ragged_decode_lengths"]
    assert out[0].shape == rec["ragged_scores"].shape and relerr(out[0], rec["ragged_scores"]) < 1e-6
    assert out[3].shape == rec["ragged_alphas"].shape and relerr(out[3], rec["ragged_alphas"]) < 1e-6


def test_tf_flavour_oracle_self_consistency():
    """oracle/ref_tf_model.py (parity unpinned, see its header): structural checks that do not need TensorFlow —
    beam 1 == greedy, the masked CE equals its definition, dropout multipliers of 1 are the identity."""
    from oracle import ref_tf_model as tfm
    V = 25
    p = tfm.init_params_tf(V, seed=2)
    p["y_W_o"] = p["y_W_o"] * 4.0
    g = torch.Generator().manual_seed(0)
    enc = torch.relu(torch.randn(2, 9, 512, generator=g))
    formula = torch.randint(0, V, (2, 5), generator=g)
    logits, alphas = tfm.decoder_train_logits(p, enc, formula)
    assert logits.shape == (2, 5, V) and torch.allclose(alphas.sum(-1), torch.ones(2, 5), atol=1e-5)
    ones = torch.ones(2, 5, 512)
    l2, _ = tfm.decoder_train_logits(p, enc, formula, ones, ones)
    assert torch.equal(logits, l2)
    lengths = torch.tensor([5, 2])
    loss, ce_words, n_words = tfm.masked_ce(logits, formula, lengths)
    lp = torch.log_softmax(logits, -1)
    want = -(lp[0, torch.arange(5), formula[0]].sum() + lp[1, torch.arange(2), formula[1, :2]].sum())
    assert abs(ce_words.item() - want.item()) < 1e-4 and n_words.item() == 7 and abs(loss.item() - want.item() / 7) < 1e-5
    gr = tfm.greedy_decode(p, enc, end_id=V - 1, max_iter=7)
    bm, _ = tfm.beam_decode(p, enc, end_id=V - 1, beam=1, max_iter=7)
    n = min(gr.shape[1], bm.shape[1])
    assert torch.equal(gr[:, :n], bm[:, :n, 0])
