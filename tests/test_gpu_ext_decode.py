"""-m gpu: greedy and beam decoding of the two-layer extension model (latex_ocr_b200/ext.py greedy_decode / beam_decode on
lo_decoder2_*) against its CPU definition (tests/ext_decode_oracle.py greedy_decode_ext / beam_decode_ext, the loop rules of
oracle/ref_decode.py).  fp32 mode: token ids must match exactly; bf16: agreement on the clear-margin steps."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from util import Cfg

import ext_decode_oracle as xo  # noqa: E402  (after util: it puts the repository root on sys.path)

pytestmark = pytest.mark.gpu


def _ext_model(V, pe, prow, pd, p2, precision, vocab=None):
    from latex_ocr_b200.ext import Img2SeqRowModel
    m = Img2SeqRowModel(Cfg(), vocab=vocab, n_tok=V, device="cuda", precision=precision,
                        impl="tc" if precision == "bf16" else "simt")
    m.build_train()
    m.encoder.load_state_dict(pe)
    m.decoder.load_state_dict(pd)
    m.row_encoder.load_state_dict(prow)
    m.layer2.load_state_dict(p2)
    m.train_mode(False)
    return m


def _params(V, seed):
    from oracle import ref_ext as rx
    from oracle import ref_model as rm
    pe, pd = rm.init_params(V, seed=seed)
    # make decoding non-degenerate (as test_gpu_decode._setup): larger output layer so the argmax moves and END appears
    g = torch.Generator().manual_seed(seed)
    pd["fc.weight"] = (torch.rand(V, 512, generator=g) * 2 - 1) * 0.5
    pd["embedding.weight"] = (torch.rand(V, 512, generator=g) * 2 - 1) * 1.0
    prow, p2 = rx.init_params_ext(seed=seed + 1)
    return pe, prow, pd, p2


def _setup(V=30, seed=4, N=3, H=32, W=80):
    from oracle import ref_ext as rx
    from oracle import ref_model as rm
    pe, prow, pd, p2 = _params(V, seed)
    img, _ = rm.synthetic_batch(N, H, W, V, 3, 5, seed=seed + 1)
    m = _ext_model(V, pe, prow, pd, p2, "fp32")
    enc = rx.row_encoder_forward(prow, rm.encoder_forward(pe, img)).reshape(N, -1, 512)
    return pd, p2, m, img, enc


def test_greedy_tokens_match_oracle():
    from latex_ocr_b200 import ext
    V = 30
    pd, p2, m, img, enc = _setup(V)
    for end_id, L in ((V - 1, 6), (7, 12)):
        want = xo.greedy_decode_ext(pd, p2, enc, V - 2, end_id, L + 1)
        got = ext.greedy_decode(m, img, start_id=V - 2, end_id=end_id, max_length_formula=L)
        assert got.shape == want.shape, (got.shape, want.shape)
        assert torch.equal(got, want)


@pytest.mark.parametrize("beam", [1, 3, 5])
def test_beam_tokens_match_oracle(beam):
    from latex_ocr_b200 import ext
    V = 30
    pd, p2, m, img, enc = _setup(V, seed=6)
    got_by_fin = {}
    for fin in ("reference", "backtrack"):
        want, wlp = xo.beam_decode_ext(pd, p2, enc, V - 2, 5, beam, 9, finalize=fin)
        got, glp = ext.beam_decode(m, img, start_id=V - 2, end_id=5, beam_size=beam, max_length_formula=8, finalize=fin)
        assert got.shape == want.permute(0, 2, 1).shape
        assert torch.equal(got, want.permute(0, 2, 1))
        assert (glp - wlp).abs().max().item() < 1e-3 * max(1.0, wlp.abs().max().item())
        got_by_fin[fin] = got
    if beam > 1:
        # the search really re-parents (some parent differs from its own beam index): back-tracking the lineage changes the
        # hypotheses, and those equal the oracle's only if layer 2's state followed the parents
        assert not torch.equal(got_by_fin["reference"], got_by_fin["backtrack"])


def test_beam_diversity_penalty_matches_oracle():
    from latex_ocr_b200 import ext
    V, beam, L = 30, 3, 8
    pd, p2, m, img, enc = _setup(V, seed=6)
    N = img.shape[0]
    u = torch.rand(L + 2, N * beam, V, generator=torch.Generator().manual_seed(77))
    want, wlp = xo.beam_decode_ext(pd, p2, enc, V - 2, 5, beam, L + 1, div_gamma=0.5, div_prob=1.0, div_u=u)
    base, _ = xo.beam_decode_ext(pd, p2, enc, V - 2, 5, beam, L + 1)
    assert want.shape != base.shape or not torch.equal(want, base)          # the penalty changes the search at these settings
    got, glp = ext.beam_decode(m, img, V - 2, 5, beam, L, div_gamma=0.5, div_prob=1.0, div_u=u)
    assert torch.equal(got, want.permute(0, 2, 1))
    assert (glp - wlp).abs().max().item() < 1e-3 * max(1.0, wlp.abs().max().item())
    a1, _ = ext.beam_decode(m, img, V - 2, 5, beam, L, div_gamma=0.5, div_prob=0.5, div_seed=9)
    a2, _ = ext.beam_decode(m, img, V - 2, 5, beam, L, div_gamma=0.5, div_prob=0.5, div_seed=9)
    assert torch.equal(a1, a2)


def test_greedy_attention_export():
    from latex_ocr_b200 import ext
    from oracle import ref_model as rm
    V = 30
    pd, p2, m, img, enc = _setup(V)
    ids, att = ext.greedy_decode(m, img, start_id=V - 2, end_id=V - 1, max_length_formula=6, return_attention=True)
    assert att.shape == (img.shape[0], ids.shape[1], enc.shape[1])
    assert (att.sum(dim=2) - 1).abs().max().item() < 1e-4
    h0, _ = rm.init_hidden_state(pd, enc)
    _, a0 = rm.attention_forward(pd, enc, h0)
    assert (att[:, 0] - a0).abs().max().item() < 1e-5


@pytest.mark.parametrize("N", [80, 16])
def test_bf16_greedy_clear_margin_agreement_160x640(N):
    """bf16 decode step kernels at 160x640 (N = 80 rows: tcgen05 GEMMs for layer 2; N = 16: the mma.sync kernel).  The fp32 oracle
    is teacher-forced on the GPU's own tokens; on every step whose fp32 top-2 logit margin exceeds 5e-2 its argmax must be the
    token the GPU chose (>= 0.99 of those steps, the rule of test_gpu_decode.test_bf16_greedy_token_match_rate_at_cfg5_widths).
    The logits go through layer 2's hidden state, which stays small at nn.LSTMCell's initialisation, so about a third of the steps
    clear the margin here (548 of 1 600 and 111 of 320 on a B200); at least a quarter must.
    The fp32 encoder output comes from the fp32 kernels (checked against the oracle in test_gpu_ext.py): a CPU CNN over 80
    images of 160x640 would dominate the test."""
    from latex_ocr_b200 import ext
    from oracle import ref_model as rm
    V, L = 500, 18
    pe, prow, pd, p2 = _params(V, seed=21)
    img, _ = rm.synthetic_batch(N, 160, 640, V, 3, 5, seed=31 + N)
    m16 = _ext_model(V, pe, prow, pd, p2, "bf16")
    m32 = _ext_model(V, pe, prow, pd, p2, "fp32")
    with torch.no_grad():
        enc = ext._encode(m32, img).float().cpu().reshape(N, -1, 512)
    got = ext.greedy_decode(m16, img, V - 2, V - 1, L)
    n = got.shape[1]
    caps = torch.cat([torch.full((N, 1), V - 2, dtype=torch.long), got], dim=1)
    # decoder2_forward teacher-forced on those tokens, with att1 hoisted (the oracle's step function) to keep the CPU time small
    step = xo.two_layer_step(pd, p2)
    with torch.no_grad():
        att1 = F.linear(enc, pd["attention.encoder_att.weight"], pd["attention.encoder_att.bias"])
        state, out = xo.initial_state(pd, enc), []
        for t in range(n):
            lg, state = step((enc, att1), state, caps[:, t])
            out.append(lg)
        ref_logits = torch.stack(out, dim=1)
    top2 = ref_logits.topk(2, dim=-1).values
    clear = (top2[..., 0] - top2[..., 1]) > 5e-2
    hit = ref_logits.argmax(-1) == got
    agree, considered = int((hit & clear).sum()), int(clear.sum())
    rate = agree / max(considered, 1)
    print("ext bf16 greedy N=%d: clear-margin agreement %d/%d = %.4f (all steps %.4f)" % (N, agree, considered, rate,
                                                                                         float(hit.float().mean())))
    assert considered >= 0.25 * N * n and rate >= 0.99


def test_write_prediction_scores_the_two_layer_model(tmp_path):
    """Img2SeqRowModel.write_prediction (what evaluate / train(..., val_set) report): the perplexity is that of the two-layer
    model (oracle teacher-forced CE) and hyp_0.txt holds ext.greedy_decode's tokens."""
    from latex_ocr_b200 import ext
    from latex_ocr_b200.data import SimpleVocab
    from oracle import ref_ext as rx
    from oracle import ref_model as rm
    V = 30
    pe, prow, pd, p2 = _params(V, seed=11)
    vocab = SimpleVocab(V)
    rng = np.random.RandomState(3)
    data = [(rng.randint(0, 256, (32, 64, 1)).astype(np.uint8), [int(x) for x in rng.randint(0, V - 3, 3 + i)]) for i in range(3)]
    cfg = Cfg(batch_size=2, max_length_formula=6, decoding="greedy", dir_answers=str(tmp_path) + "/answers/")
    m = _ext_model(V, pe, prow, pd, p2, "fp32", vocab=vocab)
    m._config = cfg
    files, perp = m.write_prediction(cfg, data)
    # oracle: teacher-forced CE of the two-layer model over every real token + END, inputs START (= PAD) + tokens
    ce, nw = 0.0, 0
    hyps = []
    for b0 in range(0, len(data), cfg.batch_size):
        batch = data[b0:b0 + cfg.batch_size]
        img = torch.from_numpy(np.stack([d[0] for d in batch])).permute(0, 3, 1, 2).float()
        T = max(len(d[1]) for d in batch) + 1
        caps = torch.full((len(batch), T + 1), vocab.id_pad, dtype=torch.long)
        for i, (_, f) in enumerate(batch):
            caps[i, 1:len(f) + 1] = torch.tensor(f)
            caps[i, len(f) + 1] = vocab.id_end
        enc = rx.row_encoder_forward(prow, rm.encoder_forward(pe, img)).reshape(len(batch), -1, 512)
        logits, _ = rx.decoder2_forward(pd, p2, enc, caps, T)
        lsm = torch.log_softmax(logits.double(), dim=-1)
        for i, (_, f) in enumerate(batch):
            n = len(f) + 1
            ce -= float(lsm[i, torch.arange(n), caps[i, 1:n + 1]].sum())
            nw += n
        ids = ext.greedy_decode(m, img, vocab.id_pad, vocab.id_end, cfg.max_length_formula)
        hyps += [" ".join(str(t) for t in (s[:s.index(vocab.id_end)] if vocab.id_end in s else s)) for s in ids.tolist()]
    want = -float(np.exp(ce / nw))
    assert abs(perp - want) <= 1e-4 * abs(want), (perp, want)
    assert open(str(tmp_path) + "/answers/hyp_0.txt").read().splitlines() == hyps
