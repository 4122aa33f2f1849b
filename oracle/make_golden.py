"""TEST INFRASTRUCTURE ONLY — generates tests/golden/*.pt by running the UNMODIFIED reference
modules (via oracle/ref_shim.py) in the build container.  Run: ``python -m oracle.make_golden``.

Weights are NOT stored (9.5 M floats): every case records the ``init_params`` seed; the
reference modules are loaded with exactly those tensors through ``load_state_dict``.  Stored:
inputs' seeds/shapes, loss, scores, alphas, encoder output, bias gradients in full, and for
the big weight gradients their sum / abs-sum / first 256 values — plus a 3-step Adam loss
trajectory.  Outputs of more than OUTPUT_FULL_MAX elements are stored as the same summaries, so
that every file stays under 1 MB.  Tests read only these files, never the reference itself.
"""
import os
import sys

import torch

from oracle import ref_model as rm
from oracle import ref_shim

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

CASES = {
    # name: B, H, W, V, tmin, tmax, train(dropout), positional
    "tiny_eval": dict(B=2, H=32, W=64, V=40, tmin=3, tmax=6, train=False, positional=True, pseed=11, dseed=21),
    "tiny_train": dict(B=3, H=32, W=80, V=40, tmin=3, tmax=7, train=True, positional=True, pseed=12, dseed=22),
    "tiny_nopos": dict(B=2, H=48, W=64, V=37, tmin=2, tmax=5, train=False, positional=False, pseed=13, dseed=23),
    "cfg1": dict(B=4, H=64, W=256, V=100, tmin=8, tmax=32, train=False, positional=True, pseed=14, dseed=24),
    # BASELINE.json configs[1] shapes (R = 14*62 = 868, T = 150, V = 500) on a B=8 sample of the batch, dropout active:
    # the exact tiles / 150-step recurrence the bench runs.  Summaries only (strided samples), ~0.6 MB.
    "cfg2": dict(B=8, H=128, W=512, V=500, tmin=150, tmax=150, train=True, positional=True, pseed=16, dseed=26, summaries_only=True),
}

SAMPLE_N = 8192
OUTPUT_FULL_MAX = 65536


def summarize(g):
    out = {}
    for k, v in g.items():
        v = v.detach()
        if v.numel() <= 4096:
            out[k] = v.clone()
        else:
            out[k] = dict(sum=v.double().sum().item(), abssum=v.double().abs().sum().item(),
                          head=v.reshape(-1)[:256].clone(), shape=tuple(v.shape))
            out[k].update(strided_sample(v))
    return out


def strided_sample(v):
    """SAMPLE_N values at a fixed stride (coprime offsets so that every row/column phase is visited) + the full-tensor
    L2 norm: lets a test bound the relative NORM error of a big tensor from the sample."""
    flat = v.detach().reshape(-1)
    n = flat.numel()
    stride = max(1, n // SAMPLE_N)
    if stride > 1 and stride % 2 == 0:
        stride += 1
    idx = (torch.arange(min(SAMPLE_N, n), dtype=torch.int64) * stride) % n
    return dict(sample_stride=stride, sample=flat[idx].clone(), norm=flat.double().norm().item())


def dropout_masks(seed, B, T, D, p=0.5):
    """Reproduces nn.Dropout's CPU draws of the reference forward (seq2seq_torch.py:316): after
    manual_seed(seed) the only RNG consumers are the T dropout calls on [B, D]."""
    torch.manual_seed(seed)
    return torch.stack([torch.nn.functional.dropout(torch.ones(B, D), p, True) for _ in range(T)], dim=1)


def run_case(name, c):
    pe, pd = rm.init_params(c["V"], seed=c["pseed"])
    enc, dec = ref_shim.build_reference_models(c["V"], positional_embeddings=c["positional"])
    enc.load_state_dict(pe)
    dec.load_state_dict(pd)
    img, formula = rm.synthetic_batch(c["B"], c["H"], c["W"], c["V"], c["tmin"], c["tmax"], seed=c["dseed"])
    T = formula.shape[1] - 1
    enc.train(c["train"])
    dec.train(c["train"])
    rec = dict(case=c, torch=torch.__version__)
    mask_seed = 1000 + c["dseed"]
    oe = torch.optim.Adam(enc.parameters(), lr=1e-3)          # img2seq_torch.py:86-87
    od = torch.optim.Adam(dec.parameters(), lr=1e-3)
    traj = []
    for step in range(3):
        torch.manual_seed(mask_seed + step)
        loss, scores, alphas = ref_shim.ref_get_loss(enc, dec, img, formula)
        od.zero_grad()
        oe.zero_grad()
        loss.backward()
        if step == 0:
            rec["loss"] = loss.item()
            for k, v in (("scores", scores), ("alphas", alphas), ("enc_out", enc(img))):
                big = c.get("summaries_only") or v.numel() > OUTPUT_FULL_MAX
                rec[k] = summarize({k: v})[k] if big else v.detach().clone()
            rec["grad_enc"] = summarize({k: v.grad for k, v in enc.named_parameters()})
            rec["grad_dec"] = summarize({k: v.grad for k, v in dec.named_parameters()})
        od.step()
        oe.step()
        traj.append(-loss.item())                              # getLoss returns -loss (:172)
    rec["get_loss_trajectory"] = traj
    rec["mask_seed"] = mask_seed
    # self-check: restatement reproduces it bit for bit right now
    mask = dropout_masks(mask_seed, c["B"], T, 512) if c["train"] else None
    l2, aux = rm.get_loss(pe, pd, img, formula, dropout_mask=mask, positional=c["positional"])
    assert abs(l2.item() - rec["loss"]) == 0.0, (name, l2.item(), rec["loss"])
    if isinstance(rec["scores"], dict):
        assert (strided_sample(aux["scores"])["sample"] - rec["scores"]["sample"]).abs().max().item() == 0.0
    else:
        assert (aux["scores"] - rec["scores"]).abs().max().item() == 0.0
    torch.save(rec, os.path.join(OUT, name + ".pt"))
    print(name, "loss", rec["loss"], "traj", traj, "T", T,
          "bytes", os.path.getsize(os.path.join(OUT, name + ".pt")))


def run_cnn_variant():
    """Encoder-only fixture for encoder_cnn='cnn' (seq2seq_torch.py:58-86): output and the gradients of sum(out * G)."""
    c = dict(B=2, H=32, W=80, V=20, pseed=15, dseed=25, gseed=35)
    pe, _ = rm.init_params(c["V"], seed=c["pseed"], encoder_cnn="cnn")
    enc, _ = ref_shim.build_reference_models(c["V"], encoder_cnn="cnn")
    enc.load_state_dict(pe)
    img, _ = rm.synthetic_batch(c["B"], c["H"], c["W"], c["V"], 3, 4, seed=c["dseed"])
    out = enc(img)
    G = torch.randn(out.shape, generator=torch.Generator().manual_seed(c["gseed"]))
    (out * G).sum().backward()
    rec = dict(case=c, torch=torch.__version__, enc_out=out.detach().clone(),
               grad_enc=summarize({k: v.grad for k, v in enc.named_parameters()}))
    assert (rm.encoder_forward(pe, img, encoder_cnn="cnn") - out).abs().max().item() == 0.0
    torch.save(rec, os.path.join(OUT, "cnn_variant.pt"))
    print("cnn_variant", tuple(out.shape), "bytes", os.path.getsize(os.path.join(OUT, "cnn_variant.pt")))


def run_reference_outputs():
    """The reference's own forward outputs, in full: getLoss (loss, scores, alphas) in eval mode, and
    DecoderWithAttention.forward with ragged caption lengths (the shrinking batch, seq2seq_torch.py:308)."""
    c = dict(B=2, H=32, W=96, V=50, tmin=3, tmax=6, pseed=21, dseed=22, lengths=[[7], [4]])
    pe, pd = rm.init_params(c["V"], seed=c["pseed"])
    enc, dec = ref_shim.build_reference_models(c["V"])
    enc.load_state_dict(pe)
    dec.load_state_dict(pd)
    dec.eval()
    img, formula = rm.synthetic_batch(c["B"], c["H"], c["W"], c["V"], c["tmin"], c["tmax"], seed=c["dseed"])
    loss, scores, alphas = ref_shim.ref_get_loss(enc, dec, img, formula)
    r_scores, _, r_lengths, r_alphas, _ = dec(enc(img), formula, torch.tensor(c["lengths"]))
    rec = dict(case=c, torch=torch.__version__, loss=loss.item(), scores=scores.detach().clone(), alphas=alphas.detach().clone(),
               ragged_scores=r_scores.detach().clone(), ragged_alphas=r_alphas.detach().clone(), ragged_decode_lengths=list(r_lengths))
    torch.save(rec, os.path.join(OUT, "reference_outputs.pt"))
    print("reference_outputs loss", rec["loss"], "bytes", os.path.getsize(os.path.join(OUT, "reference_outputs.pt")))


def main():
    if not ref_shim.reference_available():
        sys.exit("reference tree not available; golden files can only be regenerated in the build container")
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    only = set(sys.argv[1:])
    for name, c in CASES.items():
        if only and name not in only:
            continue
        run_case(name, c)
    if not only or "cnn_variant" in only:
        run_cnn_variant()
    if not only or "reference_outputs" in only:
        run_reference_outputs()


if __name__ == "__main__":
    main()
