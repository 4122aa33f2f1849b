"""Decode throughput of the two-layer extension model (Img2SeqRowModel, BASELINE.json configs[3]: CNN -> row biLSTM -> attention
LSTM -> second LSTM layer -> fc) against the one-layer Img2SeqModel on the same images, in the same process.

160x640 images (256, then 64), bf16 / tensor-core kernels, random-init weights: END never fires, so every call runs the full
max_length_formula + 2 = 152 steps.  Both models are built from the same seed, so their CNN and layer-1 weights are identical and
the difference between them is the row encoder and layer 2.  Greedy and beam-5; after one warm-up call per (model, mode, batch),
two passes alternate the models.  A decode call takes at most 1024 rows (images * beam: the attention workspace keeps one ticket
counter per row), so beam-5 over 256 images runs as two calls of 128.  Prints one JSON line with the card name and power limit."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from latex_ocr_b200 import _lib, decode, ext
from latex_ocr_b200.data import SimpleVocab
from latex_ocr_b200.img2seq import Img2SeqModel


class Cfg:
    encoder_cnn = "vanilla"; positional_embeddings = True; lr_init = 1e-3; lr_method = "adam"


V, L, STEPS, MAX_ROWS = 500, 150, 152, 1024


def build(cls):
    torch.manual_seed(0)
    m = cls(Cfg(), vocab=SimpleVocab(V), device="cuda:0", precision="bf16", impl="tc").build_pred()
    m.train_mode(False)
    return m


models = {"two_layer": (build(ext.Img2SeqRowModel), ext), "one_layer": (build(Img2SeqModel), decode)}
g = torch.Generator().manual_seed(0)
imgs = torch.where(torch.rand(256, 1, 160, 640, generator=g) < 0.1, torch.randint(0, 255, (256, 1, 160, 640), generator=g).float(),
                   torch.tensor(255.0))


def run(name, mode, n):
    """One decode of the first n images; returns (seconds, tokens of the scored hypothesis, library launches)."""
    m, mod = models[name]
    beam = 1 if mode == "greedy" else 5
    calls = -(-n * beam // MAX_ROWS)
    per = n // calls
    torch.cuda.synchronize()
    l0, t0 = _lib.launch_count(), time.perf_counter()
    toks = 0
    for c in range(calls):
        x = imgs[c * per:(c + 1) * per]
        if beam == 1:
            ids = mod.greedy_decode(m, x, V - 2, V - 1, L)
            assert ids.shape[1] == STEPS, ids.shape
            toks += ids.numel()
        else:
            ids, _ = mod.beam_decode(m, x, V - 2, V - 1, beam, L)
            assert ids.shape[2] == STEPS, ids.shape
            toks += ids.shape[0] * ids.shape[2]
    torch.cuda.synchronize()
    return time.perf_counter() - t0, toks, _lib.launch_count() - l0, calls


def row_encoder_seconds(n):
    """Time of the row biLSTM alone over the CNN features of n images (the one-off part of the two-layer model's extra cost)."""
    m = models["two_layer"][0]
    with torch.no_grad():
        feat = m.encoder.forward_raw(imgs[:n].to(m.device), need_grad=False)
        m.row_encoder.forward_raw(feat)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(2):
            m.row_encoder.forward_raw(feat)
        torch.cuda.synchronize()
    return (time.perf_counter() - t0) / 2


out = {}
for n in (256, 64):
    for mode in ("greedy", "beam5"):
        for name in models:
            run(name, mode, n)                                       # warm-up: workspaces, kernel attributes
        acc = {name: [0.0, 0, 0, 0] for name in models}
        for rep in range(2):
            for name in models:
                s, t, l, c = run(name, mode, n)
                a = acc[name]
                a[0] += s; a[1] += t; a[2] = l; a[3] = c
        for name, (s, t, l, c) in acc.items():
            out["%s_%s_%d" % (name, mode, n)] = {"tokens_per_s": t / s, "images_per_s": 2 * n / s, "seconds_2_passes": s,
                                                 "launches_per_step": l / (c * STEPS)}
        calls = acc["two_layer"][3]
        rows = row_encoder_seconds(n // calls) * calls
        d = (acc["two_layer"][0] / 2 - acc["one_layer"][0] / 2 - rows) / (calls * STEPS)
        out["row_encoder_ms_%s_%d" % (mode, n)] = rows * 1e3
        out["layer2_us_per_step_%s_%d" % (mode, n)] = d * 1e6           # two-layer minus one-layer time per call, less the row encoder
try:
    pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                        text=True, timeout=30).stdout.strip()
except Exception as e:                                               # noqa: BLE001 — report, do not fail the measurement
    pl = "unknown (%s)" % e
print(json.dumps({"workload": "160x640, 256 and 64 images, 152 steps, bf16, two-layer vs one-layer, 1 x GPU",
                  "card": torch.cuda.get_device_name(0), "power_limit": pl, **out}))
