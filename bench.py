#!/usr/bin/env python
"""bench.py — formula-images/sec of one full im2latex train step (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16|fp32] [--dump-outputs DIR]

N=1 workload = BASELINE.json configs[1]: batch 64, 1x128x512 images, 6-conv encoder + 512-d attention LSTM
decoder, vocab 500, every caption padded to T=150 decode steps (the reference trains on PADs,
img2seq_torch.py:144), bf16 storage / fp32 accumulate.  N>1 (torchrun, one rank per GPU): the same per-GPU
batch on every rank (weak scaling), NCCL all-reduce of the two gradient buckets.

A "step" = encoder fwd -> decoder fwd -> loss -> decoder bwd -> encoder bwd -> [all-reduce] -> Adam, nothing
skipped.  `value` times K steps with inputs resident in HBM (CUDA events around each step, summed; max over ranks);
`e2e` times K steps through Img2SeqModel.train_step with PINNED HOST inputs (H2D inside) and a D2H read of the loss.
`--impl reference` times the reference's CPU algorithm (oracle port, un-hoisted exactly as the reference
executes it) on the host cores of rank 0.

The batch, the initial weights and the dropout seed are seeded, and every warm-up and timed step of `value` trains
the same state (the initial weights, zero Adam moments; restored between steps, outside the timed intervals): the
backward adds partial sums with fp32 atomics in varying order, and carried from step to step those last-bit
differences grow through the recurrence, the ReLU / max-pool tie-breaks and Adam until two runs train different
models.  So a step's inputs are the same on every run, and so is its loss, which the forward computes without atomics.
`--dump-outputs DIR` writes what the last timed step returned to its caller (Img2SeqModel.train_step) as
DIR/loss.npy: [total, ce, reg, n_valid], float32.  Two builds run with the same arguments can then be compared.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG2 = dict(B=64, H=128, W=512, V=500, T=150)
# EXTENSION workload (BASELINE.json configs[3], not in the reference): row-encoder biLSTM over the CNN feature rows + a second
# decoder layer, 160x640 images (R = 18 * 78 = 1404 regions) — `--workload cfg4`, latex_ocr_b200/ext.py
CFG4 = dict(B=64, H=160, W=640, V=500, T=150)
FWD_BWD_GFLOP_PER_IMG = 56.0          # conv stack, SURVEY.md §8-d (18.67 fwd, x3 fwd+bwd)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm,power.draw,"
                 "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


METRIC = "formula-images/sec (train step, 128x512 px, seq<=150)"       # the SAME string on both arms (the driver divides them)


def run_reference(args, rank):
    """CPU reference arm: the reference's own getLoss (unmodified modules when the reference tree is importable, else the
    oracle port executing the same un-hoisted algorithm), all host threads, each step a bounded sample of the cfg2 batch
    (B=LO_REF_SAMPLE_B rows of the 64).  One extra step at twice the sample backs "linear in batch"."""
    if rank != 0:
        return
    import torch
    import bench_support as bs
    sample_b = int(os.environ.get("LO_REF_SAMPLE_B", "8"))
    c = CFG2
    dt, kind, cores = bs.cpu_arm(c, sample_b, steps=args.steps, warmup=args.warmup)
    v = sample_b / dt
    lin = None
    if os.environ.get("LO_REF_LINEARITY", "1") == "1":
        dt2, _, _ = bs.cpu_arm(c, 2 * sample_b, steps=1, warmup=1)
        lin = {"images_per_s_at_B%d" % sample_b: v, "images_per_s_at_B%d" % (2 * sample_b): 2 * sample_b / dt2}
    out = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg2: 128x512 images, 6-conv encoder + 512-d attention LSTM decoder, vocab 500, T=150 teacher-forced "
                               "steps (PADs trained on, as the reference); bounded sample of %d images per step" % sample_b,
                   "same_config": "same shapes/model as the GPU arm; batch is a %d-image sample of the 64 (throughput is linear in "
                                  "batch on the CPU, see linearity)" % sample_b,
                   "linearity": lin},
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": kind,
                         "sample": "B=%d of the B=64 batch, %d timed steps after %d warm-up, torch %s CPU fp32"
                                   % (sample_b, args.steps, args.warmup, torch.__version__)},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def log(*a):
    print("[bench %.1fs]" % (time.time() - T0), *a, file=sys.stderr, flush=True)


def dump_outputs(out_dir, loss):
    """The loss vector train_step returned, as DIR/loss.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    log("wrote %s" % os.path.join(out_dir, "loss.npy"))


T0 = time.time()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--kernels", default=os.environ.get("LO_IMPL", "tc"), help="simt | tc (tcgen05 convs/GEMMs)")
    ap.add_argument("--batch", type=int, default=CFG2["B"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-decode", action="store_true", help="omit the cfg #5 decode probe (N=1 only)")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg4"], help="cfg4 = the row-encoder / two-layer EXTENSION")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss vector of the last timed step as DIR/loss.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs dumps the GPU train step; --impl reference does not run it")
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist
    from latex_ocr_b200 import _lib
    from latex_ocr_b200.img2seq import Img2SeqModel
    from latex_ocr_b200.data import SimpleVocab
    import bench_support as bs

    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    c = dict(CFG2 if args.workload == "cfg2" else CFG4)
    c["B"] = args.batch
    args.warmup = max(args.warmup, 3)

    class Cfg:
        encoder_cnn = "vanilla"
        positional_embeddings = True
        lr_init = 1e-3
        lr_method = "adam"
        # the whole step — for N > 1 including the NCCL all-reduces of the gradient buckets — is captured in ONE CUDA graph
        # (LO_DP_GRAPH=0 falls back to eager launches on the data-parallel path)
        cuda_graph = (not args.no_graph) and (world == 1 or os.environ.get("LO_DP_GRAPH", "1") == "1")
    kernels = args.kernels
    if kernels == "tc" and not bs.tc_ready():
        kernels = "simt"
    if args.workload == "cfg4":
        from latex_ocr_b200.ext import Img2SeqRowModel as ModelCls
    else:
        ModelCls = Img2SeqModel
    torch.manual_seed(1234 + rank)             # initial weights and the decoder's dropout seed
    model = ModelCls(Cfg(), vocab=SimpleVocab(c["V"]), device="cuda:%d" % local, precision=args.precision, impl=kernels)
    model.build_train()
    model.train_mode(True)                     # dropout active, like the reference's training loop
    if world > 1:
        from latex_ocr_b200 import dist as lod
        lod.attach(model)
    img, formula = bs.synthetic_batch(c["B"], c["H"], c["W"], c["V"], c["T"], seed=1234 + rank)
    img_pin, formula_pin = img.to(torch.uint8).pin_memory(), formula.pin_memory()      # uint8 pixels as pad_batch_images yields them
    img_dev, formula_dev = img.cuda(), formula.cuda()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the state every step of the device-resident timing trains (see the module docstring)
    stores = model._stores()
    initial = [{k: getattr(S, k).clone() for k in ("master", "m", "v", "adam_state", "shadow") if getattr(S, k) is not None}
               for S in stores]

    def restore_initial_state():
        for S, snap in zip(stores, initial):
            for k, v in snap.items():
                getattr(S, k).copy_(v)

    log("model built; warm-up")
    # ---- device-resident timing ---------------------------------------------------------------------
    for _ in range(args.warmup):
        restore_initial_state()
        model.train_step(img_dev, formula_dev)
    barrier()
    log("warm-up done; timing")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for a, b in ev:
        restore_initial_state()
        a.record()
        loss = model.train_step(img_dev, formula_dev)
        b.record()
    barrier()
    ms = sum(a.elapsed_time(b) for a, b in ev) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    launches_eager = _lib.launch_count() - l0
    final_loss = float(loss[0].item())
    log("device-resident: %.2f ms/step" % ms)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss)
    # ---- end-to-end timing (pinned host inputs, H2D + loss D2H every step) -----------------------------
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(2):
        model.getLoss(img_pin, formula_pin)
    barrier()
    e0.record()
    for _ in range(args.steps):
        model.getLoss(img_pin, formula_pin)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1) / args.steps
    t = torch.tensor([ms, ms_e2e], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t[0].item(), t[1].item()
    log("e2e: %.2f ms/step" % ms_e2e)
    per_step_launches = bs.launches_per_step(model, img_dev, formula_dev)

    def finish():
        """N > 1: every rank waits here until rank 0 has printed its line, then the process leaves WITHOUT tearing the NCCL
        communicator down — ncclCommDestroy blocks while captured CUDA graphs still hold the communicator's kernels (observed
        as a teardown hang at N=2, run 46); the OS reclaims everything."""
        if world > 1:
            model._graphs.clear()
            torch.cuda.synchronize()
            dist.barrier()
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)

    if rank != 0:
        finish()
        return
    pk = peaks()
    total_imgs = c["B"] * world
    value = total_imgs / (ms / 1e3)
    if args.workload == "cfg4":
        out = {"metric": "formula-images/sec (train step, 160x640 px, seq<=150; row-encoder biLSTM + 2-layer decoder EXTENSION)",
               "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32",
               "data": "synthetic",
               "config": {"workload": "cfg4 (extension, not in the reference): batch %d/GPU, 1x160x640 images, 6-conv encoder + biLSTM(256) over "
                                      "the 18 feature rows + attention LSTM + second LSTM layer, vocab 500, T=150" % c["B"],
                          "global_batch": total_imgs, "parallelism": "dp%d" % world, "kernels": kernels, "cuda_graph": bool(Cfg.cuda_graph),
                          "loss_after": final_loss},
               "e2e": {"value": total_imgs / (ms_e2e / 1e3), "unit": "images/s", "ms_per_step": ms_e2e,
                       "h2d_bytes_per_step": int(img.numel() * 1 + formula.numel() * 8), "d2h_bytes_per_step": 4},
               "gpu_launches": int(per_step_launches * args.steps), "clocks": clocks, "roofline": None}
        print(json.dumps(out), flush=True)
        finish()
        return
    probes = bs.kernel_probes(model, c, pk)
    log("probes done")
    out = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": "cfg2: batch %d/GPU, 1x128x512 images, 6-conv encoder + 512-d attention LSTM decoder, vocab 500, "
                               "T=150 teacher-forced steps (PADs trained on, as the reference)" % c["B"],
                   "global_batch": total_imgs, "parallelism": "dp%d" % world, "kernels": kernels, "cuda_graph": bool(Cfg.cuda_graph),
                   "l2": "per-step working set (>1 GB of feature maps + 114 MB attention stream) exceeds the 126 MB L2; no explicit flush",
                   "loss_after": final_loss},
        "e2e": {"value": total_imgs / (ms_e2e / 1e3), "unit": "images/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(img.numel() * 1 + formula.numel() * 8), "d2h_bytes_per_step": 4,
                "inputs": "uint8 images (pad_batch_images layout) + int64 token ids from pinned host memory"},
        "gpu_launches": int(per_step_launches * args.steps),
        "clocks": clocks,
        "roofline": probes["dominant"],
        "roofline_all": probes["all"],
        "peaks": pk,
    }
    if not args.skip_decode and world == 1:
        try:
            out["decode"] = bs.decode_probe(model, V=c["V"])       # BASELINE.json configs[4]: greedy + beam-5 tokens/s, exact match
        except Exception as e:                                     # the headline line must survive a probe failure
            out["decode"] = {"error": repr(e)[:300]}
        log("decode probe done")
    if not args.skip_cpu_baseline and world == 1:          # reported on rank 0 at N=1 only (the scaling runs stay short)
        out["cpu_baseline"] = bs.cpu_baseline(c)
    print(json.dumps(out), flush=True)
    finish()


if __name__ == "__main__":
    main()
