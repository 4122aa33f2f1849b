"""-m gpu: parity of the CUDA path (through the C ABI and the reference-shaped Python surface) against
  (a) the committed golden fixtures produced by the UNMODIFIED reference (tests/golden, oracle/make_golden.py),
  (b) the CPU oracle restatement on the same seeded inputs.
Tolerances: fp32 mode — loss 1e-3 relative per north_star (we assert 1e-4), gradients 1e-3 of the
gradient's max-abs; bf16 mode — loss 3e-2 relative (stated tolerance), greedy tokens reported as match-rate.
"""
import pytest
import torch

from util import Cfg, build_model, grads_as_reference_layout, load_golden, relerr

pytestmark = pytest.mark.gpu


def _oracle():
    from oracle import ref_model as rm
    return rm


def _case_inputs(rec):
    rm = _oracle()
    c = rec["case"]
    pe, pd = rm.init_params(c["V"], seed=c["pseed"])
    img, formula = rm.synthetic_batch(c["B"], c["H"], c["W"], c["V"], c["tmin"], c["tmax"], seed=c["dseed"])
    return c, pe, pd, img, formula


def _close(got, want, tol, name, floor=2e-8):
    """max-abs error below tol * max|want|, with an absolute floor for gradients that are pure rounding noise
    (e.g. decoder_att.weight when every ReLU mask is constant over the regions)."""
    got, want = got.detach().double().cpu().reshape(-1), want.detach().double().cpu().reshape(-1)
    assert torch.isfinite(got).all(), name
    err = (got - want).abs().max().item()
    assert err <= tol * want.abs().max().item() + floor, (name, err, want.abs().max().item())


def _check_summary(name, got, want, tol):
    if isinstance(want, dict):
        g = got.reshape(-1)
        assert torch.isfinite(g).all(), name
        meanabs = want["abssum"] / g.numel()
        err = (g[:256].double().cpu() - want["head"].double()).abs().max().item()
        assert err <= tol * 5 * max(want["head"].abs().max().item(), meanabs) + 2e-8, (name, err)
        scale = want["abssum"] + 1e-30
        assert abs(g.double().sum().item() - want["sum"]) / scale < tol, name
        assert abs(g.double().abs().sum().item() - want["abssum"]) / scale < tol, name
    else:
        _close(got, want, tol, name)


@pytest.mark.parametrize("name", ["tiny_eval", "tiny_nopos", "cfg1"])
def test_encoder_forward_vs_golden(name):
    rec = load_golden(name)
    c, pe, pd, img, formula = _case_inputs(rec)
    m = build_model(c["V"], pe, pd, "fp32", positional=c["positional"])
    out = m.encoder(img.cuda())
    want = rec["enc_out"]
    if isinstance(want, dict):
        # cfg1 stores a strided sample of the reference output; every element is compared with the CPU oracle, the
        # restatement that tests/test_oracle_pinned.py pins to the reference
        assert tuple(out.shape) == want["shape"]
        s = _sample_of(out, want)
        assert (s - want["sample"].double()).abs().max().item() < 1e-4 * want["sample"].abs().max().item()
        want = _oracle().encoder_forward(pe, img, positional=c["positional"])
    assert out.shape == want.shape
    assert relerr(out, want) < 1e-4


@pytest.mark.parametrize("name", ["tiny_eval", "tiny_nopos", "tiny_train", "cfg1"])
def test_train_step_fp32_vs_golden(name):
    """Loss, decoder outputs, every gradient and a 3-step Adam trajectory against the reference's own run."""
    rm = _oracle()
    rec = load_golden(name)
    c, pe, pd, img, formula = _case_inputs(rec)
    m = build_model(c["V"], pe, pd, "fp32", positional=c["positional"], train=c["train"])
    B, T = c["B"], formula.shape[1] - 1
    traj = []
    for step in range(3):
        mask = None
        if c["train"]:
            torch.manual_seed(rec["mask_seed"] + step)      # reproduces nn.Dropout's CPU draws (make_golden.dropout_masks)
            mask = torch.stack([torch.nn.functional.dropout(torch.ones(B, 512), 0.5, True) for _ in range(T)], dim=1).cuda()
        loss = m._step_body(img.cuda(), formula.cuda(), [T] * B, mask)
        torch.cuda.synchronize()
        traj.append(-loss[0].item())
        if step == 0:
            assert abs(loss[0].item() - rec["loss"]) / abs(rec["loss"]) < 1e-4
            ws = m.decoder._ws[(B, T, rec["alphas"].shape[2])]["t"]
            assert relerr(ws["logits"][:, :, :c["V"]], rec["scores"]) < 1e-4
            assert relerr(ws["alphas"], rec["alphas"]) < 1e-4
            for k, g in grads_as_reference_layout(m.decoder).items():
                if k == "attention.full_att.bias":
                    assert g.abs().max().item() < 1e-6        # exactly 0 here; rounding noise (~1e-9) in the reference
                    continue
                _check_summary("dec." + k, g, rec["grad_dec"][k], 1e-3)
            for k, g in grads_as_reference_layout(m.encoder).items():
                _check_summary("enc." + k, g, rec["grad_enc"][k], 1e-3)
    # Adam turns rounding-level gradient differences on near-zero gradients into +-lr parameter moves, so the
    # trajectory is only loosely pinned after the first update (fp64 vs fp32 CPU runs of the reference equations
    # already differ by 3e-4..6e-4 at step 3): step 1 exact, step 2 tight, step 3 loose.
    ref = rec["get_loss_trajectory"]
    assert abs(traj[0] - ref[0]) / abs(ref[0]) < 1e-4 and abs(traj[1] - ref[1]) / abs(ref[1]) < 5e-4, (traj, ref)
    assert abs(traj[2] - ref[2]) / abs(ref[2]) < 1e-2, (traj, ref)


def test_train_step_fp32_vs_oracle_all_gradients():
    """Full elementwise gradient comparison against the CPU oracle (autograd of the restatement)."""
    rm = _oracle()
    V = 60
    pe, pd = rm.init_params(V, seed=5)
    img, formula = rm.synthetic_batch(3, 40, 72, V, 4, 9, seed=6)
    pe2 = {k: v.clone() for k, v in pe.items()}
    pd2 = {k: v.clone() for k, v in pd.items()}
    neg, ge, gd, aux = rm.train_step(pe2, pd2, img, formula, {}, hoist=False)
    m = build_model(V, pe, pd, "fp32")
    B, T = formula.shape[0], formula.shape[1] - 1
    loss = m._step_body(img.cuda(), formula.cuda(), [T] * B, None)
    torch.cuda.synchronize()
    assert abs(-loss[0].item() - neg) / abs(neg) < 1e-4
    for k, g in grads_as_reference_layout(m.decoder).items():
        if k == "attention.full_att.bias":
            continue
        _close(g, gd[k], 1e-3, k)
    for k, g in grads_as_reference_layout(m.encoder).items():
        _close(g, ge[k], 1e-3, k)
    # parameters after the fused Adam step == oracle Adam
    # (first Adam step = -lr * g/(|g|+eps): only elements whose gradient is at rounding level may differ by up to lr)
    for sd, ref in ((m.decoder.state_dict(), pd2), (m.encoder.state_dict(), pe2)):
        for k, v in sd.items():
            if k == "attention.full_att.bias":
                continue          # gradient is exactly 0 here, rounding noise (1e-9) in the reference -> Adam moves the
                                  # reference's copy by ~lr; the softmax is invariant to this bias, no output depends on it
            d = (v.cpu() - ref[k]).abs()
            assert d.max().item() <= 2.02e-3, k      # a sign flip of a rounding-level gradient moves a weight by 2*lr
            assert (d > 5e-5).float().mean().item() < 1e-3, k


def test_decoder_forward_api_ragged_lengths():
    """DecoderWithAttention.forward with genuinely different caption lengths (shrinking batch, :308)."""
    rm = _oracle()
    V = 50
    pe, pd = rm.init_params(V, seed=8)
    img, formula = rm.synthetic_batch(4, 32, 64, V, 3, 8, seed=9)
    lengths = torch.tensor([[9], [4], [7], [4]])
    enc = rm.encoder_forward(pe, img)
    preds, caps, dl, alphas, si = rm.decoder_forward(pd, enc, formula, lengths)
    m = build_model(V, pe, pd, "fp32")
    m.train_mode(False)
    p2, c2, dl2, a2, si2 = m.decoder(enc.cuda(), formula.cuda(), lengths)
    assert dl2 == dl and torch.equal(si2.cpu(), si) and torch.equal(c2.cpu(), caps)
    assert relerr(p2, preds) < 1e-4
    assert relerr(a2, alphas) < 1e-4


def test_attention_module_api():
    rm = _oracle()
    from latex_ocr_b200.decoder import Attention
    torch.manual_seed(3)
    att = Attention(512, 512, 512, precision="fp32")
    enc = torch.randn(5, 44, 512)
    h = torch.randn(5, 512)
    p = {"attention." + k: v.detach().cpu() for k, v in att.state_dict().items()}
    ctx, alpha = rm.attention_forward(p, enc, h)
    c2, a2 = att(enc.cuda(), h.cuda())
    assert relerr(c2, ctx) < 1e-4 and relerr(a2, alpha) < 1e-4
    with pytest.raises(Exception):
        att(enc, h)          # CPU tensors: no fallback


def _sample_of(t, want):
    """The strided sample make_golden.strided_sample took of the reference tensor, taken of ours."""
    flat = t.detach().reshape(-1)
    n = flat.numel()
    idx = (torch.arange(want["sample"].numel(), dtype=torch.int64, device=flat.device) * want["sample_stride"]) % n
    return flat[idx].double().cpu()


def _sample_norm_err(t, want):
    s = _sample_of(t, want)
    w = want["sample"].double()
    return ((s - w).norm() / (w.norm() + 1e-30)).item()


def _dropout_mask_replay(seed, B, T):
    torch.manual_seed(seed)          # reproduces nn.Dropout's CPU draws of the reference run (make_golden.dropout_masks)
    return torch.stack([torch.nn.functional.dropout(torch.ones(B, 512), 0.5, True) for _ in range(T)], dim=1)


def test_cfg2_shape_fp32_vs_golden():
    """BASELINE.json configs[1] shapes (1x128x512 -> R=868, T=150, V=500, dropout on) on a B=8 sample, fp32 CUDA-core path vs the
    UNMODIFIED reference's run (tests/golden/cfg2.pt, summaries): loss 1e-4, every gradient 1e-3, outputs 1e-4."""
    rec = load_golden("cfg2")
    c, pe, pd, img, formula = _case_inputs(rec)
    B, T = c["B"], formula.shape[1] - 1
    assert T == 150 and rec["alphas"]["shape"] == (B, T, 868)
    m = build_model(c["V"], pe, pd, "fp32", train=True)
    mask = _dropout_mask_replay(rec["mask_seed"], B, T).cuda()
    loss = m._step_body(img.cuda(), formula.cuda(), [T] * B, mask)
    torch.cuda.synchronize()
    assert abs(loss[0].item() - rec["loss"]) / abs(rec["loss"]) < 1e-4, (loss[0].item(), rec["loss"])
    ws = m.decoder._ws_for(B, T, 868)["t"]
    for name, got in (("scores", ws["logits"][:, :, :c["V"]].contiguous()), ("alphas", ws["alphas"])):
        want = rec[name]
        s = _sample_of(got, want)
        err = (s - want["sample"].double()).abs().max().item() / want["sample"].abs().max().item()
        print("cfg2 fp32", name, "max-abs sample error (rel. to max) %.2e" % err)
        assert err < 1e-4, (name, err)
    bad = []
    for mod, key in ((m.decoder, "grad_dec"), (m.encoder, "grad_enc")):
        for k, g in grads_as_reference_layout(mod).items():
            if k == "attention.full_att.bias":
                continue
            want = rec[key][k]
            if isinstance(want, dict):
                err = _sample_norm_err(g, want)
                sums = abs(g.double().sum().item() - want["sum"]) / (want["abssum"] + 1e-30)
            else:
                err = ((g.double() - want.double()).norm() / (want.double().norm() + 1e-30)).item()
                sums = 0.0
            print("cfg2 fp32 grad %-36s norm err %.2e sum err %.2e" % (k, err, sums))
            if not (err < 1e-3 and sums < 1e-3):
                bad.append((k, err, sums))
    assert not bad, bad


def test_cfg2_shape_bf16_tc_vs_golden():
    """Same shapes on the bf16 / tcgen05 + mma.sync path the bench runs.  STATED bf16 tolerances (bf16 storage of feature maps,
    att1/enc and weight shadows, fp32 accumulation, 150 recurrent steps): loss 2e-3 relative; per-tensor relative gradient NORM
    error 3e-2 (measured on the golden's strided samples; small tensors in full)."""
    rec = load_golden("cfg2")
    c, pe, pd, img, formula = _case_inputs(rec)
    B, T = c["B"], formula.shape[1] - 1
    m = build_model(c["V"], pe, pd, "bf16", train=True, impl="tc")
    mask = _dropout_mask_replay(rec["mask_seed"], B, T).cuda()
    loss = m._step_body(img.cuda(), formula.cuda(), [T] * B, mask)
    torch.cuda.synchronize()
    lerr = abs(loss[0].item() - rec["loss"]) / abs(rec["loss"])
    print("cfg2 bf16/tc loss %.6f (reference %.6f) rel.err %.2e" % (loss[0].item(), rec["loss"], lerr))
    assert lerr < 2e-3
    bad = []
    for mod, key in ((m.decoder, "grad_dec"), (m.encoder, "grad_enc")):
        for k, g in grads_as_reference_layout(mod).items():
            if k == "attention.full_att.bias":
                continue
            want = rec[key][k]
            err = _sample_norm_err(g, want) if isinstance(want, dict) else \
                ((g.double() - want.double()).norm() / (want.double().norm() + 1e-30)).item()
            print("cfg2 bf16 grad %-36s norm err %.2e" % (k, err))
            if not err < 3e-2:
                bad.append((k, err))
    assert not bad, bad


def test_bf16_mode_loss_tolerance_and_graph_replay():
    rm = _oracle()
    rec = load_golden("cfg1")
    c, pe, pd, img, formula = _case_inputs(rec)
    B, T = c["B"], formula.shape[1] - 1
    for impl in ("simt", "tc"):
        m = build_model(c["V"], pe, pd, "bf16", impl=impl)
        loss = m._step_body(img.cuda(), formula.cuda(), [T] * B, None)
        torch.cuda.synchronize()
        err = abs(loss[0].item() - rec["loss"]) / abs(rec["loss"])
        print("cfg1 bf16/%s loss rel.err %.2e" % (impl, err))
        assert err < 1e-3                                                   # stated bf16 tolerance (observed ~5e-5)
    # CUDA-graph replay gives the same numbers as eager launches
    m1 = build_model(c["V"], pe, pd, "fp32")
    m2 = build_model(c["V"], pe, pd, "fp32", graph=True)
    l1 = [m1.train_step(img, formula)[0].item() for _ in range(3)]
    l2 = [m2.train_step(img, formula)[0].item() for _ in range(3)]
    # same launches, same order; split-K / wgrad fp32 atomics make gradients differ at rounding level between any
    # two runs, which Adam amplifies from the second update on (see test_train_step_fp32_vs_golden)
    for (a, b), tol in zip(zip(l1, l2), (1e-6, 1e-5, 1e-3)):
        assert abs(a - b) / abs(a) < tol, (l1, l2)


def test_getloss_surface_and_state_dict_roundtrip(tmp_path):
    rm = _oracle()
    V = 40
    pe, pd = rm.init_params(V, seed=2)
    img, formula = rm.synthetic_batch(2, 32, 64, V, 3, 5, seed=3)
    m = build_model(V, pe, pd, "fp32")
    v = m.getLoss(img, formula, lr=123.0, dropout=0.0)
    assert isinstance(v, float) and v < 0
    path = m.save(str(tmp_path / "m.pt"))
    m2 = build_model(V, pe, pd, "fp32")
    m2.restore(path)
    for k, t in m.decoder.state_dict().items():
        assert torch.equal(t, m2.decoder.state_dict()[k])
    assert set(m.encoder.state_dict().keys()) == set(pe.keys())
    assert set(m.decoder.state_dict().keys()) == set(pd.keys())


def test_attention_kernel_versions_agree_on_a_full_step():
    """Register-streaming (att_pipe=0) and TMA-pipelined (att_pipe=1) attention kernels give the same loss/gradients."""
    from latex_ocr_b200 import _lib
    rm = _oracle()
    V = 60
    pe, pd = rm.init_params(V, seed=15)
    img, formula = rm.synthetic_batch(3, 40, 72, V, 4, 9, seed=16)
    B, T = formula.shape[0], formula.shape[1] - 1
    res = {}
    try:
        for pipe in (0, 1):
            _lib.set_option("att_pipe", pipe)
            m = build_model(V, pe, pd, "fp32")
            loss = m._step_body(img.cuda(), formula.cuda(), [T] * B, None)
            torch.cuda.synchronize()
            res[pipe] = (loss[0].item(), m.decoder.store.grad.clone(), m.encoder.store.grad.clone())
    finally:
        _lib.set_option("att_pipe", 1)
    assert abs(res[0][0] - res[1][0]) / abs(res[0][0]) < 1e-6
    for i in (1, 2):
        assert (res[0][i] - res[1][i]).abs().max().item() <= 1e-4 * res[0][i].abs().max().item() + 1e-8


def test_uint8_image_upload_equals_float_path():
    """pad_batch_images yields uint8; conv1 can take it directly (4x less H2D).  0..255 are exact in fp32 -> same loss."""
    rm = _oracle()
    V = 40
    pe, pd = rm.init_params(V, seed=2)
    img, formula = rm.synthetic_batch(2, 32, 64, V, 3, 5, seed=3)
    m1 = build_model(V, pe, pd, "fp32")
    m2 = build_model(V, pe, pd, "fp32")
    a = m1.getLoss(img, formula)
    b = m2.getLoss(img.to(torch.uint8), formula)
    assert a == b
    g1, g2 = m1.encoder.store.grad, m2.encoder.store.grad          # (wgrad split-K atomics: equal up to summation order)
    assert (g1 - g2).abs().max().item() <= 1e-5 * g1.abs().max().item()


def test_cnn_variant_encoder_vs_golden():
    """encoder_cnn='cnn' (seq2seq_torch.py:58-86: Conv2d(512,512,(2,4),stride 2,padding 1) instead of the two asymmetric pools):
    output and the gradients of sum(out * G) against the reference's own run (tests/golden/cnn_variant.pt); fp32 tight, and the
    bf16/tcgen05 path (im2col + tensor-core GEMMs) against the fp32 one."""
    from latex_ocr_b200.encoder import EncoderCNN
    from util import Cfg
    rm = _oracle()
    rec = load_golden("cnn_variant")
    c = rec["case"]
    pe, _ = rm.init_params(c["V"], seed=c["pseed"], encoder_cnn="cnn")
    img, _ = rm.synthetic_batch(c["B"], c["H"], c["W"], c["V"], 3, 4, seed=c["dseed"])
    G = torch.randn(rec["enc_out"].shape, generator=torch.Generator().manual_seed(c["gseed"]))
    grads = {}
    for precision, impl, tol in (("fp32", "simt", 1e-4), ("bf16", "tc", 3e-2)):
        enc = EncoderCNN(Cfg(encoder_cnn="cnn"), device="cuda", precision=precision, impl=impl)
        assert set(enc.state_dict()) == set(pe)
        enc.load_state_dict(pe)
        out = enc.forward_raw(img.cuda(), need_grad=True).float()
        assert out.shape == rec["enc_out"].shape
        assert relerr(out, rec["enc_out"]) < tol
        enc.backward_raw(tuple(img.shape), G.cuda().contiguous())
        torch.cuda.synchronize()
        grads[precision] = {k: p.grad.detach().float().cpu().clone() for k, p in enc.named_parameters()}
    # the random upstream gradient G makes single ReLU / pool-argmax flips (fp32 summation order) visible in the sums: big tensors
    # through their summaries at 5e-3, small ones (biases) norm-wise at 1e-2
    for k, g in grads["fp32"].items():
        want = rec["grad_enc"][k]
        if isinstance(want, dict):
            _check_summary(k, g, want, 5e-3)
        else:
            err = ((g.double() - want.double()).norm() / want.double().norm()).item()
            print("cnn variant fp32", k, "rel. norm error %.2e" % err)
            assert err < 1e-2, (k, err)
        b = grads["bf16"][k]
        assert ((b - g).norm() / g.norm()).item() < 0.15, k      # bf16 storage through 7 layers + mask flips: norm-wise 15 %


def test_in_kernel_philox_dropout_equals_injected_host_mirror_mask():
    """has_dropout=2 draws the inverted-dropout multipliers inside lstm_pw_fwd/bwd (Philox4x32-10, regenerated in the backward);
    the numpy mirror (latex_ocr_b200/philox.py, pinned to the Random123 known-answer vectors in tests/test_host_and_abi.py)
    reproduces them, and feeding that mask through the injected path gives the same loss and gradients."""
    from latex_ocr_b200 import philox
    rm = _oracle()
    V = 60
    pe, pd = rm.init_params(V, seed=5)
    img, formula = rm.synthetic_batch(3, 40, 72, V, 4, 9, seed=6)
    B, T = formula.shape[0], formula.shape[1] - 1
    m1 = build_model(V, pe, pd, "fp32", train=True)
    hw = m1.encoder.out_hw(40, 72)
    R = hw[0] * hw[1]
    m1.decoder.seed_dropout(0x1234567887654321 & 0x7FFFFFFFFFFFFFFF, call=3)
    seed = int(m1.decoder.dropout_state[0].item())
    l1 = m1._step_body(img.cuda(), formula.cuda(), [T] * B, "philox")
    torch.cuda.synchronize()
    assert int(m1.decoder.dropout_state[1].item()) == 4                      # advanced once by lo_decoder_backward
    mask = torch.from_numpy(philox.dropout_multipliers(seed, 3, B, T, 512, 0.5)).cuda()
    assert 0.4 < (mask == 0).float().mean().item() < 0.6
    m2 = build_model(V, pe, pd, "fp32", train=True)
    l2 = m2._step_body(img.cuda(), formula.cuda(), [T] * B, mask)
    torch.cuda.synchronize()
    assert l1[0].item() == l2[0].item()
    assert torch.equal(m1.decoder._ws_for(B, T, R)["t"]["hd"], m2.decoder._ws_for(B, T, R)["t"]["hd"])
    for a, b in ((m1.decoder.store.grad, m2.decoder.store.grad), (m1.encoder.store.grad, m2.encoder.store.grad)):
        assert (a - b).abs().max().item() <= 1e-5 * b.abs().max().item()    # split-K atomics: equal up to summation order
    # a second step draws a different mask
    hd1 = m1.decoder._ws_for(B, T, R)["t"]["hd"].clone()
    m1._step_body(img.cuda(), formula.cuda(), [T] * B, "philox")
    torch.cuda.synchronize()
    assert ((hd1 == 0) != (m1.decoder._ws_for(B, T, R)["t"]["hd"] == 0)).any()
