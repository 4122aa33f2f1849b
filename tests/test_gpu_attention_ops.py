"""-m gpu: the stand-alone attention entry points (lo_attention_forward, lo_attention_forward_mask, lo_attention_backward) op by op
against float64 autograd of the same step (Attention.forward seq2seq_torch.py:186-190 + the gate of :311-312), on every kernel the
backward dispatcher (bwd_launch_a, latex_ocr_b200/csrc/lo_attention.cu) can pick:
  mma   attention_bwd_mma_kernel   bf16, C = 512, mask bits given, att_bwd_mma = 1, rows per split <= 2048
  mask  attention_bwd_mask_kernel  every other case with mask bits
  pipe  attention_bwd_pipe_kernel  no mask bits: att1 is read again
each in its cluster (DSMEM combine) and ticket-counter form.  Every case id starts with the kernel it lands on.

Inputs and outputs are laid out as the decoder lays them out: alpha / de at step t of [B][T][R], att2 | gate in one out1 row,
datt2 | dgp in one dcat row, d gctx rows wider than C.  Every byte a call must not write holds a NaN guard, and so does every input
element it must not read.

Tolerances follow from the arithmetic.  Accumulation is fp32; the tensor-core kernel splits its fp32 operands into bf16 hi + lo
halves (16 mantissa bits).  So each element is bounded by K * 2^-16 times the sum of the magnitudes of the terms it adds, e.g.
|err(datt2_a)| <= |wf_a| sum_r (K 2^-16 |de_r| + bound(de_r)); a relative bound on the whole tensor would not do, since
sum_r de_r = 0 makes datt2 a cancelling sum."""
import math

import numpy as np
import pytest
import torch

from test_attention_layouts import _pack_pair_layout

K = 2.0                      # fixed factor of the per-element bounds
EPS16 = 2.0 ** -16           # what the bf16 hi + lo split keeps
T_STEPS, T_AT = 3, 1         # the step buffers hold T_STEPS steps; the calls work on step T_AT
_OPTS = ("att_pipe", "att_nsplit", "att_cluster", "att_bwd_mma")


def decode_mask_bits(buf, B, R, A):
    """[B][Rp][A/8] bytes of lo_attention_forward_mask -> bool [B][R][A], by the layout documented in include/latex_ocr_b200.h:
    bit 7 - a % 8 of the byte of (r, a / 8), which lives at (r / 2) * 2 * (A/8) + (a / 8) * 2 + (r & 1) within image b."""
    MB, Rp = A // 8, (R + 1) & ~1
    x = np.asarray(buf, dtype=np.uint8)[:B * Rp * MB].reshape(B, Rp // 2, MB, 2)      # [b][r / 2][a / 8][r & 1]
    x = x.transpose(0, 1, 3, 2).reshape(B, Rp, MB)
    return np.unpackbits(x, axis=-1, bitorder="big")[:, :R].astype(bool)


def test_decode_mask_bits_inverts_pair_layout():
    rng = np.random.RandomState(3)
    for R in (1, 2, 5, 16, 17):
        for A in (256, 512, 1024):
            bits = rng.rand(3, R, A) < 0.5
            packed = np.concatenate([_pack_pair_layout(bits[b].astype(np.uint8)) for b in range(3)])
            assert (decode_mask_bits(packed, 3, R, A) == bits).all(), (R, A)


# ---- which kernel a backward call lands on: mirrors att_pipe_splits / att_rows_per_split / use_cluster / bwd_launch_a
def _splits(B, nsplit, cluster):
    if nsplit > 0:
        return min(nsplit, 16)
    s = min(max((148 * 2) // B, 1), 16)
    return min(s, 8) if cluster else s


def _rows_per_split(R, ns):
    return ((R + ns - 1) // ns + 1) & ~1


def _use_cluster(ns, R, cluster):
    return bool(cluster) and 2 <= ns <= 8 and (R + ns - 1) // ns * 4 <= 16 * 1024


def bwd_kernel(dt, C, B, R, mask, mma, nsplit, cluster):
    ns = _splits(B, nsplit, cluster)
    if mask and dt == "bf16" and C == 512 and mma and _rows_per_split(R, ns) <= 2048:
        k = "mma"
    else:
        k = "mask" if mask else "pipe"
    return "%s_%s%d" % (k, "cluster" if _use_cluster(ns, R, cluster) else "ticket", ns)


def test_dispatch_helper_reaches_every_branch():
    """The backward matrix below must reach every kernel in both combine forms, and the > 2048-rows-per-split fallback."""
    names = {c[0].split("-")[0] for c in _BWD_CASES}
    for k in ("mma", "mask", "pipe"):
        assert any(n.startswith(k + "_cluster") for n in names), k
        assert any(n.startswith(k + "_ticket") for n in names), k
    fb = [c for c in _BWD_CASES if c[1]["dt"] == "bf16" and c[1]["C"] == 512 and c[1]["mask"] and c[1]["mma"]
          and c[0].startswith("mask")]
    assert any(c[1]["B"] == 150 and c[1]["R"] == 2100 for c in fb)


# ---- backward case matrix: (id, dict)
def _case(dt, C, B, R, mask, mma, nsplit, cluster, i, **kw):
    d = dict(dt=dt, C=C, B=B, R=R, mask=mask, mma=mma, nsplit=nsplit, cluster=cluster,
             gate=kw.pop("gate", i % 2 == 0), dreg=kw.pop("dreg", (i // 2) % 2 == 0), **kw)
    tags = [t for t in ("sreg_free", "nodgp", "chained", "zeros") if d.get(t)]
    cid = "-".join([bwd_kernel(dt, C, B, R, mask, mma, nsplit, cluster), dt, "C%d" % C, "B%d" % B, "R%d" % R,
                    "ns%d" % nsplit, "cl%d" % cluster, "mma%d" % mma, "gate%d" % d["gate"], "dreg%d" % d["dreg"]] + tags)
    return cid, d


def _bwd_matrix():
    fams = [("bf16", 512, True, 1), ("bf16", 512, True, 0), ("fp32", 512, True, 1), ("bf16", 512, False, 1), ("fp32", 512, False, 1)]
    out, i = [], 0
    for dt, C, mask, mma in fams:
        for R in (1, 2, 5, 17, 37, 180, 868):
            for ns, cl in ((0, 1), (1, 1), (2, 1), (3, 0), (8, 1), (8, 0), (16, 1)):
                out.append(_case(dt, C, 3, R, mask, mma, ns, cl, i))
                i += 1
        for B, R, ns, cl in ((1, 868, 0, 1), (1, 868, 0, 0), (64, 180, 0, 1), (64, 180, 0, 0), (150, 868, 0, 1), (150, 37, 0, 1)):
            out.append(_case(dt, C, B, R, mask, mma, ns, cl, i))
            i += 1
        out.append(_case(dt, C, 3, 37, mask, mma, 0, 1, i, dreg=True, sreg_free=True))
        out.append(_case(dt, C, 5, 17, mask, mma, 3, 0, i, gate=False, nodgp=True))
        out.append(_case(dt, C, 3, 37, mask, mma, 0, 1, i, chained=True))
        out.append(_case(dt, C, 64, 868, mask, mma, 0, 1, i + 1, chained=True))
        for ns, cl in ((0, 1), (3, 0), (1, 1)):
            out.append(_case(dt, C, 3, 37, mask, mma, ns, cl, i, zeros=True))
        i += 1
    for C in (256, 1024):
        for dt, mask, mma in (("bf16", True, 1), ("fp32", True, 1), ("bf16", False, 1), ("fp32", False, 1)):
            for R in (5, 37):
                for ns, cl in ((0, 1), (16, 1), (3, 0)):
                    out.append(_case(dt, C, 3, R, mask, mma, ns, cl, i))
                    i += 1
            out.append(_case(dt, C, 3, 37, mask, mma, 0, 1, i, zeros=True))
    # more than 2048 rows per split: the tensor-core kernel stages alpha / d reg of a split in shared memory and hands over
    out.append(_case("bf16", 512, 150, 2100, True, 1, 0, 1, 0))
    out.append(_case("bf16", 512, 2, 4200, True, 1, 2, 1, 1))
    return out


_BWD_CASES = _bwd_matrix()


# ---- GPU helpers
@pytest.fixture
def lib():
    from latex_ocr_b200 import _lib
    L = _lib.lib()
    saved = {k: L.lo_get_option(k.encode()) for k in _OPTS}
    assert all(v >= 0 for v in saved.values()), saved
    try:
        _lib.set_option("att_pipe", 1)
        yield _lib, L
    finally:
        for k, v in saved.items():
            _lib.set_option(k, v)


def _nan(*shape):
    return torch.full(shape, float("nan"), device="cuda")


def _bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t.contiguous().view(torch.uint8)


def _same_bits(a, b):
    return torch.equal(_bits(a), _bits(b))


def _plant_cancellations(att1, att2, gen):
    """att2_a = -att1_ra exactly for a sprinkling of (r, a), two whole columns included, and signed-zero pairs in two more columns."""
    B, R, A = att1.shape
    cols = torch.randperm(A, generator=gen, device="cuda")[:26]
    z = cols[24:]
    cols = cols[:24]
    a2 = att2[:, cols].to(att1.dtype)                       # representable in att1's storage type
    att2[:, cols] = a2.float()
    hit = torch.rand(B, R, len(cols), generator=gen, device="cuda") < 0.3
    hit[:, :, :2] = True
    att1[:, :, cols] = torch.where(hit, (-a2)[:, None, :].expand(B, R, len(cols)), att1[:, :, cols])
    sgn = torch.zeros(R, device="cuda")
    sgn[1::2] = -0.0
    att1[:, :, z] = sgn[None, :, None].expand(B, R, 2).to(att1.dtype)
    att2[:, z[0]] = 0.0
    att2[:, z[1]] = -0.0


class Step:
    """One attention step's buffers in the decoder's layout (fp32 state, `dt` storage for att1 / enc)."""

    def __init__(self, dt, B, R, C, seed, gate=True, zeros=False):
        A = C
        gen = torch.Generator(device="cuda").manual_seed(seed)
        tdt = torch.bfloat16 if dt == "bf16" else torch.float32
        rn = lambda *shape: torch.randn(*shape, generator=gen, device="cuda")
        self.B, self.R, self.A, self.C, self.tdt = B, R, A, C, tdt
        self.att1 = rn(B, R, A).to(tdt)
        self.enc = rn(B, R, C).to(tdt)
        att2 = rn(B, A)
        if zeros:
            _plant_cancellations(self.att1, att2, gen)
        self.o1s = A + C + 64
        self.out1 = _nan(B, self.o1s)                         # att2 | gate (pre-activation before the forward) | guard
        self.out1[:, :A] = att2
        self.gate_pre = rn(B, C) if gate else None
        if gate:
            self.out1[:, A:A + C] = self.gate_pre
        self.wf = rn(A) * (2.0 / math.sqrt(A))
        self.dgs = C + 32
        self.dgctx = _nan(B, self.dgs)
        self.dgctx[:, :C] = rn(B, C)
        self.dreg_v = rn(B, R) * 3.0
        self.work = torch.zeros(int(self._L().lo_attention_workspace_bytes(B, C)), dtype=torch.uint8, device="cuda")

    @staticmethod
    def _L():
        from latex_ocr_b200 import _lib
        return _lib.lib()

    @property
    def att2(self):
        return self.out1[:, :self.A]

    @property
    def gate(self):
        return self.out1[:, self.A:self.A + self.C] if self.gate_pre is not None else None

    def forward(self, _lib, L, mask=True, fill=0xA5):
        """Runs lo_attention_forward[_mask] on this step; returns (alpha_buf, ctx, gctx, mask_buf); writes the gate into out1.
        The mask buffer starts as `fill` bytes and has 256 guard bytes at its end."""
        B, R, A, C = self.B, self.R, self.A, self.C
        alpha = _nan(B, T_STEPS, R)
        ctx, gctx = _nan(B, C), _nan(B, C)
        MB, Rp = A // 8, (R + 1) & ~1
        mbuf = torch.full((B * Rp * MB + 256,), fill, dtype=torch.uint8, device="cuda") if mask else None
        g = self.gate_pre is not None
        args = [_lib.ptr(self.att1), _lib.ptr(self.enc), _lib.dt_of(self.att1), _lib.ptr(self.out1), self.o1s, _lib.ptr(self.wf),
                _lib.ptr(alpha[:, T_AT]), T_STEPS * R, _lib.ptr(ctx), _lib.ptr(self.gate) if g else None, self.o1s,
                _lib.ptr(gctx) if g else None]
        if mask:
            _lib.check(L.lo_attention_forward_mask(*args, _lib.ptr(mbuf), B, R, A, C, _lib.ptr(self.work), _lib.stream_ptr()))
        else:
            _lib.check(L.lo_attention_forward(*args, B, R, A, C, _lib.ptr(self.work), _lib.stream_ptr()))
        torch.cuda.synchronize()
        return alpha, ctx, gctx, mbuf


def _reference(s, dreg):
    """float64 autograd of L = <d gctx, gctx> + <d reg, alpha> on the exact values the kernels see."""
    a1, en = s.att1.double(), s.enc.double()
    a2 = s.att2.double().clone().requires_grad_()
    w = s.wf.double().clone().requires_grad_()
    pre = a1 + a2[:, None, :]
    e = torch.relu(pre) @ w
    e.retain_grad()
    al = torch.softmax(e, dim=1)
    ctx = torch.einsum("br,brc->bc", al, en)
    ctx.retain_grad()
    gp = s.gate_pre.double().clone().requires_grad_() if s.gate_pre is not None else None
    gate = torch.sigmoid(gp) if gp is not None else None
    gctx = gate * ctx if gate is not None else ctx
    loss = (s.dgctx[:, :s.C].double() * gctx).sum()
    if dreg is not None:
        loss = loss + (dreg.double() * al).sum()
    loss.backward()
    return dict(pre=pre.detach(), e=e.detach(), alpha=al.detach(), ctx=ctx.detach(), gate=None if gate is None else gate.detach(),
                de=e.grad, datt2=a2.grad, dgp=None if gp is None else gp.grad, dctx=ctx.grad, dwf=w.grad)


def _check(name, got, want, bound, ratios):
    err = (got.double() - want).abs()
    r = (err / bound.clamp_min(1e-300)).max().item()
    ratios[name] = max(ratios.get(name, 0.0), r)
    bad = ~(err <= bound)
    assert not bad.any(), "%s: %d elements out of bound, worst ratio %.3g, first at %s" % (
        name, int(bad.sum()), r, tuple(int(i) for i in bad.nonzero()[0]))


# ---- forward
_FWD_CASES = []
for _dt in ("fp32", "bf16"):
    for _C in (256, 512, 1024):
        for _B, _R, _ns, _cl in ((1, 1, 0, 1), (3, 37, 0, 1), (5, 17, 16, 1), (64, 180, 3, 0), (150, 868, 0, 1)):
            _FWD_CASES.append(pytest.param(_dt, _C, _B, _R, _ns, _cl, False, id="%s-C%d-B%d-R%d-ns%d-cl%d" % (_dt, _C, _B, _R, _ns, _cl)))
        _FWD_CASES.append(pytest.param(_dt, _C, 3, 37, 0, 1, True, id="%s-C%d-B3-R37-ns0-cl1-zeros" % (_dt, _C)))
        _FWD_CASES.append(pytest.param(_dt, _C, 4, 5, 8, 0, True, id="%s-C%d-B4-R5-ns8-cl0-zeros" % (_dt, _C)))


@pytest.mark.gpu
@pytest.mark.parametrize("dt,C,B,R,nsplit,cluster,zeros", _FWD_CASES)
def test_forward_mask_bits_and_outputs(lib, dt, C, B, R, nsplit, cluster, zeros):
    _lib, L = lib
    _lib.set_option("att_nsplit", nsplit)
    _lib.set_option("att_cluster", cluster)
    s = Step(dt, B, R, C, seed=1000 + B * 7 + R + C, zeros=zeros)
    out1_0 = s.out1.clone()
    ref = _reference(s, None)
    alpha, ctx, gctx, mbuf = s.forward(_lib, L, mask=True)
    A, MB, Rp = s.A, s.A // 8, (R + 1) & ~1
    # mask bits, bit for bit, against the fp32 comparison the header states (exact: the fp32 sum has the sign of the exact sum)
    want = (s.att1.float() + s.att2[:, None, :] > 0).cpu().numpy()
    got = decode_mask_bits(mbuf.cpu().numpy(), B, R, A)
    assert (got == want).all(), "mask bits differ at %d elements, first %s" % ((got != want).sum(), np.argwhere(got != want)[0])
    assert (mbuf[B * Rp * MB:] == 0xA5).all(), "bytes past [B][Rp][A/8] written"
    # outputs: bounds from the fp32 score sums e_r = sum_a wf_a relu(pre_ra)
    pre = ref["pre"]
    be = K * EPS16 * (torch.relu(pre) * s.wf.double().abs()).sum(-1)
    al = ref["alpha"]
    bal = al * (be + (al * be).sum(1, keepdim=True)) + 2.0 ** -22 * al
    ratios = {}
    _check("alpha", alpha[:, T_AT], al, bal, ratios)
    en = s.enc.double()
    bctx = torch.einsum("br,brc->bc", bal, en.abs()) + K * EPS16 * torch.einsum("br,brc->bc", al, en.abs())
    _check("ctx", ctx, ref["ctx"], bctx, ratios)
    g = ref["gate"]
    _check("gate", s.gate, g, 2.0 ** -21 * g, ratios)
    _check("gctx", gctx, g * ref["ctx"], g * bctx + 2.0 ** -21 * (g * ref["ctx"]).abs(), ratios)
    # nothing outside step T_AT of alpha and outside [att2 | gate] of out1 is touched
    keep = torch.ones(T_STEPS, dtype=torch.bool, device="cuda")
    keep[T_AT] = False
    assert alpha[:, keep].isnan().all()
    assert _same_bits(s.out1[:, :A], out1_0[:, :A]) and _same_bits(s.out1[:, A + C:], out1_0[:, A + C:])
    print("RATIO forward %s-C%d-B%d-R%d %s" % (dt, C, B, R, " ".join("%s=%.3g" % kv for kv in ratios.items())))
    # the mask-free forward computes the same scores: same outputs bit for bit
    s.out1.copy_(out1_0)
    alpha2, ctx2, gctx2, _ = s.forward(_lib, L, mask=False)
    assert _same_bits(alpha2, alpha) and _same_bits(ctx2, ctx) and _same_bits(gctx2, gctx)


# ---- backward
def _backward(s, _lib, L, alpha, ctx, dreg_buf, sreg_buf, mask, dwf, nodgp=False):
    B, R, A, C = s.B, s.R, s.A, s.C
    de = _nan(B, T_STEPS, R)
    dcat = _nan(B, A + C + 64)
    dctx = None if nodgp else _nan(B * C + 64)
    g = s.gate
    _lib.check(L.lo_attention_backward(
        _lib.ptr(s.att1), _lib.ptr(s.enc), _lib.dt_of(s.att1), _lib.ptr(s.out1), _lib.ptr(g) if g is not None else None, s.o1s,
        _lib.ptr(s.wf), _lib.ptr(alpha[:, T_AT]), T_STEPS * R, _lib.ptr(ctx), _lib.ptr(s.dgctx), s.dgs,
        _lib.ptr(dreg_buf), R + 4, _lib.ptr(sreg_buf[:, T_AT]) if sreg_buf is not None else None, T_STEPS,
        _lib.ptr(de[:, T_AT]), _lib.ptr(dcat), None if nodgp else _lib.ptr(dcat[:, A:]), dcat.stride(0), _lib.ptr(dctx),
        _lib.ptr(dwf), _lib.ptr(mask), B, R, A, C, _lib.ptr(s.work), _lib.stream_ptr()))
    torch.cuda.synchronize()
    return de, dcat, dctx


@pytest.mark.gpu
@pytest.mark.parametrize("cid,cfg", _BWD_CASES, ids=[c[0] for c in _BWD_CASES])
def test_backward_matches_autograd(lib, cid, cfg):
    _lib, L = lib
    dt, C, B, R = cfg["dt"], cfg["C"], cfg["B"], cfg["R"]
    _lib.set_option("att_nsplit", cfg["nsplit"])
    _lib.set_option("att_cluster", cfg["cluster"])
    _lib.set_option("att_bwd_mma", cfg["mma"])
    s = Step(dt, B, R, C, seed=B * 131 + R * 7 + C + cfg["nsplit"], gate=cfg["gate"], zeros=cfg.get("zeros", False))
    A = s.A
    ref = _reference(s, s.dreg_v if cfg["dreg"] else None)
    # forward: the mask bits (and, chained, alpha / ctx / gate) come from the forward kernel itself.  Its buffer starts all ones, and
    # the forward leaves the padding row of an odd R alone: the backward must ignore those set bits.
    mask = None
    if cfg["mask"] or cfg.get("chained"):
        fwd = s.forward(_lib, L, mask=cfg["mask"], fill=0xFF)
        mask = fwd[3]
    if cfg.get("chained"):
        alpha, ctx = fwd[0], fwd[1]
    else:
        alpha = _nan(B, T_STEPS, R)
        alpha[:, T_AT] = ref["alpha"].float()
        ctx = ref["ctx"].float()
        if s.gate is not None:
            s.out1[:, A:A + C] = ref["gate"].float()
    dreg_buf = sreg_buf = None
    al32 = alpha[:, T_AT].double()
    if cfg["dreg"]:
        dreg_buf = _nan(B, R + 4)
        dreg_buf[:, :R] = s.dreg_v
        sreg_buf = _nan(B, T_STEPS)
        gen = torch.Generator(device="cuda").manual_seed(R)
        sreg = torch.randn(B, generator=gen, device="cuda") * 5.0 if cfg.get("sreg_free") else (al32 * s.dreg_v.double()).sum(1).float()
        sreg_buf[:, T_AT] = sreg
    dwf0 = torch.randn(B * A + 64, device="cuda")
    dwf0[B * A:] = float("nan")
    dwf = dwf0.clone()
    out1_0 = s.out1.clone()

    de, dcat, dctx = _backward(s, _lib, L, alpha, ctx, dreg_buf, sreg_buf, mask, dwf, cfg.get("nodgp", False))

    # ---- expected values
    gate = s.gate.double() if s.gate is not None else None
    dg = s.dgctx[:, :C].double()
    en = s.enc.double()
    ctx64 = ctx.double()
    dcv = dg * gate if gate is not None else dg
    sr = sreg_buf[:, T_AT].double() if sreg_buf is not None else torch.zeros(B, device="cuda", dtype=torch.float64)
    dr = s.dreg_v.double() if cfg["dreg"] else torch.zeros(B, R, device="cuda", dtype=torch.float64)
    on = ref["pre"] > 0
    if cfg.get("sreg_free"):
        # the header formula with an arbitrary sreg: s = <dctx, ctx> + sreg ; de_r = alpha_r (<dctx, enc_r> + dreg_r - s)
        de_w = al32 * (torch.einsum("brc,bc->br", en, dcv) + dr - ((dcv * ctx64).sum(1) + sr)[:, None])
        datt2_w = s.wf.double() * torch.einsum("br,bra->ba", de_w, on.double())
    else:
        de_w, datt2_w = ref["de"], ref["datt2"]
    S = (torch.einsum("brc,bc->br", en.abs(), dcv.abs()) + dr.abs() + (dcv * ctx64).abs().sum(1, keepdim=True) + sr.abs()[:, None]
         + (al32 * dr.abs()).sum(1, keepdim=True))
    bde = K * EPS16 * al32 * S
    colsum = torch.einsum("br,bra->ba", K * EPS16 * de_w.abs() + bde, on.double())
    ratios = {}
    _check("de", de[:, T_AT], de_w, bde, ratios)
    _check("datt2", dcat[:, :A], datt2_w, s.wf.double().abs() * colsum, ratios)
    if not cfg.get("nodgp"):
        if gate is not None:
            # chained: ctx and gate are the forward kernel's, whose relative error on a small |ctx_c| is not the backward's to bound
            dgp_w, dctx_w = (dg * ctx64 * gate * (1 - gate), dcv) if cfg.get("chained") else (ref["dgp"], ref["dctx"])
            _check("dgp", dcat[:, A:A + C], dgp_w, 2.0 ** -20 * (dg * ctx64).abs() * gate, ratios)
            _check("dctx", dctx[:B * C].view(B, C), dctx_w, 2.0 ** -22 * dcv.abs(), ratios)
        else:
            assert (dcat[:, A:A + C] == 0).all(), "gate NULL: dgp is written with zeros"
            assert _same_bits(dctx[:B * C].view(B, C), s.dgctx[:, :C]), "gate NULL: dctx = dgctx"
    # d full_att.weight: without mask bits the whole gradient, with them its att2 term; the att1 term completes it
    a2 = s.att2.double()
    de_on = torch.einsum("br,bra->ba", de_w, on.double())
    att2_term = a2 * de_on
    att1_term = torch.einsum("br,bra->ba", de_w, on.double() * s.att1.double())
    if not cfg.get("sreg_free"):
        mag = (att2_term.abs() + att1_term.abs()).sum(0)                      # d w_full sums the per-image terms
        assert ((att2_term + att1_term).sum(0) - ref["dwf"]).abs().le(1e-9 * mag + 1e-300).all()
    inc = (dwf[:B * A].double() - dwf0[:B * A].double()).view(B, A)
    if mask is not None:
        want_w, bw = att2_term, a2.abs() * colsum
    else:
        relu = torch.relu(ref["pre"])
        want_w = att2_term + att1_term
        bw = torch.einsum("br,bra->ba", K * EPS16 * de_w.abs() + bde, relu)
    # the fp32 accumulation into dwf_part rounds once per split at most
    _check("dwf", inc, want_w, bw + 2.0 ** -19 * (dwf[:B * A].view(B, A).abs() + dwf0[:B * A].view(B, A).abs()), ratios)

    # ---- guards: nothing outside the step's slice, the A + C columns of dcat, B * C of dctx_out, B * A of dwf_part
    keep = torch.ones(T_STEPS, dtype=torch.bool, device="cuda")
    keep[T_AT] = False
    assert de[:, keep].isnan().all(), "de written outside its step"
    assert dcat[:, A + C:].isnan().all(), "dcat written past A + C"
    if cfg.get("nodgp"):
        assert dcat[:, A:A + C].isnan().all(), "datt2 written past A (into dgp)"
    else:
        assert dctx[B * C:].isnan().all(), "dctx_out written past B * C"
    assert dwf[B * A:].isnan().all(), "dwf_part written past B * A"
    assert _same_bits(s.out1, out1_0), "the backward must not write att2 / gate"

    # ---- a second call on the same workspace: the same bits (ticket counters reset, fixed combine order)
    dwf1 = dwf.clone()
    de2, dcat2, dctx2 = _backward(s, _lib, L, alpha, ctx, dreg_buf, sreg_buf, mask, dwf, cfg.get("nodgp", False))
    assert _same_bits(de2, de) and _same_bits(dcat2, dcat)
    if dctx is not None:
        assert _same_bits(dctx2, dctx)
    inc2 = (dwf[:B * A].double() - dwf1[:B * A].double()).view(B, A)
    _check("dwf", inc2, want_w, bw + 2.0 ** -19 * (dwf[:B * A].view(B, A).abs() + dwf1[:B * A].view(B, A).abs()), ratios)
    print("RATIO %s %s" % (cid, " ".join("%s=%.3g" % kv for kv in ratios.items())))
