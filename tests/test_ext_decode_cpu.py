"""CPU side of the two-layer decoding (latex_ocr_b200/ext.py greedy_decode / beam_decode): the C ABI of lo_decoder2_* without a
GPU, the two-layer decode oracle (tests/ext_decode_oracle.py) against its own teacher-forced definition
(oracle/ref_ext.py:decoder2_forward), and its step-function loops against oracle/ref_decode.py's loops on the one-layer step."""
import ctypes
import os
import subprocess

import torch

from util import ROOT  # noqa: F401  (puts the repository root on sys.path)

import ext_decode_oracle as xo  # noqa: E402

V = 30


def _params(seed=4):
    from oracle import ref_model as rm
    _, pd = rm.init_params(V, seed=seed)
    g = torch.Generator().manual_seed(seed)
    pd["fc.weight"] = (torch.rand(V, 512, generator=g) * 2 - 1) * 0.5      # non-degenerate argmax, END appears
    pd["embedding.weight"] = (torch.rand(V, 512, generator=g) * 2 - 1) * 1.0
    enc = torch.randn(3, 12, 512, generator=g) * 0.5
    return pd, enc


def test_step_function_loops_equal_ref_decode_on_the_one_layer_step():
    """With DecoderWithAttention's step the generic loops give exactly ref_decode's ids and log-probs (greedy, beam 1/3/5 x both
    finalize modes, diversity penalty)."""
    from oracle import ref_decode as rd
    from oracle import ref_model as rm
    pd, enc = _params()
    step, state = xo.one_layer_step(pd), rm.init_hidden_state(pd, enc)
    for end_id, L in ((V - 1, 6), (7, 12)):
        assert torch.equal(xo.greedy_loop(pd, enc, V - 2, end_id, L + 1, step, state), rd.greedy_decode(pd, enc, V - 2, end_id, L + 1))
    u = torch.rand(10, 3 * 3, V, generator=torch.Generator().manual_seed(77))
    for beam, fin, div in ((1, "reference", {}), (3, "reference", {}), (3, "backtrack", {}), (5, "backtrack", {}),
                           (3, "reference", dict(div_gamma=0.5, div_prob=1.0, div_u=u))):
        want, wlp = rd.beam_decode(pd, enc, V - 2, 5, beam, 9, finalize=fin, **div)
        got, glp = xo.beam_loop(pd, enc, V - 2, 5, beam, 9, step, state, finalize=fin, **div)
        assert torch.equal(got, want) and torch.equal(glp, wlp), (beam, fin, div.keys())


def test_two_layer_greedy_oracle_is_its_own_argmax():
    """Teacher-forcing decoder2_forward on greedy_decode_ext's own tokens gives logits whose argmax is those tokens."""
    from oracle import ref_ext as rx
    pd, enc = _params(seed=5)
    _, p2 = rx.init_params_ext(seed=6)
    for end_id, L in ((V - 1, 8), (7, 12)):
        ids = xo.greedy_decode_ext(pd, p2, enc, V - 2, end_id, L + 1)
        caps = torch.cat([torch.full((enc.shape[0], 1), V - 2, dtype=torch.long), ids], dim=1)
        logits, _ = rx.decoder2_forward(pd, p2, enc, caps, ids.shape[1])
        assert torch.equal(logits.argmax(-1), ids)
    # the second layer changes the search: the one-layer loop decodes something else from the same layer-1 weights
    from oracle import ref_decode as rd
    assert not torch.equal(rd.greedy_decode(pd, enc, V - 2, V - 1, 9), xo.greedy_decode_ext(pd, p2, enc, V - 2, V - 1, 9))


def test_two_layer_beam_oracle_reparents_state():
    """beam_decode_ext with beam 1 is greedy_decode_ext; with beam 3 the hypotheses re-parent (backtrack differs from the reference's
    identity finalize), and the best backtracked hypothesis re-scores to its log-prob under teacher forcing."""
    from oracle import ref_ext as rx
    pd, enc = _params(seed=5)
    _, p2 = rx.init_params_ext(seed=6)
    g = xo.greedy_decode_ext(pd, p2, enc, V - 2, 5, 9)
    b1, _ = xo.beam_decode_ext(pd, p2, enc, V - 2, 5, 1, 9)
    assert torch.equal(b1[:, :, 0][:, :g.shape[1]], g)
    ref, lp = xo.beam_decode_ext(pd, p2, enc, V - 2, 5, 3, 9, finalize="reference")
    bt, lp2 = xo.beam_decode_ext(pd, p2, enc, V - 2, 5, 3, 9, finalize="backtrack")
    assert torch.equal(lp, lp2) and not torch.equal(ref, bt)
    hyp = bt[:, :, 0]
    caps = torch.cat([torch.full((enc.shape[0], 1), V - 2, dtype=torch.long), hyp], dim=1)
    logits, _ = rx.decoder2_forward(pd, p2, enc, caps, hyp.shape[1])
    lsm = torch.log_softmax(logits, dim=-1)
    for n in range(enc.shape[0]):
        s, done = 0.0, False
        for t in range(hyp.shape[1]):
            if not done:
                s += float(lsm[n, t, hyp[n, t]])
            done = done or int(hyp[n, t]) == 5
        assert abs(s - float(lp[n, 0])) < 1e-4 * max(1.0, abs(s)), (n, s, float(lp[n, 0]))


def _lib_or_skip():
    import pytest
    from latex_ocr_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built")
    return _lib


def test_dec2_symbols_and_struct_mirror():
    _lib = _lib_or_skip()
    from latex_ocr_b200 import ext
    L = ext._bind()
    for name in ("lo_sizeof_dec2_args", "lo_dec2_workspace_bytes", "lo_decoder2_greedy_hist", "lo_decoder2_beam_div"):
        assert name in _lib.declared_symbols(), name
    out = subprocess.run(["nm", "-D", _lib.LIB_PATH], capture_output=True, text=True).stdout
    for name in ("lo_sizeof_dec2_args", "lo_dec2_workspace_bytes", "lo_decoder2_greedy_hist", "lo_decoder2_beam_div"):
        assert (" T " + name) in out, name
    assert L.lo_sizeof_dec2_args() == ctypes.sizeof(ext.Dec2Args)
    assert [f[0] for f in ext.Dec2Args._fields_] == ["D", "dt", "impl", "w_ih", "w_hh", "b_ih", "b_hh", "ws"]
    # h, c, bf16 h (two slots each) + the [B][4D] gates scratch, 256-byte aligned pieces
    assert L.lo_dec2_workspace_bytes(64, 512) == 2 * 64 * 512 * 4 * 2 + 2 * 64 * 512 * 2 + 64 * 4 * 512 * 4
    assert L.lo_dec2_workspace_bytes(0, 512) == 0


def test_dec2_entries_reject_bad_blocks_before_gpu_work():
    """Argument errors come back as -1 with a readable message, before anything touches a device (this runs without a GPU)."""
    _lib = _lib_or_skip()
    from latex_ocr_b200 import ext
    L = ext._bind()
    a = _lib.DecoderArgs()
    a.D = 512
    l2 = ext.Dec2Args()
    l2.D, l2.dt = 256, _lib.LO_F32
    for fn, extra in ((L.lo_decoder2_greedy_hist, (0, 1, 4, None, None, None, None)),
                      (L.lo_decoder2_beam_div, (0, 1, 4, None, None, None, None, 1.0, 0.0, None, None, None))):
        assert fn(ctypes.byref(a), None, *extra) == -1
        assert b"null layer-2 block" in L.lo_last_error()
        assert fn(None, ctypes.byref(l2), *extra) == -1
        assert b"args" in L.lo_last_error()
        assert fn(ctypes.byref(a), ctypes.byref(l2), *extra) == -1
        assert b"layer-2 D must equal the decoder's D" in L.lo_last_error()
        l2.D = 512
        assert fn(ctypes.byref(a), ctypes.byref(l2), *extra) == -1           # weights / workspace missing
        assert b"null layer-2 pointer" in L.lo_last_error()
        l2.D = 256

