"""EXTENSION beyond the reference — BASELINE.json configs[3]: "row-encoder biLSTM over CNN feature rows + 2-layer decoder,
160x640 images".  The reference contains neither (SURVEY.md §0: `model/decoder.py:16` only links the im2markup paper), so there
is no reference code to restate; semantics are defined HERE and checked against torch.nn.LSTM / autograd (oracle/ref_ext.py):

  RowEncoder        nn.LSTM(512, 256, bidirectional=True, batch_first=True) run over every ROW of the CNN feature map
                    ([N,H',W',512] -> [N,H',W',512], forward || backward halves), zero initial state; state_dict keys
                    ``lstm.weight_ih_l0 ... lstm.bias_hh_l0_reverse`` exactly like nn.LSTM.
  two-layer decoder the attention LSTM of DecoderWithAttention (seq2seq_torch.py:267-320) as layer 1; layer 2 =
                    nn.LSTMCell(D, D) over x_t = dropout(h1_t), zero initial state; logits_t = fc(h2_t).  Layer 2 does not feed
                    the attention, so it runs as one sequence LSTM between the time loop and the (hoisted) fc head
                    (``lo_decoder_args.phase`` 1 / 2).
  Img2SeqRowModel   EncoderCNN -> RowEncoder -> two-layer decoder, loss / regulariser / Adam exactly as Img2SeqModel.getLoss.

Both LSTMs run on ``lo_lstm_seq_forward/backward`` (csrc/lo_lstmseq.cuh): hoisted input projection, one recurrent GEMM + one cell
kernel per step, hand-derived backward with hoisted weight gradients.

Decoding (``greedy_decode`` / ``beam_decode``, same loop rules and outputs as latex_ocr_b200.decode) runs layer 2 inside the time
loop, step by step, because token t+1 depends on fc(h2_t): ``lo_decoder2_greedy_hist`` / ``lo_decoder2_beam_div``
(csrc/lo_decoder2.cuh).  In beam search layer 2's state follows the parents like layer 1's.
"""
import ctypes
import math

import torch
import torch.nn as nn

from . import _lib, decode
from ._lib import check, ptr, stream_ptr
from .img2seq import Img2SeqModel
from .params import FlatStore, LRUCache, ParamHolder


def _make_struct():
    with open(_lib.HEADER) as f:
        text = f.read()

    class LstmSeqArgs(ctypes.Structure):
        _fields_ = _lib._parse_struct(text, "lo_lstm_seq_args")

    class Dec2Args(ctypes.Structure):
        _fields_ = _lib._parse_struct(text, "lo_dec2_args")

    return LstmSeqArgs, Dec2Args


LstmSeqArgs, Dec2Args = _make_struct()
_bound = False


def _bind():
    global _bound
    L = _lib.lib()
    if _bound:
        return L
    P = ctypes.POINTER(LstmSeqArgs)
    L.lo_sizeof_lstm_seq_args.restype = ctypes.c_int64
    if L.lo_sizeof_lstm_seq_args() != ctypes.sizeof(LstmSeqArgs):
        raise _lib.LatexOcrB200Error("lo_lstm_seq_args layout mismatch — rebuild")
    L.lo_lstm_seq_workspace_bytes.restype = ctypes.c_int64
    L.lo_lstm_seq_workspace_bytes.argtypes = [P]
    for name in ("lo_lstm_seq_forward", "lo_lstm_seq_backward"):
        fn = getattr(L, name)
        fn.argtypes = [P, ctypes.c_void_p]
        fn.restype = ctypes.c_int
    L.lo_sizeof_dec2_args.restype = ctypes.c_int64
    if L.lo_sizeof_dec2_args() != ctypes.sizeof(Dec2Args):
        raise _lib.LatexOcrB200Error("lo_dec2_args layout mismatch — rebuild")
    L.lo_dec2_workspace_bytes.restype = ctypes.c_int64
    L.lo_dec2_workspace_bytes.argtypes = [ctypes.c_int, ctypes.c_int]
    PD, P2 = ctypes.POINTER(_lib.DecoderArgs), ctypes.POINTER(Dec2Args)
    vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float
    L.lo_decoder2_greedy_hist.argtypes = [PD, P2, i64, i64, i32, vp, vp, vp, vp]
    L.lo_decoder2_beam_div.argtypes = [PD, P2, i64, i64, i32, vp, vp, vp, vp, f32, f32, vp, vp, vp]
    L.lo_decoder2_greedy_hist.restype = L.lo_decoder2_beam_div.restype = ctypes.c_int
    _bound = True
    return L


def _dt(precision):
    return _lib.LO_F32 if precision == "fp32" else _lib.LO_BF16


class _Direction:
    """One direction of one layer: argument block + workspace for a given (S, M) shape."""

    def __init__(self, store, prefix, suffix, I, H, precision, impl, reverse):
        self.store, self.I, self.H, self.precision, self.impl, self.reverse = store, I, H, precision, impl, reverse
        self.names = {k: "%s%s%s" % (prefix, k, suffix) for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")}
        self._ws = LRUCache()

    def args(self, S, M):
        key = (S, M)
        ent = self._ws.get(key)
        S_ = self.store
        if ent is None:
            a = LstmSeqArgs()
            a.S, a.M, a.I, a.H = S, M, self.I, self.H
            a.dt = _dt(self.precision)
            a.impl = _lib.LO_IMPL_TC if (self.impl == "tc" and self.precision == "bf16") else _lib.LO_IMPL_SIMT
            a.reverse = 1 if self.reverse else 0
            nbytes = int(_bind().lo_lstm_seq_workspace_bytes(ctypes.byref(a)))
            ws = torch.zeros(nbytes, dtype=torch.uint8, device=S_.device)
            a.ws = ws.data_ptr()
            ent = self._ws[key] = {"a": a, "ws": ws}
        a = ent["a"]
        n = self.names
        a.w_ih, a.w_hh = S_.w(n["weight_ih"]).data_ptr(), S_.w(n["weight_hh"]).data_ptr()
        a.b_ih, a.b_hh = S_.f32(n["bias_ih"]).data_ptr(), S_.f32(n["bias_hh"]).data_ptr()
        a.g_w_ih, a.g_w_hh = S_.g(n["weight_ih"]).data_ptr(), S_.g(n["weight_hh"]).data_ptr()
        a.g_b_ih, a.g_b_hh = S_.g(n["bias_ih"]).data_ptr(), S_.g(n["bias_hh"]).data_ptr()
        return a


def _lstm_specs(prefix, suffix, I, H):
    return [("%sweight_ih%s" % (prefix, suffix), (4 * H, I)), ("%sweight_hh%s" % (prefix, suffix), (4 * H, H)),
            ("%sbias_ih%s" % (prefix, suffix), (4 * H,)), ("%sbias_hh%s" % (prefix, suffix), (4 * H,))]


class RowEncoder(nn.Module):
    """Bidirectional LSTM over the rows of the CNN feature map (extension, see module docstring)."""

    def __init__(self, channels=512, hidden=256, device="cuda", precision="bf16", impl=None):
        super().__init__()
        self.C, self.H = channels, hidden
        self.precision = precision
        self.impl = impl if impl is not None else ("tc" if precision == "bf16" else "simt")
        self.tdtype = torch.float32 if precision == "fp32" else torch.bfloat16
        specs = _lstm_specs("lstm.", "_l0", channels, hidden) + _lstm_specs("lstm.", "_l0_reverse", channels, hidden)
        self.store = FlatStore(specs, device, bf16_shadow=(precision == "bf16"))
        self.lstm = ParamHolder()
        for name, _ in specs:
            self.lstm.bind(name.split(".", 1)[1], self.store, name)
        self.dirs = (_Direction(self.store, "lstm.", "_l0", channels, hidden, precision, self.impl, False),
                     _Direction(self.store, "lstm.", "_l0_reverse", channels, hidden, precision, self.impl, True))
        b = 1.0 / math.sqrt(hidden)                       # nn.LSTM.reset_parameters
        with torch.no_grad():
            for p_ in self.lstm.parameters():
                p_.uniform_(-b, b)
        self._out = LRUCache()
        self._shadow_fresh = False

    def _load_from_state_dict(self, *a, **k):
        super()._load_from_state_dict(*a, **k)
        self._shadow_fresh = False

    def sync_shadow(self):
        if not self._shadow_fresh:
            self.store.sync_shadow()
            self._shadow_fresh = True

    def forward_raw(self, feat):
        """feat: CUDA storage-dtype [N,H',W',C] -> storage-dtype [N,H',W',2*hidden] (a cached buffer)."""
        L = _bind()
        if not feat.is_cuda:
            raise _lib.LatexOcrB200Error("RowEncoder runs on CUDA tensors only (no CPU fallback)")
        feat = feat.contiguous().to(self.tdtype)
        N, Hh, Ww, C = feat.shape
        self.sync_shadow()
        ent = self._out.get((N, Hh, Ww))
        if ent is None:
            ent = self._out[(N, Hh, Ww)] = {"out": torch.empty(N, Hh, Ww, 2 * self.H, dtype=self.tdtype, device=feat.device),
                                           "dfeat": torch.empty(N, Hh, Ww, C, dtype=torch.float32, device=feat.device)}
        out = ent["out"]
        ent["feat"] = feat
        es = out.element_size()
        for d, dr in enumerate(self.dirs):
            a = dr.args(Ww, N * Hh)
            a.x, a.x_row, a.x_step = feat.data_ptr(), Ww * C, C
            a.hs = None
            a.hs_st = out.data_ptr() + d * self.H * es
            a.hs_row, a.hs_step = Ww * 2 * self.H, 2 * self.H
            check(L.lo_lstm_seq_forward(ctypes.byref(a), stream_ptr()))
        return out

    def backward_raw(self, shape, dout):
        """dout: fp32 [N,H',W',2*hidden] -> d feat fp32 [N,H',W',C]; parameter gradients land in self.store.grad."""
        L = _bind()
        N, Hh, Ww = shape
        ent = self._out[(N, Hh, Ww)]
        dfeat, feat = ent["dfeat"], ent["feat"]
        C = feat.shape[3]
        dout = dout.contiguous()
        for d, dr in enumerate(self.dirs):
            a = dr.args(Ww, N * Hh)
            a.x, a.x_row, a.x_step = feat.data_ptr(), Ww * C, C
            a.dhs = dout.data_ptr() + d * self.H * 4
            a.hs_row, a.hs_step = Ww * 2 * self.H, 2 * self.H
            a.dx, a.dx_row, a.dx_step, a.dx_accumulate = dfeat.data_ptr(), Ww * C, C, d
            check(L.lo_lstm_seq_backward(ctypes.byref(a), stream_ptr()))
        return dfeat

    def forward(self, feat):
        with torch.no_grad():
            return self.forward_raw(feat).float()


class DecoderLayer2(nn.Module):
    """nn.LSTMCell(D, D) run over the whole sequence of dropout(h1_t) between the decoder's time loop and its fc head."""

    def __init__(self, D=512, device="cuda", precision="bf16", impl=None):
        super().__init__()
        self.D, self.precision = D, precision
        self.impl = impl if impl is not None else ("tc" if precision == "bf16" else "simt")
        self.tdtype = torch.float32 if precision == "fp32" else torch.bfloat16
        specs = _lstm_specs("cell.", "", D, D)
        self.store = FlatStore(specs, device, bf16_shadow=(precision == "bf16"))
        self.cell = ParamHolder()
        for name, _ in specs:
            self.cell.bind(name.split(".", 1)[1], self.store, name)
        self.dir = _Direction(self.store, "cell.", "", D, D, precision, self.impl, False)
        b = 1.0 / math.sqrt(D)
        with torch.no_grad():
            for p_ in self.cell.parameters():
                p_.uniform_(-b, b)
        self._shadow_fresh = False
        self._x = LRUCache()
        self._dec = LRUCache()

    def _load_from_state_dict(self, *a, **k):
        super()._load_from_state_dict(*a, **k)
        self._shadow_fresh = False

    def sync_shadow(self):
        if not self._shadow_fresh:
            self.store.sync_shadow()
            self._shadow_fresh = True

    def forward_inplace(self, hd):
        """hd: fp32 [B,T,D] (dropout(h1), batch-major) — replaced IN PLACE by h2."""
        B, T, D = hd.shape
        self.sync_shadow()
        x = self._x.get((B, T))
        if x is None:
            x = self._x[(B, T)] = torch.empty(B, T, D, dtype=self.tdtype, device=hd.device)
        x.copy_(hd)                                        # layer input in storage dtype (plumbing cast)
        a = self.dir.args(T, B)
        a.x, a.x_row, a.x_step = x.data_ptr(), T * D, D
        a.hs, a.hs_st = hd.data_ptr(), None
        a.hs_row, a.hs_step = T * D, D
        check(_bind().lo_lstm_seq_forward(ctypes.byref(a), stream_ptr()))

    def decode_args(self, B):
        """lo_dec2_args of the decode loops for B rows (layer 2 inside the time loop; workspace cached per B)."""
        self.sync_shadow()
        ent = self._dec.get(B)
        S = self.store
        if ent is None:
            nbytes = int(_bind().lo_dec2_workspace_bytes(B, self.D))
            ent = self._dec[B] = {"a": Dec2Args(), "ws": torch.empty(nbytes, dtype=torch.uint8, device=S.device)}
        a = ent["a"]
        a.D, a.dt = self.D, _dt(self.precision)
        a.impl = _lib.LO_IMPL_TC if (self.impl == "tc" and self.precision == "bf16") else _lib.LO_IMPL_SIMT
        a.w_ih, a.w_hh = S.w("cell.weight_ih").data_ptr(), S.w("cell.weight_hh").data_ptr()
        a.b_ih, a.b_hh = S.f32("cell.bias_ih").data_ptr(), S.f32("cell.bias_hh").data_ptr()
        a.ws = ent["ws"].data_ptr()
        return a

    def backward_inplace(self, dhd):
        """dhd: fp32 [B,T,D] holding d loss / d h2 — replaced IN PLACE by d loss / d dropout(h1)."""
        B, T, D = dhd.shape
        a = self.dir.args(T, B)
        a.x, a.x_row, a.x_step = self._x[(B, T)].data_ptr(), T * D, D
        a.dhs = dhd.data_ptr()
        a.hs_row, a.hs_step = T * D, D
        a.dx, a.dx_row, a.dx_step, a.dx_accumulate = dhd.data_ptr(), T * D, D, 0      # d x is scattered after the loop has read dhs
        check(_bind().lo_lstm_seq_backward(ctypes.byref(a), stream_ptr()))


def _encode(model, img):
    """CNN -> row biLSTM: the storage-dtype encoder output [N,H',W',512] the two-layer decoder attends over."""
    feat = model.encoder.forward_raw(img.to(model.device).float(), need_grad=False)
    return model.row_encoder.forward_raw(feat)


def _prepare(model, img):
    return lambda rows, steps: decode._prepare_enc(model, _encode(model, img), rows, steps)


def greedy_decode(model, img, start_id, end_id, max_length_formula=150, return_attention=False):
    """decode.greedy_decode for an Img2SeqRowModel: token ids [N, steps] (CPU int64), with ``return_attention=True`` also the
    attention weights [N, steps, R]."""
    L = _bind()
    return decode._greedy(model, _prepare(model, img),
                          lambda a, *args: L.lo_decoder2_greedy_hist(ctypes.byref(a), ctypes.byref(model.layer2.decode_args(a.B)), *args),
                          start_id, end_id, max_length_formula, return_attention)


def beam_decode(model, img, start_id, end_id, beam_size=5, max_length_formula=150, finalize="reference", div_gamma=1, div_prob=0,
                div_u=None, div_seed=None):
    """decode.beam_decode for an Img2SeqRowModel: (ids [N, beam, steps], log_probs [N, beam]) on the CPU; same finalize modes and
    diversity penalty."""
    L = _bind()
    return decode._beam(model, _prepare(model, img),
                        lambda a, *args: L.lo_decoder2_beam_div(ctypes.byref(a), ctypes.byref(model.layer2.decode_args(a.B)), *args),
                        start_id, end_id, beam_size, max_length_formula, finalize, div_gamma, div_prob, div_u, div_seed)


class Img2SeqRowModel(Img2SeqModel):
    """EncoderCNN -> RowEncoder -> attention decoder with a second LSTM layer (extension).  Same trainer surface as
    Img2SeqModel (getLoss / train_step / train / evaluate / write_prediction); evaluation decodes and scores this model
    (``ext.greedy_decode`` / ``ext.beam_decode``).  ``predict_batch`` is not offered yet: call ``ext.greedy_decode`` /
    ``ext.beam_decode`` directly."""

    def getModel(self, model_name="Img2Seq"):
        super().getModel(model_name)
        self.row_encoder = RowEncoder(512, 256, device=self.device, precision=self.precision, impl=self.impl)
        self.layer2 = DecoderLayer2(512, device=self.device, precision=self.precision, impl=self.impl)
        return self

    def getOptimizer(self, lr_method="adam", lr=0.001):
        super().getOptimizer(lr_method, lr)
        self.row_encoder.store.ensure_adam(lr)
        self.layer2.store.ensure_adam(lr)

    def set_lr(self, lr):
        super().set_lr(lr)
        self.row_encoder.store.set_lr(lr)
        self.layer2.store.set_lr(lr)

    def predict_batch(self, *a, **k):
        raise NotImplementedError("predict_batch is not offered for the row-encoder / two-layer extension: "
                                  "use latex_ocr_b200.ext.greedy_decode / ext.beam_decode")

    def _decode_ids(self, images, start_id=None, decoding=None, beam_size=None):
        return self._decode_ids_with(greedy_decode, beam_decode, images, start_id, decoding, beam_size)

    def _teacher_forced_ce(self, img, formula_t, lens, start_id):
        """Img2SeqModel._teacher_forced_ce on the two-layer model, run as _step_body runs it but without gradient or dropout:
        phase 1 (time loop of layer 1, writes hd = h1) -> layer 2 over the sequence -> phase 2 (fc head)."""
        inp = torch.cat([torch.full((formula_t.shape[0], 1), start_id, dtype=torch.int64), formula_t], dim=1)
        with torch.no_grad():
            enc = _encode(self, img)
            N, C = enc.shape[0], enc.shape[3]
            lens_s, sort_ind = (lens + 1).squeeze(1).sort(dim=0, descending=True)       # seq2seq_torch.py:286
            si = sort_ind.to(self.device)
            enc_s = enc.view(N, -1, C)[si].contiguous()
            caps = inp.to(self.device)[si].contiguous()
            dl = (lens_s - 1).tolist()
            dec = self.decoder
            ws = dec.run_forward(enc_s, caps, dl, with_loss=False, need_grad=False, phase=1)
            self.layer2.forward_inplace(ws["t"]["hd"])
            dec.run_phase(ws, 2, backward=False, with_loss=False)
            preds = ws["t"]["logits"][:, :, :dec.vocab_size]
            return self._ce_sum(preds, caps[:, 1:], dl)

    def _keepalive(self):
        keep = super()._keepalive()
        keep += [list(self.row_encoder._out.values()), list(self.layer2._x.values()), list(self.layer2.dir._ws.values())]
        keep += [list(d._ws.values()) for d in self.row_encoder.dirs]
        return keep

    def _step_body(self, img, caps, decode_lengths, dropout_mask):
        N = img.shape[0]
        feat = self.encoder.forward_raw(img, need_grad=True)                       # [N,H',W',512] incl. the timing signal
        Hh, Ww = feat.shape[1], feat.shape[2]
        enc_out = self.row_encoder.forward_raw(feat)
        R = Hh * Ww
        dec = self.decoder
        enc_flat = enc_out.view(N, R, enc_out.shape[3])
        # phase 1: time loop of layer 1 (writes hd = dropout(h1)); layer 2 over the sequence; phase 2: fc head + loss
        ws = dec.run_forward(enc_flat, caps, decode_lengths, with_loss=True, need_grad=True, dropout_mask=dropout_mask, phase=1)
        self.layer2.forward_inplace(ws["t"]["hd"])
        dec.run_phase(ws, 2, backward=False)
        dec.run_phase(ws, 2, backward=True)                                         # fc backward -> dhd = d h2
        self.layer2.backward_inplace(ws["t"]["dhd"])
        dec.run_phase(ws, 1, backward=True)                                         # BPTT of layer 1 + hoisted gradients -> denc
        scale = 1.0
        if self.dist is not None:
            self.dist.reduce_async(dec.store.grad)
            self.dist.reduce_async(self.layer2.store.grad)
            scale = 1.0 / self.dist.world_size
        dfeat = self.row_encoder.backward_raw((N, Hh, Ww), ws["t"]["denc"].view(N, Hh, Ww, enc_out.shape[3]))
        if self.dist is not None:
            self.dist.reduce_async(self.row_encoder.store.grad)
            self.encoder.backward_raw(tuple(img.shape), dfeat, on_layer_grad=self.dist.layer_hook(self.encoder))
            self.dist.wait()
        else:
            self.encoder.backward_raw(tuple(img.shape), dfeat)
        self._adam(dec.store, scale, dec)
        self._adam(self.layer2.store, scale)
        self._adam(self.row_encoder.store, scale)
        self._adam(self.encoder.store, scale, self.encoder)
        self.layer2._shadow_fresh = self.row_encoder._shadow_fresh = True          # the fused Adam refreshed the bf16 shadows
        return ws["t"]["loss"]

    def state_dict(self):
        sd = super().state_dict()
        sd["row_encoder"], sd["layer2"] = self.row_encoder.state_dict(), self.layer2.state_dict()
        return sd

    def load_state_dict(self, sd):
        super().load_state_dict(sd)
        self.row_encoder.load_state_dict(sd["row_encoder"])
        self.layer2.load_state_dict(sd["layer2"])
