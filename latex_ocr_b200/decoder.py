"""Attention / DecoderWithAttention — drop-ins for model/components/seq2seq_torch.py:160-320 on the
sm_100a kernels (lo_decoder.cu) through the C ABI.  Same constructors, forward signatures, return
tuples and ``state_dict`` keys:
  attention.{encoder_att,decoder_att,full_att}.{weight,bias}, embedding.weight,
  decode_step.{weight_ih,weight_hh,bias_ih,bias_hh}, init_h.*, init_c.*, f_beta.*, fc.*
"""
import ctypes
import math

import torch
import torch.nn as nn

from . import _lib
from ._lib import check, ptr, stream_ptr
from .params import FlatStore, LRUCache, ParamHolder


def _dt(precision):
    return _lib.LO_F32 if precision == "fp32" else _lib.LO_BF16


def decoder_specs(A, E, D, V, C):
    """Flat order: [decoder_att.W; f_beta.W; weight_hh] and their biases are contiguous so the per-step
    GEMM h -> (att2 | gate_pre | hh) and its weight gradient are single launches."""
    return [
        ("attention.encoder_att.weight", (A, C)), ("attention.encoder_att.bias", (A,)),
        ("attention.decoder_att.weight", (A, D)), ("f_beta.weight", (C, D)), ("decode_step.weight_hh", (4 * D, D)),
        ("attention.decoder_att.bias", (A,)), ("f_beta.bias", (C,)), ("decode_step.bias_hh", (4 * D,)),
        ("attention.full_att.weight", (1, A)), ("attention.full_att.bias", (1,)),
        ("embedding.weight", (V, E)),
        ("decode_step.weight_ih", (4 * D, E + C)), ("decode_step.bias_ih", (4 * D,)),
        ("init_h.weight", (D, C)), ("init_c.weight", (D, C)), ("init_h.bias", (D,)), ("init_c.bias", (D,)),
        ("fc.weight", (V, D)), ("fc.bias", (V,)),
    ]


class Attention(nn.Module):
    """seq2seq_torch.py:160-192.  Stand-alone use: forward(encoder_out[B,R,C], decoder_hidden[B,D])
    -> (context[B,C], alpha[B,R]).  Inside DecoderWithAttention the parameters are views into the
    decoder's flat store."""

    def __init__(self, encoder_dim, decoder_dim, attention_dim, device="cuda", precision="bf16", _store=None):
        super().__init__()
        self.encoder_dim, self.decoder_dim, self.attention_dim = encoder_dim, decoder_dim, attention_dim
        self.precision = precision
        self.tdtype = torch.float32 if precision == "fp32" else torch.bfloat16
        own = _store is None
        if own:
            specs = [("attention.encoder_att.weight", (attention_dim, encoder_dim)), ("attention.encoder_att.bias", (attention_dim,)),
                     ("attention.decoder_att.weight", (attention_dim, decoder_dim)), ("attention.decoder_att.bias", (attention_dim,)),
                     ("attention.full_att.weight", (1, attention_dim)), ("attention.full_att.bias", (1,))]
            _store = FlatStore(specs, device, bf16_shadow=(precision == "bf16"))
        self.store = _store
        for sub in ("encoder_att", "decoder_att", "full_att"):
            h = ParamHolder()
            h.bind("weight", _store, "attention.%s.weight" % sub)
            h.bind("bias", _store, "attention.%s.bias" % sub)
            setattr(self, sub, h)
        if own:
            with torch.no_grad():
                for sub, fan in (("encoder_att", encoder_dim), ("decoder_att", decoder_dim), ("full_att", attention_dim)):
                    b = 1.0 / math.sqrt(fan)
                    getattr(self, sub).weight.uniform_(-b, b)
                    getattr(self, sub).bias.uniform_(-b, b)
        self._work = None

    def forward(self, encoder_out, decoder_hidden):
        L = _lib.lib()
        if not encoder_out.is_cuda:
            raise _lib.LatexOcrB200Error("Attention runs on CUDA tensors only (no CPU fallback)")
        with torch.no_grad():
            S, st, dt = self.store, stream_ptr(), _dt(self.precision)
            S.sync_shadow()
            B, R, C = encoder_out.shape
            A, D = self.attention_dim, self.decoder_dim
            enc = encoder_out.contiguous().to(self.tdtype)
            att1 = torch.empty(B, R, A, dtype=self.tdtype, device=enc.device)
            check(L.lo_gemm(ptr(enc), dt, ptr(S.w("attention.encoder_att.weight")), dt, ptr(att1), dt, B * R, A, C,
                            C, 1, 1, C, A, 1, 0, 0, 0, ptr(S.f32("attention.encoder_att.bias")), 0, 0, _lib.LO_IMPL_SIMT, st))
            h = decoder_hidden.contiguous().float()
            att2 = torch.empty(B, A, dtype=torch.float32, device=enc.device)
            check(L.lo_gemm(ptr(h), _lib.LO_F32, ptr(S.w("attention.decoder_att.weight")), dt, ptr(att2), _lib.LO_F32, B, A, D,
                            D, 1, 1, D, A, 1, 0, 0, 0, ptr(S.f32("attention.decoder_att.bias")), 0, 0, _lib.LO_IMPL_SIMT, st))
            nbytes = L.lo_attention_workspace_bytes(B, C)
            if self._work is None or self._work.numel() < nbytes:
                self._work = torch.zeros(nbytes, dtype=torch.uint8, device=enc.device)
            alpha = torch.empty(B, R, dtype=torch.float32, device=enc.device)
            ctx = torch.empty(B, C, dtype=torch.float32, device=enc.device)
            check(L.lo_attention_forward(ptr(att1), ptr(enc), dt, ptr(att2), A, ptr(S.f32("attention.full_att.weight")),
                                         ptr(alpha), R, ptr(ctx), None, 0, None, B, R, A, C, ptr(self._work), st))
            return ctx, alpha


class DecoderWithAttention(nn.Module):
    def __init__(self, attention_dim, embed_dim, decoder_dim, vocab_size, encoder_dim=512, dropout=0.5,
                 device="cuda", precision="bf16", impl=None):
        super().__init__()
        self.encoder_dim, self.attention_dim = encoder_dim, attention_dim
        self.embed_dim, self.decoder_dim, self.vocab_size = embed_dim, decoder_dim, vocab_size
        self.dropout_p = dropout
        self.precision = precision
        self.impl = impl if impl is not None else ("tc" if precision == "bf16" else "simt")
        self.alpha_c = 1.0                      # img2seq_torch.py:157
        self.tdtype = torch.float32 if precision == "fp32" else torch.bfloat16
        A, E, D, V, C = attention_dim, embed_dim, decoder_dim, vocab_size, encoder_dim
        self.store = FlatStore(decoder_specs(A, E, D, V, C), device, bf16_shadow=(precision == "bf16"))
        S = self.store
        self.attention = Attention(C, D, A, device, precision, _store=S)
        self.embedding = ParamHolder()
        self.embedding.bind("weight", S, "embedding.weight")
        self.dropout = nn.Dropout(p=dropout)    # kept for train()/eval() semantics and p
        self.decode_step = ParamHolder()
        for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
            self.decode_step.bind(n, S, "decode_step." + n)
        for n in ("init_h", "init_c", "f_beta", "fc"):
            h = ParamHolder()
            h.bind("weight", S, n + ".weight")
            h.bind("bias", S, n + ".bias")
            setattr(self, n, h)
        self.reset_parameters()
        self._ws = LRUCache()     # bounded: see params.LRUCache
        self._shadow_fresh = False
        # in-kernel dropout (has_dropout=2): device {seed, call counter}; the counter is advanced by lo_decoder_backward, so
        # CUDA-graph replays draw a fresh mask every step
        self.dropout_state = torch.tensor([int(torch.initial_seed()) & 0x7FFFFFFFFFFFFFFF, 0], dtype=torch.int64, device=device)

    def seed_dropout(self, seed, call=0):
        self.dropout_state.copy_(torch.tensor([int(seed) & 0x7FFFFFFFFFFFFFFF, int(call)], dtype=torch.int64))

    def reset_parameters(self):
        A, E, D, V, C = self.attention_dim, self.embed_dim, self.decoder_dim, self.vocab_size, self.encoder_dim
        with torch.no_grad():
            def lin(h, fan):
                b = 1.0 / math.sqrt(fan)
                h.weight.uniform_(-b, b)
                h.bias.uniform_(-b, b)
            lin(self.attention.encoder_att, C)
            lin(self.attention.decoder_att, D)
            lin(self.attention.full_att, A)
            lin(self.init_h, C)
            lin(self.init_c, C)
            lin(self.f_beta, D)
            b = 1.0 / math.sqrt(D)
            for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
                getattr(self.decode_step, n).uniform_(-b, b)
            self.embedding.weight.normal_(0, 1)
            lin(self.fc, D)
        self.init_weights()
        self._shadow_fresh = False

    def init_weights(self):
        """seq2seq_torch.py:230-236."""
        with torch.no_grad():
            self.embedding.weight.uniform_(-0.1, 0.1)
            self.fc.bias.fill_(0)
            self.fc.weight.uniform_(-0.1, 0.1)
        self._shadow_fresh = False

    def load_pretrained_embeddings(self, embeddings):
        """seq2seq_torch.py:238-244 (copies into the flat store instead of re-pointing the Parameter)."""
        with torch.no_grad():
            self.embedding.weight.copy_(embeddings)
        self._shadow_fresh = False

    def fine_tune_embeddings(self, fine_tune=True):
        """seq2seq_torch.py:246-253."""
        for p in self.embedding.parameters():
            p.requires_grad = fine_tune

    def _load_from_state_dict(self, *a, **k):
        super()._load_from_state_dict(*a, **k)
        self._shadow_fresh = False

    def sync_shadow(self):
        if not self._shadow_fresh:
            self.store.sync_shadow()
            self._shadow_fresh = True

    # ---------------------------------------------------------------------------------------------
    def workspace(self, B, T, R, need_grad):
        key = (B, T, R)
        ws = self._ws.get(key)
        dev = self.store.device
        A, E, D, V, C = self.attention_dim, self.embed_dim, self.decoder_dim, self.vocab_size, self.encoder_dim
        O1, G = A + C + 4 * D, 4 * D
        f32 = torch.float32

        def z(*shape, dtype=f32):
            return torch.zeros(*shape, dtype=dtype, device=dev)

        if ws is None:
            ws = {"need_grad": False}
            t = ws["t"] = {}
            t["caps"] = z(B, T + 1, dtype=torch.int64)
            t["att1"] = z(B, R, A, dtype=self.tdtype)
            t["ptab"] = z(V, G)
            t["mean"] = z(B, C)
            t["hall"] = z(T + 1, B, D)
            t["call"] = z(T + 1, B, D)
            t["out1"] = z(T, B, O1)
            t["alphas"] = z(B, T, R)
            t["ctx"] = z(T, B, C)
            t["gctx"] = z(T, B, C)
            t["gates"] = z(T, B, G)
            t["gtmp"] = z(B, G)
            t["hd"] = z(B, T, D)
            ws["ldl"] = (V + 63) // 64 * 64
            t["logits"] = z(B, T, ws["ldl"])
            t["row_loss"] = z(B * T + B * R)
            t["loss"] = z(4)
            t["sreg"] = z(B, max(T, 2))
            t["work"] = z(int(_lib.lib().lo_decoder_workspace_bytes(B, max(A, C))), dtype=torch.uint8)
            t["dropout_mask"] = None             # [B,T,D] allocated on first use of an injected mask
            ws["bt"] = (ctypes.c_int32 * T)(*([B] * T))
            self._ws[key] = ws
        if need_grad and not ws["need_grad"]:
            t = ws["t"]
            t["wbwd1"] = z(C + D, G, dtype=self.tdtype)
            t["wbwd2"] = z(D, A + C, dtype=self.tdtype)
            t["dlogits"] = z(B, T, ws["ldl"])
            t["dhd"] = z(B, T, D)
            t["dreg"] = z(B, R)
            t["dcat"] = z(T, B, O1)
            t["dxh"] = z(B, C + D)
            t["dc"] = z(2, B, D)
            t["dctx"] = z(T, B, C)
            t["de"] = z(B, T, R)
            t["dptab"] = z(V, G)
            t["datt1"] = z(B, R, A, dtype=self.tdtype)
            t["denc"] = z(B, R, C)
            t["dinit"] = z(B, 2 * D)
            t["dmean"] = z(B, max(A, C))
            # ReLU mask bits of every step (forward attention kernel -> backward attention kernel), 1 bit per att1 element
            t["att_mask"] = torch.empty(T, B, (R + 1) // 2 * 2, A // 8, dtype=torch.uint8, device=dev)      # rows padded to an even count
            ws["need_grad"] = True
        return ws

    def _ws_for(self, B, T, R):
        """The cached workspace of an exact shape (tests / bench probes)."""
        return self._ws[(B, T, R)]

    def fill_args(self, ws, enc, B, T, R, has_dropout, dalpha_ext=None):
        S, t = self.store, ws["t"]
        a = _lib.DecoderArgs()
        a.B, a.T, a.R = B, T, R
        a.C, a.A, a.D, a.E, a.V = self.encoder_dim, self.attention_dim, self.decoder_dim, self.embed_dim, self.vocab_size
        a.dt = _dt(self.precision)
        a.impl = _lib.LO_IMPL_TC if (self.impl == "tc" and self.precision == "bf16") else _lib.LO_IMPL_SIMT
        a.has_dropout = int(has_dropout)           # 0 eval, 1 injected mask, 2 in-kernel Philox
        a.dropout_state = self.dropout_state.data_ptr()
        a.dropout_p = float(self.dropout_p)
        a.ldl = ws["ldl"]
        a.alpha_c = float(self.alpha_c)
        a.bt_host = ctypes.cast(ws["bt"], ctypes.c_void_p)
        a.caps = t["caps"].data_ptr()
        a.caps_stride = t["caps"].stride(0)
        a.enc = enc.data_ptr()

        def W(name):
            return S.w(name).data_ptr()

        def F(name):
            return S.f32(name).data_ptr()

        def Gd(name):
            return S.g(name).data_ptr()

        a.w_enc_att, a.b_enc_att = W("attention.encoder_att.weight"), F("attention.encoder_att.bias")
        a.wcat1, a.bcat1 = W("attention.decoder_att.weight"), F("attention.decoder_att.bias")
        a.w_full = F("attention.full_att.weight")
        a.emb = W("embedding.weight")
        a.w_ih, a.b_ih = W("decode_step.weight_ih"), F("decode_step.bias_ih")
        a.w_init, a.b_init = W("init_h.weight"), F("init_h.bias")
        a.w_fc, a.b_fc = W("fc.weight"), F("fc.bias")
        for k in ("att1", "ptab", "mean", "hall", "call", "out1", "alphas", "ctx", "gctx", "gates", "gtmp", "hd", "logits",
                  "row_loss", "loss", "sreg", "work"):
            setattr(a, k, t[k].data_ptr())
        if t.get("dropout_mask") is not None:
            a.dropout_mask = t["dropout_mask"].data_ptr()
        if ws["need_grad"]:
            for k in ("wbwd1", "wbwd2", "dlogits", "dhd", "dreg", "dcat", "dxh", "dc", "dctx", "de", "dptab", "datt1", "denc",
                      "dinit", "dmean", "att_mask"):
                setattr(a, k, t[k].data_ptr())
            a.g_w_enc_att, a.g_b_enc_att = Gd("attention.encoder_att.weight"), Gd("attention.encoder_att.bias")
            a.g_wcat1, a.g_bcat1 = Gd("attention.decoder_att.weight"), Gd("attention.decoder_att.bias")
            a.g_w_full, a.g_b_full = Gd("attention.full_att.weight"), Gd("attention.full_att.bias")
            a.g_emb = Gd("embedding.weight")
            a.g_w_ih, a.g_b_ih = Gd("decode_step.weight_ih"), Gd("decode_step.bias_ih")
            a.g_w_init, a.g_b_init = Gd("init_h.weight"), Gd("init_h.bias")
            a.g_w_fc, a.g_b_fc = Gd("fc.weight"), Gd("fc.bias")
        if dalpha_ext is not None:
            a.dalpha_ext = dalpha_ext.data_ptr()
        if a.impl == _lib.LO_IMPL_TC:
            if "bfwork" not in t:
                t["bfwork"] = torch.zeros(int(_lib.lib().lo_decoder_bfwork_bytes(ctypes.byref(a))), dtype=torch.uint8, device=S.device)
            a.bfwork = t["bfwork"].data_ptr()
        ws["args"] = a
        return a

    def set_lengths(self, ws, decode_lengths, B, T):
        """bt[t] = number of rows still decoding at step t (seq2seq_torch.py:308)."""
        for t in range(T):
            ws["bt"][t] = sum(1 for l in decode_lengths if l > t)

    def init_hidden_state(self, encoder_out):
        """seq2seq_torch.py:255-265 (stand-alone; the fused path computes it inside lo_decoder_forward)."""
        L = _lib.lib()
        with torch.no_grad():
            S, st, dt = self.store, stream_ptr(), _dt(self.precision)
            self.sync_shadow()
            m = encoder_out.float().mean(dim=1).contiguous()      # plumbing; the hot path uses mean_rows_kernel
            B, C, D = m.shape[0], self.encoder_dim, self.decoder_dim
            hc = torch.empty(2, B, D, dtype=torch.float32, device=m.device)
            for i, n in enumerate(("init_h", "init_c")):
                check(L.lo_gemm(ptr(m), _lib.LO_F32, ptr(S.w(n + ".weight")), dt, ptr(hc[i]), _lib.LO_F32, B, D, C, C, 1, 1, C, D,
                                1, 0, 0, 0, ptr(S.f32(n + ".bias")), 0, 0, _lib.LO_IMPL_SIMT, st))
            return hc[0], hc[1]

    def run_phase(self, ws, phase, backward, with_loss=True):
        """Extension hook (a second layer between the cell and fc, latex_ocr_b200/ext.py): re-enter the C entry points with
        ``lo_decoder_args.phase`` = 1 (time loop only) or 2 (fc head + loss only) on the argument block of run_forward.
        ``with_loss=False``: forward of the head without the loss (the workspace of a no-gradient run_forward)."""
        a = ws["args"]
        a.phase = int(phase)
        try:
            L = _lib.lib()
            if backward:
                check(L.lo_decoder_backward(ctypes.byref(a), stream_ptr()))
            else:
                check(L.lo_decoder_forward(ctypes.byref(a), 1 if with_loss else 0, stream_ptr()))
        finally:
            a.phase = 0

    def run_forward(self, enc_flat, caps_sorted, decode_lengths, with_loss, need_grad, dropout_mask=None, phase=0):
        """enc_flat: storage-dtype CUDA [B,R,C] (sorted rows); caps_sorted: CUDA int64 [B,T+1].
        dropout_mask: None (no dropout), a [B,T,D] tensor of multipliers (injected, parity tests) or the string "philox"
        (mask drawn inside the kernels)."""
        L = _lib.lib()
        B, R, _ = enc_flat.shape
        T = max(decode_lengths)
        ws = self.workspace(B, T, R, need_grad)
        self.sync_shadow()
        ws["t"]["caps"].copy_(caps_sorted[:, :T + 1])
        self.set_lengths(ws, decode_lengths, B, T)
        has_do = 0 if dropout_mask is None else (2 if isinstance(dropout_mask, str) else 1)
        if has_do == 1:
            if ws["t"].get("dropout_mask") is None:
                ws["t"]["dropout_mask"] = torch.zeros(B, T, self.decoder_dim, dtype=torch.float32, device=self.store.device)
                ws.pop("args", None)
            ws["t"]["dropout_mask"].copy_(dropout_mask)
        a = self.fill_args(ws, enc_flat, B, T, R, has_do)
        a.phase = int(phase)
        try:
            check(L.lo_decoder_forward(ctypes.byref(a), 1 if with_loss else 0, stream_ptr()))
        finally:
            a.phase = 0
        return ws

    def run_backward(self, ws):
        check(_lib.lib().lo_decoder_backward(ctypes.byref(ws["args"]), stream_ptr()))

    def make_dropout_mask(self, B, T, materialize=False):
        """Dropout of h before fc (seq2seq_torch.py:316).  Training mode: "philox" = the inverted-dropout multipliers are drawn
        inside the LSTM kernels (csrc/lo_common.cuh:philox_dropout_mult) and redrawn in the backward — no mask tensor, no torch
        RNG launch; ``materialize=True`` returns the [B,T,D] tensor of torch-drawn multipliers instead (the injected-mask path
        the parity tests use)."""
        p = self.dropout_p
        if not self.training or p <= 0.0:
            return None
        if not materialize:
            return "philox"
        keep = torch.rand(B, T, self.decoder_dim, device=self.store.device) >= p
        return keep.float() / (1.0 - p)

    def forward(self, encoder_out, encoded_captions, caption_lengths):
        """Reference signature and return tuple (seq2seq_torch.py:267-320): (predictions[B,maxT,V],
        sorted captions, decode_lengths(list), alphas[B,maxT,R], sort_ind).  Inference-style call (no
        autograd graph); training goes through Img2SeqModel.getLoss which fuses loss and backward."""
        if not encoder_out.is_cuda:
            raise _lib.LatexOcrB200Error("DecoderWithAttention runs on CUDA tensors only (no CPU fallback)")
        with torch.no_grad():
            B = encoder_out.size(0)
            C = encoder_out.size(-1)
            enc = encoder_out.reshape(B, -1, C)
            lens, sort_ind = caption_lengths.squeeze(1).sort(dim=0, descending=True)     # :286
            sort_ind_dev = sort_ind.to(enc.device)
            enc = enc[sort_ind_dev].contiguous().to(self.tdtype)
            caps = encoded_captions.to(enc.device)[sort_ind_dev].contiguous()
            decode_lengths = (lens - 1).tolist()                                           # :298
            T = max(decode_lengths)
            mask = self.make_dropout_mask(B, T)
            ws = self.run_forward(enc, caps, decode_lengths, with_loss=False, need_grad=False, dropout_mask=mask)
            if isinstance(mask, str):
                self.dropout_state[1] += 1       # forward-only call: no lo_decoder_backward to advance the Philox call counter
            preds = ws["t"]["logits"][:, :, :self.vocab_size].clone()
            alphas = ws["t"]["alphas"].clone()
            if min(decode_lengths) < T:      # rows that stopped decoding keep zeros (:301-302, :317-318)
                act = torch.arange(T, device=enc.device)[None, :] < torch.tensor(decode_lengths, device=enc.device)[:, None]
                preds = preds * act[:, :, None]
                alphas = alphas * act[:, :, None]
            return preds, caps, decode_lengths, alphas, sort_ind_dev
