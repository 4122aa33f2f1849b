"""Greedy / beam-search decoding on the B200 step kernels — the decode row of SURVEY.md §8 (a8).

Loop semantics follow the reference's TF decode loop, which is framework independent:
  dynamic_decode (model/components/dynamic_decode.py:38-61): run until every row is finished, at most
  max_length_formula + 2 steps (``finished |= time >= max_iter`` with max_iter = max_length_formula + 1, decoder.py:70);
  greedy (greedy_decoder_cell.py:53-66): id = argmax, finished |= id == END, rows keep decoding after END;
  beam (beam_search_decoder_cell.py:123-250): see include/latex_ocr_b200.h:lo_decoder_beam; ``finalize='reference'``
  reproduces the reference's identity finalize (its back-tracking loop never updates ``parents``, :237), ``'backtrack'``
  returns lineage-consistent hypotheses.
The torch flavour of the reference has no START symbol; the caller supplies ``start_id`` (SURVEY.md §8-c).
"""
import ctypes

import torch

from . import _lib
from ._lib import check, stream_ptr


def _n_steps(fin_hist):
    """fin_hist [N, steps(, beam)] int32 -> number of loop iterations the reference would have executed."""
    N = fin_hist.shape[0]
    S = fin_hist.shape[1]
    allf = fin_hist.reshape(N, S, -1).all(dim=2).all(dim=0)          # [S]
    idx = torch.nonzero(allf)
    return int(idx[0]) + 1 if idx.numel() else S


def _prepare(model, img, rows_per_img, max_steps):
    enc = model.encoder.forward_raw(img.to(model.device).float(), need_grad=False)
    return _prepare_enc(model, enc, rows_per_img, max_steps)


def _prepare_enc(model, enc, rows_per_img, max_steps):
    """enc: the storage-dtype encoder output [N,H',W',C] (CUDA) -> (decoder argument block, workspace, N)."""
    N = enc.shape[0]
    R = enc.shape[1] * enc.shape[2]
    enc_flat = enc.view(N, R, enc.shape[3])
    dec = model.decoder
    B = N * rows_per_img
    ws = dec.workspace(B, max_steps, R, need_grad=False)
    dec.sync_shadow()
    for t in range(max_steps):
        ws["bt"][t] = B
    a = dec.fill_args(ws, enc_flat, B, max_steps, R, has_dropout=False)
    a.rows_per_img = rows_per_img
    return a, ws, N


def greedy_decode(model, img, start_id, end_id, max_length_formula=150, return_attention=False):
    """Returns token ids [N, steps] (CPU int64), steps as the reference's loop would have run.  ``return_attention=True`` also
    returns the attention weights of every step, [N, steps, R] fp32 on the CPU — what the reference collects in
    ``attention_mechanism.ctx_vector`` for visualize_attention.py (attention_mechanism.py:96-121)."""
    L = _lib.lib()
    return _greedy(model, lambda rows, steps: _prepare(model, img, rows, steps),
                   lambda a, *args: L.lo_decoder_greedy_hist(ctypes.byref(a), *args),
                   start_id, end_id, max_length_formula, return_attention)


def _greedy(model, prepare, launch, start_id, end_id, max_length_formula, return_attention):
    """The greedy loop of any decoder flavour: prepare(rows_per_img, max_steps) -> (args, workspace, N) encodes the images;
    launch(args, start_id, end_id, max_steps, tokens, finished, fin_hist, stream) runs the C loop."""
    max_steps = max_length_formula + 2
    with torch.no_grad():
        a, ws, N = prepare(1, max_steps)
        dev = model.device
        tokens = torch.zeros(N, max_steps, dtype=torch.int64, device=dev)
        finished = torch.zeros(N, dtype=torch.int32, device=dev)
        hist = torch.zeros(N, max_steps, dtype=torch.int32, device=dev)
        check(launch(a, int(start_id), int(end_id), max_steps, tokens.data_ptr(), finished.data_ptr(), hist.data_ptr(), stream_ptr()))
        n = _n_steps(hist.cpu())
        if return_attention:
            return tokens[:, :n].cpu(), ws["t"]["alphas"][:, :n].float().cpu()
        return tokens[:, :n].cpu()


def attention_maps(alphas, att_h, att_w):
    """visualize_attention.py:49-72 (getOutArray): an attention vector over the R = att_h * att_w regions as a grey image,
    region r at (r // att_w, r % att_w), value (1 - alpha) * 255 (dark = attended).  alphas [..., R] -> float [..., att_h, att_w]."""
    a = torch.as_tensor(alphas, dtype=torch.float32)
    if a.shape[-1] != att_h * att_w:
        raise ValueError("attention vector of %d regions does not match a %dx%d feature map" % (a.shape[-1], att_h, att_w))
    return ((1.0 - a) * 255.0).reshape(tuple(a.shape[:-1]) + (att_h, att_w))


def beam_decode(model, img, start_id, end_id, beam_size=5, max_length_formula=150, finalize="reference",
                div_gamma=1, div_prob=0, div_u=None, div_seed=None):
    """Returns (ids [N, beam, steps], log_probs [N, beam]) on the CPU; hypothesis 0 is the one the reference scores
    (img2seq.py:210).  ``div_gamma`` / ``div_prob``: the diversity penalty of beam_search_decoder_cell.py:258-287 (off when
    gamma == 1 or prob == 0, as in configs/model.json:15-16); its Bernoulli draws come from the in-kernel Philox stream seeded
    by ``div_seed`` (default: torch's initial seed), or from ``div_u`` — uniforms [steps, N*beam, V] — when given (tests)."""
    L = _lib.lib()
    return _beam(model, lambda rows, steps: _prepare(model, img, rows, steps),
                 lambda a, *args: L.lo_decoder_beam_div(ctypes.byref(a), *args),
                 start_id, end_id, beam_size, max_length_formula, finalize, div_gamma, div_prob, div_u, div_seed)


def _beam(model, prepare, launch, start_id, end_id, beam_size, max_length_formula, finalize, div_gamma, div_prob, div_u, div_seed):
    """The beam loop of any decoder flavour (see _greedy); launch takes the arguments of lo_decoder_beam_div after the args block."""
    if finalize not in ("reference", "backtrack"):
        raise NotImplementedError("finalize must be 'reference' or 'backtrack'")
    max_steps = max_length_formula + 2
    with torch.no_grad():
        a, ws, N = prepare(beam_size, max_steps)
        dev = model.device
        ids = torch.zeros(N, max_steps, beam_size, dtype=torch.int64, device=dev)
        parents = torch.zeros_like(ids)
        hist = torch.zeros(N, max_steps, beam_size, dtype=torch.int32, device=dev)
        logp = torch.zeros(N, beam_size, dtype=torch.float32, device=dev)
        div_on = not (div_gamma == 1 or div_prob == 0)
        u_dev = state = None
        if div_on and div_u is not None:
            u_dev = torch.as_tensor(div_u, dtype=torch.float32).to(dev).contiguous()
            if tuple(u_dev.shape) != (max_steps, N * beam_size, a.V):
                raise ValueError("div_u must be [max_length_formula + 2, N * beam, V]")
        elif div_on:
            seed = torch.initial_seed() if div_seed is None else int(div_seed)
            state = torch.tensor([seed & 0x7FFFFFFFFFFFFFFF, 0], dtype=torch.int64, device=dev)
        check(launch(a, int(start_id), int(end_id), max_steps, ids.data_ptr(), parents.data_ptr(), hist.data_ptr(), logp.data_ptr(),
                     float(div_gamma), float(div_prob), u_dev.data_ptr() if u_dev is not None else None,
                     state.data_ptr() if state is not None else None, stream_ptr()))
        n = _n_steps(hist.cpu())
        ids, parents = ids[:, :n].cpu(), parents[:, :n].cpu()
        if finalize == "backtrack":
            out = torch.zeros_like(ids)
            cur = torch.arange(beam_size).unsqueeze(0).repeat(N, 1)
            for t in range(n - 1, -1, -1):
                out[:, t] = torch.gather(ids[:, t], 1, cur)
                cur = torch.gather(parents[:, t], 1, cur)
            ids = out
        return ids.permute(0, 2, 1).contiguous(), logp.cpu()      # [N, beam, time] like img2seq.py:239-241


def truncate_end(list_of_ids, id_end):
    """model/evaluation/text.py:95-104."""
    out = []
    for seq in list_of_ids:
        seq = [int(t) for t in seq]
        out.append(seq[:seq.index(id_end)] if id_end in seq else seq)
    return out
