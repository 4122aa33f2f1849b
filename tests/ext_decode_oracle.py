"""TEST INFRASTRUCTURE ONLY — CPU definition of greedy / beam decoding for the two-layer extension decoder (latex_ocr_b200/ext.py
greedy_decode / beam_decode).  "Parity unpinned — extension": the reference has no such model.

The loops follow oracle/ref_decode.py's restatement of the reference's decode loop rule for rule and reuse its bookkeeping
(cell_step, add_div_penalty, _topk_low_index_first, backtrack); they differ only in taking a step function and a state tuple, so
that the state of any number of layers is tiled per beam and gathered by parents.  With one_layer_step they return exactly what
ref_decode.greedy_decode / beam_decode return (tests/test_ext_decode_cpu.py checks it).

  step(ctx, state, tok) -> (logits, state), ctx = (enc, att1) row-aligned with the state rows
  two-layer model: layer 1 = the attention LSTM (unchanged); h2, c2 = LSTMCell(h1_t, (h2, c2)), zero initial state, gate order
  i,f,g,o; logits_t = fc(h2_t); no dropout at decode time (oracle/ref_ext.py:decoder2_forward).
"""
import torch
import torch.nn.functional as F

from oracle import ref_decode as rd
from oracle import ref_model as rm


def one_layer_step(p):
    """DecoderWithAttention's step (ref_decode.cell_step); state (h, c)."""
    def step(ctx, state, tok):
        logits, h, c = rd.cell_step(p, ctx[0], ctx[1], state[0], state[1], tok)
        return logits, (h, c)
    return step


def lstm_cell2(p2, x, h2, c2):
    """Layer 2: nn.LSTMCell(D, D), the arithmetic of ref_ext.decoder2_forward."""
    g = F.linear(x, p2["cell.weight_ih"], p2["cell.bias_ih"]) + F.linear(h2, p2["cell.weight_hh"], p2["cell.bias_hh"])
    i, f, gg, o = g.chunk(4, dim=1)
    c2 = torch.sigmoid(f) * c2 + torch.sigmoid(i) * torch.tanh(gg)
    h2 = torch.sigmoid(o) * torch.tanh(c2)
    return h2, c2


def two_layer_step(pd, p2):
    """Two-layer decode step; state (h1, c1, h2, c2).  Layer 1's own fc output is discarded."""
    def step(ctx, state, tok):
        h1, c1, h2, c2 = state
        _, h1, c1 = rd.cell_step(pd, ctx[0], ctx[1], h1, c1, tok)
        h2, c2 = lstm_cell2(p2, h1, h2, c2)
        return F.linear(h2, pd["fc.weight"], pd["fc.bias"]), (h1, c1, h2, c2)
    return step


def initial_state(pd, enc):
    """(h1, c1, h2, c2) at step 0: init_hidden_state for layer 1, zeros for layer 2."""
    h, c = rm.init_hidden_state(pd, enc)
    return h, c, torch.zeros_like(h), torch.zeros_like(c)


def greedy_loop(p, enc, start_id, end_id, max_iter, step, state):
    """ref_decode.greedy_decode with a step function.  enc [N,R,C] -> ids [N, steps]."""
    N = enc.shape[0]
    att1 = F.linear(enc, p["attention.encoder_att.weight"], p["attention.encoder_att.bias"])
    tok = torch.full((N,), start_id, dtype=torch.long)
    finished = torch.zeros(N, dtype=torch.bool)
    out = []
    time = 0
    while not bool(finished.all()):
        logits, state = step((enc, att1), state, tok)
        ids = torch.argmax(logits, dim=-1)
        out.append(ids)
        finished = finished | (ids == end_id)
        finished = finished | torch.tensor(time >= max_iter)
        tok = ids
        time += 1
    return torch.stack(out, dim=1)


def beam_loop(p, enc, start_id, end_id, beam, max_iter, step, state, finalize="reference", div_gamma=1.0, div_prob=0.0, div_u=None):
    """ref_decode.beam_decode with a step function; every tensor of `state` (one row per image) is tiled per beam and gathered by
    parents.  Returns ids [N, steps, beam] and the final log-probs [N, beam]."""
    N = enc.shape[0]
    V = p["fc.weight"].shape[0]
    att1 = F.linear(enc, p["attention.encoder_att.weight"], p["attention.encoder_att.bias"])
    ctx = (enc.repeat_interleave(beam, dim=0), att1.repeat_interleave(beam, dim=0))
    state = tuple(s.repeat_interleave(beam, dim=0) for s in state)
    tok = torch.full((N * beam,), start_id, dtype=torch.long)
    log_probs = torch.zeros(N, beam)
    finished = torch.zeros(N, beam, dtype=torch.bool)
    ids_t, parents_t = [], []
    time = 0
    fmin = torch.finfo(torch.float32).min
    while not bool(finished.all()):
        logits, state = step(ctx, state, tok)
        step_lp = torch.log_softmax(logits.view(N, beam, V), dim=-1)
        one_hot = torch.full((V,), fmin)
        one_hot[end_id] = 0.0
        f = finished.unsqueeze(-1).float()
        step_lp = (1.0 - f) * step_lp + f * one_hot
        lp = log_probs.unsqueeze(-1) + step_lp
        if div_u is not None:
            lp = rd.add_div_penalty(lp, div_gamma, div_prob, div_u[time].view(N, beam, V))
        flat = lp.reshape(N, beam * V) if time > 0 else lp[:, 0]
        new_probs, idx = rd._topk_low_index_first(flat, beam)
        new_ids = idx % V
        new_parents = idx // V
        finished = torch.gather(finished, 1, new_parents) | (new_ids == end_id)
        rows = (new_parents + torch.arange(N).unsqueeze(1) * beam).view(-1)
        state = tuple(s[rows] for s in state)
        log_probs = new_probs
        ids_t.append(new_ids)
        parents_t.append(new_parents)
        finished = finished | torch.tensor(time >= max_iter)
        tok = new_ids.view(-1)
        time += 1
    ids = torch.stack(ids_t, dim=1)
    if finalize == "reference":
        return ids, log_probs
    return rd.backtrack(ids, torch.stack(parents_t, dim=1)), log_probs


def greedy_decode_ext(pd, p2, enc, start_id, end_id, max_iter):
    return greedy_loop(pd, enc, start_id, end_id, max_iter, two_layer_step(pd, p2), initial_state(pd, enc))


def beam_decode_ext(pd, p2, enc, start_id, end_id, beam, max_iter, finalize="reference", div_gamma=1.0, div_prob=0.0, div_u=None):
    return beam_loop(pd, enc, start_id, end_id, beam, max_iter, two_layer_step(pd, p2), initial_state(pd, enc), finalize, div_gamma,
                     div_prob, div_u)
