// Greedy / beam decode loops of the torch-flavour decoder, with an optional second decoder layer (EXTENSION, BASELINE.json
// configs[3]: layer 2 = nn.LSTMCell(D, D) over h1_t, logits_t = fc(h2_t); semantics defined by oracle/ref_ext.py).  Part of the
// lo_decoder.cu translation unit, included before its C entry points because lo_decoder_greedy_hist / lo_decoder_beam_div run
// these loops too (with no layer-2 block); it needs the file-static forward_step, argmax_kernel, beam_step_kernel and
// gather_rows_kernel.
//
// Training hoists layer 2 into one sequence LSTM after the time loop (lo_decoder_args.phase 1 / 2).  Decoding cannot: token t+1
// depends on fc(h2_t), so layer 2 runs inside the loop, after forward_step(t) has written h1_t:
//   gates2 = h1_t W_ih^T            (GEMM, overwrites the gates scratch)
//   gates2 += h2_{t-1} W_hh^T       (GEMM, accumulating)
//   cell: (gates2 + b_ih + b_hh, c2_{t-1}) -> h2_t (fp32 + bf16 mirror), c2_t
// Two accumulating GEMM launches, so three dependent launches per step more than the one-layer loop.  The state lives in
// ping-pong slots: greedy alternates them; beam search keeps its state in slot 0, the cell writes slot 1 and the gather by
// parents brings it back to slot 0 (no device-to-device copy).

namespace lo {

struct Dec2Ws {
  float* h;      // f32 [2][B][D]
  float* c;      // f32 [2][B][D]
  bf16* h_bf;    // bf16 [2][B][D] mirror of h (A operand of the tensor-core GEMMs)
  float* gates;  // f32 [B][4D] pre-activations without the biases
  size_t bytes;
};

static Dec2Ws dec2_carve(void* ws, int B, int D) {
  char* base = (char*)ws;
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* {
    void* p = base ? base + off : nullptr;
    off += (bytes + 255) & ~(size_t)255;
    return p;
  };
  const size_t BD = (size_t)B * D;
  Dec2Ws w{};
  w.h = (float*)take(2 * BD * 4);
  w.c = (float*)take(2 * BD * 4);
  w.h_bf = (bf16*)take(2 * BD * 2);
  w.gates = (float*)take(4 * BD * 4);
  w.bytes = off;
  return w;
}

// nn.LSTMCell pointwise part, gate order i,f,g,o: pre = gates2 + b_ih + b_hh.  The biases and c_{t-1} are at least two launches old
// (parameters; the previous step's cell or gather), so they are fetched BEFORE griddepcontrol.wait, as in lstm_pw_fwd_kernel.
__global__ void dec2_cell_kernel(const float* __restrict__ gates, const float* __restrict__ b_ih, const float* __restrict__ b_hh,
                                 const float* __restrict__ c_prev, float* __restrict__ c_out, float* __restrict__ h_out,
                                 bf16* __restrict__ h_bf, int nrows, int D) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = idx < nrows * D;
  const int b = live ? idx / D : 0, j = live ? idx % D : 0;
  float bs[4] = {0.f, 0.f, 0.f, 0.f}, cp = 0.f;
  if (live) {
#pragma unroll
    for (int q = 0; q < 4; q++) bs[q] = b_ih[q * D + j] + b_hh[q * D + j];
    cp = c_prev[idx];
  }
  pdl_wait();
  pdl_trigger();
  if (!live) return;
  const float* g = gates + (int64_t)b * 4 * D;
  const float i = sigmoidf_(g[j] + bs[0]), f = sigmoidf_(g[D + j] + bs[1]), gg = tanhf(g[2 * D + j] + bs[2]),
              o = sigmoidf_(g[3 * D + j] + bs[3]);
  const float c = f * cp + i * gg;
  const float h = o * tanhf(c);
  c_out[idx] = c;
  h_out[idx] = h;
  if (h_bf) h_bf[idx] = __float2bfloat16_rn(h);
}

// layer-2 state by parents (gather_helper, beam_search_decoder_cell.py:370-391): dst[r] = src[rows[r]] for h, c and the bf16 h
__global__ void dec2_gather_kernel(const float* __restrict__ h_src, const float* __restrict__ c_src, const bf16* __restrict__ hb_src,
                                   const int32_t* __restrict__ rows, float* __restrict__ h_dst, float* __restrict__ c_dst,
                                   bf16* __restrict__ hb_dst, int n, int D) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * D) return;
  const int r = idx / D, j = idx % D;
  const int64_t s = (int64_t)rows[r] * D + j;
  h_dst[idx] = h_src[s];
  c_dst[idx] = c_src[s];
  if (hb_dst) hb_dst[idx] = hb_src[s];
}

static int dec2_check(const lo_decoder_args* a, const lo_dec2_args* l2) {
  LO_CHECK_ARG(l2 != nullptr, "null layer-2 block");
  LO_CHECK_ARG(a != nullptr, "args");
  LO_CHECK_ARG(l2->D == a->D, "layer-2 D must equal the decoder's D");
  // the attention workspace keeps one ticket counter per row in its first 4 KiB
  LO_CHECK_ARG(a->B <= 1024, "B <= 1024 rows (images * beam)");
  LO_CHECK_ARG(l2->dt == LO_F32 || l2->dt == LO_BF16, "layer-2 dt");
  LO_CHECK_ARG(l2->w_ih && l2->w_hh && l2->b_ih && l2->b_hh && l2->ws, "null layer-2 pointer");
  return LO_OK;
}

// zero initial state in slot 0
static int dec2_begin(const lo_dec2_args* l2, const Dims& d, cudaStream_t st) {
  const Dec2Ws w = dec2_carve(l2->ws, d.B, d.D);
  const size_t BD = (size_t)d.B * d.D;
  LO_CUDA(cudaMemsetAsync(w.h, 0, BD * 4, st));
  LO_CUDA(cudaMemsetAsync(w.c, 0, BD * 4, st));
  LO_CUDA(cudaMemsetAsync(w.h_bf, 0, BD * 2, st));
  return LO_OK;
}

// one layer-2 step after forward_step(t): reads h1_t and slot s_in, writes slot s_out
static int dec2_step(const lo_decoder_args* a, const lo_dec2_args* l2, const Dims& d, const BfViews& bv, int t, int s_in, int s_out,
                     cudaStream_t st) {
  const Dec2Ws w = dec2_carve(l2->ws, d.B, d.D);
  const int B = d.B, D = d.D, G = d.G;
  const int64_t BD = (int64_t)B * D;
  if (bv.on && l2->impl == LO_IMPL_TC && l2->dt == LO_BF16) {
    const bf16* x = bv.hall + (int64_t)(t + 1) * BD;
    const bf16* h = w.h_bf + s_in * BD;
    if (g_opt_skinny_mma && B <= 64) {
      LO_TRY(skinny_gemm_nt(x, D, (const bf16*)l2->w_ih, D, w.gates, G, B, G, D, nullptr, 1, 0, st));
      LO_TRY(skinny_gemm_nt(h, D, (const bf16*)l2->w_hh, D, w.gates, G, B, G, D, nullptr, 1, 1, st));
    } else {
      LO_TRY(tc_gemm_nt_ex(x, D, (const bf16*)l2->w_ih, D, w.gates, LO_F32, G, B, G, D, nullptr, 0, 0, 1, 0, 1, st));
      LO_TRY(tc_gemm_nt_ex(h, D, (const bf16*)l2->w_hh, D, w.gates, LO_F32, G, B, G, D, nullptr, 1, 0, 1, 0, 1, st));
    }
  } else {
    // CUDA cores (fp32: the tight-parity path); h operands from the bf16 mirrors when the decoder keeps them
    const void* x = bv.on ? (const void*)(bv.hall + (int64_t)(t + 1) * BD) : (const void*)(a->hall + (int64_t)(t + 1) * BD);
    const void* h = bv.on ? (const void*)(w.h_bf + s_in * BD) : (const void*)(w.h + s_in * BD);
    const int dtx = bv.on ? LO_BF16 : LO_F32;
    LO_TRY(gemm_nt(x, dtx, D, l2->w_ih, l2->dt, D, w.gates, LO_F32, G, B, G, D, nullptr, 0, 0, LO_IMPL_SIMT, st));
    LO_TRY(gemm_nt(h, dtx, D, l2->w_hh, l2->dt, D, w.gates, LO_F32, G, B, G, D, nullptr, 1, 0, LO_IMPL_SIMT, st));
  }
  LO_CUDA(launch_pdl(dec2_cell_kernel, dim3(cdiv(BD, 256)), dim3(256), (size_t)0, st, (const float*)w.gates, l2->b_ih, l2->b_hh,
                     (const float*)(w.c + s_in * BD), w.c + s_out * BD, w.h + s_out * BD, bv.on ? w.h_bf + s_out * BD : (bf16*)nullptr,
                     B, D));
  LO_LAUNCH_OK();
  return LO_OK;
}

// A operand of the fc head at step t: h2_t (slot s) with layer 2, else h1_t; the bf16 mirror when the decoder keeps them
struct FcInput {
  const void* x;
  int dt, impl;
};
static inline FcInput fc_input(const lo_decoder_args* a, const lo_dec2_args* l2, const Dims& d, const BfViews& bv, int t, int s) {
  const int64_t BD = (int64_t)d.B * d.D;
  if (l2) {
    const Dec2Ws w = dec2_carve(l2->ws, d.B, d.D);
    if (bv.on) return FcInput{w.h_bf + s * BD, LO_BF16, LO_IMPL_TC};
    return FcInput{w.h + s * BD, LO_F32, LO_IMPL_SIMT};
  }
  if (bv.on) return FcInput{bv.hall + (int64_t)(t + 1) * BD, LO_BF16, LO_IMPL_TC};
  return FcInput{a->hall + (int64_t)(t + 1) * BD, LO_F32, LO_IMPL_SIMT};
}

static int greedy_loop(const lo_decoder_args* a, const lo_dec2_args* l2, int64_t start_id, int64_t end_id, int max_steps,
                       int64_t* tokens, int32_t* finished, int32_t* fin_hist, cudaStream_t st) {
  LO_TRY(check_args(a));
  LO_CHECK_ARG(tokens && finished && max_steps > 0 && max_steps <= a->T, "tokens/finished/max_steps (<= T capacity)");
  const Dims d = dims(a);
  int64_t* next_tok = (int64_t*)a->sreg;          // scratch: [B] int64 fits in sreg [B][>=2] floats
  fill_i64_kernel<<<cdiv(d.B, 128), 128, 0, st>>>(next_tok, start_id, d.B);
  LO_LAUNCH_OK();
  LO_CUDA(cudaMemsetAsync(finished, 0, (size_t)d.B * 4, st));
  LO_TRY(forward_prologue(a, d, st));
  const BfViews bvg = bf_views(a, d);
  if (l2) LO_TRY(dec2_begin(l2, d, st));
  for (int t = 0; t < max_steps; t++) {
    LO_TRY(forward_step(a, d, t, Rows{0, d.B, a->work, 0}, next_tok, 1, nullptr, 0, nullptr, st));
    if (l2) LO_TRY(dec2_step(a, l2, d, bvg, t, t & 1, (t + 1) & 1, st));
    // logits_t = fc(h_t)   (no dropout at decode time); bf16 mirror: mma.sync kernel for <= 64 rows (the dispatcher falls back to
    // CUDA cores otherwise)
    const FcInput fi = fc_input(a, l2, d, bvg, t, (t + 1) & 1);
    LO_TRY(gemm_nt(fi.x, fi.dt, d.D, a->w_fc, fi.dt == LO_BF16 ? LO_BF16 : a->dt, d.D, a->logits, LO_F32, d.V, d.B, d.V, d.D, a->b_fc, 0,
                   0, fi.impl, st));
    argmax_kernel<<<cdiv(d.B, 8), 256, 0, st>>>(a->logits, d.V, tokens + t, max_steps, next_tok, finished, end_id, d.B);
    LO_LAUNCH_OK();
    if (fin_hist) {
      fin_hist_kernel<<<cdiv(d.B, 128), 128, 0, st>>>(finished, fin_hist + t, max_steps, d.B);
      LO_LAUNCH_OK();
    }
  }
  return LO_OK;
}

static int beam_loop(const lo_decoder_args* a, const lo_dec2_args* l2, int64_t start_id, int64_t end_id, int max_steps, int64_t* ids,
                     int64_t* parents, int32_t* fin_hist, float* logp, float div_gamma, float div_prob, const float* div_u,
                     const uint64_t* div_state, cudaStream_t st) {
  LO_TRY(check_args(a));
  const bool div_on = !(div_gamma == 1.f || div_prob == 0.f);               // beam_search_decoder_cell.py:270-273
  LO_CHECK_ARG(!div_on || (div_gamma > 0.f && (div_u || div_state)), "diversity penalty needs gamma > 0 and div_u or div_state");
  const int beam = a->rows_per_img;
  LO_CHECK_ARG(beam >= 1 && beam <= LO_BEAM_MAX && a->B % beam == 0, "1 <= beam (rows_per_img) <= 16, B % beam == 0");
  LO_CHECK_ARG(ids && parents && fin_hist && logp && max_steps > 0 && max_steps <= a->T, "outputs / max_steps (<= T capacity)");
  LO_CHECK_ARG((size_t)beam * a->V * 4 * (div_on ? 2 : 1) <= 200 * 1024, "beam*V too large for the shared-memory top-k");
  const Dims d = dims(a);
  const int n_img = d.B / beam;
  // scratch: next tokens (int64 [B]) in sreg, finished + parent rows (int32 [B] each) in row_loss
  int64_t* next_tok = (int64_t*)a->sreg;
  int32_t* finished = (int32_t*)a->row_loss;
  int32_t* parent_rows = finished + d.B;
  LO_CHECK_ARG((int64_t)d.B * d.T >= 2 * d.B, "row_loss scratch too small");
  fill_i64_kernel<<<cdiv(d.B, 128), 128, 0, st>>>(next_tok, start_id, d.B);
  LO_LAUNCH_OK();
  LO_CUDA(cudaMemsetAsync(finished, 0, (size_t)d.B * 4, st));
  LO_CUDA(cudaMemsetAsync(logp, 0, (size_t)d.B * 4, st));          // initial log-probs are zeros (:106-107)
  LO_TRY(forward_prologue(a, d, st));
  const BfViews bv = bf_views(a, d);
  if (l2) LO_TRY(dec2_begin(l2, d, st));
  const size_t smem = (size_t)beam * d.V * 4 * (div_on ? 2 : 1);
  static bool attr = false;
  if (!attr && smem > 48 * 1024) {
    LO_CUDA(cudaFuncSetAttribute(beam_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr = true;
  }
  for (int t = 0; t < max_steps; t++) {
    LO_TRY(forward_step(a, d, t, Rows{0, d.B, a->work, 0}, next_tok, 1, nullptr, 0, nullptr, st));
    if (l2) LO_TRY(dec2_step(a, l2, d, bv, t, 0, 1, st));
    float* h_new = a->hall + (int64_t)(t + 1) * d.B * d.D;
    float* c_new = a->call + (int64_t)(t + 1) * d.B * d.D;
    // logits; bf16 mirror -> mma.sync kernel (row blocks of 64), CUDA cores otherwise
    const FcInput fi = fc_input(a, l2, d, bv, t, 1);
    LO_TRY(gemm_nt(fi.x, fi.dt, d.D, a->w_fc, fi.dt == LO_BF16 ? LO_BF16 : a->dt, d.D, a->logits, LO_F32, d.V, d.B, d.V, d.D, a->b_fc, 0,
                   0, fi.impl, st));
    beam_step_kernel<<<n_img, 256, smem, st>>>(a->logits, d.V, beam, t, end_id, logp, finished, ids, parents, fin_hist, next_tok,
                                               parent_rows, max_steps, div_on ? logf(div_gamma) : 0.f, div_on ? div_prob : 0.f,
                                               div_u ? div_u + (int64_t)t * d.B * d.V : (const float*)nullptr,
                                               (const unsigned long long*)div_state);
    LO_LAUNCH_OK();
    // reorder the recurrent state by parents (through gtmp as a temporary)
    gather_rows_kernel<<<cdiv((long)d.B * d.D, 256), 256, 0, st>>>(h_new, parent_rows, a->gtmp, d.B, d.D);
    LO_LAUNCH_OK();
    gather_rows_kernel<<<cdiv((long)d.B * d.D, 256), 256, 0, st>>>(c_new, parent_rows, a->gtmp + (int64_t)d.B * d.D, d.B, d.D);
    LO_LAUNCH_OK();
    LO_CUDA(cudaMemcpyAsync(h_new, a->gtmp, (size_t)d.B * d.D * 4, cudaMemcpyDeviceToDevice, st));
    LO_CUDA(cudaMemcpyAsync(c_new, a->gtmp + (int64_t)d.B * d.D, (size_t)d.B * d.D * 4, cudaMemcpyDeviceToDevice, st));
    if (bv.on) LO_TRY(lo_cast(h_new, LO_F32, bv.hall + (int64_t)(t + 1) * d.B * d.D, LO_BF16, (int64_t)d.B * d.D, (void*)st));
    if (l2) {
      // layer 2: slot 1 (this step's cell) -> slot 0 by parents
      const Dec2Ws w = dec2_carve(l2->ws, d.B, d.D);
      const int64_t BD = (int64_t)d.B * d.D;
      dec2_gather_kernel<<<cdiv(BD, 256), 256, 0, st>>>(w.h + BD, w.c + BD, w.h_bf + BD, parent_rows, w.h, w.c,
                                                        bv.on ? w.h_bf : (bf16*)nullptr, d.B, d.D);
      LO_LAUNCH_OK();
    }
  }
  return LO_OK;
}

}  // namespace lo

extern "C" {

int64_t lo_sizeof_dec2_args(void) { return (int64_t)sizeof(lo_dec2_args); }

int64_t lo_dec2_workspace_bytes(int B, int D) {
  if (B <= 0 || D <= 0) return 0;
  return (int64_t)lo::dec2_carve(nullptr, B, D).bytes;
}

int lo_decoder2_greedy_hist(const lo_decoder_args* a, const lo_dec2_args* l2, int64_t start_id, int64_t end_id, int max_steps,
                            int64_t* tokens, int32_t* finished, int32_t* fin_hist, void* stream) {
  LO_TRY(lo::dec2_check(a, l2));
  return lo::greedy_loop(a, l2, start_id, end_id, max_steps, tokens, finished, fin_hist, (cudaStream_t)stream);
}

int lo_decoder2_beam_div(const lo_decoder_args* a, const lo_dec2_args* l2, int64_t start_id, int64_t end_id, int max_steps,
                         int64_t* ids, int64_t* parents, int32_t* fin_hist, float* logp, float div_gamma, float div_prob,
                         const float* div_u, const uint64_t* div_state, void* stream) {
  LO_TRY(lo::dec2_check(a, l2));
  return lo::beam_loop(a, l2, start_id, end_id, max_steps, ids, parents, fin_hist, logp, div_gamma, div_prob, div_u, div_state,
                       (cudaStream_t)stream);
}

}  // extern "C"
