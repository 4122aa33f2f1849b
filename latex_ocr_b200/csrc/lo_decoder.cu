// Attention-LSTM decoder of the torch flavour (DecoderWithAttention, seq2seq_torch.py:195-320) with the
// loss of img2seq_torch.py:147-159: forward over T teacher-forced steps, hand-derived backward.
//
// Schedule (see DESIGN.md §4): everything that does not depend on the recurrence is hoisted out of the
// time loop (att1 = encoder_att(enc), the embedding->gate projection table, logits, every weight
// gradient, d att1 and d enc).  Inside the loop each step reads enc and att1 exactly ONCE in forward
// and ONCE in backward (the HBM roofline of SURVEY.md §8-d) and runs two skinny GEMMs.
#include "lo_common.cuh"
#include "lo_ptx.cuh"

namespace lo {

#define LO_ATT_THREADS 256
#define LO_ATT_WARPS 8
#define LO_ATT_MAXSPLIT 16

static inline int att_splits(int B) {
  int s = (444 + B - 1) / B;
  if (s < 1) s = 1;
  if (s > LO_ATT_MAXSPLIT) s = LO_ATT_MAXSPLIT;
  return s;
}

__device__ __forceinline__ float ldcg_f(const float* p) { return __ldcg(p); }

// ------------------------------------------------------------------------------------------------
// K5: attention forward for one step.  grid (nsplit, B), 256 threads.  Each warp streams rows of
// att1 and enc (16 B per lane per load), keeps an online-softmax state (m, l, acc[C/32]) in registers;
// CTA combine in smem, cross-CTA combine by the last CTA to finish (threadfence + ticket).
// NV = A/256 = C/256 vectors of 8 elements per lane.
// ------------------------------------------------------------------------------------------------
template <typename T, int NV>
__global__ void __launch_bounds__(LO_ATT_THREADS) attention_fwd_kernel(
    const T* __restrict__ att1, const T* __restrict__ enc, const float* __restrict__ att2, int64_t att2_stride,
    const float* __restrict__ wf, float* __restrict__ alpha, int64_t alpha_stride, float* __restrict__ ctx,
    float* __restrict__ gate_pre, int64_t gate_stride, float* __restrict__ gctx, bf16* __restrict__ gctx_bf, int R, int nsplit,
    int* __restrict__ counters, float* __restrict__ partials, int rpi) {
  constexpr int CH = NV * 256;   // A == C == CH
  const int b = blockIdx.y, sp = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int rps = (R + nsplit - 1) / nsplit;
  const int r0 = sp * rps, r1 = min(R, r0 + rps);
  float a2[NV * 8], wv[NV * 8], acc[NV * 8];
#pragma unroll
  for (int j = 0; j < NV; j++) {
    ld8(att2 + (int64_t)b * att2_stride + (j * 32 + lane) * 8, a2 + j * 8);
    ld8(wf + (j * 32 + lane) * 8, wv + j * 8);
#pragma unroll
    for (int i = 0; i < 8; i++) acc[j * 8 + i] = 0.f;
  }
  float m = -INFINITY, l = 0.f;
  const T* a1b = att1 + (int64_t)(b / rpi) * R * CH;
  const T* eb = enc + (int64_t)(b / rpi) * R * CH;
  float* alb = alpha + (int64_t)b * alpha_stride;
  for (int r = r0 + wid; r < r1; r += 2 * LO_ATT_WARPS) {
    const int rb = r + LO_ATT_WARPS;
    const bool two = rb < r1;
    float v0[NV * 8], v1[NV * 8], u0[NV * 8], u1[NV * 8];
#pragma unroll
    for (int j = 0; j < NV; j++) {
      ld8(a1b + (int64_t)r * CH + (j * 32 + lane) * 8, v0 + j * 8);
      ld8(eb + (int64_t)r * CH + (j * 32 + lane) * 8, u0 + j * 8);
    }
    if (two) {
#pragma unroll
      for (int j = 0; j < NV; j++) {
        ld8(a1b + (int64_t)rb * CH + (j * 32 + lane) * 8, v1 + j * 8);
        ld8(eb + (int64_t)rb * CH + (j * 32 + lane) * 8, u1 + j * 8);
      }
    }
    float e0 = 0.f, e1 = 0.f;
#pragma unroll
    for (int i = 0; i < NV * 8; i++) {
      e0 = fmaf(wv[i], fmaxf(v0[i] + a2[i], 0.f), e0);
      if (two) e1 = fmaf(wv[i], fmaxf(v1[i] + a2[i], 0.f), e1);
    }
    e0 = warp_sum(e0);
    e1 = warp_sum(e1);
    if (lane == 0) {
      alb[r] = e0;
      if (two) alb[rb] = e1;
    }
    const float mn = two ? fmaxf(m, fmaxf(e0, e1)) : fmaxf(m, e0);
    const float sc = expf(m - mn);     // m = -inf on the first row -> 0
    const float p0 = expf(e0 - mn);
    const float p1 = two ? expf(e1 - mn) : 0.f;
    l = l * sc + p0 + p1;
#pragma unroll
    for (int i = 0; i < NV * 8; i++) {
      float t = acc[i] * sc;
      t = fmaf(p0, u0[i], t);
      if (two) t = fmaf(p1, u1[i], t);
      acc[i] = t;
    }
    m = mn;
  }
  // ---- CTA combine
  __shared__ float s_m[LO_ATT_WARPS], s_l[LO_ATT_WARPS];
  __shared__ float s_acc[LO_ATT_WARPS][CH];
  __shared__ float s_scale[LO_ATT_MAXSPLIT];
  __shared__ float s_ML[2];
  __shared__ int s_last;
  if (lane == 0) { s_m[wid] = m; s_l[wid] = l; }
#pragma unroll
  for (int j = 0; j < NV; j++)
#pragma unroll
    for (int i = 0; i < 8; i++) s_acc[wid][(j * 32 + lane) * 8 + i] = acc[j * 8 + i];
  __syncthreads();
  float M = -INFINITY;
#pragma unroll
  for (int w = 0; w < LO_ATT_WARPS; w++) M = fmaxf(M, s_m[w]);
  float L = 0.f;
  float wsc[LO_ATT_WARPS];
#pragma unroll
  for (int w = 0; w < LO_ATT_WARPS; w++) {
    wsc[w] = (s_m[w] == -INFINITY) ? 0.f : expf(s_m[w] - M);
    L += s_l[w] * wsc[w];
  }
  float* part = partials + ((int64_t)b * nsplit + sp) * (CH + 2);
  for (int c = threadIdx.x; c < CH; c += LO_ATT_THREADS) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < LO_ATT_WARPS; w++) t = fmaf(s_acc[w][c], wsc[w], t);
    part[2 + c] = t;
  }
  if (threadIdx.x == 0) { part[0] = M; part[1] = L; }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int ticket = atomicAdd(counters + b, 1);
    s_last = (ticket == nsplit - 1);
    if (s_last) counters[b] = 0;   // ready for the next launch
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // ---- last CTA of this batch row: global combine, write ctx (+gate), normalise alpha
  const float* pb = partials + (int64_t)b * nsplit * (CH + 2);
  if (threadIdx.x == 0) {
    float Mg = -INFINITY;
    for (int s = 0; s < nsplit; s++) Mg = fmaxf(Mg, ldcg_f(pb + (int64_t)s * (CH + 2)));
    float Lg = 0.f;
    for (int s = 0; s < nsplit; s++) {
      const float ms = ldcg_f(pb + (int64_t)s * (CH + 2));
      const float scl = (ms == -INFINITY) ? 0.f : expf(ms - Mg);
      s_scale[s] = scl;
      Lg += ldcg_f(pb + (int64_t)s * (CH + 2) + 1) * scl;
    }
    s_ML[0] = Mg;
    s_ML[1] = 1.0f / Lg;
  }
  __syncthreads();
  const float Mg = s_ML[0], invL = s_ML[1];
  for (int c = threadIdx.x; c < CH; c += LO_ATT_THREADS) {
    float t = 0.f;
    for (int s = 0; s < nsplit; s++) t = fmaf(ldcg_f(pb + (int64_t)s * (CH + 2) + 2 + c), s_scale[s], t);
    t *= invL;
    ctx[(int64_t)b * CH + c] = t;
    if (gate_pre) {
      const float g = sigmoidf_(gate_pre[(int64_t)b * gate_stride + c]);
      gate_pre[(int64_t)b * gate_stride + c] = g;
      gctx[(int64_t)b * CH + c] = g * t;
      if (gctx_bf) gctx_bf[(int64_t)b * CH + c] = __float2bfloat16_rn(g * t);
    }
  }
  for (int r = threadIdx.x; r < R; r += LO_ATT_THREADS) alb[r] = expf(ldcg_f(alb + r) - Mg) * invL;
}

// ------------------------------------------------------------------------------------------------
// K6: attention backward for one step (same streaming structure; reads enc and att1 once).
//   dctx = dgctx*gate ; dgp = dgctx*ctx*gate*(1-gate) ; s = <dctx,ctx> + sreg
//   dalpha_r = <dctx, enc_r> + dreg_r ; de_r = alpha_r (dalpha_r - s) ; datt2_a = wf_a sum_r de_r [att1_ra + att2_a > 0]
// ------------------------------------------------------------------------------------------------
template <typename T, int NV>
__global__ void __launch_bounds__(LO_ATT_THREADS) attention_bwd_kernel(
    const T* __restrict__ att1, const T* __restrict__ enc, const float* __restrict__ att2, const float* __restrict__ gate,
    int64_t o1_stride, const float* __restrict__ wf, const float* __restrict__ alpha, int64_t alpha_stride,
    const float* __restrict__ ctx, const float* __restrict__ dgctx, int64_t dg_stride, const float* __restrict__ dreg,
    int64_t dreg_stride, const float* __restrict__ sreg, int64_t sreg_stride, float* __restrict__ de, float* __restrict__ datt2,
    float* __restrict__ dgp, int64_t dcat_stride, bf16* __restrict__ datt2_bf, bf16* __restrict__ dgp_bf,
    float* __restrict__ dctx_out, int R, int nsplit, int* __restrict__ counters, float* __restrict__ partials) {
  constexpr int CH = NV * 256;
  const int b = blockIdx.y, sp = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int rps = (R + nsplit - 1) / nsplit;
  const int r0 = sp * rps, r1 = min(R, r0 + rps);
  float a2[NV * 8], dc[NV * 8], macc[NV * 8];
  float sdot = 0.f;
#pragma unroll
  for (int j = 0; j < NV; j++) {
    const int c0 = (j * 32 + lane) * 8;
    float g[8], cx[8], dg[8];
    ld8(att2 + (int64_t)b * o1_stride + c0, a2 + j * 8);
    ld8(gate + (int64_t)b * o1_stride + c0, g);
    ld8(ctx + (int64_t)b * CH + c0, cx);
    ld8(dgctx + (int64_t)b * dg_stride + c0, dg);
    float gp[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
      dc[j * 8 + i] = dg[i] * g[i];
      sdot = fmaf(dc[j * 8 + i], cx[i], sdot);
      gp[i] = dg[i] * cx[i] * g[i] * (1.f - g[i]);
      macc[j * 8 + i] = 0.f;
    }
    if (sp == 0 && wid == 0) {
      st8(dgp + (int64_t)b * dcat_stride + c0, gp);
      if (dgp_bf) st8(dgp_bf + (int64_t)b * dcat_stride + c0, gp);
      st8(dctx_out + (int64_t)b * CH + c0, dc + j * 8);
    }
  }
  const float s = warp_sum(sdot) + sreg[(int64_t)b * sreg_stride];
  const T* a1b = att1 + (int64_t)b * R * CH;
  const T* eb = enc + (int64_t)b * R * CH;
  const float* alb = alpha + (int64_t)b * alpha_stride;
  float* deb = de + (int64_t)b * alpha_stride;
  const float* drb = dreg + (int64_t)b * dreg_stride;
  for (int r = r0 + wid; r < r1; r += 2 * LO_ATT_WARPS) {
    const int rb = r + LO_ATT_WARPS;
    const bool two = rb < r1;
    float v0[NV * 8], v1[NV * 8], u0[NV * 8], u1[NV * 8];
#pragma unroll
    for (int j = 0; j < NV; j++) {
      ld8(eb + (int64_t)r * CH + (j * 32 + lane) * 8, u0 + j * 8);
      ld8(a1b + (int64_t)r * CH + (j * 32 + lane) * 8, v0 + j * 8);
    }
    if (two) {
#pragma unroll
      for (int j = 0; j < NV; j++) {
        ld8(eb + (int64_t)rb * CH + (j * 32 + lane) * 8, u1 + j * 8);
        ld8(a1b + (int64_t)rb * CH + (j * 32 + lane) * 8, v1 + j * 8);
      }
    }
    float d0 = 0.f, d1 = 0.f;
#pragma unroll
    for (int i = 0; i < NV * 8; i++) {
      d0 = fmaf(dc[i], u0[i], d0);
      if (two) d1 = fmaf(dc[i], u1[i], d1);
    }
    d0 = warp_sum(d0);
    d1 = warp_sum(d1);
    const float de0 = alb[r] * (d0 + drb[r] - s);
    const float de1 = two ? alb[rb] * (d1 + drb[rb] - s) : 0.f;
    if (lane == 0) {
      deb[r] = de0;
      if (two) deb[rb] = de1;
    }
#pragma unroll
    for (int i = 0; i < NV * 8; i++) {
      macc[i] += (v0[i] + a2[i] > 0.f) ? de0 : 0.f;
      if (two) macc[i] += (v1[i] + a2[i] > 0.f) ? de1 : 0.f;
    }
  }
  __shared__ float s_acc[LO_ATT_WARPS][CH];
  __shared__ int s_last;
#pragma unroll
  for (int j = 0; j < NV; j++)
#pragma unroll
    for (int i = 0; i < 8; i++) s_acc[wid][(j * 32 + lane) * 8 + i] = macc[j * 8 + i];
  __syncthreads();
  float* part = partials + ((int64_t)b * nsplit + sp) * (CH + 2);
  for (int c = threadIdx.x; c < CH; c += LO_ATT_THREADS) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < LO_ATT_WARPS; w++) t += s_acc[w][c];
    part[2 + c] = t;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int ticket = atomicAdd(counters + b, 1);
    s_last = (ticket == nsplit - 1);
    if (s_last) counters[b] = 0;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const float* pb = partials + (int64_t)b * nsplit * (CH + 2);
  for (int c = threadIdx.x; c < CH; c += LO_ATT_THREADS) {
    float t = 0.f;
    for (int sidx = 0; sidx < nsplit; sidx++) t += ldcg_f(pb + (int64_t)sidx * (CH + 2) + 2 + c);
    datt2[(int64_t)b * dcat_stride + c] = t * wf[c];
    if (datt2_bf) datt2_bf[(int64_t)b * dcat_stride + c] = __float2bfloat16_rn(t * wf[c]);
  }
}

// ------------------------------------------------------------------------------------------------
// hoisted d att1 / d w_full: ONE sweep over att1 after the time loop.
//   datt1[b,r,a] = wf[a] * sum_t de[b,t,r] * [att1[b,r,a] + att2[t,b,a] > 0]
//   dwf[a]      += sum_{b,r,t} de[b,t,r] * relu(att1[b,r,a] + att2[t,b,a])
// grid (A/64, ceil(R/32), B), 128 threads, thread tile 4(r) x 4(a), time chunks of 32 staged in smem.
// ------------------------------------------------------------------------------------------------
// WACC: 0 = d att1 only; 1 = also all of d w_full; 2 = only the `x * (sum_t on * de)` term of d w_full (ReLU): the other term,
// sum_{t,b} att2_t[b,a] * sum_r on * de_t[b,r], was accumulated per step by the mask-bit attention backward kernels (dwf_part)
template <typename T, int WACC, int ACT = 0>
__global__ void __launch_bounds__(128) datt1_kernel(const T* __restrict__ att1, const float* __restrict__ out1,
                                                     int64_t o1_row, int64_t o1_step, const float* __restrict__ de,
                                                     const float* __restrict__ wf, T* __restrict__ datt1,
                                                     float* __restrict__ dwf, int Tn, int R, int A) {
  constexpr int TT = 32;
  __shared__ __align__(16) float s_a2[TT][64];
  __shared__ __align__(16) float s_de[TT][32];
  __shared__ float s_w[8][64];
  const int b = blockIdx.z, r0 = blockIdx.y * 32, a0 = blockIdx.x * 64;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;   // a = a0 + tx*4.., r = r0 + ty*4..
  float x[4][4], nx[4][4], acc[4][4], wacc[4];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    wacc[i] = 0.f;
    const int r = r0 + ty * 4 + i;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      acc[i][j] = 0.f;
      x[i][j] = (r < R) ? ldf(att1 + ((int64_t)b * R + r) * A + a0 + tx * 4 + j) : -INFINITY;
      nx[i][j] = -x[i][j];
    }
  }
  for (int t0 = 0; t0 < Tn; t0 += TT) {
    for (int i = threadIdx.x; i < TT * 64; i += 128) {
      const int tt = i / 64, a = i % 64;
      s_a2[tt][a] = (t0 + tt < Tn) ? out1[(int64_t)(t0 + tt) * o1_step + (int64_t)b * o1_row + a0 + a] : 0.f;
    }
    for (int i = threadIdx.x; i < TT * 32; i += 128) {
      const int tt = i / 32, r = i % 32;
      s_de[tt][r] = (t0 + tt < Tn && r0 + r < R) ? de[((int64_t)b * Tn + t0 + tt) * R + r0 + r] : 0.f;
    }
    __syncthreads();
#pragma unroll 4
    for (int tt = 0; tt < TT; tt++) {
      const float4 q = *reinterpret_cast<const float4*>(&s_a2[tt][tx * 4]);
      const float4 d4 = *reinterpret_cast<const float4*>(&s_de[tt][ty * 4]);
      const float a2v[4] = {q.x, q.y, q.z, q.w}, dv[4] = {d4.x, d4.y, d4.z, d4.w};
      if constexpr (ACT == 0 && WACC == 1) {
        // d w_full[a] = sum de * relu(x + a2) = sum_i x[i][a] * (sum_t on * de) + sum_t a2_t[a] * (sum_i on * de): the first term is
        // x * acc at the very end (x does not depend on t), the second needs only the per-step column sums s[j]
        float sc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const bool on = a2v[j] > nx[i][j];
            if (on) { acc[i][j] += dv[i]; sc[j] += dv[i]; }
          }
#pragma unroll
        for (int j = 0; j < 4; j++) wacc[j] = fmaf(a2v[j], sc[j], wacc[j]);
      } else
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
          if constexpr (ACT == 0) {
            // x + a2 > 0  <=>  a2 > -x exactly (an fp32 sum has the sign of the exact sum): one compare + one predicated add
            const bool on = a2v[j] > nx[i][j];
            acc[i][j] += on ? dv[i] : 0.f;
          } else {
            const float pre = x[i][j] + a2v[j];
            // tanh score (Genthial cell); padded rows: tanh(-inf) = -1 -> derivative 0, dv = 0
            const float post = tanhf(pre);
            acc[i][j] = fmaf(dv[i], 1.f - post * post, acc[i][j]);
            if (WACC) wacc[j] = fmaf(dv[i], post, wacc[j]);
          }
        }
    }
    __syncthreads();
  }
  float wv[4];
#pragma unroll
  for (int j = 0; j < 4; j++) wv[j] = wf[a0 + tx * 4 + j];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int r = r0 + ty * 4 + i;
    if (r >= R) continue;
#pragma unroll
    for (int j = 0; j < 4; j++) stf(datt1 + ((int64_t)b * R + r) * A + a0 + tx * 4 + j, acc[i][j] * wv[j]);
  }
  if (!WACC) return;
  if constexpr (ACT == 0) {
#pragma unroll
    for (int i = 0; i < 4; i++)
      if (r0 + ty * 4 + i < R) {
#pragma unroll
        for (int j = 0; j < 4; j++) wacc[j] = fmaf(x[i][j], acc[i][j], wacc[j]);      // the x * (sum_t on * de) term
      }
  }
#pragma unroll
  for (int j = 0; j < 4; j++) s_w[ty][tx * 4 + j] = wacc[j];
  __syncthreads();
  if (threadIdx.x < 64) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; k++) t += s_w[k][threadIdx.x];
    atomicAdd(dwf + a0 + threadIdx.x, t);
  }
}

// ------------------------------------------------------------------------------------------------
// small pointwise / reduction kernels
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void mean_rows_kernel(const T* __restrict__ enc, float* __restrict__ mean, int R, int C, int rpi) {
  const int b = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.f;
  for (int r = 0; r < R; r++) s += ldf(enc + ((int64_t)(b / rpi) * R + r) * C + c);
  mean[(int64_t)b * C + c] = s / (float)R;
}

// LSTM cell pointwise (nn.LSTMCell, gate order i,f,g,o).  pre = gtmp + ptab[tok] + hh_pre.
__global__ void lstm_pw_fwd_kernel(const float* __restrict__ gtmp, const float* __restrict__ ptab,
                                   const int64_t* __restrict__ tok, int64_t tok_stride, const float* __restrict__ hh,
                                   int64_t hh_stride, const float* __restrict__ c_prev, float* __restrict__ gates,
                                   float* __restrict__ c_out, float* __restrict__ h_out, bf16* __restrict__ h_bf,
                                   float* __restrict__ hd, int64_t hd_stride, const float* __restrict__ dmask, int nrows, int D,
                                   int V, const unsigned long long* __restrict__ dstate, float dp, int row0, int t_idx) {
  // Everything but the gates GEMM result is at least two launches old (token -> table row, the recurrent projection of this step,
  // c_t; the dropout draw depends on nothing): fetched / computed BEFORE griddepcontrol.wait, so only one L2 round trip (gtmp) is left
  // on the critical path of the time loop instead of two dependent ones.
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = idx < nrows * D;
  const int b = live ? idx / D : 0, j = live ? idx % D : 0;
  float a4[4] = {0.f, 0.f, 0.f, 0.f}, cp = 0.f, mult = 1.f;
  if (live) {
    int64_t tk = tok[(int64_t)b * tok_stride];
    if (tk < 0) tk = 0;
    if (tk >= V) tk = V - 1;
    const float* pt = ptab + tk * 4 * D;
    const float* h0 = hh + (int64_t)b * hh_stride;
#pragma unroll
    for (int q = 0; q < 4; q++) a4[q] = pt[q * D + j] + h0[q * D + j];
    cp = c_prev[(int64_t)b * D + j];
    if (hd) {
      if (dmask) mult = dmask[(int64_t)b * hd_stride + j];                                           // injected mask (parity tests)
      else if (dstate) mult = philox_dropout_mult(dstate, row0 + b, t_idx, j, dp, 1.f / (1.f - dp));  // drawn here, redrawn in the backward
    }
  }
  pdl_wait();
  pdl_trigger();
  if (!live) return;
  const float* g0 = gtmp + (int64_t)b * 4 * D;
  const float pi = g0[j] + a4[0];
  const float pf = g0[D + j] + a4[1];
  const float pg = g0[2 * D + j] + a4[2];
  const float po = g0[3 * D + j] + a4[3];
  const float i = sigmoidf_(pi), f = sigmoidf_(pf), g = tanhf(pg), o = sigmoidf_(po);
  const float c = f * cp + i * g;
  const float h = o * tanhf(c);
  float* gt = gates + (int64_t)b * 4 * D;
  gt[j] = i; gt[D + j] = f; gt[2 * D + j] = g; gt[3 * D + j] = o;
  c_out[(int64_t)b * D + j] = c;
  h_out[(int64_t)b * D + j] = h;
  if (h_bf) h_bf[(int64_t)b * D + j] = __float2bfloat16_rn(h);
  if (hd) hd[(int64_t)b * hd_stride + j] = h * mult;
}

// backward of the cell pointwise part: dh = dhd[b,t] + dh_next ; writes d(pre-activations), dc_prev in place
__global__ void lstm_pw_bwd_kernel(const float* __restrict__ dhd, int64_t dhd_stride, const float* __restrict__ dmask,
                                   const float* __restrict__ dh_next,
                                   int64_t dhn_stride, float* __restrict__ dc, const float* __restrict__ gates,
                                   const float* __restrict__ c_prev, const float* __restrict__ c_cur,
                                   float* __restrict__ dG, int64_t dG_stride, bf16* __restrict__ dG_bf, float* __restrict__ dxh_zero,
                                   int C, int nrows, int D, const unsigned long long* __restrict__ dstate, float dp, int row0,
                                   int t_idx) {
  // gates / cells come from the forward pass, dhd from the hoisted fc backward, dc from this kernel's previous launch (three launches
  // back), the dropout draw depends on nothing: all fetched before griddepcontrol.wait; only dh_next (the GEMM just before) is after it
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = idx < nrows * D;
  const int b = live ? idx / D : 0, j = live ? idx % D : 0;
  float i = 0.f, f = 0.f, g = 0.f, o = 0.f, tc = 0.f, cpv = 0.f, dhv = 0.f, dcv = 0.f;
  if (live) {
    const float* gt = gates + (int64_t)b * 4 * D;
    i = gt[j]; f = gt[D + j]; g = gt[2 * D + j]; o = gt[3 * D + j];
    tc = tanhf(c_cur[(int64_t)b * D + j]);
    cpv = c_prev[(int64_t)b * D + j];
    dhv = dhd[(int64_t)b * dhd_stride + j];
    if (dmask) dhv *= dmask[(int64_t)b * dhd_stride + j];
    else if (dstate) dhv *= philox_dropout_mult(dstate, row0 + b, t_idx, j, dp, 1.f / (1.f - dp));
    dcv = dc[(int64_t)b * D + j];
  }
  pdl_wait();
  pdl_trigger();
  if (!live) return;
  const float dh = dhv + dh_next[(int64_t)b * dhn_stride + j];
  const float dct = dcv + dh * o * (1.f - tc * tc);
  float* d = dG + (int64_t)b * dG_stride;
  d[j] = dct * g * i * (1.f - i);
  d[D + j] = dct * cpv * f * (1.f - f);
  d[2 * D + j] = dct * i * (1.f - g * g);
  d[3 * D + j] = dh * tc * o * (1.f - o);
  dc[(int64_t)b * D + j] = dct * f;
  if (dG_bf) {
    bf16* q = dG_bf + (int64_t)b * dG_stride;
    q[j] = __float2bfloat16_rn(d[j]);
    q[D + j] = __float2bfloat16_rn(d[D + j]);
    q[2 * D + j] = __float2bfloat16_rn(d[2 * D + j]);
    q[3 * D + j] = __float2bfloat16_rn(d[3 * D + j]);
  }
  if (dxh_zero) {
    // the tcgen05 split-K GEMMs that follow accumulate with atomics: clear [dgctx | dh] (dh_next was consumed above;
    // entry C+j is this thread's own read location, entries < C are never read here)
    float* z = dxh_zero + (int64_t)b * (C + D);
    z[C + j] = 0.f;
    for (int q = j; q < C; q += D) z[q] = 0.f;
  }
}

// fused cross-entropy forward/backward: warp per (b,t) row.  target = caps[b][t+1]; rows with b >= bt[t] get 0.
__global__ void ce_kernel(const float* __restrict__ logits, const int64_t* __restrict__ caps, int64_t caps_stride,
                          const int32_t* __restrict__ dlen, float* __restrict__ row_loss, float* __restrict__ dlogits,
                          bf16* __restrict__ dlogits_bf, int B, int Tn, int V, int ld, float inv_n) {
  const int row = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= B * Tn) return;
  const int b = row / Tn, t = row % Tn;
  const float* lg = logits + (int64_t)row * ld;
  float* dl = dlogits ? dlogits + (int64_t)row * ld : nullptr;
  bf16* dlb = dlogits_bf ? dlogits_bf + (int64_t)row * ld : nullptr;
  if (t >= dlen[b]) {
    if (lane == 0) row_loss[row] = 0.f;
    if (dl) for (int v = lane; v < ld; v += 32) dl[v] = 0.f;
    if (dlb) for (int v = lane; v < ld; v += 32) dlb[v] = __float2bfloat16_rn(0.f);
    return;
  }
  float mx = -INFINITY;
  for (int v = lane; v < V; v += 32) mx = fmaxf(mx, lg[v]);
  mx = warp_max(mx);
  float se = 0.f;
  for (int v = lane; v < V; v += 32) se += expf(lg[v] - mx);
  se = warp_sum(se);
  const float lse = mx + logf(se);
  int64_t tg = caps[(int64_t)b * caps_stride + t + 1];
  if (tg < 0) tg = 0;
  if (tg >= V) tg = V - 1;
  if (lane == 0) row_loss[row] = lse - lg[tg];
  if (dl)
    for (int v = lane; v < ld; v += 32) {
      const float g = v < V ? (expf(lg[v] - lse) - (v == (int)tg ? 1.f : 0.f)) * inv_n : 0.f;
      dl[v] = g;
      if (dlb) dlb[v] = __float2bfloat16_rn(g);
    }
}

// doubly-stochastic regulariser: S = sum_t alpha ; sq -> row_loss tail ; dreg = -2 alpha_c (1-S)/(B R)
__global__ void reg_kernel(const float* __restrict__ alphas, float* __restrict__ sq, float* __restrict__ dreg, int B, int Tn,
                           int R, float alpha_c) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * R) return;
  const int b = idx / R, r = idx % R;
  float S = 0.f;
  for (int t = 0; t < Tn; t++) S += alphas[((int64_t)b * Tn + t) * R + r];
  const float d = 1.f - S;
  sq[idx] = d * d;
  if (dreg) dreg[idx] = -2.f * alpha_c * d / ((float)B * (float)R);
}

// sreg[b,t] = sum_r alpha[b,t,r] dreg[b,r]  (warp per (b,t))
__global__ void sreg_kernel(const float* __restrict__ alphas, const float* __restrict__ dreg, int64_t dreg_bstride,
                            int64_t dreg_tstride, float* __restrict__ sreg, int B, int Tn, int R) {
  const int row = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= B * Tn) return;
  const int b = row / Tn, t = row % Tn;
  float s = 0.f;
  for (int r = lane; r < R; r += 32)
    s = fmaf(alphas[(int64_t)row * R + r], dreg[(int64_t)b * dreg_bstride + (int64_t)t * dreg_tstride + r], s);
  s = warp_sum(s);
  if (lane == 0) sreg[row] = s;
}

// deterministic final reduction: loss[0]=total, [1]=ce, [2]=reg, [3]=n_valid
__global__ void loss_finalize_kernel(const float* __restrict__ row_loss, int n_rows, const float* __restrict__ sq, int n_sq,
                                     float inv_n, float alpha_c, float* __restrict__ loss) {
  __shared__ float red[2][32];
  float a = 0.f, c = 0.f;
  for (int i = threadIdx.x; i < n_rows; i += blockDim.x) a += row_loss[i];
  for (int i = threadIdx.x; i < n_sq; i += blockDim.x) c += sq[i];
  a = warp_sum(a);
  c = warp_sum(c);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a; red[1][threadIdx.x >> 5] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float ta = 0.f, tcq = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) { ta += red[0][w]; tcq += red[1][w]; }
    const float ce = ta * inv_n, reg = n_sq ? tcq / (float)n_sq : 0.f;
    loss[0] = ce + alpha_c * reg;
    loss[1] = ce;
    loss[2] = reg;
    loss[3] = 1.f / inv_n;
  }
}

// dptab[v][:] = sum over (t,b) with caps[b][t] == v (and t < dlen[b]) of dG[t][b][:]   (deterministic order)
__global__ void dptab_kernel(const float* __restrict__ dcat, int64_t row_stride, int64_t step_stride, int col0,
                             const int64_t* __restrict__ caps, int64_t caps_stride, const int32_t* __restrict__ dlen,
                             float* __restrict__ dptab, int B, int Tn, int G) {
  const int v = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  __shared__ unsigned s_bits[8];
  float acc = 0.f;
  const int total = B * Tn;
  for (int base = 0; base < total; base += 256) {
    const int idx = base + threadIdx.x;
    bool hit = false;
    if (idx < total) {
      const int b = idx / Tn, t = idx % Tn;
      hit = (t < dlen[b]) && (caps[(int64_t)b * caps_stride + t] == (int64_t)v);
    }
    const unsigned bal = __ballot_sync(0xffffffffu, hit);
    if ((threadIdx.x & 31) == 0) s_bits[threadIdx.x >> 5] = bal;
    __syncthreads();
    if (j < G) {
#pragma unroll
      for (int w = 0; w < 8; w++) {
        unsigned bits = s_bits[w];
        while (bits) {                                  // ascending index order -> deterministic sum
          const int k = __ffs(bits) - 1;
          bits &= bits - 1;
          const int id = base + w * 32 + k;
          const int b = id / Tn, t = id % Tn;
          acc += dcat[(int64_t)t * step_stride + (int64_t)b * row_stride + col0 + j];
        }
      }
    }
    __syncthreads();
  }
  if (j < G) dptab[(int64_t)v * G + j] = acc;
}

// one-hot rows (t,b) x Vp for the tensor-core form of the embedding-table gradient: dptab = onehot^T @ dG
__global__ void onehot_kernel(const int64_t* __restrict__ caps, int64_t caps_stride, const int32_t* __restrict__ dlen,
                              bf16* __restrict__ oh, int B, int Tn, int Vp) {
  const int64_t total = (int64_t)B * Tn * Vp;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int v = (int)(i % Vp);
    const int64_t row = i / Vp;
    const int b = (int)(row % B), t = (int)(row / B);
    const bool hit = (t < dlen[b]) && (caps[(int64_t)b * caps_stride + t] == (int64_t)v);
    oh[i] = __float2bfloat16_rn(hit ? 1.f : 0.f);
  }
}

// bf16 operands of the batched tensor-core GEMM d enc[b] += alphas[b]^T dctx[:, b, :]:
//   alphas fp32 [B*T][R] -> bf16 [B*T][Rp] (rows padded to a multiple of 8 elements = 16 bytes, a TMA stride requirement)
__global__ void cast_pad_rows_kernel(const float* __restrict__ x, bf16* __restrict__ y, int64_t rows, int R, int Rp) {
  const int64_t total = rows * Rp;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / Rp;
    const int c = (int)(i % Rp);
    y[i] = __float2bfloat16_rn(c < R ? x[r * R + c] : 0.f);
  }
}
//   dctx fp32 [T][B][C] -> bf16 [B][T][C]
__global__ void cast_tb_to_bt_kernel(const float* __restrict__ x, bf16* __restrict__ y, int T, int B, int C) {
  const int64_t total = (int64_t)T * B * (C / 8);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c8 = (int)(i % (C / 8));
    const int64_t tb = i / (C / 8);
    const int b = (int)(tb % B), t = (int)(tb / B);
    float v[8];
    ld8(x + tb * C + c8 * 8, v);
    st8(y + ((int64_t)b * T + t) * C + c8 * 8, v);
  }
}

// denc[b][r][:] += dmean[b][:] / R
__global__ void add_rowbcast_kernel(float* __restrict__ denc, const float* __restrict__ dmean, int R, int C, float scale,
                                    int64_t total) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const int64_t b = i / ((int64_t)R * C);
    denc[i] += dmean[b * C + c] * scale;
  }
}

// out[n][k] = in[k][n]  (in [K][ld_in] -> out [N][ld_out]), generic small transpose with dtype
template <typename T>
__global__ void transpose_kernel(const T* __restrict__ in, int64_t ld_in, T* __restrict__ out, int64_t ld_out, int K, int N) {
  __shared__ float tile[32][33];
  const int k0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += 8)
    if (k0 + i < K && n0 + threadIdx.x < N) tile[i][threadIdx.x] = ldf(in + (int64_t)(k0 + i) * ld_in + n0 + threadIdx.x);
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8)
    if (n0 + i < N && k0 + threadIdx.x < K) stf(out + (int64_t)(n0 + i) * ld_out + k0 + threadIdx.x, tile[threadIdx.x][i]);
}

__global__ void argmax_kernel(const float* __restrict__ logits, int V, int64_t* __restrict__ tokens, int64_t tok_stride,
                              int64_t* __restrict__ next_tok, int32_t* __restrict__ finished, int64_t end_id, int B) {
  const int b = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  float best = -INFINITY;
  int bi = 0;
  for (int v = lane; v < V; v += 32) {
    const float x = logits[(int64_t)b * V + v];
    if (x > best) { best = x; bi = v; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }   // lowest index wins ties (torch.argmax)
  }
  if (lane == 0) {
    tokens[(int64_t)b * tok_stride] = bi;
    next_tok[b] = bi;
    if (bi == end_id) finished[b] = 1;
  }
}


// ------------------------------------------------------------------------------------------------
// beam search step (beam_search_decoder_cell.py:123-187): one block per image.
//   lp = log_softmax(logits) ; finished beams -> [END: 0, else: dtype.min] ; total = prev + lp ;
//   time 0: beam 0 only ; top-k(beam) over beam*V (lower flat index wins ties) ; id = idx % V ; parent = idx / V
// ------------------------------------------------------------------------------------------------
#define LO_BEAM_MAX 16
__global__ void __launch_bounds__(256) beam_step_kernel(const float* __restrict__ logits, int V, int beam, int t, int64_t end_id,
                                                        float* __restrict__ logp, int32_t* __restrict__ finished,
                                                        int64_t* __restrict__ ids, int64_t* __restrict__ parents,
                                                        int32_t* __restrict__ fin_hist, int64_t* __restrict__ next_tok,
                                                        int32_t* __restrict__ parent_rows, int max_steps, float div_log_gamma,
                                                        float div_prob, const float* __restrict__ div_u,
                                                        const unsigned long long* __restrict__ div_state) {
  extern __shared__ float s_tot[];            // [beam*V] (+ [beam*V] penalties when the diversity penalty is on)
  __shared__ float s_red[8];
  __shared__ int s_redi[8];
  __shared__ float s_lse[LO_BEAM_MAX];
  __shared__ float s_newp[LO_BEAM_MAX];
  __shared__ int s_newi[LO_BEAM_MAX];
  const int img = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int row0 = img * beam;
  // log-sum-exp per beam row (warp w handles rows w, w+8, ...)
  for (int k = wid; k < beam; k += 8) {
    const float* lg = logits + (int64_t)(row0 + k) * V;
    float mx = -INFINITY;
    for (int v = lane; v < V; v += 32) mx = fmaxf(mx, lg[v]);
    mx = warp_max(mx);
    float se = 0.f;
    for (int v = lane; v < V; v += 32) se += expf(lg[v] - mx);
    se = warp_sum(se);
    if (lane == 0) s_lse[k] = mx + logf(se);
  }
  __syncthreads();
  const int nb = (t == 0) ? 1 : beam;          // beam_search_decoder_cell.py:159-160
  const int total = nb * V;
  for (int i = tid; i < total; i += 256) {
    const int k = i / V, v = i % V;
    float lp = logits[(int64_t)(row0 + k) * V + v] - s_lse[k];
    if (finished[row0 + k]) lp = (v == (int)end_id) ? 0.f : -3.4028234663852886e38f;   // mask_probs :353-367
    s_tot[i] = logp[row0 + k] + lp;
  }
  __syncthreads();
  if (div_log_gamma != 0.f && div_prob > 0.f) {
    // add_div_penalty (beam_search_decoder_cell.py:258-287, Li et al. 2016): rank of every candidate inside its beam row
    // (0 = best; tf.nn.top_k(sorted) puts the lower index first among equals), penalty = log(gamma) * rank, applied where
    // div_prob > u with u ~ U[0,1) per (image, beam, token) — injected (div_u, parity tests) or drawn from Philox
    float* s_pen = s_tot + beam * V;
    for (int i = tid; i < total; i += 256) {
      const int k = i / V, v = i % V;
      const float x = s_tot[i];
      const float* rowp = s_tot + k * V;
      int rank = 0;
      for (int q = 0; q < V; q++) {
        const float y = rowp[q];
        rank += (y > x || (y == x && q < v)) ? 1 : 0;
      }
      float u;
      if (div_u) u = div_u[(int64_t)(row0 + k) * V + v];
      else {
        const uint4 r = philox4x32_10(make_uint4((uint32_t)(v >> 2), (uint32_t)t, (uint32_t)(row0 + k), (uint32_t)div_state[1]),
                                      make_uint2((uint32_t)div_state[0], (uint32_t)(div_state[0] >> 32)));
        u = u01((v & 3) == 0 ? r.x : ((v & 3) == 1 ? r.y : ((v & 3) == 2 ? r.z : r.w)));
      }
      s_pen[i] = div_prob > u ? div_log_gamma * (float)rank : 0.f;
    }
    __syncthreads();
    for (int i = tid; i < total; i += 256) s_tot[i] += s_pen[i];
    __syncthreads();
  }
  for (int j = 0; j < beam; j++) {
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = tid; i < total; i += 256) {
      const float x = s_tot[i];
      if (x > best || (x == best && i < bi)) { best = x; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
    }
    if (lane == 0) { s_red[wid] = best; s_redi[wid] = bi; }
    __syncthreads();
    if (tid == 0) {
      float b2 = s_red[0];
      int i2 = s_redi[0];
      for (int w = 1; w < 8; w++)
        if (s_red[w] > b2 || (s_red[w] == b2 && s_redi[w] < i2)) { b2 = s_red[w]; i2 = s_redi[w]; }
      if (i2 == 0x7fffffff) i2 = 0;          // fewer candidates than beams (beam*V < beam): cannot happen for V >= beam
      s_newp[j] = b2;
      s_newi[j] = i2;
      s_tot[i2] = -INFINITY;                  // remove from the candidate set
    }
    __syncthreads();
  }
  if (tid < beam) {
    const int idx = s_newi[tid];
    const int id = idx % V, par = idx / V;
    const int fin = finished[row0 + par] | (id == (int)end_id ? 1 : 0);
    const int64_t o = ((int64_t)img * max_steps + t) * beam + tid;
    ids[o] = id;
    parents[o] = par;
    fin_hist[o] = fin;
    next_tok[row0 + tid] = id;
    parent_rows[row0 + tid] = row0 + par;
    logp[row0 + tid] = s_newp[tid];           // (every read of the old logp happened before the top-k loop)
  }
  __syncthreads();                            // finished[] of the parents is read above, overwritten below
  if (tid < beam) {
    const int64_t o = ((int64_t)img * max_steps + t) * beam + tid;
    finished[row0 + tid] = fin_hist[o];
  }
}

// dst[r][:] = src[rows[r]][:]  (state gather by parents, gather_helper beam_search_decoder_cell.py:370-391)
__global__ void gather_rows_kernel(const float* __restrict__ src, const int32_t* __restrict__ rows, float* __restrict__ dst, int n,
                                   int D) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * D) return;
  const int r = idx / D, j = idx % D;
  dst[idx] = src[(int64_t)rows[r] * D + j];
}

__global__ void fin_hist_kernel(const int32_t* __restrict__ finished, int32_t* __restrict__ hist, int64_t stride, int B) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) hist[(int64_t)i * stride] = finished[i];
}

__global__ void fill_i64_kernel(int64_t* p, int64_t v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

__global__ void bump_counter_kernel(unsigned long long* c) { *c += 1ull; }

__global__ void dlen_kernel(int32_t* dlen, int B, int Tn, int full) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) dlen[i] = full;
  (void)Tn;
}

// ------------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------------
struct Dims {
  int B, T, R, C, A, D, E, V, O1, G, Vl;
};
static inline Dims dims(const lo_decoder_args* a) {
  return Dims{a->B, a->T, a->R, a->C, a->A, a->D, a->E, a->V, a->A + a->C + 4 * a->D, 4 * a->D, a->ldl > 0 ? a->ldl : a->V};
}

// bf16 staging used when impl == TC: mirrors written by the step kernels feed the tcgen05 GEMMs directly
struct BfViews {
  bool on;
  bf16 *dcat, *hall, *gctx, *wet, *onehot, *hd, *dlogits, *wfct, *wil, *alphas, *dctx, *dptab, *wihT;
};
static inline int64_t rpad8(int64_t r) { return (r + 7) / 8 * 8; }
static BfViews bf_views(const lo_decoder_args* a, const Dims& d) {
  BfViews v{false, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  if (a->impl == LO_IMPL_TC && a->dt == LO_BF16 && a->bfwork && tc_available()) {
    const int64_t TB = (int64_t)d.T * d.B;
    v.on = true;
    v.dcat = (bf16*)a->bfwork;
    v.hall = v.dcat + TB * d.O1;
    v.gctx = v.hall + (TB + d.B) * d.D;
    v.wet = v.gctx + TB * d.C;
    v.onehot = v.wet + (int64_t)d.A * d.C;
    v.hd = v.onehot + TB * ((d.V + 7) / 8 * 8);
    v.dlogits = v.hd + TB * d.D;
    v.wfct = v.dlogits + TB * d.Vl;
    v.wil = v.wfct + (int64_t)d.D * d.Vl;
    v.alphas = v.wil + (int64_t)4 * d.D * d.C;            // [B][T][roundup8(R)] (zero padded): A operand of the batched alpha^T dctx GEMM
    v.dctx = v.alphas + TB * rpad8(d.R);                   // [B][T][C]
    v.dptab = v.dctx + TB * d.C;                           // [V][4D] bf16 copy of the embedding-table gradient
    v.wihT = v.dptab + (int64_t)d.V * d.G;                 // [E][4D] = (weight_ih[:, :E])^T
  }
  return v;
}

static int check_args(const lo_decoder_args* a) {
  LO_CHECK_ARG(a != nullptr, "args");
  LO_CHECK_ARG(a->B > 0 && a->T > 0 && a->R > 0 && a->V > 1, "B,T,R,V");
  LO_CHECK_ARG(a->A == a->C && (a->C == 256 || a->C == 512 || a->C == 1024), "attention_dim == encoder_dim in {256,512,1024}");
  LO_CHECK_ARG(a->D % 8 == 0 && a->E % 8 == 0, "D, E multiples of 8");
  LO_CHECK_ARG(a->dt == LO_F32 || a->dt == LO_BF16, "dt");
  LO_CHECK_ARG(a->ldl == 0 || a->ldl >= a->V, "ldl >= V");
  LO_CHECK_ARG(a->rows_per_img <= 1 || a->B % a->rows_per_img == 0, "B must be a multiple of rows_per_img");
  LO_CHECK_ARG(a->bt_host && a->caps && a->enc && a->work, "null pointer");
  LO_CHECK_ARG(a->has_dropout != 2 || (a->dropout_state && a->dropout_p >= 0.f && a->dropout_p < 1.f &&
                                       (!g_opt_fuse_lstm || g_opt_skinny_mma)),
               "has_dropout=2 needs dropout_state, 0 <= dropout_p < 1 (and the mma.sync kernel when fuse_lstm=1)");
  for (int t = 0; t < a->T; t++) {
    LO_CHECK_ARG(a->bt_host[t] >= 1 && a->bt_host[t] <= a->B, "bt_host out of range");
    if (t) LO_CHECK_ARG(a->bt_host[t] <= a->bt_host[t - 1], "bt_host must be non-increasing");
  }
  return LO_OK;
}

static int* work_counters(const lo_decoder_args* a) { return (int*)a->work; }
// ReLU mask bits of step t, first row r0 (NULL when the scheme is off)
static inline uint8_t* att_mask_at(const lo_decoder_args* a, int t, int64_t r0) {
  if (!a->att_mask || !g_opt_att_maskbits || !g_opt_att_pipe || a->rows_per_img > 1) return nullptr;
  return a->att_mask + ((int64_t)t * a->B + r0) * ((a->R + 1) & ~1) * (a->A / 8);      // rows padded to an even count (pair layout)
}
static float* work_partials(const lo_decoder_args* a) { return (float*)((char*)a->work + 4096); }
static int32_t* work_dlen(const lo_decoder_args* a) { return (int32_t*)((char*)a->work + 2048); }

static int attention_forward_launch(const void* att1, const void* enc, int dt, const float* att2, int64_t att2_stride,
                                    const float* wf, float* alpha, int64_t alpha_stride, float* ctx, float* gate_pre,
                                    int64_t gate_stride, float* gctx, bf16* gctx_bf, int B, int R, int C, void* work, cudaStream_t st,
                                    int rpi = 1, int nsplit_hint = 0, uint8_t* mask_out = nullptr, int abi = 0) {
  if (rpi < 1) rpi = 1;
  if (g_opt_att_pipe) {
    AttFwdArgs x{att1, enc, att2, att2_stride, wf, alpha, alpha_stride, ctx, gate_pre, gate_stride, gctx, gctx_bf, B, R, work, rpi,
                 nsplit_hint, 0, 0, mask_out, abi};
    return attention_fwd_pipe(x, dt, C, st);
  }
  const int ns = att_splits(B);
  int* cnt = (int*)work;
  float* part = (float*)((char*)work + 4096);
  dim3 grid(ns, B);
#define LO_ATT_FWD(T, NV)                                                                                           \
  attention_fwd_kernel<T, NV><<<grid, LO_ATT_THREADS, 0, st>>>((const T*)att1, (const T*)enc, att2, att2_stride, wf, \
                                                               alpha, alpha_stride, ctx, gate_pre, gate_stride, gctx, gctx_bf, R, ns, cnt, part, rpi)
  if (dt == LO_F32) {
    if (C == 256) LO_ATT_FWD(float, 1); else if (C == 512) LO_ATT_FWD(float, 2); else LO_ATT_FWD(float, 4);
  } else {
    if (C == 256) LO_ATT_FWD(bf16, 1); else if (C == 512) LO_ATT_FWD(bf16, 2); else LO_ATT_FWD(bf16, 4);
  }
#undef LO_ATT_FWD
  LO_LAUNCH_OK();
  return LO_OK;
}

// builds dlen[b] (device) = number of steps row b decodes, from the host bt[] array, via tiny memcpy-free kernels
static int upload_dlen(const lo_decoder_args* a, cudaStream_t st) {
  // dlen[b] = #{t : bt[t] > b}.  bt is non-increasing, so rows [bt[t], bt[t-1]) have dlen = t.
  int32_t* dl = work_dlen(a);
  LO_CHECK_ARG(a->B <= 512, "B <= 512 (dlen scratch)");
  LO_CUDA(cudaMemsetAsync(dl, 0, (size_t)a->B * 4, st));   // rows that never decode (caption length 1)
  // rows below bt[T-1] decode all T steps
  dlen_kernel<<<cdiv(a->B, 128), 128, 0, st>>>(dl, a->bt_host[a->T - 1], a->T, a->T);
  LO_LAUNCH_OK();
  for (int t = a->T - 1; t >= 1; t--) {
    const int lo_ = a->bt_host[t], hi_ = a->bt_host[t - 1];
    if (hi_ > lo_) {
      dlen_kernel<<<cdiv(hi_ - lo_, 128), 128, 0, st>>>(dl + lo_, hi_ - lo_, a->T, t);
      LO_LAUNCH_OK();
    }
  }
  return LO_OK;
}

// x = hi + lo with hi = bf16(x), lo = bf16(x - hi): two bf16 GEMMs then reproduce an fp32-input GEMM to ~2^-17 relative
__global__ void split_bf16_kernel(const float* __restrict__ x, bf16* __restrict__ hi, bf16* __restrict__ lo, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = x[i];
    const bf16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

int g_opt_fuse_lstm = 0;   // measured slower (23.0 vs 20.1 ms/step): 128 epilogue threads cannot hide the dependent global loads
                           // (tok -> table row, recurrent projection, c) that 32 K threads of lstm_pw_fwd_kernel hide
// wil[4*j + g][c] = w_ih[g*D + j][E + c]: gate-interleaved copy of the context half of weight_ih, so that one 32-column
// accumulator chunk of the tcgen05 GEMM holds whole hidden units and the LSTM cell can run in its epilogue
__global__ void interleave_wih_kernel(const bf16* __restrict__ w_ih, bf16* __restrict__ wil, int D, int E, int C) {
  const int64_t total = (int64_t)4 * D * (C / 8);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c8 = (int)(i % (C / 8));
    const int n = (int)(i / (C / 8));        // interleaved row 4*j + g
    const int j = n >> 2, g = n & 3;
    *reinterpret_cast<uint4*>(wil + (int64_t)n * C + c8 * 8) =
        *reinterpret_cast<const uint4*>(w_ih + ((int64_t)g * D + j) * (E + C) + E + c8 * 8);
  }
}

static int forward_prologue(const lo_decoder_args* a, const Dims& d, cudaStream_t st) {
  const int dt = a->dt;
  const int rpi = a->rows_per_img > 1 ? a->rows_per_img : 1;
  // att1 = enc @ W_e^T + b_e   (hoisted: the reference recomputes it every step, seq2seq_torch.py:186)
  LO_TRY(gemm_nt(a->enc, dt, d.C, a->w_enc_att, dt, d.C, a->att1, dt, d.A, (d.B / rpi) * d.R, d.A, d.C, a->b_enc_att, 0, 0, a->impl, st));
  const BfViews bv0 = bf_views(a, d);
  // embedding -> gate projection table (replaces embedding lookup + x[:, :E] @ W_ih[:, :E]^T, seq2seq_torch.py:291,:313)
  if (bv0.on && d.E % 64 == 0) {
    LO_TRY(tc_gemm_nt_ex((const bf16*)a->emb, d.E, (const bf16*)a->w_ih, d.E + d.C, a->ptab, LO_F32, d.G, d.V, d.G, d.E, a->b_ih, 0, 0, 1,
                         0, 0, st));
  } else {
    LO_TRY(gemm_nt(a->emb, dt, d.E, a->w_ih, dt, d.E + d.C, a->ptab, LO_F32, d.G, d.V, d.G, d.E, a->b_ih, 0, 0, LO_IMPL_SIMT, st));
  }
  // init_hidden_state (seq2seq_torch.py:255-265)
  {
    dim3 grid(cdiv(d.C, 256), d.B);
    LO_DISPATCH_DT(dt, T, (mean_rows_kernel<T><<<grid, 256, 0, st>>>((const T*)a->enc, a->mean, d.R, d.C, rpi)));
    LO_LAUNCH_OK();
  }
  const size_t es = dt == LO_F32 ? 4 : 2;
  if (bv0.on && d.C % 64 == 0 && d.T >= 2) {
    // the row means stay fp32-accurate: hi/lo bf16 split (staged in the not-yet-used gctx mirrors of steps 0 and 1)
    bf16* mean_hi = bv0.gctx;
    bf16* mean_lo = bv0.gctx + (int64_t)d.B * d.C;
    split_bf16_kernel<<<cdiv((long)d.B * d.C, 256), 256, 0, st>>>(a->mean, mean_hi, mean_lo, (int64_t)d.B * d.C);
    LO_LAUNCH_OK();
    const bf16* w_h = (const bf16*)a->w_init;
    const bf16* w_c = w_h + (int64_t)d.D * d.C;
    LO_TRY(tc_gemm_nt_ex(mean_hi, d.C, w_h, d.C, a->hall, LO_F32, d.D, d.B, d.D, d.C, a->b_init, 0, 0, 1, 0, 1, st));
    LO_TRY(tc_gemm_nt_ex(mean_lo, d.C, w_h, d.C, a->hall, LO_F32, d.D, d.B, d.D, d.C, nullptr, 1, 0, 1, 0, 1, st));
    LO_TRY(tc_gemm_nt_ex(mean_hi, d.C, w_c, d.C, a->call, LO_F32, d.D, d.B, d.D, d.C, a->b_init + d.D, 0, 0, 1, 0, 1, st));
    LO_TRY(tc_gemm_nt_ex(mean_lo, d.C, w_c, d.C, a->call, LO_F32, d.D, d.B, d.D, d.C, nullptr, 1, 0, 1, 0, 1, st));
  } else {
    LO_TRY(gemm_nt(a->mean, LO_F32, d.C, a->w_init, dt, d.C, a->hall, LO_F32, d.D, d.B, d.D, d.C, a->b_init, 0, 0, LO_IMPL_SIMT, st));
    LO_TRY(gemm_nt(a->mean, LO_F32, d.C, (const char*)a->w_init + (size_t)d.D * d.C * es, dt, d.C, a->call, LO_F32, d.D, d.B,
                   d.D, d.C, a->b_init + d.D, 0, 0, LO_IMPL_SIMT, st));
  }
  const BfViews bv = bf_views(a, d);
  if (bv.on) {
    LO_TRY(lo_cast(a->hall, LO_F32, bv.hall, LO_BF16, (int64_t)d.B * d.D, (void*)st));
    if ((g_opt_fuse_lstm || g_opt_dec_fuse || g_opt_dec_cl) && d.E % 8 == 0 && d.C % 8 == 0) {
      interleave_wih_kernel<<<148 * 2, 256, 0, st>>>((const bf16*)a->w_ih, bv.wil, d.D, d.E, d.C);
      LO_LAUNCH_OK();
    }
  }
  return LO_OK;
}

// a contiguous slice of batch rows processed on one stream.  The rows of a batch never interact inside the time loop
// (only the hoisted weight-gradient GEMMs mix them), so the loop can run as independent half-batch chains on two
// streams: while one chain streams att1/enc (HBM bound, all SMs) the other runs its latency-bound GEMM / LSTM kernels.
struct Rows {
  int row0, nrows;
  void* work;       // attention workspace of this chain
  int nsplit;       // attention split hint (0 = automatic)
};
int g_opt_dec_streams = 1;
// timing dissection only (tools/dec_breakdown.py; results are garbage): 1 = skip the hoisted part of the backward, 2 = skip the
// attention launches of the time loops, 4 = skip the per-step GEMM / LSTM launches, 8 = skip the hoisted part of the forward
int g_opt_dbg_skip = 0;

// one decoder step t for the rows of `rs`; tok: token ids consumed at this step (row 0 of the batch)
static int forward_step(const lo_decoder_args* a, const Dims& d, int t, const Rows& rs, const int64_t* tok, int64_t tok_stride,
                        float* hd_t, int64_t hd_stride, const float* dmask_t, cudaStream_t st) {
  const int dt = a->dt;
  const int nrows = rs.nrows;
  const int64_t r0 = rs.row0;
  if (nrows <= 0) return LO_OK;
  const size_t es = dt == LO_F32 ? 4 : 2;
  float* h_prev = a->hall + ((int64_t)t * d.B + r0) * d.D;
  float* c_prev = a->call + ((int64_t)t * d.B + r0) * d.D;
  float* o1 = a->out1 + ((int64_t)t * d.B + r0) * d.O1;
  float* gtmp = a->gtmp + r0 * d.G;
  const int rpi = a->rows_per_img > 1 ? a->rows_per_img : 1;
  const char* att1 = (const char*)a->att1 + (size_t)(r0 / rpi) * d.R * d.A * es;
  const char* enc = (const char*)a->enc + (size_t)(r0 / rpi) * d.R * d.C * es;
  // [att2 | gate_pre | hh_pre] = h_prev @ [W_d; W_beta; W_hh]^T + b   (seq2seq_torch.py:187, :311, LSTMCell hh part)
  const BfViews bv = bf_views(a, d);
  if (g_opt_dbg_skip & 4) {
  } else if (bv.on && g_opt_skinny_mma && nrows <= 64) {
    LO_TRY(skinny_gemm_nt(bv.hall + ((int64_t)t * d.B + r0) * d.D, d.D, (const bf16*)a->wcat1, d.D, o1, d.O1, nrows, d.O1, d.D, a->bcat1, 1,
                          0, st));
  } else if (bv.on) {
    LO_TRY(tc_gemm_nt_ex(bv.hall + ((int64_t)t * d.B + r0) * d.D, d.D, (const bf16*)a->wcat1, d.D, o1, LO_F32, d.O1, nrows, d.O1, d.D,
                         a->bcat1, 0, 0, 1, 0, 1, st));
  } else {
    LO_TRY(gemm_nt(h_prev, LO_F32, d.D, a->wcat1, dt, d.D, o1, LO_F32, d.O1, nrows, d.O1, d.D, a->bcat1, 0, 0, LO_IMPL_SIMT, st));
  }
  if (!(g_opt_dbg_skip & 2))
  LO_TRY(attention_forward_launch(att1, enc, dt, o1, d.O1, a->w_full, a->alphas + (r0 * d.T + t) * d.R, (int64_t)d.T * d.R,
                                  a->ctx + ((int64_t)t * d.B + r0) * d.C, o1 + d.A, d.O1, a->gctx + ((int64_t)t * d.B + r0) * d.C,
                                  bv.on ? bv.gctx + ((int64_t)t * d.B + r0) * d.C : nullptr, nrows, d.R, d.C, rs.work, st,
                                  a->rows_per_img, rs.nsplit, hd_t ? att_mask_at(a, t, r0) : nullptr));
  if (g_opt_dbg_skip & 4) return LO_OK;
  // gates_x = (gate*ctx) @ W_ih[:, E:]^T
  if (bv.on && g_opt_fuse_lstm) {
    // ... with the LSTM cell fused into the GEMM epilogue (no gates_x round trip, one launch less per step)
    TcLstmEpi e{a->ptab, tok + r0 * tok_stride, tok_stride, o1 + d.A + d.C, d.O1, c_prev, a->gates + ((int64_t)t * d.B + r0) * d.G,
                a->call + ((int64_t)(t + 1) * d.B + r0) * d.D, a->hall + ((int64_t)(t + 1) * d.B + r0) * d.D,
                bv.hall + ((int64_t)(t + 1) * d.B + r0) * d.D, hd_t ? hd_t + r0 * hd_stride : (float*)nullptr, hd_stride,
                dmask_t ? dmask_t + r0 * hd_stride : (const float*)nullptr, d.D, d.V,
                (const unsigned long long*)((hd_t && a->has_dropout == 2) ? a->dropout_state : nullptr), a->dropout_p, (int)r0, t};
    if (g_opt_skinny_mma && nrows <= 64 && d.C <= 512)
      return skinny_gemm_nt_lstm(bv.gctx + ((int64_t)t * d.B + r0) * d.C, d.C, bv.wil, d.C, nrows, d.D, d.C, e, st);
    return tc_gemm_nt_lstm(bv.gctx + ((int64_t)t * d.B + r0) * d.C, d.C, bv.wil, d.C, nrows, d.D, d.C, e, st);
  }
  if (bv.on && g_opt_skinny_mma && nrows <= 64) {
    LO_TRY(skinny_gemm_nt(bv.gctx + ((int64_t)t * d.B + r0) * d.C, d.C, (const bf16*)a->w_ih + d.E, d.E + d.C, gtmp, d.G, nrows, d.G, d.C,
                          nullptr, 1, 0, st));
  } else if (bv.on) {
    LO_TRY(tc_gemm_nt_ex(bv.gctx + ((int64_t)t * d.B + r0) * d.C, d.C, (const bf16*)a->w_ih + d.E, d.E + d.C, gtmp, LO_F32, d.G, nrows,
                         d.G, d.C, nullptr, 0, 0, 1, 0, 1, st));
  } else {
    LO_TRY(gemm_nt(a->gctx + ((int64_t)t * d.B + r0) * d.C, LO_F32, d.C, (const char*)a->w_ih + (size_t)d.E * es, dt, d.E + d.C, gtmp,
                   LO_F32, d.G, nrows, d.G, d.C, nullptr, 0, 0, LO_IMPL_SIMT, st));
  }
  LO_CUDA(launch_pdl(lstm_pw_fwd_kernel, dim3(cdiv((long)nrows * d.D, 256)), dim3(256), (size_t)0, st, (const float*)gtmp,
                     (const float*)a->ptab, tok + r0 * tok_stride, tok_stride, (const float*)(o1 + d.A + d.C), (int64_t)d.O1,
                     (const float*)c_prev, a->gates + ((int64_t)t * d.B + r0) * d.G, a->call + ((int64_t)(t + 1) * d.B + r0) * d.D,
                     a->hall + ((int64_t)(t + 1) * d.B + r0) * d.D,
                     bv.on ? bv.hall + ((int64_t)(t + 1) * d.B + r0) * d.D : (bf16*)nullptr,
                     hd_t ? hd_t + r0 * hd_stride : (float*)nullptr, hd_stride,
                     dmask_t ? dmask_t + r0 * hd_stride : (const float*)nullptr, nrows, d.D, d.V,
                     (const unsigned long long*)((hd_t && a->has_dropout == 2) ? a->dropout_state : nullptr), a->dropout_p, (int)r0, t));
  LO_LAUNCH_OK();
  return LO_OK;
}

// fork/join helpers for the two-chain time loop (legal inside stream capture: the side stream joins back)
static cudaStream_t g_side = nullptr;
static cudaEvent_t g_ev_fork = nullptr, g_ev_join = nullptr;
static int side_stream_init() {
  if (g_side) return LO_OK;
  LO_CUDA(cudaStreamCreateWithFlags(&g_side, cudaStreamNonBlocking));
  LO_CUDA(cudaEventCreateWithFlags(&g_ev_fork, cudaEventDisableTiming));
  LO_CUDA(cudaEventCreateWithFlags(&g_ev_join, cudaEventDisableTiming));
  return LO_OK;
}
static inline bool two_chains(const lo_decoder_args* a, const Dims& d) {
  return g_opt_dec_streams >= 2 && d.B >= 32 && a->rows_per_img <= 1;
}
static inline Rows chain_rows(const lo_decoder_args* a, const Dims& d, int chain, int nchains, int active) {
  // rows [0, half) -> chain 0, [half, B) -> chain 1; `active` = rows still decoding at this step (sorted by length)
  const int half = nchains == 2 ? (d.B + 1) / 2 : d.B;
  Rows r;
  r.row0 = chain * half;
  const int hi = chain == 0 ? (active < half ? active : half) : active;
  r.nrows = hi - r.row0 > 0 ? hi - r.row0 : 0;
  if (chain == 0 && nchains == 1) r.nrows = active;
  r.work = (char*)a->work + (size_t)chain * lo_attention_workspace_bytes(d.B, d.C);
  r.nsplit = nchains == 2 ? (148 / (half > 0 ? half : 1) > 0 ? 148 / half : 1) : 0;   // each chain fills one CTA slot per SM
  return r;
}

}  // namespace lo

// greedy / beam decode loops (one- and two-layer decoder) and the two-layer decode entry points
#include "lo_decoder2.cuh"

using namespace lo;

extern "C" {

int64_t lo_decoder_bfwork_bytes(const lo_decoder_args* a) {
  if (!a) return 0;
  const int64_t TB = (int64_t)a->T * a->B, O1 = a->A + a->C + 4 * a->D;
  const int64_t Vp = (a->V + 7) / 8 * 8;
  const int64_t Vl = a->ldl > 0 ? a->ldl : a->V;
  return (TB * (O1 + a->D + a->C + Vp + a->D + Vl) + (int64_t)a->B * a->D + (int64_t)a->A * a->C + (int64_t)a->D * Vl +
          (int64_t)4 * a->D * a->C + TB * ((a->R + 7) / 8 * 8) + TB * a->C + (int64_t)(a->V + a->E) * 4 * a->D) * 2 + 1024;
}

int64_t lo_sizeof_decoder_args(void) { return (int64_t)sizeof(lo_decoder_args); }

int64_t lo_attention_workspace_bytes(int B, int C) {
  return 4096 + (int64_t)B * LO_ATT_MAXSPLIT * (C + 2) * 4;
}
/* the decoder entry points use two such regions (one per row chain) */
int64_t lo_decoder_workspace_bytes(int B, int C) { return 2 * lo_attention_workspace_bytes(B, C); }

int lo_attention_forward(const void* att1, const void* enc, int dt, const float* att2, int64_t att2_stride, const float* wf,
                         float* alpha, int64_t alpha_stride, float* ctx, float* gate_pre, int64_t gate_stride, float* gctx,
                         int B, int R, int A, int C, void* work, void* stream) {
  LO_CHECK_ARG(att1 && enc && att2 && wf && alpha && ctx && work, "null pointer");
  LO_CHECK_ARG(A == C && (C == 256 || C == 512 || C == 1024), "attention_dim == encoder_dim in {256,512,1024}");
  LO_CHECK_ARG(B > 0 && B <= 512 && R > 0, "B in 1..512, R > 0");
  LO_CHECK_ARG(att2_stride % 4 == 0, "att2 rows must be 16-byte aligned");
  return attention_forward_launch(att1, enc, dt, att2, att2_stride, wf, alpha, alpha_stride, ctx, gate_pre, gate_stride, gctx, nullptr,
                                  B, R, C, work, (cudaStream_t)stream, 1, 0, nullptr, 1);
}

int lo_attention_forward_mask(const void* att1, const void* enc, int dt, const float* att2, int64_t att2_stride, const float* wf,
                              float* alpha, int64_t alpha_stride, float* ctx, float* gate_pre, int64_t gate_stride, float* gctx,
                              uint8_t* relu_mask_out, int B, int R, int A, int C, void* work, void* stream) {
  LO_CHECK_ARG(att1 && enc && att2 && wf && alpha && ctx && work, "null pointer");
  LO_CHECK_ARG(A == C && (C == 256 || C == 512 || C == 1024), "attention_dim == encoder_dim in {256,512,1024}");
  LO_CHECK_ARG(B > 0 && B <= 512 && R > 0, "B in 1..512, R > 0");
  LO_CHECK_ARG(att2_stride % 4 == 0, "att2 rows must be 16-byte aligned");
  LO_CHECK_ARG(!relu_mask_out || g_opt_att_pipe, "mask bits are written by the TMA-ring kernel (option att_pipe=1)");
  return attention_forward_launch(att1, enc, dt, att2, att2_stride, wf, alpha, alpha_stride, ctx, gate_pre, gate_stride, gctx, nullptr,
                                  B, R, C, work, (cudaStream_t)stream, 1, 0, relu_mask_out, 1);
}

int lo_attention_backward(const void* att1, const void* enc, int dt, const float* att2, const float* gate, int64_t o1_stride,
                          const float* wf, const float* alpha, int64_t alpha_stride, const float* ctx, const float* dgctx,
                          int64_t dg_stride, const float* dreg, int64_t dreg_stride, const float* sreg, int64_t sreg_stride, float* de,
                          float* datt2, float* dgp, int64_t dcat_stride, float* dctx_out, float* dwf_part, const uint8_t* relu_mask,
                          int B, int R, int A, int C, void* work, void* stream) {
  LO_CHECK_ARG(att1 && enc && att2 && wf && alpha && ctx && dgctx && de && datt2 && work, "null pointer");
  LO_CHECK_ARG(A == C && (C == 256 || C == 512 || C == 1024), "attention_dim == encoder_dim in {256,512,1024}");
  LO_CHECK_ARG(B > 0 && B <= 512 && R > 0, "B in 1..512, R > 0");
  LO_CHECK_ARG(g_opt_att_pipe, "stand-alone attention backward runs on the TMA-ring kernel (option att_pipe=1)");
  AttBwdArgs x{att1, enc, att2, gate, o1_stride, wf, alpha, alpha_stride, ctx, dgctx, dg_stride, dreg, dreg_stride, sreg, sreg_stride,
               de, datt2, dgp, dcat_stride, nullptr, nullptr, dctx_out, B, R, work, dwf_part, 0, 0, 0, relu_mask};
  x.abi = 1;
  return attention_bwd_pipe(x, dt, C, (cudaStream_t)stream);
}

int lo_decoder_forward(const lo_decoder_args* a, int with_loss, void* stream) {
  LO_TRY(check_args(a));
  cudaStream_t st = (cudaStream_t)stream;
  const Dims d = dims(a);
  const bool ragged = a->bt_host[d.T - 1] < d.B;
  if (ragged && a->phase != 2) {
    LO_CUDA(cudaMemsetAsync(a->alphas, 0, (size_t)d.B * d.T * d.R * 4, st));
    LO_CUDA(cudaMemsetAsync(a->hd, 0, (size_t)d.B * d.T * d.D * 4, st));
  }
  LO_TRY(upload_dlen(a, st));
  if (a->phase != 2) {
  LO_TRY(forward_prologue(a, d, st));
  const int nchains = two_chains(a, d) ? 2 : 1;
  if (nchains == 2) {
    LO_TRY(side_stream_init());
    LO_CUDA(cudaEventRecord(g_ev_fork, st));
    LO_CUDA(cudaStreamWaitEvent(g_side, g_ev_fork, 0));
  }
  const BfViews bvs = bf_views(a, d);
  const bool fused = bvs.on && g_opt_dec_fuse && g_opt_skinny_mma && !g_opt_fuse_lstm && g_opt_att_pipe && nchains == 1 && d.B <= 64 &&
                     d.C == d.D && d.D <= 512 && d.D % 16 == 0 && d.O1 % 16 == 0 && d.E % 8 == 0 && a->rows_per_img <= 1;
  const bool clf = bvs.on && !fused && !(g_opt_dbg_skip & 4) && g_opt_skinny_mma && !g_opt_fuse_lstm && g_opt_att_pipe && nchains == 1 && d.E % 8 == 0 &&
                   a->rows_per_img <= 1 && dec_cl_fwd_ok(d.D, d.C, d.O1);
  if (clf) {
    // two launches per step: attention(t) -> dec_cl_fwd(t) = [gates GEMM + LSTM cell | cluster all-gather | projection of h_{t+1}],
    // one 16-CTA cluster per block of 16 batch rows (lo_cluster.cu)
    LO_TRY(skinny_gemm_nt(bvs.hall, d.D, (const bf16*)a->wcat1, d.D, a->out1, d.O1, a->bt_host[0], d.O1, d.D, a->bcat1, 1, 0, st));
    for (int t = 0; t < d.T; t++) {
      const int nrows = a->bt_host[t];
      float* o1 = a->out1 + (int64_t)t * d.B * d.O1;
      if (!(g_opt_dbg_skip & 2))
      LO_TRY(attention_forward_launch(a->att1, a->enc, a->dt, o1, d.O1, a->w_full, a->alphas + (int64_t)t * d.R, (int64_t)d.T * d.R,
                                      a->ctx + (int64_t)t * d.B * d.C, o1 + d.A, d.O1, a->gctx + (int64_t)t * d.B * d.C,
                                      bvs.gctx + (int64_t)t * d.B * d.C, nrows, d.R, d.C, a->work, st, 1, 0, att_mask_at(a, t, 0)));
      DecStepFwd p{};
      p.gctx = bvs.gctx + (int64_t)t * d.B * d.C; p.ld_gctx = d.C;
      p.wil = bvs.wil; p.ld_wil = d.C;
      const float* dm = (a->has_dropout == 1 && a->dropout_mask) ? a->dropout_mask + (int64_t)t * d.D : nullptr;
      p.e = TcLstmEpi{a->ptab, a->caps + t, a->caps_stride, o1 + d.A + d.C, d.O1, a->call + (int64_t)t * d.B * d.D,
                      a->gates + (int64_t)t * d.B * d.G, a->call + (int64_t)(t + 1) * d.B * d.D, a->hall + (int64_t)(t + 1) * d.B * d.D,
                      bvs.hall + (int64_t)(t + 1) * d.B * d.D, a->hd + (int64_t)t * d.D, (int64_t)d.T * d.D, dm, d.D, d.V,
                      (const unsigned long long*)(a->has_dropout == 2 ? a->dropout_state : nullptr), a->dropout_p, 0, t};
      p.wcat = (const bf16*)a->wcat1; p.ld_wcat = d.D; p.bcat = a->bcat1;
      p.o1_next = t + 1 < d.T ? a->out1 + (int64_t)(t + 1) * d.B * d.O1 : nullptr;
      p.ld_o1 = d.O1; p.N2 = d.O1;
      p.M = nrows; p.K = d.C;
      LO_TRY(dec_cl_fwd(p, st));
    }
  } else if (fused) {
    // two launches per step: attention(t) -> dec_step_fwd(t) = [gates GEMM + LSTM cell | grid barrier | projection of h_{t+1}]
    unsigned int* bar = (unsigned int*)((char*)a->work + lo_attention_workspace_bytes(d.B, d.C));      // chain-1 region is unused here
    LO_CUDA(cudaMemsetAsync(bar, 0, 16 * 128, st));                                                    // 16 arrival counters, one cache line each
    const int grid = cdiv(d.O1, 16) > cdiv(d.G, 16) ? cdiv(d.O1, 16) : cdiv(d.G, 16);
    LO_TRY(skinny_gemm_nt(bvs.hall, d.D, (const bf16*)a->wcat1, d.D, a->out1, d.O1, a->bt_host[0], d.O1, d.D, a->bcat1, 1, 0, st));
    unsigned int epoch = 0;
    for (int t = 0; t < d.T; t++) {
      const int nrows = a->bt_host[t];
      float* o1 = a->out1 + (int64_t)t * d.B * d.O1;
      if (!(g_opt_dbg_skip & 2))
      LO_TRY(attention_forward_launch(a->att1, a->enc, a->dt, o1, d.O1, a->w_full, a->alphas + (int64_t)t * d.R, (int64_t)d.T * d.R,
                                      a->ctx + (int64_t)t * d.B * d.C, o1 + d.A, d.O1, a->gctx + (int64_t)t * d.B * d.C,
                                      bvs.gctx + (int64_t)t * d.B * d.C, nrows, d.R, d.C, a->work, st, 1, 0, att_mask_at(a, t, 0)));
      DecStepFwd p{};
      p.gctx = bvs.gctx + (int64_t)t * d.B * d.C; p.ld_gctx = d.C;
      p.wil = bvs.wil; p.ld_wil = d.C;
      const float* dm = (a->has_dropout == 1 && a->dropout_mask) ? a->dropout_mask + (int64_t)t * d.D : nullptr;
      p.e = TcLstmEpi{a->ptab, a->caps + t, a->caps_stride, o1 + d.A + d.C, d.O1, a->call + (int64_t)t * d.B * d.D,
                      a->gates + (int64_t)t * d.B * d.G, a->call + (int64_t)(t + 1) * d.B * d.D, a->hall + (int64_t)(t + 1) * d.B * d.D,
                      bvs.hall + (int64_t)(t + 1) * d.B * d.D, a->hd + (int64_t)t * d.D, (int64_t)d.T * d.D, dm, d.D, d.V,
                      (const unsigned long long*)(a->has_dropout == 2 ? a->dropout_state : nullptr), a->dropout_p, 0, t};
      p.wcat = (const bf16*)a->wcat1; p.ld_wcat = d.D; p.bcat = a->bcat1;
      const bool more = t + 1 < d.T;
      p.o1_next = more ? a->out1 + (int64_t)(t + 1) * d.B * d.O1 : nullptr;
      p.ld_o1 = d.O1; p.N2 = d.O1;
      p.bar = bar; p.bar_target = more ? (++epoch) * (unsigned int)grid : 0u;
      p.M = nrows; p.K = d.C;
      LO_TRY(dec_step_fwd(p, st));
    }
  } else
  for (int chain = 0; chain < nchains; chain++) {
    cudaStream_t cs = chain == 0 ? st : g_side;
    for (int t = 0; t < d.T; t++) {
      const float* dm = (a->has_dropout == 1 && a->dropout_mask) ? a->dropout_mask + (int64_t)t * d.D : nullptr;
      const Rows rs = chain_rows(a, d, chain, nchains, a->bt_host[t]);
      LO_TRY(forward_step(a, d, t, rs, a->caps + t, a->caps_stride, a->hd + (int64_t)t * d.D, (int64_t)d.T * d.D, dm, cs));
    }
  }
  if (nchains == 2) {
    LO_CUDA(cudaEventRecord(g_ev_join, g_side));
    LO_CUDA(cudaStreamWaitEvent(st, g_ev_join, 0));
  }
  }   // phase != 2
  if (a->phase == 1) return LO_OK;       // extension: the caller runs a second layer over hd before the head
  if (g_opt_dbg_skip & 8) return LO_OK;
  // predictions = fc(dropout(h))  (seq2seq_torch.py:316), hoisted out of the loop
  const BfViews bvf = bf_views(a, d);
  const bool fc_tc = bvf.on && d.Vl % 64 == 0 && d.D % 64 == 0;
  if (fc_tc) {
    LO_TRY(lo_cast(a->hd, LO_F32, bvf.hd, LO_BF16, (int64_t)d.B * d.T * d.D, stream));
    LO_TRY(tc_gemm_nt_ex(bvf.hd, d.D, (const bf16*)a->w_fc, d.D, a->logits, LO_F32, d.Vl, d.B * d.T, d.V, d.D, a->b_fc, 0, 0, 1, 0, 0, st));
  } else {
    LO_TRY(gemm_nt(a->hd, LO_F32, d.D, a->w_fc, a->dt, d.D, a->logits, LO_F32, d.Vl, d.B * d.T, d.V, d.D, a->b_fc, 0, 0, LO_IMPL_SIMT, st));
  }
  if (ragged) {
    // rows that stopped decoding keep zeros in `predictions` (seq2seq_torch.py:301): re-zero what the GEMM wrote (bias)
    // handled by the CE kernel (ignores them) and by the Python side for the returned tensor.
  }
  if (with_loss) {
    long nvalid = 0;
    for (int t = 0; t < d.T; t++) nvalid += a->bt_host[t];
    const float inv_n = 1.0f / (float)nvalid;
    ce_kernel<<<cdiv((long)d.B * d.T, 8), 256, 0, st>>>(a->logits, a->caps, a->caps_stride, work_dlen(a), a->row_loss, a->dlogits,
                                                         (fc_tc && a->dlogits) ? bvf.dlogits : nullptr, d.B, d.T, d.V, d.Vl, inv_n);
    LO_LAUNCH_OK();
    reg_kernel<<<cdiv((long)d.B * d.R, 256), 256, 0, st>>>(a->alphas, a->row_loss + (int64_t)d.B * d.T, a->dreg, d.B, d.T, d.R, a->alpha_c);
    LO_LAUNCH_OK();
    loss_finalize_kernel<<<1, 1024, 0, st>>>(a->row_loss, d.B * d.T, a->row_loss + (int64_t)d.B * d.T, d.B * d.R, inv_n, a->alpha_c, a->loss);
    LO_LAUNCH_OK();
  }
  return LO_OK;
}

int lo_decoder_pack_bwd_weights(const lo_decoder_args* a, void* stream) {
  LO_TRY(check_args(a));
  LO_CHECK_ARG(a->wbwd1 && a->wbwd2, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const Dims d = dims(a);
  const size_t es = a->dt == LO_F32 ? 4 : 2;
  dim3 blk(32, 8);
  // wbwd1 [C+D][4D]: rows 0..C-1 <- (w_ih[:, E:])^T ; rows C.. <- w_hh^T
  const char* w_hh = (const char*)a->wcat1 + (size_t)(d.A + d.C) * d.D * es;
  const char* w_dec = (const char*)a->wcat1;
  const char* w_beta = (const char*)a->wcat1 + (size_t)d.A * d.D * es;
  LO_DISPATCH_DT(a->dt, T, {
    transpose_kernel<T><<<dim3(cdiv(d.C, 32), cdiv(d.G, 32)), blk, 0, st>>>((const T*)a->w_ih + d.E, d.E + d.C, (T*)a->wbwd1, d.G, d.G, d.C);
    transpose_kernel<T><<<dim3(cdiv(d.D, 32), cdiv(d.G, 32)), blk, 0, st>>>((const T*)w_hh, d.D, (T*)a->wbwd1 + (int64_t)d.C * d.G, d.G, d.G, d.D);
    // wbwd2 [D][A+C]: [n][k<A] = w_dec[k][n] ; [n][A+k] = w_beta[k][n]
    transpose_kernel<T><<<dim3(cdiv(d.D, 32), cdiv(d.A, 32)), blk, 0, st>>>((const T*)w_dec, d.D, (T*)a->wbwd2, d.A + d.C, d.A, d.D);
    transpose_kernel<T><<<dim3(cdiv(d.D, 32), cdiv(d.C, 32)), blk, 0, st>>>((const T*)w_beta, d.D, (T*)a->wbwd2 + d.A, d.A + d.C, d.C, d.D);
  });
  lo::g_launches += 3;
  LO_LAUNCH_OK();
  return LO_OK;
}

int lo_decoder_backward(const lo_decoder_args* a, void* stream) {
  LO_TRY(check_args(a));
  cudaStream_t st = (cudaStream_t)stream;
  const Dims d = dims(a);
  const int dt = a->dt;
  const bool ragged = a->bt_host[d.T - 1] < d.B;
  const int ns = att_splits(d.B);
  const int64_t BT = (int64_t)d.B * d.T;
  const float* dal = a->dalpha_ext ? a->dalpha_ext : a->dreg;
  const int64_t dal_b = a->dalpha_ext ? (int64_t)d.T * d.R : d.R, dal_t = a->dalpha_ext ? d.R : 0;
  if (a->phase != 2) {
    LO_TRY(lo_decoder_pack_bwd_weights(a, stream));
    // sreg[b,t] = sum_r alpha dreg
    sreg_kernel<<<cdiv(BT, 8), 256, 0, st>>>(a->alphas, dal, dal_b, dal_t, a->sreg, d.B, d.T, d.R);
    LO_LAUNCH_OK();
  }
  // fc backward (hoisted): g_w_fc = dlogits^T hd ; g_b_fc ; dhd = dlogits @ W_fc (* dropout mask)
  const BfViews bvf = bf_views(a, d);
  const bool fc_tc = bvf.on && d.Vl % 64 == 0 && d.D % 64 == 0 && !a->dalpha_ext;
  if (a->phase == 1) {
    // extension: d hd was put there by the caller (backward of the layer between the cell and fc)
  } else if (fc_tc) {
    // (dlogits bf16 mirror was written by ce_kernel; generic-autograd callers that fill dlogits themselves use the SIMT path)
    LO_CUDA(cudaMemsetAsync(a->g_w_fc, 0, (size_t)d.V * d.D * 4, st));
    LO_TRY(tc_gemm_tn(bvf.dlogits, d.Vl, bvf.hd, d.D, a->g_w_fc, d.D, d.V, d.D, (int)BT, st));
    transpose_kernel<bf16><<<dim3(cdiv(d.D, 32), cdiv(d.V, 32)), dim3(32, 8), 0, st>>>((const bf16*)a->w_fc, d.D, bvf.wfct, d.Vl, d.V, d.D);
    LO_LAUNCH_OK();
    LO_TRY(tc_gemm_nt_ex(bvf.dlogits, d.Vl, bvf.wfct, d.Vl, a->dhd, LO_F32, d.D, (int)BT, d.D, d.Vl, nullptr, 0, 0, 1, 0, 0, st));
  } else {
    LO_TRY(gemm_tn(a->dlogits, LO_F32, d.Vl, a->hd, LO_F32, d.D, a->g_w_fc, LO_F32, d.D, d.V, d.D, (int)BT, 0, LO_IMPL_SIMT, st));
    LO_TRY(gemm_nn(a->dlogits, LO_F32, d.Vl, a->w_fc, dt, d.D, a->dhd, LO_F32, d.D, (int)BT, d.D, d.V, 0, LO_IMPL_SIMT, st));
  }
  if (a->phase != 1) LO_TRY(colsum(a->dlogits, LO_F32, a->g_b_fc, (int)BT, d.V, d.Vl, 0, st));
  if (a->phase == 2) return LO_OK;
  LO_CUDA(cudaMemsetAsync(a->dxh, 0, (size_t)d.B * (d.C + d.D) * 4, st));
  LO_CUDA(cudaMemsetAsync(a->dc, 0, (size_t)d.B * d.D * 4, st));
  if (ragged) {
    LO_CUDA(cudaMemsetAsync(a->dcat, 0, (size_t)d.T * d.B * d.O1 * 4, st));
    LO_CUDA(cudaMemsetAsync(a->de, 0, (size_t)BT * d.R * 4, st));
    LO_CUDA(cudaMemsetAsync(a->dctx, 0, (size_t)d.T * d.B * d.C * 4, st));
    const BfViews bz = bf_views(a, d);
    if (bz.on) LO_CUDA(cudaMemsetAsync(bz.dcat, 0, (size_t)d.T * d.B * d.O1 * 2, st));
  }
  const BfViews bv = bf_views(a, d);
  if (g_opt_att_pipe) LO_CUDA(cudaMemsetAsync(a->dmean, 0, (size_t)d.B * d.A * 4, st));    // [B][A] scratch for d w_full
  const int nchains = two_chains(a, d) ? 2 : 1;
  if (nchains == 2) {
    LO_TRY(side_stream_init());
    LO_CUDA(cudaEventRecord(g_ev_fork, st));
    LO_CUDA(cudaStreamWaitEvent(g_side, g_ev_fork, 0));
  }
  const cudaStream_t st_main = st;
  const bool fusedb = bv.on && g_opt_dec_fuse_bwd && g_opt_skinny_mma && g_opt_att_pipe && nchains == 1 && d.B <= 64 && d.C == d.D &&
                      (d.A + d.C) % 512 == 0 && d.G % 512 == 0 && ((d.C + d.D) / 16) * (d.G / 512) <= 296 && a->rows_per_img <= 1;
  const bool clb = bv.on && !fusedb && !(g_opt_dbg_skip & 4) && g_opt_skinny_mma && g_opt_att_pipe && nchains == 1 && a->rows_per_img <= 1 &&
                   dec_cl_bwd_ok(d.D, d.C, d.A);
  if (clb) {
    // two launches per step: attention_bwd(t) -> dec_cl_bwd = [dh_t += (datt2|dgate)_t W | LSTM bwd (t-1) | cluster all-gather | dG_{t-1} W]
    auto fill_bc = [&](DecStepBwd& p, int t) {       // LSTM backward + dG projection of step t
      p.dhd = a->dhd + (int64_t)t * d.D; p.dhd_stride = (int64_t)d.T * d.D;
      p.dmask = (a->has_dropout == 1 && a->dropout_mask) ? a->dropout_mask + (int64_t)t * d.D : nullptr;
      p.dstate = (const unsigned long long*)(a->has_dropout == 2 ? a->dropout_state : nullptr);
      p.dp = a->dropout_p; p.t_idx = t;
      p.dc = a->dc; p.gates = a->gates + (int64_t)t * d.B * d.G;
      p.c_prev = a->call + (int64_t)t * d.B * d.D; p.c_cur = a->call + (int64_t)(t + 1) * d.B * d.D;
      p.dG = a->dcat + (int64_t)t * d.B * d.O1 + d.A + d.C; p.dG_bf = bv.dcat + (int64_t)t * d.B * d.O1 + d.A + d.C; p.dG_stride = d.O1;
      p.Mb = a->bt_host[t];
    };
    auto fill_common = [&](DecStepBwd& p) {
      p.wbwd1 = (const bf16*)a->wbwd1; p.ld_w1 = d.G; p.K1 = d.G;
      p.wbwd2 = (const bf16*)a->wbwd2; p.ld_w2 = d.A + d.C; p.K2 = d.A + d.C;
      p.dxh = a->dxh; p.C = d.C; p.D = d.D; p.ld_dcat = d.O1;
    };
    {
      DecStepBwd p{};
      fill_common(p);
      fill_bc(p, d.T - 1);
      LO_TRY(dec_cl_bwd(p, st));
    }
    for (int t = d.T - 1; t >= 0; t--) {
      const int nrows = a->bt_host[t];
      float* dcat_t = a->dcat + (int64_t)t * d.B * d.O1;
      bf16* dcat_bf_t = bv.dcat + (int64_t)t * d.B * d.O1;
      const float* o1 = a->out1 + (int64_t)t * d.B * d.O1;
      AttBwdArgs x{a->att1, a->enc, o1, o1 + d.A, d.O1, a->w_full, a->alphas + (int64_t)t * d.R, (int64_t)d.T * d.R,
                   a->ctx + (int64_t)t * d.B * d.C, a->dxh, d.C + d.D, dal + (int64_t)t * dal_t, dal_b, a->sreg + t, d.T,
                   a->de + (int64_t)t * d.R, dcat_t, dcat_t + d.A, d.O1, dcat_bf_t, dcat_bf_t + d.A, a->dctx + (int64_t)t * d.B * d.C,
                   nrows, d.R, a->work, a->dmean, 0, 0, 0, att_mask_at(a, t, 0)};
      if (!(g_opt_dbg_skip & 2)) LO_TRY(attention_bwd_pipe(x, dt, d.C, st));
      DecStepBwd p{};
      fill_common(p);
      p.dcat_a = dcat_bf_t; p.Ma = nrows;
      if (t > 0) fill_bc(p, t - 1);
      LO_TRY(dec_cl_bwd(p, st));
    }
  } else if (fusedb) {
    // two launches per step: attention_bwd(t) -> dec_step_bwd = [dh += (datt2|dgate) W | barrier | LSTM bwd (t-1) | barrier | dG W]
    unsigned int* bar = (unsigned int*)((char*)a->work + lo_attention_workspace_bytes(d.B, d.C)) + 1024;   // chain-1 region, unused here
    LO_CUDA(cudaMemsetAsync(bar, 0, 16 * 128, st));
    const unsigned int grid = (unsigned int)(((d.C + d.D) / 16) * (d.G / 512));
    unsigned int nb = 0;
    auto fill_bc = [&](DecStepBwd& p, int t) {       // phases B/C for step t
      p.dhd = a->dhd + (int64_t)t * d.D; p.dhd_stride = (int64_t)d.T * d.D;
      p.dmask = (a->has_dropout == 1 && a->dropout_mask) ? a->dropout_mask + (int64_t)t * d.D : nullptr;
      p.dstate = (const unsigned long long*)(a->has_dropout == 2 ? a->dropout_state : nullptr);
      p.dp = a->dropout_p; p.t_idx = t;
      p.dc = a->dc; p.gates = a->gates + (int64_t)t * d.B * d.G;
      p.c_prev = a->call + (int64_t)t * d.B * d.D; p.c_cur = a->call + (int64_t)(t + 1) * d.B * d.D;
      p.dG = a->dcat + (int64_t)t * d.B * d.O1 + d.A + d.C; p.dG_bf = bv.dcat + (int64_t)t * d.B * d.O1 + d.A + d.C; p.dG_stride = d.O1;
      p.wbwd1 = (const bf16*)a->wbwd1; p.ld_w1 = d.G; p.K1 = d.G; p.Mb = a->bt_host[t];
    };
    {
      DecStepBwd p{};
      fill_bc(p, d.T - 1);
      p.wbwd2 = (const bf16*)a->wbwd2; p.ld_w2 = d.A + d.C; p.K2 = d.A + d.C;
      p.dxh = a->dxh; p.C = d.C; p.D = d.D; p.bar = bar; p.bar_target = (nb + 1) * grid;
      nb += 1;
      LO_TRY(dec_step_bwd(p, st));
    }
    for (int t = d.T - 1; t >= 0; t--) {
      const int nrows = a->bt_host[t];
      float* dcat_t = a->dcat + (int64_t)t * d.B * d.O1;
      bf16* dcat_bf_t = bv.dcat + (int64_t)t * d.B * d.O1;
      const float* o1 = a->out1 + (int64_t)t * d.B * d.O1;
      AttBwdArgs x{a->att1, a->enc, o1, o1 + d.A, d.O1, a->w_full, a->alphas + (int64_t)t * d.R, (int64_t)d.T * d.R,
                   a->ctx + (int64_t)t * d.B * d.C, a->dxh, d.C + d.D, dal + (int64_t)t * dal_t, dal_b, a->sreg + t, d.T,
                   a->de + (int64_t)t * d.R, dcat_t, dcat_t + d.A, d.O1, dcat_bf_t, dcat_bf_t + d.A, a->dctx + (int64_t)t * d.B * d.C,
                   nrows, d.R, a->work, a->dmean, 0, 0, 0, att_mask_at(a, t, 0)};
      LO_TRY(attention_bwd_pipe(x, dt, d.C, st));
      DecStepBwd p{};
      p.dcat_a = dcat_bf_t; p.ld_dcat = d.O1; p.wbwd2 = (const bf16*)a->wbwd2; p.ld_w2 = d.A + d.C; p.K2 = d.A + d.C; p.Ma = nrows;
      p.dxh = a->dxh; p.C = d.C; p.D = d.D; p.bar = bar;
      p.K1 = d.G;                                  // grid size (phase C tiling) even when phases B/C are skipped
      if (t > 0) {
        fill_bc(p, t - 1);
        p.bar_target = (nb + 1) * grid;
        nb += 2;
      }
      LO_TRY(dec_step_bwd(p, st));
    }
  } else
  for (int chain = 0; chain < nchains; chain++) {
   st = chain == 0 ? st_main : g_side;
   for (int t = d.T - 1; t >= 0; t--) {
    const Rows rs = chain_rows(a, d, chain, nchains, a->bt_host[t]);
    const int nrows = rs.nrows;
    const int64_t r0 = rs.row0;
    if (nrows <= 0) continue;
    const size_t es = dt == LO_F32 ? 4 : 2;
    float* dcat_t = a->dcat + ((int64_t)t * d.B + r0) * d.O1;
    bf16* dcat_bf_t = bv.on ? bv.dcat + ((int64_t)t * d.B + r0) * d.O1 : nullptr;
    const float* o1 = a->out1 + ((int64_t)t * d.B + r0) * d.O1;
    float* dxh = a->dxh + r0 * (d.C + d.D);
    const float* dmul = (a->has_dropout == 1 && a->dropout_mask) ? a->dropout_mask + (int64_t)t * d.D + r0 * d.T * d.D : nullptr;
    if (!(g_opt_dbg_skip & 4))
    LO_CUDA(launch_pdl(lstm_pw_bwd_kernel, dim3(cdiv((long)nrows * d.D, 256)), dim3(256), (size_t)0, st,
                       (const float*)(a->dhd + (int64_t)t * d.D + r0 * d.T * d.D), (int64_t)d.T * d.D, dmul, (const float*)(dxh + d.C),
                       (int64_t)(d.C + d.D), a->dc + r0 * d.D, (const float*)(a->gates + ((int64_t)t * d.B + r0) * d.G),
                       (const float*)(a->call + ((int64_t)t * d.B + r0) * d.D),
                       (const float*)(a->call + ((int64_t)(t + 1) * d.B + r0) * d.D), dcat_t + d.A + d.C, (int64_t)d.O1,
                       bv.on ? dcat_bf_t + d.A + d.C : (bf16*)nullptr, bv.on ? dxh : (float*)nullptr, d.C, nrows, d.D,
                       (const unsigned long long*)(a->has_dropout == 2 ? a->dropout_state : nullptr), a->dropout_p, (int)r0, t));
    LO_LAUNCH_OK();
    // [dgctx | dh_prev] = dG @ [W_ih[:, E:] | W_hh]
    if (g_opt_dbg_skip & 4) {
    } else if (bv.on && g_opt_skinny_mma && nrows <= 64) {
      LO_TRY(skinny_gemm_nt(dcat_bf_t + d.A + d.C, d.O1, (const bf16*)a->wbwd1, d.G, dxh, d.C + d.D, nrows, d.C + d.D, d.G, nullptr, 4, 1,
                            st));
    } else if (bv.on) {
      LO_TRY(tc_gemm_nt_ex(dcat_bf_t + d.A + d.C, d.O1, (const bf16*)a->wbwd1, d.G, dxh, LO_F32, d.C + d.D, nrows, d.C + d.D, d.G,
                           nullptr, 0, 0, 4, 1, 1, st));
    } else {
      LO_TRY(gemm_nt(dcat_t + d.A + d.C, LO_F32, d.O1, a->wbwd1, dt, d.G, dxh, LO_F32, d.C + d.D, nrows, d.C + d.D, d.G, nullptr, 0,
                     0, LO_IMPL_SIMT, st));
    }
    const char* att1 = (const char*)a->att1 + (size_t)r0 * d.R * d.A * es;
    const char* enc = (const char*)a->enc + (size_t)r0 * d.R * d.C * es;
    const float* alpha_t = a->alphas + (r0 * d.T + t) * d.R;
    const float* ctx_t = a->ctx + ((int64_t)t * d.B + r0) * d.C;
    const float* dal_t_ptr = dal + (int64_t)t * dal_t + r0 * dal_b;
    const float* sreg_t = a->sreg + r0 * d.T + t;
    float* de_t = a->de + (r0 * d.T + t) * d.R;
    float* dctx_t = a->dctx + ((int64_t)t * d.B + r0) * d.C;
    if (g_opt_dbg_skip & 2) {
    } else if (g_opt_att_pipe) {
      AttBwdArgs x{att1, enc, o1, o1 + d.A, d.O1, a->w_full, alpha_t, (int64_t)d.T * d.R, ctx_t, dxh, d.C + d.D, dal_t_ptr, dal_b, sreg_t,
                   d.T, de_t, dcat_t, dcat_t + d.A, d.O1, dcat_bf_t, dcat_bf_t ? dcat_bf_t + d.A : nullptr, dctx_t, nrows, d.R, rs.work,
                   a->dmean + r0 * d.A, rs.nsplit, 0, 0, att_mask_at(a, t, r0)};
      LO_TRY(attention_bwd_pipe(x, dt, d.C, st));
    } else {
    int* cnt_c = (int*)rs.work;
    float* part_c = (float*)((char*)rs.work + 4096);
    dim3 grid(ns, nrows);
#define LO_ATT_BWD(TY_, NV)                                                                                                       \
  attention_bwd_kernel<TY_, NV><<<grid, LO_ATT_THREADS, 0, st>>>(                                                                 \
      (const TY_*)att1, (const TY_*)enc, o1, o1 + d.A, d.O1, a->w_full, alpha_t, (int64_t)d.T * d.R, ctx_t, dxh, d.C + d.D, dal_t_ptr, \
      dal_b, sreg_t, d.T, de_t, dcat_t, dcat_t + d.A, d.O1, dcat_bf_t, dcat_bf_t ? dcat_bf_t + d.A : nullptr, dctx_t, d.R, ns, cnt_c,  \
      part_c)
    if (dt == LO_F32) {
      if (d.C == 256) LO_ATT_BWD(float, 1); else if (d.C == 512) LO_ATT_BWD(float, 2); else LO_ATT_BWD(float, 4);
    } else {
      if (d.C == 256) LO_ATT_BWD(bf16, 1); else if (d.C == 512) LO_ATT_BWD(bf16, 2); else LO_ATT_BWD(bf16, 4);
    }
#undef LO_ATT_BWD
    LO_LAUNCH_OK();
    }
    // dh_prev += [datt2 | dgate_pre] @ [W_d ; W_beta]
    if (g_opt_dbg_skip & 4) {
    } else if (bv.on && g_opt_skinny_mma && nrows <= 64) {
      LO_TRY(skinny_gemm_nt(dcat_bf_t, d.O1, (const bf16*)a->wbwd2, d.A + d.C, dxh + d.C, d.C + d.D, nrows, d.D, d.A + d.C, nullptr, 4, 1,
                            st));
    } else if (bv.on) {
      LO_TRY(tc_gemm_nt_ex(dcat_bf_t, d.O1, (const bf16*)a->wbwd2, d.A + d.C, dxh + d.C, LO_F32, d.C + d.D, nrows, d.D, d.A + d.C,
                           nullptr, 0, 0, 4, 1, 1, st));
    } else {
      LO_TRY(gemm_nt(dcat_t, LO_F32, d.O1, a->wbwd2, dt, d.A + d.C, dxh + d.C, LO_F32, d.C + d.D, nrows, d.D, d.A + d.C, nullptr, 1,
                     0, LO_IMPL_SIMT, st));
    }
   }
  }
  st = st_main;
  if (nchains == 2) {
    LO_CUDA(cudaEventRecord(g_ev_join, g_side));
    LO_CUDA(cudaStreamWaitEvent(st, g_ev_join, 0));
  }
  // dinit = [dh0 | dc0]
  LO_CUDA(cudaMemcpy2DAsync(a->dinit, (size_t)2 * d.D * 4, a->dxh + d.C, (size_t)(d.C + d.D) * 4, (size_t)d.D * 4, d.B,
                            cudaMemcpyDeviceToDevice, st));
  LO_CUDA(cudaMemcpy2DAsync(a->dinit + d.D, (size_t)2 * d.D * 4, a->dc, (size_t)d.D * 4, (size_t)d.D * 4, d.B,
                            cudaMemcpyDeviceToDevice, st));
  if (g_opt_dbg_skip & 1) return LO_OK;
  // ---- hoisted gradients
  const bool tc = bv.on;
  bf16* dcat_bf = bv.dcat;
  bf16* hall_bf = bv.hall;
  bf16* gctx_bf = bv.gctx;
  bf16* wet_bf = bv.wet;
  // [W_d; W_beta; W_hh] and biases: dcat^T @ h_prev
  if (tc) {
    LO_CUDA(cudaMemsetAsync(a->g_wcat1, 0, (size_t)d.O1 * d.D * 4, st));
    LO_TRY(tc_gemm_tn(dcat_bf, d.O1, hall_bf, d.D, a->g_wcat1, d.D, d.O1, d.D, d.T * d.B, st));
  } else {
    LO_TRY(gemm_tn(a->dcat, LO_F32, d.O1, a->hall, LO_F32, d.D, a->g_wcat1, LO_F32, d.D, d.O1, d.D, d.T * d.B, 0, LO_IMPL_SIMT, st));
  }
  LO_TRY(colsum(a->dcat, LO_F32, a->g_bcat1, d.T * d.B, d.O1, d.O1, 0, st));
  // W_ih[:, E:] : dG^T @ gctx ; b_ih = colsum(dG) (== g_b_hh)
  if (tc) {
    LO_CUDA(cudaMemset2DAsync(a->g_w_ih + d.E, (size_t)(d.E + d.C) * 4, 0, (size_t)d.C * 4, d.G, st));
    LO_TRY(tc_gemm_tn(dcat_bf + d.A + d.C, d.O1, gctx_bf, d.C, a->g_w_ih + d.E, d.E + d.C, d.G, d.C, d.T * d.B, st));
  } else {
    LO_TRY(gemm_tn(a->dcat + d.A + d.C, LO_F32, d.O1, a->gctx, LO_F32, d.C, a->g_w_ih + d.E, LO_F32, d.E + d.C, d.G, d.C, d.T * d.B, 0,
                   LO_IMPL_SIMT, st));
  }
  LO_TRY(colsum(a->dcat + d.A + d.C, LO_F32, a->g_b_ih, d.T * d.B, d.G, d.O1, 0, st));
  // embedding path through the projection table
  if (tc) {
    const int Vp = (d.V + 7) / 8 * 8;
    onehot_kernel<<<148 * 8, 256, 0, st>>>(a->caps, a->caps_stride, work_dlen(a), bv.onehot, d.B, d.T, Vp);
    LO_LAUNCH_OK();
    LO_CUDA(cudaMemsetAsync(a->dptab, 0, (size_t)d.V * d.G * 4, st));
    LO_TRY(tc_gemm_tn(bv.onehot, Vp, dcat_bf + d.A + d.C, d.O1, a->dptab, d.G, d.V, d.G, d.T * d.B, st));
  } else {
    dim3 grid(cdiv(d.G, 256), d.V);
    dptab_kernel<<<grid, 256, 0, st>>>(a->dcat, d.O1, (int64_t)d.B * d.O1, d.A + d.C, a->caps, a->caps_stride, work_dlen(a), a->dptab,
                                       d.B, d.T, d.G);
    LO_LAUNCH_OK();
  }
  if (tc && d.E % 64 == 0 && d.G % 64 == 0 && d.V >= 64) {
    // g_emb = dptab W_ih[:, :E] and g_W_ih[:, :E] = dptab^T emb on tcgen05 (bf16 copy of dptab, transposed weight slice)
    LO_TRY(lo_cast(a->dptab, LO_F32, bv.dptab, LO_BF16, (int64_t)d.V * d.G, stream));
    transpose_kernel<bf16><<<dim3(cdiv(d.E, 32), cdiv(d.G, 32)), dim3(32, 8), 0, st>>>((const bf16*)a->w_ih, d.E + d.C, bv.wihT, d.G, d.G, d.E);
    LO_LAUNCH_OK();
    LO_TRY(tc_gemm_nt(bv.dptab, d.G, bv.wihT, d.G, a->g_emb, LO_F32, d.E, d.V, d.E, d.G, nullptr, 0, 0, st));
    LO_CUDA(cudaMemset2DAsync(a->g_w_ih, (size_t)(d.E + d.C) * 4, 0, (size_t)d.E * 4, d.G, st));
    LO_TRY(tc_gemm_tn(bv.dptab, d.G, (const bf16*)a->emb, d.E, a->g_w_ih, d.E + d.C, d.G, d.E, d.V, st));
  } else {
    LO_TRY(gemm_nn(a->dptab, LO_F32, d.G, a->w_ih, dt, d.E + d.C, a->g_emb, LO_F32, d.E, d.V, d.E, d.G, 0, LO_IMPL_SIMT, st));
    LO_TRY(gemm_tn(a->dptab, LO_F32, d.G, a->emb, dt, d.E, a->g_w_ih, LO_F32, d.E + d.C, d.G, d.E, d.V, 0, LO_IMPL_SIMT, st));
  }
  // d att1 + d w_full in one sweep over att1
  LO_CUDA(cudaMemsetAsync(a->g_w_full, 0, (size_t)d.A * 4, st));
  LO_CUDA(cudaMemsetAsync(a->g_b_full, 0, 4, st));   // sum_r de = 0 exactly (softmax); reference value is rounding noise
  {
    dim3 grid(d.A / 64, cdiv(d.R, 32), d.B);
    if (g_opt_att_pipe && !att_mask_at(a, 0, 0)) {
      // d w_full was accumulated per batch row by the attention backward kernels (dmean doubles as the [B][A] scratch)
      LO_TRY(colsum(a->dmean, LO_F32, a->g_w_full, d.B, d.A, d.A, 0, st));
      LO_DISPATCH_DT(dt, T, (datt1_kernel<T, 0><<<grid, 128, 0, st>>>((const T*)a->att1, a->out1, d.O1, (int64_t)d.B * d.O1, a->de,
                                                                       a->w_full, (T*)a->datt1, a->g_w_full, d.T, d.R, d.A)));
    } else if (g_opt_att_pipe) {
      // mask-bit scheme: the att2 term of d w_full came out of the per-step kernels (dmean scratch), the sweep adds the x term
      LO_TRY(colsum(a->dmean, LO_F32, a->g_w_full, d.B, d.A, d.A, 0, st));
      LO_DISPATCH_DT(dt, T, (datt1_kernel<T, 2><<<grid, 128, 0, st>>>((const T*)a->att1, a->out1, d.O1, (int64_t)d.B * d.O1, a->de,
                                                                       a->w_full, (T*)a->datt1, a->g_w_full, d.T, d.R, d.A)));
    } else {
      LO_DISPATCH_DT(dt, T, (datt1_kernel<T, 1><<<grid, 128, 0, st>>>((const T*)a->att1, a->out1, d.O1, (int64_t)d.B * d.O1, a->de,
                                                                       a->w_full, (T*)a->datt1, a->g_w_full, d.T, d.R, d.A)));
    }
    LO_LAUNCH_OK();
  }
  // encoder_att: g_W = datt1^T enc ; g_b = colsum(datt1) ; denc = datt1 @ W_e
  if (tc) {
    LO_CUDA(cudaMemsetAsync(a->g_w_enc_att, 0, (size_t)d.A * d.C * 4, st));
    LO_TRY(tc_gemm_tn((const bf16*)a->datt1, d.A, (const bf16*)a->enc, d.C, a->g_w_enc_att, d.C, d.A, d.C, d.B * d.R, st));
    transpose_kernel<bf16><<<dim3(cdiv(d.C, 32), cdiv(d.A, 32)), dim3(32, 8), 0, st>>>((const bf16*)a->w_enc_att, d.C, wet_bf, d.A, d.A, d.C);
    LO_LAUNCH_OK();
    LO_TRY(tc_gemm_nt((const bf16*)a->datt1, d.A, wet_bf, d.A, a->denc, LO_F32, d.C, d.B * d.R, d.C, d.A, nullptr, 0, 0, st));
  } else {
    LO_TRY(gemm_tn(a->datt1, dt, d.A, a->enc, dt, d.C, a->g_w_enc_att, LO_F32, d.C, d.A, d.C, d.B * d.R, 0, LO_IMPL_SIMT, st));
    LO_TRY(gemm_nn(a->datt1, dt, d.A, a->w_enc_att, dt, d.C, a->denc, LO_F32, d.C, d.B * d.R, d.C, d.A, 0, LO_IMPL_SIMT, st));
  }
  LO_TRY(colsum(a->datt1, dt, a->g_b_enc_att, d.B * d.R, d.A, d.A, 0, st));
  // denc[b] += alphas[b]^T @ dctx[:, b, :]   (the context read, summed over time — a batched GEMM instead of a per-step RMW)
  if (tc && d.C % 8 == 0) {
    // tcgen05, one launch (3-D tensor maps, grid.y = batch); bf16 operands cast once after the loop
    const int Rp = (int)rpad8(d.R);
    cast_pad_rows_kernel<<<148 * 8, 256, 0, st>>>(a->alphas, bv.alphas, BT, d.R, Rp);
    LO_LAUNCH_OK();
    cast_tb_to_bt_kernel<<<148 * 8, 256, 0, st>>>(a->dctx, bv.dctx, d.T, d.B, d.C);
    LO_LAUNCH_OK();
    LO_TRY(tc_gemm_tn_batched(bv.alphas, Rp, (int64_t)d.T * Rp, bv.dctx, d.C, (int64_t)d.T * d.C, a->denc, d.C, (int64_t)d.R * d.C, d.R,
                              d.C, d.T, d.B, st));
  } else {
    GemmDesc g{d.R, d.C, d.T, 1, d.R, (int64_t)d.B * d.C, 1, d.C, d.B, (int64_t)d.T * d.R, d.C, (int64_t)d.R * d.C, nullptr, 1, 0};
    LO_TRY(gemm(a->alphas, LO_F32, a->dctx, LO_F32, a->denc, LO_F32, g, LO_IMPL_SIMT, st));
  }
  // init_h / init_c
  LO_TRY(gemm_tn(a->dinit, LO_F32, 2 * d.D, a->mean, LO_F32, d.C, a->g_w_init, LO_F32, d.C, 2 * d.D, d.C, d.B, 0, LO_IMPL_SIMT, st));
  LO_TRY(colsum(a->dinit, LO_F32, a->g_b_init, d.B, 2 * d.D, 2 * d.D, 0, st));
  LO_TRY(gemm_nn(a->dinit, LO_F32, 2 * d.D, a->w_init, dt, d.C, a->dmean, LO_F32, d.C, d.B, d.C, 2 * d.D, 0, LO_IMPL_SIMT, st));
  {
    const int64_t total = (int64_t)d.B * d.R * d.C;
    add_rowbcast_kernel<<<148 * 8, 256, 0, st>>>(a->denc, a->dmean, d.R, d.C, 1.0f / (float)d.R, total);
    LO_LAUNCH_OK();
  }
  if (a->has_dropout == 2) {
    // forward and backward of this step drew the same Philox stream; the next step (also a graph replay) gets a new one
    bump_counter_kernel<<<1, 1, 0, st>>>((unsigned long long*)a->dropout_state + 1);
    LO_LAUNCH_OK();
  }
  return LO_OK;
}

int lo_decoder_greedy_hist(const lo_decoder_args* a, int64_t start_id, int64_t end_id, int max_steps, int64_t* tokens,
                           int32_t* finished, int32_t* fin_hist, void* stream) {
  return greedy_loop(a, nullptr, start_id, end_id, max_steps, tokens, finished, fin_hist, (cudaStream_t)stream);
}

int lo_decoder_greedy(const lo_decoder_args* a, int64_t start_id, int64_t end_id, int max_steps, int64_t* tokens,
                      int32_t* finished, void* stream) {
  return lo_decoder_greedy_hist(a, start_id, end_id, max_steps, tokens, finished, nullptr, stream);
}

int lo_decoder_beam(const lo_decoder_args* a, int64_t start_id, int64_t end_id, int max_steps, int64_t* ids, int64_t* parents,
                    int32_t* fin_hist, float* logp, void* stream) {
  return lo_decoder_beam_div(a, start_id, end_id, max_steps, ids, parents, fin_hist, logp, 1.f, 0.f, nullptr, nullptr, stream);
}

int lo_decoder_beam_div(const lo_decoder_args* a, int64_t start_id, int64_t end_id, int max_steps, int64_t* ids, int64_t* parents,
                        int32_t* fin_hist, float* logp, float div_gamma, float div_prob, const float* div_u,
                        const uint64_t* div_state, void* stream) {
  return beam_loop(a, nullptr, start_id, end_id, max_steps, ids, parents, fin_hist, logp, div_gamma, div_prob, div_u, div_state,
                   (cudaStream_t)stream);
}

}  // extern "C"

// TensorFlow-flavour (Genthial) decoder: same translation unit, shares the kernels above
#include "lo_tfdecoder.cuh"
// generic sequence LSTM (extension: row-encoder biLSTM, second decoder layer)
#include "lo_lstmseq.cuh"
