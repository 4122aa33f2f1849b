// Attention step kernels, version 2: the att1 / enc row streams go through a TMA bulk-copy (cp.async.bulk) ->
// shared-memory ring fed by a dedicated producer warp, so the bytes in flight per SM (2 CTAs x 3 stages x 32 KB)
// no longer depend on register-limited occupancy.  Same math, same combine order, same outputs as the register
// versions in lo_decoder.cu (attention_fwd_kernel / attention_bwd_kernel), which remain the fallback.
//   forward : e_r = w . relu(att1_r + att2) ; online softmax ; ctx = sum_r alpha_r enc_r      (seq2seq_torch.py:186-190)
//   backward: dalpha_r = <dctx, enc_r> + dreg_r ; de_r = alpha_r (dalpha_r - s) ; datt2 = w * sum_r de_r [att1_r + att2 > 0]
// L2 policy: enc is read again by the next step (and by the backward) -> evict_last; att1 likewise is re-read every
// step; which of the two to pin is a run-time option (lo_set_option) because together they are as large as the L2.
#include <cooperative_groups.h>

#include "lo_common.cuh"
#include "lo_ptx.cuh"

namespace cg = cooperative_groups;

namespace lo {

int g_opt_att_pipe = 1;
int g_opt_pdl = 1;               // programmatic dependent launch for the per-step kernels
int g_opt_att_policy_enc = 1;    // 0 normal, 1 evict_last, 2 evict_first
int g_opt_att_policy_att1 = 2;
int g_opt_att_nsplit = 0;        // 0 = automatic
int g_opt_att_cluster = 1;
int g_opt_att_abi_pdl = 0;       // 1: the stand-alone attention entry points may use programmatic dependent launch too (bench probes)
int g_opt_att_bwd_mma = 1;       // 1: 512-wide bf16 backward with both contractions on mma.sync (attention_bwd_mma_kernel)
int g_opt_att_maskbits = 1;      // 1: the forward attention kernel stores the ReLU mask bits, the backward streams them instead of att1       // 1: the splits of one batch row form a thread-block cluster and combine through DSMEM

#ifndef LO_ATT_RPW
#define LO_ATT_RPW 2          // rows per consumer warp per stage (bf16): 2 -> 32 KB stages, 2 CTAs/SM ; 1 -> 16 KB stages, 3 CTAs/SM
#endif
#ifndef LO_ATT_MINB
#define LO_ATT_MINB 2
#endif
#define AP_THREADS 288
#define AP_CWARPS 8
#define AP_STAGES 3
#define AP_MAXSPLIT 16


// ---- timing build only (-DLO_ATT_TIMING, tools/att_timeline.py): per-CTA %globaltimer stamps of the last attention launch
#ifdef LO_ATT_TIMING
__device__ long long* g_att_ts = nullptr;
__device__ __forceinline__ void att_ts(int k) {
  if (g_att_ts) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_att_ts[((int64_t)blockIdx.y * gridDim.x + blockIdx.x) * 16 + k] = t;
  }
}
#define ATT_TS(k, cond) do { if (cond) att_ts(k); } while (0)
#else
#define ATT_TS(k, cond) do { } while (0)
#endif

__device__ __forceinline__ uint64_t make_policy(int kind) {
  return kind == 1 ? l2_policy_evict_last() : (kind == 2 ? l2_policy_evict_first() : l2_policy_evict_normal());
}

// score non-linearity: ACT 0 = ReLU (torch flavour, seq2seq_torch.py:188), 1 = tanh (Genthial cell, attention_mechanism.py:82)
template <int ACT, bool APPROX>
__device__ __forceinline__ float att_act(float x) {
  if constexpr (ACT == 0) return fmaxf(x, 0.f);
  else if constexpr (APPROX) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
  } else return tanhf(x);
}
// derivative given the pre-activation (ReLU) / the activation value (tanh)
template <int ACT>
__device__ __forceinline__ float att_dact(float pre, float post) {
  if constexpr (ACT == 0) return pre > 0.f ? 1.f : 0.f;
  else return 1.f - post * post;
}

// rows per split of the BACKWARD mask kernels: even, so that every stage starts on an (even, odd) row pair of the mask layout
__host__ __device__ __forceinline__ int att_rows_per_split(int R, int nsplit) { return (((R + nsplit - 1) / nsplit) + 1) & ~1; }

// NVA / NVC: 256-element groups per att1 row / per enc row (the torch flavour has A = C; the Genthial cell dim_e = 256 < C = 512)
template <typename T, int NVA, int NVC>
struct ApCfg {
  static constexpr int CHA = NVA * 256;
  static constexpr int CHC = NVC * 256;
  static constexpr int NVM = NVA > NVC ? NVA : NVC;
  static constexpr int RPW = (sizeof(T) == 2 && NVM <= 2) ? LO_ATT_RPW : 1;      // rows per consumer warp per stage
  static constexpr int ROWS = AP_CWARPS * RPW;
  static constexpr int HALF_A = ROWS * CHA;                             // att1 part
  static constexpr int HALF_C = ROWS * CHC;                             // enc part
  static constexpr int STAGE_ELEMS = HALF_A + HALF_C;
  static constexpr int STAGE_BYTES = STAGE_ELEMS * (int)sizeof(T);
  static constexpr int SMEM = AP_STAGES * STAGE_BYTES + 128;
};

template <typename T, int NVA, int NVC, bool CL, int ACT, bool MK>
__global__ void __launch_bounds__(AP_THREADS, LO_ATT_MINB) attention_fwd_pipe_kernel(
    const T* __restrict__ att1, const T* __restrict__ enc, const float* __restrict__ att2, int64_t att2_stride,
    const float* __restrict__ wf, float* __restrict__ alpha, int64_t alpha_stride, float* __restrict__ ctx,
    float* __restrict__ gate_pre, int64_t gate_stride, float* __restrict__ gctx, bf16* __restrict__ gctx_bf, int R, int nsplit,
    int* __restrict__ counters, float* __restrict__ partials, int pol_enc, int pol_att1, int rpi, uint8_t* __restrict__ mask_out) {
  using C = ApCfg<T, NVA, NVC>;
  constexpr int CHA = C::CHA, CHC = C::CHC;
  extern __shared__ __align__(128) uint8_t ap_smem[];
  T* ring = reinterpret_cast<T*>(ap_smem);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ap_smem + AP_STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + AP_STAGES;
  float* s_e = reinterpret_cast<float*>(ap_smem + AP_STAGES * C::STAGE_BYTES + 128);   // cluster mode: raw scores of this CTA's rows
  __shared__ float s_m[AP_CWARPS], s_l[AP_CWARPS];
  __shared__ float s_scale[AP_MAXSPLIT];
  __shared__ float s_ML[2];
  __shared__ int s_last;

  const int b = blockIdx.y, sp = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int rps = (R + nsplit - 1) / nsplit;
  const int r0 = sp * rps, r1 = min(R, r0 + rps);
  const int nst = r1 > r0 ? (r1 - r0 + C::ROWS - 1) / C::ROWS : 0;
  const T* a1b = att1 + (int64_t)(b / rpi) * R * CHA;      // beam search: rpi consecutive rows attend over one image
  const T* eb = enc + (int64_t)(b / rpi) * R * CHC;
  float* alb = alpha + (int64_t)b * alpha_stride;
  ATT_TS(0, threadIdx.x == 0);

  if (threadIdx.x == 0) {
    for (int s = 0; s < AP_STAGES; s++) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, AP_CWARPS);
    }
    fence_barrier_init();
  }
  __syncthreads();
  // PDL: the producer's bulk copies read only loop-invariant tensors (att1, enc: written long before the preceding kernel), so they
  // are issued BEFORE griddepcontrol.wait and overlap the tail of the preceding launch; consumers wait before touching its results.
  float m = -INFINITY, l = 0.f;
  float gate_pf = 0.f;
  float acc[NVC * 8];
#pragma unroll
  for (int i = 0; i < NVC * 8; i++) acc[i] = 0.f;

  if (wid == AP_CWARPS) {
    // ===== producer warp: one lane issues the bulk copies =====
    if (lane == 0) {
      const uint64_t pe = make_policy(pol_enc), pa = make_policy(pol_att1);
      for (int i = 0; i < nst; i++) {
        const int s = i % AP_STAGES;
        const uint32_t ph = (i / AP_STAGES) & 1;
        mbar_wait(empty_bar + s, ph ^ 1);
        const int row = r0 + i * C::ROWS;
        const int rows = min(C::ROWS, r1 - row);
        const uint32_t bytes_a = (uint32_t)rows * CHA * (uint32_t)sizeof(T), bytes_c = (uint32_t)rows * CHC * (uint32_t)sizeof(T);
        T* sa = ring + (size_t)s * C::STAGE_ELEMS;
        mbar_expect_tx(full_bar + s, bytes_a + bytes_c);
        ATT_TS(6, i == 0);
        ATT_TS(7, i == nst - 1);
        if (pol_att1 == 3) bulk_g2s_nohint(sa, a1b + (int64_t)row * CHA, bytes_a, full_bar + s);
        else bulk_g2s(sa, a1b + (int64_t)row * CHA, bytes_a, full_bar + s, pa);
        if (pol_enc == 3) bulk_g2s_nohint(sa + C::HALF_A, eb + (int64_t)row * CHC, bytes_c, full_bar + s);
        else bulk_g2s(sa + C::HALF_A, eb + (int64_t)row * CHC, bytes_c, full_bar + s, pe);
      }
    }
    __syncwarp();
    pdl_wait();          // the producer warp joins the combine below, which reads the preceding kernel's results
  } else {
    // ===== consumer warps =====
    float a2[NVA * 8], wv[NVA * 8];
#pragma unroll
    for (int j = 0; j < NVA; j++) ld8(wf + (j * 32 + lane) * 8, wv + j * 8);        // a parameter: independent of the preceding launch
    pdl_wait();
    ATT_TS(1, threadIdx.x == 0);
    pdl_trigger();
#pragma unroll
    for (int j = 0; j < NVA; j++) ld8(att2 + (int64_t)b * att2_stride + (j * 32 + lane) * 8, a2 + j * 8);
    // mask bits: the score loop works on n = (0 - att2) - att1 = -(att1 + att2), whose SIGN bit is set exactly when att1 + att2 > 0.
    // The negation rounds symmetrically, an exact cancellation gives +0, and 0 - att2 is never -0, so no pair of zeros gives -0 either.
    if constexpr (MK) {
#pragma unroll
      for (int i = 0; i < NVA * 8; i++) a2[i] = 0.f - a2[i];
    }
    // cluster mode: the gate pre-activation of the channel this thread finalises after the combine (one L2 round trip off the tail)
    if (CL && gate_pre && (int)threadIdx.x < (CHC + nsplit - 1) / nsplit && sp * ((CHC + nsplit - 1) / nsplit) + (int)threadIdx.x < CHC)
      gate_pf = gate_pre[(int64_t)b * gate_stride + sp * ((CHC + nsplit - 1) / nsplit) + threadIdx.x];
    ATT_TS(2, threadIdx.x == 0);
    for (int i = 0; i < nst; i++) {
      const int s = i % AP_STAGES;
      const uint32_t ph = (i / AP_STAGES) & 1;
      const int row = r0 + i * C::ROWS;
      const int rows = min(C::ROWS, r1 - row);
      mbar_wait(full_bar + s, ph);
      ATT_TS(3, threadIdx.x == 0 && i == 0);
      const uint32_t sa = smem_u32(ring + (size_t)s * C::STAGE_ELEMS);
      const uint32_t se = sa + C::HALF_A * (uint32_t)sizeof(T);
      constexpr uint32_t ES = (uint32_t)sizeof(T);
      const int ra = wid, rb = wid + AP_CWARPS;
      const bool one = ra < rows;
      const bool two = (C::RPW == 2) && (rb < rows);
      if (one) {
        float e0 = 0.f, e1 = 0.f;
        // training (ReLU score): bit 7 - (c % 8) of byte c/8 of row r = (att1[r][c] + att2[c] > 0); the backward reads these
        // 64 bytes per row instead of the 1 KB att1 row
        // layout: byte (r, c/8) at (r/2) * 2*(CHA/8) + (c/8)*2 + (r&1) — the bytes of an (even, odd) row pair are adjacent, which
        // is what the tensor-core backward wants (one 32-bit word per lane = its four A fragments of a 16 x 16 block)
        uint8_t* mrow = MK ? mask_out + (int64_t)b * ((R + 1) & ~1) * (CHA / 8) : nullptr;
#pragma unroll
        for (int j = 0; j < NVA; j++) {
          float v[8];
          lds8(sa + ((uint32_t)ra * CHA + (j * 32 + lane) * 8) * ES, v, (const T*)nullptr);
          uint32_t bits = 0;
#pragma unroll
          for (int q = 0; q < 8; q++) {
            // one funnel shift per element collects the sign bits of n = -pre (element q -> bit 7-q): bit = pre > 0, +0 included
            float pre;
            if constexpr (MK) {
              const float n = a2[j * 8 + q] - v[q];
              bits = __funnelshift_l(__float_as_uint(n), bits, 1);
              pre = -n;
            } else {
              pre = v[q] + a2[j * 8 + q];
            }
            e0 = fmaf(wv[j * 8 + q], att_act<ACT, sizeof(T) == 2>(pre), e0);
          }
          if (MK) mrow[(int64_t)((row + ra) >> 1) * (CHA / 4) + (j * 32 + lane) * 2 + ((row + ra) & 1)] = (uint8_t)bits;
          if (two) {
            lds8(sa + ((uint32_t)rb * CHA + (j * 32 + lane) * 8) * ES, v, (const T*)nullptr);
            bits = 0;
#pragma unroll
            for (int q = 0; q < 8; q++) {
              float pre;
              if constexpr (MK) {
                const float n = a2[j * 8 + q] - v[q];
                bits = __funnelshift_l(__float_as_uint(n), bits, 1);
                pre = -n;
              } else {
                pre = v[q] + a2[j * 8 + q];
              }
              e1 = fmaf(wv[j * 8 + q], att_act<ACT, sizeof(T) == 2>(pre), e1);
            }
            if (MK) mrow[(int64_t)((row + rb) >> 1) * (CHA / 4) + (j * 32 + lane) * 2 + ((row + rb) & 1)] = (uint8_t)bits;
          }
        }
        e0 = warp_sum(e0);
        e1 = warp_sum(e1);
        if (lane == 0) {
          if constexpr (CL) {
            s_e[row + ra - r0] = e0;
            if (two) s_e[row + rb - r0] = e1;
          } else {
            alb[row + ra] = e0;
            if (two) alb[row + rb] = e1;
          }
        }
        const float mn = two ? fmaxf(m, fmaxf(e0, e1)) : fmaxf(m, e0);
        const float sc = expf(m - mn);
        const float p0 = expf(e0 - mn);
        const float p1 = two ? expf(e1 - mn) : 0.f;
        l = l * sc + p0 + p1;
#pragma unroll
        for (int j = 0; j < NVC; j++) {
          float u[8];
          lds8(se + ((uint32_t)ra * CHC + (j * 32 + lane) * 8) * ES, u, (const T*)nullptr);
#pragma unroll
          for (int q = 0; q < 8; q++) acc[j * 8 + q] = fmaf(p0, u[q], acc[j * 8 + q] * sc);
          if (two) {
            lds8(se + ((uint32_t)rb * CHC + (j * 32 + lane) * 8) * ES, u, (const T*)nullptr);
#pragma unroll
            for (int q = 0; q < 8; q++) acc[j * 8 + q] = fmaf(p1, u[q], acc[j * 8 + q]);
          }
        }
        m = mn;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_bar + s);
    }
  }
  ATT_TS(4, threadIdx.x == 0);
  __syncthreads();     // every TMA write has landed and been consumed: the ring can be reused for the combine
  ATT_TS(8, threadIdx.x == 0);
  float* s_acc = reinterpret_cast<float*>(ap_smem);          // [AP_CWARPS][CHC]
  if (wid < AP_CWARPS) {
    if (lane == 0) { s_m[wid] = m; s_l[wid] = l; }
#pragma unroll
    for (int j = 0; j < NVC; j++)
#pragma unroll
      for (int i = 0; i < 8; i++) s_acc[wid * CHC + (j * 32 + lane) * 8 + i] = acc[j * 8 + i];
  }
  __syncthreads();
  float M = -INFINITY;
#pragma unroll
  for (int w = 0; w < AP_CWARPS; w++) M = fmaxf(M, s_m[w]);
  float L = 0.f;
  float wsc[AP_CWARPS];
#pragma unroll
  for (int w = 0; w < AP_CWARPS; w++) {
    wsc[w] = (s_m[w] == -INFINITY) ? 0.f : expf(s_m[w] - M);
    L += s_l[w] * wsc[w];
  }
  if constexpr (CL) {
    // ===== cluster combine: the nsplit CTAs of this batch row exchange (M, L, acc) through distributed shared memory =====
    cg::cluster_group cluster = cg::this_cluster();
    float* s_part = s_acc + AP_CWARPS * CHC;                 // [CHC] combined accumulator of this CTA (still inside the ring)
    __shared__ float s_MLp[2];
    for (int c = threadIdx.x; c < CHC; c += AP_THREADS) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < AP_CWARPS; w++) t = fmaf(s_acc[w * CHC + c], wsc[w], t);
      s_part[c] = t;
    }
    if (threadIdx.x == 0) { s_MLp[0] = M; s_MLp[1] = L; }
    cluster.sync();
    float Mg = -INFINITY;
    for (int q = 0; q < nsplit; q++) Mg = fmaxf(Mg, cluster.map_shared_rank(s_MLp, q)[0]);
    float Lg = 0.f;
    float scl[8];
#pragma unroll
    for (int q = 0; q < 8; q++) {
      scl[q] = 0.f;
      if (q < nsplit) {
        const float* ml = cluster.map_shared_rank(s_MLp, q);
        const float ms = ml[0];
        scl[q] = (ms == -INFINITY) ? 0.f : expf(ms - Mg);
        Lg += ml[1] * scl[q];
      }
    }
    const float invL = 1.0f / Lg;
    // this CTA finalises its slice of the channels ...
    const int cps = (CHC + nsplit - 1) / nsplit;
    for (int c = sp * cps + threadIdx.x; c < min(CHC, (sp + 1) * cps); c += AP_THREADS) {
      float t = 0.f;
#pragma unroll
      for (int q = 0; q < 8; q++)
        if (q < nsplit) t = fmaf(cluster.map_shared_rank(s_part, q)[c], scl[q], t);
      t *= invL;
      ctx[(int64_t)b * CHC + c] = t;
      if (gate_pre) {
        const bool pf = c == sp * cps + (int)threadIdx.x && (int)threadIdx.x < AP_CWARPS * 32;     // fetched before the main loop
        const float g = sigmoidf_(pf ? gate_pf : gate_pre[(int64_t)b * gate_stride + c]);
        gate_pre[(int64_t)b * gate_stride + c] = g;
        gctx[(int64_t)b * CHC + c] = g * t;
        if (gctx_bf) gctx_bf[(int64_t)b * CHC + c] = __float2bfloat16_rn(g * t);
      } else if (gctx_bf) {
        gctx_bf[(int64_t)b * CHC + c] = __float2bfloat16_rn(t);      // no gate (Genthial cell): bf16 mirror of the context itself
      }
    }
    // ... and normalises the attention weights of its own rows (scores never leave shared memory)
    for (int r = r0 + threadIdx.x; r < r1; r += AP_THREADS) alb[r] = expf(s_e[r - r0] - Mg) * invL;
    cluster.sync();                                          // peers may still be reading this CTA's shared memory
    ATT_TS(5, threadIdx.x == 0);
    return;
  }
  float* part = partials + ((int64_t)b * nsplit + sp) * (CHC + 2);
  for (int c = threadIdx.x; c < CHC; c += AP_THREADS) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < AP_CWARPS; w++) t = fmaf(s_acc[w * CHC + c], wsc[w], t);
    part[2 + c] = t;
  }
  if (threadIdx.x == 0) { part[0] = M; part[1] = L; }
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
  const float* pb = partials + (int64_t)b * nsplit * (CHC + 2);
  if (threadIdx.x == 0) {
    float Mg = -INFINITY;
    for (int s = 0; s < nsplit; s++) Mg = fmaxf(Mg, __ldcg(pb + (int64_t)s * (CHC + 2)));
    float Lg = 0.f;
    for (int s = 0; s < nsplit; s++) {
      const float ms = __ldcg(pb + (int64_t)s * (CHC + 2));
      const float scl = (ms == -INFINITY) ? 0.f : expf(ms - Mg);
      s_scale[s] = scl;
      Lg += __ldcg(pb + (int64_t)s * (CHC + 2) + 1) * scl;
    }
    s_ML[0] = Mg;
    s_ML[1] = 1.0f / Lg;
  }
  __syncthreads();
  const float Mg = s_ML[0], invL = s_ML[1];
  for (int c = threadIdx.x; c < CHC; c += AP_THREADS) {
    float t = 0.f;
    for (int s = 0; s < nsplit; s++) t = fmaf(__ldcg(pb + (int64_t)s * (CHC + 2) + 2 + c), s_scale[s], t);
    t *= invL;
    ctx[(int64_t)b * CHC + c] = t;
    if (gate_pre) {
      const float g = sigmoidf_(gate_pre[(int64_t)b * gate_stride + c]);
      gate_pre[(int64_t)b * gate_stride + c] = g;
      gctx[(int64_t)b * CHC + c] = g * t;
      if (gctx_bf) gctx_bf[(int64_t)b * CHC + c] = __float2bfloat16_rn(g * t);
    } else if (gctx_bf) {
      gctx_bf[(int64_t)b * CHC + c] = __float2bfloat16_rn(t);
    }
  }
  for (int r = threadIdx.x; r < R; r += AP_THREADS) alb[r] = expf(__ldcg(alb + r) - Mg) * invL;
}

template <typename T, int NVA, int NVC, bool CL, int ACT>
__global__ void __launch_bounds__(AP_THREADS) attention_bwd_pipe_kernel(
    const T* __restrict__ att1, const T* __restrict__ enc, const float* __restrict__ att2, const float* __restrict__ gate,
    int64_t o1_stride, const float* __restrict__ wf, const float* __restrict__ alpha, int64_t alpha_stride,
    const float* __restrict__ ctx, const float* __restrict__ dgctx, int64_t dg_stride, const float* __restrict__ dreg,
    int64_t dreg_stride, const float* __restrict__ sreg, int64_t sreg_stride, float* __restrict__ de, float* __restrict__ datt2,
    float* __restrict__ dgp, int64_t dcat_stride, bf16* __restrict__ datt2_bf, bf16* __restrict__ dgp_bf,
    float* __restrict__ dctx_out, int R, int nsplit, int* __restrict__ counters, float* __restrict__ partials, int pol_enc,
    int pol_att1, float* __restrict__ dwf_part) {
  using C = ApCfg<T, NVA, NVC>;
  constexpr int CHA = C::CHA, CHC = C::CHC;
  extern __shared__ __align__(128) uint8_t ap_smem[];
  T* ring = reinterpret_cast<T*>(ap_smem);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ap_smem + AP_STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + AP_STAGES;
  __shared__ int s_last;
  const int b = blockIdx.y, sp = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int rps = (R + nsplit - 1) / nsplit;
  const int r0 = sp * rps, r1 = min(R, r0 + rps);
  const int nst = r1 > r0 ? (r1 - r0 + C::ROWS - 1) / C::ROWS : 0;
  const T* a1b = att1 + (int64_t)b * R * CHA;
  const T* eb = enc + (int64_t)b * R * CHC;
  if (threadIdx.x == 0) {
    for (int s = 0; s < AP_STAGES; s++) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, AP_CWARPS);
    }
    fence_barrier_init();
  }
  __syncthreads();
  // PDL: the producer's bulk copies read only loop-invariant tensors (att1, enc: written long before the preceding kernel), so they
  // are issued BEFORE griddepcontrol.wait and overlap the tail of the preceding launch; consumers wait before touching its results.
  float macc[NVA * 8], wacc[NVA * 8];     // wacc: d w_full partial = sum_r de_r * relu(att1_r + att2)   (full_att.weight gradient)
#pragma unroll
  for (int i = 0; i < NVA * 8; i++) { macc[i] = 0.f; wacc[i] = 0.f; }

  if (wid == AP_CWARPS) {
    if (lane == 0) {
      const uint64_t pe = make_policy(pol_enc), pa = make_policy(pol_att1);
      for (int i = 0; i < nst; i++) {
        const int s = i % AP_STAGES;
        const uint32_t ph = (i / AP_STAGES) & 1;
        mbar_wait(empty_bar + s, ph ^ 1);
        const int row = r0 + i * C::ROWS;
        const int rows = min(C::ROWS, r1 - row);
        const uint32_t bytes_a = (uint32_t)rows * CHA * (uint32_t)sizeof(T), bytes_c = (uint32_t)rows * CHC * (uint32_t)sizeof(T);
        T* sa = ring + (size_t)s * C::STAGE_ELEMS;
        mbar_expect_tx(full_bar + s, bytes_a + bytes_c);
        if (pol_att1 == 3) bulk_g2s_nohint(sa, a1b + (int64_t)row * CHA, bytes_a, full_bar + s);
        else bulk_g2s(sa, a1b + (int64_t)row * CHA, bytes_a, full_bar + s, pa);
        if (pol_enc == 3) bulk_g2s_nohint(sa + C::HALF_A, eb + (int64_t)row * CHC, bytes_c, full_bar + s);
        else bulk_g2s(sa + C::HALF_A, eb + (int64_t)row * CHC, bytes_c, full_bar + s, pe);
      }
    }
    __syncwarp();
    pdl_wait();          // the producer warp joins the combine below, which reads the preceding kernel's results
  } else {
    float a2[NVA * 8], dc[NVC * 8];
    float sdot = 0.f;
    // att2 / gate / ctx / sreg were saved by the forward pass: they are fetched BEFORE griddepcontrol.wait (overlapping the tail of
    // the preceding launch); only d gctx comes from the preceding kernel
    float gv[NVC * 8], cxv[NVC * 8];
#pragma unroll
    for (int j = 0; j < NVA; j++) ld8(att2 + (int64_t)b * o1_stride + (j * 32 + lane) * 8, a2 + j * 8);
#pragma unroll
    for (int j = 0; j < NVC; j++) {
      const int c0 = (j * 32 + lane) * 8;
      if (gate) ld8(gate + (int64_t)b * o1_stride + c0, gv + j * 8);
      ld8(ctx + (int64_t)b * CHC + c0, cxv + j * 8);
    }
    const float sreg_b = sreg ? sreg[(int64_t)b * sreg_stride] : 0.f;
    pdl_wait();
    pdl_trigger();
#pragma unroll
    for (int j = 0; j < NVC; j++) {
      const int c0 = (j * 32 + lane) * 8;
      float dg[8], gp[8];
      const float* g = gv + j * 8;
      const float* cx = cxv + j * 8;
      ld8(dgctx + (int64_t)b * dg_stride + c0, dg);
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const float gi = gate ? g[i] : 1.f;                // Genthial cell: the context is used ungated
        dc[j * 8 + i] = dg[i] * gi;
        sdot = fmaf(dc[j * 8 + i], cx[i], sdot);
        gp[i] = dg[i] * cx[i] * gi * (1.f - gi);
      }
      if (sp == 0 && wid == 0) {
        if (dgp) st8(dgp + (int64_t)b * dcat_stride + c0, gp);
        if (dgp_bf) st8(dgp_bf + (int64_t)b * dcat_stride + c0, gp);
        if (dctx_out) st8(dctx_out + (int64_t)b * CHC + c0, dc + j * 8);
      }
    }
    const float sall = warp_sum(sdot) + sreg_b;
    const float* alb = alpha + (int64_t)b * alpha_stride;
    float* deb = de + (int64_t)b * alpha_stride;
    const float* drb = dreg + (int64_t)b * dreg_stride;
    // per-row scalars (alpha, d reg) are fetched one stage ahead: a dependent global load after the warp reduction would sit on
    // the critical path of every stage
    float pa0 = 0.f, pa1 = 0.f, pd0 = 0.f, pd1 = 0.f;
    auto prefetch = [&](int i) {
      const int row = r0 + i * C::ROWS;
      const int rows = min(C::ROWS, r1 - row);
      const int ra = wid, rb = wid + AP_CWARPS;
      if (i < nst && ra < rows) {
        pa0 = alb[row + ra];
        pd0 = dreg ? drb[row + ra] : 0.f;
        if (C::RPW == 2 && rb < rows) {
          pa1 = alb[row + rb];
          pd1 = dreg ? drb[row + rb] : 0.f;
        }
      }
    };
    prefetch(0);
    for (int i = 0; i < nst; i++) {
      const int s = i % AP_STAGES;
      const uint32_t ph = (i / AP_STAGES) & 1;
      const int row = r0 + i * C::ROWS;
      const int rows = min(C::ROWS, r1 - row);
      const float al0 = pa0, al1 = pa1, dr0 = pd0, dr1 = pd1;
      prefetch(i + 1);
      mbar_wait(full_bar + s, ph);
      const T* sa = ring + (size_t)s * C::STAGE_ELEMS;
      const T* se = sa + C::HALF_A;
      const int ra = wid, rb = wid + AP_CWARPS;
      const bool one = ra < rows;
      const bool two = (C::RPW == 2) && (rb < rows);
      if (one) {
        float d0 = 0.f, d1 = 0.f;
#pragma unroll
        for (int j = 0; j < NVC; j++) {
          float u[8];
          ld8(se + (size_t)ra * CHC + (j * 32 + lane) * 8, u);
#pragma unroll
          for (int q = 0; q < 8; q++) d0 = fmaf(dc[j * 8 + q], u[q], d0);
          if (two) {
            ld8(se + (size_t)rb * CHC + (j * 32 + lane) * 8, u);
#pragma unroll
            for (int q = 0; q < 8; q++) d1 = fmaf(dc[j * 8 + q], u[q], d1);
          }
        }
        d0 = warp_sum(d0);
        d1 = warp_sum(d1);
        const float de0 = al0 * (d0 + dr0 - sall);
        const float de1 = two ? al1 * (d1 + dr1 - sall) : 0.f;
        if (lane == 0) {
          deb[row + ra] = de0;
          if (two) deb[row + rb] = de1;
        }
#pragma unroll
        for (int j = 0; j < NVA; j++) {
          float v[8];
          ld8(sa + (size_t)ra * CHA + (j * 32 + lane) * 8, v);
#pragma unroll
          for (int q = 0; q < 8; q++) {
            const float pre = v[q] + a2[j * 8 + q];
            const float post = att_act<ACT, sizeof(T) == 2>(pre);
            macc[j * 8 + q] = fmaf(de0, att_dact<ACT>(pre, post), macc[j * 8 + q]);
            wacc[j * 8 + q] = fmaf(de0, post, wacc[j * 8 + q]);
          }
          if (two) {
            ld8(sa + (size_t)rb * CHA + (j * 32 + lane) * 8, v);
#pragma unroll
            for (int q = 0; q < 8; q++) {
              const float pre = v[q] + a2[j * 8 + q];
              const float post = att_act<ACT, sizeof(T) == 2>(pre);
              macc[j * 8 + q] = fmaf(de1, att_dact<ACT>(pre, post), macc[j * 8 + q]);
              wacc[j * 8 + q] = fmaf(de1, post, wacc[j * 8 + q]);
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_bar + s);
    }
  }
  __syncthreads();
  float* s_acc = reinterpret_cast<float*>(ap_smem);            // [8][CHA] mask sums | [2][CHA] CTA totals | [8][CHA] w_full sums
  float* s_part = s_acc + AP_CWARPS * CHA;
  float* s_wacc = s_part + 2 * CHA;
  if (wid < AP_CWARPS) {
#pragma unroll
    for (int j = 0; j < NVA; j++)
#pragma unroll
      for (int i = 0; i < 8; i++) {
        s_acc[wid * CHA + (j * 32 + lane) * 8 + i] = macc[j * 8 + i];
        s_wacc[wid * CHA + (j * 32 + lane) * 8 + i] = wacc[j * 8 + i];
      }
  }
  __syncthreads();
  if constexpr (CL) {
    cg::cluster_group cluster = cg::this_cluster();
    for (int c = threadIdx.x; c < CHA; c += AP_THREADS) {
      float t = 0.f, u = 0.f;
#pragma unroll
      for (int w = 0; w < AP_CWARPS; w++) { t += s_acc[w * CHA + c]; u += s_wacc[w * CHA + c]; }
      s_part[c] = t;
      s_part[CHA + c] = u;
    }
    cluster.sync();
    const int cps = (CHA + nsplit - 1) / nsplit;
    for (int c = sp * cps + threadIdx.x; c < min(CHA, (sp + 1) * cps); c += AP_THREADS) {
      float t = 0.f, u = 0.f;
      for (int q = 0; q < nsplit; q++) {                       // fixed order -> deterministic
        const float* rp = cluster.map_shared_rank(s_part, q);
        t += rp[c];
        u += rp[CHA + c];
      }
      datt2[(int64_t)b * dcat_stride + c] = t * wf[c];
      if (datt2_bf) datt2_bf[(int64_t)b * dcat_stride + c] = __float2bfloat16_rn(t * wf[c]);
      if (dwf_part) dwf_part[(int64_t)b * CHA + c] += u;       // one writer per (b, c): plain accumulate over the time loop
    }
    cluster.sync();
    return;
  }
  if (dwf_part) {
    for (int c = threadIdx.x; c < CHA; c += AP_THREADS) {
      float u = 0.f;
#pragma unroll
      for (int w = 0; w < AP_CWARPS; w++) u += s_wacc[w * CHA + c];
      atomicAdd(dwf_part + (int64_t)b * CHA + c, u);
    }
  }
  float* part = partials + ((int64_t)b * nsplit + sp) * (CHA + 2);
  for (int c = threadIdx.x; c < CHA; c += AP_THREADS) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < AP_CWARPS; w++) t += s_acc[w * CHA + c];
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
  const float* pb = partials + (int64_t)b * nsplit * (CHA + 2);
  for (int c = threadIdx.x; c < CHA; c += AP_THREADS) {
    float t = 0.f;
    for (int sidx = 0; sidx < nsplit; sidx++) t += __ldcg(pb + (int64_t)sidx * (CHA + 2) + 2 + c);
    datt2[(int64_t)b * dcat_stride + c] = t * wf[c];
    if (datt2_bf) datt2_bf[(int64_t)b * dcat_stride + c] = __float2bfloat16_rn(t * wf[c]);
  }
}

// ------------------------------------------------------------------------------------------------------------------------------
// Attention backward, mask-bit version (ReLU score): the forward kernel left 1 bit per att1 element (att1 + att2 > 0), so the
// backward streams enc rows (CHC elements) + CHA/8 mask bytes per region instead of enc + att1 rows: 60.5 MB instead of
// 114 MB per step at cfg #2.  Same math, same masks (the bits ARE the forward's comparisons), same combine order.
// d w_full: only its att2 term (sum_r on * de times att2) is accumulated here (dwf_part); the term that needs att1 itself is added by
// the post-loop sweep (datt1_kernel<.., WACC = 2>).
// ------------------------------------------------------------------------------------------------------------------------------
#define APM_STAGES 5
template <typename T, int NVA, int NVC>
struct ApmCfg {
  static constexpr int CHA = NVA * 256, CHC = NVC * 256;
  static constexpr int RPW = (sizeof(T) == 2 && NVC <= 2) ? LO_ATT_RPW : 1;
  static constexpr int ROWS = AP_CWARPS * RPW;
  static constexpr int ENC_BYTES = ROWS * CHC * (int)sizeof(T);
  static constexpr int MSK_BYTES = ROWS * (CHA / 8);
  static constexpr int STAGE_BYTES = ENC_BYTES + MSK_BYTES;
  static constexpr int SMEM = APM_STAGES * STAGE_BYTES + 128;
  static_assert(APM_STAGES * STAGE_BYTES >= (AP_CWARPS + 2) * CHA * 4, "combine scratch must fit in the ring");
};

template <typename T, int NVA, int NVC, bool CL>
__global__ void __launch_bounds__(AP_THREADS, LO_ATT_MINB) attention_bwd_mask_kernel(
    const uint8_t* __restrict__ mask, const T* __restrict__ enc, const float* __restrict__ gate, int64_t o1_stride,
    const float* __restrict__ wf, const float* __restrict__ alpha, int64_t alpha_stride, const float* __restrict__ ctx,
    const float* __restrict__ dgctx, int64_t dg_stride, const float* __restrict__ dreg, int64_t dreg_stride,
    const float* __restrict__ sreg, int64_t sreg_stride, float* __restrict__ de, float* __restrict__ datt2, float* __restrict__ dgp,
    int64_t dcat_stride, bf16* __restrict__ datt2_bf, bf16* __restrict__ dgp_bf, float* __restrict__ dctx_out, int R, int nsplit,
    int* __restrict__ counters, float* __restrict__ partials, int pol_enc, const float* __restrict__ att2,
    float* __restrict__ dwf_part) {
  using C = ApmCfg<T, NVA, NVC>;
  constexpr int CHA = C::CHA, CHC = C::CHC, MB = CHA / 8;
  extern __shared__ __align__(128) uint8_t ap_smem[];
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ap_smem + APM_STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + APM_STAGES;
  __shared__ int s_last;
  const int b = blockIdx.y, sp = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int rps = att_rows_per_split(R, nsplit);          // even (and ROWS is even): stages start on an (even, odd) row pair
  const int r0 = sp * rps, r1 = min(R, r0 + rps);
  const int nst = r1 > r0 ? (r1 - r0 + C::ROWS - 1) / C::ROWS : 0;
  const T* eb = enc + (int64_t)b * R * CHC;
  const uint8_t* mb = mask + (int64_t)b * ((R + 1) & ~1) * MB;      // pair layout, see attention_fwd_pipe_kernel
  if (threadIdx.x == 0) {
    for (int s = 0; s < APM_STAGES; s++) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, AP_CWARPS);
    }
    fence_barrier_init();
  }
  __syncthreads();
  float macc[NVA * 8];
#pragma unroll
  for (int i = 0; i < NVA * 8; i++) macc[i] = 0.f;

  if (wid == AP_CWARPS) {
    // producer: enc is loop-invariant (prefetchable before griddepcontrol.wait); the mask bits of this step were written by the
    // forward pass long ago as well
    if (lane == 0) {
      const uint64_t pe = make_policy(pol_enc), pm = l2_policy_evict_first();
      for (int i = 0; i < nst; i++) {
        const int s = i % APM_STAGES;
        const uint32_t ph = (i / APM_STAGES) & 1;
        mbar_wait(empty_bar + s, ph ^ 1);
        const int row = r0 + i * C::ROWS;
        const int rows = min(C::ROWS, r1 - row);
        const uint32_t bytes_c = (uint32_t)rows * CHC * (uint32_t)sizeof(T), bytes_m = (uint32_t)((rows + 1) >> 1) * 2u * MB;
        uint8_t* st = ap_smem + (size_t)s * C::STAGE_BYTES;
        mbar_expect_tx(full_bar + s, bytes_c + bytes_m);
        bulk_g2s(st, eb + (int64_t)row * CHC, bytes_c, full_bar + s, pe);
        bulk_g2s(st + C::ENC_BYTES, mb + (int64_t)row * MB, bytes_m, full_bar + s, pm);
      }
    }
    __syncwarp();
    pdl_wait();
  } else {
    float dc[NVC * 8];
    float sdot = 0.f;
    float gv[NVC * 8], cxv[NVC * 8];
#pragma unroll
    for (int j = 0; j < NVC; j++) {
      const int c0 = (j * 32 + lane) * 8;
      if (gate) ld8(gate + (int64_t)b * o1_stride + c0, gv + j * 8);
      ld8(ctx + (int64_t)b * CHC + c0, cxv + j * 8);
    }
    const float sreg_b = sreg ? sreg[(int64_t)b * sreg_stride] : 0.f;
    pdl_wait();
    pdl_trigger();
#pragma unroll
    for (int j = 0; j < NVC; j++) {
      const int c0 = (j * 32 + lane) * 8;
      float dg[8], gp[8];
      ld8(dgctx + (int64_t)b * dg_stride + c0, dg);
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const float gi = gate ? gv[j * 8 + i] : 1.f;
        dc[j * 8 + i] = dg[i] * gi;
        sdot = fmaf(dc[j * 8 + i], cxv[j * 8 + i], sdot);
        gp[i] = dg[i] * cxv[j * 8 + i] * gi * (1.f - gi);
      }
      if (sp == 0 && wid == 0) {
        if (dgp) st8(dgp + (int64_t)b * dcat_stride + c0, gp);
        if (dgp_bf) st8(dgp_bf + (int64_t)b * dcat_stride + c0, gp);
        if (dctx_out) st8(dctx_out + (int64_t)b * CHC + c0, dc + j * 8);
      }
    }
    const float sall = warp_sum(sdot) + sreg_b;
    const float* alb = alpha + (int64_t)b * alpha_stride;
    float* deb = de + (int64_t)b * alpha_stride;
    const float* drb = dreg + (int64_t)b * dreg_stride;
    float pa0 = 0.f, pa1 = 0.f, pd0 = 0.f, pd1 = 0.f;
    auto prefetch = [&](int i) {
      const int row = r0 + i * C::ROWS;
      const int rows = min(C::ROWS, r1 - row);
      const int ra = wid, rb = wid + AP_CWARPS;
      if (i < nst && ra < rows) {
        pa0 = alb[row + ra];
        pd0 = dreg ? drb[row + ra] : 0.f;
        if (C::RPW == 2 && rb < rows) {
          pa1 = alb[row + rb];
          pd1 = dreg ? drb[row + rb] : 0.f;
        }
      }
    };
    prefetch(0);
    for (int i = 0; i < nst; i++) {
      const int s = i % APM_STAGES;
      const uint32_t ph = (i / APM_STAGES) & 1;
      const int row = r0 + i * C::ROWS;
      const int rows = min(C::ROWS, r1 - row);
      const float al0 = pa0, al1 = pa1, dr0 = pd0, dr1 = pd1;
      prefetch(i + 1);
      mbar_wait(full_bar + s, ph);
      const uint32_t se = smem_u32(ap_smem + (size_t)s * C::STAGE_BYTES);
      constexpr uint32_t ES = (uint32_t)sizeof(T);
      const uint8_t* sm = ap_smem + (size_t)s * C::STAGE_BYTES + C::ENC_BYTES;
      const int ra = wid, rb = wid + AP_CWARPS;
      const bool one = ra < rows;
      const bool two = (C::RPW == 2) && (rb < rows);
      if (one) {
        float d0 = 0.f, d1 = 0.f;
#pragma unroll
        for (int j = 0; j < NVC; j++) {
          float u[8];
          lds8(se + ((uint32_t)ra * CHC + (j * 32 + lane) * 8) * ES, u, (const T*)nullptr);
#pragma unroll
          for (int q = 0; q < 8; q++) d0 = fmaf(dc[j * 8 + q], u[q], d0);
          if (two) {
            lds8(se + ((uint32_t)rb * CHC + (j * 32 + lane) * 8) * ES, u, (const T*)nullptr);
#pragma unroll
            for (int q = 0; q < 8; q++) d1 = fmaf(dc[j * 8 + q], u[q], d1);
          }
        }
        d0 = warp_sum(d0);
        d1 = warp_sum(d1);
        const float de0 = al0 * (d0 + dr0 - sall);
        const float de1 = two ? al1 * (d1 + dr1 - sall) : 0.f;
        if (lane == 0) {
          deb[row + ra] = de0;
          if (two) deb[row + rb] = de1;
        }
#pragma unroll
        for (int j = 0; j < NVA; j++) {
          const uint32_t m0 = sm[(ra >> 1) * 2 * MB + (j * 32 + lane) * 2 + (ra & 1)];
          const uint32_t m1 = two ? sm[(rb >> 1) * 2 * MB + (j * 32 + lane) * 2 + (rb & 1)] : 0u;
#pragma unroll
          for (int q = 0; q < 8; q++) {
            if (m0 & (0x80u >> q)) macc[j * 8 + q] += de0;
            if (m1 & (0x80u >> q)) macc[j * 8 + q] += de1;
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_bar + s);
    }
  }
  __syncthreads();
  float* s_acc = reinterpret_cast<float*>(ap_smem);            // [8][CHA] mask sums | [CHA] CTA totals
  float* s_part = s_acc + AP_CWARPS * CHA;
  if (wid < AP_CWARPS) {
#pragma unroll
    for (int j = 0; j < NVA; j++)
#pragma unroll
      for (int i = 0; i < 8; i++) s_acc[wid * CHA + (j * 32 + lane) * 8 + i] = macc[j * 8 + i];
  }
  __syncthreads();
  if constexpr (CL) {
    cg::cluster_group cluster = cg::this_cluster();
    for (int c = threadIdx.x; c < CHA; c += AP_THREADS) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < AP_CWARPS; w++) t += s_acc[w * CHA + c];
      s_part[c] = t;
    }
    cluster.sync();
    const int cps = (CHA + nsplit - 1) / nsplit;
    for (int c = sp * cps + threadIdx.x; c < min(CHA, (sp + 1) * cps); c += AP_THREADS) {
      float t = 0.f;
      for (int q = 0; q < nsplit; q++) t += cluster.map_shared_rank(s_part, q)[c];      // fixed order -> deterministic
      if (dwf_part) dwf_part[(int64_t)b * CHA + c] += t * att2[(int64_t)b * o1_stride + c];    // att2 term of d w_full (one owner per (b, c))
      datt2[(int64_t)b * dcat_stride + c] = t * wf[c];
      if (datt2_bf) datt2_bf[(int64_t)b * dcat_stride + c] = __float2bfloat16_rn(t * wf[c]);
    }
    cluster.sync();
    return;
  }
  float* part = partials + ((int64_t)b * nsplit + sp) * (CHA + 2);
  for (int c = threadIdx.x; c < CHA; c += AP_THREADS) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < AP_CWARPS; w++) t += s_acc[w * CHA + c];
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
  const float* pb = partials + (int64_t)b * nsplit * (CHA + 2);
  for (int c = threadIdx.x; c < CHA; c += AP_THREADS) {
    float t = 0.f;
    for (int sidx = 0; sidx < nsplit; sidx++) t += __ldcg(pb + (int64_t)sidx * (CHA + 2) + 2 + c);
    if (dwf_part) dwf_part[(int64_t)b * CHA + c] += t * att2[(int64_t)b * o1_stride + c];
    datt2[(int64_t)b * dcat_stride + c] = t * wf[c];
    if (datt2_bf) datt2_bf[(int64_t)b * dcat_stride + c] = __float2bfloat16_rn(t * wf[c]);
  }
}

// ------------------------------------------------------------------------------------------------------------------------------
// [r2b] Tensor-core backward for the 512-wide torch flavour (bf16): the two contractions of the step run on mma.sync instead of
// CUDA-core FMAs / predicated adds (2.5x fewer warp instructions).  Measured: the launch was NOT issue-bound — 17.35 vs 17.44 us
// (run 60); what it loses it loses at its ends (DESIGN.md section 4) — but the tensor-core version frees the issue slots and,
// with alpha / d reg staged in shared memory and the tail operands fetched up front, runs at 15.7 us:
//   d[r]     = sum_c enc[r][c] * dctx[c]          A = 16 enc rows straight from the ring (ldmatrix), B = dctx split into bf16 hi+lo
//                                                  (columns 0/1 of B, products exact, fp32 accumulation)
//   datt2[a] = sum_r bit[r][a] * de[r]            A = mask bits expanded to bf16 {0, 2.0} with ONE shift + ONE and per register,
//                                                  B = de split into bf16 hi+lo
// A stage is 16 region rows; all 8 consumer warps share it: warp w takes channels [64w, 64w+64) of the dot product (4 k-steps),
// the 16 partial sums per warp meet in shared memory behind one 256-thread named barrier, every warp then forms de for the 16
// rows (redundantly: 16 lanes) and runs the mask contraction for ITS 64 attention columns (4 blocks of 16).  ~110 warp
// instructions per warp and stage instead of ~260 per 2 rows.
// Ring rows are padded to 1040 B (one bulk copy per row) so that the 8 rows of an ldmatrix phase hit 8 different 16-byte bank
// groups.  Mask layout (written by the forward kernel): byte (r, a/8) lives at (r/2) * 2*(A/8) + (a/8)*2 + (r&1), i.e. the bytes
// of an even/odd row pair are adjacent: a lane's four A registers per 16 x 16 block are then shifts of ONE 32-bit word
// [even(q) | even(q+4) | odd(q) | odd(q+4)] (q = lane % 4: fragment k index = region row).  Fragment row m = g + 8h of block j
// stands for attention column 64w + 8g + 2j + h (g = lane / 4): any bijection works, this one makes a lane's 8 columns one byte.
// ------------------------------------------------------------------------------------------------------------------------------
constexpr int ABM_STAGES = 5;
constexpr int ABM_ROWS = 16;
constexpr int ABM_CH = 512;
constexpr int ABM_PITCH = ABM_CH * 2 + 16;                    // bytes per ring row
constexpr int ABM_ENC_BYTES = ABM_ROWS * ABM_PITCH;
constexpr int ABM_MSK_BYTES = ABM_ROWS * (ABM_CH / 8);
constexpr int ABM_STAGE_BYTES = ABM_ENC_BYTES + ABM_MSK_BYTES;
constexpr int ABM_SMEM = ABM_STAGES * ABM_STAGE_BYTES + 128 + 2 * AP_CWARPS * ABM_ROWS * 4;
static_assert(ABM_STAGE_BYTES % 128 == 0, "stage alignment");

__device__ __forceinline__ void att_ldsm_x4(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3, uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(saddr));
}
__device__ __forceinline__ void att_mma_16816(float* c, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// (x, y) -> packed bf16 pair of the high parts (sel 0) or of the residuals x - hi(x) (sel 1); low half = x
__device__ __forceinline__ uint32_t pack_split(float x, float y, int sel) {
  const bf16 hx = __float2bfloat16_rn(x), hy = __float2bfloat16_rn(y);
  __nv_bfloat162 r;
  if (sel == 0) {
    r.x = hx; r.y = hy;
  } else {
    r.x = __float2bfloat16_rn(x - __bfloat162float(hx));
    r.y = __float2bfloat16_rn(y - __bfloat162float(hy));
  }
  return *reinterpret_cast<uint32_t*>(&r);
}

template <bool CL>
__global__ void __launch_bounds__(AP_THREADS, 2) attention_bwd_mma_kernel(
    const uint8_t* __restrict__ mask, const bf16* __restrict__ enc, const float* __restrict__ gate, int64_t o1_stride,
    const float* __restrict__ wf, const float* __restrict__ alpha, int64_t alpha_stride, const float* __restrict__ ctx,
    const float* __restrict__ dgctx, int64_t dg_stride, const float* __restrict__ dreg, int64_t dreg_stride,
    const float* __restrict__ sreg, int64_t sreg_stride, float* __restrict__ de, float* __restrict__ datt2, float* __restrict__ dgp,
    int64_t dcat_stride, bf16* __restrict__ datt2_bf, bf16* __restrict__ dgp_bf, float* __restrict__ dctx_out, int R, int nsplit,
    int* __restrict__ counters, float* __restrict__ partials, int pol_enc, const float* __restrict__ att2,
    float* __restrict__ dwf_part) {
  constexpr int CH = ABM_CH, MB = CH / 8;
  extern __shared__ __align__(128) uint8_t ap_smem[];
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ap_smem + ABM_STAGES * ABM_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + ABM_STAGES;
  float* s_pd = reinterpret_cast<float*>(ap_smem + ABM_STAGES * ABM_STAGE_BYTES + 128);      // [2][8 warps][16 rows] partial dots
  __shared__ int s_last;
  const int b = blockIdx.y, sp = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int rps = att_rows_per_split(R, nsplit);                // even: a stage starts on an even/odd row pair
  const int r0 = sp * rps, r1 = min(R, r0 + rps);
  const int nst = r1 > r0 ? (r1 - r0 + ABM_ROWS - 1) / ABM_ROWS : 0;
  const int Rp = (R + 1) & ~1;
  ATT_TS(0, threadIdx.x == 0);
  const bf16* eb = enc + (int64_t)b * R * CH;
  const uint8_t* mb = mask + (int64_t)b * Rp * MB;
  if (threadIdx.x == 0) {
    for (int s = 0; s < ABM_STAGES; s++) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, AP_CWARPS);
    }
    fence_barrier_init();
  }
  __syncthreads();
  const int g = lane >> 2, q = lane & 3;
  // cluster mode: the full_att weight and the att2 value of the column this thread finalises after the combine are forward-pass
  // data -> fetched up front, off the tail
  const int cps_pf = (CH + nsplit - 1) / nsplit;
  const int c_pf = sp * cps_pf + (int)threadIdx.x;
  float wf_pf = 0.f, a2_pf = 0.f;
  if (CL && (int)threadIdx.x < cps_pf && c_pf < CH) {
    wf_pf = wf[c_pf];
    if (dwf_part) a2_pf = att2[(int64_t)b * o1_stride + c_pf];
  }
  float macc[4][4];
#pragma unroll
  for (int j = 0; j < 4; j++)
#pragma unroll
    for (int i = 0; i < 4; i++) macc[j][i] = 0.f;

  if (wid == AP_CWARPS) {
    // producer warp: enc and the mask bits of this step were written long before the preceding launch -> no griddepcontrol.wait
    const uint64_t pe = make_policy(pol_enc), pm = l2_policy_evict_first();
    for (int i = 0; i < nst; i++) {
      const int s = i % ABM_STAGES;
      const uint32_t ph = (i / ABM_STAGES) & 1;
      const int row = r0 + i * ABM_ROWS;
      const int rows = min(ABM_ROWS, r1 - row);
      const uint32_t bytes_m = (uint32_t)((rows + 1) >> 1) * 2u * MB;
      uint8_t* st = ap_smem + (size_t)s * ABM_STAGE_BYTES;
      if (lane == 0) {
        mbar_wait(empty_bar + s, ph ^ 1);
        mbar_expect_tx(full_bar + s, (uint32_t)rows * CH * 2u + bytes_m);
        ATT_TS(6, i == 0);
        ATT_TS(7, i == nst - 1);
      }
      __syncwarp();
      if (lane < rows) bulk_g2s(st + lane * ABM_PITCH, eb + (int64_t)(row + lane) * CH, CH * 2u, full_bar + s, pe);
      else if (lane == ABM_ROWS) bulk_g2s(st + ABM_ENC_BYTES, mb + (int64_t)(row >> 1) * 2 * MB, bytes_m, full_bar + s, pm);
    }
    __syncwarp();
    pdl_wait();
  } else {
    float sdot = 0.f;
    float gv[16], cxv[16];
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const int c0 = (j * 32 + lane) * 8;
      if (gate) ld8(gate + (int64_t)b * o1_stride + c0, gv + j * 8);
      ld8(ctx + (int64_t)b * CH + c0, cxv + j * 8);
    }
    // this lane's slice of the B operand of the dot product: k = 64*wid + 16*s + 2q + {0,1,8,9}; columns 0 / 1 = hi / lo parts
    float gq[4][4];
#pragma unroll
    for (int s = 0; s < 4; s++) {
      const int k0 = 64 * wid + 16 * s + 2 * q;
      if (gate && g < 2) {
        const float2 u = *reinterpret_cast<const float2*>(gate + (int64_t)b * o1_stride + k0);
        const float2 v = *reinterpret_cast<const float2*>(gate + (int64_t)b * o1_stride + k0 + 8);
        gq[s][0] = u.x; gq[s][1] = u.y; gq[s][2] = v.x; gq[s][3] = v.y;
      } else {
        gq[s][0] = gq[s][1] = gq[s][2] = gq[s][3] = 1.f;
      }
    }
    const float sreg_b = sreg ? sreg[(int64_t)b * sreg_stride] : 0.f;
    // alpha and the regulariser gradient of this CTA's rows are forward-pass results: ALL of them are staged in shared memory before
    // the wait.  (Fetching them stage by stage with a one-stage lookahead made every 16-row stage cost one L2 round trip, ~0.8 us: the
    // main loop then ran at 3.5 TB/s whatever the arithmetic was — run 62 timeline.)
    const float* alb = alpha + (int64_t)b * alpha_stride;
    float* deb = de + (int64_t)b * alpha_stride;
    const float* drb = dreg + (int64_t)b * dreg_stride;
    const int rr = lane & 15;
    float* s_al = s_pd + 2 * AP_CWARPS * ABM_ROWS;      // [rps] alpha | [rps] d reg
    float* s_dr = s_al + rps;
    for (int r = threadIdx.x; r < r1 - r0; r += AP_CWARPS * 32) {
      s_al[r] = alb[r0 + r];
      s_dr[r] = dreg ? drb[r0 + r] : 0.f;
    }
    pdl_wait();
    ATT_TS(1, threadIdx.x == 0);
    pdl_trigger();
    uint32_t bd[4][2];
#pragma unroll
    for (int s = 0; s < 4; s++) {
      bd[s][0] = bd[s][1] = 0u;
      if (g < 2) {
        const int k0 = 64 * wid + 16 * s + 2 * q;
        const float2 u = *reinterpret_cast<const float2*>(dgctx + (int64_t)b * dg_stride + k0);
        const float2 v = *reinterpret_cast<const float2*>(dgctx + (int64_t)b * dg_stride + k0 + 8);
        bd[s][0] = pack_split(u.x * gq[s][0], u.y * gq[s][1], g);
        bd[s][1] = pack_split(v.x * gq[s][2], v.y * gq[s][3], g);
      }
    }
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const int c0 = (j * 32 + lane) * 8;
      float dg[8], gp[8], dc[8];
      ld8(dgctx + (int64_t)b * dg_stride + c0, dg);
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const float gi = gate ? gv[j * 8 + i] : 1.f;
        dc[i] = dg[i] * gi;
        sdot = fmaf(dc[i], cxv[j * 8 + i], sdot);
        gp[i] = dg[i] * cxv[j * 8 + i] * gi * (1.f - gi);
      }
      if (sp == 0 && wid == 0) {
        if (dgp) st8(dgp + (int64_t)b * dcat_stride + c0, gp);
        if (dgp_bf) st8(dgp_bf + (int64_t)b * dcat_stride + c0, gp);
        if (dctx_out) st8(dctx_out + (int64_t)b * CH + c0, dc);
      }
    }
    const float sall = warp_sum(sdot) + sreg_b;
    ATT_TS(2, threadIdx.x == 0);
    const uint32_t ring = smem_u32(ap_smem);
    const uint32_t a_off = (uint32_t)((lane & 7) + ((lane >> 3) & 1) * 8) * ABM_PITCH + (uint32_t)(64 * wid + (lane >> 4) * 8) * 2u;
    const uint32_t m_off = ABM_ENC_BYTES + (uint32_t)q * 2u * MB + (uint32_t)(8 * wid + g) * 2u;
    asm volatile("bar.sync 1, 256;" ::: "memory");     // s_al / s_dr complete
    for (int i = 0; i < nst; i++) {
      const int s = i % ABM_STAGES;
      const uint32_t ph = (i / ABM_STAGES) & 1;
      const int row = r0 + i * ABM_ROWS;
      const int rows = min(ABM_ROWS, r1 - row);
      const float al = rr < rows ? s_al[i * ABM_ROWS + rr] : 0.f, dr = rr < rows ? s_dr[i * ABM_ROWS + rr] : 0.f;
      mbar_wait(full_bar + s, ph);
      ATT_TS(3, threadIdx.x == 0 && i == 0);
      const uint32_t sb = ring + (uint32_t)s * ABM_STAGE_BYTES;
      // ---- partial dot products of the 16 rows over this warp's 64 channels
      float d4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int k = 0; k < 4; k++) {
        uint32_t a0, a1, a2, a3;
        att_ldsm_x4(a0, a1, a2, a3, sb + a_off + k * 32);
        att_mma_16816(d4, a0, a1, a2, a3, bd[k][0], bd[k][1]);
      }
      // this lane's mask word (read now: the ring slot is released right after the barrier-independent part)
      const uint32_t u_lo = *reinterpret_cast<const uint16_t*>(ap_smem + (size_t)s * ABM_STAGE_BYTES + m_off);
      const uint32_t u_hi = *reinterpret_cast<const uint16_t*>(ap_smem + (size_t)s * ABM_STAGE_BYTES + m_off + 4 * 2 * MB);
      const uint32_t mw = __byte_perm(u_lo, u_hi, 0x5140);      // [even(q) | even(q+4) | odd(q) | odd(q+4)]
      float* pdw = s_pd + (i & 1) * (AP_CWARPS * ABM_ROWS);
      if (q == 0) {
        pdw[wid * ABM_ROWS + g] = d4[0] + d4[1];
        pdw[wid * ABM_ROWS + g + 8] = d4[2] + d4[3];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_bar + s);                 // every lane of this warp has read what it needs from the slot
      asm volatile("bar.sync 1, 256;" ::: "memory");
      float dsum = 0.f;
#pragma unroll
      for (int w = 0; w < AP_CWARPS; w++) dsum += pdw[w * ABM_ROWS + rr];
      const float dev = rr < rows ? al * (dsum + dr - sall) : 0.f;
      if (wid == (i & 7) && lane < rows) deb[row + lane] = dev;
      // ---- mask contraction: B = de of rows (2q, 2q+1, 2q+8, 2q+9), hi parts in column 0 (g == 0), residuals in column 1
      const float v0 = __shfl_sync(0xffffffffu, dev, 2 * q), v1 = __shfl_sync(0xffffffffu, dev, 2 * q + 1);
      const float v2 = __shfl_sync(0xffffffffu, dev, 2 * q + 8), v3 = __shfl_sync(0xffffffffu, dev, 2 * q + 9);
      uint32_t bm0 = 0u, bm1 = 0u;
      if (g < 2) {
        bm0 = pack_split(v0, v1, g);
        bm1 = pack_split(v2, v3, g);
      }
#pragma unroll
      for (int j = 0; j < 4; j++) {
        uint32_t af[4];
#pragma unroll
        for (int ii = 0; ii < 4; ii++) {
          // element e=0 (low half): bit 8*rs + 7 - (2j + h); e=1: 16 above.  -> bit 14 / 30 (bf16 2.0)
          const int h = ii & 1, rs = ii >> 1;
          const int sh = 14 - (8 * rs + 7 - (2 * j + h));
          af[ii] = (sh >= 0 ? (mw << sh) : (mw >> (-sh))) & 0x40004000u;
        }
        att_mma_16816(macc[j], af[0], af[1], af[2], af[3], bm0, bm1);
      }
    }
  }
  ATT_TS(4, threadIdx.x == 0);
  __syncthreads();
  ATT_TS(8, threadIdx.x == 0);
  float* s_part = reinterpret_cast<float*>(ap_smem);             // [CH] mask sums of this CTA (every column has ONE owner lane)
  if (wid < AP_CWARPS && q == 0) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
      s_part[64 * wid + 8 * g + 2 * j] = 0.5f * (macc[j][0] + macc[j][1]);
      s_part[64 * wid + 8 * g + 2 * j + 1] = 0.5f * (macc[j][2] + macc[j][3]);
    }
  }
  __syncthreads();
  if constexpr (CL) {
    cg::cluster_group cluster = cg::this_cluster();
    cluster.sync();
    const int cps = (CH + nsplit - 1) / nsplit;
    for (int c = sp * cps + threadIdx.x; c < min(CH, (sp + 1) * cps); c += AP_THREADS) {
      float t = 0.f;
      for (int qq = 0; qq < nsplit; qq++) t += cluster.map_shared_rank(s_part, qq)[c];      // fixed order -> deterministic
      const bool pf = c == c_pf;
      const float wfc = pf ? wf_pf : wf[c];
      if (dwf_part) dwf_part[(int64_t)b * CH + c] += t * (pf ? a2_pf : att2[(int64_t)b * o1_stride + c]);      // att2 term of d w_full (one owner per (b, c))
      datt2[(int64_t)b * dcat_stride + c] = t * wfc;
      if (datt2_bf) datt2_bf[(int64_t)b * dcat_stride + c] = __float2bfloat16_rn(t * wfc);
    }
    cluster.sync();
    ATT_TS(5, threadIdx.x == 0);
    return;
  }
  float* part = partials + ((int64_t)b * nsplit + sp) * (CH + 2);
  for (int c = threadIdx.x; c < CH; c += AP_THREADS) part[2 + c] = s_part[c];
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
  for (int c = threadIdx.x; c < CH; c += AP_THREADS) {
    float t = 0.f;
    for (int sidx = 0; sidx < nsplit; sidx++) t += __ldcg(pb + (int64_t)sidx * (CH + 2) + 2 + c);
    if (dwf_part) dwf_part[(int64_t)b * CH + c] += t * att2[(int64_t)b * o1_stride + c];
    datt2[(int64_t)b * dcat_stride + c] = t * wf[c];
    if (datt2_bf) datt2_bf[(int64_t)b * dcat_stride + c] = __float2bfloat16_rn(t * wf[c]);
  }
}

int att_pipe_splits(int B, int hint = 0) {
  if (g_opt_att_nsplit > 0) return g_opt_att_nsplit > AP_MAXSPLIT ? AP_MAXSPLIT : g_opt_att_nsplit;      // explicit option wins
  if (hint > 0) return hint > 8 ? 8 : hint;
  // two CTAs per SM are resident (smem): one full wave of <= 296 CTAs.  Measured at B=64, R=868 (bf16): 4 splits
  // (256 CTAs, 14 stages each) 25.9 us vs 9 splits (576 CTAs = 2 waves) 32.8 us — per-CTA start-up/combine
  // costs dominate short CTAs (profiles/r1_attention_nsplit_sweep.txt)
  int s = (148 * LO_ATT_MINB) / B;
  if (s < 1) s = 1;
  if (s > AP_MAXSPLIT) s = AP_MAXSPLIT;
  if (g_opt_att_cluster && s > 8) s = 8;       // portable cluster size limit
  return s;
}

// optional L2 access-policy window attached to every attention launch (lo_set_l2_window): as a LAUNCH attribute it is also
// recorded in CUDA-graph kernel nodes, which a stream attribute is not
static cudaAccessPolicyWindow g_att_window{};

static inline bool att_pdl_ok(int abi) { return !abi || g_opt_att_abi_pdl; }

// launch with (optional) cluster dimension {ns,1,1} and the PDL attribute.
// pdl = false (stand-alone C entry points): these kernels read operands BEFORE griddepcontrol.wait — loop-invariant inputs in the
// forward (att1, enc, full_att weight), forward-pass results in the backward (alpha, ctx, gate, att2, d reg).  Inside the decoder's
// time loops those are at least two launches old; a caller of the C ABI may have produced them with the launch enqueued just before,
// which would be allowed to overlap.  Without the attribute the launch is fully stream-ordered (the wait is a no-op).
template <typename... KArgs, typename... Args>
static cudaError_t launch_att(void (*kernel)(KArgs...), dim3 grid, size_t smem, int cluster_x, cudaStream_t st, bool pdl, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(AP_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[3];
  int n = 0;
  if (g_att_window.num_bytes) {
    attr[n].id = cudaLaunchAttributeAccessPolicyWindow;
    attr[n].val.accessPolicyWindow = g_att_window;
    n++;
  }
  if (g_opt_pdl && pdl) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    n++;
  }
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    n++;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

static inline bool use_cluster(int ns, int R) {
  // cluster mode keeps the raw scores of a CTA's rows in shared memory: ceil(R/ns) floats next to the ring
  return g_opt_att_cluster && ns >= 2 && ns <= 8 && ((R + ns - 1) / ns) * 4 <= 16 * 1024;
}

template <typename T, int NVA, int NVC, int ACT, bool MK>
static int fwd_launch_m(const AttFwdArgs& x, cudaStream_t st) {
  using C = ApCfg<T, NVA, NVC>;
  constexpr int SM_MAX = C::SMEM + 16 * 1024;
  static bool attr = false;
  if (!attr) {
    LO_CUDA(cudaFuncSetAttribute(attention_fwd_pipe_kernel<T, NVA, NVC, false, ACT, MK>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
    LO_CUDA(cudaFuncSetAttribute(attention_fwd_pipe_kernel<T, NVA, NVC, true, ACT, MK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_MAX));
    attr = true;
  }
  const int ns = att_pipe_splits(x.B, x.nsplit_hint);
  const int rpi = x.rows_per_img > 1 ? x.rows_per_img : 1;
  if (use_cluster(ns, x.R)) {
    const size_t smem = C::SMEM + (size_t)((x.R + ns - 1) / ns) * 4;
    LO_CUDA(launch_att(attention_fwd_pipe_kernel<T, NVA, NVC, true, ACT, MK>, dim3(ns, x.B), smem, ns, st, att_pdl_ok(x.abi), (const T*)x.att1, (const T*)x.enc,
                       x.att2, x.att2_stride, x.wf, x.alpha, x.alpha_stride, x.ctx, x.gate_pre, x.gate_stride, x.gctx, x.gctx_bf, x.R, ns,
                       (int*)x.work, (float*)((char*)x.work + 4096), g_opt_att_policy_enc, g_opt_att_policy_att1, rpi, x.mask_out));
  } else {
    LO_CUDA(launch_att(attention_fwd_pipe_kernel<T, NVA, NVC, false, ACT, MK>, dim3(ns, x.B), (size_t)C::SMEM, 1, st, att_pdl_ok(x.abi), (const T*)x.att1,
                       (const T*)x.enc, x.att2, x.att2_stride, x.wf, x.alpha, x.alpha_stride, x.ctx, x.gate_pre, x.gate_stride, x.gctx,
                       x.gctx_bf, x.R, ns, (int*)x.work, (float*)((char*)x.work + 4096), g_opt_att_policy_enc, g_opt_att_policy_att1, rpi,
                       x.mask_out));
  }
  LO_LAUNCH_OK();
  return LO_OK;
}

template <typename T, int NVA, int NVC, int ACT>
static int fwd_launch_a(const AttFwdArgs& x, cudaStream_t st) {
  if constexpr (ACT == 0) {
    if (x.mask_out) return fwd_launch_m<T, NVA, NVC, ACT, true>(x, st);        // training: also emit the ReLU mask bits
  }
  return fwd_launch_m<T, NVA, NVC, ACT, false>(x, st);
}

template <typename T, int NVA, int NVC>
static int fwd_launch(const AttFwdArgs& x, cudaStream_t st) {
  return x.act == 1 ? fwd_launch_a<T, NVA, NVC, 1>(x, st) : fwd_launch_a<T, NVA, NVC, 0>(x, st);
}

// C: enc channels; x.a_ch: att1 channels (0 = C).  Supported: A == C in {256, 512, 1024} and (A, C) = (256, 512)
template <typename T>
static int fwd_dispatch(const AttFwdArgs& x, int C, cudaStream_t st) {
  const int A = x.a_ch > 0 ? x.a_ch : C;
  if (A == 256 && C == 512) return fwd_launch<T, 1, 2>(x, st);
  if (A != C) return fail(LO_EINVAL, "%s: attention width pair (%ld, %ld) not instantiated", __func__, A, C);
  if (C == 256) return fwd_launch<T, 1, 1>(x, st);
  if (C == 512) return fwd_launch<T, 2, 2>(x, st);
  return fwd_launch<T, 4, 4>(x, st);
}
int attention_fwd_pipe(const AttFwdArgs& x, int dt, int C, cudaStream_t st) {
  return dt == LO_F32 ? fwd_dispatch<float>(x, C, st) : fwd_dispatch<bf16>(x, C, st);
}

template <typename T, int NVA, int NVC, int ACT>
static int bwd_launch_a(const AttBwdArgs& x, cudaStream_t st) {
  using C = ApCfg<T, NVA, NVC>;
  static bool attr = false;
  if (!attr) {
    LO_CUDA(cudaFuncSetAttribute(attention_bwd_pipe_kernel<T, NVA, NVC, false, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
    LO_CUDA(cudaFuncSetAttribute(attention_bwd_pipe_kernel<T, NVA, NVC, true, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
    attr = true;
  }
  const int ns = att_pipe_splits(x.B, x.nsplit_hint);
  if constexpr (ACT == 0 && sizeof(T) == 2 && NVA == 2 && NVC == 2)
  if (x.mask_in && g_opt_att_bwd_mma && att_rows_per_split(x.R, ns) <= 2048) {
    static bool attr_t = false;
    if (!attr_t) {
      LO_CUDA(cudaFuncSetAttribute(attention_bwd_mma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ABM_SMEM + 2048 * 8));
      LO_CUDA(cudaFuncSetAttribute(attention_bwd_mma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ABM_SMEM + 2048 * 8));
      attr_t = true;
    }
#define LO_BWDT_ARGS                                                                                                                  \
  x.mask_in, (const bf16*)x.enc, x.gate, x.o1_stride, x.wf, x.alpha, x.alpha_stride, x.ctx, x.dgctx, x.dg_stride, x.dreg,            \
      x.dreg_stride, x.sreg, x.sreg_stride, x.de, x.datt2, x.dgp, x.dcat_stride, x.datt2_bf, x.dgp_bf, x.dctx_out, x.R, ns,           \
      (int*)x.work, (float*)((char*)x.work + 4096), g_opt_att_policy_enc, x.att2, x.dwf_part
    const size_t smem_t = (size_t)ABM_SMEM + (size_t)att_rows_per_split(x.R, ns) * 8;      // + alpha / d reg of the CTA's rows
    if (use_cluster(ns, x.R)) {
      LO_CUDA(launch_att(attention_bwd_mma_kernel<true>, dim3(ns, x.B), smem_t, ns, st, att_pdl_ok(x.abi), LO_BWDT_ARGS));
    } else {
      LO_CUDA(launch_att(attention_bwd_mma_kernel<false>, dim3(ns, x.B), smem_t, 1, st, att_pdl_ok(x.abi), LO_BWDT_ARGS));
    }
#undef LO_BWDT_ARGS
    LO_LAUNCH_OK();
    return LO_OK;
  }
  if constexpr (ACT == 0) if (x.mask_in) {
    using CM = ApmCfg<T, NVA, NVC>;
    static bool attr_m = false;
    if (!attr_m) {
      LO_CUDA(cudaFuncSetAttribute(attention_bwd_mask_kernel<T, NVA, NVC, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CM::SMEM));
      LO_CUDA(cudaFuncSetAttribute(attention_bwd_mask_kernel<T, NVA, NVC, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CM::SMEM));
      attr_m = true;
    }
#define LO_BWDM_ARGS                                                                                                                  \
  x.mask_in, (const T*)x.enc, x.gate, x.o1_stride, x.wf, x.alpha, x.alpha_stride, x.ctx, x.dgctx, x.dg_stride, x.dreg, x.dreg_stride, \
      x.sreg, x.sreg_stride, x.de, x.datt2, x.dgp, x.dcat_stride, x.datt2_bf, x.dgp_bf, x.dctx_out, x.R, ns, (int*)x.work,           \
      (float*)((char*)x.work + 4096), g_opt_att_policy_enc, x.att2, x.dwf_part
    if (use_cluster(ns, x.R)) {
      LO_CUDA(launch_att(attention_bwd_mask_kernel<T, NVA, NVC, true>, dim3(ns, x.B), (size_t)CM::SMEM, ns, st, att_pdl_ok(x.abi), LO_BWDM_ARGS));
    } else {
      LO_CUDA(launch_att(attention_bwd_mask_kernel<T, NVA, NVC, false>, dim3(ns, x.B), (size_t)CM::SMEM, 1, st, att_pdl_ok(x.abi), LO_BWDM_ARGS));
    }
#undef LO_BWDM_ARGS
    LO_LAUNCH_OK();
    return LO_OK;
  }
#define LO_BWD_ARGS                                                                                                              \
  (const T*)x.att1, (const T*)x.enc, x.att2, x.gate, x.o1_stride, x.wf, x.alpha, x.alpha_stride, x.ctx, x.dgctx, x.dg_stride, x.dreg, \
      x.dreg_stride, x.sreg, x.sreg_stride, x.de, x.datt2, x.dgp, x.dcat_stride, x.datt2_bf, x.dgp_bf, x.dctx_out, x.R, ns,       \
      (int*)x.work, (float*)((char*)x.work + 4096), g_opt_att_policy_enc, g_opt_att_policy_att1, x.dwf_part
  if (use_cluster(ns, x.R)) {
    LO_CUDA(launch_att(attention_bwd_pipe_kernel<T, NVA, NVC, true, ACT>, dim3(ns, x.B), (size_t)C::SMEM, ns, st, att_pdl_ok(x.abi), LO_BWD_ARGS));
  } else {
    LO_CUDA(launch_att(attention_bwd_pipe_kernel<T, NVA, NVC, false, ACT>, dim3(ns, x.B), (size_t)C::SMEM, 1, st, att_pdl_ok(x.abi), LO_BWD_ARGS));
  }
#undef LO_BWD_ARGS
  LO_LAUNCH_OK();
  return LO_OK;
}

template <typename T, int NVA, int NVC>
static int bwd_launch(const AttBwdArgs& x, cudaStream_t st) {
  return x.act == 1 ? bwd_launch_a<T, NVA, NVC, 1>(x, st) : bwd_launch_a<T, NVA, NVC, 0>(x, st);
}

template <typename T>
static int bwd_dispatch(const AttBwdArgs& x, int C, cudaStream_t st) {
  const int A = x.a_ch > 0 ? x.a_ch : C;
  if (A == 256 && C == 512) return bwd_launch<T, 1, 2>(x, st);
  if (A != C) return fail(LO_EINVAL, "%s: attention width pair (%ld, %ld) not instantiated", __func__, A, C);
  if (C == 256) return bwd_launch<T, 1, 1>(x, st);
  if (C == 512) return bwd_launch<T, 2, 2>(x, st);
  return bwd_launch<T, 4, 4>(x, st);
}
int attention_bwd_pipe(const AttBwdArgs& x, int dt, int C, cudaStream_t st) {
  return dt == LO_F32 ? bwd_dispatch<float>(x, C, st) : bwd_dispatch<bf16>(x, C, st);
}

}  // namespace lo

namespace lo { extern long long* g_tc_dbg; }
extern "C" int lo_debug_buffer(void* p) {
  lo::g_tc_dbg = (long long*)p;
  LO_TRY(lo::cl_set_ts((long long*)p));
  LO_TRY(lo::sk_set_ts((long long*)p));
#ifdef LO_ATT_TIMING
  long long* q = (long long*)p;
  LO_CUDA(cudaMemcpyToSymbol(lo::g_att_ts, &q, sizeof(q)));
#endif
  return LO_OK;
}

// L2 persistence experiment: access-policy window of `stream` over [base, base+bytes) (hit -> persisting, miss -> streaming) and
// the persisting carve-out sized to fit; bytes = 0 resets both.  Attention loads honour it with att_policy_* = 3 (no cache hint).
extern "C" int lo_set_l2_window(const void* base, int64_t bytes, float hit_ratio, void* stream) {
  int dev = 0, max_persist = 0, max_window = 0;
  LO_CUDA(cudaGetDevice(&dev));
  LO_CUDA(cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev));
  LO_CUDA(cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, dev));
  cudaStreamAttrValue v{};
  if (bytes <= 0 || !base) {
    v.accessPolicyWindow.num_bytes = 0;
    lo::g_att_window = v.accessPolicyWindow;
    LO_CUDA(cudaStreamSetAttribute((cudaStream_t)stream, cudaStreamAttributeAccessPolicyWindow, &v));
    LO_CUDA(cudaCtxResetPersistingL2Cache());
    return LO_OK;
  }
  const size_t carve = (size_t)(bytes < max_persist ? bytes : max_persist);
  LO_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve));
  v.accessPolicyWindow.base_ptr = const_cast<void*>(base);
  v.accessPolicyWindow.num_bytes = (size_t)(bytes < max_window ? bytes : max_window);
  v.accessPolicyWindow.hitRatio = hit_ratio;
  v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  lo::g_att_window = v.accessPolicyWindow;
  LO_CUDA(cudaStreamSetAttribute((cudaStream_t)stream, cudaStreamAttributeAccessPolicyWindow, &v));
  lo::fail(LO_OK, "l2 window%s: carve %ld B (device max %ld B)", "", (long)carve, (long)max_persist);      // readable via lo_last_error()
  return LO_OK;
}

extern "C" int lo_get_option(const char* name) {
  if (!name) return -1;
  if (!strcmp(name, "att_pipe")) return lo::g_opt_att_pipe;
  if (!strcmp(name, "att_maskbits")) return lo::g_opt_att_maskbits;
  if (!strcmp(name, "att_bwd_mma")) return lo::g_opt_att_bwd_mma;
  if (!strcmp(name, "att_abi_pdl")) return lo::g_opt_att_abi_pdl;
  if (!strcmp(name, "dbg_skip")) return lo::g_opt_dbg_skip;
  if (!strcmp(name, "conv_mc")) return lo::g_opt_conv_mc;
  if (!strcmp(name, "att_cluster")) return lo::g_opt_att_cluster;
  if (!strcmp(name, "att_nsplit")) return lo::g_opt_att_nsplit;
  if (!strcmp(name, "pdl")) return lo::g_opt_pdl;
  if (!strcmp(name, "conv_persist")) return lo::g_opt_conv_persist;
  if (!strcmp(name, "wgrad256")) return lo::g_opt_wgrad256;
  if (!strcmp(name, "conv_mt2")) return lo::g_opt_conv_mt2;
  if (!strcmp(name, "dec_fuse")) return lo::g_opt_dec_fuse;
  if (!strcmp(name, "dec_cl")) return lo::g_opt_dec_cl;
  if (!strcmp(name, "dec_cl_bwd")) return lo::g_opt_dec_cl_bwd;
  if (!strcmp(name, "dec_fuse_bwd")) return lo::g_opt_dec_fuse_bwd;
  if (!strcmp(name, "fuse_lstm")) return lo::g_opt_fuse_lstm;
  if (!strcmp(name, "skinny_mma")) return lo::g_opt_skinny_mma;
  if (!strcmp(name, "skinny_tma")) return lo::g_opt_skinny_tma;
  if (!strcmp(name, "dec_streams")) return lo::g_opt_dec_streams;
  return -1;
}

extern "C" int lo_set_option(const char* name, int value) {
  if (!name) return LO_EINVAL;
  if (!strcmp(name, "att_pipe")) lo::g_opt_att_pipe = value;
  else if (!strcmp(name, "att_policy_enc")) lo::g_opt_att_policy_enc = value;
  else if (!strcmp(name, "att_policy_att1")) lo::g_opt_att_policy_att1 = value;
  else if (!strcmp(name, "att_nsplit")) lo::g_opt_att_nsplit = value;
  else if (!strcmp(name, "pdl")) lo::g_opt_pdl = value;
  else if (!strcmp(name, "att_cluster")) lo::g_opt_att_cluster = value;
  else if (!strcmp(name, "att_maskbits")) lo::g_opt_att_maskbits = value;
  else if (!strcmp(name, "att_bwd_mma")) lo::g_opt_att_bwd_mma = value;
  else if (!strcmp(name, "att_abi_pdl")) lo::g_opt_att_abi_pdl = value;
  else if (!strcmp(name, "dbg_skip")) lo::g_opt_dbg_skip = value;
  else if (!strcmp(name, "conv_mc")) lo::g_opt_conv_mc = value;
  else if (!strcmp(name, "conv_persist")) lo::g_opt_conv_persist = value;
  else if (!strcmp(name, "wgrad256")) lo::g_opt_wgrad256 = value;
  else if (!strcmp(name, "conv_mt2")) lo::g_opt_conv_mt2 = value;
  else if (!strcmp(name, "dec_streams")) { lo::g_opt_dec_streams = value; lo::g_opt_skinny8 = value >= 2 ? 0 : 1; }
  else if (!strcmp(name, "skinny8")) lo::g_opt_skinny8 = value;
  else if (!strcmp(name, "fuse_lstm")) lo::g_opt_fuse_lstm = value;
  else if (!strcmp(name, "dec_fuse")) lo::g_opt_dec_fuse = value;
  else if (!strcmp(name, "dec_cl")) lo::g_opt_dec_cl = value;
  else if (!strcmp(name, "dec_cl_bwd")) lo::g_opt_dec_cl_bwd = value;
  else if (!strcmp(name, "dec_fuse_bwd")) lo::g_opt_dec_fuse_bwd = value;
  else if (!strcmp(name, "skinny_mma")) lo::g_opt_skinny_mma = value;
  else if (!strcmp(name, "skinny_tma")) lo::g_opt_skinny_tma = value;
  else if (!strcmp(name, "l2_persist_mb")) {
    // size of the L2 set-aside that evict_last / persisting accesses may occupy (0 = driver default)
    cudaError_t e = cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)value << 20);
    if (e != cudaSuccess) return lo::fail(LO_ECUDA, "lo_set_option(l2_persist_mb): %s (%ld)", cudaGetErrorString(e), (long)e);
  }
  else return lo::fail(LO_EINVAL, "lo_set_option: unknown option %s", name);
  return LO_OK;
}
