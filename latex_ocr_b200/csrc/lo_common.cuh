// Shared device/host helpers for the latex_ocr_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/latex_ocr_b200.h"

typedef __nv_bfloat16 bf16;

namespace lo {

// ---- error plumbing ---------------------------------------------------------------------------
extern char g_err[512];
extern int64_t g_launches;

inline int fail(int code, const char* fmt, const char* a = "", long b = 0, long c = 0) {
  snprintf(g_err, sizeof(g_err), fmt, a, b, c);
  return code;
}

#define LO_CHECK_ARG(cond, what)                                                        \
  do {                                                                                  \
    if (!(cond)) return lo::fail(LO_EINVAL, "%s: invalid argument: " what " (line %ld)", __func__, __LINE__); \
  } while (0)

#define LO_CUDA(call)                                                                   \
  do {                                                                                  \
    cudaError_t e__ = (call);                                                           \
    if (e__ != cudaSuccess)                                                             \
      return lo::fail(LO_ECUDA, "%s: CUDA error %ld at line %ld", cudaGetErrorString(e__), (long)e__, __LINE__); \
  } while (0)

// call after every <<<>>> launch
#define LO_LAUNCH_OK()                                                                  \
  do {                                                                                  \
    lo::g_launches++;                                                                   \
    cudaError_t e__ = cudaGetLastError();                                               \
    if (e__ != cudaSuccess)                                                             \
      return lo::fail(LO_ECUDA, "%s: launch failed (%ld) at line %ld", cudaGetErrorString(e__), (long)e__, __LINE__); \
  } while (0)

#define LO_TRY(call)                                                                    \
  do {                                                                                  \
    int r__ = (call);                                                                   \
    if (r__ != LO_OK) return r__;                                                       \
  } while (0)

inline int cdiv(long a, long b) { return (int)((a + b - 1) / b); }

// kernel launch with (optionally) the programmatic-dependent-launch attribute; kernels launched this way call
// pdl_wait() before touching global memory
extern int g_opt_pdl;
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_opt_pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- dtype helpers ----------------------------------------------------------------------------
__device__ __forceinline__ float ldf(const float* p) { return *p; }
__device__ __forceinline__ float ldf(const bf16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void stf(float* p, float v) { *p = v; }
__device__ __forceinline__ void stf(bf16* p, float v) { *p = __float2bfloat16_rn(v); }
// value as it will be read back after a store to T (used so fwd masks == bwd masks)
__device__ __forceinline__ float roundto(float v, const float*) { return v; }
__device__ __forceinline__ float roundto(float v, const bf16*) { return __bfloat162float(__float2bfloat16_rn(v)); }

// 8 consecutive elements -> 8 floats (16-byte aligned for bf16, 32-byte for float)
__device__ __forceinline__ void ld8(const float* p, float* v) {
  float4 a = *reinterpret_cast<const float4*>(p);
  float4 b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void ld8(const bf16* p, float* v) {
  uint4 u = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; i++) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
// the same from SHARED memory through a 32-bit shared-window address (ld.shared: no generic-address translation, 32-bit
// address arithmetic)
__device__ __forceinline__ void lds8(uint32_t saddr, float* v, const float*) {
  float4 a, b;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w) : "r"(saddr));
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(saddr + 16));
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void lds8(uint32_t saddr, float* v, const bf16*) {
  uint32_t w[4];
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]) : "r"(saddr));
#pragma unroll
  for (int i = 0; i < 4; i++) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ void st8(float* p, const float* v) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void st8(bf16* p, const float* v) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&h);
  }
  *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// Philox4x32-10 (Salmon et al., SC'11), counter-based: the same (key, counter) gives the same 4 words in the forward and the
// backward kernel, so dropout masks are regenerated instead of stored.  Host mirror: latex_ocr_b200/philox.py.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}
// uniform in [0, 1) with 24 bits
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }
// inverted-dropout multiplier of element (row b, step t, unit j): state = {seed, call counter} in device memory
__device__ __forceinline__ float philox_dropout_mult(const unsigned long long* state, int b, int t, int j, float p, float scale) {
  const unsigned long long seed = state[0], call = state[1];
  const uint4 r = philox4x32_10(make_uint4((uint32_t)(j >> 2), (uint32_t)t, (uint32_t)b, (uint32_t)call),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const uint32_t w = (j & 3) == 0 ? r.x : ((j & 3) == 1 ? r.y : ((j & 3) == 2 ? r.z : r.w));
  return u01(w) >= p ? scale : 0.f;
}

// host-side dtype dispatch: calls f(T*) with T = float or bf16
#define LO_DISPATCH_DT(dt, T, ...)                   \
  do {                                               \
    if ((dt) == LO_F32) { typedef float T; __VA_ARGS__; } \
    else if ((dt) == LO_BF16) { typedef bf16 T; __VA_ARGS__; } \
    else return lo::fail(LO_EINVAL, "%s: bad dtype %ld", __func__, (long)(dt)); \
  } while (0)

// ---- internal launchers shared between translation units ---------------------------------------
struct GemmDesc {
  int M, N, K;
  int64_t sam, sak, sbk, sbn, ldc;
  int batch;
  int64_t sA, sB, sC;
  const float* bias;
  int accumulate, relu;
};
int gemm(const void* A, int dtA, const void* B, int dtB, void* C, int dtC, const GemmDesc& d, int impl, cudaStream_t st);
// C[M][N] (+)= A[M][K] * W[N][K]^T + bias  (row-major, K contiguous)
int gemm_nt(const void* A, int dtA, int64_t lda, const void* W, int dtW, int64_t ldw, void* C, int dtC, int64_t ldc,
            int M, int N, int K, const float* bias, int accumulate, int relu, int impl, cudaStream_t st);
// C[M][N] (+)= A[K][M]^T * B[K][N]   (weight gradients)
int gemm_tn(const void* A, int dtA, int64_t lda, const void* B, int dtB, int64_t ldb, void* C, int dtC, int64_t ldc,
            int M, int N, int K, int accumulate, int impl, cudaStream_t st);
// C[M][N] (+)= A[M][K] * B[K][N]
int gemm_nn(const void* A, int dtA, int64_t lda, const void* B, int dtB, int64_t ldb, void* C, int dtC, int64_t ldc,
            int M, int N, int K, int accumulate, int impl, cudaStream_t st);
int colsum(const void* X, int dt, float* out, int M, int N, int64_t ld, int accumulate, cudaStream_t st);

// attention step kernels, TMA-pipelined version (lo_attention.cu)
struct AttFwdArgs {
  const void *att1, *enc;
  const float* att2; int64_t att2_stride;
  const float* wf;
  float* alpha; int64_t alpha_stride;
  float* ctx; float* gate_pre; int64_t gate_stride; float* gctx; bf16* gctx_bf;
  int B, R;
  void* work;
  int rows_per_img;
  int nsplit_hint;
  int act;             // 0 ReLU score (torch flavour), 1 tanh (Genthial cell)
  int a_ch;            // channels of att1 / att2 / wf (0 = same as enc)
  uint8_t* mask_out;   // optional (ReLU score only): [B][R][A/8] bits (att1 + att2 > 0) of this step, for the backward
  int abi = 0;         // 1: called through a stand-alone C entry point -> launched WITHOUT programmatic dependent launch (see launch_att)
};
struct AttBwdArgs {
  const void *att1, *enc;
  const float *att2, *gate; int64_t o1_stride;
  const float* wf; const float* alpha; int64_t alpha_stride;
  const float* ctx; const float* dgctx; int64_t dg_stride;
  const float* dreg; int64_t dreg_stride; const float* sreg; int64_t sreg_stride;
  float* de; float* datt2; float* dgp; int64_t dcat_stride; bf16* datt2_bf; bf16* dgp_bf; float* dctx_out;
  int B, R;
  void* work;
  float* dwf_part;     // [B][A] running sum over the time loop of the full_att.weight gradient contributions (optional)
  int nsplit_hint;
  int act;
  int a_ch;
  const uint8_t* mask_in;   // optional (ReLU score only): the forward's mask bits; the kernel then streams enc + 1 bit per att1
                            // element instead of enc + att1 (dwf_part then receives only the att2 term of d w_full; the att1 term
                            // comes from the post-loop sweep)
  int abi = 0;         // as in AttFwdArgs
};
extern int g_opt_att_pipe;
extern int g_opt_att_maskbits;
extern int g_opt_dbg_skip;
extern int g_opt_conv_mc;
extern int g_opt_conv_persist;
extern int g_opt_wgrad256;
extern int g_opt_conv_mt2;
extern int g_opt_dec_streams;
extern int g_opt_skinny8;
int attention_fwd_pipe(const AttFwdArgs& x, int dt, int C, cudaStream_t st);
int attention_bwd_pipe(const AttBwdArgs& x, int dt, int C, cudaStream_t st);

// tcgen05 paths (lo_tc.cu)
bool tc_available();
int tc_gemm_nt(const bf16* A, int64_t lda, const bf16* W, int64_t ldw, void* C, int dtC, int64_t ldc,
               int M, int N, int K, const float* bias, int accumulate, int relu, cudaStream_t st);
int tc_gemm_nt_ex(const bf16* A, int64_t lda, const bf16* W, int64_t ldw, void* C, int dtC, int64_t ldc, int M, int N, int K,
                  const float* bias, int accumulate, int relu, int splits, int atomic_acc, int small_n_tile, cudaStream_t st);
struct TcLstmEpi {
  const float* ptab; const int64_t* tok; int64_t tok_stride;
  const float* hh; int64_t hh_stride;
  const float* c_prev; float* gates; float* c_out; float* h_out; bf16* h_bf;
  float* hd; int64_t hd_stride; const float* dmask;
  int D, V;
  // in-kernel dropout (has_dropout = 2): Philox state, drop probability, first batch row of this launch, step index
  const unsigned long long* dstate; float dp; int row0, t_idx;
};
// fused decoder forward step (lo_skinny.cu): [gates GEMM + LSTM cell] -> grid barrier -> [projection of h_{t+1} for step t+1]
struct DecStepFwd {
  const bf16* gctx; int64_t ld_gctx;       // A of phase 1: gate * context of step t, [M][K]
  const bf16* wil; int64_t ld_wil;         // gate-interleaved context half of weight_ih [4D][K]
  TcLstmEpi e;                             // LSTM epilogue (writes h_{t+1} fp32 + bf16 mirror, c, gates, hd)
  const bf16* wcat; int64_t ld_wcat;       // [N2][D] = [decoder_att; f_beta; weight_hh]
  const float* bcat; float* o1_next; int64_t ld_o1; int N2;   // phase 2 output (NULL: last step, phase 2 skipped)
  unsigned int* bar; unsigned int bar_target;                 // monotonic arrival counter of the grid barrier
  int M, K;
};
int dec_step_fwd(const DecStepFwd& p, cudaStream_t st);
// fused decoder backward step (lo_skinny.cu), launched after the attention backward of step t:
//   phase A: dh_{t-1} += [datt2 | dgate_pre]_t [W_d ; W_beta]          (K = A+C, two K slices, fp32 atomics)
//   grid barrier ; phase B: LSTM-cell backward of step t-1 (pointwise, spread over the whole grid) ; grid barrier
//   phase C: [dgctx | dh]_{t-1} = dG_{t-1} [W_ih[:, E:] | W_hh]          (K = 4D, four K slices, fp32 atomics)
struct DecStepBwd {
  // phase A (skipped when dcat_a == NULL: first launch of the loop)
  const bf16* dcat_a; int64_t ld_dcat;      // [Ma][A+C] bf16 mirror of datt2 | dgate_pre of step t
  const bf16* wbwd2; int64_t ld_w2; int K2; // [D][A+C]
  int Ma;
  // phase B/C (skipped when gates == NULL: last launch of the loop)
  const float* dhd; int64_t dhd_stride; const float* dmask; const unsigned long long* dstate; float dp; int t_idx;
  float* dc; const float* gates; const float* c_prev; const float* c_cur;
  float* dG; bf16* dG_bf; int64_t dG_stride;      // d pre-activations of step t-1 (fp32 + bf16 mirror), row stride O1
  const bf16* wbwd1; int64_t ld_w1; int K1;       // [C+D][4D]
  int Mb;
  float* dxh; int C, D;                            // [B][C+D]: dgctx | dh (accumulated with atomics, cleared in phase B)
  unsigned int* bar; unsigned int bar_target;      // target of the FIRST barrier of this launch (the second is + gridDim.x)
};
int dec_step_bwd(const DecStepBwd& p, cudaStream_t st);
extern int g_opt_dec_fuse_bwd;
extern int g_opt_dec_fuse;
// cluster-fused step kernels (lo_cluster.cu): the same DecStepFwd / DecStepBwd contracts, rows split into blocks of 16 (one 16-CTA cluster
// each), no grid barrier (bar / bar_target unused), dxh written instead of accumulated
extern int g_opt_dec_cl, g_opt_dec_cl_bwd;
bool dec_cl_fwd_ok(int D, int C, int N2);
bool dec_cl_bwd_ok(int D, int C, int A);
int dec_cl_fwd(const DecStepFwd& p, cudaStream_t st);
int dec_cl_bwd(const DecStepBwd& p, cudaStream_t st);
int cl_set_ts(long long* p);      // timing build only
int sk_set_ts(long long* p);      // timing build only
int tc_gemm_nt_lstm(const bf16* A, int64_t lda, const bf16* Wil, int64_t ldw, int M, int D, int K, const TcLstmEpi& e, cudaStream_t st);
extern int g_opt_fuse_lstm;
extern int g_opt_skinny_mma;
extern int g_opt_skinny_tma;
int skinny_gemm_nt_lstm(const bf16* A, int64_t lda, const bf16* Wil, int64_t ldw, int M, int D, int K, const TcLstmEpi& e, cudaStream_t st);
int skinny_gemm_nt(const bf16* A, int64_t lda, const bf16* W, int64_t ldw, float* C, int64_t ldc, int M, int N, int K, const float* bias,
                   int splits, int atomic_acc, cudaStream_t st);
int tc_gemm_tn(const bf16* A, int64_t lda, const bf16* B, int64_t ldb, float* C, int64_t ldc, int M, int N, int K, cudaStream_t st);
int tc_gemm_tn_batched(const bf16* A, int64_t sAk, int64_t sAb, const bf16* B, int64_t sBk, int64_t sBb, float* C, int64_t ldc,
                       int64_t sCb, int M, int N, int K, int batch, cudaStream_t st);
int tc_conv3x3_wgrad(const bf16* x, const bf16* dy, float* dw, int N, int H, int W, int Cin, int Cout, int pad, cudaStream_t st);
int tc_conv3x3(const bf16* x, const bf16* w, const float* bias, const bf16* mask, bf16* y,
               int N, int H, int W, int Cin, int Cout, int pad, int relu, cudaStream_t st);

}  // namespace lo
