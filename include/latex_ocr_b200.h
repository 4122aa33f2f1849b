/*
 * latex_ocr_b200 — C ABI of the B200-native (sm_100a) im2latex hot path.
 *
 * The reference (LinXueyuanStdio/LaTeX_OCR) has no FFI: its boundary is the Python class surface
 * (SURVEY.md §8-b).  Each entry point below replaces the library call(s) the reference makes at the
 * cited lines; the Python mirror in latex_ocr_b200/ (EncoderCNN, Attention, DecoderWithAttention,
 * Img2SeqModel) reaches them through ctypes.  Conventions:
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - stream-ordered on `stream` (a cudaStream_t passed as void*); no allocation, no synchronisation,
 *     no host-visible global state -> every call is CUDA-graph capturable;
 *   - programmatic dependent launch: most kernels are launched so that they may become resident while the preceding
 *     launch of the stream drains, and read their PARAMETER operands (weights, biases, projection tables — never
 *     activations) before they wait for it.  A parameter must therefore not be produced by the launch enqueued
 *     immediately before the call that consumes it (an optimiser step followed by anything else is fine: every
 *     entry point enqueues more than one launch or waits first).  The stand-alone attention entry points
 *     (lo_attention_forward / _forward_mask / _backward), whose early reads include activations (att1, enc; alpha,
 *     ctx, gate of the forward pass), are launched WITHOUT that overlap unless lo_set_option("att_abi_pdl", 1) says the
 *     caller guarantees those tensors are older than the preceding launch; lo_set_option("pdl", 0) turns the overlap
 *     off everywhere;
 *   - return 0 on success, negative LO_E* otherwise (never throws); lo_last_error() gives the text;
 *   - dtype arguments are LO_F32 or LO_BF16 and name the STORAGE type of the "big" tensors
 *     (feature maps, conv/linear weight shadows, encoder_out, att1).  Small per-step state is fp32.
 *     Accumulation is always fp32.
 */
#ifndef LATEX_OCR_B200_H
#define LATEX_OCR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LO_F32 0
#define LO_BF16 1

#define LO_OK 0
#define LO_EINVAL (-1)   /* bad argument / unsupported shape */
#define LO_ECUDA (-2)    /* a CUDA runtime call or launch failed */
#define LO_ENOTSUP (-3)  /* path not available on this device (needs sm_100) */

#define LO_IMPL_SIMT 0   /* CUDA-core kernels (fp32 or bf16 storage) — the tight-parity path */
#define LO_IMPL_TC 1     /* tcgen05 + TMA kernels (bf16 storage only) */

int lo_version(void);
const char* lo_last_error(void);
/* number of kernels launched through this library since load (bench.py's gpu_launches) */
int64_t lo_launch_count(void);
/* tuning knobs: "att_pipe" (1: TMA-pipelined attention kernels, 0: register-streaming), "att_policy_enc" /
 * "att_policy_att1" (L2 policy 0 normal, 1 evict_last, 2 evict_first), "att_nsplit" (0 = automatic), "pdl", "att_abi_pdl" (above);
 * schedule variants, each parity-tested against the default (tests/test_gpu_tc.py, DESIGN.md §8): "att_maskbits", "att_bwd_mma",
 * "skinny_mma", "skinny_tma", "fuse_lstm", "dec_streams", "dec_fuse", "dec_fuse_bwd", "dec_cl", "dec_cl_bwd", "conv_persist",
 * "conv_mt2", "conv_mc", "wgrad256"; "dbg_skip" is a timing-dissection aid (results are garbage).  LO_OPTS=name=value,... in the
 * environment sets them at load time (Python side). */
int lo_set_option(const char* name, int value);
/* current value of a tuning knob (-1: unknown name) */
int lo_get_option(const char* name);
/* L2 persistence: access-policy window of `stream` over [base, base+bytes) (hits persist, misses stream) with the
 * persisting carve-out sized to fit; bytes = 0 resets.  The attention kernels honour it with att_policy_enc/att1 = 3
 * (bulk copies without an explicit cache hint). */
int lo_set_l2_window(const void* base, int64_t bytes, float hit_ratio, void* stream);
/* development aid: device buffer (>= 16 int64) that CTA (0,0,0) of the tcgen05 NT GEMM stamps with clock64 at its
 * pipeline milestones; NULL disables */
int lo_debug_buffer(void* p);
/* 1 if the tcgen05/TMA kernels are built in and the current device is sm_100 */
int lo_tc_available(void);

/* ------------------------------------------------------------------------------------------------
 * Generic strided (batched) GEMM:  C[b][m][n] (+)= sum_k A[b][m*sam + k*sak] * B[b][k*sbk + n*sbn] (+ bias[n]) (ReLU)
 * Replaces nn.Linear / torch.mm call sites: seq2seq_torch.py:172-176, :223-227 and their autograd.
 * dtA/dtB/dtC in {LO_F32, LO_BF16}; supported combos: (f,f,f) (f,bf,f) (bf,bf,bf) (bf,bf,f).
 * impl=LO_IMPL_TC requires bf16 A and B, sak==1, sbk==1 (both K-major), K%64==0, 16B-aligned rows.
 */
int lo_gemm(const void* A, int dtA, const void* B, int dtB, void* C, int dtC,
            int M, int N, int K,
            int64_t sam, int64_t sak, int64_t sbk, int64_t sbn, int64_t ldc,
            int batch, int64_t sA, int64_t sB, int64_t sC,
            const float* bias, int accumulate, int relu, int impl, void* stream);

/* column sums: out[n] (+)= sum_m X[m*ld + n]  (bias gradients) ; X fp32 or bf16 */
int lo_colsum(const void* X, int dt, float* out, int M, int N, int64_t ld, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Encoder.  Feature maps are NHWC; conv weights are [Cout][3][3][Cin] ("KRSC", K-major for the
 * implicit GEMM); replaces nn.Conv2d/nn.ReLU/nn.MaxPool2d at seq2seq_torch.py:35-56 and
 * convolution_backward (autograd of img2seq_torch.py:165).
 */
/* conv1 (Cin=1) + bias + ReLU + 2x2/2 max-pool fused; img fp32 [N][H][W] raw 0..255
 * (img2seq_torch.py:115-117); out [N][H/2][W/2][64] */
int lo_conv1_pool_forward(const float* img, const float* w, const float* bias, void* out, int dt,
                          int N, int H, int W, void* stream);
/* same with the image as uint8 pixels [N][H][W] (what pad_batch_images produces, model/utils/image.py:27-64): 4x less
 * host->device traffic; pixel values 0..255 are exact in fp32, so results are identical */
int lo_conv1_pool_forward_u8(const uint8_t* img, const float* w, const float* bias, void* out, int dt,
                             int N, int H, int W, void* stream);
int lo_conv1_pool_wgrad_u8(const uint8_t* img, const float* w, const float* bias, const void* dpool, int dt,
                           float* dw, float* db, int N, int H, int W, void* stream);
/* conv1 weight/bias gradient from the POOLED output gradient; recomputes conv1 to find the
 * ReLU mask and pool argmax (first maximum in window scan order, as PyTorch) */
int lo_conv1_pool_wgrad(const float* img, const float* w, const float* bias, const void* dpool, int dt,
                        float* dw, float* db, int N, int H, int W, void* stream);
/* the same two kernels with the pixel normalisation x' = x * scale + offset applied to in-bounds pixels (zero padding stays
 * zero in the normalised space): the TF flavour feeds (img - 128) / 128 (model/encoder.py:26-27) -> scale 1/128, offset -1.
 * img: fp32 or uint8 [N][H][W] (img_is_u8). */
int lo_conv1_pool_forward_norm(const void* img, int img_is_u8, float scale, float offset, const float* w,
                               const float* bias, void* out, int dt, int N, int H, int W, void* stream);
int lo_conv1_pool_wgrad_norm(const void* img, int img_is_u8, float scale, float offset, const float* w,
                             const float* bias, const void* dpool, int dt, float* dw, float* db, int N, int H, int W,
                             void* stream);
/* Training variant: the forward additionally stores one byte per pooled output and channel, [N][H/2][W/2][64] — bits 0-1 the
 * window index (py*2+px) of the pool arg-max (first maximum in scan order, as nn.MaxPool2d), bit 2 the ReLU bit — and the
 * weight gradient reads the codes instead of recomputing conv1.  img fp32 or uint8 (img_is_u8); scale/offset as above (1, 0 for
 * the torch flavour). */
int lo_conv1_pool_forward_code(const void* img, int img_is_u8, float scale, float offset, const float* w, const float* bias,
                               void* out, uint8_t* code, int dt, int N, int H, int W, void* stream);
int lo_conv1_pool_wgrad_code(const void* img, int img_is_u8, float scale, float offset, const uint8_t* code, const void* dpool,
                             int dt, float* dw, float* db, int N, int H, int W, void* stream);
/* General strided convolution = im2col + lo_gemm: the 'cnn' encoder variant's Conv2d(512,512,(2,4),stride=2,padding=1)
 * (seq2seq_torch.py:80).  col [N*Ho*Wo][R*S*C], taps-major, C % 8 == 0; forward y = relu(col W^T + b) with W [Cout][R][S][C];
 * weight gradient dW = dy^T col; data gradient dcol = dy W then lo_col2im (a gather over the windows covering each input
 * pixel, optional ReLU mask of the producing layer). */
int lo_im2col(const void* x, void* col, int dt, int N, int H, int W, int C, int R, int S, int stride, int pad,
              void* stream);
int lo_col2im(const void* dcol, const void* mask, void* dx, int dt, int N, int H, int W, int C, int R, int S,
              int stride, int pad, void* stream);
/* out[n][k] = in[k][n] for k < K, n < N */
int lo_transpose(const void* in, int64_t ld_in, void* out, int64_t ld_out, int dt, int K, int N, void* stream);
/* y = [relu](conv3x3(x, w, pad) + bias) [* (mask > 0)] ; x [N][H][W][Cin], y [N][H+2pad-2][W+2pad-2][Cout];
 * pad in {0,1,2}.  mask (optional, same shape/dtype as y) implements the ReLU backward when this
 * call computes a data gradient.  bias may be NULL. */
int lo_conv3x3(const void* x, const void* w, const float* bias, const void* mask, void* y, int dt,
               int N, int H, int W, int Cin, int Cout, int pad, int relu, int impl, void* stream);
/* dw[Cout][3][3][Cin] = sum x (*) dy ; db[Cout] = sum dy ; x [N][H][W][Cin], dy [N][Ho][Wo][Cout] */
int lo_conv3x3_wgrad(const void* x, const void* dy, float* dw, float* db, int dt,
                     int N, int H, int W, int Cin, int Cout, int pad, int impl, void* stream);
/* wt[Cin][3][3][Cout] = w[Cout][2-r][2-s][Cin]  (weights of the data-gradient convolution) */
int lo_conv_weight_flip(const void* w, void* wt, int dt, int Cin, int Cout, void* stream);
/* floor-mode max-pool kh x kw, stride = kernel (nn.MaxPool2d seq2seq_torch.py:37,42,49,52) */
int lo_maxpool_forward(const void* x, void* y, int dt, int N, int H, int W, int C, int kh, int kw, void* stream);
/* dx = route dy to the first maximum of each window, times (x > 0) (x is a ReLU output) */
int lo_maxpool_backward(const void* x, const void* y, const void* dy, void* dx, int dt,
                        int N, int H, int W, int C, int kh, int kw, void* stream);
/* out = y + timing_signal (seq2seq_torch.py:115-157); table fp32 [H][W][C] built once by the host */
int lo_add_table(const void* y, const float* table, void* out, int dt, int N, int64_t HWC, void* stream);
/* dY6 = denc (fp32) * (y6 > 0), cast to dt */
int lo_relu_mask_cast(const float* g, const void* y, void* out, int dt, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Attention (single step): Attention.forward seq2seq_torch.py:178-192 with att1 hoisted.
 * att1,enc [B][R][A|C] (dt) ; att2 [B][A] fp32 (= decoder_att(h)) ; wf [A] fp32 (full_att.weight; its bias
 * cancels in the softmax) ; alpha out fp32 [B][alpha_stride>=R] ; ctx out fp32 [B][C].
 * gate_pre (optional) [B][gate_stride]: if given, gate = sigmoid(gate_pre) is written back in place and
 * gctx [B][C] = gate*ctx (seq2seq_torch.py:311-312).  work: lo_attention_workspace_bytes(B, C) bytes.
 */
int64_t lo_attention_workspace_bytes(int B, int C);
int64_t lo_decoder_workspace_bytes(int B, int C);   /* `work` of lo_decoder_args: two attention regions (two row chains) */
int lo_attention_forward(const void* att1, const void* enc, int dt, const float* att2, int64_t att2_stride,
                         const float* wf, float* alpha, int64_t alpha_stride, float* ctx,
                         float* gate_pre, int64_t gate_stride, float* gctx,
                         int B, int R, int A, int C, void* work, void* stream);
/* the same, additionally storing the ReLU mask bits for lo_attention_backward(relu_mask = ...): relu_mask_out is
 * [B][Rp][A/8] bytes with Rp = R rounded up to an even count; bit 7 - a % 8 of the byte of (r, a / 8) = att1 + att2 > 0, and that
 * byte lives at (r / 2) * 2 * (A/8) + (a / 8) * 2 + (r & 1) within image b (the bytes of an even/odd row pair are adjacent).
 * The buffer is opaque to callers: only its size matters. */
int lo_attention_forward_mask(const void* att1, const void* enc, int dt, const float* att2, int64_t att2_stride,
                              const float* wf, float* alpha, int64_t alpha_stride, float* ctx,
                              float* gate_pre, int64_t gate_stride, float* gctx, uint8_t* relu_mask_out,
                              int B, int R, int A, int C, void* work, void* stream);

/* Backward of one attention step (autograd of seq2seq_torch.py:186-190 + the gate of :311-312), reading att1 and enc ONCE:
 *   dctx = dgctx * gate ; dgp = dgctx * ctx * gate (1 - gate) ; s = <dctx, ctx> + sreg[b]
 *   dalpha_r = <dctx, enc_r> + dreg[b][r] ; de_r = alpha_r (dalpha_r - s) ; datt2_a = wf_a sum_r de_r [att1_ra + att2_a > 0]
 * att2 / gate [B][o1_stride] fp32 as the forward left them (gate after the sigmoid; NULL = ungated context) ; alpha / de
 * [B][alpha_stride] ; ctx / dctx_out [B][C] ; dgctx [B][dg_stride] ; dreg [B][dreg_stride] and sreg [B][sreg_stride] may be NULL ;
 * datt2 / dgp [B][dcat_stride] ; dwf_part (optional) [B][A] += sum_r de_r relu(att1_r + att2) (full_att.weight gradient).
 * dgp and dctx_out may be NULL; with gate NULL, dctx = dgctx and dgp (when given) is written with zeros.
 * d att1 and d enc are NOT produced here: they are hoisted out of the time loop (see lo_decoder_backward).
 * relu_mask (optional): the bits lo_attention_forward_mask stored; att1 is then NOT read, and dwf_part (optional) receives only the
 * att2 term of the full_att.weight gradient, sum_r de_r [on] att2_a — the term that needs att1 itself, sum_r de_r [on] att1_ra, is
 * added by lo_decoder_backward's single sweep over att1 after the time loop. */
int lo_attention_backward(const void* att1, const void* enc, int dt, const float* att2, const float* gate, int64_t o1_stride,
                          const float* wf, const float* alpha, int64_t alpha_stride, const float* ctx, const float* dgctx,
                          int64_t dg_stride, const float* dreg, int64_t dreg_stride, const float* sreg, int64_t sreg_stride,
                          float* de, float* datt2, float* dgp, int64_t dcat_stride, float* dctx_out, float* dwf_part,
                          const uint8_t* relu_mask, int B, int R, int A, int C, void* work, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Whole teacher-forced decoder: DecoderWithAttention.forward seq2seq_torch.py:267-320 (+ the loss of
 * img2seq_torch.py:147-159) and its hand-derived backward.  One struct carries every buffer; the
 * Python side (latex_ocr_b200/decoder.py) parses THIS header to build the ctypes mirror.
 * Shapes: B rows (already sorted by length), T steps, R regions, C=enc dim, A=att dim, D=decoder dim,
 * E=embed dim, V=vocab.  "f32" fields are float*, "big" fields are `dt` storage.
 */
typedef struct lo_decoder_args {
  int32_t B, T, R, C, A, D, E, V;
  int32_t dt;              /* storage of enc/att1/weight shadows */
  int32_t impl;            /* LO_IMPL_SIMT | LO_IMPL_TC for the hoisted GEMMs */
  int32_t has_dropout;     /* 0: eval ; 1: multiply h by dropout_mask before fc (injected mask: parity tests) ;
                              2: draw the inverted-dropout mask inside the LSTM kernels (Philox4x32-10 keyed by dropout_state,
                                 regenerated in the backward; nothing is stored) */
  int32_t ldl;             /* row stride of logits/dlogits (>= V; a multiple of 64 enables the tcgen05 fc GEMMs); 0 -> V */
  float alpha_c;           /* doubly-stochastic regulariser weight (img2seq_torch.py:157) */
  int32_t rows_per_img;    /* decode only: consecutive rows that share one image (beam size); 0/1 for training */
  int32_t phase;           /* 0: whole call (default).  EXTENSION (a second decoder layer between the cell and fc): 1 = time loop
                              only — lo_decoder_forward stops after writing hd, lo_decoder_backward starts from the dhd the caller
                              put there; 2 = head only — logits + loss from whatever the caller left in hd, backward of fc -> dhd */
  const int32_t* bt_host;  /* HOST int[T]: rows active at step t (seq2seq_torch.py:308); non-increasing */
  const int64_t* caps;     /* [B][caps_stride] token ids (sorted rows) */
  int64_t caps_stride;
  /* inputs */
  const void* enc;         /* big [B][R][C] */
  /* parameters: weight shadows in `dt`, biases fp32.  Wcat1 = [decoder_att; f_beta; weight_hh] rows
   * (contiguous [A+C+4D][D]), bcat1 likewise.  w_ih is [4D][E+C]. */
  const void* w_enc_att; const float* b_enc_att;   /* [A][C] */
  const void* wcat1; const float* bcat1;           /* [A+C+4D][D] */
  const float* w_full;                             /* [A] fp32 */
  const void* emb;                                 /* [V][E] */
  const void* w_ih; const float* b_ih;             /* [4D][E+C] */
  const void* w_init; const float* b_init;         /* [2D][C]: init_h rows then init_c rows */
  const void* w_fc; const float* b_fc;             /* [V][D] */
  /* transposed shadows for the backward per-step GEMMs (built by lo_decoder_pack_bwd_weights) */
  void* wbwd1;             /* [C+D][4D]: rows 0..C-1 = w_ih[:,E+j]^T, rows C.. = w_hh[:,j]^T */
  void* wbwd2;             /* [D][A+C]: [n][k] = k<A ? w_dec_att[k][n] : w_f_beta[k-A][n] */
  /* forward state (f32 unless noted) */
  void* att1;              /* big [B][R][A] */
  float* ptab;             /* [V][4D] = emb @ w_ih[:, :E]^T + b_ih */
  float* mean;             /* [B][C] */
  float* hall;             /* [T+1][B][D] */
  float* call;             /* [T+1][B][D] */
  float* out1;             /* [T][B][A+C+4D]: att2 | gate (sigmoid applied) | h@w_hh^T+b_hh */
  float* alphas;           /* [B][T][R] */
  uint8_t* att_mask;       /* optional, training only: [T][B][Rp][A/8], Rp = R rounded up to even (layout: lo_attention_forward_mask) — bit = (att1[b][r][a] + att2_t[b][a] > 0),
                              written by the forward attention kernel; the backward then streams enc + these 64 bytes per region
                              instead of enc + att1 (60.5 MB instead of 114 MB per step at cfg #2).  NULL: att1 is re-read. */
  float* ctx;              /* [T][B][C] */
  float* gctx;             /* [T][B][C] */
  float* gates;            /* [T][B][4D] post-activation i,f,g,o */
  float* gtmp;             /* [B][4D] scratch */
  const float* dropout_mask; /* [B][T][D] multipliers or NULL */
  const uint64_t* dropout_state; /* has_dropout=2: device {seed, call counter}; lo_decoder_backward increments the counter */
  float dropout_p;         /* has_dropout=2: drop probability (seq2seq_torch.py:216 nn.Dropout(p)) */
  float* hd;               /* [B][T][D] h after dropout */
  float* logits;           /* [B][T][ldl]  (== predictions in the first V columns) */
  /* loss */
  float* row_loss;         /* [B*T + B*R]: per-position CE, then the B*R regulariser partials (1 - sum_t alpha)^2 */
  float* loss;             /* [4]: total, ce, reg, n_valid */
  /* backward state */
  float* dlogits;          /* [B][T][ldl] */
  float* dhd;              /* [B][T][D] */
  float* dreg;             /* [B][R] gradient of the regulariser w.r.t. alpha (same for every t) */
  const float* dalpha_ext; /* optional external d loss/d alphas [B][T][R] (generic autograd mode); overrides dreg */
  float* sreg;             /* [B][T] */
  float* dcat;             /* [T][B][A+C+4D]: datt2 | dgate_pre | dgates_pre */
  float* dxh;              /* [B][C+D] scratch: dgctx | dh_prev */
  float* dc;               /* [2][B][D] ping-pong dc */
  float* dctx;             /* [T][B][C] */
  float* de;               /* [B][T][R] */
  float* dptab;            /* [V][4D] */
  void* datt1;             /* big [B][R][A] */
  float* denc;             /* f32 [B][R][C]  (output: gradient w.r.t. encoder_out) */
  float* dinit;            /* [B][2D] = dh0 | dc0 */
  float* dmean;            /* [B][max(A,C)]: d mean_r(enc); doubles as the [B][A] d full_att.weight scratch of the time loop */
  /* parameter gradients (fp32, reference layouts) */
  float* g_w_enc_att; float* g_b_enc_att;
  float* g_wcat1; float* g_bcat1;
  float* g_w_full; float* g_b_full;
  float* g_emb;
  float* g_w_ih; float* g_b_ih;
  float* g_w_init; float* g_b_init;
  float* g_w_fc; float* g_b_fc;
  void* work;              /* lo_decoder_workspace_bytes(B, max(A,C)), zero-initialised once */
  void* bfwork;            /* optional (impl=TC, dt=bf16): bf16 staging for the hoisted tcgen05 GEMMs,
                              lo_decoder_bfwork_bytes(args) bytes */
} lo_decoder_args;

int64_t lo_decoder_bfwork_bytes(const lo_decoder_args* a);
/* sizeof(lo_decoder_args) as compiled into the library (the ctypes mirror checks it) */
int64_t lo_sizeof_decoder_args(void);
/* forward through all T steps + logits ; if with_loss, also CE + regulariser into loss[] */
int lo_decoder_forward(const lo_decoder_args* a, int with_loss, void* stream);
/* backward of loss[0]; fills every g_* and denc.  Requires lo_decoder_forward(with_loss=1) state. */
int lo_decoder_backward(const lo_decoder_args* a, void* stream);
int lo_decoder_pack_bwd_weights(const lo_decoder_args* a, void* stream);

/* greedy decode on the same step kernels (decode loop semantics of dynamic_decode.py:17-74 +
 * greedy_decoder_cell.py:46-66): tokens out [B][max_steps] int64, first input token = start_id */
int lo_decoder_greedy(const lo_decoder_args* a, int64_t start_id, int64_t end_id, int max_steps,
                      int64_t* tokens, int32_t* finished, void* stream);
/* greedy: tokens [B][max_steps]; fin_hist (optional) [B][max_steps] int32 = finished flag after each step */
int lo_decoder_greedy_hist(const lo_decoder_args* a, int64_t start_id, int64_t end_id, int max_steps,
                           int64_t* tokens, int32_t* finished, int32_t* fin_hist, void* stream);

/* beam search on the same step kernels: beam_search_decoder_cell.py:98-187 (log-softmax, finished mask with
 * dtype.min, only beam 0 at time 0, top-k over beam*V with the lower index winning ties, state gather by parents;
 * no length normalisation, diversity penalty off as in configs/model.json:15-16).  a->B = n_img*beam rows,
 * a->rows_per_img = beam, a->enc holds n_img images.  ids/parents out [n_img][max_steps][beam] int64,
 * fin_hist [n_img][max_steps][beam] int32 (finished flags after each step), logp [n_img][beam] final scores. */
int lo_decoder_beam(const lo_decoder_args* a, int64_t start_id, int64_t end_id, int max_steps, int64_t* ids,
                    int64_t* parents, int32_t* fin_hist, float* logp, void* stream);
/* the same with the diversity penalty of beam_search_decoder_cell.py:258-287 (Li et al. 2016; configs/model.json:15-16
 * div_gamma / div_prob): every candidate's accumulated log-prob gets log(div_gamma) * (its rank inside its beam row, 0 = best)
 * where div_prob > u, u ~ U[0,1) per (image, beam, token).  Off when div_gamma == 1 or div_prob == 0 (:270-273).
 * div_u (optional) injects the uniforms [max_steps][B][V] (parity tests); otherwise they are drawn in the kernel from
 * Philox4x32-10 keyed by div_state = device {seed, call counter}. */
int lo_decoder_beam_div(const lo_decoder_args* a, int64_t start_id, int64_t end_id, int max_steps, int64_t* ids,
                        int64_t* parents, int32_t* fin_hist, float* logp, float div_gamma, float div_prob,
                        const float* div_u, const uint64_t* div_state, void* stream);

/* ------------------------------------------------------------------------------------------------
 * TensorFlow-flavour decoder (SURVEY.md §8-a row a7): the Genthial attention cell of
 * model/components/attention_cell.py:58-89 + attention_mechanism.py:43-94,145-153, driven like
 * model/decoder.py:24-72 (teacher forcing = tf.nn.dynamic_rnn over [start_token ; E[formula[:, :-1]]]),
 * masked cross-entropy of model/img2seq.py:68-71, hand-derived backward, greedy / beam decode.
 *   per step:  [i j f o] = [emb_{t-1}; o_{t-1}; h_{t-1}] K + b        (TF LSTMCell, forget_bias 1)
 *              e_r = beta . tanh(att_img_r + h_t W_h) ; alpha = softmax ; ctx = sum alpha_r img_r
 *              o_t = tanh(h_t o_W_h + ctx o_W_c) ; logits_t = o_t y_W_o
 * Parameter storage is [out][in] (K-major for the forward GEMMs; the Python side exposes TF-shaped
 * [in][out] views of the same memory).  Shapes: B rows, T steps (buffer capacity), R regions, C channels,
 * A=dim_e ((A, C) equal or (256, 512): the instantiated widths of the attention kernels), D=num_units, O=dim_o,
 * E=dim_embeddings, V=vocab.
 */
typedef struct lo_tfdec_args {
  int32_t B, T, R, C, A, D, O, E, V;
  int32_t dt;              /* storage of enc / att_img / weight shadows */
  int32_t impl;            /* LO_IMPL_SIMT | LO_IMPL_TC */
  int32_t ldl;             /* row stride of logits / dlogits (>= V, multiple of 8) */
  int32_t rows_per_img;    /* decode only: beam size (consecutive rows share one image); 0/1 otherwise */
  float inv_n_words;       /* 1 / sum(lengths): the loss is the mean over valid tokens */
  const void* enc;         /* big [B/rows_per_img][R][C] */
  const int64_t* formula;  /* [B][formula_stride] target ids; step t consumes formula[:, t-1], predicts formula[:, t] */
  int64_t formula_stride;
  const int32_t* lengths;  /* device [B]: valid tokens per row incl. END (sequence_mask, img2seq.py:69) */
  const float* keep_h;     /* optional [T][B][D] dropout multipliers for new_h (attention_cell.py:72), pre-scaled by 1/keep */
  const float* keep_o;     /* optional [T][B][O] for new_o (:83) */
  /* parameters: weight shadows in `dt`, biases / beta fp32 */
  const void* w_img;       /* [A][C]          att_img.kernel^T */
  const void* w_cat2;      /* [A+O][D]        att_h.kernel^T rows, then o_W_h^T rows */
  const float* beta;       /* [A]             att_beta */
  const void* w_lstm;      /* [4D][E+O+D]     lstm.kernel^T (gate rows i, j, f, o) */
  const float* b_lstm;     /* [4D] */
  const void* w_oc;        /* [O][C]          o_W_c^T */
  const void* w_y;         /* [V][O]          y_W_o^T */
  const void* w_init;      /* [2D+O][C]       W_c_0^T, W_h_0^T, W_o_0^T */
  const float* b_init;     /* [2D+O] */
  const void* emb;         /* [V+1][E]        embedding_table rows, then start_token */
  /* parameter gradients, fp32, same layouts */
  float* g_w_img; float* g_w_cat2; float* g_beta; float* g_w_lstm; float* g_b_lstm; float* g_w_oc; float* g_w_y;
  float* g_w_init; float* g_b_init; float* g_emb;
  /* results */
  float* logits;           /* [T][B][ldl] time-major */
  float* alphas;           /* [B][T][R] */
  uint8_t* att_mask;       /* optional, training only: [T][B][Rp][A/8], Rp = R rounded up to even (layout: lo_attention_forward_mask) — bit = (att1[b][r][a] + att2_t[b][a] > 0),
                              written by the forward attention kernel; the backward then streams enc + these 64 bytes per region
                              instead of enc + att1 (60.5 MB instead of 114 MB per step at cfg #2).  NULL: att1 is re-read. */
  float* loss;             /* [4]: mean CE over valid tokens (x2), 0, n_words — ce_words (img2seq.py:74) = loss[0] * loss[3] */
  float* denc;             /* f32 [B][R][C] gradient w.r.t. the encoder output */
  void* ws;                /* lo_tfdec_workspace_bytes(args) bytes, zero-initialised once by the caller */
} lo_tfdec_args;

int64_t lo_sizeof_tfdec_args(void);
int64_t lo_tfdec_workspace_bytes(const lo_tfdec_args* a);
/* all T steps + logits; with_loss: masked CE into loss[] (and d logits kept for the backward) */
int lo_tfdec_forward(const lo_tfdec_args* a, int with_loss, void* stream);
/* backward of loss[0]: fills every g_* and denc (requires lo_tfdec_forward(with_loss=1) state in ws) */
int lo_tfdec_backward(const lo_tfdec_args* a, void* stream);
/* greedy decode (greedy_decoder_cell.py:38-66 + dynamic_decode.py:38-61): tokens [B][max_steps], fin_hist (optional)
 * [B][max_steps] finished flags after each step; max_steps <= T */
int lo_tfdec_greedy(const lo_tfdec_args* a, int64_t end_id, int max_steps, int64_t* tokens, int32_t* fin_hist, void* stream);
/* beam search (beam_search_decoder_cell.py:98-187): B = n_img*beam rows, rows_per_img = beam; ids/parents/fin_hist
 * [n_img][max_steps][beam], logp [n_img][beam] */
int lo_tfdec_beam(const lo_tfdec_args* a, int64_t end_id, int max_steps, int64_t* ids, int64_t* parents, int32_t* fin_hist,
                  float* logp, void* stream);
/* with the diversity penalty (see lo_decoder_beam_div) */
int lo_tfdec_beam_div(const lo_tfdec_args* a, int64_t end_id, int max_steps, int64_t* ids, int64_t* parents, int32_t* fin_hist,
                      float* logp, float div_gamma, float div_prob, const float* div_u, const uint64_t* div_state, void* stream);

/* ------------------------------------------------------------------------------------------------
 * EXTENSION (not in the reference; BASELINE.json configs[3]): generic sequence LSTM with nn.LSTM semantics (gate order i,f,g,o,
 * two bias vectors), forward over S steps for M independent sequences + hand-derived backward.  Used for the row-encoder biLSTM
 * over the CNN feature rows (two calls, `reverse` = 0 / 1, writing the two halves of the output channels) and for a second decoder
 * layer.  Element (t, m) of x / dx lives at m * row + t * step (+ channel); of hs / hs_st / dhs at m * hs_row + t * hs_step.
 */
typedef struct lo_lstm_seq_args {
  int32_t S, M, I, H;      /* steps, sequences, input width, hidden width (I, H multiples of 8) */
  int32_t dt;              /* storage of x / hs_st / the weight shadows: LO_F32 | LO_BF16 */
  int32_t impl;            /* LO_IMPL_SIMT | LO_IMPL_TC (bf16 only) */
  int32_t reverse;         /* 1: process t = S-1 .. 0 */
  int32_t dx_accumulate;   /* backward: add onto dx instead of overwriting (second direction of a bidirectional layer) */
  const void* x;           /* dt */
  int64_t x_row, x_step;
  const void* w_ih;        /* dt [4H][I] */
  const void* w_hh;        /* dt [4H][H] */
  const float* b_ih; const float* b_hh;   /* fp32 [4H] */
  const float* h0; const float* c0;       /* optional fp32 [M][H] (NULL = zeros) */
  float* hs;               /* optional out fp32 */
  void* hs_st;             /* optional out, storage dtype */
  int64_t hs_row, hs_step;
  const float* dhs;        /* backward in: d loss / d hs (fp32, hs strides); NULL = zeros */
  float* dx;               /* optional backward out fp32 */
  int64_t dx_row, dx_step;
  float* g_w_ih; float* g_w_hh; float* g_b_ih; float* g_b_hh;   /* backward out, fp32, overwritten */
  float* dh0; float* dc0;  /* optional backward out fp32 [M][H] */
  void* ws;                /* lo_lstm_seq_workspace_bytes(args) bytes; forward state is kept there for the backward */
} lo_lstm_seq_args;
int64_t lo_sizeof_lstm_seq_args(void);
int64_t lo_lstm_seq_workspace_bytes(const lo_lstm_seq_args* a);
int lo_lstm_seq_forward(const lo_lstm_seq_args* a, void* stream);
int lo_lstm_seq_backward(const lo_lstm_seq_args* a, void* stream);

/* EXTENSION: greedy / beam decoding of the two-layer decoder (layer 1 = the attention LSTM of lo_decoder_args, layer 2 =
 * nn.LSTMCell(D, D) over h1_t with zero initial state, logits_t = fc(h2_t); no dropout at decode time).  Layer 2 runs inside the
 * time loop, one step per step: gates2 = h1_t W_ih^T + h2_{t-1} W_hh^T + b_ih + b_hh, then the cell (gate order i,f,g,o).
 * In beam search its state (h2, c2) is gathered by parents like layer 1's.  Loop rules, outputs and limits are those of
 * lo_decoder_greedy_hist / lo_decoder_beam_div. */
typedef struct lo_dec2_args {
  int32_t D;               /* hidden width; must equal lo_decoder_args.D */
  int32_t dt;              /* storage of the weight shadows: LO_F32 | LO_BF16 */
  int32_t impl;            /* LO_IMPL_SIMT | LO_IMPL_TC (tensor-core GEMMs; used when the decoder runs its bf16 mirrors) */
  const void* w_ih;        /* dt [4D][D] */
  const void* w_hh;        /* dt [4D][D] */
  const float* b_ih; const float* b_hh;   /* fp32 [4D] */
  void* ws;                /* lo_dec2_workspace_bytes(B, D) bytes, B = lo_decoder_args.B; no initialisation needed */
} lo_dec2_args;
int64_t lo_sizeof_dec2_args(void);
int64_t lo_dec2_workspace_bytes(int B, int D);
int lo_decoder2_greedy_hist(const lo_decoder_args* a, const lo_dec2_args* l2, int64_t start_id, int64_t end_id, int max_steps,
                            int64_t* tokens, int32_t* finished, int32_t* fin_hist, void* stream);
int lo_decoder2_beam_div(const lo_decoder_args* a, const lo_dec2_args* l2, int64_t start_id, int64_t end_id, int max_steps,
                         int64_t* ids, int64_t* parents, int32_t* fin_hist, float* logp, float div_gamma, float div_prob,
                         const float* div_u, const uint64_t* div_state, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Optimiser: torch.optim.Adam defaults (img2seq_torch.py:86-87, :168-170) on one flat buffer.
 * state_dev: float[2] = {step (as float), lr}; step is incremented on the device so the call is
 * graph-replayable.  shadow (optional) receives the bf16 copy of the updated parameters.
 */
int lo_adam_step(float* p, const float* g, float* m, float* v, void* shadow_bf16, int64_t n,
                 float* state_dev, float beta1, float beta2, float eps, float grad_scale, void* stream);
/* Same update restricted to n_ranges element ranges {offset, count} (host array of 2*n_ranges int64) of the flat buffers:
 * parameters outside the ranges are frozen (requires_grad=False after fine_tune(), seq2seq_torch.py:102-113, :246-253 —
 * torch.optim.Adam skips them: no moment decay, no update).  One step-counter increment for the whole call. */
int lo_adam_step_ranges(float* p, const float* g, float* m, float* v, void* shadow_bf16, const int64_t* ranges,
                        int n_ranges, float* state_dev, float beta1, float beta2, float eps, float grad_scale,
                        void* stream);
/* The optimisers of the TF trainer (model/img2seq.py:98-111) with TensorFlow 1.12's update rules, on one flat buffer:
 * kind 1 AdamOptimizer (epsilon outside the bias correction: lr_t = lr sqrt(1-b2^t)/(1-b1^t), p -= lr_t m/(sqrt(v)+eps)),
 * 2 GradientDescentOptimizer, 3 AdagradOptimizer (s1 = accumulator, initial value 0.1), 4 RMSPropOptimizer (s1 = rms slot,
 * initial value 1; beta2 = decay 0.9, eps 1e-10, momentum 0).  state_dev as in lo_adam_step. */
int lo_tf_optim_step(int kind, float* p, const float* g, float* s1, float* s2, void* shadow_bf16, int64_t n,
                     float* state_dev, float beta1, float beta2, float eps, float grad_scale, void* stream);
int lo_cast(const void* src, int dt_src, void* dst, int dt_dst, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LATEX_OCR_B200_H */
