/*
 * bnn_b200.h — C ABI of libbnn_b200.so: the B200 (sm_100a) variational hot path of
 * pytorch_bayesian (Mirko-Nava/BayesianNeuralNetworks).
 *
 * The reference has no FFI of its own (it is pure Python on torch ops); each entry point below
 * replaces the torch-op sequence of one reference call site, cited as file:line relative to the
 * reference checkout.  All pointers are raw DEVICE pointers to fp32 unless stated otherwise; the
 * caller owns every buffer (outputs and workspaces included) and passes the CUDA stream to
 * launch on.  The library never allocates or frees device memory, never synchronises the
 * stream, keeps no mutable global state besides lazily-set kernel attributes, and has no CPU
 * fallback.  Every function returns a bnn_status (0 = ok); no C++ exception crosses the boundary.
 *
 * Random numbers: eps is a pure function of (seed, step, tensor_id, global sample index,
 * element index) through Philox4x32-10 + Box-Muller (see bnn_rng), so any partition of the
 * samples over GPUs or launches regenerates the same stream, and the backward pass regenerates
 * the forward's eps from the same counters.  When `eps` pointers are non-NULL the kernels read
 * eps from memory instead (layout [S][numel], the test-only "eps-injected" mode used for parity
 * against the reference's torch.randn_like tensors).
 */
#ifndef BNN_B200_H
#define BNN_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BNN_B200_ABI_VERSION 1

typedef enum bnn_status {
  BNN_OK = 0,
  BNN_ERR_BAD_ARGUMENT = 1,   /* null pointer, negative size, inconsistent shapes           */
  BNN_ERR_MISALIGNED = 2,     /* pointer or leading dimension violates a stated alignment   */
  BNN_ERR_UNSUPPORTED_ARCH = 3, /* current device is not compute capability 10.x            */
  BNN_ERR_CUDA = 4,           /* a CUDA runtime call failed; see bnn_last_error_string()    */
  BNN_ERR_WORKSPACE = 5,      /* workspace too small; query the matching *_workspace_size   */
  BNN_ERR_UNSUPPORTED = 6     /* valid request the kernels do not implement (stated limits) */
} bnn_status;

/* Arithmetic mode of the sampled contractions.  TF32: tcgen05 kind::tf32, fp32 accumulate
 * (2e-3 parity class).  FP32X3: three-term TF32 split (hi*hi + hi*lo + lo*hi), fp32-class
 * accuracy (1e-5 parity class) on the same tensor-core path. */
typedef enum bnn_precision {
  BNN_PREC_TF32 = 0,
  BNN_PREC_FP32X3 = 1
} bnn_precision;

/* Philox stream selector.  eps(seed, step, tensor_id, sample, element):
 *   key     = (seed_lo, seed_hi)
 *   counter = ((element + elem_offset) / 4, sample, tensor_id, step_lo) with step_hi folded into key.y
 * `step_dev` (optional, device pointer to one uint64) is ADDED to `step` inside the kernel, so a
 * captured CUDA graph can advance the stream without re-capturing. */
typedef struct bnn_rng {
  uint64_t seed;
  uint64_t step;
  const uint64_t* step_dev;
  uint64_t elem_offset;   /* added to every element index: lets a launch address a slice (one conv
                             group) of a tensor and still draw the tensor-global stream */
  uint32_t tensor_id;
  uint32_t reserved;
  /* Rank-one sign noise (Flipout, Wen et al. 2018; reference dense.py:63-83): when row_sign != NULL the eps of weight
   * element (n, k) for sample index s is  row_sign[s * rows + n] * col_sign[s * cols + k]  (values +-1) instead of a Philox
   * normal, so  y = x (mu + sigma o (r s^T))^T = x mu^T + ((x o s) sigma^T) o r  comes out of ONE sampled contraction and
   * the backward kernels form d mu, d rho with the same eps.  s is the GLOBAL sample index (sample_begin + local index):
   * pass pointers offset accordingly.  cols = row length of the weight matrix; rows = its row count. */
  const float* row_sign;
  const float* col_sign;
  int32_t rows;
  int32_t cols;
} bnn_rng;

/* A dense matrix operand seen through an NCHW window: logical element (m, n), m in [0, M),
 * n in [0, N), lives at  base[(m / P) * batch_stride + n * P + (m % P)].
 * P = 1, batch_stride = ld  describes an ordinary row-major matrix (Linear activations);
 * P = OH*OW, batch_stride = C*OH*OW describes a conv feature map with m = (b, oh, ow). */
typedef struct bnn_view {
  float* base;
  int64_t batch_stride;
  int32_t P;
  int32_t reserved;
} bnn_view;

/* ---- library ---- */
int bnn_abi_version(void);
const char* bnn_last_error_string(void);           /* thread-local, never NULL */
int bnn_device_supported(int device);              /* BNN_OK iff compute capability 10.x */

/* sigma = 1e-10 + softplus(rho), softplus beta=1 threshold=20.
 * Replaces WeightNormal.stddev — pytorch_bayesian/nn/core.py:25-27. */
int bnn_stddev(const float* rho, float* sigma, int64_t numel, void* stream);

/* out[s][i] = mu[i] + sigma[i] * eps(s0 + s, i) for s in [0, S).
 * Replaces WeightNormal.sample — pytorch_bayesian/nn/core.py:44-45 (only needed when the caller
 * wants the sampled tensor in memory: `.sampled`, tests; the contractions never materialise it).
 * `eps_out` (optional, [S][numel]) receives the eps used.  `eps_in` (optional) injects eps. */
int bnn_materialize(const float* mu, const float* sigma, const float* eps_in, float* out,
                    float* eps_out, int64_t numel, int32_t S, uint32_t sample_begin,
                    const bnn_rng* rng, void* stream);

/* ---- sampled contractions ----
 * Forward:  Y[s] = A[s] * W_s^T + b_s,  W_s = mu_w + sigma_w * eps_w(s),  b_s likewise.
 * Replaces NormalLinear.sample/.forward — pytorch_bayesian/nn/dense.py:46-60 — and, with the
 * im2col matrix as A and an NCHW view as Y, NormalConv2d.forward — pytorch_bayesian/nn/conv.py:
 * 65-73,112-119 — for all S Monte-Carlo samples of container.py:32-37 in one launch.
 *   a            [S or 1][M][K] row-major, leading dimension lda (floats); a_sample_stride = 0
 *                when all samples share the same activations (first Bayesian layer).
 *   mu_w/sigma_w [N][K] row-major contiguous; mu_b/sigma_b [N] or NULL (no bias).
 *   eps_w [S][N*K], eps_b [S][N]: optional injected eps (NULL = Philox).
 *   y            view of [M][N] per sample; y_sample_stride floats between samples.
 * rng_w / rng_b select the streams of the weight and the bias tensor. */
int bnn_sampled_gemm_fwd(const float* a, int64_t lda, int64_t a_sample_stride,
                         const float* mu_w, const float* sigma_w,
                         const float* mu_b, const float* sigma_b,
                         const float* eps_w, const float* eps_b,
                         bnn_view y, int64_t y_sample_stride,
                         int32_t M, int32_t N, int32_t K, int32_t S, uint32_t sample_begin,
                         const bnn_rng* rng_w, const bnn_rng* rng_b,
                         int32_t precision, void* stream);

/* Data gradient: dA[s] = dY[s] * W_s  (W_s regenerated from the same counters).
 * With a_sample_stride == 0 the S contributions are summed into one dA (shared activations).
 * Autograd of F.linear / F.conv2d w.r.t. the input at dense.py:60 / conv.py:116-119. */
int bnn_sampled_gemm_dgrad(bnn_view dy, int64_t dy_sample_stride,
                           const float* mu_w, const float* sigma_w, const float* eps_w,
                           float* da, int64_t lda, int64_t a_sample_stride,
                           int32_t M, int32_t N, int32_t K, int32_t S, uint32_t sample_begin,
                           const bnn_rng* rng_w, int32_t precision, void* stream);

/* Weight gradient with the reparameterisation chain fused into the epilogue:
 *   G_s = dY[s]^T * A[s];  dmu_w += sum_s G_s;  drho_w += (sum_s G_s o eps_w(s)) o sigmoid(rho_w)
 * (SURVEY §3.2; autograd of core.py:44-45 + dense.py:60).  dmu_w / drho_w are ACCUMULATED INTO
 * (atomic adds when the launch splits the reduction), so zero them first for a fresh gradient.
 * rho_w is the raw scale parameter ([N][K]). */
int bnn_sampled_gemm_wgrad(bnn_view dy, int64_t dy_sample_stride,
                           const float* a, int64_t lda, int64_t a_sample_stride,
                           const float* rho_w, const float* eps_w,
                           float* dmu_w, float* drho_w,
                           int32_t M, int32_t N, int32_t K, int32_t S, uint32_t sample_begin,
                           const bnn_rng* rng_w, int32_t precision, void* stream);

/* Bias gradient: c_s[n] = sum_m dY[s][m][n]; dmu_b += sum_s c_s;
 * drho_b += (sum_s c_s * eps_b(s, n)) * sigmoid(rho_b[n]).  Accumulates (atomics). */
int bnn_bias_grad(bnn_view dy, int64_t dy_sample_stride, const float* rho_b, const float* eps_b,
                  float* dmu_b, float* drho_b, int32_t M, int32_t N, int32_t S,
                  uint32_t sample_begin, const bnn_rng* rng_b, void* stream);

/* ---- conv2d lowering helpers (NCHW, fp32) ----
 * col[(b*OH*OW + oh*OW + ow)][(c*KH + kh)*KW + kw] = x[b][c0 + c][oh*sh - ph + kh*dh][...] (0 outside).
 * c runs over `Cg` channels starting at c0 (one conv group). */
typedef struct bnn_conv2d_geom {
  int32_t B, C, H, W;          /* input batch, total channels, height, width */
  int32_t c0, Cg;              /* first channel and channel count of this group */
  int32_t KH, KW, OH, OW;
  int32_t sh, sw, ph, pw, dh, dw;
} bnn_conv2d_geom;
int bnn_im2col(const float* x, float* col, const bnn_conv2d_geom* g, void* stream);
/* dx[b][c0 + c][h][w] (+)= sum over (kh, kw, oh, ow) hitting (h, w) of dcol[...]; gather form, no
 * atomics; `accumulate` != 0 adds into dx instead of overwriting the group's channels. */
int bnn_col2im(const float* dcol, float* dx, const bnn_conv2d_geom* g, int32_t accumulate,
               void* stream);

/* ---- implicit-GEMM convolution (no im2col matrix) ----
 * NormalConv2d.forward — pytorch_bayesian/nn/conv.py:65-73,112-119 (F.conv2d(x, W_s, b_s, stride, padding, dilation)
 * for S Monte-Carlo samples) — and its autograd, for groups == 1 layers with in_channels % 32 == 0, TF32.
 * Layouts: activations NHWC (torch.channels_last memory) [S or 1][B][H][W][C] (x_sample_stride = 0: all samples share x,
 * else B*H*W*C); weights, sigma, rho, injected eps and the weight gradients in (o, kh, kw, c) order [Cout][KH][KW][C] —
 * bnn_conv2d_weight_layout / _unlayout convert from / to the reference's OIHW parameters; the eps stream of the tensor is
 * keyed by the element index in THAT order.  The activation operand reaches the tensor cores through an im2col tensor
 * map (cuTensorMapEncodeIm2col): a k-block is one filter tap x 32 channels.
 *   fwd    y[s] = conv2d(x[s], W_s) + b_s; y: view of [B*OH*OW][Cout] per sample (P = 1, batch_stride = Cout: NHWC;
 *          P = OH*OW, batch_stride = Cout*OH*OW: NCHW), y_sample_stride floats between samples
 *   dgrad  dx[s] = conv2d_transpose(dy[s], W_s) in the transposed-filter (gather) form, stride 1 only, Cout % 32 == 0;
 *          dy NHWC [S][B][OH][OW][Cout], dx NHWC; x_sample_stride = 0 sums the S contributions into one dx
 *   wgrad  G_s = dy[s]^T im2col(x[s]); dmu_w += sum_s G_s; drho_w += (sum_s G_s o eps_s) o sigmoid(rho_w) (accumulated)
 * BNN_ERR_UNSUPPORTED when a requirement is not met (callers then lower explicitly: bnn_im2col_nhwc + bnn_sampled_gemm_*). */
typedef struct bnn_conv2d_nhwc {
  int32_t B;                 /* images per Monte-Carlo sample */
  int32_t H, W, C;           /* input height, width, channels */
  int32_t OH, OW, Cout;
  int32_t KH, KW;
  int32_t sh, sw, ph, pw, dh, dw;
  int32_t reserved;
} bnn_conv2d_nhwc;
int bnn_sampled_conv2d_fwd(const float* x, int64_t x_sample_stride, const float* mu_w, const float* sigma_w,
                           const float* mu_b, const float* sigma_b, const float* eps_w, const float* eps_b, bnn_view y,
                           int64_t y_sample_stride, const bnn_conv2d_nhwc* g, int32_t S, uint32_t sample_begin,
                           const bnn_rng* rng_w, const bnn_rng* rng_b, void* stream);
int bnn_sampled_conv2d_dgrad(const float* dy, const float* mu_w, const float* sigma_w, const float* eps_w, float* dx,
                             int64_t x_sample_stride, const bnn_conv2d_nhwc* g, int32_t S, uint32_t sample_begin,
                             const bnn_rng* rng_w, void* stream);
int bnn_sampled_conv2d_wgrad(const float* dy, const float* x, int64_t x_sample_stride, const float* rho_w,
                             const float* eps_w, float* dmu_w, float* drho_w, const bnn_conv2d_nhwc* g, int32_t S,
                             uint32_t sample_begin, const bnn_rng* rng_w, void* stream);
/* ---- transposed convolution on the same kernels ----
 * NormalConvTranspose2d.forward (F.conv_transpose2d(x, W_s, b_s, stride, padding, output_padding, 1, dilation) for S
 * Monte-Carlo samples) and its autograd.  W [Cin][Cout][KH][KW]; `g` describes the CONV VIEW of the layer, the convolution
 * from the transposed output to the transposed input with the same W read as OIHW: g->C = Cout and g->H, g->W = output
 * size; g->Cout = Cin and g->OH, g->OW = input size; KH, KW, stride, padding, dilation as given (output_padding is the
 * part of g->H, g->W the conv view rounds away, so it must be below the stride).  Weights, sigma, rho, eps and gradients
 * in the conv view's (o, kh, kw, c) order = [Cin][KH][KW][Cout] (bnn_conv2d_weight_layout with Cout = Cin).
 *   fwd    y[s] = conv_transpose2d(x[s], W_s) + b_s: x NHWC [S or 1][B][OH][OW][Cin] (x_sample_stride = 0: shared), y NHWC
 *          [S][B][H][W][Cout] contiguous.  The outputs are cut into sh x sw phases (h % sh, w % sw); each phase is a
 *          stride-1 transposed-filter gather over its own taps (one launch per phase), phases without a tap get b_s.
 *          Needs Cin % 32 == 0, Cout % 4 == 0, stride <= 8.
 *   dgrad  dx[s] = conv2d(dy[s], W_s) (the conv view's forward, no bias); dy NHWC [S][B][H][W][Cout], dx NHWC;
 *          x_sample_stride = 0 sums the S contributions into one dx.  Needs Cout % 32 == 0, Cin % 4 == 0.
 *   wgrad  G_s = x[s]^T im2col(dy[s]) accumulated as bnn_sampled_conv2d_wgrad; x_sample_stride = 0: all samples read x.
 *          Needs Cout % 32 == 0, Cin % 4 == 0.
 * No allocation, no stream synchronisation.  BNN_ERR_UNSUPPORTED when a requirement is not met (callers then lower
 * explicitly: bnn_sampled_gemm_dgrad + bnn_col2im_nhwc for the forward, bnn_im2col_nhwc + bnn_sampled_gemm_fwd / _wgrad
 * for the gradients). */
int bnn_sampled_conv_transpose2d_fwd(const float* x, int64_t x_sample_stride, const float* mu_w, const float* sigma_w,
                                     const float* mu_b, const float* sigma_b, const float* eps_w, const float* eps_b, float* y,
                                     const bnn_conv2d_nhwc* g, int32_t S, uint32_t sample_begin, const bnn_rng* rng_w,
                                     const bnn_rng* rng_b, void* stream);
int bnn_sampled_conv_transpose2d_dgrad(const float* dy, const float* mu_w, const float* sigma_w, const float* eps_w,
                                       float* dx, int64_t x_sample_stride, const bnn_conv2d_nhwc* g, int32_t S,
                                       uint32_t sample_begin, const bnn_rng* rng_w, void* stream);
int bnn_sampled_conv_transpose2d_wgrad(const float* dy, const float* x, int64_t x_sample_stride, const float* rho_w,
                                       const float* eps_w, float* dmu_w, float* drho_w, const bnn_conv2d_nhwc* g, int32_t S,
                                       uint32_t sample_begin, const bnn_rng* rng_w, void* stream);
/* Host only (test aid): the phase plan of bnn_sampled_conv_transpose2d_fwd, 14 ints per phase {rh, rw, rows_h, rows_w,
 * taps_h, taps_w, last tap h, last tap w, tap step h, tap step w, first input row h, w, input step h, w}: walked tap j of
 * the phase is kh = last - j * tap step, read at input row i + first + j * input step for output row rh + sh * i.  Returns
 * the number of phases (may exceed max_phases; only max_phases are written) or a negative bnn_status. */
int bnn_debug_conv_transpose_phases(const bnn_conv2d_nhwc* g, int32_t* out, int32_t max_phases);
/* ---- 3-d transposed convolution (NormalConvTranspose3d) ----
 * The same three passes with a depth: activations NDHWC (torch.channels_last_3d memory), W [Cin][Cout][KD][KH][KW] and
 * `g` the conv view with the 2-d convention above (g->C = Cout, g->D, g->H, g->W = output size; g->Cout = Cin, g->OD,
 * g->OH, g->OW = input size).  Weights, sigma, rho, eps and gradients in (o, kd, kh, kw, c) order = [Cin][KD][KH][KW][Cout]
 * (bnn_conv2d_weight_layout with Cout = Cin, taps = KD*KH*KW).  The activation operand reaches the tensor cores through a
 * rank-5 im2col tensor map; GEMM row m = (img, d, h, w).  The forward cuts the outputs into sd x sh x sw phases.
 * One predicate for all three passes: Cin % 32 == 0, Cout % 32 == 0, stride <= 8, 16-byte aligned tensors, and every
 * phase corner and conv-view corner within [-16, 15] with every filter extent (k - 1) d below 32 (the rank-5 im2col
 * descriptor).  BNN_ERR_UNSUPPORTED when it does not hold; callers then contract materialised samples. */
typedef struct bnn_conv3d_nhwc {
  int32_t B;                 /* images per Monte-Carlo sample */
  int32_t D, H, W, C;        /* input depth, height, width, channels */
  int32_t OD, OH, OW, Cout;
  int32_t KD, KH, KW;
  int32_t sd, sh, sw, pd, ph, pw, dd, dh, dw;
  int32_t reserved;
} bnn_conv3d_nhwc;
int bnn_sampled_conv_transpose3d_fwd(const float* x, int64_t x_sample_stride, const float* mu_w, const float* sigma_w,
                                     const float* mu_b, const float* sigma_b, const float* eps_w, const float* eps_b, float* y,
                                     const bnn_conv3d_nhwc* g, int32_t S, uint32_t sample_begin, const bnn_rng* rng_w,
                                     const bnn_rng* rng_b, void* stream);
int bnn_sampled_conv_transpose3d_dgrad(const float* dy, const float* mu_w, const float* sigma_w, const float* eps_w,
                                       float* dx, int64_t x_sample_stride, const bnn_conv3d_nhwc* g, int32_t S,
                                       uint32_t sample_begin, const bnn_rng* rng_w, void* stream);
int bnn_sampled_conv_transpose3d_wgrad(const float* dy, const float* x, int64_t x_sample_stride, const float* rho_w,
                                       const float* eps_w, float* dmu_w, float* drho_w, const bnn_conv3d_nhwc* g, int32_t S,
                                       uint32_t sample_begin, const bnn_rng* rng_w, void* stream);
/* Host only (test aid): the phase plan of bnn_sampled_conv_transpose3d_fwd, 21 ints per phase: the seven fields of
 * bnn_debug_conv_transpose_phases, each for d, h, w {rd, rh, rw, rows_d, rows_h, rows_w, taps_d, ...}.  Returns the
 * number of phases (may exceed max_phases) or a negative bnn_status. */
int bnn_debug_conv_transpose3d_phases(const bnn_conv3d_nhwc* g, int32_t* out, int32_t max_phases);
/* Host only: whether the transposed-convolution kernels take ALL THREE passes (fwd, dgrad, wgrad) of the conv-view
 * geometry `g` — channel counts, strides, every phase corner of the forward and every conv-view corner of the gradients.
 * In 2-d the entry points check these one pass at a time, and with stride >= 2 the forward's phase corners (divided by
 * the stride) admit geometries whose conv view the gradients refuse; a caller that must not mix paths within one call
 * asks here before launching anything.  Tensor alignment is the caller's (16-byte bases).  BNN_OK when taken,
 * BNN_ERR_UNSUPPORTED when not, BNN_ERR_BAD_ARGUMENT for a NULL or inconsistent geometry.  No device needed. */
int bnn_conv_transpose2d_supported(const bnn_conv2d_nhwc* g);
int bnn_conv_transpose3d_supported(const bnn_conv3d_nhwc* g);
/* OIHW parameters [Cout][Cg][taps] -> (o, kh, kw, c) order: mu_p, and optionally sigma_p = 1e-10 + softplus(rho) and
 * rho_p (NULL to skip); the inverse for `n_arrays` arrays stored back to back (gradients of mean and scale). */
int bnn_conv2d_weight_layout(const float* mu, const float* rho, float* mu_p, float* sigma_p, float* rho_p, int32_t Cout,
                             int32_t Cg, int32_t taps, void* stream);
int bnn_conv2d_weight_unlayout(const float* in, float* out, int32_t n_arrays, int32_t Cout, int32_t Cg, int32_t taps,
                               void* stream);
/* dY of a conv layer as autograd delivers it for an NCHW-contiguous output ([n_imgs][N][P], P = OH*OW, n_imgs = S*B
 * sample-major) -> the row-major [n_imgs*P][N] (NHWC) matrix the gradient kernels read, one coalesced pass through shared
 * memory; with dmu_b / drho_b non-NULL the same pass accumulates the reparameterised bias gradient (see bnn_bias_grad;
 * eps_b [S][N] optional injected eps).  BNN_ERR_UNSUPPORTED when an image's (N + 1) x P floats exceed 48 KiB. */
int bnn_nchw_to_nhwc_bias_grad(const float* dy, float* dy_nhwc, int64_t n_imgs, int32_t B, int32_t N, int32_t P,
                               const float* rho_b, const float* eps_b, float* dmu_b, float* drho_b, uint32_t sample_begin,
                               const bnn_rng* rng_b, void* stream);
/* explicit lowering in the same column order (kh, kw, c), NHWC tensors of n_imgs images, C % 4 == 0:
 *   col[(n, oh, ow)][(kh*KW + kw)*C + c] = x[n][oh*sh - ph + kh*dh][ow*sw - pw + kw*dw][c]  (0 outside)
 *   dx[n][h][w][c] = sum of the dcol entries that read (n, h, w, c)  (gather form, overwrites dx) */
int bnn_im2col_nhwc(const float* x, float* col, const bnn_conv2d_nhwc* g, int64_t n_imgs, void* stream);
int bnn_col2im_nhwc(const float* dcol, float* dx, const bnn_conv2d_nhwc* g, int64_t n_imgs, void* stream);
/* ---- Flipout sign passes (FlipOutNormalConvTranspose1d / 2d / 3d) ----
 * Tensors of n images with C channels and P pixels per image (P = L, H*W or D*H*W); sign [n][C] of +-1.  "Channels-last"
 * is [n][P][C], "NC(D)HW" is [n][C][P].  The arithmetic is torch's: the sign product is exact, then one fp32 add, so the
 * outputs are bit-identical to `a * sign` and `a + b * sign`.  No size limit per image; 64-bit indexing.
 *   split    reads a once ([n][C][P], or channels-last when a_channels_last != 0) and writes sa_cl = sign * a in
 *            channels-last and, unless a already is channels-last (a_cl is then ignored and may be NULL), a_cl = a in
 *            channels-last.
 *   combine  reads channels-last a and b and writes out = a + sign * b, channels-last when out_channels_last != 0,
 *            else NC(D)HW-contiguous.
 * No allocation, no stream synchronisation.  BNN_ERR_BAD_ARGUMENT for NULL pointers, non-positive sizes or n*C*P beyond
 * 64 bits. */
int bnn_flipout_split(const float* a, int32_t a_channels_last, const float* sign, float* a_cl, float* sa_cl, int64_t n,
                      int32_t C, int64_t P, void* stream);
int bnn_flipout_combine(const float* a, const float* b, const float* sign, float* out, int32_t out_channels_last,
                        int64_t n, int32_t C, int64_t P, void* stream);

/* ---- KL divergence, closed form, many tensors per launch ----
 * For tensor t with posterior N(mu, sigma = 1e-10 + softplus(rho)) and scalar prior N(loc, scale):
 *   kl_sum[t] = sum_i 0.5*[(sigma/scale)^2 + ((mu-loc)/scale)^2 - 1 - log((sigma/scale)^2)]
 * Replaces KLDivergence.compute_kl — pytorch_bayesian/nn/loss.py:16-28 — and torch's
 * _kl_normal_normal (torch/distributions/kl.py:468-471); the caller applies the reference's
 * mean-of-means / n_batches reduction (loss.py:38) to the per-tensor sums.
 * Optional gradients (both NULL or both set per tensor), written not accumulated:
 *   grad_mu = c_t*(mu-loc)/scale^2,  grad_rho = c_t*(sigma/scale^2 - 1/sigma)*sigmoid(rho),
 *   c_t = grad_coeff[t] * (grad_scale_dev ? *grad_scale_dev : 1).
 * `kl_sum` and `kl_total` may both be NULL for a gradient-only pass. */
typedef struct bnn_kl_tensor {
  const float* mu;
  const float* rho;
  float* grad_mu;      /* optional */
  float* grad_rho;     /* optional */
  int64_t numel;
  float prior_loc;
  float prior_scale;
  float grad_coeff;
  float reserved;
} bnn_kl_tensor;
size_t bnn_kl_workspace_size(int32_t n_tensors);
int bnn_kl(const bnn_kl_tensor* tensors /* HOST array */, int32_t n_tensors,
           double* kl_sum /* device [n_tensors] or NULL */,
           float* kl_total /* device scalar or NULL: sum_t grad_coeff[t] * kl_sum[t], i.e. the
                              reference's mean-of-means / n_batches when grad_coeff[t] =
                              1 / (numel_t * n_tensors * n_batches) (loss.py:28,38) */,
           const float* grad_scale_dev, void* workspace, size_t workspace_bytes, void* stream);

/* ---- optimizer step with the KL gradient folded in (SURVEY 8f-3) ----
 * For every (mu, rho) pair: g = likelihood gradient (g_mu / g_rho, NULL = zero) + kl_coeff * dKL/d(mu, rho) with the
 * closed forms given for bnn_kl above, then torch.optim.Adam's update (no weight decay, no amsgrad; the optimizer of
 * examples/MNIST/train.py:43) of the parameters and their moment buffers, all in one pass.  `step_dev` (device scalar,
 * float) holds the number of THIS step (1, 2, ...), so that a captured CUDA graph replays with a fresh bias correction;
 * when NULL, `step_host` is used.  kl_coeff = 1 / (numel_t * n_tensors * n_batches) reproduces the gradient of
 * KLDivergence.forward (pytorch_bayesian/nn/loss.py:28,38); kl_coeff = 0 is plain Adam. */
typedef struct bnn_adam_tensor {
  float* mu;
  float* rho;
  const float* g_mu;   /* optional */
  const float* g_rho;  /* optional */
  float* m_mu;
  float* v_mu;
  float* m_rho;
  float* v_rho;
  int64_t numel;
  float prior_loc;
  float prior_scale;
  float kl_coeff;
  float reserved;
} bnn_adam_tensor;
int bnn_adam_kl_step(const bnn_adam_tensor* tensors /* HOST array */, int32_t n_tensors, float lr, float beta1, float beta2,
                     float eps, const float* step_dev, int64_t step_host, void* stream);
/* A tensor with rho == NULL (then g_rho, m_rho, v_rho are ignored and kl_coeff must be 0) is a plain parameter updated
 * by Adam alone: the deterministic layers of a model (examples/MNIST/model.py:21-27) ride in the same launch. */

/* ---- the same step with the multi-GPU gradient exchange folded in (SURVEY 8e: "one allreduce (avg) of the flat
 * [dmu, drho] gradient buffer") ----
 * One process per GPU on one NVLink node.  Every rank keeps ALL its gradients in one flat buffer that every other rank
 * has mapped into its address space (CUDA IPC / symmetric memory; `base[r]` = rank r's buffer as seen from THIS process,
 * base[rank] = the local one).  g_mu / g_rho of the table point into the local buffer; the kernel reads the element at
 * the same offset from all `world` buffers, averages in rank order (bit-identical result on every rank) and applies the
 * update: a one-shot all-reduce without a reduced gradient ever being written.  Callers bracket it with
 * bnn_peer_barrier: once after the backward pass (every rank's gradients are complete) and once after this call (every
 * rank has finished reading, the buffers may be overwritten).  Replaces the loop body's loss.backward(); optimizer.step()
 * (examples/MNIST/train.py:63-65) under data / sample parallelism. */
#define BNN_MAX_PEERS 8
typedef struct bnn_peer_grads {
  int32_t world;
  int32_t rank;
  const float* base[BNN_MAX_PEERS];
} bnn_peer_grads;
int bnn_adam_kl_step_peers(const bnn_adam_tensor* tensors /* HOST array */, int32_t n_tensors, float lr, float beta1,
                           float beta2, float eps, const float* step_dev, int64_t step_host,
                           const bnn_peer_grads* peers, void* stream);
/* In-place average of the ranks' flat gradient buffers (numel floats each) in two hops: every rank averages ITS slice
 * of the buffer over all ranks and writes the result into every rank's buffer (reduce-scatter + all-gather over peer
 * memory).  Launch between two bnn_peer_barrier calls; afterwards bnn_adam_kl_step runs on the local buffer.  Moves
 * (R - 1) / R of the buffer per direction and rank where bnn_adam_kl_step_peers pulls R - 1 whole buffers: the choice for
 * more than two ranks.  Replaces the same call site (the gradient all-reduce of SURVEY 8e). */
int bnn_peer_average(const bnn_peer_grads* peers, int64_t numel, void* stream);
/* Gathers separately stored gradients into the flat (peer-visible) buffer in one launch: dst[dst_offset .. + numel) =
 * src[0 .. numel) (src NULL: zeros).  The alternative — gradients as views of the flat buffer — costs a fill plus one
 * accumulation kernel per parameter in every backward pass. */
typedef struct bnn_pack_item {
  const float* src;
  int64_t dst_offset;      /* in floats */
  int64_t numel;
} bnn_pack_item;
int bnn_pack_gradients(const bnn_pack_item* items /* HOST array */, int32_t n_items, float* dst, void* stream);
/* Flag barrier between the ranks (one launch per rank, same point of every rank's stream; a rank that never arrives
 * traps the waiting kernels after 10 s instead of hanging).  flags[r] (HOST array of `world` pointers): rank r's flag
 * block — BNN_MAX_PEERS uint32 words in peer-visible memory, zero before first use — as mapped into this process.
 * epoch_dev: local device counter (zero before first use), advanced by every launch, so a captured graph replays it. */
int bnn_peer_barrier(uint32_t* const* flags /* HOST array */, int32_t world, int32_t rank, uint32_t* epoch_dev,
                     void* stream);

/* ---- likelihood tail: mean cross-entropy over the S Monte-Carlo predictions (SURVEY 8f-3) ----
 * Replaces the loop body `torch.stack([criterion(pred, y) for pred in preds]).mean()` with criterion =
 * CrossEntropyLoss() — examples/MNIST/train.py:59-61 — when the S predictions are the row blocks of one
 * [rows = S*labels][classes] matrix x (row pitch ldx floats): row r is scored against target[r % labels], so the B
 * labels are shared by the samples and never replicated.
 *   loss  = sum_r (logsumexp(x[r,:]) - x[r, target]) / count over the rows whose target != ignore_index
 *           (torch.nn.functional.cross_entropy, reduction 'mean'; a target outside [0, classes) that is not
 *           ignore_index makes the loss NaN instead of torch's device assert)
 *   lse   [rows]: logsumexp of every row, kept for the backward pass;  count: number of rows that counted (float).
 *   dx    = grad_loss / count * (softmax(x[r,:]) - onehot(target)), 0 for ignored rows; written, not accumulated.
 * Forward reads x once (one warp per row, online max/sum), backward reads x once and writes dx once.
 * `workspace`: bnn_mc_cross_entropy_workspace_size() bytes, 16-byte aligned, ZERO when first used; a call leaves it
 * ready for the next call on the same stream.  loss / count / grad_loss are device scalars. */
size_t bnn_mc_cross_entropy_workspace_size(void);
int bnn_mc_cross_entropy_fwd(const float* x, int64_t ldx, const int64_t* target, int64_t rows, int64_t labels,
                             int32_t classes, int64_t ignore_index, float* lse, float* loss, float* count,
                             void* workspace, size_t workspace_bytes, void* stream);
int bnn_mc_cross_entropy_bwd(const float* x, int64_t ldx, const int64_t* target, int64_t rows, int64_t labels,
                             int32_t classes, int64_t ignore_index, const float* lse, const float* count,
                             const float* grad_loss, float* dx, int64_t lddx, void* stream);

/* ---- pruning ----
 * key_i = log N(0; mu_i, sigma_i) evaluated with the exact op order of torch's Normal.log_prob
 * (torch/distributions/normal.py:87-102) on softplus(rho)+1e-10; the k largest keys get
 * mu <- 0, rho <- -30.  Replaces PruneNormal.prune_param — pytorch_bayesian/prune/prune.py:10-17.
 * Ties at the k-th key are broken towards the lowest element index (torch.topk's tie order is
 * unspecified; identical masks whenever the k-th key is unique).
 * All tensors of one call are processed by the same launches.  `mask_out` (optional, uint8
 * [numel]) receives the selection.  `keys_out` (optional) receives the keys.
 * Two exact implementations are chosen per tensor on the device: a sampled two-sweep path (a grid
 * around the k-th key from a sample; sweep 1 histograms a certified interval of every key and proves
 * which bins hold the k-th key; sweep 2 prunes what is certainly above, defers the ~1000 elements that
 * overlap and resolves those by their exact keys) and the general three-pass radix select over a key
 * workspace, which also catches every case the first declines.  NaN keys rank first, as in torch.topk. */
#define BNN_PRUNE_GENERAL 1u   /* flags: force the general radix-select path (tests; implied by keys_out) */
typedef struct bnn_prune_tensor {
  float* mu;
  float* rho;
  uint8_t* mask_out;   /* optional */
  float* keys_out;     /* optional */
  int64_t numel;
  int64_t k;
  uint32_t flags;
  uint32_t reserved;
} bnn_prune_tensor;
size_t bnn_prune_workspace_size(const bnn_prune_tensor* tensors, int32_t n_tensors);
int bnn_prune(const bnn_prune_tensor* tensors /* HOST array */, int32_t n_tensors,
              void* workspace, size_t workspace_bytes, void* stream);

/* The same selection OUT OF PLACE, in ONE sweep over (mu, rho): 8 bytes read + 8 bytes written per pair, against two
 * reads and a write in place (where nothing may be modified before the selection is proven).  mu_out / rho_out receive
 * the pruned tensors (every element is written); the inputs are read only.  Same keys, same tie rule, same masks as
 * bnn_prune.  Callers that own the parameters swap their storage for the outputs (prune/prune.py does). */
typedef struct bnn_prune_into_tensor {
  const float* mu;
  const float* rho;
  float* mu_out;
  float* rho_out;
  uint8_t* mask_out;   /* optional */
  int64_t numel;
  int64_t k;
  uint32_t flags;      /* BNN_PRUNE_GENERAL: force the general path (on a copy in the outputs) */
  uint32_t reserved;
  /* optional by-product of the same sweep (north_star: "the pruning mask reuses that same pass"): the element sum of
   * KL(N(mu, sigma) || N(prior_loc, prior_scale)) over the INPUT tensor, i.e. the per-tensor sum bnn_kl reports
   * (loss.py:16-38), formed from the sigma / log sigma the key arithmetic computes anyway.  Agrees with bnn_kl to a few
   * 1e-6 relative (approximate softplus / log2).  NULL: not computed.  numel == 0 leaves it untouched. */
  double* kl_sum_out;
  float prior_loc;
  float prior_scale;
} bnn_prune_into_tensor;
size_t bnn_prune_into_workspace_size(const bnn_prune_into_tensor* tensors, int32_t n_tensors);
int bnn_prune_into(const bnn_prune_into_tensor* tensors /* HOST array */, int32_t n_tensors, void* workspace,
                   size_t workspace_bytes, void* stream);

/* ---- self test of the prune path's certified key intervals: for every element writes the interval [lo, hi] that the
 * two sweeps of bnn_prune use to classify it, in "key2" units: key2 = (log N(0; mu, sigma) + log sqrt(2 pi)) * log2(e).
 * The exact fp32 key that torch computes (prune.py:11) must lie inside.  variant 0: the fast path taken when every
 * rho of a 4-element group is <= ln(1/4) (only valid for such rho); variant 1: the path for any rho. */
int bnn_selftest_prune_interval(const float* mu, const float* rho, int64_t numel, float* lo_out, float* hi_out,
                                int32_t variant, void* stream);

/* ---- self test of the tcgen05 path (one 128xNx32 TF32 tile against a serial fp32 loop run by
 * the same kernel's thread 0); returns BNN_OK and writes max |err| to *max_err_dev. */
int bnn_selftest_umma(float* max_err_dev, void* stream);
/* same for MN-major (transposed) operand tiles, the layout the data- and weight-gradient kernels use */
int bnn_selftest_umma_mn(float* max_err_dev, void* stream);

/* ---- test aid: force the TMA-fed forward / data-gradient contraction onto one kernel variant so that small test
 * shapes reach all of them: 0 = CTA pair (needs more than four 128-row blocks), 1 / 2 / 4 = row blocks per CTA,
 * -1 = the launcher's cost model (default).  Process-wide; not for production use. */
int bnn_debug_force_contract_variant(int32_t variant);
/* test aid, host arithmetic only: the heterogeneous tile list of the CTA-pair kernel for `samples` samples of `m_blocks`
 * 128-row blocks on `pair_slots` SM pairs (narrow layers: one column tile).  out7 = {on, n_a, s1, a1, b1, a2, b2}: samples
 * [0, s1) are cut into a1 tiles of 8 row blocks followed by b1 tiles of 6, the others into a2 / b2; n_a = number of
 * 8-block tiles; on = 0: the uniform grid is kept. */
int bnn_debug_pair_tile_plan(int32_t m_blocks, int32_t samples, int32_t pair_slots, int32_t* out7);
/* test aid, host arithmetic only: the plan of the TMA-fed TF32 weight gradient (dmu / drho of an M x N x K contraction
 * over S samples) on `sms` SMs, including a forced override.  out5 = {pair, n_chunks, chunk_blocks, units_per_cta,
 * groups}: each sample's M rows are cut into n_chunks chunks of chunk_blocks 64-row stages (the last one may be shorter),
 * a work unit is (sample, chunk) numbered u = sample * n_chunks + chunk, and CTA group z (gridDim.z = groups) walks
 * units [z * units_per_cta, min((z + 1) * units_per_cta, S * n_chunks)); pair = 1: CTA pairs over adjacent 128-row
 * n-tiles.  BNN_ERR_BAD_ARGUMENT when a forced value does not fit the shape. */
int bnn_debug_wgrad_plan(int32_t M, int32_t N, int32_t K, int32_t S, int32_t sms, int32_t* out5);
/* test aid: force parts of that plan for every later weight-gradient launch: pair (0 / 1), n_chunks, units_per_cta;
 * -1 each = the cost model's choice (default).  A forced value the shape cannot take (pair with one n-tile, an n_chunks
 * that does not give exactly that many non-empty chunks, more units per CTA than S * n_chunks, more than 65535 groups,
 * a units_per_cta whose ceil(S * n_chunks / groups) is smaller)
 * makes the launch fail with BNN_ERR_BAD_ARGUMENT instead of running another plan.  Process-wide; not for production
 * use. */
int bnn_debug_force_wgrad_plan(int32_t pair, int32_t n_chunks, int32_t units_per_cta);

#ifdef __cplusplus
}
#endif
#endif /* BNN_B200_H */
