// contract.cuh — pieces shared by the register-staged (sampled_gemm.cu) and the TMA-fed
// (sampled_gemm_tma.cu) sample-and-contract kernels.
#pragma once
#include "common.cuh"
#include "umma.cuh"

namespace bnn {
namespace contract {

using namespace umma;

constexpr int kBK = 32;                      // contraction elements per stage (one 128-byte row)
constexpr int kTileRows = 128;
constexpr int kTileBytes = kTileRows * kRowBytes;   // 16 KiB
constexpr int kProducerWarps = 8;
constexpr int kProducerThreads = kProducerWarps * 32;
constexpr int kMmaWarp = 8;
constexpr int kEpiWarp0 = 9;
constexpr int kEpiThreads = 128;
constexpr int kThreads = 13 * 32;
constexpr int kStageBudget = 208 * 1024;     // bytes of the operand ring
constexpr int kMaxStages = 8;
constexpr int kSmemAux = 2048;               // barriers, tmem pointer, bias row
constexpr int kEpiBarrier = 1;               // named barrier id of the epilogue warps

struct View {
  float* base;
  int64_t bs;
  int P;
  // phase view (TMA kernels' staged row-major drain only; pw == 0: off): row m = (img, i, j) of an img x (pimg / pw) x pw
  // grid lands at base + img * s_img + i * s_i + j * bs — one output phase of a strided transposed convolution
  int pw = 0, pimg = 0;
  int64_t s_i = 0, s_img = 0;
  // depth level of the phase view (3-d data-gradient drain only): row m = (img, a, i, j) of an img x (pimg / pplane) x
  // (pplane / pw) x pw grid lands at base + img * s_img + a * s_a + i * s_i + j * bs
  int pplane = 0;
  int64_t s_a = 0;
};
__device__ __forceinline__ float* phase_row(const View& v, int m) {
  const int img = m / v.pimg, r = m - img * v.pimg, i = r / v.pw, j = r - i * v.pw;
  return v.base + static_cast<int64_t>(img) * v.s_img + static_cast<int64_t>(i) * v.s_i + static_cast<int64_t>(j) * v.bs;
}
// the offset within an image in 32 bits (an image below 2^31 floats, checked by the host)
__device__ __forceinline__ float* phase_row3(const View& v, int m) {
  const int img = m / v.pimg, r = m - img * v.pimg, a = r / v.pplane, r2 = r - a * v.pplane, i = r2 / v.pw,
            j = r2 - i * v.pw;
  return v.base + static_cast<int64_t>(img) * v.s_img +
         (a * static_cast<int>(v.s_a) + i * static_cast<int>(v.s_i) + j * static_cast<int>(v.bs));
}
__device__ __forceinline__ int64_t view_off(const View& v, int m, int n) {
  if (v.P == 1) return static_cast<int64_t>(m) * v.bs + n;
  const int b = m / v.P, p = m - b * v.P;
  return static_cast<int64_t>(b) * v.bs + static_cast<int64_t>(n) * v.P + p;
}

// eps source of one (tensor, sample): injected array or the Philox stream
struct EpsSrc {
  const float* inj;   // already offset to the sample's [numel] block, or nullptr
  RngKey key;
  uint32_t sample;
};
// rank-one sign noise (Flipout): element idx = (n, k) of a [rows][cols] weight matrix (plus the slice offset)
__device__ __forceinline__ float eps_rank_one(const EpsSrc& e, int64_t idx) {
  const int64_t el = idx + static_cast<int64_t>(e.key.elem_offset);
  const int64_t n = el / e.key.cols;
  const int k = static_cast<int>(el - n * e.key.cols);
  return __ldg(e.key.row_sign + static_cast<int64_t>(e.sample) * e.key.rows + n) *
         __ldg(e.key.col_sign + static_cast<int64_t>(e.sample) * e.key.cols + k);
}
// kSigns: 1 = the launch uses rank-one sign noise, 0 = it does not (the TMA kernels are instantiated per case: the sign
// vectors' pointers kept live across the generator loop cost registers those kernels do not have), -1 = decided at run time
template <int kSigns = -1>
__device__ __forceinline__ float4 eps_vec4(const EpsSrc& e, int64_t idx) {   // idx % 4 == 0
  if (e.inj != nullptr) return __ldg(reinterpret_cast<const float4*>(e.inj + idx));
  if (kSigns == 1 || (kSigns == -1 && e.key.row_sign != nullptr)) {
    if ((e.key.cols & 3) == 0 && (e.key.elem_offset & 3u) == 0) {      // the four elements share a row
      const int64_t el = idx + static_cast<int64_t>(e.key.elem_offset);
      const int64_t n = el / e.key.cols;
      const int k = static_cast<int>(el - n * e.key.cols);
      const float r = __ldg(e.key.row_sign + static_cast<int64_t>(e.sample) * e.key.rows + n);
      const float* c = e.key.col_sign + static_cast<int64_t>(e.sample) * e.key.cols + k;
      return make_float4(r * __ldg(c), r * __ldg(c + 1), r * __ldg(c + 2), r * __ldg(c + 3));
    }
    return make_float4(eps_rank_one(e, idx), eps_rank_one(e, idx + 1), eps_rank_one(e, idx + 2), eps_rank_one(e, idx + 3));
  }
  return eps4(e.key, e.sample, static_cast<uint32_t>(idx >> 2));
}
template <int kSigns = -1>
__device__ __forceinline__ float eps_one(const EpsSrc& e, int64_t idx) {
  if (e.inj != nullptr) return __ldg(e.inj + idx);
  if (kSigns == 1 || (kSigns == -1 && e.key.row_sign != nullptr)) return eps_rank_one(e, idx);
  return eps1(e.key, e.sample, static_cast<uint64_t>(idx));
}

__device__ __forceinline__ int mma_n(int valid) {   // MMA N extent: multiple of 16 in [16, 128]
  int n = (valid + 15) & ~15;
  return n < 16 ? 16 : (n > 128 ? 128 : n);
}

// one 16-column chunk of an output row -> global memory through a view
__device__ __forceinline__ void store_chunk(const View& out, int m, int n, int N, const float* v,
                                            bool vec) {
  if (out.P == 1) {
    float* dst = out.base + static_cast<int64_t>(m) * out.bs + n;
    if (vec && n + 16 <= N) {
#pragma unroll
      for (int j = 0; j < 16; j += 4)
        *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (n + j < N) dst[j] = v[j];
    }
  } else {
    const int b = m / out.P, p = m - b * out.P;
    float* dst = out.base + static_cast<int64_t>(b) * out.bs + p;
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (n + j < N) dst[static_cast<int64_t>(n + j) * out.P] = v[j];
  }
}

__device__ __forceinline__ void red_add4(float* dst, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(dst), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}

// the same chunk ADDED to a row-major output (several CTAs contribute partial sums over the samples)
__device__ __forceinline__ void add_chunk(const View& out, int m, int n, int N, const float* v, bool vec) {
  float* dst = out.base + static_cast<int64_t>(m) * out.bs + n;
  if (vec && n + 16 <= N) {
#pragma unroll
    for (int j = 0; j < 16; j += 4) red_add4(dst + j, v[j], v[j + 1], v[j + 2], v[j + 3]);
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (n + j < N) atomicAdd(dst + j, v[j]);
  }
}


// ---- TMA-fed TF32 kernels (sampled_gemm_tma.cu).  Each returns kNotEligible when the request does not meet
// its alignment / layout requirements; the caller then takes the register-staged kernels.
constexpr int kNotEligible = -1;
int tma_fwd(const float* a, int64_t lda, int64_t a_sample_stride, const float* mu_w, const float* sigma_w,
            const float* mu_b, const float* sigma_b, const float* eps_w, const float* eps_b, bnn_view y,
            int64_t y_sample_stride, int M, int N, int K, int S, uint32_t sample_begin, const bnn_rng* rng_w,
            const bnn_rng* rng_b, cudaStream_t st);
int tma_dgrad(bnn_view dy, int64_t dy_sample_stride, const float* mu_w, const float* sigma_w, const float* eps_w,
              float* da, int64_t lda, int64_t a_sample_stride, int M, int N, int K, int S, uint32_t sample_begin,
              const bnn_rng* rng_w, cudaStream_t st);
int tma_wgrad(bnn_view dy, int64_t dy_sample_stride, const float* a, int64_t lda, int64_t a_sample_stride,
              const float* rho_w, const float* eps_w, float* dmu_w, float* drho_w, int M, int N, int K, int S,
              uint32_t sample_begin, const bnn_rng* rng_w, cudaStream_t st);
// implicit-GEMM convolution (NHWC activations through an im2col tensor map, weights [Cout][KH][KW][C]).  Geometry of
// the launchers: a 3-d convolution (vol: NDHWC tensors, rank-5 maps, the kMode 3 kernels) or a 2-d one as depth 1
// (D = OD = KD = sd = dd = 1, pd = 0: rank-4 maps, the kMode 1 kernels)
struct ConvGeom {
  bnn_conv3d_nhwc g;
  bool vol;
};
ConvGeom conv_geom_2d(const bnn_conv2d_nhwc& g);
int tma_conv_fwd(const float* x, int64_t x_sample_stride, const float* mu_w, const float* sigma_w, const float* mu_b,
                 const float* sigma_b, const float* eps_w, const float* eps_b, bnn_view y, int64_t y_sample_stride,
                 const ConvGeom& g, int S, uint32_t sample_begin, const bnn_rng* rng_w, const bnn_rng* rng_b,
                 cudaStream_t st);
// the weight gradient of a conv layer takes (dy, x), that of a transposed conv its conv view's operands (x, dy)
int tma_conv_wgrad(const float* dy, bool shared_dy, const float* a, bool shared_a, const float* rho_w, const float* eps_w,
                   float* dmu_w, float* drho_w, const ConvGeom& g, int S, uint32_t sample_begin,
                   const bnn_rng* rng_w, cudaStream_t st);
// transposed-filter gather: the stride-1 conv input gradient (x = dy, sum_samples for a shared input) and the forward of a
// transposed convolution in its conv view's geometry (see bnn_b200.h; one launch per output phase); input gradient of a
// transposed convolution = the conv view's forward
int tma_conv_gather(const float* x, bool shared_x, const float* mu_w, const float* sigma_w, const float* mu_b,
                    const float* sigma_b, const float* eps_w, const float* eps_b, float* y, int64_t y_sample_stride,
                    bool sum_samples, const ConvGeom& g, int S, uint32_t sample_begin, const bnn_rng* rng_w,
                    const bnn_rng* rng_b, cudaStream_t st);
int tma_conv_transpose_dgrad(const float* dy, const float* mu_w, const float* sigma_w, const float* eps_w, float* dx,
                             int64_t x_sample_stride, const ConvGeom& g, int S, uint32_t sample_begin,
                             const bnn_rng* rng_w, cudaStream_t st);
// host: the phase plan, 7 ints per phase dimension (14 per phase in 2-d, 21 in 3-d)
int conv_transpose_phases(const ConvGeom& g, int32_t* out, int max_phases);
// host: geometry part of the 3-d transposed convolution's eligibility (channels, strides, every conv-view and phase corner)
bool conv_transpose_ok(const ConvGeom& g);
int tma_selftest(float* max_err_dev, cudaStream_t st);
int tma_pair_tile_plan(int m_blocks, int S, int slots, int32_t* out7);   // test aid: TilePlan fields {on, n_a, s1, a1, b1, a2, b2}
int tma_force_variant(int variant);   // test aid: 0 = CTA pair, 1 / 2 / 4 = row blocks per CTA, -1 = cost model (default)
// host: the weight-gradient launch plan on `sms` SMs (including a forced override); the launcher runs exactly this plan
struct WgradPlan {
  int pair;           // CTA pairs over adjacent n-tiles
  int n_chunks;       // M-chunks per sample; a work unit = (sample, chunk)
  int chunk_blocks;   // 64-row stages per chunk (the last chunk may be shorter)
  int per;            // work units per CTA: ceil(S * n_chunks / groups), as the kernel derives it
  int groups;         // gridDim.z
};
int wgrad_plan(int M, int N, int K, int S, int sms, WgradPlan* plan);
int tma_force_wgrad_plan(int pair, int n_chunks, int units_per_cta);   // test aid: -1 = the cost model's choice
int tma_stage_counters(unsigned long long* out8, int reset);  // profiling builds only: CTA timeline of the pair kernels
int tma_wait_counters(unsigned long long* out8, int reset);   // profiling builds (-DBNN_PROFILE_WAITS) only

}  // namespace contract
}  // namespace bnn
