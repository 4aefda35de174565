// sampled_gemm_tma.cu — TMA-fed TF32 variants of the sample-and-contract kernels for aligned row-major operands (the
// large-shape path: BASELINE config C4 and the im2col matrices of the conv layers).
//
//   forward / data gradient   Activations (or dY) arrive by TMA (cp.async.bulk.tensor.3d, 128B swizzle, TF32 conversion in
//     contract_tma_kernel     the copy engine): the MB tiles of a k-block land in one of two slot groups on one
//     contract_pair_kernel    transaction barrier.  Sixteen generator warps in four groups do nothing but produce
//                             W_s = mu + sigma * eps_s (Philox) — group j owns weight slot j and the k-blocks
//                             it % 4 == j, so four tiles are in flight.  One thread issues tcgen05.mma and ONE
//                             tcgen05.commit per k-block ("k-block consumed": frees the weight slot and, two k-blocks
//                             later, the activation group).  Four warps drain TMEM.  The data gradient stores the
//                             generated tile in the MN-major canonical layout, i.e. in W's natural [n][k] orientation.
//                             The pair kernel runs the same protocol over a cluster of two CTAs (cta_group::2): each
//                             generates half of the weight tile, the leader issues M = 256 MMAs and multicast commits.
//   weight gradient           BOTH operands (dY^T and A^T) are MN-major tiles loaded by TMA — no thread touches
//     wgrad_tma_kernel        operand data; twelve epilogue warps regenerate eps per work unit and keep the running
//                             sums of G_s and G_s o eps_s in TMEM.
// Eligibility (else the caller uses sampled_gemm.cu): TF32 precision, row-major operands (view P == 1 for everything
// that is READ), 16-byte aligned bases and leading dimensions.
// Profiling builds (-DBNN_PROFILE_WAITS) add wait-cycle counters and elimination switches (BNN_EXP_FLAGS).
#include <cuda.h>

#include <cstdlib>
#include <mutex>

#include <algorithm>
#include <array>
#include <vector>

#include "contract.cuh"

namespace bnn {
namespace contract {
#ifdef BNN_PROFILE_WAITS
// profiling builds: cycles spent waiting, summed over CTAs: [0] kernel, [1] MMA on full_w, [2] MMA on full_a,
// [3] generator warp 0 on empty_w, [4] TMA thread on the consumed barrier, [5] CTAs
__device__ unsigned long long g_wait_cycles[8];
// CTA timeline of the CTA-pair kernels, cycles since the CTA's first instruction summed over CTAs: [0] prologue done,
// [1] generator warp 0 done, [2] accumulator complete (epilogue warp 0), [3] epilogue done, [4] CTA end, [5] CTAs;
// [6] / [7] globaltimer (ns) of the first CTA start / last CTA end
__device__ unsigned long long g_stage_cycles[8];
#define BNN_STAGE(i, t0) atomicAdd(&g_stage_cycles[i], (unsigned long long)(clock64() - (t0)))
#define BNN_T0() const long long _t0 = clock64()
#define BNN_ACC(var) var += clock64() - _t0
#else
#define BNN_T0()
#define BNN_ACC(var)
#endif
namespace {

constexpr int kASlots = 8;                   // activation tile slots (16 KiB each): two k-block groups of up to 4 tiles
constexpr int kWSlots = 4;                   // generated weight tile ring (the k-block bookkeeping assumes 4)
// warp roles of the forward / data-gradient kernel: 16 weight generators (the Philox chains are latency bound:
// four warps per scheduler hide them), MMA issuer, four epilogue warps (TMEM lane quarter = warp % 4), TMA issuer
constexpr int kGenWarps = 16;
constexpr int kGenGroups = 4;                       // generator groups: group j produces the k-blocks it % 4 == j into
constexpr int kGroupWarps = kGenWarps / kGenGroups; // weight slot j, so four tiles are in flight at different phases
constexpr int kGroupThreads = kGroupWarps * 32;     // (one tile's latency — loads, Philox chain — is hidden by the others)
constexpr int kMmaWarpT = kGenWarps;
constexpr int kEpiWarp0T = kGenWarps + 1;
constexpr int kTmaWarp = kGenWarps + 5;
constexpr int kThreadsTma = (kGenWarps + 6) * 32;
constexpr uint32_t kMnLbo = 4096, kMnSbo = 512;    // MN-major 128 x 32 tile: 4 groups of 32 MN, 8 atoms of 4 K-rows
constexpr uint32_t kMnKStep = 2 * kMnSbo;            // one UMMA K-step (8 TF32) = two 4-row atoms

// ---------------------------------------------------------------------------------------------- tensor maps
using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                              const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                              CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn encode_fn() {
  static EncodeFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  });
  return fn;
}

// fp32 matrix [samples][rows][cols] (row stride ld, sample stride ss floats) -> 3-d map with a box of
// 32 columns x box_rows rows, 128B swizzle, TF32 conversion, zero fill outside [cols) x [rows) x [samples)
int make_map(CUtensorMap* map, const float* base, int64_t cols, int64_t rows, int64_t samples, int64_t ld, int64_t ss,
             int box_rows, bool mn_major = false) {
  EncodeFn fn = encode_fn();
  if (fn == nullptr) return kNotEligible;
  const cuuint64_t dims[3] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows),
                              static_cast<cuuint64_t>(samples)};
  const cuuint64_t strides[2] = {static_cast<cuuint64_t>(ld) * 4u,
                                 static_cast<cuuint64_t>(samples > 1 ? ss : ld * rows) * 4u};
  const cuuint32_t box[3] = {32u, static_cast<cuuint32_t>(box_rows), 1u};
  const cuuint32_t estr[3] = {1u, 1u, 1u};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE,
                        mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return kNotEligible;
  return BNN_OK;
}

// NHWC fp32 tensor [n_imgs][H][W][C] seen through the filter's bounding box (cuTensorMapEncodeIm2col): a load delivers
// `box_pixels` base pixels (traversed w, h, n with the given stride, starting at the lower corner) x 32 channels, TF32
// conversion, zero fill outside the image.  lower / upper corner: first base pixel and (last base pixel + 1 - extent).
using EncodeIm2colFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);
EncodeIm2colFn encode_im2col_fn() {
  static EncodeIm2colFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeIm2colFn>(p);
  });
  return fn;
}

// Depth: the rank-5 map of an NDHWC tensor [n_imgs][D][H][W][C] (3-d convolutions, vol); without it the rank-4 map.
struct Im2colDepth {
  bool vol;
  int64_t D;
  int lower, upper, stride;
};
int make_im2col_map(CUtensorMap* map, const float* base, int64_t C, int64_t W, int64_t H, int64_t n_imgs, int lower_w,
                    int lower_h, int upper_w, int upper_h, int stride_w, int stride_h, int box_pixels, bool mn_major,
                    const Im2colDepth& dep = Im2colDepth{false, 1, 0, 0, 1}) {
  EncodeIm2colFn fn = encode_im2col_fn();
  if (fn == nullptr) return kNotEligible;
  const int64_t D = dep.vol ? dep.D : 1;
  const cuuint32_t rank = dep.vol ? 5u : 4u;
  const cuuint64_t dims[5] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H),
                              static_cast<cuuint64_t>(dep.vol ? D : n_imgs), static_cast<cuuint64_t>(n_imgs)};
  const cuuint64_t strides[4] = {static_cast<cuuint64_t>(C) * 4u, static_cast<cuuint64_t>(W * C) * 4u,
                                 static_cast<cuuint64_t>(H * W * C) * 4u, static_cast<cuuint64_t>(D * H * W * C) * 4u};
  const int lower[3] = {lower_w, lower_h, dep.lower}, upper[3] = {upper_w, upper_h, dep.upper};
  const cuuint32_t estr[5] = {1u, static_cast<cuuint32_t>(stride_w), static_cast<cuuint32_t>(stride_h),
                              dep.vol ? static_cast<cuuint32_t>(dep.stride) : 1u, 1u};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, rank, const_cast<float*>(base), dims, strides, lower, upper,
                        32u, static_cast<cuuint32_t>(box_pixels), estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return kNotEligible;
  // Known driver issue (CUDA <= 13.1, the workaround CUTLASS applies in cute/atom/copy_traits_sm90_im2col.hpp): for tensors
  // smaller than 128 KiB the encoder sets bit 21 of the descriptor's second word, which makes the copy engine misread the
  // extent; clear it (rank 4 and rank 5 alike).
  int driver = 0;
  if (cudaDriverGetVersion(&driver) == cudaSuccess && driver <= 13010 && n_imgs * D * H * W * C * 4 < 131072)
    reinterpret_cast<uint64_t*>(map)[1] &= ~(1ull << 21);
  return BNN_OK;
}

bool tma_ok(const void* base, int64_t ld, int64_t ss) {
  return aligned16(base) && ld % 4 == 0 && ss % 4 == 0 && ld > 0;
}

// ---------------------------------------------------------------------------------------------- forward / dgrad
// Implicit-GEMM addressing of the TMA-loaded operand (conv layers): the operand is never an im2col MATRIX, it is the NHWC
// tensor itself seen through an im2col tensor map; row m of the GEMM is the pixel (img, p, q) of a P = rows x OW grid
// (output pixels for forward / weight gradient, input pixels for the data gradient), k-block rb is (filter tap, 32
// channels).  on == 0: plain row-major matrix; 1: 2-d (rank-4 map), 2: 3-d (rank-5 map, kMode 3 kernels).
struct ConvCoords {
  int on;
  int P, OW;                // pixel grid of the GEMM rows
  int imgs;                 // images per sample: n coordinate = sample * imgs + img
  int sh, sw;               // traversal stride (the conv stride; 1 for the data gradient)
  int lh, lw;               // lower corner: base pixel of grid pixel 0
  int dh, dw;               // dilation
  int KW, taps;             // filter width, KH * KW
  int cblocks;              // 32-channel k-blocks per tap (channels of the LOADED tensor / 32)
  int w_rows;               // data gradient: rows of the weight matrix (Cout); its row pitch is wtaps * K floats
  int chans;                // channels of the loaded tensor (weight gradient: groups beyond K load channel `chans` = zeros)
  // data gradient: flipped tap t = (jh, jw) of the walk (jh = t / KW) is the weight's tap (tkh - jh tdh, tkw - jw tdw) of a
  // wtaps = KH x wKW filter.  Stride 1: every tap (tkh = KH - 1, tdh = 1, ...); one phase of a strided transposed
  // convolution: the taps of that phase only, tdh = sh / gcd(sh, dh) apart
  int wtaps, wKW, tkh, tkw, tdh, tdw;
  // 3-d convolutions (kMode 3, rank-5 map): row m = (img, d, h, w), HW pixels per depth plane; depth stride, lower corner
  // and dilation; KH x KW = KHW walked taps per depth plane; data gradient: walked tap (jd, jh, jw) is the weight's tap
  // (tkd - jd tdd, tkh - jh tdh, tkw - jw tdw) of a filter wKH high
  int HW, sd, ld, dd, KH, KHW, tkd, tdd, wKH;
};
__device__ __forceinline__ int64_t conv_dgrad_tap(const ConvCoords& c, int tapf) {
  const int jh = tapf / c.KW, jw = tapf - jh * c.KW;
  return static_cast<int64_t>((c.tkh - jh * c.tdh) * c.wKW + c.tkw - jw * c.tdw);
}
__device__ __forceinline__ int64_t conv_dgrad_tap3d(const ConvCoords& c, int tapf) {
  const int jd = tapf / c.KHW, r = tapf - jd * c.KHW, jh = r / c.KW, jw = r - jh * c.KW;
  return static_cast<int64_t>(((c.tkd - jd * c.tdd) * c.wKH + c.tkh - jh * c.tdh) * c.wKW + c.tkw - jw * c.tdw);
}
__device__ __forceinline__ void conv_pixel(const ConvCoords& c, int m, int smp, int* w, int* h, int* n) {
  const int img = m / c.P, rem = m - img * c.P;
  const int ph = rem / c.OW, q = rem - ph * c.OW;
  *w = q * c.sw + c.lw;
  *h = ph * c.sh + c.lh;
  *n = smp * c.imgs + img;
}
__device__ __forceinline__ void conv_pixel3d(const ConvCoords& c, int m, int smp, int* w, int* h, int* d, int* n) {
  const int img = m / c.P, rem = m - img * c.P;
  const int pd = rem / c.HW, r2 = rem - pd * c.HW;
  const int ph = r2 / c.OW, q = r2 - ph * c.OW;
  *w = q * c.sw + c.lw;
  *h = ph * c.sh + c.lh;
  *d = pd * c.sd + c.ld;
  *n = smp * c.imgs + img;
}

// Heterogeneous tile list of the CTA-pair kernel (narrow layers whose uniform 1024-row tiles need between one and two
// waves): a sample's rows are cut into `a` tiles of 8 row blocks followed by `b` tiles of 6; samples [0, s1) use (a1, b1),
// the others (a2, b2).  The grid lists every 8-block tile first, then the 6-block ones, so that a pair slot runs one of
// each instead of two full ones (C3 conv forward: 74 + 72 tiles on 74 slots: 1.75 wave-equivalents instead of 2).
struct TilePlan {
  int on;
  int n_a;                  // number of 8-block tiles of the launch
  int s1, a1, b1, a2, b2;
};

struct TmaContractParams {
  TilePlan plan;
  CUtensorMap map_l;        // fwd: activations [S or 1][M][K]; dgrad: dY [S][M][N]; conv: the NHWC tensor (im2col map)
  ConvCoords conv;
  int64_t w_numel;          // elements of the weight tensor (injected eps: stride between samples)
  View out;                 // fwd: y view; dgrad: da as a row-major view
  int64_t out_sample_stride;
  const float* mu_w;
  const float* sigma_w;
  const float* eps_w;
  const float* mu_b;
  const float* sigma_b;
  const float* eps_b;
  int M, N, K, S;
  uint32_t sample_begin;
  bnn_rng rng_w, rng_b;
  int shared_l;             // all samples read sample 0 of the L operand (shared activations)
  int sum_samples;          // dgrad with shared activations: one output, summed over the samples
  int z_per;                // sum_samples: samples per CTA (grid.z = sample groups); more than one group -> the partial
  int atomic_out;           //   sums are ADDED to the (zeroed) output
  int vec_out;
  int exp_flags;            // profiling builds: 1 = skip weight generation, 2 = eps read from memory; single CTA only:
                            //   4 = skip TMA loads, 8 = skip MMA issue
};

struct TmaPipe {
  uint64_t* full_a;      // [2]        TMA transaction barriers: the MB activation tiles of one k-block group
  uint64_t* full_w;      // [kWSlots]  one arrival per warp of the generator group that owns the slot
  uint64_t* empty_w;     // [kWSlots]  "k-block consumed": one tcgen05.commit per k-block
  uint64_t* accum_full;  // accumulators complete
  uint32_t* tmem_slot;
  float* aux;            // 128 floats: the sampled bias row of this CTA's columns
  uint32_t ring_a, ring_w;
};

__device__ __forceinline__ TmaPipe carve_tma(uint8_t* smem_raw) {
  TmaPipe p;
  p.full_a = reinterpret_cast<uint64_t*>(smem_raw);
  p.full_w = p.full_a + 2;
  p.empty_w = p.full_w + kWSlots;
  p.accum_full = p.empty_w + kWSlots;
  p.tmem_slot = reinterpret_cast<uint32_t*>(p.accum_full + 1);
  p.aux = reinterpret_cast<float*>(smem_raw + 512);
  const uint32_t base = smem_u32(smem_raw) + kSmemAux;
  p.ring_a = (base + 1023u) & ~1023u;
  p.ring_w = p.ring_a + kASlots * kTileBytes;
  return p;
}

// W_s = mu + sigma * eps_s for a (kRows x 32) piece of the weight matrix, written as an operand tile by ONE generator
// group (kGroupThreads threads, four float4 per thread and trip: all loads first, then the Philox chains).
//   kMnMajor = false: K-major tile, tile rows = n (kRows of them), columns = k          (forward)
//   kMnMajor = true : MN-major tile, K-rows = n (32), MN = k (kRows of them)            (data gradient)
// Element (n, k) of the weight matrix lives at n * ldw + woff + k (ldw = K, woff = 0 for a plain [N][K] matrix; the
// conv data gradient walks the (o, kh, kw, c) tensor with n = o, ldw = taps * C, woff = tap * C, k = c).
template <int kRows, bool kMnMajor, int kSigns>
__device__ __forceinline__ void gen_w_tile(uint32_t tile, const float* __restrict__ mu, const float* __restrict__ sigma,
                                           const EpsSrc& eps, int n0, int N, int k0, int K, int tid, int64_t ldw,
                                           int64_t woff) {
  constexpr int kItems = kRows * 8;                       // float4 items
  constexpr int kTrips = kItems / (4 * kGroupThreads);
  static_assert(kItems % (4 * kGroupThreads) == 0, "tile does not divide over the generator group");
#pragma unroll 1
  for (int trip = 0; trip < kTrips; ++trip) {
    float4 m[4], sg[4];
    int64_t idx[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int item = (trip * 4 + u) * kGroupThreads + tid;
      int n, k;
      if (!kMnMajor) { n = n0 + (item >> 3); k = k0 + ((item & 7) << 2); }
      else { n = n0 + item / (kRows / 4); k = k0 + ((item % (kRows / 4)) << 2); }
      idx[u] = -1;
      if (n < N && k < K) {
        idx[u] = static_cast<int64_t>(n) * ldw + woff + k;
        m[u] = __ldg(reinterpret_cast<const float4*>(mu + idx[u]));
        sg[u] = __ldg(reinterpret_cast<const float4*>(sigma + idx[u]));
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int item = (trip * 4 + u) * kGroupThreads + tid;
      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      if (idx[u] >= 0) {
        const float4 e = eps_vec4<kSigns>(eps, idx[u]);
        w.x = fmaf(sg[u].x, e.x, m[u].x);
        w.y = fmaf(sg[u].y, e.y, m[u].y);
        w.z = fmaf(sg[u].z, e.z, m[u].z);
        w.w = fmaf(sg[u].w, e.w, m[u].w);
      }
      uint32_t off;
      if (!kMnMajor) off = tile_offset(item >> 3, item & 7);
      else off = tile_offset_mn((item % (kRows / 4)) << 2, item / (kRows / 4), kMnLbo, kMnSbo);
      sts128(tile + off, to_tf32(w.x), to_tf32(w.y), to_tf32(w.z), to_tf32(w.w));
    }
  }
}

// ---------------------------------------------------------------------------------------------- staged epilogue
// A TMEM lane is an output row, so an epilogue thread that stores its own 16-column chunk writes 16 bytes of 32
// different rows per warp instruction: 32 memory wavefronts per 512 bytes (measured: 25 k cycles to drain the 512 x 128
// accumulator of one CTA, a quarter of a C3 conv tile's time).  Each epilogue warp therefore passes its 32 rows through
// a private shared-memory buffer, 64 columns at a time, and writes whole row segments:
//   row-major output (view P == 1): staging rows of 64 + 4 floats (float4 writes of a quarter warp hit 32 different
//     banks); two rows per store instruction, 256 contiguous bytes each;
//   NCHW output (P = OH*OW, P % 4 == 0): staging [column][32 rows + 4]; four rows of a lane's group are four consecutive
//     pixels of one image, i.e. one aligned float4 of out[img][n][p..p+3]; a store instruction covers 4 columns x 8 row
//     groups: for P = 16 two runs of 256 contiguous bytes (was: two runs of 64 bytes per scalar store).
// kStageWarpBytes per warp; the kernels alias the operand ring (dead once the accumulator is complete).
constexpr int kStageWarpBytes = 64 * 36 * 4;     // 9216: [64 columns][32 + 4] floats; the row-major form needs 32 x 68 x 4 = 8704
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ bool stage_eligible(const View& out, bool vec_out, int cols_here) {
  if ((cols_here & 3) != 0 || (reinterpret_cast<uintptr_t>(out.base) & 15) != 0 || (out.bs & 3) != 0) return false;
  return out.P == 1 ? vec_out : (out.P & 3) == 0;
}
// Halves [h_begin, h_end) (64 columns each) of one 128-row block, drained by one warp (TMEM lanes [32 quad, +32), rows
// m0 .. m0 + 31 of the output, columns col0 .. col0 + cols_here): two tcgen05.ld per round trip, then (+ bias) ->
// staging -> coalesced stores / adds.
// kPhase: the output may be a phase view (View::pw; conv data-gradient instantiations only — the others keep the plain
// row addressing); 2: with the depth level (3-d conv data gradient)
template <bool kBias, int kPhase = 0>
__device__ __forceinline__ void drain_block_staged(uint32_t taddr, uint32_t stage, const float* aux, const View& out,
                                                   int m0, int M, int col0, int cols_here, int lane, bool add,
                                                   int h_begin = 0, int h_end = 2) {
  const bool nchw = out.P != 1;
  // per-lane destination of the write-out phase
  float* dst;
  bool ok;
  if (!nchw) {
    dst = out.base + static_cast<int64_t>(m0 + (lane >> 4)) * out.bs + col0 + ((lane & 15) << 2);
    ok = true;
  } else {
    const int m = m0 + ((lane & 7) << 2);                  // first of the lane's four rows (one image: P % 4 == 0)
    const int b = m / out.P, px = m - b * out.P;
    dst = out.base + static_cast<int64_t>(b) * out.bs + static_cast<int64_t>(col0 + (lane >> 3)) * out.P + px;
    ok = m < M;
  }
  for (int h = h_begin; h < h_end && h * 64 < cols_here; ++h) {
#pragma unroll 1
    for (int pr = 0; pr < 2 && (h * 4 + pr * 2) * 16 < cols_here; ++pr) {      // two 16-column chunks per TMEM round trip
      uint32_t r[2][16];
      tmem_ld16_nowait(taddr + (h * 4 + pr * 2) * 16, r[0]);
      if ((h * 4 + pr * 2 + 1) * 16 < cols_here) tmem_ld16_nowait(taddr + (h * 4 + pr * 2 + 1) * 16, r[1]);
      tmem_ld_wait();
#pragma unroll
      for (int q2 = 0; q2 < 2; ++q2) {
        const int cc = pr * 2 + q2;
        if ((h * 4 + cc) * 16 >= cols_here) break;
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[q2][j]);
        if (kBias) {
          const float4* a4 = reinterpret_cast<const float4*>(aux + (h * 4 + cc) * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 q = a4[j];
            v[4 * j] += q.x; v[4 * j + 1] += q.y; v[4 * j + 2] += q.z; v[4 * j + 3] += q.w;
          }
        }
        if (!nchw) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            sts128(stage + lane * 272 + cc * 64 + j * 16, __float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]),
                   __float_as_uint(v[4 * j + 2]), __float_as_uint(v[4 * j + 3]));
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) sts32(stage + ((cc * 16 + j) * 36 + lane) * 4, __float_as_uint(v[j]));
        }
      }
    }
    __syncwarp();
    const int cols_half = cols_here - h * 64 < 64 ? cols_here - h * 64 : 64;
    if (!nchw) {
      const int c4 = lane & 15;
#pragma unroll 8
      for (int i = 0; i < 16; ++i) {
        const int row = 2 * i + (lane >> 4);
        if (c4 * 4 < cols_half && m0 + row < M) {
          const float4 q = lds128(stage + row * 272 + c4 * 16);
          float* d = (!kPhase || out.pw == 0) ? dst + static_cast<int64_t>(2 * i) * out.bs + h * 64
                                              : (kPhase == 2 ? phase_row3(out, m0 + row) : phase_row(out, m0 + row)) +
                                                    col0 + (c4 << 2) + h * 64;
          if (add) red_add4(d, q.x, q.y, q.z, q.w);
          else *reinterpret_cast<float4*>(d) = q;
        }
      }
    } else {
      const int rg = lane & 7, ns = lane >> 3;
#pragma unroll 8
      for (int i = 0; i < 16; ++i) {
        const int n = i * 4 + ns;
        if (n < cols_half && ok) {
          const float4 q = lds128(stage + (n * 36 + rg * 4) * 4);
          float* d = dst + static_cast<int64_t>(h * 64 + i * 4) * out.P;
          if (add) red_add4(d, q.x, q.y, q.z, q.w);
          else *reinterpret_cast<float4*>(d) = q;
        }
      }
    }
    __syncwarp();
  }
}
// The accumulator of one CTA (mb_count row blocks of 128 rows x cols_here columns) drained by kDrainPerQuad warps per
// TMEM lane quarter — the epilogue warp of the quarter (idx 0) and generator warps with the same warp % 4, idle once
// their loop has ended: work items = (row block, 64-column half), item i goes to warp i % kDrainPerQuad.
constexpr int kDrainPerQuad = 4;
constexpr int kDrainThreads = 4 * kDrainPerQuad * 32;
constexpr int kDrainBarrier = 2;
template <bool kBias, int kPhase = 0>
__device__ __forceinline__ void drain_tile_shared(uint32_t tmem, uint32_t stage_base, const float* aux, const View& out,
                                                  int row0, int M, int mb_count, int col0, int cols_here, int quad,
                                                  int idx, int lane, bool add) {
  const uint32_t stage = stage_base + static_cast<uint32_t>(idx * 4 + quad) * kStageWarpBytes;
  const int halves = (cols_here + 63) / 64;
  for (int item = idx; item < mb_count * halves; item += kDrainPerQuad) {
    const int mb = item / halves, h = item - mb * halves;
    if (row0 + mb * 128 >= M) break;
    drain_block_staged<kBias, kPhase>(tmem + (static_cast<uint32_t>(quad * 32) << 16) + mb * 128, stage, aux, out,
                              row0 + mb * 128 + quad * 32, M, col0, cols_here, lane, add, h, h + 1);
  }
}

// Forward / data gradient.  kPair: the same contraction over a cluster of two CTAs (cta_group::2): the pair computes
// 2 x MB x 128 output rows against ONE 128-column weight tile of which each CTA generates only its half (64 n-rows forward
// / 64 k-columns dgrad) — half the Philox work per SM and per MMA cycle.  Each CTA loads its own activation tiles by TMA
// (transaction bytes land on the LEADER's barrier), the generator warps of the peer arrive on the leader's barrier through
// the cluster address space, the leader's single MMA thread issues tcgen05.mma.cta_group::2 (M = 256) and frees the slots
// of BOTH CTAs with multicast commits.  Epilogue: every CTA drains its own TMEM.
// The pair's weight ring holds kWSlots 8 KiB half tiles.  Eight slots were measured: the generators wait less (19 k
// instead of 26 k cycles per C3 tile), the MMA thread's 8.8 k cycles of waiting for weights do not move — they are the
// cold start of a tile (first mu / sigma loads, instruction cache), not a lack of slack in the ring.
constexpr int kHalfTileBytes = kTileBytes / 2;

// One body, contract_body.inc (see there why it is included rather than called)
template <int MB, bool kDgrad, int kMode>
__global__ void __launch_bounds__(kThreadsTma, 1) contract_tma_kernel(const __grid_constant__ TmaContractParams p) {
  constexpr bool kPair = false;
#include "contract_body.inc"
}
template <int MB, bool kDgrad, int kMode>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreadsTma, 1)
contract_pair_kernel(const __grid_constant__ TmaContractParams p) {
  constexpr bool kPair = true;
#include "contract_body.inc"
}

// The conv variants (im2col tensor maps, tap-major weight rows) are separate instantiations: folded into one kernel, the
// conv state kept live across the generator loop pushed every input-gradient variant over its register budget (116-152
// bytes of spill stores in the hot loop: C4 input gradient 2.33 -> 2.86 ms).
template <bool kPair, int MB, bool kDgrad, int kMode>
int launch_contract_v(const TmaContractParams& p, dim3 grid, cudaStream_t st) {
  constexpr size_t kSmem = kSmemAux + 1024 + static_cast<size_t>(kASlots) * kTileBytes +
                           static_cast<size_t>(kWSlots) * (kPair ? kHalfTileBytes : kTileBytes);
  void (*kernel)(TmaContractParams);
  if constexpr (kPair) kernel = contract_pair_kernel<MB, kDgrad, kMode>;
  else kernel = contract_tma_kernel<MB, kDgrad, kMode>;
  static SmemOptIn opt_in;
  const int rc = allow_dynamic_smem(kernel, kSmem, &opt_in);
  if (rc != BNN_OK) return rc;
  kernel<<<grid, kThreadsTma, kSmem, st>>>(p);
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}
template <bool kPair, int MB, bool kDgrad>
int launch_contract(const TmaContractParams& p, dim3 grid, cudaStream_t st) {
  if (p.conv.on == 2) return launch_contract_v<kPair, MB, kDgrad, 3>(p, grid, st);
  if (p.conv.on) return launch_contract_v<kPair, MB, kDgrad, 1>(p, grid, st);
  if (p.rng_w.row_sign != nullptr) return launch_contract_v<kPair, MB, kDgrad, 2>(p, grid, st);
  return launch_contract_v<kPair, MB, kDgrad, 0>(p, grid, st);
}

// Test aid: force one kernel variant (0 = pair, 1 / 2 / 4 = rows blocks per CTA, -1 = cost model) so that small test
// shapes reach every variant.  Set through bnn_debug_force_contract_variant.
std::atomic<int> g_forced_variant{-1};

// Tile plan of the CTA-pair kernel (TilePlan): when the uniform grid needs a fraction of a wave more than a whole
// number (1 < tiles / slots < 2 is the case that matters: the example conv layers), look for a cut of every sample into
// 8- and 6-row-block tiles — at most two kinds of samples — whose list schedule (all 8-block tiles first) finishes
// earlier.  Cost unit: one row block of MMAs per k-block; the fixed cost per tile is ignored, so a plan must win by 8 %.
bool solve_pair_tiles(TilePlan* plan, int m_blocks, int S, int slots);
bool plan_pair_tiles(TilePlan* plan, int m_blocks, int S, int gx, int gz, bool sum_samples, int slots) {
  plan->on = 0;
  if (sum_samples || gx != 1 || gz != S || S < 1 || slots < 1) return false;
  // the search costs milliseconds: one result per (rows, samples, machine) for the life of the process
  static std::mutex mu;
  static std::vector<std::pair<std::array<int, 3>, TilePlan>> cache;
  const std::array<int, 3> key = {m_blocks, S, slots};
  std::lock_guard<std::mutex> lock(mu);
  for (const auto& e : cache)
    if (e.first == key) { *plan = e.second; return plan->on != 0; }
  TilePlan found{};
  solve_pair_tiles(&found, m_blocks, S, slots);
  cache.emplace_back(key, found);
  *plan = found;
  return plan->on != 0;
}
bool solve_pair_tiles(TilePlan* plan, int m_blocks, int S, int slots) {
  plan->on = 0;
  const int units = (m_blocks + 1) / 2;                        // row-block pairs per sample (one row block per CTA)
  const int uniform_tiles = S * ((units + 3) / 4);
  if (uniform_tiles <= slots || uniform_tiles > 4 * slots) return false;
  auto makespan = [&](int n_a, int n_b) {                      // greedy list schedule on `slots` machines
    std::vector<int> load(static_cast<size_t>(slots), 0);
    auto place = [&](int cost) { auto it = std::min_element(load.begin(), load.end()); *it += cost; };
    for (int i = 0; i < n_a; ++i) place(4);
    for (int i = 0; i < n_b; ++i) place(3);
    return *std::max_element(load.begin(), load.end());
  };
  const int base = makespan(uniform_tiles, 0);
  struct Cut { int a, b; };
  std::vector<Cut> cuts;                                       // 4 a + 3 b covers the units with at most 2 to spare
  for (int a = 0; a * 4 <= units + 3; ++a)
    for (int b = 0; b <= (units + 2) / 3 + 1; ++b) {
      const int cover = 4 * a + 3 * b;
      if (cover >= units && cover <= units + 2 && (a > 0 || b > 0)) cuts.push_back({a, b});
    }
  int best = base;
  TilePlan found = *plan;
  for (const Cut& c1 : cuts)
    for (const Cut& c2 : cuts)
      for (int s1 = 0; s1 <= S; ++s1) {
        if ((s1 == 0 && (&c1 != &cuts[0])) || (s1 == S && (&c2 != &cuts[0]))) continue;      // unused class: one representative
        const int n_a = s1 * c1.a + (S - s1) * c2.a, n_b = s1 * c1.b + (S - s1) * c2.b;
        const int ms = makespan(n_a, n_b);
        if (ms < best) { best = ms; found = TilePlan{1, n_a, s1, c1.a, c1.b, c2.a, c2.b}; }
      }
  if (best * 100 > base * 92) return false;
  *plan = found;
  return true;
}

template <bool kDgrad>
int dispatch_tma_contract(TmaContractParams& p, int n_cols, cudaStream_t st) {
  const int m_blocks = (p.M + 127) / 128;
  const int gx = (n_cols + 127) / 128;
  const int sms = sm_count();
  const int n_red = kDgrad ? p.N : p.K;
  // Shared activations (one output summed over the samples): a CTA walks `z_per` samples; when the output has too few
  // tiles to fill the machine the samples are split over grid.z and the partial sums are added to the zeroed output.
  int gz = p.S;
  if (p.sum_samples) {
    const int64_t tiles = static_cast<int64_t>(gx) * ((m_blocks + 3) / 4);
    int groups = static_cast<int>((sms + tiles - 1) / tiles);
    if (groups > p.S) groups = p.S;
    if (groups < 1 || p.out.P != 1) groups = 1;
    p.z_per = (p.S + groups - 1) / groups;
    gz = (p.S + p.z_per - 1) / p.z_per;
    p.atomic_out = gz > 1 ? 1 : 0;
    if (p.atomic_out)
      BNN_CUDA_OK(cudaMemset2DAsync(p.out.base, static_cast<size_t>(p.out.bs) * 4, 0, static_cast<size_t>(n_cols) * 4,
                                    static_cast<size_t>(p.M), st));
  }
  // Rows per CTA by a cost model of the measured kernels (DESIGN §4), in cycles per 32-wide k-block: a CTA generates
  // its weight tile at ~1.86 weights/clk whatever the number of 128-row blocks that reuse it (128 x 32 tile: ~2200
  // cycles; half of it per CTA of a pair), its MMAs + operand delivery cost ~425 cycles per block (~468 per block pair
  // with cta_group::2), so a k-block takes the larger of the two; a launch takes waves x (fixed cost + k-blocks x that).
  // Small problems thereby keep few rows per CTA (every SM gets a short k-loop) and large ones share each generated
  // tile between 1024 rows — without insisting on a CTA for every SM: 144 busy SMs with 4x the reuse beat 148.
  const double iters = static_cast<double>((n_red + kBK - 1) / kBK) * (p.sum_samples ? p.z_per : 1);
  const double w_rows = n_cols < 128 ? n_cols : 128;
  auto cost_single = [&](int mb) {
    const int64_t ctas = static_cast<int64_t>(gx) * ((m_blocks + mb - 1) / mb) * gz;
    const double waves = static_cast<double>((ctas + sms - 1) / sms);
    const double gen = w_rows * kBK / 1.86, mma = 425.0 * (mb < m_blocks ? mb : m_blocks);
    return waves * (4000.0 + 600.0 * mb + iters * ((gen > mma ? gen : mma) + 100.0));
  };
  auto cost_pair = [&]() {
    const int64_t pairs = static_cast<int64_t>(gx) * ((m_blocks + 7) / 8) * gz;
    const int slots = sms / 2;
    const double waves = static_cast<double>((pairs + slots - 1) / slots);
    const double gen = (w_rows > 64 ? 64 : w_rows) * kBK / 1.86, mma = 468.0 * 4;
    return waves * (5000.0 + 600.0 * 4 + iters * ((gen > mma ? gen : mma) + 100.0));
  };
  int best = 1;
  double best_cost = cost_single(1);
  for (int mb = 2; mb <= 4; mb *= 2) {
    if (m_blocks < mb) break;
    const double c = cost_single(mb);
    if (c < best_cost) { best_cost = c; best = mb; }
  }
  if (m_blocks > 4 && cost_pair() < 0.9 * best_cost) best = 0;       // a clear win only: the model is coarse
  const int forced = g_forced_variant.load(std::memory_order_relaxed);
  if (forced > 0 || (forced == 0 && m_blocks > 4)) best = forced;
  if (best == 0) {                                                // two CTAs (one cluster) per 1024 rows
    const int pairs = (m_blocks + 7) / 8;
    if (plan_pair_tiles(&p.plan, m_blocks, p.S, gx, gz, p.sum_samples != 0, sms / 2))
      return launch_contract<true, 4, kDgrad>(p, dim3(2 * (p.plan.n_a + p.plan.s1 * p.plan.b1 + (p.S - p.plan.s1) * p.plan.b2), 1, 1), st);
    return launch_contract<true, 4, kDgrad>(p, dim3(2 * pairs, gx, gz), st);
  }
  if (best == 4) return launch_contract<false, 4, kDgrad>(p, dim3(gx, (m_blocks + 3) / 4, gz), st);
  if (best == 2) return launch_contract<false, 2, kDgrad>(p, dim3(gx, (m_blocks + 1) / 2, gz), st);
  return launch_contract<false, 1, kDgrad>(p, dim3(gx, m_blocks, gz), st);
}

// ---------------------------------------------------------------------------------------------- weight gradient
// CTA (k-tile, n-tile, sample group).  Stage = dY^T tile (MN = n) + A^T tile (MN = k), each 4 TMA boxes of
// 32 MN x 32 K-rows (m).  TMEM columns: [0,128) G0 | [128,256) sum G | [256,384) sum G o eps | [384,512) G1.
constexpr int kWgStages = 3;                 // stages of 64 contraction rows: 8 MMAs per barrier wait / tcgen05.commit
constexpr int kWgRows = 64;                  // contraction rows (m) per stage
constexpr int kWgOperandBytes = 4 * kWgRows * kRowBytes;      // 4 MN groups x 64 K-rows x 128 B = 32 KiB per operand
constexpr uint32_t kWgLbo = kWgRows * kRowBytes;              // next 32 MN elements: 8 KiB further
constexpr int kWgEpiWarps = 12;              // three warps per TMEM lane quarter share the 8 column chunks of a tile:
constexpr int kWgThreads = (2 + kWgEpiWarps) * 32;   // regenerating eps for 128 x 128 per sample is the long pole
                                             // warp 0 TMA, warp 1 MMA (+TMEM owner), warps 2.. epilogue
constexpr size_t kWgradSmem = kSmemAux + 1024 + static_cast<size_t>(kWgStages) * 2 * kWgOperandBytes;

struct TmaWgradParams {
  CUtensorMap map_dy;       // dY [S][M][N], box 32 x 32
  CUtensorMap map_a;        // A  [S or 1][M][K], box 32 x 32; conv: the NHWC input (im2col map, 32 channels x 64 pixels)
  ConvCoords conv;
  const float* rho_w;
  const float* eps_w;
  float* dmu_w;
  float* drho_w;
  int M, N, K, S;
  uint32_t sample_begin;
  bnn_rng rng_w;
  int shared_a;
  int shared_dy;            // all samples read sample 0 of dY (the weight gradient of a transposed conv with shared input)
  int n_chunks;             // the M reduction of every sample is cut into n_chunks pieces of chunk_blocks k-blocks:
  int chunk_blocks;         // a work unit = (sample, chunk); (sum_chunks G) o eps = sum_chunks (G o eps), so units are independent
};

// kPair: the same kernel over a cluster of two CTAs (launched with cluster dimension (2,1,1)): the pair owns two adjacent
// n-tiles and ONE k-tile, tcgen05.mma.cta_group::2 computes 256 (n) x 128 (k) per instruction, and each CTA loads its own
// dY^T tile but only HALF of the shared A^T tile (48 instead of 64 KiB per stage and CTA: the kernel is paced by operand
// delivery).  TMA bytes and the epilogue's buffer releases land on the leader's barriers; commits are multicast.
// kVol: 3-d convolutions (rank-5 im2col map of A)
template <bool kPair, bool kSignNoise, bool kVol = false>
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_tma_kernel(const __grid_constant__ TmaWgradParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  constexpr uint32_t kTmemCols = 512;
  constexpr uint32_t kColG0 = 0, kColMu = 128, kColRho = 256, kColG1 = 384;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* empty = full + kWgStages;
  uint64_t* accum_full = empty + kWgStages;
  uint64_t* accum_empty = accum_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_empty + 2);
  const uint32_t ring = (smem_u32(smem_raw) + kSmemAux + 1023u) & ~1023u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kWgStages; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(accum_full + i, 1); mbar_init(accum_empty + i, (kPair ? 2 : 1) * kWgEpiWarps); }
    fence_mbar_init();
    tma_prefetch_desc(&p.map_dy);
    tma_prefetch_desc(&p.map_a);
  }
  if (warp == 1) { if (kPair) tmem_alloc_pair(tmem_slot, kTmemCols); else tmem_alloc(tmem_slot, kTmemCols); }
  tc_fence_before_sync();
  if (kPair) cluster_sync_all(); else __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;      // 0 = leader

  const int n0 = blockIdx.x * 128;                          // this CTA's rows of dmu / drho (pairs are adjacent in x)
  const int k0 = blockIdx.y * 128;
  const int groups = gridDim.z;
  const int units = p.S * p.n_chunks;
  const int per = (units + groups - 1) / groups;
  const int s_begin = blockIdx.z * per;                          // work units [s_begin, s_end)
  const int s_end = s_begin + per < units ? s_begin + per : units;
  const int m_total = (p.M + kWgRows - 1) / kWgRows;        // stages of 64 rows
  auto unit_blocks = [&](int u, int* mb0) {                      // k-block range of unit u
    const int c = u % p.n_chunks;
    *mb0 = c * p.chunk_blocks;
    const int left = m_total - *mb0;
    return left < p.chunk_blocks ? left : p.chunk_blocks;
  };

  if (s_begin < s_end) {
    if (warp == 0) {
      if (lane == 0) {
        int it = 0;
        // conv: the 32-column group kc .. kc + 31 of the im2col matrix = (tap, channels c0 ..) of the NHWC input — fixed per
        // CTA; groups beyond K read channel `chans` (outside the tensor: zeros, the transaction still completes)
        int g_c0[4] = {0, 0, 0, 0};
        uint16_t g_ow[4] = {0, 0, 0, 0}, g_oh[4] = {0, 0, 0, 0};
        uint16_t g_od[kVol ? 4 : 1] = {0};
        if (p.conv.on) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const int kc = k0 + g * 32;
            if (kc >= p.K) { g_c0[g] = p.conv.chans; continue; }
            int tap = kc / p.conv.chans;
            g_c0[g] = kc - tap * p.conv.chans;
            if constexpr (kVol) {
              const int kd = tap / p.conv.KHW;
              g_od[g] = static_cast<uint16_t>(kd * p.conv.dd);
              tap -= kd * p.conv.KHW;
            }
            const int kh = tap / p.conv.KW, kw = tap - kh * p.conv.KW;
            g_ow[g] = static_cast<uint16_t>(kw * p.conv.dw);
            g_oh[g] = static_cast<uint16_t>(kh * p.conv.dh);
          }
        }
        for (int u = s_begin; u < s_end; ++u) {
          const int s = u / p.n_chunks;
          const int sa = p.shared_a ? 0 : s, sd = p.shared_dy ? 0 : s;
          int mb0;
          const int m_blocks = unit_blocks(u, &mb0);
          for (int mb = mb0; mb < mb0 + m_blocks; ++mb, ++it) {
            const int stage = it % kWgStages;
            mbar_wait(empty + stage, ((it / kWgStages) & 1) ^ 1);
            const uint32_t base = ring + stage * 2 * kWgOperandBytes;
            int cw = 0, ch = 0, cn = 0, cd = 0;
            if constexpr (kVol) conv_pixel3d(p.conv, mb * kWgRows, sa, &cw, &ch, &cd, &cn);
            else if (p.conv.on) conv_pixel(p.conv, mb * kWgRows, sa, &cw, &ch, &cn);
            (void)cd;
            if (!kPair) {
              mbar_arrive_expect_tx(full + stage, 2 * kWgOperandBytes);
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                tma_load_3d(base + g * kWgLbo, &p.map_dy, n0 + g * 32, mb * kWgRows, sd, full + stage);
                if constexpr (kVol) {
                  tma_load_im2col_5d(base + kWgOperandBytes + g * kWgLbo, &p.map_a, g_c0[g], cw, ch, cd, cn, g_ow[g], g_oh[g],
                                     g_od[g], full + stage);
                } else if (!p.conv.on) {
                  tma_load_3d(base + kWgOperandBytes + g * kWgLbo, &p.map_a, k0 + g * 32, mb * kWgRows, sa, full + stage);
                } else {
                  tma_load_im2col_4d(base + kWgOperandBytes + g * kWgLbo, &p.map_a, g_c0[g], cw, ch, cn, g_ow[g], g_oh[g],
                                     full + stage);
                }
              }
            } else {
              const uint32_t lead_full = mapa_u32(smem_u32(full + stage), 0);
              if (rank == 0) mbar_arrive_expect_tx(full + stage, 2 * (kWgOperandBytes + kWgOperandBytes / 2));
#pragma unroll
              for (int g = 0; g < 4; ++g)
                tma_load_3d_pair(base + g * kWgLbo, &p.map_dy, n0 + g * 32, mb * kWgRows, sd, lead_full);
#pragma unroll
              for (int g = 0; g < 2; ++g) {     // this CTA's half (64 columns) of the shared A^T tile
                const int kc = k0 + static_cast<int>(rank) * 64 + g * 32;
                if constexpr (kVol) {
                  const int gi = static_cast<int>(rank) * 2 + g;
                  tma_load_im2col_5d_pair(base + kWgOperandBytes + g * kWgLbo, &p.map_a, g_c0[gi], cw, ch, cd, cn, g_ow[gi],
                                          g_oh[gi], g_od[gi], lead_full);
                } else if (!p.conv.on) {
                  tma_load_3d_pair(base + kWgOperandBytes + g * kWgLbo, &p.map_a, kc, mb * kWgRows, sa, lead_full);
                } else {
                  const int gi = static_cast<int>(rank) * 2 + g;
                  tma_load_im2col_4d_pair(base + kWgOperandBytes + g * kWgLbo, &p.map_a, g_c0[gi], cw, ch, cn, g_ow[gi],
                                          g_oh[gi], lead_full);
                }
              }
            }
          }
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      if (lane == 0 && rank == 0) {
        const uint32_t idesc = kPair ? make_idesc_tf32(256, 128, true, true) : make_idesc_tf32(128, mma_n(p.K - k0), true, true);
        const uint64_t desc_dy0 = make_smem_desc_mn(ring, kWgLbo, kMnSbo);
        const uint64_t desc_a0 = make_smem_desc_mn(ring + kWgOperandBytes, kWgLbo, kMnSbo);
        int it = 0;
        for (int u = s_begin, i = 0; u < s_end; ++u, ++i) {
          const int buf = i & 1;
          if (kPair) mbar_wait_cluster(accum_empty + buf, ((i >> 1) & 1) ^ 1); else mbar_wait(accum_empty + buf, ((i >> 1) & 1) ^ 1);
          tc_fence_after_sync();
          const uint32_t d = tmem + (buf ? kColG1 : kColG0);
          int mb0;
          const int m_blocks = unit_blocks(u, &mb0);
          for (int mb = 0; mb < m_blocks; ++mb, ++it) {
            const int stage = it % kWgStages;
            if (kPair) mbar_wait_cluster(full + stage, (it / kWgStages) & 1); else mbar_wait(full + stage, (it / kWgStages) & 1);
            tc_fence_after_sync();
            const uint64_t da0 = desc_advance(desc_dy0, static_cast<uint32_t>(stage) * (2 * kWgOperandBytes >> 4));
            const uint64_t db0 = desc_advance(desc_a0, static_cast<uint32_t>(stage) * (2 * kWgOperandBytes >> 4));
#pragma unroll
            for (int ks = 0; ks < kWgRows / 8; ++ks) {
              if (kPair)
                mma_tf32_pair(d, desc_advance(da0, ks * (kMnKStep >> 4)), desc_advance(db0, ks * (kMnKStep >> 4)), idesc,
                              mb > 0 || ks > 0);
              else
                mma_tf32(d, desc_advance(da0, ks * (kMnKStep >> 4)), desc_advance(db0, ks * (kMnKStep >> 4)), idesc,
                         mb > 0 || ks > 0);
            }
            if (kPair) mma_commit_pair(empty + stage, 3); else mma_commit(empty + stage);
          }
          if (kPair) mma_commit_pair(accum_full + buf, 3); else mma_commit(accum_full + buf);
        }
      }
      __syncwarp();
    } else {
      const int quad = warp & 3;                    // TMEM lane quarter this warp may access
      const int sub = (warp - 2) >> 2;              // which third of the column chunks it handles
      const int n = n0 + quad * 32 + lane;
      const uint32_t lane_addr = tmem + (static_cast<uint32_t>(quad * 32) << 16);
      const RngKey key = resolve_rng(p.rng_w);
      const int cols_here = p.K - k0 < 128 ? p.K - k0 : 128;
      for (int u = s_begin, i = 0; u < s_end; ++u, ++i) {
        const int s = u / p.n_chunks;
        const int buf = i & 1;
        const bool first = (u == s_begin), last = (u + 1 == s_end);
        EpsSrc eps;
        eps.inj = p.eps_w ? p.eps_w + static_cast<int64_t>(s) * p.N * p.K : nullptr;
        eps.key = key;
        eps.sample = p.sample_begin + s;
        mbar_wait(accum_full + buf, (i >> 1) & 1);
        tc_fence_after_sync();
        for (int c = sub; c * 16 < cols_here; c += kWgEpiWarps / 4) {
          float g[16], dm[16], dr[16];
          tmem_ld16(lane_addr + (buf ? kColG1 : kColG0) + c * 16, g);
          if (!first) {
            tmem_ld16(lane_addr + kColMu + c * 16, dm);
            tmem_ld16(lane_addr + kColRho + c * 16, dr);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) dm[j] = dr[j] = 0.f;
          }
          const int k = k0 + c * 16;
          if (n < p.N) {
            const int64_t row = static_cast<int64_t>(n) * p.K;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              if (k + q * 4 < p.K) {
                const float4 e = eps_vec4<kSignNoise ? 1 : 0>(eps, row + k + q * 4);
                dm[q * 4 + 0] += g[q * 4 + 0]; dr[q * 4 + 0] = fmaf(g[q * 4 + 0], e.x, dr[q * 4 + 0]);
                dm[q * 4 + 1] += g[q * 4 + 1]; dr[q * 4 + 1] = fmaf(g[q * 4 + 1], e.y, dr[q * 4 + 1]);
                dm[q * 4 + 2] += g[q * 4 + 2]; dr[q * 4 + 2] = fmaf(g[q * 4 + 2], e.z, dr[q * 4 + 2]);
                dm[q * 4 + 3] += g[q * 4 + 3]; dr[q * 4 + 3] = fmaf(g[q * 4 + 3], e.w, dr[q * 4 + 3]);
              }
            }
          }
          if (!last) {
            tmem_st16(lane_addr + kColMu + c * 16, dm);
            tmem_st16(lane_addr + kColRho + c * 16, dr);
          } else if (n < p.N) {
            const int64_t row = static_cast<int64_t>(n) * p.K;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              if (k + q * 4 < p.K) {
                const int64_t i0 = row + k + q * 4;
                const float4 r = __ldg(reinterpret_cast<const float4*>(p.rho_w + i0));
                red_add4(p.dmu_w + i0, dm[q * 4], dm[q * 4 + 1], dm[q * 4 + 2], dm[q * 4 + 3]);
                red_add4(p.drho_w + i0, dr[q * 4] * sigmoid_fast(r.x), dr[q * 4 + 1] * sigmoid_fast(r.y),
                         dr[q * 4 + 2] * sigmoid_fast(r.z), dr[q * 4 + 3] * sigmoid_fast(r.w));
              }
            }
          }
        }
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) {
          if (kPair) mbar_arrive_cluster(mapa_u32(smem_u32(accum_empty + buf), 0)); else mbar_arrive(accum_empty + buf);
        }
      }
    }
  }
  tc_fence_before_sync();
  if (kPair) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    if (kPair) tmem_dealloc_pair(tmem, kTmemCols); else tmem_dealloc(tmem, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------- self test
// MN-major operand tiles: D(128 x 64) = A^T-tile(MN-major, 128 x 32) * B^T-tile(MN-major, 64 x 32)^T against a
// serial fp32 loop over the TF32-rounded values.
__device__ __forceinline__ float st_a(int r, int c) {
  return __uint_as_float(to_tf32(0.01f * static_cast<float>((r * 7 + c * 13) % 97) - 0.4f));
}
__device__ __forceinline__ float st_b(int r, int c) {
  return __uint_as_float(to_tf32(0.02f * static_cast<float>((r * 5 + c * 3) % 89) - 0.7f));
}
__global__ void __launch_bounds__(128, 1) selftest_mn_kernel(float* max_err, int variant) {
  __shared__ __align__(1024) uint8_t tiles[2 * kTileBytes];
  __shared__ uint64_t bar;
  __shared__ uint32_t slot;
  __shared__ float red[4];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t ta = smem_u32(tiles), tb = ta + kTileBytes;
  const bool a_mn = variant & 1, b_mn = variant & 2;
  const uint32_t lbo = kMnLbo, sbo = kMnSbo;
  for (int i = tid; i < 128 * 32; i += 128) {
    const int mn = i & 127, k = i >> 7;
    const uint32_t va = __float_as_uint(st_a(mn, k)), vb = __float_as_uint(mn < 64 ? st_b(mn, k) : 0.f);
    if (a_mn) sts32(ta + tile_offset_mn(mn, k, lbo, sbo), va);
    else sts32(ta + tile_offset(mn, k >> 2) + ((k & 3) << 2), va);
    if (b_mn) sts32(tb + tile_offset_mn(mn, k, lbo, sbo), vb);
    else sts32(tb + tile_offset(mn, k >> 2) + ((k & 3) << 2), vb);
  }
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(&slot, 64);
  fence_proxy_async_smem();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(&slot);
  if (tid == 0) {
    const uint32_t idesc = make_idesc_tf32(128, 64, a_mn, b_mn);
    for (int ks = 0; ks < 4; ++ks) {
      const uint64_t da = a_mn ? make_smem_desc_mn(ta + ks * kMnKStep, lbo, sbo) : make_smem_desc(ta + ks * 32);
      const uint64_t db = b_mn ? make_smem_desc_mn(tb + ks * kMnKStep, lbo, sbo) : make_smem_desc(tb + ks * 32);
      mma_tf32(tmem, da, db, idesc, ks > 0);
    }
    mma_commit(&bar);
  }
  mbar_wait(&bar, 0);
  tc_fence_after_sync();
  float err = (ta & 1023u) ? 1e30f : 0.f;
  for (int c = 0; c < 4; ++c) {
    float v[16];
    tmem_ld16(tmem + (static_cast<uint32_t>(warp * 32) << 16) + c * 16, v);
    for (int j = 0; j < 16; ++j) {
      float ref = 0.f;
      for (int k = 0; k < 32; ++k) ref = fmaf(st_a(tid, k), st_b(c * 16 + j, k), ref);
      err = fmaxf(err, fabsf(ref - v[j]));
    }
  }
  for (int o = 16; o > 0; o >>= 1) err = fmaxf(err, __shfl_xor_sync(0xffffffffu, err, o));
  if (lane == 0) red[warp] = err;
  tc_fence_before_sync();
  __syncthreads();
  if (tid == 0) *max_err = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
  if (warp == 0) {
    tc_fence_after_sync();
    tmem_dealloc(tmem, 64);
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------- host entry points
int tma_fwd(const float* a, int64_t lda, int64_t a_sample_stride, const float* mu_w, const float* sigma_w,
            const float* mu_b, const float* sigma_b, const float* eps_w, const float* eps_b, bnn_view y,
            int64_t y_sample_stride, int M, int N, int K, int S, uint32_t sample_begin, const bnn_rng* rng_w,
            const bnn_rng* rng_b, cudaStream_t st) {
  const bool shared = a_sample_stride == 0;
  if (!tma_ok(a, lda, a_sample_stride) || K % 4 != 0 || rng_w->elem_offset % 4 != 0 || !aligned16(mu_w) ||
      !aligned16(sigma_w) || (eps_w != nullptr && !aligned16(eps_w)))
    return kNotEligible;
  TmaContractParams p{};
  int rc = make_map(&p.map_l, a, K, M, shared ? 1 : S, lda, a_sample_stride, 128);
  if (rc != BNN_OK) return rc;
  p.out.base = y.base; p.out.bs = y.batch_stride; p.out.P = y.P; p.out_sample_stride = y_sample_stride;
  p.mu_w = mu_w; p.sigma_w = sigma_w; p.eps_w = eps_w; p.mu_b = mu_b; p.sigma_b = sigma_b; p.eps_b = eps_b;
  p.M = M; p.N = N; p.K = K; p.S = S; p.sample_begin = sample_begin;
  p.w_numel = static_cast<int64_t>(N) * K;
  p.rng_w = *rng_w; p.rng_b = rng_b ? *rng_b : *rng_w;
  p.shared_l = shared ? 1 : 0;
  p.sum_samples = 0;
#ifdef BNN_PROFILE_WAITS
  { const char* e = getenv("BNN_EXP_FLAGS"); p.exp_flags = e ? atoi(e) : 0; }
#endif
  p.vec_out = (y.P == 1) && (y.batch_stride % 4 == 0) && (y_sample_stride % 4 == 0) && aligned16(y.base);
  return dispatch_tma_contract<false>(p, N, st);
}

int tma_dgrad(bnn_view dy, int64_t dy_sample_stride, const float* mu_w, const float* sigma_w, const float* eps_w,
              float* da, int64_t lda, int64_t a_sample_stride, int M, int N, int K, int S, uint32_t sample_begin,
              const bnn_rng* rng_w, cudaStream_t st) {
  if (dy.P != 1 || !tma_ok(dy.base, dy.batch_stride, dy_sample_stride) || K % 4 != 0 || rng_w->elem_offset % 4 != 0 ||
      !aligned16(mu_w) || !aligned16(sigma_w) || (eps_w != nullptr && !aligned16(eps_w)))
    return kNotEligible;
  TmaContractParams p{};
  int rc = make_map(&p.map_l, dy.base, N, M, S, dy.batch_stride, dy_sample_stride, 128);
  if (rc != BNN_OK) return rc;
  p.out.base = da; p.out.bs = lda; p.out.P = 1; p.out_sample_stride = a_sample_stride;
  p.mu_w = mu_w; p.sigma_w = sigma_w; p.eps_w = eps_w;
  p.M = M; p.N = N; p.K = K; p.S = S; p.sample_begin = sample_begin;
  p.w_numel = static_cast<int64_t>(N) * K;
  p.rng_w = *rng_w; p.rng_b = *rng_w;
  p.shared_l = 0;
  p.sum_samples = (a_sample_stride == 0) ? 1 : 0;
  p.vec_out = (lda % 4 == 0) && (a_sample_stride % 4 == 0) && aligned16(da);
  return dispatch_tma_contract<true>(p, K, st);
}

namespace {
// Test aid (bnn_debug_force_wgrad_plan): forced {pair, n_chunks, units per CTA}, -1 = the cost model's choice.  Unlike
// the contraction variant, a forced value the shape cannot take is an error, never a silent fall-back to another plan.
std::atomic<int> g_forced_wgrad[3] = {-1, -1, -1};
}  // namespace

// Work-unit plan of the weight gradient (host arithmetic) on `sms` SMs.  Work units = (sample, M-chunk); a CTA =
// (tile, group) walks `per` consecutive units, the epilogue of one unit (TMEM drain + eps regeneration for 128 x 128
// weights, ~6 stage times) overlapping the MMAs of the next.  The plan minimises  waves x (per x (stages per unit + 0.5)
// + 6)  over the number of M-chunks and units per CTA: small layers get ONE wave of CTAs with long units instead of
// several waves of short ones (every extra unit costs an epilogue), and no CTA is launched without work.  The cost
// model cuts the m_total 64-row stages of a sample into at most min(ceil(m_total / 4), 64) chunks, i.e. no more chunks
// than 256-row pieces; every chunk holds chunk_blocks = ceil(m_total / n_chunks) stages except the last, which holds
// what is left and may be shorter (m_total = 5: 3 + 2 stages; m_total = 13: 4 + 4 + 4 + 1).
int wgrad_plan(int M, int N, int K, int S, int sms, WgradPlan* out) {
  const int tiles = ((N + 127) / 128) * ((K + 127) / 128);
  const int m_total = (M + kWgRows - 1) / kWgRows;         // 64-row stages
  const int f_pair = g_forced_wgrad[0].load(std::memory_order_relaxed);
  const int f_chunks = g_forced_wgrad[1].load(std::memory_order_relaxed);
  const int f_per = g_forced_wgrad[2].load(std::memory_order_relaxed);
  if (f_chunks > 0) {
    const int cb = (m_total + f_chunks - 1) / f_chunks;
    BNN_REQUIRE((m_total + cb - 1) / cb == f_chunks, BNN_ERR_BAD_ARGUMENT,
                "forced weight-gradient plan: n_chunks = %d does not cut %d stages of 64 rows into %d non-empty chunks",
                f_chunks, m_total, f_chunks);
  }
  const int max_chunks = (m_total + 3) / 4 < 64 ? (m_total + 3) / 4 : 64;
  double best_cost = 0.0;
  int best_cb = m_total, best_n = 1, best_per = S;
  bool have = false;
  const int n_first = f_chunks > 0 ? f_chunks : 1, n_last = f_chunks > 0 ? f_chunks : (max_chunks < 1 ? 1 : max_chunks);
  for (int n = n_first; n <= n_last; ++n) {
    const int cb = (m_total + n - 1) / n, n_eff = (m_total + cb - 1) / cb;
    if (n_eff != n) continue;
    const int64_t units = static_cast<int64_t>(S) * n;
    for (int c = 0; c < (f_per > 0 ? 1 : 32); ++c) {
      const int64_t per = f_per > 0 ? f_per : c < 16 ? c + 1 : (units + (c - 16)) / (c - 15);   // 1..16, then units / (1..16) rounded up
      if (per < 1 || per > units) continue;
      const int64_t groups = (units + per - 1) / per;
      if (groups > 65535) continue;
      if (f_per > 0 && (units + groups - 1) / groups != per) continue;       // the kernel would walk fewer units per CTA
      const int64_t ctas = static_cast<int64_t>(tiles) * groups;
      const double waves = static_cast<double>((ctas + sms - 1) / sms);
      const double cost = waves * (static_cast<double>(per) * (cb + 0.5) + 6.0);
      if (!have || cost < best_cost * 0.999 || (cost <= best_cost * 1.001 && ctas < static_cast<int64_t>(tiles) * ((static_cast<int64_t>(S) * best_n + best_per - 1) / best_per))) {
        have = true; best_cost = cost; best_cb = cb; best_n = n; best_per = static_cast<int>(per);
      }
    }
  }
  BNN_REQUIRE(have || f_per <= 0, BNN_ERR_BAD_ARGUMENT,
              "forced weight-gradient plan: units_per_cta = %d fits no plan of %d samples (more than S x n_chunks units, "
              "more than 65535 groups, or the last group would be short enough to shrink every CTA's share)", f_per, S);
  const int64_t units = static_cast<int64_t>(S) * best_n;
  const int groups = static_cast<int>((units + best_per - 1) / best_per);
  const int n_tiles = (N + 127) / 128;
  bool pair = n_tiles >= 2 && static_cast<int64_t>(tiles) * groups >= 2 * sms;
  if (f_pair >= 0) {
    BNN_REQUIRE(f_pair == 0 || n_tiles >= 2, BNN_ERR_BAD_ARGUMENT,
                "forced weight-gradient plan: pair = 1 needs at least two 128-row n-tiles, N = %d has one", N);
    pair = f_pair == 1;
  }
  out->pair = pair ? 1 : 0;
  out->n_chunks = best_n;
  out->chunk_blocks = best_cb;
  out->per = static_cast<int>((units + groups - 1) / groups);           // what the kernel derives from gridDim.z
  out->groups = groups;
  return BNN_OK;
}

int tma_force_wgrad_plan(int pair, int n_chunks, int units_per_cta) {
  BNN_REQUIRE(pair >= -1 && pair <= 1 && (n_chunks == -1 || n_chunks >= 1) && (units_per_cta == -1 || units_per_cta >= 1),
              BNN_ERR_BAD_ARGUMENT, "bnn_debug_force_wgrad_plan: pair in {-1, 0, 1}, n_chunks and units_per_cta -1 or >= 1");
  g_forced_wgrad[0].store(pair, std::memory_order_relaxed);
  g_forced_wgrad[1].store(n_chunks, std::memory_order_relaxed);
  g_forced_wgrad[2].store(units_per_cta, std::memory_order_relaxed);
  return BNN_OK;
}

// Plan + launch shared by the matrix and the implicit-GEMM (conv) weight gradient
int wgrad_plan_and_launch(TmaWgradParams& p, int M, int N, int K, int S, cudaStream_t st) {
  WgradPlan plan{};
  int rc = wgrad_plan(M, N, K, S, sm_count(), &plan);
  if (rc != BNN_OK) return rc;
  p.chunk_blocks = plan.chunk_blocks;
  p.n_chunks = plan.n_chunks;
  const int groups = plan.groups;
  static SmemOptIn opt_in[6];
  const bool signs = p.rng_w.row_sign != nullptr, vol = p.conv.on == 2;
  rc = allow_dynamic_smem(wgrad_tma_kernel<false, false>, kWgradSmem, &opt_in[0]);
  if (rc == BNN_OK) rc = allow_dynamic_smem(wgrad_tma_kernel<true, false>, kWgradSmem, &opt_in[1]);
  if (rc == BNN_OK) rc = allow_dynamic_smem(wgrad_tma_kernel<false, true>, kWgradSmem, &opt_in[2]);
  if (rc == BNN_OK) rc = allow_dynamic_smem(wgrad_tma_kernel<true, true>, kWgradSmem, &opt_in[3]);
  if (rc == BNN_OK) rc = allow_dynamic_smem(wgrad_tma_kernel<false, false, true>, kWgradSmem, &opt_in[4]);
  if (rc == BNN_OK) rc = allow_dynamic_smem(wgrad_tma_kernel<true, false, true>, kWgradSmem, &opt_in[5]);
  if (rc != BNN_OK) return rc;
  const int n_tiles = (N + 127) / 128, k_tiles = (K + 127) / 128;
  if (plan.pair) {
    // CTA pairs over adjacent n-tiles (large problems: the kernel is paced by operand delivery, a pair halves the A^T traffic)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((n_tiles + 1) / 2 * 2, k_tiles, groups);
    cfg.blockDim = dim3(kWgThreads);
    cfg.dynamicSmemBytes = kWgradSmem;
    cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    if (vol) BNN_CUDA_OK(cudaLaunchKernelEx(&cfg, wgrad_tma_kernel<true, false, true>, p));
    else if (signs) BNN_CUDA_OK(cudaLaunchKernelEx(&cfg, wgrad_tma_kernel<true, true>, p));
    else BNN_CUDA_OK(cudaLaunchKernelEx(&cfg, wgrad_tma_kernel<true, false>, p));
  } else {
    if (vol) wgrad_tma_kernel<false, false, true><<<dim3(n_tiles, k_tiles, groups), kWgThreads, kWgradSmem, st>>>(p);
    else if (signs) wgrad_tma_kernel<false, true><<<dim3(n_tiles, k_tiles, groups), kWgThreads, kWgradSmem, st>>>(p);
    else wgrad_tma_kernel<false, false><<<dim3(n_tiles, k_tiles, groups), kWgThreads, kWgradSmem, st>>>(p);
  }
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}


int tma_wgrad(bnn_view dy, int64_t dy_sample_stride, const float* a, int64_t lda, int64_t a_sample_stride,
              const float* rho_w, const float* eps_w, float* dmu_w, float* drho_w, int M, int N, int K, int S,
              uint32_t sample_begin, const bnn_rng* rng_w, cudaStream_t st) {
  const bool shared = a_sample_stride == 0;
  if (dy.P != 1 || !tma_ok(dy.base, dy.batch_stride, dy_sample_stride) || !tma_ok(a, lda, a_sample_stride) ||
      K % 4 != 0 || rng_w->elem_offset % 4 != 0 || !aligned16(rho_w) || !aligned16(dmu_w) || !aligned16(drho_w) ||
      (eps_w != nullptr && !aligned16(eps_w)))
    return kNotEligible;
  TmaWgradParams p{};
  int rc = make_map(&p.map_dy, dy.base, N, M, S, dy.batch_stride, dy_sample_stride, kWgRows, true);
  if (rc != BNN_OK) return rc;
  rc = make_map(&p.map_a, a, K, M, shared ? 1 : S, lda, a_sample_stride, kWgRows, true);
  if (rc != BNN_OK) return rc;
  p.rho_w = rho_w; p.eps_w = eps_w; p.dmu_w = dmu_w; p.drho_w = drho_w;
  p.M = M; p.N = N; p.K = K; p.S = S; p.sample_begin = sample_begin;
  p.rng_w = *rng_w;
  p.shared_a = shared ? 1 : 0;
  return wgrad_plan_and_launch(p, M, N, K, S, st);
}

// ---------------------------------------------------------------------------------------------- implicit-GEMM convolution
// The same kernels with the activation operand addressed through an im2col tensor map over the NHWC tensor: no im2col
// matrix exists.  Weights are [Cout][KH][KW][C] (k = (kh, kw, c), c fastest), so a 32-wide k-block is one filter tap and
// 32 consecutive channels — C % 32 == 0 is the eligibility condition.  3-d convolutions (ConvGeom::vol) take the same
// path with NDHWC tensors, [Cout][KD][KH][KW][C] weights, rank-5 maps and the kMode 3 kernels.
namespace {
// im2col descriptor limits (cuTensorMapEncodeIm2col): box corners within [-128, 127] at rank 4 and [-16, 15] at rank 5;
// the copy's tap offsets address the box, so a filter extent (k - 1) d must stay below its span (256 / 32)
bool corner_ok(int v, bool vol) { return vol ? (v >= -16 && v <= 15) : (v >= -128 && v <= 127); }
bool extent_ok(int e, bool vol) { return e < (vol ? 32 : 256); }

ConvCoords conv_coords_fwd(const ConvGeom& cg) {
  const bnn_conv3d_nhwc& g = cg.g;
  ConvCoords c{};
  c.on = cg.vol ? 2 : 1; c.P = g.OD * g.OH * g.OW; c.OW = g.OW; c.imgs = g.B;
  c.sh = g.sh; c.sw = g.sw; c.lh = -g.ph; c.lw = -g.pw; c.dh = g.dh; c.dw = g.dw;
  c.KW = g.KW; c.taps = g.KD * g.KH * g.KW; c.cblocks = g.C / kBK; c.w_rows = g.Cout; c.chans = g.C;
  c.HW = g.OH * g.OW; c.sd = g.sd; c.ld = -g.pd; c.dd = g.dd; c.KH = g.KH; c.KHW = g.KH * g.KW;
  return c;
}
bool conv_ok(const ConvGeom& cg) {
  const bnn_conv3d_nhwc& g = cg.g;
  auto dim_ok = [&](int pad, int k, int d, int s) {
    return corner_ok(-pad, cg.vol) && corner_ok(pad - (k - 1) * d, cg.vol) && extent_ok((k - 1) * d, cg.vol) && s >= 1 &&
           s <= 8;
  };
  return g.C % kBK == 0 && dim_ok(g.ph, g.KH, g.dh, g.sh) && dim_ok(g.pw, g.KW, g.dw, g.sw) &&
         (!cg.vol || dim_ok(g.pd, g.KD, g.dd, g.sd));
}
Im2colDepth depth_fwd(const ConvGeom& cg) {
  const bnn_conv3d_nhwc& g = cg.g;
  return Im2colDepth{cg.vol, g.D, -g.pd, g.pd - (g.KD - 1) * g.dd, g.sd};
}
}  // namespace

ConvGeom conv_geom_2d(const bnn_conv2d_nhwc& g) {
  ConvGeom cg{};
  cg.vol = false;
  cg.g = bnn_conv3d_nhwc{g.B, 1, g.H, g.W, g.C, 1, g.OH, g.OW, g.Cout, 1, g.KH, g.KW, 1, g.sh, g.sw, 0, g.ph, g.pw,
                         1, g.dh, g.dw, 0};
  return cg;
}

namespace {
// sum_samples: every sample reads its own x and the S results are summed into one y (the input gradient of a transposed
// convolution with shared input); else x_sample_stride == 0 means all samples share x
int conv_fwd_launch(const float* x, int64_t x_sample_stride, const float* mu_w, const float* sigma_w, const float* mu_b,
                    const float* sigma_b, const float* eps_w, const float* eps_b, bnn_view y, int64_t y_sample_stride,
                    const ConvGeom& cg, int S, uint32_t sample_begin, const bnn_rng* rng_w, const bnn_rng* rng_b,
                    bool sum_samples, cudaStream_t st) {
  const bnn_conv3d_nhwc* g = &cg.g;
  const bool shared = x_sample_stride == 0 && !sum_samples;
  if (!conv_ok(cg) || !aligned16(x) || rng_w->elem_offset % 4 != 0 || !aligned16(mu_w) || !aligned16(sigma_w) ||
      (eps_w != nullptr && !aligned16(eps_w)))
    return kNotEligible;
  TmaContractParams p{};
  int rc = make_im2col_map(&p.map_l, x, g->C, g->W, g->H, static_cast<int64_t>(shared ? 1 : S) * g->B, -g->pw, -g->ph,
                           g->pw - (g->KW - 1) * g->dw, g->ph - (g->KH - 1) * g->dh, g->sw, g->sh, 128, false,
                           depth_fwd(cg));
  if (rc != BNN_OK) return rc;
  p.conv = conv_coords_fwd(cg);
  p.out.base = y.base; p.out.bs = y.batch_stride; p.out.P = y.P; p.out_sample_stride = y_sample_stride;
  p.mu_w = mu_w; p.sigma_w = sigma_w; p.eps_w = eps_w; p.mu_b = mu_b; p.sigma_b = sigma_b; p.eps_b = eps_b;
  p.M = g->B * g->OD * g->OH * g->OW; p.N = g->Cout; p.K = g->KD * g->KH * g->KW * g->C; p.S = S;
  p.sample_begin = sample_begin;
  p.w_numel = static_cast<int64_t>(p.N) * p.K;
  p.rng_w = *rng_w; p.rng_b = rng_b ? *rng_b : *rng_w;
  p.shared_l = shared ? 1 : 0;
  p.sum_samples = sum_samples ? 1 : 0;
#ifdef BNN_PROFILE_WAITS
  { const char* e = getenv("BNN_EXP_FLAGS"); p.exp_flags = e ? atoi(e) : 0; }
#endif
  p.vec_out = (y.P == 1) && (y.batch_stride % 4 == 0) && (y_sample_stride % 4 == 0) && aligned16(y.base);
  return dispatch_tma_contract<false>(p, p.N, st);
}
}  // namespace

int tma_conv_fwd(const float* x, int64_t x_sample_stride, const float* mu_w, const float* sigma_w, const float* mu_b,
                 const float* sigma_b, const float* eps_w, const float* eps_b, bnn_view y, int64_t y_sample_stride,
                 const ConvGeom& g, int S, uint32_t sample_begin, const bnn_rng* rng_w, const bnn_rng* rng_b,
                 cudaStream_t st) {
  return conv_fwd_launch(x, x_sample_stride, mu_w, sigma_w, mu_b, sigma_b, eps_w, eps_b, y, y_sample_stride, g, S,
                         sample_begin, rng_w, rng_b, false, st);
}

// Weight gradient of the implicit GEMM: G = dY^T A with dY [S or 1][B*OH*OW][Cout] (map_dy) and A the NHWC tensor
// [S or 1][B][H][W][C] seen through the im2col map (map_a).  A convolution passes (dy, x), shared_a when all samples
// share x; a transposed convolution passes its conv view's operands (x, dy), shared_dy when all samples share x.
int tma_conv_wgrad(const float* dy, bool shared_dy, const float* a, bool shared_a, const float* rho_w, const float* eps_w,
                   float* dmu_w, float* drho_w, const ConvGeom& cg, int S, uint32_t sample_begin,
                   const bnn_rng* rng_w, cudaStream_t st) {
  const bnn_conv3d_nhwc* g = &cg.g;
  const int M = g->B * g->OD * g->OH * g->OW, N = g->Cout, K = g->KD * g->KH * g->KW * g->C;
  if (!conv_ok(cg) || N % 4 != 0 || !aligned16(dy) || !aligned16(a) || rng_w->elem_offset % 4 != 0 || !aligned16(rho_w) ||
      !aligned16(dmu_w) || !aligned16(drho_w) || (eps_w != nullptr && !aligned16(eps_w)))
    return kNotEligible;
  TmaWgradParams p{};
  int rc = make_map(&p.map_dy, dy, N, M, shared_dy ? 1 : S, N, static_cast<int64_t>(M) * N, kWgRows, true);
  if (rc != BNN_OK) return rc;
  rc = make_im2col_map(&p.map_a, a, g->C, g->W, g->H, static_cast<int64_t>(shared_a ? 1 : S) * g->B, -g->pw, -g->ph,
                       g->pw - (g->KW - 1) * g->dw, g->ph - (g->KH - 1) * g->dh, g->sw, g->sh, kWgRows, true,
                       depth_fwd(cg));
  if (rc != BNN_OK) return rc;
  p.conv = conv_coords_fwd(cg);
  p.rho_w = rho_w; p.eps_w = eps_w; p.dmu_w = dmu_w; p.drho_w = drho_w;
  p.M = M; p.N = N; p.K = K; p.S = S; p.sample_begin = sample_begin;
  p.rng_w = *rng_w;
  p.shared_a = shared_a ? 1 : 0;
  p.shared_dy = shared_dy ? 1 : 0;
  return wgrad_plan_and_launch(p, M, N, K, S, st);
}

// ---------------------------------------------------------------------------------------------- transposed-filter gather
// The input gradient of a stride-1 convolution is a gather like the forward pass, no column matrix and no scatter:
//   dX[n][h][w][c] = sum_{kh, kw, o} dY[n][h + ph - kh dh][w + pw - kw dw][o] W[o][kh][kw][c]
// an im2col load of dY with lower corner p - (K - 1) d, taps walked in flipped order.
// A transposed convolution with weight W [Cin][Cout][KH][KW] is the adjoint of its CONV VIEW, the convolution from the
// transposed output (C = Cout channels, H x W) to the transposed input (Cout_view = Cin channels, OH x OW) with the same W
// read as OIHW.  Its forward is therefore the conv view's data gradient plus a bias:
//   y[n][h][w][c] = b[c] + sum_{kh, kw, o : (h + ph - kh dh) % sh == 0, ...} x[n][(h + ph - kh dh) / sh][..][o] W[o][kh][kw][c]
// Split the outputs into sh x sw phases (h % sh, w % sw).  In phase r a tap contributes iff (r + ph - kh dh) % sh == 0,
// and then from input row i + (r + ph - kh dh) / sh for output row r + sh i: every phase is a STRIDE-1 gather over x with
// its own taps (tdh = sh / gcd(sh, dh) apart, dh / gcd(sh, dh) input rows apart) and its own im2col corner.  One launch of
// the data-gradient kernel per phase walks exactly that phase's taps x 32-channel blocks (no MMA on inserted zeros) and
// writes its rows through a phase view; phases without a tap get the bias alone.  At stride 1 there is one phase with
// every tap: the conv input gradient above, written through the plain row view.  A 3-d transposed convolution adds the
// depth as a third phase dimension (sd x sh x sw phases) and a depth level to the phase view.
namespace {
struct PhaseDim {
  int r, rows;              // phase offset, output rows of the phase
  int taps, tlast, tstep;   // taps of the phase, the last one, their spacing
  int lo, dstep;            // input row of (phase row 0, last tap) and input-row distance of consecutive walked taps
};
int gcd_int(int a, int b) { while (b != 0) { const int t = a % b; a = b; b = t; } return a; }
// one dimension of output size n_out (the conv view's input size)
PhaseDim phase_dim(int r, int n_out, int s, int pad, int d, int k) {
  PhaseDim pd{};
  pd.r = r;
  pd.rows = (n_out - r + s - 1) / s;
  const int gd = gcd_int(s, d);
  pd.tstep = s / gd;
  pd.dstep = d / gd;
  pd.taps = 0;
  pd.tlast = -1;
  for (int kk = 0; kk < k; ++kk)
    if ((((r + pad - kk * d) % s) + s) % s == 0) { ++pd.taps; pd.tlast = kk; }
  pd.lo = pd.taps > 0 ? (r + pad - pd.tlast * d) / s : 0;     // exact division
  return pd;
}

// the phases of a request, depth-major: (d, h, w) phase dimensions; a 2-d request has one depth phase of one row
struct Phase {
  PhaseDim d, h, w;
};
template <class F>
void for_each_phase(const ConvGeom& cg, F&& f) {
  const bnn_conv3d_nhwc& g = cg.g;
  const int ph_d = g.sd < g.D ? g.sd : g.D, ph_h = g.sh < g.H ? g.sh : g.H, ph_w = g.sw < g.W ? g.sw : g.W;
  for (int rd = 0; rd < ph_d; ++rd)
    for (int rh = 0; rh < ph_h; ++rh)
      for (int rw = 0; rw < ph_w; ++rw)
        f(Phase{phase_dim(rd, g.D, g.sd, g.pd, g.dd, g.KD), phase_dim(rh, g.H, g.sh, g.ph, g.dh, g.KH),
                phase_dim(rw, g.W, g.sw, g.pw, g.dw, g.KW)});
}
// every phase's corners and tap offsets within the im2col descriptor's range
bool phases_ok(const ConvGeom& cg) {
  const bnn_conv3d_nhwc& g = cg.g;
  bool ok = true;
  auto dim_ok = [&](const PhaseDim& a, int n_in) {
    return corner_ok(a.lo, cg.vol) && corner_ok(a.lo + a.rows - n_in, cg.vol) && extent_ok((a.taps - 1) * a.dstep, cg.vol);
  };
  for_each_phase(cg, [&](const Phase& ph) {
    if (ph.d.taps == 0 || ph.h.taps == 0 || ph.w.taps == 0) return;
    ok = ok && dim_ok(ph.h, g.OH) && dim_ok(ph.w, g.OW) && (!cg.vol || dim_ok(ph.d, g.OD));
  });
  return ok;
}

__global__ void phase_bias_kernel(float* y, int64_t ss, int64_t s_img, int64_t s_a, int64_t s_i, int64_t s_j, int S, int B,
                                  int planes, int rows, int cols, int C, const float* mu_b, const float* sigma_b,
                                  const float* eps_b, uint32_t sample_begin, bnn_rng rng_b) {
  const int64_t total = static_cast<int64_t>(S) * B * planes * rows * cols * C;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int64_t q = t;
    const int c = static_cast<int>(q % C); q /= C;
    const int j = static_cast<int>(q % cols); q /= cols;
    const int i = static_cast<int>(q % rows); q /= rows;
    const int a = static_cast<int>(q % planes); q /= planes;
    const int img = static_cast<int>(q % B);
    const int s = static_cast<int>(q / B);
    float b = 0.f;
    if (mu_b != nullptr) {
      const float e = eps_b ? __ldg(eps_b + static_cast<int64_t>(s) * C + c)
                            : eps1(resolve_rng(rng_b), sample_begin + s, static_cast<uint64_t>(c));
      b = fmaf(__ldg(sigma_b + c), e, __ldg(mu_b + c));
    }
    y[s * ss + img * s_img + a * s_a + i * s_i + j * s_j + c] = b;
  }
}
}  // namespace

int conv_transpose_phases(const ConvGeom& cg, int32_t* out, int max_phases) {
  const int per = cg.vol ? 21 : 14;
  int n = 0;
  for_each_phase(cg, [&](const Phase& ph) {
    if (n < max_phases) {
      int32_t* o = out + per * n;
      const PhaseDim* dims[3] = {&ph.d, &ph.h, &ph.w};
      const int first = cg.vol ? 0 : 1, nd = 3 - first;
      for (int k = 0; k < nd; ++k) {
        const PhaseDim& a = *dims[first + k];
        const int32_t v[7] = {a.r, a.rows, a.taps, a.tlast, a.tstep, a.lo, a.dstep};
        for (int f = 0; f < 7; ++f) o[f * nd + k] = v[f];
      }
    }
    ++n;
  });
  return n;
}

bool conv_transpose_ok(const ConvGeom& cg) {
  const bnn_conv3d_nhwc& g = cg.g;
  // the 3-d phase view addresses within an output image in 32 bits
  return g.Cout % kBK == 0 && static_cast<int64_t>(g.D) * g.H * g.W * g.C < (int64_t(1) << 31) && conv_ok(cg) &&
         phases_ok(cg);
}

// x: the gathered NHWC tensor [S or 1][B][OH][OW][Cout] (conv view), shared_x: all samples read sample 0 of x; y: the
// NHWC output [S][B][H][W][C] with the optional sampled bias, or with sum_samples one output summed over the samples
int tma_conv_gather(const float* x, bool shared_x, const float* mu_w, const float* sigma_w, const float* mu_b,
                    const float* sigma_b, const float* eps_w, const float* eps_b, float* y, int64_t y_sample_stride,
                    bool sum_samples, const ConvGeom& cg, int S, uint32_t sample_begin, const bnn_rng* rng_w,
                    const bnn_rng* rng_b, cudaStream_t st) {
  const bnn_conv3d_nhwc* g = &cg.g;
  // conv view: C = gathered output channels (the drained columns), Cout = channels of x (reduction)
  if (g->Cout % kBK != 0 || g->C % 4 != 0 || g->sh > 8 || g->sw > 8 || g->sd > 8 || !aligned16(x) || !aligned16(y) ||
      rng_w->elem_offset % 4 != 0 || !aligned16(mu_w) || !aligned16(sigma_w) || (eps_w != nullptr && !aligned16(eps_w)))
    return kNotEligible;
  // checked for every phase before anything is launched
  if (!phases_ok(cg)) return kNotEligible;
  const bool phased = g->sh != 1 || g->sw != 1 || g->sd != 1;
  const int64_t C = g->C, img_y = static_cast<int64_t>(g->D) * g->H * g->W * C;
  int rc = BNN_OK;
  for_each_phase(cg, [&](const Phase& ph) {
    if (rc != BNN_OK) return;
    const PhaseDim &e = ph.d, &a = ph.h, &b = ph.w;
    float* base = y + ((static_cast<int64_t>(e.r) * g->H + a.r) * g->W + b.r) * C;
    if (e.taps == 0 || a.taps == 0 || b.taps == 0) {
      const int64_t total = static_cast<int64_t>(S) * g->B * e.rows * a.rows * b.rows * C;
      const int blocks = static_cast<int>(std::min<int64_t>((total + 255) / 256, 4 * sm_count()));
      phase_bias_kernel<<<blocks, 256, 0, st>>>(base, y_sample_stride, img_y, g->sd * g->H * g->W * C, g->sh * g->W * C,
                                                g->sw * C, S, g->B, e.rows, a.rows, b.rows, g->C, mu_b, sigma_b, eps_b,
                                                sample_begin, rng_b ? *rng_b : *rng_w);
      const cudaError_t err = cudaGetLastError();
      if (err != cudaSuccess) rc = fail(BNN_ERR_CUDA, "phase_bias_kernel: %s", cudaGetErrorString(err));
      return;
    }
    TmaContractParams p{};
    const int up_h = a.lo + a.rows - g->OH, up_w = b.lo + b.rows - g->OW;
    rc = make_im2col_map(&p.map_l, x, g->Cout, g->OW, g->OH, static_cast<int64_t>(shared_x ? 1 : S) * g->B, b.lo, a.lo,
                         up_w, up_h, 1, 1, 128, false, Im2colDepth{cg.vol, g->OD, e.lo, e.lo + e.rows - g->OD, 1});
    if (rc != BNN_OK) return;
    ConvCoords c{};
    c.on = cg.vol ? 2 : 1; c.P = e.rows * a.rows * b.rows; c.OW = b.rows; c.imgs = g->B; c.sh = 1; c.sw = 1;
    c.lh = a.lo; c.lw = b.lo; c.dh = a.dstep; c.dw = b.dstep; c.KW = b.taps; c.taps = e.taps * a.taps * b.taps;
    c.cblocks = g->Cout / kBK; c.w_rows = g->Cout; c.chans = g->Cout;
    c.wtaps = g->KD * g->KH * g->KW; c.wKW = g->KW; c.tkh = a.tlast; c.tkw = b.tlast; c.tdh = a.tstep; c.tdw = b.tstep;
    c.HW = a.rows * b.rows; c.sd = 1; c.ld = e.lo; c.dd = e.dstep; c.KH = a.taps; c.KHW = a.taps * b.taps;
    c.tkd = e.tlast; c.tdd = e.tstep; c.wKH = g->KH;
    p.conv = c;
    p.out.base = base; p.out.bs = g->sw * C; p.out.P = 1;
    if (phased) {
      p.out.pw = b.rows; p.out.pimg = c.P; p.out.s_i = g->sh * g->W * C; p.out.s_img = img_y;
      p.out.pplane = a.rows * b.rows; p.out.s_a = static_cast<int64_t>(g->sd) * g->H * g->W * C;
    }
    p.out_sample_stride = y_sample_stride;
    p.mu_w = mu_w; p.sigma_w = sigma_w; p.eps_w = eps_w; p.mu_b = mu_b; p.sigma_b = sigma_b; p.eps_b = eps_b;
    p.M = g->B * c.P; p.N = c.taps * g->Cout; p.K = g->C; p.S = S; p.sample_begin = sample_begin;
    p.w_numel = static_cast<int64_t>(g->Cout) * c.wtaps * g->C;
    p.rng_w = *rng_w; p.rng_b = rng_b ? *rng_b : *rng_w;
    p.shared_l = shared_x ? 1 : 0;
    p.sum_samples = sum_samples ? 1 : 0;
    // C % 4 == 0: with a 4-aligned sample stride every CTA takes the staged drain, the only one with the phase view
    p.vec_out = (y_sample_stride % 4 == 0);
    rc = dispatch_tma_contract<true>(p, p.K, st);
  });
  return rc;
}

int tma_conv_transpose_dgrad(const float* dy, const float* mu_w, const float* sigma_w, const float* eps_w, float* dx,
                             int64_t x_sample_stride, const ConvGeom& cg, int S, uint32_t sample_begin,
                             const bnn_rng* rng_w, cudaStream_t st) {
  const bnn_conv3d_nhwc* g = &cg.g;
  if (!conv_ok(cg) || g->Cout % 4 != 0 || !aligned16(dy) || !aligned16(dx) || rng_w->elem_offset % 4 != 0 ||
      !aligned16(mu_w) || !aligned16(sigma_w) || (eps_w != nullptr && !aligned16(eps_w)))
    return kNotEligible;
  bnn_view v{};
  v.base = dx; v.batch_stride = g->Cout; v.P = 1;
  return conv_fwd_launch(dy, static_cast<int64_t>(g->B) * g->D * g->H * g->W * g->C, mu_w, sigma_w, nullptr, nullptr, eps_w,
                         nullptr, v, x_sample_stride, cg, S, sample_begin, rng_w, nullptr, x_sample_stride == 0, st);
}

int tma_wait_counters(unsigned long long* out8, int reset) {
#ifdef BNN_PROFILE_WAITS
  BNN_CUDA_OK(cudaMemcpyFromSymbol(out8, g_wait_cycles, 8 * sizeof(unsigned long long)));
  if (reset) {
    unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    BNN_CUDA_OK(cudaMemcpyToSymbol(g_wait_cycles, z, sizeof(z)));
  }
  return BNN_OK;
#else
  (void)out8; (void)reset;
  return kNotEligible;
#endif
}

int tma_stage_counters(unsigned long long* out8, int reset) {
#ifdef BNN_PROFILE_WAITS
  BNN_CUDA_OK(cudaMemcpyFromSymbol(out8, g_stage_cycles, 8 * sizeof(unsigned long long)));
  if (reset) {
    unsigned long long z[8] = {0, 0, 0, 0, 0, 0, ~0ull, 0};
    BNN_CUDA_OK(cudaMemcpyToSymbol(g_stage_cycles, z, sizeof(z)));
  }
  return BNN_OK;
#else
  (void)out8; (void)reset;
  return kNotEligible;
#endif
}

int tma_pair_tile_plan(int m_blocks, int S, int slots, int32_t* out7) {      // host only: the plan the launcher would use
  TilePlan plan{};
  solve_pair_tiles(&plan, m_blocks, S, slots);
  out7[0] = plan.on; out7[1] = plan.n_a; out7[2] = plan.s1; out7[3] = plan.a1; out7[4] = plan.b1; out7[5] = plan.a2; out7[6] = plan.b2;
  return BNN_OK;
}

int tma_force_variant(int variant) {
  const bool ok = variant == -1 || variant == 0 || variant == 1 || variant == 2 || variant == 4;
  g_forced_variant.store(ok ? variant : -1, std::memory_order_relaxed);
  return BNN_OK;
}

int tma_selftest(float* max_err_dev, cudaStream_t st) {
  selftest_mn_kernel<<<1, 128, 0, st>>>(max_err_dev, 3);
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}

}  // namespace contract
}  // namespace bnn
