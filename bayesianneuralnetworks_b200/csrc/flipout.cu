// flipout.cu — the sign algebra around the two contractions of the Flipout transposed convolution layers
// (FlipOutNormalConvTranspose1d / 2d / 3d):  y = convT(x, mu) + R o convT(x o S, sigma), and in the backward pass
// dx = convT^T(g, mu) + S o convT^T(R o g, sigma).  The contraction kernels read and write channels-last activations.
//
//   bnn_flipout_split    a ([n][C][P] or channels-last [n][P][C]) -> a in channels-last (skipped when it already is)
//                        and sign[n][c] * a in channels-last, one read of a
//   bnn_flipout_combine  channels-last a, b -> a + sign[n][c] * b, NC(D)HW-contiguous or channels-last
//
// The arithmetic is torch's: the sign product is exact, then one fp32 add, so the results are bit-identical to
// `a * s` and `a + b * s`.  A layout change goes through a 32-channel x 64-pixel shared-memory tile (both sides
// coalesced; no limit on the size of an image); a layout-preserving call is one flat vectorised pass.  Indices are
// 64-bit.
#include "common.cuh"

namespace bnn {
namespace {

constexpr int kThreads = 256;              // 32 x 8
constexpr int kTileC = 32, kTileP = 64;
constexpr int kPitch = kTileP + 1;         // [c][p] tile, odd pitch: conflict-free along c and along p

int grid_for(int64_t items, int waves) {
  const int64_t cap = static_cast<int64_t>(sm_count()) * waves;
  return static_cast<int>(items < 1 ? 1 : (items < cap ? items : cap));
}

// kCombine = false: a is [n][C][P]; writes a_cl (channels-last copy) and sa_cl = sign * a (channels-last).
// kCombine = true:  a, b are [n][P][C]; writes out = a + sign * b as [n][C][P].
template <bool kCombine>
__global__ void __launch_bounds__(kThreads) flipout_transpose_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                                     const float* __restrict__ sign, float* __restrict__ out0,
                                                                     float* __restrict__ out1, int64_t n, int C, int64_t P) {
  __shared__ float tile[kTileC * kPitch];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t p_tiles = (P + kTileP - 1) / kTileP;
  const int64_t c_tiles = (C + kTileC - 1) / kTileC;
  const int64_t tiles = n * c_tiles * p_tiles;
  const int64_t CP = static_cast<int64_t>(C) * P;
  for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
    const int64_t pt = t % p_tiles, rest = t / p_tiles;
    const int c0 = static_cast<int>(rest % c_tiles) * kTileC;
    const int64_t img = rest / c_tiles;
    const int64_t p0 = pt * kTileP;
    const float* sg = sign + img * C;
    __syncthreads();                       // the previous tile has been written out
    if (!kCombine) {
      // NCHW side: rows c, pixels contiguous
      float v[kTileC / 8][kTileP / 32];
#pragma unroll
      for (int i = 0; i < kTileC / 8; ++i)
#pragma unroll
        for (int j = 0; j < kTileP / 32; ++j) {
          const int c = c0 + ty + 8 * i;
          const int64_t p = p0 + tx + 32 * j;
          v[i][j] = (c < C && p < P) ? __ldg(a + img * CP + static_cast<int64_t>(c) * P + p) : 0.f;
        }
#pragma unroll
      for (int i = 0; i < kTileC / 8; ++i)
#pragma unroll
        for (int j = 0; j < kTileP / 32; ++j) tile[(ty + 8 * i) * kPitch + tx + 32 * j] = v[i][j];
      __syncthreads();
      // channels-last side: rows p, channels contiguous; this thread's channel is fixed
      const int c = c0 + tx;
      if (c < C) {
        const float s = __ldg(sg + c);
#pragma unroll
        for (int i = 0; i < kTileP / 8; ++i) {
          const int pl = ty + 8 * i;
          const int64_t p = p0 + pl;
          if (p < P) {
            const float x = tile[tx * kPitch + pl];
            const int64_t o = img * CP + p * C + c;
            if (out0 != nullptr) out0[o] = x;
            out1[o] = s * x;
          }
        }
      }
    } else {
      // channels-last side: rows p, channels contiguous; the sign of this thread's channel is applied on the way in
      const int c = c0 + tx;
      const float s = c < C ? __ldg(sg + c) : 0.f;
      float va[kTileP / 8], vb[kTileP / 8];
#pragma unroll
      for (int i = 0; i < kTileP / 8; ++i) {
        const int64_t p = p0 + ty + 8 * i;
        const bool in = c < C && p < P;
        const int64_t o = img * CP + p * C + c;
        va[i] = in ? __ldg(a + o) : 0.f;
        vb[i] = in ? __ldg(b + o) : 0.f;
      }
#pragma unroll
      for (int i = 0; i < kTileP / 8; ++i) tile[tx * kPitch + ty + 8 * i] = __fadd_rn(va[i], __fmul_rn(s, vb[i]));
      __syncthreads();
      // NCHW side: rows c, pixels contiguous
#pragma unroll
      for (int i = 0; i < kTileC / 8; ++i)
#pragma unroll
        for (int j = 0; j < kTileP / 32; ++j) {
          const int cl = ty + 8 * i;
          const int64_t p = p0 + tx + 32 * j;
          if (c0 + cl < C && p < P) out0[img * CP + static_cast<int64_t>(c0 + cl) * P + p] = tile[cl * kPitch + tx + 32 * j];
        }
    }
  }
}

// Layout-preserving form over channels-last tensors [n][P][C] seen as one flat array: kCombine = false writes
// out = sign * a, kCombine = true writes out = a + sign * b.  A block takes kSpan consecutive elements per step; their
// channel is (start % C + offset) % C in 32 bits (an image boundary is a multiple of C), their image advances past
// image boundaries without a 64-bit division per element.  kVec: float4 of four channels of one pixel (C % 4 == 0,
// 16-byte aligned tensors).
constexpr int kSpan = 4096;
template <bool kCombine, bool kVec>
__global__ void __launch_bounds__(kThreads) flipout_flat_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                                const float* __restrict__ sign, float* __restrict__ out,
                                                                int64_t n, int C, int64_t P) {
  constexpr int kW = kVec ? 4 : 1;
  constexpr int kPer = kSpan / (kThreads * kW);
  const int64_t CP = static_cast<int64_t>(C) * P, total = n * CP;
  for (int64_t start = static_cast<int64_t>(blockIdx.x) * kSpan; start < total;
       start += static_cast<int64_t>(gridDim.x) * kSpan) {
    const int64_t img0 = start / CP, rem = start - img0 * CP;
    const uint32_t c_start = static_cast<uint32_t>(rem % C);
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int off = (u * kThreads + static_cast<int>(threadIdx.x)) * kW;
      const int64_t e = start + off;
      if (e >= total) break;
      const int64_t into = rem + off;      // offset from the start of image img0
      const int64_t img = img0 + (CP > kSpan ? static_cast<int64_t>(into >= CP)
                                             : static_cast<int64_t>(static_cast<uint32_t>(into) / static_cast<uint32_t>(CP)));
      const uint32_t c = (c_start + static_cast<uint32_t>(off)) % static_cast<uint32_t>(C);
      const float* sg = sign + img * C + c;
      if (kVec) {
        const float4 s = __ldg(reinterpret_cast<const float4*>(sg));
        const float4 x = ldg_stream4(a + e);
        float4 r;
        if (kCombine) {
          const float4 y = ldg_stream4(b + e);
          r = make_float4(__fadd_rn(x.x, __fmul_rn(s.x, y.x)), __fadd_rn(x.y, __fmul_rn(s.y, y.y)),
                          __fadd_rn(x.z, __fmul_rn(s.z, y.z)), __fadd_rn(x.w, __fmul_rn(s.w, y.w)));
        } else {
          r = make_float4(s.x * x.x, s.y * x.y, s.z * x.z, s.w * x.w);
        }
        *reinterpret_cast<float4*>(out + e) = r;
      } else {
        const float s = __ldg(sg);
        out[e] = kCombine ? __fadd_rn(__ldg(a + e), __fmul_rn(s, __ldg(b + e))) : s * __ldg(a + e);
      }
    }
  }
}

int check_sizes(int64_t n, int32_t C, int64_t P, const char* who) {
  BNN_REQUIRE(n > 0 && C > 0 && P > 0, BNN_ERR_BAD_ARGUMENT, "%s: bad shape (n = %lld, C = %d, P = %lld)", who,
              static_cast<long long>(n), C, static_cast<long long>(P));
  BNN_REQUIRE(P <= INT64_MAX / C && n <= INT64_MAX / (static_cast<int64_t>(C) * P), BNN_ERR_BAD_ARGUMENT,
              "%s: n * C * P overflows 64 bits", who);
  return BNN_OK;
}

int launch_flat(bool combine, const float* a, const float* b, const float* sign, float* out, int64_t n, int32_t C,
                int64_t P, cudaStream_t stream) {
  const bool vec = C % 4 == 0 && aligned16(a) && aligned16(out) && aligned16(sign) && (b == nullptr || aligned16(b));
  const int grid = grid_for((n * C * P + kSpan - 1) / kSpan, 8);
  if (combine) {
    if (vec) flipout_flat_kernel<true, true><<<grid, kThreads, 0, stream>>>(a, b, sign, out, n, C, P);
    else flipout_flat_kernel<true, false><<<grid, kThreads, 0, stream>>>(a, b, sign, out, n, C, P);
  } else {
    if (vec) flipout_flat_kernel<false, true><<<grid, kThreads, 0, stream>>>(a, b, sign, out, n, C, P);
    else flipout_flat_kernel<false, false><<<grid, kThreads, 0, stream>>>(a, b, sign, out, n, C, P);
  }
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}

int64_t transpose_tiles(int64_t n, int32_t C, int64_t P) {
  return n * ((C + kTileC - 1) / kTileC) * ((P + kTileP - 1) / kTileP);
}

}  // namespace
}  // namespace bnn

using namespace bnn;

extern "C" {

int bnn_flipout_split(const float* a, int32_t a_channels_last, const float* sign, float* a_cl, float* sa_cl, int64_t n,
                      int32_t C, int64_t P, void* stream) {
  int rc = check_sizes(n, C, P, "bnn_flipout_split");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(a && sign && sa_cl && (a_channels_last || a_cl), BNN_ERR_BAD_ARGUMENT,
              "bnn_flipout_split: NULL pointer (a_cl is required unless a is channels-last)");
  rc = check_device();
  if (rc != BNN_OK) return rc;
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (a_channels_last) return launch_flat(false, a, nullptr, sign, sa_cl, n, C, P, s);
  flipout_transpose_kernel<false><<<grid_for(transpose_tiles(n, C, P), 8), kThreads, 0, s>>>(a, nullptr, sign, a_cl, sa_cl,
                                                                                             n, C, P);
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}

int bnn_flipout_combine(const float* a, const float* b, const float* sign, float* out, int32_t out_channels_last,
                        int64_t n, int32_t C, int64_t P, void* stream) {
  int rc = check_sizes(n, C, P, "bnn_flipout_combine");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(a && b && sign && out, BNN_ERR_BAD_ARGUMENT, "bnn_flipout_combine: NULL pointer");
  rc = check_device();
  if (rc != BNN_OK) return rc;
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (out_channels_last) return launch_flat(true, a, b, sign, out, n, C, P, s);
  flipout_transpose_kernel<true><<<grid_for(transpose_tiles(n, C, P), 8), kThreads, 0, s>>>(a, b, sign, out, nullptr, n,
                                                                                            C, P);
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}

}  // extern "C"
