// conv.cu — entry points of the implicit-GEMM convolution path (NormalConv2d / NormalConv1d, reference conv.py:65-73,
// 89-96,112-119 and their autograd) and the small layout kernels around it.
//
// Layouts.  Activations NHWC (torch.channels_last memory): [S*B][H][W][C].  Weights in (o, kh, kw, c) order, so that the
// GEMM's k index (tap, channel) walks memory contiguously and a 32-wide k-block is one filter tap x 32 channels — exactly
// the box an im2col tensor map delivers.  bnn_conv2d_weight_layout produces that order (and sigma) from the reference's
// OIHW parameters once per step; the layer's eps stream is DEFINED over the (o, kh, kw, c) order (eps is i.i.d., so the
// distribution of the sampled weights is the reference's; `.sampled` and eps injection permute on the way in and out).
//
// bnn_im2col_nhwc / bnn_col2im_nhwc are the explicit lowering in the same (kh, kw, c) column order, for the requests
// the TMA path does not take: fp32 (3xTF32) mode and the input gradient of strided layers.
//
// The transposed layers (NormalConvTranspose1d / 2d / 3d) run on the same kernels through their conv view; the 3-d entry
// points (NDHWC tensors, rank-5 im2col maps) check one eligibility predicate for their three passes.
#include "contract.cuh"

namespace bnn {
namespace {

constexpr int kThreads = 256;

__global__ void __launch_bounds__(kThreads) weight_layout_kernel(const float* __restrict__ mu, const float* __restrict__ rho,
                                                                 float* __restrict__ mu_p, float* __restrict__ sigma_p,
                                                                 float* __restrict__ rho_p, int Cg, int taps, int64_t total) {
  for (int64_t j = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; j < total;
       j += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(j % Cg);
    const int64_t t = j / Cg;
    const int tap = static_cast<int>(t % taps);
    const int64_t o = t / taps;
    const int64_t i = (o * Cg + c) * taps + tap;          // OIHW index
    const float r = __ldg(rho + i);
    mu_p[j] = __ldg(mu + i);
    if (sigma_p != nullptr) sigma_p[j] = stddev_exact(r);
    if (rho_p != nullptr) rho_p[j] = r;
  }
}

// out (OIHW) <- in ((o, kh, kw, c) order), n_arrays arrays back to back (the gradients of mean and scale)
__global__ void __launch_bounds__(kThreads) weight_unlayout_kernel(const float* __restrict__ in, float* __restrict__ out, int Cg,
                                                                   int taps, int64_t per_array, int64_t total) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t a = i / per_array, e = i - a * per_array;
    const int tap = static_cast<int>(e % taps);
    const int64_t t = e / taps;
    const int c = static_cast<int>(t % Cg);
    const int64_t o = t / Cg;
    out[i] = __ldg(in + a * per_array + (o * taps + tap) * Cg + c);
  }
}

// col[m][(kh * KW + kw) * C + c] = x[n][oh*sh - ph + kh*dh][ow*sw - pw + kw*dw][c]  (0 outside), m = (n, oh, ow); one
// float4 of channels per thread: both sides coalesced
__global__ void __launch_bounds__(kThreads) im2col_nhwc_kernel(const float* __restrict__ x, float* __restrict__ col,
                                                               const bnn_conv2d_nhwc g, int64_t n_imgs) {
  const int c4s = g.C / 4, taps = g.KH * g.KW;
  const int64_t total = n_imgs * g.OH * g.OW * taps * c4s;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c4 = static_cast<int>(i % c4s);
    int64_t t = i / c4s;
    const int tap = static_cast<int>(t % taps);
    t /= taps;
    const int ow = static_cast<int>(t % g.OW);
    t /= g.OW;
    const int oh = static_cast<int>(t % g.OH);
    const int64_t n = t / g.OH;
    const int kh = tap / g.KW, kw = tap - kh * g.KW;
    const int h = oh * g.sh - g.ph + kh * g.dh, w = ow * g.sw - g.pw + kw * g.dw;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (h >= 0 && h < g.H && w >= 0 && w < g.W)
      v = __ldg(reinterpret_cast<const float4*>(x + ((n * g.H + h) * g.W + w) * g.C) + c4);
    reinterpret_cast<float4*>(col)[i] = v;
  }
}

// dx[n][h][w][c] = sum over the (oh, kh), (ow, kw) that hit (h, w) of dcol[(n, oh, ow)][(kh*KW + kw)*C + c]: gather form
__global__ void __launch_bounds__(kThreads) col2im_nhwc_kernel(const float* __restrict__ dcol, float* __restrict__ dx,
                                                               const bnn_conv2d_nhwc g, int64_t n_imgs) {
  const int c4s = g.C / 4, taps = g.KH * g.KW;
  const int64_t total = n_imgs * g.H * g.W * c4s;
  const int64_t K4 = static_cast<int64_t>(taps) * c4s;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c4 = static_cast<int>(i % c4s);
    int64_t t = i / c4s;
    const int w = static_cast<int>(t % g.W);
    t /= g.W;
    const int h = static_cast<int>(t % g.H);
    const int64_t n = t / g.H;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int kh = 0; kh < g.KH; ++kh) {
      const int hh = h + g.ph - kh * g.dh;
      if (hh < 0 || hh % g.sh != 0) continue;
      const int oh = hh / g.sh;
      if (oh >= g.OH) continue;
      for (int kw = 0; kw < g.KW; ++kw) {
        const int ww = w + g.pw - kw * g.dw;
        if (ww < 0 || ww % g.sw != 0) continue;
        const int ow = ww / g.sw;
        if (ow >= g.OW) continue;
        const float4 v = __ldg(reinterpret_cast<const float4*>(dcol) + ((n * g.OH + oh) * g.OW + ow) * K4 +
                               static_cast<int64_t>(kh * g.KW + kw) * c4s + c4);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
    }
    reinterpret_cast<float4*>(dx)[i] = acc;
  }
}

// dY of a conv layer arrives from autograd NCHW-contiguous ([R][N][P], P = OH*OW) whenever the layer's output was; the
// implicit-GEMM kernels want it as rows [R*P][N] (NHWC).  One block transposes `ipb` images through shared memory — an
// image's N*P block is contiguous on both sides, so reads and writes are fully coalesced — and, while the values are
// there, sums every column: the reparameterised bias gradient (SURVEY §3.2: c_s[n] = sum_m dY[s][m][n]; dmu_b += sum_s
// c_s; drho_b += sum_s c_s eps_b(s, n) sigmoid(rho_b[n])) costs no second pass over dY.
// division of a 32-bit index by a launch constant without the ~20-instruction integer divide (Granlund-Montgomery):
// q = (umulhi(n, mul) + n) >> shift, exact for every n < 2^31 (the indices here are < 2^27)
struct FastDiv {
  uint32_t mul, shift, d;
};
inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f;
  f.d = d;
  uint32_t s = 0;
  while ((1u << s) < d) ++s;
  f.shift = s;
  f.mul = static_cast<uint32_t>(((uint64_t(1) << 32) * ((uint64_t(1) << s) - d)) / d + 1);
  return f;
}
__device__ __forceinline__ uint32_t fdiv(uint32_t n, const FastDiv& f) {
  return static_cast<uint32_t>((static_cast<uint64_t>(__umulhi(n, f.mul)) + n) >> f.shift);
}

__global__ void __launch_bounds__(kThreads) nchw_to_nhwc_bias_kernel(const float* __restrict__ dy, float* __restrict__ out,
                                                                     int64_t n_imgs, int B, int N, int P, int ipt, int passes,
                                                                     const float* __restrict__ rho_b,
                                                                     const float* __restrict__ eps_b, float* __restrict__ dmu_b,
                                                                     float* __restrict__ drho_b, uint32_t sample_begin,
                                                                     bnn_rng rng, int vec, FastDiv dNP, FastDiv dP, FastDiv dN) {
  extern __shared__ float s_tile[];          // ipt images x [P][N + 1]
  const int pitch = N + 1, NP = N * P, img_smem = P * pitch;
  const bool want_bias = dmu_b != nullptr;
  const RngKey key = resolve_rng(rng);
  float acc = 0.f;                           // column sum of thread n = threadIdx.x over the images of one sample
  int cur_s = -1;
  auto flush = [&](int s) {
    if (!want_bias || s < 0) return;
    const int n = threadIdx.x;               // N <= kThreads on this path (checked by the host)
    if (n < N) {
      const float e = eps_b != nullptr ? __ldg(eps_b + static_cast<int64_t>(s) * N + n)
                                       : eps1(key, sample_begin + s, static_cast<uint64_t>(n));
      atomicAdd(dmu_b + n, acc);
      atomicAdd(drho_b + n, acc * e * sigmoid_fast(__ldg(rho_b + n)));
    }
    acc = 0.f;
  };
  // element i of the block's run of images -> (image, n, p) on the NCHW side, (image, p, n) on the NHWC side
  auto split_nchw = [&](int i, int& im, int& n, int& pp) {
    im = static_cast<int>(fdiv(i, dNP));
    const int r = i - im * NP;
    n = static_cast<int>(fdiv(r, dP));
    pp = r - n * P;
  };
  auto split_nhwc = [&](int i, int& im, int& pp, int& n) {
    im = static_cast<int>(fdiv(i, dNP));
    const int r = i - im * NP;
    pp = static_cast<int>(fdiv(r, dN));
    n = r - pp * N;
  };
  for (int pass = 0; pass < passes; ++pass) {
    const int64_t img0 = (static_cast<int64_t>(blockIdx.x) * passes + pass) * ipt;
    if (img0 >= n_imgs) break;
    const int here = n_imgs - img0 < ipt ? static_cast<int>(n_imgs - img0) : ipt;
    const int total = here * NP;
    const float* src = dy + img0 * NP;
    float* dst = out + img0 * NP;
    __syncthreads();
    // several independent loads in flight per thread before the first (dependent) shared-memory store
    if (vec) {                               // P % 4 == 0: a float4 holds (n, p .. p + 3)
      for (int i0 = threadIdx.x * 4; i0 < total; i0 += kThreads * 16) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + u * (kThreads * 4);
          if (i < total) v[u] = ldg_stream4(src + i);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + u * (kThreads * 4);
          if (i < total) {
            int im, n, pp;
            split_nchw(i, im, n, pp);
            float* t = s_tile + im * img_smem + pp * pitch + n;
            t[0] = v[u].x; t[pitch] = v[u].y; t[2 * pitch] = v[u].z; t[3 * pitch] = v[u].w;
          }
        }
      }
    } else {
      for (int i0 = threadIdx.x; i0 < total; i0 += kThreads * 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = i0 + u * kThreads;
          if (i < total) v[u] = __ldg(src + i);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = i0 + u * kThreads;
          if (i < total) {
            int im, n, pp;
            split_nchw(i, im, n, pp);
            s_tile[im * img_smem + pp * pitch + n] = v[u];
          }
        }
      }
    }
    __syncthreads();
    if (vec && N % 4 == 0) {
      for (int i = threadIdx.x * 4; i < total; i += kThreads * 4) {
        int im, pp, n;
        split_nhwc(i, im, pp, n);
        const float* t = s_tile + im * img_smem + pp * pitch + n;
        *reinterpret_cast<float4*>(dst + i) = make_float4(t[0], t[1], t[2], t[3]);
      }
    } else {
      for (int i = threadIdx.x; i < total; i += kThreads) {
        int im, pp, n;
        split_nhwc(i, im, pp, n);
        dst[i] = s_tile[im * img_smem + pp * pitch + n];
      }
    }
    if (want_bias) {
      for (int im = 0; im < here; ++im) {
        const int s = static_cast<int>((img0 + im) / B);
        if (s != cur_s) { flush(cur_s); cur_s = s; }
        if (static_cast<int>(threadIdx.x) < N) {
          const float* t = s_tile + im * img_smem + threadIdx.x;
          float c = 0.f;
          for (int pp = 0; pp < P; ++pp) c += t[pp * pitch];
          acc += c;
        }
      }
    }
  }
  flush(cur_s);
}

// The same pass with ONE WARP PER IMAGE (images whose [P][N + 1] block fits 8 KiB-class shared-memory slices, i.e. the
// example conv layers): no block-wide barrier, all of an image's 128-bit loads in flight before the first dependent
// shared-memory store (16 per lane at C3), a warp walks `ipw` consecutive images and keeps the column sums of N <= 256
// channels in registers.  The block-per-pass kernel above is sync bound at small images (3.4 TB/s at C3).
constexpr int kWarpImgMaxN = 256;
__global__ void __launch_bounds__(kThreads) nchw_to_nhwc_bias_warp_kernel(
    const float* __restrict__ dy, float* __restrict__ out, int64_t n_imgs, int B, int N, int P, int ipw,
    const float* __restrict__ rho_b, const float* __restrict__ eps_b, float* __restrict__ dmu_b, float* __restrict__ drho_b,
    uint32_t sample_begin, bnn_rng rng, FastDiv dP, FastDiv dN) {
  extern __shared__ float s_tile[];          // one [P][N + 1] block per warp
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  const int pitch = N + 1, NP = N * P;
  float* const tile = s_tile + warp * (P * pitch);
  const bool want_bias = dmu_b != nullptr;
  const RngKey key = resolve_rng(rng);
  float acc[kWarpImgMaxN / 32];              // column sums of channels lane, lane + 32, ... over the images of one sample
#pragma unroll
  for (int c = 0; c < kWarpImgMaxN / 32; ++c) acc[c] = 0.f;
  int cur_s = -1;
  auto flush = [&](int s) {
    if (!want_bias || s < 0) return;
#pragma unroll
    for (int c = 0; c < kWarpImgMaxN / 32; ++c) {
      const int n = c * 32 + lane;
      if (n < N) {
        const float e = eps_b != nullptr ? __ldg(eps_b + static_cast<int64_t>(s) * N + n)
                                         : eps1(key, sample_begin + s, static_cast<uint64_t>(n));
        atomicAdd(dmu_b + n, acc[c]);
        atomicAdd(drho_b + n, acc[c] * e * sigmoid_fast(__ldg(rho_b + n)));
      }
      acc[c] = 0.f;
    }
  };
  const int64_t img_begin = (static_cast<int64_t>(blockIdx.x) * warps + warp) * ipw;
  for (int j = 0; j < ipw; ++j) {
    const int64_t img = img_begin + j;
    if (img >= n_imgs) break;
    const float* src = dy + img * NP;
    float* dst = out + img * NP;
    // NCHW side: a float4 holds (n, p .. p + 3), P % 4 == 0 on this path
    for (int i0 = lane * 4; i0 < NP; i0 += 32 * 4 * 8) {
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * 128;
        if (i < NP) v[u] = ldg_stream4(src + i);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * 128;
        if (i < NP) {
          const int n = static_cast<int>(fdiv(i, dP)), pp = i - n * P;
          float* t = tile + pp * pitch + n;
          t[0] = v[u].x; t[pitch] = v[u].y; t[2 * pitch] = v[u].z; t[3 * pitch] = v[u].w;
        }
      }
    }
    __syncwarp();
    // NHWC side: N % 4 == 0 on this path
    for (int i = lane * 4; i < NP; i += 128) {
      const int pp = static_cast<int>(fdiv(i, dN)), n = i - pp * N;
      const float* t = tile + pp * pitch + n;
      *reinterpret_cast<float4*>(dst + i) = make_float4(t[0], t[1], t[2], t[3]);      // read next by the gradient kernels: keep it in L2
    }
    if (want_bias) {
      const int s = static_cast<int>(img / B);
      if (s != cur_s) { flush(cur_s); cur_s = s; }
#pragma unroll
      for (int c = 0; c < kWarpImgMaxN / 32; ++c) {
        const int n = c * 32 + lane;
        if (n < N) {
          float sum = 0.f;
          for (int pp = 0; pp < P; ++pp) sum += tile[pp * pitch + n];
          acc[c] += sum;
        }
      }
    }
    __syncwarp();
  }
  flush(cur_s);
}

int grid_for(int64_t items) {
  const int64_t blocks = (items + kThreads - 1) / kThreads;
  const int64_t cap = static_cast<int64_t>(sm_count()) * 16;
  return static_cast<int>(blocks < 1 ? 1 : (blocks < cap ? blocks : cap));
}

int check_geom(const bnn_conv2d_nhwc* g, const char* who) {
  BNN_REQUIRE(g != nullptr, BNN_ERR_BAD_ARGUMENT, "%s: geometry is NULL", who);
  BNN_REQUIRE(g->B > 0 && g->H > 0 && g->W > 0 && g->C > 0 && g->Cout > 0 && g->KH > 0 && g->KW > 0 && g->OH > 0 &&
                  g->OW > 0 && g->sh > 0 && g->sw > 0 && g->dh > 0 && g->dw > 0 && g->ph >= 0 && g->pw >= 0,
              BNN_ERR_BAD_ARGUMENT, "%s: bad geometry", who);
  BNN_REQUIRE(g->OH == (g->H + 2 * g->ph - g->dh * (g->KH - 1) - 1) / g->sh + 1 &&
                  g->OW == (g->W + 2 * g->pw - g->dw * (g->KW - 1) - 1) / g->sw + 1,
              BNN_ERR_BAD_ARGUMENT, "%s: OH / OW do not match the geometry", who);
  return BNN_OK;
}

}  // namespace
}  // namespace bnn

using namespace bnn;

extern "C" {

int bnn_conv2d_weight_layout(const float* mu, const float* rho, float* mu_p, float* sigma_p, float* rho_p, int32_t Cout,
                             int32_t Cg, int32_t taps, void* stream) {
  BNN_REQUIRE(mu && rho && mu_p, BNN_ERR_BAD_ARGUMENT, "bnn_conv2d_weight_layout: NULL pointer");
  BNN_REQUIRE(Cout > 0 && Cg > 0 && taps > 0, BNN_ERR_BAD_ARGUMENT, "bnn_conv2d_weight_layout: bad shape");
  int rc = check_device();
  if (rc != BNN_OK) return rc;
  const int64_t total = static_cast<int64_t>(Cout) * Cg * taps;
  weight_layout_kernel<<<grid_for(total), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(mu, rho, mu_p, sigma_p, rho_p, Cg,
                                                                                            taps, total);
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}

int bnn_conv2d_weight_unlayout(const float* in, float* out, int32_t n_arrays, int32_t Cout, int32_t Cg, int32_t taps,
                               void* stream) {
  BNN_REQUIRE(in && out, BNN_ERR_BAD_ARGUMENT, "bnn_conv2d_weight_unlayout: NULL pointer");
  BNN_REQUIRE(n_arrays > 0 && Cout > 0 && Cg > 0 && taps > 0, BNN_ERR_BAD_ARGUMENT, "bnn_conv2d_weight_unlayout: bad shape");
  int rc = check_device();
  if (rc != BNN_OK) return rc;
  const int64_t per = static_cast<int64_t>(Cout) * Cg * taps;
  weight_unlayout_kernel<<<grid_for(per * n_arrays), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(in, out, Cg, taps, per,
                                                                                                      per * n_arrays);
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}

int bnn_im2col_nhwc(const float* x, float* col, const bnn_conv2d_nhwc* g, int64_t n_imgs, void* stream) {
  int rc = check_geom(g, "bnn_im2col_nhwc");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(x && col && n_imgs > 0, BNN_ERR_BAD_ARGUMENT, "bnn_im2col_nhwc: NULL pointer or no images");
  BNN_REQUIRE(g->C % 4 == 0 && aligned16(x) && aligned16(col), BNN_ERR_MISALIGNED,
              "bnn_im2col_nhwc: needs C %% 4 == 0 and 16-byte aligned pointers");
  rc = check_device();
  if (rc != BNN_OK) return rc;
  const int64_t total = n_imgs * g->OH * g->OW * g->KH * g->KW * (g->C / 4);
  im2col_nhwc_kernel<<<grid_for(total), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(x, col, *g, n_imgs);
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}

int bnn_col2im_nhwc(const float* dcol, float* dx, const bnn_conv2d_nhwc* g, int64_t n_imgs, void* stream) {
  int rc = check_geom(g, "bnn_col2im_nhwc");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(dcol && dx && n_imgs > 0, BNN_ERR_BAD_ARGUMENT, "bnn_col2im_nhwc: NULL pointer or no images");
  BNN_REQUIRE(g->C % 4 == 0 && aligned16(dcol) && aligned16(dx), BNN_ERR_MISALIGNED,
              "bnn_col2im_nhwc: needs C %% 4 == 0 and 16-byte aligned pointers");
  rc = check_device();
  if (rc != BNN_OK) return rc;
  const int64_t total = n_imgs * g->H * g->W * (g->C / 4);
  col2im_nhwc_kernel<<<grid_for(total), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(dcol, dx, *g, n_imgs);
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}

int bnn_nchw_to_nhwc_bias_grad(const float* dy, float* dy_nhwc, int64_t n_imgs, int32_t B, int32_t N, int32_t P,
                               const float* rho_b, const float* eps_b, float* dmu_b, float* drho_b, uint32_t sample_begin,
                               const bnn_rng* rng_b, void* stream) {
  BNN_REQUIRE(dy && dy_nhwc && n_imgs > 0 && B > 0 && N > 0 && P > 0, BNN_ERR_BAD_ARGUMENT,
              "bnn_nchw_to_nhwc_bias_grad: NULL pointer or bad shape");
  BNN_REQUIRE((dmu_b == nullptr) == (drho_b == nullptr) && (dmu_b == nullptr || (rho_b != nullptr && rng_b != nullptr)),
              BNN_ERR_BAD_ARGUMENT, "bnn_nchw_to_nhwc_bias_grad: the bias gradient needs dmu_b, drho_b, rho_b and rng_b");
  const size_t img_smem = static_cast<size_t>(N + 1) * P * sizeof(float);
  BNN_REQUIRE(img_smem <= 48 * 1024 && (dmu_b == nullptr || N <= kThreads), BNN_ERR_UNSUPPORTED,
              "bnn_nchw_to_nhwc_bias_grad: one image's (N + 1) x P block must fit 48 KiB of shared memory (and N <= 256 with "
              "the bias gradient)");
  int rc = check_device();
  if (rc != BNN_OK) return rc;
  int ipt = static_cast<int>((32 * 1024) / img_smem);      // images per pass: at most ~32 KiB of shared memory per block ...
  if (ipt < 1) ipt = 1;
  if (ipt > 64) ipt = 64;
  const int64_t want_blocks = static_cast<int64_t>(sm_count()) * 4;      // ... but enough blocks to fill the machine
  if (n_imgs / ipt < want_blocks) ipt = static_cast<int>(n_imgs / want_blocks > 1 ? n_imgs / want_blocks : 1);
  // a few passes per block keep the number of (atomic) bias flushes down without starving the machine of blocks
  const int64_t tiles = (n_imgs + ipt - 1) / ipt;
  int passes = static_cast<int>(tiles / (static_cast<int64_t>(sm_count()) * 4));
  if (passes < 1) passes = 1;
  if (passes > 8) passes = 8;
  const int64_t blocks = (tiles + passes - 1) / passes;
  BNN_REQUIRE(blocks <= 0x7fffffff, BNN_ERR_UNSUPPORTED, "bnn_nchw_to_nhwc_bias_grad: too many images");
  const int vec = (P % 4 == 0) && aligned16(dy) && aligned16(dy_nhwc) && ((static_cast<int64_t>(N) * P) % 4 == 0);
  bnn_rng rng = rng_b ? *rng_b : bnn_rng{};
  // one warp per image when an image's block is small and everything is 128-bit friendly
  if (vec && N % 4 == 0 && N <= kWarpImgMaxN && img_smem <= 12 * 1024) {
    int warps = static_cast<int>((64 * 1024) / img_smem);
    if (warps > kThreads / 32) warps = kThreads / 32;
    const int64_t want_warps = static_cast<int64_t>(sm_count()) * 24;
    int ipw = static_cast<int>((n_imgs + want_warps - 1) / want_warps);
    if (ipw < 1) ipw = 1;
    if (ipw > 16) ipw = 16;
    const int64_t wblocks = (n_imgs + static_cast<int64_t>(warps) * ipw - 1) / (static_cast<int64_t>(warps) * ipw);
    const size_t smem = static_cast<size_t>(warps) * img_smem;
    static SmemOptIn opt_in;
    rc = allow_dynamic_smem(nchw_to_nhwc_bias_warp_kernel, 64 * 1024, &opt_in);
    if (rc != BNN_OK) return rc;
    nchw_to_nhwc_bias_warp_kernel<<<static_cast<int>(wblocks), warps * 32, smem, static_cast<cudaStream_t>(stream)>>>(
        dy, dy_nhwc, n_imgs, B, N, P, ipw, rho_b, eps_b, dmu_b, drho_b, sample_begin, rng,
        make_fastdiv(static_cast<uint32_t>(P)), make_fastdiv(static_cast<uint32_t>(N)));
    BNN_CUDA_OK(cudaGetLastError());
    return BNN_OK;
  }
  nchw_to_nhwc_bias_kernel<<<static_cast<int>(blocks), kThreads, static_cast<size_t>(ipt) * img_smem,
                             static_cast<cudaStream_t>(stream)>>>(dy, dy_nhwc, n_imgs, B, N, P, ipt, passes, rho_b, eps_b, dmu_b,
                                                                  drho_b, sample_begin, rng, vec,
                                                                  make_fastdiv(static_cast<uint32_t>(N) * P),
                                                                  make_fastdiv(static_cast<uint32_t>(P)),
                                                                  make_fastdiv(static_cast<uint32_t>(N)));
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}

int bnn_sampled_conv2d_fwd(const float* x, int64_t x_sample_stride, const float* mu_w, const float* sigma_w,
                           const float* mu_b, const float* sigma_b, const float* eps_w, const float* eps_b, bnn_view y,
                           int64_t y_sample_stride, const bnn_conv2d_nhwc* g, int32_t S, uint32_t sample_begin,
                           const bnn_rng* rng_w, const bnn_rng* rng_b, void* stream) {
  int rc = check_geom(g, "bnn_sampled_conv2d_fwd");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(x && mu_w && sigma_w && y.base && rng_w && S > 0 && S <= 65535, BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv2d_fwd: NULL pointer or bad sample count");
  BNN_REQUIRE((mu_b == nullptr) == (sigma_b == nullptr) && (mu_b == nullptr || rng_b != nullptr), BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv2d_fwd: bias needs mu_b, sigma_b and rng_b");
  BNN_REQUIRE(y.P >= 1, BNN_ERR_BAD_ARGUMENT, "bnn_sampled_conv2d_fwd: bad output view");
  rc = check_device();
  if (rc != BNN_OK) return rc;
  rc = contract::tma_conv_fwd(x, x_sample_stride, mu_w, sigma_w, mu_b, sigma_b, eps_w, eps_b, y, y_sample_stride,
                              contract::conv_geom_2d(*g), S,
                              sample_begin, rng_w, rng_b, static_cast<cudaStream_t>(stream));
  if (rc == contract::kNotEligible)
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv2d_fwd: needs C %% 32 == 0, 16-byte aligned tensors and a filter "
                                     "window within the im2col descriptor's limits (use bnn_im2col_nhwc + bnn_sampled_gemm_fwd)");
  return rc;
}

int bnn_sampled_conv2d_dgrad(const float* dy, const float* mu_w, const float* sigma_w, const float* eps_w, float* dx,
                             int64_t x_sample_stride, const bnn_conv2d_nhwc* g, int32_t S, uint32_t sample_begin,
                             const bnn_rng* rng_w, void* stream) {
  int rc = check_geom(g, "bnn_sampled_conv2d_dgrad");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(dy && mu_w && sigma_w && dx && rng_w && S > 0 && S <= 65535, BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv2d_dgrad: NULL pointer or bad sample count");
  rc = check_device();
  if (rc != BNN_OK) return rc;
  // strided layers keep the explicit lowering (col2im of the column gradients)
  rc = g->sh != 1 || g->sw != 1
           ? contract::kNotEligible
           : contract::tma_conv_gather(dy, false, mu_w, sigma_w, nullptr, nullptr, eps_w, nullptr, dx, x_sample_stride,
                                       x_sample_stride == 0, contract::conv_geom_2d(*g), S, sample_begin, rng_w, nullptr,
                                       static_cast<cudaStream_t>(stream));
  if (rc == contract::kNotEligible)
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv2d_dgrad: needs stride 1, Cout %% 32 == 0, C %% 4 == 0 and 16-byte "
                                     "aligned tensors (use bnn_sampled_gemm_dgrad + bnn_col2im_nhwc)");
  return rc;
}

int bnn_sampled_conv2d_wgrad(const float* dy, const float* x, int64_t x_sample_stride, const float* rho_w,
                             const float* eps_w, float* dmu_w, float* drho_w, const bnn_conv2d_nhwc* g, int32_t S,
                             uint32_t sample_begin, const bnn_rng* rng_w, void* stream) {
  int rc = check_geom(g, "bnn_sampled_conv2d_wgrad");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(dy && x && rho_w && dmu_w && drho_w && rng_w && S > 0 && S <= 65535, BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv2d_wgrad: NULL pointer or bad sample count");
  rc = check_device();
  if (rc != BNN_OK) return rc;
  rc = contract::tma_conv_wgrad(dy, false, x, x_sample_stride == 0, rho_w, eps_w, dmu_w, drho_w, contract::conv_geom_2d(*g),
                                S, sample_begin, rng_w,
                                static_cast<cudaStream_t>(stream));
  if (rc == contract::kNotEligible)
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv2d_wgrad: needs C %% 32 == 0, Cout %% 4 == 0 and 16-byte aligned "
                                     "tensors (use bnn_im2col_nhwc + bnn_sampled_gemm_wgrad)");
  return rc;
}


int bnn_sampled_conv_transpose2d_fwd(const float* x, int64_t x_sample_stride, const float* mu_w, const float* sigma_w,
                                     const float* mu_b, const float* sigma_b, const float* eps_w, const float* eps_b, float* y,
                                     const bnn_conv2d_nhwc* g, int32_t S, uint32_t sample_begin, const bnn_rng* rng_w,
                                     const bnn_rng* rng_b, void* stream) {
  int rc = check_geom(g, "bnn_sampled_conv_transpose2d_fwd");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(x && mu_w && sigma_w && y && rng_w && S > 0 && S <= 65535, BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv_transpose2d_fwd: NULL pointer or bad sample count");
  BNN_REQUIRE((mu_b == nullptr) == (sigma_b == nullptr) && (mu_b == nullptr || rng_b != nullptr), BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv_transpose2d_fwd: bias needs mu_b, sigma_b and rng_b");
  rc = check_device();
  if (rc != BNN_OK) return rc;
  rc = contract::tma_conv_gather(x, x_sample_stride == 0, mu_w, sigma_w, mu_b, sigma_b, eps_w, eps_b, y,
                                 static_cast<int64_t>(g->B) * g->H * g->W * g->C, false, contract::conv_geom_2d(*g), S,
                                 sample_begin, rng_w, rng_b,
                                 static_cast<cudaStream_t>(stream));
  if (rc == contract::kNotEligible)
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv_transpose2d_fwd: needs Cout %% 32 == 0, C %% 4 == 0, stride <= 8, "
                                     "16-byte aligned tensors and phase corners within the im2col descriptor's limits "
                                     "(use bnn_sampled_gemm_dgrad + bnn_col2im_nhwc)");
  return rc;
}

int bnn_sampled_conv_transpose2d_dgrad(const float* dy, const float* mu_w, const float* sigma_w, const float* eps_w,
                                       float* dx, int64_t x_sample_stride, const bnn_conv2d_nhwc* g, int32_t S,
                                       uint32_t sample_begin, const bnn_rng* rng_w, void* stream) {
  int rc = check_geom(g, "bnn_sampled_conv_transpose2d_dgrad");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(dy && mu_w && sigma_w && dx && rng_w && S > 0 && S <= 65535, BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv_transpose2d_dgrad: NULL pointer or bad sample count");
  rc = check_device();
  if (rc != BNN_OK) return rc;
  rc = contract::tma_conv_transpose_dgrad(dy, mu_w, sigma_w, eps_w, dx, x_sample_stride, contract::conv_geom_2d(*g), S,
                                          sample_begin, rng_w,
                                          static_cast<cudaStream_t>(stream));
  if (rc == contract::kNotEligible)
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv_transpose2d_dgrad: needs C %% 32 == 0, Cout %% 4 == 0, 16-byte "
                                     "aligned tensors and a filter window within the im2col descriptor's limits (use "
                                     "bnn_im2col_nhwc + bnn_sampled_gemm_fwd)");
  return rc;
}

int bnn_sampled_conv_transpose2d_wgrad(const float* dy, const float* x, int64_t x_sample_stride, const float* rho_w,
                                       const float* eps_w, float* dmu_w, float* drho_w, const bnn_conv2d_nhwc* g, int32_t S,
                                       uint32_t sample_begin, const bnn_rng* rng_w, void* stream) {
  int rc = check_geom(g, "bnn_sampled_conv_transpose2d_wgrad");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(dy && x && rho_w && dmu_w && drho_w && rng_w && S > 0 && S <= 65535, BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv_transpose2d_wgrad: NULL pointer or bad sample count");
  rc = check_device();
  if (rc != BNN_OK) return rc;
  // conv view: the "dY" operand is the transposed input x (shared by the samples when x_sample_stride == 0), A = dy
  rc = contract::tma_conv_wgrad(x, x_sample_stride == 0, dy, false, rho_w, eps_w, dmu_w, drho_w, contract::conv_geom_2d(*g),
                                S, sample_begin, rng_w,
                                static_cast<cudaStream_t>(stream));
  if (rc == contract::kNotEligible)
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv_transpose2d_wgrad: needs C %% 32 == 0, Cout %% 4 == 0 and 16-byte "
                                     "aligned tensors (use bnn_im2col_nhwc + bnn_sampled_gemm_wgrad)");
  return rc;
}

int bnn_debug_conv_transpose_phases(const bnn_conv2d_nhwc* g, int32_t* out, int32_t max_phases) {
  const int rc = check_geom(g, "bnn_debug_conv_transpose_phases");
  if (rc != BNN_OK) return -rc;
  if (out == nullptr && max_phases > 0) return -fail(BNN_ERR_BAD_ARGUMENT, "bnn_debug_conv_transpose_phases: NULL output");
  return contract::conv_transpose_phases(contract::conv_geom_2d(*g), out, max_phases);
}

// ---- 3-d transposed convolution: one eligibility predicate for the three passes (bnn_b200.h)
namespace {
int check_geom3d(const bnn_conv3d_nhwc* g, const char* who) {
  BNN_REQUIRE(g != nullptr, BNN_ERR_BAD_ARGUMENT, "%s: geometry is NULL", who);
  BNN_REQUIRE(g->B > 0 && g->D > 0 && g->H > 0 && g->W > 0 && g->C > 0 && g->Cout > 0 && g->KD > 0 && g->KH > 0 &&
                  g->KW > 0 && g->OD > 0 && g->OH > 0 && g->OW > 0 && g->sd > 0 && g->sh > 0 && g->sw > 0 && g->dd > 0 &&
                  g->dh > 0 && g->dw > 0 && g->pd >= 0 && g->ph >= 0 && g->pw >= 0,
              BNN_ERR_BAD_ARGUMENT, "%s: bad geometry", who);
  BNN_REQUIRE(g->OD == (g->D + 2 * g->pd - g->dd * (g->KD - 1) - 1) / g->sd + 1 &&
                  g->OH == (g->H + 2 * g->ph - g->dh * (g->KH - 1) - 1) / g->sh + 1 &&
                  g->OW == (g->W + 2 * g->pw - g->dw * (g->KW - 1) - 1) / g->sw + 1,
              BNN_ERR_BAD_ARGUMENT, "%s: OD / OH / OW do not match the geometry", who);
  return BNN_OK;
}
contract::ConvGeom geom3d(const bnn_conv3d_nhwc* g) {
  contract::ConvGeom cg{};
  cg.g = *g;
  cg.vol = true;
  return cg;
}
// the predicate: channels, strides, every conv-view and phase corner (contract::conv_transpose_ok), alignment
bool transpose3d_ok(const bnn_conv3d_nhwc* g, std::initializer_list<const void*> tensors, const bnn_rng* rng_w) {
  for (const void* t : tensors)
    if (t != nullptr && !aligned16(t)) return false;
  return g->C % 32 == 0 && rng_w->elem_offset % 4 == 0 && contract::conv_transpose_ok(geom3d(g));
}
constexpr const char* kT3dLimits = "needs Cin %% 32 == 0, Cout %% 32 == 0, stride <= 8, 16-byte aligned tensors and every "
                                   "phase and conv-view corner within the rank-5 im2col descriptor's limits";
}  // namespace

int bnn_sampled_conv_transpose3d_fwd(const float* x, int64_t x_sample_stride, const float* mu_w, const float* sigma_w,
                                     const float* mu_b, const float* sigma_b, const float* eps_w, const float* eps_b, float* y,
                                     const bnn_conv3d_nhwc* g, int32_t S, uint32_t sample_begin, const bnn_rng* rng_w,
                                     const bnn_rng* rng_b, void* stream) {
  int rc = check_geom3d(g, "bnn_sampled_conv_transpose3d_fwd");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(x && mu_w && sigma_w && y && rng_w && S > 0 && S <= 65535, BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv_transpose3d_fwd: NULL pointer or bad sample count");
  BNN_REQUIRE((mu_b == nullptr) == (sigma_b == nullptr) && (mu_b == nullptr || rng_b != nullptr), BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv_transpose3d_fwd: bias needs mu_b, sigma_b and rng_b");
  if (!transpose3d_ok(g, {x, mu_w, sigma_w, eps_w, y}, rng_w))
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv_transpose3d_fwd: %s", kT3dLimits);
  rc = check_device();
  if (rc != BNN_OK) return rc;
  rc = contract::tma_conv_gather(x, x_sample_stride == 0, mu_w, sigma_w, mu_b, sigma_b, eps_w, eps_b, y,
                                 static_cast<int64_t>(g->B) * g->D * g->H * g->W * g->C, false, geom3d(g), S, sample_begin,
                                 rng_w, rng_b, static_cast<cudaStream_t>(stream));
  if (rc == contract::kNotEligible)
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv_transpose3d_fwd: %s", kT3dLimits);
  return rc;
}

int bnn_sampled_conv_transpose3d_dgrad(const float* dy, const float* mu_w, const float* sigma_w, const float* eps_w,
                                       float* dx, int64_t x_sample_stride, const bnn_conv3d_nhwc* g, int32_t S,
                                       uint32_t sample_begin, const bnn_rng* rng_w, void* stream) {
  int rc = check_geom3d(g, "bnn_sampled_conv_transpose3d_dgrad");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(dy && mu_w && sigma_w && dx && rng_w && S > 0 && S <= 65535, BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv_transpose3d_dgrad: NULL pointer or bad sample count");
  if (!transpose3d_ok(g, {dy, mu_w, sigma_w, eps_w, dx}, rng_w))
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv_transpose3d_dgrad: %s", kT3dLimits);
  rc = check_device();
  if (rc != BNN_OK) return rc;
  rc = contract::tma_conv_transpose_dgrad(dy, mu_w, sigma_w, eps_w, dx, x_sample_stride, geom3d(g), S, sample_begin, rng_w,
                                          static_cast<cudaStream_t>(stream));
  if (rc == contract::kNotEligible)
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv_transpose3d_dgrad: %s", kT3dLimits);
  return rc;
}

int bnn_sampled_conv_transpose3d_wgrad(const float* dy, const float* x, int64_t x_sample_stride, const float* rho_w,
                                       const float* eps_w, float* dmu_w, float* drho_w, const bnn_conv3d_nhwc* g, int32_t S,
                                       uint32_t sample_begin, const bnn_rng* rng_w, void* stream) {
  int rc = check_geom3d(g, "bnn_sampled_conv_transpose3d_wgrad");
  if (rc != BNN_OK) return rc;
  BNN_REQUIRE(dy && x && rho_w && dmu_w && drho_w && rng_w && S > 0 && S <= 65535, BNN_ERR_BAD_ARGUMENT,
              "bnn_sampled_conv_transpose3d_wgrad: NULL pointer or bad sample count");
  if (!transpose3d_ok(g, {dy, x, rho_w, eps_w, dmu_w, drho_w}, rng_w))
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv_transpose3d_wgrad: %s", kT3dLimits);
  rc = check_device();
  if (rc != BNN_OK) return rc;
  rc = contract::tma_conv_wgrad(x, x_sample_stride == 0, dy, false, rho_w, eps_w, dmu_w, drho_w, geom3d(g), S, sample_begin,
                                rng_w, static_cast<cudaStream_t>(stream));
  if (rc == contract::kNotEligible)
    return fail(BNN_ERR_UNSUPPORTED, "bnn_sampled_conv_transpose3d_wgrad: %s", kT3dLimits);
  return rc;
}

int bnn_conv_transpose2d_supported(const bnn_conv2d_nhwc* g) {
  const int rc = check_geom(g, "bnn_conv_transpose2d_supported");
  if (rc != BNN_OK) return rc;
  // the forward's phase corners and the input / weight gradients' conv-view corners (conv_ok) in one predicate
  if (!contract::conv_transpose_ok(contract::conv_geom_2d(*g)))
    return fail(BNN_ERR_UNSUPPORTED, "bnn_conv_transpose2d_supported: needs Cin %% 32 == 0, Cout %% 32 == 0, stride <= 8 and "
                                     "every phase and conv-view corner within the im2col descriptor's limits");
  return BNN_OK;
}

int bnn_conv_transpose3d_supported(const bnn_conv3d_nhwc* g) {
  const int rc = check_geom3d(g, "bnn_conv_transpose3d_supported");
  if (rc != BNN_OK) return rc;
  if (g->C % 32 != 0 || !contract::conv_transpose_ok(geom3d(g)))
    return fail(BNN_ERR_UNSUPPORTED, "bnn_conv_transpose3d_supported: %s", kT3dLimits);
  return BNN_OK;
}

int bnn_debug_conv_transpose3d_phases(const bnn_conv3d_nhwc* g, int32_t* out, int32_t max_phases) {
  const int rc = check_geom3d(g, "bnn_debug_conv_transpose3d_phases");
  if (rc != BNN_OK) return -rc;
  if (out == nullptr && max_phases > 0) return -fail(BNN_ERR_BAD_ARGUMENT, "bnn_debug_conv_transpose3d_phases: NULL output");
  return contract::conv_transpose_phases(geom3d(g), out, max_phases);
}

}  // extern "C"
