// adam.cu — bnn_adam_kl_step: the optimizer half of the ELBO tail (SURVEY §8f-3).
//
// One pass over the variational parameters that (a) forms the closed-form KL gradient of every element
//     dKL/dmu = c (mu - loc) / scale^2,   dKL/drho = c (sigma / scale^2 - 1 / sigma) sigmoid(rho),   sigma = 1e-10 + softplus(rho)
// (SURVEY §3.2; the gradient of KLDivergence.forward, pytorch_bayesian/nn/loss.py:16-38, with c = 1 / (numel_t n_tensors
// n_batches)), (b) adds it to the likelihood gradient that autograd (and the gradient all-reduce) left in g_mu / g_rho, and
// (c) applies torch.optim.Adam's update (examples/MNIST/train.py:43,65: Adam over all parameters, no weight decay, no
// amsgrad) to mu, rho and their moment buffers.  The separate path reads and writes the gradients three more times (KL
// gradient kernel, autograd accumulation, optimizer).  Bandwidth bound: 8 loads + 6 stores of 4 bytes per (mu, rho) pair.
// A tensor with rho == NULL is a plain (deterministic) parameter: Adam on `mu` alone, so one launch updates a whole model.
//
// bnn_adam_kl_step_peers folds the data-/sample-parallel gradient exchange (SURVEY §8e: ONE all-reduce of the flat
// gradient buffer) into the same pass: every rank keeps its gradients in a buffer that all ranks of the node have mapped
// (NVLink peer memory), and each rank's optimizer kernel reads the R copies of a gradient element straight from the R
// buffers, averages them and applies the update — a one-shot all-reduce whose only output is the updated parameters.
// bnn_peer_barrier is the flag barrier around it (all gradients written before anyone reads; all reads done before
// anyone overwrites), so the whole training step is one capturable graph without a NCCL call.
#include "common.cuh"

namespace bnn {
namespace {

constexpr int kThreads = 256;
constexpr int kMaxTensors = 16;       // per launch: the table travels by value in the kernel parameters

struct AdamDesc {
  float* mu; float* rho;
  const float* g_mu; const float* g_rho;
  float* m_mu; float* v_mu; float* m_rho; float* v_rho;
  int64_t numel;
  int64_t block_begin;       // first global block-chunk of this tensor
  float loc, inv_scale2, coeff;
  int vec;                   // every pointer 16-byte aligned
};
struct AdamTable {
  AdamDesc t[kMaxTensors];
  int n;
  int world;                 // > 1: gradients are averaged over `world` peer buffers (bnn_adam_kl_step_peers)
  const float* peer[BNN_MAX_PEERS];   // rank r's flat gradient buffer, mapped here; peer[rank] is the local one
  int rank;
  int pad;
  int64_t total_chunks;
  float lr, beta1, beta2, eps;
  const float* step_dev;     // device scalar: number of this step (1, 2, ...), as torch's capturable Adam keeps it
  float step_host;           // used when step_dev is NULL
};

constexpr int kPerThread = 4;                               // elements per thread per chunk (one float4 per array)
constexpr int kChunk = kThreads * kPerThread;               // 1024 elements

struct Hyper { float lr_over_bc1, inv_sqrt_bc2, beta1, beta2, eps; };

__device__ __forceinline__ void adam_element(float& p, float g, float& m, float& v, const Hyper& h) {
  m = fmaf(g - m, 1.0f - h.beta1, m);                      // exp_avg.lerp_(grad, 1 - beta1)
  v = fmaf(h.beta2, v, (1.0f - h.beta2) * g * g);          // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
  const float denom = fmaf(sqrtf(v), h.inv_sqrt_bc2, h.eps);
  p = fmaf(-h.lr_over_bc1, m / denom, p);
}

__device__ __forceinline__ void elbo_adam_pair(float& mu, float& rho, float g_mu, float g_rho, float& m_mu, float& v_mu,
                                               float& m_rho, float& v_rho, float loc, float inv_scale2, float coeff,
                                               const Hyper& h) {
  if (coeff != 0.0f) {
    const float sigma = stddev_exact(rho);
    const float sig = 1.0f / (1.0f + expf(-rho));
    g_mu = fmaf(coeff * (mu - loc), inv_scale2, g_mu);
    g_rho = fmaf(coeff * (sigma * inv_scale2 - 1.0f / sigma), sig, g_rho);
  }
  adam_element(mu, g_mu, m_mu, v_mu, h);
  adam_element(rho, g_rho, m_rho, v_rho, h);
}

// loads that bypass the (non-coherent) L1: peer buffers are rewritten by their owners between launches
__device__ __forceinline__ float4 ld_peer4(const float* p) { return __ldcv(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float ld_peer1(const float* p) { return __ldcv(p); }

// mean over the ranks of the gradient element(s) at `g` (a pointer into the LOCAL buffer): same offset in every peer
// buffer, summed in rank order so that every rank obtains bit-identical parameters
template <bool kPeers>
__device__ __forceinline__ float4 grad4(const AdamTable& tab, const float* g) {
  if (g == nullptr) return make_float4(0.f, 0.f, 0.f, 0.f);
  if (!kPeers) return ldg_stream4(g);
  const int64_t off = g - tab.peer[tab.rank];
  float4 acc = ld_peer4(tab.peer[0] + off);
  for (int r = 1; r < tab.world; ++r) {
    const float4 v = ld_peer4(tab.peer[r] + off);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  const float inv = 1.0f / static_cast<float>(tab.world);
  return make_float4(acc.x * inv, acc.y * inv, acc.z * inv, acc.w * inv);
}
template <bool kPeers>
__device__ __forceinline__ float grad1(const AdamTable& tab, const float* g) {
  if (g == nullptr) return 0.f;
  if (!kPeers) return *g;
  const int64_t off = g - tab.peer[tab.rank];
  float acc = ld_peer1(tab.peer[0] + off);
  for (int r = 1; r < tab.world; ++r) acc += ld_peer1(tab.peer[r] + off);
  return acc * (1.0f / static_cast<float>(tab.world));     // as grad4 and bnn_peer_average: alignment changes no bit
}

template <bool kPeers>
__global__ void __launch_bounds__(kThreads) adam_kl_kernel(const __grid_constant__ AdamTable tab) {
  __shared__ int64_t s_begin[kMaxTensors];
  if (threadIdx.x < tab.n) s_begin[threadIdx.x] = tab.t[threadIdx.x].block_begin;
  __syncthreads();
  const double step = tab.step_dev != nullptr ? static_cast<double>(*tab.step_dev) : static_cast<double>(tab.step_host);
  Hyper h;
  h.beta1 = tab.beta1; h.beta2 = tab.beta2; h.eps = tab.eps;
  h.lr_over_bc1 = static_cast<float>(static_cast<double>(tab.lr) / (1.0 - pow(static_cast<double>(tab.beta1), step)));
  h.inv_sqrt_bc2 = static_cast<float>(1.0 / sqrt(1.0 - pow(static_cast<double>(tab.beta2), step)));
  int t = 0;
  for (int64_t chunk = blockIdx.x; chunk < tab.total_chunks; chunk += gridDim.x) {
    while (t + 1 < tab.n && chunk >= s_begin[t + 1]) ++t;
    const AdamDesc& d = tab.t[t];
    const int64_t i0 = (chunk - d.block_begin) * kChunk + threadIdx.x * kPerThread;
    if (i0 >= d.numel) continue;
    if (d.rho == nullptr) {                       // plain parameter: Adam on mu alone
      if (d.vec && i0 + kPerThread <= d.numel) {
        float4 mu = *reinterpret_cast<const float4*>(d.mu + i0);
        const float4 gm = grad4<kPeers>(tab, d.g_mu ? d.g_mu + i0 : nullptr);
        float4 mm = *reinterpret_cast<const float4*>(d.m_mu + i0), vm = *reinterpret_cast<const float4*>(d.v_mu + i0);
        adam_element(mu.x, gm.x, mm.x, vm.x, h);
        adam_element(mu.y, gm.y, mm.y, vm.y, h);
        adam_element(mu.z, gm.z, mm.z, vm.z, h);
        adam_element(mu.w, gm.w, mm.w, vm.w, h);
        *reinterpret_cast<float4*>(d.mu + i0) = mu;
        *reinterpret_cast<float4*>(d.m_mu + i0) = mm; *reinterpret_cast<float4*>(d.v_mu + i0) = vm;
      } else {
        for (int e = 0; e < kPerThread; ++e) {
          const int64_t i = i0 + e;
          if (i >= d.numel) break;
          float mu = d.mu[i], mm = d.m_mu[i], vm = d.v_mu[i];
          adam_element(mu, grad1<kPeers>(tab, d.g_mu ? d.g_mu + i : nullptr), mm, vm, h);
          d.mu[i] = mu; d.m_mu[i] = mm; d.v_mu[i] = vm;
        }
      }
      continue;
    }
    if (d.vec && i0 + kPerThread <= d.numel) {
      float4 mu = *reinterpret_cast<const float4*>(d.mu + i0), rho = *reinterpret_cast<const float4*>(d.rho + i0);
      const float4 gm = grad4<kPeers>(tab, d.g_mu ? d.g_mu + i0 : nullptr);
      const float4 gr = grad4<kPeers>(tab, d.g_rho ? d.g_rho + i0 : nullptr);
      float4 mm = *reinterpret_cast<const float4*>(d.m_mu + i0), vm = *reinterpret_cast<const float4*>(d.v_mu + i0);
      float4 mr = *reinterpret_cast<const float4*>(d.m_rho + i0), vr = *reinterpret_cast<const float4*>(d.v_rho + i0);
      elbo_adam_pair(mu.x, rho.x, gm.x, gr.x, mm.x, vm.x, mr.x, vr.x, d.loc, d.inv_scale2, d.coeff, h);
      elbo_adam_pair(mu.y, rho.y, gm.y, gr.y, mm.y, vm.y, mr.y, vr.y, d.loc, d.inv_scale2, d.coeff, h);
      elbo_adam_pair(mu.z, rho.z, gm.z, gr.z, mm.z, vm.z, mr.z, vr.z, d.loc, d.inv_scale2, d.coeff, h);
      elbo_adam_pair(mu.w, rho.w, gm.w, gr.w, mm.w, vm.w, mr.w, vr.w, d.loc, d.inv_scale2, d.coeff, h);
      *reinterpret_cast<float4*>(d.mu + i0) = mu; *reinterpret_cast<float4*>(d.rho + i0) = rho;
      *reinterpret_cast<float4*>(d.m_mu + i0) = mm; *reinterpret_cast<float4*>(d.v_mu + i0) = vm;
      *reinterpret_cast<float4*>(d.m_rho + i0) = mr; *reinterpret_cast<float4*>(d.v_rho + i0) = vr;
    } else {
      for (int e = 0; e < kPerThread; ++e) {
        const int64_t i = i0 + e;
        if (i >= d.numel) break;
        float mu = d.mu[i], rho = d.rho[i], mm = d.m_mu[i], vm = d.v_mu[i], mr = d.m_rho[i], vr = d.v_rho[i];
        elbo_adam_pair(mu, rho, grad1<kPeers>(tab, d.g_mu ? d.g_mu + i : nullptr),
                       grad1<kPeers>(tab, d.g_rho ? d.g_rho + i : nullptr), mm, vm, mr, vr, d.loc, d.inv_scale2, d.coeff, h);
        d.mu[i] = mu; d.rho[i] = rho; d.m_mu[i] = mm; d.v_mu[i] = vm; d.m_rho[i] = mr; d.v_rho[i] = vr;
      }
    }
  }
}

int adam_launch(const bnn_adam_tensor* tensors, int32_t n_tensors, float lr, float beta1, float beta2, float eps,
                const float* step_dev, int64_t step_host, const bnn_peer_grads* peers, void* stream, const char* who) {
  BNN_REQUIRE(n_tensors >= 0, BNN_ERR_BAD_ARGUMENT, "%s: n_tensors < 0", who);
  if (n_tensors == 0) return BNN_OK;
  BNN_REQUIRE(tensors != nullptr, BNN_ERR_BAD_ARGUMENT, "%s: tensor table is NULL", who);
  BNN_REQUIRE(lr >= 0.f && beta1 >= 0.f && beta1 < 1.f && beta2 >= 0.f && beta2 < 1.f && eps >= 0.f, BNN_ERR_BAD_ARGUMENT,
              "%s: need lr >= 0, 0 <= beta < 1, eps >= 0", who);
  BNN_REQUIRE(step_dev != nullptr || step_host >= 1, BNN_ERR_BAD_ARGUMENT,
              "%s: the step number starts at 1 (pass step_dev or step_host >= 1)", who);
  const bool use_peers = peers != nullptr && peers->world > 1;
  if (peers != nullptr) {
    BNN_REQUIRE(peers->world >= 1 && peers->world <= BNN_MAX_PEERS && peers->rank >= 0 && peers->rank < peers->world,
                BNN_ERR_BAD_ARGUMENT, "%s: need 1 <= world <= %d and 0 <= rank < world", who, BNN_MAX_PEERS);
    for (int r = 0; r < peers->world; ++r)
      BNN_REQUIRE(peers->base[r] != nullptr && aligned16(peers->base[r]), BNN_ERR_BAD_ARGUMENT,
                  "%s: peer gradient buffer %d is NULL or not 16-byte aligned", who, r);
  }
  for (int i = 0; i < n_tensors; ++i) {
    const bnn_adam_tensor& t = tensors[i];
    BNN_REQUIRE(t.numel >= 0, BNN_ERR_BAD_ARGUMENT, "%s: tensor %d has numel < 0", who, i);
    BNN_REQUIRE(t.numel == 0 || (t.mu && t.m_mu && t.v_mu), BNN_ERR_BAD_ARGUMENT,
                "%s: tensor %d has a NULL parameter or moment pointer", who, i);
    BNN_REQUIRE(t.numel == 0 || t.rho == nullptr || (t.m_rho && t.v_rho), BNN_ERR_BAD_ARGUMENT,
                "%s: tensor %d has rho but no moment buffers for it", who, i);
    // an empty tensor has NULL pointers (torch's data_ptr() of zero elements): it is skipped, whatever its kind
    BNN_REQUIRE(t.numel == 0 || t.rho != nullptr || (t.kl_coeff == 0.f && t.g_rho == nullptr), BNN_ERR_BAD_ARGUMENT,
                "%s: tensor %d is a plain parameter (rho NULL): kl_coeff must be 0 and g_rho NULL", who, i);
    BNN_REQUIRE(t.kl_coeff == 0.f || t.prior_scale > 0.f, BNN_ERR_BAD_ARGUMENT, "%s: tensor %d needs prior scale > 0", who, i);
    if (use_peers) {
      BNN_REQUIRE((t.g_mu == nullptr || t.g_mu >= peers->base[peers->rank]) &&
                      (t.g_rho == nullptr || t.g_rho >= peers->base[peers->rank]),
                  BNN_ERR_BAD_ARGUMENT, "%s: tensor %d: gradients must live inside this rank's peer-visible buffer", who, i);
    }
  }
  int rc = check_device();
  if (rc != BNN_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int max_grid = sm_count() * 8;
  for (int first = 0; first < n_tensors; first += kMaxTensors) {
    const int n = n_tensors - first < kMaxTensors ? n_tensors - first : kMaxTensors;
    AdamTable tab;
    tab.n = 0; tab.pad = 0;
    tab.world = use_peers ? peers->world : 1;
    tab.rank = use_peers ? peers->rank : 0;
    for (int r = 0; r < BNN_MAX_PEERS; ++r) tab.peer[r] = (use_peers && r < peers->world) ? peers->base[r] : nullptr;
    tab.lr = lr; tab.beta1 = beta1; tab.beta2 = beta2; tab.eps = eps;
    tab.step_dev = step_dev; tab.step_host = static_cast<float>(step_host);
    int64_t chunks = 0;
    for (int i = 0; i < n; ++i) {
      const bnn_adam_tensor& t = tensors[first + i];
      if (t.numel == 0) continue;
      AdamDesc& d = tab.t[tab.n++];
      d.mu = t.mu; d.rho = t.rho; d.g_mu = t.g_mu; d.g_rho = t.g_rho;
      d.m_mu = t.m_mu; d.v_mu = t.v_mu; d.m_rho = t.m_rho; d.v_rho = t.v_rho;
      d.numel = t.numel; d.block_begin = chunks;
      d.loc = t.prior_loc; d.coeff = t.kl_coeff;
      d.inv_scale2 = t.kl_coeff != 0.f ? 1.0f / (t.prior_scale * t.prior_scale) : 0.f;
      d.vec = aligned16(t.mu) && aligned16(t.m_mu) && aligned16(t.v_mu) &&
              (t.rho == nullptr || (aligned16(t.rho) && aligned16(t.m_rho) && aligned16(t.v_rho))) &&
              (t.g_mu == nullptr || aligned16(t.g_mu)) && (t.g_rho == nullptr || aligned16(t.g_rho));
      chunks += (t.numel + kChunk - 1) / kChunk;
    }
    if (tab.n == 0) continue;
    tab.total_chunks = chunks;
    const int grid = static_cast<int>(chunks < max_grid ? chunks : max_grid);
    if (use_peers) adam_kl_kernel<true><<<grid, kThreads, 0, st>>>(tab);
    else adam_kl_kernel<false><<<grid, kThreads, 0, st>>>(tab);
    BNN_CUDA_OK(cudaGetLastError());
  }
  return BNN_OK;
}

// ---- flag barrier between the ranks of one node (one rank per GPU; every rank launches it at the same point of its
// stream).  flags[r] = rank r's flag block (BNN_MAX_PEERS uint32 words, zero before first use) as mapped here.  Thread p
// publishes this rank's arrival number in peer p's block (release, system scope: the gradient stores of the earlier
// kernels of this stream are visible to whoever acquires the flag), then waits until peer p's arrival shows up in the
// local block.  The arrival number lives in device memory and advances by one per launch, so a captured graph replays it.
struct BarrierParams {
  uint32_t* flags[BNN_MAX_PEERS];
  uint32_t* epoch;
  int world, rank;
};
__global__ void __launch_bounds__(32) peer_barrier_kernel(const __grid_constant__ BarrierParams p) {
  const int t = threadIdx.x;
  const uint32_t e = *p.epoch + 1u;
  __syncwarp();
  if (t < p.world && t != p.rank) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.flags[t] + p.rank), "r"(e) : "memory");
    const uint32_t* mine = p.flags[p.rank] + t;
    uint64_t t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
      uint32_t v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
      if (static_cast<int32_t>(v - e) >= 0) break;
      uint64_t t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > 10000000000ull) __trap();      // 10 s: a rank that never arrives must fail the launch, not hang the box
    }
    __threadfence_system();
  }
  __syncwarp();
  if (t == 0) *p.epoch = e;
}

// ---- bnn_peer_average: in-place average of the ranks' flat gradient buffers in two hops instead of R - 1 reads of
// everything by everyone: rank r owns the r-th slice of the buffer, reads that slice from every rank (all R loads of an
// element are in flight together), averages in rank order and writes the result back into EVERY rank's buffer
// (reduce-scatter + all-gather over NVLink peer memory, (R - 1) / R of the buffer in each direction per rank instead of
// R - 1 buffers inbound).  An element is read and rewritten by its owner only, so the update is safe in place.  Between
// two bnn_peer_barrier launches; afterwards every rank holds the same averaged gradients locally and the plain
// optimizer kernel runs on them.
struct AverageParams {
  float* peer[BNN_MAX_PEERS];
  int world, rank;
  int64_t begin, end;        // this rank's slice [begin, end) in floats, multiples of 4 (except the very end of the buffer)
};
__global__ void __launch_bounds__(kThreads) peer_average_kernel(const __grid_constant__ AverageParams p) {
  const float inv = 1.0f / static_cast<float>(p.world);
  const int64_t n4 = (p.end - p.begin) / 4;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(kThreads) + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * kThreads) {
    const int64_t off = p.begin + 4 * i;
    float4 v[BNN_MAX_PEERS];
#pragma unroll
    for (int r = 0; r < BNN_MAX_PEERS; ++r)
      if (r < p.world) v[r] = ld_peer4(p.peer[r] + off);
    float4 acc = v[0];
#pragma unroll
    for (int r = 1; r < BNN_MAX_PEERS; ++r)
      if (r < p.world) { acc.x += v[r].x; acc.y += v[r].y; acc.z += v[r].z; acc.w += v[r].w; }
    acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
#pragma unroll
    for (int r = 0; r < BNN_MAX_PEERS; ++r)
      if (r < p.world) *reinterpret_cast<float4*>(p.peer[r] + off) = acc;
  }
  // tail of the buffer (numel not a multiple of 4): the last rank's slice ends there
  const int64_t tail = p.begin + 4 * n4;
  if (blockIdx.x == 0 && threadIdx.x < p.end - tail) {
    const int64_t off = tail + threadIdx.x;
    float acc = 0.f;
    for (int r = 0; r < p.world; ++r) acc += ld_peer1(p.peer[r] + off);
    acc *= inv;
    for (int r = 0; r < p.world; ++r) p.peer[r][off] = acc;
  }
}

// ---- bnn_pack_gradients: the gradients autograd left in separate tensors -> one flat (peer-visible) buffer, one launch.
// Replaces "gradients are views of the flat buffer" (a fill of the buffer plus one accumulation kernel per parameter
// in every backward pass) by a single gather after the backward pass.
constexpr int kPackMax = 32;
struct PackItem { const float* src; int64_t dst; int64_t numel; int64_t chunk_begin; };
struct PackTable {
  PackItem t[kPackMax];
  int n;
  int pad;
  int64_t total_chunks;
  float* dst_base;
};
__global__ void __launch_bounds__(kThreads) pack_kernel(const __grid_constant__ PackTable tab) {
  __shared__ int64_t s_begin[kPackMax];
  if (threadIdx.x < tab.n) s_begin[threadIdx.x] = tab.t[threadIdx.x].chunk_begin;
  __syncthreads();
  int t = 0;
  for (int64_t chunk = blockIdx.x; chunk < tab.total_chunks; chunk += gridDim.x) {
    while (t + 1 < tab.n && chunk >= s_begin[t + 1]) ++t;
    const PackItem& it = tab.t[t];
    const int64_t i0 = (chunk - it.chunk_begin) * kChunk + threadIdx.x * kPerThread;
    if (i0 >= it.numel) continue;
    float* dst = tab.dst_base + it.dst + i0;
    const bool vec = it.src != nullptr ? ((reinterpret_cast<uintptr_t>(it.src + i0) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0
                                       : (reinterpret_cast<uintptr_t>(dst) & 15u) == 0;
    if (vec && i0 + kPerThread <= it.numel) {
      *reinterpret_cast<float4*>(dst) = it.src != nullptr ? ldg_stream4(it.src + i0) : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
      for (int e = 0; e < kPerThread && i0 + e < it.numel; ++e) dst[e] = it.src != nullptr ? it.src[i0 + e] : 0.f;
    }
  }
}

}  // namespace
}  // namespace bnn

using namespace bnn;

extern "C" int bnn_pack_gradients(const bnn_pack_item* items, int32_t n_items, float* dst, void* stream) {
  BNN_REQUIRE(n_items >= 0, BNN_ERR_BAD_ARGUMENT, "bnn_pack_gradients: n_items < 0");
  if (n_items == 0) return BNN_OK;
  BNN_REQUIRE(items != nullptr && dst != nullptr, BNN_ERR_BAD_ARGUMENT, "bnn_pack_gradients: NULL pointer");
  for (int i = 0; i < n_items; ++i)
    BNN_REQUIRE(items[i].numel >= 0 && items[i].dst_offset >= 0, BNN_ERR_BAD_ARGUMENT,
                "bnn_pack_gradients: item %d has a negative size or offset", i);
  int rc = check_device();
  if (rc != BNN_OK) return rc;
  const int max_grid = sm_count() * 4;
  for (int first = 0; first < n_items; first += kPackMax) {
    const int n = n_items - first < kPackMax ? n_items - first : kPackMax;
    PackTable tab;
    tab.n = 0; tab.pad = 0; tab.dst_base = dst;
    int64_t chunks = 0;
    for (int i = 0; i < n; ++i) {
      const bnn_pack_item& it = items[first + i];
      if (it.numel == 0) continue;
      tab.t[tab.n++] = PackItem{it.src, it.dst_offset, it.numel, chunks};
      chunks += (it.numel + kChunk - 1) / kChunk;
    }
    if (tab.n == 0) continue;
    tab.total_chunks = chunks;
    const int grid = static_cast<int>(chunks < max_grid ? chunks : max_grid);
    pack_kernel<<<grid, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(tab);
    BNN_CUDA_OK(cudaGetLastError());
  }
  return BNN_OK;
}

extern "C" int bnn_adam_kl_step(const bnn_adam_tensor* tensors, int32_t n_tensors, float lr, float beta1, float beta2,
                                float eps, const float* step_dev, int64_t step_host, void* stream) {
  return adam_launch(tensors, n_tensors, lr, beta1, beta2, eps, step_dev, step_host, nullptr, stream, "bnn_adam_kl_step");
}

extern "C" int bnn_adam_kl_step_peers(const bnn_adam_tensor* tensors, int32_t n_tensors, float lr, float beta1, float beta2,
                                      float eps, const float* step_dev, int64_t step_host, const bnn_peer_grads* peers,
                                      void* stream) {
  BNN_REQUIRE(peers != nullptr, BNN_ERR_BAD_ARGUMENT, "bnn_adam_kl_step_peers: peers is NULL");
  return adam_launch(tensors, n_tensors, lr, beta1, beta2, eps, step_dev, step_host, peers, stream,
                     "bnn_adam_kl_step_peers");
}

extern "C" int bnn_peer_average(const bnn_peer_grads* peers, int64_t numel, void* stream) {
  BNN_REQUIRE(peers != nullptr && numel >= 0, BNN_ERR_BAD_ARGUMENT, "bnn_peer_average: NULL table or negative size");
  BNN_REQUIRE(peers->world >= 1 && peers->world <= BNN_MAX_PEERS && peers->rank >= 0 && peers->rank < peers->world,
              BNN_ERR_BAD_ARGUMENT, "bnn_peer_average: need 1 <= world <= %d and 0 <= rank < world", BNN_MAX_PEERS);
  if (numel == 0 || peers->world == 1) return BNN_OK;
  int rc = check_device();
  if (rc != BNN_OK) return rc;
  AverageParams p;
  for (int r = 0; r < BNN_MAX_PEERS; ++r) {
    p.peer[r] = r < peers->world ? const_cast<float*>(peers->base[r]) : nullptr;
    BNN_REQUIRE(r >= peers->world || (p.peer[r] != nullptr && aligned16(p.peer[r])), BNN_ERR_BAD_ARGUMENT,
                "bnn_peer_average: peer gradient buffer %d is NULL or not 16-byte aligned", r);
  }
  p.world = peers->world; p.rank = peers->rank;
  const int64_t per = ((numel + peers->world - 1) / peers->world + 3) / 4 * 4;      // slice length, a multiple of 4
  p.begin = per * peers->rank < numel ? per * peers->rank : numel;
  p.end = p.begin + per < numel ? p.begin + per : numel;
  if (p.end <= p.begin) return BNN_OK;
  const int64_t n4 = (p.end - p.begin + 3) / 4;
  const int64_t blocks = (n4 + kThreads - 1) / kThreads;
  const int grid = static_cast<int>(blocks < sm_count() * 8 ? blocks : sm_count() * 8);
  peer_average_kernel<<<grid, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(p);
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}

extern "C" int bnn_peer_barrier(uint32_t* const* flags, int32_t world, int32_t rank, uint32_t* epoch_dev, void* stream) {
  BNN_REQUIRE(flags != nullptr && epoch_dev != nullptr, BNN_ERR_BAD_ARGUMENT, "bnn_peer_barrier: NULL pointer");
  BNN_REQUIRE(world >= 1 && world <= BNN_MAX_PEERS && rank >= 0 && rank < world, BNN_ERR_BAD_ARGUMENT,
              "bnn_peer_barrier: need 1 <= world <= %d and 0 <= rank < world", BNN_MAX_PEERS);
  int rc = check_device();
  if (rc != BNN_OK) return rc;
  BarrierParams p;
  for (int r = 0; r < BNN_MAX_PEERS; ++r) {
    p.flags[r] = r < world ? flags[r] : nullptr;
    BNN_REQUIRE(r >= world || flags[r] != nullptr, BNN_ERR_BAD_ARGUMENT, "bnn_peer_barrier: flag block %d is NULL", r);
  }
  p.epoch = epoch_dev; p.world = world; p.rank = rank;
  peer_barrier_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(p);
  BNN_CUDA_OK(cudaGetLastError());
  return BNN_OK;
}
