// umma.cuh — thin inline-PTX wrappers for the sm_100a tensor-core path (tcgen05 + TMEM + mbarrier)
// and the canonical K-major SWIZZLE_128B shared-memory tile the kernels stage operands in.
//
// Tile convention (one "K-major SW128" operand tile of fp32/TF32 data):
//   R rows (R % 8 == 0) x 32 columns; a row is 128 bytes; 8 rows form a 1024-byte swizzle atom;
//   the 16-byte chunk c16 of row r lives at   (r/8)*1024 + (r%8)*128 + ((c16 ^ (r%8)) * 16).
// The matching UMMA shared-memory descriptor has SBO = 1024 B, layout SWIZZLE_128B, version 1;
// a UMMA K-step (8 TF32 = 32 B) advances the start address by 32 B inside the atom.
#pragma once
#include <cstdint>

namespace bnn {
namespace umma {

constexpr int kTileCols = 32;            // fp32 elements per 128-byte row
constexpr int kRowBytes = 128;
constexpr int kAtomBytes = 1024;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t tile_offset(int row, int c16) {
  return static_cast<uint32_t>((row >> 3) * kAtomBytes + (row & 7) * kRowBytes + (((c16 ^ row) & 7) << 4));
}

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must fail the launch (trap), never hang the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint64_t t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  while (!mbar_try_wait(bar, parity)) {
    uint64_t t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > 4000000000ull) __trap();   // 4 s
  }
}

// ---- proxy / tcgen05 fences -------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---- TMEM -------------------------------------------------------------------------------------
// whole warp; ncols power of two in [32, 512]; the base address lands in *dst_smem
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// 32 lanes x 16 consecutive columns: thread t of the warp receives lane (base_lane + t)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// 32 lanes x 16 consecutive columns, registers -> TMEM (same lane mapping as tmem_ld16)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      :
      : "r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
        "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
        "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])),
        "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])),
        "r"(__float_as_uint(v[15]))
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// issue-only variant of tmem_ld16: pair with tmem_ld_wait() before the registers are read
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- mbarrier arrive (generic threads) / named barriers ---------------------------------------
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- shared-memory stores by 32-bit shared address ---------------------------------------------
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t a) {
  asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(a) : "memory");
}

// ---- descriptors + MMA ------------------------------------------------------------------------
// K-major, SWIZZLE_128B, SBO 1024 B, LBO (ignored) 1, descriptor version 1 (sm_100)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  return static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu) | (uint64_t(1) << 16) |
         (uint64_t(kAtomBytes >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
// descriptor of the tile `units16` 16-byte units after the tile that `base_desc` describes (the 14-bit start-address
// field cannot overflow: shared memory is < 256 KiB) — one 32-bit add per MMA instead of rebuilding the descriptor
__device__ __forceinline__ uint64_t desc_advance(uint64_t base_desc, uint32_t units16) {
  return base_desc + units16;
}
// kind::tf32, fp32 accumulate, M x N tile; a_mn / b_mn select MN-major (transposed) operand tiles
__device__ __forceinline__ uint32_t make_idesc_tf32(int m, int n, bool a_mn = false, bool b_mn = false) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (a_mn ? (1u << 15) : 0u) | (b_mn ? (1u << 16) : 0u) |
         (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
// MN-major operand tile of fp32/TF32 data.  For 32-bit MN-major operands the only swizzled layout tcgen05 accepts is
// SWIZZLE_128B_BASE32B (CuTe: Layout_MN_SW128_32B_Atom = Swizzle<2,5,2> o (32 MN x 4 K) : (1, 32)): 32 consecutive MN
// elements form a 128-byte row, 4 K-rows form a 512-byte swizzle atom in which the 32-BYTE chunk c32 of K-row r sits
// at r*128 + ((c32 ^ r) * 32); the next 4 K-rows follow at SBO, the next 32 MN elements at LBO.  It is what TMA
// writes with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.  One UMMA K-step (8 TF32) = two atoms.
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu) | (static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         (static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32) | (uint64_t(1) << 46) | (uint64_t(1) << 61);
}
// byte offset of element (mn, k) inside an MN-major tile with the given LBO / SBO
__device__ __forceinline__ uint32_t tile_offset_mn(int mn, int k, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  const int r = k & 3;
  return static_cast<uint32_t>(mn >> 5) * lbo_bytes + static_cast<uint32_t>(k >> 2) * sbo_bytes +
         static_cast<uint32_t>(r * kRowBytes) + static_cast<uint32_t>(((((mn & 31) >> 3) ^ r) << 5) + ((mn & 7) << 2));
}

// ---- TMA (cp.async.bulk.tensor) -----------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 3-d tile load: coordinates (c0 = innermost element, c1 = row, c2 = sample); out-of-bounds elements are zero
__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const void* tmap, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// 2-d tile load: coordinates (c0 = innermost element index, c1 = row index); completes on `bar` (tx bytes)
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const void* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, one K-step of 8 TF32 elements; issued by ONE thread
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                         uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate ? 1u : 0u)
      : "memory");
}
// arrive on an mbarrier once every MMA issued so far by this thread has completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---- CTA pairs (cta_group::2): two SMs of one TPC compute one 256-row MMA tile; the B operand is split between
// their shared memories, so each SM stages only half of it -----------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local_smem_addr` in the CTA of rank `cta`
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_smem_addr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  uint64_t t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  while (!mbar_try_wait_cluster(bar, parity)) {
    uint64_t t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > 4000000000ull) __trap();   // 4 s
  }
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A * B^T for a 256 x N tile; issued by ONE thread of the leader CTA (rank 0)
__device__ __forceinline__ void mma_tf32_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate ? 1u : 0u)
      : "memory");
}
// arrive on the barrier at the same shared-memory offset in every CTA of `cta_mask` once the MMAs issued so far finish
__device__ __forceinline__ void mma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}
// 3-d TMA tile load of a CTA pair: data lands in THIS CTA's shared memory, the transaction bytes complete on the
// barrier at `mbar_cluster_addr` (the leader CTA's barrier)
__device__ __forceinline__ void tma_load_3d_pair(uint32_t smem_dst, const void* tmap, int c0, int c1, int c2,
                                                 uint32_t mbar_cluster_addr) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(mbar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// ---- TMA im2col mode (implicit-GEMM convolution): the tensor map describes an NHWC activation tensor (dims C, W, H, N)
// with the filter's bounding box; a load delivers `pixelsPerColumn` consecutive OUTPUT pixels (traversed w, then h, then
// n, with the convolution stride) x `channelsPerPixel` channels, read at (base pixel + filter-tap offset), zero outside
// the image — i.e. one (rows x 32) tile of the im2col matrix for the k-block (tap, c0 .. c0 + 31) without the matrix.
// (w, h, n) = the first base pixel = output pixel * stride + lower corner; (off_w, off_h) = tap * dilation.
__device__ __forceinline__ void tma_load_im2col_4d(uint32_t smem_dst, const void* tmap, int c, int w, int h, int n,
                                                   uint16_t off_w, uint16_t off_h, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2], {%7, %8};"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(n),
        "h"(off_w), "h"(off_h)
      : "memory");
}
// CTA-pair form: data lands in THIS CTA's shared memory, the bytes complete on the barrier at `mbar_cluster_addr`
__device__ __forceinline__ void tma_load_im2col_4d_pair(uint32_t smem_dst, const void* tmap, int c, int w, int h, int n,
                                                        uint16_t off_w, uint16_t off_h, uint32_t mbar_cluster_addr) {
  asm volatile(
      "cp.async.bulk.tensor.4d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], "
      "[%1, {%3, %4, %5, %6}], [%2], {%7, %8};"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(mbar_cluster_addr), "r"(c), "r"(w), "r"(h), "r"(n),
        "h"(off_w), "h"(off_h)
      : "memory");
}
// 3-d convolutions: NDHWC tensor {c, w, h, d, n} through a rank-5 im2col map, tap offsets {w, h, d}
__device__ __forceinline__ void tma_load_im2col_5d(uint32_t smem_dst, const void* tmap, int c, int w, int h, int d, int n,
                                                   uint16_t off_w, uint16_t off_h, uint16_t off_d, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes [%0], "
      "[%1, {%3, %4, %5, %6, %7}], [%2], {%8, %9, %10};"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c), "r"(w), "r"(h), "r"(d), "r"(n),
        "h"(off_w), "h"(off_h), "h"(off_d)
      : "memory");
}
__device__ __forceinline__ void tma_load_im2col_5d_pair(uint32_t smem_dst, const void* tmap, int c, int w, int h, int d,
                                                        int n, uint16_t off_w, uint16_t off_h, uint16_t off_d,
                                                        uint32_t mbar_cluster_addr) {
  asm volatile(
      "cp.async.bulk.tensor.5d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], "
      "[%1, {%3, %4, %5, %6, %7}], [%2], {%8, %9, %10};"
      :
      : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(mbar_cluster_addr), "r"(c), "r"(w), "r"(h), "r"(d),
        "r"(n), "h"(off_w), "h"(off_h), "h"(off_d)
      : "memory");
}

__host__ __device__ constexpr uint32_t tmem_cols_pow2(uint32_t need) {
  return need <= 32 ? 32u : need <= 64 ? 64u : need <= 128 ? 128u : need <= 256 ? 256u : 512u;
}

}  // namespace umma
}  // namespace bnn
