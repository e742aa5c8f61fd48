// Inline-PTX wrappers for the Blackwell (sm_100a) features the lfmq kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld), clusters + DSMEM.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace lfmq {
namespace sm100 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// cluster-scope variants (remote arrive = release.cluster on a mapa address; wait = acquire.cluster)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t remote_bar_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait_cluster(bar, parity)) {
  }
}

__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// release at gpu scope (cumulative: covers what this thread has observed, e.g. across a preceding bar.sync)
__device__ __forceinline__ void red_release_gpu_add(unsigned int* p, unsigned int v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long v;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v));
  return v;
}

// ---- proxies / fences -------------------------------------------------------------------------
// generic-proxy smem writes -> visible to the async proxy (TMA, tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- clusters / DSMEM -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() {
  cluster_arrive();
  cluster_wait();
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void st_cluster_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}

// ---- TMA --------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
// TMA store of a 3-D box shared::cta -> global as one bulk async-group member; rows outside the tensor are clipped.
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// 1-D bulk copy global -> shared::cta (size a multiple of 16 B), completing tx-bytes on a local mbarrier
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the committed groups have finished READING shared memory (the source may be overwritten)
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all but the most recent committed group have finished reading shared memory
__device__ __forceinline__ void bulk_wait_group_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
// the committed groups are complete (their global writes are done)
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// multicast: the box lands at the same CTA-relative offset (and signals the same-offset mbarrier) in every CTA
// of `cta_mask`.
__device__ __forceinline__ void tma_load_2d_mcast(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                                  uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster "
      "[%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask)
      : "memory");
}
// Bulk copy local smem -> (remote) smem of a cluster peer; completes `bytes` of tx on the peer's mbarrier.
// dst / bar are shared::cluster addresses (mapa), src is a shared::cta address; bytes % 16 == 0.
__device__ __forceinline__ void bulk_copy_s2c(uint32_t dst_cluster_addr, uint32_t src_cta_addr, uint32_t bytes,
                                              uint32_t bar_cluster_addr) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   dst_cluster_addr),
               "r"(src_cta_addr), "r"(bytes), "r"(bar_cluster_addr)
               : "memory");
}
// Asynchronous L2 prefetch of `bytes` (multiple of 16) starting at a 16-byte aligned global address.
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// generic-proxy global writes (acquired from a peer) -> ordered before this thread's async-proxy (TMA) global reads
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- programmatic dependent launch ----------------------------------------------------------------
// wait: returns once the preceding kernel of the stream has completed and its writes are visible (a no-op when the
// kernel was not launched with the programmatic-stream-serialization attribute); launch_dependents: the next kernel's
// CTAs may be dispatched as soon as every CTA of this grid has executed it (or exited).
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- register re-allocation between warpgroups (4 aligned consecutive warps execute it together) ---------
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// ---- TMEM allocation ---------------------------------------------------------------------------
// Whole-warp calls.  ncols: power of two in [32, 512].
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ---- UMMA descriptors --------------------------------------------------------------------------
constexpr uint32_t LAYOUT_NONE = 0, LAYOUT_SW128 = 2, LAYOUT_SW64 = 4, LAYOUT_SW32 = 6;

// 64-bit shared-memory matrix descriptor (sm_100 format: version field = 1 at bit 46).
//   K-major,  SWIZZLE_128B: rows of 128 B; SBO = byte stride between 8-row groups (1024 when dense); LBO unused.
//   K-major,  SWIZZLE_64B : rows of  64 B; SBO = 512 when dense.
//   MN-major, SWIZZLE_128B: 128 B (64 elements of MN) per k row; SBO = byte stride between 8-k-row groups (1024),
//                           LBO = byte stride between successive 64-element MN blocks.
__host__ __device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                            uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}

// 32-bit instruction descriptor for kind::f16, bf16 x bf16 -> fp32.
__host__ __device__ __forceinline__ uint32_t make_idesc_bf16(uint32_t M, uint32_t N, bool a_mn_major, bool b_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;    // D format = F32
  d |= 1u << 7;    // A format = BF16
  d |= 1u << 10;   // B format = BF16
  d |= (a_mn_major ? 1u : 0u) << 15;
  d |= (b_mn_major ? 1u : 0u) << 16;
  d |= (N >> 3) << 17;
  d |= (M >> 4) << 24;
  return d;
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrives on `bar` when all previously issued MMAs of this thread have completed (implies fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// the same arrive on the barrier at this offset in every CTA of `cta_mask` (multicast operand rings: a stage is free
// only when all CTAs that received it have consumed it)
__device__ __forceinline__ void umma_commit_mcast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

// ---- TMEM loads ---------------------------------------------------------------------------------
// 32x32b: thread i of the warp reads TMEM lane (lane_base + i), `n` consecutive 32-bit columns.
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t v[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t v[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t v[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- TMEM stores (registers -> TMEM), same 32x32b addressing as the loads ---------------------------------
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t v[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t v[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- 256-bit global accesses (sm_100: STG/LDG .256) -- one full 32-byte sector per thread ----------------
__device__ __forceinline__ void st_global_v8(void* p, const uint32_t v[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]),
               "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void st_global_v8f(void* p, const float v[8]) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]),
               "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}
__device__ __forceinline__ void ld_global_v8(const void* p, uint32_t v[8]) {
  asm volatile("ld.global.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void ld_global_v8f(const void* p, float v[8]) {
  asm volatile("ld.global.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}

// ---- math ---------------------------------------------------------------------------------------
__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sigmoid_approx(float x) { return fmaf(0.5f, tanh_approx(0.5f * x), 0.5f); }
// packed bf16x2 helpers (one MUFU op evaluates two tanh)
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t tanh_bf16x2(uint32_t x) {
  uint32_t y;
  asm("tanh.approx.bf16x2 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}
__device__ __forceinline__ uint32_t fma_bf16x2(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("fma.rn.bf16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t mul_bf16x2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t add_bf16x2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("add.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t neg_bf16x2(uint32_t a) { return a ^ 0x80008000u; }
constexpr uint32_t BF16X2_ONE = 0x3F803F80u;
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

}  // namespace sm100
}  // namespace lfmq
