// sm_100a primitives used by the tensor-core kernels: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (TMEM alloc / mma / commit / ld / st) and the shared-memory / instruction descriptors.
// Hand-written inline PTX; nothing here depends on CUTLASS.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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
// Bounded spin: a protocol bug must never hang the GPU box.  After ~2^18 failed probes the waiter records
// a site code (read back by lg_debug_timeout_code()) and gives up; the kernel then finishes with garbage instead
// of dead-locking, and the host can report where it stalled.
// dbg points at 32 words; word `site` keeps the first code recorded there: 0x80000000 | extra << 12 | thread;
// word 31 is the "some wait has timed out" flag: once it is set every other long wait gives up after 64 probes,
// so a broken pipeline drains in milliseconds instead of minutes.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, unsigned int* dbg, uint32_t site,
                                          uint32_t extra = 0) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    ++spins;
    if (spins == 64 && dbg && *reinterpret_cast<volatile unsigned int*>(dbg + 31) != 0u) return;
    if (spins > (1u << 18)) {
      if (dbg) {
        atomicCAS(dbg + (site & 31), 0u, 0x80000000u | ((extra & 0xffff) << 12) | (threadIdx.x & 0xfff));
        atomicExch(dbg + 31, 1u);
      }
      return;
    }
  }
}
// same, acquiring at cluster scope (the arrival may come from the peer CTA of a pair)
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
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity, unsigned int* dbg, uint32_t site,
                                                  uint32_t extra = 0) {
  uint32_t spins = 0;
  while (!mbar_try_wait_cluster(bar, parity)) {
    ++spins;
    if (spins == 64 && dbg && *reinterpret_cast<volatile unsigned int*>(dbg + 31) != 0u) return;
    if (spins > (1u << 18)) {
      if (dbg) {
        atomicCAS(dbg + (site & 31), 0u, 0x80000000u | ((extra & 0xffff) << 12) | (threadIdx.x & 0xfff));
        atomicExch(dbg + 31, 1u);
      }
      return;
    }
  }
}
// CTA pairs (cta_group::2): in the shared::cluster window bit 24 of a shared-memory address selects the CTA of the
// pair; clearing it addresses the same offset in the even ("leader") CTA
constexpr uint32_t PAIR_LEADER_MASK = 0xFEFFFFFFu;
// arrive on the barrier at this offset in the LEADER CTA of the pair (from either CTA).  Plain arrive (no
// cluster-scope release: that costs a MEMBAR + ERRBAR per arrival, 10-16 % of the epilogue's stall samples): what the
// barrier orders here are TMEM reads against later MMAs, which the tcgen05 fences on both sides cover.
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PAIR_LEADER_MASK) : "memory");
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// CTA-pair loads (cta_group::2): the box lands in THIS CTA's shared memory, the transaction bytes complete on the
// barrier at `bar`'s offset in the LEADER CTA (the single MMA-issuing thread of the pair waits there)
__device__ __forceinline__ void tma_load_2d_cg2(void* smem_dst, const CUtensorMap* m, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(m), "r"(smem_u32(bar) & PAIR_LEADER_MASK), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_cg2(void* smem_dst, const CUtensorMap* m, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(m), "r"(smem_u32(bar) & PAIR_LEADER_MASK), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// TMA stores (shared -> global), tracked by per-thread bulk async-groups
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(m), "r"(smem_u32(smem_src)),
               "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(m),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all of this thread's stores have finished READING shared memory (the buffers may be rewritten)
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all but the most recent bulk store group have finished READING their shared-memory source
__device__ __forceinline__ void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
// all of this thread's stores have completed
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---------------------------------------------------------------- tcgen05 / TMEM
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "n"(NCOLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
// CTA-pair variants: the same warp of BOTH CTAs of the pair executes them with the same shared-memory offset
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "n"(NCOLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]      (single CTA, kind::f16: fp16 / bf16 operands, fp32 accumulate)
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// CTA pair: D[tmem of both CTAs] (+)= A[256 rows: 128 in each CTA's smem] * B[N rows: N/2 in each CTA's smem];
// issued by one thread of the LEADER CTA, descriptors are shared-memory offsets valid in both CTAs
__device__ __forceinline__ void mma_ss_cg2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once the pair's MMAs issued so far have completed) on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void mma_commit_cg2(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp gets lane (base_lane + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// Programmatic dependent launch (kernels launched with cudaLaunchAttributeProgrammaticStreamSerialization):
// `pdl_launch_dependents` lets the next kernel of the stream become resident as SMs drain, `pdl_wait` blocks until
// every kernel this one depends on has completed and its memory is visible.  Nothing before `pdl_wait` may touch
// global memory a predecessor writes; both are no-ops in a plain launch.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor, K-major operand tile whose rows are 128 bytes (64 x 16-bit) with
// the 128-byte swizzle (matches CU_TENSOR_MAP_SWIZZLE_128B boxes of inner extent 64 elements):
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (= 1, unused for swizzled K-major) |
//   [32,46) SBO >> 4 (= 1024 B: eight 128-byte rows) | [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_sdesc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// Instruction descriptor, kind::f16, fp32 accumulate, both operands K-major.
//   [4,6) D format (1 = f32) | [7,10) A format | [10,13) B format (0 = f16, 1 = bf16) | [15] A major | [16] B major
//   [17,23) N >> 3 | [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc(int m, int n, bool bf16) {
  return (1u << 4) | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(m >> 4) << 24);
}

// bf16 packing without per-element F2F conversions (those run on the slow XU pipe): one cvt.rn.bf16x2.f32 per pair,
// and the hi values are recovered for the lo split with integer shifts
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {  // a -> low half
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_bf16x2_lo(float a, float b, uint32_t hi) {  // bf16(a - hi.a), bf16(b - hi.b)
  return pack_bf16x2(a - __uint_as_float(hi << 16), b - __uint_as_float(hi & 0xffff0000u));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

}  // namespace tc

// ---------------------------------------------------------------- host: tensor maps
// cuTensorMapEncodeTiled is fetched through the runtime (no link-time dependency on libcuda).
int tc_make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner, uint64_t outer, uint64_t row_stride_bytes,
                    uint32_t box_inner, uint32_t box_outer, bool swizzle128 = true);
int tc_make_tmap_3d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t d0, uint64_t d1, uint64_t d2,
                    uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t b0, uint32_t b1, uint32_t b2);
