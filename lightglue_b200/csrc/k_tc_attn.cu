// tcgen05 flash attention for the tensor-core path (lightglue.py:113-137: softmax(q k^T / 8) v, no mask).
//
// One CTA owns 256 query rows (two 128-row tiles) of one (sequence, head) and sweeps the key/value
// sequence in blocks of 64:
//   S_t = Q_t K_j^T      tcgen05.mma  M=128 N=64 K=64    operands in shared memory (TMA, 128B swizzle)
//   P_t = exp2(c S_t - c m_t)   softmax warpgroup t: TMEM -> registers -> fp16 -> TMEM (in place over S_t)
//   O_t += P_t V_j       tcgen05.mma  M=128 N=64 K=64    A = P_t from TMEM, B = V^T tile in shared memory
// O(N) softmax against a lazily moved reference maximum: a block's exponentials are taken against the reference of the
// earlier blocks WITHOUT looking for the row maximum first; the block's row sum (needed anyway) shows whether any P left the
// safe fp16 range, and only then the true maximum is taken, O / l are rescaled and the block is redone.  The denominator is
// summed in registers (packed f32x2 adds), one division at the end.
// 256 TMEM columns and ~100 KB of shared memory per CTA, so TWO CTAs are resident per SM: four softmax warps per
// scheduler hide the TMEM-load / barrier latencies of a block.  TMEM map: S0 0-63 | S1 64-127 | O0 128-191 | O1 192-255.
// Warp roles (384 threads = 3 warpgroups): warpgroup 0 = {warp 0 TMA producer, warp 1 TMEM owner + MMA issuer of
// tile 0, warp 2 MMA issuer of tile 1, 1 idle warp} shrinks its registers (setmaxnreg.dec); warpgroups 1 and 2 are
// the softmax warpgroups of query tile 0 / 1 (one query row per thread; warp w reads TMEM lanes 32*(w%4)..).
#include "lg_handle.h"
#include "tc_common.cuh"

using namespace tc;

namespace {

constexpr int QT = 128;          // query rows per tile
constexpr int KB = 64;           // keys per block
constexpr int Q_TILE_BYTES = QT * 64 * 2;   // 16 KB
constexpr int K_TILE_BYTES = KB * 64 * 2;   // 8 KB
constexpr float SCALE_LOG2 = 0.125f * 1.4426950408889634f;  // dh^-0.5 * log2(e)

struct AttnParams {
  CUtensorMap q_map;   // (64, Lp, S*H)   box (64, 128, 1)
  CUtensorMap k_map;   // (64, Lp, S*H)   box (64, 64, 1)
  CUtensorMap vt_map;  // (Lp, 64, S*H)   box (64, 64, 1)
  __nv_bfloat16* ctxh; __nv_bfloat16* ctxl;
  int kv_shift;
  int rows_per_cta;  // 256 (two query tiles per CTA) or 128 (one: small problems that would not fill the SMs)
  SeqState st;
  unsigned int* dbg;
};

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// packed fp32 pairs (sm_100 FFMA2 / FADD2: one issue slot for two elements)
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// pipeline waits of this kernel: try_wait with a suspend-time hint, so that a waiting warp sleeps in hardware instead
// of spending issue slots on polling (the softmax warps need them); bounded like tc::mbar_wait
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity, unsigned int* dbg, uint32_t site, uint32_t extra = 0) {
  uint32_t spins = 0;
  for (;;) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(20000u)
        : "memory");
    if (ok) return;
    ++spins;
    if (spins == 8 && dbg && *reinterpret_cast<volatile unsigned int*>(dbg + 31) != 0u) return;
    if (spins > (1u << 14)) {
      if (dbg) {
        atomicCAS(dbg + (site & 31), 0u, 0x80000000u | ((extra & 0xffff) << 12) | (threadIdx.x & 0xfff));
        atomicExch(dbg + 31, 1u);
      }
      return;
    }
  }
}
__device__ __forceinline__ float max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// One softmax warpgroup: query tile t (of nt in this CTA), one query row per thread.  ts / to: TMEM addresses of S_t / O_t
// (lane offset of this warp included); r: global row of this thread, off: its offset in the context images.
__device__ __forceinline__ void softmax_tile(const AttnParams& p, int t, int nt, uint32_t ts, uint32_t to, uint64_t* s_full,
                                             uint64_t* p_full, uint64_t* o_final, int nkv, int len_kv, int len_q, int r, long off) {
        float m_used = -INFINITY, l = 0.f;
        uint32_t sv[2][32];
        // The two query tiles of the CTA alternate their exponential phases (a token per scheduler, below).  Measured
        // alternatives on B200 (B = 32, N = 2048, per launch; this kernel: 385 - 390 us):
        //  * FOUR tiles in one 640-thread CTA per SM with a ring of four tokens: +10 %;
        //  * a persistent one-CTA-per-SM kernel with DOUBLE-BUFFERED S (S_{j+1} = Q K_{j+1}^T issued under the exponentials of
        //    block j, so the wait for S disappears from the tile's chain; 2 tiles x (2 x 64 S + 64 O) = 384 TMEM columns):
        //    448 us with alternating tiles, 479 free-running; with two threads per row (eight softmax warps per tile,
        //    barrier.red over the warp pair for the lazy-maximum decision) 450 / 490; with mbarrier tokens per
        //    scheduler 497; degree-3 polynomial exp2 for 1/8 - 4/8 of the elements on top of any of them: no gain.
        //    A softmax warp spends ~1100 cycles per 64-key block outside its exponentials even when S is ready (barrier
        //    round trips ~90-200 cycles each, TMEM load, store drain, branches), and only TMEM for two tiles fits with
        //    double buffering: four resident tiles that wait for their MMAs beat two that do not.
        //  (tools/micro/micro_exp.cu: the exponential phase alone runs at 9.8 cycles per MUFU with one warp per scheduler and
        //  8.2 with two -- the 8-cycle MUFU issue rate -- so the phase itself is not what is slow.)
        const bool pingpong = nt > 1;
        // One token per SCHEDULER: the warp of tile 0 and the warp of tile 1 that own the same row quarter share a
        // scheduler and its MUFU; named barrier 2 + 2 q + t (64 threads) hands the exponential phase from one to the other,
        // so a hand-over never waits for the slowest of the four schedulers (a CTA-wide token, barriers 2 / 3 with 256
        // threads, measured 1 % slower; passing the token after half of the block's exponentials measured the same).
        const int qd = (threadIdx.x / 32) % 4;
        const int bar_self = 2 + 2 * qd + t, bar_next = 2 + 2 * qd + (t ^ 1);
        const bool ring_last = t + 1 == nt;
        if (pingpong && ring_last) asm volatile("bar.arrive %0, 64;" ::"r"(bar_next) : "memory");  // tile 0 goes first
        // P = exp2(c s - c m_used) of one 64-key block: scale-and-shift and row sum as packed f32x2 operations, P stored
        // in place over S; returns the row sum of the block.  (A degree-3 Cody-Waite polynomial for 12 - 50 % of the
        // exponentials on the FMA pipe, packed f32x2, was measured on B200: 405 - 468 us per launch against 412 with
        // every exponential on the MUFU -- no gain; measured again with a degree-4 polynomial and the per-scheduler token:
        // 397 us for 1 pair in 8, 411 for 2 in 8, against 389, profiles/r2_y_attention_poly_exp2.log.)
        auto exp_block = [&](float m) -> float {
          const uint64_t sc2 = pack2(SCALE_LOG2, SCALE_LOG2);
          const float nmc = -m * SCALE_LOG2;
          const uint64_t nm2 = pack2(nmc, nmc);
          uint64_t la = pack2(0.f, 0.f), lb = pack2(0.f, 0.f);
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint32_t pk[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              float x0, x1;
              unpack2(fma2(pack2(__uint_as_float(sv[c][2 * i]), __uint_as_float(sv[c][2 * i + 1])), sc2, nm2), x0, x1);
              const float e0 = ex2(x0), e1 = ex2(x1);
              if (i & 1) lb = add2(lb, pack2(e0, e1));
              else la = add2(la, pack2(e0, e1));
              const __half2 hh = __floats2half2_rn(e0, e1);
              pk[i] = *reinterpret_cast<const uint32_t*>(&hh);
            }
            tmem_st16(ts + c * 16, pk);
          }
          float a0, a1;
          unpack2(add2(la, lb), a0, a1);
          return a0 + a1;
        };
        for (int j = 0; j < nkv; ++j) {
          mbar_wait_sleep(&s_full[t], j & 1, p.dbg, 6, j * 2 + t);
          tc_fence_after();
          const int valid = len_kv - j * KB;
          tmem_ld32(ts, sv[0]);
          tmem_ld32(ts + 32, sv[1]);
          tmem_ld_wait();
          if (valid < KB) {
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (c * 32 + i >= valid) sv[c][i] = 0xff800000u;
          }
          // Fast path: NO row maximum.  The exponentials are taken against the reference maximum m_used of the earlier
          // blocks and the block's row sum (needed anyway) tells whether that was safe: sum <= 2^14 means every P <= 2^14,
          // far inside fp16; anything else (a larger value, +inf) sends the WARP through the slow path below, which takes
          // the true row maximum, rescales O / l and redoes the block.  m_used only moves when it has to, so the slow
          // path runs in the first block and a few more per row (the row-maximum pass cost 430 - 780 cycles of the ~2900
          // per block in the clock trace, on the critical chain of the tile).
          // Ping-pong between the two query tiles of the CTA (named barriers 2 / 3): the exponentials of tile t run
          // while tile 1-t waits for its MMAs, and vice versa (measured on B200: 410 us per launch against 427 without).
          float bsum = 0.f;
          bool slow = j == 0;
          if (j > 0) {
            if (pingpong) asm volatile("bar.sync %0, 64;" ::"r"(bar_self) : "memory");
            bsum = exp_block(m_used);
            if (pingpong && !(ring_last && j + 1 == nkv)) asm volatile("bar.arrive %0, 64;" ::"r"(bar_next) : "memory");  // the other tile's turn
            slow = !(bsum <= 16384.f);
          } else if (pingpong) {
            asm volatile("bar.sync %0, 64;" ::"r"(bar_self) : "memory");
            if (!(ring_last && j + 1 == nkv)) asm volatile("bar.arrive %0, 64;" ::"r"(bar_next) : "memory");
          }
          if (__any_sync(0xffffffffu, slow)) {
            tmem_st_wait();  // the block's first P store must have landed before it is stored again
            float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                mx0 = max3(mx0, __uint_as_float(sv[c][i]), __uint_as_float(sv[c][i + 1]));
                mx1 = max3(mx1, __uint_as_float(sv[c][i + 2]), __uint_as_float(sv[c][i + 3]));
              }
            const float mx = fmaxf(mx0, mx1);
            float alpha = 1.f;
            if (slow && mx > m_used) {
              if (m_used != -INFINITY) alpha = ex2((m_used - mx) * SCALE_LOG2);
              m_used = mx;
            }
            if (j > 0) {  // S_t(j) was issued after P_t(j-1) V: that MMA has retired, O_t may be rescaled
#pragma unroll 1
              for (int c = 0; c < 4; ++c) {
                uint32_t o16[16];
                tmem_ld16(to + c * 16, o16);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; ++i) o16[i] = __float_as_uint(__uint_as_float(o16[i]) * alpha);
                tmem_st16(to + c * 16, o16);
              }
              l *= alpha;
            }
            bsum = exp_block(m_used);  // lanes whose reference did not move reproduce their block bit for bit
          }
          l += bsum;
          tmem_st_wait();
          tc_fence_before();
          mbar_arrive(&p_full[t]);
        }
        mbar_wait_sleep(&o_final[t], 0, p.dbg, 8, t);
        tc_fence_after();
        const float inv = l > 0.f ? 1.f / l : 0.f;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          tmem_ld32(to + c * 32, sv[c]);
          tmem_ld_wait();
          if (r < len_q) {
            uint32_t ph[16], pl[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float a = __uint_as_float(sv[c][2 * i]) * inv, b = __uint_as_float(sv[c][2 * i + 1]) * inv;
              ph[i] = pack_bf16x2(a, b);
              pl[i] = pack_bf16x2_lo(a, b, ph[i]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              reinterpret_cast<uint4*>(p.ctxh + off + c * 32)[i] = make_uint4(ph[4 * i], ph[4 * i + 1], ph[4 * i + 2], ph[4 * i + 3]);
              if (p.ctxl)
                reinterpret_cast<uint4*>(p.ctxl + off + c * 32)[i] = make_uint4(pl[4 * i], pl[4 * i + 1], pl[4 * i + 2], pl[4 * i + 3]);
            }
          }
        }
}

constexpr int B_KV_STAGES = 4;
constexpr int B_V_TILE_BYTES = 64 * 128;                      // [64 d rows][64 keys]
constexpr int B_STAGE_BYTES = K_TILE_BYTES + B_V_TILE_BYTES;  // 16 KB

__global__ void __launch_bounds__(384, 2) tc_attention2_kernel(const __grid_constant__ AttnParams p) {
  pdl_launch_dependents();
  pdl_wait();  // the sequence lengths read right below belong to the dependency chain
  const int s = blockIdx.z, h = blockIdx.y, r0 = blockIdx.x * p.rows_per_cta;
  const int len_q = p.st.len[s];
  if (r0 >= len_q || lg_pair_stopped(p.st, s)) return;
  const int skv = (s + p.kv_shift) % p.st.S;
  const int len_kv = p.st.len[skv];
  const int nkv = (len_kv + KB - 1) / KB;
  const int nt = (p.rows_per_cta > QT && len_q - r0 > QT) ? 2 : 1;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // align by OFFSETTING the shared array (not by rebuilding a pointer from an integer): the compiler keeps the
  // shared address space and emits LDS / STS instead of generic LD / ST for everything derived from it
  uint8_t* smem = smem_raw + ((1024u - (static_cast<uint32_t>(reinterpret_cast<uintptr_t>(smem_raw)) & 1023u)) & 1023u);
  uint8_t* sq = smem;                                  // 2 x 16 KB
  uint8_t* skvb = smem + 2 * Q_TILE_BYTES;             // B_KV_STAGES x 16 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(skvb + B_KV_STAGES * B_STAGE_BYTES);
  uint64_t* q_full = bars;
  uint64_t* kv_full = bars + 1;
  uint64_t* kv_empty = kv_full + B_KV_STAGES;
  uint64_t* s_full = kv_empty + B_KV_STAGES;  // [2]
  uint64_t* p_full = s_full + 2;              // [2]
  uint64_t* o_final = p_full + 2;             // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_final + 2);

  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.q_map);
    tma_prefetch_desc(&p.k_map);
    tma_prefetch_desc(&p.vt_map);
    mbar_init(q_full, 1);
    for (int i = 0; i < B_KV_STAGES; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], nt); }
    for (int t = 0; t < 2; ++t) { mbar_init(&s_full[t], 1); mbar_init(&p_full[t], 128); mbar_init(&o_final[t], 1); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<256>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");  // 80 -> 32 frees 6144 registers = exactly what 2 x 128 x (104 - 80) needs
    if (nkv > 0) {
      if (warp == 0) {
        if (elect_one()) {
          mbar_arrive_expect_tx(q_full, 2 * Q_TILE_BYTES);
          tma_load_3d(sq, &p.q_map, 0, r0, s * LG_HEADS + h, q_full);
          tma_load_3d(sq + Q_TILE_BYTES, &p.q_map, 0, r0 + QT, s * LG_HEADS + h, q_full);
          for (int j = 0; j < nkv; ++j) {
            const int stage = j % B_KV_STAGES, round = j / B_KV_STAGES;
            mbar_wait_sleep(&kv_empty[stage], (round & 1) ^ 1, p.dbg, 1, j);
            uint8_t* dst = skvb + stage * B_STAGE_BYTES;
            mbar_arrive_expect_tx(&kv_full[stage], B_STAGE_BYTES);
            tma_load_3d(dst, &p.k_map, 0, j * KB, skv * LG_HEADS + h, &kv_full[stage]);
            tma_load_3d(dst + K_TILE_BYTES, &p.vt_map, j * KB, 0, skv * LG_HEADS + h, &kv_full[stage]);
          }
        }
      } else if (warp - 1 < nt) {
        // MMA issuer of tile t: S_t(0); then per block: wait P_t(j) -> O_t += P_t V_j ; S_t(j+1) = Q_t K_{j+1}^T
        const int t = warp - 1;
        constexpr uint32_t idesc_qk = make_idesc(QT, KB, false);  // M=128 N=64, fp16
        constexpr uint32_t idesc_pv = make_idesc(QT, 64, false);  // M=128 N=64, fp16
        const uint64_t qdesc = make_sdesc_sw128(smem_u32(sq + t * Q_TILE_BYTES));
        const uint64_t kdesc0 = make_sdesc_sw128(smem_u32(skvb));
        const uint64_t vdesc0 = make_sdesc_sw128(smem_u32(skvb + K_TILE_BYTES));
        const uint32_t ts_addr = tmem_base + t * 64;
        const uint32_t to_addr = tmem_base + 128 + t * 64;
        auto issue_qk = [&](int j) {
          const uint64_t kdesc = kdesc0 + (uint64_t)((j % B_KV_STAGES) * (B_STAGE_BYTES >> 4));
#pragma unroll
          for (int k = 0; k < 4; ++k) mma_ss(ts_addr, qdesc + 2 * k, kdesc + 2 * k, idesc_qk, k > 0 ? 1u : 0u);
          mma_commit(&s_full[t]);
        };
        mbar_wait_sleep(q_full, 0, p.dbg, 2);
        mbar_wait_sleep(&kv_full[0], 0, p.dbg, 3);
        tc_fence_after();
        if (elect_one()) issue_qk(0);
        __syncwarp();
        for (int j = 0; j < nkv; ++j) {
          const int stage = j % B_KV_STAGES;
          if (j + 1 < nkv) mbar_wait_sleep(&kv_full[(j + 1) % B_KV_STAGES], ((j + 1) / B_KV_STAGES) & 1, p.dbg, 4, j);
          mbar_wait_sleep(&p_full[t], j & 1, p.dbg, 5, j * 2 + t);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t vdesc = vdesc0 + (uint64_t)(stage * (B_STAGE_BYTES >> 4));
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              mma_ts(to_addr, ts_addr + ks * 8, vdesc + 2 * ks, idesc_pv, (j > 0 || ks > 0) ? 1u : 0u);
            mma_commit(&kv_empty[stage]);
            // in-order tensor pipe: S_t(j+1) overwrites S_t / P_t(j) only after P_t(j) V_j has consumed it
            if (j + 1 < nkv) issue_qk(j + 1);
            else mma_commit(&o_final[t]);
          }
          __syncwarp();
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    const int t = (warp - 4) / 4;
    const int quarter = warp % 4;
    const int row = quarter * 32 + lane;
    const int r = r0 + t * QT + row;
    const long off = ((long)s * p.st.Lp + r) * LG_DIM + h * LG_HDIM;
    if (nkv > 0) {
      if (t < nt) {
        const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
        softmax_tile(p, t, nt, tmem_base + lane_off + t * 64, tmem_base + lane_off + 128 + t * 64, s_full, p_full, o_final, nkv,
                     len_kv, len_q, r, off);
      }
    } else if (r < len_q) {
      for (int i = 0; i < 8; ++i) {
        reinterpret_cast<uint4*>(p.ctxh + off)[i] = make_uint4(0, 0, 0, 0);
        if (p.ctxl) reinterpret_cast<uint4*>(p.ctxl + off)[i] = make_uint4(0, 0, 0, 0);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<256>(tmem_base);
}


struct AttnMapCache {
  const void* q; const void* k; const void* vt; int S, Lp;
  CUtensorMap qm, km, vm;
};
}  // namespace

int tc_attention(LgHandle* h, const TcBuffers& b, const SeqState& st, int kv_shift, const __half* kbuf, cudaStream_t stream) {
  h->launches += 1;
  // tensor maps depend only on (buffers, S, Lp): cache the last two sets (self: k = b.k, cross: k = b.q); the
  // buffer addresses are unique per device (UVA), so the cache is safe with several devices in one process
  static thread_local AttnMapCache cache[2];
  AttnMapCache* c = nullptr;
  for (auto& e : cache)
    if (e.q == b.q && e.k == kbuf && e.vt == b.vt && e.S == st.S && e.Lp == st.Lp) c = &e;
  if (!c) {
    c = &cache[kbuf == b.q ? 1 : 0];
    const uint64_t SH = (uint64_t)st.S * LG_HEADS, Lp = st.Lp;
    int r;
    if ((r = tc_make_tmap_3d(&c->qm, b.q, 2, 64, Lp, SH, 128, Lp * 128, 64, QT, 1))) return r;
    if ((r = tc_make_tmap_3d(&c->km, kbuf, 2, 64, Lp, SH, 128, Lp * 128, 64, KB, 1))) return r;
    if ((r = tc_make_tmap_3d(&c->vm, b.vt, 2, Lp, 64, SH, Lp * 2, 64 * Lp * 2, 64, 64, 1))) return r;
    c->q = b.q; c->k = kbuf; c->vt = b.vt; c->S = st.S; c->Lp = st.Lp;
  }
  AttnParams p;
  p.q_map = c->qm; p.k_map = c->km; p.vt_map = c->vm;
  p.ctxh = b.ctxh; p.ctxl = b.ctxl; p.kv_shift = kv_shift; p.st = st; p.dbg = h->tc.dbg;
  dim3 grid((st.Lp + 2 * QT - 1) / (2 * QT), LG_HEADS, st.S);
  p.rows_per_cta = 2 * QT;
  if ((long)grid.x * grid.y * grid.z < 2 * lg_num_sms()) {  // fewer CTAs than resident slots: one query tile per CTA instead
    p.rows_per_cta = QT;
    grid.x = st.Lp / QT;
  }
  constexpr int smem2 = 2 * Q_TILE_BYTES + B_KV_STAGES * B_STAGE_BYTES + 1024 + 256;
  if (int r = lg_func_smem_once((const void*)tc_attention2_kernel, smem2)) return r;
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute at[1];
  cfg.gridDim = grid; cfg.blockDim = dim3(384); cfg.dynamicSmemBytes = smem2; cfg.stream = stream;
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, tc_attention2_kernel, p);
  if (e != cudaSuccess) return lg_set_cuda_error(e, __FILE__, __LINE__);
  return 0;
}
