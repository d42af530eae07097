// tcgen05 / TMA linear layers for the LG_PREC_BF16 and LG_PREC_BF16X3 paths.
//
//   C[128 rows, 256 cols per accumulator slot] = A[rows, K] * W[cols, K]^T     (fp32 accumulate in TMEM)
//
// * operands are bf16, K-major; tiles are staged by TMA (128-byte swizzle) into a shared-memory ring, one elected
//   thread of a CTA pair issues tcgen05.mma (M=256 over the pair, N=256, K=16), tcgen05.commit releases the ring
//   slot and finally signals the epilogue warps, which read the accumulator back with tcgen05.ld;
// * LG_PREC_BF16X3 runs three passes over K into the same accumulator: A_lo*W_hi + A_hi*W_lo +
//   A_hi*W_hi with x = hi + lo, hi = bf16(x), lo = bf16(x - hi)  (~16 mantissa bits per operand);
// * A may be the concatenation of two sources along K (the FFN input cat([x, msg]), lightglue.py:172);
// * fused epilogues: bias (+ RoPE, head split, V transpose) for the QKV projections, bias +
//   LayerNorm(512) + exact GELU for ffn.0 (two 256-column accumulator slots = the whole 512-column TMEM),
//   bias + residual for ffn.3, bias * scale for input_proj / final_proj.
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2-5 = epilogue
// (warp w reads TMEM lanes 32*(w%4) .. +31, one accumulator row per thread).
#include <stdio.h>

#include <unordered_map>

#include "lg_handle.h"
#include "tc_common.cuh"

using namespace tc;

namespace {

constexpr int BM = 128, BN = 256, BK = 64;
constexpr int A_TILE_BYTES = BM * BK * 2;  // 16 KB
constexpr int W_TILE_BYTES = BN * BK * 2;  // 32 KB

enum { TEPI_QKV = 0, TEPI_LN_GELU = 2, TEPI_RESID = 3, TEPI_F32 = 4, TEPI_LSE = 5, TEPI_ARGMAX = 6, TEPI_CONV = 7 };

struct TcLinParams {
  CUtensorMap a_hi[2], a_lo[2];  // A segment 0 / 1
  CUtensorMap w_hi, w_lo;        // 3-D: (K, Nout, select), box 64 x 128 rows (mma_n / 2): each CTA of a pair holds one half of the N tile
  int kb0, kb_total, passes, n_tiles;
  int epi, rope;
  SeqState st;
  int w_select;                  // 1: third TMA coordinate / bias offset = stop_layer[pair] - 1
                                 // 2: third TMA coordinate = partner sequence (similarity sweeps of the assignment)
  float* part; int* part_arg; int part_stride;  // TEPI_LSE: (max, sumexp) pairs; TEPI_ARGMAX: best / arg, [S*Lp, part_stride]
  const float* term;             // TEPI_ARGMAX: logsigmoid(z) - LSE per token, [S, Lp]
  int reverse;  // walk the tile list from its end: a kernel that reads what the previous kernel wrote LAST finds it in L2
  float* logmat; int mat_m, mat_n;  // TEPI_ARGMAX, optional: materialise the [B, M+1, N+1] log-assignment matrix (core block)
  const float* bias; long bias_sel_stride;
  float scale;
  float* out_f32; int ldo;
  __nv_bfloat16* out_h; __nv_bfloat16* out_l; int ldb;
  __half* q; __half* k; __half* vt; const float* cs;
  const float* ln_g; const float* ln_b;
  unsigned int* dbg;
  // 3x3 convolution as a GEMM over a zero-padded NHWC image [rows = B (H+2) (W+2), Cin] (SuperPoint encoder): K block kb
  // = (tap, 64-channel block); the A tile of a tap is the same matrix shifted by (dy (W+2) + dx) rows (TMA fills the
  // rows outside the tensor with zeros).  conv_cb = Cin / 64 (0: not a convolution).  TEPI_CONV zeroes the padding
  // pixels again on the way out (conv_w2 = W + 2, conv_plane = (H+2)(W+2), conv_rows = B conv_plane) and applies ReLU.
  int conv_cb, conv_w2, conv_h, conv_w, relu;
  long conv_plane, conv_rows;
  int mma_n;  // N of the MMAs when fewer than 256 output columns exist (64 / 128; 0 = 256): each CTA then
              // holds mma_n / 2 rows of the W tile and the accumulator uses the first mma_n columns of its slot
  // epilogue tensor maps (all boxes are 32 rows x 128 bytes, 128B swizzle)
  CUtensorMap o_h;          // bf16 hi output [rows, ldb], box 64 cols x 32 rows, 128B swizzle (two chunks per store)
  CUtensorMap o_l32;        // bf16 lo output, box 32 cols x 32 rows, no swizzle (one chunk per store)
  CUtensorMap o_h32;        // bf16 hi output, same dense box (LayerNorm variant)
  CUtensorMap o_f32;        // fp32 output / residual [rows, 256], box 32 cols (TEPI_RESID loads and stores through it)
  CUtensorMap o_q, o_k;     // fp16 [S*H, Lp, 64], box (64, 32, 1)
  CUtensorMap cs_map;       // fp32 [rows, 64] cos | sin, box 32 cols
};

// ------------------------------------------------------------------------------------------------
// Persistent kernel: grid = #SMs, every CTA walks the tile list (n-tile fastest, so neighbouring CTAs
// share A tiles in L2).  320 threads: warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 2-9
// epilogue.  With one 256-column accumulator slot per tile TMEM holds two accumulators, so the epilogue
// of tile i overlaps the MMAs of tile i+1; the LayerNorm variant needs all 512 columns for one tile.
// Epilogue data path: TMEM -> registers (one row per thread) -> per-warp 32x32 fp32 staging tile in
// shared memory (XOR-swizzled, conflict-free both ways) -> registers in a row-contiguous layout (8 lanes
// x 16 B per row) -> coalesced global loads / stores.
// ------------------------------------------------------------------------------------------------

// CTA pairs (cta_group::2).  The two CTAs of a cluster take the two row tiles of a "tile pair" with the same
// n-tile; one thread of the leader CTA issues M=256 MMAs that read A (128 rows) and HALF of the W tile (128 of its
// 256 rows) from each CTA's shared memory, so every SM receives only half of the weight bytes and a ring stage is
// 32 KB.  X3: split-bf16 with the K block outermost -- one stage holds A_hi, A_lo, W_hi, W_lo of a 64-wide K block
// and feeds all three passes (A_lo W_hi, A_hi W_lo, A_hi W_hi): the W_hi / A_hi tiles are loaded once instead of
// twice.  With two accumulator slots (LayerNorm variant) the slots take consecutive stages of the same format.
template <int NSLOT, bool X3>
struct LinCfg {
  // accumulator hand-over barriers: NSLOT == 1: two 256-column buffers used by alternate tiles; NSLOT == 2 (LayerNorm):
  // the two 256-column SLOTS of one tile, completed and released one after the other
  static constexpr int NBUF = 2;
  // epilogue warps: 8 (two per TMEM lane quarter, 128 columns each); the LayerNorm variant (512 columns, the
  // instruction-heaviest epilogue) runs 16 so that four warps per scheduler hide its latencies
  static constexpr int EW = NSLOT == 1 ? 8 : 16;
  static constexpr int GROUPS = EW / 4;
  // control warps ahead of the epilogue warps: TMA producer, MMA issuer
  static constexpr int CTRL = 2;
  static constexpr int THREADS = (CTRL + EW) * 32;
  static constexpr int W_PART = W_TILE_BYTES / 2;  // bytes of one W tile held by this CTA
  static constexpr int STAGE_BYTES = X3 ? 2 * A_TILE_BYTES + 2 * W_PART : A_TILE_BYTES + W_PART;
  static constexpr int COLS = NSLOT * BN;
  // per epilogue warp: box A (4 KB: fp32 32x32 output box / rotary cos), box B (4 KB: 16-bit 32x64 box, hi or
  // fp16), box C (4 KB: rotary sin, or the dense 32x32 bf16 "lo" box).  The LayerNorm variant has no box A.
  // (NSLOT == 2: one dense 32x32 bf16 box, 2 KB, shared by the hi and lo images)
  static constexpr int WARP_BYTES = NSLOT == 1 ? 3 * 4096 : 2048;
  // LayerNorm variant: 16 of the 64 slot-0 values every epilogue thread keeps across the MMAs of slot 1 live in shared
  // memory, the other 48 in registers (576 threads leave 96 registers per thread)
  static constexpr int STASH_SMEM = NSLOT == 2 ? 16 : 0;
  static constexpr int STASH_BYTES = STASH_SMEM * EW * 32 * 4;
  static constexpr int BOXB_OFF = NSLOT == 1 ? 4096 : 0;
  static constexpr int BOXC_OFF = NSLOT == 1 ? 8192 : 0;
  static constexpr int VEC_BYTES = (NSLOT == 1 ? 1 : 3) * COLS * 4;     // bias (| ln gamma | ln beta)
  static constexpr int LNP_BYTES = NSLOT == 1 ? 0 : 128 * GROUPS * 2 * 8;  // LayerNorm partial (mean, M2) per row, slot and column group
  static constexpr int FIXED_BYTES = EW * WARP_BYTES + VEC_BYTES + LNP_BYTES + STASH_BYTES + 512 + 1024;
  static constexpr int SMEM_MAX = 232448;  // 227 KB per CTA
  static constexpr int FIT = (SMEM_MAX - FIXED_BYTES) / STAGE_BYTES;
  static constexpr int STAGES = FIT > 6 ? 6 : FIT;
  static_assert(STAGES >= 2, "the TMA ring needs at least two stages");
  static constexpr int SMEM = STAGES * STAGE_BYTES + FIXED_BYTES;
};

__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
template <int NTHREADS>
__device__ __forceinline__ void epi_bar_n() { asm volatile("bar.sync 1, %0;" ::"n"(NTHREADS) : "memory"); }  // the epilogue warps

// Row tiles ("slots") per sequence.  With per-tile weight selection the two CTAs of a pair share one W tile, so a pair
// must not straddle two sequences: an odd tile count gets one more slot, a dead tile past the sequence's end (its A rows
// are the next sequence's or TMA zero fill; its epilogue stores nothing).  Without weight selection pairs may cross.
__host__ __device__ __forceinline__ int row_slots(const SeqState& st, int w_select) {
  const int tiles = st.Lp / BM;
  return tiles + (w_select != 0 && tiles % 2 != 0);
}
// tiles of the launch; S is even, so they come in pairs
__host__ __device__ __forceinline__ int total_tiles(const TcLinParams& p) {
  return p.n_tiles * p.st.S * row_slots(p.st, p.w_select);
}

struct TileInfo {
  int s, r0, n_tile, sel, len;
  long grow0;
};
// decode tile t (n-tile fastest); returns false for tiles with nothing to do (all fields are filled either way)
__device__ __forceinline__ bool decode_tile(const TcLinParams& p, int t, int n_tiles, TileInfo& ti) {
  const int slots = row_slots(p.st, p.w_select);
  ti.n_tile = t % n_tiles;
  const int rt = t / n_tiles;
  ti.s = rt / slots;
  ti.r0 = (rt % slots) * BM;
  ti.len = p.st.len[ti.s];
  ti.grow0 = (long)ti.s * p.st.Lp + ti.r0;
  ti.sel = 0;
  const int pair = ti.s >= p.st.B ? ti.s - p.st.B : ti.s;
  const int sl = p.st.stop_layer[pair];
  bool live = ti.r0 < ti.len;
  if (p.w_select == 1) ti.sel = sl > 0 ? sl - 1 : 0;
  else if (p.w_select == 2) {
    ti.sel = ti.s >= p.st.B ? ti.s - p.st.B : ti.s + p.st.B;
    live = live && ti.n_tile * BN < p.st.len[ti.sel];  // no live columns otherwise
  } else if (sl != 0) live = false;                      // pair already exited (lightglue.py:549-550)
  return live;
}

// Tile schedule: the two CTAs of a cluster take the two row tiles of a "tile pair" with the same n-tile; both walk
// the same list of tile pairs.
struct TileWalk {
  int cur, step, end, rank, n_tiles;
  __device__ TileWalk(int total_tiles, int n_tiles_) : n_tiles(n_tiles_) {
    rank = (int)cluster_ctarank();
    cur = blockIdx.x / 2; step = gridDim.x / 2; end = total_tiles / 2;
  }
  // returns false when done; `mine` = this CTA's tile (decoded), `store` = its epilogue may write (the pair runs loads
  // and MMAs as long as either tile is live)
  __device__ bool next(const TcLinParams& p, TileInfo& mine, bool& store) {
    while (cur < end) {
      const int id = p.reverse ? end - 1 - cur : cur;
      cur += step;
      const int n_tile = id % n_tiles, rtp = id / n_tiles;
      TileInfo peer;
      const bool lm = decode_tile(p, (rtp * 2 + rank) * n_tiles + n_tile, n_tiles, mine);
      const bool lp = decode_tile(p, (rtp * 2 + (rank ^ 1)) * n_tiles + n_tile, n_tiles, peer);
      if (!lm && !lp) continue;
      store = lm;
      return true;
    }
    return false;
  }
};

template <int NSLOT, int EPI, bool X3>
__global__ void __launch_bounds__(LinCfg<NSLOT, X3>::THREADS, 1) tc_linear_kernel(const __grid_constant__ TcLinParams p) {
  using C = LinCfg<NSLOT, X3>;
  constexpr int EPI_WARPS = C::EW;
  auto epi_bar = [] { epi_bar_n<C::EW * 32>(); };
  constexpr int STAGES = C::STAGES, NBUF = C::NBUF, STAGE_BYTES = C::STAGE_BYTES, COLS = C::COLS;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // align by OFFSETTING the shared array (not by rebuilding a pointer from an integer): the compiler keeps the
  // shared address space and emits LDS / STS instead of generic LD / ST for everything derived from it
  uint8_t* smem = smem_raw + ((1024u - (static_cast<uint32_t>(reinterpret_cast<uintptr_t>(smem_raw)) & 1023u)) & 1023u);
  uint8_t* epi_smem = smem + STAGES * STAGE_BYTES;  // 1024-aligned: per-warp TMA boxes
  float* s_bias = reinterpret_cast<float*>(epi_smem + EPI_WARPS * C::WARP_BYTES);
  float* s_gamma = s_bias + (NSLOT == 1 ? 0 : COLS);       // LayerNorm variant only
  float* s_beta = s_gamma + (NSLOT == 1 ? 0 : COLS);
  float2* s_lnp = reinterpret_cast<float2*>(s_bias + C::VEC_BYTES / 4);  // [GROUPS][128 rows]
  float* s_stash = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(s_lnp) + C::LNP_BYTES);  // [STASH_SMEM][epilogue threads]
  uint64_t* full = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(s_stash) + C::STASH_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* acc_full = empty + STAGES;
  uint64_t* acc_empty = acc_full + NBUF;
  uint64_t* ldbar = acc_empty + NBUF;  // [EPI_WARPS] per-warp TMA-load barriers (residual / rotary boxes)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ldbar + EPI_WARPS);

  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int n_tiles = p.n_tiles;
  const int tiles = total_tiles(p);
  // ring iterations per tile: (K block, accumulator slot), split-bf16 passes inside an iteration
  const int iters = p.kb_total * NSLOT;
  const int rank = (int)cluster_ctarank();

  pdl_launch_dependents();  // the next kernel's CTAs may take this SM as soon as this CTA has left it
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.a_hi[0]);
    tma_prefetch_desc(&p.w_hi);
    // only the leader's `full` / `acc_empty` barriers are waited on (its TMA bytes AND the peer's complete there; both
    // CTAs' epilogue warps arrive there); `empty` / `acc_full` exist in both CTAs and receive the leader's multicast
    // commits
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < NBUF; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 2 * EPI_WARPS); }
    for (int i = 0; i < EPI_WARPS; ++i) mbar_init(&ldbar[i], 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_cg2<512>(tmem_slot);
  if (EPI == TEPI_LN_GELU && warp >= C::CTRL) {
    for (int i = threadIdx.x - C::CTRL * 32; i < COLS; i += EPI_WARPS * 32) { s_gamma[i] = p.ln_g[i]; s_beta[i] = p.ln_b[i]; }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer's barriers are initialised before anything can arrive on them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // everything above (barriers, TMEM, descriptor prefetch, LayerNorm vectors = weights) overlapped the tail of the
  // previous kernel; activations, lengths and stop flags are only read from here on
  pdl_wait();

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      int g = 0;  // global k-block counter across tiles (ring position)
      TileWalk walk(tiles, n_tiles);
      TileInfo ti;
      bool store;
      while (walk.next(p, ti, store)) {
        for (int it = 0; it < iters; ++it, ++g) {
          const int stage = g % STAGES, round = g / STAGES;
          mbar_wait(&empty[stage], (round & 1) ^ 1, p.dbg, 17, it);
          uint8_t* sa = smem + stage * STAGE_BYTES;
          // this CTA's A rows and its half (128 of 256 rows) of the W tile; the bytes of BOTH CTAs complete on the
          // leader's barrier, which only the leader arms
          const int sl_ = it / p.kb_total, kb = it % p.kb_total;  // slot outermost: slot 0 completes (and is normalised) first
          int seg = kb >= p.kb0 ? 1 : 0;
          int kc = (seg ? kb - p.kb0 : kb) * BK;
          int arow = (int)ti.grow0;
          if (p.conv_cb) {  // convolution tap: shifted rows of the padded image, channel block kb % conv_cb
            const int tap = kb / p.conv_cb;
            arow += (tap / 3 - 1) * p.conv_w2 + (tap % 3 - 1);
            kc = (kb % p.conv_cb) * BK;
            seg = 0;
          }
          const int wpart = p.mma_n ? p.mma_n * (BK * 2 / 2) : C::W_PART;  // bytes of this CTA's half of the W tile
          const int wrow = (ti.n_tile * NSLOT + sl_) * BN + rank * (p.mma_n ? p.mma_n / 2 : BN / 2);
          if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * (X3 ? 2 * A_TILE_BYTES + 2 * wpart : A_TILE_BYTES + wpart));
          if (X3) {
            tma_load_2d_cg2(sa, &p.a_hi[seg], kc, arow, &full[stage]);
            tma_load_2d_cg2(sa + A_TILE_BYTES, &p.a_lo[seg], kc, arow, &full[stage]);
            tma_load_3d_cg2(sa + 2 * A_TILE_BYTES, &p.w_hi, kb * BK, wrow, ti.sel, &full[stage]);
            tma_load_3d_cg2(sa + 2 * A_TILE_BYTES + C::W_PART, &p.w_lo, kb * BK, wrow, ti.sel, &full[stage]);
          } else {
            tma_load_2d_cg2(sa, &p.a_hi[seg], kc, arow, &full[stage]);
            tma_load_3d_cg2(sa + A_TILE_BYTES, &p.w_hi, kb * BK, wrow, ti.sel, &full[stage]);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    const uint32_t idesc = make_idesc(2 * BM, p.mma_n ? p.mma_n : BN, true);
    int g = 0, li = 0;  // li: index among this CTA's live tiles
#ifdef LG_TC_TRACE
    long long trm[8][4];
    const bool tracing = EPI == TEPI_LN_GELU && blockIdx.x == 0;
#endif
    TileWalk walk(tiles, n_tiles);
    TileInfo ti;
    bool store;
    while (rank == 0 && walk.next(p, ti, store)) {  // the leader issues for both CTAs
      const int buf = NSLOT == 1 ? li % NBUF : 0;
      const uint32_t par = NSLOT == 1 ? (uint32_t)((li / NBUF) & 1) : (uint32_t)(li & 1);
      // the epilogue warps of both CTAs have drained this accumulator; the LayerNorm variant waits per slot, right
      // before the slot's first MMA, so that slot 0 of the next tile overlaps the normalisation of slot 1
      if (NSLOT == 1) {
        mbar_wait_cluster(&acc_empty[buf], par ^ 1, p.dbg, 20, li);
        tc_fence_after();
      }
      const uint32_t acc = tmem_base + buf * BN;
      for (int it = 0; it < iters; ++it, ++g) {
        const int stage = g % STAGES, round = g / STAGES;
        if (NSLOT == 2 && it % p.kb_total == 0) {
          mbar_wait_cluster(&acc_empty[it / p.kb_total], par ^ 1, p.dbg, 20, li);
          tc_fence_after();
        }
#ifdef LG_TC_TRACE
        if (tracing && li < 8 && it % p.kb_total == 0) trm[li][(it / p.kb_total) * 2] = clock64();  // slot free
#endif
        mbar_wait(&full[stage], round & 1, p.dbg, 18, it);
        tc_fence_after();
#ifdef LG_TC_TRACE
        if (tracing && li < 8 && it % p.kb_total == p.kb_total - 1) trm[li][(it / p.kb_total) * 2 + 1] = clock64();  // last stage of the slot arrived
#endif
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const int sl_ = it / p.kb_total, kb = it % p.kb_total;
          const uint32_t d = acc + sl_ * BN;
          if (X3) {
            const uint64_t ahi = make_sdesc_sw128(sa), alo = make_sdesc_sw128(sa + A_TILE_BYTES);
            const uint64_t whi = make_sdesc_sw128(sa + 2 * A_TILE_BYTES), wlo = make_sdesc_sw128(sa + 2 * A_TILE_BYTES + C::W_PART);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) mma_ss_cg2(d, alo + 2 * k, whi + 2 * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) mma_ss_cg2(d, ahi + 2 * k, wlo + 2 * k, idesc, 1u);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) mma_ss_cg2(d, ahi + 2 * k, whi + 2 * k, idesc, 1u);
          } else {
            const uint64_t adesc = make_sdesc_sw128(sa), bdesc = make_sdesc_sw128(sa + A_TILE_BYTES);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) mma_ss_cg2(d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          mma_commit_cg2(&empty[stage], (uint16_t)3);  // frees the stage in both CTAs
          if (kb == p.kb_total - 1) mma_commit_cg2(&acc_full[buf + sl_], (uint16_t)3);  // this 256-column accumulator is complete
        }
        __syncwarp();
      }
      ++li;
    }
#ifdef LG_TC_TRACE
    if (tracing && lane == 0 && rank == 0)
      for (int i = 0; i < li && i < 8; ++i)
        printf("TRM tile %d slot0_free %lld slot0_last_full %lld slot1_free %lld slot1_last_full %lld\n", i, trm[i][0], trm[i][1], trm[i][2], trm[i][3]);
#endif
  } else if (warp >= C::CTRL) {
    // ------------------------------------------------------------------ epilogue (8 or 16 warps)
    // Everything stays in the row-per-thread layout tcgen05.ld delivers: results are packed into 32-row x
    // 128-byte shared-memory boxes in the 128B-swizzle pattern and leave through TMA stores; the fp32
    // residual and the rotary tables arrive the same way through TMA loads.  No per-lane global traffic.
    const int ew = warp - C::CTRL;
    const int quarter = warp % 4;                 // TMEM lane group this warp may read
    const int half = ew / 4;                      // which column group of the tile this warp owns
    constexpr int HCOLS = COLS / C::GROUPS;       // columns per warp (128)
    const int te = threadIdx.x - C::CTRL * 32;    // index among the epilogue threads
    uint8_t* wsm = epi_smem + ew * C::WARP_BYTES;
    uint8_t* boxA = wsm;                          // fp32 box / cos (NSLOT == 1 only)
    uint8_t* boxB = wsm + C::BOXB_OFF;            // 16-bit box: 32 rows x 64 elements, swizzled
    uint8_t* boxC = wsm + C::BOXC_OFF;            // sin box (swizzled fp32) or dense bf16 lo box (32 rows x 64 B)
    const int row = quarter * 32 + lane;          // accumulator row of this thread
    const int sw = lane & 7;                      // swizzle key of this thread's box row
    uint8_t* arow = boxA + lane * 128;
    uint8_t* brow = boxB + lane * 128;
    uint8_t* crow_sw = boxC + lane * 128;         // as a swizzled 128-byte row (sin)
    uint8_t* crow_lo = boxC + lane * 64;          // as a dense 64-byte row (lo)
    uint32_t ld_phase = 0;
    int li = 0;
#ifdef LG_TC_TRACE
    long long tre[8][6];
    const bool tracing = EPI == TEPI_LN_GELU && blockIdx.x == 0 && ew == 0;
#endif
    TileWalk walk(tiles, n_tiles);
    TileInfo ti;
    bool store;
    while (walk.next(p, ti, store)) {
      const int buf = NSLOT == 1 ? li % NBUF : 0;
      const uint32_t par = NSLOT == 1 ? (uint32_t)((li / NBUF) & 1) : (uint32_t)(li & 1);
      auto release_acc = [&](int bb) {  // this warp has finished reading accumulator bb
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(&acc_empty[bb]);
      };
      if (!store) {  // dead tile of a live pair: drain the accumulator(s), write nothing
        for (int bb = 0; bb < (NSLOT == 1 ? 1 : 2); ++bb) {
          mbar_wait(&acc_full[buf + bb], par, p.dbg, 23, li);
          tc_fence_after();
          release_acc(buf + bb);
        }
        ++li;
        continue;
      }
      const float* bias = p.bias + (p.w_select == 1 ? (long)ti.sel * p.bias_sel_stride : 0) + ti.n_tile * COLS;
      const int grow_w = (int)ti.grow0 + quarter * 32;   // first global row of this warp
      const bool is_sweep = EPI == TEPI_LSE || EPI == TEPI_ARGMAX;
      // which output a QKV tile feeds: packed channel order [q | k | v] (self) or [qk | v] (cross)
      const int which = ti.n_tile;  // COLS == 256 == one of q / k / v
      const bool qkv_v = EPI == TEPI_QKV && (p.rope ? which == 2 : which == 1);
      const bool use_rope = EPI == TEPI_QKV && p.rope && !qkv_v;
      if (NSLOT == 1 && use_rope && lane == 0) {
        tma_store_wait_read();              // boxes of the previous tile are free again
        mbar_arrive_expect_tx(&ldbar[ew], 8192);  // cos | sin of this warp's 32 rows (shared by all heads)
        tma_load_2d(boxA, &p.cs_map, 0, grow_w, &ldbar[ew]);
        tma_load_2d(boxC, &p.cs_map, 32, grow_w, &ldbar[ew]);
      }
      epi_bar();  // previous tile's readers of s_bias / s_lnp are done
      if (!is_sweep)
        for (int i = te; i < COLS; i += EPI_WARPS * 32) s_bias[i] = bias[i];
      epi_bar();
      if (EPI == TEPI_LN_GELU) {
        // ---------------------------------------------------------------- LayerNorm(512) + GELU, slot by slot
        // Warp (quarter, group g) owns rows 32 quarter .. +31 and columns 64 g .. +63 of BOTH 256-column slots.
        // Slot 0 is complete half an MMA phase before slot 1 (the slot is the outer loop of the K ring).  Its statistics
        // pass keeps the 64 biased values of every thread in REGISTERS and hands the slot back at once, so the tensor
        // pipe starts the next tile's slot 0 the moment this tile's slot 1 is complete: the whole normalisation (slot 0
        // from registers, then slot 1 from TMEM) runs under the next tile's MMAs.  (In-kernel clock trace before this
        // change, cycles per tile: MMAs 21.4 k + 15.5 k, then 15.8 k with the tensor pipe idle -- drain + statistics 3.4 k,
        // normalisation of slot 0 out of TMEM 11.6 k -- before the next tile could start.)
        constexpr int GC = 64;
        const uint32_t tq = tmem_base + ((uint32_t)(quarter * 32) << 16);
        constexpr int SREG = GC - C::STASH_SMEM;  // slot-0 values of this thread kept in registers (the rest: s_stash)
        uint32_t stash_u[GC];  // raw accumulators, then + bias, then the finished GELU values (bit patterns)
        float* stash = reinterpret_cast<float*>(stash_u);
        float* my_stash = s_stash + te;  // element i of this thread: my_stash[i * EPI_WARPS * 32] (conflict-free)
        {
          mbar_wait(&acc_full[0], par, p.dbg, 19, li);
          tc_fence_after();
#ifdef LG_TC_TRACE
          if (tracing && li < 8) tre[li][0] = clock64();
#endif
          float sh = 0.f, s1 = 0.f, s2 = 0.f;
          uint32_t tail[16];
          tmem_ld32(tq + half * GC, *reinterpret_cast<uint32_t(*)[32]>(stash_u));
          if constexpr (SREG == GC) {
            tmem_ld32(tq + half * GC + 32, *reinterpret_cast<uint32_t(*)[32]>(stash_u + 32));
          } else {
            tmem_ld16(tq + half * GC + 32, *reinterpret_cast<uint32_t(*)[16]>(stash_u + 32));
            tmem_ld16(tq + half * GC + 48, tail);
          }
          tmem_ld_wait();
          release_acc(0);  // slot 0 lives in registers now: the next tile's MMAs may overwrite it
          const float4* b4 = reinterpret_cast<const float4*>(s_bias + half * GC);
#pragma unroll
          for (int j4 = 0; j4 < GC / 4; ++j4) {
            const float4 bb = b4[j4];
            float v0, v1, v2, v3;
            if (4 * j4 < SREG) {
              v0 = stash[(4 * j4) % SREG] + bb.x; v1 = stash[(4 * j4 + 1) % SREG] + bb.y;
              v2 = stash[(4 * j4 + 2) % SREG] + bb.z; v3 = stash[(4 * j4 + 3) % SREG] + bb.w;
              stash[(4 * j4) % SREG] = v0; stash[(4 * j4 + 1) % SREG] = v1; stash[(4 * j4 + 2) % SREG] = v2; stash[(4 * j4 + 3) % SREG] = v3;
            } else {
              const int t4 = (4 * j4 - SREG) % 16;
              v0 = __uint_as_float(tail[t4]) + bb.x; v1 = __uint_as_float(tail[t4 + 1]) + bb.y;
              v2 = __uint_as_float(tail[t4 + 2]) + bb.z; v3 = __uint_as_float(tail[t4 + 3]) + bb.w;
              my_stash[(t4) * EPI_WARPS * 32] = v0; my_stash[(t4 + 1) * EPI_WARPS * 32] = v1;
              my_stash[(t4 + 2) * EPI_WARPS * 32] = v2; my_stash[(t4 + 3) * EPI_WARPS * 32] = v3;
            }
            if (j4 == 0) sh = v0;  // shift by the first element: cancellation-free E[(v-sh)^2]
            const float d0 = v0 - sh, d1 = v1 - sh, d2 = v2 - sh, d3 = v3 - sh;
            s1 += (d0 + d1) + (d2 + d3);
            s2 = fmaf(d0, d0, s2); s2 = fmaf(d1, d1, s2); s2 = fmaf(d2, d2, s2); s2 = fmaf(d3, d3, s2);
          }
          // this group: mean_g = sh + s1/GC, M2_g = sum (v - mean_g)^2 = s2 - s1^2/GC (shifted -> no cancellation)
          s_lnp[half * 128 + quarter * 32 + lane] = make_float2(sh + s1 * (1.f / GC), s2 - s1 * s1 * (1.f / GC));
        }
        {
          mbar_wait(&acc_full[1], par, p.dbg, 19, li);
          tc_fence_after();
#ifdef LG_TC_TRACE
          if (tracing && li < 8) tre[li][1] = clock64();
#endif
          float sh = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll
          for (int c0 = 0; c0 < GC; c0 += 16) {
            const int tcol = BN + half * GC + c0;
            uint32_t raw[16];
            tmem_ld16(tq + tcol, raw);
            tmem_ld_wait();
            const float4* b4 = reinterpret_cast<const float4*>(s_bias + tcol);
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const float4 bb = b4[j4];
              const float v0 = __uint_as_float(raw[4 * j4]) + bb.x, v1 = __uint_as_float(raw[4 * j4 + 1]) + bb.y;
              const float v2 = __uint_as_float(raw[4 * j4 + 2]) + bb.z, v3 = __uint_as_float(raw[4 * j4 + 3]) + bb.w;
              if (c0 == 0 && j4 == 0) sh = v0;
              const float d0 = v0 - sh, d1 = v1 - sh, d2 = v2 - sh, d3 = v3 - sh;
              s1 += (d0 + d1) + (d2 + d3);
              s2 = fmaf(d0, d0, s2); s2 = fmaf(d1, d1, s2); s2 = fmaf(d2, d2, s2); s2 = fmaf(d3, d3, s2);
            }
          }
          s_lnp[(C::GROUPS + half) * 128 + quarter * 32 + lane] = make_float2(sh + s1 * (1.f / GC), s2 - s1 * s1 * (1.f / GC));
        }
#ifdef LG_TC_TRACE
        if (tracing && li < 8) tre[li][2] = clock64();
#endif
        epi_bar();
#ifdef LG_TC_TRACE
        if (tracing && li < 8) tre[li][3] = clock64();
#endif
        // equal-sized groups merge with Chan's formula: mean = avg(mean_g), M2 = sum M2_g + GC * sum (mean_g - mean)^2
        float msum = 0.f, m2 = 0.f;
#pragma unroll
        for (int g = 0; g < 2 * C::GROUPS; ++g) { const float2 a = s_lnp[g * 128 + quarter * 32 + lane]; msum += a.x; m2 += a.y; }
        const float mean = msum * (1.f / (2 * C::GROUPS));
        float dev = 0.f;
#pragma unroll
        for (int g = 0; g < 2 * C::GROUPS; ++g) { const float dm = s_lnp[g * 128 + quarter * 32 + lane].x - mean; dev = fmaf(dm, dm, dev); }
        const float rstd = rsqrtf(fmaxf((m2 + dev * GC) * (1.f / COLS), 0.f) + 1e-5f);
        const bool haslo = p.out_l != nullptr;
        // per warp: one dense 32 x 32 bf16 box for the hi image and (pair kernels) a second one for the lo image, so that a
        // box is rewritten while the bulk store of the OTHER one is still reading (wait_group.read 1)
        uint8_t* box_hi = epi_smem + ew * C::WARP_BYTES;
        uint8_t* box_lo = box_hi + (C::WARP_BYTES > 2048 ? 2048 : 0);
        constexpr bool two_boxes = C::WARP_BYTES > 2048;
        const int grow_w2 = (int)ti.grow0 + quarter * 32;
        // exact (erf) GELU of the normalised value; erf via Abramowitz-Stegun 7.1.26 (|err| < 1.5e-7): 1 MUFU.RCP + 1 MUFU.EX2
        auto ln_gelu = [&](float xb, float g, float be) -> float {
          const float y = fmaf((xb - mean) * rstd, g, be);
          const float z = fabsf(y) * 0.70710678118654752f;
          const float tt = rcp_approx(fmaf(0.3275911f, z, 1.f));
          float pl = fmaf(1.061405429f, tt, -1.453152027f);
          pl = fmaf(pl, tt, 1.421413741f); pl = fmaf(pl, tt, -0.284496736f); pl = fmaf(pl, tt, 0.254829592f);
          const float ez = ex2_approx(-1.4426950408889634f * z * z);
          const float erf_abs = fmaf(-pl * tt, ez, 1.f);
          const float hy = 0.5f * y;
          return fmaf(copysignf(erf_abs, y), hy, hy);
        };
        // v[0..31]: 32 finished columns of this thread's row -> hi (and lo) bf16 images through the box(es)
        auto store32 = [&](const float* v, int tcol) {
          for (int pass = 0; pass < (haslo ? 2 : 1); ++pass) {
            uint8_t* box = pass == 0 ? box_hi : box_lo;
            if (lane == 0) { if (two_boxes && haslo) tma_store_wait_read1(); else tma_store_wait_read(); }  // the box may be rewritten
            __syncwarp();
            uint8_t* brow32 = box + lane * 64;
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) {
              uint32_t w[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float a = v[8 * j8 + 2 * e], b = v[8 * j8 + 2 * e + 1];
                const uint32_t hi = pack_bf16x2(a, b);
                w[e] = pass == 0 ? hi : pack_bf16x2_lo(a, b, hi);
              }
              *reinterpret_cast<uint4*>(brow32 + (j8 << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(pass == 0 ? &p.o_h32 : &p.o_l32, box, tcol, grow_w2);
              tma_store_commit();
            }
          }
        };
        // slot 0 out of the registers (and the shared-memory part of the stash)
#pragma unroll
        for (int c0 = 0; c0 < GC; c0 += 32) {
          const int tcol = half * GC + c0;
          const float4* g4 = reinterpret_cast<const float4*>(s_gamma + tcol);
          const float4* e4 = reinterpret_cast<const float4*>(s_beta + tcol);
          float* v = stash + c0;  // in place: every value is read once
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 g = g4[j4], be = e4[j4];
            const int i0 = c0 + 4 * j4;
            float x0, x1, x2, x3;
            if (i0 < SREG) { x0 = stash[i0]; x1 = stash[i0 + 1]; x2 = stash[i0 + 2]; x3 = stash[i0 + 3]; }
            else {
              const int t4 = (i0 - SREG) % 16;
              x0 = my_stash[t4 * EPI_WARPS * 32]; x1 = my_stash[(t4 + 1) * EPI_WARPS * 32];
              x2 = my_stash[(t4 + 2) * EPI_WARPS * 32]; x3 = my_stash[(t4 + 3) * EPI_WARPS * 32];
            }
            v[4 * j4] = ln_gelu(x0, g.x, be.x); v[4 * j4 + 1] = ln_gelu(x1, g.y, be.y);
            v[4 * j4 + 2] = ln_gelu(x2, g.z, be.z); v[4 * j4 + 3] = ln_gelu(x3, g.w, be.w);
          }
          store32(v, tcol);
        }
#ifdef LG_TC_TRACE
        if (tracing && li < 8) tre[li][4] = clock64();
#endif
        // slot 1 out of TMEM
#pragma unroll 1
        for (int c0 = 0; c0 < GC; c0 += 32) {
          const int tcol = BN + half * GC + c0;
          uint32_t raw[32];
          tmem_ld32(tq + tcol, raw);
          tmem_ld_wait();
          const float4* b4 = reinterpret_cast<const float4*>(s_bias + tcol);
          const float4* g4 = reinterpret_cast<const float4*>(s_gamma + tcol);
          const float4* e4 = reinterpret_cast<const float4*>(s_beta + tcol);
          float v[32];
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 bb = b4[j4], g = g4[j4], be = e4[j4];
            v[4 * j4] = ln_gelu(__uint_as_float(raw[4 * j4]) + bb.x, g.x, be.x);
            v[4 * j4 + 1] = ln_gelu(__uint_as_float(raw[4 * j4 + 1]) + bb.y, g.y, be.y);
            v[4 * j4 + 2] = ln_gelu(__uint_as_float(raw[4 * j4 + 2]) + bb.z, g.z, be.z);
            v[4 * j4 + 3] = ln_gelu(__uint_as_float(raw[4 * j4 + 3]) + bb.w, g.w, be.w);
          }
          if (c0 + 32 >= GC) release_acc(1);  // the last TMEM read of slot 1 is done: the next tile's MMAs may overwrite it
          store32(v, tcol);
        }
#ifdef LG_TC_TRACE
        if (tracing && li < 8) tre[li][5] = clock64();
#endif
        ++li;
        continue;
      }
      mbar_wait(&acc_full[buf], par, p.dbg, 19, li);
      tc_fence_after();
      const uint32_t tl = tmem_base + buf * BN + ((uint32_t)(quarter * 32) << 16) + half * HCOLS;
      const int r = ti.r0 + row;
      const bool live = r < ti.len;
      const long grow = ti.grow0 + row;
      uint32_t raw[32];

      if (is_sweep) {
        // Assignment sweeps (lightglue.py:265-277, 302-305) on a 128 x 256 tile of S = p_s p_partner^T; every
        // row reduction is thread-local, the transposed problem (partner as rows) is just another tile row.
        const int ncols = p.st.len[ti.sel] - ti.n_tile * BN - half * HCOLS;  // live columns of this warp's half
        const int slot = ti.n_tile * 2 + half;
        if (EPI == TEPI_LSE) {
          // online (max, sum-exp) in base 2: exp(x - m) = ex2(x * log2e - m * log2e), one FFMA + one MUFU per element
          constexpr float L2E = 1.4426950408889634f;
          float m = -INFINITY, se = 0.f;
          for (int c0 = 0; c0 < HCOLS && c0 < ncols; c0 += 32) {
            tmem_ld32(tl + c0, raw);
            tmem_ld_wait();
            if (c0 + 32 > ncols) {  // ragged last chunk: padding columns count as -inf
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (c0 + j >= ncols) raw[j] = 0xff800000u;
            }
            float cm = __uint_as_float(raw[0]);
#pragma unroll
            for (int j = 1; j < 32; ++j) cm = fmaxf(cm, __uint_as_float(raw[j]));
            if (cm > m) { se *= ex2_approx((m - cm) * L2E); m = cm; }
            const float mb = -m * L2E;
            float s0 = 0.f, s1 = 0.f;
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              s0 += ex2_approx(fmaf(__uint_as_float(raw[j]), L2E, mb));
              s1 += ex2_approx(fmaf(__uint_as_float(raw[j + 1]), L2E, mb));
            }
            se += s0 + s1;
          }
          if (live) reinterpret_cast<float2*>(p.part)[grow * p.part_stride + slot] = make_float2(m, se);
        } else {
          // score = 2 S + term_s[i] + term_partner[j]; the row term does not move the arg-max
          const float* ct = p.term + (long)ti.sel * p.st.Lp + ti.n_tile * BN + half * HCOLS;
          const float rterm = live ? p.term[grow] : 0.f;
          // the matrix is written from the image0 side only (rows = image0 points, columns = image1 points)
          const bool write_mat = NSLOT == 1 && p.logmat != nullptr && ti.s < p.st.B;
          float best = -INFINITY; int arg = 0;
          const int col0 = ti.n_tile * BN + half * HCOLS;
          const int rbase = ti.r0 + quarter * 32;                 // first row of this warp inside its sequence
          const int rows_ok = min(32, ti.len - rbase);            // live rows of this warp (may be <= 0)
          const long pitch = p.mat_n + 1;
          for (int c0 = 0; c0 < HCOLS && c0 < ncols; c0 += 32) {
            tmem_ld32(tl + c0, raw);
            tmem_ld_wait();
            const int nlive = ncols - c0;  // >= 32 on every chunk but a ragged last one
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const float4 c4v = __ldg(reinterpret_cast<const float4*>(ct + c0) + j4);
              const float cc[4] = {c4v.x, c4v.y, c4v.z, c4v.w};
#pragma unroll
              for (int jj = 0; jj < 4; ++jj) {
                const int j = j4 * 4 + jj;
                float sc = fmaf(2.f, __uint_as_float(raw[j]), cc[jj]);
                raw[j] = __float_as_uint(sc + rterm);
                if (j >= nlive) sc = -INFINITY;                    // uniform, false on full chunks
                if (sc > best) { best = sc; arg = col0 + c0 + j; }  // ascending j: first max wins
              }
            }
            if (write_mat && rows_ok > 0) {
              // stage the 32 x 32 block (swizzled), then every row leaves as one 128-byte store of the warp:
              // the (N+1)-float row pitch of the reference's matrix is only 4-byte aligned, so no TMA here
              __syncwarp();
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4)
                *reinterpret_cast<uint4*>(arow + ((j4 ^ sw) << 4)) = make_uint4(raw[4 * j4], raw[4 * j4 + 1], raw[4 * j4 + 2], raw[4 * j4 + 3]);
              __syncwarp();
              if (lane < nlive) {  // this lane's column exists
                float* mo = p.logmat + ((long)ti.s * (p.mat_m + 1) + rbase) * pitch + (col0 + c0 + lane);
                const uint8_t* src = boxA + ((lane & 3) << 2);
                const int l4 = lane >> 2;
                if (rows_ok == 32) {
#pragma unroll
                  for (int rr = 0; rr < 32; ++rr, mo += pitch)
                    *mo = *reinterpret_cast<const float*>(src + rr * 128 + ((l4 ^ (rr & 7)) << 4));
                } else {
                  for (int rr = 0; rr < rows_ok; ++rr, mo += pitch)
                    *mo = *reinterpret_cast<const float*>(src + rr * 128 + ((l4 ^ (rr & 7)) << 4));
                }
              }
            }
          }
          if (live) {
            p.part[grow * p.part_stride + slot] = best + rterm;
            p.part_arg[grow * p.part_stride + slot] = arg;
          }
        }
      } else {
        // residual row segments (x + ffn(...), lightglue.py:172 / 228-229) are fetched one chunk ahead: the load of
        // chunk c + 1 is in flight while chunk c is processed (its HBM latency was the top stall of this epilogue)
        float4 xr[8], xn[8];
        if (NSLOT == 1 && EPI == TEPI_RESID) {
          const float4* xp = reinterpret_cast<const float4*>(p.out_f32 + grow * p.ldo + ti.n_tile * COLS + half * HCOLS);
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) xn[j4] = xp[j4];
        }
        for (int c0 = 0; c0 < HCOLS; c0 += 32) {
          const int ci = c0 / 32;                      // chunk index inside this warp's half
          const int tcol = half * HCOLS + c0;          // column inside the tile
          const int col = ti.n_tile * COLS + tcol;     // output channel of element 0 of this chunk
          if (EPI == TEPI_CONV && col >= p.ldb) break; // Cout < 256: the weight rows beyond it are zero padding
          tmem_ld32(tl + c0, raw);
          if (NSLOT == 1 && EPI == TEPI_RESID) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) xr[j4] = xn[j4];
            if (c0 + 32 < HCOLS) {
              const float4* xp = reinterpret_cast<const float4*>(p.out_f32 + grow * p.ldo + col + 32);
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4) xn[j4] = xp[j4];
            }
          }
          if (lane == 0) tma_store_wait_read();        // every box of this warp may be rewritten
          tmem_ld_wait();
          __syncwarp();
          const float4* b4 = reinterpret_cast<const float4*>(s_bias + tcol);
          float v[32];
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 bb = b4[j4];
            v[4 * j4] = __uint_as_float(raw[4 * j4]) + bb.x; v[4 * j4 + 1] = __uint_as_float(raw[4 * j4 + 1]) + bb.y;
            v[4 * j4 + 2] = __uint_as_float(raw[4 * j4 + 2]) + bb.z; v[4 * j4 + 3] = __uint_as_float(raw[4 * j4 + 3]) + bb.w;
          }
          if (qkv_v) {
            // V is stored transposed [S, H, 64, Lp] (K-major B operand of P*V): 32 lanes = 32 consecutive rows
            if (live) {
              const int hh = tcol / LG_HDIM, d0 = tcol % LG_HDIM;
              __half* dst = p.vt + (((long)ti.s * LG_HEADS + hh) * LG_HDIM + d0) * p.st.Lp + r;
#pragma unroll
              for (int j = 0; j < 32; ++j) dst[(long)j * p.st.Lp] = __float2half_rn(v[j]);
            }
            continue;
          }
          if (p.scale != 1.f) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= p.scale;
          }
          if (EPI == TEPI_CONV) {  // ReLU, and the padding pixels of the NHWC image stay zero for the next layer's taps
            const long pp = grow % p.conv_plane;
            const int yy = (int)(pp / p.conv_w2), xx = (int)(pp % p.conv_w2);
            const bool inside = grow < p.conv_rows && yy >= 1 && yy <= p.conv_h && xx >= 1 && xx <= p.conv_w;
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = inside ? ((p.relu && v[j] < 0.f) ? 0.f : v[j]) : 0.f;
          }
          if (NSLOT == 1 && EPI == TEPI_RESID) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              v[4 * j4] += xr[j4].x; v[4 * j4 + 1] += xr[j4].y; v[4 * j4 + 2] += xr[j4].z; v[4 * j4 + 3] += xr[j4].w;
            }
          }
          // ---- rotary embedding on q / k (lightglue.py:58-65, 168-169); freq index = d / 2
          if (NSLOT == 1 && use_rope) {
            if (ci == 0) { mbar_wait(&ldbar[ew], ld_phase & 1, p.dbg, 22, 0); ld_phase++; }
            const int f0 = (tcol % LG_HDIM) / 2;  // 0 or 16
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const int chunk = (f0 >> 2) + j4;
              const float4 c4v = *reinterpret_cast<const float4*>(arow + ((chunk ^ sw) << 4));
              const float4 s4v = *reinterpret_cast<const float4*>(crow_sw + ((chunk ^ sw) << 4));
              const float cc[4] = {c4v.x, c4v.y, c4v.z, c4v.w}, ss[4] = {s4v.x, s4v.y, s4v.z, s4v.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float a = v[8 * j4 + 2 * e], b = v[8 * j4 + 2 * e + 1];
                v[8 * j4 + 2 * e] = a * cc[e] - b * ss[e];
                v[8 * j4 + 2 * e + 1] = b * cc[e] + a * ss[e];
              }
            }
          }
          const bool f32out = NSLOT == 1 && (EPI == TEPI_RESID || EPI == TEPI_F32);
          const bool fp16 = EPI == TEPI_QKV;
          const bool has16 = fp16 || EPI == TEPI_CONV || EPI == TEPI_RESID ||
                             (EPI == TEPI_F32 && p.out_h != nullptr);
          const bool haslo = has16 && !fp16 && p.out_l != nullptr;
          if (f32out) {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4)
              *reinterpret_cast<float4*>(arow + ((j4 ^ sw) << 4)) = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
          }
          if (has16) {
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) {
              uint32_t wh[4], wl[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float a = v[8 * j8 + 2 * e], b = v[8 * j8 + 2 * e + 1];
                if (fp16) {
                  const __half2 hh2 = __floats2half2_rn(a, b);
                  wh[e] = *reinterpret_cast<const uint32_t*>(&hh2);
                } else {
                  wh[e] = pack_bf16x2(a, b);
                  if (haslo) wl[e] = pack_bf16x2_lo(a, b, wh[e]);
                }
              }
              const int chunk = (ci & 1) * 4 + j8;  // 16-byte chunk inside the 64-element box row
              *reinterpret_cast<uint4*>(brow + ((chunk ^ sw) << 4)) = make_uint4(wh[0], wh[1], wh[2], wh[3]);
              if (haslo) *reinterpret_cast<uint4*>(crow_lo + (j8 << 4)) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            if (f32out) tma_store_2d(&p.o_f32, boxA, col, grow_w);
            if (haslo) tma_store_2d(&p.o_l32, boxC, col, grow_w);
            if (has16 && (ci & 1)) {  // the 64-element box is complete
              if (fp16) tma_store_3d(which == 0 ? &p.o_q : &p.o_k, boxB, 0, ti.r0 + quarter * 32, ti.s * LG_HEADS + tcol / LG_HDIM);
              else tma_store_2d(&p.o_h, boxB, col - 32, grow_w);
            }
            tma_store_commit();
          }
          __syncwarp();
        }
      }
      // accumulator drained: hand the TMEM buffer back to the MMA warp
      release_acc(buf);
      ++li;
    }
    if (lane == 0) tma_store_wait_all();
#ifdef LG_TC_TRACE
    if (tracing && lane == 0)
      for (int i = 0; i < li && i < 8; ++i)
        printf("TRE tile %d full0 %lld full1 %lld stats %lld merged %lld rel0 %lld rel1 %lld\n", i, tre[i][0], tre[i][1], tre[i][2], tre[i][3], tre[i][4], tre[i][5]);
#endif
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // no CTA leaves while the leader may still read its operands / arrive on its barriers
  if (warp == 1) tmem_dealloc_cg2<512>(tmem_base);
}

// fp32 -> bf16 hi (/ lo) for rows < len
__global__ void __launch_bounds__(256) shadow_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ hi,
                                                     __nv_bfloat16* __restrict__ lo, int cols, SeqState st) {
  const int row = blockIdx.x;
  const int s = row / st.Lp, r = row % st.Lp;
  if (r >= st.len[s]) return;
  for (int c = threadIdx.x * 4; c < cols; c += 1024) {
    const float4 t = *reinterpret_cast<const float4*>(x + (long)row * cols + c);
    const float v[4] = {t.x, t.y, t.z, t.w};
    uint2 h, l;
    h.x = pack_bf16x2(v[0], v[1]); h.y = pack_bf16x2(v[2], v[3]);
    l.x = pack_bf16x2_lo(v[0], v[1], h.x); l.y = pack_bf16x2_lo(v[2], v[3], h.y);
    *reinterpret_cast<uint2*>(hi + (long)row * cols + c) = h;
    if (lo) *reinterpret_cast<uint2*>(lo + (long)row * cols + c) = l;
  }
}

__global__ void split_weights_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                     size_t n) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = w[i];
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[i] = h;
  lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// ------------------------------------------------------------------------------------------------
// host: tensor maps (cached per handle), launches
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn get_encode() {
  static EncodeFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeFn)p;
  }
  return fn;
}
}  // namespace

int tc_make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner, uint64_t outer, uint64_t row_stride_bytes,
                    uint32_t box_inner, uint32_t box_outer, bool swizzle128) {
  EncodeFn enc = get_encode();
  if (!enc) return lg_set_error("cuTensorMapEncodeTiled unavailable");
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return lg_set_error("cuTensorMapEncodeTiled (2d) failed");
  return 0;
}

int tc_make_tmap_3d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t d0, uint64_t d1, uint64_t d2,
                    uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t b0, uint32_t b1, uint32_t b2) {
  EncodeFn enc = get_encode();
  if (!enc) return lg_set_error("cuTensorMapEncodeTiled unavailable");
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {b0, b1, b2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(out, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return lg_set_error("cuTensorMapEncodeTiled (3d) failed");
  return 0;
}

namespace {
struct MapKey {
  const void* p; uint64_t a, b, c, d;
  bool operator==(const MapKey& o) const { return p == o.p && a == o.a && b == o.b && c == o.c && d == o.d; }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = (size_t)k.p;
    for (uint64_t v : {k.a, k.b, k.c, k.d}) h = h * 1000003u ^ (size_t)v;
    return h;
  }
};
struct MapCache {
  std::unordered_map<MapKey, CUtensorMap, MapKeyHash> m;
};

// A operand: [rows, K] bf16 row-major, box 64 x 128
int amap(LgHandle* h, CUtensorMap* out, const void* base, uint64_t rows, uint64_t K) {
  MapCache* mc = static_cast<MapCache*>(h->tc.map_cache);
  MapKey key{base, rows, K, 1, 0};
  auto it = mc->m.find(key);
  if (it != mc->m.end()) { *out = it->second; return 0; }
  if (mc->m.size() > 4096) mc->m.clear();
  int r = tc_make_tmap_2d(out, base, 2, K, rows, K * 2, BK, BM);
  if (r) return r;
  mc->m.emplace(key, *out);
  return 0;
}
// W operand: nsel x [Nout, K] bf16, box 64 x box_rows x 1
int wmap(LgHandle* h, CUtensorMap* out, const void* base, uint64_t Nout, uint64_t K, uint64_t nsel, uint64_t sel_stride_elems,
         uint32_t box_rows) {
  MapCache* mc = static_cast<MapCache*>(h->tc.map_cache);
  MapKey key{base, Nout, K, nsel | ((uint64_t)box_rows << 32), sel_stride_elems + 2};
  auto it = mc->m.find(key);
  if (it != mc->m.end()) { *out = it->second; return 0; }
  if (mc->m.size() > 4096) mc->m.clear();
  int r = tc_make_tmap_3d(out, base, 2, K, Nout, nsel, K * 2, (nsel > 1 ? sel_stride_elems : Nout * K) * 2, BK, box_rows, 1);
  if (r) return r;
  mc->m.emplace(key, *out);
  return 0;
}

// epilogue boxes: 2-D [rows, cols] tensors, 32-row boxes
int omap2d(LgHandle* h, CUtensorMap* out, const void* base, int elem_bytes, uint64_t cols, uint64_t rows, uint32_t box_cols,
           bool swizzle) {
  MapCache* mc = static_cast<MapCache*>(h->tc.map_cache);
  MapKey key{base, cols, rows, (uint64_t)box_cols | ((uint64_t)swizzle << 16) | ((uint64_t)elem_bytes << 20), 7};
  auto it = mc->m.find(key);
  if (it != mc->m.end()) { *out = it->second; return 0; }
  if (mc->m.size() > 4096) mc->m.clear();
  int r = tc_make_tmap_2d(out, base, elem_bytes, cols, rows, cols * elem_bytes, box_cols, 32, swizzle);
  if (r) return r;
  mc->m.emplace(key, *out);
  return 0;
}
// q / k fp16 [S*H, Lp, 64]: box (64, 32, 1)
int omap_qk(LgHandle* h, CUtensorMap* out, const void* base, uint64_t Lp, uint64_t SH) {
  MapCache* mc = static_cast<MapCache*>(h->tc.map_cache);
  MapKey key{base, Lp, SH, 32, 9};
  auto it = mc->m.find(key);
  if (it != mc->m.end()) { *out = it->second; return 0; }
  if (mc->m.size() > 4096) mc->m.clear();
  int r = tc_make_tmap_3d(out, base, 2, 64, Lp, SH, 128, Lp * 128, 64, 32, 1);
  if (r) return r;
  mc->m.emplace(key, *out);
  return 0;
}

template <int NSLOT, int EPI>
int launch_linear_t(TcLinParams& p, int n_tiles, cudaStream_t stream) {
  const bool x3 = p.passes == 3;
  void (*kernel)(TcLinParams) = x3 ? tc_linear_kernel<NSLOT, EPI, true> : tc_linear_kernel<NSLOT, EPI, false>;
  const int smem = x3 ? LinCfg<NSLOT, true>::SMEM : LinCfg<NSLOT, false>::SMEM;
  if (int r = lg_func_smem_once((const void*)kernel, smem)) return r;
  const int num_sms = lg_num_sms();
  p.n_tiles = n_tiles;
  const int total = total_tiles(p);
  int grid = total < num_sms ? total : num_sms;
  grid &= ~1;  // whole clusters of two (total is even)
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 2;
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(LinCfg<NSLOT, false>::THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, p);
  if (e != cudaSuccess) return lg_set_cuda_error(e, __FILE__, __LINE__);
  return 0;
}
int launch_linear(TcLinParams& p, int n_tiles, cudaStream_t stream) {
  switch (p.epi) {
    case TEPI_QKV: return launch_linear_t<1, TEPI_QKV>(p, n_tiles, stream);
    case TEPI_LN_GELU: return launch_linear_t<2, TEPI_LN_GELU>(p, 1, stream);
    case TEPI_RESID: return launch_linear_t<1, TEPI_RESID>(p, n_tiles, stream);
    case TEPI_F32: return launch_linear_t<1, TEPI_F32>(p, n_tiles, stream);
    case TEPI_CONV: return launch_linear_t<1, TEPI_CONV>(p, n_tiles, stream);
    case TEPI_LSE: return launch_linear_t<1, TEPI_LSE>(p, n_tiles, stream);
    case TEPI_ARGMAX: return launch_linear_t<1, TEPI_ARGMAX>(p, n_tiles, stream);
  }
  return lg_set_error("launch_linear: bad epilogue");
}

struct LinDesc {
  const __nv_bfloat16 *a0h, *a0l; int k0;   // A segment 0: [S * Lp rows, k0]
  const __nv_bfloat16 *a1h, *a1l; int k1;   // A segment 1 (k1 = 0: none)
  const __nv_bfloat16 *wh, *wl; int nout;   // W: nsel x [nout, K] (bf16 hi / lo)
  int nsel; size_t sel_stride;
};

// A / W tensor maps, output maps and launch of one tensor-core GEMM (linears, assignment sweeps, convolutions)
int run_linear(LgHandle* h, const SeqState& st, const LinDesc& d, TcLinParams& p, cudaStream_t stream) {
  const bool x3 = h->cfg.precision == LG_PREC_BF16X3;
  const uint64_t rows = (uint64_t)st.S * st.Lp;
  const int K = p.conv_cb ? 9 * d.k0 : d.k0 + d.k1;  // a 3x3 convolution runs K over the nine taps of one A matrix
  const uint32_t wbox = (p.mma_n ? p.mma_n : BN) / 2;  // each CTA of a pair holds half of the W tile's rows
  int r;
  if ((r = amap(h, &p.a_hi[0], d.a0h, rows, d.k0))) return r;
  p.a_hi[1] = p.a_hi[0];
  if (d.k1 && (r = amap(h, &p.a_hi[1], d.a1h, rows, d.k1))) return r;
  p.a_lo[0] = p.a_hi[0]; p.a_lo[1] = p.a_hi[1];
  if (x3) {
    if ((r = amap(h, &p.a_lo[0], d.a0l, rows, d.k0))) return r;
    p.a_lo[1] = p.a_lo[0];
    if (d.k1 && (r = amap(h, &p.a_lo[1], d.a1l, rows, d.k1))) return r;
  }
  if ((r = wmap(h, &p.w_hi, d.wh, d.nout, K, d.nsel, d.sel_stride, wbox))) return r;
  p.w_lo = p.w_hi;
  if (x3 && (r = wmap(h, &p.w_lo, d.wl, d.nout, K, d.nsel, d.sel_stride, wbox))) return r;
  if (p.out_h && (r = omap2d(h, &p.o_h, p.out_h, 2, p.ldb, rows, 64, true))) return r;
  if (p.out_l && (r = omap2d(h, &p.o_l32, p.out_l, 2, p.ldb, rows, 32, false))) return r;
  if (p.out_h && p.epi == TEPI_LN_GELU && (r = omap2d(h, &p.o_h32, p.out_h, 2, p.ldb, rows, 32, false))) return r;
  if ((p.epi == TEPI_RESID || p.epi == TEPI_F32) && (r = omap2d(h, &p.o_f32, p.out_f32, 4, p.ldo, rows, 32, true))) return r;
  if (p.epi == TEPI_QKV) {
    if ((r = omap_qk(h, &p.o_q, p.q, st.Lp, (uint64_t)st.S * LG_HEADS))) return r;
    if ((r = omap_qk(h, &p.o_k, p.k, st.Lp, (uint64_t)st.S * LG_HEADS))) return r;
    if (p.rope && (r = omap2d(h, &p.cs_map, p.cs, 4, 64, rows, 32, true))) return r;
  }
  p.kb0 = d.k0 / BK;
  p.kb_total = K / BK;
  p.passes = x3 ? 3 : 1;
  p.st = st;
  if (p.w_select != 2) p.w_select = d.nsel > 1;
  p.dbg = h->tc.dbg;
  h->launches += 1;
  return launch_linear(p, (d.nout + BN - 1) / BN, stream);
}
}  // namespace

// ------------------------------------------------------------------------------------------------
// entry points used by lg_api.cu
// ------------------------------------------------------------------------------------------------

// ------------------------------------------------------------------------------------------------
// Assignment tail on the tensor cores (matches-only variant: the log-assignment matrix is never written)
// ------------------------------------------------------------------------------------------------
// launches: sweep 1 (LSE partials), z + term, sweep 2 (arg-max partials, optionally the matrix), [dustbin], tail
int tc_assign_sweeps(LgHandle* h, const TcBuffers& b, const SeqState& st, const AssignArgs& a, float* part, int* part_arg,
                     float* term, cudaStream_t stream) {
  float* logmat = a.log_assignment;
  const int M = a.M, N = a.N;
  const int ntc = (st.Lp + BN - 1) / BN;
  for (int sweep = 0; sweep < 2; ++sweep) {
    TcLinParams p{};
    p.epi = sweep == 0 ? TEPI_LSE : TEPI_ARGMAX;
    p.scale = 1.f; p.bias = h->wpk;  // unused
    p.part = part; p.part_arg = part_arg; p.part_stride = 2 * ntc; p.term = term;
    p.logmat = sweep == 1 ? logmat : nullptr; p.mat_m = M; p.mat_n = N;
    p.w_select = 2;
    // W = the partner sequence's rows of p: one [Lp, 256] matrix per sequence
    LinDesc ld{b.msgh, b.msgl, LG_DIM, nullptr, nullptr, 0, b.msgh, b.msgl, st.Lp, st.S, (size_t)st.Lp * LG_DIM};
    int r;
    {
      Timer tm(h, LG_K_ASSIGN_MATRIX, stream, sweep == 1 && logmat != nullptr);  // the matrix-writing sweep on its own
      if ((r = run_linear(h, st, ld, p, stream))) return r;
    }
    if (sweep == 0) {
      if ((r = misc_assign_term(a, st, part, 2 * ntc, BN / 2, term, stream))) return r;
      h->launches += 1;
    }
  }
  if (logmat) { if (int rd = misc_assign_dustbin(a, st, stream)) return rd; h->launches += 1; }
  int r = misc_assign_tail(a, st, part, part_arg, 2 * ntc, BN / 2, stream);
  h->launches += 1;
  return r;
}

unsigned int tc_debug_timeout_code(LgHandle* h, unsigned int* words32) {
  unsigned int v[32] = {0};
  if (!h->tc.dbg) return 0;
  if (cudaMemcpy(v, h->tc.dbg, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return 0xffffffffu;
  unsigned int first = 0;
  for (int i = 0; i < 32; ++i) {
    if (words32) words32[i] = v[i];
    if (v[i] && !first) first = (unsigned)i << 24 | (v[i] & 0x80ffffffu);
  }
  if (first) cudaMemset(h->tc.dbg, 0, sizeof(v));
  return first;
}

int tc_pack_weights(LgHandle* h, cudaStream_t stream) {
  TcWeights& w = h->tc;
  const size_t n = h->wpk_floats;
  cudaError_t e = cudaMalloc(&w.w_hi, n * sizeof(__nv_bfloat16));
  if (e != cudaSuccess) return lg_set_cuda_error(e, __FILE__, __LINE__);
  e = cudaMalloc(&w.w_lo, n * sizeof(__nv_bfloat16));
  if (e != cudaSuccess) return lg_set_cuda_error(e, __FILE__, __LINE__);
  split_weights_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(h->wpk, w.w_hi, w.w_lo, n);
  LG_CHECK_LAUNCH();
  w.map_cache = new MapCache();
  e = cudaMalloc(&w.dbg, 32 * sizeof(unsigned int));
  if (e != cudaSuccess) return lg_set_cuda_error(e, __FILE__, __LINE__);
  cudaMemsetAsync(w.dbg, 0, 32 * sizeof(unsigned int), stream);
  if (!get_encode()) return lg_set_error("cuTensorMapEncodeTiled unavailable (driver too old?)");
  return 0;
}

void tc_free_weights(TcWeights* w) {
  if (w->w_hi) cudaFree(w->w_hi);
  if (w->w_lo) cudaFree(w->w_lo);
  if (w->map_cache) delete static_cast<MapCache*>(w->map_cache);
  if (w->dbg) cudaFree(w->dbg);
  w->dbg = nullptr;
  w->w_hi = w->w_lo = nullptr;
  w->map_cache = nullptr;
}

void tc_carve(size_t* off, char* base, size_t S, int Lp, const LgHandle* h, TcBuffers* b) {
  const size_t R = S * Lp;
  const bool x3 = h->cfg.precision == LG_PREC_BF16X3;
  auto take = [&](size_t bytes) -> void* {
    *off = (*off + 1023) & ~(size_t)1023;
    void* p = base ? base + *off : nullptr;
    *off += bytes;
    return p;
  };
  b->xh = (__nv_bfloat16*)take(R * 256 * 2);
  b->xl = x3 ? (__nv_bfloat16*)take(R * 256 * 2) : nullptr;
  b->ctxh = (__nv_bfloat16*)take(R * 256 * 2);
  b->ctxl = x3 ? (__nv_bfloat16*)take(R * 256 * 2) : nullptr;
  b->msgh = (__nv_bfloat16*)take(R * 256 * 2);
  b->msgl = x3 ? (__nv_bfloat16*)take(R * 256 * 2) : nullptr;
  b->hh = (__nv_bfloat16*)take(R * 512 * 2);
  b->hl = x3 ? (__nv_bfloat16*)take(R * 512 * 2) : nullptr;
  b->q = (__half*)take(R * 256 * 2);
  b->k = (__half*)take(R * 256 * 2);
  b->vt = (__half*)take(R * 256 * 2);
}

int tc_refresh_shadow(LgHandle* h, const TcBuffers& b, const float* x, const SeqState& st, cudaStream_t stream) {
  shadow_kernel<<<st.S * st.Lp, 256, 0, stream>>>(x, b.xh, b.xl, LG_DIM, st);
  LG_CHECK_LAUNCH();
  return 0;
}

int tc_input_proj(LgHandle* h, const TcBuffers& b, const SeqState& st, const float* desc_packed, float* x, cudaStream_t stream) {
  const int d = h->cfg.input_dim;
  if (d % BK != 0) return lg_set_error("tensor-core input_proj needs input_dim % 64 == 0");
  shadow_kernel<<<st.S * st.Lp, 256, 0, stream>>>(desc_packed, b.hh, b.hl, d, st);
  LG_CHECK_LAUNCH();
  h->launches += 1;
  TcLinParams p{};
  p.epi = TEPI_F32; p.scale = 1.f; p.bias = h->wpk + h->o_inb;
  p.out_f32 = x; p.ldo = LG_DIM; p.out_h = b.xh; p.out_l = b.xl; p.ldb = LG_DIM;
  LinDesc ld{b.hh, b.hl, d, nullptr, nullptr, 0, h->tc.w_hi + h->o_inw, h->tc.w_lo + h->o_inw, LG_DIM, 1, 0};
  return run_linear(h, st, ld, p, stream);
}

int tc_final_proj(LgHandle* h, const TcBuffers& b, const SeqState& st, float* p_out, cudaStream_t stream) {
  TcLinParams p{};
  p.epi = TEPI_F32; p.scale = 0.25f;  // / 256^(1/4) (lightglue.py:291)
  p.bias = h->wpk + h->o_assign + AO_FB; p.bias_sel_stride = ASSIGN_BLOB_PAD;
  p.out_f32 = p_out; p.ldo = LG_DIM; p.out_h = b.msgh; p.out_l = b.msgl; p.ldb = LG_DIM;  // bf16 images feed the sweeps
  const size_t fw = h->o_assign + AO_FW;
  LinDesc ld{b.xh, b.xl, LG_DIM, nullptr, nullptr, 0, h->tc.w_hi + fw, h->tc.w_lo + fw, LG_DIM, h->cfg.n_layers, ASSIGN_BLOB_PAD};
  return run_linear(h, st, ld, p, stream);
}

int tc_conv(LgHandle* h, const SeqState& st, const __nv_bfloat16* in_h, const __nv_bfloat16* in_l, int cin, int taps, size_t w_off,
            const float* bias, int relu, int B, int H, int W, __nv_bfloat16* out_h, __nv_bfloat16* out_l, int cout, float* out_f32,
            int ldo, cudaStream_t stream) {
  const bool x3 = h->cfg.precision == LG_PREC_BF16X3;
  if (cin % BK != 0 || (taps != 1 && taps != 9)) return lg_set_error("tc_conv: Cin must be a multiple of 64, 1x1 or 3x3");
  TcLinParams p{};
  p.epi = out_f32 ? TEPI_F32 : TEPI_CONV;
  p.scale = 1.f; p.bias = bias; p.relu = relu;
  p.out_f32 = out_f32; p.ldo = ldo; p.out_h = out_h; p.out_l = x3 ? out_l : nullptr; p.ldb = cout;
  const int mma_n = cout <= 64 ? 64 : cout <= 128 ? 128 : BN;  // no MMA columns for the zero rows of a narrow layer
  p.mma_n = mma_n == BN ? 0 : mma_n;
  p.conv_cb = taps == 9 ? cin / BK : 0;
  p.conv_w2 = W + 2; p.conv_h = H; p.conv_w = W;
  p.conv_plane = (long)(H + 2) * (W + 2); p.conv_rows = (long)B * p.conv_plane;
  LinDesc ld{in_h, in_l, cin, nullptr, nullptr, 0, h->tc.w_hi + w_off, h->tc.w_lo + w_off, BN, 1, 0};
  return run_linear(h, st, ld, p, stream);
}

int tc_block(LgHandle* h, const TcBuffers& b, const SeqState& st, int layer, int blk, float* x, const float* cs,
             cudaStream_t stream) {
  const BlockOff& o = blk == 0 ? h->bself : h->bcross;
  const size_t base = h->o_layers + (size_t)layer * h->layer_stride + (blk == 0 ? 0 : h->bself.total);
  const float* bw = h->wpk + base;
  const __nv_bfloat16 *wh = h->tc.w_hi + base, *wl = h->tc.w_lo + base;
  // Tile order against the 126 MB L2: every kernel of the chain reads what its predecessor wrote, and only the part written
  // LAST is still resident.  QKV and ffn.0 walk their tile lists backwards, ffn.3 (and the attention grid) forwards: ffn.3
  // starts on the hidden tiles ffn.0 finished with, the next QKV on the x images ffn.3 finished with, attention on the
  // q / k / v of the sequences QKV wrote last, ffn.0 on the context of the sequences attention wrote last.
  {  // QKV (+RoPE) / [to_qk | to_v] projection
    Timer t(h, LG_K_LINEAR, stream);
    Timer t2(h, LG_K_QKV, stream);
    TcLinParams p{};
    p.epi = TEPI_QKV; p.rope = blk == 0; p.scale = 1.f; p.bias = bw + o.bp; p.reverse = 1;
    p.q = b.q; p.k = b.k; p.vt = b.vt; p.cs = cs;
    LinDesc ld{b.xh, b.xl, LG_DIM, nullptr, nullptr, 0, wh + o.wp, wl + o.wp, blk == 0 ? 3 * LG_DIM : 2 * LG_DIM, 1, 0};
    int r = run_linear(h, st, ld, p, stream);
    if (r) return r;
  }
  {
    Timer t(h, LG_K_ATTENTION, stream);
    int r = tc_attention(h, b, st, blk == 0 ? 0 : st.B, blk == 0 ? b.k : b.q, stream);
    if (r) return r;
  }
  Timer t(h, LG_K_LINEAR, stream);
  {  // ffn.0 on cat([x, msg]) + LayerNorm + GELU -> h; the output projection is folded into the weights (W1f, b1f:
     // lg_handle.h), so the GEMM reads cat([x, ctx]) and `msg` is never formed
    TcLinParams p{};
    p.epi = TEPI_LN_GELU; p.scale = 1.f; p.bias = bw + o.b1f; p.ln_g = bw + o.g; p.ln_b = bw + o.be;
    p.reverse = 1;
    p.out_h = b.hh; p.out_l = b.hl; p.ldb = LG_FFN;
    LinDesc ld{b.xh, b.xl, LG_DIM, b.ctxh, b.ctxl, LG_DIM, wh + o.w1f, wl + o.w1f, LG_FFN, 1, 0};
    Timer t2(h, LG_K_FFN0, stream);
    int r = run_linear(h, st, ld, p, stream);
    if (r) return r;
  }
  {  // ffn.3 + residual -> x (fp32 master + bf16 shadows)
    TcLinParams p{};
    p.epi = TEPI_RESID; p.scale = 1.f; p.bias = bw + o.b2; p.out_f32 = x; p.ldo = LG_DIM;
    p.out_h = b.xh; p.out_l = b.xl; p.ldb = LG_DIM;
    LinDesc ld{b.hh, b.hl, LG_FFN, nullptr, nullptr, 0, wh + o.w2, wl + o.w2, LG_DIM, 1, 0};
    Timer t2(h, LG_K_FFN3, stream);
    int r = run_linear(h, st, ld, p, stream);
    if (r) return r;
  }
  return 0;
}
