// K2: staged, warp-specialised EdgeConv kernel (bf16 operands, fp32 accumulation in TMEM).
//
// Replaces StaticGraph_module.forward of checkerpose/model/pipeline.py:45-59 (get_graph_feature :27-40 +
// Conv2d 1x1 + BatchNorm2d + LeakyReLU + max over K) in the factored form of cp_fold_edgeconv, fused with
// the GEMM of the layer that consumes the aggregated feature.  One persistent CTA of 32 warps (8 warpgroups) per SM;
// the unit of work ("round") is one 64-channel slice of one tile of 128 plan-order nodes:
//
//   warps 0-15  aggregators.  A quarter-warp owns one node PAIR of the plan: it takes the max over the staged rows the
//               two nodes share once, then over the rest of each (40 - C row reads of 128 bits per lane instead of 40),
//               adds the nodes' own Q slices, applies LeakyReLU and writes the bf16 A operand slice straight into the
//               SWIZZLE_128B layout tcgen05.mma reads.  The plan's overlap-sorted pair groups rotate over the warps
//               from slice to slice, so every warp reads about the same number of rows per tile;
//   warps 16-23 epilogue (two warps per TMEM lane quarter, every second 32-column block each): TMEM -> registers ->
//               bias / LeakyReLU -> bf16 -> a swizzled shared-memory tile -> global with TMA tensor stores (or fp32
//               logits with plain stores); waits for / releases the accumulator per 128-column block;
//   warp 24     weight producer: streams the packed weight tiles (16 KB) with cp.async.bulk (TMA engine);
//   warp 25     MMA issuer: tcgen05.mma (M=128, N<=128, K=16) slice by slice as A slices complete; warp-uniform loop,
//               the instructions are issued under elect.sync (see mma_issuer: this warp is the critical path);
//   warps 26-27 idle (they complete the control warpgroup);
//   warps 28-31 stagers: copy every round's DISTINCT neighbour row slices (plan.ulist, ~245 rows x 128 B instead of
//               128 x K gathered rows) from the [P|Q] table into a shared-memory ring with cp.async (LDGSTS) and
//               signal the round with cp.async.mbarrier.arrive.noinc (asynchronous: they never wait for their own
//               copies and run ahead as far as the ring has room).  Ring positions are a pure function of the plan's
//               list lengths: stagers and aggregators recompute them and never exchange positions.
// The register file is re-divided with setmaxnreg (REGS_* below; the kernel is launched at 64 registers per thread).
//
// The aggregation of tile i+1 overlaps the MMAs and the epilogue of tile i; every hand-off is an mbarrier.
// What bounds the kernel: DESIGN.md section 5.
//
// A CTA-pair variant (cta_group::2, two tiles sharing every MMA) was measured no faster and removed: DESIGN.md section 8.
#include <cuda.h>
#include <string.h>

#include "common.cuh"
#include "sm100.cuh"

using bf16 = __nv_bfloat16;
using namespace sm100;

namespace {

constexpr int TILE_M = CP_PLAN_TILE;
constexpr int NUM_AGG_WARPS = 16;            // 64 quarter-warps = the 64 node pairs of a tile
constexpr int NUM_QW = NUM_AGG_WARPS * 4;
constexpr int EPI_WARP0 = NUM_AGG_WARPS;                 // TMEM lane quarter = warp % 4; NUM_EPI_WARPS / 4 warps share a quarter's columns
constexpr int NUM_EPI_WARPS = 8;
// The SM's warp scheduler favours higher warp ids, and a warp that spins on an mbarrier still competes for issue
// slots, so the single-thread roles everything else waits on get the highest warp ids.
constexpr int W_WARP = EPI_WARP0 + NUM_EPI_WARPS;                   // weight producer (+ TMEM alloc/dealloc)
constexpr int MMA_WARP = W_WARP + 1;
constexpr int STG_WARP0 = MMA_WARP + 3;         // two idle warps complete the control warpgroup; then the stagers
constexpr int NUM_STG_WARPS = 4;
constexpr int STG_THREADS = NUM_STG_WARPS * 32;
constexpr int NUM_WARPS = STG_WARP0 + NUM_STG_WARPS;
// measured (ms per launch, 256->512 / 256->256 + a_out): 72/64/56/40 0.623 / 0.600; 80/56/56/24 0.655 / 0.601;
// 80/56/48/32 0.632 / 0.601; 80/48/56/40 0.668 / 0.607; 80/56/40/40 0.663 / 0.688 (the stagers need 56, the MMA warp
// spills below 40, the epilogue slows below 64)
constexpr int REGS_AGG = 72, REGS_EPI = 64, REGS_CTRL = 40, REGS_STG = 56;   // the kernel is launched at 64
static_assert(NUM_WARPS == 32 && NUM_AGG_WARPS * REGS_AGG + NUM_EPI_WARPS * REGS_EPI + 4 * REGS_CTRL + NUM_STG_WARPS * REGS_STG <= NUM_WARPS * 64,
              "register budget");
constexpr int NTHREADS = NUM_WARPS * 32;
constexpr int A_BUF_BYTES = TILE_M * 128;    // one K slice of the A operand: 128 rows x 64 bf16
constexpr int A_BUFS = 3;
constexpr int B_STAGE_BYTES = 128 * 128;     // one K slice of a packed 128-row weight tile (the N of one tcgen05.mma)
constexpr int B_STAGES = 3;
constexpr int NBAR = 4;                      // staging rounds that may be unreleased at any time
constexpr int UI = CP_PLAN_UMAX / NUM_QW;    // list entries per quarter-warp
constexpr int TBUF_BYTES = 32 * 64;          // per epilogue warp: a tile of 32 rows x 32 bf16 (SWIZZLE_64B) for the TMA stores
constexpr int BIAS_BYTES = 512 * 4;
constexpr int TMEM_COLS = 512;
constexpr int MAX_WTILES = 16;
constexpr int SMEM_BYTES = 227 * 1024;
static_assert(UI == 8 && NUM_QW == CP_PLAN_LIST_LANES, "the issue path loads a quarter-warp's 8 uint16 list entries as one uint4");

constexpr int OFF_A = 0;
constexpr int OFF_B = OFF_A + A_BUFS * A_BUF_BYTES;
constexpr int OFF_TBUF = OFF_B + B_STAGES * B_STAGE_BYTES;
constexpr int OFF_BIAS = OFF_TBUF + NUM_EPI_WARPS * TBUF_BYTES;
constexpr int OFF_BAR = OFF_BIAS + BIAS_BYTES;
constexpr int OFF_WQ = OFF_BAR + 256;                          // per stager warp: virtual ring position of the last NBAR rounds
constexpr int OFF_PROG = OFF_WQ + NUM_STG_WARPS * 16 + 64;
__host__ __device__ constexpr int prog_width(int KCH) { return 8 * KCH + 8; }      // uint16 per pair entry (= 2 KP + 8)
__host__ __device__ constexpr int prog_bytes(int KCH) { return CP_PLAN_PAIRS * prog_width(KCH) * 2; }
__host__ __device__ constexpr int off_ring(int KCH) { return (OFF_PROG + 2 * prog_bytes(KCH) + 127) & ~127; }
__host__ __device__ constexpr int ring_rows(int KCH) { return (SMEM_BYTES - 1024 - off_ring(KCH)) / 128; }

struct EcParams {
  cp_edgeconv_params p;
  int KC;            // 64-channel slices of the aggregated feature (= GEMM K chunks) = rounds per tile
  int NB;            // 128-column blocks of the GEMM output
  int npad;          // nout rounded up to 16
  int num_tiles;     // B * ceil(N / 128)
  int tiles_per_roi;
  int tpr_shift;     // log2(tiles_per_roi) when it is a power of two (every shipped N), else -1
  int tma_out;       // bf16 output with nout % 32 == 0: the epilogue stores through the tensor map
  cp::WTile wt[MAX_WTILES];  // order: slice-major, then column block
};

// Tiles of this CTA: blockIdx.x, then every gridDim.x-th tile.
struct TileIt {
  int first, step, count, last;
  __device__ __forceinline__ explicit TileIt(const EcParams& kp) {
    last = kp.num_tiles - 1;
    first = (int)blockIdx.x;
    step = (int)gridDim.x;
    count = first < kp.num_tiles ? (kp.num_tiles - first + step - 1) / step : 0;
  }
  __device__ __forceinline__ int tile(int i) const {
    const int t = first + i * step;
    return t < last ? t : last;
  }
};

struct Bars {
  uint64_t stg_full[NBAR], stg_empty[NBAR];
  uint64_t a_full[A_BUFS], a_empty[A_BUFS];
  uint64_t b_full[B_STAGES], b_empty[B_STAGES];
  uint64_t acc_full[4], acc_empty[4];   // per 128-column block of the accumulator: the next tile's MMAs follow the epilogue block by block
  uint32_t tmem_slot;
  uint32_t bias_blocks;   // bit i: columns [32 i, 32 i + 32) have a non-zero bias (the P half of a [P|Q] layer has none)
};
static_assert(sizeof(Bars) <= 256, "barrier block");

__device__ __forceinline__ uint32_t bf2_max3(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(r), "r"(c));   // ptxas fuses the pair into one 3-input VHMNMX
  return r;
}
__device__ __forceinline__ uint4 bf8_max3(uint4 a, uint4 b, uint4 c) {
  return make_uint4(bf2_max3(a.x, b.x, c.x), bf2_max3(a.y, b.y, c.y), bf2_max3(a.z, b.z, c.z), bf2_max3(a.w, b.w, c.w));
}
__device__ __forceinline__ uint2 lds64(uint32_t addr) {
  uint2 r;
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(addr));
  return r;
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
  uint32_t r;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(addr));
  return r;
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ uint32_t a_offset(int buf, int row, int chunk) {
  return (uint32_t)(OFF_A + buf * A_BUF_BYTES + row * 128 + ((chunk ^ (row & 7)) << 4));
}
__device__ __forceinline__ int tile_roi(const EcParams& kp, int tile) {
  return kp.tpr_shift >= 0 ? (tile >> kp.tpr_shift) : tile / kp.tiles_per_roi;
}
__device__ __forceinline__ void tile_coords(const EcParams& kp, int tile, int& b, int& t, int& g) {
  b = tile_roi(kp, tile);
  t = tile - b * kp.tiles_per_roi;
  g = kp.p.graph_sel ? __ldg(kp.p.graph_sel + b) : 0;
}

// ------------------------------------------------------------------------------------------------------
// weight producer / MMA issuer
// ------------------------------------------------------------------------------------------------------
__device__ void weight_producer(const EcParams& kp, uint8_t* sm, Bars* bars) {
  const int NB = kp.NB;
  const TileIt tiles(kp);
  uint32_t cnt = 0;
  for (int ti = 0; ti < tiles.count; ++ti) {
    for (int c = 0; c < kp.KC; ++c)
      for (int nb = 0; nb < NB; ++nb, ++cnt) {
        const int s = cnt % B_STAGES;
        const uint32_t use = cnt / B_STAGES;
        if (use > 0) mbar_wait(&bars->b_empty[s], (use - 1) & 1);
        const cp::WTile& w = kp.wt[c * NB + nb];
        if (elect_one()) {
          mbar_arrive_expect_tx(&bars->b_full[s], w.bytes);
          bulk_g2s(sm + OFF_B + s * B_STAGE_BYTES, w.ptr, w.bytes, &bars->b_full[s]);
        }
        __syncwarp();
      }
  }
}

// The MMA warp is the kernel's critical path (DESIGN.md section 5): every instruction between two tcgen05.mma costs
// tile time, so the loop keeps running ring positions / parities / descriptor words in registers (no modulo, no
// constant-bank table look-ups, no 64-bit descriptor rebuild per MMA) and issues under elect.sync.
__device__ void mma_issuer(const EcParams& kp, uint8_t* sm, Bars* bars, uint32_t tmem_base) {
  const uint32_t a_lo0 = smem_desc_lo(smem_u32(sm + OFF_A)), b_lo0 = smem_desc_lo(smem_u32(sm + OFF_B));
  const uint32_t a_full0 = smem_u32(&bars->a_full[0]), a_empty0 = smem_u32(&bars->a_empty[0]);
  const uint32_t b_full0 = smem_u32(&bars->b_full[0]), b_empty0 = smem_u32(&bars->b_empty[0]);
  const uint32_t acc_full0 = smem_u32(&bars->acc_full[0]), acc_empty0 = smem_u32(&bars->acc_empty[0]);
  const int KC = kp.KC, NB = kp.NB;
  const uint32_t idesc_full = make_idesc_bf16_m128(128);
  const uint32_t idesc_last = make_idesc_bf16_m128((uint32_t)(kp.npad - (NB - 1) * 128));
  uint32_t ab = 0, a_par = 0;     // A slice ring position and the parity to wait for
  uint32_t bs = 0, b_par = 0;     // weight stage ring position and parity
  uint32_t acc_par = 0;           // parity of acc_empty to wait for (flips per tile; nothing to wait for on the first)
  bool first_tile = true;
  auto wait_s = [](uint32_t bar_s, uint32_t parity) {   // mbarrier wait on a shared-space address
    uint32_t ok, spins = 0;
    do {
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(ok) : "r"(bar_s), "r"(parity) : "memory");
      if (!ok && ++spins > (1u << 27)) __trap();   // a broken pipeline traps instead of hanging the GPU box
    } while (!ok);
  };
  auto commit_s = [](uint32_t bar_s) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_s) : "memory");
  };
  const TileIt tiles(kp);
  for (int ti = 0; ti < tiles.count; ++ti) {
    for (int c = 0; c < KC; ++c) {
      wait_s(a_full0 + ab * 8, a_par);
      const uint32_t a_lo = a_lo0 + ab * (A_BUF_BYTES >> 4);
      const bool last_slice = c == KC - 1;
      for (int nb = 0; nb < NB; ++nb) {
        wait_s(b_full0 + bs * 8, b_par);
        if (c == 0 && !first_tile) wait_s(acc_empty0 + nb * 8, acc_par);   // the previous tile's columns are drained
        tc_fence_after_sync();
        const uint32_t b_lo = b_lo0 + bs * (B_STAGE_BYTES >> 4);
        const uint32_t idesc = nb == NB - 1 ? idesc_last : idesc_full;
        const uint32_t d = tmem_base + (uint32_t)(nb * 128);
        if (elect_one()) {
          mma_bf16_ss_lo(d, a_lo, b_lo, idesc, (uint32_t)(c != 0));
          mma_bf16_ss_lo(d, a_lo + 2, b_lo + 2, idesc, 1u);
          mma_bf16_ss_lo(d, a_lo + 4, b_lo + 4, idesc, 1u);
          mma_bf16_ss_lo(d, a_lo + 6, b_lo + 6, idesc, 1u);
          commit_s(b_empty0 + bs * 8);
          if (last_slice) commit_s(acc_full0 + nb * 8);
          if (nb == NB - 1) commit_s(a_empty0 + ab * 8);
        }
        __syncwarp();
        if (++bs == B_STAGES) { bs = 0; b_par ^= 1; }
      }
      if (++ab == A_BUFS) { ab = 0; a_par ^= 1; }
    }
    if (!first_tile) acc_par ^= 1;
    first_tile = false;
  }
}

// Ring position of the next round (U rows, contiguous): a pure function of the list lengths of the tiles this CTA
// processes, so the stagers and every aggregator warp compute it on their own and never exchange positions.
__device__ __forceinline__ uint32_t ring_place(uint32_t& ph, uint32_t U, uint32_t R) {
  if (ph + U > R) ph = 0;
  const uint32_t at = ph;
  ph += U;
  return at;
}

// ------------------------------------------------------------------------------------------------------
// stagers: one warpgroup copies every round's distinct neighbour row slices into the ring
// ------------------------------------------------------------------------------------------------------
template <int KCH>
__device__ void stager(const EcParams& kp, uint8_t* sm, Bars* bars, int pw, int lane) {
  constexpr int PROG_BYTES = prog_bytes(KCH), OFF_RING = off_ring(KCH);
  constexpr uint32_t R = ring_rows(KCH);
  const cp_edgeconv_params& p = kp.p;
  const cp_graph_plan& pl = p.plan;
  const int q = pw * 4 + (lane >> 3), sub = lane & 7;   // copying quarter-warp 0..15: ring rows q, q + 16, ... of a round
  const int tid = pw * 32 + lane;
  const uint32_t sm_base = smem_u32(sm);
  const uint32_t vs = sm_base + OFF_WQ + pw * 16;        // per-warp copy of vstart[NBAR] (same-value stores by all lanes)
  const uint32_t row_bytes = (uint32_t)p.ld_z * 2;
  const uint32_t KC = (uint32_t)kp.KC;
  const TileIt tiles(kp);
  const int my_tiles = tiles.count;
  uint32_t vh = 0, ph = 0;      // ring head: virtual (monotonic) and physical row
  uint32_t rel = 0;             // rounds < rel are known to be released by all aggregator warps
  uint32_t r = 0;               // round being copied
  for (int ti = 0; ti < my_tiles; ++ti) {
    int b, t, g;
    tile_coords(kp, tiles.tile(ti), b, t, g);
    const size_t gt = (size_t)g * pl.T + t;
    const uint32_t U = (uint32_t)__ldg(pl.ucount + gt);
    // ring row j of a round holds list entry (lane j % 64, slot j / 64): this thread copies rows j = q, q + 16, ...
    // (the 1 KB list stays in L1 over the tile's rounds)
    const uint16_t* lst = pl.ulist + gt * NUM_QW * UI;
    if (ti + 1 < my_tiles) {   // next tile's list -> L2
      int b2, t2, g2;
      tile_coords(kp, tiles.tile(ti + 1), b2, t2, g2);
      const size_t gt2 = (size_t)g2 * pl.T + t2;
      if (tid < 8) prefetch_l2(pl.ulist + gt2 * NUM_QW * UI + tid * 64);
      if (tid == 8) prefetch_l2(pl.ucount + gt2);
    }
    {  // the tile's own Q halves -> L2 (128 rows x Co bf16 = 2 Co lines of 128 B); the aggregators read them 2-3 rounds later
      const uint8_t* qn = reinterpret_cast<const uint8_t*>(p.z) + ((size_t)b * p.N + (size_t)t * TILE_M) * row_bytes + p.Co * 2;
      const int lines_per_row = p.Co >> 6;
      const int rows_t = min(TILE_M, p.N - t * TILE_M);
      for (int l = tid; l < rows_t * lines_per_row; l += STG_THREADS)
        prefetch_l2(qn + (size_t)(l / lines_per_row) * row_bytes + (l % lines_per_row) * 128);
    }
    const uint8_t* zb = reinterpret_cast<const uint8_t*>(p.z) + (size_t)b * p.N * row_bytes + sub * 16;
    for (uint32_t c = 0; c < KC; ++c, ++r) {
      uint32_t nvh = vh, nph = ph;
      if (nph + U > R) {   // a round is contiguous in the ring: skip the tail
        nvh += R - nph;
        nph = 0;
      }
      // rounds that must have been released by ALL aggregator warps before this one is copied: whatever still occupies
      // the ring rows, the round whose barrier pair is reused, and (first round of a tile) the last round of the tile
      // whose program buffer is overwritten
      int need_rel = (int)r - NBAR;
      if (c == 0) need_rel = max(need_rel, (int)r - (int)KC - 1);
      while (rel < r) {
        const uint32_t oldest_v = lds32(vs + (rel % NBAR) * 4);
        if (nvh + U - oldest_v <= R && (int)rel > need_rel) break;
        mbar_wait(&bars->stg_empty[rel % NBAR], (rel / NBAR) & 1);
        ++rel;
      }
      sts32(vs + (r % NBAR) * 4, nvh);
      __syncwarp();      // every lane stores the same value and reads it back later: order the lanes explicitly (racecheck)
      vh = nvh + U;
      ph = nph + U;
      const uint32_t dst = sm_base + OFF_RING + (nph + q) * 128u + sub * 16;
      const uint8_t* src = zb + c * 128;
#pragma unroll 4
      for (uint32_t j = (uint32_t)q; j < U; j += 16) {
        const uint32_t row = __ldg(lst + (j & (NUM_QW - 1)) * UI + (j >> 6));
        cp_async16(dst + (j - (uint32_t)q) * 128u, src + (size_t)row * row_bytes);
      }
      if (c == 0) {  // the tile's pair programs ride along with its first round
        const uint32_t pd = sm_base + OFF_PROG + (ti & 1) * PROG_BYTES;
        const uint8_t* prog_src = reinterpret_cast<const uint8_t*>(pl.prog) + gt * PROG_BYTES;
        for (int piece = tid; piece < PROG_BYTES / 16; piece += STG_THREADS) cp_async16(pd + piece * 16, prog_src + piece * 16);
      }
      // asynchronous arrival: fires when all of this thread's copies so far have landed; nobody waits here
      cp_async_arrive_noinc(&bars->stg_full[r % NBAR]);
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// aggregators
// ------------------------------------------------------------------------------------------------------
// max over the four staged row slices whose byte offsets are packed in w0, w1 (two uint16 each)
__device__ __forceinline__ uint4 max_quad(uint4 m, uint32_t stg, uint32_t w0, uint32_t w1) {
  const uint4 v0 = lds128(stg + (w0 & 0xffffu)), v1 = lds128(stg + (w0 >> 16));
  const uint4 v2 = lds128(stg + (w1 & 0xffffu)), v3 = lds128(stg + (w1 >> 16));
  return bf8_max3(bf8_max3(m, v0, v1), v2, v3);
}

__device__ __forceinline__ uint4 finish_node(uint4 m, uint4 q, float slope, bool fast_lrelu) {
  const uint32_t mw[4] = {m.x, m.y, m.z, m.w}, qv[4] = {q.x, q.y, q.z, q.w};
  uint32_t ow[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 a = bf2_to_f2(mw[e]), d = bf2_to_f2(qv[e]);
    const float x = a.x + d.x, y = a.y + d.y;
    ow[e] = fast_lrelu ? f2_to_bf2(fmaxf(x, x * slope), fmaxf(y, y * slope)) : f2_to_bf2(cp::lrelu(x, slope), cp::lrelu(y, slope));
  }
  return make_uint4(ow[0], ow[1], ow[2], ow[3]);
}

template <int KCH>
__device__ void aggregator(const EcParams& kp, uint8_t* sm, Bars* bars, int aw, int lane) {
  constexpr int KP = 4 * KCH, PW = prog_width(KCH), PROG_BYTES = prog_bytes(KCH), OFF_RING = off_ring(KCH);
  constexpr uint32_t R = ring_rows(KCH);
  constexpr uint32_t NEG_INF2 = 0xFF80FF80u;  // bf16x2 (-inf, -inf)
  const cp_edgeconv_params& p = kp.p;
  const cp_graph_plan& pl = p.plan;
  const int grp = lane >> 3, sub = lane & 7;
  const uint32_t sm_base = smem_u32(sm);
  const float slope = p.agg_slope;
  const bool fast_lrelu = slope >= 0.f && slope <= 1.f;   // then lrelu(x) == max(x, slope * x)
  const uint32_t KC = (uint32_t)kp.KC;
  uint32_t it = 0;      // round being reduced
  uint32_t ph = 0;      // ring head (replica of the stagers')
  auto tile_U = [&](int tile) -> uint32_t {
    int b, t, g;
    tile_coords(kp, tile, b, t, g);
    return (uint32_t)__ldg(pl.ucount + (size_t)g * pl.T + t);
  };
  const TileIt tiles(kp);
  uint32_t U_next = tiles.count > 0 ? tile_U(tiles.tile(0)) : 0u;
  for (uint32_t ti = 0; ti < (uint32_t)tiles.count; ++ti) {
    const int tile = tiles.tile((int)ti);
    const int b = tile_roi(kp, tile), t = tile - b * kp.tiles_per_roi;
    const int n0 = t * TILE_M;
    const uint32_t row0 = (uint32_t)(b * p.N + n0);   // B * N < 2^31 (checked by the host)
    const uint32_t prog_s = sm_base + OFF_PROG + (ti & 1) * PROG_BYTES;
    const uint32_t U = U_next;
    if ((int)ti + 1 < tiles.count) U_next = tile_U(tiles.tile((int)ti + 1));
    for (uint32_t c = 0; c < KC; ++c, ++it) {
      const uint32_t stg = sm_base + OFF_RING + ring_place(ph, U, R) * 128u + sub * 16;
      mbar_wait(&bars->stg_full[it % NBAR], (it / NBAR) & 1);

      // ---- this quarter-warp's pair; the overlap-sorted pair groups rotate over the warps from slice to slice so that
      //      every warp sees the same mix of cheap (large C) and expensive pairs over a tile ----
      const uint32_t pair = (((uint32_t)aw + 4 * c) & (NUM_AGG_WARPS - 1)) * 4 + grp;
      const uint32_t pe = prog_s + pair * (PW * 2);
      const uint32_t info = lds32(pe + 2 * KP * 2);
      const int na = info & 255, nb = (info >> 8) & 255;
      const uint32_t nc4 = info >> 18;              // chunks (of 4 rows) the pair shares        } warp-uniform
      const uint32_t nr4 = (uint32_t)KCH - nc4;     // chunks of each node's own rows            }
      // own Q slices: issued first, their (L2) latency hides behind the row reads
      const bf16* zq = reinterpret_cast<const bf16*>(p.z) + p.Co + c * 64 + sub * 8;
      const uint4 qa = na != 255 ? ldg_nc_na_v4(zq + (size_t)(row0 + na) * p.ld_z) : make_uint4(0, 0, 0, 0);
      const uint4 qb = nb != 255 ? ldg_nc_na_v4(zq + (size_t)(row0 + nb) * p.ld_z) : make_uint4(0, 0, 0, 0);

      uint4 acc = make_uint4(NEG_INF2, NEG_INF2, NEG_INF2, NEG_INF2);
      uint32_t pa = pe;
      for (uint32_t j = 0; j < nc4; ++j, pa += 8) {       // rows both nodes need
        const uint2 o = lds64(pa);
        acc = max_quad(acc, stg, o.x, o.y);
      }
      uint4 accb = acc;
      uint32_t pb = pe + KP * 2;
      for (uint32_t j = 0; j < nr4; ++j, pa += 8, pb += 8) {   // the rest of each
        const uint2 oa = lds64(pa), ob = lds64(pb);
        acc = max_quad(acc, stg, oa.x, oa.y);
        accb = max_quad(accb, stg, ob.x, ob.y);
      }

      const uint32_t ab = it % A_BUFS;
      if (it >= A_BUFS) mbar_wait(&bars->a_empty[ab], ((it / A_BUFS) - 1) & 1);   // MMAs that read this buffer are done
      if (na != 255) {
        const uint4 o = finish_node(acc, qa, slope, fast_lrelu);
        sts128(sm_base + a_offset(ab, na, sub), o);
        if (p.a_out) *reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(p.a_out) + (size_t)(row0 + na) * p.ld_a_out + c * 64 + sub * 8) = o;
      }
      if (nb != 255) {
        const uint4 o = finish_node(accb, qb, slope, fast_lrelu);
        sts128(sm_base + a_offset(ab, nb, sub), o);
        if (p.a_out) *reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(p.a_out) + (size_t)(row0 + nb) * p.ld_a_out + c * 64 + sub * 8) = o;
      }
      fence_proxy_async_smem();  // generic-proxy writes of A -> visible to the tensor core's async proxy
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&bars->a_full[ab]);
        mbar_arrive(&bars->stg_empty[it % NBAR]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// epilogue: warp q drains TMEM lanes [32 q, 32 q + 32), 32 columns at a time
// ------------------------------------------------------------------------------------------------------
template <bool ACT, bool TMA_OUT>
__device__ void epilogue_warps(const EcParams& kp, const CUtensorMap* out_map, uint8_t* sm, Bars* bars, uint32_t tmem_base, int ew, int lane) {
  constexpr int ACC_BLK = 128;      // columns per accumulator block (= per MMA)
  constexpr int ACC_SH = 7;
  const TileIt tiles(kp);
  const cp_edgeconv_params& p = kp.p;
  const cp_chain_layer& L = p.layer;
  const int q = ew & 3, h = ew >> 2;
  const int row = q * 32 + lane;
  const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16);
  const uint32_t sm_base = smem_u32(sm);
  const uint32_t tbuf = sm_base + OFF_TBUF + ew * TBUF_BYTES;
  const uint32_t bias_s = sm_base + OFF_BIAS;
  const float slope = L.slope;
  const uint32_t bias_blocks = bars->bias_blocks;
  const int sw = (lane >> 1) & 3;   // SWIZZLE_64B: 16-byte chunk index ^= bits 1-2 of the row
  for (int ti = 0; ti < tiles.count; ++ti) {
    const int tile = tiles.tile(ti);
    const int b = tile_roi(kp, tile), t = tile - b * kp.tiles_per_roi;
    const int n0 = t * TILE_M;
    const int rows_valid = min(TILE_M, p.N - n0);
    const bool row_ok = row < rows_valid;
    const size_t grow0 = (size_t)b * p.N + n0;
    for (int c0 = h * 32; c0 < kp.NB * ACC_BLK; c0 += 32 * (NUM_EPI_WARPS / 4)) {
      if ((c0 & (ACC_BLK - 1)) == h * 32) {   // this warp's first block of an accumulator block
        mbar_wait(&bars->acc_full[c0 >> ACC_SH], ti & 1);
        tc_fence_after_sync();
      }
      const bool last_of_block = (c0 & (ACC_BLK - 1)) == h * 32 + ACC_BLK - 32 * (NUM_EPI_WARPS / 4);
      if (c0 >= kp.npad) {          // nothing to drain in a ragged block's tail; still release the block
        if (last_of_block) {
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bars->acc_empty[c0 >> ACC_SH]);
        }
        continue;
      }
      uint32_t r[32];
      const int ncols = min(32, kp.npad - c0);   // 16 or 32 (npad is a multiple of 16)
      if (TMA_OUT || ncols == 32) {
        tmem_ld32(tbase + (uint32_t)c0, r);
      } else {
        uint32_t hh[16];
        tmem_ld16(tbase + (uint32_t)c0, hh);
#pragma unroll
        for (int e = 0; e < 16; ++e) { r[e] = hh[e]; r[16 + e] = 0; }
      }
      tmem_ld_wait();
      float v[32];
#pragma unroll
      for (int e = 0; e < 32; ++e) v[e] = __uint_as_float(r[e]);
      if ((bias_blocks >> (c0 >> 5)) & 1) {
#pragma unroll
        for (int e4 = 0; e4 < 8; ++e4) {
          const uint4 bb = lds128(bias_s + (uint32_t)(c0 + e4 * 4) * 4);
          v[e4 * 4 + 0] += __uint_as_float(bb.x);
          v[e4 * 4 + 1] += __uint_as_float(bb.y);
          v[e4 * 4 + 2] += __uint_as_float(bb.z);
          v[e4 * 4 + 3] += __uint_as_float(bb.w);
        }
      }
      if (ACT) {
#pragma unroll
        for (int e = 0; e < 32; ++e) v[e] = cp::lrelu(v[e], slope);
      }
      if (TMA_OUT) {
        // 32 rows x 64 B tile in the SWIZZLE_64B layout of the tensor map; the TMA engine writes it to
        // out[b, n0 + 32 q .. +32, c0 .. c0+32) and clips rows beyond N
        if (lane == 0) bulk_wait_read<0>();   // the warp's previous store is done reading the tile
        __syncwarp();
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const uint4 w = make_uint4(f2_to_bf2(v[e * 8], v[e * 8 + 1]), f2_to_bf2(v[e * 8 + 2], v[e * 8 + 3]),
                                     f2_to_bf2(v[e * 8 + 4], v[e * 8 + 5]), f2_to_bf2(v[e * 8 + 6], v[e * 8 + 7]));
          sts128(tbuf + lane * 64 + ((e ^ sw) << 4), w);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && q * 32 < rows_valid) {
          tma_store_3d(out_map, tbuf, c0, n0 + q * 32, b);
          bulk_commit();
        }
      } else if (row_ok) {
        if (p.out_mode == CP_OUT_BF16) {
          bf16* o = reinterpret_cast<bf16*>(p.out) + (grow0 + row) * p.ld_out + c0;
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (e * 8 < ncols)
              *reinterpret_cast<uint4*>(o + e * 8) = make_uint4(f2_to_bf2(v[e * 8], v[e * 8 + 1]), f2_to_bf2(v[e * 8 + 2], v[e * 8 + 3]),
                                                                f2_to_bf2(v[e * 8 + 4], v[e * 8 + 5]), f2_to_bf2(v[e * 8 + 6], v[e * 8 + 7]));
        } else {
          float* o = reinterpret_cast<float*>(p.out) + (grow0 + row) * p.ld_out;
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (c0 + e < p.n_valid) o[c0 + e] = v[e];
        }
      }
      if (last_of_block) {   // this warp is done with the accumulator block: the next tile's MMAs may overwrite it
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->acc_empty[c0 >> ACC_SH]);
      }
    }
  }
  if (TMA_OUT && lane == 0) bulk_wait_read<0>();   // shared memory must outlive the last stores' reads
}

template <int KCH>
__global__ void __launch_bounds__(NTHREADS, 1) edgeconv_kernel(const __grid_constant__ EcParams kp, const __grid_constant__ CUtensorMap out_map) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  Bars* bars = reinterpret_cast<Bars*>(sm + OFF_BAR);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NBAR; ++s) {
      mbar_init(&bars->stg_full[s], STG_THREADS);     // every stager thread, asynchronously, once its copies of the round landed
      mbar_init(&bars->stg_empty[s], NUM_AGG_WARPS);
    }
    for (int c = 0; c < A_BUFS; ++c) {
      mbar_init(&bars->a_full[c], NUM_AGG_WARPS);
      mbar_init(&bars->a_empty[c], 1);
    }
    for (int s = 0; s < B_STAGES; ++s) {
      mbar_init(&bars->b_full[s], 1);
      mbar_init(&bars->b_empty[s], 1);
    }
    for (int nb = 0; nb < 4; ++nb) {
      mbar_init(&bars->acc_full[nb], 1);
      mbar_init(&bars->acc_empty[nb], NUM_EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == W_WARP) tmem_alloc(&bars->tmem_slot, TMEM_COLS);
  for (int i = threadIdx.x; i < BIAS_BYTES / 4; i += NTHREADS)   // bias row (zero-padded) for the epilogue's broadcast loads
    reinterpret_cast<float*>(sm + OFF_BIAS)[i] = (kp.p.layer.bias && i < kp.p.layer.nout) ? kp.p.layer.bias[i] : 0.f;
  if (warp == 0) {
    bool nz = false;
    if (kp.p.layer.bias && lane < 16)
      for (int e = lane * 32; e < min(lane * 32 + 32, kp.p.layer.nout); ++e) nz |= kp.p.layer.bias[e] != 0.f;
    const uint32_t m = __ballot_sync(0xffffffffu, nz);
    if (lane == 0) bars->bias_blocks = m;
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = bars->tmem_slot;

  if (warp >= STG_WARP0) {
    if (REGS_STG < 64) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_STG));
    stager<KCH>(kp, sm, bars, warp - STG_WARP0, lane);
  } else if (warp >= W_WARP) {   // control warpgroup
    if (REGS_CTRL < 64) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_CTRL));
    if (warp == MMA_WARP) mma_issuer(kp, sm, bars, tmem_base);
    else if (warp == W_WARP) weight_producer(kp, sm, bars);
    __syncwarp();
  } else if (warp >= EPI_WARP0) {
    if (REGS_EPI < 64) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_EPI));
    const int q = warp - EPI_WARP0;
    const bool tma_out = kp.tma_out != 0;
    if (kp.p.layer.act) {
      if (tma_out) epilogue_warps<true, true>(kp, &out_map, sm, bars, tmem_base, q, lane);
      else epilogue_warps<true, false>(kp, &out_map, sm, bars, tmem_base, q, lane);
    } else {
      if (tma_out) epilogue_warps<false, true>(kp, &out_map, sm, bars, tmem_base, q, lane);
      else epilogue_warps<false, false>(kp, &out_map, sm, bars, tmem_base, q, lane);
    }
  } else {
    if (REGS_AGG > 64) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_AGG));
    aggregator<KCH>(kp, sm, bars, warp, lane);
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == W_WARP) tmem_dealloc(tmem_base, TMEM_COLS);
}

template <int KCH>
cudaError_t launch(const EcParams& kp, const CUtensorMap& map, int grid, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(edgeconv_kernel<KCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  if (e != cudaSuccess) return e;
  edgeconv_kernel<KCH><<<grid, NTHREADS, SMEM_BYTES, s>>>(kp, map);
  return cudaSuccess;
}

}  // namespace

extern "C" int cp_edgeconv_ring_rows(int KP) {
  switch (KP) {
    case 8: return ring_rows(2);
    case 16: return ring_rows(4);
    case 20: return ring_rows(5);
    case 32: return ring_rows(8);
    case 40: return ring_rows(10);
    default: return -1;
  }
}

extern "C" int cp_edgeconv_fwd(const cp_edgeconv_params* pp, cp_stream_t s) {
  CP_REQUIRE(pp, CP_E_INVALID, "cp_edgeconv_fwd: null params");
  const cp_edgeconv_params& p = *pp;
  const cp_graph_plan& pl = p.plan;
  const cp_chain_layer& L = p.layer;
  CP_REQUIRE(p.B > 0 && p.N > 0 && p.z && p.out, CP_E_INVALID, "cp_edgeconv_fwd: bad B=%d N=%d or null tensor", p.B, p.N);
  CP_REQUIRE(p.Co == 64 || p.Co == 128 || p.Co == 256, CP_E_UNSUPPORTED, "cp_edgeconv_fwd: Co=%d not in {64,128,256}", p.Co);
  CP_REQUIRE(p.ld_z >= 2 * p.Co && (p.ld_z % 8) == 0 && (reinterpret_cast<uintptr_t>(p.z) & 15) == 0, CP_E_INVALID,
             "cp_edgeconv_fwd: z must be 16-byte aligned with ld_z %% 8 == 0 and ld_z >= 2*Co (ld_z=%d)", p.ld_z);
  CP_REQUIRE((size_t)p.N * p.ld_z * 2 < (1ull << 32) && (size_t)p.B * p.N < (1ull << 31), CP_E_UNSUPPORTED,
             "cp_edgeconv_fwd: one RoI's table must be < 4 GB and B * N < 2^31");
  CP_REQUIRE(pl.ucount && pl.ulist && pl.prog && pl.N == p.N && pl.T == (p.N + TILE_M - 1) / TILE_M && pl.G >= 1, CP_E_INVALID,
             "cp_edgeconv_fwd: graph plan does not match N=%d", p.N);
  CP_REQUIRE(pl.K >= 1 && pl.KP == cp_graph_plan_kp(pl.K), CP_E_UNSUPPORTED, "cp_edgeconv_fwd: K=%d / KP=%d not supported", pl.K, pl.KP);
  CP_REQUIRE(pl.umax == CP_PLAN_UMAX, CP_E_INVALID, "cp_edgeconv_fwd: plan.umax=%d, expected %d", pl.umax, CP_PLAN_UMAX);
  CP_REQUIRE(pl.max_unique >= 1 && pl.max_unique <= pl.umax && pl.max_unique <= cp_edgeconv_ring_rows(pl.KP), CP_E_UNSUPPORTED,
             "cp_edgeconv_fwd: a tile of this graph has %d distinct neighbour rows, the staging ring holds %d (use cp_chain_fwd(CP_PRO_AGG))",
             pl.max_unique, cp_edgeconv_ring_rows(pl.KP));
  CP_REQUIRE((reinterpret_cast<uintptr_t>(pl.prog) & 15) == 0 && (reinterpret_cast<uintptr_t>(pl.ulist) & 15) == 0, CP_E_INVALID,
             "cp_edgeconv_fwd: plan.prog / plan.ulist must be 16-byte aligned");
  CP_REQUIRE(!p.a_out || (p.ld_a_out >= p.Co && (p.ld_a_out % 8) == 0 && (reinterpret_cast<uintptr_t>(p.a_out) & 15) == 0), CP_E_INVALID,
             "cp_edgeconv_fwd: bad a_out / ld_a_out");
  CP_REQUIRE(L.w_packed && L.kin == p.Co && L.nout >= 1, CP_E_INVALID, "cp_edgeconv_fwd: layer kin=%d must equal Co=%d", L.kin, p.Co);
  CP_REQUIRE((reinterpret_cast<uintptr_t>(L.w_packed) & 15) == 0, CP_E_INVALID, "cp_edgeconv_fwd: weights not 16-byte aligned");
  EcParams kp;
  kp.p = p;
  kp.KC = p.Co / 64;
  kp.npad = (L.nout + 15) & ~15;
  CP_REQUIRE(kp.npad <= TMEM_COLS, CP_E_UNSUPPORTED, "cp_edgeconv_fwd: nout=%d > 512", L.nout);
  kp.NB = (kp.npad + 127) / 128;
  kp.tiles_per_roi = (p.N + TILE_M - 1) / TILE_M;
  kp.tpr_shift = -1;
  for (int sft = 0; sft < 30; ++sft)
    if ((1 << sft) == kp.tiles_per_roi) kp.tpr_shift = sft;
  kp.num_tiles = p.B * kp.tiles_per_roi;
  if (p.out_mode == CP_OUT_BF16)
    CP_REQUIRE((p.ld_out % 8) == 0 && p.ld_out >= kp.npad, CP_E_INVALID, "cp_edgeconv_fwd: bf16 output needs ld_out %% 8 == 0 and >= %d", kp.npad);
  else
    CP_REQUIRE(p.out_mode == CP_OUT_F32 && p.n_valid >= 1 && p.n_valid <= p.ld_out && p.n_valid <= kp.npad, CP_E_INVALID,
               "cp_edgeconv_fwd: bad f32 output spec");
  for (int c = 0; c < kp.KC; ++c)
    for (int nb = 0; nb < kp.NB; ++nb) kp.wt[c * kp.NB + nb] = cp::packed_tile(L.w_packed, nb, c, L.kin, kp.npad);
  const int num_sms = cp::num_sms();
  const int grid = kp.num_tiles < num_sms ? kp.num_tiles : num_sms;
  // bf16 outputs whose width is a multiple of 32 columns leave through TMA tensor stores: a 3-D map (columns, nodes, RoIs)
  // with a 32 x 32 box, so that rows beyond N of a ragged last tile are clipped instead of landing in the next RoI
  CUtensorMap map;
  memset(&map, 0, sizeof(map));
  kp.tma_out = (p.out_mode == CP_OUT_BF16 && kp.npad % 32 == 0 && kp.npad == L.nout && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0) ? 1 : 0;
  if (kp.tma_out) {
    const int rc = cp::make_out_tensor_map(&map, p.out, kp.npad, p.ld_out, p.N, p.B, "cp_edgeconv_fwd");
    if (rc != CP_OK) return rc;
  }
  cudaError_t e;
  switch (pl.KP) {
    case 8: e = launch<2>(kp, map, grid, (cudaStream_t)s); break;
    case 16: e = launch<4>(kp, map, grid, (cudaStream_t)s); break;
    case 20: e = launch<5>(kp, map, grid, (cudaStream_t)s); break;
    case 32: e = launch<8>(kp, map, grid, (cudaStream_t)s); break;
    default: e = launch<10>(kp, map, grid, (cudaStream_t)s); break;
  }
  CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "cp_edgeconv_fwd: launch failed: %s", cudaGetErrorString(e));
  CP_CHECK_LAUNCH("cp_edgeconv_fwd");
  return CP_OK;
}
