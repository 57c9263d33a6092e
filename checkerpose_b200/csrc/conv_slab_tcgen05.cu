// Slab convolution on tcgen05: the bf16 image branch over zero-bordered NHWC maps, every activation read once
// (SURVEY.md section 8f rank 1; get_gdrn_upsample_module checkerpose/model/pipeline.py:183-211, Index2Feat_module's
// patch_generator :144-145).
//
// cp_conv_bf16 (conv_bf16_tcgen05.cu) gathers the rows of every kernel tap again -- 9 x 16 KB of cp.async traffic and
// shared-memory writes per 64-channel slice of a 3 x 3 convolution, next to 9 x 32 KB of weights: with operand reads on top the
// shared-memory port, not the tensor pipe, sets its pace (64 % of the MMA rate).  Here the map carries its own zero border,
// (an image (H, W) is stored as (H+1, W+1) with a zero last row and column: over the flat index these are all four borders),
// so over the flat pixel index g = (b * Hp + py) * Wp + px a tap is a constant row shift:
//   out[g] = act(sum_t x[g + shift_t, :] . W_t^T + bias)
// and a tile of 128 consecutive positions needs ONE slab of 128 + max shift - min shift rows per channel slice (262 rows for
// 3 x 3 on a 64 x 64 map: 34 KB instead of 144 KB).  The slab is loaded by two TMA tensor copies (SWIZZLE_128B; rows before /
// after the matrix zero-filled), and tap t is the same shared memory read through a descriptor whose start address is moved
// by shift_t rows.  Measured on B200: tcgen05.mma applies the 128-byte swizzle on ABSOLUTE shared-memory address bits (the
// pattern TMA wrote), so a start address that is not a multiple of 8 rows needs nothing else -- putting the row phase into
// the descriptor's base-offset field (bits 49-51) gives wrong results.  No loader warps.
//
// CTA pairs (cluster of 2, tcgen05.mma.cta_group::2, M = 256): each CTA holds the slab of its own 128 positions and HALF of
// every weight tile; the leader's MMA reads both halves.  Weight traffic into each SM's shared memory halves again.
//   warp 0      weight producer: this CTA's (half) weight tile per (slice, tap) through the TMA engine, ring of WS stages;
//   warp 3      slab producer: two cp.async.bulk.tensor.2d per (tile, slice), double-buffered;
//   warp 1      leader: MMA issuer (4 MMAs of K = 16 per tap; commits release the stage / slab / accumulator in both CTAs);
//               peer: relays "my half has landed" to the leader's barriers;
//   warps 4-7   epilogue: tcgen05.ld -> + bias (BatchNorm folded) -> ReLU -> bf16 -> either 32 x 32 tiles through TMA stores
//               onto the same zero-bordered grid (positions outside the valid window written as zeros), or direct stores of
//               the window rows to a strided destination (patch maps; the four parities of a transposed convolution).
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "sm100.cuh"

using bf16 = __nv_bfloat16;
using namespace sm100;

namespace {

constexpr int TILE_M = 128;
constexpr int NTHREADS = 256;            // TMA-fed kernel: 8 warps
constexpr int EPI_WARP0 = 4;
constexpr int MAX_AB = 6;
constexpr int MAX_WS = 8;
constexpr int EPI_TILE_BYTES = 32 * 64;   // 32 rows x 32 bf16 (SWIZZLE_64B) per TMA store
constexpr int TMEM_COLS = 512;            // two accumulators of 256 columns
constexpr int SMEM_LIMIT = 227 * 1024;
constexpr int BAR_BYTES = 384;
constexpr int SEG_MAX = 4;
constexpr int SEG_BYTES = SEG_MAX * 256 * 4;    // fused 1x1 head: its weights (seg_n x Nout fp32), after the barrier block

struct Bars {
  uint64_t a_full[MAX_AB], a_empty[MAX_AB];
  uint64_t w_full[MAX_WS], w_empty[MAX_WS];
  uint64_t acc_full[2], acc_empty[2];
  uint32_t tmem_slot;
};

struct SlabParams {
  cp_conv_slab_params p;
  int c_chunks, row_tiles, npad, tma_out, img;
  int lo;             // smallest tap shift: the slab of tile rt starts at row rt * 128 + lo
  int RB;             // rows per TMA box (two boxes per slab)
  int a_buf_bytes, w_slot_bytes, AB, WS, off_w, off_epi, off_bar;   // AB slab buffers, WS weight stages
  int64_t G;
};

// Work units: (phase, 128-row tile), phase-major (tiles of one phase cost the same).  A CTA pair takes two neighbouring row
// tiles of ONE phase (the leader issues one tap list for both); with an odd tile count the peer's last tile lies beyond the
// matrix: its loads are zero-filled and nothing is stored.
template <bool PAIR>
struct Units {
  int first, step, count, per_phase;
  __device__ __forceinline__ explicit Units(const SlabParams& kp) {
    per_phase = PAIR ? (kp.row_tiles + 1) >> 1 : kp.row_tiles;
    const int total = per_phase * kp.p.num_phases;
    first = PAIR ? (int)blockIdx.x >> 1 : (int)blockIdx.x;
    step = PAIR ? (int)gridDim.x >> 1 : (int)gridDim.x;
    count = first < total ? (total - first + step - 1) / step : 0;
  }
  __device__ __forceinline__ void at(int i, int& ph, int& rt) const {
    const int u = first + i * step;
    ph = u / per_phase;
    const int r = u - ph * per_phase;
    rt = PAIR ? 2 * r + (int)(blockIdx.x & 1) : r;
  }
};

// ------------------------------------------------------------------------------------------------------
template <bool PAIR>
__device__ void slab_producer(const SlabParams& kp, const CUtensorMap* x_map, uint8_t* sm, Bars* bars) {
  const Units<PAIR> units(kp);
  const uint32_t sm_base = smem_u32(sm);
  const uint32_t box_bytes = (uint32_t)kp.RB * 128u;
  uint32_t ab = 0, around = 0;
  for (int i = 0; i < units.count; ++i) {
    int ph, rt;
    units.at(i, ph, rt);
    const int row_start = rt * TILE_M + kp.lo;
    for (int cc = 0; cc < kp.c_chunks; ++cc) {
      if (around > 0) mbar_wait(&bars->a_empty[ab], (around - 1) & 1);
      if (elect_one()) {
        const uint32_t dst = sm_base + ab * (uint32_t)kp.a_buf_bytes;
        mbar_arrive_expect_tx(&bars->a_full[ab], 2 * box_bytes);
        tma_load_2d(dst, x_map, cc * 64, row_start, &bars->a_full[ab]);
        tma_load_2d(dst + box_bytes, x_map, cc * 64, row_start + kp.RB, &bars->a_full[ab]);
      }
      __syncwarp();
      if (++ab == (uint32_t)kp.AB) { ab = 0; ++around; }
    }
  }
}

template <bool PAIR>
__device__ void weight_producer(const SlabParams& kp, uint8_t* sm, Bars* bars) {
  const cp_conv_slab_params& p = kp.p;
  const uint8_t* wb = reinterpret_cast<const uint8_t*>(p.w_packed);
  const Units<PAIR> units(kp);
  const uint32_t rank = PAIR ? (blockIdx.x & 1) : 0;
  const int npad = kp.npad;
  uint32_t s = 0, round = 0;
  for (int i = 0; i < units.count; ++i) {
    int ph, rt;
    units.at(i, ph, rt);
    const cp_slab_phase& P = p.phase[ph];
    for (int cc = 0; cc < kp.c_chunks; ++cc) {
      for (int t = 0; t < P.ntaps; ++t) {
        if (round > 0) mbar_wait(&bars->w_empty[s], (round - 1) & 1);
        if (elect_one()) {
          const size_t kc = (size_t)P.wtap[t] * kp.c_chunks + cc;
          uint8_t* w_s = sm + kp.off_w + s * kp.w_slot_bytes;
          if (PAIR) {
            // this CTA's half of the tile's rows (= output columns): a whole 128-row block of the packed matrix when the tile
            // has 256 columns, half of the single block otherwise
            const uint32_t half = (uint32_t)(npad / 2) * 128u;
            const uint8_t* src = npad == 256 ? wb + cp::packed_tile_offset(rank, kc, 128, p.K)
                                             : wb + cp::packed_tile_offset(0, kc, npad, p.K) + (size_t)rank * half;
            mbar_arrive_expect_tx(&bars->w_full[s], half);
            bulk_g2s(w_s, src, half, &bars->w_full[s]);
          } else {
            const int rows0 = min(128, npad), rows1 = npad - rows0;
            mbar_arrive_expect_tx(&bars->w_full[s], (uint32_t)npad * 128u);
            bulk_g2s(w_s, wb + cp::packed_tile_offset(0, kc, rows0, p.K), (uint32_t)rows0 * 128u, &bars->w_full[s]);
            if (rows1 > 0) bulk_g2s(w_s + 128 * 128, wb + cp::packed_tile_offset(1, kc, rows1, p.K), (uint32_t)rows1 * 128u, &bars->w_full[s]);
          }
        }
        __syncwarp();
        if (++s == (uint32_t)kp.WS) { s = 0; ++round; }
      }
    }
  }
}

template <bool PAIR>
__device__ void mma_issuer(const SlabParams& kp, uint8_t* sm, Bars* bars, uint32_t tmem_base) {
  const cp_conv_slab_params& p = kp.p;
  const uint32_t sm_base = smem_u32(sm);
  const uint32_t idesc = make_idesc_bf16(PAIR ? 256u : 128u, (uint32_t)kp.npad);
  const Units<PAIR> units(kp);
  uint32_t s = 0, wround = 0, ab = 0, around = 0, tcount = 0;
  for (int i = 0; i < units.count; ++i, ++tcount) {
    int ph, rt;
    units.at(i, ph, rt);
    const cp_slab_phase& P = p.phase[ph];
    const uint32_t slot = tcount & 1;
    // CTA pairs: the peer arrives on these barriers as well.  The data behind them is only read by the MMA unit (async
    // proxy), never by this thread, so the default CTA-scope wait is enough, as in CUTLASS' 2-SM pipelines.
    if (tcount >= 2) mbar_wait(&bars->acc_empty[slot], ((tcount >> 1) - 1) & 1);
    const uint32_t d = tmem_base + slot * 256;
    for (int cc = 0; cc < kp.c_chunks; ++cc) {
      mbar_wait(&bars->a_full[ab], around & 1);
      const uint32_t a_lo0 = smem_desc_lo(sm_base + ab * (uint32_t)kp.a_buf_bytes);
      for (int t = 0; t < P.ntaps; ++t) {
        mbar_wait(&bars->w_full[s], wround & 1);
        tc_fence_after_sync();
        const uint32_t rel = (uint32_t)(P.shift[t] - kp.lo);            // rows from the start of the slab
        const uint32_t a_lo = a_lo0 + rel * 8;                          // 128 bytes per row, in units of 16
        const uint32_t w_lo = smem_desc_lo(sm_base + kp.off_w + s * kp.w_slot_bytes);
        const bool last_t = t == P.ntaps - 1;
        if (elect_one()) {
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k) {
            const uint32_t acc = (uint32_t)((cc | t | (int)k) != 0);
            if (PAIR) mma2_bf16_ss_lo(d, a_lo + 2 * k, w_lo + 2 * k, idesc, acc);
            else mma_bf16_ss_lo(d, a_lo + 2 * k, w_lo + 2 * k, idesc, acc);
          }
          if (PAIR) {
            mma2_commit_both(smem_u32(&bars->w_empty[s]));
            if (last_t) mma2_commit_both(smem_u32(&bars->a_empty[ab]));
            if (last_t && cc == kp.c_chunks - 1) mma2_commit_both(smem_u32(&bars->acc_full[slot]));
          } else {
            mma_commit(&bars->w_empty[s]);
            if (last_t) mma_commit(&bars->a_empty[ab]);
            if (last_t && cc == kp.c_chunks - 1) mma_commit(&bars->acc_full[slot]);
          }
        }
        __syncwarp();
        if (++s == (uint32_t)kp.WS) { s = 0; ++wround; }
      }
      if (++ab == (uint32_t)kp.AB) { ab = 0; ++around; }
    }
  }
}

// CTA pairs: the peer's MMA warp has nothing to issue; in the leader's order of consumption it tells the leader's barriers
// when the peer's slab / weight half has landed.
__device__ void relay_peer(const SlabParams& kp, Bars* bars) {
  const cp_conv_slab_params& p = kp.p;
  const uint32_t a_full_leader0 = mapa_rank(smem_u32(&bars->a_full[0]), 0);
  const uint32_t w_full_leader0 = mapa_rank(smem_u32(&bars->w_full[0]), 0);
  const Units<true> units(kp);
  uint32_t s = 0, wround = 0, ab = 0, around = 0;
  for (int i = 0; i < units.count; ++i) {
    int ph, rt;
    units.at(i, ph, rt);
    const int ntaps = p.phase[ph].ntaps;
    for (int cc = 0; cc < kp.c_chunks; ++cc) {
      mbar_wait(&bars->a_full[ab], around & 1);
      if (elect_one()) mbar_arrive_remote(a_full_leader0 + ab * 8);
      __syncwarp();
      for (int t = 0; t < ntaps; ++t) {
        mbar_wait(&bars->w_full[s], wround & 1);
        if (elect_one()) mbar_arrive_remote(w_full_leader0 + s * 8);
        __syncwarp();
        if (++s == (uint32_t)kp.WS) { s = 0; ++wround; }
      }
      if (++ab == (uint32_t)kp.AB) { ab = 0; ++around; }
    }
  }
}

template <bool PAIR>
__device__ void epilogue(const SlabParams& kp, const CUtensorMap* out_map, uint8_t* sm, Bars* bars, uint32_t tmem_base, int q, int lane) {
  const cp_conv_slab_params& p = kp.p;
  const bool bias_vec = p.bias && (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0;
  const bool out_vec = (p.ld_out & 7) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0;
  const uint32_t tbuf0 = smem_u32(sm) + kp.off_epi + q * 2 * EPI_TILE_BYTES;
  const uint32_t acc_empty_leader0 = PAIR ? mapa_rank(smem_u32(&bars->acc_empty[0]), 0) : 0u;
  const int sw = (lane >> 1) & 3;      // SWIZZLE_64B: 16-byte chunk index ^= bits 1-2 of the row
  bf16* out = reinterpret_cast<bf16*>(p.out);
  const Units<PAIR> units(kp);
  uint32_t tcount = 0, nstore = 0;
  for (int i = 0; i < units.count; ++i, ++tcount) {
    int ph, rt;
    units.at(i, ph, rt);
    const uint32_t slot = tcount & 1;
    // this row's grid position: inside the window of real outputs?
    const int64_t row0 = (int64_t)rt * TILE_M + q * 32;
    const int64_t g = row0 + lane;
    bool valid = g < kp.G;
    int64_t orow = g;
    if (valid) {
      const int b = (int)(g / kp.img);
      const int rem = (int)(g - (int64_t)b * kp.img);
      const int py = rem / p.Wp, px = rem - py * p.Wp;
      valid = py >= p.vy0 && py < p.vy1 && px >= p.vx0 && px < p.vx1;
      if (p.compact) orow = (int64_t)b * p.out_sb + (int64_t)(py - p.vy0) * p.out_sy + (int64_t)(px - p.vx0) * p.out_sx + p.phase[ph].out_off;
    }
    while (!mbar_try_wait(&bars->acc_full[slot], (tcount >> 1) & 1)) __nanosleep(64);   // idle for a whole K loop: do not spin
    tc_fence_after_sync();
    const uint32_t tb = tmem_base + ((uint32_t)(q * 32) << 16) + slot * 256;
    float seg_acc[SEG_MAX] = {0.f, 0.f, 0.f, 0.f};
    for (int n0 = 0; n0 < kp.npad; n0 += 32) {
      if (n0 >= p.Nout) break;
      uint32_t r[32];
      tmem_ld32(tb + (uint32_t)n0, r);
      float bv[32];
      if (bias_vec && n0 + 32 <= p.Nout) {
#pragma unroll
        for (int e4 = 0; e4 < 8; ++e4) {
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + n0) + e4);
          bv[e4 * 4] = b4.x; bv[e4 * 4 + 1] = b4.y; bv[e4 * 4 + 2] = b4.z; bv[e4 * 4 + 3] = b4.w;
        }
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e) bv[e] = (p.bias && n0 + e < p.Nout) ? __ldg(p.bias + n0 + e) : 0.f;
      }
      tmem_ld_wait();
      uint32_t w[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        float x0 = __uint_as_float(r[2 * e]) + bv[2 * e], x1 = __uint_as_float(r[2 * e + 1]) + bv[2 * e + 1];
        if (p.act) { x0 = cp::lrelu(x0, p.slope); x1 = cp::lrelu(x1, p.slope); }
        w[e] = valid ? f2_to_bf2(x0, x1) : 0u;      // outside the window the grid keeps its zero border
      }
      if (p.seg_w) {      // fused 1x1 head over the bf16 values this row stores
        const float4* sw4 = reinterpret_cast<const float4*>(sm + kp.off_bar + BAR_BYTES);
#pragma unroll
        for (int j = 0; j < SEG_MAX; ++j) {
          if (j >= p.seg_n) break;
          float a = seg_acc[j];
#pragma unroll
          for (int e4 = 0; e4 < 8; ++e4) {
            const float4 c = sw4[j * 64 + (n0 >> 2) + e4];
            a = fmaf(__uint_as_float(w[2 * e4] << 16), c.x, a);
            a = fmaf(__uint_as_float(w[2 * e4] & 0xffff0000u), c.y, a);
            a = fmaf(__uint_as_float(w[2 * e4 + 1] << 16), c.z, a);
            a = fmaf(__uint_as_float(w[2 * e4 + 1] & 0xffff0000u), c.w, a);
          }
          seg_acc[j] = a;
        }
      }
      if (kp.tma_out) {
        const uint32_t tbuf = tbuf0 + (nstore & 1) * EPI_TILE_BYTES;
        ++nstore;
        if (lane == 0) bulk_wait_read<1>();
        __syncwarp();
#pragma unroll
        for (int e = 0; e < 4; ++e) sts128(tbuf + lane * 64 + ((e ^ sw) << 4), make_uint4(w[e * 4], w[e * 4 + 1], w[e * 4 + 2], w[e * 4 + 3]));
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && row0 < kp.G) {
          tma_store_3d(out_map, tbuf, n0, (int)row0, 0);
          bulk_commit();
        }
      } else if (p.compact ? valid : g < kp.G) {
        bf16* o = out + orow * p.ld_out + n0;
        if (out_vec && n0 + 32 <= p.Nout) {
#pragma unroll
          for (int e = 0; e < 4; ++e) reinterpret_cast<uint4*>(o)[e] = make_uint4(w[e * 4], w[e * 4 + 1], w[e * 4 + 2], w[e * 4 + 3]);
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (n0 + e < p.Nout) o[e] = __ushort_as_bfloat16((unsigned short)((e & 1) ? (w[e >> 1] >> 16) : (w[e >> 1] & 0xffffu)));
        }
      }
    }
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) {
      if (PAIR) mbar_arrive_remote(acc_empty_leader0 + slot * 8);
      else mbar_arrive(&bars->acc_empty[slot]);
    }
    if (p.seg_w && valid) {
      const int Hs = p.vy1 - p.vy0, Ws = p.vx1 - p.vx0;
      const int b = (int)(g / kp.img);
      const int rem = (int)(g - (int64_t)b * kp.img);
      const int py = rem / p.Wp, px = rem - py * p.Wp;
#pragma unroll
      for (int j = 0; j < SEG_MAX; ++j)
        if (j < p.seg_n) p.seg_out[(((int64_t)b * p.seg_n + j) * Hs + (py - p.vy0)) * Ws + (px - p.vx0)] = seg_acc[j] + __ldg(p.seg_b + j);
    }
  }
  if (kp.tma_out && lane == 0) bulk_wait_read<0>();
}

template <bool PAIR>
__global__ void __launch_bounds__(NTHREADS, 1) conv_slab_kernel(const __grid_constant__ SlabParams kp, const __grid_constant__ CUtensorMap x_map,
                                                                 const __grid_constant__ CUtensorMap out_map) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  Bars* bars = reinterpret_cast<Bars*>(sm + kp.off_bar);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool leader = !PAIR || (blockIdx.x & 1) == 0;
  if (threadIdx.x == 0) {
    // pairs: the leader's "full" barriers also collect the peer's relay, its acc_empty both CTAs' epilogue warps
    for (int a = 0; a < MAX_AB; ++a) {
      mbar_init(&bars->a_full[a], PAIR && leader ? 2 : 1);
      mbar_init(&bars->a_empty[a], 1);
    }
    for (int s = 0; s < MAX_WS; ++s) {
      mbar_init(&bars->w_full[s], PAIR && leader ? 2 : 1);
      mbar_init(&bars->w_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&bars->acc_full[a], 1);
      mbar_init(&bars->acc_empty[a], PAIR ? 8 : 4);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    if (PAIR) tmem_alloc_pair(&bars->tmem_slot, TMEM_COLS);
    else tmem_alloc(&bars->tmem_slot, TMEM_COLS);
  }
  if (kp.p.seg_w) {   // fused 1x1 head: weights zero-padded to npad columns
    float* sw = reinterpret_cast<float*>(sm + kp.off_bar + BAR_BYTES);
    for (int i = threadIdx.x; i < kp.p.seg_n * 256; i += blockDim.x) {
      const int j = i >> 8, n = i & 255;
      sw[i] = n < kp.p.Nout ? __ldg(kp.p.seg_w + (size_t)j * kp.p.Nout + n) : 0.f;
    }
  }
  tc_fence_before_sync();
  if (PAIR) cluster_sync_all();     // both CTAs' barriers exist before anyone arrives remotely
  else __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = bars->tmem_slot;

  if (warp >= EPI_WARP0) epilogue<PAIR>(kp, &out_map, sm, bars, tmem_base, warp - EPI_WARP0, lane);
  else if (warp == 0) weight_producer<PAIR>(kp, sm, bars);
  else if (warp == 3) slab_producer<PAIR>(kp, &x_map, sm, bars);
  else if (warp == 1) {
    if (leader) mma_issuer<PAIR>(kp, sm, bars, tmem_base);
    else relay_peer(kp, bars);
  }

  tc_fence_before_sync();
  if (PAIR) cluster_sync_all();     // no CTA leaves while the peer may still read its shared memory / arrive on its barriers
  else __syncthreads();
  if (warp == 2) {
    if (PAIR) tmem_dealloc_pair(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <bool PAIR>
cudaError_t launch(const SlabParams& kp, const CUtensorMap& x_map, const CUtensorMap& out_map, int grid, int smem, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(conv_slab_kernel<PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(NTHREADS);
  cfg.dynamicSmemBytes = (size_t)smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = PAIR ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, conv_slab_kernel<PAIR>, kp, x_map, out_map);
}

}  // namespace

extern "C" int cp_conv_slab(const cp_conv_slab_params* pp, cp_stream_t s) {
  CP_REQUIRE(pp, CP_E_INVALID, "cp_conv_slab: null params");
  const cp_conv_slab_params& p = *pp;
  CP_REQUIRE(p.x && p.w_packed && p.out && p.B > 0 && p.Hp > 0 && p.Wp > 0 && p.Nout > 0, CP_E_INVALID, "cp_conv_slab: bad arguments");
  CP_REQUIRE(p.C > 0 && p.C % 64 == 0 && (reinterpret_cast<uintptr_t>(p.w_packed) & 15) == 0 &&
             p.ldx >= p.C && (p.ldx & 7) == 0 && (reinterpret_cast<uintptr_t>(p.x) & 15) == 0, CP_E_UNSUPPORTED,
             "cp_conv_slab: C=%d must be a multiple of 64, pixel rows and weights 16-byte aligned", p.C);
  CP_REQUIRE(p.Nout <= 256 && p.ld_out >= p.Nout, CP_E_UNSUPPORTED, "cp_conv_slab: Nout=%d must be <= 256 and <= ld_out", p.Nout);
  CP_REQUIRE(p.num_phases >= 1 && p.num_phases <= CP_SLAB_MAX_PHASES && (p.num_phases == 1 || p.compact), CP_E_INVALID,
             "cp_conv_slab: %d phases (several phases need a compact destination)", p.num_phases);
  CP_REQUIRE(p.vy0 >= 0 && p.vy1 <= p.Hp && p.vx0 >= 0 && p.vx1 <= p.Wp && p.vy0 < p.vy1 && p.vx0 < p.vx1, CP_E_INVALID, "cp_conv_slab: bad output window");
  CP_REQUIRE(!p.seg_w || (p.seg_b && p.seg_out && p.seg_n >= 1 && p.seg_n <= SEG_MAX && !p.compact && p.num_phases == 1), CP_E_INVALID,
             "cp_conv_slab: the fused 1x1 head needs bias, output, 1..%d channels and a same-grid destination", SEG_MAX);
  SlabParams kp;
  memset(&kp, 0, sizeof(kp));
  kp.p = p;
  kp.c_chunks = p.C / 64;
  int lo = 0, hi = 0, wt_max = 0;
  for (int ph = 0; ph < p.num_phases; ++ph) {
    const cp_slab_phase& P = p.phase[ph];
    CP_REQUIRE(P.ntaps >= 1 && P.ntaps <= CP_SLAB_MAX_TAPS, CP_E_INVALID, "cp_conv_slab: phase %d has %d taps", ph, P.ntaps);
    for (int t = 0; t < P.ntaps; ++t) {
      CP_REQUIRE(P.wtap[t] >= 0, CP_E_INVALID, "cp_conv_slab: negative weight tap");
      if (ph == 0 && t == 0) lo = hi = P.shift[t];
      lo = P.shift[t] < lo ? P.shift[t] : lo;
      hi = P.shift[t] > hi ? P.shift[t] : hi;
      wt_max = P.wtap[t] > wt_max ? P.wtap[t] : wt_max;
    }
  }
  CP_REQUIRE((int64_t)(wt_max + 1) * p.C <= p.K && p.K % 64 == 0, CP_E_INVALID, "cp_conv_slab: weight tap %d beyond K=%d", wt_max, p.K);
  kp.lo = lo;
  const int R = TILE_M + hi - lo;
  kp.RB = ((R + 1) / 2 + 7) / 8 * 8;
  CP_REQUIRE(kp.RB <= 256, CP_E_UNSUPPORTED, "cp_conv_slab: tap span %d rows too wide for one slab (map width %d)", hi - lo, p.Wp);
  kp.img = p.Hp * p.Wp;
  kp.G = (int64_t)p.B * kp.img;
  CP_REQUIRE(kp.G + TILE_M + kp.RB * 2 < (1ll << 31), CP_E_UNSUPPORTED, "cp_conv_slab: too many rows");
  kp.row_tiles = (int)((kp.G + TILE_M - 1) / TILE_M);
  kp.npad = (p.Nout + 15) / 16 * 16;
  const char* pair_env = getenv("CP_SLAB_PAIR");
  const bool pair = !(pair_env && pair_env[0] == '0') && (kp.npad == 256 || kp.npad <= 128) && kp.row_tiles >= 2;
  kp.a_buf_bytes = 2 * kp.RB * 128;
  const int w_rows = pair ? kp.npad / 2 : kp.npad;
  kp.w_slot_bytes = (w_rows * 128 + 1023) / 1024 * 1024;
  // shared memory: 4 weight stages first, then as many slab buffers as fit (2..6: the narrow convolutions are bound by the
  // activation stream and want it deep), the rest goes back to the weight ring
  const int avail = SMEM_LIMIT - (1024 + 4 * 2 * EPI_TILE_BYTES + BAR_BYTES + SEG_BYTES);
  kp.AB = (avail - 4 * kp.w_slot_bytes) / kp.a_buf_bytes;
  kp.AB = kp.AB > MAX_AB ? MAX_AB : kp.AB;
  CP_REQUIRE(kp.AB >= 2, CP_E_UNSUPPORTED, "cp_conv_slab: no room for two activation slabs");
  kp.WS = (avail - kp.AB * kp.a_buf_bytes) / kp.w_slot_bytes;
  kp.WS = kp.WS > MAX_WS ? MAX_WS : kp.WS;
  CP_REQUIRE(kp.WS >= 2, CP_E_UNSUPPORTED, "cp_conv_slab: no room for the weight ring");
  kp.off_w = kp.AB * kp.a_buf_bytes;
  kp.off_epi = kp.off_w + kp.WS * kp.w_slot_bytes;
  kp.off_bar = kp.off_epi + 4 * 2 * EPI_TILE_BYTES;
  const int smem = kp.off_bar + BAR_BYTES + SEG_BYTES + 1024;
  static_assert(sizeof(Bars) <= BAR_BYTES, "barrier block");

  CUtensorMap x_map, out_map;
  memset(&x_map, 0, sizeof(x_map));
  memset(&out_map, 0, sizeof(out_map));
  int rc = cp::make_bf16_operand_map(&x_map, p.x, p.C, kp.G, p.ldx, "cp_conv_slab", kp.RB);
  if (rc != CP_OK) return rc;
  kp.tma_out = (!p.compact && (p.ld_out & 7) == 0 && p.Nout % 32 == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0) ? 1 : 0;
  if (kp.tma_out) {
    rc = cp::make_out_tensor_map(&out_map, p.out, p.Nout, p.ld_out, (int)kp.G, 1, "cp_conv_slab");
    if (rc != CP_OK) return rc;
  }
  const int num_sms = cp::num_sms();
  cudaError_t e;
  if (pair) {
    const int units = (kp.row_tiles + 1) / 2 * p.num_phases;
    const int clusters = units < num_sms / 2 ? units : num_sms / 2;
    e = launch<true>(kp, x_map, out_map, 2 * clusters, smem, (cudaStream_t)s);
  } else {
    const int units = kp.row_tiles * p.num_phases;
    const int grid = units < num_sms ? units : num_sms;
    e = launch<false>(kp, x_map, out_map, grid, smem, (cudaStream_t)s);
  }
  CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "cp_conv_slab: launch failed: %s", cudaGetErrorString(e));
  CP_CHECK_LAUNCH("cp_conv_slab");
  return CP_OK;
}
