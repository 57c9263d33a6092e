// K3: warp-specialised Index2Feat gather + pre-graph MLP + first [P|Q] GEMM (bf16 operands, fp32 accumulation in TMEM).
//
// Replaces, for one refine stage, Index2Feat_module's 4-tap integer gather (checkerpose/model/pipeline.py:156-163), the
// roi-mask multiply and concat with the previous graph feature (:280-283), pre_graph_module = Linear+LeakyReLU x2
// (:284-286) and the [P|Q] GEMM of the stage's first EdgeConv layer (cp_fold_edgeconv) -- three chained GEMMs
//   h0 = lrelu([taps | gf] W0^T + b0)   K = 256 + Cg -> 256
//   h1 = lrelu(h0 W1^T + b1)            256 -> 256
//   z  = h1 W2^T + b2                   256 -> 256 or 512
// per tile of 128 nodes, with nothing but z going back to HBM.  One persistent CTA of 16 warps per SM:
//
//   warps 0-3   gather producers: cp.async (LDGSTS, zero-fill for masked / missing rows) of the four 128-byte taps and
//               of the graph-feature row slices straight into 64-channel A-operand chunks (SWIZZLE_128B) of a 4-slot
//               ring; the taps' addresses of the NEXT tile are computed while the current one is copied;
//   warps 4-11  epilogue: TMEM -> registers -> + bias (shared memory) -> LeakyReLU -> bf16 -> either the next GEMM's A
//               operand in shared memory (h0, h1) or, for z, a swizzled 32 x 32 tile that leaves through a TMA tensor
//               store (a thread owns a row: direct stores would write 32 half-filled sectors per instruction);
//   warp 12     weight producer: the 40 packed 16 KB weight tiles of a node tile through the TMA engine, 4-stage ring;
//   warp 13     one thread issues tcgen05.mma (M=128, N=128, K=16).
//
// TMEM holds two accumulators of 256 columns; the GEMM stages of a tile (L0, L1, L2 first half, L2 second half)
// alternate between them, so the MMAs of a stage overlap the epilogue of the one before wherever the data allows
// (L2b over L2a's epilogue, the next tile's L0 over L2b's), and the gathers run a tile ahead of both.
// cp_chain_fwd (chain_tcgen05.cu) dispatches here for the shipped layer shapes and keeps the generic kernel otherwise.
#include <cuda.h>

#include "common.cuh"
#include "sm100.cuh"

using bf16 = __nv_bfloat16;
using namespace sm100;

namespace {

constexpr int TILE_M = 128;
constexpr int NUM_G_WARPS = 4, G_THREADS = NUM_G_WARPS * 32;
constexpr int NUM_E_WARPS = 8;              // a multiple of 4: NUM_E_WARPS / 4 warps per TMEM lane quarter
constexpr int E_WARP0 = 4;
constexpr int W_WARP = E_WARP0 + NUM_E_WARPS, MMA_WARP = W_WARP + 1;
constexpr int NUM_WARPS = 16;               // two idle warps: 512 threads leave 128 registers per thread
static_assert(NUM_E_WARPS % 4 == 0 && E_WARP0 % 4 == 0 && NUM_G_WARPS <= E_WARP0 && TILE_M % (NUM_G_WARPS * 4) == 0, "epilogue warp w drains TMEM lane quarter w % 4");
constexpr int NTHREADS = NUM_WARPS * 32;
constexpr int CHUNK_BYTES = TILE_M * 128;   // 128 rows x 64 bf16
constexpr int NX = 4;                       // gather ring slots
constexpr int NH = 4;                       // chunks of h0 / h1 (256 channels)
constexpr int B_STAGES = 4, B_STAGE_BYTES = 128 * 128;
constexpr int TBUF_BYTES = 32 * 64;          // per epilogue warp: a tile of 32 rows x 32 bf16 (SWIZZLE_64B) for the TMA stores
constexpr int BIAS_FLOATS = 1024;           // 256 + 256 + 512
constexpr int ACC_COLS = 256;
constexpr int MAX_WT = 48;

constexpr int OFF_X = 0;
constexpr int OFF_H = OFF_X + NX * CHUNK_BYTES;
constexpr int OFF_B = OFF_H + NH * CHUNK_BYTES;
constexpr int OFF_TBUF = OFF_B + B_STAGES * B_STAGE_BYTES;
constexpr int OFF_BIAS = OFF_TBUF + NUM_E_WARPS * TBUF_BYTES;
constexpr int OFF_BAR = OFF_BIAS + BIAS_FLOATS * 4;
constexpr int SMEM_BYTES = OFF_BAR + 512;
static_assert(SMEM_BYTES + 1024 <= 227 * 1024, "shared memory budget");

struct TcParams {
  cp_chain_params p;
  int tiles_per_roi, num_tiles;
  int KX;        // A chunks of layer 0: 4 taps + Cg / 64
  int P2;        // 128-column blocks of layer 2 per half (1: nout2 = 256, one half; 2: nout2 = 512, two halves)
  int halves2;   // 1 or 2 accumulator passes for layer 2
  int T;         // weight tiles per node tile
  cp::WTile wt[MAX_WT]; // in the order the MMA thread consumes them
};

struct Bars {
  uint64_t x_full[NX], x_empty[NX];
  uint64_t b_full[B_STAGES], b_empty[B_STAGES];
  uint64_t h_full[NH], h_free;   // h_full per 64-channel chunk: the next GEMM starts on chunk 0 while the epilogue writes chunk 1
  uint64_t acc_full[2], acc_empty[2];
  uint32_t tmem_slot;
};
static_assert(sizeof(Bars) <= 512, "barrier block");

__device__ __forceinline__ uint32_t chunk_off(int row, int piece) { return (uint32_t)(row * 128 + ((piece ^ (row & 7)) << 4)); }

// ------------------------------------------------------------------------------------------------------
// gather producers
// ------------------------------------------------------------------------------------------------------
__device__ void gather_warps(const TcParams& kp, uint8_t* sm, Bars* bars, int gw, int lane) {
  const cp_chain_params& p = kp.p;
  const int rg = lane >> 3, piece = lane & 7;
  const uint32_t sm_base = smem_u32(sm);
  constexpr int RPT = TILE_M / (NUM_G_WARPS * 4);   // rows per thread: 8
  // byte offset of tap (0,0) of each of this thread's rows inside the RoI's patch map, -1 = masked / no row
  int toff[RPT], toff_next[RPT];
  auto load_ids = [&](int tile, int (&o)[RPT]) {
    const int b = tile / kp.tiles_per_roi, n0 = (tile - b * kp.tiles_per_roi) * TILE_M;
    const int rows_valid = min(TILE_M, p.N - n0);
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
      const int r = 4 * (gw + NUM_G_WARPS * i) + rg;
      o[i] = -1;
      if (r < rows_valid) {
        const size_t e = (size_t)b * p.N + n0 + r;
        const float mk = p.mask ? __ldg(p.mask + e) : 1.f;
        const int yy = (int)(2 * __ldg(p.y_id + e)), xx = (int)(2 * __ldg(p.x_id + e));
        // caller error (the reference raises a device-side index assert, pipeline.py:158-161): never read out of bounds
        if (yy < 0 || xx < 0 || yy + p.tap_step >= p.Hp || xx + p.tap_step >= p.Wp) __trap();
        if (mk != 0.f) o[i] = (yy * p.Wp + xx) * 128;
      }
    }
  };
  if ((int)blockIdx.x < kp.num_tiles) load_ids(blockIdx.x, toff_next);
  uint32_t cnt = 0;   // chunks produced
  for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x) {
    const int b = tile / kp.tiles_per_roi, n0 = (tile - b * kp.tiles_per_roi) * TILE_M;
    const int rows_valid = min(TILE_M, p.N - n0);
#pragma unroll
    for (int i = 0; i < RPT; ++i) toff[i] = toff_next[i];
    if (tile + (int)gridDim.x < kp.num_tiles) load_ids(tile + gridDim.x, toff_next);   // in flight while this tile is copied
    const uint8_t* pb = reinterpret_cast<const uint8_t*>(p.patches) + (size_t)b * p.Hp * p.Wp * 128 + piece * 16;
    const uint8_t* gf = reinterpret_cast<const uint8_t*>(p.graph_feat) + ((size_t)b * p.N + n0) * p.ld_gf * 2 + piece * 16;
    for (int c = 0; c < kp.KX; ++c, ++cnt) {
      const uint32_t slot = cnt % NX;
      if (cnt >= NX) mbar_wait(&bars->x_empty[slot], ((cnt / NX) - 1) & 1);
      const uint32_t dst = sm_base + OFF_X + slot * CHUNK_BYTES;
      if (c < 4) {
        const int tap_off = (((c & 1) ? p.tap_step : 0) * p.Wp + ((c & 2) ? p.tap_step : 0)) * 128;
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
          const int r = 4 * (gw + NUM_G_WARPS * i) + rg;
          const bool ok = toff[i] >= 0;
          cp_async16_zfill(dst + chunk_off(r, piece), pb + (ok ? toff[i] + tap_off : 0), ok ? 16u : 0u);
        }
      } else {
        const uint8_t* src = gf + (c - 4) * 128;
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
          const int r = 4 * (gw + NUM_G_WARPS * i) + rg;
          const bool ok = r < rows_valid;
          cp_async16_zfill(dst + chunk_off(r, piece), src + (ok ? (size_t)r * p.ld_gf * 2 : 0), ok ? 16u : 0u);
        }
      }
      cp_async_arrive_noinc(&bars->x_full[slot]);
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// weight producer / MMA issuer
// ------------------------------------------------------------------------------------------------------
__device__ void weight_producer(const TcParams& kp, uint8_t* sm, Bars* bars) {
  uint32_t cnt = 0;
  for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x) {
    for (int w = 0; w < kp.T; ++w, ++cnt) {
      const int s = cnt % B_STAGES;
      const uint32_t use = cnt / B_STAGES;
      if (use > 0) mbar_wait(&bars->b_empty[s], (use - 1) & 1);
      if (elect_one()) {
        mbar_arrive_expect_tx(&bars->b_full[s], kp.wt[w].bytes);
        bulk_g2s(sm + OFF_B + s * B_STAGE_BYTES, kp.wt[w].ptr, kp.wt[w].bytes, &bars->b_full[s]);
      }
      __syncwarp();
    }
  }
}

__device__ void mma_issuer(const TcParams& kp, uint8_t* sm, Bars* bars, uint32_t tmem_base) {
  uint32_t wcnt = 0;    // weight tiles consumed
  uint32_t xcnt = 0;    // gather chunks consumed
  uint32_t st = 0;      // accumulator stages issued (slot = st & 1)
  uint32_t hcnt = 0;    // h_full phases consumed
  const uint32_t idesc = make_idesc_bf16_m128(128);
  const uint32_t b_lo0 = smem_desc_lo(smem_u32(sm + OFF_B));
  auto gemm_block = [&](uint32_t a_addr, uint32_t d, bool accumulate) {   // one 128 x 128 x 64 block against the next weight tile
    const int s = wcnt % B_STAGES;
    mbar_wait(&bars->b_full[s], (wcnt / B_STAGES) & 1);
    tc_fence_after_sync();
    const uint32_t a_lo = smem_desc_lo(a_addr), b_lo = b_lo0 + s * (B_STAGE_BYTES >> 4);
    if (elect_one()) {
      mma_bf16_ss_lo(d, a_lo, b_lo, idesc, (uint32_t)accumulate);
      mma_bf16_ss_lo(d, a_lo + 2, b_lo + 2, idesc, 1u);
      mma_bf16_ss_lo(d, a_lo + 4, b_lo + 4, idesc, 1u);
      mma_bf16_ss_lo(d, a_lo + 6, b_lo + 6, idesc, 1u);
      mma_commit(&bars->b_empty[s]);
    }
    __syncwarp();
    ++wcnt;
  };
  auto acquire_acc = [&]() -> uint32_t {   // TMEM columns of the next stage, once its previous contents are drained
    const uint32_t slot = st & 1;
    if (st >= 2) {
      mbar_wait(&bars->acc_empty[slot], ((st >> 1) - 1) & 1);
      tc_fence_after_sync();
    }
    return tmem_base + slot * ACC_COLS;
  };
  for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x) {
    // ---- L0: [taps | gf] -> 256, chunk by chunk as the gathers land ----
    {
      const uint32_t d = acquire_acc();
      for (int c = 0; c < kp.KX; ++c, ++xcnt) {
        const uint32_t slot = xcnt % NX;
        mbar_wait(&bars->x_full[slot], (xcnt / NX) & 1);
        tc_fence_after_sync();
        const uint32_t a_addr = smem_u32(sm + OFF_X + slot * CHUNK_BYTES);
        gemm_block(a_addr, d, c != 0);
        gemm_block(a_addr, d + 128, c != 0);
        if (elect_one()) mma_commit(&bars->x_empty[slot]);
        __syncwarp();
      }
      if (elect_one()) mma_commit(&bars->acc_full[st & 1]);
      __syncwarp();
      ++st;
    }
    // ---- L1: h0 -> 256 ----
    {
      const uint32_t d = acquire_acc();
      for (int c = 0; c < NH; ++c) {
        mbar_wait(&bars->h_full[c], hcnt & 1);
        tc_fence_after_sync();
        const uint32_t a_addr = smem_u32(sm + OFF_H + c * CHUNK_BYTES);
        gemm_block(a_addr, d, c != 0);
        gemm_block(a_addr, d + 128, c != 0);
      }
      ++hcnt;
      if (elect_one()) {
        mma_commit(&bars->h_free);            // h0 consumed: the epilogue may write h1 over it
        mma_commit(&bars->acc_full[st & 1]);
      }
      __syncwarp();
      ++st;
    }
    // ---- L2: h1 -> 256 (one pass) or 512 (two passes of 256 columns) ----
    for (int half = 0; half < kp.halves2; ++half) {
      const uint32_t d = acquire_acc();
      for (int c = 0; c < NH; ++c) {
        if (half == 0) {
          mbar_wait(&bars->h_full[c], hcnt & 1);
          tc_fence_after_sync();
        }
        const uint32_t a_addr = smem_u32(sm + OFF_H + c * CHUNK_BYTES);
        for (int nb = 0; nb < kp.P2; ++nb) gemm_block(a_addr, d + nb * 128, c != 0);
      }
      if (half == 0) ++hcnt;
      if (elect_one()) {
        if (half == kp.halves2 - 1) mma_commit(&bars->h_free);   // h1 consumed: the next tile's h0 may be written
        mma_commit(&bars->acc_full[st & 1]);
      }
      __syncwarp();
      ++st;
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// epilogue: warp (q = w & 3, half = w >> 2) drains TMEM lanes [32 q, 32 q + 32), every second 32-column block
// ------------------------------------------------------------------------------------------------------
__device__ void epilogue_warps(const TcParams& kp, const CUtensorMap* out_map, uint8_t* sm, Bars* bars, uint32_t tmem_base, int ew, int lane) {
  const cp_chain_params& p = kp.p;
  const int q = ew & 3, hh = ew >> 2;
  const int row = q * 32 + lane;
  const uint32_t sm_base = smem_u32(sm);
  const uint32_t bias_s = sm_base + OFF_BIAS;
  const uint32_t tbuf = sm_base + OFF_TBUF + ew * TBUF_BYTES;
  const int sw = (lane >> 1) & 3;   // SWIZZLE_64B: 16-byte chunk index ^= bits 1-2 of the row
  uint32_t st = 0, hfree = 0;
  for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x) {
    const int b = tile / kp.tiles_per_roi, n0 = (tile - b * kp.tiles_per_roi) * TILE_M;
    const int rows_valid = min(TILE_M, p.N - n0);
    const int nstages = 2 + kp.halves2;
    for (int k = 0; k < nstages; ++k, ++st) {
      const uint32_t slot = st & 1;
      const int layer = k < 2 ? k : 2;
      const cp_chain_layer& L = p.layers[layer];
      const int ncols = k < 2 ? ACC_COLS : kp.P2 * 128;                  // columns of this stage
      const int col0 = k < 2 ? 0 : (k - 2) * ACC_COLS;                   // first output column of the stage
      const uint32_t bias_l = bias_s + (uint32_t)(layer * 256 + col0) * 4;   // layers 0, 1: 256 floats each; layer 2 after them
      mbar_wait(&bars->acc_full[slot], (st >> 1) & 1);
      tc_fence_after_sync();
      if (k < 2) {   // the H buffer must be free: h1 of the previous tile (k = 0) / h0 of this tile (k = 1) consumed
        if (hfree > 0) mbar_wait(&bars->h_free, (hfree - 1) & 1);
        ++hfree;
      }
      const uint32_t tbase = tmem_base + slot * ACC_COLS + ((uint32_t)(q * 32) << 16);
      for (int c0 = hh * 32; c0 < ncols; c0 += 32 * (NUM_E_WARPS / 4)) {
        uint32_t r[32];
        tmem_ld32(tbase + (uint32_t)c0, r);
        float v[32];
        uint4 bb[8];
#pragma unroll
        for (int e4 = 0; e4 < 8; ++e4) bb[e4] = lds128(bias_l + (uint32_t)(c0 + e4 * 4) * 4);   // zero-filled without bias
        tmem_ld_wait();
#pragma unroll
        for (int e4 = 0; e4 < 8; ++e4) {
          v[e4 * 4 + 0] = __uint_as_float(r[e4 * 4 + 0]) + __uint_as_float(bb[e4].x);
          v[e4 * 4 + 1] = __uint_as_float(r[e4 * 4 + 1]) + __uint_as_float(bb[e4].y);
          v[e4 * 4 + 2] = __uint_as_float(r[e4 * 4 + 2]) + __uint_as_float(bb[e4].z);
          v[e4 * 4 + 3] = __uint_as_float(r[e4 * 4 + 3]) + __uint_as_float(bb[e4].w);
        }
        if (L.act) {
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = cp::lrelu(v[e], L.slope);
        }
        uint4 w[4];
#pragma unroll
        for (int e = 0; e < 4; ++e)
          w[e] = make_uint4(f2_to_bf2(v[e * 8], v[e * 8 + 1]), f2_to_bf2(v[e * 8 + 2], v[e * 8 + 3]),
                            f2_to_bf2(v[e * 8 + 4], v[e * 8 + 5]), f2_to_bf2(v[e * 8 + 6], v[e * 8 + 7]));
        if (k < 2) {   // next GEMM's A operand: column c -> chunk c / 64, 16-byte piece (c % 64) / 8
          const uint32_t hb = sm_base + OFF_H + (uint32_t)(c0 >> 6) * CHUNK_BYTES;
#pragma unroll
          for (int e = 0; e < 4; ++e) sts128(hb + chunk_off(row, ((c0 & 63) >> 3) + e), w[e]);
          fence_proxy_async_smem();   // generic-proxy writes of H -> visible to the tensor core's async proxy
          __syncwarp();
          if (lane == 0) mbar_arrive(&bars->h_full[c0 >> 6]);   // this warp's half of chunk c0 / 64 is in place
        } else {
          if (lane == 0) bulk_wait_read<0>();   // the warp's previous store is done reading the tile
          __syncwarp();
#pragma unroll
          for (int e = 0; e < 4; ++e) sts128(tbuf + lane * 64 + ((e ^ sw) << 4), w[e]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0 && q * 32 < rows_valid) {
            tma_store_3d(out_map, tbuf, col0 + c0, n0 + q * 32, b);
            bulk_commit();
          }
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->acc_empty[slot]);
    }
  }
  if (lane == 0) bulk_wait_read<0>();   // shared memory must outlive the last stores' reads
}

__global__ void __launch_bounds__(NTHREADS, 1) taps_chain_kernel(const __grid_constant__ TcParams kp, const __grid_constant__ CUtensorMap out_map) {
  extern __shared__ __align__(1024) uint8_t sm[];
  if ((smem_u32(sm) & 1023u) != 0) __trap();   // SWIZZLE_128B operand tiles need 1024-byte alignment
  Bars* bars = reinterpret_cast<Bars*>(sm + OFF_BAR);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < NX; ++s) {
      mbar_init(&bars->x_full[s], G_THREADS);
      mbar_init(&bars->x_empty[s], 1);
    }
    for (int s = 0; s < B_STAGES; ++s) {
      mbar_init(&bars->b_full[s], 1);
      mbar_init(&bars->b_empty[s], 1);
    }
    for (int c = 0; c < NH; ++c) mbar_init(&bars->h_full[c], 8);   // 4 lane quarters x the 2 32-column blocks of the chunk
    mbar_init(&bars->h_free, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bars->acc_full[s], 1);
      mbar_init(&bars->acc_empty[s], NUM_E_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == W_WARP) tmem_alloc(&bars->tmem_slot, 2 * ACC_COLS);
  // biases: layer 0 at [0,256), layer 1 at [256,512), layer 2 at [512, 1024); zero where a layer has none
  for (int i = threadIdx.x; i < BIAS_FLOATS; i += NTHREADS) {
    const int layer = i < 256 ? 0 : i < 512 ? 1 : 2;
    const int c = i - (layer == 2 ? 512 : layer * 256);
    const cp_chain_layer& L = kp.p.layers[layer];
    reinterpret_cast<float*>(sm + OFF_BIAS)[i] = (L.bias && c < L.nout) ? L.bias[c] : 0.f;
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = bars->tmem_slot;

  if (warp < NUM_G_WARPS) {
    gather_warps(kp, sm, bars, warp, lane);
  } else if (warp >= E_WARP0 && warp < E_WARP0 + NUM_E_WARPS) {
    epilogue_warps(kp, &out_map, sm, bars, tmem_base, warp - E_WARP0, lane);
  } else if (warp == W_WARP) {
    weight_producer(kp, sm, bars);     // whole warp, warp-uniform control flow; an elected lane issues
  } else if (warp == MMA_WARP) {
    mma_issuer(kp, sm, bars, tmem_base);
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == W_WARP) tmem_dealloc(tmem_base, 2 * ACC_COLS);
}

}  // namespace

namespace cp {

// true if the launch was taken (status in *rc); false = shape not covered, use the generic chain kernel
bool taps_chain_try(const cp_chain_params& p, cudaStream_t s, int* rc) {
  *rc = CP_OK;
  if (p.prologue != CP_PRO_TAPS || p.num_layers != 3 || p.out_mode != CP_OUT_BF16 || p.a_out) return false;
  const cp_chain_layer &L0 = p.layers[0], &L1 = p.layers[1], &L2 = p.layers[2];
  if (p.E != 64 || (p.Cg != 64 && p.Cg != 128 && p.Cg != 256) || L0.kin != 256 + p.Cg || L0.nout != 256 || L1.kin != 256 ||
      L1.nout != 256 || L2.kin != 256 || (L2.nout != 256 && L2.nout != 512) || p.ld_out < L2.nout || (p.ld_out % 8) != 0 ||
      (p.ld_gf % 8) != 0 || (reinterpret_cast<uintptr_t>(p.patches) & 15) || (reinterpret_cast<uintptr_t>(p.graph_feat) & 15) ||
      (reinterpret_cast<uintptr_t>(p.out) & 15) || (size_t)p.Hp * p.Wp * 128 >= (1ull << 31))
    return false;
  TcParams kp;
  kp.p = p;
  kp.tiles_per_roi = (p.N + TILE_M - 1) / TILE_M;
  kp.num_tiles = kp.tiles_per_roi * p.B;
  kp.KX = 4 + p.Cg / 64;
  kp.halves2 = L2.nout / 256;
  kp.P2 = 2;
  int T = 0;
  auto tile = [](const cp_chain_layer& L, int nb, int kc) { return cp::packed_tile(L.w_packed, nb, kc, L.kin, L.nout); };
  for (int c = 0; c < kp.KX; ++c)
    for (int nb = 0; nb < 2; ++nb) kp.wt[T++] = tile(L0, nb, c);
  for (int c = 0; c < NH; ++c)
    for (int nb = 0; nb < 2; ++nb) kp.wt[T++] = tile(L1, nb, c);
  for (int half = 0; half < kp.halves2; ++half)
    for (int c = 0; c < NH; ++c)
      for (int nb = 0; nb < kp.P2; ++nb) kp.wt[T++] = tile(L2, half * 2 + nb, c);
  kp.T = T;
  const int num_sms = cp::num_sms();
  const int grid = kp.num_tiles < num_sms ? kp.num_tiles : num_sms;
  cudaError_t e = cudaFuncSetAttribute(taps_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  if (e != cudaSuccess) {
    cp::set_error("cp_chain_fwd(TAPS): cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
    *rc = CP_E_CUDA;
    return true;
  }
  CUtensorMap map;
  *rc = cp::make_out_tensor_map(&map, p.out, L2.nout, p.ld_out, p.N, p.B, "cp_chain_fwd(TAPS)");
  if (*rc != CP_OK) return true;
  taps_chain_kernel<<<grid, NTHREADS, SMEM_BYTES, s>>>(kp, map);
  e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    cp::set_error("cp_chain_fwd(TAPS): CUDA error %d (%s)", (int)e, cudaGetErrorString(e));
    (void)cudaGetLastError();
    *rc = CP_E_CUDA;
  }
  return true;
}

}  // namespace cp
