// bf16 implicit-GEMM convolution on tcgen05: the image branch of the bf16 mode without a library call
// (SURVEY.md section 8f rank 1; get_gdrn_upsample_module checkerpose/model/pipeline.py:183-211, Index2Feat_module's
// patch_generator :144-145, seg_block :349,383, InitNet_GNN.conv1x1 init.py:112).
//
// Same skeleton as the split-precision kernel of the float32 mode (gemm_x3_tcgen05.cu, which runs the tensor pipe at 96 % of
// the sustained bf16 peak), with bf16 operands and ONE tcgen05.mma per K step:
//   out[m, :Nout] = act(A[m, :K] . W^T + bias),  A[m] = the kernel taps of output pixel m of an NHWC map, zero-padded  (CONV / CONVT)
// One persistent CTA of 16 warps per SM; tile = 128 rows x <= 256 output columns; K chunks of 64 channels; FOUR operand
// stages of 48 KB (A 16 KB + W 32 KB) -- an MMA chunk is only 512 clk here, so the ring has to cover the L2 latency:
//   warps 8-15  A loaders: cp.async (LDGSTS, 16 bytes, zero-fill outside the map) straight into the SWIZZLE_128B operand tile,
//               completion signalled asynchronously (cp.async.mbarrier.arrive.noinc): they never wait for their own data
//               and run up to four chunks ahead; chunk position (tap, channel slice) advanced incrementally, no division;
//   warp 0      weight producer: packed weight tiles through the TMA engine (cp.async.bulk);
//   warp 1      MMA issuer: 4 tcgen05.mma (M=128, N<=256, K=16) per chunk; tcgen05.commit releases the stage;
//   warps 4-7   epilogue: tcgen05.ld -> + bias (BatchNorm folded) -> ReLU / LeakyReLU -> bf16 -> 32 x 32 tiles (SWIZZLE_64B) -> TMA
//               tensor stores; two accumulators of 256 TMEM columns.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "sm100.cuh"

using bf16 = __nv_bfloat16;
using namespace sm100;

namespace {

constexpr int TILE_M = 128;
constexpr int BN = 256;
constexpr int NUM_WARPS = 16;
constexpr int NTHREADS = NUM_WARPS * 32;
constexpr int LOAD_WARP0 = 8, NUM_LOAD_WARPS = 8, LOAD_THREADS = NUM_LOAD_WARPS * 32;
constexpr int EPI_WARP0 = 4;
constexpr int STAGES = 4;
constexpr int A_BYTES = TILE_M * 128;
constexpr int W_BYTES = BN * 128;
constexpr int STAGE_BYTES = A_BYTES + W_BYTES;            // 48 KB
constexpr int EPI_TILE_BYTES = 32 * 64;                   // 32 rows x 32 bf16 (SWIZZLE_64B) per TMA store
constexpr int OFF_EPI = STAGES * STAGE_BYTES;             // 4 epilogue warps x 2 tiles
constexpr int OFF_BAR = OFF_EPI + 4 * 2 * EPI_TILE_BYTES;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
constexpr int TMEM_COLS = 512;
constexpr int RPT = TILE_M / (LOAD_THREADS / 8);          // rows per loader thread: 4 (8 lanes copy one 128-byte row piece)

struct Bars {
  uint64_t full[STAGES], empty[STAGES];
  uint64_t acc_full[2], acc_empty[2];
  uint32_t tmem_slot;
};

struct CvParams {
  cp_conv_bf16_params p;
  int KC, c_chunks, num_m_tiles, nblk, num_tiles, npad, tma_out;
};

// Tiles of this CTA.  MC (weight multicast over a cluster of 2 CTAs, nblk == 1): cluster c takes tile pairs (2p, 2p + 1), the
// CTA of rank r tile 2p + r; with an odd tile count the last pair's second CTA repeats the last tile (same values stored twice).
template <bool MC>
struct TileIt {
  int first, step, count, last;
  __device__ __forceinline__ explicit TileIt(const CvParams& kp) {
    last = kp.num_tiles - 1;
    if (MC) {
      const int cid = (int)blockIdx.x >> 1, ncl = (int)gridDim.x >> 1, npairs = (kp.num_tiles + 1) >> 1;
      first = 2 * cid + (int)(blockIdx.x & 1);
      step = 2 * ncl;
      count = cid < npairs ? (npairs - cid + ncl - 1) / ncl : 0;
    } else {
      first = (int)blockIdx.x;
      step = (int)gridDim.x;
      count = first < kp.num_tiles ? (kp.num_tiles - first + step - 1) / step : 0;
    }
  }
  __device__ __forceinline__ int tile(int i) const {
    const int t = first + i * step;
    return t < last ? t : last;
  }
};

// ------------------------------------------------------------------------------------------------------
// A loaders
// ------------------------------------------------------------------------------------------------------
struct RowInfo {       // per thread: its 4 rows of the current tile
  int64_t base[RPT];   // CONV: element offset of input pixel (b, oy - pad, ox - pad) (may be negative: only dereferenced for
                       // taps inside the map).  CONVT: pixel index b * H * W, -1 = beyond M
  int oyx[RPT];        // CONV / CONVT: oy | ox << 16 (CONV marks rows beyond M with 0x7fff7fff: every tap fails the bounds check)
};

__device__ __forceinline__ void rows_of_tile(const CvParams& kp, int m_tile, int tl, RowInfo& ri) {
  const cp_conv_bf16_params& p = kp.p;
#pragma unroll
  for (int i = 0; i < RPT; ++i) {
    const int64_t m = (int64_t)m_tile * TILE_M + (tl >> 3) + 32 * i;
    ri.oyx[i] = 0;
    if (m >= p.M) {
      ri.base[i] = -1;
      ri.oyx[i] = 0x7fff7fff;
    } else {
      const int hw = p.Ho * p.Wo;
      const int64_t b = m / hw;
      const int rem = (int)(m - b * hw);
      const int oy = rem / p.Wo, ox = rem - oy * p.Wo;
      ri.oyx[i] = oy | (ox << 16);
      ri.base[i] = p.mode == CP_X3_CONV ? ((b * p.H + (oy - p.pad)) * p.W + (ox - p.pad)) * p.k1 : b * p.H * p.W;
    }
  }
}

struct ChunkPos {
  int ky, kx, cc;
  __device__ __forceinline__ void reset() { ky = kx = cc = 0; }
  __device__ __forceinline__ void next(int c_chunks, int KW) {
    if (++cc == c_chunks) {
      cc = 0;
      if (++kx == KW) { kx = 0; ++ky; }
    }
  }
};

template <bool MC>
__device__ void a_loader(const CvParams& kp, uint8_t* sm, Bars* bars, int tl) {
  const cp_conv_bf16_params& p = kp.p;
  const int piece = tl & 7;
  const uint32_t sm_base = smem_u32(sm);
  const bf16* a1 = reinterpret_cast<const bf16*>(p.a1);
  RowInfo ri;
  ChunkPos pos;
  uint32_t it = 0;
  const TileIt<MC> tiles(kp);
  for (int ti = 0; ti < tiles.count; ++ti) {
    const int tile = tiles.tile(ti);
    rows_of_tile(kp, tile / kp.nblk, tl, ri);
    pos.reset();
    for (int kc = 0; kc < kp.KC; ++kc, ++it) {
      const uint32_t s = it % STAGES;
      if (it >= STAGES) mbar_wait(&bars->empty[s], ((it / STAGES) - 1) & 1);
      const uint32_t a_s = sm_base + s * STAGE_BYTES;
      if (p.mode == CP_X3_CONV) {
        const int dy = pos.ky - p.pad, dx = pos.kx - p.pad;
        const bf16* src = a1 + ((int64_t)pos.ky * p.W + pos.kx) * p.k1 + pos.cc * 64 + piece * 8;
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
          const int r = (tl >> 3) + 32 * i;
          const int iy = (ri.oyx[i] & 0xffff) + dy, ix = (ri.oyx[i] >> 16) + dx;
          const bool ok = (unsigned)iy < (unsigned)p.H && (unsigned)ix < (unsigned)p.W;
          cp_async16_zfill(a_s + r * 128 + ((piece ^ (r & 7)) << 4), ok ? src + ri.base[i] : a1, ok ? 16u : 0u);
        }
      } else {   // transposed convolution, stride 2
        const bf16* src = a1 + pos.cc * 64 + piece * 8;
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
          const int r = (tl >> 3) + 32 * i;
          const int ty = (ri.oyx[i] & 0xffff) + p.pad - pos.ky, tx = (ri.oyx[i] >> 16) + p.pad - pos.kx;
          const int iy = ty >> 1, ix = tx >> 1;
          const bool ok = ri.base[i] >= 0 && ((ty | tx) & 1) == 0 && ty >= 0 && tx >= 0 && iy < p.H && ix < p.W;
          cp_async16_zfill(a_s + r * 128 + ((piece ^ (r & 7)) << 4), ok ? src + (ri.base[i] + (int64_t)iy * p.W + ix) * p.k1 : a1, ok ? 16u : 0u);
        }
      }
      cp_async_arrive_noinc(&bars->full[s]);     // fires when this thread's copies have landed
      pos.next(kp.c_chunks, p.KW);
    }
  }
}

// ------------------------------------------------------------------------------------------------------
template <bool MC>
__device__ void weight_producer(const CvParams& kp, uint8_t* sm, Bars* bars) {
  const cp_conv_bf16_params& p = kp.p;
  const uint8_t* wb = reinterpret_cast<const uint8_t*>(p.w_packed);
  uint32_t it = 0;
  const TileIt<MC> tiles(kp);
  for (int ti = 0; ti < tiles.count; ++ti) {
    const int tile = tiles.tile(ti);
    const int nb = tile % kp.nblk;
    const int col0 = nb * BN;
    const int cols = min(BN, kp.npad - col0);
    const int rows0 = min(128, cols), rows1 = cols - rows0;
    for (int kc = 0; kc < kp.KC; ++kc, ++it) {
      const uint32_t s = it % STAGES;
      if (it >= STAGES) mbar_wait(&bars->empty[s], ((it / STAGES) - 1) & 1);
      if (MC) {
        // both CTAs of the cluster consume the same weight tile (nblk == 1): each fetches HALF of its rows from L2 and
        // multicasts them into both CTAs' stage s; every CTA's barrier expects the whole tile
        if (elect_one()) {
          uint8_t* w_s = sm + s * STAGE_BYTES + A_BYTES;
          const uint32_t half = (uint32_t)(cols / 2) * 128u, rank = blockIdx.x & 1;
          mbar_arrive_expect_tx(&bars->full[s], (uint32_t)cols * 128u);
          const uint8_t* src = cols == 256 ? wb + cp::packed_tile_offset(rank, kc, 128, p.K)                 // packed 128-row block `rank`
                                           : wb + cp::packed_tile_offset(0, kc, cols, p.K) + (size_t)rank * half;   // half of the single block
          bulk_g2s_multicast(w_s + rank * half, src, half, &bars->full[s], (uint16_t)3);
        }
        __syncwarp();
        continue;
      }
      if (elect_one()) {
        uint8_t* w_s = sm + s * STAGE_BYTES + A_BYTES;
        mbar_arrive_expect_tx(&bars->full[s], (uint32_t)cols * 128u);
        bulk_g2s(w_s, wb + cp::packed_tile_offset(col0 / 128, kc, rows0, p.K), (uint32_t)rows0 * 128u, &bars->full[s]);
        if (rows1 > 0)
          bulk_g2s(w_s + 128 * 128, wb + cp::packed_tile_offset(col0 / 128 + 1, kc, rows1, p.K), (uint32_t)rows1 * 128u, &bars->full[s]);
      }
      __syncwarp();
    }
  }
}

template <bool MC>
__device__ void mma_issuer(const CvParams& kp, uint8_t* sm, Bars* bars, uint32_t tmem_base) {
  const uint32_t sm_base = smem_u32(sm);
  uint32_t it = 0, tcount = 0;
  const TileIt<MC> tiles(kp);
  for (int ti = 0; ti < tiles.count; ++ti, ++tcount) {
    const int tile = tiles.tile(ti);
    const int nb = tile % kp.nblk;
    const int cols = min(BN, kp.npad - nb * BN);
    const uint32_t idesc = make_idesc_bf16_m128((uint32_t)cols);
    const uint32_t slot = tcount & 1;
    if (tcount >= 2) mbar_wait(&bars->acc_empty[slot], ((tcount >> 1) - 1) & 1);
    const uint32_t d = tmem_base + slot * BN;
    for (int kc = 0; kc < kp.KC; ++kc, ++it) {
      const uint32_t s = it % STAGES;
      mbar_wait(&bars->full[s], (it / STAGES) & 1);
      tc_fence_after_sync();
      const uint32_t a_lo = smem_desc_lo(sm_base + s * STAGE_BYTES), w_lo = a_lo + (A_BYTES >> 4);
      if (elect_one()) {
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) mma_bf16_ss_lo(d, a_lo + 2 * k, w_lo + 2 * k, idesc, (uint32_t)((kc | (int)k) != 0));
        if (MC) mma_commit_multicast(&bars->empty[s], (uint16_t)3);   // stage s is refilled (by either CTA) only when BOTH have consumed it
        else mma_commit(&bars->empty[s]);
        if (kc == kp.KC - 1) mma_commit(&bars->acc_full[slot]);
      }
      __syncwarp();
    }
  }
}

template <bool MC>
__device__ void epilogue(const CvParams& kp, const CUtensorMap* out_map, uint8_t* sm, Bars* bars, uint32_t tmem_base, int q, int lane) {
  const cp_conv_bf16_params& p = kp.p;
  const bool bias_vec = p.bias && (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0;
  const uint32_t tbuf0 = smem_u32(sm) + OFF_EPI + q * 2 * EPI_TILE_BYTES;
  const int sw = (lane >> 1) & 3;      // SWIZZLE_64B: 16-byte chunk index ^= bits 1-2 of the row
  bf16* out = reinterpret_cast<bf16*>(p.out);
  uint32_t tcount = 0, nstore = 0;
  const TileIt<MC> tiles(kp);
  for (int ti = 0; ti < tiles.count; ++ti, ++tcount) {
    const int tile = tiles.tile(ti);
    const int m_tile = tile / kp.nblk, nb = tile - m_tile * kp.nblk;
    const int col0 = nb * BN;
    const int cols = min(BN, kp.npad - col0);
    const uint32_t slot = tcount & 1;
    while (!mbar_try_wait(&bars->acc_full[slot], (tcount >> 1) & 1)) __nanosleep(64);   // idle for a whole K loop: do not spin
    tc_fence_after_sync();
    const int64_t row0 = (int64_t)m_tile * TILE_M + q * 32;
    const int64_t row = row0 + lane;
    const bool row_ok = row < p.M;
    const uint32_t tb = tmem_base + ((uint32_t)(q * 32) << 16) + slot * BN;
    for (int c0 = 0; c0 < cols; c0 += 32) {
      const int n0 = col0 + c0;
      if (n0 >= p.Nout) break;
      uint32_t r[32];
      tmem_ld32(tb + (uint32_t)c0, r);
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
      float v[32];
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const float x = __uint_as_float(r[e]) + bv[e];
        v[e] = p.act ? cp::lrelu(x, p.slope) : x;
      }
      if (kp.tma_out) {
        const uint32_t tbuf = tbuf0 + (nstore & 1) * EPI_TILE_BYTES;
        ++nstore;
        if (lane == 0) bulk_wait_read<1>();
        __syncwarp();
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const uint4 w = make_uint4(f2_to_bf2(v[e * 8], v[e * 8 + 1]), f2_to_bf2(v[e * 8 + 2], v[e * 8 + 3]),
                                     f2_to_bf2(v[e * 8 + 4], v[e * 8 + 5]), f2_to_bf2(v[e * 8 + 6], v[e * 8 + 7]));
          sts128(tbuf + lane * 64 + ((e ^ sw) << 4), w);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && row0 < p.M) {
          tma_store_3d(out_map, tbuf, n0, (int)row0, 0);
          bulk_commit();
        }
      } else if (row_ok) {
        bf16* orow = out + row * p.ld_out;
#pragma unroll
        for (int e = 0; e < 32; ++e)
          if (n0 + e < p.Nout) orow[n0 + e] = __float2bfloat16_rn(v[e]);
      }
    }
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(&bars->acc_empty[slot]);
  }
  if (kp.tma_out && lane == 0) bulk_wait_read<0>();
}

template <bool MC>
__global__ void __launch_bounds__(NTHREADS, 1) conv_bf16_kernel(const __grid_constant__ CvParams kp, const __grid_constant__ CUtensorMap out_map) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  Bars* bars = reinterpret_cast<Bars*>(sm + OFF_BAR);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&bars->full[s], 1 + LOAD_THREADS);     // weight producer (with the byte count) + every loader thread (asynchronously)
      mbar_init(&bars->empty[s], MC ? 2 : 1);          // multicast: the MMA streams of both CTAs
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&bars->acc_full[a], 1);
      mbar_init(&bars->acc_empty[a], 4);
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(&bars->tmem_slot, TMEM_COLS);
  tc_fence_before_sync();
  if (MC) cluster_sync_all();     // the peer's barriers exist before its multicast copies / commits arrive
  else __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = bars->tmem_slot;

  if (warp >= LOAD_WARP0) a_loader<MC>(kp, sm, bars, threadIdx.x - LOAD_WARP0 * 32);
  else if (warp >= EPI_WARP0) epilogue<MC>(kp, &out_map, sm, bars, tmem_base, warp - EPI_WARP0, lane);
  else if (warp == 0) weight_producer<MC>(kp, sm, bars);
  else if (warp == 1) mma_issuer<MC>(kp, sm, bars, tmem_base);

  tc_fence_before_sync();
  if (MC) cluster_sync_all();     // no CTA leaves while the peer may still write into / arrive on its shared memory
  else __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

}  // namespace

extern "C" int cp_conv_bf16(const cp_conv_bf16_params* pp, cp_stream_t s) {
  CP_REQUIRE(pp, CP_E_INVALID, "cp_conv_bf16: null params");
  const cp_conv_bf16_params& p = *pp;
  CP_REQUIRE(p.a1 && p.w_packed && p.out && p.M > 0 && p.Nout > 0 && p.K > 0, CP_E_INVALID, "cp_conv_bf16: bad arguments");
  CP_REQUIRE(p.K % 64 == 0 && (reinterpret_cast<uintptr_t>(p.w_packed) & 15) == 0 && p.ld_out >= p.Nout, CP_E_UNSUPPORTED,
             "cp_conv_bf16: K=%d must be a multiple of 64, weights 16-byte aligned, ld_out >= Nout", p.K);
  CvParams kp;
  kp.p = p;
  CP_REQUIRE(p.mode == CP_X3_CONV || p.mode == CP_X3_CONVT, CP_E_INVALID, "cp_conv_bf16: bad mode %d", p.mode);
  CP_REQUIRE(p.k1 > 0 && p.k1 % 64 == 0 && p.KH > 0 && p.KW > 0 && p.KH * p.KW * p.k1 == p.K, CP_E_UNSUPPORTED,
             "cp_conv_bf16: conv needs Cin %% 64 == 0 and K == KH*KW*Cin (Cin=%d KH=%d KW=%d K=%d)", p.k1, p.KH, p.KW, p.K);
  CP_REQUIRE(p.H > 0 && p.W > 0 && p.Ho > 0 && p.Wo > 0 && p.Ho < 32768 && p.Wo < 32768 && p.pad >= 0 && p.M % ((int64_t)p.Ho * p.Wo) == 0 &&
             (reinterpret_cast<uintptr_t>(p.a1) & 15) == 0, CP_E_INVALID, "cp_conv_bf16: bad map sizes H=%d W=%d Ho=%d Wo=%d", p.H, p.W, p.Ho, p.Wo);
  kp.c_chunks = p.k1 / 64;
  kp.KC = p.K / 64;
  kp.npad = (p.Nout + 15) / 16 * 16;
  kp.nblk = (kp.npad + BN - 1) / BN;
  CP_REQUIRE(p.M < (1ll << 31) && (p.M + TILE_M - 1) / TILE_M * kp.nblk < (1ll << 31), CP_E_UNSUPPORTED, "cp_conv_bf16: too many rows / tiles");
  kp.num_m_tiles = (int)((p.M + TILE_M - 1) / TILE_M);
  kp.num_tiles = kp.num_m_tiles * kp.nblk;
  CUtensorMap map;
  memset(&map, 0, sizeof(map));
  kp.tma_out = ((p.ld_out & 7) == 0 && p.Nout % 32 == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0) ? 1 : 0;
  if (kp.tma_out) {
    const int rc = cp::make_out_tensor_map(&map, p.out, p.Nout, p.ld_out, (int)p.M, 1, "cp_conv_bf16");
    if (rc != CP_OK) return rc;
  }
  const int num_sms = cp::num_sms();
  // weight multicast over clusters of 2 CTAs when every tile uses the same weight tile sequence (one column block) and its
  // halves are whole swizzle atoms; CP_CONV_MULTICAST=0 forces the single-CTA kernel (A/B measurements)
  const char* mc_env = getenv("CP_CONV_MULTICAST");
  const bool mc = !(mc_env && mc_env[0] == '0') && kp.nblk == 1 && kp.num_tiles >= 2 && (kp.npad == 256 || kp.npad <= 128);
  cudaError_t e;
  if (!mc) {
    const int grid = kp.num_tiles < num_sms ? kp.num_tiles : num_sms;
    e = cudaFuncSetAttribute(conv_bf16_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "cp_conv_bf16: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
    conv_bf16_kernel<false><<<grid, NTHREADS, SMEM_BYTES, (cudaStream_t)s>>>(kp, map);
  } else {
    const int want = 2 * ((kp.num_tiles + 1) / 2);
    const int grid = want < (num_sms & ~1) ? want : (num_sms & ~1);
    e = cudaFuncSetAttribute(conv_bf16_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "cp_conv_bf16: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(NTHREADS);
    cfg.dynamicSmemBytes = SMEM_BYTES;
    cfg.stream = (cudaStream_t)s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, conv_bf16_kernel<true>, kp, map);
    CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "cp_conv_bf16: cluster launch failed: %s", cudaGetErrorString(e));
  }
  CP_CHECK_LAUNCH("cp_conv_bf16");
  return CP_OK;
}
