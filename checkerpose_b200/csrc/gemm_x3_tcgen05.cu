// Split-precision tensor-core GEMM / implicit-GEMM convolution: the float32 mode of the head on tcgen05.
//
// The reference is fp32 end to end and north_star asks for decoded codes that match it on >= 99.9 % of keypoints;
// one bf16 rounding per tensor is ~100x too coarse for 13 cascaded sign tests (DESIGN.md section 6), and the
// SIMT FFMA GEMM (cp_linear_f32) left the tensor cores idle.  Here every fp32 operand x is split on the fly into
// two bf16 values  x = hi + lo + O(2^-17 |x|)  and the product is taken as
//     a . w  ~=  a_hi . w_hi  +  a_hi . w_lo  +  a_lo . w_hi            (three tcgen05.mma, fp32 accumulation in TMEM)
// -- relative error ~2^-16 per product, storage between layers stays fp32.  The same kernel is
//   * Linear(+bias+LeakyReLU) on node-major fp32 rows, with an optional second operand [a1 | a2] (the concat of
//     pipeline.py:283)                                                           -> replaces cp_linear_f32;
//   * Conv2d k x k (stride 1, zero padding) / ConvTranspose2d (stride 2) over an NHWC fp32 map as an IMPLICIT GEMM:
//     the A tile of a K chunk is the 64-channel slice of one kernel tap of 128 output pixels, gathered (zero-filled
//     outside the map) by the same loader warps -- the image branch of the float32 mode (pipeline.py:183-211, 144-145).
//
// One persistent CTA of 16 warps per SM; tile = 128 rows x up to 256 output columns; K chunks of 64:
//   warps 8-15  A loaders: ld.global fp32 (next chunk's loads in flight while this one is converted) -> hi / lo bf16 ->
//               two SWIZZLE_128B K-major operand tiles in shared memory;
//   warp 0      weight producer: packed hi / lo weight tiles (cp_pack_weight_split) through the TMA engine (cp.async.bulk);
//   warp 1      MMA issuer: 3 x 4 tcgen05.mma (M=128, N<=256, K=16) per chunk, tcgen05.commit releases the stage;
//   warps 4-7   epilogue: tcgen05.ld -> + bias -> LeakyReLU / ReLU -> 32 x 32 fp32 tiles in shared memory -> TMA tensor stores
//               (1.27 -> 0.57 ms for 1M x 256 -> 256: per-thread row stores kept the epilogue, not the MMAs, on the critical path);
// two stages of operands (96 KB each), two accumulators of 256 TMEM columns (the epilogue of tile i overlaps the MMAs
// of tile i + 1).
#include <cuda.h>
#include <string.h>

#include "common.cuh"
#include "sm100.cuh"

using bf16 = __nv_bfloat16;
using namespace sm100;

namespace {

constexpr int TILE_M = 128;
constexpr int BN = 256;                        // output columns per tile pass
constexpr int NUM_WARPS = 16;
constexpr int NTHREADS = NUM_WARPS * 32;
constexpr int LOAD_WARP0 = 8, NUM_LOAD_WARPS = 8;
constexpr int EPI_WARP0 = 4;
constexpr int STAGES = 2;
constexpr int A_BYTES = TILE_M * 128;          // one 64-wide bf16 K chunk of 128 rows
constexpr int W_BYTES = BN * 128;
constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * W_BYTES;   // A_hi, A_lo, W_hi, W_lo
constexpr int EPI_TILE_BYTES = 32 * 128;                 // 32 rows x 32 fp32 (SWIZZLE_128B) per TMA store
constexpr int OFF_EPI = STAGES * STAGE_BYTES;            // 4 epilogue warps x 2 tiles
constexpr int OFF_BAR = OFF_EPI + 4 * 2 * EPI_TILE_BYTES;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;         // + alignment slack
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
constexpr int TMEM_COLS = 512;

struct Bars {
  uint64_t full[STAGES], empty[STAGES];
  uint64_t acc_full[2], acc_empty[2];
  uint32_t tmem_slot;
};

struct X3Params {
  cp_gemm_x3_params p;
  int KC;            // K chunks of 64
  int c_chunks;      // conv: 64-channel chunks per tap (Cin / 64)
  int num_m_tiles, nblk, num_tiles;
  int npad;
  int tma_out;       // the epilogue leaves through TMA tensor stores (ld_out % 4 == 0, Nout % 4 == 0, 16-byte aligned base)
};

__device__ __forceinline__ float bf_round(float a) { return __bfloat162float(__float2bfloat16_rn(a)); }

__device__ __forceinline__ void sts64(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}

// ------------------------------------------------------------------------------------------------------
// A loaders
// ------------------------------------------------------------------------------------------------------
constexpr int RPT = TILE_M / (NUM_LOAD_WARPS * 2);   // rows per thread: 8 (a warp instruction covers 2 rows x 16 float4)

struct RowInfo {       // per thread: its 8 rows of the current tile
  int64_t base[RPT];   // LINEAR: row index.  CONV: element offset of input pixel (b, oy - pad, ox - pad), channel 0 (may lie outside
                       // the map, even negative: only dereferenced for taps that land inside).  CONVT: pixel index b * H * W.
                       // LINEAR / CONVT: -1 = row beyond M (CONV marks those rows in oyx)
  int oyx[RPT];        // CONV / CONVT: oy | ox << 16
};

__device__ __forceinline__ void rows_of_tile(const X3Params& kp, int m_tile, int lw, int lane, RowInfo& ri) {
  const cp_gemm_x3_params& p = kp.p;
#pragma unroll
  for (int i = 0; i < RPT; ++i) {
    const int64_t m = (int64_t)m_tile * TILE_M + lw * 16 + i * 2 + (lane >> 4);
    ri.oyx[i] = 0;
    if (m >= p.M) {
      ri.base[i] = -1;
      ri.oyx[i] = 0x7fff7fff;      // CONV: every tap of such a row fails the bounds check (its base may be negative for real rows too)
    } else if (p.mode == CP_X3_LINEAR) {
      ri.base[i] = m;
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

// Position of a K chunk inside the reduction: LINEAR = which operand and column; CONV / CONVT = kernel tap and 64-channel
// slice.  Advanced incrementally (no division per chunk: the loader warps are issue-bound on exactly this arithmetic --
// ncu r02: 1150 warp instructions per loader warp and chunk with the division per row, 22 % of all samples).
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

// this thread's float4 of its 8 rows for the chunk at `cp` (LINEAR: chunk index kc); zero fill outside the matrix / the map
__device__ __forceinline__ void load_chunk(const X3Params& kp, const RowInfo& ri, const ChunkPos& cp, int kc, int c4, float4 (&v)[RPT]) {
  const cp_gemm_x3_params& p = kp.p;
  if (p.mode == CP_X3_LINEAR) {
    const int k = kc * 64 + c4 * 4;
    const bool first = k < p.k1;
    const float* src = first ? p.a1 + k : p.a2 + (k - p.k1);
    const int64_t ld = first ? p.ld1 : p.ld2;
#pragma unroll
    for (int i = 0; i < RPT; ++i)
      v[i] = ri.base[i] >= 0 ? __ldg(reinterpret_cast<const float4*>(src + ri.base[i] * ld)) : make_float4(0.f, 0.f, 0.f, 0.f);
  } else if (p.mode == CP_X3_CONV) {
    const int dy = cp.ky - p.pad, dx = cp.kx - p.pad;
    const float* src = p.a1 + ((int64_t)cp.ky * p.W + cp.kx) * p.k1 + cp.cc * 64 + c4 * 4;   // + base[i] = pixel (oy + dy, ox + dx)
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
      const int iy = (ri.oyx[i] & 0xffff) + dy, ix = (ri.oyx[i] >> 16) + dx;
      const bool ok = (unsigned)iy < (unsigned)p.H && (unsigned)ix < (unsigned)p.W;
      v[i] = ok ? __ldg(reinterpret_cast<const float4*>(src + ri.base[i])) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  } else {   // transposed convolution, stride 2: out[oy] += in[iy] * w[ky] with oy = 2 iy - pad + ky
    const float* src = p.a1 + cp.cc * 64 + c4 * 4;
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
      const int ty = (ri.oyx[i] & 0xffff) + p.pad - cp.ky, tx = (ri.oyx[i] >> 16) + p.pad - cp.kx;
      const int iy = ty >> 1, ix = tx >> 1;
      const bool ok = ri.base[i] >= 0 && ((ty | tx) & 1) == 0 && ty >= 0 && tx >= 0 && iy < p.H && ix < p.W;
      v[i] = ok ? __ldg(reinterpret_cast<const float4*>(src + (ri.base[i] + (int64_t)iy * p.W + ix) * p.k1)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
}

__device__ void a_loader(const X3Params& kp, uint8_t* sm, Bars* bars, int lw, int lane) {
  const int c4 = lane & 15;                  // float4 index inside the 64-wide chunk
  const uint32_t sm_base = smem_u32(sm);
  RowInfo ri;
  float4 cur[RPT], nxt[RPT];
  ChunkPos pos;                              // position of the chunk being PREFETCHED
  uint32_t it = 0;                           // chunk counter over all tiles of this CTA
  for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x) {
    const int m_tile = tile / kp.nblk;
    rows_of_tile(kp, m_tile, lw, lane, ri);
    pos.reset();
    load_chunk(kp, ri, pos, 0, c4, cur);
    for (int kc = 0; kc < kp.KC; ++kc, ++it) {
      if (kc + 1 < kp.KC) {                  // next chunk's loads in flight while this one is converted
        pos.next(kp.c_chunks, kp.p.KW);
        load_chunk(kp, ri, pos, kc + 1, c4, nxt);
      }
      const uint32_t s = it % STAGES;
      if (it >= STAGES) mbar_wait(&bars->empty[s], ((it / STAGES) - 1) & 1);
      const uint32_t a_hi = sm_base + s * STAGE_BYTES, a_lo = a_hi + A_BYTES;
#pragma unroll
      for (int i = 0; i < RPT; ++i) {
        const int r = lw * 16 + i * 2 + (lane >> 4);
        const float4 v = cur[i];
        const float hx = bf_round(v.x), hy = bf_round(v.y), hz = bf_round(v.z), hw = bf_round(v.w);
        const uint32_t off = (uint32_t)(r * 128 + (((c4 >> 1) ^ (r & 7)) << 4) + (c4 & 1) * 8);
        sts64(a_hi + off, f2_to_bf2(hx, hy), f2_to_bf2(hz, hw));
        sts64(a_lo + off, f2_to_bf2(v.x - hx, v.y - hy), f2_to_bf2(v.z - hz, v.w - hw));
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->full[s]);
      if (kc + 1 < kp.KC) {
#pragma unroll
        for (int i = 0; i < RPT; ++i) cur[i] = nxt[i];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------
__device__ void weight_producer(const X3Params& kp, uint8_t* sm, Bars* bars) {
  const cp_gemm_x3_params& p = kp.p;
  uint32_t it = 0;
  for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x) {
    const int nb = tile % kp.nblk;
    const int col0 = nb * BN;
    const int cols = min(BN, kp.npad - col0);                 // multiple of 16
    const int rows0 = min(128, cols), rows1 = cols - rows0;    // the two packed 128-row blocks of this pass
    for (int kc = 0; kc < kp.KC; ++kc, ++it) {
      const uint32_t s = it % STAGES;
      if (it >= STAGES) mbar_wait(&bars->empty[s], ((it / STAGES) - 1) & 1);
      if (elect_one()) {
        uint8_t* w_hi = sm + s * STAGE_BYTES + 2 * A_BYTES;
        uint8_t* w_lo = w_hi + W_BYTES;
        mbar_arrive_expect_tx(&bars->full[s], (uint32_t)cols * 128u * 2u);
        const size_t o0 = cp::packed_tile_offset(col0 / 128, kc, rows0, p.K);
        bulk_g2s(w_hi, reinterpret_cast<const uint8_t*>(p.w_hi) + o0, (uint32_t)rows0 * 128u, &bars->full[s]);
        bulk_g2s(w_lo, reinterpret_cast<const uint8_t*>(p.w_lo) + o0, (uint32_t)rows0 * 128u, &bars->full[s]);
        if (rows1 > 0) {
          const size_t o1 = cp::packed_tile_offset(col0 / 128 + 1, kc, rows1, p.K);
          bulk_g2s(w_hi + 128 * 128, reinterpret_cast<const uint8_t*>(p.w_hi) + o1, (uint32_t)rows1 * 128u, &bars->full[s]);
          bulk_g2s(w_lo + 128 * 128, reinterpret_cast<const uint8_t*>(p.w_lo) + o1, (uint32_t)rows1 * 128u, &bars->full[s]);
        }
      }
      __syncwarp();
    }
  }
}

__device__ void mma_issuer(const X3Params& kp, uint8_t* sm, Bars* bars, uint32_t tmem_base) {
  const uint32_t sm_base = smem_u32(sm);
  uint32_t it = 0, tcount = 0;
  for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x, ++tcount) {
    const int nb = tile % kp.nblk;
    const int cols = min(BN, kp.npad - nb * BN);
    const uint32_t idesc = make_idesc_bf16_m128((uint32_t)cols);
    const uint32_t slot = tcount & 1;
    if (tcount >= 2) mbar_wait(&bars->acc_empty[slot], ((tcount >> 1) - 1) & 1);   // the epilogue drained this accumulator
    const uint32_t d = tmem_base + slot * BN;
    for (int kc = 0; kc < kp.KC; ++kc, ++it) {
      const uint32_t s = it % STAGES;
      mbar_wait(&bars->full[s], (it / STAGES) & 1);
      tc_fence_after_sync();
      const uint32_t a_hi = smem_desc_lo(sm_base + s * STAGE_BYTES), a_lo = a_hi + (A_BYTES >> 4);
      const uint32_t w_hi = a_hi + (2 * A_BYTES >> 4), w_lo = w_hi + (W_BYTES >> 4);
      if (elect_one()) {
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) {
          mma_bf16_ss_lo(d, a_hi + 2 * k, w_hi + 2 * k, idesc, (uint32_t)((kc | (int)k) != 0));
          mma_bf16_ss_lo(d, a_hi + 2 * k, w_lo + 2 * k, idesc, 1u);
          mma_bf16_ss_lo(d, a_lo + 2 * k, w_hi + 2 * k, idesc, 1u);
        }
        mma_commit(&bars->empty[s]);
        if (kc == kp.KC - 1) mma_commit(&bars->acc_full[slot]);
      }
      __syncwarp();
    }
  }
}

// warp q drains TMEM lanes [32 q, 32 q + 32): 32 columns at a time -> + bias -> activation -> a 32 x 32 fp32 tile in shared
// memory (SWIZZLE_128B) -> one TMA tensor store (full 128-byte rows; rows beyond M / columns beyond Nout are clipped by the
// tensor map).  Outputs whose rows are not 16-byte aligned (the 7 / 2 / 13 logits) are stored directly.
__device__ void epilogue(const X3Params& kp, const CUtensorMap* out_map, uint8_t* sm, Bars* bars, uint32_t tmem_base, int q, int lane) {
  const cp_gemm_x3_params& p = kp.p;
  const bool bias_vec = p.bias && (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0;
  const uint32_t tbuf0 = smem_u32(sm) + OFF_EPI + q * 2 * EPI_TILE_BYTES;
  uint32_t tcount = 0, nstore = 0;
  for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x, ++tcount) {
    const int m_tile = tile / kp.nblk, nb = tile - m_tile * kp.nblk;
    const int col0 = nb * BN;
    const int cols = min(BN, kp.npad - col0);
    const uint32_t slot = tcount & 1;
    // the epilogue warps share their schedulers with the loader warps and idle for a whole K loop (36-72 chunks of a
    // convolution): back off instead of spinning on the barrier (their spin was 22 % of all issue samples, ncu r02)
    while (!mbar_try_wait(&bars->acc_full[slot], (tcount >> 1) & 1)) __nanosleep(128);
    tc_fence_after_sync();
    const int64_t row0 = (int64_t)m_tile * TILE_M + q * 32;
    const int64_t row = row0 + lane;
    const bool row_ok = row < p.M;
    float* orow = p.out + (row_ok ? row : 0) * p.ld_out;
    const uint32_t tb = tmem_base + ((uint32_t)(q * 32) << 16) + slot * BN;
    for (int c0 = 0; c0 < cols; c0 += 32) {
      const int n0 = col0 + c0;
      if (n0 >= p.Nout) break;
      uint32_t r[32];
      tmem_ld32(tb + (uint32_t)c0, r);      // columns beyond `cols` hold stale data and are never stored
      float bv[32];
      if (bias_vec && n0 + 32 <= p.Nout) {  // the bias loads fly while the TMEM read does
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
        if (lane == 0) bulk_wait_read<1>();   // the store that last used this tile has read it
        __syncwarp();
#pragma unroll
        for (int e4 = 0; e4 < 8; ++e4)
          sts128(tbuf + lane * 128 + ((e4 ^ (lane & 7)) << 4), v[e4 * 4], v[e4 * 4 + 1], v[e4 * 4 + 2], v[e4 * 4 + 3]);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && row0 < p.M) {
          tma_store_2d(out_map, tbuf, n0, (int)row0);
          bulk_commit();
        }
      } else if (row_ok) {
#pragma unroll
        for (int e = 0; e < 32; ++e)
          if (n0 + e < p.Nout) orow[n0 + e] = v[e];
      }
    }
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(&bars->acc_empty[slot]);
  }
  if (kp.tma_out && lane == 0) bulk_wait_read<0>();   // shared memory outlives the last stores' reads
}

__global__ void __launch_bounds__(NTHREADS, 1) gemm_x3_kernel(const __grid_constant__ X3Params kp, const __grid_constant__ CUtensorMap out_map) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  Bars* bars = reinterpret_cast<Bars*>(sm + OFF_BAR);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&bars->full[s], 1 + NUM_LOAD_WARPS);   // weight producer (with the byte count) + every loader warp
      mbar_init(&bars->empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&bars->acc_full[a], 1);
      mbar_init(&bars->acc_empty[a], 4);
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(&bars->tmem_slot, TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = bars->tmem_slot;

  if (warp >= LOAD_WARP0) a_loader(kp, sm, bars, warp - LOAD_WARP0, lane);
  else if (warp >= EPI_WARP0) epilogue(kp, &out_map, sm, bars, tmem_base, warp - EPI_WARP0, lane);
  else if (warp == 0) weight_producer(kp, sm, bars);
  else if (warp == 1) mma_issuer(kp, sm, bars, tmem_base);

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

__global__ void pack_weight_split_kernel(const float* __restrict__ w, int Nout, int K, int Npad, bf16* __restrict__ hi, bf16* __restrict__ lo) {
  const int64_t total = (int64_t)Npad * K;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(e / K), k = (int)(e - (int64_t)n * K);
    const int nb = n >> 7, r = n & 127, kk = k & 63;
    const size_t off = cp::packed_tile_offset(nb, k >> 6, cp::packed_block_rows(nb, Npad), K) / 2 + (size_t)r * 64 + (size_t)(((kk >> 3) ^ (r & 7)) << 3) + (kk & 7);
    const float v = (n < Nout) ? w[(size_t)n * K + k] : 0.f;
    const bf16 h = __float2bfloat16_rn(v);
    hi[off] = h;
    lo[off] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

}  // namespace

extern "C" int cp_pack_weight_split(const float* w, int Nout, int K, void* packed_hi, void* packed_lo, cp_stream_t s) {
  CP_REQUIRE(w && packed_hi && packed_lo && Nout > 0 && K > 0, CP_E_INVALID, "cp_pack_weight_split: bad arguments");
  CP_REQUIRE(K % 64 == 0, CP_E_UNSUPPORTED, "cp_pack_weight_split: K=%d must be a multiple of 64", K);
  const int npad = (Nout + 15) / 16 * 16;
  const int64_t total = (int64_t)npad * K;
  const int grid = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  pack_weight_split_kernel<<<grid, 256, 0, (cudaStream_t)s>>>(w, Nout, K, npad, (bf16*)packed_hi, (bf16*)packed_lo);
  CP_CHECK_LAUNCH("cp_pack_weight_split");
  return CP_OK;
}

extern "C" int cp_gemm_x3(const cp_gemm_x3_params* pp, cp_stream_t s) {
  CP_REQUIRE(pp, CP_E_INVALID, "cp_gemm_x3: null params");
  const cp_gemm_x3_params& p = *pp;
  CP_REQUIRE(p.a1 && p.w_hi && p.w_lo && p.out && p.M > 0 && p.Nout > 0 && p.K > 0, CP_E_INVALID, "cp_gemm_x3: bad arguments");
  CP_REQUIRE(p.K % 64 == 0, CP_E_UNSUPPORTED, "cp_gemm_x3: K=%d must be a multiple of 64", p.K);
  CP_REQUIRE(((reinterpret_cast<uintptr_t>(p.w_hi) | reinterpret_cast<uintptr_t>(p.w_lo)) & 15) == 0, CP_E_INVALID, "cp_gemm_x3: weights not 16-byte aligned");
  CP_REQUIRE(p.ld_out >= p.Nout, CP_E_INVALID, "cp_gemm_x3: ld_out=%d < Nout=%d", p.ld_out, p.Nout);
  X3Params kp;
  kp.p = p;
  kp.c_chunks = 1;
  if (p.mode == CP_X3_LINEAR) {
    CP_REQUIRE(p.k1 > 0 && p.k1 % 64 == 0 && p.k2 >= 0 && p.k2 % 64 == 0 && p.k1 + p.k2 == p.K, CP_E_UNSUPPORTED,
               "cp_gemm_x3: k1=%d, k2=%d must be multiples of 64 summing to K=%d", p.k1, p.k2, p.K);
    CP_REQUIRE(p.k2 == 0 || p.a2, CP_E_INVALID, "cp_gemm_x3: a2 is NULL but k2=%d", p.k2);
    CP_REQUIRE(p.ld1 >= p.k1 && (p.ld1 & 3) == 0 && (reinterpret_cast<uintptr_t>(p.a1) & 15) == 0 &&
               (p.k2 == 0 || (p.ld2 >= p.k2 && (p.ld2 & 3) == 0 && (reinterpret_cast<uintptr_t>(p.a2) & 15) == 0)), CP_E_INVALID,
               "cp_gemm_x3: operand rows must be 16-byte aligned (ld %% 4 == 0)");
  } else {
    CP_REQUIRE(p.mode == CP_X3_CONV || p.mode == CP_X3_CONVT, CP_E_INVALID, "cp_gemm_x3: bad mode %d", p.mode);
    CP_REQUIRE(p.k1 > 0 && p.k1 % 64 == 0 && p.KH > 0 && p.KW > 0 && p.KH * p.KW * p.k1 == p.K, CP_E_UNSUPPORTED,
               "cp_gemm_x3: conv needs Cin %% 64 == 0 and K == KH*KW*Cin (Cin=%d KH=%d KW=%d K=%d)", p.k1, p.KH, p.KW, p.K);
    CP_REQUIRE(p.H > 0 && p.W > 0 && p.Ho > 0 && p.Wo > 0 && p.Ho < 32768 && p.Wo < 32768 && p.pad >= 0 && p.M % ((int64_t)p.Ho * p.Wo) == 0, CP_E_INVALID,
               "cp_gemm_x3: bad map sizes H=%d W=%d Ho=%d Wo=%d (M must be B*Ho*Wo)", p.H, p.W, p.Ho, p.Wo);
    CP_REQUIRE((reinterpret_cast<uintptr_t>(p.a1) & 15) == 0, CP_E_INVALID, "cp_gemm_x3: input map not 16-byte aligned");
    kp.c_chunks = p.k1 / 64;
  }
  kp.KC = p.K / 64;
  kp.npad = (p.Nout + 15) / 16 * 16;
  kp.nblk = (kp.npad + BN - 1) / BN;
  CP_REQUIRE((p.M + TILE_M - 1) / TILE_M * kp.nblk < (1ll << 31), CP_E_UNSUPPORTED, "cp_gemm_x3: too many tiles");
  kp.num_m_tiles = (int)((p.M + TILE_M - 1) / TILE_M);
  kp.num_tiles = kp.num_m_tiles * kp.nblk;
  CP_REQUIRE(p.M < (1ll << 31), CP_E_UNSUPPORTED, "cp_gemm_x3: M must be < 2^31");
  CUtensorMap map;
  memset(&map, 0, sizeof(map));
  // (the TMA engine clips the inner dimension in 16-byte units: a row length that is not a multiple of 4 floats would spill
  //  into the next columns -- measured on B200 -- so those outputs take the direct path)
  kp.tma_out = ((p.ld_out & 3) == 0 && (p.Nout & 3) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0) ? 1 : 0;
  if (kp.tma_out) {
    const int rc = cp::make_f32_tensor_map_2d(&map, p.out, p.Nout, p.M, p.ld_out, "cp_gemm_x3");
    if (rc != CP_OK) return rc;
  }
  const int num_sms = cp::num_sms();
  const int grid = kp.num_tiles < num_sms ? kp.num_tiles : num_sms;
  cudaError_t e = cudaFuncSetAttribute(gemm_x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "cp_gemm_x3: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
  gemm_x3_kernel<<<grid, NTHREADS, SMEM_BYTES, (cudaStream_t)s>>>(kp, map);
  CP_CHECK_LAUNCH("cp_gemm_x3");
  return CP_OK;
}
