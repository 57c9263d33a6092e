// K4: the tail of a refine stage in one launch -- query MLP 256 -> 64 -> 2 fused with the sign-bit decode and the id update.
//
// Replaces, per refine stage, MLP_QueryNet's last two Linear layers (checkerpose/model/pipeline.py:174-180; the first one is
// fused into the last EdgeConv launch) and the decode of pipeline.py:375-381:  new_x_bit / new_y_bit planes of
// output_x_bits / output_y_bits,  pred_id = pred_id * 2 + (sigmoid(bit) > 0.5),  plus the keypoint-order ids the caller sees
// after the last stage.  Before: a generic chain launch (0.19 ms, 3.0 TB/s on its 565 MB input) writing fp32 logits, then a
// decode launch reading them back.
//
// One persistent CTA of 8 warps per SM, tile = 128 plan-order nodes:
//   warp 0      producer: the tile's A operand (128 rows x 256 bf16) as four TMA TENSOR loads (cp.async.bulk.tensor.2d, box
//               64 channels x 128 rows, SWIZZLE_128B: lands in the K-major layout tcgen05.mma reads; rows beyond B*N are
//               zero-filled by the TMA unit) into a 2-stage ring; the 64 x 256 weight tile (32 KB) is loaded once per CTA;
//   warp 1      MMA issuer: 16 x tcgen05.mma (M=128, N=64, K=16) per tile into one of two 64-column accumulators;
//   warps 4-7   epilogue: tcgen05.ld -> + b1 -> LeakyReLU -> the 64 -> 2 layer as register dot products in fp32 -> logits ->
//               bit planes, id = 2 id + bit (plan order, in place), keypoint-order ids (last stage).
// HBM-bound: N * 256 * 2 bytes read per RoI, ~50 bytes written per keypoint.
#include <cuda.h>
#include <string.h>

#include "common.cuh"
#include "sm100.cuh"

using namespace sm100;

namespace {

constexpr int TILE_M = 128;
constexpr int NTHREADS = 256;
constexpr int STAGES = 2;
constexpr int KMAX = 256, NMID = 64;
constexpr int A_CHUNK_BYTES = TILE_M * 128;                 // 128 rows x 64 bf16
constexpr int A_STAGE_BYTES = (KMAX / 64) * A_CHUNK_BYTES;  // 64 KB
constexpr int W_BYTES = NMID * KMAX * 2;                    // 32 KB: 4 chunks of 64 rows x 128 B
constexpr int OFF_W = STAGES * A_STAGE_BYTES;
constexpr int OFF_CONST = OFF_W + W_BYTES;                  // b1[64], w2[2][64], b2[2] as fp32
constexpr int OFF_BAR = OFF_CONST + (64 + 128 + 8) * 4;
constexpr int SMEM_BYTES = OFF_BAR + 128 + 1024;
constexpr int TMEM_COLS = 128;

struct Bars {
  uint64_t full[STAGES], empty[STAGES], acc_full[2], acc_empty[2], w_full;
  uint32_t tmem_slot;
};

struct QtParams {
  cp_query_decode_params p;
  int KC;            // K chunks of 64
  int64_t M;         // B * N
  int num_tiles;
  int wsel;          // object-indexed weights: p.graph_sel selects them; every tile then holds rows of one RoI
  int tiles_per_roi; // with wsel
};

// First row of a tile and its valid rows (the RoI's rows with wsel, else the flat rows of B * N); RoI of the tile with wsel
__device__ __forceinline__ void tile_rows(const QtParams& kp, int tile, int64_t& row0, int& rows_valid, int& b) {
  if (kp.wsel) {
    b = tile / kp.tiles_per_roi;
    const int n0 = (tile - b * kp.tiles_per_roi) * TILE_M;
    row0 = (int64_t)b * kp.p.N + n0;
    rows_valid = min(TILE_M, kp.p.N - n0);
  } else {
    b = 0;
    row0 = (int64_t)tile * TILE_M;
    rows_valid = (int)min((int64_t)TILE_M, kp.M - row0);
  }
}

// b1[64], w2[2][64], b2[2] of object obj -> cst
__device__ __forceinline__ void load_consts(const cp_query_decode_params& p, float* cst, int64_t obj, int tid, int nthreads) {
  for (int i = tid; i < 64 + 128 + 2; i += nthreads) {
    float v;
    if (i < 64) v = p.b1 ? p.b1[obj * p.b1_stride + i] : 0.f;
    else if (i < 192) v = p.w2[obj * p.w2_stride + i - 64];          // (2, 64) row-major
    else v = p.b2 ? p.b2[obj * p.b2_stride + i - 192] : 0.f;
    cst[i] = v;
  }
}

__global__ void __launch_bounds__(NTHREADS, 1) query_tail_kernel(const __grid_constant__ QtParams kp, const __grid_constant__ CUtensorMap src_map) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  Bars* bars = reinterpret_cast<Bars*>(sm + OFF_BAR);
  float* cst = reinterpret_cast<float*>(sm + OFF_CONST);
  const cp_query_decode_params& p = kp.p;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&bars->full[s], 1);
      mbar_init(&bars->empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&bars->acc_full[a], 1);
      mbar_init(&bars->acc_empty[a], 4);
    }
    mbar_init(&bars->w_full, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(&bars->tmem_slot, TMEM_COLS);
  load_consts(p, cst, 0, threadIdx.x, NTHREADS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = bars->tmem_slot;
  const int KC = kp.KC;

  if (warp == 0) {
    // ---- producer ----
    uint32_t it = 0;
    int wobj = -1;   // object whose W1 is resident
    for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x, ++it) {
      int64_t row0;
      int rows_valid, b;
      tile_rows(kp, tile, row0, rows_valid, b);
      const int obj = cp::weight_obj(p.graph_sel, kp.wsel != 0, b);
      if (obj != wobj) {
        // the previous tile's MMAs read the resident W1: wait until they are done before overwriting it
        if (it > 0) mbar_wait(&bars->empty[(it - 1) % STAGES], ((it - 1) / STAGES) & 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&bars->w_full, (uint32_t)(NMID * KC * 128));
          // the whole packed matrix (cp::packed_tile_offset): one block of 64 rows, chunk c at c * 64 * 128 bytes
          bulk_g2s(sm + OFF_W, reinterpret_cast<const uint8_t*>(p.w1_packed) + (int64_t)obj * p.w1_stride, (uint32_t)(NMID * KC * 128),
                   &bars->w_full);
        }
        __syncwarp();
        wobj = obj;
      }
      const uint32_t s = it % STAGES;
      if (it >= STAGES) mbar_wait(&bars->empty[s], ((it / STAGES) - 1) & 1);
      if (elect_one()) {
        mbar_arrive_expect_tx(&bars->full[s], (uint32_t)(KC * A_CHUNK_BYTES));
        for (int c = 0; c < KC; ++c) tma_load_2d(smem_u32(sm + s * A_STAGE_BYTES + c * A_CHUNK_BYTES), &src_map, c * 64, (int)row0, &bars->full[s]);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ---- MMA issuer ----
    const uint32_t idesc = make_idesc_bf16_m128(NMID);
    const uint32_t w_lo0 = smem_desc_lo(smem_u32(sm + OFF_W));
    uint32_t it = 0, wn = 0;
    int wobj = -1;
    for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x, ++it) {
      const uint32_t s = it % STAGES, slot = it & 1;
      int64_t row0;
      int rows_valid, b;
      tile_rows(kp, tile, row0, rows_valid, b);
      const int obj = cp::weight_obj(p.graph_sel, kp.wsel != 0, b);
      if (obj != wobj) {   // the producer loaded this object's W1
        mbar_wait(&bars->w_full, wn & 1);
        ++wn;
        wobj = obj;
      }
      if (it >= 2) mbar_wait(&bars->acc_empty[slot], ((it >> 1) - 1) & 1);
      mbar_wait(&bars->full[s], (it / STAGES) & 1);
      tc_fence_after_sync();
      const uint32_t a_lo0 = smem_desc_lo(smem_u32(sm + s * A_STAGE_BYTES));
      const uint32_t d = tmem_base + slot * NMID;
      if (elect_one()) {
        for (int c = 0; c < KC; ++c) {
          const uint32_t a_lo = a_lo0 + c * (A_CHUNK_BYTES >> 4), w_lo = w_lo0 + c * ((NMID * 128) >> 4);
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k) mma_bf16_ss_lo(d, a_lo + 2 * k, w_lo + 2 * k, idesc, (uint32_t)((c | (int)k) != 0));
        }
        mma_commit(&bars->empty[s]);
        mma_commit(&bars->acc_full[slot]);
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ---- epilogue: query layer 2 (64 -> 2) and the decode, one thread per node ----
    const int q = warp - 4;
    const float slope = p.slope;
    uint32_t it = 0;
    int cur_obj = 0;   // object whose b1 / W2 / b2 are in cst (the kernel loads object 0's)
    for (int tile = blockIdx.x; tile < kp.num_tiles; tile += gridDim.x, ++it) {
      const uint32_t slot = it & 1;
      int64_t row0;
      int rows_valid, tb_roi;
      tile_rows(kp, tile, row0, rows_valid, tb_roi);
      const int obj = cp::weight_obj(p.graph_sel, kp.wsel != 0, tb_roi);
      if (obj != cur_obj) {   // every epilogue warp is past the previous tile's reads, then all see the new constants
        cp::named_bar_sync(1, 128);
        load_consts(p, cst, obj, q * 32 + lane, 128);
        cp::named_bar_sync(1, 128);
        cur_obj = obj;
      }
      mbar_wait(&bars->acc_full[slot], (it >> 1) & 1);
      tc_fence_after_sync();
      const uint32_t tb = tmem_base + ((uint32_t)(q * 32) << 16) + slot * NMID;
      float lx = cst[192], ly = cst[193];
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t r[32];
        tmem_ld32(tb + half * 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const int c = half * 32 + e;
          const float h = cp::lrelu(__uint_as_float(r[e]) + cst[c], slope);
          lx = fmaf(h, cst[64 + c], lx);
          ly = fmaf(h, cst[128 + c], ly);
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->acc_empty[slot]);     // the accumulator is in registers: the next tile's MMAs may run
      const int64_t e = row0 + q * 32 + lane;
      if (q * 32 + lane < rows_valid) {
        const int b = kp.wsel ? tb_roi : (int)(e / p.N), n = (int)(e - (int64_t)b * p.N);
        int kpt = n;
        if (p.perm) kpt = p.perm[(size_t)(p.graph_sel ? p.graph_sel[b] : 0) * p.N + n];
        if (p.logits) {
          p.logits[e * p.ld_logits] = lx;
          p.logits[e * p.ld_logits + 1] = ly;
        }
        p.x_bits[((size_t)b * p.Ltot + p.plane) * p.N + kpt] = lx;
        p.y_bits[((size_t)b * p.Ltot + p.plane) * p.N + kpt] = ly;
        const int64_t xi = p.x_id[e] * 2 + (lx > 0.f ? 1 : 0), yi = p.y_id[e] * 2 + (ly > 0.f ? 1 : 0);
        p.x_id[e] = xi;
        p.y_id[e] = yi;
        if (p.x_id_kp) {
          p.x_id_kp[(size_t)b * p.N + kpt] = xi;
          p.y_id_kp[(size_t)b * p.N + kpt] = yi;
        }
      }
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

}  // namespace

extern "C" int cp_query_decode_fwd(const cp_query_decode_params* pp, cp_stream_t s) {
  CP_REQUIRE(pp, CP_E_INVALID, "cp_query_decode_fwd: null params");
  const cp_query_decode_params& p = *pp;
  CP_REQUIRE(p.B > 0 && p.N > 0 && p.src && p.w1_packed && p.w2 && p.x_bits && p.y_bits && p.x_id && p.y_id, CP_E_INVALID,
             "cp_query_decode_fwd: bad arguments");
  CP_REQUIRE((p.kin == 64 || p.kin == 128 || p.kin == 256) && p.nmid == NMID && p.nout == 2, CP_E_UNSUPPORTED,
             "cp_query_decode_fwd: supports kin in {64,128,256}, 64 hidden channels, 2 logits (kin=%d nmid=%d nout=%d)", p.kin, p.nmid, p.nout);
  CP_REQUIRE(p.ld_src >= p.kin && (p.ld_src % 8) == 0 && (reinterpret_cast<uintptr_t>(p.src) & 15) == 0 &&
             (reinterpret_cast<uintptr_t>(p.w1_packed) & 15) == 0, CP_E_INVALID, "cp_query_decode_fwd: src / weights must be 16-byte aligned, ld %% 8 == 0");
  CP_REQUIRE((p.x_id_kp == nullptr) == (p.y_id_kp == nullptr) && p.plane >= 0 && p.plane < p.Ltot && (!p.logits || p.ld_logits >= 2), CP_E_INVALID,
             "cp_query_decode_fwd: bad decode arguments");
  QtParams kp;
  kp.p = p;
  kp.KC = p.kin / 64;
  kp.M = (int64_t)p.B * p.N;
  CP_REQUIRE(kp.M < (1ll << 31), CP_E_UNSUPPORTED, "cp_query_decode_fwd: B * N must be < 2^31");
  CP_REQUIRE(p.w1_stride >= 0 && (p.w1_stride % 16) == 0 && p.b1_stride >= 0 && p.w2_stride >= 0 && p.b2_stride >= 0, CP_E_INVALID,
             "cp_query_decode_fwd: strides must be >= 0, w1_stride a multiple of 16");
  kp.wsel = (p.w1_stride != 0 || p.b1_stride != 0 || p.w2_stride != 0 || p.b2_stride != 0) ? 1 : 0;
  kp.tiles_per_roi = (p.N + TILE_M - 1) / TILE_M;
  kp.num_tiles = kp.wsel ? kp.tiles_per_roi * p.B : (int)((kp.M + TILE_M - 1) / TILE_M);
  CUtensorMap map;
  memset(&map, 0, sizeof(map));
  const int rc = cp::make_bf16_operand_map(&map, p.src, p.kin, kp.M, p.ld_src, "cp_query_decode_fwd");
  if (rc != CP_OK) return rc;
  const int num_sms = cp::num_sms();
  const int grid = kp.num_tiles < num_sms ? kp.num_tiles : num_sms;
  cudaError_t e = cudaFuncSetAttribute(query_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "cp_query_decode_fwd: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
  query_tail_kernel<<<grid, NTHREADS, SMEM_BYTES, (cudaStream_t)s>>>(kp, map);
  CP_CHECK_LAUNCH("cp_query_decode_fwd");
  return CP_OK;
}
