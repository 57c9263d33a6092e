// Fused tcgen05 "chain" kernel: the bf16 tensor-core path of the GNN keypoint head.
//
// One persistent CTA (256 threads, two CTAs per SM) walks over tiles of 128 keypoints ("nodes") of
// one RoI.  Per tile:
//
//   PROLOGUE  builds the A operand (128 nodes x K channels, bf16) straight in shared memory, in the
//             K-major SWIZZLE_128B layout tcgen05.mma reads -- it never exists in HBM:
//               LOAD : rows of a node-major tensor
//               AGG  : EdgeConv aggregation  lrelu(max_k P[idx[i,k]] + Q[i])  with the max taken in
//                      registers over packed bf16x2 (replaces get_graph_feature + conv + BN + LeakyReLU +
//                      max of checkerpose/model/pipeline.py:27-59; see cp_fold_edgeconv for the algebra)
//               TAPS : Index2Feat 4-tap gather x roi mask (pipeline.py:156-163, 280), then (second K
//                      phase) the previous graph feature, i.e. the concat of pipeline.py:283
//   GEMMs     up to three chained Linear(+bias+LeakyReLU) layers on tcgen05: weights are pre-packed
//             tile images streamed by one producer thread with cp.async.bulk (TMA engine) into a
//             2-stage mbarrier ring; one elected thread issues tcgen05.mma (M=128, N<=128, K=16) with
//             fp32 accumulators in TMEM (256 columns per CTA); tcgen05.commit signals stage release and
//             accumulator-ready.  Between layers the epilogue converts TMEM -> bf16 and writes the
//             next A operand back into the same shared-memory tile.
//   OUTPUT    bf16 [P|Q] table for the next EdgeConv layer, or fp32 logits.
//
// Roofline: with the factored EdgeConv the layer is bandwidth-bound (DESIGN.md section 5); the tensor
// work per tile (128 x 512 x 256 MACs) is ~4k cycles against a gather of 128 x K x 512 B from L2.
#include "common.cuh"
#include "sm100.cuh"

using bf16 = __nv_bfloat16;
using namespace sm100;

namespace {

constexpr int TILE_M = 128;
constexpr int NTHREADS = 256;
constexpr int NWARPS = 8;
constexpr int KCHUNK = 64;                       // bf16 elements per 128-byte swizzle row
constexpr int A_CHUNK_BYTES = TILE_M * 128;      // 16 KB: 128 rows x 64 bf16
constexpr int A_CHUNKS = 4;                      // K <= 256 resident at a time
constexpr int B_STAGE_BYTES = 128 * 128;         // 16 KB: <=128 weight rows x 64 bf16
constexpr int STAGES = 3;
constexpr int TMEM_COLS = 256;
constexpr int MAX_WTILES = 48;
// two CTAs per SM: 2 x (SMEM_BYTES + 1 KB reserved) must stay within 227 KB, so there is no alignment slack -- the
// kernel traps if the dynamic shared-memory window is not 1024-byte aligned (it is: windows are 1 KB granular)
constexpr int SMEM_BYTES = A_CHUNKS * A_CHUNK_BYTES + STAGES * B_STAGE_BYTES + 256;
static_assert(2 * (SMEM_BYTES + 1024) <= 227 * 1024, "two CTAs per SM");

struct KParams {
  cp_chain_params p;
  int tiles_per_roi;
  int num_node_tiles;
  int T;  // weight tiles per node tile
  cp::WTile wt[MAX_WTILES];
};

struct Smem {
  uint8_t* A;
  uint8_t* Bst;
  uint64_t* full;
  uint64_t* empty;
  uint64_t* acc;
  uint32_t* tmem_slot;
};

__device__ __forceinline__ uint32_t a_offset(int kc, int row, int chunk) {
  return (uint32_t)(kc * A_CHUNK_BYTES + row * 128 + ((chunk ^ (row & 7)) << 4));
}

__device__ __forceinline__ uint32_t bf2_max(uint32_t a, uint32_t b) {
  __nv_bfloat162 x = *reinterpret_cast<__nv_bfloat162*>(&a), y = *reinterpret_cast<__nv_bfloat162*>(&b);
  __nv_bfloat162 m = __hmax2(x, y);
  return *reinterpret_cast<uint32_t*>(&m);
}

// ---- prologues: all 256 threads fill A chunks [0, C/64) for the 128 rows of the tile -----------------

// rows of a node-major bf16 tensor; C in {64,128,256}.  cp.async (LDGSTS) straight into the swizzled operand layout,
// zero-filled beyond rows_valid: all of a thread's 16-byte pieces (up to 16 at C = 256) are in flight at once -- one
// memory round trip per tile instead of the four of the register-staged version (0.224 -> see DESIGN.md section 8).
__device__ __forceinline__ void fill_rows(uint8_t* A, const bf16* src, int ld, int C, int64_t row0, int rows_valid) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cpr = C >> 3;  // 16-byte chunks per row
  const int rpi = 32 / cpr;
  const int sub = lane / cpr, chunk = lane - sub * cpr;
  const uint32_t a_s = sm100::smem_u32(A);
  for (int r = warp * rpi + sub; r < TILE_M; r += NWARPS * rpi) {
    const bool ok = r < rows_valid;
    const void* g = src + (ok ? (row0 + r) * ld + chunk * 8 : 0);
    cp_async16_zfill(a_s + a_offset(chunk >> 3, r, chunk & 7), g, ok ? 16u : 0u);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// EdgeConv aggregation; Co in {64,128,256}
__device__ __forceinline__ void fill_agg(uint8_t* A, const cp_chain_params& p, int b, int n0, int rows_valid) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int Co = p.Co, K = p.K;
  const int cpr = Co >> 3;
  const int rpi = 32 / cpr;
  const int sub = lane / cpr, chunk = lane - sub * cpr;
  const int g = p.graph_sel ? p.graph_sel[b] : 0;
  const int32_t* idx_g = p.idx + (size_t)g * p.N * K;
  const bf16* zb = reinterpret_cast<const bf16*>(p.z) + (size_t)b * p.N * p.ld_z;
  bf16* aout = p.a_out ? reinterpret_cast<bf16*>(p.a_out) + (size_t)b * p.N * p.ld_a_out : nullptr;
  const float slope = p.agg_slope;
  for (int r = warp * rpi + sub; r < TILE_M; r += NWARPS * rpi) {
    uint4 o = make_uint4(0, 0, 0, 0);
    if (r < rows_valid) {
      const int i = n0 + r;
      const int32_t* nb = idx_g + (size_t)i * K;
      const bf16* zc = zb + chunk * 8;
      // seed with the first neighbour (no -inf constants; correct for graphs without self loops too)
      uint4 m = ldg_nc_v4(zc + (size_t)__ldg(nb) * p.ld_z);
      int k = 1;
      for (; k + 4 <= K; k += 4) {
        const int j0 = __ldg(nb + k), j1 = __ldg(nb + k + 1), j2 = __ldg(nb + k + 2), j3 = __ldg(nb + k + 3);
        const uint4 v0 = ldg_nc_v4(zc + (size_t)j0 * p.ld_z);
        const uint4 v1 = ldg_nc_v4(zc + (size_t)j1 * p.ld_z);
        const uint4 v2 = ldg_nc_v4(zc + (size_t)j2 * p.ld_z);
        const uint4 v3 = ldg_nc_v4(zc + (size_t)j3 * p.ld_z);
        m.x = bf2_max(bf2_max(m.x, v0.x), bf2_max(v1.x, bf2_max(v2.x, v3.x)));
        m.y = bf2_max(bf2_max(m.y, v0.y), bf2_max(v1.y, bf2_max(v2.y, v3.y)));
        m.z = bf2_max(bf2_max(m.z, v0.z), bf2_max(v1.z, bf2_max(v2.z, v3.z)));
        m.w = bf2_max(bf2_max(m.w, v0.w), bf2_max(v1.w, bf2_max(v2.w, v3.w)));
      }
      for (; k < K; ++k) {
        const uint4 v = ldg_nc_v4(zc + (size_t)__ldg(nb + k) * p.ld_z);
        m.x = bf2_max(m.x, v.x); m.y = bf2_max(m.y, v.y); m.z = bf2_max(m.z, v.z); m.w = bf2_max(m.w, v.w);
      }
      const uint4 q = ldg_nc_v4(zc + (size_t)i * p.ld_z + Co);
      const uint32_t mm[4] = {m.x, m.y, m.z, m.w}, qq[4] = {q.x, q.y, q.z, q.w};
      uint32_t oo[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float2 a = bf2_to_f2(mm[t]), c = bf2_to_f2(qq[t]);
        oo[t] = f2_to_bf2(cp::lrelu(a.x + c.x, slope), cp::lrelu(a.y + c.y, slope));
      }
      o = make_uint4(oo[0], oo[1], oo[2], oo[3]);
      if (aout) *reinterpret_cast<uint4*>(aout + (size_t)i * p.ld_a_out + chunk * 8) = o;
    }
    *reinterpret_cast<uint4*>(A + a_offset(chunk >> 3, r, chunk & 7)) = o;
  }
}

// Index2Feat taps (E == 64: one tap = one 128-byte K chunk), masked
__device__ __forceinline__ void fill_taps(uint8_t* A, const cp_chain_params& p, int b, int n0, int rows_valid) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tap = lane >> 3, chunk = lane & 7;
  const bf16* pb = reinterpret_cast<const bf16*>(p.patches) + (size_t)b * p.Hp * p.Wp * 64;
  // a thread owns rows warp, warp + 8, ...: first all the ids and masks, then all the tap loads, then the stores, so
  // that the two dependent global-load latencies are paid once per tile instead of once per row
  constexpr int RPT = TILE_M / NWARPS;
  int off[RPT];   // element offset of the tap inside the RoI's patch map, -1 = masked / no row
#pragma unroll
  for (int u = 0; u < RPT; ++u) {
    const int r = warp + u * NWARPS;
    off[u] = -1;
    if (r < rows_valid) {
      const size_t e = (size_t)b * p.N + n0 + r;
      const float mk = p.mask ? __ldg(p.mask + e) : 1.f;
      const int yy = (int)(2 * __ldg(p.y_id + e)) + ((tap & 1) ? p.tap_step : 0);
      const int xx = (int)(2 * __ldg(p.x_id + e)) + ((tap & 2) ? p.tap_step : 0);
      if (yy < 0 || xx < 0 || yy >= p.Hp || xx >= p.Wp) __trap();   // caller error (the reference raises an index assert)
      if (mk != 0.f) off[u] = (yy * p.Wp + xx) * 64 + chunk * 8;
    }
  }
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    uint4 v[RPT / 2];
#pragma unroll
    for (int u = 0; u < RPT / 2; ++u) {
      const int o = off[h * (RPT / 2) + u];
      v[u] = make_uint4(0, 0, 0, 0);
      if (o >= 0) v[u] = ldg_nc_v4(pb + o);
    }
#pragma unroll
    for (int u = 0; u < RPT / 2; ++u) {
      const int r = warp + (h * (RPT / 2) + u) * NWARPS;
      *reinterpret_cast<uint4*>(A + a_offset(tap, r, chunk)) = v[u];
    }
  }
}

// ---- epilogue: TMEM accumulator columns [0, pcols) of this pass -> bias/act -> destination -----------
enum { EPI_SMEM = 0, EPI_BF16 = 1, EPI_F32 = 2 };

__device__ __forceinline__ void epilogue(uint32_t tmem_base, int pcols, int col0_global, const float* bias, int nout_valid, int act,
                                         float slope, int mode, uint8_t* A, void* out, int ld_out, int n_valid,
                                         int64_t row0, int rows_valid) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = warp & 3, half = warp >> 2;
  const int row = q * 32 + lane;
  const bool row_ok = row < rows_valid;
  const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16);
  const int nch = pcols >> 4;  // 16-column chunks
  for (int ch = half; ch < nch; ch += 2) {
    uint32_t r[16];
    tmem_ld16(tbase + (uint32_t)(ch * 16), r);
    const int c0 = ch * 16;  // column within the pass
    float4 bv[4];            // bias of the 16 columns, loaded while the TMEM read is in flight
#pragma unroll
    for (int t = 0; t < 4; ++t) bv[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias) {
      if (col0_global + c0 + 16 <= nout_valid && (reinterpret_cast<uintptr_t>(bias) & 15) == 0) {
#pragma unroll
        for (int t = 0; t < 4; ++t) bv[t] = __ldg(reinterpret_cast<const float4*>(bias + col0_global + c0) + t);
      } else {
        float* bs = reinterpret_cast<float*>(bv);
#pragma unroll
        for (int t = 0; t < 16; ++t) bs[t] = (col0_global + c0 + t < nout_valid) ? __ldg(bias + col0_global + c0 + t) : 0.f;
      }
    }
    tmem_ld_wait();
    float v[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) {
      float x = __uint_as_float(r[t]) + reinterpret_cast<const float*>(bv)[t];
      if (act) x = cp::lrelu(x, slope);
      v[t] = x;
    }
    if (mode == EPI_F32) {
      if (row_ok) {
        float* o = reinterpret_cast<float*>(out) + (row0 + row) * ld_out;
#pragma unroll
        for (int t = 0; t < 16; ++t)
          if (col0_global + c0 + t < n_valid) o[col0_global + c0 + t] = v[t];
      }
    } else {
      uint4 w0 = make_uint4(f2_to_bf2(v[0], v[1]), f2_to_bf2(v[2], v[3]), f2_to_bf2(v[4], v[5]), f2_to_bf2(v[6], v[7]));
      uint4 w1 = make_uint4(f2_to_bf2(v[8], v[9]), f2_to_bf2(v[10], v[11]), f2_to_bf2(v[12], v[13]), f2_to_bf2(v[14], v[15]));
      if (mode == EPI_SMEM) {
        // next layer's A operand: column c -> K chunk c/64, 16-byte chunk (c%64)/8
        const int c = col0_global + c0;
        *reinterpret_cast<uint4*>(A + a_offset(c >> 6, row, (c & 63) >> 3)) = w0;
        *reinterpret_cast<uint4*>(A + a_offset((c + 8) >> 6, row, ((c + 8) & 63) >> 3)) = w1;
      } else if (row_ok) {
        bf16* o = reinterpret_cast<bf16*>(out) + (row0 + row) * ld_out + col0_global + c0;
        *reinterpret_cast<uint4*>(o) = w0;
        *reinterpret_cast<uint4*>(o + 8) = w1;
      }
    }
  }
}

template <int PRO>
__global__ void __launch_bounds__(NTHREADS, 2) chain_kernel(const __grid_constant__ KParams kp) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const cp_chain_params& p = kp.p;
  uint8_t* base = smem_raw;
  if ((smem_u32(base) & 1023u) != 0) __trap();   // SWIZZLE_128B operand tiles need 1024-byte alignment
  Smem sm;
  sm.A = base;
  sm.Bst = base + A_CHUNKS * A_CHUNK_BYTES;
  sm.full = reinterpret_cast<uint64_t*>(sm.Bst + STAGES * B_STAGE_BYTES);
  sm.empty = sm.full + STAGES;
  sm.acc = sm.empty + STAGES;
  sm.tmem_slot = reinterpret_cast<uint32_t*>(sm.acc + 1);

  const int warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&sm.full[s], 1);
      mbar_init(&sm.empty[s], 1);
    }
    mbar_init(sm.acc, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(sm.tmem_slot, TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *sm.tmem_slot;

  const int my_tiles = (kp.num_node_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const long long total_w = (long long)my_tiles * kp.T;
  long long pc = 0;       // weight tiles issued (producer warp only)
  long long mc = 0;       // weight tiles consumed (tracked uniformly by all threads)
  uint32_t acc_n = 0;     // accumulator-barrier phases consumed (uniform)
  // warps 0 / 1 run the MMA issue / weight streaming loops warp-uniformly; an elected lane issues the single-thread
  // instructions (under an `if (lane == 0)` region ptxas wraps every tcgen05.mma in a uniform-register broadcast loop)

  for (int tile = blockIdx.x; tile < kp.num_node_tiles; tile += gridDim.x) {
    const int b = tile / kp.tiles_per_roi;
    const int n0 = (tile - b * kp.tiles_per_roi) * TILE_M;
    const int rows_valid = min(TILE_M, p.N - n0);
    const int64_t row0 = (int64_t)b * p.N + n0;

    // ---------------- prologue -> A ----------------
    if (PRO == CP_PRO_LOAD) fill_rows(sm.A, reinterpret_cast<const bf16*>(p.src), p.ld_src, p.C, row0, rows_valid);
    else if (PRO == CP_PRO_AGG) fill_agg(sm.A, p, b, n0, rows_valid);
    else fill_taps(sm.A, p, b, n0, rows_valid);
    fence_proxy_async_smem();
    __syncthreads();

    int widx = 0;  // index into the per-node-tile weight table
    for (int l = 0; l < p.num_layers; ++l) {
      const cp_chain_layer& L = p.layers[l];
      const int npad = (L.nout + 15) & ~15;
      const int npass = (npad + TMEM_COLS - 1) / TMEM_COLS;
      const bool last = (l == p.num_layers - 1);
      const int nphase = (PRO == CP_PRO_TAPS && l == 0) ? 2 : 1;
      for (int pass = 0; pass < npass; ++pass) {
        const int col0 = pass * TMEM_COLS;
        const int pcols = min(TMEM_COLS, npad - col0);
        const int nblk = (pcols + 127) >> 7;
        for (int ph = 0; ph < nphase; ++ph) {
          const int kc_count = (nphase == 2) ? (ph == 0 ? 4 : (p.Cg >> 6)) : (L.kin >> 6);
          if (ph == 1) {
            // second K phase of the pre-graph GEMM: A <- previous graph feature (all MMAs of phase 0 done)
            fill_rows(sm.A, reinterpret_cast<const bf16*>(p.graph_feat), p.ld_gf, p.Cg, row0, rows_valid);
            fence_proxy_async_smem();
            __syncthreads();
          }
          const int ntiles = nblk * kc_count;
          const long long mc_end = mc + ntiles;
          if (warp == 0) {
            {
              tc_fence_after_sync();
              for (int nbi = 0; nbi < nblk; ++nbi) {
                for (int kci = 0; kci < kc_count; ++kci) {
                  const cp::WTile& wt = kp.wt[widx + nbi * kc_count + kci];
                  const long long it = mc + nbi * kc_count + kci;
                  const int s = (int)(it % STAGES);
                  mbar_wait(&sm.full[s], (uint32_t)((it / STAGES) & 1));
                  tc_fence_after_sync();
                  const uint32_t idesc = make_idesc_bf16_m128(wt.bytes >> 7);
                  const uint32_t a_addr = smem_u32(sm.A + kci * A_CHUNK_BYTES);
                  const uint32_t b_addr = smem_u32(sm.Bst + s * B_STAGE_BYTES);
                  const uint32_t d = tmem_base + (uint32_t)(nbi * 128);
                  if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < KCHUNK / 16; ++k) {
                      mma_bf16_ss(d, make_smem_desc_sw128(a_addr + k * 32), make_smem_desc_sw128(b_addr + k * 32), idesc,
                                  (uint32_t)((kci | k | ph) != 0));
                    }
                    mma_commit(&sm.empty[s]);
                  }
                  __syncwarp();
                }
              }
              if (elect_one()) mma_commit(sm.acc);
            }
            __syncwarp();
          } else if (warp == 1) {
            {
              long long limit = mc_end + STAGES;
              if (limit > total_w) limit = total_w;
              while (pc < limit) {
                const int s = (int)(pc % STAGES);
                const long long use = pc / STAGES;
                if (use > 0) mbar_wait(&sm.empty[s], (uint32_t)((use - 1) & 1));
                const cp::WTile& wt = kp.wt[(int)(pc % kp.T)];
                if (elect_one()) {
                  mbar_arrive_expect_tx(&sm.full[s], wt.bytes);
                  bulk_g2s(sm.Bst + s * B_STAGE_BYTES, wt.ptr, wt.bytes, &sm.full[s]);
                }
                __syncwarp();
                ++pc;
              }
            }
            __syncwarp();
          }
          mc = mc_end;
          widx += ntiles;
          // ---------------- wait for the accumulator ----------------
          mbar_wait(sm.acc, acc_n & 1);
          ++acc_n;
          tc_fence_after_sync();
        }
        // ---------------- epilogue of this pass ----------------
        int mode;
        if (!last) mode = EPI_SMEM;
        else mode = (p.out_mode == CP_OUT_BF16) ? EPI_BF16 : EPI_F32;
        epilogue(tmem_base, pcols, col0, L.bias, L.nout, L.act, L.slope, mode, sm.A, p.out, p.ld_out, p.n_valid, row0, rows_valid);
        tc_fence_before_sync();
        if (mode == EPI_SMEM) fence_proxy_async_smem();
        __syncthreads();
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, TMEM_COLS);
}

bool pow2_64_256(int c) { return c == 64 || c == 128 || c == 256; }

}  // namespace

namespace cp {
bool taps_chain_try(const cp_chain_params& p, cudaStream_t s, int* rc);   // taps_chain_tcgen05.cu
}

extern "C" int cp_chain_fwd(const cp_chain_params* pp, cp_stream_t s) {
  CP_REQUIRE(pp, CP_E_INVALID, "cp_chain_fwd: null params");
  const cp_chain_params& p = *pp;
  CP_REQUIRE(p.B > 0 && p.N > 0, CP_E_INVALID, "cp_chain_fwd: bad B=%d N=%d", p.B, p.N);
  CP_REQUIRE(p.num_layers >= 1 && p.num_layers <= 3, CP_E_INVALID, "cp_chain_fwd: num_layers=%d outside [1,3]", p.num_layers);
  CP_REQUIRE(p.out && p.ld_out > 0, CP_E_INVALID, "cp_chain_fwd: no output buffer");
  int kin0 = 0;
  switch (p.prologue) {
    case CP_PRO_LOAD:
      CP_REQUIRE(p.src && pow2_64_256(p.C) && p.ld_src >= p.C && (p.ld_src % 8) == 0, CP_E_UNSUPPORTED,
                 "cp_chain_fwd(LOAD): need C in {64,128,256}, ld %% 8 == 0 (C=%d ld=%d)", p.C, p.ld_src);
      kin0 = p.C;
      break;
    case CP_PRO_AGG:
      CP_REQUIRE(p.z && p.idx && pow2_64_256(p.Co) && p.ld_z >= 2 * p.Co && (p.ld_z % 8) == 0, CP_E_UNSUPPORTED,
                 "cp_chain_fwd(AGG): need Co in {64,128,256} (Co=%d ld_z=%d)", p.Co, p.ld_z);
      CP_REQUIRE(p.K >= 1 && p.K <= 64, CP_E_UNSUPPORTED, "cp_chain_fwd(AGG): K=%d outside [1,64]", p.K);
      CP_REQUIRE(!p.a_out || (p.ld_a_out >= p.Co && (p.ld_a_out % 8) == 0), CP_E_INVALID, "cp_chain_fwd(AGG): bad ld_a_out");
      kin0 = p.Co;
      break;
    case CP_PRO_TAPS:
      CP_REQUIRE(p.patches && p.x_id && p.y_id && p.graph_feat, CP_E_INVALID, "cp_chain_fwd(TAPS): null pointer");
      CP_REQUIRE(p.E == 64 && pow2_64_256(p.Cg) && p.ld_gf >= p.Cg && (p.ld_gf % 8) == 0 && p.tap_step > 0, CP_E_UNSUPPORTED,
                 "cp_chain_fwd(TAPS): need E == 64 and Cg in {64,128,256} (E=%d Cg=%d)", p.E, p.Cg);
      kin0 = 4 * p.E + p.Cg;
      break;
    default:
      CP_REQUIRE(false, CP_E_INVALID, "cp_chain_fwd: bad prologue %d", p.prologue);
  }
  if (p.prologue == CP_PRO_TAPS) {   // the shipped refine-stage shapes run on the warp-specialised kernel
    bool shapes_ok = true;
    for (int l = 0; l < p.num_layers; ++l) shapes_ok = shapes_ok && p.layers[l].w_packed && (reinterpret_cast<uintptr_t>(p.layers[l].w_packed) & 15) == 0;
    int rc = CP_OK;
    if (shapes_ok && (p.ld_out % 8) == 0 && cp::taps_chain_try(p, (cudaStream_t)s, &rc)) return rc;
  }
  KParams kp;
  kp.p = p;
  kp.tiles_per_roi = (p.N + TILE_M - 1) / TILE_M;
  kp.num_node_tiles = kp.tiles_per_roi * p.B;
  int T = 0;
  int kin_expected = kin0;
  for (int l = 0; l < p.num_layers; ++l) {
    const cp_chain_layer& L = p.layers[l];
    const bool last = (l == p.num_layers - 1);
    CP_REQUIRE(L.w_packed && L.nout >= 1, CP_E_INVALID, "cp_chain_fwd: layer %d has no weights", l);
    CP_REQUIRE(L.kin == kin_expected, CP_E_INVALID, "cp_chain_fwd: layer %d kin=%d but its input has %d channels", l, L.kin, kin_expected);
    CP_REQUIRE((reinterpret_cast<uintptr_t>(L.w_packed) & 15) == 0, CP_E_INVALID, "cp_chain_fwd: layer %d weights not 16-byte aligned", l);
    const int npad = (L.nout + 15) & ~15;
    const int max_n = (last && p.out_mode == CP_OUT_BF16) ? 512 : 256;
    CP_REQUIRE(npad <= max_n, CP_E_UNSUPPORTED, "cp_chain_fwd: layer %d nout=%d too wide", l, L.nout);
    CP_REQUIRE(last || (npad % 64) == 0, CP_E_UNSUPPORTED, "cp_chain_fwd: chained layer %d needs nout %% 64 == 0", l);
    const bool two_phase = (p.prologue == CP_PRO_TAPS && l == 0);
    CP_REQUIRE(two_phase || L.kin <= 256, CP_E_UNSUPPORTED, "cp_chain_fwd: layer %d kin=%d > 256", l, L.kin);
    const int npass = (npad + TMEM_COLS - 1) / TMEM_COLS;
    for (int pass = 0; pass < npass; ++pass) {
      const int col0 = pass * TMEM_COLS;
      const int pcols = (npad - col0 < TMEM_COLS) ? (npad - col0) : TMEM_COLS;
      const int nblk = (pcols + 127) / 128;
      const int nphase = two_phase ? 2 : 1;
      for (int ph = 0; ph < nphase; ++ph) {
        const int kc_begin = (two_phase && ph == 1) ? 4 : 0;
        const int kc_count = two_phase ? (ph == 0 ? 4 : p.Cg / 64) : L.kin / 64;
        for (int nbi = 0; nbi < nblk; ++nbi) {
          for (int kci = 0; kci < kc_count; ++kci) {
            CP_REQUIRE(T < MAX_WTILES, CP_E_UNSUPPORTED, "cp_chain_fwd: weight tile table overflow");
            kp.wt[T++] = cp::packed_tile(L.w_packed, col0 / 128 + nbi, kc_begin + kci, L.kin, npad);
          }
        }
      }
    }
    kin_expected = npad;
    if (!last) CP_REQUIRE(npad == L.nout, CP_E_UNSUPPORTED, "cp_chain_fwd: chained layer %d nout must be a multiple of 16", l);
  }
  kp.T = T;
  if (p.out_mode == CP_OUT_BF16)
    CP_REQUIRE((p.ld_out % 8) == 0, CP_E_INVALID, "cp_chain_fwd: bf16 output needs ld_out %% 8 == 0");
  else
    CP_REQUIRE(p.out_mode == CP_OUT_F32 && p.n_valid >= 1 && p.n_valid <= p.ld_out, CP_E_INVALID, "cp_chain_fwd: bad f32 output spec");

  const int num_sms = cp::num_sms();
  int grid = kp.num_node_tiles < 2 * num_sms ? kp.num_node_tiles : 2 * num_sms;
  cudaStream_t st = (cudaStream_t)s;
  cudaError_t e = cudaSuccess;
  switch (p.prologue) {
    case CP_PRO_LOAD:
      e = cudaFuncSetAttribute(chain_kernel<CP_PRO_LOAD>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
      if (e == cudaSuccess) chain_kernel<CP_PRO_LOAD><<<grid, NTHREADS, SMEM_BYTES, st>>>(kp);
      break;
    case CP_PRO_AGG:
      e = cudaFuncSetAttribute(chain_kernel<CP_PRO_AGG>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
      if (e == cudaSuccess) chain_kernel<CP_PRO_AGG><<<grid, NTHREADS, SMEM_BYTES, st>>>(kp);
      break;
    default:
      e = cudaFuncSetAttribute(chain_kernel<CP_PRO_TAPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
      if (e == cudaSuccess) chain_kernel<CP_PRO_TAPS><<<grid, NTHREADS, SMEM_BYTES, st>>>(kp);
      break;
  }
  CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "cp_chain_fwd: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
  CP_CHECK_LAUNCH("cp_chain_fwd");
  return CP_OK;
}
