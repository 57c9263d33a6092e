// K1 for wide features (C > 64): kNN on node features, e.g. knn(x, k) + get_graph_feature in the DGCNN style.
//
// Contract = knn_kernel's (knn.cu), bit for bit: the k nearest by the fp32 direct-difference distance
//     d_ij = fmaf(t, t, d) over c = 0 .. C-1 in that order, t = x[c, j] - x[c, i],
// ordered by (d, j).  At C = 3 a distance is three FMAs; at C = 64 ... 1024 it is a dot product, and the tensor pipe
// can take the N x N x C part of the work.  It cannot decide the result (bf16 operands, an accumulation order we do
// not control), so here the tensor cores only prune and exact fp32 decides:
//
//   Gram tile.  One CTA per (RoI, 128 query points).  Candidates come in tiles of 128 points; per K chunk of 64
//   channels, loader warps read x coalesced along N (one thread per point), split each fp32 value into bf16 hi + lo
//   (the scheme of gemm_x3_tcgen05.cu) and write the K-major SWIZZLE_128B operand tiles; the same threads accumulate
//   each point's fp32 squared norm n_j.  One thread issues g~ = A_hi B_hi^T + A_hi B_lo^T + A_lo B_hi^T (3 x 4
//   tcgen05.mma, M = N = 128, K = 16) into one of two 128-column TMEM accumulators.
//   Approximate distance  d~_ij = n_i + n_j - 2 g~_ij  (fp32), with a bound |d~_ij - d_ij| <= eps_ij (below).
//
//   Two passes over the candidate tiles, both on the tensor cores:
//     pass 1  T_i = k-th smallest of d~_ij + eps_ij over all j (a per-row sorted list in shared memory).  At least k
//             candidates have d_ij <= T_i, so the row's k-th exact distance is <= T_i.
//     pass 2  the same tiles again; a candidate with d~_ij - eps_ij <= T_i (every j with d_ij <= T_i passes) is rescored
//             exactly from x in channel order and inserted into the row's sorted (d, j) list.  Candidates arrive in
//             increasing j and are inserted after equal distances, so the list is the (d, j)-ordered top k, exactly
//             what knn_kernel keeps.  Ties and duplicates only widen the band; nothing is ever dropped, so no overflow
//             path is needed.  When eps is larger than the spread of the distances (a large common offset, n_i >> d_ij)
//             every candidate passes and pass 2 is an exact scan.
//
// The bound, u = 2^-24, gamma_n = n u / (1 - n u), N_i = exact squared norm, D_ij = exact real distance:
//   * bf16 split: |x - hi| <= 2^-8 |x|, lo = bf16(x - hi), |x - hi - lo| <= 2^-16 |x|; the dropped terms
//     a_lo b_lo + r_a b + a r_b + r_a r_b are <= 3.01 * 2^-16 |a||b| per channel.
//   * tensor-core accumulation of the 3 * 64 * KC bf16 products (each exact in fp32): assumed <= 2^-20 relative per
//     addition w.r.t. the sum of |terms| (8x the truncating fp32 adder's 2^-23, to allow for alignment loss), i.e.
//     gamma'_n * 1.02 * sum_c |a_c||b_c|, n = 3 * 64 * KC.
//     With Cauchy-Schwarz, sum_c |a_c||b_c| <= sqrt(N_i N_j):   |g~ - G| <= (3.1 * 2^-16 + 1.02 gamma'_n) sqrt(N_i N_j).
//   * norms: |n_i - N_i| <= gamma_C N_i.   Evaluating n_i + n_j - 2 g~ in fp32: <= 3.2 u (n_i + n_j).
//   * the exact path's own rounding: |d_ij - D_ij| <= gamma_{C+2} D_ij, and D_ij <= 2 (N_i + N_j).
//   * denormals: bf16 lo parts below 2^-126 and products below 2^-126 may be flushed by the tensor pipe:
//     <= 2^-126 * 1.01 * sqrt(C) (sqrt(N_i) + sqrt(N_j)) + 3 * 64 * KC * 2^-126.
//   With N_i <= n_i / (1 - gamma_C) this gives
//     eps_ij = alpha sqrt(n_i n_j) + beta (n_i + n_j) + gamma (sqrt(n_i) + sqrt(n_j)) + eps0,
//   whose coefficients the host evaluates in double and doubles, which covers the fp32 evaluation of eps, d~ +- eps
//   and the comparisons.
//
// Roles (13 warps, one CTA per SM: 194 KB of shared memory):
//   warps 0-3   selection: warp q owns TMEM lanes / query rows [32 q, 32 q + 32), one row per thread; sorted lists in
//               shared memory ([slot][row], 128 x 64 x (4 + 4) bytes); pass 2 rescoring reads x from global memory
//               (L1 / L2: a query's column is coalesced across the warp, candidates are gathered);
//   warp 4      TMEM allocation + MMA issue;
//   warps 5-12  loaders: threads 0-127 the query tile rows, 128-255 the candidate tile rows; two operand stages.
// No N x N buffer exists anywhere; the kernel allocates nothing.
#include "common.cuh"
#include "sm100.cuh"

using namespace sm100;

namespace {

constexpr int TILE = 128;                       // query rows per CTA = candidates per tile
constexpr int NUM_SEL_WARPS = 4, MMA_WARP = 4, LOAD_WARP0 = 5, NUM_LOAD_WARPS = 8;
constexpr int NTHREADS = (LOAD_WARP0 + NUM_LOAD_WARPS) * 32;
constexpr int STAGES = 2;
constexpr int OP_BYTES = TILE * 128;            // one 64-wide bf16 K chunk of 128 rows
constexpr int STAGE_BYTES = 4 * OP_BYTES;       // A_hi, A_lo, B_hi, B_lo
constexpr int KMAX = 64;
constexpr int OFF_LIST_D = STAGES * STAGE_BYTES;
constexpr int OFF_LIST_J = OFF_LIST_D + KMAX * TILE * 4;
constexpr int OFF_NORM = OFF_LIST_J + KMAX * TILE * 4;   // float normA[2][128] (n, sqrt n), normB[2 slots][2][128]
constexpr int OFF_BAR = OFF_NORM + 6 * TILE * 4;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;        // + alignment slack
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
constexpr uint32_t TMEM_COLS = 256;                      // two 128-column accumulators

struct Bars {
  uint64_t full[STAGES], empty[STAGES];
  uint64_t acc_full[2], acc_empty[2], norm_full[2];
  uint32_t tmem_slot;
};

struct KnnParams {
  const float* x;
  int C, N, k, KC, NT;    // K chunks of 64 channels; candidate tiles
  float alpha, beta, gamma, eps0;
  int64_t* idx64;
  int32_t* idx32;
};

__device__ __forceinline__ float bf_round(float a) { return __bfloat162float(__float2bfloat16_rn(a)); }

// ------------------------------------------------------------------------------------------------------
// loaders: thread t < 128 owns query row t, t >= 128 candidate row t - 128 of the current tile.  Per K chunk: 64 scalar
// loads (coalesced along N across the warp), hi / lo split, two 16-byte stores per 8 channels into the swizzled tiles.
__device__ void loader(const KnnParams& kp, uint8_t* sm, Bars* bars, float* norms, int t) {
  const bool is_a = t < TILE;
  const int r = t & (TILE - 1);
  const int lane = t & 31;
  const float* xb = kp.x + (size_t)blockIdx.y * kp.C * kp.N;
  const uint32_t op = smem_u32(sm) + (is_a ? 0u : 2u * OP_BYTES);
  const int q = blockIdx.x * TILE + r;
  uint32_t it = 0;
  for (int tile = 0; tile < 2 * kp.NT; ++tile) {
    const int n = is_a ? q : (tile % kp.NT) * TILE + r;
    const bool ok = n < kp.N;
    float nrm = 0.f;
    for (int kc = 0; kc < kp.KC; ++kc, ++it) {
      float v[64];
      const int c0 = kc * 64;
#pragma unroll
      for (int e = 0; e < 64; ++e) v[e] = (ok && c0 + e < kp.C) ? __ldg(xb + (size_t)(c0 + e) * kp.N + n) : 0.f;
      const uint32_t s = it % STAGES;
      if (it >= STAGES) mbar_wait(&bars->empty[s], ((it / STAGES) - 1) & 1);
      const uint32_t hi = op + s * STAGE_BYTES, lo = hi + OP_BYTES;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        uint32_t h[4], l[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float a = v[u * 8 + 2 * e], b = v[u * 8 + 2 * e + 1];
          const float ha = bf_round(a), hb = bf_round(b);
          h[e] = f2_to_bf2(ha, hb);
          l[e] = f2_to_bf2(a - ha, b - hb);
          nrm = fmaf(a, a, nrm);
          nrm = fmaf(b, b, nrm);
        }
        const uint32_t off = (uint32_t)(r * 128 + ((u ^ (r & 7)) << 4));
        sts128(hi + off, make_uint4(h[0], h[1], h[2], h[3]));
        sts128(lo + off, make_uint4(l[0], l[1], l[2], l[3]));
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->full[s]);
    }
    // norms of this tile: the selection warps read them once the accumulator slot's previous tile is done with
    const uint32_t slot = tile & 1;
    if (tile >= 2) mbar_wait(&bars->acc_empty[slot], ((tile >> 1) - 1) & 1);
    if (!is_a) {
      norms[2 * TILE + slot * 2 * TILE + r] = nrm;
      norms[2 * TILE + slot * 2 * TILE + TILE + r] = sqrtf(nrm);
    } else if (tile == 0) {
      norms[r] = nrm;
      norms[TILE + r] = sqrtf(nrm);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&bars->norm_full[slot]);
  }
}

__device__ void mma_issuer(const KnnParams& kp, uint8_t* sm, Bars* bars, uint32_t tmem_base) {
  const uint32_t sm_base = smem_u32(sm);
  const uint32_t idesc = make_idesc_bf16_m128(TILE);
  uint32_t it = 0;
  for (int tile = 0; tile < 2 * kp.NT; ++tile) {
    const uint32_t slot = tile & 1;
    if (tile >= 2) mbar_wait(&bars->acc_empty[slot], ((tile >> 1) - 1) & 1);
    tc_fence_after_sync();
    const uint32_t d = tmem_base + slot * TILE;
    for (int kc = 0; kc < kp.KC; ++kc, ++it) {
      const uint32_t s = it % STAGES;
      mbar_wait(&bars->full[s], (it / STAGES) & 1);
      tc_fence_after_sync();
      const uint32_t a_hi = smem_desc_lo(sm_base + s * STAGE_BYTES), a_lo = a_hi + (OP_BYTES >> 4);
      const uint32_t b_hi = a_hi + (2 * OP_BYTES >> 4), b_lo = b_hi + (OP_BYTES >> 4);
      if (elect_one()) {
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) {
          mma_bf16_ss_lo(d, a_hi + 2 * k, b_hi + 2 * k, idesc, (uint32_t)((kc | (int)k) != 0));
          mma_bf16_ss_lo(d, a_hi + 2 * k, b_lo + 2 * k, idesc, 1u);
          mma_bf16_ss_lo(d, a_lo + 2 * k, b_hi + 2 * k, idesc, 1u);
        }
        mma_commit(&bars->empty[s]);
        if (kc == kp.KC - 1) mma_commit(&bars->acc_full[slot]);
      }
      __syncwarp();
    }
  }
}

// exact fp32 direct-difference distance, channels in order (knn_kernel's arithmetic)
__device__ __forceinline__ float exact_dist(const float* __restrict__ xb, int C, int N, int i, int j) {
  const float* pi = xb + i;
  const float* pj = xb + j;
  float d = 0.f;
  int c = 0;
  for (; c + 8 <= C; c += 8) {
    float a[8], b[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      a[e] = __ldg(pj + (size_t)(c + e) * N);
      b[e] = __ldg(pi + (size_t)(c + e) * N);
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float t = a[e] - b[e];
      d = fmaf(t, t, d);
    }
  }
  for (; c < C; ++c) {
    const float t = __ldg(pj + (size_t)c * N) - __ldg(pi + (size_t)c * N);
    d = fmaf(t, t, d);
  }
  return d;
}

// selection warp q, thread = query row 32 q + lane
__device__ void selector(const KnnParams& kp, uint8_t* sm, Bars* bars, const float* norms, uint32_t tmem_base, int q, int lane) {
  const int r = q * 32 + lane;
  const int i = blockIdx.x * TILE + r;
  const bool row_ok = i < kp.N;
  const int k = kp.k;
  const float* xb = kp.x + (size_t)blockIdx.y * kp.C * kp.N;
  float* ld = reinterpret_cast<float*>(sm + OFF_LIST_D) + r;   // element p at ld[p * TILE]
  int* lj = reinterpret_cast<int*>(sm + OFF_LIST_J) + r;
  const float INF = __int_as_float(0x7f800000);
  for (int p = 0; p < k; ++p) ld[p * TILE] = INF;
  float thr = INF;          // pass 1: current k-th smallest upper bound;  pass 2: current k-th exact distance
  float T = INF;            // pass 2: the certified threshold of pass 1
  float ni = 0.f, ri = 0.f;
  for (int tile = 0; tile < 2 * kp.NT; ++tile) {
    const bool pass2 = tile >= kp.NT;
    const int j0 = (tile % kp.NT) * TILE;
    const uint32_t slot = tile & 1, ph = (tile >> 1) & 1;
    mbar_wait(&bars->norm_full[slot], ph);
    mbar_wait(&bars->acc_full[slot], ph);
    tc_fence_after_sync();
    if (tile == 0) {
      ni = norms[r];
      ri = norms[TILE + r];
    }
    const float* nb = norms + 2 * TILE + slot * 2 * TILE;
    const uint32_t tb = tmem_base + ((uint32_t)(q * 32) << 16) + slot * TILE;
    uint32_t mask[TILE / 32];
#pragma unroll
    for (int c0 = 0; c0 < TILE; c0 += 32) {
      uint32_t g[32];
      tmem_ld32(tb + (uint32_t)c0, g);
      tmem_ld_wait();
      uint32_t m = 0;
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const int jl = c0 + e;
        const float nj = nb[jl], rj = nb[TILE + jl];
        const float dt = fmaf(-2.f, __uint_as_float(g[e]), ni + nj);
        const float eps = fmaf(kp.alpha, ri * rj, fmaf(kp.beta, ni + nj, fmaf(kp.gamma, ri + rj, kp.eps0)));
        const bool cand = row_ok && j0 + jl < kp.N;
        if (!pass2) {
          const float ub = dt + eps;
          if (cand && ub < thr) {   // sorted insertion of the upper bound
            int p = k - 1;
            while (p > 0 && ld[(p - 1) * TILE] > ub) {
              ld[p * TILE] = ld[(p - 1) * TILE];
              --p;
            }
            ld[p * TILE] = ub;
            thr = ld[(k - 1) * TILE];
          }
        } else if (cand && dt - eps <= T) {
          m |= 1u << e;
        }
      }
      if (pass2) mask[c0 >> 5] = m;
    }
    // the accumulator and this slot's norms are no longer needed
    tc_fence_before_sync();
    __syncwarp();
    if (lane == 0) mbar_arrive(&bars->acc_empty[slot]);
    if (!pass2) {
      if (tile == kp.NT - 1) {   // end of pass 1: certified threshold, fresh list for the exact distances
        T = thr;
        thr = INF;
        for (int p = 0; p < k; ++p) {
          ld[p * TILE] = INF;
          lj[p * TILE] = -1;
        }
      }
      continue;
    }
#pragma unroll 1
    for (int w = 0; w < TILE / 32; ++w) {
      uint32_t m = mask[w];
      while (m) {
        const int j = j0 + w * 32 + __ffs(m) - 1;
        m &= m - 1;
        const float d = exact_dist(xb, kp.C, kp.N, i, j);
        if (d < thr) {   // after every equal distance: candidates arrive in increasing j
          int p = k - 1;
          while (p > 0 && ld[(p - 1) * TILE] > d) {
            ld[p * TILE] = ld[(p - 1) * TILE];
            lj[p * TILE] = lj[(p - 1) * TILE];
            --p;
          }
          ld[p * TILE] = d;
          lj[p * TILE] = j;
          thr = ld[(k - 1) * TILE];
        }
      }
    }
  }
  if (!row_ok) return;
  const size_t o = ((size_t)blockIdx.y * kp.N + i) * k;
  for (int p = 0; p < k; ++p) {
    const int j = lj[p * TILE];
    kp.idx64[o + p] = j;
    if (kp.idx32) kp.idx32[o + p] = j;
  }
}

__global__ void __launch_bounds__(NTHREADS, 1) knn_tcgen05_kernel(const __grid_constant__ KnnParams kp) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  Bars* bars = reinterpret_cast<Bars*>(sm + OFF_BAR);
  float* norms = reinterpret_cast<float*>(sm + OFF_NORM);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&bars->full[s], NUM_LOAD_WARPS);
      mbar_init(&bars->empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&bars->acc_full[a], 1);
      mbar_init(&bars->acc_empty[a], NUM_SEL_WARPS);
      mbar_init(&bars->norm_full[a], NUM_LOAD_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == MMA_WARP) tmem_alloc(&bars->tmem_slot, TMEM_COLS);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = bars->tmem_slot;

  if (warp >= LOAD_WARP0) loader(kp, sm, bars, norms, threadIdx.x - LOAD_WARP0 * 32);
  else if (warp == MMA_WARP) mma_issuer(kp, sm, bars, tmem_base);
  else selector(kp, sm, bars, norms, tmem_base, warp, lane);

  tc_fence_before_sync();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc(tmem_base, TMEM_COLS);
}

}  // namespace

// C > 64: called by cp_knn (knn.cu) after its argument checks
int cp::knn_wide(const float* x, int B, int C, int N, int k, int64_t* idx64, int32_t* idx32, cudaStream_t st) {
  KnnParams kp;
  kp.x = x;
  kp.C = C;
  kp.N = N;
  kp.k = k;
  kp.KC = cp::ceil_div(C, 64);
  kp.NT = cp::ceil_div(N, TILE);
  kp.idx64 = idx64;
  kp.idx32 = idx32;
  // eps coefficients (header comment), evaluated in double and doubled
  const double u = 1.0 / (1 << 24), tiny = 1.1754943508222875e-38;   // 2^-24, 2^-126
  const double nprod = 3.0 * 64.0 * kp.KC;
  const double gC = C * u < 0.5 ? C * u / (1.0 - C * u) : INFINITY;
  const double gC2 = (C + 2) * u < 0.5 ? (C + 2) * u / (1.0 - (C + 2) * u) : INFINITY;
  const double ua = 1.0 / (1 << 20);
  const double gacc = nprod * ua < 0.5 ? nprod * ua / (1.0 - nprod * ua) : INFINITY;
  const double inv = 1.0 / (1.0 - gC);
  kp.alpha = (float)(2.0 * 2.0 * (3.1 / 65536.0 + 1.02 * gacc) * inv);
  kp.beta = (float)(2.0 * (gC * inv + 3.2 * u + 2.0 * gC2 * inv));
  kp.gamma = (float)(2.0 * 2.0 * tiny * 1.01 * sqrt((double)C) * sqrt(inv));
  kp.eps0 = (float)(2.0 * 2.0 * nprod * tiny);
  const dim3 grid(kp.NT, B);
  cudaError_t e = cudaFuncSetAttribute(knn_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "cp_knn: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
  knn_tcgen05_kernel<<<grid, NTHREADS, SMEM_BYTES, st>>>(kp);
  CP_CHECK_LAUNCH("cp_knn");
  return CP_OK;
}
