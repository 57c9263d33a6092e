// K1: kNN graph construction.
//
// Replaces knn(x, k) of checkerpose/model/pipeline.py:18-23 (identical copies in init.py:27-32,
// pipeline_lm.py:18-23, init_lm.py:27-32): negative squared pairwise distance + topk(k).
//
// The graph is static (built once per module in __init__ on C=3 normalised keypoints), so this
// kernel is off the per-RoI loop; it must however be fp32-exact: on the shipped FPS clouds the gap
// between the k-th and (k+1)-th neighbour is ~1e-4 relative, which bf16/TF32 distance tiles would
// not resolve (SURVEY.md section 8c).  A C=3 distance is three FMAs, so the tensor pipe has nothing to
// offer here and selection is the cost: distances are formed by direct differences in fp32
// registers (more accurate than the reference's  -|x|^2 + 2x.y - |y|^2  expansion) and each warp
// keeps its query's k best in a register-resident sorted list (two slots per lane, k <= 64) that is
// updated with ballot/shuffle insertion -- no per-query N-long row ever exists in memory, whereas
// the reference materialises the (N,N) matrix (64 MB per object at N=4096).
//
// Block = 8 warps = 8 queries at a time; candidate points are staged through shared memory in
// coalesced tiles shared by the 8 warps.  C <= 64 only: wider inputs (feature-space graphs) go to
// knn_tcgen05.cu, which returns the same (d, j)-ordered result with tensor-core pruning.
#include "common.cuh"

namespace {

constexpr int KNN_WARPS = 8;
constexpr int KNN_TILE = 256;  // candidates per smem tile

template <int CMAX>
__global__ void __launch_bounds__(KNN_WARPS * 32)
knn_kernel(const float* __restrict__ x, int C, int N, int k, int64_t* __restrict__ idx64,
           int32_t* __restrict__ idx32) {
  extern __shared__ float smem[];
  float* tile = smem;                       // [C][KNN_TILE]
  float* qbuf = smem + (size_t)C * KNN_TILE;  // [KNN_WARPS][C]
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* xb = x + (size_t)b * C * N;
  const int q = blockIdx.x * KNN_WARPS + warp;  // query handled by this warp
  const bool active = q < N;
  float* myq = qbuf + warp * C;
  if (active)
    for (int c = lane; c < C; c += 32) myq[c] = xb[(size_t)c * N + q];
  float qreg[CMAX > 0 ? CMAX : 1];
  __syncwarp();
  if (CMAX > 0 && active) {
#pragma unroll
    for (int c = 0; c < CMAX; ++c) qreg[c] = myq[c];
  }

  const float INF = __int_as_float(0x7f800000);
  float d0 = INF, d1 = INF;  // slots lane and lane+32 of the sorted list
  int i0 = -1, i1 = -1;
  float thresh = INF;

  for (int base = 0; base < N; base += KNN_TILE) {
    __syncthreads();
    for (int e = threadIdx.x; e < C * KNN_TILE; e += blockDim.x) {
      int c = e / KNN_TILE, j = e - c * KNN_TILE;
      tile[e] = (base + j < N) ? xb[(size_t)c * N + base + j] : 0.f;
    }
    __syncthreads();
    if (!active) continue;
    const int lim = min(KNN_TILE, N - base);
    for (int j0 = 0; j0 < lim; j0 += 32) {
      const int j = j0 + lane;
      float d = INF;
      if (j < lim) {
        d = 0.f;
        if (CMAX > 0) {
#pragma unroll
          for (int c = 0; c < CMAX; ++c) {
            float t = tile[c * KNN_TILE + j] - qreg[c];
            d = fmaf(t, t, d);
          }
        } else {
          for (int c = 0; c < C; ++c) {
            float t = tile[c * KNN_TILE + j] - myq[c];
            d = fmaf(t, t, d);
          }
        }
      }
      unsigned m = __ballot_sync(0xffffffffu, d < thresh);
      while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const float dj = __shfl_sync(0xffffffffu, d, src);
        if (!(dj < thresh)) continue;  // warp-uniform
        const int jj = base + j0 + src;
        // number of list entries <= dj  (list is sorted, so this is the insertion slot)
        const int pos = __popc(__ballot_sync(0xffffffffu, d0 <= dj)) + __popc(__ballot_sync(0xffffffffu, d1 <= dj));
        const float up0 = __shfl_up_sync(0xffffffffu, d0, 1);
        const int ui0 = __shfl_up_sync(0xffffffffu, i0, 1);
        float up1 = __shfl_up_sync(0xffffffffu, d1, 1);
        int ui1 = __shfl_up_sync(0xffffffffu, i1, 1);
        const float t31 = __shfl_sync(0xffffffffu, d0, 31);
        const int ti31 = __shfl_sync(0xffffffffu, i0, 31);
        if (lane == 0) { up1 = t31; ui1 = ti31; }
        if (lane > pos) { d0 = up0; i0 = ui0; } else if (lane == pos) { d0 = dj; i0 = jj; }
        const int s1 = lane + 32;
        if (s1 > pos) { d1 = up1; i1 = ui1; } else if (s1 == pos) { d1 = dj; i1 = jj; }
        thresh = (k - 1 < 32) ? __shfl_sync(0xffffffffu, d0, k - 1) : __shfl_sync(0xffffffffu, d1, k - 1 - 32);
      }
    }
  }
  if (!active) return;
  const size_t o = ((size_t)b * N + q) * k;
  if (lane < k) {
    idx64[o + lane] = i0;
    if (idx32) idx32[o + lane] = i0;
  }
  if (lane + 32 < k) {
    idx64[o + lane + 32] = i1;
    if (idx32) idx32[o + lane + 32] = i1;
  }
}

}  // namespace

extern "C" int cp_knn(const float* x, int B, int C, int N, int k, int64_t* idx64, int32_t* idx32, cp_stream_t s) {
  CP_REQUIRE(x && idx64, CP_E_INVALID, "cp_knn: null pointer");
  CP_REQUIRE(B > 0 && C > 0 && N > 0, CP_E_INVALID, "cp_knn: bad shape B=%d C=%d N=%d", B, C, N);
  CP_REQUIRE(k >= 1 && k <= 64 && k <= N, CP_E_UNSUPPORTED, "cp_knn: need 1 <= k <= min(64, N), got k=%d N=%d", k, N);
  cudaStream_t st = (cudaStream_t)s;
  if (C > 64) return cp::knn_wide(x, B, C, N, k, idx64, idx32, st);
  dim3 grid(cp::ceil_div(N, KNN_WARPS), B);
  size_t smem = ((size_t)C * KNN_TILE + (size_t)KNN_WARPS * C) * sizeof(float);
  if (C == 3) {
    knn_kernel<3><<<grid, KNN_WARPS * 32, smem, st>>>(x, C, N, k, idx64, idx32);
  } else {
    if (smem > 48 * 1024) cudaFuncSetAttribute(knn_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    knn_kernel<0><<<grid, KNN_WARPS * 32, smem, st>>>(x, C, N, k, idx64, idx32);
  }
  CP_CHECK_LAUNCH("cp_knn");
  return CP_OK;
}
