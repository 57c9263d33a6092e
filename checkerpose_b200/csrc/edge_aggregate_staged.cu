// float32 EdgeConv aggregation on the graph plan:  y[b,i,:] = lrelu(max_k P[b, nbr(i,k), :] + Q[b,i,:]),  z = [P|Q] fp32.
//
// The float32 mode keeps fp32 tensors between layers (the GEMMs run on cp_gemm_x3), so the aggregation is a pure
// gather + max over fp32 rows.  The unstaged kernel (cp_edge_aggregate: one warp per node, rows gathered from L2) moves
// N * K * Co * 4 bytes per RoI through L2 (21 GB per launch at the benchmark shape, 3.6 ms).  This kernel uses the same
// graph plan as the bf16 tcgen05 kernel (graph_plan.cu): per tile of 128 plan-order nodes and 32-channel slice (128-byte
// row pieces, so the plan's byte offsets apply unchanged) the tile's DISTINCT neighbour rows are staged in shared memory
// once with cp.async (double-buffered over the slices), and a quarter-warp reduces one node PAIR of the plan's programs
// (shared rows once) with 128-bit shared-memory loads.
#include "common.cuh"
#include "sm100.cuh"

using sm100::cp_async16;

namespace {

constexpr int TILE = CP_PLAN_TILE;
constexpr int NTHREADS = 512;                  // 64 quarter-warps = the 64 node pairs of a tile
constexpr int UI = CP_PLAN_UMAX / CP_PLAN_LIST_LANES;

__device__ __forceinline__ float4 lds128f(uint32_t addr) {
  float4 r;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
  return r;
}
__device__ __forceinline__ float4 max4(float4 a, float4 b) {
  return make_float4(fmaxf(a.x, b.x), fmaxf(a.y, b.y), fmaxf(a.z, b.z), fmaxf(a.w, b.w));
}

__global__ void __launch_bounds__(NTHREADS, 2)
edge_aggregate_staged_kernel(const float* __restrict__ z, float* __restrict__ y, cp_graph_plan pl, const int32_t* __restrict__ graph_sel,
                             float slope, int B, int N, int Co, int rows_cap, int num_tiles) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int KP = pl.KP, KCH = KP / 4, PW = 2 * KP + 8;
  const int prog_bytes = CP_PLAN_PAIRS * PW * 2;
  const uint32_t sm_base = (uint32_t)__cvta_generic_to_shared(smem);
  const uint32_t prog_s = sm_base, ring_s = sm_base + ((prog_bytes + 127) & ~127);
  const int tid = threadIdx.x, qw = tid >> 3, sub = tid & 7;
  const int KC = Co / 32;
  const int ld = 2 * Co;
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int b = tile / pl.T, t = tile - b * pl.T;
    const int g = graph_sel ? graph_sel[b] : 0;
    const size_t gt = (size_t)g * pl.T + t;
    const int U = pl.ucount[gt];
    const uint16_t* lst = pl.ulist + gt * CP_PLAN_UMAX;
    const float* zb = z + (size_t)b * N * ld;
    auto stage = [&](int c, int buf) {
      const uint32_t dst = ring_s + (uint32_t)buf * rows_cap * 128u + sub * 16;
      const float* src = zb + c * 32 + sub * 4;
      for (int j = qw; j < U; j += 64) {
        const int row = lst[(j & 63) * UI + (j >> 6)];
        cp_async16(dst + j * 128u, src + (size_t)row * ld);
      }
    };
    __syncthreads();     // the previous tile's readers are done with the programs and both buffers
    {
      const uint8_t* psrc = reinterpret_cast<const uint8_t*>(pl.prog) + gt * prog_bytes;
      for (int piece = tid; piece < prog_bytes / 16; piece += NTHREADS) cp_async16(prog_s + piece * 16, psrc + piece * 16);
    }
    stage(0, 0);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const int n0 = t * TILE;
    for (int c = 0; c < KC; ++c) {
      if (c + 1 < KC) stage(c + 1, (c + 1) & 1);
      asm volatile("cp.async.commit_group;" ::: "memory");
      asm volatile("cp.async.wait_group 1;" ::: "memory");
      __syncthreads();
      const uint32_t stg = ring_s + (uint32_t)(c & 1) * rows_cap * 128u + sub * 16;
      const uint32_t pe = prog_s + qw * (PW * 2);
      uint32_t info;
      asm volatile("ld.shared.u32 %0, [%1];" : "=r"(info) : "r"(pe + 2 * KP * 2));
      const int na = info & 255, nb = (info >> 8) & 255;
      const int nc4 = info >> 18, nr4 = KCH - nc4;
      const float NEG = -__int_as_float(0x7f800000);
      float4 acc = make_float4(NEG, NEG, NEG, NEG);
      uint32_t pa = pe;
      auto quad = [&](float4 m, uint32_t pp) {
        uint32_t w0, w1;
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(w0), "=r"(w1) : "r"(pp));
        const float4 v0 = lds128f(stg + (w0 & 0xffffu)), v1 = lds128f(stg + (w0 >> 16));
        const float4 v2 = lds128f(stg + (w1 & 0xffffu)), v3 = lds128f(stg + (w1 >> 16));
        return max4(max4(m, max4(v0, v1)), max4(v2, v3));
      };
      for (int j = 0; j < nc4; ++j, pa += 8) acc = quad(acc, pa);
      float4 accb = acc;
      uint32_t pb = pe + KP * 2;
      for (int j = 0; j < nr4; ++j, pa += 8, pb += 8) {
        acc = quad(acc, pa);
        accb = quad(accb, pb);
      }
      const int ch = c * 32 + sub * 4;
      if (na != 255) {
        const size_t node = (size_t)b * N + n0 + na;
        const float4 q = __ldg(reinterpret_cast<const float4*>(z + node * ld + Co + ch));
        *reinterpret_cast<float4*>(y + node * Co + ch) =
            make_float4(cp::lrelu(acc.x + q.x, slope), cp::lrelu(acc.y + q.y, slope), cp::lrelu(acc.z + q.z, slope), cp::lrelu(acc.w + q.w, slope));
      }
      if (nb != 255) {
        const size_t node = (size_t)b * N + n0 + nb;
        const float4 q = __ldg(reinterpret_cast<const float4*>(z + node * ld + Co + ch));
        *reinterpret_cast<float4*>(y + node * Co + ch) =
            make_float4(cp::lrelu(accb.x + q.x, slope), cp::lrelu(accb.y + q.y, slope), cp::lrelu(accb.z + q.z, slope), cp::lrelu(accb.w + q.w, slope));
      }
      __syncthreads();   // buffer (c & 1) is refilled by the next iteration's stage(c + 2)
    }
  }
}

}  // namespace

extern "C" int cp_edge_aggregate_staged_f32(const float* z, const cp_graph_plan* plan, const int32_t* graph_sel, float slope, float* y,
                                            int B, int N, int Co, cp_stream_t s) {
  CP_REQUIRE(z && y && plan && B > 0 && N > 0, CP_E_INVALID, "cp_edge_aggregate_staged_f32: bad arguments");
  const cp_graph_plan& pl = *plan;
  CP_REQUIRE(Co > 0 && Co % 32 == 0 && ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(y)) & 15) == 0, CP_E_UNSUPPORTED,
             "cp_edge_aggregate_staged_f32: Co=%d must be a multiple of 32, tensors 16-byte aligned", Co);
  CP_REQUIRE(pl.ucount && pl.ulist && pl.prog && pl.N == N && pl.T == (N + TILE - 1) / TILE && pl.KP == cp_graph_plan_kp(pl.K) && pl.KP > 0 &&
             pl.umax == CP_PLAN_UMAX, CP_E_INVALID, "cp_edge_aggregate_staged_f32: graph plan does not match N=%d", N);
  CP_REQUIRE(pl.max_unique >= 1 && pl.max_unique <= CP_PLAN_UMAX, CP_E_UNSUPPORTED,
             "cp_edge_aggregate_staged_f32: a tile has %d distinct neighbour rows (> %d): use cp_edge_aggregate", pl.max_unique, CP_PLAN_UMAX);
  CP_REQUIRE((size_t)N * 2 * Co * 4 < (1ull << 32), CP_E_UNSUPPORTED, "cp_edge_aggregate_staged_f32: one RoI's table must be < 4 GB");
  const int rows_cap = (pl.max_unique + 7) & ~7;
  const int prog_bytes = CP_PLAN_PAIRS * (2 * pl.KP + 8) * 2;
  const int smem = ((prog_bytes + 127) & ~127) + 2 * rows_cap * 128;
  const int num_tiles = B * pl.T;
  cudaError_t e = cudaFuncSetAttribute(edge_aggregate_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "cp_edge_aggregate_staged_f32: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
  const int ctas_per_sm = smem <= 110 * 1024 ? 2 : 1;
  const int cap = cp::num_sms() * ctas_per_sm;
  const int grid = num_tiles < cap ? num_tiles : cap;
  edge_aggregate_staged_kernel<<<grid, NTHREADS, smem, (cudaStream_t)s>>>(z, y, pl, graph_sel, slope, B, N, Co, rows_cap, num_tiles);
  CP_CHECK_LAUNCH("cp_edge_aggregate_staged_f32");
  return CP_OK;
}
