// CUDA-core kernels of the GNN keypoint head: layout conversion, weight folding/packing, the fp32
// validation path (FFMA GEMM + EdgeConv aggregation + 4-tap gather) and the sign-bit decode.
// All of them are HBM/L2-bound byte movers or tiny; the tensor-core path lives in chain_tcgen05.cu.
#include "common.cuh"

using bf16 = __nv_bfloat16;

namespace {

// ------------------------------------------------------------------------------------------------
// (B, R, S) -> (B, S, R) tiled transpose with dtype conversion.  src[b][r][s], dst[b][s][r].
// ------------------------------------------------------------------------------------------------
template <typename TS, typename TD>
__global__ void transpose_kernel(const TS* __restrict__ src, TD* __restrict__ dst, int R, int S) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int s0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const TS* sb = src + (size_t)b * R * S;
  TD* db = dst + (size_t)b * R * S;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int r = r0 + i, sidx = s0 + threadIdx.x;
    if (r < R && sidx < S) tile[i][threadIdx.x] = cp::to_f32<TS>(sb[(size_t)r * S + sidx]);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int sidx = s0 + i, r = r0 + threadIdx.x;
    if (r < R && sidx < S) db[(size_t)sidx * R + r] = cp::from_f32<TD>(tile[threadIdx.x][i]);
  }
}

// bf16 -> bf16 with R and S multiples of 64 (NCHW <-> NHWC of the HRNet maps, (B,hw,N) -> (B,N,hw) of the init head):
// 64 x 64 tiles, 128-bit global accesses on both sides (a 128-byte line per 8 threads), transposition through a
// shared-memory tile of bf16 pairs with an odd row stride (conflict-free in both directions).
__global__ void __launch_bounds__(256) transpose_bf16_64_kernel(const uint16_t* __restrict__ src, uint16_t* __restrict__ dst, int R, int S) {
  __shared__ uint32_t tile[64][33];   // [r][pair of s]
  const int b = blockIdx.z;
  const int s0 = blockIdx.x * 64, r0 = blockIdx.y * 64;
  const uint16_t* sb = src + (size_t)b * R * S;
  uint16_t* db = dst + (size_t)b * R * S;
  const int t = threadIdx.x, v = t & 7, row = t >> 3;   // 8 threads x 16 B per 128-byte row, 32 rows per pass
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int r = row + 32 * h;
    const uint4 x = *reinterpret_cast<const uint4*>(sb + (size_t)(r0 + r) * S + s0 + v * 8);
    tile[r][v * 4 + 0] = x.x; tile[r][v * 4 + 1] = x.y; tile[r][v * 4 + 2] = x.z; tile[r][v * 4 + 3] = x.w;
  }
  __syncthreads();
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int sidx = row + 32 * h;   // output row = source column
    const int sel = (sidx & 1) ? 0x7632 : 0x5410;   // take the high / low halves of two words
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t a = tile[v * 8 + 2 * j][sidx >> 1], c = tile[v * 8 + 2 * j + 1][sidx >> 1];
      w[j] = __byte_perm(a, c, sel);
    }
    *reinterpret_cast<uint4*>(db + (size_t)(s0 + sidx) * R + r0 + v * 8) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// (B, R, S) -> (B, S, R) like the kernel above (R == 64: one output row = one 128-byte line), fused with the two steps
// that follow the init head's conv1x1 (init.py:113-114): + bias[s] (the conv bias: s = keypoint = conv channel) and the
// move of row s to row row_map[g(b)][s] (keypoint order -> plan order).
__global__ void __launch_bounds__(256) transpose_scatter_bf16_64_kernel(const uint16_t* __restrict__ src, uint16_t* __restrict__ dst, int R, int S,
                                                                        const float* __restrict__ bias, const int32_t* __restrict__ row_map,
                                                                        const int32_t* __restrict__ graph_sel) {
  __shared__ uint32_t tile[64][33];   // [r][pair of s]
  const int b = blockIdx.z;
  const int s0 = blockIdx.x * 64, r0 = blockIdx.y * 64;
  const uint16_t* sb = src + (size_t)b * R * S;
  uint16_t* db = dst + (size_t)b * R * S;
  const int t = threadIdx.x, v = t & 7, row = t >> 3;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int r = row + 32 * h;
    const uint4 x = *reinterpret_cast<const uint4*>(sb + (size_t)(r0 + r) * S + s0 + v * 8);
    tile[r][v * 4 + 0] = x.x; tile[r][v * 4 + 1] = x.y; tile[r][v * 4 + 2] = x.z; tile[r][v * 4 + 3] = x.w;
  }
  __syncthreads();
  const int g = (row_map && graph_sel) ? graph_sel[b] : 0;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int sidx = row + 32 * h;   // output row = source column
    const int sel = (sidx & 1) ? 0x7632 : 0x5410;
    const float bs = bias ? bias[s0 + sidx] : 0.f;
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t a = tile[v * 8 + 2 * j][sidx >> 1], c = tile[v * 8 + 2 * j + 1][sidx >> 1];
      w[j] = __byte_perm(a, c, sel);
      if (bias) {   // bf16 + f32 bias, rounded once (the reference adds the bias in the conv's accumulation type)
        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
        const __nv_bfloat162 o = __floats2bfloat162_rn(f.x + bs, f.y + bs);
        w[j] = *reinterpret_cast<const uint32_t*>(&o);
      }
    }
    const int drow = row_map ? row_map[(size_t)g * S + s0 + sidx] : s0 + sidx;
    *reinterpret_cast<uint4*>(db + (size_t)drow * R + r0 + v * 8) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// x (rows, C) bf16 += bias (C) f32, in place, 128-bit accesses: the bias of a library convolution that has no fused
// activation (torch runs it as a separate broadcast add at a fraction of the HBM rate).
__global__ void __launch_bounds__(256) bias_add_rows_kernel(uint4* __restrict__ x, const float* __restrict__ bias, int64_t vecs, int cv, int relu) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < vecs; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % cv) * 8;
    uint4 t = x[e];
    uint32_t w[4] = {t.x, t.y, t.z, t.w};
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + c)), b1 = __ldg(reinterpret_cast<const float4*>(bias + c + 4));
    const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
      float lo = f.x + bb[2 * i], hi = f.y + bb[2 * i + 1];
      if (relu) { lo = fmaxf(lo, 0.f); hi = fmaxf(hi, 0.f); }
      const __nv_bfloat162 o = __floats2bfloat162_rn(lo, hi);
      w[i] = *reinterpret_cast<const uint32_t*>(&o);
    }
    x[e] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

template <typename TS, typename TD>
int launch_transpose(const void* src, void* dst, int B, int R, int S, cudaStream_t st) {
  if (sizeof(TS) == 2 && sizeof(TD) == 2 && R % 64 == 0 && S % 64 == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
    dim3 grid(S / 64, R / 64, B);
    transpose_bf16_64_kernel<<<grid, 256, 0, st>>>((const uint16_t*)src, (uint16_t*)dst, R, S);
    return 0;
  }
  dim3 grid(cp::ceil_div(S, 32), cp::ceil_div(R, 32), B), block(32, 8);
  transpose_kernel<TS, TD><<<grid, block, 0, st>>>((const TS*)src, (TD*)dst, R, S);
  return 0;
}

int transpose_dispatch(const void* src, int sd, void* dst, int dd, int B, int R, int S, cudaStream_t st) {
  if (sd == CP_F32 && dd == CP_F32) return launch_transpose<float, float>(src, dst, B, R, S, st);
  if (sd == CP_F32 && dd == CP_BF16) return launch_transpose<float, bf16>(src, dst, B, R, S, st);
  if (sd == CP_BF16 && dd == CP_F32) return launch_transpose<bf16, float>(src, dst, B, R, S, st);
  if (sd == CP_BF16 && dd == CP_BF16) return launch_transpose<bf16, bf16>(src, dst, B, R, S, st);
  return -1;
}

template <typename TS, typename TD>
__global__ void convert_kernel(const TS* __restrict__ src, TD* __restrict__ dst, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) dst[i] = cp::from_f32<TD>(cp::to_f32<TS>(src[i]));
}

// ------------------------------------------------------------------------------------------------
// get_graph_feature (pipeline.py:27-40): out[b, c, n, k] = x[b,c,idx[n,k]] - x[b,c,n]; out[b, C+c, n, k] = x[b,c,n]
// ------------------------------------------------------------------------------------------------
__global__ void graph_feature_kernel(const float* __restrict__ x, const int32_t* __restrict__ idx,
                                     const int32_t* __restrict__ graph_sel, float* __restrict__ out, int C,
                                     int N, int K) {
  const int b = blockIdx.z, c = blockIdx.y;
  const int g = graph_sel ? graph_sel[b] : 0;
  const float* xr = x + ((size_t)b * C + c) * N;
  const int32_t* ig = idx + (size_t)g * N * K;
  float* o1 = out + (((size_t)b * 2 * C + c) * N) * K;
  float* o2 = out + (((size_t)b * 2 * C + C + c) * N) * K;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < N * K; e += gridDim.x * blockDim.x) {
    const int n = e / K;
    const float ctr = xr[n];
    o1[e] = xr[ig[e]] - ctr;
    o2[e] = ctr;
  }
}

// ------------------------------------------------------------------------------------------------
// weight preparation
// ------------------------------------------------------------------------------------------------
__global__ void fold_edgeconv_kernel(const float* __restrict__ w, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, const float* __restrict__ mean,
                                     const float* __restrict__ var, float eps, int C, int Co,
                                     float* __restrict__ wf, float* __restrict__ bf) {
  const int o = blockIdx.x;  // output channel
  // same arithmetic as F.batch_norm in eval mode: scale = gamma / sqrt(var + eps)
  const float sc = gamma[o] / sqrtf(var[o] + eps);
  const float sh = beta[o] - sc * mean[o];
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float w1 = w[(size_t)o * 2 * C + c], w2 = w[(size_t)o * 2 * C + C + c];
    wf[(size_t)o * C + c] = sc * w1;
    wf[(size_t)(Co + o) * C + c] = sc * (w2 - w1);
  }
  if (threadIdx.x == 0) {
    bf[o] = 0.f;
    bf[Co + o] = sh;
  }
}

// Packed weight image for the tcgen05 kernels (layout: cp::packed_tile_offset)
__global__ void pack_weight_kernel(const float* __restrict__ w, int Nout, int K, int Npad, bf16* __restrict__ out) {
  const int64_t total = (int64_t)Npad * K;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(e / K), k = (int)(e - (int64_t)n * K);
    const int nb = n >> 7, r = n & 127, kk = k & 63;
    const int chunk = kk >> 3, within = kk & 7;
    const size_t off = cp::packed_tile_offset(nb, k >> 6, cp::packed_block_rows(nb, Npad), K) / 2 + (size_t)r * 64 + (size_t)((chunk ^ (r & 7)) << 3) + within;
    const float v = (n < Nout) ? w[(size_t)n * K + k] : 0.f;
    out[off] = __float2bfloat16_rn(v);
  }
}

// ------------------------------------------------------------------------------------------------
// fp32 GEMM: y = act([a1|a2] . w^T + bias).  64x64 tile, BK=16, 256 threads, 4x4 per thread.
// ------------------------------------------------------------------------------------------------
constexpr int GM = 64, GN = 64, GK = 16;

__global__ void __launch_bounds__(256)
linear_f32_kernel(const float* __restrict__ a1, int lda1, int K1, const float* __restrict__ a2, int lda2, int K2,
                  const float* __restrict__ w, const float* __restrict__ bias, int act, float slope,
                  float* __restrict__ y, int ldy, int64_t M, int Nout) {
  __shared__ float As[GK][GM + 4];
  __shared__ float Ws[GK][GN + 4];
  const int K = K1 + K2;
  const int64_t m0 = (int64_t)blockIdx.x * GM;
  const int n0 = blockIdx.y * GN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += GK) {
    // 64x16 elements each for A and W: 1024 / 256 threads = 4 per thread
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int e = threadIdx.x + t * 256;
      const int r = e >> 4, kk = e & 15;
      const int k = k0 + kk;
      float av = 0.f, wv = 0.f;
      const int64_t m = m0 + r;
      if (m < M && k < K) av = (k < K1) ? a1[m * lda1 + k] : a2[m * lda2 + (k - K1)];
      const int n = n0 + r;
      if (n < Nout && k < K) wv = w[(size_t)n * K + k];
      As[kk][r] = av;
      Ws[kk][r] = wv;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < GK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Ws[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= Nout) continue;
      float v = acc[i][j] + (bias ? bias[n] : 0.f);
      if (act) v = cp::lrelu(v, slope);
      y[m * ldy + n] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// EdgeConv aggregation: y[b,i,c] = lrelu(max_k z[b, idx[i,k], c] + z[b, i, Co+c]).  One warp per node,
// lanes across channels (coalesced row segments), neighbour ids broadcast by shuffle.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
edge_aggregate_kernel(const T* __restrict__ z, const int32_t* __restrict__ idx, const int32_t* __restrict__ graph_sel,
                      float slope, T* __restrict__ y, int N, int K, int Co) {
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + warp;
  if (i >= N) return;
  const int g = graph_sel ? graph_sel[b] : 0;
  const int32_t* nb = idx + ((size_t)g * N + i) * K;
  const T* zb = z + (size_t)b * N * 2 * Co;
  int my0 = (lane < K) ? nb[lane] : 0;
  int my1 = (lane + 32 < K) ? nb[lane + 32] : 0;
  for (int c = lane; c < Co; c += 32) {
    float m = -__int_as_float(0x7f800000);
    for (int k = 0; k < K; ++k) {
      const int j = (k < 32) ? __shfl_sync(0xffffffffu, my0, k) : __shfl_sync(0xffffffffu, my1, k - 32);
      m = fmaxf(m, cp::to_f32<T>(zb[(size_t)j * 2 * Co + c]));
    }
    const float q = cp::to_f32<T>(zb[(size_t)i * 2 * Co + Co + c]);
    y[((size_t)b * N + i) * Co + c] = cp::from_f32<T>(cp::lrelu(m + q, slope));
  }
}

// ------------------------------------------------------------------------------------------------
// Index2Feat 4-tap gather * mask.  One warp per keypoint; E channels per tap are contiguous (NHWC).
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
sample_taps_kernel(const T* __restrict__ patches, int Hp, int Wp, int E, int step, const int64_t* __restrict__ x_id,
                   const int64_t* __restrict__ y_id, const float* __restrict__ mask, T* __restrict__ out, int N) {
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.x * 8 + warp;
  if (n >= N) return;
  const int64_t xi = x_id[(size_t)b * N + n], yi = y_id[(size_t)b * N + n];
  const float mk = mask ? mask[(size_t)b * N + n] : 1.f;
  const T* pb = patches + (size_t)b * Hp * Wp * E;
  T* ob = out + ((size_t)b * N + n) * 4 * E;
  for (int t = 0; t < 4; ++t) {
    // tap order of pipeline.py:158-162: (2y,2x), (2y+k,2x), (2y,2x+k), (2y+k,2x+k)
    const int yy = (int)(2 * yi) + ((t & 1) ? step : 0);
    const int xx = (int)(2 * xi) + ((t & 2) ? step : 0);
    // an id outside the patch map is a caller error: the reference's advanced indexing raises a device-side index
    // assert for it (pipeline.py:158-161); so does this kernel, instead of reading out of bounds
    if (yi < 0 || xi < 0 || yy >= Hp || xx >= Wp) __trap();
    const T* src = pb + ((size_t)yy * Wp + xx) * E;
    for (int e = lane; e < E; e += 32) ob[t * E + e] = cp::from_f32<T>(cp::to_f32<T>(src[e]) * mk);
  }
}

// ------------------------------------------------------------------------------------------------
// decode
// ------------------------------------------------------------------------------------------------
// Node-major tensors inside the head are in PLAN order (cp_graph_plan_build); the reference's outputs are in
// keypoint order.  perm (G,N): plan position -> keypoint id; NULL = identity.
__device__ __forceinline__ int plan_to_keypoint(const int32_t* perm, const int32_t* graph_sel, int b, int n, int N) {
  if (!perm) return n;
  const int g = graph_sel ? graph_sel[b] : 0;
  return perm[(size_t)g * N + n];
}

__global__ void decode_init_kernel(const float* __restrict__ logits, int ld, int L, int Ltot, float* __restrict__ roi_bit,
                                   float* __restrict__ x_bits, float* __restrict__ y_bits, float* __restrict__ roi_mask,
                                   int64_t* __restrict__ x_id, int64_t* __restrict__ y_id, int B, int N,
                                   const int32_t* __restrict__ perm, const int32_t* __restrict__ graph_sel) {
  const int64_t total = (int64_t)B * N;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / N), n = (int)(e - (int64_t)b * N);
    const int kp = plan_to_keypoint(perm, graph_sel, b, n, N);
    const float* row = logits + e * ld;
    const float r = row[0];
    roi_bit[(size_t)b * N + kp] = r;
    if (roi_mask) roi_mask[e] = r > 0.f ? 1.f : 0.f;
    int64_t xi = 0, yi = 0;
    for (int l = 0; l < L; ++l) {
      const float xv = row[1 + l], yv = row[1 + L + l];
      x_bits[((size_t)b * Ltot + l) * N + kp] = xv;
      y_bits[((size_t)b * Ltot + l) * N + kp] = yv;
      xi = xi * 2 + (xv > 0.f ? 1 : 0);
      yi = yi * 2 + (yv > 0.f ? 1 : 0);
    }
    x_id[e] = xi;
    y_id[e] = yi;
  }
}

__global__ void decode_refine_kernel(const float* __restrict__ logits, int ld, int plane, int Ltot,
                                     float* __restrict__ x_bits, float* __restrict__ y_bits, int64_t* __restrict__ x_id,
                                     int64_t* __restrict__ y_id, int64_t* __restrict__ x_id_kp, int64_t* __restrict__ y_id_kp,
                                     int B, int N, const int32_t* __restrict__ perm, const int32_t* __restrict__ graph_sel) {
  const int64_t total = (int64_t)B * N;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / N), n = (int)(e - (int64_t)b * N);
    const int kp = plan_to_keypoint(perm, graph_sel, b, n, N);
    const float xv = logits[e * ld], yv = logits[e * ld + 1];
    x_bits[((size_t)b * Ltot + plane) * N + kp] = xv;
    y_bits[((size_t)b * Ltot + plane) * N + kp] = yv;
    const int64_t xi = x_id[e] * 2 + (xv > 0.f ? 1 : 0), yi = y_id[e] * 2 + (yv > 0.f ? 1 : 0);
    x_id[e] = xi;
    y_id[e] = yi;
    if (x_id_kp) {   // last stage: the ids the caller sees, in keypoint order
      x_id_kp[(size_t)b * N + kp] = xi;
      y_id_kp[(size_t)b * N + kp] = yi;
    }
  }
}

// dst[b, perm[n], :] = src[b, n, :] (to_keypoint_order != 0) or dst[b, n, :] = src[b, perm[n], :] (== 0); rows of
// `row_bytes` bytes (multiple of 4) moved as 32-bit words, one warp per row.
__global__ void __launch_bounds__(256)
permute_rows_kernel(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, int words, int B, int N,
                    const int32_t* __restrict__ perm, const int32_t* __restrict__ graph_sel, int to_keypoint_order) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t total = (int64_t)B * N;
  for (int64_t e = (int64_t)blockIdx.x * 8 + warp; e < total; e += (int64_t)gridDim.x * 8) {
    const int b = (int)(e / N), n = (int)(e - (int64_t)b * N);
    const int kp = plan_to_keypoint(perm, graph_sel, b, n, N);
    const int64_t s = to_keypoint_order ? e : (int64_t)b * N + kp;
    const int64_t d = to_keypoint_order ? (int64_t)b * N + kp : e;
    for (int w = lane; w < words; w += 32) dst[d * words + w] = src[s * words + w];
  }
}

__global__ void correspondences_kernel(const float* __restrict__ roi_bit, const float* __restrict__ seg,
                                       const float* __restrict__ bbox, const int64_t* __restrict__ x_id,
                                       const int64_t* __restrict__ y_id, cp_corr_record* __restrict__ out, int B, int N,
                                       int S) {
  const int64_t total = (int64_t)B * N;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / N);
    const int xi = (int)x_id[e], yi = (int)y_id[e];
    const float* bb = bbox + (size_t)b * 4;
    // roi_xy_ori[v,u] = (ratio_x*u + x0, ratio_y*v + y0), ratio = w/S (bop_dataset_pytorch.py:231-235), in fp64
    const double u = ((double)bb[2] / (double)S) * (double)xi + (double)bb[0];
    const double v = ((double)bb[3] / (double)S) * (double)yi + (double)bb[1];
    uint32_t f = roi_bit[e] > 0.f ? 1u : 0u;
    if (f) {
      const size_t pix = (size_t)yi * S + xi;
      const float* sb = seg + (size_t)b * 2 * S * S;
      if (sb[(size_t)S * S + pix] > 0.f) f |= 2u;  // channel 1 = full mask (test.py:314)
      if (sb[pix] > 0.f) f |= 4u;                  // channel 0 = visible mask (test.py:313)
    }
    cp_corr_record r;
    r.u = (float)u;
    r.v = (float)v;
    r.flags = f;
    out[e] = r;
  }
}

// Packed form of the same records for the multi-GPU gather / the device->host read-back: per RoI one row of
// 16 + 2 N bytes = { f32 bbox[4]; u16 rec[N] }, rec = x_id | y_id << 6 | flags << 12 (S <= 64).  u, v are an affine
// function of (bbox, id) that the consumer evaluates (cp_correspondences_unpack, or numpy on the host).
__global__ void correspondences_pack_kernel(const float* __restrict__ roi_bit, const float* __restrict__ seg,
                                            const float* __restrict__ bbox, const int64_t* __restrict__ x_id,
                                            const int64_t* __restrict__ y_id, uint8_t* __restrict__ out, int B, int N, int S) {
  const int64_t total = (int64_t)B * N;
  const size_t row_bytes = 16 + 2 * (size_t)N;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / N), n = (int)(e - (int64_t)b * N);
    const int xi = (int)x_id[e], yi = (int)y_id[e];
    uint32_t f = roi_bit[e] > 0.f ? 1u : 0u;
    if (f) {
      const size_t pix = (size_t)yi * S + xi;
      const float* sb = seg + (size_t)b * 2 * S * S;
      if (sb[(size_t)S * S + pix] > 0.f) f |= 2u;
      if (sb[pix] > 0.f) f |= 4u;
    }
    uint8_t* row = out + (size_t)b * row_bytes;
    reinterpret_cast<uint16_t*>(row + 16)[n] = (uint16_t)((uint32_t)xi | ((uint32_t)yi << 6) | (f << 12));
    if (n < 4) reinterpret_cast<float*>(row)[n] = bbox[(size_t)b * 4 + n];
  }
}

__global__ void correspondences_unpack_kernel(const uint8_t* __restrict__ packed, cp_corr_record* __restrict__ out, int B, int N, int S) {
  const int64_t total = (int64_t)B * N;
  const size_t row_bytes = 16 + 2 * (size_t)N;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / N), n = (int)(e - (int64_t)b * N);
    const uint8_t* row = packed + (size_t)b * row_bytes;
    const float* bb = reinterpret_cast<const float*>(row);
    const uint32_t w = reinterpret_cast<const uint16_t*>(row + 16)[n];
    const int xi = w & 63, yi = (w >> 6) & 63;
    cp_corr_record r;   // the same fp64 arithmetic as correspondences_kernel: bit-identical u, v
    r.u = (float)(((double)bb[2] / (double)S) * (double)xi + (double)bb[0]);
    r.v = (float)(((double)bb[3] / (double)S) * (double)yi + (double)bb[1]);
    r.flags = w >> 12;
    out[e] = r;
  }
}

__global__ void threshold_kernel(const float* __restrict__ x, float thr, int apply_sigmoid, void* __restrict__ out,
                                 int out_dtype, int64_t n) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    float v = x[e];
    if (apply_sigmoid) v = 1.0f / (1.0f + expf(-v));
    const bool on = v > thr;
    if (out_dtype == 0) ((float*)out)[e] = on ? 1.f : 0.f;
    else ((int64_t*)out)[e] = on ? 1 : 0;
  }
}

__global__ void bits_to_id_kernel(const float* __restrict__ in, int64_t outer, int L, int64_t inner, int64_t so,
                                  int64_t sl, int64_t si, int binarize, float thr, int base, void* __restrict__ out,
                                  int out_dtype) {
  const int64_t total = outer * inner;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t o = e / inner, i = e - o * inner;
    // float accumulation mirrors the reference (sum of value * base**(L-1-l)); exact for ids < 2^24
    double acc = 0.0;
    double wgt = 1.0;
    for (int l = L - 1; l >= 0; --l) {
      float v = in[o * so + l * sl + i * si];
      if (binarize) v = v > thr ? 1.f : 0.f;
      acc += (double)v * wgt;
      wgt *= (double)base;
    }
    if (out_dtype == 0) ((float*)out)[e] = (float)acc;
    else ((int64_t*)out)[e] = (int64_t)acc;
  }
}

__global__ void id_to_bits_kernel(const int64_t* __restrict__ ids, int64_t count, int L, int shift, float* __restrict__ out) {
  const int64_t total = count * L;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / L;
    const int l = (int)(e - i * L);
    const int64_t v = ids[i];
    const int64_t s1 = v >> (shift * (L - 1 - l));
    const int64_t s2 = v >> (shift * (L - l));
    out[e] = (float)(s1 - (s2 << shift));
  }
}

__global__ void group_argmax_kernel(const float* __restrict__ x, int64_t G, int D, int64_t inner, int64_t* __restrict__ out) {
  const int64_t total = G * inner;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = e / inner, i = e - g * inner;
    const float* p = x + g * D * inner + i;
    float best = p[0];
    int arg = 0;
    for (int d = 1; d < D; ++d) {
      const float v = p[(int64_t)d * inner];
      if (v > best) { best = v; arg = d; }
    }
    out[e] = arg;
  }
}

inline int grid_for(int64_t n, int block = 256) {
  int64_t g = (n + block - 1) / block;
  return (int)(g < 1 ? 1 : (g > 148 * 16 ? 148 * 16 : g));
}

}  // namespace

// 1-based object ids -> 0-based graph selector (pipeline_lm.py:56-57: self.knn_idx[obj_ids-1]); an id outside [1, G]
// traps, like the reference's device-side index assert
__global__ void graph_sel_kernel(const int64_t* __restrict__ obj_ids, int64_t n, int G, int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t g = obj_ids[i] - 1;
  if (g < 0 || g >= G) __trap();
  out[i] = (int32_t)g;
}

// ================================================================================================
extern "C" {

int cp_graph_sel(const int64_t* obj_ids, int64_t n, int G, int32_t* out, cp_stream_t s) {
  CP_REQUIRE(obj_ids && out && n > 0 && G > 0, CP_E_INVALID, "cp_graph_sel: bad arguments");
  graph_sel_kernel<<<cp::ceil_div(n, 256), 256, 0, (cudaStream_t)s>>>(obj_ids, n, G, out);
  CP_CHECK_LAUNCH("cp_graph_sel");
  return CP_OK;
}

int cp_transpose_cn_to_nc(const void* src, int sd, void* dst, int dd, int B, int C, int N, cp_stream_t s) {
  CP_REQUIRE(src && dst && B > 0 && C > 0 && N > 0, CP_E_INVALID, "cp_transpose_cn_to_nc: bad arguments");
  CP_REQUIRE(transpose_dispatch(src, sd, dst, dd, B, C, N, (cudaStream_t)s) == 0, CP_E_INVALID,
             "cp_transpose_cn_to_nc: bad dtype");
  CP_CHECK_LAUNCH("cp_transpose_cn_to_nc");
  return CP_OK;
}

int cp_transpose_scatter_bf16(const void* src, void* dst, int B, int R, int S, const float* bias, const int32_t* row_map,
                              const int32_t* graph_sel, cp_stream_t s) {
  CP_REQUIRE(src && dst && src != dst && B > 0 && R > 0 && S > 0, CP_E_INVALID, "cp_transpose_scatter_bf16: bad arguments");
  CP_REQUIRE(R % 64 == 0 && S % 64 == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0, CP_E_UNSUPPORTED,
             "cp_transpose_scatter_bf16: R=%d and S=%d must be multiples of 64, pointers 16-byte aligned", R, S);
  dim3 grid(S / 64, R / 64, B);
  transpose_scatter_bf16_64_kernel<<<grid, 256, 0, (cudaStream_t)s>>>((const uint16_t*)src, (uint16_t*)dst, R, S, bias, row_map, graph_sel);
  CP_CHECK_LAUNCH("cp_transpose_scatter_bf16");
  return CP_OK;
}

int cp_bias_add_rows_bf16(void* x, const float* bias, int64_t rows, int C, int relu, cp_stream_t s) {
  CP_REQUIRE(x && bias && rows >= 0 && C > 0, CP_E_INVALID, "cp_bias_add_rows_bf16: bad arguments");
  CP_REQUIRE(C % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(bias) & 15) == 0, CP_E_UNSUPPORTED,
             "cp_bias_add_rows_bf16: C=%d must be a multiple of 8, pointers 16-byte aligned", C);
  if (rows == 0) return CP_OK;
  const int64_t vecs = rows * (C / 8);
  bias_add_rows_kernel<<<grid_for(vecs), 256, 0, (cudaStream_t)s>>>((uint4*)x, bias, vecs, C / 8, relu);
  CP_CHECK_LAUNCH("cp_bias_add_rows_bf16");
  return CP_OK;
}

int cp_transpose_nc_to_cn(const void* src, int sd, void* dst, int dd, int B, int N, int C, cp_stream_t s) {
  CP_REQUIRE(src && dst && B > 0 && C > 0 && N > 0, CP_E_INVALID, "cp_transpose_nc_to_cn: bad arguments");
  CP_REQUIRE(transpose_dispatch(src, sd, dst, dd, B, N, C, (cudaStream_t)s) == 0, CP_E_INVALID,
             "cp_transpose_nc_to_cn: bad dtype");
  CP_CHECK_LAUNCH("cp_transpose_nc_to_cn");
  return CP_OK;
}

int cp_convert(const void* src, int sd, void* dst, int dd, int64_t n, cp_stream_t s) {
  CP_REQUIRE(src && dst && n >= 0, CP_E_INVALID, "cp_convert: bad arguments");
  if (n == 0) return CP_OK;
  cudaStream_t st = (cudaStream_t)s;
  const int g = grid_for(n);
  if (sd == CP_F32 && dd == CP_BF16) convert_kernel<float, bf16><<<g, 256, 0, st>>>((const float*)src, (bf16*)dst, n);
  else if (sd == CP_BF16 && dd == CP_F32) convert_kernel<bf16, float><<<g, 256, 0, st>>>((const bf16*)src, (float*)dst, n);
  else if (sd == CP_F32 && dd == CP_F32) convert_kernel<float, float><<<g, 256, 0, st>>>((const float*)src, (float*)dst, n);
  else if (sd == CP_BF16 && dd == CP_BF16) convert_kernel<bf16, bf16><<<g, 256, 0, st>>>((const bf16*)src, (bf16*)dst, n);
  else CP_REQUIRE(false, CP_E_INVALID, "cp_convert: bad dtype");
  CP_CHECK_LAUNCH("cp_convert");
  return CP_OK;
}

int cp_graph_feature(const float* x, const int32_t* idx, const int32_t* graph_sel, float* out, int B, int C, int N,
                     int K, cp_stream_t s) {
  CP_REQUIRE(x && idx && out && B > 0 && C > 0 && N > 0 && K > 0, CP_E_INVALID, "cp_graph_feature: bad arguments");
  dim3 grid(min(cp::ceil_div((int64_t)N * K, 256), 64), C, B);
  graph_feature_kernel<<<grid, 256, 0, (cudaStream_t)s>>>(x, idx, graph_sel, out, C, N, K);
  CP_CHECK_LAUNCH("cp_graph_feature");
  return CP_OK;
}

int cp_fold_edgeconv(const float* conv_w, const float* gamma, const float* beta, const float* mean, const float* var,
                     float eps, int C, int Co, float* w_fold, float* b_fold, cp_stream_t s) {
  CP_REQUIRE(conv_w && gamma && beta && mean && var && w_fold && b_fold && C > 0 && Co > 0, CP_E_INVALID,
             "cp_fold_edgeconv: bad arguments");
  fold_edgeconv_kernel<<<Co, 128, 0, (cudaStream_t)s>>>(conv_w, gamma, beta, mean, var, eps, C, Co, w_fold, b_fold);
  CP_CHECK_LAUNCH("cp_fold_edgeconv");
  return CP_OK;
}

size_t cp_packed_weight_bytes(int Nout, int K) {
  if (Nout <= 0 || K <= 0 || (K % 64) != 0) return 0;
  const size_t npad = (size_t)((Nout + 15) / 16) * 16;
  return npad * (size_t)K * 2;
}

int cp_pack_weight(const float* w, int Nout, int K, void* packed, cp_stream_t s) {
  CP_REQUIRE(w && packed && Nout > 0 && K > 0, CP_E_INVALID, "cp_pack_weight: bad arguments");
  CP_REQUIRE(K % 64 == 0, CP_E_UNSUPPORTED, "cp_pack_weight: K=%d must be a multiple of 64", K);
  const int npad = (Nout + 15) / 16 * 16;
  pack_weight_kernel<<<grid_for((int64_t)npad * K), 256, 0, (cudaStream_t)s>>>(w, Nout, K, npad, (bf16*)packed);
  CP_CHECK_LAUNCH("cp_pack_weight");
  return CP_OK;
}

int cp_linear_f32(const float* a1, int lda1, int K1, const float* a2, int lda2, int K2, const float* w,
                  const float* bias, int act, float slope, float* y, int ldy, int64_t M, int Nout, cp_stream_t s) {
  CP_REQUIRE(a1 && w && y && K1 > 0 && K2 >= 0 && M > 0 && Nout > 0, CP_E_INVALID, "cp_linear_f32: bad arguments");
  CP_REQUIRE(K2 == 0 || a2, CP_E_INVALID, "cp_linear_f32: a2 is NULL but K2=%d", K2);
  CP_REQUIRE(M / GM < 2147483647LL, CP_E_UNSUPPORTED, "cp_linear_f32: M too large");
  dim3 grid(cp::ceil_div(M, GM), cp::ceil_div(Nout, GN));
  linear_f32_kernel<<<grid, 256, 0, (cudaStream_t)s>>>(a1, lda1, K1, a2, lda2, K2, w, bias, act, slope, y, ldy, M, Nout);
  CP_CHECK_LAUNCH("cp_linear_f32");
  return CP_OK;
}

int cp_edge_aggregate(const void* z, int dtype, const int32_t* idx, const int32_t* graph_sel, float slope, void* y,
                      int B, int N, int K, int Co, cp_stream_t s) {
  CP_REQUIRE(z && idx && y && B > 0 && N > 0 && Co > 0, CP_E_INVALID, "cp_edge_aggregate: bad arguments");
  CP_REQUIRE(K >= 1 && K <= 64, CP_E_UNSUPPORTED, "cp_edge_aggregate: K=%d outside [1,64]", K);
  dim3 grid(cp::ceil_div(N, 8), B);
  if (dtype == CP_F32)
    edge_aggregate_kernel<float><<<grid, 256, 0, (cudaStream_t)s>>>((const float*)z, idx, graph_sel, slope, (float*)y, N, K, Co);
  else if (dtype == CP_BF16)
    edge_aggregate_kernel<bf16><<<grid, 256, 0, (cudaStream_t)s>>>((const bf16*)z, idx, graph_sel, slope, (bf16*)y, N, K, Co);
  else CP_REQUIRE(false, CP_E_INVALID, "cp_edge_aggregate: bad dtype %d", dtype);
  CP_CHECK_LAUNCH("cp_edge_aggregate");
  return CP_OK;
}

int cp_sample_taps(const void* patches, int dtype, int Hp, int Wp, int E, int tap_step, const int64_t* x_id,
                   const int64_t* y_id, const float* mask, void* out, int B, int N, cp_stream_t s) {
  CP_REQUIRE(patches && x_id && y_id && out && B > 0 && N > 0 && E > 0 && Hp > 0 && Wp > 0 && tap_step > 0, CP_E_INVALID,
             "cp_sample_taps: bad arguments");
  dim3 grid(cp::ceil_div(N, 8), B);
  if (dtype == CP_F32)
    sample_taps_kernel<float><<<grid, 256, 0, (cudaStream_t)s>>>((const float*)patches, Hp, Wp, E, tap_step, x_id, y_id, mask, (float*)out, N);
  else if (dtype == CP_BF16)
    sample_taps_kernel<bf16><<<grid, 256, 0, (cudaStream_t)s>>>((const bf16*)patches, Hp, Wp, E, tap_step, x_id, y_id, mask, (bf16*)out, N);
  else CP_REQUIRE(false, CP_E_INVALID, "cp_sample_taps: bad dtype %d", dtype);
  CP_CHECK_LAUNCH("cp_sample_taps");
  return CP_OK;
}

int cp_decode_init(const float* logits, int ld, int L, int Ltot, float* roi_bit, float* x_bits, float* y_bits,
                   float* roi_mask, int64_t* x_id, int64_t* y_id, int B, int N, const int32_t* perm,
                   const int32_t* graph_sel, cp_stream_t s) {
  CP_REQUIRE(logits && roi_bit && x_bits && y_bits && x_id && y_id && B > 0 && N > 0, CP_E_INVALID,
             "cp_decode_init: bad arguments");
  CP_REQUIRE(L >= 1 && L <= Ltot && ld >= 1 + 2 * L, CP_E_INVALID, "cp_decode_init: bad L=%d Ltot=%d ld=%d", L, Ltot, ld);
  decode_init_kernel<<<grid_for((int64_t)B * N), 256, 0, (cudaStream_t)s>>>(logits, ld, L, Ltot, roi_bit, x_bits, y_bits,
                                                                            roi_mask, x_id, y_id, B, N, perm, graph_sel);
  CP_CHECK_LAUNCH("cp_decode_init");
  return CP_OK;
}

int cp_decode_refine(const float* logits, int ld, int plane, int Ltot, float* x_bits, float* y_bits, int64_t* x_id,
                     int64_t* y_id, int64_t* x_id_kp, int64_t* y_id_kp, int B, int N, const int32_t* perm,
                     const int32_t* graph_sel, cp_stream_t s) {
  CP_REQUIRE((x_id_kp == nullptr) == (y_id_kp == nullptr), CP_E_INVALID, "cp_decode_refine: x_id_kp / y_id_kp must be given together");
  CP_REQUIRE(logits && x_bits && y_bits && x_id && y_id && B > 0 && N > 0, CP_E_INVALID, "cp_decode_refine: bad arguments");
  CP_REQUIRE(plane >= 0 && plane < Ltot && ld >= 2, CP_E_INVALID, "cp_decode_refine: bad plane=%d Ltot=%d ld=%d", plane, Ltot, ld);
  decode_refine_kernel<<<grid_for((int64_t)B * N), 256, 0, (cudaStream_t)s>>>(logits, ld, plane, Ltot, x_bits, y_bits, x_id,
                                                                              y_id, x_id_kp, y_id_kp, B, N, perm, graph_sel);
  CP_CHECK_LAUNCH("cp_decode_refine");
  return CP_OK;
}

int cp_permute_rows(const void* src, void* dst, int row_bytes, int B, int N, const int32_t* perm, const int32_t* graph_sel,
                    int to_keypoint_order, cp_stream_t s) {
  CP_REQUIRE(src && dst && perm && B > 0 && N > 0 && row_bytes > 0 && (row_bytes % 4) == 0 && src != dst, CP_E_INVALID,
             "cp_permute_rows: bad arguments (row_bytes=%d must be a multiple of 4, out of place)", row_bytes);
  int64_t g = ((int64_t)B * N + 7) / 8;
  if (g > 148 * 16) g = 148 * 16;
  permute_rows_kernel<<<(int)g, 256, 0, (cudaStream_t)s>>>((const uint32_t*)src, (uint32_t*)dst, row_bytes / 4, B, N, perm,
                                                           graph_sel, to_keypoint_order);
  CP_CHECK_LAUNCH("cp_permute_rows");
  return CP_OK;
}

int cp_correspondences(const float* roi_bit, const float* seg, const float* bbox, const int64_t* x_id,
                       const int64_t* y_id, cp_corr_record* out, int B, int N, int S, cp_stream_t s) {
  CP_REQUIRE(roi_bit && seg && bbox && x_id && y_id && out && B > 0 && N > 0 && S > 0, CP_E_INVALID,
             "cp_correspondences: bad arguments");
  correspondences_kernel<<<grid_for((int64_t)B * N), 256, 0, (cudaStream_t)s>>>(roi_bit, seg, bbox, x_id, y_id, out, B, N, S);
  CP_CHECK_LAUNCH("cp_correspondences");
  return CP_OK;
}

int cp_correspondences_pack(const float* roi_bit, const float* seg, const float* bbox, const int64_t* x_id,
                            const int64_t* y_id, uint8_t* out, int B, int N, int S, cp_stream_t s) {
  CP_REQUIRE(roi_bit && seg && bbox && x_id && y_id && out && B > 0 && N > 0, CP_E_INVALID, "cp_correspondences_pack: bad arguments");
  CP_REQUIRE(S > 0 && S <= 64 && N >= 4 && N % 2 == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0, CP_E_UNSUPPORTED,
             "cp_correspondences_pack: needs S <= 64 (6-bit ids), even N >= 4, 4-byte aligned rows (S=%d N=%d)", S, N);
  correspondences_pack_kernel<<<grid_for((int64_t)B * N), 256, 0, (cudaStream_t)s>>>(roi_bit, seg, bbox, x_id, y_id, out, B, N, S);
  CP_CHECK_LAUNCH("cp_correspondences_pack");
  return CP_OK;
}

int cp_correspondences_unpack(const uint8_t* packed, cp_corr_record* out, int B, int N, int S, cp_stream_t s) {
  CP_REQUIRE(packed && out && B > 0 && N > 0 && S > 0 && S <= 64 && N % 2 == 0, CP_E_INVALID, "cp_correspondences_unpack: bad arguments");
  correspondences_unpack_kernel<<<grid_for((int64_t)B * N), 256, 0, (cudaStream_t)s>>>(packed, out, B, N, S);
  CP_CHECK_LAUNCH("cp_correspondences_unpack");
  return CP_OK;
}

int cp_threshold(const float* x, float thr, int apply_sigmoid, void* out, int out_dtype, int64_t count, cp_stream_t s) {
  CP_REQUIRE(x && out && count >= 0 && (out_dtype == 0 || out_dtype == 1), CP_E_INVALID, "cp_threshold: bad arguments");
  if (count == 0) return CP_OK;
  threshold_kernel<<<grid_for(count), 256, 0, (cudaStream_t)s>>>(x, thr, apply_sigmoid, out, out_dtype, count);
  CP_CHECK_LAUNCH("cp_threshold");
  return CP_OK;
}

int cp_bits_to_id(const float* in, int64_t outer, int L, int64_t inner, int64_t stride_o, int64_t stride_l,
                  int64_t stride_i, int binarize, float thr, int base, void* out, int out_dtype, cp_stream_t s) {
  CP_REQUIRE(in && out && outer >= 0 && inner >= 0 && L >= 1 && base >= 2 && (out_dtype == 0 || out_dtype == 1),
             CP_E_INVALID, "cp_bits_to_id: bad arguments");
  if (outer * inner == 0) return CP_OK;
  bits_to_id_kernel<<<grid_for(outer * inner), 256, 0, (cudaStream_t)s>>>(in, outer, L, inner, stride_o, stride_l, stride_i,
                                                                          binarize, thr, base, out, out_dtype);
  CP_CHECK_LAUNCH("cp_bits_to_id");
  return CP_OK;
}

int cp_id_to_bits(const int64_t* ids, int64_t count, int L, int base, float* out, cp_stream_t s) {
  CP_REQUIRE(ids && out && count >= 0 && L >= 1, CP_E_INVALID, "cp_id_to_bits: bad arguments");
  int shift = 0;
  while ((1 << shift) < base) ++shift;
  CP_REQUIRE(base >= 2 && (1 << shift) == base, CP_E_UNSUPPORTED, "cp_id_to_bits: base=%d is not a power of two", base);
  CP_REQUIRE(shift * L < 63, CP_E_UNSUPPORTED, "cp_id_to_bits: code too long");
  if (count == 0) return CP_OK;
  id_to_bits_kernel<<<grid_for(count * L), 256, 0, (cudaStream_t)s>>>(ids, count, L, shift, out);
  CP_CHECK_LAUNCH("cp_id_to_bits");
  return CP_OK;
}

int cp_group_argmax(const float* x, int64_t G, int D, int64_t inner, int64_t* out, cp_stream_t s) {
  CP_REQUIRE(x && out && G >= 0 && D >= 1 && inner >= 0, CP_E_INVALID, "cp_group_argmax: bad arguments");
  if (G * inner == 0) return CP_OK;
  group_argmax_kernel<<<grid_for(G * inner), 256, 0, (cudaStream_t)s>>>(x, G, D, inner, out);
  CP_CHECK_LAUNCH("cp_group_argmax");
  return CP_OK;
}

}  // extern "C"
