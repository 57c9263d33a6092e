// Shared host/device helpers for the checkerpose_b200 CUDA library.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/checkerpose_b200.h"

namespace cp {

void set_error(const char* fmt, ...);

#define CP_REQUIRE(cond, code, ...)          \
  do {                                        \
    if (!(cond)) {                            \
      cp::set_error(__VA_ARGS__);             \
      return (code);                          \
    }                                         \
  } while (0)

// Check the launch that was just issued.  cudaPeekAtLastError does not clear sticky state and is
// legal during stream capture.
#define CP_CHECK_LAUNCH(name)                                                      \
  do {                                                                             \
    cudaError_t e__ = cudaPeekAtLastError();                                       \
    if (e__ != cudaSuccess) {                                                      \
      cp::set_error("%s: CUDA error %d (%s)", name, (int)e__, cudaGetErrorString(e__)); \
      (void)cudaGetLastError();                                                    \
      return CP_E_CUDA;                                                            \
    }                                                                              \
  } while (0)

// 3-D TMA tensor map (columns, nodes, RoIs) of a bf16 node-major output (B, N, ld_out) with a 32 x 32 box in the
// SWIZZLE_64B layout: the epilogues store 32-row x 64-byte tiles through it, and rows beyond N of a ragged last tile are
// clipped instead of landing in the next RoI.  map128 points at 128 bytes (a CUtensorMap).  CP_OK or an error code.
int make_out_tensor_map(void* map128, void* out, int ncols, int ld_out, int N, int B, const char* who);

// 2-D TMA tensor map (channels, rows) of a bf16 row-major matrix with a 64 x 128 box, SWIZZLE_128B: one box = one K chunk of a
// 128-row A operand tile in the layout tcgen05.mma reads (TMA tensor LOADS; rows beyond the matrix are zero-filled).
int make_bf16_operand_map(void* map128, const void* src, int64_t ncols, int64_t nrows, int64_t ld, const char* who, int box_rows = 128);

// 2-D TMA tensor map (columns, rows) of an fp32 row-major matrix (rows, ld) with a 32 x 32 box in the SWIZZLE_128B layout
// (one box row = 32 floats = 128 bytes): epilogues store 32 x 32 tiles through it; rows / columns beyond the matrix are clipped.
int make_f32_tensor_map_2d(void* map128, void* out, int64_t ncols, int64_t nrows, int64_t ld, const char* who);

// SM count of the CURRENT device (cached per device index; the persistent kernels size their grids with it)
int num_sms();

// cp_knn for C > 64 (knn_tcgen05.cu): arguments already checked by cp_knn
int knn_wide(const float* x, int B, int C, int N, int k, int64_t* idx64, int32_t* idx32, cudaStream_t st);

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// Packed weight layout, written by cp_pack_weight / cp_pack_weight_split and sized by cp_packed_weight_bytes: an (Nout x K)
// matrix, K a multiple of 64, zero-padded to npad = Nout rounded up to 16 rows, in bf16.  The rows form blocks of 128 (the
// last block holds the npad - 128 nb rows left), each block is stored as its K chunks of 64 columns one after the other,
// and a chunk of `rows` rows is a rows x 128-byte tile in the K-major SWIZZLE_128B layout tcgen05.mma reads: row r at
// r * 128, its 16-byte piece j at ((j ^ (r & 7)) << 4).  One bulk copy moves one tile into shared memory.
__host__ __device__ __forceinline__ int packed_block_rows(int nb, int npad) { return npad - 128 * nb < 128 ? npad - 128 * nb : 128; }
// byte offset of the tile of block nb (rows = packed_block_rows(nb, npad)), K chunk kc
__host__ __device__ __forceinline__ size_t packed_tile_offset(size_t nb, size_t kc, size_t rows, size_t K) {
  return nb * 128 * K * 2 + kc * rows * 128;
}

// One packed weight tile in the tile tables of the persistent kernels: the tile of object 0, and the index of the layer
// whose w_stride moves it to another object's weights (cp_chain_layer)
struct WTile {
  const uint8_t* ptr;
  uint32_t bytes;
  uint32_t layer;
};
static inline WTile packed_tile(const void* w_packed, int nb, int kc, int K, int npad, int layer = 0) {
  const int rows = packed_block_rows(nb, npad);
  return {static_cast<const uint8_t*>(w_packed) + packed_tile_offset(nb, kc, rows, K), (uint32_t)rows * 128u, (uint32_t)layer};
}
// Object of RoI b for the weights of a launch: graph_sel[b] when the launch has object-indexed weights, else 0
__device__ __forceinline__ int weight_obj(const int32_t* sel, bool wsel, int b) { return (wsel && sel) ? __ldg(sel + b) : 0; }
// Named barrier over `nthreads` threads (whole warps) of the CTA; id 0 is __syncthreads
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.f ? v : v * slope; }

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

}  // namespace cp
