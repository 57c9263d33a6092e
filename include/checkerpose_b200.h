/*
 * checkerpose_b200 -- C ABI of the B200 (sm_100a) kernels behind CheckerPose's GNN keypoint head.
 *
 * The reference (RuyiLian/CheckerPose) has no native code and no FFI: the "operator interface" of
 * this path is the Python nn.Module / function API of checkerpose/model/{init,init_lm,pipeline,
 * pipeline_lm}.py.  Each entry point below names the reference function(s) it replaces; the
 * Python drop-in modules in checkerpose_b200/model/ bind them with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless stated otherwise; the caller owns all buffers
 *     (inputs, outputs, packed weights); the library never allocates or frees device memory;
 *   - every launch goes to the cudaStream_t passed in (an opaque void* here), is asynchronous and
 *     CUDA-graph capturable; no internal synchronisation, no mutable global state;
 *   - "node-major" = (B, N, C) row-major with C contiguous.  The reference's (B, C, N) tensors are
 *     converted at the module boundary (cp_transpose_*), or are zero-copy permuted views;
 *   - return value: 0 on success, negative on error (CP_E_*); cp_last_error_string() gives the
 *     message for the calling thread.  Nothing throws or aborts across the ABI;
 *   - there is no CPU fallback anywhere.
 */
#ifndef CHECKERPOSE_B200_H_
#define CHECKERPOSE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* cp_stream_t; /* cudaStream_t */

enum { CP_F32 = 0, CP_BF16 = 1 };
enum {
  CP_OK = 0,
  CP_E_INVALID = -1,     /* bad argument / null pointer / misaligned */
  CP_E_UNSUPPORTED = -2, /* shape outside what the kernel handles */
  CP_E_CUDA = -3         /* CUDA runtime error captured at launch */
};

const char* cp_last_error_string(void);
int cp_version(void);
/* Compute capability of the current device as major*10+minor (100 on B200), or <0 on error. */
int cp_device_arch(void);

/* ---- K1: kNN graph -------------------------------------------------------------------------
 * knn(x, k)  pipeline.py:18-23 == init.py:27-32 == pipeline_lm.py:18-23 == init_lm.py:27-32.
 * x (B, C, N) f32 -> idx64 (B, N, k) int64, nearest first (self is entry 0); optional int32 copy
 * idx32 (may be NULL).  fp32 direct-difference distances, ties broken towards the lower index.
 * 1 <= k <= 64, k <= N, any C >= 1 (C > 64: tensor-core pruning, the same exact fp32 result). */
int cp_knn(const float* x, int B, int C, int N, int k, int64_t* idx64, int32_t* idx32, cp_stream_t s);

/* ---- layout conversion at the module boundary ----------------------------------------------
 * (B, C, N) <-> (B, N, C), with dtype conversion (CP_F32 / CP_BF16 on either side). */
int cp_transpose_cn_to_nc(const void* src, int src_dtype, void* dst, int dst_dtype, int B, int C, int N, cp_stream_t s);
int cp_transpose_nc_to_cn(const void* src, int src_dtype, void* dst, int dst_dtype, int B, int N, int C, cp_stream_t s);
int cp_convert(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t count, cp_stream_t s);
/* The layout change after the init head's conv1x1 (init.py:113-114, `out.view(-1, N, 64)` of the channels-last conv
 * output) fused with the conv bias and the keypoint -> plan renumbering: bf16 src (B, R, S) -> dst (B, S, R) with
 * dst[b, row_map[g(b)][s], r] = src[b, r, s] + bias[s].  bias (S) f32 or NULL; row_map (G, S) int32 or NULL (identity);
 * graph_sel (B) int32 or NULL (graph 0).  R and S multiples of 64, out of place. */
int cp_transpose_scatter_bf16(const void* src, void* dst, int B, int R, int S, const float* bias, const int32_t* row_map,
                              const int32_t* graph_sel, cp_stream_t s);
/* x (rows, C) bf16 = [relu](x + bias (C) f32) in place: the bias of a library convolution without fused activation
 * (Index2Feat_module.patch_generator pipeline.py:144-145, seg_block :349, the folded BN shift of up_net[0]'s
 * ConvTranspose2d :186-197) on its channels-last output.  C multiple of 8. */
int cp_bias_add_rows_bf16(void* x, const float* bias, int64_t rows, int C, int relu, cp_stream_t s);

/* ---- get_graph_feature(x, knn_idx, batch_indices)  pipeline.py:27-40 ------------------------
 * Kept for API completeness (the fused path never materialises it).
 * x (B, C, N) f32, idx (G, N, K) int32, graph_sel (B) int32 or NULL (=> graph 0) -> out (B, 2C, N, K). */
int cp_graph_feature(const float* x, const int32_t* idx, const int32_t* graph_sel, float* out,
                     int B, int C, int N, int K, cp_stream_t s);

/* ---- weight preparation (module-owned, derived lazily after load_state_dict) ----------------
 * EdgeConv folding: StaticGraph_module = Conv2d(2C->Co,1x1,no bias)+BatchNorm2d(eval)+LeakyReLU+max_k
 * (pipeline.py:45-59).  With W=[W1|W2], s=gamma/sqrt(var+eps), t=beta-s*mean:
 *   max_k lrelu(s*(W1(x_j-x_i)+W2 x_i)+t) = lrelu(max_k P_j + Q_i),  P=(s.W1)x, Q=(s.(W2-W1))x+t
 * (max commutes because lrelu is increasing; folding s into the rows removes the sign problem of
 * negative gammas).  w_fold (2Co, C) f32 = [s.W1 ; s.(W2-W1)], b_fold (2Co) = [0 ; t]. */
int cp_fold_edgeconv(const float* conv_w, const float* gamma, const float* beta, const float* mean,
                     const float* var, float eps, int C, int Co, float* w_fold, float* b_fold, cp_stream_t s);
/* Pack an (Nout, K) f32 row-major weight into the bf16 tile image the tcgen05 kernels stream with
 * bulk copies: N blocks of <=128 rows (Nout padded to 16), K chunks of 64, each tile K-major
 * SWIZZLE_128B.  K % 64 == 0. */
size_t cp_packed_weight_bytes(int Nout, int K);
int cp_pack_weight(const float* w, int Nout, int K, void* packed, cp_stream_t s);

/* ---- fp32 SIMT GEMM (FFMA): shapes the tensor-core kernel below does not take (K not a multiple of 64) ----
 * y[m, :] = act([a1[m, :K1] | a2[m, :K2]] . w^T + bias);  w (Nout, K1+K2) row-major;  a2 may be NULL.
 * act: 0 = none, 1 = LeakyReLU(slope).  Replaces nn.Linear(+LeakyReLU) (pipeline.py:61-69) and the
 * folded EdgeConv node GEMM. */
int cp_linear_f32(const float* a1, int lda1, int K1, const float* a2, int lda2, int K2, const float* w,
                  const float* bias, int act, float slope, float* y, int ldy, int64_t M, int Nout, cp_stream_t s);

/* ---- float32 mode on the tensor cores: split-bf16 x3 GEMM / implicit-GEMM convolution (tcgen05) ----
 * out[m, :Nout] = act(A[m, :K] . W^T + bias) with every fp32 operand split on the fly into bf16 hi + lo and the
 * product taken as hi.hi + hi.lo + lo.hi (fp32 accumulation in TMEM; ~2^-16 relative per product; fp32 in, fp32 out).
 *   CP_X3_LINEAR : A[m] = [a1[m, :k1] | a2[m, :k2]]  (k1 + k2 == K; a2 may be NULL with k2 == 0) -- nn.Linear
 *                  (+LeakyReLU) of pipeline.py:61-69, the folded EdgeConv node GEMM, the concat of pipeline.py:283.
 *   CP_X3_CONV   : a1 = NHWC map (B, H, W, k1 = Cin); row m = output pixel (b, oy, ox) of a (B, Ho, Wo) grid;
 *                  A[m, (ky*KW + kx)*Cin + c] = a1[b, oy - pad + ky, ox - pad + kx, c] (0 outside the map): Conv2d
 *                  KH x KW, stride 1 (pipeline.py:144-145, 195-208).  W row n = weight[n] in (ky, kx, c) order.
 *   CP_X3_CONVT  : the same gather for ConvTranspose2d stride 2 (pipeline.py:187-197): tap (ky, kx) reads
 *                  a1[b, (oy + pad - ky) / 2, (ox + pad - kx) / 2, c] when both are even and inside the map.
 * act: 0 = none, 1 = LeakyReLU(slope) (slope 0 = ReLU).  K, k1, k2 multiples of 64; weights packed by
 * cp_pack_weight_split (two images of cp_pack_weight's layout: bf16(w) and bf16(w - bf16(w))). */
enum { CP_X3_LINEAR = 0, CP_X3_CONV = 1, CP_X3_CONVT = 2 };
typedef struct {
  int mode;
  const float* a1; int ld1; int k1;
  const float* a2; int ld2; int k2;
  int H, W, Ho, Wo, KH, KW, pad;
  int64_t M; int K;
  const void* w_hi; const void* w_lo;
  const float* bias; int act; float slope;
  float* out; int ld_out; int Nout;
} cp_gemm_x3_params;
int cp_pack_weight_split(const float* w, int Nout, int K, void* packed_hi, void* packed_lo, cp_stream_t s);
int cp_gemm_x3(const cp_gemm_x3_params* p, cp_stream_t s);

/* ---- bf16 implicit-GEMM convolution on tcgen05 (conv_bf16_tcgen05.cu): the image branch of the bf16 mode ----
 * Same operand gather as cp_gemm_x3 (CP_X3_CONV / CP_X3_CONVT) with bf16 activations and one MMA per K step:
 * out[m, :Nout] = act(A[m, :K] . W^T + bias), bf16 in / bf16 out, fp32 accumulation; W packed by cp_pack_weight with rows in
 * (ky, kx, c) order; BatchNorm folded into W / bias by the caller; act: 0 = none, 1 = LeakyReLU(slope) (slope 0 = ReLU).
 * Replaces the cuDNN calls of get_gdrn_upsample_module (pipeline.py:183-211), patch_generator (:144-145), seg_block (:349,383)
 * and conv1x1 (init.py:112) when the tcgen05 image branch is selected. */
typedef struct {
  int mode;
  const void* a1; int ld1; int k1;
  int H, W, Ho, Wo, KH, KW, pad;
  int64_t M; int K;
  const void* w_packed;
  const float* bias; int act; float slope;
  void* out; int ld_out; int Nout;
} cp_conv_bf16_params;
int cp_conv_bf16(const cp_conv_bf16_params* p, cp_stream_t s);

/* ---- slab convolution (conv_slab_tcgen05.cu): the same convolutions over ZERO-BORDERED maps, each activation read once ----
 * x is a stored NHWC map (B, Hp, Wp, C) bf16 that includes its own zero border (one zero row after and one zero column right
 * of every image are enough: over the flat index they are the top / left border of what follows; rows before the first and
 * after the last image are zero-filled by the TMA unit), seen as a matrix of G = B*Hp*Wp rows.  Over
 * that flat row index a kernel tap is a CONSTANT row shift: the output at grid position g reads rows g + shift[t], so one
 * tile of 128 consecutive positions needs one slab of 128 + max(shift) - min(shift) rows per 64-channel slice -- loaded ONCE
 * by TMA (SWIZZLE_128B, rows outside the matrix zero-filled) and presented to tcgen05.mma once per tap through a descriptor
 * whose start address is moved by shift rows (cp_conv_bf16 gathers every tap's rows again: 9x the activation traffic of a
 * 3x3 convolution).  CTA pairs (cta_group::2, M = 256) share each weight tile: every CTA loads half of it.
 *   out[g, :Nout] = act(sum_t x[g + shift[t], :C] . W[:, wtap[t]*C : (wtap[t]+1)*C]^T + bias)   for positions g = (b, py, px)
 *   with vy0 <= py < vy1, vx0 <= px < vx1 (the window that holds real outputs);
 *   compact == 0: out has the grid of x ((G, ld_out) rows); rows outside the window are written as ZEROS, so the result is again
 *                 a zero-bordered map (Conv2d 3x3 pad 1 chains: get_gdrn_upsample_module pipeline.py:195-208);
 *   compact == 1: only window rows are written, to row b*out_sb + (py-vy0)*out_sy + (px-vx0)*out_sx + phase.out_off (pixels):
 *                 patch_generator (Conv2d 2x2 pad 1, pipeline.py:144-145: 65 x 65 outputs of a 64 x 64 map) and the four
 *                 output parities ("phases") of ConvTranspose2d stride 2 (pipeline.py:187-197), each with its own tap list.
 * W: cp_pack_weight of the (Nout, K) matrix, K = (number of weight taps) * C in tap-major order; C % 64 == 0; Nout <= 256. */
#define CP_SLAB_MAX_TAPS 9
#define CP_SLAB_MAX_PHASES 4
typedef struct {
  int ntaps;
  int wtap[CP_SLAB_MAX_TAPS];
  int shift[CP_SLAB_MAX_TAPS];
  int out_off;
} cp_slab_phase;
typedef struct {
  const void* x; int B, Hp, Wp, C, ldx;
  const void* w_packed; int K;
  const float* bias; int act; float slope;
  void* out; int ld_out; int Nout;
  int num_phases; cp_slab_phase phase[CP_SLAB_MAX_PHASES];
  int vy0, vy1, vx0, vx1;
  int compact; int64_t out_sb; int out_sy, out_sx;
  /* Fused 1x1 head on the convolution's own output (seg_w != NULL; needs compact == 0): seg_block of pipeline.py:349,383.
   * seg_out[b, j, py - vy0, px - vx0] = seg_b[j] + sum_n bf16(out[g, n]) * seg_w[j, n]  (fp32, NCHW (B, seg_n, vy1-vy0, vx1-vx0)),
   * computed in the epilogue from the values being stored: the map is not read again.  seg_n <= 4. */
  const float* seg_w; const float* seg_b; float* seg_out; int seg_n;
} cp_conv_slab_params;
int cp_conv_slab(const cp_conv_slab_params* p, cp_stream_t s);
/* zero the border of a bordered NHWC map (B, Hp, Wp, C) of elem_bytes-wide elements (row pitch C): the LAST row and the LAST
 * column of every image (over the flat pixel index they serve as the right / left and bottom / top borders at once) */
int cp_zero_border_nhwc(void* x, int B, int Hp, int Wp, int C, int elem_bytes, cp_stream_t s);

/* ---- K2: EdgeConv -----------------------------------------------------------------------------
 * Aggregation half:  y[b,i,c] = lrelu(max_k z[b, idx[g(b), i, k], c] + z[b, i, Co + c]),  z (B,N,2Co).
 * idx (G, N, K) int32; graph_sel (B) int32 selects the per-RoI graph (pipeline_lm.py:55-57), NULL =>
 * shared graph 0 (pipeline.py:55).  dtype applies to z and y. */
int cp_edge_aggregate(const void* z, int dtype, const int32_t* idx, const int32_t* graph_sel, float slope,
                      void* y, int B, int N, int K, int Co, cp_stream_t s);

/* Fused tcgen05 chain (bf16 operands, fp32 accumulation in TMEM).  One launch does, per tile of 128
 * nodes:  PROLOGUE -> A tile in shared memory -> up to 3 chained GEMM(+bias+LeakyReLU) layers whose
 * weights are streamed with bulk-async copies -> OUTPUT.
 *   prologue CP_PRO_LOAD : A = src[b, n, :C]                                   (bf16 node-major)
 *            CP_PRO_AGG  : A = lrelu(max_k z[b, idx[n,k], :Co] + z[b, n, Co:])  (EdgeConv aggregation)
 *            CP_PRO_TAPS : A = [4-tap gather of patches * roi mask | graph_feat] (Index2Feat + concat,
 *                          pipeline.py:147-164, 278-283)
 *   output   CP_OUT_BF16 : out (B*N, ld_out) bf16, all Nout columns (EdgeConv [P|Q] table)
 *            CP_OUT_F32  : out (B*N, ld_out) f32, first n_valid columns (logits)
 * See DESIGN.md for the tile/pipeline description. */
enum { CP_PRO_LOAD = 0, CP_PRO_AGG = 1, CP_PRO_TAPS = 2 };
enum { CP_OUT_BF16 = 0, CP_OUT_F32 = 1 };

typedef struct {
  const void* w_packed; /* cp_pack_weight image of the (nout, kin) weight */
  const float* bias;    /* (nout) or NULL */
  int kin;              /* multiple of 64, <= 512 for layer 0 of TAPS, else <= 256 */
  int nout;             /* <= 512 for the last layer with CP_OUT_BF16, else <= 256 */
  int act;              /* 0 none, 1 LeakyReLU */
  float slope;
} cp_chain_layer;

typedef struct {
  int prologue;
  int B, N;
  /* LOAD */
  const void* src; int ld_src; int C;
  /* AGG */
  const void* z; int ld_z; int Co; const int32_t* idx; const int32_t* graph_sel; int K; float agg_slope;
  /* TAPS: patches (B, Hp, Wp, E) bf16 NHWC, ids (B,N) int64, mask (B,N) f32 {0,1}, graph_feat (B,N,Cg) bf16 */
  const void* patches; int Hp, Wp, E, tap_step; const int64_t* x_id; const int64_t* y_id; const float* mask;
  const void* graph_feat; int ld_gf; int Cg;
  /* optional copy of the prologue's A tile (first C / Co channels) to global, bf16 (B*N, ld_a_out) */
  void* a_out; int ld_a_out;
  int num_layers;
  cp_chain_layer layers[3];
  int out_mode; void* out; int ld_out; int n_valid;
} cp_chain_params;

int cp_chain_fwd(const cp_chain_params* p, cp_stream_t s);

/* ---- K2, staged form: graph plan + warp-specialised EdgeConv kernel ----------------------------------
 * cp_graph_plan_build (HOST pointers, host code; run once per graph next to the knn() call of
 * pipeline.py:248 / init.py:98): renumbers the keypoints of each graph by recursive coordinate bisection
 * so that consecutive nodes form compact patches, lists for every tile of CP_PLAN_TILE (128) consecutive
 * nodes the distinct neighbour rows the kernel stages in shared memory, and matches the tile's nodes into
 * CP_PLAN_PAIRS (64) pairs that share most of their neighbours (the kernel reads the shared rows once).
 *   in : xyz (G,3,N) f32 or NULL (keep numbering), idx (G,N,K) int32, umax = capacity of a tile's list
 *        (multiple of 128, <= 512)
 *   out: perm (G,N) int32      perm[g][n'] = original keypoint stored at plan position n'
 *        idx_p (G,N,K) int32   neighbour lists in plan numbering
 *        ucount (G,T) int32    distinct neighbour rows per tile, T = ceil(N/128)
 *        ulist (G,T,64,umax/64) uint16  entry [q][i] = (64 i + q)-th distinct row (ascending), 0xFFFF beyond ucount
 *                              (N < 65535)
 *        prog (G,T,64,PW) uint16, PW = 2 KP + 8, KP = cp_graph_plan_kp(K): per pair
 *              [0,KP)    node a: byte offsets (128 x position in the tile's list) of its neighbours, the C rows it
 *                        shares with b first; padding repeats entry 0
 *              [KP,2KP)  node b: its neighbours outside those C rows; padding repeats a real neighbour
 *              [2KP]     a | b << 8 (node positions inside the tile; 255 = none)
 *              [2KP+1]   C (multiple of 4, the same for the 4 consecutive pairs a warp works on)
 * Returns the largest per-tile count of distinct rows or a negative CP_E_* code. */
int cp_graph_plan_kp(int K); /* neighbour-list length the kernel is instantiated for: 8,16,20,32,40; -1 if K > 40 */
int cp_graph_plan_build(const float* xyz, const int32_t* idx, int G, int N, int K, int umax, int32_t* perm,
                        int32_t* idx_p, int32_t* ucount, uint16_t* ulist, uint16_t* prog);
#define CP_PLAN_TILE 128  /* nodes per tile of cp_edgeconv_fwd */
#define CP_PLAN_PAIRS 64  /* node pairs per tile */
#define CP_PLAN_UMAX 512  /* capacity of a tile's distinct-row list */
#define CP_PLAN_LIST_LANES 64 /* ulist is stored transposed: one row of umax/64 entries per copying quarter-warp */
/* Rows of 128 B the kernel's staging ring holds for a plan with list length KP (a tile's rows must fit; the
 * kernel keeps up to three slices in flight when they do). */
int cp_edgeconv_ring_rows(int KP);

typedef struct { /* DEVICE pointers to the arrays cp_graph_plan_build produced */
  int G, N, K, KP, T, umax;
  int max_unique; /* return value of cp_graph_plan_build: the largest ucount */
  const int32_t* ucount;
  const uint16_t* ulist;
  const uint16_t* prog;
} cp_graph_plan;

/* float32 aggregation half of the factored EdgeConv on the graph plan: y (B,N,Co) fp32 = lrelu(max_k P[nbr] + Q),
 * z (B,N,2Co) fp32 = [P|Q], both in PLAN order.  Stages every tile's distinct neighbour rows in shared memory once per
 * 32-channel slice and reduces the plan's node pairs (the float32 mode's counterpart of cp_edgeconv_fwd's aggregators).
 * Co % 32 == 0; every tile's distinct-row count <= CP_PLAN_UMAX (else use cp_edge_aggregate). */
int cp_edge_aggregate_staged_f32(const float* z, const cp_graph_plan* plan, const int32_t* graph_sel, float slope, float* y,
                                 int B, int N, int Co, cp_stream_t s);

/* StaticGraph_module (pipeline.py:45-59) in the factored form, fused with the GEMM that consumes it:
 *   A[i,:]  = lrelu(max_k z[b, nbr(i,k), :Co] + z[b, i, Co:2Co])       (never leaves the SM)
 *   out     = act(A . W^T + bias)                                       (tcgen05, fp32 accumulate in TMEM)
 * One persistent CTA of 32 warps per SM (csrc/edgeconv_tcgen05.cu).  Per tile of 128 nodes and 64-channel slice a
 * stager warpgroup copies the tile's DISTINCT neighbour row slices (128 B each, plan.ulist) into a shared-memory ring
 * with cp.async and signals the slice asynchronously (cp.async.mbarrier.arrive.noinc); sixteen aggregator warps -- a
 * quarter-warp per node pair of plan.prog -- take the max in registers with 128-bit shared-memory loads and write
 * the bf16 A operand; one thread issues the MMAs against weights streamed through the TMA engine by another, and
 * eight epilogue warps drain TMEM into TMA tensor stores -- all overlapped through mbarriers.
 * All node-major tensors are in PLAN order.  Co in {64,128,256}; layer.kin == Co; layer.nout <= 512;
 * K <= 40; every tile's distinct-row count <= min(umax, cp_edgeconv_ring_rows(KP)) (else use
 * cp_chain_fwd(CP_PRO_AGG)). */
typedef struct {
  int B, N;
  const void* z; int ld_z; int Co;
  cp_graph_plan plan; const int32_t* graph_sel; float agg_slope;
  void* a_out; int ld_a_out;          /* optional bf16 copy of A (the EdgeConv output feature) */
  cp_chain_layer layer;
  int out_mode; void* out; int ld_out; int n_valid;
} cp_edgeconv_params;
int cp_edgeconv_fwd(const cp_edgeconv_params* p, cp_stream_t s);

/* ---- K3: Index2Feat 4-tap integer gather (pipeline.py:156-163) + roi-mask multiply (:280) ------
 * patches (B, Hp, Wp, E) NHWC in `dtype`; taps (2y,2x),(2y+k,2x),(2y,2x+k),(2y+k,2x+k), channel order
 * [tap1 | tap2 | tap3 | tap4]; out (B, N, 4E) node-major in `dtype`; mask (B,N) f32 or NULL.
 * Precondition (as for the CP_PRO_TAPS prologue of cp_chain_fwd): 0 <= 2*id and 2*id + tap_step < Hp / Wp.  An id
 * outside the patch map traps the kernel (the reference's indexing raises a device-side assert); nothing is read
 * out of bounds. */
int cp_sample_taps(const void* patches, int dtype, int Hp, int Wp, int E, int tap_step, const int64_t* x_id,
                   const int64_t* y_id, const float* mask, void* out, int B, int N, cp_stream_t s);

/* ---- image branch glue (pipeline.py:372-373 + nn.UpsamplingBilinear2d of pipeline.py:201) -------
 * out (B, 2H, 2W, Ca+Cb) NHWC = bilinear x2 upsampling (align_corners=True) of cat([a, b], channel).
 * a, b are NHWC views: channel stride 1, element strides (sb, sh, sw) given; Cb may be 0 (b NULL).
 * Channels and strides must be multiples of 16 bytes.  The convolutions around it stay on cuDNN. */
int cp_upsample2x_cat_nhwc(const void* a, int64_t a_sb, int64_t a_sh, int64_t a_sw, int Ca, const void* b,
                           int64_t b_sb, int64_t b_sh, int64_t b_sw, int Cb, int dtype, void* out, int B,
                           int H, int W, cp_stream_t s);
/* the same with the output's element strides (o_sb, o_sh, o_sw >= Ca+Cb) given: writes the interior of a zero-bordered map */
int cp_upsample2x_cat_nhwc_to(const void* a, int64_t a_sb, int64_t a_sh, int64_t a_sw, int Ca, const void* b,
                              int64_t b_sb, int64_t b_sh, int64_t b_sw, int Cb, int dtype, void* out, int64_t o_sb,
                              int64_t o_sh, int64_t o_sw, int B, int H, int W, cp_stream_t s);

/* ---- K4: sign-bit decode ------------------------------------------------------------------------
 * Init stage (pipeline.py:363-369): logits (B*N, ld) f32 rows = [roi, x_0..x_{L-1}, y_0..y_{L-1}].
 * Writes roi_bit (B,1,N), planes 0..L-1 of x_bits / y_bits (B, Ltot, N), roi_mask (B,N) f32 {0,1} and
 * ids (B,N) int64 = sum_i bit_i 2^(L-1-i).  bit = logit > 0  (== sigmoid > 0.5 up to |logit| < 2e-7).
 * Logit rows, roi_mask and ids are in PLAN order (row n of RoI b is keypoint perm[g(b)][n]; perm (G,N) int32 from
 * cp_graph_plan_build, graph_sel (B) int32 or NULL => graph 0; perm NULL => identity); roi_bit / x_bits / y_bits
 * are written in the reference's keypoint order. */
/* 1-based object ids (n) int64 -> 0-based graph selector int32 (pipeline_lm.py:56-57: self.knn_idx[obj_ids-1]).
 * An id outside [1, G] traps on the device -- the reference raises a device-side index assert for it. */
int cp_graph_sel(const int64_t* obj_ids, int64_t n, int G, int32_t* out, cp_stream_t s);

int cp_decode_init(const float* logits, int ld, int L, int Ltot, float* roi_bit, float* x_bits, float* y_bits,
                   float* roi_mask, int64_t* x_id, int64_t* y_id, int B, int N, const int32_t* perm,
                   const int32_t* graph_sel, cp_stream_t s);
/* Refine stage (pipeline.py:375-381): logits (B*N, ld) rows = [x_new, y_new]; writes plane `plane` of
 * x_bits / y_bits and updates id = 2*id + bit in place; x_id_kp / y_id_kp (B, N) int64 or both NULL: the updated ids
 * also in keypoint order (the last stage's: what PoseNet_GNNskip.forward returns). */
int cp_decode_refine(const float* logits, int ld, int plane, int Ltot, float* x_bits, float* y_bits,
                     int64_t* x_id, int64_t* y_id, int64_t* x_id_kp, int64_t* y_id_kp, int B, int N,
                     const int32_t* perm, const int32_t* graph_sel, cp_stream_t s);

/* ---- K4 fused: tail of a refine stage = query MLP layers 2 and 3 + decode_refine, one launch (query_tail_tcgen05.cu) ----
 * src (B*N, kin) bf16 plan-order rows = lrelu(W_q0 h + b_q0) (the first query layer is fused into the last EdgeConv launch);
 *   hid   = lrelu(src . W1^T + b1)      kin -> 64      tcgen05, A tiles by TMA tensor loads      (MLP_QueryNet, pipeline.py:174-180)
 *   [x,y] = hid . W2^T + b2             64 -> 2        fp32 register dot products
 * then exactly cp_decode_refine on [x, y] (pipeline.py:375-381).  logits (B*N, ld_logits) f32 may be NULL.
 * kin in {64, 128, 256}; nmid == 64; nout == 2; w1_packed from cp_pack_weight; w2 (2, 64) f32 row-major. */
typedef struct {
  int B, N;
  const void* src; int ld_src; int kin;
  const void* w1_packed; const float* b1; int nmid; float slope;
  const float* w2; const float* b2; int nout;
  float* logits; int ld_logits;
  int plane, Ltot;
  float* x_bits; float* y_bits; int64_t* x_id; int64_t* y_id; int64_t* x_id_kp; int64_t* y_id_kp;
  const int32_t* perm; const int32_t* graph_sel;
} cp_query_decode_params;
int cp_query_decode_fwd(const cp_query_decode_params* p, cp_stream_t s);
/* Plan order <-> keypoint order for node-major rows of row_bytes bytes (multiple of 4), out of place:
 * to_keypoint_order != 0: dst[b, perm[g(b)][n], :] = src[b, n, :];  == 0: dst[b, n, :] = src[b, perm[g(b)][n], :]. */
int cp_permute_rows(const void* src, void* dst, int row_bytes, int B, int N, const int32_t* perm,
                    const int32_t* graph_sel, int to_keypoint_order, cp_stream_t s);
/* Correspondence records, first half of from_id_to_pose (test_network_with_test_data.py:50-66) for the
 * three calls of test.py:335-368, with roi_xy_ori of bop_dataset_pytorch.py:223-235,266-269:
 *   u = bbox.x + x_id * bbox.w / S,  v = bbox.y + y_id * bbox.h / S
 *   flags bit0 = roi logit > 0; bit1 = bit0 & seg[1 (full)][y,x] > 0; bit2 = bit0 & seg[0 (visib)][y,x] > 0
 * roi_bit (B,1,N) f32 logits, seg (B,2,S,S) f32 logits NCHW, bbox (B,4) f32 [x,y,w,h]. */
typedef struct { float u, v; uint32_t flags; } cp_corr_record;
int cp_correspondences(const float* roi_bit, const float* seg, const float* bbox, const int64_t* x_id,
                       const int64_t* y_id, cp_corr_record* out, int B, int N, int S, cp_stream_t s);
/* The same records packed for the multi-GPU gather and the device->host read-back (2 bytes per keypoint instead
 * of 12): per RoI one row of 16 + 2 N bytes = { f32 bbox[4]; u16 rec[N] }, rec = x_id | y_id << 6 | flags << 12.
 * Needs S <= 64 (6-bit ids) and an even N >= 4.  cp_correspondences_unpack evaluates u, v with the arithmetic of
 * cp_correspondences (bit-identical records). */
int cp_correspondences_pack(const float* roi_bit, const float* seg, const float* bbox, const int64_t* x_id,
                            const int64_t* y_id, uint8_t* out, int B, int N, int S, cp_stream_t s);
int cp_correspondences_unpack(const uint8_t* packed, cp_corr_record* out, int B, int N, int S, cp_stream_t s);

/* ---- SURVEY 8(f) rank 2: batched RANSAC PnP over the packed records -----------------------------------------
 * Second half of from_id_to_pose (test_network_with_test_data.py:97-115), where the reference calls
 * cv2.solvePnPRansac(valid_p3d, valid_p2d, cam_K, None, reprojectionError, iterationsCount, flags=SOLVEPNP_EPNP) per RoI
 * on the CPU.  One CTA per RoI: valid correspondences (record flags & flag_mask: 1 = roi bit, 2 = & full mask, 4 = &
 * visible mask) -> `iterations` (rounded up to a multiple of 256) P3P hypotheses scored against all of them -> Gauss-Newton
 * refit on the inliers.  Exactly one of: packed (B, 16 + 2N) rows of cp_correspondences_pack, records (B, N) 12-byte records
 * of cp_correspondences.  p3d (G, N, 3) f32 object keypoints (mm) in
 * keypoint order; graph_sel (B) int32 or NULL; cam_K (B, 9) f32 row-major if k_batched else (9).
 * pose_out (B, 12) f32 = R row-major (9) | t (3) with x_cam = R x_obj + t; ninl_out (B) int32 inlier count;
 * inlier_mask_out (B, N) u8 or NULL.  Fewer than 4 valid correspondences give R = I, t = 0, 0 inliers (reference :111-114).
 * Deterministic for a given seed.  Not a port of OpenCV: parity is agreement of the estimated pose (tests/test_gpu_pnp.py). */
int cp_pnp_ransac(const uint8_t* packed, const cp_corr_record* records, const float* p3d, const int32_t* graph_sel, const float* cam_K, int k_batched,
                  int flag_mask, float reproj_thresh, int iterations, uint64_t seed, float* pose_out, int32_t* ninl_out,
                  uint8_t* inlier_mask_out, int B, int N, int S, cp_stream_t s);

/* Elementwise helpers behind common_ops.py:5-27 and pipeline.py:84-127.
 * out = sigmoid(x) > thr ? 1 : 0 as f32 (out_dtype 0) or int64 (out_dtype 1). */
int cp_threshold(const float* x, float thr, int apply_sigmoid, void* out, int out_dtype, int64_t count, cp_stream_t s);
/* MSB-first code -> id (pipeline.py:72-82; class_id_encoder_decoder.py:17-63).
 * in element (o, l, i) at in[o*stride_o + l*stride_l + i*stride_i] (f32); digit = binarize ? (in > thr) : in;
 * out[o*inner + i] = sum_l digit * base^(L-1-l), written as int64 (out_dtype 1) or f32 (out_dtype 0). */
int cp_bits_to_id(const float* in, int64_t outer, int L, int64_t inner, int64_t stride_o, int64_t stride_l,
                  int64_t stride_i, int binarize, float thr, int base, void* out, int out_dtype, cp_stream_t s);

/* Inverse of cp_bits_to_id for power-of-two bases (class_id_encoder_decoder.py:65-101):
 * out[e*L + l] = (ids[e] >> (log2(base)*(L-1-l))) - ((ids[e] >> (log2(base)*(L-l))) << log2(base)), as f32. */
int cp_id_to_bits(const int64_t* ids, int64_t count, int L, int base, float* out, cp_stream_t s);
/* CE branch of from_output_to_class_binary_code (common_ops.py:29-38): x viewed as (G, D, inner) f32,
 * out[g*inner + i] = argmax_d x[g, d, i] (first maximum wins, like numpy.argmax) as int64. */
int cp_group_argmax(const float* x, int64_t G, int D, int64_t inner, int64_t* out, cp_stream_t s);

/* ---- offline keypoint preparation (SURVEY.md section 8f, rank 4) ---------------------------------
 * farthest_point_sample_init_center(xyz, npoint)  preprocess_data/get_fps_points.py:65-90, float64, the reference's
 * operation order (bit-exact ids).  xyz (V,3) f64 vertices; center (3) f64 HOST values = (max + min) / 2 and
 * init_dist = 10 * |max - min| (computed by the caller as the reference does, :74-80); dist_ws (V) f64 workspace;
 * ids (npoint) int64 and fps_xyz (npoint,3) f64 outputs.  One CTA; O(npoint * V). */
int cp_fps(const double* xyz, int V, int npoint, const double* center, double init_dist, double* dist_ws,
           int64_t* ids, double* fps_xyz, cp_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* CHECKERPOSE_B200_H_ */
