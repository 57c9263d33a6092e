// Batched RANSAC PnP over the decoded correspondence records: the second half of from_id_to_pose
// (checkerpose/test_network_with_test_data.py:97-115), which the reference runs per RoI on the CPU with
//     cv2.solvePnPRansac(valid_p3d, valid_p2d, cam_K, None, reprojectionError=2, iterationsCount=150, flags=SOLVEPNP_EPNP)
// (OpenCV is a third-party dependency of the reference, not vendored; this container has opencv-python 4.13.0).  SURVEY.md
// section 8(f) rank 2: the consumer of the records, serial on the CPU three times per RoI (test.py:335-368).
//
// This is NOT a port of OpenCV's solver: it is a GPU formulation of the same estimator family -- RANSAC over minimal
// samples, then a least-squares refit on the inliers -- chosen for one CTA per RoI:
//   1. the RoI's valid correspondences (flag bit of the record) are compacted into shared memory in keypoint order
//      (deterministic: ballot / prefix, no atomics): 3-D point (mm) + normalised image point;
//   2. every thread draws one hypothesis: 4 distinct correspondences from a counter-based generator, Grunert's P3P on the
//      first three (law of cosines -> one quartic in v = s3 / s1, derived in scripts/pnp/derive_p3p.py; roots by
//      Durand-Kerner in float64; absolute orientation from the two triangles), disambiguated by the fourth point;
//   3. every thread scores its hypothesis against all correspondences (broadcast reads of shared memory), the block
//      takes the arg-max of the inlier counts (ties: lowest hypothesis index);
//   4. Gauss-Newton on the reprojection error of the inliers (6 x 6 normal equations accumulated by the block, solved in
//      float64 by one thread), inliers re-selected once, refit again.
// Like the reference, fewer than 4 valid correspondences (or no valid hypothesis) give R = I, t = 0.
// Parity: pose agreement with cv2.solvePnPRansac on the same records (tests/test_gpu_pnp.py; tolerance stated there) --
// RANSAC draws differ, so the comparison is on the estimate, not on bits.
#include "common.cuh"

namespace {

constexpr int NT = 256;            // threads per CTA = hypotheses per round

struct Pose {
  float R[9];
  float t[3];
};

struct cplx {
  double re, im;
};
__device__ __forceinline__ cplx cmul(cplx a, cplx b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
__device__ __forceinline__ cplx csub(cplx a, cplx b) { return {a.re - b.re, a.im - b.im}; }
__device__ __forceinline__ cplx cdiv(cplx a, cplx b) {
  const double d = b.re * b.re + b.im * b.im;
  return {(a.re * b.re + a.im * b.im) / d, (a.im * b.re - a.re * b.im) / d};
}

// real roots of x^4 + a3 x^3 + a2 x^2 + a1 x + a0 (Durand-Kerner, then two Newton steps on the real part)
__device__ int quartic_real_roots(double a0, double a1, double a2, double a3, double* out) {
  const double sc = 1.0 + fmax(fmax(fabs(a0), fabs(a1)), fmax(fabs(a2), fabs(a3)));
  cplx r[4] = {{0.4 * sc, 0.9 * sc}, {-0.65 * sc, 0.72 * sc}, {0.1 * sc, -1.1 * sc}, {-0.9 * sc, -0.3 * sc}};
  for (int it = 0; it < 60; ++it) {
    double moved = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      cplx p = {r[i].re + a3, r[i].im};
      p = cmul(p, r[i]); p.re += a2;
      p = cmul(p, r[i]); p.re += a1;
      p = cmul(p, r[i]); p.re += a0;
      cplx d = {1.0, 0.0};
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j != i) d = cmul(d, csub(r[i], r[j]));
      if (d.re * d.re + d.im * d.im < 1e-300) continue;
      const cplx s = cdiv(p, d);
      r[i] = csub(r[i], s);
      moved = fmax(moved, fabs(s.re) + fabs(s.im));
    }
    if (moved < 1e-14 * sc) break;
  }
  int n = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (fabs(r[i].im) < 1e-6 * (1.0 + fabs(r[i].re))) {
      double x = r[i].re;
      for (int k = 0; k < 2; ++k) {
        const double p = (((x + a3) * x + a2) * x + a1) * x + a0;
        const double dp = ((4.0 * x + 3.0 * a3) * x + 2.0 * a2) * x + a1;
        if (dp != 0.0) x -= p / dp;
      }
      out[n++] = x;
    }
  }
  return n;
}

__device__ __forceinline__ void cross3(const double* a, const double* b, double* c) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ bool normalize3(double* a) {
  const double n = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
  if (n < 1e-12) return false;
  a[0] /= n; a[1] /= n; a[2] /= n;
  return true;
}
// orthonormal frame of a triangle: columns e1 = (Q1 - Q0)^, e2 = e3 x e1, e3 = (e1 x (Q2 - Q0))^   (row-major 3x3)
__device__ bool tri_frame(const double Q[3][3], double* F) {
  double e1[3] = {Q[1][0] - Q[0][0], Q[1][1] - Q[0][1], Q[1][2] - Q[0][2]};
  double d2[3] = {Q[2][0] - Q[0][0], Q[2][1] - Q[0][1], Q[2][2] - Q[0][2]};
  double e3[3], e2[3];
  if (!normalize3(e1)) return false;
  cross3(e1, d2, e3);
  if (!normalize3(e3)) return false;
  cross3(e3, e1, e2);
  for (int r = 0; r < 3; ++r) {
    F[r * 3 + 0] = e1[r];
    F[r * 3 + 1] = e2[r];
    F[r * 3 + 2] = e3[r];
  }
  return true;
}

// Grunert's P3P on three correspondences (X world points, x normalised image points), best of the <= 4 solutions by
// the reprojection error of a fourth correspondence.  Returns false when no solution puts the points in front.
__device__ bool p3p_best(const float* Xs, const float* xs, const int idx[4], float fx, float fy, Pose& out) {
  double X[3][3], f[3][3];
  for (int i = 0; i < 3; ++i) {
    for (int a = 0; a < 3; ++a) X[i][a] = Xs[idx[i] * 3 + a];
    f[i][0] = xs[idx[i] * 2];
    f[i][1] = xs[idx[i] * 2 + 1];
    f[i][2] = 1.0;
    normalize3(f[i]);
  }
  auto d2 = [&](int i, int j) {
    const double a = X[i][0] - X[j][0], b = X[i][1] - X[j][1], c = X[i][2] - X[j][2];
    return a * a + b * b + c * c;
  };
  auto dot = [&](int i, int j) { return f[i][0] * f[j][0] + f[i][1] * f[j][1] + f[i][2] * f[j][2]; };
  const double a2 = d2(1, 2), b2 = d2(0, 2), c2 = d2(0, 1);
  if (b2 < 1e-12) return false;
  const double ca = dot(1, 2), cb = dot(0, 2), cg = dot(0, 1);
  const double q1 = (a2 - c2) / b2, q2 = c2 / b2;
  // coefficients printed by scripts/pnp/derive_p3p.py
  const double A0 = -4 * cg * cg * q1 - 4 * cg * cg * q2 + q1 * q1 + 2 * q1 + 1;
  const double A1 = -4 * (-ca * cg * q1 - 2 * ca * cg * q2 + ca * cg - 2 * cb * cg * cg * q1 - 2 * cb * cg * cg * q2 + cb * q1 * q1 + cb * q1);
  const double A2 = 2 * (-2 * ca * ca * q2 + 2 * ca * ca - 4 * ca * cb * cg * q1 - 8 * ca * cb * cg * q2 + 2 * cb * cb * q1 * q1 -
                         2 * cg * cg * q1 - 2 * cg * cg * q2 + 2 * cg * cg + q1 * q1 - 1);
  const double A3 = -4 * (-2 * ca * ca * cb * q2 - ca * cg * q1 - 2 * ca * cg * q2 + ca * cg + cb * q1 * q1 - cb * q1);
  const double A4 = -4 * ca * ca * q2 + q1 * q1 - 2 * q1 + 1;
  if (fabs(A4) < 1e-12) return false;
  double roots[4];
  const int nr = quartic_real_roots(A0 / A4, A1 / A4, A2 / A4, A3 / A4, roots);
  double FX[9];
  if (!tri_frame(X, FX)) return false;
  const double X4[3] = {Xs[idx[3] * 3], Xs[idx[3] * 3 + 1], Xs[idx[3] * 3 + 2]};
  const double x4 = xs[idx[3] * 2], y4 = xs[idx[3] * 2 + 1];
  double best = 1e300;
  bool found = false;
  for (int k = 0; k < nr; ++k) {
    const double v = roots[k];
    const double den = 2.0 * (cg - v * ca);
    const double w = 1.0 + v * v - 2.0 * v * cb;
    if (!(v > 0.0) || fabs(den) < 1e-12 || !(w > 0.0)) continue;
    const double u = (q1 * w - v * v + 1.0) / den;
    if (!(u > 0.0)) continue;
    const double s1 = sqrt(b2 / w), s2 = u * s1, s3 = v * s1;
    const double P[3][3] = {{s1 * f[0][0], s1 * f[0][1], s1 * f[0][2]}, {s2 * f[1][0], s2 * f[1][1], s2 * f[1][2]},
                            {s3 * f[2][0], s3 * f[2][1], s3 * f[2][2]}};
    double FP[9];
    if (!tri_frame(P, FP)) continue;
    double R[9];
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) R[r * 3 + c] = FP[r * 3 + 0] * FX[c * 3 + 0] + FP[r * 3 + 1] * FX[c * 3 + 1] + FP[r * 3 + 2] * FX[c * 3 + 2];
    double t[3];
    for (int r = 0; r < 3; ++r) t[r] = P[0][r] - (R[r * 3] * X[0][0] + R[r * 3 + 1] * X[0][1] + R[r * 3 + 2] * X[0][2]);
    double Y[3];
    for (int r = 0; r < 3; ++r) Y[r] = R[r * 3] * X4[0] + R[r * 3 + 1] * X4[1] + R[r * 3 + 2] * X4[2] + t[r];
    if (!(Y[2] > 0.0)) continue;
    const double ex = fx * (Y[0] / Y[2] - x4), ey = fy * (Y[1] / Y[2] - y4);
    const double e = ex * ex + ey * ey;
    if (e < best) {
      best = e;
      found = true;
      for (int i = 0; i < 9; ++i) out.R[i] = (float)R[i];
      for (int i = 0; i < 3; ++i) out.t[i] = (float)t[i];
    }
  }
  return found;
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t& s) {
  uint64_t z = (s += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

__device__ __forceinline__ bool is_inlier(const Pose& P, const float* X, const float* x, float fx, float fy, float thr2) {
  const float Yx = P.R[0] * X[0] + P.R[1] * X[1] + P.R[2] * X[2] + P.t[0];
  const float Yy = P.R[3] * X[0] + P.R[4] * X[1] + P.R[5] * X[2] + P.t[1];
  const float Yz = P.R[6] * X[0] + P.R[7] * X[1] + P.R[8] * X[2] + P.t[2];
  if (!(Yz > 0.f)) return false;
  const float iz = 1.f / Yz;
  const float ex = fx * (Yx * iz - x[0]), ey = fy * (Yy * iz - x[1]);
  return ex * ex + ey * ey < thr2;
}

// block-wide sum of NV per-thread doubles; the result lands in red[0..NV) (read after the trailing __syncthreads)
template <int NV>
__device__ void block_sum(const float* v, double* red, int tid) {
  const int lane = tid & 31, warp = tid >> 5;
  for (int k = 0; k < NV; ++k) {
    double s = (double)v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) red[NV + warp * NV + k] = s;
  }
  __syncthreads();
  if (tid < NV) {
    double s = 0.0;
    for (int w = 0; w < NT / 32; ++w) s += red[NV + w * NV + tid];
    red[tid] = s;
  }
  __syncthreads();
}

// One Gauss-Newton step on the reprojection error of the correspondences marked in `mask`; every thread ends with the
// same updated pose.  Returns false when the normal equations are not positive definite (pose left unchanged).
__device__ bool gn_step(Pose& P, const float* Xs, const float* xs, const uint8_t* mask, int M, float fx, float fy, double* red, int tid) {
  float acc[27];
#pragma unroll
  for (int i = 0; i < 27; ++i) acc[i] = 0.f;
  for (int k = tid; k < M; k += NT) {
    if (!mask[k]) continue;
    const float* X = Xs + k * 3;
    const float yr0 = P.R[0] * X[0] + P.R[1] * X[1] + P.R[2] * X[2];
    const float yr1 = P.R[3] * X[0] + P.R[4] * X[1] + P.R[5] * X[2];
    const float yr2 = P.R[6] * X[0] + P.R[7] * X[1] + P.R[8] * X[2];
    const float Yx = yr0 + P.t[0], Yy = yr1 + P.t[1], Yz = yr2 + P.t[2];
    const float iz = 1.f / Yz;
    const float rx = fx * (Yx * iz - xs[k * 2]), ry = fy * (Yy * iz - xs[k * 2 + 1]);
    // d(residual)/dY = [a 0 c; 0 b d];  dY = -[yr]x w + dt
    const float a = fx * iz, b = fy * iz, c = -fx * Yx * iz * iz, d = -fy * Yy * iz * iz;
    float J0[6], J1[6];
    // -[yr]x = [0 yr2 -yr1; -yr2 0 yr0; yr1 -yr0 0]
    J0[0] = c * yr1;             J0[1] = a * yr2 - c * yr0;   J0[2] = -a * yr1;   J0[3] = a;   J0[4] = 0.f; J0[5] = c;
    J1[0] = -b * yr2 + d * yr1;  J1[1] = -d * yr0;            J1[2] = b * yr0;    J1[3] = 0.f; J1[4] = b;   J1[5] = d;
    int o = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
#pragma unroll
      for (int j = i; j < 6; ++j) acc[o++] += J0[i] * J0[j] + J1[i] * J1[j];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) acc[21 + i] += J0[i] * rx + J1[i] * ry;
  }
  block_sum<27>(acc, red, tid);
  __shared__ double delta[7];
  if (tid == 0) {
    double H[6][6], g[6];
    int o = 0;
    for (int i = 0; i < 6; ++i)
      for (int j = i; j < 6; ++j) H[i][j] = H[j][i] = red[o++];
    for (int i = 0; i < 6; ++i) g[i] = -red[21 + i];
    for (int i = 0; i < 6; ++i) H[i][i] += 1e-9 * (1.0 + H[i][i]);
    bool ok = true;        // Cholesky H = L L^T, in place (lower triangle)
    for (int i = 0; i < 6 && ok; ++i)
      for (int j = 0; j <= i; ++j) {
        double s = H[i][j];
        for (int k = 0; k < j; ++k) s -= H[i][k] * H[j][k];
        if (i == j) {
          if (!(s > 0.0)) { ok = false; break; }
          H[i][i] = sqrt(s);
        } else {
          H[i][j] = s / H[j][j];
        }
      }
    if (ok) {
      for (int i = 0; i < 6; ++i) {
        double s = g[i];
        for (int k = 0; k < i; ++k) s -= H[i][k] * g[k];
        g[i] = s / H[i][i];
      }
      for (int i = 5; i >= 0; --i) {
        double s = g[i];
        for (int k = i + 1; k < 6; ++k) s -= H[k][i] * g[k];
        g[i] = s / H[i][i];
      }
    }
    for (int i = 0; i < 6; ++i) delta[i] = ok ? g[i] : 0.0;
    delta[6] = ok ? 1.0 : 0.0;
  }
  __syncthreads();
  const bool ok = delta[6] != 0.0;
  if (ok) {   // R <- exp([w]x) R, t <- t + dt   (every thread, same arithmetic)
    const double wx = delta[0], wy = delta[1], wz = delta[2];
    const double th2 = wx * wx + wy * wy + wz * wz, th = sqrt(th2);
    const double A = th < 1e-9 ? 1.0 : sin(th) / th, Bc = th < 1e-9 ? 0.5 : (1.0 - cos(th)) / th2;
    const double K[9] = {0, -wz, wy, wz, 0, -wx, -wy, wx, 0};
    double E[9];
    for (int r = 0; r < 3; ++r)
      for (int c2 = 0; c2 < 3; ++c2) {
        double kk = 0.0;
        for (int m = 0; m < 3; ++m) kk += K[r * 3 + m] * K[m * 3 + c2];
        E[r * 3 + c2] = (r == c2 ? 1.0 : 0.0) + A * K[r * 3 + c2] + Bc * kk;
      }
    float Rn[9];
    for (int r = 0; r < 3; ++r)
      for (int c2 = 0; c2 < 3; ++c2) Rn[r * 3 + c2] = (float)(E[r * 3] * P.R[c2] + E[r * 3 + 1] * P.R[3 + c2] + E[r * 3 + 2] * P.R[6 + c2]);
    for (int i = 0; i < 9; ++i) P.R[i] = Rn[i];
    for (int i = 0; i < 3; ++i) P.t[i] += (float)delta[3 + i];
  }
  __syncthreads();
  return ok;
}

struct FlagSets {
  uint32_t mask[3];
};

// grid (B, V): CTA (b, v) solves RoI b on the correspondences of validity set flag_masks.mask[v] and writes row v * B + b of
// the outputs; its hypotheses are keyed on rng_index[b] (b when NULL), so every (b, v) is what a launch of one set computes.
__global__ void __launch_bounds__(NT, 1)
pnp_ransac_kernel(const uint8_t* __restrict__ packed, const cp_corr_record* __restrict__ rec12, const float* __restrict__ p3d, const int32_t* __restrict__ graph_sel,
                  const float* __restrict__ cam_K, int k_stride, FlagSets flag_masks, const int32_t* __restrict__ rng_index, float thresh, int rounds,
                  uint64_t seed, float* __restrict__ pose_out, int32_t* __restrict__ ninl_out, uint8_t* __restrict__ inl_mask_out, int B, int N, int S) {
  extern __shared__ __align__(16) uint8_t smem[];
  float* Xs = reinterpret_cast<float*>(smem);                 // (N, 3) compacted 3-D points
  float* xs = Xs + (size_t)N * 3;                             // (N, 2) normalised image points
  uint16_t* src = reinterpret_cast<uint16_t*>(xs + (size_t)N * 2);   // (N) keypoint id of the compacted entry
  uint8_t* mask = reinterpret_cast<uint8_t*>(src + N);        // (N) inlier flags of the compacted entries
  __shared__ double red[27 + (NT / 32) * 27];
  __shared__ int warp_cnt[NT / 32], s_best_cnt, s_best_h;
  __shared__ Pose s_pose;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t flag_mask = blockIdx.y == 0 ? flag_masks.mask[0] : blockIdx.y == 1 ? flag_masks.mask[1] : flag_masks.mask[2];
  const size_t o = (size_t)blockIdx.y * B + b;                // output row
  const int rb = rng_index ? rng_index[b] : b;                // hypothesis stream
  // records: packed rows (bbox + u16 per keypoint) or the 12-byte {u, v, flags} records of cp_correspondences
  const size_t row_bytes = 16 + 2 * (size_t)N;
  const uint8_t* row = packed ? packed + (size_t)b * row_bytes : nullptr;
  const float* bb = reinterpret_cast<const float*>(row);
  const uint16_t* rec = reinterpret_cast<const uint16_t*>(row + 16);
  const cp_corr_record* r12 = rec12 ? rec12 + (size_t)b * N : nullptr;
  const float* Kc = cam_K + (size_t)b * k_stride;
  const float fx = Kc[0], fy = Kc[4], cx = Kc[2], cy = Kc[5];
  const int g = graph_sel ? graph_sel[b] : 0;
  const float* Xg = p3d + (size_t)g * N * 3;

  // ---- 1. ordered compaction of the valid correspondences ----
  int base = 0;
  for (int n0 = 0; n0 < N; n0 += NT) {
    const int n = n0 + tid;
    uint32_t w = 0;
    bool v = false;
    float ru = 0.f, rv = 0.f;
    if (n < N) {
      if (r12) {
        const cp_corr_record q = r12[n];
        ru = q.u;
        rv = q.v;
        v = (q.flags & flag_mask) != 0;
      } else {
        w = rec[n];
        v = ((w >> 12) & flag_mask) != 0;
      }
    }
    const uint32_t bal = __ballot_sync(0xffffffffu, v);
    if (lane == 0) warp_cnt[warp] = __popc(bal);
    __syncthreads();
    int off = base;
    for (int q = 0; q < warp; ++q) off += warp_cnt[q];
    int tot = 0;
    for (int q = 0; q < NT / 32; ++q) tot += warp_cnt[q];
    if (v) {
      const int k = off + __popc(bal & ((1u << lane) - 1u));
      double u, vv;
      if (r12) {
        u = ru;
        vv = rv;
      } else {   // the same fp64 arithmetic as cp_correspondences (bit-identical u, v)
        const int xi = w & 63, yi = (w >> 6) & 63;
        u = (double)(float)(((double)bb[2] / (double)S) * (double)xi + (double)bb[0]);
        vv = (double)(float)(((double)bb[3] / (double)S) * (double)yi + (double)bb[1]);
      }
      xs[k * 2] = (float)((u - (double)cx) / (double)fx);
      xs[k * 2 + 1] = (float)((vv - (double)cy) / (double)fy);
      Xs[k * 3] = Xg[n * 3];
      Xs[k * 3 + 1] = Xg[n * 3 + 1];
      Xs[k * 3 + 2] = Xg[n * 3 + 2];
      src[k] = (uint16_t)n;
    }
    base += tot;
    __syncthreads();
  }
  const int M = base;
  if (inl_mask_out)
    for (int n = tid; n < N; n += NT) inl_mask_out[o * N + n] = 0;
  Pose P;
  for (int i = 0; i < 9; ++i) P.R[i] = (i % 4 == 0) ? 1.f : 0.f;
  P.t[0] = P.t[1] = P.t[2] = 0.f;
  int ninl = 0;
  if (M >= 4) {
    const float thr2 = thresh * thresh;
    // ---- 2 + 3. hypotheses and scores, `rounds` rounds of NT ----
    if (tid == 0) { s_best_cnt = -1; s_best_h = 0x7fffffff; }
    __syncthreads();
    Pose mine;
    int my_cnt = -1, my_h = 0x7fffffff;
    for (int r = 0; r < rounds; ++r) {
      const int h = r * NT + tid;
      uint64_t st = seed ^ (0xD1B54A32D192ED03ull * (uint64_t)(rb + 1)) ^ (0x8CB92BA72F3D8DD7ull * (uint64_t)(h + 1));
      int idx[4];
      bool ok = true;
      for (int i = 0; i < 4 && ok; ++i) {
        int tries = 0;
        bool dup;
        do {
          idx[i] = (int)(splitmix64(st) % (uint64_t)M);
          dup = false;
          for (int j = 0; j < i; ++j) dup |= idx[j] == idx[i];
        } while (dup && ++tries < 16);
        ok = !dup;
      }
      Pose cand;
      if (ok) ok = p3p_best(Xs, xs, idx, fx, fy, cand);
      if (ok) {
        int cnt = 0;
        for (int k = 0; k < M; ++k) cnt += is_inlier(cand, Xs + k * 3, xs + k * 2, fx, fy, thr2) ? 1 : 0;
        if (cnt > my_cnt) { my_cnt = cnt; my_h = h; mine = cand; }
      }
    }
    // ---- arg-max over the block (ties: lowest hypothesis index, so the result does not depend on scheduling) ----
    atomicMax(&s_best_cnt, my_cnt);
    __syncthreads();
    if (my_cnt == s_best_cnt && my_cnt >= 0) atomicMin(&s_best_h, my_h);
    __syncthreads();
    if (s_best_cnt >= 4) {
      if (my_cnt == s_best_cnt && my_h == s_best_h) s_pose = mine;
      __syncthreads();
      P = s_pose;
      // ---- 4. least-squares refit on the inliers, inliers re-selected once ----
      for (int pass = 0; pass < 2; ++pass) {
        for (int k = tid; k < M; k += NT) mask[k] = is_inlier(P, Xs + k * 3, xs + k * 2, fx, fy, thr2) ? 1 : 0;
        __syncthreads();
        for (int it = 0; it < (pass == 0 ? 10 : 5); ++it)
          if (!gn_step(P, Xs, xs, mask, M, fx, fy, red, tid)) break;
      }
      float c = 0.f;
      for (int k = tid; k < M; k += NT) {
        const bool in = is_inlier(P, Xs + k * 3, xs + k * 2, fx, fy, thr2);
        c += in ? 1.f : 0.f;
        if (in && inl_mask_out) inl_mask_out[o * N + src[k]] = 1;
      }
      block_sum<1>(&c, red, tid);
      ninl = (int)(red[0] + 0.5);
    } else {
      __syncthreads();
    }
  }
  if (tid == 0) {
    for (int i = 0; i < 9; ++i) pose_out[o * 12 + i] = P.R[i];
    for (int i = 0; i < 3; ++i) pose_out[o * 12 + 9 + i] = P.t[i];
    ninl_out[o] = ninl;
  }
}

}  // namespace

// shared by the two entry points; `name` prefixes the error messages
static int pnp_launch(const char* name, const uint8_t* packed, const cp_corr_record* records, const float* p3d, const int32_t* graph_sel,
                      const float* cam_K, int k_batched, const int32_t* flag_masks, int num_sets, const int32_t* rng_index, float reproj_thresh,
                      int iterations, uint64_t seed, float* pose_out, int32_t* ninl_out, uint8_t* inlier_mask_out, int B, int N, int S,
                      cp_stream_t s) {
  CP_REQUIRE((packed != nullptr) != (records != nullptr) && p3d && cam_K && pose_out && ninl_out && B > 0 && N >= 4, CP_E_INVALID,
             "%s: bad arguments (exactly one of packed / records)", name);
  CP_REQUIRE(S > 0 && S <= 64 && N % 2 == 0 && N <= 8192, CP_E_UNSUPPORTED, "%s: needs S <= 64 and an even N <= 8192 (S=%d N=%d)", name, S, N);
  FlagSets sets = {{0u, 0u, 0u}};
  bool masks_ok = true;
  for (int v = 0; v < num_sets; ++v) {
    masks_ok &= flag_masks[v] >= 1 && flag_masks[v] <= 7;
    sets.mask[v] = (uint32_t)flag_masks[v];
  }
  CP_REQUIRE(masks_ok && reproj_thresh > 0.f && iterations >= 1, CP_E_INVALID, "%s: flag_mask in [1,7], reproj_thresh > 0, iterations >= 1", name);
  const int rounds = (iterations + NT - 1) / NT;
  const size_t smem = (size_t)N * (3 * 4 + 2 * 4 + 2 + 1);
  cudaError_t e = cudaFuncSetAttribute(pnp_ransac_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  CP_REQUIRE(e == cudaSuccess, CP_E_CUDA, "%s: cudaFuncSetAttribute failed: %s", name, cudaGetErrorString(e));
  pnp_ransac_kernel<<<dim3(B, num_sets), NT, smem, (cudaStream_t)s>>>(packed, records, p3d, graph_sel, cam_K, k_batched ? 9 : 0, sets, rng_index,
                                                                     reproj_thresh, rounds, seed, pose_out, ninl_out, inlier_mask_out, B, N, S);
  CP_CHECK_LAUNCH(name);
  return CP_OK;
}

extern "C" int cp_pnp_ransac(const uint8_t* packed, const cp_corr_record* records, const float* p3d, const int32_t* graph_sel, const float* cam_K, int k_batched,
                             int flag_mask, float reproj_thresh, int iterations, uint64_t seed, float* pose_out, int32_t* ninl_out,
                             uint8_t* inlier_mask_out, int B, int N, int S, cp_stream_t s) {
  const int32_t mask = flag_mask;
  return pnp_launch("cp_pnp_ransac", packed, records, p3d, graph_sel, cam_K, k_batched, &mask, 1, nullptr, reproj_thresh, iterations, seed,
                    pose_out, ninl_out, inlier_mask_out, B, N, S, s);
}

extern "C" int cp_pnp_ransac_sets(const uint8_t* packed, const cp_corr_record* records, const float* p3d, const int32_t* graph_sel,
                                  const float* cam_K, int k_batched, int num_sets, const int32_t* flag_masks, const int32_t* rng_index,
                                  float reproj_thresh, int iterations, uint64_t seed, float* pose_out, int32_t* ninl_out,
                                  uint8_t* inlier_mask_out, int B, int N, int S, cp_stream_t s) {
  CP_REQUIRE(flag_masks && num_sets >= 1 && num_sets <= 3, CP_E_INVALID, "cp_pnp_ransac_sets: needs 1 to 3 flag masks (got %d)", num_sets);
  for (int v = 0; v < num_sets; ++v)
    for (int u = 0; u < v; ++u)
      CP_REQUIRE(flag_masks[u] != flag_masks[v], CP_E_INVALID, "cp_pnp_ransac_sets: flag masks %d and %d are both %d", u, v, flag_masks[v]);
  return pnp_launch("cp_pnp_ransac_sets", packed, records, p3d, graph_sel, cam_K, k_batched, flag_masks, num_sets, rng_index, reproj_thresh,
                    iterations, seed, pose_out, ninl_out, inlier_mask_out, B, N, S, s);
}
