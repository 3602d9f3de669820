// Support-function network (HomogeneousICNN, dair_pll/deep_support_function.py:213-266; used by
// DeepSupportConvex.get_vertices, geometry.py:309-325): the memory-bound layers around the three
// (D x W) x (W x W) products.  The products themselves are plain FP64 library GEMMs (cuBLAS reaches
// 34 TFLOP/s = 92% of the FP64 peak on these shapes, tools/time_icnn.py); everything else -- the K = 3
// input layers, the LeakyReLU slope masks, the (D x W) -> (D x 3) output contraction and the two
// (3 x W) weight-gradient reductions -- is fused here into four passes so that each (D x W) array
// crosses HBM once per use instead of once per elementwise op.  All kernels are HBM-bound.
//
// Notation (depth 2, width W, D direction rows, slope s of the LeakyReLU):
//   h0 = lrelu(d Wd0)                         m0 = slope mask of h0 (recomputed from the sign of h0)
//   z1 = h0 |Wh| + d Wd1                      = [h0 | d | 0] [|Wh| ; Wd1 ; 0]   (one product, K = W + 8)
//   m1 = slope mask of z1
//   T  = m1 (|wout| * |Wh|^T)                 a0 = T o m0
//   p  = m1 (|wout| * Wd1^T) + a0 Wd0^T       (D x 3)  = d f / d d, the support point
// Backward for a cotangent gp (D x 3):  t = (gp Wd0) o m0,  G = t^T m1 (third product),
//   g1 = gp^T m1,  gWd0 = gp^T a0  (3 x W each, reduced here per block, summed by the caller).
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/dair_pll_b200.h"
#include "cn_launch.cuh"

namespace {

constexpr int kRowsPerBlock = 64;

// h0aug (D, W + 8): columns [0, W) = lrelu(d Wd0), [W, W+3) = d, rest 0.  One thread per column.
__global__ void icnn_input_kernel(const double* __restrict__ d, const double* __restrict__ Wd0, int64_t D, int W,
                                  double slope, double* __restrict__ h0aug) {
  const int Wa = W + 8;
  const int64_t r0 = (int64_t)blockIdx.x * kRowsPerBlock;
  const int64_t r1 = r0 + kRowsPerBlock < D ? r0 + kRowsPerBlock : D;
  for (int j = threadIdx.x; j < Wa; j += blockDim.x) {
    double w0 = 0, w1 = 0, w2 = 0;
    if (j < W) { w0 = Wd0[j]; w1 = Wd0[W + j]; w2 = Wd0[2 * W + j]; }
    for (int64_t r = r0; r < r1; ++r) {
      const double dx = d[3 * r], dy = d[3 * r + 1], dz = d[3 * r + 2];
      double v;
      if (j < W) {
        const double lin = dx * w0 + dy * w1 + dz * w2;
        v = lin > 0 ? lin : slope * lin;
      } else {
        v = j == W ? dx : (j == W + 1 ? dy : (j == W + 2 ? dz : 0.0));
      }
      h0aug[r * Wa + j] = v;
    }
  }
}

// z1 -> m1 in place
__global__ void icnn_mask_kernel(double* __restrict__ z, int64_t n, double slope) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) z[i] = z[i] > 0 ? 1.0 : slope;
}

// T -> a0 = T o m0 in place;  p = m1 V1^T + a0 Wd0^T with V1 = |wout| * Wd1 (3 x W).  One warp per row.
__global__ void icnn_output_kernel(double* __restrict__ T, const double* __restrict__ h0aug, const double* __restrict__ m1,
                                   const double* __restrict__ Wd0, const double* __restrict__ V1, int64_t D, int W,
                                   double slope, double* __restrict__ p) {
  const int Wa = W + 8;
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < D; r += nwarps) {
    double s0 = 0, s1 = 0, s2 = 0;
    for (int j = lane; j < W; j += 32) {
      const double m0 = h0aug[r * Wa + j] > 0 ? 1.0 : slope;
      const double a = T[r * W + j] * m0;
      const double m = m1[r * W + j];
      T[r * W + j] = a;
      s0 += m * V1[j] + a * Wd0[j];
      s1 += m * V1[W + j] + a * Wd0[W + j];
      s2 += m * V1[2 * W + j] + a * Wd0[2 * W + j];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s0 += __shfl_xor_sync(0xffffffffu, s0, o);
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (lane == 0) { p[3 * r] = s0; p[3 * r + 1] = s1; p[3 * r + 2] = s2; }
  }
}

// t = (gp Wd0) o m0;  per-block partial sums part[block][0..2][j] = sum_r gp[r,k] m1[r,j],
// part[block][3..5][j] = sum_r gp[r,k] a0[r,j].  One thread per column, fixed row order (deterministic).
__global__ void icnn_backward_kernel(const double* __restrict__ gp, const double* __restrict__ h0aug,
                                     const double* __restrict__ m1, const double* __restrict__ a0,
                                     const double* __restrict__ Wd0, int64_t D, int W, double slope, int rows_per_block,
                                     double* __restrict__ t, double* __restrict__ part) {
  const int Wa = W + 8;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = r0 + rows_per_block < D ? r0 + rows_per_block : D;
  for (int j = threadIdx.x; j < W; j += blockDim.x) {
    const double w0 = Wd0[j], w1 = Wd0[W + j], w2 = Wd0[2 * W + j];
    double a[6] = {0, 0, 0, 0, 0, 0};
    for (int64_t r = r0; r < r1; ++r) {
      const double gx = gp[3 * r], gy = gp[3 * r + 1], gz = gp[3 * r + 2];
      const double m0 = h0aug[r * Wa + j] > 0 ? 1.0 : slope;
      t[r * W + j] = (gx * w0 + gy * w1 + gz * w2) * m0;
      const double m = m1[r * W + j], av = a0[r * W + j];
      a[0] += gx * m; a[1] += gy * m; a[2] += gz * m;
      a[3] += gx * av; a[4] += gy * av; a[5] += gz * av;
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) part[((int64_t)blockIdx.x * 6 + k) * W + j] = a[k];
  }
}

// Support directions of the two elbow links against the ground (GeometryCollider.collide_plane_convex,
// geometry.py:560-567: minus the third row of the link's world rotation) and their n_query perturbed, normalised copies
// (DeepSupportConvex.get_vertices, geometry.py:309-325).  One thread per sample.
__global__ void elbow_support_directions_kernel(const double* __restrict__ q, int64_t q_stride, const double* __restrict__ axis,
                                                const double* __restrict__ pert0, const double* __restrict__ pert1, int nq,
                                                int64_t B, double* __restrict__ dirs0, double* __restrict__ dirs1) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const double* qb = q + b * q_stride;
  const double w = qb[0], x = qb[1], y = qb[2], z = qb[3], th = qb[7];
  const double s = 2.0 / (w * w + x * x + y * y + z * z);
  const double r[3] = {s * (x * z - w * y), s * (y * z + w * x), 1 - s * (x * x + y * y)};      // R1[2, :]
  const double a[3] = {axis[0], axis[1], axis[2]};
  // third row of R2 = R1 Rot(axis, th):  r Rot = r cos + (r x a) sin + a (a.r)(1 - cos)
  const double c = cos(th), sn = sin(th), ar = r[0] * a[0] + r[1] * a[1] + r[2] * a[2];
  const double rxa[3] = {r[1] * a[2] - r[2] * a[1], r[2] * a[0] - r[0] * a[2], r[0] * a[1] - r[1] * a[0]};
  double r2[3];
  for (int i = 0; i < 3; ++i) r2[i] = r[i] * c + rxa[i] * sn + a[i] * ar * (1 - c);
  for (int g = 0; g < 2; ++g) {
    const double* base = g == 0 ? r : r2;
    const double* pert = g == 0 ? pert0 : pert1;
    double* out = (g == 0 ? dirs0 : dirs1) + b * nq * 3;
    for (int k = 0; k < nq; ++k) {
      const double vx = -base[0] + pert[3 * k], vy = -base[1] + pert[3 * k + 1], vz = -base[2] + pert[3 * k + 2];
      const double n = sqrt(vx * vx + vy * vy + vz * vz);
      out[3 * k] = vx / n; out[3 * k + 1] = vy / n; out[3 * k + 2] = vz / n;
    }
  }
}

// Support directions of a single floating body against the ground (minus the third row of its world rotation, s = 2 / |q|^2
// for the unnormalised quaternion) and their n_query perturbed, normalised copies, as elbow_support_directions_kernel for
// one link.  One thread per sample.
__global__ void body_support_directions_kernel(const double* __restrict__ q, int64_t q_stride, const double* __restrict__ pert,
                                               int nq, int64_t B, double* __restrict__ dirs) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const double* qb = q + b * q_stride;
  const double w = qb[0], x = qb[1], y = qb[2], z = qb[3];
  const double s = 2.0 / (w * w + x * x + y * y + z * z);
  const double r[3] = {s * (x * z - w * y), s * (y * z + w * x), 1 - s * (x * x + y * y)};      // R[2, :]
  double* out = dirs + b * nq * 3;
  for (int k = 0; k < nq; ++k) {
    const double vx = -r[0] + pert[3 * k], vy = -r[1] + pert[3 * k + 1], vz = -r[2] + pert[3 * k + 2];
    const double n = sqrt(vx * vx + vy * vy + vz * vz);
    out[3 * k] = vx / n; out[3 * k + 1] = vy / n; out[3 * k + 2] = vz / n;
  }
}

}  // namespace

extern "C" {

int dpll_icnn_input_f64(const double* d, const double* Wd0, int64_t D, int32_t W, double slope, double* h0aug,
                        void* stream) {
  if (D < 0 || W <= 0 || !Wd0) return DPLL_EINVAL;
  if (D == 0) return DPLL_OK;
  if (!d || !h0aug) return DPLL_EINVAL;
  icnn_input_kernel<<<cn::grid_for(D, kRowsPerBlock), 288, 0, static_cast<cudaStream_t>(stream)>>>(d, Wd0, D, W, slope, h0aug);
  return cn::launch_status();
}

int dpll_elbow_support_directions_f64(const double* q, int64_t q_stride, const double* axis, const double* pert0,
                                      const double* pert1, int32_t n_query, int64_t B, double* dirs0, double* dirs1,
                                      void* stream) {
  if (B < 0 || n_query <= 0 || q_stride < 8 || !axis || !pert0 || !pert1) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  if (!q || !dirs0 || !dirs1) return DPLL_EINVAL;
  elbow_support_directions_kernel<<<cn::grid_for(B, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      q, q_stride, axis, pert0, pert1, n_query, B, dirs0, dirs1);
  return cn::launch_status();
}

int dpll_body_support_directions_f64(const double* q, int64_t q_stride, const double* pert, int32_t n_query, int64_t B,
                                     double* dirs, void* stream) {
  if (B < 0 || n_query <= 0 || q_stride < 4 || !pert) return DPLL_EINVAL;
  if (B == 0) return DPLL_OK;
  if (!q || !dirs) return DPLL_EINVAL;
  body_support_directions_kernel<<<cn::grid_for(B, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(q, q_stride, pert, n_query,
                                                                                                  B, dirs);
  return cn::launch_status();
}

int dpll_icnn_mask_f64(double* z, int64_t n, double slope, void* stream) {
  if (n < 0) return DPLL_EINVAL;
  if (n == 0) return DPLL_OK;
  if (!z) return DPLL_EINVAL;
  int blocks = cn::grid_for(n, 256 * 8);
  if (blocks > 148 * 16) blocks = 148 * 16;
  icnn_mask_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(z, n, slope);
  return cn::launch_status();
}

int dpll_icnn_output_f64(double* T, const double* h0aug, const double* m1, const double* Wd0, const double* V1, int64_t D,
                         int32_t W, double slope, double* p, void* stream) {
  if (D < 0 || W <= 0 || !Wd0 || !V1) return DPLL_EINVAL;
  if (D == 0) return DPLL_OK;
  if (!T || !h0aug || !m1 || !p) return DPLL_EINVAL;
  int blocks = cn::grid_for(D, 8);                 // 8 warps (rows) per block of 256 threads
  if (blocks > 148 * 8) blocks = 148 * 8;
  icnn_output_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(T, h0aug, m1, Wd0, V1, D, W, slope, p);
  return cn::launch_status();
}

// rows per block: 512 for large batches; small batches (the active rows of a step) still get ~4 blocks per SM
static int backward_rows_per_block(int64_t D) {
  int rows = 512;
  while (rows > 32 && D / rows < 148 * 4) rows >>= 1;
  return rows;
}

int dpll_icnn_backward_blocks(int64_t D) { return cn::grid_for(D, backward_rows_per_block(D)); }

int dpll_icnn_backward_f64(const double* gp, const double* h0aug, const double* m1, const double* a0, const double* Wd0,
                           int64_t D, int32_t W, double slope, double* t, double* part, void* stream) {
  if (D < 0 || W <= 0 || !Wd0) return DPLL_EINVAL;
  if (D == 0) return DPLL_OK;
  if (!gp || !h0aug || !m1 || !a0 || !t || !part) return DPLL_EINVAL;
  icnn_backward_kernel<<<dpll_icnn_backward_blocks(D), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      gp, h0aug, m1, a0, Wd0, D, W, slope, backward_rows_per_block(D), t, part);
  return cn::launch_status();
}

}  // extern "C"
