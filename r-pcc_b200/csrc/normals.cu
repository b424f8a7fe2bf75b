// normals.cu -- point-to-plane PSNR for range images: exact k-NN normals of a cloud, and the point-to-plane error
// between two clouds over the same ray table, B frames per launch.
//
// The reference's calc_point_to_point_plane_psnr (utils/evaluate_metrics.py:48-72) takes its normals from open3d's
// estimate_normals(KDTreeSearchParamHybrid(radius, max_nn)) (:133).  open3d is not available, so this file implements
// the definition written down in DESIGN.md ("Point-to-plane PSNR"); parity with open3d's normals is unpinned.
//
//   neighbourhood  the `knn` nearest points of the point's own cloud, the point itself included, restricted to those
//                  within `radius` (cham_d <= radius^2 in f32); distance ties go to the smaller flat pixel index.
//                  Found by the window search of window.cuh, which stops once the k-th best distance (or radius^2
//                  while fewer than k are found) lies below the bound for every pixel outside the window: exact.
//   normal         f64 covariance of the neighbourhood (two-pass: mean first, / n), cyclic Jacobi eigen-solve, the
//                  eigenvector of the smallest eigenvalue oriented so that n . p <= 0.  (0,0,0) = no normal: fewer
//                  than 3 neighbours, lambda2 == 0, or lambda1 - lambda0 <= 1e-6 lambda2 (e.g. one scan line).
//   error          for a point a of one cloud, b = its nearest point in the other (window_nn: the chamfer's
//                  neighbour), err = ((a - b) . n(b))^2 in f64, or cham_d(a, b) when b has no normal.
#include <math.h>

#include "window.cuh"

namespace rpcc {

constexpr int kNrThreads = 128;
constexpr int kP2Threads = 256;
constexpr int kP2Cols = RPCC_P2PLANE_COLS;
constexpr int kP2Sums = kP2Cols - 1;      // the last column, the whole-image scans, comes from the counters

// (d, p) < (bd, bi): distance first, then flat pixel index
__device__ __forceinline__ bool nn_less(float d, int p, float bd, int bi) { return d < bd || (d == bd && p < bi); }

// One Jacobi rotation of the symmetric 3x3 matrix (a) zeroing a_pq; r is the third index.  v's columns p, q rotate with it.
__device__ __forceinline__ void jacobi_rot(double& app, double& aqq, double& apq, double& arp, double& arq, double* vp,
                                           double* vq) {
  if (apq == 0.0) return;
  const double theta = 0.5 * (aqq - app) / apq;
  double t = 1.0 / (fabs(theta) + sqrt(1.0 + theta * theta));
  if (theta < 0.0) t = -t;
  const double c = 1.0 / sqrt(1.0 + t * t), s = t * c;
  app -= t * apq;
  aqq += t * apq;
  apq = 0.0;
  const double gp = arp, gq = arq;
  arp = c * gp - s * gq;
  arq = s * gp + c * gq;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double x = vp[i], y = vq[i];
    vp[i] = c * x - s * y;
    vq[i] = s * x + c * y;
  }
}

// Unit normal of the symmetric covariance (a00 a11 a22 a01 a02 a12) oriented against (px,py,pz); false = no normal.
__device__ __forceinline__ bool pca_normal(double a00, double a11, double a22, double a01, double a02, double a12, double px, double py,
                           double pz, double* n) {
  double v0[3] = {1.0, 0.0, 0.0}, v1[3] = {0.0, 1.0, 0.0}, v2[3] = {0.0, 0.0, 1.0};
  for (int sweep = 0; sweep < 32; ++sweep) {
    const double off = fabs(a01) + fabs(a02) + fabs(a12);
    if (off == 0.0 || off <= 1e-18 * (fabs(a00) + fabs(a11) + fabs(a22))) break;
    jacobi_rot(a00, a11, a01, a02, a12, v0, v1);   // p=0 q=1 r=2: a_rp = a02, a_rq = a12
    jacobi_rot(a00, a22, a02, a01, a12, v0, v2);   // p=0 q=2 r=1: a_rp = a01, a_rq = a21
    jacobi_rot(a11, a22, a12, a01, a02, v1, v2);   // p=1 q=2 r=0: a_rp = a10, a_rq = a20
  }
  // eigenvalues a00, a11, a22 with eigenvectors v0, v1, v2: the smallest, the middle, the largest
  double l0 = a00, l1 = a11, l2 = a22;
  double e0 = v0[0], e1 = v0[1], e2 = v0[2];
  if (l1 < l0) { const double t = l0; l0 = l1; l1 = t; e0 = v1[0]; e1 = v1[1]; e2 = v1[2]; }
  if (a22 < l0) { l2 = l1; l1 = l0; l0 = a22; e0 = v2[0]; e1 = v2[1]; e2 = v2[2]; }
  else if (a22 < l1) { l2 = l1; l1 = a22; }
  if (!(l2 != 0.0) || l1 - l0 <= 1e-6 * l2) return false;
  const double inv = 1.0 / sqrt(e0 * e0 + e1 * e1 + e2 * e2);
  const double sgn = (e0 * px + e1 * py + e2 * pz) > 0.0 ? -inv : inv;
  n[0] = e0 * sgn; n[1] = e1 * sgn; n[2] = e2 * sgn;
  return true;
}

// One thread per pixel: the k-NN neighbourhood of its point (list sorted by (distance, index), KMAX >= knn entries in
// registers), then its normal.
template <int KMAX>
__global__ void __launch_bounds__(kNrThreads)
normals_kernel(const float* __restrict__ range_all, const float* __restrict__ lut, int H, int W, int knn, float rad2,
               EvalGeom g, float* __restrict__ normals, unsigned* __restrict__ fallback, const unsigned* __restrict__ neg) {
  const int f = blockIdx.y, HW = H * W;
  const int p = blockIdx.x * kNrThreads + threadIdx.x;
  if (p >= HW) return;
  const float* rg = range_all + (size_t)f * HW;
  float* out = normals + ((size_t)f * HW + p) * 3;
  const float inf = __int_as_float(0x7f800000);
  float qx, qy, qz;
  if (!image_point(rg, lut, p, qx, qy, qz)) { out[0] = 0.f; out[1] = 0.f; out[2] = 0.f; return; }
  float bd[KMAX];
  int bi[KMAX];
  int cnt = 0;                 // accepted candidates (within the radius) so far
  float kd = inf;              // key of the knn-th entry (inf while fewer are held)
  int ki = 0x7fffffff;
  auto reset = [&]() {
#pragma unroll
    for (int j = 0; j < KMAX; ++j) { bd[j] = inf; bi[j] = 0x7fffffff; }
    cnt = 0; kd = inf; ki = 0x7fffffff;
  };
  reset();
  auto probe = [&](int hh, int ww) {
    const int c = hh * W + ww;
    float x, y, z;
    if (!image_point(rg, lut, c, x, y, z)) return;
    float d = cham_d(qx, qy, qz, x, y, z);
    if (!(d <= rad2) || !nn_less(d, c, kd, ki)) return;
    ++cnt;
    int cc = c;
#pragma unroll
    for (int j = 0; j < KMAX; ++j) {          // sorted insertion; entries past knn-1 are overflow, never read
      if (j < knn && nn_less(d, cc, bd[j], bi[j])) {
        const float td = bd[j]; const int ti = bi[j];
        bd[j] = d; bi[j] = cc; d = td; cc = ti;
      }
      if (j == knn - 1) { kd = bd[j]; ki = bi[j]; }
    }
  };
  window_search(H, W, p / W, p - (p / W) * W, __ldg(rg + p), g, neg[f] != 0u, fallback + f, probe,
                [&]() { return fminf(kd, rad2); }, reset);
  const int m = cnt < knn ? cnt : knn;
  if (m < 3) { out[0] = 0.f; out[1] = 0.f; out[2] = 0.f; return; }
  double sx = 0.0, sy = 0.0, sz = 0.0;
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    if (j < m) {
      float x, y, z;
      image_point(rg, lut, bi[j], x, y, z);
      sx += (double)x; sy += (double)y; sz += (double)z;
    }
  }
  const double inv_m = 1.0 / (double)m;
  const double mx = sx * inv_m, my = sy * inv_m, mz = sz * inv_m;
  double c00 = 0.0, c11 = 0.0, c22 = 0.0, c01 = 0.0, c02 = 0.0, c12 = 0.0;
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    if (j < m) {
      float x, y, z;
      image_point(rg, lut, bi[j], x, y, z);
      const double dx = (double)x - mx, dy = (double)y - my, dz = (double)z - mz;
      c00 += dx * dx; c11 += dy * dy; c22 += dz * dz; c01 += dx * dy; c02 += dx * dz; c12 += dy * dz;
    }
  }
  double n[3];
  if (!pca_normal(c00 * inv_m, c11 * inv_m, c22 * inv_m, c01 * inv_m, c02 * inv_m, c12 * inv_m, (double)qx, (double)qy,
                  (double)qz, n)) {
    out[0] = 0.f; out[1] = 0.f; out[2] = 0.f;
    return;
  }
  out[0] = (float)n[0]; out[1] = (float)n[1]; out[2] = (float)n[2];
}

// err of point (ax,ay,az) against its nearest neighbour j of image rb (window_nn); *no_normal when n(j) = (0,0,0)
__device__ __forceinline__ double p2plane_err(const float* __restrict__ rb, const float* __restrict__ lut,
                                              const float* __restrict__ nb, int j, float d, float ax, float ay, float az,
                                              bool* no_normal) {
  *no_normal = false;
  if (j < 0) return (double)d;                  // empty cloud on the other side: +inf
  const float nx = __ldg(nb + 3 * j), ny = __ldg(nb + 3 * j + 1), nz = __ldg(nb + 3 * j + 2);
  if (nx == 0.f && ny == 0.f && nz == 0.f) { *no_normal = true; return (double)d; }
  float bx, by, bz;
  image_point(rb, lut, j, bx, by, bz);
  const double e = ((double)ax - (double)bx) * (double)nx + ((double)ay - (double)by) * (double)ny +
                   ((double)az - (double)bz) * (double)nz;
  return e * e;
}

// One thread per pixel, both directions; per-CTA partial sums in a fixed layout, added up in CTA order by
// p2plane_finish_kernel (as eval_pixels_kernel / eval_finish_kernel), so the figures do not depend on scheduling.
__global__ void __launch_bounds__(kP2Threads)
p2plane_pixels_kernel(const float* __restrict__ ra_all, const float* __restrict__ rb_all, const float* __restrict__ lut,
                      const float* __restrict__ na_all, const float* __restrict__ nb_all, int H, int W, EvalGeom g,
                      double* __restrict__ part, unsigned* __restrict__ fallback, const unsigned* __restrict__ neg) {
  const int f = blockIdx.y, HW = H * W;
  const int p = blockIdx.x * kP2Threads + threadIdx.x;
  const float* ra = ra_all + (size_t)f * HW;
  const float* rb = rb_all + (size_t)f * HW;
  double v[kP2Sums];
#pragma unroll
  for (int q = 0; q < kP2Sums; ++q) v[q] = 0.0;
  if (p < HW) {
    const int h = p / W, w = p - h * W;
    const bool exhaustive = neg[f] != 0u;
#pragma unroll 1
    for (int dir = 0; dir < 2; ++dir) {        // ref -> rec, then rec -> ref
      const float* rq = dir ? rb : ra;
      const float* ro = dir ? ra : rb;
      const float* no = (dir ? na_all : nb_all) + (size_t)f * HW * 3;
      float qx, qy, qz;
      if (!image_point(rq, lut, p, qx, qy, qz)) continue;
      int j;
      const float d = nearest_in_window<true>(ro, lut, H, W, h, w, __ldg(rq + p), qx, qy, qz, g, exhaustive, fallback + f, &j);
      bool nn;
      const double e = p2plane_err(ro, lut, no, j, d, qx, qy, qz, &nn);
      if (dir == 0) { v[0] = 1.0; v[1] = e; v[2] = nn ? 1.0 : 0.0; }
      else { v[3] = 1.0; v[4] = e; v[5] = nn ? 1.0 : 0.0; }
    }
  }
  __shared__ double s_part[kP2Threads / 32][kP2Sums];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < kP2Sums; ++q) {
    double x = v[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) s_part[warp][q] = x;
  }
  __syncthreads();
  if (threadIdx.x < kP2Sums) {
    const int q = threadIdx.x;
    double x = s_part[0][q];
    for (int k = 1; k < kP2Threads / 32; ++k) x += s_part[k][q];
    part[((size_t)f * gridDim.x + blockIdx.x) * kP2Sums + q] = x;
  }
}

__global__ void p2plane_finish_kernel(const double* __restrict__ part, int nblk, const unsigned* __restrict__ fallback,
                                      double* __restrict__ metrics) {
  const int f = blockIdx.x, q = threadIdx.x;
  if (q >= kP2Cols) return;
  double x = 0.0;
  if (q == kP2Sums) {
    x = (double)fallback[f];
  } else {
    for (int k = 0; k < nblk; ++k) x += part[((size_t)f * nblk + k) * kP2Sums + q];
  }
  metrics[(size_t)f * kP2Cols + q] = x;
}

}  // namespace rpcc

using namespace rpcc;

extern "C" size_t rpcc_normals_workspace_bytes(int B, int H, int W) {
  (void)H; (void)W;
  return 2 * sizeof(unsigned) * (size_t)(B > 0 ? B : 0) + 64;
}

extern "C" int rpcc_normals_batch(const float* range, const float* lut, int B, int H, int W, double hfov, double vmax,
                                  double vmin, int knn, float radius, float* normals, void* workspace, void* stream) {
  RPCC_REQUIRE(range && lut && normals && workspace, "null pointer");
  RPCC_REQUIRE(H >= 2 && W >= 1 && B >= 0 && B <= 65535, "bad sizes");
  RPCC_REQUIRE(fabs(hfov - 6.283185307179586) < 1e-6, "the window search needs a 360-degree sensor (columns wrap around)");
  RPCC_REQUIRE(knn >= 3 && knn <= 32, "knn must be in [3, 32]");
  RPCC_REQUIRE(radius > 0.f, "radius must be positive");
  if (B == 0) return RPCC_OK;
  const EvalGeom g = make_eval_geom(H, W, hfov, vmax, vmin);
  const int HW = H * W;
  unsigned* fallback = static_cast<unsigned*>(workspace);
  unsigned* neg = fallback + B;
  cudaStream_t st = as_stream(stream);
  RPCC_CUDA(cudaMemsetAsync(fallback, 0, 2 * sizeof(unsigned) * (size_t)B, st));
  if (int rc = eval_neg_flags(range, range, B, HW, neg, st)) return rc;
  const float rad2 = radius * radius;             // one f32 rounding, as the oracle computes it
  const dim3 grid((HW + kNrThreads - 1) / kNrThreads, B);
  if (knn <= 16)
    normals_kernel<16><<<grid, kNrThreads, 0, st>>>(range, lut, H, W, knn, rad2, g, normals, fallback, neg);
  else
    normals_kernel<32><<<grid, kNrThreads, 0, st>>>(range, lut, H, W, knn, rad2, g, normals, fallback, neg);
  RPCC_LAUNCH_CHECK("normals_kernel");
  return RPCC_OK;
}

extern "C" size_t rpcc_p2plane_workspace_bytes(int B, int H, int W) {
  const size_t nblk = ((size_t)H * W + kP2Threads - 1) / kP2Threads;
  return sizeof(double) * (size_t)B * nblk * kP2Sums + 2 * sizeof(unsigned) * (size_t)B + 64;
}

extern "C" int rpcc_p2plane_batch(const float* range_ref, const float* range_rec, const float* lut,
                                  const float* normals_ref, const float* normals_rec, int B, int H, int W, double hfov,
                                  double vmax, double vmin, double* metrics, void* workspace, void* stream) {
  RPCC_REQUIRE(range_ref && range_rec && lut && normals_ref && normals_rec && metrics && workspace, "null pointer");
  RPCC_REQUIRE(H >= 2 && W >= 1 && B >= 0 && B <= 65535, "bad sizes");
  RPCC_REQUIRE(fabs(hfov - 6.283185307179586) < 1e-6, "the window search needs a 360-degree sensor (columns wrap around)");
  if (B == 0) return RPCC_OK;
  const EvalGeom g = make_eval_geom(H, W, hfov, vmax, vmin);
  const int HW = H * W, nblk = (HW + kP2Threads - 1) / kP2Threads;
  double* part = static_cast<double*>(workspace);
  unsigned* fallback = reinterpret_cast<unsigned*>(part + (size_t)B * nblk * kP2Sums);
  unsigned* neg = fallback + B;
  cudaStream_t st = as_stream(stream);
  RPCC_CUDA(cudaMemsetAsync(fallback, 0, 2 * sizeof(unsigned) * (size_t)B, st));
  if (int rc = eval_neg_flags(range_ref, range_rec, B, HW, neg, st)) return rc;
  p2plane_pixels_kernel<<<dim3(nblk, B), kP2Threads, 0, st>>>(range_ref, range_rec, lut, normals_ref, normals_rec, H, W, g,
                                                             part, fallback, neg);
  RPCC_LAUNCH_CHECK("p2plane_pixels_kernel");
  p2plane_finish_kernel<<<B, 32, 0, st>>>(part, nblk, fallback, metrics);
  RPCC_LAUNCH_CHECK("p2plane_finish_kernel");
  return RPCC_OK;
}
