// evalq.cu -- stage 6 for range images: the reconstruction-quality figures the reference prints under --eval
// (tools/compress.py:157-192, tools/compress_datalist.py:166-199), for B frame pairs per launch.
//
//   depth error  max / mean |range_rec - range|                          (compress_datalist.py:180-182)
//   chamfer      calc_chamfer_distance(point_cloud, point_cloud_rec)     (utils/evaluate_metrics.py:9-45):
//                for every point of one cloud the squared distance to its nearest neighbour in the other
//                (NmDistanceKernel, chamfer3D.cu:12-154), then mean sqrt both ways and the F-score counts
//                (fscore.py:12-16)
//
// The reference's kernel is an O(N*M) scan: 8.8e9 pair evaluations per direction for a 64E frame.  Here both
// clouds are range images over the SAME ray table (cloud = range x LUT), which bounds the search exactly: a
// candidate on a ray at angle t from the query's ray is at least r_query * sin(t) away, whatever its range.  So
// the search starts at the query's own pixel and grows a window of rows / columns until every pixel outside it is
// provably farther than the best distance found (for encode -> decode pairs, where |range_rec - range| <= step/2,
// that is 1 to 5 candidates per point instead of ~94,000).  Distances use the reference's arithmetic
// (d = fma(z,z, fma(x,x, y*y)) on b - a), and the minimum over the window equals the minimum over the whole cloud,
// so dist1 / dist2 are bit-identical to the brute-force kernel's (tests/test_gpu_eval.py compares them with
// rpcc_chamfer_batch, which is itself pinned to oracle.chamfer_nn by test_plugin_fps_and_chamfer_drop_in).
//
// The search itself (window_nn, its bound and its tables) is in window.cuh, shared with normals.cu.
#include <math.h>

#include "window.cuh"

namespace rpcc {

constexpr int kEvThreads = 256;
constexpr int kEvCols = RPCC_EVAL_COLS;

// A negative range puts a point on the far side of the sensor, where the window bound does not hold: frames that
// contain one (possible only when the int16 symbols wrapped, i.e. at an accuracy far below the sensor's) are flagged
// here and searched exhaustively.
__global__ void eval_flags_kernel(const float* __restrict__ ra, const float* __restrict__ rb, int HW, unsigned* __restrict__ neg) {
  const int f = blockIdx.y;
  bool bad = false;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += gridDim.x * blockDim.x)
    bad = bad || ra[(size_t)f * HW + p] < 0.f || rb[(size_t)f * HW + p] < 0.f;
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(neg + f, 1u);
}

// One thread per pixel; per-CTA partial sums go to `part` in a fixed layout and are added up in CTA order by
// eval_finish_kernel, so the figures do not depend on scheduling.
__global__ void __launch_bounds__(kEvThreads)
eval_pixels_kernel(const float* __restrict__ ra_all, const float* __restrict__ rb_all, const float* __restrict__ lut,
                   const uint8_t* __restrict__ la_all, const uint8_t* __restrict__ lb_all, int H, int W, float thr,
                   EvalGeom g, float* __restrict__ dist1, float* __restrict__ dist2, double* __restrict__ part,
                   unsigned* __restrict__ fallback, const unsigned* __restrict__ neg) {
  const int f = blockIdx.y, HW = H * W;
  const int p = blockIdx.x * kEvThreads + threadIdx.x;
  const float* ra = ra_all + (size_t)f * HW;
  const float* rb = rb_all + (size_t)f * HW;
  double v[kEvCols];
#pragma unroll
  for (int q = 0; q < kEvCols; ++q) v[q] = 0.0;
  if (p < HW) {
    const int h = p / W, w = p - h * W;
    const bool exhaustive = neg[f] != 0u;
    const float a = __ldg(ra + p), b = __ldg(rb + p);
    const float lx = __ldg(lut + 3 * p), ly = __ldg(lut + 3 * p + 1), lz = __ldg(lut + 3 * p + 2);
    const float e = fabsf(b - a);                           // np.abs(range_image_rec - range_image)
    v[0] = (double)e; v[1] = (double)e;
    if (la_all && lb_all) v[11] = la_all[(size_t)f * HW + p] != lb_all[(size_t)f * HW + p] ? 1.0 : 0.0;
    const float ax = a * lx, ay = a * ly, az = a * lz;      // PCTransformer.range_image_to_point_cloud
    const float bx = b * lx, by = b * ly, bz = b * lz;
    const bool va = (ax + ay) + az != 0.f, vb = (bx + by) + bz != 0.f;
    float d1 = 0.f, d2 = 0.f;
    if (va) {
      d1 = window_nn(rb, lut, H, W, h, w, a, ax, ay, az, g, exhaustive, fallback + f);
      v[2] = 1.0; v[3] = (double)sqrtf(d1); v[4] = d1 < thr ? 1.0 : 0.0; v[5] = (double)d1;
    }
    if (vb) {
      d2 = window_nn(ra, lut, H, W, h, w, b, bx, by, bz, g, exhaustive, fallback + f);
      v[6] = 1.0; v[7] = (double)sqrtf(d2); v[8] = d2 < thr ? 1.0 : 0.0; v[9] = (double)d2;
    }
    if (dist1) dist1[(size_t)f * HW + p] = va ? d1 : -1.f;
    if (dist2) dist2[(size_t)f * HW + p] = vb ? d2 : -1.f;
  }
  __shared__ double s_part[kEvThreads / 32][kEvCols];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < kEvCols; ++q) {
    double x = v[q];
    if (q == 0) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(0xffffffffu, x, o));
    } else {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    }
    if (lane == 0) s_part[warp][q] = x;
  }
  __syncthreads();
  if (threadIdx.x < kEvCols) {
    const int q = threadIdx.x;
    double x = s_part[0][q];
    for (int k = 1; k < kEvThreads / 32; ++k) x = q == 0 ? fmax(x, s_part[k][q]) : x + s_part[k][q];
    part[((size_t)f * gridDim.x + blockIdx.x) * kEvCols + q] = x;
  }
}

__global__ void eval_finish_kernel(const double* __restrict__ part, int nblk, const unsigned* __restrict__ fallback,
                                   double* __restrict__ metrics) {
  const int f = blockIdx.x, q = threadIdx.x;
  if (q >= kEvCols) return;
  double x = 0.0;
  for (int k = 0; k < nblk; ++k) {
    const double y = part[((size_t)f * nblk + k) * kEvCols + q];
    x = q == 0 ? fmax(x, y) : x + y;
  }
  if (q == 10) x = (double)fallback[f];
  metrics[(size_t)f * kEvCols + q] = x;
}

// steps[b][l] (f64) for decoding what the encoder just wrote: uniform -> step; non-uniform -> step + level_dacc[salience]
// as QuantizationModule does in double precision (utils/compress_utils.py:48,124-131)
__global__ void eval_steps_kernel(const uint8_t* __restrict__ salience, int n, double step, const double* __restrict__ dacc8,
                                  double* __restrict__ steps) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s = step;
  if (salience) { const int lv = salience[i]; s = lv < 8 ? step + dacc8[lv] : step; }
  steps[i] = s;
}

int eval_neg_flags(const float* range_a, const float* range_b, int B, int HW, unsigned* neg, cudaStream_t st) {
  eval_flags_kernel<<<dim3(8, B), 256, 0, st>>>(range_a, range_b, HW, neg);
  RPCC_LAUNCH_CHECK("eval_flags_kernel");
  return RPCC_OK;
}

}  // namespace rpcc

using namespace rpcc;

extern "C" size_t rpcc_eval_workspace_bytes(int B, int H, int W) {
  const size_t nblk = ((size_t)H * W + kEvThreads - 1) / kEvThreads;
  return sizeof(double) * (size_t)B * nblk * kEvCols + 2 * sizeof(unsigned) * (size_t)B + 64;
}

extern "C" int rpcc_eval_batch(const float* range_ref, const float* range_rec, const float* lut, const uint8_t* labels_ref,
                               const uint8_t* labels_rec, int B, int H, int W, double hfov, double vmax, double vmin,
                               float threshold_sq, float* dist1, float* dist2, double* metrics, void* workspace,
                               void* stream) {
  RPCC_REQUIRE(range_ref && range_rec && lut && metrics && workspace, "null pointer");
  RPCC_REQUIRE(H >= 2 && W >= 1 && B >= 0 && B <= 65535, "bad sizes");
  RPCC_REQUIRE(fabs(hfov - 6.283185307179586) < 1e-6, "the window search needs a 360-degree sensor (columns wrap around)");
  if (B == 0) return RPCC_OK;
  const EvalGeom g = make_eval_geom(H, W, hfov, vmax, vmin);
  const int HW = H * W, nblk = (HW + kEvThreads - 1) / kEvThreads;
  double* part = static_cast<double*>(workspace);
  unsigned* fallback = reinterpret_cast<unsigned*>(part + (size_t)B * nblk * kEvCols);
  cudaStream_t st = as_stream(stream);
  unsigned* neg = fallback + B;
  RPCC_CUDA(cudaMemsetAsync(fallback, 0, 2 * sizeof(unsigned) * (size_t)B, st));
  if (int rc = eval_neg_flags(range_ref, range_rec, B, HW, neg, st)) return rc;
  eval_pixels_kernel<<<dim3(nblk, B), kEvThreads, 0, st>>>(range_ref, range_rec, lut, labels_ref, labels_rec, H, W,
                                                          threshold_sq, g, dist1, dist2, part, fallback, neg);
  RPCC_LAUNCH_CHECK("eval_pixels_kernel");
  eval_finish_kernel<<<B, 32, 0, st>>>(part, nblk, fallback, metrics);
  RPCC_LAUNCH_CHECK("eval_finish_kernel");
  return RPCC_OK;
}

extern "C" int rpcc_eval_steps_batch(const uint8_t* salience, int B, int K, double step, const double* level_dacc8_dev,
                                     double* steps, void* stream) {
  RPCC_REQUIRE(steps && (!salience || level_dacc8_dev), "null pointer");
  const int n = B * K;
  if (n == 0) return RPCC_OK;
  eval_steps_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(salience, n, step, level_dacc8_dev, steps);
  RPCC_LAUNCH_CHECK("eval_steps_kernel");
  return RPCC_OK;
}
