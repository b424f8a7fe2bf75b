// window.cuh -- the exact nearest-neighbour search in range-image space shared by evalq.cu (chamfer / --eval figures)
// and normals.cu (k-NN normals, point-to-plane error).
//
// Both clouds are range images over the same ray table.  Pixel (h, w) looks along elevation alt_h = vfov*h/(H-1) + vmin
// and azimuth az_w = hfov*w/W (dataset/transformer.py:41-54).  A candidate on a ray at angle t from the query's ray is at
// least r_query * sin(t) away, whatever its range.  Two rays whose rows differ by k are at least k*dalt apart (a
// great-circle distance is never smaller than the latitude difference); two rays whose columns differ by k (circularly)
// satisfy sin(t/2) >= cmin * sin(k*daz/2), cmin = the smallest cos(alt) of the sensor.  EvalGeom holds sin^2 of those
// angles less an absolute slack kEvTau, and the stop rule takes a relative margin of 2e-3 off the squared distance.
// A search grows a window of rows / columns around the query's own pixel until every pixel outside it is provably
// farther than what it still needs.
//
// Why both: the points are f32(r * f32(ray)), so each coordinate is off its exact value by at most
// r * (2^-25 + 2^-24) (the table's rounding, then the product's), and the difference vector of two points at ranges
// near r by at most 2 * sqrt(3) * 1.5 * 2^-24 * r = 3.1e-7 r.  That is an error in the ANGLE, absolute: relative to
// the bound r * sin(t) it grows as 3.1e-7 / t, and at fine angular pitches (t = 8.7e-5 rad for 65536 columns at -25
// degrees, 3.7e-5 rad for 16384 rows over 35 degrees) it outgrows any fixed relative margin.  kEvTau = 1e-6 rad
// covers it more than three times over: |b - a| >= r sin(t) - 3.1e-7 r >= r sin(t - kEvTau) while t - kEvTau stays
// below 90 degrees.  What is left is relative: the rounding of the subtraction, the squares and the two FMAs of
// cham_d (a few 2^-24), of the f32 tables and of r2 * table; the 2e-3 margin covers it, also near 90 degrees where
// the slack buys nothing.  The bound holds for any ray table that rounds each unit-vector component once, as
// transform_map does.  At the reference lidars (t >= 2.4e-3 rad) the slack is below 5e-4 of the pitch.
#pragma once
#include <math.h>

#include "common.cuh"

namespace rpcc {

constexpr int kEvR = 48;              // largest window half-size held in the tables; beyond it: whole-image scan
constexpr double kEvTau = 1e-6;       // absolute angular slack of the tables (rad), see the top of this file

struct EvalGeom {
  float row_s2[kEvR + 2];             // sin^2(smallest angle to any ray >= k rows away - kEvTau)
  float col_s2[kEvR + 2];             // same for >= k columns away (circular)
};

inline EvalGeom make_eval_geom(int H, int W, double hfov, double vmax, double vmin) {
  EvalGeom g;
  const double dalt = (vmax - vmin) / (double)(H - 1), daz = hfov / (double)W;
  const double cmin = cos(fmax(fabs(vmax), fabs(vmin)));
  const double half_pi = 1.57079632679489661923;
  for (int k = 0; k < kEvR + 2; ++k) {
    const double tr = fmax(0.0, k * dalt - kEvTau);
    g.row_s2[k] = tr >= half_pi ? 1.0f : (float)(sin(tr) * sin(tr));
    const double az = fmin(k * daz, 3.14159265358979323846);
    const double sh = cmin * sin(az / 2);                    // <= sin(t/2)
    const double t = fmax(0.0, 2.0 * asin(fmin(sh, 1.0)) - kEvTau);
    g.col_s2[k] = t >= half_pi ? 1.0f : (float)(sin(t) * sin(t));
  }
  return g;
}

__device__ __forceinline__ float cham_d(float ax, float ay, float az, float bx, float by, float bz) {
  const float x = bx - ax, y = by - ay, z = bz - az;   // chamfer3D.cu:29-35 with nvcc's contraction
  return __fmaf_rn(z, z, __fmaf_rn(x, x, __fmul_rn(y, y)));
}

// A negative range puts a point on the far side of the sensor, where the window bound does not hold: neg[f] is set for
// every frame f in which range_a or range_b ([B][HW] each; they may be the same array) holds one, and searches of such
// a frame are exhaustive (evalq.cu).
int eval_neg_flags(const float* range_a, const float* range_b, int B, int HW, unsigned* neg, cudaStream_t st);

// The walk every search here shares.  probe(hh, ww) visits the query's own pixel (h, w) first, then the pixels of a
// window grown one row pair or one column pair at a time, on the side whose bound is smaller, until limit() -- the
// squared distance the search still has to beat -- lies below the bound for everything outside the window.  No pixel
// is visited twice.  Past kEvR rows or columns, or at once when `exhaustive`, it calls restart(), counts the query in
// *fallback and visits every pixel of the image in raster order (the query's pixel again among them).
template <class Probe, class Limit, class Restart>
__device__ __forceinline__ void window_search(int H, int W, int h, int w, float rq, const EvalGeom& g, bool exhaustive,
                                              unsigned* fallback, Probe&& probe, Limit&& limit, Restart&& restart) {
  const float inf = __int_as_float(0x7f800000);
  probe(h, w);
  const float r2 = rq * rq * (1.0f - 2e-3f);
  int dr = 0, dc = 0;
  while (!exhaustive) {
    const float lb_row = (h - dr <= 0 && h + dr >= H - 1) ? inf : r2 * g.row_s2[dr + 1];
    const float lb_col = (2 * dc + 1 >= W) ? inf : r2 * g.col_s2[dc + 1];
    if (limit() < fminf(lb_row, lb_col)) return;
    if (lb_row == inf && lb_col == inf) return;            // the window is the whole image
    if (dr >= kEvR || dc >= kEvR) break;
    if (lb_row <= lb_col) {
      ++dr;
      for (int s = -1; s <= 1; s += 2) {
        const int hh = h + s * dr;
        if (hh < 0 || hh >= H) continue;
        for (int k = -dc; k <= dc; ++k) { int ww = w + k; ww += ww < 0 ? W : 0; ww -= ww >= W ? W : 0; probe(hh, ww); }
      }
    } else {
      ++dc;
      const int h0 = max(0, h - dr), h1 = min(H - 1, h + dr);
      for (int s = -1; s <= 1; s += 2) {
        int ww = w + s * dc; ww += ww < 0 ? W : 0; ww -= ww >= W ? W : 0;
        if (s == 1 && 2 * dc == W) continue;               // the two new columns coincide
        for (int hh = h0; hh <= h1; ++hh) probe(hh, ww);
      }
    }
  }
  // the tabulated window did not settle the search (for a nearest neighbour never the case in an encode -> decode
  // pair): scan everything
  restart();
  atomicAdd(fallback, 1u);
  for (int hh = 0; hh < H; ++hh)
    for (int ww = 0; ww < W; ++ww) probe(hh, ww);
}

// The point of image `rb` at flat pixel p, as PCTransformer.range_image_to_point_cloud computes it; false for an empty
// pixel and for a point with x + y + z == 0 (np.sum(points, -1) != 0, utils/evaluate_metrics.py:14-15).
__device__ __forceinline__ bool image_point(const float* __restrict__ rb, const float* __restrict__ lut, int p, float& x,
                                            float& y, float& z) {
  const float r = __ldg(rb + p);
  if (r == 0.f) return false;
  x = r * __ldg(lut + 3 * p); y = r * __ldg(lut + 3 * p + 1); z = r * __ldg(lut + 3 * p + 2);
  return (x + y) + z != 0.f;
}

// nearest valid point of image `rb` to the point (qx,qy,qz) = rq * ray(h,w); exact (see the top of this file).  With
// kIdx the flat pixel index of that point goes to *idx (-1 if the image has none): the first minimum in raster order,
// the neighbour the brute-force chamfer kernel picks.  Inlined into its caller; window_nn below is the out-of-line form.
template <bool kIdx>
__device__ __forceinline__ float nearest_in_window(const float* __restrict__ rb, const float* __restrict__ lut, int H,
                                                   int W, int h, int w, float rq, float qx, float qy, float qz,
                                                   const EvalGeom& g, bool exhaustive, unsigned* fallback, int* idx) {
  float best = __int_as_float(0x7f800000);
  int bi = -1;
  auto probe = [&](int hh, int ww) {
    const int p = hh * W + ww;
    float x, y, z;
    if (!image_point(rb, lut, p, x, y, z)) return;
    const float d = cham_d(qx, qy, qz, x, y, z);
    if constexpr (kIdx) {
      if (d < best || (d == best && p < bi)) { best = d; bi = p; }
    } else {
      best = d < best ? d : best;
    }
  };
  window_search(H, W, h, w, rq, g, exhaustive, fallback, probe, [&]() { return best; }, []() {});
  if constexpr (kIdx) *idx = bi;
  return best;
}

__device__ inline float window_nn(const float* __restrict__ rb, const float* __restrict__ lut, int H, int W, int h, int w,
                                  float rq, float qx, float qy, float qz, const EvalGeom& g, bool exhaustive,
                                  unsigned* fallback) {
  return nearest_in_window<false>(rb, lut, H, W, h, w, rq, qx, qy, qz, g, exhaustive, fallback, nullptr);
}

}  // namespace rpcc
