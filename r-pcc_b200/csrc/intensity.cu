// intensity.cu -- the optional intensity section of a `.rpcc` (DESIGN.md §4, "Intensity"): the owners' intensities
// (project.cu, rpcc_intensity_owner_batch) quantised to one byte per non-empty pixel in raster order, and the inverse.
//
// The reference drops the fourth column of a KITTI `.bin` (dataset/dataset.py:62) and writes zeros in its place
// (:72-81); this is a capability of this project's own.  The quantiser follows the geometry's conventions: step =
// 2 * intensity_accuracy in f64, q = clamp(round_half_away((double)i / step), 0, 255) with NaN -> 0, and the decoder's
// value is (float)((double)q * step), the form of the residual's dequantisation.
//
// One CTA of 1024 threads per frame walks the image in 1024-pixel steps; a pixel's rank among the frame's non-empty
// pixels is a block scan of a ballot, so the bytes land back to back at the frame's base without a second pass.
#include "common.cuh"

namespace rpcc {

constexpr int kIntThreads = 1024;

// exclusive rank of `flag` among the CTA's threads (raster order = thread order) and, in *total, how many are set
__device__ __forceinline__ unsigned cta_rank(bool flag, unsigned* s_w, unsigned* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned m = __ballot_sync(0xffffffffu, flag);
  if (lane == 0) s_w[warp] = __popc(m);
  __syncthreads();
  if (warp == 0) {
    const unsigned c = s_w[lane];
    unsigned incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    s_w[lane] = incl - c;
    if (lane == 31) s_w[32] = incl;
  }
  __syncthreads();
  const unsigned r = s_w[warp] + __popc(m & lanemask_lt());
  *total = s_w[32];
  __syncthreads();   // s_w is rewritten by the next step
  return r;
}

__device__ __forceinline__ uint8_t quantize_intensity(float v, double step, bool& clamped) {
  const double q = round((double)v / step);   // half away from zero
  if (q != q) return 0;                        // NaN
  if (q < 0.0) { clamped = true; return 0; }
  if (q > 255.0) { clamped = true; return 255; }
  return (uint8_t)q;
}

__global__ void __launch_bounds__(kIntThreads)
intensity_pack_kernel(const float* __restrict__ intensity, const float* __restrict__ range, int HW, double step,
                      const unsigned long long* __restrict__ base, uint8_t* __restrict__ out,
                      rpcc_frame_result* __restrict__ results) {
  __shared__ unsigned s_w[33];
  const int f = blockIdx.x;
  const float* im = intensity + (size_t)f * HW;
  const float* rg = range + (size_t)f * HW;
  uint8_t* o = out + base[f];
  unsigned at = 0;
  bool clamped = false;
  for (int p0 = 0; p0 < HW; p0 += kIntThreads) {
    const int p = p0 + threadIdx.x;
    const bool full = p < HW && rg[p] != 0.f;
    unsigned n;
    const unsigned r = cta_rank(full, s_w, &n);
    if (full) o[at + r] = quantize_intensity(im[p], step, clamped);
    at += n;
  }
  if (__syncthreads_or(clamped) && threadIdx.x == 0 && results) results[f].flags |= 8u;
}

// non-empty = label != 1; a frame whose stream (base[f] .. base[f+1]) is shorter than its non-empty pixels reads zeros
// past its end (the caller compares the lengths)
__global__ void __launch_bounds__(kIntThreads)
intensity_unpack_kernel(const uint8_t* __restrict__ labels, int HW, double step, const unsigned long long* __restrict__ base,
                        const uint8_t* __restrict__ in, float* __restrict__ intensity) {
  __shared__ unsigned s_w[33];
  const int f = blockIdx.x;
  const uint8_t* lb = labels + (size_t)f * HW;
  const uint8_t* q = in + base[f];
  const unsigned long long len = base[f + 1] - base[f];
  float* out = intensity + (size_t)f * HW;
  unsigned at = 0;
  for (int p0 = 0; p0 < HW; p0 += kIntThreads) {
    const int p = p0 + threadIdx.x;
    const bool full = p < HW && lb[p] != 1;
    unsigned n;
    const unsigned r = cta_rank(full, s_w, &n);
    if (p < HW) out[p] = (full && at + r < len) ? (float)((double)q[at + r] * step) : 0.f;
    at += n;
  }
}

}  // namespace rpcc

using namespace rpcc;

extern "C" int rpcc_intensity_pack_batch(const float* intensity, const float* range, int B, int H, int W, double step,
                                         const uint64_t* sym_base, uint8_t* out, rpcc_frame_result* results, void* stream) {
  RPCC_REQUIRE(intensity && range && sym_base && out, "null pointer");
  RPCC_REQUIRE(B >= 0 && H >= 1 && W >= 1, "bad shape");
  RPCC_REQUIRE(step > 0, "step must be positive");
  if (B == 0) return RPCC_OK;
  intensity_pack_kernel<<<B, kIntThreads, 0, as_stream(stream)>>>(intensity, range, H * W, step,
                                                                  reinterpret_cast<const unsigned long long*>(sym_base),
                                                                  out, results);
  RPCC_LAUNCH_CHECK("intensity_pack_kernel");
  return RPCC_OK;
}

extern "C" int rpcc_intensity_unpack_batch(const uint8_t* labels, const uint8_t* in, const uint64_t* base, int B, int H,
                                           int W, double step, float* intensity, void* stream) {
  RPCC_REQUIRE(labels && in && base && intensity, "null pointer");
  RPCC_REQUIRE(B >= 0 && H >= 1 && W >= 1, "bad shape");
  RPCC_REQUIRE(step > 0, "step must be positive");
  if (B == 0) return RPCC_OK;
  intensity_unpack_kernel<<<B, kIntThreads, 0, as_stream(stream)>>>(labels, H * W, step,
                                                                    reinterpret_cast<const unsigned long long*>(base), in,
                                                                    intensity);
  RPCC_LAUNCH_CHECK("intensity_unpack_kernel");
  return RPCC_OK;
}
