// fps.cu -- stage 2a: furthest point sampling.
//
// Replaces ops/fps/src/sampling_gpu.cu:24-184 (furthest_point_sampling_kernel + launcher) and,
// in the fused form, the mask + FPS lines of PointCloudSegment.segment
// (utils/segment_utils.py:137-141).
//
// Exactness contract (SURVEY A.2): the seed sequence is identical to the reference kernel's:
//   d  = fma(dz,dz, fma(dx,dx, dy*dy))            (the contraction nvcc emits for sampling_gpu.cu:64)
//   t[k] = min(d, t[k]), t starts at 1e10
//   winner = max t, ties -> min bitrev(k mod bs) over log2(bs) bits, then min k
// (the reference's per-thread strided scan with strict '>' followed by a shared-memory tree that
// keeps the lower slot on ties, sampling_gpu.cu:16-21,54-134; bs = min(1024, 2^floor(log2 n))).
// Every kernel below orders candidates by (t, ~tiekey) with
// tiekey = (bitrev(k mod bs) << (32-log2 bs)) | (k / bs); the pipeline has bs = 1024 (H*W >= 1024).
//
// Two paths:
//  * fps_generic_kernel: any (B,n,3) input, one CTA per batch item, state in global memory --
//    the drop-in for furthest_point_sampling_wrapper.  (bits(t) << 32) | ~tiekey in one 64-bit key,
//    so one unsigned max does it.
//  * the pipeline: mask + FPS fused, the masked point cloud built straight from range x LUT.  A
//    first-pass kernel does round 1 over every pixel, then one CTA per frame runs the remaining
//    rounds with exact bucket pruning over 64-pixel buckets (segment_fps_wide_kernel), at most
//    131 072 pixels.  Images whose pixel count is not a multiple of 4, or whose range / LUT / owner
//    bases are off a 16-byte boundary, are first staged into padded copies (segment_fps_launch);
//    m = 1 takes the same kernels.
//
// Owner hints (the encoder's chain; assign.cu reads them).  The rounds compute, for every pixel, the minimum t[p] over
// the centres of fps_dist(p, c); the pipeline path also leaves one byte per pixel saying which centre gave it, so that
// the label assignment can evaluate that one centre instead of searching all of them.  owner[p] = c < m promises
//   fps_dist(p, c) = t_final[p] (unmasked coordinates: the pixel is not masked) and
//   fps_dist(p, c') > t_final[p] * (1 + eps') for every other centre c',   eps' = 3.8e-6;
// owner[p] = 255 means "no hint", and any pixel may carry it.  The rules (eps = 4e-6, tau = 1e-30):
//  * first pass: 0 if the pixel is not an origin and tau <= t < 1e10 * (1 - eps) (the initial clamp, masked and empty
//    pixels and zero distances get 255), else 255;
//  * round j, touched non-origin pixel, d = fps_dist, told its running distance: d < told * (1 - eps) and d >= tau
//    -> j (every earlier centre is at least told away, and told > d * (1 + eps')); otherwise d <= told * (1 + eps)
//    -> 255 (a rival within eps: ties, duplicate centres); otherwise the byte stays;
//  * pruned buckets need nothing: a bucket is skipped only if fl(lb * 0.99999) >= its max t, and lb is a true lower
//    bound of fps_dist over the bucket (monotone roundings of non-negative terms), so a skipped centre lies beyond
//    t * (1 + 1e-5 - 2^-23) for every pixel of it -- the pruning slack must stay above eps;
//  * the last centre gets its update pass (without a winner search) when hints are asked for.
// eps' is eps less the rounding of the f32 constants and of the threshold products (< 1e-7 each).  Why a hint is exact
// in torch arithmetic: fps_dist (fma form) and assign.cu's torch_sum3 of rounded squares sum the same rounded
// differences with three roundings each, so both lie within 3 x 2^-24 (relative) of the exact non-negative sum once
// that sum is at least tau (far above the subnormals).  A rival's torch square then exceeds the owner's by a factor of
// at least (1 + eps')(1 - 12 x 2^-24) > 1 + 3e-6, and its correctly rounded square root the owner's by more than 1.5e-6
// less the 2^-24 of either rounding: strictly greater, so torch's first-index rule cannot hand the pixel to a
// lower-index rival either.  Staged images get no hints: their launch fills owner[] with 255.
#include <type_traits>

#include "common.cuh"

namespace rpcc {

__device__ __forceinline__ float fps_dist(float x, float y, float z, float x1, float y1, float z1) {
  const float dx = x - x1, dy = y - y1, dz = z - z1;
  return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}

__device__ __forceinline__ unsigned long long warp_key_max(unsigned long long k) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, k, o);
    k = other > k ? other : k;
  }
  return k;
}

__device__ __forceinline__ unsigned long long make_key(float d2, unsigned tiekey) {
  // d2 >= 0 (NaN coordinates are not supported): its bit pattern orders like the value
  return ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned long long)(0xFFFFFFFFu - tiekey);
}

// ------------------------------------------------------------------------------------------------
// generic kernel: one CTA per batch item, temp in global memory (the reference's buffer)
// ------------------------------------------------------------------------------------------------
constexpr int kGenThreads = 1024;

__global__ void __launch_bounds__(kGenThreads, 1)
fps_generic_kernel(const float* __restrict__ points, int n, int m, int log2bs, float* __restrict__ temp,
                   int* __restrict__ idx) {
  if (m <= 0) return;
  const int b = blockIdx.x;
  points += (size_t)b * n * 3;
  temp += (size_t)b * n;
  idx += (size_t)b * m;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned bsmask = (1u << log2bs) - 1u;
  __shared__ unsigned long long s_part[2][32];

  for (int k = tid; k < n; k += kGenThreads) temp[k] = 1e10f;
  if (tid == 0) idx[0] = 0;
  int old = 0;
  for (int j = 1; j < m; ++j) {
    const float x1 = points[(size_t)old * 3], y1 = points[(size_t)old * 3 + 1], z1 = points[(size_t)old * 3 + 2];
    unsigned long long best = 0;
    for (int k = tid; k < n; k += kGenThreads) {
      const float d = fps_dist(points[(size_t)k * 3], points[(size_t)k * 3 + 1], points[(size_t)k * 3 + 2], x1, y1, z1);
      const float d2 = fminf(d, temp[k]);
      temp[k] = d2;
      const unsigned t = (unsigned)k & bsmask;
      const unsigned tiekey = log2bs ? (__brev(t) & ~(0xFFFFFFFFu >> log2bs)) | ((unsigned)k >> log2bs) : (unsigned)k;
      const unsigned long long key = make_key(d2, tiekey);
      best = key > best ? key : best;
    }
    best = warp_key_max(best);
    if (lane == 0) s_part[j & 1][warp] = best;
    __syncthreads();
    best = warp_key_max(s_part[j & 1][lane]);
    const unsigned tiekey = 0xFFFFFFFFu - (unsigned)(best & 0xFFFFFFFFull);
    if (log2bs) {
      const unsigned t = __brev(tiekey & ~(0xFFFFFFFFu >> log2bs));
      old = (int)(((tiekey & (0xFFFFFFFFu >> log2bs)) << log2bs) | t);
    } else {
      old = (int)tiekey;
    }
    if (tid == 0) idx[j] = old;
  }
}

// torch float32 semantics of utils/segment_utils.py:137-139 for one pixel:
// |sum(pc*g)+g3| / norm(g) > thr ? pc : 0   (size-3 reductions associate as torch_sum3)
__device__ __forceinline__ void masked_point(float r, const float* __restrict__ lut3, float g0, float g1, float g2,
                                             float g3, float gnorm, float thr, float& x, float& y, float& z) {
  x = r * lut3[0]; y = r * lut3[1]; z = r * lut3[2];
  const float s = torch_sum3(x * g0, y * g1, z * g2);
  const float dif = fabsf(s + g3) / gnorm;
  if (!(dif > thr)) { x = 0.f; y = 0.f; z = 0.f; }
}

// ------------------------------------------------------------------------------------------------
// fused mask + FPS with exact bucket pruning: one CTA per frame, state in L2
// ------------------------------------------------------------------------------------------------
// Round j of FPS only lowers the running distance t[k] of points that are closer to the new centre
// than to every earlier one -- a few per cent of the image.  Pixels are grouped into buckets of 64
// consecutive pixels (neighbours on one beam); a bucket keeps its bounding box and its maximum t.
// A bucket whose box is farther from the new centre than sqrt(max t) cannot change (the test
// carries a 1e-5 relative slack, two orders of magnitude above the rounding of either side), so a
// round touches only the buckets around the new centre and the argmax comes from the per-bucket
// maxima.  Touched points are updated with the reference's own arithmetic, and maxima are exact,
// so the seed sequence is the reference's, bit for bit.
// Per frame this replaces 99 passes over 128 000 points by one pass plus ~50 buckets per round:
// a single CTA per frame suffices, no cross-SM exchange, 148+ frames in flight.
//   state in global memory (L2-resident): t[HW] per frame, bit 31 = "masked to the origin"
//   state on chip: boxes in shared memory (6 floats per bucket), max t in registers.
constexpr unsigned kNoTie = 0xFFFFFFFFu;
constexpr int kRoundThreads = 1024;   // the round kernel: CTAs of 1024 threads, two resident per SM
// owner hints (see the header): 1 -/+ eps and the floor tau
constexpr float kHintLo = 1.0f - 4e-6f, kHintHi = 1.0f + 4e-6f, kHintTau = 1e-30f;
constexpr unsigned kNoHint = 255u;

// ---- first pass as its own kernel: round 1 over every bucket is plain streaming work -- it wants registers
//      and many independent warps, the round loop below wants two resident CTAs of 1024 threads at 32 registers.  One warp
//      takes a run of consecutive buckets of one frame and leaves, per bucket, a 32-byte record {box, max t, unused} and,
//      per pixel, t (bit 31 = "masked to the origin") for the round kernel.
struct __align__(16) FpsBucket { float x0, y0, z0, x1, y1, z1; unsigned bmax, unused; };
constexpr int kFirstThreads = 256;

// Four consecutive pixels per lane (H*W a multiple of 4): 128-bit loads and stores, a bucket is 16 lanes, a warp does 2
// buckets at a time and the per-bucket reductions are 4-step shuffles.  The ground mask is decided by a * (1/|g|) wherever
// that is more than 1e-6 (relative) away from the threshold -- the correctly rounded quotient the reference compares is
// then on the same side -- and by the division itself for the lanes that are not.
__device__ __forceinline__ float seg16_min(float v) {
#pragma unroll
  for (int o = 1; o < 16; o <<= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float seg16_max(float v) {
#pragma unroll
  for (int o = 1; o < 16; o <<= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ unsigned seg16_umax(unsigned v) {
#pragma unroll
  for (int o = 1; o < 16; o <<= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__global__ void __launch_bounds__(kFirstThreads)
fps_first_pass4_kernel(const float* __restrict__ range, const float* __restrict__ lut, const float* __restrict__ ground,
                       int B, int HW, int NB, int runs, float thr, unsigned* __restrict__ temp_ws, FpsBucket* __restrict__ rec,
                       int* __restrict__ work, uint8_t* __restrict__ owner) {
  const int lane = threadIdx.x & 31;
  const int w = blockIdx.x * (kFirstThreads / 32) + (threadIdx.x >> 5);
  const int f = w / runs, c = w - f * runs;
  if (f >= B) return;                                        // warp-uniform
  int nlive = 0;                                             // buckets of this warp's run that can still change
  const int NG = (HW + 127) >> 7;                            // groups of 2 buckets
  const int per = (NG + runs - 1) / runs;
  const int ga = c * per, gb = min(NG, ga + per);
  const float* rg = range + (size_t)f * HW;
  uint4* temp4 = reinterpret_cast<uint4*>(temp_ws + (size_t)f * HW);
  const float4* lut4 = reinterpret_cast<const float4*>(lut);
  const float g0 = ground[f * 4], g1 = ground[f * 4 + 1], g2 = ground[f * 4 + 2], g3 = ground[f * 4 + 3];
  const float gnorm = sqrtf(torch_sum3(g0 * g0, g1 * g1, g2 * g2));
  const float rgn = 1.0f / gnorm, thi = thr + fabsf(thr) * 1e-6f, tlo = thr - fabsf(thr) * 1e-6f;
  float sx, sy, sz;                                          // seed 0 is flat index 0 (sampling_gpu.cu:44-46)
  masked_point(rg[0], lut, g0, g1, g2, g3, gnorm, thr, sx, sy, sz);
  const float INF = __int_as_float(0x7f800000), QNAN = __int_as_float(0x7fc00000);
  for (int g = ga; g < gb; ++g) {
    const int p0 = (g << 7) + 4 * lane;
    const bool inb = p0 < HW;                                // H*W % 4 == 0: all four pixels or none
    float4 r = make_float4(0.f, 0.f, 0.f, 0.f), l0 = r, l1 = r, l2 = r;
    if (inb) {
      r = ld_stream_f4(reinterpret_cast<const float4*>(rg + p0));
      const float4* lp = lut4 + (size_t)(p0 >> 2) * 3;
      l0 = __ldg(lp); l1 = __ldg(lp + 1); l2 = __ldg(lp + 2);
    }
    float x[4] = {r.x * l0.x, r.y * l0.w, r.z * l1.z, r.w * l2.y};
    float y[4] = {r.x * l0.y, r.y * l1.x, r.z * l1.w, r.w * l2.z};
    float z[4] = {r.x * l0.z, r.y * l1.y, r.z * l2.x, r.w * l2.w};
    // ---- ground mask (utils/segment_utils.py:137-139)
    float a[4];
    bool keep[4], unsure = false;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      a[i] = fabsf(torch_sum3(x[i] * g0, y[i] * g1, z[i] * g2) + g3);
      const float qa = a[i] * rgn;
      keep[i] = qa > thi;
      unsure = unsure || !(keep[i] || qa < tlo);
    }
    if (__any_sync(0xffffffffu, unsure)) {
#pragma unroll
      for (int i = 0; i < 4; ++i) keep[i] = a[i] / gnorm > thr;
    }
    // ---- round 1: t = min(d(point, seed 0), 1e10)
    float t[4];
    unsigned word[4], hints = 0u;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (!keep[i]) { x[i] = 0.f; y[i] = 0.f; z[i] = 0.f; }
      const bool origin = (x[i] == 0.f) && (y[i] == 0.f) && (z[i] == 0.f);
      t[i] = fminf(fps_dist(x[i], y[i], z[i], sx, sy, sz), 1e10f);
      word[i] = __float_as_uint(t[i]) | (origin ? 0x80000000u : 0u);
      hints |= (!origin && t[i] >= kHintTau && t[i] < 1e10f * kHintLo ? 0u : kNoHint) << (8 * i);   // owner: seed 0
    }
    if (inb) temp4[p0 >> 2] = make_uint4(word[0], word[1], word[2], word[3]);
    if (inb && owner) reinterpret_cast<unsigned*>(owner + (size_t)f * HW)[p0 >> 2] = hints;
    const unsigned t0 = inb ? __float_as_uint(t[0]) : 0u, t1 = inb ? __float_as_uint(t[1]) : 0u;
    const unsigned t2 = inb ? __float_as_uint(t[2]) : 0u, t3 = inb ? __float_as_uint(t[3]) : 0u;
    const unsigned bmax = seg16_umax(max(max(t0, t1), max(t2, t3)));
    const int b = (g << 1) + (lane >> 4);                    // this lane's bucket
    nlive += __popc(__ballot_sync(0xffffffffu, (lane & 15) == 0 && b < NB && bmax != 0u));
    FpsBucket o = {INF, INF, INF, -INF, -INF, -INF, 0u, 0u};
    // A bucket whose running distances are all zero -- ground and empty pixels when seed 0 is one of them, about half of
    // a frame's buckets -- can never change and keeps the defaults (maximum 0, empty box); when every bucket is at zero
    // the round kernel picks pixel 0 without looking at them.
    if (__any_sync(0xffffffffu, bmax != 0u)) {
      o.bmax = bmax;
      // box over the points that can still change (t > 0): the others are NaN, which min / max skip
      float mn[3] = {QNAN, QNAN, QNAN}, mx[3] = {QNAN, QNAN, QNAN};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool live = inb && t[i] > 0.f;
        const float lx = live ? x[i] : QNAN, ly = live ? y[i] : QNAN, lz = live ? z[i] : QNAN;
        mn[0] = fminf(mn[0], lx); mn[1] = fminf(mn[1], ly); mn[2] = fminf(mn[2], lz);
        mx[0] = fmaxf(mx[0], lx); mx[1] = fmaxf(mx[1], ly); mx[2] = fmaxf(mx[2], lz);
      }
      o.x0 = seg16_min(mn[0]); o.y0 = seg16_min(mn[1]); o.z0 = seg16_min(mn[2]);
      o.x1 = seg16_max(mx[0]); o.y1 = seg16_max(mx[1]); o.z1 = seg16_max(mx[2]);
      if (!(o.x0 == o.x0)) { o.x0 = INF; o.y0 = INF; o.z0 = INF; o.x1 = -INF; o.y1 = -INF; o.z1 = -INF; }   // no live point
    }
    if ((lane & 15) == 0 && b < NB) {
      float4* dst = reinterpret_cast<float4*>(rec + (size_t)f * NB + b);
      dst[0] = make_float4(o.x0, o.y0, o.z0, o.x1);
      dst[1] = make_float4(o.y1, o.z1, __uint_as_float(o.bmax), 0.f);
    }
  }
  if (work && lane == 0 && nlive) atomicAdd(work + f, nlive);
}

// The round kernels give one frame at a time to a CTA, and a frame's rounds cost in proportion to its buckets that can
// change (30 ... 60 % of them).  Handing the frames out longest first keeps the CTAs' finishing times together: queue[i] =
// the frame with the i-th largest count (ties by index; any order gives the same seeds), followed by `tail` entries B that
// send the CTAs home.  work == nullptr: index order.
constexpr int kOrderMaxFrames = 8192;
__global__ void __launch_bounds__(256)
fps_order_kernel(const int* __restrict__ work, int B, int tail, int* __restrict__ queue) {
  __shared__ int s_w[256];
  const int f = blockIdx.x * 256 + threadIdx.x;
  if (work == nullptr) {                                     // index order
    if (f < B + tail) queue[f] = f < B ? f : B;
    return;
  }
  const int w = f < B ? work[f] : 0;
  int rank = 0;
  for (int g0 = 0; g0 < B; g0 += 256) {                      // every thread of the block walks the same counts: a tile at a time
    __syncthreads();
    s_w[threadIdx.x] = g0 + (int)threadIdx.x < B ? work[g0 + threadIdx.x] : -1;
    __syncthreads();
    const int n = min(256, B - g0);
#pragma unroll 8
    for (int i = 0; i < n; ++i) {
      const int v = s_w[i];
      rank += (v > w || (v == w && g0 + i < f)) ? 1 : 0;
    }
  }
  if (f < B) queue[rank] = f;
  else if (f < B + tail) queue[f] = B;
}

__device__ __forceinline__ unsigned fps_tie_key(unsigned p) { return (__brev(p) & 0xFFC00000u) | (p >> 10); }

// ---- the rounds.  Most of a round's instructions, and its longest dependent chain, are the bucket updates: a warp walks
//      its touched buckets one at a time, one trip to L2 each.  A bucket is one warp wide at two consecutive pixels per
//      lane (64-bit loads): against 32-pixel buckets, half as many boxes to keep (48 KB per frame at 64 x 2000) and to
//      test, half as many update steps.  No tie key is kept per bucket: a round's winner is found by scanning the one
//      bucket that holds the frame's maximum (the load warp 0 makes anyway to fetch the centre's coordinates); only when
//      several buckets hold the very same maximum -- the origin points when seed 0 is not one of them, or equal
//      distances -- do all warps scan their candidates (TIE below).  Takes what segment_fps_launch guarantees: H*W a
//      multiple of 4 and 16-byte aligned range / LUT.
//      Measured on 1184 frames of 64 x 2000 (profiles/r02h_fps_pair_ab.txt, r02j_fps_wide_ab.txt): one 32-pixel bucket
//      per step 2.70 ms, two per step (16 lanes x 2 pixels each) 2.43-2.47 ms, 64-pixel buckets 2.26 ms at two CTAs of
//      1024 threads per SM -- and 2.51 ms at FOUR CTAs of 512 threads (a third fewer instructions, 46 % issue
//      utilisation): what shortens a round is warps working on the same frame, not more frames per SM.
//      Also measured (profiles/r02j_fps_wide_smemcoords_ab.txt): the point holding every bucket's maximum kept in shared
//      memory (first pass and update steps leave it), so that all warps reduce the candidates themselves -- one barrier
//      per round, no global load before the box tests.  Seeds identical, but a third more instructions (the capture in
//      every update step, the redundant reduction) at the same 63 % issue utilisation: 2.57-2.66 ms.  Not kept.
template <int Q>
__global__ void __launch_bounds__(kRoundThreads, 2)
segment_fps_wide_kernel(const float* __restrict__ range, const float* __restrict__ lut, const float* __restrict__ ground,
                        int B, int HW, int m, float thr, unsigned* __restrict__ temp_ws, const FpsBucket* __restrict__ rec,
                        int* __restrict__ next_frame, int* __restrict__ center_idx, float* __restrict__ centers,
                        uint8_t* __restrict__ owner) {
  constexpr int NW = kRoundThreads / 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int NB = (HW + 63) >> 6;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4* s_boxa = reinterpret_cast<float4*>(smem_raw);          // [Q][kRoundThreads]: x0, y0, z0, x1 of bucket (q, tid)
  float2* s_boxb = reinterpret_cast<float2*>(s_boxa + Q * kRoundThreads);   // [Q][kRoundThreads]: y1, z1
  __shared__ uint2 s_part[2][32];
  __shared__ float4 s_win[2];
  __shared__ int s_frame;
  const float INF = __int_as_float(0x7f800000);

  for (;;) {
    // queue: next_frame[0] = head, next_frame[64 ...] = the frames, longest first, then one B per CTA (fps_order_kernel)
    if (tid == 0) s_frame = next_frame[64 + atomicAdd(next_frame, 1)];
    __syncthreads();
    const int f = s_frame;
    if (f >= B) break;
    const float* rg = range + (size_t)f * HW;
    unsigned* temp = temp_ws + (size_t)f * HW;
    float sx, sy, sz;                                          // seed 0 is flat index 0 (sampling_gpu.cu:44-46)
    {
      const float g0 = ground[f * 4], g1 = ground[f * 4 + 1], g2 = ground[f * 4 + 2], g3 = ground[f * 4 + 3];
      masked_point(rg[0], lut, g0, g1, g2, g3, sqrtf(torch_sum3(g0 * g0, g1 * g1, g2 * g2)), thr, sx, sy, sz);
    }
    const bool seed0_origin = (sx == 0.f) && (sy == 0.f) && (sz == 0.f);
    if (tid == 0) {
      center_idx[(size_t)f * m] = 0;
      float* c = centers + (size_t)f * m * 3;
      c[0] = sx; c[1] = sy; c[2] = sz;
    }
    // ---- round 1 was done by the first-pass kernel: fetch this thread's records (boxes, maxima)
    unsigned bmax[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int b = warp + NW * (q * 32 + lane);
      float4 ra = make_float4(INF, INF, INF, -INF), rb = make_float4(-INF, -INF, 0.f, 0.f);
      if (b < NB) {
        const float4* src = reinterpret_cast<const float4*>(rec + (size_t)f * NB + b);
        ra = ld_stream_f4(src); rb = ld_stream_f4(src + 1);
      }
      s_boxa[q * kRoundThreads + tid] = ra;
      s_boxb[q * kRoundThreads + tid] = make_float2(rb.x, rb.y);
      bmax[q] = __float_as_uint(rb.z);
    }
    float x1 = sx, y1 = sy, z1 = sz;

    for (int j = 1; j < m; ++j) {
      // ---- winner of the previous round: the largest bucket maximum, then the point inside that bucket
      {
        unsigned d = bmax[0];
        int bq = 0, same = 1;                                  // how many of this lane's buckets hold d
#pragma unroll
        for (int q = 1; q < Q; ++q) {
          same = bmax[q] > d ? 1 : same + (bmax[q] == d ? 1 : 0);
          bq = bmax[q] > d ? q : bq;
          d = max(d, bmax[q]);
        }
        const unsigned dw = __reduce_max_sync(0xffffffffu, d);
        const unsigned holders = __reduce_add_sync(0xffffffffu, d == dw ? (unsigned)same : 0u);
        const unsigned code = __reduce_min_sync(0xffffffffu, d == dw ? (unsigned)(bq * 32 + lane) : 0xFFFFu);
        if (lane == 0) s_part[j & 1][warp] = make_uint2(dw, (unsigned)(warp + NW * (int)code) | (holders > 1u ? 0x80000000u : 0u));
        __syncthreads();
        if (warp == 0) {
          const uint2 v = lane < NW ? s_part[j & 1][lane] : make_uint2(0u, 0u);
          const unsigned dmax = __reduce_max_sync(0xffffffffu, v.x);
          const unsigned cand = __ballot_sync(0xffffffffu, lane < NW && v.x == dmax);
          const bool several = (cand & (cand - 1u)) != 0u || __any_sync(0xffffffffu, v.x == dmax && (v.y >> 31) != 0u);
          if (dmax == 0u) {
            // every running distance is zero: the tie rule picks pixel 0, which is seed 0 again
            if (lane == 0) {
              s_win[j & 1] = make_float4(sx, sy, sz, 0.f);
              center_idx[(size_t)f * m + j] = 0;
              float* c = centers + ((size_t)f * m + j) * 3;
              c[0] = sx; c[1] = sy; c[2] = sz;
            }
          } else if (!several) {
            const int bstar = (int)(__shfl_sync(0xffffffffu, v.y, __ffs(cand) - 1) & 0x7fffffffu);
            const int p = (bstar << 6) + (lane << 1);
            uint2 tb = make_uint2(0u, 0u);
            float2 r = make_float2(0.f, 0.f), la = r, lb2 = r, lc = r;
            if (p < HW) {                                      // H*W is even: both pixels or none
              tb = *reinterpret_cast<const uint2*>(temp + p);
              r = __ldg(reinterpret_cast<const float2*>(rg + p));
              const float2* l2 = reinterpret_cast<const float2*>(lut + (size_t)p * 3);
              la = __ldg(l2); lb2 = __ldg(l2 + 1); lc = __ldg(l2 + 2);
            }
            const unsigned ka = (p < HW && (tb.x & 0x7fffffffu) == dmax) ? fps_tie_key((unsigned)p) : kNoTie;
            const unsigned kb = (p < HW && (tb.y & 0x7fffffffu) == dmax) ? fps_tie_key((unsigned)p + 1u) : kNoTie;
            const unsigned tk = min(ka, kb);
            const unsigned tkmin = __reduce_min_sync(0xffffffffu, tk);
            if (tk == tkmin) {                                 // tie keys are unique: one lane (the bucket holds dmax)
              const bool second = kb < ka;
              const bool org = ((second ? tb.y : tb.x) >> 31) != 0u;
              const float rr = second ? r.y : r.x;
              const float wx = second ? lb2.y : la.x, wy = second ? lc.x : la.y, wz = second ? lc.y : lb2.x;
              const float cx = org ? 0.f : rr * wx, cy = org ? 0.f : rr * wy, cz = org ? 0.f : rr * wz;
              s_win[j & 1] = make_float4(cx, cy, cz, 0.f);
              center_idx[(size_t)f * m + j] = p + (second ? 1 : 0);
              float* c = centers + ((size_t)f * m + j) * 3;
              c[0] = cx; c[1] = cy; c[2] = cz;
            }
          } else if (lane == 0) {
            s_win[j & 1] = make_float4(__uint_as_float(dmax), 0.f, 0.f, 1.f);    // TIE: resolved by all warps below
          }
        }
        __syncthreads();
        float4 w = s_win[j & 1];
        if (w.w != 0.f) {                                      // block-uniform
          // TIE: every warp scans its buckets that hold the maximum for the smallest tie key
          const unsigned dmax = __float_as_uint(w.x);
          unsigned tkw = kNoTie;
#pragma unroll
          for (int q = 0; q < Q; ++q) {
            unsigned cm = __ballot_sync(0xffffffffu, bmax[q] == dmax);
            while (cm) {
              const int t = __ffs(cm) - 1;
              cm &= cm - 1;
              const int p = ((warp + NW * (q * 32 + t)) << 6) + (lane << 1);
              unsigned tk = kNoTie;
              if (p < HW) {
                const uint2 tb = *reinterpret_cast<const uint2*>(temp + p);
                if ((tb.x & 0x7fffffffu) == dmax) tk = fps_tie_key((unsigned)p);
                if ((tb.y & 0x7fffffffu) == dmax) tk = min(tk, fps_tie_key((unsigned)p + 1u));
              }
              tkw = min(tkw, __reduce_min_sync(0xffffffffu, tk));
            }
          }
          if (lane == 0) s_part[j & 1][warp] = make_uint2(tkw, 0u);      // (warp 0 read the maxima before the last barrier)
          __syncthreads();
          if (warp == 0) {
            const unsigned tkmin = __reduce_min_sync(0xffffffffu, lane < NW ? s_part[j & 1][lane].x : kNoTie);
            if (lane == 0) {
              const int k = (int)(((tkmin & 0x3FFFFFu) << 10) | __brev(tkmin & 0xFFC00000u));
              const float r = ld_stream_f(rg + k);
              const float wx = ld_stream_f(lut + (size_t)k * 3), wy = ld_stream_f(lut + (size_t)k * 3 + 1), wz = ld_stream_f(lut + (size_t)k * 3 + 2);
              const bool org = (temp[k] >> 31) != 0u;
              const float cx = org ? 0.f : r * wx, cy = org ? 0.f : r * wy, cz = org ? 0.f : r * wz;
              s_win[j & 1] = make_float4(cx, cy, cz, 0.f);
              center_idx[(size_t)f * m + j] = k;
              float* c = centers + ((size_t)f * m + j) * 3;
              c[0] = cx; c[1] = cy; c[2] = cz;
            }
          }
          __syncthreads();
          w = s_win[j & 1];
        }
        x1 = w.x; y1 = w.y; z1 = w.z;
      }
      if (j == m - 1 && owner == nullptr) break;             // the last centre needs an update pass only for the hints
      // ---- per q: which of my buckets can change, then update them with the reference arithmetic.  When seed 0 is an
      //      origin point (a ground or empty pixel 0: the usual case) every origin point sits at t = 0 for good --
      //      min(d, 0) = 0 whatever coordinates go in -- so the masked points need not be re-zeroed.  A pixel can
      //      change its running distance or its owner hint only if d <= told * (1 + eps): one compare on the common path.
      auto update = [&](auto simple, auto hints) {
#pragma unroll
        for (int q = 0; q < Q; ++q) {
          unsigned act;
          {
            const float4 ba = s_boxa[q * kRoundThreads + tid];
            const float2 bb = s_boxb[q * kRoundThreads + tid];
            const float ox = fmaxf(fmaxf(ba.x - x1, x1 - ba.w), 0.f);
            const float oy = fmaxf(fmaxf(ba.y - y1, y1 - bb.x), 0.f);
            const float oz = fmaxf(fmaxf(ba.z - z1, z1 - bb.y), 0.f);
            const float lb = __fmaf_rn(oz, oz, __fmaf_rn(oy, oy, ox * ox));
            act = __ballot_sync(0xffffffffu, lb * 0.99999f < __uint_as_float(bmax[q]));
          }
          while (act) {                                        // warp-uniform
            const int t = __ffs(act) - 1;
            act &= act - 1;
            const int p = ((warp + NW * (q * 32 + t)) << 6) + (lane << 1);
            unsigned nb = 0u;
            if (p < HW) {                                      // H*W is even: both pixels or none
              const uint2 told = *reinterpret_cast<const uint2*>(temp + p);
              const float2 r = __ldg(reinterpret_cast<const float2*>(rg + p));
              const float2* l2 = reinterpret_cast<const float2*>(lut + (size_t)p * 3);
              const float2 la = __ldg(l2), lb2 = __ldg(l2 + 1), lc = __ldg(l2 + 2);
              float xa = r.x * la.x, ya = r.x * la.y, za = r.x * lb2.x;
              float xb = r.y * lb2.y, yb = r.y * lc.x, zb = r.y * lc.y;
              if (!decltype(simple)::value) {
                const bool oa = (told.x >> 31) != 0u, ob = (told.y >> 31) != 0u;
                xa = oa ? 0.f : xa; ya = oa ? 0.f : ya; za = oa ? 0.f : za;
                xb = ob ? 0.f : xb; yb = ob ? 0.f : yb; zb = ob ? 0.f : zb;
              }
              const float oa_ = __uint_as_float(told.x & 0x7fffffffu), ob_ = __uint_as_float(told.y & 0x7fffffffu);
              const float da = fps_dist(xa, ya, za, x1, y1, z1), db = fps_dist(xb, yb, zb, x1, y1, z1);
              const float na = fminf(da, oa_), nb_ = fminf(db, ob_);                   // sampling_gpu.cu:64-66
              const bool ca = da <= oa_ * kHintHi, cb = db <= ob_ * kHintHi;
              if (ca || cb) {
                *reinterpret_cast<uint2*>(temp + p) = make_uint2(__float_as_uint(na) | (told.x & 0x80000000u),
                                                                 __float_as_uint(nb_) | (told.y & 0x80000000u));
                if (decltype(hints)::value) {                  // origin pixels keep their 255 (SIMPLE: t = 0 for good)
                  uint8_t* o = owner + (size_t)f * HW + p;
                  const bool ra = (decltype(simple)::value || (told.x >> 31) == 0u) && da < oa_ * kHintLo && da >= kHintTau;
                  const bool rb = (decltype(simple)::value || (told.y >> 31) == 0u) && db < ob_ * kHintLo && db >= kHintTau;
                  if (ca) o[0] = (uint8_t)(ra ? (unsigned)j : kNoHint);
                  if (cb) o[1] = (uint8_t)(rb ? (unsigned)j : kNoHint);
                }
              }
              nb = max(__float_as_uint(na), __float_as_uint(nb_));
            }
            const unsigned newmax = __reduce_max_sync(0xffffffffu, nb);
            bmax[q] = lane == t ? newmax : bmax[q];
          }
        }
      };
      if (owner == nullptr) {
        if (seed0_origin) update(std::true_type(), std::false_type()); else update(std::false_type(), std::false_type());
      } else {
        if (seed0_origin) update(std::true_type(), std::true_type()); else update(std::false_type(), std::true_type());
      }
    }
    __syncthreads();   // the next frame rewrites the boxes, s_part and s_frame
  }
}

// Copies B range images to [B][P] and the LUT to [P][3], P = H*W rounded up to a multiple of 4; each pad pixel is a copy
// of pixel 0 of its frame (see segment_fps_launch).
__global__ void __launch_bounds__(256)
fps_stage_kernel(const float* __restrict__ range, const float* __restrict__ lut, int B, int HW, int P,
                 float* __restrict__ range_s, float* __restrict__ lut_s) {
  const size_t n = (size_t)(B + 1) * P;                      // the B frames, then the LUT
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
    const size_t f = i / P;
    const int p = (int)(i - f * P), src = p < HW ? p : 0;
    if (f < (size_t)B) {
      range_s[i] = range[f * HW + src];
    } else {
      for (int c = 0; c < 3; ++c) lut_s[(size_t)p * 3 + c] = lut[(size_t)src * 3 + c];
    }
  }
}

// The pipeline's FPS (mask + rounds) for B frames; owner: nullptr, or [B][H*W] bytes that receive the owner hints of
// the header (the encoder passes its label buffer, which assign.cu then overwrites in place).
int segment_fps_launch(const float* range, const float* lut, const float* ground, int B, int H, int W, int m, float ground_thr,
                       int32_t* center_idx, float* centers, uint8_t* owner, cudaStream_t st) {
  RPCC_REQUIRE(range && lut && ground && center_idx && centers, "null pointer");
  const int HW = H * W;
  RPCC_REQUIRE(HW >= 1024, "range image must have at least 1024 pixels");
  RPCC_REQUIRE(m >= 1, "need at least one seed");
  RPCC_REQUIRE(owner == nullptr || m < (int)kNoHint, "owner hints need fewer than 255 seeds");
  if (B == 0) return RPCC_OK;
  const int NB = (HW + 63) / 64;                             // 64-pixel buckets: at most 2 per thread
  if (NB > 2048) {
    set_error("rpcc_segment_fps_batch: H*W = %d exceeds the on-chip capacity (131072 pixels)", HW);
    return RPCC_ERR_CAPACITY;
  }
  const int Q = NB <= 1024 ? 1 : 2;
  auto kern = Q == 1 ? segment_fps_wide_kernel<1> : segment_fps_wide_kernel<2>;
  const size_t smem = sizeof(float) * 6 * Q * kRoundThreads;
  RPCC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  RPCC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kRoundThreads, smem));
  if (per_sm < 1) per_sm = 1;
  int grid = per_sm * sm_count();
  if (grid > B) grid = B;
  // The kernels take H*W a multiple of 4 and range / LUT / owner on 16-byte boundaries (every lidar of the reference,
  // buffers from cudaMalloc).  Any other input is staged: the frames are copied to [B][P] and the LUT to [P][3],
  // P = H*W rounded up to a multiple of 4, and the same kernels run with H*W := P.  Each pad pixel is a copy of pixel 0
  // of its frame (range and ray), so the first pass masks it with the same arithmetic as seed 0 and it is bit-identical
  // to seed 0.  So:
  //  * its running distance is exactly 0 from the first pass on, and min(d, 0) keeps it there;
  //  * it is never in a box, which covers only t > 0;
  //  * it never wins a round: dmax == 0 picks pixel 0 explicitly, and the tie scan looks only at t == dmax > 0.
  // The seeds are those of the unpadded image, every centre index below the real H*W.  The staged rounds run without
  // owner hints (owner[] holds H*W bytes per frame, not P): the caller's bytes are all set to 255, "no hint".
  const bool direct = HW % 4 == 0 && (reinterpret_cast<uintptr_t>(range) | reinterpret_cast<uintptr_t>(lut) |
                                      reinterpret_cast<uintptr_t>(owner)) % 16 == 0;
  const int P = (HW + 3) & ~3;
  // scratch: running distances, bucket records, frame queue head + queue + live buckets per frame, staged images
  const size_t temp_bytes = sizeof(unsigned) * (size_t)B * P;
  const size_t rec_off = (temp_bytes + 255) & ~(size_t)255;
  const size_t ctr_off = rec_off + ((sizeof(FpsBucket) * (size_t)B * NB + 255) & ~(size_t)255);
  const size_t stage_off = ctr_off + ((256 + sizeof(int) * ((size_t)2 * B + grid) + 255) & ~(size_t)255);
  const size_t lut_off = stage_off + ((temp_bytes + 255) & ~(size_t)255);
  const bool ordered = B > grid && B <= kOrderMaxFrames;     // more frames than CTAs: longest first
  void* ws = nullptr;
  cudaMemPool_t pool = nullptr;
  { const int rc = scratch_pool(&pool); if (rc != RPCC_OK) return rc; }
  RPCC_CUDA(cudaMallocFromPoolAsync(&ws, direct ? stage_off : lut_off + sizeof(float) * 3 * (size_t)P, pool, st));
  unsigned char* base = static_cast<unsigned char*>(ws);
  unsigned* temp = static_cast<unsigned*>(ws);
  FpsBucket* rec = reinterpret_cast<FpsBucket*>(base + rec_off);
  int* counter = reinterpret_cast<int*>(base + ctr_off);     // queue head (256 bytes), the queue (B + grid entries), live buckets per frame (B)
  int* queue = counter + 64;
  int* work = queue + B + grid;
  cudaError_t le = cudaMemsetAsync(counter, 0, 256, st);
  if (le == cudaSuccess && ordered) le = cudaMemsetAsync(work, 0, sizeof(int) * (size_t)B, st);
  if (le == cudaSuccess && !direct) {
    float* range_s = reinterpret_cast<float*>(base + stage_off);
    float* lut_s = reinterpret_cast<float*>(base + lut_off);
    if (owner) le = cudaMemsetAsync(owner, (int)kNoHint, (size_t)B * HW, st);
    if (le == cudaSuccess) {
      const size_t blocks = ((size_t)(B + 1) * P + 255) / 256, cap = (size_t)8 * sm_count();
      fps_stage_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(range, lut, B, HW, P, range_s, lut_s);
      le = cudaGetLastError();
      count_launch();
    }
    range = range_s; lut = lut_s; owner = nullptr;
  }
  if (le == cudaSuccess) {
    const int runs = 32;                                     // warps per frame: ~63 buckets each at 64 x 2000
    const unsigned blocks = (unsigned)(((long long)B * runs + kFirstThreads / 32 - 1) / (kFirstThreads / 32));
    fps_first_pass4_kernel<<<blocks, kFirstThreads, 0, st>>>(range, lut, ground, B, P, NB, runs, ground_thr, temp, rec,
                                                              ordered ? work : nullptr, owner);
    le = cudaGetLastError();
    count_launch();
  }
  if (le == cudaSuccess) {
    fps_order_kernel<<<(B + grid + 255) / 256, 256, 0, st>>>(ordered ? work : nullptr, B, grid, queue);
    le = cudaGetLastError();
    count_launch();
  }
  if (le == cudaSuccess) {
    kern<<<grid, kRoundThreads, smem, st>>>(range, lut, ground, B, P, m, ground_thr, temp, rec, counter, center_idx, centers,
                                            owner);
    le = cudaGetLastError();
  }
  RPCC_CUDA(cudaFreeAsync(ws, st));
  RPCC_CUDA(le);
  count_launch();
  return RPCC_OK;
}

}  // namespace rpcc

using namespace rpcc;

extern "C" int rpcc_fps_batch(const float* points, int B, int n, int m, float* temp, int32_t* idx, void* stream) {
  RPCC_REQUIRE(points && temp && idx, "null pointer");
  RPCC_REQUIRE(B >= 0 && n >= 1 && m >= 0, "bad shape");
  if (B == 0 || m == 0) return RPCC_OK;
  int log2bs = 0;
  while ((2 << log2bs) <= n && log2bs < 10) ++log2bs;  // bs = min(1024, 2^floor(log2 n)), sampling_gpu.cu:9-13
  fps_generic_kernel<<<B, kGenThreads, 0, as_stream(stream)>>>(points, n, m, log2bs, temp, idx);
  RPCC_LAUNCH_CHECK("fps_generic_kernel");
  return RPCC_OK;
}

extern "C" int rpcc_segment_fps_batch(const float* range, const float* lut, const float* ground, int B, int H, int W,
                                      int m, float ground_thr, int32_t* center_idx, float* centers, void* stream) {
  return segment_fps_launch(range, lut, ground, B, H, W, m, ground_thr, center_idx, centers, nullptr, as_stream(stream));
}
