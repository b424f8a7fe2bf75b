// ground.cu -- stage 2 prologue: deterministic ground-plane RANSAC on the device.
//
// Stands in for open3d's PointCloud.segment_plane(distance_threshold=0.1, ransac_n=10,
// num_iterations=100) as PointCloudSegment.segment calls it (utils/segment_utils.py:74-82,101-108).
// open3d is a third-party dependency that is neither vendored nor pinned by the reference, and the
// reference feeds it an UNSEEDED random subsample (segment_utils.py:103), so two reference runs do
// not produce the same bytes: there is nothing to be bit-exact against ("parity unpinned", DESIGN.md).
// What is kept: the candidate rule (z < -1.5; more than 5000 -> subsample to 5000; fewer than 800 ->
// every pixel), the hypothesis shape (10-point least-squares planes, 100 of them), the score
// (inlier count at 0.1 m, ties by lower rmse) and the final least-squares refit on the inliers of
// the best hypothesis (SURVEY App. G).  What changes: sampling is counter-based and keyed by
// (seed, frame key), the subsample is an even stride over the candidates in raster order.  The frame key
// is 0 unless the caller supplies one per frame (frame_keys), so by default a frame's plane -- and with
// it the frame's .rpcc bytes -- depends on the frame's content alone: not on its position in a batch, a
// datalist or a shard, nor on the GPU count (tests/test_gpu_datalist.py).
//
// One CTA per frame; the <= 5000 candidates live in shared memory, one warp scores one hypothesis.
// The image is read once (pass 1: candidate bit masks + running counts); the kept candidates are then
// located in the masks by rank, so their loads are independent of one another and all in flight together.
// oracle/rpcc_oracle.c:orc_ground_fit restates this kernel (samples, summation orders, kGfThreads = 512) and
// tests/test_gpu_stages.py compares the fitted planes bit for bit: a change of the arithmetic here must be mirrored there.
#include "ransac.cuh"

namespace rpcc {

constexpr int kGfThreads = 512;
constexpr int kGfOcc = 2;                                 // resident CTAs per SM
constexpr int kGfMaxPts = 5000;
constexpr int kGfPad = (kGfMaxPts + 127) / 128 * 128;   // slots padded so that a lane scores 4 consecutive points per load
constexpr int kGfIters = 100;
constexpr int kGfSample = 10;
constexpr int kGfSlots = (kGfMaxPts + kGfThreads - 1) / kGfThreads;   // slots gathered per thread

// point-plane distance of the scoring and refit passes (this kernel's own arithmetic, not the reference's: three fused
// multiply-adds; both passes must use the same expression so that the refit sees the inliers that were counted)
__device__ __forceinline__ float plane_dist(float a, float b, float c, float d, float x, float y, float z) {
  return fabsf(__fmaf_rn(a, x, __fmaf_rn(b, y, __fmaf_rn(c, z, d))));
}

__global__ void __launch_bounds__(kGfThreads, kGfOcc)
ground_fit_kernel(const float* __restrict__ range, const float* __restrict__ lut, int HW, unsigned long long seed,
                  const unsigned long long* __restrict__ frame_keys, float z_below, float inlier_thr,
                  float* __restrict__ ground) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* px = reinterpret_cast<float*>(smem_raw);
  float* py = px + kGfPad;
  float* pz = py + kGfPad;
  constexpr int NW = kGfThreads / 32;
  const int seg_len = (HW + NW - 1) / NW;
  const int seg_words = (seg_len + 31) / 32;
  unsigned* s_mask = reinterpret_cast<unsigned*>(pz + kGfPad);            // [NW][seg_words] candidate bits
  unsigned short* s_pref = reinterpret_cast<unsigned short*>(s_mask + NW * seg_words);  // [NW][seg_words] candidates before the word, in its segment
  __shared__ int s_warp[NW], s_base[NW + 1];
  __shared__ double s_plane[kGfIters][4];
  __shared__ unsigned long long s_score[kGfIters];  // (inliers << 40) | ~quantised rmse | ~iteration  (max wins)
  __shared__ double s_sums[10];
  __shared__ double s_part[NW][10];
  __shared__ double s_best[4];

  const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* rg = range + (size_t)f * HW;
  const unsigned long long fkey = frame_keys ? frame_keys[f] : 0ull;

  // Each warp owns a contiguous segment of the image, so the candidate order is the raster order.
  const int p_begin = warp * seg_len;
  const int p_end = min(HW, p_begin + seg_len);
  // pass 1: candidates (z < z_below; empty pixels have z = 0) as one bit per pixel, with the running count in front
  // of every word, in arrays private to the warp's segment
  {
    unsigned* wmask = s_mask + warp * seg_words;
    unsigned short* wpref = s_pref + warp * seg_words;
    int cnt = 0;
#pragma unroll 8
    for (int w = 0; w < seg_words; ++w) {      // every word is written: pass 2 searches wpref[] over the whole segment
      const int p = p_begin + w * 32 + lane;
      const bool c = p < p_end && (__ldg(rg + p) * __ldg(lut + 3 * p + 2) < z_below);
      const unsigned b = __ballot_sync(0xffffffffu, c);
      if (lane == 0) { wmask[w] = b; wpref[w] = (unsigned short)cnt; }
      cnt += __popc(b);
    }
    if (lane == 0) s_warp[warp] = cnt;
  }
  __syncthreads();
  int nc = 0;
  {
    int base = 0;
    for (int q = 0; q < NW; ++q) { const int c = s_warp[q]; if (q < tid) base += c; nc += c; }
    if (tid <= NW) s_base[tid] = base;      // s_base[w] = candidates before warp w's segment, s_base[NW] = all
  }
  const bool use_all = nc < 800;  // segment_utils.py:105-106
  if (use_all) nc = HW;
  const int ns = nc < kGfMaxPts ? nc : kGfMaxPts;
  const bool narrow = (unsigned long long)HW * (unsigned long long)kGfMaxPts < 0xFFFFFFFFull;
  __syncthreads();

  // pass 2: an even stride of the candidates, in raster order: candidate number r goes to slot floor(r * ns / nc) and
  // the first one there is kept, i.e. slot s holds candidate ceil(s * nc / ns).  Every thread locates the pixels of
  // its slots in the bit masks first and then loads them all at once.
  {
    const float qnan = __int_as_float(0x7fc00000);
    int pp[kGfSlots];
#pragma unroll
    for (int i = 0; i < kGfSlots; ++i) {
      const int s = tid + i * kGfThreads;
      pp[i] = -1;
      if (s < ns) {
        int r = s;
        if (ns != nc) {
          if (narrow) r = (int)(((unsigned)s * (unsigned)nc + (unsigned)ns - 1u) / (unsigned)ns);
          else r = (int)(((long long)s * nc + ns - 1) / ns);
        }
        if (use_all) {
          pp[i] = r;
        } else {
          int w = 0;                                         // the segment holding candidate r
#pragma unroll
          for (int step = NW / 2; step > 0; step >>= 1) if (s_base[w + step] <= r) w += step;
          const int rr = r - s_base[w];
          const unsigned short* wpref = s_pref + w * seg_words;
          int lo = 0, hi = seg_words - 1;                    // last word with wpref <= rr (empty words share their successor's count)
          while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if ((int)wpref[mid] <= rr) lo = mid; else hi = mid - 1;
          }
          const unsigned bits = s_mask[w * seg_words + lo];
          const int bit = (int)__fns(bits, 0u, rr - (int)wpref[lo] + 1);
          pp[i] = w * seg_len + lo * 32 + bit;
        }
      }
    }
    float rv[kGfSlots], lx[kGfSlots], ly[kGfSlots], lz[kGfSlots];
#pragma unroll
    for (int i = 0; i < kGfSlots; ++i) {
      rv[i] = 0.f; lx[i] = 0.f; ly[i] = 0.f; lz[i] = 0.f;
      if (pp[i] >= 0) {
        const int p = pp[i];
        rv[i] = __ldg(rg + p); lx[i] = __ldg(lut + 3 * p); ly[i] = __ldg(lut + 3 * p + 1); lz[i] = __ldg(lut + 3 * p + 2);
      }
    }
#pragma unroll
    for (int i = 0; i < kGfSlots; ++i) {
      const int s = tid + i * kGfThreads;
      if (pp[i] >= 0) { px[s] = rv[i] * lx[i]; py[s] = rv[i] * ly[i]; pz[s] = rv[i] * lz[i]; }
      else if (s < kGfPad) { px[s] = qnan; py[s] = qnan; pz[s] = qnan; }   // padding: |NaN| < thr is false, never an inlier
    }
    for (int s = tid + kGfSlots * kGfThreads; s < kGfPad; s += kGfThreads) { px[s] = qnan; py[s] = qnan; pz[s] = qnan; }
  }
  __syncthreads();
  const int ns4 = (ns + 3) >> 2;   // groups of 4 slots

  // hypotheses: one warp each
  for (int it = warp; it < kGfIters; it += NW) {
    // sample j is the (j+1)-th link of one splitmix64 chain: lane j walks the chain to its own link and
    // reduces it modulo ns (the 64-bit remainder is the expensive part), lane 0 then adds the ten points in order
    int myk = 0;
    if (lane < kGfSample) {
      unsigned long long st = splitmix64(splitmix64(seed + fkey) ^ ((unsigned long long)it << 40));
      for (int j = 0; j <= lane; ++j) st = splitmix64(st);
      myk = (int)(st % (unsigned long long)ns);
    }
    int ks[kGfSample];
#pragma unroll
    for (int j = 0; j < kGfSample; ++j) ks[j] = __shfl_sync(0xffffffffu, myk, j);
    if (lane == 0) {
      double s[10];
      for (int q = 0; q < 10; ++q) s[q] = 0.0;
#pragma unroll
      for (int j = 0; j < kGfSample; ++j) {
        const int k = ks[j];
        const double x = px[k], y = py[k], z = pz[k];
        s[0] += 1.0; s[1] += x; s[2] += y; s[3] += z;
        s[4] += x * x; s[5] += x * y; s[6] += x * z; s[7] += y * y; s[8] += y * z; s[9] += z * z;
      }
      double pl[4] = {0, 0, 0, 0};
      const bool ok = plane_from_sums(s, pl);
      s_plane[it][0] = ok ? pl[0] : 0.0; s_plane[it][1] = ok ? pl[1] : 0.0;
      s_plane[it][2] = ok ? pl[2] : 0.0; s_plane[it][3] = ok ? pl[3] : 0.0;
    }
    __syncwarp();
    const float a = (float)s_plane[it][0], b = (float)s_plane[it][1], c = (float)s_plane[it][2], d = (float)s_plane[it][3];
    int inl = 0;
    float err = 0.f;
    if (a != 0.f || b != 0.f || c != 0.f) {
      // a lane scores 4 consecutive slots per iteration (three 16-byte shared loads)
      for (int k4 = lane; k4 < ns4; k4 += 32) {
        const float4 X = reinterpret_cast<const float4*>(px)[k4];
        const float4 Y = reinterpret_cast<const float4*>(py)[k4];
        const float4 Z = reinterpret_cast<const float4*>(pz)[k4];
        const float d0 = plane_dist(a, b, c, d, X.x, Y.x, Z.x), d1 = plane_dist(a, b, c, d, X.y, Y.y, Z.y);
        const float d2 = plane_dist(a, b, c, d, X.z, Y.z, Z.z), d3 = plane_dist(a, b, c, d, X.w, Y.w, Z.w);
        if (d0 < inlier_thr) { ++inl; err += d0 * d0; }
        if (d1 < inlier_thr) { ++inl; err += d1 * d1; }
        if (d2 < inlier_thr) { ++inl; err += d2 * d2; }
        if (d3 < inlier_thr) { ++inl; err += d3 * d3; }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      inl += __shfl_xor_sync(0xffffffffu, inl, o);
      err += __shfl_xor_sync(0xffffffffu, err, o);
    }
    if (lane == 0) {
      const float rmse = inl > 0 ? sqrtf(err / (float)inl) : 1e9f;
      // larger is better: inliers first, then smaller rmse, then smaller iteration index
      s_score[it] = ((unsigned long long)inl << 40) | ((unsigned long long)(0xFFFFFFu - min(0xFFFFFFu, (unsigned)(rmse * 1e6f))) << 8) |
                    (unsigned long long)(0xFFu - it);
    }
  }
  __syncthreads();
  if (warp == 0) {
    // the scores are distinct (the iteration index is part of them): one maximum
    unsigned long long best = 0ull;
    for (int it = lane; it < kGfIters; it += 32) best = s_score[it] > best ? s_score[it] : best;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
      best = other > best ? other : best;
    }
    const int bi = 0xFF - (int)(best & 0xFFull);
    if (lane < 4) s_best[lane] = s_plane[bi][lane];
  }
  __syncthreads();
  // refit on the inliers of the best hypothesis (f64 sums)
  {
    const float a = (float)s_best[0], b = (float)s_best[1], c = (float)s_best[2], d = (float)s_best[3];
    double s[10];
    for (int q = 0; q < 10; ++q) s[q] = 0.0;
    for (int k = tid; k < ns; k += kGfThreads) {
      const double x = px[k], y = py[k], z = pz[k];
      if (plane_dist(a, b, c, d, px[k], py[k], pz[k]) < inlier_thr) {
        s[0] += 1.0; s[1] += x; s[2] += y; s[3] += z;
        s[4] += x * x; s[5] += x * y; s[6] += x * z; s[7] += y * y; s[8] += y * z; s[9] += z * z;
      }
    }
    // fixed reduction order (xor tree inside the warp, warps in index order): the plane must be
    // bit-reproducible from run to run
    for (int q = 0; q < 10; ++q) {
      double v = s[q];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) s_part[warp][q] = v;
    }
  }
  __syncthreads();
  if (tid < 10) {
    double v = 0.0;
    for (int w = 0; w < NW; ++w) v += s_part[w][tid];
    s_sums[tid] = v;
  }
  __syncthreads();
  if (tid == 0) {
    double pl[4];
    if (!plane_from_sums(s_sums, pl)) {
      if (s_best[0] != 0.0 || s_best[1] != 0.0 || s_best[2] != 0.0) { for (int q = 0; q < 4; ++q) pl[q] = s_best[q]; }
      else { pl[0] = 0.0; pl[1] = 0.0; pl[2] = 1.0; pl[3] = 1.73; }  // no usable plane: a level ground at sensor height
    }
    for (int q = 0; q < 4; ++q) ground[f * 4 + q] = (float)pl[q];
  }
}

}  // namespace rpcc

using namespace rpcc;

extern "C" int rpcc_ground_fit_batch(const float* range, const float* lut, int B, int H, int W, uint64_t seed,
                                     const uint64_t* frame_keys, float* ground, void* stream) {
  RPCC_REQUIRE(range && lut && ground, "null pointer");
  if (B == 0) return RPCC_OK;
  const size_t seg_words = (((size_t)H * W + kGfThreads / 32 - 1) / (kGfThreads / 32) + 31) / 32;
  RPCC_REQUIRE((size_t)H * W <= 65535u * (size_t)(kGfThreads / 32), "range image too large for the ground fit");
  const size_t smem = sizeof(float) * 3 * kGfPad + (sizeof(unsigned) + sizeof(unsigned short)) * (size_t)(kGfThreads / 32) * seg_words + 16;
  RPCC_CUDA(cudaFuncSetAttribute(ground_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ground_fit_kernel<<<B, kGfThreads, smem, as_stream(stream)>>>(
      range, lut, H * W, (unsigned long long)seed, reinterpret_cast<const unsigned long long*>(frame_keys), -1.5f, 0.1f, ground);
  RPCC_LAUNCH_CHECK("ground_fit_kernel");
  return RPCC_OK;
}
