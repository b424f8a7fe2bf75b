// assign.cu -- stage 2b + stage 3 accumulation.
//
// Replaces the torch eager block of PointCloudSegment.segment
// (utils/segment_utils.py:143-148,168-169: ground residual along the ray, 100 centre distances,
// argmax of -|.|, relabel) -- which materialises a (H,W,100,3) temporary of 153.6 MB per frame --
// by one fused per-pixel kernel, and accumulates what point_modeling
// (ops/cpp_modules/src/cpp_modules.cpp:471-518) and the stable label-major symbol order need.
//
// Arithmetic (SURVEY A.3): every torch op is its own kernel, so each elementwise result is
// rounded to f32 before the next; size-3 reductions associate as torch_sum3 (common.cuh).
//   channel 0   : | range - ( -g3 / sum3(g*lut) ) |
//   channel c>=1: sqrt( sum3( (pc - centre_c)^2 ) )          pc = range * lut
//   label = first argmin; label>0 -> +1; range==0 -> 1
// Centres that cannot win for any pixel of a warp are culled with bounding-box distance bounds first
// (see the kernel); the evaluated ones use exactly the arithmetic above.
//
// Per-label statistics are exact: range * 2^28 is an integer for range in [2^-5, 256), summed in
// u64 -- identical to the reference's double accumulation in raster order, whose partial sums are
// then all exactly representable (SURVEY H5).  Ranges outside that interval raise flags bit 0 and
// the frame's means are recomputed sequentially by model.cu.
#include "book.cuh"

namespace rpcc {

constexpr int kTile = RPCC_TILE;  // 1024 threads, one pixel each
constexpr int kMaxQ = 8;          // centres per lane in the bound pass: up to 256 centres

// order-preserving float <-> int maps, so that the warp-wide REDUX min / max work on floats
__device__ __forceinline__ int f2ord(float f) { const int b = __float_as_int(f); return b ^ ((b >> 31) & 0x7fffffff); }
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }
__device__ __forceinline__ float sqrt_approx(float v) { float r; asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(v)); return r; }

constexpr int kAsWarps = 8;        // one 1024-pixel tile per warp, 8 tiles of one frame per CTA
constexpr int kAsOcc = 6;          // resident CTAs per SM

// One warp walks one tile, 32 consecutive pixels (a slice) at a time -- neighbours on one beam -- and
// needs no block-level synchronisation after the centres are staged.  Per slice the warp bounds every
// centre against the slice's bounding sphere (centre o, radius R): a centre can be nearest to some
// pixel of the slice only if |c - o| <= min_c' |c' - o| + 2R.  That test costs 6 flops per centre
// (centres spread over the lanes) and leaves a handful of survivors, which all lanes then evaluate with
// the reference arithmetic verbatim, in ascending centre index with a strict '<' (torch.max's
// first-index rule).  The slack of 1e-5 relative on both sides of the test is two orders of magnitude
// above the rounding of the quantities compared, so a culled centre can neither win nor tie.
// Label statistics go to per-warp bins in shared memory (no atomics: one leader lane per label and
// slice) and are flushed once per tile.
//
// hinted: labels[] holds, on entry, the owner hints the FPS rounds of these very centres left (fps.cu's header): a
// byte c < m promises that centre c is the unique nearest one with a margin that keeps it the strict argmin of the
// reference arithmetic too.  A lane is resolved without the cull when its pixel is empty, when its ground residual is
// below the skip threshold (label 0, see below), or when it carries a hint: it then evaluates that one centre, and
// channel 0 against it decides as in the search (first index on ties).  The cull runs only for slices with an
// unresolved lane, over those lanes alone (sphere, reach, survivors).  Each lane reads its hint before it overwrites
// the byte with its label, hence no __restrict__ on labels.
template <int MQ>   // centres per lane in the bound pass (32 * MQ >= m; the padding sits at +inf)
__global__ void __launch_bounds__(kAsWarps * 32, kAsOcc)
assign_labels_kernel(const float* __restrict__ range, const float* __restrict__ lut, const float* __restrict__ ground,
                     const float* __restrict__ centers, int HW, int W, int m, int T, uint8_t* labels, Book bk, bool hinted) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int K = m + 2;
  constexpr int mq = MQ;
  float4* s_c = reinterpret_cast<float4*>(smem_raw);                               // [MQ * 32] x, y, z, -
  unsigned long long* s_sum = reinterpret_cast<unsigned long long*>(s_c + mq * 32); // [kAsWarps][K]
  unsigned* s_cnt = reinterpret_cast<unsigned*>(s_sum + kAsWarps * K);            // [kAsWarps][K]

  const int f = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tile = blockIdx.x * kAsWarps + warp;
  for (int c = tid; c < mq * 32; c += kAsWarps * 32) {
    // padding centres sit at +inf: they never survive
    const float inf = __int_as_float(0x7f800000);
    const float* cp = centers + ((size_t)f * m + c) * 3;
    s_c[c] = c < m ? make_float4(cp[0], cp[1], cp[2], 0.f) : make_float4(inf, inf, inf, 0.f);
  }
  unsigned long long* sum = s_sum + warp * K;
  unsigned* cnt = s_cnt + warp * K;
  for (int l = lane; l < K; l += 32) { cnt[l] = 0; sum[l] = 0; }
  __syncthreads();
  if (tile >= T) return;

  const float g0 = ground[f * 4], g1 = ground[f * 4 + 1], g2 = ground[f * 4 + 2], g3 = ground[f * 4 + 3];
  const float* rg = range + (size_t)f * HW;
  uint8_t* lb = labels + (size_t)f * HW;
  const int p_tile = tile * RPCC_TILE;
  int next_row = ((p_tile + W - 1) / W) * W;       // next pixel that starts an image row
  int carry = -1;                                  // label left of the slice (none for the tile's first pixel)
  unsigned ccnt = 0, flag = 0;

  // A centre at distance D from the ground plane cannot take a pixel whose ground residual is below D / 2: the residual
  // |r - rplane| along the ray bounds the pixel's own distance to the plane, so |p - c| >= D - residual > residual.  With
  // D the smallest such distance over the frame's centres (the FPS seeds lie beyond the ground threshold of it), a slice
  // whose residuals all stay below D / 2 (minus a margin that covers the f32 rounding of both sides up to ranges of
  // hundreds of metres) is ground without looking at any centre.  The argument holds pixel by pixel.
  float skip_thr;
  {
    float dpl = __int_as_float(0x7f800000);
#pragma unroll
    for (int q = 0; q < MQ; ++q) {
      const float4 c = s_c[q * 32 + lane];
      if (q * 32 + lane < m) dpl = fminf(dpl, fabsf(torch_sum3(c.x * g0, c.y * g1, c.z * g2) + g3));
    }
    dpl = __uint_as_float(__reduce_min_sync(0xffffffffu, __float_as_uint(dpl)));
    const float gn = sqrtf(g0 * g0 + g1 * g1 + g2 * g2);
    skip_thr = 0.5f * (dpl / gn) * 0.99f - 2e-4f;       // NaN / inf planes: the comparison below is false, nothing is skipped
    if (!(gn > 0.f) || !(dpl < 1e30f)) skip_thr = -1.f;
  }
  // the loads of slice s + 1 are issued before slice s is worked on (the body is several hundred dependent instructions)
  float rn = 0.f, tn0 = 0.f, tn1 = 0.f, tn2 = 0.f;
  unsigned hn = 255u;
  auto fetch = [&](int pp) {
    rn = 0.f; tn0 = 0.f; tn1 = 0.f; tn2 = 0.f; hn = 255u;
    if (pp < HW) {
      rn = ld_stream_f(rg + pp);
      const float* l3 = lut + 3 * pp;
      tn0 = __ldg(l3); tn1 = __ldg(l3 + 1); tn2 = __ldg(l3 + 2);
      if (hinted) hn = lb[pp];
    }
  };
  fetch(p_tile + lane);
#pragma unroll 1
  for (int s = 0; s < RPCC_TILE / 32; ++s) {
    const int p0 = p_tile + s * 32, p = p0 + lane;
    if (p0 >= HW) break;
    const bool inb = p < HW;
    int label = 1;
    const float r = rn, t0 = tn0, t1 = tn1, t2 = tn2;
    const unsigned hint = hn;
    if (s + 1 < RPCC_TILE / 32) fetch(p + 32);
    float x = 0.f, y = 0.f, z = 0.f, best = 0.f;
    if (r != 0.0f) {                                  // (out-of-bounds lanes carry r = 0)
      x = r * t0; y = r * t1; z = r * t2;
      const float rplane = (-g3) / torch_sum3(g0 * t0, g1 * t1, g2 * t2);
      best = fabsf(r - rplane);                       // channel 0 (utils/segment_utils.py:143)
    }
    const bool valid = inb && r != 0.0f;
    bool act = valid && !(best < skip_thr);           // unresolved: needs the search
    if (valid) label = 0;                             // a residual below the skip threshold: ground (the others: below)
    if (act && hint < (unsigned)m) {                  // the FPS owner hint: one centre, the reference arithmetic
      const float4 cc = s_c[hint];
      const float dx = x - cc.x, dy = y - cc.y, dz = z - cc.z;
      const float s2 = torch_sum3(dx * dx, dy * dy, dz * dz);
      // sqrtf(s2) < best, decided on the squares where they are clear of each other: s2 below RD(RD(best^2) * (1 - 1e-6))
      // puts sqrt(s2) below best * (1 - 4.7e-7), which its rounding (2^-24 relative) cannot reach; s2 >= RU(best^2) gives
      // sqrtf(s2) >= best (see the search below).  In between, and for NaN / inf, the square root decides.
      const bool win = s2 < __fmul_rd(__fmul_rd(best, best), 0.999999f) ||
                       (!(s2 >= __fmul_ru(best, best)) && sqrtf(s2) < best);
      label = win ? (int)hint + 2 : 0;
      act = false;
    }
    if (__any_sync(0xffffffffu, act)) {
      const float maxb = __uint_as_float(__reduce_max_sync(0xffffffffu, act ? __float_as_uint(best) : 0u));
      // bounding sphere of the slice's unresolved points: box centre, farthest such point.  Any centre will do -- the radius
      // below is taken from the points themselves -- so the box comes from coordinates shifted by +256 m, whose bit
      // patterns order like the values for anything a lidar returns (one REDUX per face, no order-preserving transform);
      // beyond that range the centre is merely a poor one and the sphere a large one.
      const unsigned ux = __float_as_uint(x + 256.f), uy = __float_as_uint(y + 256.f), uz = __float_as_uint(z + 256.f);
      const float ox = __fmaf_rn(0.5f, __uint_as_float(__reduce_min_sync(0xffffffffu, act ? ux : 0x7f7fffffu)) +
                                       __uint_as_float(__reduce_max_sync(0xffffffffu, act ? ux : 0u)), -256.f);
      const float oy = __fmaf_rn(0.5f, __uint_as_float(__reduce_min_sync(0xffffffffu, act ? uy : 0x7f7fffffu)) +
                                       __uint_as_float(__reduce_max_sync(0xffffffffu, act ? uy : 0u)), -256.f);
      const float oz = __fmaf_rn(0.5f, __uint_as_float(__reduce_min_sync(0xffffffffu, act ? uz : 0x7f7fffffu)) +
                                       __uint_as_float(__reduce_max_sync(0xffffffffu, act ? uz : 0u)), -256.f);
      const float ex = x - ox, ey = y - oy, ez = z - oz;
      const float e2 = act ? __fmaf_rn(ez, ez, __fmaf_rn(ey, ey, ex * ex)) : 0.f;
      // (bounds only: the approximate square root's 2 ulp disappear in the 1e-5 slack)
      const float R = sqrt_approx(__uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(e2)))) * 1.00001f;
      // squared distance of every centre to the sphere centre (centre q * 32 + lane), and the smallest
      float d2[MQ];
      float dmin = __int_as_float(0x7f800000);
#pragma unroll
      for (int q = 0; q < MQ; ++q) {
        const float4 c = s_c[q * 32 + lane];
        const float ax = c.x - ox, ay = c.y - oy, az = c.z - oz;
        d2[q] = __fmaf_rn(az, az, __fmaf_rn(ay, ay, ax * ax));
        dmin = fminf(dmin, d2[q]);                  // NaN centres drop out here and below (comparisons are false)
      }
      dmin = __uint_as_float(__reduce_min_sync(0xffffffffu, __float_as_uint(dmin)));
      // a centre takes a pixel only with |p - c| < best_p (the pixel's ground residual), so it must also lie within
      // max(best) + R of the sphere centre: slices of ground pixels (residuals of centimetres) keep no centre at all
      const float reach = fminf(sqrt_approx(dmin) * 1.00001f + 2.0f * R, (maxb * 1.00001f + R) * 1.00001f);
      const float thr2 = reach * reach * 1.00001f;
      // Survivors are evaluated in ascending centre index with a strict '<' (torch.max's first-index rule).  The square
      // root is taken only when some lane can still improve: sqrtf is correctly rounded and monotone, so a squared
      // distance s >= RU(best * best) gives sqrtf(s) >= best and cannot win.  (NaN / inf on either side fail the
      // comparison below and take the square root, as before.)
      int bi = 0;
      float best2 = __fmul_ru(best, best);
#pragma unroll
      for (int q = 0; q < MQ; ++q) {
        unsigned surv = __ballot_sync(0xffffffffu, d2[q] * 0.99999f <= thr2);
        while (surv) {
          const int b = __ffs(surv) - 1;
          surv &= surv - 1;
          const int ci = q * 32 + b;
          const float4 cc = s_c[ci];
          const float dx = x - cc.x, dy = y - cc.y, dz = z - cc.z;
          const float s2 = torch_sum3(dx * dx, dy * dy, dz * dz);
          if (__any_sync(0xffffffffu, act && !(s2 >= best2))) {
            const float v = sqrtf(s2);                                     // channel ci + 1 (:144, :25-26)
            if (v < best) { best = v; bi = ci + 1; best2 = __fmul_ru(v, v); }
          }
        }
      }
      if (act) label = bi > 0 ? bi + 1 : 0;            // :168-169
    }
    if (inb) lb[p] = (uint8_t)label;
    // ---- per-label count and exact range sum (range * 2^28 as u64, see the header), private bins: the lanes of a
    //      label form a group (match_any), the group's sums come from two reductions over that group, its lowest
    //      lane adds them to the warp's bins -- one pass, however many labels the slice holds
    {
      const bool exact = !(inb && label >= 2) || (r >= 0.03125f && r < 256.0f);
      if (!__all_sync(0xffffffffu, exact)) flag |= 1u;
      const unsigned long long v = inb ? (unsigned long long)((double)r * 268435456.0) : 0ull;
      const int key = inb ? label : 0x7fffffff;                // out-of-image lanes: a group of their own, not counted
      const unsigned grp = __match_any_sync(0xffffffffu, key);
      // v < 2^36: split so that 32 addends cannot overflow 32 bits
      const unsigned slo = __reduce_add_sync(grp, (unsigned)(v & 0xFFFFFu));
      const unsigned shi = __reduce_add_sync(grp, (unsigned)(v >> 20));
      if (inb && (grp & lanemask_lt()) == 0u) {
        cnt[label] += (unsigned)__popc(grp);
        if (label >= 2) sum[label] += ((unsigned long long)shi << 20) + slo;
      }
      __syncwarp();
    }
    // ---- contour bits inside the tile, its first pixel excluded (extract_contour, cpp_modules.cpp:534-545)
    {
      int left = __shfl_up_sync(0xffffffffu, label, 1);
      if (lane == 0) left = carry;
      carry = __shfl_sync(0xffffffffu, label, 31);
      bool rowstart = false;
      if (W >= 32) {
        if (next_row < p0 + 32) { rowstart = (p == next_row); next_row += W; }
      } else {
        rowstart = (p % W) == 0;
      }
      const bool c = inb && p != p_tile && (rowstart || label != left);
      ccnt += __popc(__ballot_sync(0xffffffffu, c));
    }
  }
  // ---- flush the tile: histogram row, frame totals, contour count
  for (int l = lane; l < K; l += 32) {
    const unsigned c = cnt[l];
    bk.tile_hist[((size_t)f * T + tile) * K + l] = (uint16_t)c;
    if (c) {
      atomicAdd(&bk.label_cnt[(size_t)f * K + l], c);
      if (l >= 2) atomicAdd(&bk.label_sum[(size_t)f * K + l], sum[l]);
    }
  }
  if (lane == 0) {
    bk.tile_ccnt[(size_t)f * T + tile] = (uint16_t)ccnt;
    if (flag) atomicOr(&bk.flags[f], flag);
  }
}

// statistics only (caller-supplied labels)
__global__ void __launch_bounds__(kTile, 2)
label_stats_kernel(const float* __restrict__ range, const uint8_t* __restrict__ labels, int HW, int W, int K, int T,
                   Book bk) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* s_sum = reinterpret_cast<unsigned long long*>(smem_raw);
  unsigned* s_cnt = reinterpret_cast<unsigned*>(s_sum + K);
  unsigned* s_flag = s_cnt + K;
  unsigned* s_ccnt = s_flag + 1;
  unsigned* s_last = s_ccnt + 1;
  const int f = blockIdx.y, tile = blockIdx.x, tid = threadIdx.x;
  for (int l = tid; l < K; l += kTile) { s_cnt[l] = 0; s_sum[l] = 0; }
  if (tid == 0) { *s_flag = 0; *s_ccnt = 0; }
  __syncthreads();
  const int p = tile * kTile + tid;
  const bool inb = p < HW;
  int label = 1;
  float r = 0.f;
  if (inb) {
    label = labels[(size_t)f * HW + p];
    r = range[(size_t)f * HW + p];
    // a label without a model row counts as empty, as dequant_reconstruct_kernel decodes it: counted under K-1 it
    // would shift the symbols of label K-1 in every later tile
    if (label >= K) { label = 1; atomicOr(s_flag, 2u); }
  }
  warp_label_stats(label, inb, r, s_cnt, s_sum, s_flag);
  tile_contour_count(label, inb, p, W, s_last, s_ccnt);
  __syncthreads();
  flush_tile_stats(K, f, tile, T, s_cnt, s_sum, s_flag, s_ccnt, bk);
}

}  // namespace rpcc

using namespace rpcc;

static int zero_book(const Book& bk, int B, int K, cudaStream_t st) {
  RPCC_CUDA(cudaMemsetAsync(bk.label_sum, 0, book_zero_bytes(B, K), st));
  RPCC_CUDA(cudaMemsetAsync(bk.flags, 0, sizeof(unsigned) * (size_t)B, st));
  return RPCC_OK;
}

extern "C" size_t rpcc_book_bytes(int B, int H, int W, int K) {
  const int T = (H * W + kTile - 1) / kTile;
  return book_bytes(B, T, K);
}


namespace rpcc {
// hinted: labels[] holds the owner hints of segment_fps_launch for these centres (see the kernel)
int assign_labels_launch(const float* range, const float* lut, const float* ground, const float* centers, int B, int H, int W,
                         int m, uint8_t* labels, void* book, cudaStream_t st, bool hinted) {
  RPCC_REQUIRE(range && lut && ground && centers && labels && book, "null pointer");
  RPCC_REQUIRE(m >= 1 && m + 2 <= RPCC_MAX_LABELS, "cluster_num must be in [1, 254]");
  RPCC_REQUIRE(B <= 65535, "at most 65535 frames per launch");
  if (B == 0) return RPCC_OK;
  const int HW = H * W, K = m + 2, T = (HW + kTile - 1) / kTile;
  const Book bk = make_book(book, B, T, K);
  int rc = zero_book(bk, B, K, st);
  if (rc != RPCC_OK) return rc;
  const int mq = (m + 31) / 32;
  const int MQ = mq <= 1 ? 1 : mq <= 2 ? 2 : mq <= 4 ? 4 : 8;
  const size_t smem = sizeof(float4) * 32 * MQ + (sizeof(unsigned long long) + sizeof(unsigned)) * K * kAsWarps;
  const dim3 grid((T + kAsWarps - 1) / kAsWarps, B);
#define RPCC_ASSIGN_GO(Q) assign_labels_kernel<Q><<<grid, kAsWarps * 32, smem, st>>>(range, lut, ground, centers, HW, W, m, T, labels, bk, hinted)
  if (MQ == 1) RPCC_ASSIGN_GO(1); else if (MQ == 2) RPCC_ASSIGN_GO(2); else if (MQ == 4) RPCC_ASSIGN_GO(4); else RPCC_ASSIGN_GO(8);
#undef RPCC_ASSIGN_GO
  RPCC_LAUNCH_CHECK("assign_labels_kernel");
  return RPCC_OK;
}
}  // namespace rpcc

// arbitrary centres: no hints
extern "C" int rpcc_assign_labels_batch(const float* range, const float* lut, const float* ground, const float* centers,
                                        int B, int H, int W, int m, uint8_t* labels, void* book,
                                        void* stream) {
  return assign_labels_launch(range, lut, ground, centers, B, H, W, m, labels, book, as_stream(stream), false);
}

extern "C" int rpcc_label_stats_batch(const float* range, const uint8_t* labels, int B, int H, int W, int K,
                                      void* book, void* stream) {
  RPCC_REQUIRE(range && labels && book, "null pointer");
  RPCC_REQUIRE(K >= 2 && K <= RPCC_MAX_LABELS, "K must be in [2, 256]");
  RPCC_REQUIRE(B <= 65535, "at most 65535 frames per launch");
  if (B == 0) return RPCC_OK;
  const int HW = H * W, T = (HW + kTile - 1) / kTile;
  cudaStream_t st = as_stream(stream);
  const Book bk = make_book(book, B, T, K);
  int rc = zero_book(bk, B, K, st);
  if (rc != RPCC_OK) return rc;
  const size_t smem = (sizeof(unsigned long long) + sizeof(unsigned)) * K + sizeof(unsigned) * 34;
  label_stats_kernel<<<dim3(T, B), kTile, smem, st>>>(range, labels, HW, W, K, T, bk);
  RPCC_LAUNCH_CHECK("label_stats_kernel");
  return RPCC_OK;
}
