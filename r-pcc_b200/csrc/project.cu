// project.cu -- stage 1: spherical range-image projection, B frames per launch.
//
// Replaces dataset_utils_cpp.point_cloud_to_range_image_even
// (reference ops/cpp_modules/src/cpp_modules.cpp:427-467) and the numpy multiply of
// dataset/transformer.py:94-101.
//
// Design (HBM-bound: 16 B/point in, 4 B/pixel out):
//   one persistent CTA of 1024 threads per SM; a CTA owns a whole frame at a time, so the
//   frame's range image lives in L2 from its sentinel fill, through the z-buffer reductions
//   (RED.MIN.U32 on the order-preserving bit pattern of the non-negative depth), to the
//   in-place finalisation -- DRAM sees the points once and the image once.
//   Points are read as coalesced float4 rows (x,y,z,intensity) with L1 bypass.
// Exactness: pixel indices use a device port of glibc's atan2f (the reference calls libm;
// CUDA's own atan2f differs in the last ulp and flips ~10 pixels per frame).  All float ops
// are unfused (-fmad=false), division and sqrt are IEEE.

#include "async.cuh"

namespace rpcc {

// ---- glibc 2.39 atanf/atan2f float sequence (fdlibm), see oracle/rpcc_oracle.c and SURVEY App. F
__device__ __forceinline__ float dev_atanf(float x) {
  const int hx = __float_as_int(x);
  const int ix = hx & 0x7fffffff;
  int id;
  if (ix >= 0x50800000) {
    if (ix > 0x7f800000) return x + x;
    const float r = __int_as_float(0x3fc90fda) + __int_as_float(0x33a22168);
    return hx > 0 ? r : -r;
  }
  float hi = 0.f, lo = 0.f;
  if (ix < 0x3ee00000) {
    if (ix < 0x31000000) return x;
    id = -1;
  } else {
    x = fabsf(x);
    if (ix < 0x3f980000) {
      if (ix < 0x3f300000) { id = 0; x = (2.0f * x - 1.0f) / (2.0f + x); hi = __int_as_float(0x3eed6338); lo = __int_as_float(0x31ac3769); }
      else                 { id = 1; x = (x - 1.0f) / (x + 1.0f);        hi = __int_as_float(0x3f490fda); lo = __int_as_float(0x33222168); }
    } else {
      if (ix < 0x401c0000) { id = 2; x = (x - 1.5f) / (1.0f + 1.5f * x); hi = __int_as_float(0x3f7b985e); lo = __int_as_float(0x33140fb4); }
      else                 { id = 3; x = -1.0f / x;                       hi = __int_as_float(0x3fc90fda); lo = __int_as_float(0x33a22168); }
    }
  }
  const float z = x * x;
  const float w = z * z;
  const float s1 = z * (__int_as_float(0x3eaaaaab) + w * (__int_as_float(0x3e124925) + w * (__int_as_float(0x3dba2e6e) +
                   w * (__int_as_float(0x3d886b35) + w * (__int_as_float(0x3d4bda59) + w * __int_as_float(0x3c8569d7))))));
  const float s2 = w * (__int_as_float(0xbe4ccccd) + w * (__int_as_float(0xbde38e38) + w * (__int_as_float(0xbd9d8795) +
                   w * (__int_as_float(0xbd6ef16b) + w * __int_as_float(0xbd15a221)))));
  if (id < 0) return x - x * (s1 + s2);
  const float r = hi - ((x * (s1 + s2) - lo) - x);
  return hx < 0 ? -r : r;
}

__device__ __forceinline__ float dev_atan2f(float y, float x) {
  const float tiny = 1.0e-30f;
  const float pi_o_2 = __int_as_float(0x3fc90fdb), pi = __int_as_float(0x40490fdb);
  const float pi_lo = __int_as_float(0xb3bbbd2e);
  const int hx = __float_as_int(x), hy = __float_as_int(y);
  const int ix = hx & 0x7fffffff, iy = hy & 0x7fffffff;
  if (ix > 0x7f800000 || iy > 0x7f800000) return x + y;
  if (hx == 0x3f800000) return dev_atanf(y);
  const int m = ((hy >> 31) & 1) | ((hx >> 30) & 2);
  if (iy == 0) return m < 2 ? y : (m == 2 ? pi + tiny : -pi - tiny);
  if (ix == 0) return hy < 0 ? -pi_o_2 - tiny : pi_o_2 + tiny;
  if (ix == 0x7f800000) {
    const float pi_o_4 = __int_as_float(0x3f490fdb);
    if (iy == 0x7f800000) {
      return m == 0 ? pi_o_4 + tiny : m == 1 ? -pi_o_4 - tiny : m == 2 ? 3.0f * pi_o_4 + tiny : -3.0f * pi_o_4 - tiny;
    }
    return m == 0 ? 0.0f : m == 1 ? -0.0f : m == 2 ? pi + tiny : -pi - tiny;
  }
  if (iy == 0x7f800000) return hy < 0 ? -pi_o_2 - tiny : pi_o_2 + tiny;
  const int k = (iy - ix) >> 23;
  float z;
  if (k > 24) z = pi_o_2 + 0.5f * pi_lo;
  else if (hx < 0 && k < -26) z = 0.0f;
  else z = dev_atanf(fabsf(y / x));
  switch (m) {
    case 0: return z;
    case 1: return -z;
    case 2: return pi - (z - pi_lo);
    default: return (z - pi_lo) - pi;
  }
}

struct Pixel { int pix; float depth; float d2; };

// cpp_modules.cpp:443-458, expression for expression.
__device__ __forceinline__ Pixel point_to_pixel(float x, float y, float z, int H, int W, float hfov, float vmin, float vres) {
  Pixel p;
  p.d2 = x * x + y * y + z * z;
  p.depth = sqrtf(p.d2);
  float ha = dev_atan2f(y, x);
  if (ha < 0) ha = (float)((double)ha + 2 * 3.14159265);
  const float va = dev_atan2f(z, sqrtf(x * x + y * y));
  int col = (int)roundf(ha / hfov * (float)W);
  col = col % W;
  int row = (int)roundf((va - vmin) / vres);
  row = row >= H ? H - 1 : row;
  row = row < 0 ? 0 : row;
  p.pix = row * W + col;
  return p;
}

constexpr unsigned kEmpty = 0xFFFFFFFFu;
constexpr int kPPT = 2;             // independent points per thread and chunk
// ring of point chunks staged in shared memory by bulk async copies: 128 KB per CTA (stage count a power of two)
template <int THREADS> struct ProjStages { static constexpr int value = 8192 / (THREADS * kPPT); };
constexpr int kDeferCap = 2048;     // points per CTA and frame whose pixel is re-derived with the exact libm sequence
template <int THREADS>
constexpr size_t proj_smem() { return sizeof(float4) * (ProjStages<THREADS>::value * THREADS * kPPT + kDeferCap) + 16 * ProjStages<THREADS>::value + 64; }

// mbarrier / bulk-copy primitives: async.cuh (SASS: SYNCS.*, UBLKCP)

// Fast pixel derivation with a proof obligation instead of exactness.  Division-free arctangents
// (odd minimax polynomials: degree 17 on [0,1] for the azimuth, |error| <= 1.0e-7 rad evaluated in f32;
// degree 13 on [0,0.62] for the elevation, <= 6.5e-8 rad), approximate reciprocal / reciprocal square
// root (<= 2 ulp) and fused multiply-adds give continuous column / row coordinates that differ from
// the reference's (glibc atan2f <= 1 ulp, then IEEE divisions) by at most
//   col: ~9e-4 px at W = 2000 (1.4e-6 rad of angle error scaled by W / hfov, plus a few ulp(W) of rounding)
//   row: ~6e-5 rows at vres = 0.00745 rad (3e-7 rad of angle error, plus a few ulp(H))
// `mcol` / `mrow` (host, from the lidar table) are 4x those bounds.  If the fast coordinate is farther
// than the margin from every rounding boundary (k + 0.5), rounding it gives the reference's integer;
// otherwise -- about 1 % of the points -- the caller re-derives the pixel with the exact sequence.
// Zero / tiny / huge coordinates and elevations beyond +-31.8 degrees always take the exact path.
struct ProjParams {
  int H, W;
  float hfov, vmin, vres;        // exact path
  float col_scale, row_scale;    // fast path: W / hfov, 1 / vres
  float mcol, mrow, hm1;         // margins, (float)(H - 1)
};

__device__ __forceinline__ bool fast_point(float x, float y, float z, const ProjParams& P, int& pix, float& d2) {
  const float p2 = x * x + y * y;          // unfused, as the reference: also feeds the exact depth
  d2 = p2 + z * z;                         // depth = sqrtf(d2), cpp_modules.cpp:444; taken once per pixel at the end
  // elevation = atan(z / planar)
  float inv;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(p2));
  const float tv = z * inv, uv = tv * tv;
  float pv = 0.02573351562023163f;
  pv = __fmaf_rn(pv, uv, -0.06798829138278961f);
  pv = __fmaf_rn(pv, uv, 0.10521461814641953f);
  pv = __fmaf_rn(pv, uv, -0.1420031487941742f);
  pv = __fmaf_rn(pv, uv, 0.1999349743127823f);
  pv = __fmaf_rn(pv, uv, -0.3333311378955841f);
  pv = __fmaf_rn(pv, uv, 1.0f);
  const float va = pv * tv;
  // azimuth in [0, 2 pi]
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
  float rmx;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rmx) : "f"(mx));
  const float t = mn * rmx, u = t * t;
  float p = 0.002456609858199954f;
  p = __fmaf_rn(p, u, -0.01440086867660284f);
  p = __fmaf_rn(p, u, 0.03978036344051361f);
  p = __fmaf_rn(p, u, -0.07234777510166168f);
  p = __fmaf_rn(p, u, 0.10498903691768646f);
  p = __fmaf_rn(p, u, -0.14161217212677002f);
  p = __fmaf_rn(p, u, 0.19985905289649963f);
  p = __fmaf_rn(p, u, -0.33332598209381104f);
  p = __fmaf_rn(p, u, 0.9999998807907104f);
  float a = p * t;
  a = ay > ax ? 1.5707963705062866f - a : a;
  a = x < 0.0f ? 3.1415927410125732f - a : a;
  a = y < 0.0f ? 6.2831853071795862f - a : a;
  // column: boundaries of round() are the integers of ct = coordinate + 0.5
  const float ct = __fmaf_rn(a, P.col_scale, 0.5f);
  const bool cbad = fabsf(ct - rintf(ct)) < P.mcol;
  int col = __float2int_rd(ct);            // in [0, W]
  col = col >= P.W ? col - P.W : col;      // cpp_modules.cpp:452 (col % W)
  // row: only the integers 1 .. H-1 of rt separate two rows (beyond them the clamp decides either way)
  const float rt = __fmaf_rn(va - P.vmin, P.row_scale, 0.5f);
  const float rn = rintf(rt);
  const bool rbad = (fabsf(rt - rn) < P.mrow) && (rn >= 1.0f) && (rn <= P.hm1);
  const int row = min(max(__float2int_rd(rt), 0), P.H - 1);
  pix = row * P.W + col;
  // 1e-24 < p2 < 1e24 as one unsigned range check on the bit pattern (also rejects NaN/inf/negative zero sums)
  const bool sane = (__float_as_uint(p2) - 0x17800000u) < (0x67000000u - 0x17800000u);
  return sane && !cbad && !rbad && (fabsf(tv) <= 0.62f);
}

template <int STRIDE>
__device__ __forceinline__ void load_point(const float* __restrict__ pts, int64_t i, float& x, float& y, float& z) {
  if (STRIDE == 4) {
    const float4 v = ld_stream_f4(reinterpret_cast<const float4*>(pts) + i);
    x = v.x; y = v.y; z = v.z;
  } else {
    x = ld_stream_f(pts + i * 3); y = ld_stream_f(pts + i * 3 + 1); z = ld_stream_f(pts + i * 3 + 2);
  }
}

__device__ __forceinline__ void team_barrier() {
  // all threads of all CTAs of the cluster; release/acquire at cluster scope covers global memory
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned team_rank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }

// scratch: int32[B][4] = {lastZero+1 (slot col==0), pix, lastZero+1 (slot col!=0), pix}, zeroed by the caller.
//
// A cluster of kTeam CTAs (one per SM) owns a frame at a time: few frames are in flight (74 x 512 KB),
// so a frame's range image lives in L2 from its sentinel fill, through the z-buffer reductions
// (RED.MIN.U32 on the bit pattern of the non-negative depth), to the in-place finalisation, and DRAM
// sees the points once and the image once.  Chunk c of a frame (1024 points) belongs to CTA c mod kTeam.
// STRIDE 4 (KITTI .bin rows): every CTA streams its chunks through a ring of kStages shared-memory
// buffers filled by cp.async.bulk (one elected thread issues, an mbarrier per stage counts the bytes, a
// second mbarrier per stage collects one "consumed" arrival per warp).  The ring runs ahead across
// frame boundaries, so 100+ KB per SM are in flight regardless of what the warps are doing -- including
// the sentinel fill and the finalisation -- which is what hides the HBM latency.
// STRIDE 3 (the numpy-facing op): frames need not start 16-byte aligned, points are loaded directly.
template <int STRIDE, int kTeam, int kProjThreads>
__global__ void __launch_bounds__(kProjThreads, 1)
project_kernel(const float* __restrict__ points, const int64_t* __restrict__ offsets, int B, ProjParams P,
               unsigned* __restrict__ range, int* __restrict__ scratch) {
  constexpr int kChunk = kProjThreads * kPPT;   // points per stage
  constexpr int kStages = ProjStages<kProjThreads>::value;
  const int H = P.H, W = P.W, HW = H * W;
  const int tid = threadIdx.x, lane = tid & 31;
  const int rank = (int)team_rank();
  const int team = blockIdx.x / kTeam, nteams = gridDim.x / kTeam;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float4* s_pts = reinterpret_cast<float4*>(smem_raw);                    // [kStages][kChunk]
  float4* s_defer = s_pts + kStages * kChunk;                             // [kDeferCap] x, y, z, bits(index in frame)
  const unsigned a_full = smem_addr(s_defer + kDeferCap);                 // kStages mbarriers
  const unsigned a_empty = a_full + 8 * kStages;                          // kStages mbarriers
  __shared__ int s_zero[4];
  __shared__ unsigned s_fix[2];
  __shared__ int s_ndefer;

  // ---- producer state (thread 0 only): next chunk to request
  int pf = team;                // frame
  int64_t pbase = 0;            // first point of that frame
  int pn = 0, pc = rank;        // points in that frame, next chunk of this CTA inside it
  unsigned pg = 0;              // chunks requested so far (ring position)
  unsigned cg = 0;              // chunks consumed so far (all threads)
  auto producer_seek = [&]() {  // position on the next frame in which this CTA has a chunk
    while (pf < B) {
      pbase = offsets[pf];
      pn = (int)(offsets[pf + 1] - pbase);
      if (pn > rank * kChunk) break;
      pf += nteams;
    }
    pc = rank;
  };
  auto produce = [&]() {        // request one chunk (no-op when this CTA's frames are exhausted)
    if (pf >= B) return;
    const unsigned st = pg % kStages;
    mbar_wait(a_empty + 8 * st, ((pg / kStages) & 1u) ^ 1u);   // every warp has taken chunk pg - kStages
    const int first = pc * kChunk;
    const int cnt = min(kChunk, pn - first);
    mbar_arrive_expect_tx(a_full + 8 * st, (unsigned)cnt * 16u);
    bulk_load(smem_addr(s_pts + st * kChunk), reinterpret_cast<const float4*>(points) + pbase + first, (unsigned)cnt * 16u,
              a_full + 8 * st);
    ++pg;
    pc += kTeam;
    if (pc * kChunk >= pn) { pf += nteams; producer_seek(); }
  };
  if (STRIDE == 4) {
    if (tid == 0) {
      for (int s = 0; s < kStages; ++s) { mbar_init(a_full + 8 * s, 1); mbar_init(a_empty + 8 * s, kProjThreads / 32); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
      producer_seek();
      for (int s = 0; s < kStages - 1; ++s) produce();
    }
  }

  const unsigned a_pts = smem_addr(s_pts) + (unsigned)tid * 16u;

  // ---- image passes.  A frame's image is (1) filled with the sentinel, (2) reduced into, (3) finalised in
  // place (sentinel -> 0.0f, squared depth -> depth with the IEEE sqrt of cpp_modules.cpp:444), all
  // through L2.  Passes (1) of the NEXT frame and (3) of the PREVIOUS frame are sliced into the
  // streaming loop of the current one (one 16-byte step per thread and chunk), so the only
  // synchronisation is one team barrier per frame.  Step k of a pass touches uint4 number
  // (k * kTeam + rank) * kProjThreads + tid of the image.
  const bool vec = (HW & 3) == 0;            // every frame's image is 16-byte aligned
  const int n4 = vec ? (HW >> 2) : 0;
  const int ksteps = (n4 + kTeam * kProjThreads - 1) / (kTeam * kProjThreads);
  auto fin = [](unsigned b) { return b == kEmpty ? 0u : __float_as_uint(sqrtf(__uint_as_float(b))); };
  auto fill_step = [&](unsigned* im, int k) {
    const int i = (k * kTeam + rank) * kProjThreads + tid;
    if (i < n4) reinterpret_cast<uint4*>(im)[i] = make_uint4(kEmpty, kEmpty, kEmpty, kEmpty);
  };
  auto fin_load = [&](unsigned* im, int k, uint4& w) {
    const int i = (k * kTeam + rank) * kProjThreads + tid;
    if (i < n4) w = __ldcg(reinterpret_cast<uint4*>(im) + i);
  };
  auto fin_store = [&](unsigned* im, int k, uint4 w) {
    const int i = (k * kTeam + rank) * kProjThreads + tid;
    if (i < n4) {
      // a finished image is dead weight in L2 until the next kernel: evict-first, so that LRU does not
      // push out the live images (sentinel-filled long ago, not yet touched again) instead
      w.x = fin(w.x); w.y = fin(w.y); w.z = fin(w.z); w.w = fin(w.w);
      asm volatile("st.global.L2::cache_hint.v4.u32 [%0], {%1,%2,%3,%4}, %5;"
                   ::"l"(reinterpret_cast<uint4*>(im) + i), "r"(w.x), "r"(w.y), "r"(w.z), "r"(w.w), "l"(0x12F0000000000000ull) : "memory");
    }
  };
  auto fill_rest = [&](unsigned* im, int k) {     // steps k.. of the fill, and the scalar path
    for (; k < ksteps; ++k) fill_step(im, k);
    if (!vec) for (int i = rank * kProjThreads + tid; i < HW; i += kTeam * kProjThreads) im[i] = kEmpty;
  };
  auto fin_rest = [&](unsigned* im, int k) {
    for (; k < ksteps; ++k) { uint4 w = make_uint4(0, 0, 0, 0); fin_load(im, k, w); fin_store(im, k, w); }
    if (!vec) for (int i = rank * kProjThreads + tid; i < HW; i += kTeam * kProjThreads) im[i] = fin(__ldcg(im + i));
  };

  if (team < B) fill_rest(range + (size_t)team * HW, 0);
  if (tid == 0) s_ndefer = 0;
  team_barrier();
  unsigned* prev = nullptr;                  // image waiting for its finalisation
  for (int f = team; f < B; f += nteams) {
    unsigned* img = range + (size_t)f * HW;
    unsigned* next = (f + nteams < B) ? range + (size_t)(f + nteams) * HW : nullptr;
    int kf = next ? 0 : ksteps, kz = prev ? 0 : ksteps;
    // z-buffer on the SQUARED depth (sqrt is monotone: the square root of the minimum is the minimum of
    // the square roots, bit for bit)
    const int64_t p0 = offsets[f], p1 = offsets[f + 1];
    int* zs = scratch + (size_t)f * 4;
    // exact derivation + z-buffer update of one point (also the zero-depth bookkeeping)
    auto exact_update = [&](float x, float y, float z, int rel) {
      const Pixel p = point_to_pixel(x, y, z, H, W, P.hfov, P.vmin, P.vres);
      if (p.depth == 0.0f) {
        // zero depth re-opens the pixel in the reference's sequential loop (cpp_modules.cpp:459)
        const int slot = (p.pix % W == 0) ? 0 : 2;
        atomicMax(&zs[slot], rel + 1);
        zs[slot + 1] = p.pix;
      } else {
        atomicMin(&img[p.pix], __float_as_uint(p.d2));
      }
    };
    const int npts = (int)(p1 - p0);
    // the next image is filled during the LAST ksteps iterations (it should not sit in L2 for a whole frame)
    int wait_fill = (npts - rank * kChunk + kTeam * kChunk - 1) / (kTeam * kChunk) - ksteps;
    for (int i0 = rank * kChunk; i0 < npts; i0 += kTeam * kChunk) {
      float4 v[kPPT];
      uint4 w = make_uint4(0, 0, 0, 0);
      if (kz < ksteps) fin_load(prev, kz, w);           // consumed at the end of the iteration
      if (STRIDE == 4) {
        const unsigned st = cg & (kStages - 1);
        if (tid == 0) produce();                  // keep kStages - 1 chunks ahead of the consumers
        mbar_wait(a_full + 8 * st, (cg / kStages) & 1u);
#pragma unroll
        for (int u = 0; u < kPPT; ++u) v[u] = lds_f4(a_pts + (st * kChunk + u * kProjThreads) * 16u);
        __syncwarp();
        if (lane == 0) mbar_arrive(a_empty + 8 * st);   // this warp's slice is in registers
        ++cg;
      }
      if (--wait_fill < 0 && kf < ksteps) { fill_step(next, kf); ++kf; }
      bool bad[kPPT];
#pragma unroll
      for (int u = 0; u < kPPT; ++u) {
        const int i = i0 + u * kProjThreads + tid;
        const bool have = i < npts;
        float x = 1.f, y = 0.f, z = 0.f;
        if (STRIDE == 4) { if (have) { x = v[u].x; y = v[u].y; z = v[u].z; } }
        else if (have) load_point<STRIDE>(points, p0 + i, x, y, z);
        v[u].x = x; v[u].y = y; v[u].z = z;
        int pix;
        float d2;
        const bool ok = fast_point(x, y, z, P, pix, d2);
        if (have && ok) atomicMin(&img[pix], __float_as_uint(d2));
        bad[u] = have && !ok;
      }
      // the rest (~1 %) is parked in shared memory and redone densely below
      bool any_bad = false;
#pragma unroll
      for (int u = 0; u < kPPT; ++u) any_bad = any_bad || bad[u];
      if (__any_sync(0xffffffffu, any_bad)) {
#pragma unroll
        for (int u = 0; u < kPPT; ++u) {
          if (bad[u]) {
            const int i = i0 + u * kProjThreads + tid;
            const int slot = atomicAdd(&s_ndefer, 1);
            if (slot < kDeferCap) s_defer[slot] = make_float4(v[u].x, v[u].y, v[u].z, __int_as_float(i));
            else exact_update(v[u].x, v[u].y, v[u].z, i);          // list full: do it in place
          }
        }
      }
      if (kz < ksteps) { fin_store(prev, kz, w); ++kz; }
    }
    __syncthreads();
    {
      const int nd = min(s_ndefer, kDeferCap);
      for (int e = tid; e < nd; e += kProjThreads) {
        const float4 q = s_defer[e];
        exact_update(q.x, q.y, q.z, __float_as_int(q.w));
      }
    }
    if (next) fill_rest(next, kf);
    if (prev) fin_rest(prev, kz);
    team_barrier();   // every reduction of frame f has been performed; the next image is filled
    if (tid < 4) s_zero[tid] = __ldcg(zs + tid);
    if (tid < 2) s_fix[tid] = kEmpty;
    if (tid == 0) s_ndefer = 0;
    __syncthreads();
    if (s_zero[0] > 0 || s_zero[2] > 0) {   // same decision in every CTA of the team
      // rare: only points after the last zero-depth hit of a pixel count for that pixel
      if (rank == 0) {
        for (int64_t i = p0 + tid; i < p1; i += kProjThreads) {
          float x, y, z;
          load_point<STRIDE>(points, i, x, y, z);
          const Pixel p = point_to_pixel(x, y, z, H, W, P.hfov, P.vmin, P.vres);
          if (p.depth == 0.0f) continue;
          const int rel = (int)(i - p0);
          if (s_zero[0] > 0 && p.pix == s_zero[1] && rel >= s_zero[0]) atomicMin(&s_fix[0], __float_as_uint(p.d2));
          if (s_zero[2] > 0 && p.pix == s_zero[3] && rel >= s_zero[2]) atomicMin(&s_fix[1], __float_as_uint(p.d2));
        }
        __syncthreads();
        if (tid == 0) {
          if (s_zero[0] > 0) img[s_zero[1]] = s_fix[0];
          if (s_zero[2] > 0) img[s_zero[3]] = s_fix[1];
        }
      }
      team_barrier();
    }
    prev = img;
    __syncthreads();   // s_zero is rewritten after the next frame
  }
  if (prev) fin_rest(prev, 0);
}

// Intensity owner of every pixel (DESIGN.md §4, "Intensity"): the point the reference's sequential z-buffer loop stored
// last.  A point is a candidate when sqrtf(d2) has the finalised range's bits and it comes after the pixel's last
// zero-depth point (the projection's `scratch`); the owner is the candidate with the smallest in-frame index, i.e. the
// first to reach the final depth after the pixel was last re-opened.  The pixel comes from the projection's own
// derivation (fast_point, the exact sequence where it declines), so it is the pixel the point was reduced into.
// owner [B][HW] u32 must hold 0xFFFFFFFF on entry.  grid (x, B): the CTAs of column x stride over the frame's points.
__global__ void __launch_bounds__(256)
intensity_owner_kernel(const float4* __restrict__ points, const int64_t* __restrict__ offsets, ProjParams P,
                       const unsigned* __restrict__ range, const int* __restrict__ scratch, unsigned* __restrict__ owner) {
  const int f = blockIdx.y, HW = P.H * P.W;
  const int64_t p0 = offsets[f];
  const int n = (int)(offsets[f + 1] - p0);
  const int* zs = scratch + (size_t)f * 4;
  const int z0 = zs[0], z0pix = zs[1], z2 = zs[2], z2pix = zs[3];
  const unsigned* img = range + (size_t)f * HW;
  unsigned* own = owner + (size_t)f * HW;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 v = ld_stream_f4(points + p0 + i);
    int pix;
    float d2;
    if (!fast_point(v.x, v.y, v.z, P, pix, d2)) {
      const Pixel q = point_to_pixel(v.x, v.y, v.z, P.H, P.W, P.hfov, P.vmin, P.vres);
      pix = q.pix;
      d2 = q.d2;
    }
    const unsigned dbits = __float_as_uint(sqrtf(d2));
    if (dbits == 0u || dbits != __ldg(img + pix)) continue;       // zero depth, or not the pixel's final depth
    if ((z0 > 0 && pix == z0pix && i < z0) || (z2 > 0 && pix == z2pix && i < z2)) continue;   // before a re-opening
    atomicMin(own + pix, (unsigned)i);
  }
}

// intensity [B][HW] = the owner's fourth column, 0 where the pixel has no owner
__global__ void intensity_gather_kernel(const float4* __restrict__ points, const int64_t* __restrict__ offsets, int HW,
                                        const unsigned* __restrict__ owner, float* __restrict__ intensity) {
  const int f = blockIdx.y;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const unsigned o = owner[(size_t)f * HW + p];
  intensity[(size_t)f * HW + p] = o == kEmpty ? 0.f : __ldg(&points[offsets[f] + o].w);
}

__global__ void range_to_xyz_kernel(const float* __restrict__ range, const float* __restrict__ lut, int64_t total,
                                    int HW, float* __restrict__ xyz) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float r = range[i];
  const int p = (int)(i % HW);
  xyz[i * 3 + 0] = r * lut[p * 3 + 0];
  xyz[i * 3 + 1] = r * lut[p * 3 + 1];
  xyz[i * 3 + 2] = r * lut[p * 3 + 2];
}

}  // namespace rpcc

using namespace rpcc;

// the pixel derivation's parameters, shared by the projection and the intensity owner pass
static ProjParams proj_params(int H, int W, float hfov, float vmax, float vmin) {
  // margins of fast_point(): 4x the worst-case distance between the fast and the reference
  // coordinate.  col: 3 ulp of an angle in [4,8) (4.77e-7 each) scaled to columns + 4 ulp of W;
  // row: 3 ulp of an angle in [1,2) (1.19e-7 each) scaled to rows + 4 ulp of H.
  ProjParams P;
  P.H = H; P.W = W; P.hfov = hfov; P.vmin = vmin;
  P.vres = (vmax - vmin) / (float)(H - 1);
  P.col_scale = (float)W / hfov; P.row_scale = 1.0f / P.vres; P.hm1 = (float)(H - 1);
  const float ulp_w = ldexpf(1.0f, ilogbf((float)(W > 1 ? W : 2)) - 23), ulp_h = ldexpf(1.0f, ilogbf((float)H) - 23);
  P.mcol = 4.0f * (3.0f * 4.77e-7f * (float)W / fabsf(hfov) + 4.0f * ulp_w);
  P.mrow = 4.0f * (3.0f * 1.2e-7f / fabsf(P.vres) + 4.0f * ulp_h);
  // margins this large (or a table the fast path was not derived for) send every point down the exact path
  if (!(P.mcol < 0.25f) || !(hfov > 6.28f && hfov < 6.29f)) P.mcol = 1.0f;
  if (!(P.mrow < 0.25f) || !(P.vres > 0.0f)) P.mrow = 1.0f;
  return P;
}

template <int STRIDE, int TEAM, int THREADS>
static int launch_project(const float* points, const int64_t* offsets, int B, const ProjParams& P, unsigned* img,
                          int* scratch, cudaStream_t st) {
  auto kern = project_kernel<STRIDE, TEAM, THREADS>;
  RPCC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)proj_smem<THREADS>()));
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = TEAM; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = proj_smem<THREADS>();
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cfg.gridDim = dim3(TEAM);
  int nteams = 0;
  if (cudaOccupancyMaxActiveClusters(&nteams, kern, &cfg) != cudaSuccess || nteams <= 0) {
    cudaGetLastError();
    nteams = sm_count() / TEAM;
  }
  if (nteams > B) nteams = B;
  cfg.gridDim = dim3(TEAM * nteams);
  RPCC_CUDA(cudaLaunchKernelEx(&cfg, kern, points, offsets, B, P, img, scratch));
  return RPCC_OK;
}

extern "C" int rpcc_project_batch(const float* points, int stride, const int64_t* offsets, int B, int H, int W,
                                  float hfov, float vmax, float vmin, float* range, int32_t* scratch, void* stream) {
  RPCC_REQUIRE(points && offsets && range && scratch, "null pointer");
  RPCC_REQUIRE(stride == 3 || stride == 4, "stride must be 3 or 4");
  RPCC_REQUIRE(B >= 0 && H >= 2 && W >= 1, "bad shape");
  RPCC_REQUIRE(stride != 4 || (reinterpret_cast<uintptr_t>(points) & 15) == 0, "stride-4 points must be 16-byte aligned");
  if (B == 0) return RPCC_OK;
  cudaStream_t st = as_stream(stream);
  RPCC_CUDA(cudaMemsetAsync(scratch, 0, sizeof(int32_t) * 4 * (size_t)B, st));
  const ProjParams P = proj_params(H, W, hfov, vmax, vmin);
  // template arguments: point stride, CTAs per frame (cluster size), threads per CTA
  unsigned* img = reinterpret_cast<unsigned*>(range);
  const int rc = stride == 3 ? launch_project<3, 2, 512>(points, offsets, B, P, img, scratch, st)
                             : launch_project<4, 2, 1024>(points, offsets, B, P, img, scratch, st);
  if (rc != RPCC_OK) return rc;
  RPCC_LAUNCH_CHECK("project_kernel");
  return RPCC_OK;
}

extern "C" int rpcc_intensity_owner_batch(const float* points, const int64_t* offsets, int B, int H, int W, float hfov,
                                          float vmax, float vmin, const float* range, const int32_t* scratch,
                                          uint32_t* owner, float* intensity, void* stream) {
  RPCC_REQUIRE(points && offsets && range && scratch && owner && intensity, "null pointer");
  RPCC_REQUIRE(B >= 0 && B <= 65535 && H >= 2 && W >= 1, "bad shape");
  RPCC_REQUIRE((reinterpret_cast<uintptr_t>(points) & 15) == 0, "points must be 16-byte aligned rows of 4 floats");
  if (B == 0) return RPCC_OK;
  cudaStream_t st = as_stream(stream);
  const int HW = H * W;
  RPCC_CUDA(cudaMemsetAsync(owner, 0xFF, sizeof(uint32_t) * (size_t)B * HW, st));
  // 32 CTAs per frame: ~15 points per thread for a 64E frame, thousands of CTAs for a batch
  intensity_owner_kernel<<<dim3(32, B), 256, 0, st>>>(reinterpret_cast<const float4*>(points), offsets,
                                                       proj_params(H, W, hfov, vmax, vmin),
                                                       reinterpret_cast<const unsigned*>(range), scratch, owner);
  RPCC_LAUNCH_CHECK("intensity_owner_kernel");
  intensity_gather_kernel<<<dim3((HW + 255) / 256, B), 256, 0, st>>>(reinterpret_cast<const float4*>(points), offsets, HW,
                                                                      owner, intensity);
  RPCC_LAUNCH_CHECK("intensity_gather_kernel");
  return RPCC_OK;
}

extern "C" int rpcc_range_to_xyz_batch(const float* range, const float* lut, int B, int HW, float* xyz, void* stream) {
  RPCC_REQUIRE(range && lut && xyz, "null pointer");
  const int64_t total = (int64_t)B * HW;
  if (total == 0) return RPCC_OK;
  range_to_xyz_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(range, lut, total, HW, xyz);
  RPCC_LAUNCH_CHECK("range_to_xyz_kernel");
  return RPCC_OK;
}
