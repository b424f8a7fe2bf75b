// dbscan.cu -- DBSCAN segmentation of range images, B frames per launch, stream-ordered, no host synchronisation.
// The definition is this project's own (DESIGN.md §4, "DBSCAN (this project's definition)"; oracle/dbscan.py):
//
//   points   non-empty pixels the FPS path masks as non-ground (fps.cu masked_point: |sum(pc*g)+g3| / |g| > thr)
//   q ~ p    cham_d(p, q) <= e2, e2 = (float)(eps * eps) computed in double; p ~ p
//   core     a point with at least min_points neighbours; clusters = connected components of the cores
//   border   a non-core point with a core neighbour: joins the cluster of its nearest core (cham_d, then pixel index)
//   labels   0 ground, 1 empty, 2 .. cluster_num the cluster_num - 1 largest clusters (cores + borders; on equal size
//            the smaller first core pixel first), numbered in order of their first core pixel; cluster_num + 1 noise
//            and every other cluster
//
// Neighbourhoods are found in range-image space (window.cuh): a pixel whose ray is at angle t from the query's ray is
// at least r_q sin t away, so all neighbours lie in the rows and columns whose angle stays below asin(eps / r_q).  The
// window is sized per query from that angle; where eps is not below r_q, or the frame holds a negative range (a point
// behind the sensor, where the bound does not hold), the query scans the whole image and is counted.
//
// Kernels: points (mask) -> count (core flags; stops at min_points) -> link (union-find over core-core edges, the
// larger root hooked under the smaller, so that a component's root is its smallest core pixel whatever the thread
// order; nearest core of the other points) -> resolve (roots, cluster sizes, a list of roots per frame) -> select (one
// CTA per frame: radix select of the kept clusters and their labels) -> labels.
#include <math.h>

#include "window.cuh"

namespace rpcc {

constexpr int kDbThreads = 256;
constexpr int kDbSelThreads = 1024;

// state bits per pixel: bit 0 = a point, bit 1 = a core point (the count kernel sets bit 1 of its own pixel only, so
// bit 0 -- what its neighbours read -- never changes while they read it)
constexpr uint8_t kPoint = 1, kCore = 3;

struct DbGeom { float dalt, daz, cmin; };

struct DbWs {
  unsigned* fallback;   // [B] points whose neighbourhood needed a whole-image scan
  unsigned* nroots;     // [B] clusters found
  unsigned* neg;        // [B] the frame holds a negative range
  uint8_t* state;       // [B][HW]
  int* parent;          // [B][HW] union-find parent (cores), nearest core (other points) or -1
  int* size;            // [B][HW] cluster size at the root pixel, then the root's label
  int* roots;           // [B][HW] roots of the frame, first nroots[f] valid
};

inline size_t db_align(size_t x) { return (x + 255) & ~(size_t)255; }

inline DbWs db_carve(void* ws, int B, size_t HW) {
  unsigned char* p = static_cast<unsigned char*>(ws);
  const size_t n = (size_t)B * HW;
  DbWs w;
  w.fallback = reinterpret_cast<unsigned*>(p);
  w.nroots = w.fallback + B;
  w.neg = w.nroots + B;
  p += db_align(3 * sizeof(unsigned) * (size_t)B);
  w.state = p;                                p += db_align(n);
  w.parent = reinterpret_cast<int*>(p);       p += db_align(sizeof(int) * n);
  w.size = reinterpret_cast<int*>(p);         p += db_align(sizeof(int) * n);
  w.roots = reinterpret_cast<int*>(p);
  return w;
}

// Half-sizes (rows kr, columns kc) of the window that holds every point within eps of a query at range rq, or false
// when eps is not below rq (with window.cuh's relative margin of 2e-3 on the squared distance): then a neighbour can
// lie in any direction.  The angle gets a relative margin of 1e-3 for the f32 asin / sin / division here, and an
// absolute one of 1e-6 rad (window.cuh's kEvTau) for the f32 points: their rounding moves the difference of two points
// by up to 3.1e-7 r, an angular error that no relative margin covers at fine pitches (see window.cuh).  Rows k apart
// are at least k * dalt apart; columns k apart satisfy sin(t/2) >= cmin sin(k daz / 2).
__device__ __forceinline__ bool db_window(float rq, float e2, const DbGeom& g, int H, int W, int& kr, int& kc) {
  const float r2 = rq * rq * (1.0f - 2e-3f);
  if (!(e2 < r2)) return false;
  const float t = asinf(sqrtf(e2 / r2)) * 1.001f + 1e-6f;
  kr = min(H - 1, (int)(t / g.dalt));
  const float sh = sinf(0.5f * t) / g.cmin;
  kc = sh >= 1.0f ? W : min(W, (int)(2.0f * asinf(sh) / g.daz));
  return true;
}

// probe(q) for every pixel q of the window (rows outward from the query's, columns outward inside a row: the nearest
// pixels come first, which is what lets the count stop early), or of the whole image in raster order when `all`.
// probe returns true to stop the walk.
template <class Probe>
__device__ __forceinline__ void db_walk(int H, int W, int h, int w, bool all, int kr, int kc, Probe&& probe) {
  if (all) {
    for (int q = 0; q < H * W; ++q) if (probe(q)) return;
    return;
  }
  const bool wrap_all = 2 * kc + 1 >= W;
  for (int d = 0; d <= kr; ++d) {
    for (int s = d ? -1 : 1; s <= 1; s += 2) {
      const int hh = h + s * d;
      if (hh < 0 || hh >= H) continue;
      const int row = hh * W;
      if (wrap_all) {
        for (int ww = 0; ww < W; ++ww) if (probe(row + ww)) return;
        continue;
      }
      if (probe(row + w)) return;
      for (int k = 1; k <= kc; ++k) {
        int a = w + k; a -= a >= W ? W : 0;
        int b = w - k; b += b < 0 ? W : 0;
        if (probe(row + a) || probe(row + b)) return;
      }
    }
  }
}

__device__ __forceinline__ void db_point(const float* __restrict__ rg, const float* __restrict__ lut, int q, float& x,
                                         float& y, float& z) {
  const float r = rg[q];
  x = r * __ldg(lut + 3 * q); y = r * __ldg(lut + 3 * q + 1); z = r * __ldg(lut + 3 * q + 2);
}

// ECL-CC style union-find on frame-local pixel indices: parent[x] <= x always, so a root is its tree's smallest pixel;
// find halves paths (benign races: every store writes an ancestor), unite hooks the larger root under the smaller
// with a CAS that only a root can pass.
__device__ __forceinline__ int uf_find(volatile int* par, int x) {
  int cur = par[x];
  if (cur != x) {
    int prev = x, nxt;
    while (cur > (nxt = par[cur])) { par[prev] = nxt; prev = cur; cur = nxt; }
  }
  return cur;
}

__device__ __forceinline__ void uf_unite(volatile int* par, int a, int b) {
  int ra = uf_find(par, a), rb = uf_find(par, b);
  while (ra != rb) {
    if (ra < rb) {
      const int old = atomicCAS((int*)&par[rb], rb, ra);
      if (old == rb) return;
      rb = old;
    } else {
      const int old = atomicCAS((int*)&par[ra], ra, rb);
      if (old == ra) return;
      ra = old;
    }
  }
}

__global__ void __launch_bounds__(kDbThreads)
dbscan_points_kernel(const float* __restrict__ range, const float* __restrict__ lut, const float* __restrict__ ground,
                     int HW, float thr, DbWs ws) {
  const int f = blockIdx.y, p = blockIdx.x * kDbThreads + threadIdx.x;
  if (p >= HW) return;
  const size_t o = (size_t)f * HW + p;
  const float g0 = ground[f * 4], g1 = ground[f * 4 + 1], g2 = ground[f * 4 + 2], g3 = ground[f * 4 + 3];
  const float gnorm = sqrtf(torch_sum3(g0 * g0, g1 * g1, g2 * g2));
  const float r = range[o];
  bool pt = false;
  if (r != 0.f) {
    const float x = r * __ldg(lut + 3 * p), y = r * __ldg(lut + 3 * p + 1), z = r * __ldg(lut + 3 * p + 2);
    const float s = torch_sum3(x * g0, y * g1, z * g2);
    pt = fabsf(s + g3) / gnorm > thr;
  }
  ws.state[o] = pt ? kPoint : 0;
  ws.parent[o] = -1;
  ws.size[o] = 0;
}

__global__ void __launch_bounds__(kDbThreads)
dbscan_count_kernel(const float* __restrict__ range, const float* __restrict__ lut, int H, int W, DbGeom g, float e2,
                    unsigned min_points, DbWs ws) {
  const int f = blockIdx.y, HW = H * W, p = blockIdx.x * kDbThreads + threadIdx.x;
  if (p >= HW) return;
  const size_t base = (size_t)f * HW;
  const uint8_t* st = ws.state + base;
  if (!(st[p] & kPoint)) return;
  const float* rg = range + base;
  float px, py, pz;
  db_point(rg, lut, p, px, py, pz);
  unsigned n = 0;
  auto probe = [&](int q) -> bool {
    if (st[q] & kPoint) {
      float x, y, z;
      db_point(rg, lut, q, x, y, z);
      if (cham_d(px, py, pz, x, y, z) <= e2) ++n;
    }
    return n >= min_points;
  };
  int kr = 0, kc = 0;
  const bool all = ws.neg[f] != 0u || !db_window(rg[p], e2, g, H, W, kr, kc);
  if (all) atomicAdd(ws.fallback + f, 1u);
  db_walk(H, W, p / W, p % W, all, kr, kc, probe);
  if (n >= min_points) {
    ws.state[base + p] = kCore;
    ws.parent[base + p] = p;
  }
}

__global__ void __launch_bounds__(kDbThreads)
dbscan_link_kernel(const float* __restrict__ range, const float* __restrict__ lut, int H, int W, DbGeom g, float e2,
                   DbWs ws) {
  const int f = blockIdx.y, HW = H * W, p = blockIdx.x * kDbThreads + threadIdx.x;
  if (p >= HW) return;
  const size_t base = (size_t)f * HW;
  const uint8_t* st = ws.state + base;
  const uint8_t sp = st[p];
  if (!(sp & kPoint)) return;
  const float* rg = range + base;
  volatile int* par = ws.parent + base;
  float px, py, pz;
  db_point(rg, lut, p, px, py, pz);
  int kr = 0, kc = 0;
  const bool all = ws.neg[f] != 0u || !db_window(rg[p], e2, g, H, W, kr, kc);
  if (sp == kCore) {
    // every core-core edge once, from its smaller end; an edge to a point whose parent is p's last known root (an
    // ancestor of p, so the same set) changes nothing
    int rp = uf_find(par, p);
    db_walk(H, W, p / W, p % W, all, kr, kc, [&](int q) -> bool {
      if (q > p && st[q] == kCore && par[q] != rp) {
        float x, y, z;
        db_point(rg, lut, q, x, y, z);
        if (cham_d(px, py, pz, x, y, z) <= e2) { uf_unite(par, p, q); rp = uf_find(par, p); }
      }
      return false;
    });
  } else {
    float best = __int_as_float(0x7f800000);
    int bi = -1;
    db_walk(H, W, p / W, p % W, all, kr, kc, [&](int q) -> bool {
      if (st[q] == kCore) {
        float x, y, z;
        db_point(rg, lut, q, x, y, z);
        const float d = cham_d(px, py, pz, x, y, z);
        if (d <= e2 && (d < best || (d == best && q < bi))) { best = d; bi = q; }
      }
      return false;
    });
    ws.parent[base + p] = bi;    // a non-core entry: no find ever walks through it
  }
}

__global__ void __launch_bounds__(kDbThreads)
dbscan_resolve_kernel(int HW, DbWs ws) {
  const int f = blockIdx.y, p = blockIdx.x * kDbThreads + threadIdx.x;
  if (p >= HW) return;
  const size_t base = (size_t)f * HW;
  const uint8_t sp = ws.state[base + p];
  if (!(sp & kPoint)) return;
  volatile int* par = ws.parent + base;
  // parent is left as it is: a store of the root here could be overwritten by another thread's path halving (with an
  // ancestor that is not the root); the label kernel walks to the root instead
  int root;
  if (sp == kCore) {
    root = uf_find(par, p);
    if (root == p) ws.roots[base + atomicAdd(ws.nroots + f, 1u)] = p;
  } else {
    const int c = par[p];
    if (c < 0) return;                                   // noise
    root = uf_find(par, c);
  }
  atomicAdd(ws.size + base + root, 1);
}

__device__ __forceinline__ unsigned long long db_key(const int* size, int root) {
  // larger clusters first; on equal size the smaller first core pixel
  return ((unsigned long long)(unsigned)size[root] << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)root);
}

// One CTA per frame: the keep = min(cluster_num - 1, clusters) largest keys by an 8-bit radix select (keys are
// distinct, so exactly `keep` reach the threshold), then size[root] := the root's label.
__global__ void __launch_bounds__(kDbSelThreads)
dbscan_select_kernel(int HW, int m, DbWs ws) {
  __shared__ unsigned hist[256];
  __shared__ unsigned long long s_prefix;
  __shared__ unsigned s_need;
  __shared__ int s_kept[RPCC_MAX_LABELS];
  __shared__ unsigned s_nk;
  const int f = blockIdx.x, tid = threadIdx.x;
  const size_t base = (size_t)f * HW;
  const int* roots = ws.roots + base;
  int* size = ws.size + base;
  const unsigned n = ws.nroots[f];
  const unsigned keep = min(n, (unsigned)(m - 1));
  unsigned long long thr = 0ull;
  if (keep < n) {
    unsigned long long prefix = 0ull, mask = 0ull;
    unsigned need = keep;
    for (int shift = 56; shift >= 0 && need > 0; shift -= 8) {
      for (int i = tid; i < 256; i += kDbSelThreads) hist[i] = 0u;
      __syncthreads();
      for (unsigned i = tid; i < n; i += kDbSelThreads) {
        const unsigned long long k = db_key(size, roots[i]);
        if ((k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 255u], 1u);
      }
      __syncthreads();
      if (tid == 0) {
        unsigned cum = 0;
        for (int d = 255; d >= 0; --d) {
          if (cum + hist[d] >= need) { s_prefix = prefix | ((unsigned long long)d << shift); s_need = need - cum; break; }
          cum += hist[d];
        }
      }
      __syncthreads();
      prefix = s_prefix; need = s_need; mask |= 0xFFull << shift;
      __syncthreads();
    }
    thr = keep ? prefix : ~0ull;
  }
  if (tid == 0) s_nk = 0u;
  __syncthreads();
  for (unsigned i = tid; i < n; i += kDbSelThreads) {
    const int r = roots[i];
    if (keep > 0 && db_key(size, r) >= thr) s_kept[atomicAdd(&s_nk, 1u)] = r;
  }
  __syncthreads();
  const unsigned nk = s_nk;
  for (unsigned i = tid; i < n; i += kDbSelThreads) {
    const int r = roots[i];
    int lab = m + 1;
    if (keep > 0 && db_key(size, r) >= thr) {
      lab = 2;
      for (unsigned j = 0; j < nk; ++j) lab += s_kept[j] < r;
    }
    size[r] = lab;
  }
}

__global__ void __launch_bounds__(kDbThreads)
dbscan_labels_kernel(const float* __restrict__ range, int HW, int m, DbWs ws, uint8_t* __restrict__ labels) {
  const int f = blockIdx.y, p = blockIdx.x * kDbThreads + threadIdx.x;
  if (p >= HW) return;
  const size_t o = (size_t)f * HW + p;
  const int* par = ws.parent + (size_t)f * HW;
  const uint8_t sp = ws.state[o];
  int lab;
  if (!(sp & kPoint)) {
    lab = range[o] == 0.f ? 1 : 0;
  } else {
    int x = sp == kCore ? p : par[p];                    // a border starts from its nearest core; noise: -1
    if (x < 0) {
      lab = m + 1;
    } else {
      for (int y = par[x]; y != x; y = par[x]) x = y;    // read-only: no union-find writes are left in flight
      lab = ws.size[(size_t)f * HW + x];
    }
  }
  labels[o] = (uint8_t)lab;
}

}  // namespace rpcc

using namespace rpcc;

extern "C" size_t rpcc_dbscan_workspace_bytes(int B, int H, int W) {
  const size_t n = (size_t)B * H * W;
  return db_align(3 * sizeof(unsigned) * (size_t)B) + db_align(n) + 3 * db_align(sizeof(int) * n);
}

extern "C" int rpcc_dbscan_segment_batch(const float* range, const float* lut, const float* ground, int B, int H, int W,
                                         double hfov, double vmax, double vmin, double eps, int min_points,
                                         int cluster_num, float ground_thr, uint8_t* labels, void* workspace,
                                         void* stream) {
  RPCC_REQUIRE(range && lut && ground && labels && workspace, "null pointer");
  RPCC_REQUIRE(H >= 2 && W >= 1 && B >= 0 && B <= 65535, "bad sizes");
  RPCC_REQUIRE(fabs(hfov - 6.283185307179586) < 1e-6, "the window search needs a 360-degree sensor (columns wrap around)");
  RPCC_REQUIRE(eps > 0, "eps must be positive");
  RPCC_REQUIRE(min_points >= 1, "min_points must be at least 1");
  RPCC_REQUIRE(cluster_num >= 1 && cluster_num + 2 <= 254, "cluster_num must be in [1, 252]");
  if (B == 0) return RPCC_OK;
  const int HW = H * W;
  const float e2 = (float)(eps * eps);
  DbGeom g;
  g.dalt = (float)((vmax - vmin) / (double)(H - 1));
  g.daz = (float)(hfov / (double)W);
  g.cmin = (float)cos(fmax(fabs(vmax), fabs(vmin)));
  const DbWs ws = db_carve(workspace, B, (size_t)HW);
  cudaStream_t st = as_stream(stream);
  RPCC_CUDA(cudaMemsetAsync(ws.fallback, 0, 3 * sizeof(unsigned) * (size_t)B, st));
  if (int rc = eval_neg_flags(range, range, B, HW, ws.neg, st)) return rc;
  const dim3 grid((HW + kDbThreads - 1) / kDbThreads, B);
  dbscan_points_kernel<<<grid, kDbThreads, 0, st>>>(range, lut, ground, HW, ground_thr, ws);
  RPCC_LAUNCH_CHECK("dbscan_points_kernel");
  dbscan_count_kernel<<<grid, kDbThreads, 0, st>>>(range, lut, H, W, g, e2, (unsigned)min_points, ws);
  RPCC_LAUNCH_CHECK("dbscan_count_kernel");
  dbscan_link_kernel<<<grid, kDbThreads, 0, st>>>(range, lut, H, W, g, e2, ws);
  RPCC_LAUNCH_CHECK("dbscan_link_kernel");
  dbscan_resolve_kernel<<<grid, kDbThreads, 0, st>>>(HW, ws);
  RPCC_LAUNCH_CHECK("dbscan_resolve_kernel");
  dbscan_select_kernel<<<B, kDbSelThreads, 0, st>>>(HW, cluster_num, ws);
  RPCC_LAUNCH_CHECK("dbscan_select_kernel");
  dbscan_labels_kernel<<<grid, kDbThreads, 0, st>>>(range, HW, cluster_num, ws, labels);
  RPCC_LAUNCH_CHECK("dbscan_labels_kernel");
  return RPCC_OK;
}
