// quantize.cu -- stage 4: intra-prediction + residual quantisation + stable label-major scatter
// + contour bitmap / index sequence, fused in one pass over the range image.
//
// Replaces, per pixel and bit for bit:
//   segment_utils_cpp.intra_predict        (ops/cpp_modules/src/cpp_modules.cpp:248-285)
//   residual = range - pred                (tools/compress.py:106, numpy f32)
//   quantization_utils_cpp.uniform_quantize / nonuniform_quantize   (:288-334 / :337-424):
//       q = (int)roundf(residual / step_l), emitted label-major (0,2,3,..), raster inside a label
//   .astype(np.int16)                      (utils/compress_utils.py:142, wraps)
//   contour_utils_cpp.extract_contour + np.packbits + astype(uint16)   (:521-558, compress_utils.py:155-160)
//
// Reads 4 B (range) + 1 B (label) per pixel, writes 2 B per valid pixel + 1 bit per pixel + 2 B per run.
// One WARP = one 1024-pixel tile, 8 tiles of a frame per CTA; the tile's range values and labels arrive in shared
// memory through two bulk copies (TMA engine) that complete on the warp's own mbarrier.  The stable rank of a pixel
// inside (tile, label) is a per-warp counter in shared memory, seeded from tile_off (model.cu), plus the pixel's
// rank among the same-label lanes of its 32-pixel slice (match_any): no block-level synchronisation.
#include "async.cuh"
#include "book.cuh"

namespace rpcc {

constexpr int kQWarps = 8;                  // one 1024-pixel tile per warp, 8 tiles per CTA
constexpr int kQThreads = kQWarps * 32;
constexpr int kQOcc = 4;                    // resident CTAs per SM, both quantize kernels
constexpr int kQSlices = 2;                 // 32-pixel slices per step: that many independent loads in flight per lane

// stores into the two output streams: 64-bit base (kept in one register pair) + 32-bit element index
__device__ __forceinline__ void stg_elem(int16_t* base, unsigned i, int v) {
  asm volatile("st.global.u16 [%0], %1;" :: "l"(base + i), "h"((short)v) : "memory");
}
__device__ __forceinline__ void stg_elem(int32_t* base, unsigned i, int v) {
  asm volatile("st.global.u32 [%0], %1;" :: "l"(base + i), "r"(v) : "memory");
}
__device__ __forceinline__ void stg_elem(uint16_t* base, unsigned i, int v) {
  asm volatile("st.global.u16 [%0], %1;" :: "l"(base + i), "h"((unsigned short)v) : "memory");
}

// One warp walks one tile in raster order, 32 consecutive pixels (a slice) at a time, and needs no
// block-level synchronisation: its private counters cnt[label] start at tile_off (the position, in the frame's
// label-major symbol stream, of the tile's first symbol of that label) and advance as the slices go by, so that the
// stable rank of a pixel is counter + (same-label lanes below it) -- one match_any per slice.  Contour bits come from
// one ballot per slice, MSB-first bytes from brev.
//
// The kernel is bound by instruction issue before it is bound by HBM (ncu: 77 % issue-active at 28 % of the HBM peak
// in round 1, 108 warp instructions per slice), so the slice body is written for a short, branch-free instruction
// stream:
//   * the label left of a pixel is a second byte load (same L1 sector) instead of two shuffles and a select;
//   * the two rare per-pixel cases -- a plane row instead of a constant prediction, a quotient too close to a rounding
//     boundary for the reciprocal product -- are taken by the whole warp behind ONE vote per step of 4 slices, so the
//     common path carries no divergence bookkeeping;
//   * a tile holds at most one row start when W >= 1024 (every lidar of the reference): its pixel index is computed
//     once per tile (WIDE), the generic `p % W` stays for narrower images;
//   * shared-memory tables are addressed by 32-bit shared addresses, global streams by a 64-bit base + 32-bit index.
// FULL: the whole tile lies inside the image (no bounds predicates).  CLAMP: labels may exceed K-1 (caller-supplied
// label maps; the encoder's own labels never do).
// STAGED: the tile's range values and labels are in shared memory (rng_addr / lab_addr, brought there by the bulk
// copies of quantize_pack_staged_kernel; lab_addr - 1 holds the label left of the tile), else they are read from
// global memory per slice.
template <typename SymT, bool FULL, bool CLAMP, bool WIDE, bool STAGED>
__device__ __forceinline__ void quantize_tile(const float* __restrict__ rg, const uint8_t* __restrict__ lb, unsigned rng_addr,
                                              unsigned lab_addr,
                                              const float* __restrict__ lut, unsigned model_addr, unsigned tab_addr,
                                              unsigned cnt_addr, SymT* __restrict__ sym, uint16_t* __restrict__ sq,
                                              uint8_t* __restrict__ cbits, int cbytes, int p_tile, int HW, int W, int K,
                                              unsigned lane) {
  const unsigned lt = lanemask_lt();
  // the one pixel of this tile that starts an image row (cpp_modules.cpp:537): slice row_sl, lane row_ln -- or none.
  // Every per-slice test below compares against the slice counter, the only induction variable besides the two
  // shared-memory cursors.
  int row_sl = -1;
  if (WIDE) {
    const int nr = ((p_tile + W - 1) / W) * W - p_tile;      // offset of the next row start inside the tile
    if (nr < RPCC_TILE && (nr & 31) == (int)lane) row_sl = nr >> 5;
  }
  const float* rp = rg + p_tile + (int)lane;     // this lane's pixel of the current slice
  const uint8_t* lp = lb + p_tile + (int)lane;
  unsigned rcur = rng_addr + 4u * lane, lcur = lab_addr + lane;   // STAGED: the same in shared memory
  unsigned nseq = 0;                             // idx_sequence entries emitted by this tile so far
  unsigned myword = 0;                           // contour word of slice `lane` of the tile
  asm volatile("" : "+l"(sym), "+l"(sq));        // keep the two stream bases in one register pair each

#pragma unroll 1
  for (int k = 0; k < RPCC_TILE / 32; k += kQSlices) {       // k: first slice of the step
    const int p_step = p_tile + k * 32;
    if (!FULL && p_step >= HW) break;
    float r[kQSlices];
    int lab[kQSlices], lft[kQSlices];
#pragma unroll
    for (int j = 0; j < kQSlices; ++j) {
      const int p = p_step + j * 32 + (int)lane;
      const bool inb = FULL || p < HW;
      if (STAGED) {
        r[j] = inb ? lds_f32(rcur + 128u * j) : 0.f;
        lab[j] = inb ? (int)lds_u8(lcur + 32u * j) : 1;
        lft[j] = (int)lds_u8(lcur + 32u * j - 1u);
      } else {
        r[j] = inb ? ld_stream_f(rp + j * 32) : 0.f;
        lab[j] = inb ? (int)__ldg(lp + j * 32) : 1;
        // label of the pixel to the left (the frame's first pixel has none: it starts a row, the value is not used)
        lft[j] = (inb && (j > 0 || p > 0)) ? (int)__ldg(lp + j * 32 - 1) : -1;
      }
      if (CLAMP && lab[j] >= K) lab[j] = 1;      // flagged by label_stats; never emitted
      if (CLAMP && lft[j] >= K) lft[j] = 1;
    }
    rp += 32 * kQSlices;
    lp += 32 * kQSlices;
    rcur += 128u * kQSlices;
    lcur += 32u * kQSlices;
    // ---- table look-ups; the ray directions of the pixels whose row is a plane are requested now (L2) and used after
    //      the rank / contour work of the step, which needs neither them nor the prediction
    float pred[kQSlices], inv[kQSlices];
    bool plane[kQSlices], some_plane = false;    // slice j's row is a plane: its 1 / step is stored negated
#pragma unroll
    for (int j = 0; j < kQSlices; ++j) {
      const float2 tb = lds_f2(tab_addr + (unsigned)lab[j] * 16u);
      pred[j] = tb.x;
      inv[j] = tb.y;
      plane[j] = tb.y < 0.0f;
      some_plane = some_plane || plane[j];
    }
    const bool any_plane = __any_sync(0xffffffffu, some_plane);   // the ground row is a plane, in every frame
    float lx[kQSlices], ly[kQSlices], lz[kQSlices];
    if (any_plane) {
#pragma unroll
      for (int j = 0; j < kQSlices; ++j) {
        lx[j] = 0.f; ly[j] = 0.f; lz[j] = 0.f;
        if (plane[j]) {
          const float* t3 = lut + (size_t)(p_step + j * 32 + (int)lane) * 3;
          lx[j] = __ldg(t3); ly[j] = __ldg(t3 + 1); lz[j] = __ldg(t3 + 2);
        }
      }
    }
    // ---- stable positions, contour bits, idx_sequence
    unsigned pos[kQSlices];
#pragma unroll
    for (int j = 0; j < kQSlices; ++j) {
      const int p = p_step + j * 32 + (int)lane;
      const bool inb = FULL || p < HW;
      const int l = lab[j];
      // private counter + rank among the slice's lanes with the same label
      const unsigned grp = __match_any_sync(0xffffffffu, l);
      const unsigned ca = cnt_addr + (unsigned)l * 4u;
      const unsigned base = lds_u32(ca);             // same address for the whole group: one broadcast read
      __syncwarp();
      if ((grp & lt) == 0u) sts_u32(ca, base + __popc(grp));   // the group's lowest lane
      __syncwarp();
      pos[j] = base + __popc(grp & lt);
      // contour bit (cpp_modules.cpp:534-545) and idx_sequence
      const bool rowstart = WIDE ? (row_sl == k + j) : (p % W) == 0;
      const bool c = inb && (rowstart || l != lft[j]);
      const unsigned cb = __ballot_sync(0xffffffffu, c);
      if (c) stg_elem(sq, nseq + __popc(cb & lt), l);
      nseq += __popc(cb);
      if ((int)lane == k + j) myword = cb;
    }
    // ---- symbols (cpp_modules.cpp:264-281, tools/compress.py:106, cpp_modules.cpp:311-331)
    if (any_plane) {
      // (measured and not kept: a branch-free form in which every lane divides, 0.456 ms against 0.385; the plane
      //  prediction by a reciprocal product with an exact fallback for the lanes near a rounding boundary, 0.381 ms --
      //  one per cent for an error analysis that would have to hold for every model a caller can pass)
#pragma unroll
      for (int j = 0; j < kQSlices; ++j) {
        if (plane[j]) {
          const float4 m = lds_f4(model_addr + (unsigned)lab[j] * 16u);
          pred[j] = -m.w / (m.x * lx[j] + m.y * ly[j] + m.z * lz[j]);   // cpp_modules.cpp:273-279
        }
      }
    }
    // q = (int)roundf(res / step) (cpp_modules.cpp:318).  The reciprocal product t is within 1.8e-7 |t| of the
    // IEEE quotient, so unless t lies within 1e-6 |t| of a rounding boundary (k + 0.5) both round to the same
    // integer -- and away from a boundary round-to-nearest-even IS round-half-away.  The few that are near
    // (and NaN / huge values, whose conversion does not round-trip) take the division.
    int q[kQSlices];
    bool near = false;
#pragma unroll
    for (int j = 0; j < kQSlices; ++j) {
      const float t = (r[j] - pred[j]) * fabsf(inv[j]);
      q[j] = __float2int_rn(t);
      near = near || !(__fmaf_rn(fabsf(t), 1e-6f, fabsf(t - (float)q[j])) < 0.5f);
    }
    if (__any_sync(0xffffffffu, near)) {
#pragma unroll
      for (int j = 0; j < kQSlices; ++j) {
        const float res = r[j] - pred[j];
        const float t = res * fabsf(inv[j]);
        if (!(__fmaf_rn(fabsf(t), 1e-6f, fabsf(t - (float)q[j])) < 0.5f))
          q[j] = (int)roundf(res / lds_f32(tab_addr + (unsigned)lab[j] * 16u + 8u));
      }
    }
#pragma unroll
    for (int j = 0; j < kQSlices; ++j)
      if (lab[j] != 1) stg_elem(sym, pos[j], q[j]);   // int16: wraps like astype(np.int16)
  }
  // ---- contour bytes of the tile: lane i holds the word of slice i (np.packbits bytes 4i .. 4i+3 of the tile)
  {
    myword = __byte_perm(__brev(myword), 0, 0x0123);   // np.packbits: pixel p0+i -> byte i/8, bit 7-(i%8)
    const int byte0 = (p_tile >> 3) + 4 * (int)lane;
    if ((cbytes & 3) == 0 && byte0 + 4 <= cbytes) {
      *reinterpret_cast<unsigned*>(cbits + byte0) = myword;
    } else {
#pragma unroll
      for (int b = 0; b < 4; ++b)
        if (byte0 + b < cbytes) cbits[byte0 + b] = (uint8_t)(myword >> (8 * b));
    }
  }
}

template <typename SymT, bool CLAMP, bool WIDE>
__global__ void __launch_bounds__(kQThreads, kQOcc)
quantize_pack_kernel(const float* __restrict__ range, const uint8_t* __restrict__ labels, const float* __restrict__ model,
                     const float* __restrict__ lut, Book bk, const float* __restrict__ step_per_label, float step,
                     int HW, int W, int K, int T, SymT* __restrict__ symbols, size_t sym_stride,
                     uint8_t* __restrict__ contour_bits, int cbytes, uint16_t* __restrict__ seq, size_t seq_stride,
                     const unsigned long long* __restrict__ sym_base, const unsigned long long* __restrict__ seq_base) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4* s_model = reinterpret_cast<float4*>(smem_raw);            // [K]
  float4* s_tab = s_model + K;                                      // [K] constant prediction, 1 / step (negated: the row is a plane), step, -
  unsigned* s_cnt = reinterpret_cast<unsigned*>(s_tab + K);         // [kQWarps][K] next symbol position per label

  const int f = blockIdx.y, tid = threadIdx.x;
  const unsigned lane = tid & 31, warp = tid >> 5;
  const int tile = blockIdx.x * kQWarps + (int)warp;
  for (int l = tid; l < K; l += kQThreads) {
    const float4 m = reinterpret_cast<const float4*>(model)[(size_t)f * K + l];
    s_model[l] = m;
    const float st = step_per_label ? step_per_label[(size_t)f * K + l] : step;
    s_tab[l] = make_float4(m.w, (m.x + m.y + m.z == 0) ? 1.0f / st : -(1.0f / st), st, 0.0f);
  }
  unsigned* cnt = s_cnt + warp * K;
  if (tile < T)
    for (int l = lane; l < K; l += 32) cnt[l] = bk.tile_off[((size_t)f * T + tile) * K + l];
  __syncthreads();
  if (tile >= T) return;

  const size_t fbase = (size_t)f * HW;
  SymT* sym = symbols + (sym_base ? (size_t)sym_base[f] : (size_t)f * sym_stride);
  uint16_t* sq = seq + (seq_base ? (size_t)seq_base[f] : (size_t)f * seq_stride) + bk.tile_coff[(size_t)f * T + tile];
  const int p_tile = tile * RPCC_TILE;
  const unsigned model_addr = (unsigned)__cvta_generic_to_shared(s_model);
  const unsigned tab_addr = (unsigned)__cvta_generic_to_shared(s_tab);
  const unsigned cnt_addr = (unsigned)__cvta_generic_to_shared(cnt);
  uint8_t* cb = contour_bits + (size_t)f * cbytes;
  if (p_tile + RPCC_TILE <= HW)
    quantize_tile<SymT, true, CLAMP, WIDE, false>(range + fbase, labels + fbase, 0u, 0u, lut, model_addr, tab_addr, cnt_addr,
                                                  sym, sq, cb, cbytes, p_tile, HW, W, K, lane);
  else
    quantize_tile<SymT, false, CLAMP, WIDE, false>(range + fbase, labels + fbase, 0u, 0u, lut, model_addr, tab_addr, cnt_addr,
                                                   sym, sq, cb, cbytes, p_tile, HW, W, K, lane);
}

// The same with the inputs staged through shared memory by the TMA engine: one elected lane per warp issues two bulk
// copies (cp.async.bulk: the tile's 4 KB of range values and 1 KB of labels) that complete on the warp's own mbarrier;
// the warp then works entirely out of shared memory.  No per-slice global load sits in the dependency chain any more,
// a whole tile per warp is in flight from the first instruction, and the 4 resident CTAs of an SM overlap the copies
// of one with the arithmetic of the others.  Needs 16-byte aligned bases and HW % 16 == 0 (every lidar of the
// reference; otherwise the launcher falls back to quantize_pack_kernel).
constexpr int kQsLabPad = 16;                                         // bytes in front of a warp's labels: [15] = left label
constexpr int kQsWarpBytes = RPCC_TILE * 4 + kQsLabPad + RPCC_TILE;   // 5136

template <typename SymT, bool CLAMP, bool WIDE>
__global__ void __launch_bounds__(kQThreads, kQOcc)
quantize_pack_staged_kernel(const float* __restrict__ range, const uint8_t* __restrict__ labels, const float* __restrict__ model,
                            const float* __restrict__ lut, Book bk, const float* __restrict__ step_per_label, float step,
                            int HW, int W, int K, int T, SymT* __restrict__ symbols, size_t sym_stride,
                            uint8_t* __restrict__ contour_bits, int cbytes, uint16_t* __restrict__ seq, size_t seq_stride,
                            const unsigned long long* __restrict__ sym_base, const unsigned long long* __restrict__ seq_base) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* s_stage = smem_raw;                                              // [kQWarps][kQsWarpBytes]
  unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(s_stage + kQWarps * kQsWarpBytes);   // [kQWarps]
  float4* s_model = reinterpret_cast<float4*>(s_bar + kQWarps);                   // [K]
  float4* s_tab = s_model + K;                                                    // [K]
  unsigned* s_cnt = reinterpret_cast<unsigned*>(s_tab + K);                       // [kQWarps][K]

  const int f = blockIdx.y, tid = threadIdx.x;
  const unsigned lane = tid & 31, warp = tid >> 5;
  const int tile = blockIdx.x * kQWarps + (int)warp;
  const int p_tile = tile * RPCC_TILE;
  const size_t fbase = (size_t)f * HW;
  const unsigned stage = smem_addr(s_stage + warp * kQsWarpBytes);
  const unsigned rng_addr = stage, lab_addr = stage + RPCC_TILE * 4 + kQsLabPad;
  const unsigned bar = smem_addr(s_bar + warp);
  // every global load of the prologue is issued before any of them is consumed: one memory latency, not four
  const bool live = tile < T;
  if (live && lane == 0) {
    const int n = min(RPCC_TILE, HW - p_tile);
    mbar_init(bar, 1);
    mbar_init_fence();
    mbar_arrive_expect_tx(bar, (unsigned)n * 5u);
    bulk_load(rng_addr, range + fbase + p_tile, (unsigned)n * 4u, bar);
    bulk_load(lab_addr, labels + fbase + p_tile, (unsigned)n, bar);
  }
  // the label left of the tile (the frame's first pixel has none: it starts a row, the value is not used)
  unsigned left0 = 0xFFu;
  if (live && lane == 0 && p_tile > 0) left0 = (unsigned)__ldg(labels + fbase + p_tile - 1);
  unsigned toff[(RPCC_MAX_LABELS + 31) / 32];
#pragma unroll
  for (int i = 0; i < (RPCC_MAX_LABELS + 31) / 32; ++i) {
    const int l = (int)lane + 32 * i;
    toff[i] = (live && l < K) ? __ldg(bk.tile_off + ((size_t)f * T + tile) * K + l) : 0u;
  }
  unsigned coff = 0;
  if (live) coff = __ldg(bk.tile_coff + (size_t)f * T + tile);
  constexpr int kRows = (254 + kQThreads - 1) / kQThreads;          // model rows per thread (K <= 254)
  float4 m[kRows];
  float st[kRows];
#pragma unroll
  for (int i = 0; i < kRows; ++i) {
    const int l = tid + i * kQThreads;
    m[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    st[i] = step;
    if (l < K) {
      m[i] = __ldg(reinterpret_cast<const float4*>(model) + (size_t)f * K + l);
      if (step_per_label) st[i] = __ldg(step_per_label + (size_t)f * K + l);
    }
  }
  const unsigned long long sbase = sym_base ? __ldg(sym_base + f) : (unsigned long long)f * sym_stride;
  const unsigned long long qbase = seq_base ? __ldg(seq_base + f) : (unsigned long long)f * seq_stride;
#pragma unroll
  for (int i = 0; i < kRows; ++i) {
    const int l = tid + i * kQThreads;
    if (l < K) {
      s_model[l] = m[i];
      s_tab[l] = make_float4(m[i].w, (m[i].x + m[i].y + m[i].z == 0) ? 1.0f / st[i] : -(1.0f / st[i]), st[i], 0.0f);
    }
  }
  unsigned* cnt = s_cnt + warp * K;
#pragma unroll
  for (int i = 0; i < (RPCC_MAX_LABELS + 31) / 32; ++i) {
    const int l = (int)lane + 32 * i;
    if (live && l < K) cnt[l] = toff[i];
  }
  if (live && lane == 0) sts_u8(lab_addr - 1u, left0);
  __syncthreads();
  if (!live) return;

  SymT* sym = symbols + (size_t)sbase;
  uint16_t* sq = seq + (size_t)qbase + coff;
  const unsigned model_addr = smem_addr(s_model), tab_addr = smem_addr(s_tab), cnt_addr = smem_addr(cnt);
  uint8_t* cb = contour_bits + (size_t)f * cbytes;
  mbar_wait(bar, 0);
  if (p_tile + RPCC_TILE <= HW)
    quantize_tile<SymT, true, CLAMP, WIDE, true>(nullptr, nullptr, rng_addr, lab_addr, lut, model_addr, tab_addr, cnt_addr, sym,
                                                 sq, cb, cbytes, p_tile, HW, W, K, lane);
  else
    quantize_tile<SymT, false, CLAMP, WIDE, true>(nullptr, nullptr, rng_addr, lab_addr, lut, model_addr, tab_addr, cnt_addr, sym,
                                                  sq, cb, cbytes, p_tile, HW, W, K, lane);
}

// exclusive scan of the per-frame symbol / sequence counts (one CTA; B <= 65535)
__global__ void __launch_bounds__(1024)
frame_offsets_kernel(const rpcc_frame_result* __restrict__ results, int B, unsigned long long* __restrict__ sym_base,
                     unsigned long long* __restrict__ seq_base) {
  __shared__ unsigned long long s_a[32], s_b[32];
  __shared__ unsigned long long s_run[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { s_run[0] = 0; s_run[1] = 0; }
  __syncthreads();
  for (int b0 = 0; b0 < B; b0 += 1024) {
    const int b = b0 + tid;
    const unsigned long long a = b < B ? results[b].sym_count : 0ull;
    const unsigned long long c = b < B ? results[b].seq_count : 0ull;
    unsigned long long ia = a, ic = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long va = __shfl_up_sync(0xffffffffu, ia, o), vc = __shfl_up_sync(0xffffffffu, ic, o);
      if (lane >= o) { ia += va; ic += vc; }
    }
    if (lane == 31) { s_a[warp] = ia; s_b[warp] = ic; }
    __syncthreads();
    unsigned long long wa = 0, wc = 0;
    for (int q = 0; q < warp; ++q) { wa += s_a[q]; wc += s_b[q]; }
    if (b < B) { sym_base[b] = s_run[0] + wa + ia - a; seq_base[b] = s_run[1] + wc + ic - c; }
    __syncthreads();
    if (tid == 1023) { s_run[0] += wa + ia; s_run[1] += wc + ic; }
    __syncthreads();
  }
  if (tid == 0) { sym_base[B] = s_run[0]; seq_base[B] = s_run[1]; }
}

}  // namespace rpcc

using namespace rpcc;

extern "C" int rpcc_frame_offsets_batch(const rpcc_frame_result* results, int B, uint64_t* sym_base, uint64_t* seq_base,
                                        void* stream) {
  RPCC_REQUIRE(results && sym_base && seq_base, "null pointer");
  frame_offsets_kernel<<<1, 1024, 0, as_stream(stream)>>>(results, B, reinterpret_cast<unsigned long long*>(sym_base),
                                                          reinterpret_cast<unsigned long long*>(seq_base));
  RPCC_LAUNCH_CHECK("frame_offsets_kernel");
  return RPCC_OK;
}

namespace rpcc {

// SymT = int16_t: the bitstream type (utils/compress_utils.py:142); int32_t: what
// uniform_quantize / nonuniform_quantize themselves return (cpp_modules.cpp:322,408).
template <typename SymT>
int quantize_pack_launch(const float* range, const uint8_t* labels, const float* model, const float* lut, void* book,
                         const float* step_per_label, float step, int B, int H, int W, int K, SymT* symbols,
                         size_t sym_stride, uint8_t* contour_bits, uint16_t* seq, size_t seq_stride,
                         const uint64_t* sym_base, const uint64_t* seq_base, void* stream, bool trusted_labels) {
  RPCC_REQUIRE(range && labels && model && lut && book && symbols && contour_bits && seq, "null pointer");
  RPCC_REQUIRE(K >= 2 && K <= 254, "K must be in [2, 254]");
  RPCC_REQUIRE(B <= 65535, "at most 65535 frames per launch");
  if (B == 0) return RPCC_OK;
  const int HW = H * W, T = (HW + RPCC_TILE - 1) / RPCC_TILE;
  const Book bk = make_book(book, B, T, K);
  const size_t smem = 2 * sizeof(float4) * K + sizeof(unsigned) * (size_t)kQWarps * K;
  const dim3 grid((T + kQWarps - 1) / kQWarps, B);
  cudaStream_t st = as_stream(stream);
  const int cbytes = (HW + 7) / 8;
  const unsigned long long* sb = reinterpret_cast<const unsigned long long*>(sym_base);
  const unsigned long long* qb = reinterpret_cast<const unsigned long long*>(seq_base);
#define RPCC_Q_LAUNCH(CLAMP, WIDE)                                                                                       \
  quantize_pack_kernel<SymT, CLAMP, WIDE><<<grid, kQThreads, smem, st>>>(range, labels, model, lut, bk, step_per_label,  \
                                                                         step, HW, W, K, T, symbols, sym_stride,          \
                                                                         contour_bits, cbytes, seq, seq_stride, sb, qb)
  const bool wide = W >= RPCC_TILE;      // at most one row start per 1024-pixel tile
  // bulk copies need 16-byte aligned sources and sizes
  const bool staged = wide && (HW % 16) == 0 && ((uintptr_t)range % 16) == 0 && ((uintptr_t)labels % 16) == 0;
  if (staged) {
    const size_t smem_s = (size_t)kQWarps * kQsWarpBytes + 8 * kQWarps + smem;
#define RPCC_QS_LAUNCH(CLAMP)                                                                                            \
  do {                                                                                                                   \
    RPCC_CUDA(cudaFuncSetAttribute(quantize_pack_staged_kernel<SymT, CLAMP, true>,                                       \
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_s));                           \
    quantize_pack_staged_kernel<SymT, CLAMP, true><<<grid, kQThreads, smem_s, st>>>(                                     \
        range, labels, model, lut, bk, step_per_label, step, HW, W, K, T, symbols, sym_stride, contour_bits, cbytes,     \
        seq, seq_stride, sb, qb);                                                                                        \
  } while (0)
    if (trusted_labels) RPCC_QS_LAUNCH(false); else RPCC_QS_LAUNCH(true);
#undef RPCC_QS_LAUNCH
  } else if (trusted_labels) { if (wide) RPCC_Q_LAUNCH(false, true); else RPCC_Q_LAUNCH(false, false); }
  else { if (wide) RPCC_Q_LAUNCH(true, true); else RPCC_Q_LAUNCH(true, false); }
#undef RPCC_Q_LAUNCH
  RPCC_LAUNCH_CHECK("quantize_pack_kernel");
  return RPCC_OK;
}
template int quantize_pack_launch<int32_t>(const float*, const uint8_t*, const float*, const float*, void*, const float*, float,
                                           int, int, int, int, int32_t*, size_t, uint8_t*, uint16_t*, size_t, const uint64_t*,
                                           const uint64_t*, void*, bool);
template int quantize_pack_launch<int16_t>(const float*, const uint8_t*, const float*, const float*, void*, const float*, float,
                                           int, int, int, int, int16_t*, size_t, uint8_t*, uint16_t*, size_t, const uint64_t*,
                                           const uint64_t*, void*, bool);
}  // namespace rpcc

extern "C" int rpcc_quantize_pack_batch(const float* range, const uint8_t* labels, const float* model, const float* lut,
                                        void* book, const float* step_per_label, float step, int B, int H, int W, int K,
                                        int16_t* symbols, size_t sym_stride, uint8_t* contour_bits, uint16_t* seq,
                                        size_t seq_stride, const uint64_t* sym_base, const uint64_t* seq_base,
                                        void* stream) {
  return quantize_pack_launch<int16_t>(range, labels, model, lut, book, step_per_label, step, B, H, W, K, symbols, sym_stride,
                                       contour_bits, seq, seq_stride, sym_base, seq_base, stream, false);
}
