// points.cu -- the last step of decoding: reconstructed range images -> the rows of the output `.bin` files.
//
// Replaces PCTransformer.range_image_to_point_cloud (reference dataset/transformer.py:94-101) followed by
// save_point_cloud_to_file's filter (dataset/dataset.py:72-81): xyz = range_rec * LUT (f32), keep the pixels whose
// float32 sum x + y + z is not zero, append the intensity (the decoded intensity image, or zero).  Frames come out packed back to back in raster order
// (frame b's rows are rows[row_base[b] .. row_base[b+1])), so one device -> host copy per batch carries exactly the
// bytes that go to disk and the host never touches the 1.5 MB xyz image of a frame.
#include "common.cuh"

namespace rpcc {

constexpr int kPtWarps = 8;

__device__ __forceinline__ bool point_at(const float* __restrict__ rg, const float* __restrict__ lut, int p, float4& out) {
  const float r = __ldg(rg + p);
  out.x = r * __ldg(lut + 3 * (size_t)p);
  out.y = r * __ldg(lut + 3 * (size_t)p + 1);
  out.z = r * __ldg(lut + 3 * (size_t)p + 2);
  out.w = 0.f;
  return (out.x + out.y) + out.z != 0.f;      // np.sum(point_cloud, -1) != 0
}

// one warp per 1024-pixel tile: points in the tile
__global__ void __launch_bounds__(kPtWarps * 32)
points_count_kernel(const float* __restrict__ range, const float* __restrict__ lut, int HW, int T, unsigned* __restrict__ tile_cnt) {
  const int f = blockIdx.y, lane = threadIdx.x & 31, tile = blockIdx.x * kPtWarps + (threadIdx.x >> 5);
  if (tile >= T) return;
  const float* rg = range + (size_t)f * HW;
  unsigned n = 0;
  for (int s = 0; s < RPCC_TILE / 32; ++s) {
    const int p = tile * RPCC_TILE + s * 32 + lane;
    float4 v;
    const bool ok = p < HW && point_at(rg, lut, p, v);
    n += __popc(__ballot_sync(0xffffffffu, ok));
  }
  if (lane == 0) tile_cnt[(size_t)f * T + tile] = n;
}

// per frame: tile counts -> offsets inside the frame (in place), and the frame's total
__global__ void __launch_bounds__(1024)
points_frame_scan_kernel(unsigned* __restrict__ tile_cnt, int T, unsigned* __restrict__ frame_cnt) {
  __shared__ unsigned s_w[32];
  const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned c = tid < T ? tile_cnt[(size_t)f * T + tid] : 0u;
  unsigned incl = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    unsigned w = s_w[lane], wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += v; }
    s_w[lane] = wi - w;
    if (lane == 31) frame_cnt[f] = wi;
  }
  __syncthreads();
  if (tid < T) tile_cnt[(size_t)f * T + tid] = s_w[warp] + incl - c;
}

// row_base[b] = points of frames 0..b-1 (u64), row_base[B] = all; a single CTA walks the frames in chunks of 1024
__global__ void __launch_bounds__(1024)
points_base_kernel(const unsigned* __restrict__ frame_cnt, int B, unsigned long long* __restrict__ row_base) {
  __shared__ unsigned long long s_w[32];
  __shared__ unsigned long long s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_carry = 0ull;
  __syncthreads();
  for (int b0 = 0; b0 < B; b0 += 1024) {
    const int b = b0 + tid;
    const unsigned long long c = b < B ? (unsigned long long)frame_cnt[b] : 0ull;
    unsigned long long incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      unsigned long long w = s_w[lane], wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const unsigned long long v = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += v; }
      s_w[lane] = wi - w;
    }
    __syncthreads();
    const unsigned long long carry = s_carry;
    if (b < B) row_base[b] = carry + s_w[warp] + incl - c;
    __syncthreads();
    if (tid == 1023) s_carry = carry + s_w[warp] + incl;
    __syncthreads();
  }
  if (tid == 0) row_base[B] = s_carry;
}

__global__ void __launch_bounds__(kPtWarps * 32)
points_write_kernel(const float* __restrict__ range, const float* __restrict__ lut, const float* __restrict__ intensity,
                    int HW, int T, const unsigned* __restrict__ tile_off, const unsigned long long* __restrict__ row_base,
                    float4* __restrict__ rows) {
  const int f = blockIdx.y, lane = threadIdx.x & 31, tile = blockIdx.x * kPtWarps + (threadIdx.x >> 5);
  if (tile >= T) return;
  const float* rg = range + (size_t)f * HW;
  float4* out = rows + row_base[f] + tile_off[(size_t)f * T + tile];
  unsigned at = 0;
  for (int s = 0; s < RPCC_TILE / 32; ++s) {
    const int p = tile * RPCC_TILE + s * 32 + lane;
    float4 v;
    const bool ok = p < HW && point_at(rg, lut, p, v);
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (ok && intensity) v.w = __ldg(intensity + (size_t)f * HW + p);
    if (ok) out[at + __popc(m & lanemask_lt())] = v;
    at += __popc(m);
  }
}

}  // namespace rpcc

using namespace rpcc;

extern "C" size_t rpcc_points_workspace_bytes(int B, int H, int W) {
  const size_t T = ((size_t)H * W + RPCC_TILE - 1) / RPCC_TILE;
  return sizeof(unsigned) * ((size_t)B * T + (size_t)B) + 64;
}

extern "C" int rpcc_points_out_intensity_batch(const float* range_rec, const float* lut, const float* intensity, int B,
                                               int H, int W, float* rows, uint64_t* row_base, void* workspace, void* stream) {
  RPCC_REQUIRE(range_rec && lut && rows && row_base && workspace, "null pointer");
  RPCC_REQUIRE(B >= 0 && B <= 65535, "at most 65535 frames per launch");
  const int HW = H * W, T = (HW + RPCC_TILE - 1) / RPCC_TILE;
  RPCC_REQUIRE(T >= 1 && T <= 1024, "range image too large");
  cudaStream_t st = as_stream(stream);
  unsigned* tile_cnt = static_cast<unsigned*>(workspace);
  unsigned* frame_cnt = tile_cnt + (size_t)B * T;
  if (B == 0) { RPCC_CUDA(cudaMemsetAsync(row_base, 0, sizeof(uint64_t), st)); return RPCC_OK; }
  const dim3 grid((T + kPtWarps - 1) / kPtWarps, B);
  points_count_kernel<<<grid, kPtWarps * 32, 0, st>>>(range_rec, lut, HW, T, tile_cnt);
  RPCC_LAUNCH_CHECK("points_count_kernel");
  points_frame_scan_kernel<<<B, 1024, 0, st>>>(tile_cnt, T, frame_cnt);
  RPCC_LAUNCH_CHECK("points_frame_scan_kernel");
  points_base_kernel<<<1, 1024, 0, st>>>(frame_cnt, B, reinterpret_cast<unsigned long long*>(row_base));
  RPCC_LAUNCH_CHECK("points_base_kernel");
  points_write_kernel<<<grid, kPtWarps * 32, 0, st>>>(range_rec, lut, intensity, HW, T, tile_cnt,
                                                     reinterpret_cast<const unsigned long long*>(row_base),
                                                     reinterpret_cast<float4*>(rows));
  RPCC_LAUNCH_CHECK("points_write_kernel");
  return RPCC_OK;
}

extern "C" int rpcc_points_out_batch(const float* range_rec, const float* lut, int B, int H, int W, float* rows,
                                     uint64_t* row_base, void* workspace, void* stream) {
  return rpcc_points_out_intensity_batch(range_rec, lut, nullptr, B, H, W, rows, row_base, workspace, stream);
}
