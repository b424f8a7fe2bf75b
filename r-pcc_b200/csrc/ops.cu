// ops.cu -- one-frame, host-pointer entry points: the one-to-one replacements of the reference's
// pybind11 functions (ops/cpp_modules/src/cpp_modules.cpp:597-636), of
// furthest_point_sampling_wrapper (ops/fps/src/sampling.cpp:24-37) and of chamfer_3D.forward
// (utils/ChamferDistancePytorch/chamfer3D/chamfer_cuda.cpp:17-19).  Each one uploads its numpy-shaped
// arguments, runs the same batch kernels the pipeline uses with B = 1, and downloads the result;
// they are synchronous like the functions they replace.  Labels arrive as int32 (what
// py::array_t<int> delivers) and must lie in [0, 253].
#include <vector>

#include "book.cuh"

using namespace rpcc;

namespace rpcc {
template <typename SymT>
int quantize_pack_launch(const float* range, const uint8_t* labels, const float* model, const float* lut, void* book,
                         const float* step_per_label, float step, int B, int H, int W, int K, SymT* symbols,
                         size_t sym_stride, uint8_t* contour_bits, uint16_t* seq, size_t seq_stride,
                         const uint64_t* sym_base, const uint64_t* seq_base, void* stream, bool trusted_labels);
}

namespace {

struct DevBuf {
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  int alloc(size_t bytes) { return check_cuda(cudaMalloc(&p, bytes ? bytes : 16), "cudaMalloc"); }
  template <typename T> T* as() { return static_cast<T*>(p); }
};

int upload(DevBuf& d, const void* src, size_t bytes) {
  int rc = d.alloc(bytes);
  if (rc != RPCC_OK) return rc;
  return check_cuda(cudaMemcpy(d.p, src, bytes, cudaMemcpyHostToDevice), "cudaMemcpy H2D");
}

int download(void* dst, const void* src, size_t bytes) {
  return check_cuda(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost), "cudaMemcpy D2H");
}

// int32 labels -> u8; *kmax = highest label.  Rejects labels outside [0, 253].
int narrow_labels(const int32_t* seg, size_t n, std::vector<uint8_t>& out, int* kmax) {
  out.resize(n);
  int mx = 0;
  for (size_t i = 0; i < n; ++i) {
    const int v = seg[i];
    if (v < 0 || v > 253) { set_error("label %d at pixel %zu is outside [0, 253]", v, i); return RPCC_ERR_ARG; }
    out[i] = (uint8_t)v;
    mx = v > mx ? v : mx;
  }
  *kmax = mx;
  return RPCC_OK;
}

#define TRY(x) do { int _r = (x); if (_r != RPCC_OK) return _r; } while (0)

// labels + "range" -> book through point_model (offsets, counts); optionally the means.
struct FrameBook {
  DevBuf labels, range, book, model, results, ground;
  int K = 0;
  rpcc_frame_result res{};
  int build(const float* range_host, const int32_t* seg, int H, int W, bool want_model, int K_min = 2) {
    const size_t HW = (size_t)H * W;
    std::vector<uint8_t> lab;
    int kmax = 0;
    TRY(narrow_labels(seg, HW, lab, &kmax));
    K = kmax + 1 > K_min ? kmax + 1 : K_min;
    TRY(upload(labels, lab.data(), HW));
    TRY(upload(range, range_host, HW * sizeof(float)));
    TRY(book.alloc(rpcc_book_bytes(1, H, W, K)));
    TRY(results.alloc(sizeof(rpcc_frame_result)));
    TRY(rpcc_label_stats_batch(range.as<float>(), labels.as<uint8_t>(), 1, H, W, K, book.p, nullptr));
    if (want_model) {
      const float zero[4] = {0, 0, 0, 0};
      TRY(upload(ground, zero, sizeof(zero)));
      TRY(model.alloc(sizeof(float) * 4 * K));
    }
    TRY(rpcc_point_model_batch(range.as<float>(), labels.as<uint8_t>(), want_model ? ground.as<float>() : nullptr, book.p, 1,
                               H, W, K, want_model ? model.as<float>() : nullptr, results.as<rpcc_frame_result>(), nullptr));
    TRY(download(&res, results.p, sizeof(res)));
    return RPCC_OK;
  }
};

__global__ void intra_predict_kernel(const int32_t* __restrict__ seg, const float* __restrict__ model, int K,
                                     const float* __restrict__ lut, int HW, float* __restrict__ pred) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const int l = seg[p];
  // the reference reads model[label] unchecked (cpp_modules.cpp:266-270); out-of-range labels give NaN here
  if (l < 0 || l >= K) { pred[p] = __int_as_float(0x7fc00000); return; }
  const float m0 = model[l * 4], m1 = model[l * 4 + 1], m2 = model[l * 4 + 2], m3 = model[l * 4 + 3];
  if (m0 + m1 + m2 == 0) pred[p] = m3;
  else pred[p] = -m3 / (m0 * lut[(size_t)p * 3] + m1 * lut[(size_t)p * 3 + 1] + m2 * lut[(size_t)p * 3 + 2]);
}

__global__ void kp_count_kernel(const uint8_t* __restrict__ labels, const int32_t* __restrict__ kp, int HW, int K,
                                unsigned* __restrict__ kp_cnt) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const int l = labels[p];
  if (l != 1 && l < K && kp[p] > 0) atomicAdd(&kp_cnt[l], 1u);
}

// shared tail of the two quantisers: symbols as int32 in the reference's order
int quantize_common(FrameBook& fb, int H, int W, const float* step_per_label_dev, float step, int32_t* out, int64_t* n_out) {
  const size_t HW = (size_t)H * W;
  DevBuf zero_model, lut, sym, contour, seq;
  std::vector<float> zm((size_t)fb.K * 4, 0.f);
  TRY(upload(zero_model, zm.data(), zm.size() * sizeof(float)));   // pred == 0: the "range" input IS the residual
  TRY(lut.alloc(16));                                              // never read: every model row is a point model
  TRY(sym.alloc(HW * sizeof(int32_t)));
  TRY(contour.alloc((HW + 7) / 8));
  TRY(seq.alloc(HW * sizeof(uint16_t)));
  // int32 symbols, as the reference's quantisers return them (narrowing to int16 happens later,
  // utils/compress_utils.py:142)
  TRY(quantize_pack_launch<int32_t>(fb.range.as<float>(), fb.labels.as<uint8_t>(), zero_model.as<float>(), lut.as<float>(),
                                    fb.book.p, step_per_label_dev, step, 1, H, W, fb.K, sym.as<int32_t>(), HW,
                                    contour.as<uint8_t>(), seq.as<uint16_t>(), HW, nullptr, nullptr, nullptr, false));
  *n_out = (int64_t)fb.res.sym_count;
  return download(out, sym.p, (size_t)fb.res.sym_count * sizeof(int32_t));
}

}  // namespace

extern "C" int rpcc_op_point_cloud_to_range_image_even(const float* points, int64_t n, int stride, int H, int W, float hfov,
                                                       float vmax, float vmin, float* range_out) {
  RPCC_REQUIRE(points || n == 0, "null pointer");
  RPCC_REQUIRE(range_out && n >= 0, "bad argument");
  DevBuf d_pts, d_off, d_rng, d_scr;
  TRY(upload(d_pts, points, sizeof(float) * stride * (size_t)n));
  const int64_t off[2] = {0, n};
  TRY(upload(d_off, off, sizeof(off)));
  TRY(d_rng.alloc(sizeof(float) * (size_t)H * W));
  TRY(d_scr.alloc(sizeof(int32_t) * 4));
  TRY(rpcc_project_batch(d_pts.as<float>(), stride, d_off.as<int64_t>(), 1, H, W, hfov, vmax, vmin, d_rng.as<float>(),
                         d_scr.as<int32_t>(), nullptr));
  return download(range_out, d_rng.p, sizeof(float) * (size_t)H * W);
}

extern "C" int rpcc_op_point_modeling(const float* range, const int32_t* seg, int H, int W, float* out, int cap, int* K_out) {
  RPCC_REQUIRE(range && seg && out && K_out, "null pointer");
  FrameBook fb;
  TRY(fb.build(range, seg, H, W, true));
  // the reference sizes its output by the highest label (cpp_modules.cpp:481-486,505)
  const int K = (int)fb.res.model_rows > 1 ? (int)fb.res.model_rows : 1;
  int kmax = 0;
  for (size_t i = 0; i < (size_t)H * W; ++i) kmax = seg[i] > kmax ? seg[i] : kmax;
  const int Kref = kmax + 1;
  (void)K;
  RPCC_REQUIRE(cap >= Kref, "output too small");
  std::vector<float> m((size_t)fb.K * 4);
  TRY(download(m.data(), fb.model.p, m.size() * sizeof(float)));
  for (int l = 0; l < Kref; ++l) out[l] = l < 2 ? 0.0f : m[(size_t)l * 4 + 3];
  *K_out = Kref;
  return RPCC_OK;
}

extern "C" int rpcc_op_intra_predict(const int32_t* seg, const float* model, int K, const float* lut, int H, int W, float* pred) {
  RPCC_REQUIRE(seg && model && lut && pred && K >= 1, "bad argument");
  const size_t HW = (size_t)H * W;
  DevBuf d_seg, d_model, d_lut, d_pred;
  TRY(upload(d_seg, seg, HW * sizeof(int32_t)));
  TRY(upload(d_model, model, sizeof(float) * 4 * K));
  TRY(upload(d_lut, lut, HW * 3 * sizeof(float)));
  TRY(d_pred.alloc(HW * sizeof(float)));
  intra_predict_kernel<<<(unsigned)((HW + 255) / 256), 256>>>(d_seg.as<int32_t>(), d_model.as<float>(), K, d_lut.as<float>(),
                                                              (int)HW, d_pred.as<float>());
  count_launch();
  TRY(check_cuda(cudaGetLastError(), "intra_predict_kernel"));
  return download(pred, d_pred.p, HW * sizeof(float));
}

extern "C" int rpcc_op_uniform_quantize(const int32_t* seg, const float* residual, int H, int W, float acc, int32_t* out,
                                        int64_t* n_out) {
  RPCC_REQUIRE(seg && residual && out && n_out, "null pointer");
  FrameBook fb;
  TRY(fb.build(residual, seg, H, W, false));
  return quantize_common(fb, H, W, nullptr, acc, out, n_out);
}

extern "C" int rpcc_op_extract_features_with_segment(const float* range, const int32_t* seg, int H, int W, int region,
                                                     int segments, int sharp_num, int less_sharp_num, int flat_num,
                                                     float* feature_map, int32_t* key_point_map) {
  RPCC_REQUIRE(range && seg && key_point_map, "null pointer");
  const size_t HW = (size_t)H * W;
  std::vector<uint8_t> lab;
  int kmax = 0;
  TRY(narrow_labels(seg, HW, lab, &kmax));
  const int K = kmax + 1 > 2 ? kmax + 1 : 2;
  DevBuf d_lab, d_rng, d_kp, d_feat, d_cnt;
  TRY(upload(d_lab, lab.data(), HW));
  TRY(upload(d_rng, range, HW * sizeof(float)));
  TRY(d_kp.alloc(HW));
  TRY(d_cnt.alloc(sizeof(uint32_t) * K));
  if (feature_map) TRY(d_feat.alloc(HW * sizeof(float)));
  TRY(rpcc_keypoints_salience_batch(d_rng.as<float>(), d_lab.as<uint8_t>(), nullptr, 1, H, W, K, region, segments, sharp_num,
                                    less_sharp_num, flat_num, nullptr, nullptr, 0, 0, d_kp.as<uint8_t>(),
                                    feature_map ? d_feat.as<float>() : nullptr, nullptr, nullptr, d_cnt.as<uint32_t>(), nullptr));
  std::vector<uint8_t> kp(HW);
  TRY(download(kp.data(), d_kp.p, HW));
  for (size_t i = 0; i < HW; ++i) key_point_map[i] = kp[i];
  if (feature_map) TRY(download(feature_map, d_feat.p, HW * sizeof(float)));
  return RPCC_OK;
}

extern "C" int rpcc_op_nonuniform_quantize(const int32_t* seg, const float* residual, const int32_t* key_point_map, int H,
                                           int W, const int32_t* level_kp_num, const float* level_acc, int level_num,
                                           int ground_level, int32_t* out, int64_t* n_out, int32_t* salience, int* K_out) {
  RPCC_REQUIRE(seg && residual && key_point_map && level_kp_num && level_acc && out && n_out && salience && K_out, "null pointer");
  RPCC_REQUIRE(level_num >= 1 && level_num <= 8, "1..8 salience levels");
  const size_t HW = (size_t)H * W;
  FrameBook fb;
  TRY(fb.build(residual, seg, H, W, false));
  int kmax = 0;
  for (size_t i = 0; i < HW; ++i) kmax = seg[i] > kmax ? seg[i] : kmax;
  const int Kref = kmax + 1;  // the reference's cluster_num (cpp_modules.cpp:355-360)
  // salience rule on the host from device counts (cpp_modules.cpp:388-405)
  DevBuf d_kp, d_cnt, d_step;
  TRY(upload(d_kp, key_point_map, HW * sizeof(int32_t)));
  TRY(d_cnt.alloc(sizeof(uint32_t) * fb.K));
  TRY(check_cuda(cudaMemset(d_cnt.p, 0, sizeof(uint32_t) * fb.K), "memset"));
  kp_count_kernel<<<(unsigned)((HW + 255) / 256), 256>>>(fb.labels.as<uint8_t>(), d_kp.as<int32_t>(), (int)HW, fb.K, d_cnt.as<uint32_t>());
  count_launch();
  TRY(check_cuda(cudaGetLastError(), "kp_count_kernel"));
  std::vector<uint32_t> kpn(fb.K), pn(fb.K);
  TRY(download(kpn.data(), d_cnt.p, sizeof(uint32_t) * fb.K));
  {
    const int T = ((int)HW + RPCC_TILE - 1) / RPCC_TILE;
    const Book bk = make_book(fb.book.p, 1, T, fb.K);
    TRY(download(pn.data(), bk.label_cnt, sizeof(uint32_t) * fb.K));
  }
  std::vector<float> steps(fb.K, level_acc[level_num - 1]);
  for (int l = 0; l < fb.K; ++l) {
    int lev = 0;
    if (l == 0) lev = ground_level;
    else if (l == 1) lev = level_num - 1;
    else if (pn[l] < 30u) lev = level_num - 1;
    else for (int q = 0; q < level_num; ++q) if ((int)kpn[l] >= level_kp_num[q]) { lev = q; break; }
    RPCC_REQUIRE(lev >= 0 && lev < level_num, "ground_level out of range");
    if (l < Kref) salience[l] = lev;
    steps[l] = level_acc[lev];
  }
  *K_out = Kref;
  TRY(upload(d_step, steps.data(), steps.size() * sizeof(float)));
  return quantize_common(fb, H, W, d_step.as<float>(), 0.f, out, n_out);
}

extern "C" int rpcc_op_extract_contour(const int32_t* seg, int H, int W, int32_t* contour, int32_t* seq, int64_t* L_out) {
  RPCC_REQUIRE(seg && contour && seq && L_out, "null pointer");
  const size_t HW = (size_t)H * W;
  std::vector<float> zeros(HW, 0.f);
  FrameBook fb;
  TRY(fb.build(zeros.data(), seg, H, W, false));
  DevBuf zero_model, lut, sym, cb, sq;
  std::vector<float> zm((size_t)fb.K * 4, 0.f);
  TRY(upload(zero_model, zm.data(), zm.size() * sizeof(float)));
  TRY(lut.alloc(16));
  TRY(sym.alloc(HW * sizeof(int16_t)));
  TRY(cb.alloc((HW + 7) / 8));
  TRY(sq.alloc(HW * sizeof(uint16_t)));
  TRY(rpcc_quantize_pack_batch(fb.range.as<float>(), fb.labels.as<uint8_t>(), zero_model.as<float>(), lut.as<float>(), fb.book.p,
                               nullptr, 1.0f, 1, H, W, fb.K, sym.as<int16_t>(), HW, cb.as<uint8_t>(), sq.as<uint16_t>(), HW,
                               nullptr, nullptr, nullptr));
  std::vector<uint8_t> bits((HW + 7) / 8);
  std::vector<uint16_t> s16(fb.res.seq_count);
  TRY(download(bits.data(), cb.p, bits.size()));
  TRY(download(s16.data(), sq.p, s16.size() * sizeof(uint16_t)));
  for (size_t p = 0; p < HW; ++p) contour[p] = (bits[p >> 3] >> (7 - (p & 7))) & 1;
  for (size_t i = 0; i < s16.size(); ++i) seq[i] = s16[i];
  *L_out = (int64_t)s16.size();
  return RPCC_OK;
}

extern "C" int rpcc_op_recover_map(const int32_t* contour, const int32_t* seq, int64_t L, int H, int W, int32_t* seg_out) {
  RPCC_REQUIRE(contour && seq && seg_out && L >= 0, "bad argument");
  const size_t HW = (size_t)H * W;
  std::vector<uint8_t> bits((HW + 7) / 8, 0);
  for (size_t p = 0; p < HW; ++p) if (contour[p] != 0) bits[p >> 3] |= (uint8_t)(1u << (7 - (p & 7)));
  std::vector<uint16_t> s16((size_t)L);
  int kmax = 1;
  for (int64_t i = 0; i < L; ++i) {
    RPCC_REQUIRE(seq[i] >= 0 && seq[i] <= 253, "sequence label outside [0, 253]");
    s16[i] = (uint16_t)seq[i];
    kmax = seq[i] > kmax ? seq[i] : kmax;
  }
  const int K = kmax + 1;
  DevBuf d_bits, d_seq, d_cnt, d_sym, d_model, d_steps, d_lut, d_lab, d_rng, d_book, d_res;
  TRY(upload(d_bits, bits.data(), bits.size()));
  TRY(upload(d_seq, s16.data(), s16.size() * sizeof(uint16_t)));
  const uint32_t cnt = (uint32_t)L;
  TRY(upload(d_cnt, &cnt, sizeof(cnt)));
  std::vector<float> zm((size_t)K * 4, 0.f);
  std::vector<double> st((size_t)K, 1.0);
  std::vector<float> lutz(HW * 3, 0.f);
  TRY(upload(d_model, zm.data(), zm.size() * sizeof(float)));
  TRY(upload(d_steps, st.data(), st.size() * sizeof(double)));
  TRY(upload(d_lut, lutz.data(), lutz.size() * sizeof(float)));
  TRY(d_sym.alloc(HW * sizeof(int16_t)));
  TRY(check_cuda(cudaMemset(d_sym.p, 0, HW * sizeof(int16_t)), "memset"));
  TRY(d_lab.alloc(HW));
  TRY(d_rng.alloc(HW * sizeof(float)));
  TRY(d_book.alloc(rpcc_book_bytes(1, H, W, K)));
  TRY(d_res.alloc(sizeof(rpcc_frame_result)));
  TRY(rpcc_decode_batch(d_bits.as<uint8_t>(), d_seq.as<uint16_t>(), (size_t)L, d_cnt.as<uint32_t>(), d_sym.as<int16_t>(), HW,
                        nullptr, d_model.as<float>(), d_steps.as<double>(), d_lut.as<float>(), 1, H, W, K, d_lab.as<uint8_t>(),
                        d_rng.as<float>(), nullptr, d_book.p, d_res.as<rpcc_frame_result>(), nullptr));
  std::vector<uint8_t> lab(HW);
  TRY(download(lab.data(), d_lab.p, HW));
  for (size_t p = 0; p < HW; ++p) seg_out[p] = lab[p];
  return RPCC_OK;
}

extern "C" int rpcc_op_furthest_point_sample(const float* points, int B, int n, int m, int32_t* idx_out) {
  RPCC_REQUIRE(points && idx_out && B >= 1 && n >= 1 && m >= 1, "bad argument");
  DevBuf d_pts, d_tmp, d_idx;
  TRY(upload(d_pts, points, sizeof(float) * 3 * (size_t)B * n));
  TRY(d_tmp.alloc(sizeof(float) * (size_t)B * n));
  TRY(d_idx.alloc(sizeof(int32_t) * (size_t)B * m));
  TRY(rpcc_fps_batch(d_pts.as<float>(), B, n, m, d_tmp.as<float>(), d_idx.as<int32_t>(), nullptr));
  return download(idx_out, d_idx.p, sizeof(int32_t) * (size_t)B * m);
}

extern "C" int rpcc_op_segment(const float* range, const float* lut, const float* ground, int H, int W, int m,
                               float ground_thr, int32_t* seg_out, int32_t* center_idx_out) {
  RPCC_REQUIRE(range && lut && ground && seg_out, "null pointer");
  const size_t HW = (size_t)H * W;
  DevBuf d_rng, d_lut, d_g, d_ci, d_c, d_lab, d_book;
  TRY(upload(d_rng, range, HW * sizeof(float)));
  TRY(upload(d_lut, lut, HW * 3 * sizeof(float)));
  TRY(upload(d_g, ground, 4 * sizeof(float)));
  TRY(d_ci.alloc(sizeof(int32_t) * m));
  TRY(d_c.alloc(sizeof(float) * 3 * m));
  TRY(d_lab.alloc(HW));
  TRY(d_book.alloc(rpcc_book_bytes(1, H, W, m + 2)));
  TRY(rpcc_segment_fps_batch(d_rng.as<float>(), d_lut.as<float>(), d_g.as<float>(), 1, H, W, m, ground_thr, d_ci.as<int32_t>(),
                             d_c.as<float>(), nullptr));
  TRY(rpcc_assign_labels_batch(d_rng.as<float>(), d_lut.as<float>(), d_g.as<float>(), d_c.as<float>(), 1, H, W, m,
                               d_lab.as<uint8_t>(), d_book.p, nullptr));
  std::vector<uint8_t> lab(HW);
  TRY(download(lab.data(), d_lab.p, HW));
  for (size_t p = 0; p < HW; ++p) seg_out[p] = lab[p];
  if (center_idx_out) TRY(download(center_idx_out, d_ci.p, sizeof(int32_t) * m));
  return RPCC_OK;
}

extern "C" int rpcc_op_segment_dbscan(const float* range, const float* lut, const float* ground, int H, int W, double hfov,
                                      double vmax, double vmin, double eps, int min_points, int cluster_num, float ground_thr,
                                      int32_t* seg_out, uint32_t* exhaustive_out, uint32_t* clusters_out) {
  RPCC_REQUIRE(range && lut && ground && seg_out, "null pointer");
  RPCC_REQUIRE(H >= 2 && W >= 1, "bad sizes");
  const size_t HW = (size_t)H * W;
  DevBuf d_rng, d_lut, d_g, d_lab, d_ws;
  TRY(upload(d_rng, range, HW * sizeof(float)));
  TRY(upload(d_lut, lut, HW * 3 * sizeof(float)));
  TRY(upload(d_g, ground, 4 * sizeof(float)));
  TRY(d_lab.alloc(HW));
  TRY(d_ws.alloc(rpcc_dbscan_workspace_bytes(1, H, W)));
  TRY(rpcc_dbscan_segment_batch(d_rng.as<float>(), d_lut.as<float>(), d_g.as<float>(), 1, H, W, hfov, vmax, vmin, eps,
                                min_points, cluster_num, ground_thr, d_lab.as<uint8_t>(), d_ws.p, nullptr));
  std::vector<uint8_t> lab(HW);
  TRY(download(lab.data(), d_lab.p, HW));
  for (size_t p = 0; p < HW; ++p) seg_out[p] = lab[p];
  uint32_t counts[2];
  TRY(download(counts, d_ws.p, sizeof(counts)));   // the workspace starts with [fallback][clusters] for B = 1
  if (exhaustive_out) *exhaustive_out = counts[0];
  if (clusters_out) *clusters_out = counts[1];
  return RPCC_OK;
}

extern "C" int rpcc_op_chamfer(const float* xyz1, int n, const float* xyz2, int m, float* dist1, int32_t* idx1, float* dist2,
                               int32_t* idx2) {
  RPCC_REQUIRE(xyz1 && xyz2 && dist1 && idx1 && dist2 && idx2 && n >= 1 && m >= 1, "bad argument");
  DevBuf a, b, d1, i1, d2, i2, scr;
  TRY(upload(a, xyz1, sizeof(float) * 3 * (size_t)n));
  TRY(upload(b, xyz2, sizeof(float) * 3 * (size_t)m));
  TRY(d1.alloc(sizeof(float) * n)); TRY(i1.alloc(sizeof(int32_t) * n));
  TRY(d2.alloc(sizeof(float) * m)); TRY(i2.alloc(sizeof(int32_t) * m));
  TRY(scr.alloc(sizeof(unsigned long long) * ((size_t)n + m)));
  TRY(rpcc_chamfer_batch(a.as<float>(), n, b.as<float>(), m, d1.as<float>(), i1.as<int32_t>(), d2.as<float>(), i2.as<int32_t>(),
                         scr.p, nullptr));
  TRY(download(dist1, d1.p, sizeof(float) * n)); TRY(download(idx1, i1.p, sizeof(int32_t) * n));
  TRY(download(dist2, d2.p, sizeof(float) * m)); TRY(download(idx2, i2.p, sizeof(int32_t) * m));
  return RPCC_OK;
}

extern "C" int rpcc_op_range_to_xyz(const float* range, const float* lut, int H, int W, float* xyz) {
  RPCC_REQUIRE(range && lut && xyz, "null pointer");
  const size_t HW = (size_t)H * W;
  DevBuf d_r, d_l, d_x;
  TRY(upload(d_r, range, HW * sizeof(float)));
  TRY(upload(d_l, lut, HW * 3 * sizeof(float)));
  TRY(d_x.alloc(HW * 3 * sizeof(float)));
  TRY(rpcc_range_to_xyz_batch(d_r.as<float>(), d_l.as<float>(), 1, (int)HW, d_x.as<float>(), nullptr));
  return download(xyz, d_x.p, HW * 3 * sizeof(float));
}

extern "C" int rpcc_op_ground_fit(const float* range, const float* lut, int H, int W, uint64_t seed, float* ground_out) {
  RPCC_REQUIRE(range && lut && ground_out, "null pointer");
  const size_t HW = (size_t)H * W;
  DevBuf d_r, d_l, d_g;
  TRY(upload(d_r, range, HW * sizeof(float)));
  TRY(upload(d_l, lut, HW * 3 * sizeof(float)));
  TRY(d_g.alloc(4 * sizeof(float)));
  TRY(rpcc_ground_fit_batch(d_r.as<float>(), d_l.as<float>(), 1, H, W, seed, nullptr, d_g.as<float>(), nullptr));
  return download(ground_out, d_g.p, 4 * sizeof(float));
}

// QuantizationModule.dequantize_residual (utils/compress_utils.py:114-132): symbols (n,) i16 label-major,
// seg (H,W) i32, steps [K] f64 (K > max label) -> residual (H,W) f32.  *consumed = symbols the label map asks for.
extern "C" int rpcc_op_dequantize(const int16_t* symbols, int64_t n, const int32_t* seg, int H, int W, const double* steps,
                                  int K, float* residual_out, int64_t* consumed) {
  RPCC_REQUIRE(symbols && seg && steps && residual_out, "null pointer");
  const size_t HW = (size_t)H * W;
  std::vector<uint8_t> lab;
  int kmax = 0;
  TRY(narrow_labels(seg, HW, lab, &kmax));
  RPCC_REQUIRE(K > kmax && K >= 2, "steps must cover every label");
  DevBuf d_lab, d_sym, d_cnt, d_model, d_steps, d_lut, d_rng, d_book, d_res;
  TRY(upload(d_lab, lab.data(), HW));
  TRY(upload(d_sym, symbols, (size_t)(n > 0 ? n : 1) * sizeof(int16_t)));
  const uint32_t cnt = (uint32_t)n;
  TRY(upload(d_cnt, &cnt, sizeof(cnt)));
  std::vector<float> zm((size_t)K * 4, 0.f);
  std::vector<float> lutz(HW * 3, 0.f);
  TRY(upload(d_model, zm.data(), zm.size() * sizeof(float)));
  TRY(upload(d_steps, steps, sizeof(double) * K));
  TRY(upload(d_lut, lutz.data(), lutz.size() * sizeof(float)));
  TRY(d_rng.alloc(HW * sizeof(float)));
  TRY(d_book.alloc(rpcc_book_bytes(1, H, W, K)));
  TRY(d_res.alloc(sizeof(rpcc_frame_result)));
  TRY(rpcc_dequantize_batch(d_lab.as<uint8_t>(), d_sym.as<int16_t>(), (size_t)n, d_cnt.as<uint32_t>(), d_model.as<float>(),
                            d_steps.as<double>(), d_lut.as<float>(), 1, H, W, K, d_rng.as<float>(), nullptr, d_book.p,
                            d_res.as<rpcc_frame_result>(), 0, nullptr));
  rpcc_frame_result r{};
  TRY(download(&r, d_res.p, sizeof(r)));
  if (consumed) *consumed = r.sym_count;
  return download(residual_out, d_rng.p, HW * sizeof(float));
}

extern "C" int rpcc_op_plane_modeling(const float* range, const int32_t* seg, const float* lut, int H, int W,
                                      float angle_threshold_deg, uint64_t seed, float* rows_out, int cap_rows, int* rows) {
  RPCC_REQUIRE(range && seg && lut && rows_out && rows, "null pointer");
  const size_t HW = (size_t)H * W;
  FrameBook fb;
  TRY(fb.build(range, seg, H, W, true));
  RPCC_REQUIRE(cap_rows >= fb.K - 1, "rows_out too small");
  DevBuf d_lut, d_order;
  TRY(upload(d_lut, lut, HW * 3 * sizeof(float)));
  TRY(d_order.alloc(HW * sizeof(uint32_t)));
  TRY(rpcc_label_order_batch(fb.labels.as<uint8_t>(), fb.book.p, 1, H, W, fb.K, d_order.as<uint32_t>(), HW, nullptr));
  TRY(rpcc_plane_model_batch(fb.range.as<float>(), d_lut.as<float>(), d_order.as<uint32_t>(), HW, fb.book.p, 1, H, W, fb.K,
                             30, 0.1f, 4, 10, angle_threshold_deg, seed, nullptr, fb.model.as<float>(), nullptr));
  *rows = fb.K - 1;
  return download(rows_out, fb.model.as<float>() + 4, sizeof(float) * 4 * (size_t)(fb.K - 1));
}

// The intensity section of one frame (rpcc_intensity_owner_batch / _pack_batch / _unpack_batch with B = 1).
extern "C" int rpcc_op_intensity_owner(const float* points, int64_t n, int H, int W, float hfov, float vmax, float vmin,
                                       uint32_t* owner_out, float* intensity_out) {
  RPCC_REQUIRE(points || n == 0, "null pointer");
  RPCC_REQUIRE(intensity_out && n >= 0, "bad argument");
  const size_t HW = (size_t)H * W;
  DevBuf d_pts, d_off, d_rng, d_scr, d_own, d_int;
  TRY(upload(d_pts, points, sizeof(float) * 4 * (size_t)n));
  const int64_t off[2] = {0, n};
  TRY(upload(d_off, off, sizeof(off)));
  TRY(d_rng.alloc(sizeof(float) * HW));
  TRY(d_scr.alloc(sizeof(int32_t) * 4));
  TRY(d_own.alloc(sizeof(uint32_t) * HW));
  TRY(d_int.alloc(sizeof(float) * HW));
  TRY(rpcc_project_batch(d_pts.as<float>(), 4, d_off.as<int64_t>(), 1, H, W, hfov, vmax, vmin, d_rng.as<float>(),
                         d_scr.as<int32_t>(), nullptr));
  TRY(rpcc_intensity_owner_batch(d_pts.as<float>(), d_off.as<int64_t>(), 1, H, W, hfov, vmax, vmin, d_rng.as<float>(),
                                 d_scr.as<int32_t>(), d_own.as<uint32_t>(), d_int.as<float>(), nullptr));
  if (owner_out) TRY(download(owner_out, d_own.p, sizeof(uint32_t) * HW));
  return download(intensity_out, d_int.p, sizeof(float) * HW);
}

extern "C" int rpcc_op_intensity_pack(const float* intensity, const float* range, int H, int W, double step, uint8_t* out,
                                      int64_t* n_out, uint32_t* flags_out) {
  RPCC_REQUIRE(intensity && range && out && n_out, "null pointer");
  const size_t HW = (size_t)H * W;
  int64_t n = 0;
  for (size_t i = 0; i < HW; ++i) n += range[i] != 0.f;
  DevBuf d_int, d_rng, d_base, d_out, d_res;
  TRY(upload(d_int, intensity, sizeof(float) * HW));
  TRY(upload(d_rng, range, sizeof(float) * HW));
  const uint64_t base[2] = {0, (uint64_t)n};
  TRY(upload(d_base, base, sizeof(base)));
  TRY(d_out.alloc((size_t)n));
  const rpcc_frame_result r0{};
  TRY(upload(d_res, &r0, sizeof(r0)));
  TRY(rpcc_intensity_pack_batch(d_int.as<float>(), d_rng.as<float>(), 1, H, W, step, d_base.as<uint64_t>(),
                                d_out.as<uint8_t>(), d_res.as<rpcc_frame_result>(), nullptr));
  rpcc_frame_result r{};
  TRY(download(&r, d_res.p, sizeof(r)));
  *n_out = n;
  if (flags_out) *flags_out = r.flags;
  return download(out, d_out.p, (size_t)n);
}

extern "C" int rpcc_op_intensity_unpack(const uint8_t* q, int64_t n, const int32_t* seg, int H, int W, double step,
                                        float* intensity_out) {
  RPCC_REQUIRE((q || n == 0) && seg && intensity_out, "null pointer");
  const size_t HW = (size_t)H * W;
  std::vector<uint8_t> empty(HW);
  int64_t want = 0;
  for (size_t i = 0; i < HW; ++i) { empty[i] = seg[i] == 1 ? 1 : 0; want += seg[i] != 1; }
  if (n != want) {
    set_error("rpcc_op_intensity_unpack: intensity section holds %lld bytes, the label map has %lld non-empty pixels",
              (long long)n, (long long)want);
    return RPCC_ERR_ARG;
  }
  DevBuf d_lab, d_q, d_base, d_int;
  TRY(upload(d_lab, empty.data(), HW));
  TRY(upload(d_q, q, (size_t)n));
  const uint64_t base[2] = {0, (uint64_t)n};
  TRY(upload(d_base, base, sizeof(base)));
  TRY(d_int.alloc(sizeof(float) * HW));
  TRY(rpcc_intensity_unpack_batch(d_lab.as<uint8_t>(), d_q.as<uint8_t>(), d_base.as<uint64_t>(), 1, H, W, step,
                                  d_int.as<float>(), nullptr));
  return download(intensity_out, d_int.p, sizeof(float) * HW);
}
