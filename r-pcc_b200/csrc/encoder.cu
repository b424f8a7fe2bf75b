// encoder.cu -- the batched encoder: project -> [ground fit] -> FPS -> labels (or DBSCAN -> label statistics) ->
// [key points] -> point models -> quantise + pack, B frames per call, plus the host-buffer entry point that
// pipelines H2D copy / kernels / D2H copy over several stream slots.
//
// This is what tools/compress_datalist.py's per-frame closure (reference
// tools/compress_datalist.py:91-134: dataset[index] -> segment -> cluster_modeling ->
// intra_predict -> quantize_residual -> compress_point_cloud up to, not including, the entropy
// coder) becomes when many frames are processed per launch.  The entropy coder (bz2/deflate) stays
// on host threads, fed by the sections this returns.
#include <math.h>
#include <string.h>

#include <new>
#include <vector>

#include "book.cuh"

using namespace rpcc;

namespace rpcc {
// quantize.cu; trusted_labels: the labels come from assign_labels_kernel and are < K by construction
template <typename SymT>
int quantize_pack_launch(const float* range, const uint8_t* labels, const float* model, const float* lut, void* book,
                         const float* step_per_label, float step, int B, int H, int W, int K, SymT* symbols,
                         size_t sym_stride, uint8_t* contour_bits, uint16_t* seq, size_t seq_stride,
                         const uint64_t* sym_base, const uint64_t* seq_base, void* stream, bool trusted_labels);
// fps.cu: owner receives the per-pixel owner hints; assign.cu: hinted reads them from labels and overwrites them
int segment_fps_launch(const float* range, const float* lut, const float* ground, int B, int H, int W, int m, float ground_thr,
                       int32_t* center_idx, float* centers, uint8_t* owner, cudaStream_t st);
int assign_labels_launch(const float* range, const float* lut, const float* ground, const float* centers, int B, int H, int W,
                         int m, uint8_t* labels, void* book, cudaStream_t st, bool hinted);
}

namespace {

struct Slot {
  cudaStream_t stream = nullptr;
  cudaEvent_t done = nullptr;   // all work of the slot's current chunk (including D2H of results)
  float* points = nullptr;      // host path staging [max_points][4]
  int64_t* offsets = nullptr;   // [max_batch+1]
  float* range = nullptr;       // [B][HW]
  int32_t* scratch = nullptr;   // [B][4]
  float* ground = nullptr;      // [B][4]
  uint64_t* keys = nullptr;     // [B] caller-supplied RANSAC keys of the chunk (host path staging)
  int32_t* center_idx = nullptr;
  float* centers = nullptr;
  uint8_t* labels = nullptr;
  void* book = nullptr;
  float* model = nullptr;       // [B][K][4]
  rpcc_frame_result* results = nullptr;
  uint64_t* sym_base = nullptr; // [B+1]
  uint64_t* seq_base = nullptr; // [B+1]
  int16_t* symbols = nullptr;   // packed, capacity B*HW
  uint16_t* seq = nullptr;      // packed, capacity B*HW
  uint8_t* contour = nullptr;   // [B][cbytes]
  uint8_t* key_points = nullptr;
  uint8_t* salience = nullptr;
  float* step_per_label = nullptr;
  uint32_t* kp_cnt = nullptr;
  uint32_t* order = nullptr;    // plane modelling: pixels in label-major order [B][HW]
  void* db_ws = nullptr;        // segment_method 1: rpcc_dbscan_segment_batch's workspace
  // cfg.eval: decode what was just written and compare (tools/compress_datalist.py:166-199)
  uint8_t* ev_labels = nullptr; // [B][HW]
  float* ev_range = nullptr;    // [B][HW]
  void* ev_book = nullptr;
  rpcc_frame_result* ev_results = nullptr;
  double* ev_steps = nullptr;   // [B][K]
  double* ev_metrics = nullptr; // [B][RPCC_EVAL_COLS]
  void* ev_ws = nullptr;
  // cfg.eval == 2: point-to-plane PSNR (normals.cu)
  float* ev_nref = nullptr;     // [B][HW][3] normals of the encoded frame
  float* ev_nrec = nullptr;     // [B][HW][3] normals of the reconstruction
  double* ev_p2 = nullptr;      // [B][RPCC_P2PLANE_COLS]
  void* ev_nws = nullptr;
  void* ev_p2ws = nullptr;
  // cfg.intensity_step > 0: the intensity section (project.cu owner pass, intensity.cu)
  uint32_t* int_owner = nullptr; // [B][HW]
  float* inten = nullptr;        // [B][HW] the owners' intensities
  uint8_t* int_stream = nullptr; // packed at sym_base, capacity B*HW
  // pinned host mirrors for the small per-chunk tables
  rpcc_frame_result* h_results = nullptr;
  int64_t* h_offsets = nullptr;
  int last_B = 0;
  // optional per-stage timing (bench.py roofline): ring of event sets, one set per chain call
  cudaEvent_t* ev = nullptr;    // [kEvRing][kStages + 1]
  int* ev_frames = nullptr;     // frames of each recorded call
  int ev_head = 0, ev_count = 0;
};

constexpr int kSlots = 3;
constexpr int kStages = 8;     // project, ground, fps, assign, keypoints, model, quantize, eval
constexpr int kEvRing = 256;   // chain calls per slot whose stage events are kept

}  // namespace

struct rpcc_encoder {
  rpcc_encoder_config cfg;
  int HW, K, T, cbytes;
  int host_chunk;   // frames per pipeline stage of encode_host
  float hfov, vmax, vmin;
  float level_acc[8];
  float* lut = nullptr;
  double* dacc8 = nullptr;      // level_dacc on the device (cfg.eval, non-uniform)
  Slot slot[kSlots];
  uint64_t ground_seed = 0x5EEDull;
  bool profiling = false;
};

namespace {

template <typename Tp>
int dev_alloc(Tp** p, size_t count) {
  void* q = nullptr;
  RPCC_CUDA(cudaMalloc(&q, count * sizeof(Tp) > 0 ? count * sizeof(Tp) : 16));
  *p = static_cast<Tp*>(q);
  return RPCC_OK;
}

int alloc_slot(rpcc_encoder* e, Slot& s) {
  const size_t B = e->cfg.max_batch, HW = e->HW, K = e->K, m = e->cfg.cluster_num;
  RPCC_CUDA(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
  RPCC_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
  int rc;
#define A(ptr, n) if ((rc = dev_alloc(&s.ptr, (n))) != RPCC_OK) return rc
  A(points, (size_t)e->cfg.max_points * 4);
  A(offsets, B + 1);
  A(range, B * HW);
  A(scratch, B * 4);
  A(ground, B * 4);
  A(keys, B);
  A(center_idx, B * m);
  A(centers, B * m * 3);
  A(labels, B * HW);
  A(model, B * K * 4);
  A(results, B);
  A(sym_base, B + 1);
  A(seq_base, B + 1);
  A(symbols, B * HW);
  A(seq, B * HW);
  A(contour, B * (size_t)e->cbytes);
  if (e->cfg.nonuniform) {
    A(key_points, B * HW);
    A(salience, B * K);
    A(step_per_label, B * K);
    A(kp_cnt, B * K);
  }
  if (e->cfg.model_method == 1) { A(order, B * HW); }
  if (e->cfg.intensity_step > 0) {
    A(int_owner, B * HW);
    A(inten, B * HW);
    A(int_stream, B * HW);
  }
  if (e->cfg.segment_method == 1) RPCC_CUDA(cudaMalloc(&s.db_ws, rpcc_dbscan_workspace_bytes((int)B, e->cfg.H, e->cfg.W)));
  if (e->cfg.eval) {
    A(ev_labels, B * HW);
    A(ev_range, B * HW);
    A(ev_results, B);
    A(ev_steps, B * K);
    A(ev_metrics, B * RPCC_EVAL_COLS);
    void* p = nullptr;
    RPCC_CUDA(cudaMalloc(&p, book_bytes((int)B, e->T, (int)K)));
    s.ev_book = p;
    RPCC_CUDA(cudaMalloc(&s.ev_ws, rpcc_eval_workspace_bytes((int)B, e->cfg.H, e->cfg.W)));
    if (e->cfg.eval == 2) {
      A(ev_nref, B * HW * 3);
      A(ev_nrec, B * HW * 3);
      A(ev_p2, B * RPCC_P2PLANE_COLS);
      RPCC_CUDA(cudaMalloc(&s.ev_nws, rpcc_normals_workspace_bytes((int)B, e->cfg.H, e->cfg.W)));
      RPCC_CUDA(cudaMalloc(&s.ev_p2ws, rpcc_p2plane_workspace_bytes((int)B, e->cfg.H, e->cfg.W)));
    }
  }
#undef A
  void* bk = nullptr;
  RPCC_CUDA(cudaMalloc(&bk, book_bytes((int)B, e->T, (int)K)));
  s.book = bk;
  RPCC_CUDA(cudaMallocHost(reinterpret_cast<void**>(&s.h_results), sizeof(rpcc_frame_result) * B));
  RPCC_CUDA(cudaMallocHost(reinterpret_cast<void**>(&s.h_offsets), sizeof(int64_t) * (B + 1)));
  return RPCC_OK;
}

void free_slot(Slot& s) {
  void* ptrs[] = {s.points, s.offsets, s.range, s.scratch, s.ground, s.keys, s.center_idx, s.centers, s.labels, s.book, s.model,
                  s.results, s.sym_base, s.seq_base, s.symbols, s.seq, s.contour, s.key_points, s.salience,
                  s.step_per_label, s.kp_cnt, s.order, s.db_ws, s.ev_labels, s.ev_range, s.ev_book,
                  s.ev_results, s.ev_steps, s.ev_metrics, s.ev_ws, s.ev_nref, s.ev_nrec, s.ev_p2, s.ev_nws, s.ev_p2ws,
                  s.int_owner, s.inten, s.int_stream};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (s.ev) {
    for (int i = 0; i < kEvRing * (kStages + 1); ++i) if (s.ev[i]) cudaEventDestroy(s.ev[i]);
    delete[] s.ev;
    delete[] s.ev_frames;
  }
  if (s.h_results) cudaFreeHost(s.h_results);
  if (s.h_offsets) cudaFreeHost(s.h_offsets);
  if (s.done) cudaEventDestroy(s.done);
  if (s.stream) cudaStreamDestroy(s.stream);
  s = Slot();
}

// the kernel chain for B frames whose points are already on the device; frame_keys: device [B] or NULL (key 0: the
// deterministic RANSACs then depend on the frame's content alone)
int run_chain(rpcc_encoder* e, Slot& s, const float* points, int stride, const int64_t* offsets, int B,
              const float* ground_in, const uint64_t* frame_keys) {
  const rpcc_encoder_config& c = e->cfg;
  void* st = s.stream;
  int rc;
  RPCC_REQUIRE(stride == 4 || !(c.intensity_step > 0), "an intensity encoder needs stride-4 points (x, y, z, intensity)");
  cudaEvent_t* ev = nullptr;
  if (e->profiling && s.ev) {
    ev = s.ev + (size_t)s.ev_head * (kStages + 1);
    s.ev_frames[s.ev_head] = B;
    s.ev_head = (s.ev_head + 1) % kEvRing;
    if (s.ev_count < kEvRing) ++s.ev_count;
  }
#define MARK(i) do { if (ev) RPCC_CUDA(cudaEventRecord(ev[i], s.stream)); } while (0)
  MARK(0);
  if ((rc = rpcc_project_batch(points, stride, offsets, B, c.H, c.W, e->hfov, e->vmax, e->vmin, s.range, s.scratch, st))) return rc;
  if (c.intensity_step > 0) {
    if ((rc = rpcc_intensity_owner_batch(points, offsets, B, c.H, c.W, e->hfov, e->vmax, e->vmin, s.range, s.scratch,
                                         s.int_owner, s.inten, st))) return rc;
  }
  MARK(1);
  if (ground_in) {
    if (ground_in != s.ground)
      RPCC_CUDA(cudaMemcpyAsync(s.ground, ground_in, sizeof(float) * 4 * (size_t)B, cudaMemcpyDefault, s.stream));
  } else {
    if ((rc = rpcc_ground_fit_batch(s.range, e->lut, B, c.H, c.W, e->ground_seed, frame_keys, s.ground, st))) return rc;
  }
  MARK(2);
  if (c.segment_method == 1) {
    // DBSCAN's time goes to the "fps" stage slot, the label statistics to "assign"
    if ((rc = rpcc_dbscan_segment_batch(s.range, e->lut, s.ground, B, c.H, c.W, c.hfov, c.vmax, c.vmin, c.dbscan_eps,
                                        c.dbscan_min_points, c.cluster_num, c.ground_threshold, s.labels, s.db_ws, st))) return rc;
    MARK(3);
    if ((rc = rpcc_label_stats_batch(s.range, s.labels, B, c.H, c.W, e->K, s.book, st))) return rc;
  } else {
    // the FPS rounds leave, per pixel, which centre is its nearest (owner hints, fps.cu) in the label buffer; the label
    // assignment evaluates that one centre where there is a hint and overwrites the byte with the label
    if ((rc = segment_fps_launch(s.range, e->lut, s.ground, B, c.H, c.W, c.cluster_num, c.ground_threshold,
                                 s.center_idx, s.centers, s.labels, s.stream))) return rc;
    MARK(3);
    if ((rc = assign_labels_launch(s.range, e->lut, s.ground, s.centers, B, c.H, c.W, c.cluster_num, s.labels, s.book, s.stream,
                                   true))) return rc;
  }
  MARK(4);
  if (c.nonuniform) {
    if ((rc = rpcc_keypoints_salience_batch(s.range, s.labels, s.book, B, c.H, c.W, e->K, c.feature_region, c.segments,
                                            c.sharp_num, c.less_sharp_num, c.flat_num, c.level_kp_num, e->level_acc,
                                            c.level_num, c.ground_level, s.key_points, nullptr, s.salience,
                                            s.step_per_label, s.kp_cnt, st))) return rc;
  }
  MARK(5);
  if ((rc = rpcc_point_model_batch(s.range, s.labels, s.ground, s.book, B, c.H, c.W, e->K, s.model, s.results, st))) return rc;
  if (c.model_method == 1) {
    if ((rc = rpcc_label_order_batch(s.labels, s.book, B, c.H, c.W, e->K, s.order, (size_t)e->HW, st))) return rc;
    if ((rc = rpcc_plane_model_batch(s.range, e->lut, s.order, (size_t)e->HW, s.book, B, c.H, c.W, e->K, 30, 0.1f, 4, 10,
                                     c.plane_angle_threshold, e->ground_seed ^ 0x9E3779B97F4A7C15ull, frame_keys, s.model, st))) return rc;
  }
  if ((rc = rpcc_frame_offsets_batch(s.results, B, s.sym_base, s.seq_base, st))) return rc;
  MARK(6);
  if ((rc = quantize_pack_launch<int16_t>(s.range, s.labels, s.model, e->lut, s.book, c.nonuniform ? s.step_per_label : nullptr,
                                          (float)c.step, B, c.H, c.W, e->K, s.symbols, 0, s.contour, s.seq, 0, s.sym_base,
                                          s.seq_base, st, true))) return rc;
  if (c.intensity_step > 0 &&
      (rc = rpcc_intensity_pack_batch(s.inten, s.range, B, c.H, c.W, c.intensity_step, s.sym_base, s.int_stream, s.results, st)))
    return rc;
  MARK(7);
  if (c.eval) {
    // decode the sections exactly as they go to the file, then compare with the frame that was encoded
    if ((rc = rpcc_eval_steps_batch(c.nonuniform ? s.salience : nullptr, B, e->K, c.step, e->dacc8, s.ev_steps, st))) return rc;
    if ((rc = rpcc_decode_packed_batch(s.contour, s.seq, s.seq_base, s.symbols, s.sym_base, s.model, s.ev_steps, e->lut, B,
                                       c.H, c.W, e->K, s.ev_labels, s.ev_range, nullptr, s.ev_book, s.ev_results, st))) return rc;
    if ((rc = rpcc_eval_batch(s.range, s.ev_range, e->lut, s.labels, s.ev_labels, B, c.H, c.W, c.hfov, c.vmax, c.vmin,
                              c.eval_threshold_sq, nullptr, nullptr, s.ev_metrics, s.ev_ws, st))) return rc;
    if (c.eval == 2) {
      if ((rc = rpcc_normals_batch(s.range, e->lut, B, c.H, c.W, c.hfov, c.vmax, c.vmin, RPCC_NORMAL_KNN, RPCC_NORMAL_RADIUS,
                                   s.ev_nref, s.ev_nws, st))) return rc;
      if ((rc = rpcc_normals_batch(s.ev_range, e->lut, B, c.H, c.W, c.hfov, c.vmax, c.vmin, RPCC_NORMAL_KNN, RPCC_NORMAL_RADIUS,
                                   s.ev_nrec, s.ev_nws, st))) return rc;
      if ((rc = rpcc_p2plane_batch(s.range, s.ev_range, e->lut, s.ev_nref, s.ev_nrec, B, c.H, c.W, c.hfov, c.vmax, c.vmin,
                                   s.ev_p2, s.ev_p2ws, st))) return rc;
    }
  }
  MARK(8);
#undef MARK
  s.last_B = B;
  return RPCC_OK;
}

}  // namespace

extern "C" int rpcc_encoder_create(const rpcc_encoder_config* cfg, rpcc_encoder** out) {
  RPCC_REQUIRE(cfg && out, "null pointer");
  RPCC_REQUIRE(cfg->H >= 2 && cfg->W >= 1 && (size_t)cfg->H * cfg->W >= 1024, "range image must have >= 1024 pixels");
  RPCC_REQUIRE(cfg->cluster_num >= 1 && cfg->cluster_num + 2 <= 254, "cluster_num must be in [1, 252]");
  RPCC_REQUIRE(cfg->max_batch >= 1 && cfg->max_batch <= 65535, "max_batch must be in [1, 65535]");
  RPCC_REQUIRE(cfg->max_points >= 1, "max_points must be positive");
  RPCC_REQUIRE(cfg->step > 0, "step must be positive");
  RPCC_REQUIRE(!cfg->nonuniform || (cfg->level_num >= 1 && cfg->level_num <= 8), "1..8 salience levels");
  RPCC_REQUIRE(cfg->model_method == 0 || cfg->model_method == 1, "model_method must be 0 (point) or 1 (plane)");
  RPCC_REQUIRE(cfg->segment_method == 0 || cfg->segment_method == 1, "segment_method must be 0 (FPS) or 1 (DBSCAN)");
  RPCC_REQUIRE(cfg->segment_method == 0 || cfg->dbscan_eps > 0, "DBSCAN eps must be positive");
  RPCC_REQUIRE(cfg->segment_method == 0 || cfg->dbscan_min_points >= 1, "DBSCAN min_points must be at least 1");
  RPCC_REQUIRE(cfg->segment_method == 0 || fabs(cfg->hfov - 6.283185307179586) < 1e-6, "DBSCAN needs a 360-degree sensor");
  RPCC_REQUIRE(cfg->intensity_step >= 0, "intensity_step must be 0 (off) or positive");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    set_error("rpcc_encoder_create: no CUDA device (this library has no CPU fallback)");
    return RPCC_ERR_NO_DEVICE;
  }
  RPCC_CUDA(cudaSetDevice(cfg->device));
  rpcc_encoder* e = new (std::nothrow) rpcc_encoder();
  RPCC_REQUIRE(e != nullptr, "out of host memory");
  e->cfg = *cfg;
  e->HW = cfg->H * cfg->W;
  e->K = cfg->cluster_num + 2;
  e->T = (e->HW + RPCC_TILE - 1) / RPCC_TILE;
  e->cbytes = (e->HW + 7) / 8;
  {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device) != cudaSuccess) { cudaGetLastError(); sms = 0; }
    // default: three quarters of a frame per SM -- measured on 1184-frame calls (profiles/r02k_host_chunk.txt): 74 or 111
    // frames per stage 37.0 k frames/s, 148: 36.3 k, 296: 34.1 k (the last stage's kernels and download run with the
    // upload link idle, so short stages cost less at the end of a call)
    const int want = cfg->host_chunk > 0 ? cfg->host_chunk : (sms > 0 ? (3 * sms) / 4 : cfg->max_batch);
    e->host_chunk = want < cfg->max_batch ? want : cfg->max_batch;
  }
  // the pybind boundary narrows the Python doubles to float (cpp_modules.cpp:427-428)
  e->hfov = (float)cfg->hfov; e->vmax = (float)cfg->vmax; e->vmin = (float)cfg->vmin;
  // QuantizationModule.__init__: acc = base + delta in f64 (utils/compress_utils.py:48), narrowed to
  // f32 when nonuniform_quantize receives it (py::array_t<float>, cpp_modules.cpp:339)
  for (int q = 0; q < 8; ++q) e->level_acc[q] = q < cfg->level_num ? (float)(cfg->step + cfg->level_dacc[q]) : 0.f;
  int rc = RPCC_OK;
  std::vector<float> lut((size_t)e->HW * 3);
  rc = rpcc_transform_map(cfg->H, cfg->W, cfg->hfov, cfg->vmax, cfg->vmin, lut.data());
  if (rc == RPCC_OK) rc = dev_alloc(&e->lut, lut.size());
  if (rc == RPCC_OK) rc = check_cuda(cudaMemcpy(e->lut, lut.data(), lut.size() * sizeof(float), cudaMemcpyHostToDevice), "lut upload");
  if (rc == RPCC_OK && cfg->eval) {
    rc = dev_alloc(&e->dacc8, 8);
    if (rc == RPCC_OK) rc = check_cuda(cudaMemcpy(e->dacc8, cfg->level_dacc, 8 * sizeof(double), cudaMemcpyHostToDevice), "dacc upload");
  }
  for (int i = 0; i < kSlots && rc == RPCC_OK; ++i) rc = alloc_slot(e, e->slot[i]);
  if (rc != RPCC_OK) { rpcc_encoder_destroy(e); return rc; }
  *out = e;
  return RPCC_OK;
}

extern "C" void rpcc_encoder_destroy(rpcc_encoder* e) {
  if (!e) return;
  cudaSetDevice(e->cfg.device);
  for (int i = 0; i < kSlots; ++i) free_slot(e->slot[i]);
  if (e->lut) cudaFree(e->lut);
  if (e->dacc8) cudaFree(e->dacc8);
  delete e;
}

extern "C" int rpcc_encoder_slots(void) { return kSlots; }

// Per-stage device timing with CUDA events on the slots' own streams.  enable=1 starts a fresh
// recording (events are recorded between the stages of every chain call, at most kEvRing calls per
// slot are kept).  rpcc_encoder_stage_times synchronises and returns, per stage, the summed
// milliseconds and the frames they cover: stages = project, ground, fps, assign, keypoints, model, quantize.
extern "C" int rpcc_encoder_profile(rpcc_encoder* e, int enable) {
  RPCC_REQUIRE(e, "null pointer");
  RPCC_CUDA(cudaSetDevice(e->cfg.device));
  for (int i = 0; i < kSlots; ++i) {
    Slot& s = e->slot[i];
    if (enable && !s.ev) {
      s.ev = new (std::nothrow) cudaEvent_t[(size_t)kEvRing * (kStages + 1)]();
      s.ev_frames = new (std::nothrow) int[kEvRing]();
      RPCC_REQUIRE(s.ev && s.ev_frames, "out of host memory");
      for (int q = 0; q < kEvRing * (kStages + 1); ++q) RPCC_CUDA(cudaEventCreate(&s.ev[q]));
    }
    s.ev_head = 0; s.ev_count = 0;
  }
  e->profiling = enable != 0;
  return RPCC_OK;
}

extern "C" int rpcc_encoder_stage_times(rpcc_encoder* e, double* ms_out, long long* frames_out, int* calls_out) {
  RPCC_REQUIRE(e && ms_out && frames_out, "null pointer");
  RPCC_CUDA(cudaSetDevice(e->cfg.device));
  for (int q = 0; q < kStages; ++q) ms_out[q] = 0.0;
  long long frames = 0;
  int calls = 0;
  for (int i = 0; i < kSlots; ++i) {
    Slot& s = e->slot[i];
    if (!s.ev) continue;
    RPCC_CUDA(cudaStreamSynchronize(s.stream));
    for (int k = 0; k < s.ev_count; ++k) {
      cudaEvent_t* ev = s.ev + (size_t)k * (kStages + 1);
      for (int q = 0; q < kStages; ++q) {
        float ms = 0.f;
        RPCC_CUDA(cudaEventElapsedTime(&ms, ev[q], ev[q + 1]));
        ms_out[q] += ms;
      }
      frames += s.ev_frames[k];
      ++calls;
    }
  }
  *frames_out = frames;
  if (calls_out) *calls_out = calls;
  return RPCC_OK;
}

extern "C" int rpcc_encoder_encode_device(rpcc_encoder* e, int slot, const float* points, int stride,
                                          const int64_t* offsets, int B, const float* ground_in,
                                          const uint64_t* frame_keys) {
  RPCC_REQUIRE(e && points && offsets, "null pointer");
  RPCC_REQUIRE(slot >= 0 && slot < kSlots, "bad slot");
  if (B > e->cfg.max_batch) { set_error("rpcc_encoder_encode_device: B=%d exceeds max_batch=%d", B, e->cfg.max_batch); return RPCC_ERR_CAPACITY; }
  RPCC_CUDA(cudaSetDevice(e->cfg.device));
  return run_chain(e, e->slot[slot], points, stride, offsets, B, ground_in, frame_keys);
}

extern "C" int rpcc_encoder_sync(rpcc_encoder* e) {
  RPCC_REQUIRE(e, "null pointer");
  RPCC_CUDA(cudaSetDevice(e->cfg.device));
  for (int i = 0; i < kSlots; ++i) RPCC_CUDA(cudaStreamSynchronize(e->slot[i].stream));
  return RPCC_OK;
}

extern "C" void* rpcc_encoder_stream(rpcc_encoder* e, int slot) {
  return (e && slot >= 0 && slot < kSlots) ? (void*)e->slot[slot].stream : nullptr;
}

extern "C" void* rpcc_encoder_device_buffer(rpcc_encoder* e, int slot, const char* name) {
  if (!e || !name || slot < 0 || slot >= kSlots) return nullptr;
  Slot& s = e->slot[slot];
  struct { const char* n; void* p; } tab[] = {
      {"range", s.range}, {"labels", s.labels}, {"model", s.model}, {"symbols", s.symbols}, {"seq", s.seq},
      {"contour", s.contour}, {"results", s.results}, {"center_idx", s.center_idx}, {"centers", s.centers},
      {"ground", s.ground}, {"key_points", s.key_points}, {"salience", s.salience}, {"step_per_label", s.step_per_label},
      {"sym_base", s.sym_base}, {"seq_base", s.seq_base}, {"lut", e->lut}, {"points", s.points}, {"offsets", s.offsets}, {"order", s.order},
      {"eval_range", s.ev_range}, {"eval_labels", s.ev_labels}, {"eval_metrics", s.ev_metrics},
      {"eval_normals_ref", s.ev_nref}, {"eval_normals_rec", s.ev_nrec}, {"eval_p2plane", s.ev_p2}, {"dbscan_workspace", s.db_ws},
      {"intensity_owner", s.int_owner}, {"intensity", s.inten}, {"intensity_stream", s.int_stream}};
  for (auto& t : tab) if (strcmp(t.n, name) == 0) return t.p;
  return nullptr;
}

// Host buffers in, host sections out.  Frames are cut into chunks of <= max_batch and pipelined over
// the stream slots: while chunk c runs its kernels, chunk c+1's points are on their way up and chunk
// c-1's sections on their way down.
extern "C" int rpcc_encoder_encode_host(rpcc_encoder* e, const float* points_host, int stride,
                                        const int64_t* offsets_host, int B, const float* ground_host,
                                        rpcc_frame_result* results, float* model, uint8_t* contour_bits,
                                        uint16_t* seq, size_t seq_cap, int16_t* symbols, size_t sym_cap,
                                        uint8_t* salience, const uint64_t* frame_keys, double* eval_metrics) {
  return rpcc_encoder_encode_host_intensity(e, points_host, stride, offsets_host, B, ground_host, results, model, contour_bits,
                                            seq, seq_cap, symbols, sym_cap, salience, frame_keys, eval_metrics, nullptr);
}

extern "C" int rpcc_encoder_encode_host_intensity(rpcc_encoder* e, const float* points_host, int stride,
                                                  const int64_t* offsets_host, int B, const float* ground_host,
                                                  rpcc_frame_result* results, float* model, uint8_t* contour_bits,
                                                  uint16_t* seq, size_t seq_cap, int16_t* symbols, size_t sym_cap,
                                                  uint8_t* salience, const uint64_t* frame_keys, double* eval_metrics,
                                                  uint8_t* intensity) {
  RPCC_REQUIRE(!eval_metrics || e == nullptr || e->cfg.eval, "eval_metrics needs an encoder created with eval = 1 or 2");
  RPCC_REQUIRE(e && points_host && offsets_host && results && model && contour_bits && seq && symbols, "null pointer");
  RPCC_REQUIRE(!intensity || e->cfg.intensity_step > 0, "intensity output needs an encoder created with intensity_step > 0");
  RPCC_REQUIRE(intensity || !(e->cfg.intensity_step > 0),
               "this encoder carries intensity: call rpcc_encoder_encode_host_intensity with an intensity output");
  RPCC_REQUIRE(stride == 3 || stride == 4, "stride must be 3 or 4");
  RPCC_REQUIRE(B >= 0, "bad batch");
  RPCC_CUDA(cudaSetDevice(e->cfg.device));
  const int MB = e->host_chunk, K = e->K, cb = e->cbytes;
  const size_t ecols = RPCC_EVAL_COLS + (e->cfg.eval == 2 ? RPCC_P2PLANE_COLS : 0);   // eval_metrics row width
  const int nchunks = (B + MB - 1) / MB;
  size_t sym_done = 0, seq_done = 0;
  struct Pending { int slot, f0, nb; };
  std::vector<Pending> pend;

  auto finish = [&](const Pending& p) -> int {
    Slot& s = e->slot[p.slot];
    RPCC_CUDA(cudaEventSynchronize(s.done));   // results of the chunk are on the host
    size_t ns = 0, nq = 0;
    for (int i = 0; i < p.nb; ++i) { results[p.f0 + i] = s.h_results[i]; ns += s.h_results[i].sym_count; nq += s.h_results[i].seq_count; }
    if (sym_done + ns > sym_cap || seq_done + nq > seq_cap) {
      set_error("rpcc_encoder_encode_host: output capacity exceeded (symbols %zu/%zu, seq %zu/%zu)", sym_done + ns, sym_cap, seq_done + nq, seq_cap);
      return RPCC_ERR_CAPACITY;
    }
    RPCC_CUDA(cudaMemcpyAsync(symbols + sym_done, s.symbols, ns * sizeof(int16_t), cudaMemcpyDeviceToHost, s.stream));
    RPCC_CUDA(cudaMemcpyAsync(seq + seq_done, s.seq, nq * sizeof(uint16_t), cudaMemcpyDeviceToHost, s.stream));
    if (intensity) RPCC_CUDA(cudaMemcpyAsync(intensity + sym_done, s.int_stream, ns, cudaMemcpyDeviceToHost, s.stream));
    RPCC_CUDA(cudaMemcpyAsync(model + (size_t)p.f0 * K * 4, s.model, sizeof(float) * 4 * K * (size_t)p.nb, cudaMemcpyDeviceToHost, s.stream));
    RPCC_CUDA(cudaMemcpyAsync(contour_bits + (size_t)p.f0 * cb, s.contour, (size_t)cb * p.nb, cudaMemcpyDeviceToHost, s.stream));
    if (salience && e->cfg.nonuniform)
      RPCC_CUDA(cudaMemcpyAsync(salience + (size_t)p.f0 * K, s.salience, (size_t)K * p.nb, cudaMemcpyDeviceToHost, s.stream));
    if (eval_metrics) {
      RPCC_CUDA(cudaMemcpy2DAsync(eval_metrics + (size_t)p.f0 * ecols, sizeof(double) * ecols, s.ev_metrics,
                                  sizeof(double) * RPCC_EVAL_COLS, sizeof(double) * RPCC_EVAL_COLS, (size_t)p.nb,
                                  cudaMemcpyDeviceToHost, s.stream));
      if (e->cfg.eval == 2)
        RPCC_CUDA(cudaMemcpy2DAsync(eval_metrics + (size_t)p.f0 * ecols + RPCC_EVAL_COLS, sizeof(double) * ecols, s.ev_p2,
                                    sizeof(double) * RPCC_P2PLANE_COLS, sizeof(double) * RPCC_P2PLANE_COLS, (size_t)p.nb,
                                    cudaMemcpyDeviceToHost, s.stream));
    }
    RPCC_CUDA(cudaEventRecord(s.done, s.stream));
    sym_done += ns; seq_done += nq;
    return RPCC_OK;
  };

  // every exit of the loop -- CUDA error, capacity error -- falls through to the stream synchronisation below: no
  // copy into the caller's buffers is left in flight when this call returns
  auto run = [&]() -> int {
  int rc = RPCC_OK;
  for (int c = 0; c < nchunks && rc == RPCC_OK; ++c) {
    // Slot c % kSlots was last used by chunk c - kSlots, which has been finished below (at most two
    // chunks are ever pending); its D2H copies precede this chunk's work in stream order.
    const int sl = c % kSlots;
    Slot& s = e->slot[sl];
    const int f0 = c * MB, nb = (B - f0) < MB ? (B - f0) : MB;
    const int64_t p0 = offsets_host[f0], p1 = offsets_host[f0 + nb];
    if (p1 - p0 > e->cfg.max_points) {
      set_error("rpcc_encoder_encode_host: chunk has %lld points, max_points=%lld", (long long)(p1 - p0), (long long)e->cfg.max_points);
      rc = RPCC_ERR_CAPACITY;
      break;
    }
    for (int i = 0; i <= nb; ++i) s.h_offsets[i] = offsets_host[f0 + i] - p0;
    RPCC_CUDA(cudaMemcpyAsync(s.offsets, s.h_offsets, sizeof(int64_t) * (nb + 1), cudaMemcpyHostToDevice, s.stream));
    RPCC_CUDA(cudaMemcpyAsync(s.points, points_host + (size_t)p0 * stride, sizeof(float) * stride * (size_t)(p1 - p0), cudaMemcpyHostToDevice, s.stream));
    const float* gin = nullptr;
    if (ground_host) {
      RPCC_CUDA(cudaMemcpyAsync(s.ground, ground_host + (size_t)f0 * 4, sizeof(float) * 4 * nb, cudaMemcpyHostToDevice, s.stream));
      gin = s.ground;
    }
    const uint64_t* kin = nullptr;
    if (frame_keys) {
      RPCC_CUDA(cudaMemcpyAsync(s.keys, frame_keys + f0, sizeof(uint64_t) * nb, cudaMemcpyHostToDevice, s.stream));
      kin = s.keys;
    }
    rc = run_chain(e, s, s.points, stride, s.offsets, nb, gin, kin);
    if (rc) break;
    RPCC_CUDA(cudaMemcpyAsync(s.h_results, s.results, sizeof(rpcc_frame_result) * nb, cudaMemcpyDeviceToHost, s.stream));
    RPCC_CUDA(cudaEventRecord(s.done, s.stream));
    pend.push_back({sl, f0, nb});
    // with this chunk queued, collect every older one: the host blocks on chunk c-1's results while
    // chunk c's upload and kernels proceed
    while (pend.size() > 1 && rc == RPCC_OK) { rc = finish(pend.front()); pend.erase(pend.begin()); }
  }
  while (!pend.empty() && rc == RPCC_OK) { rc = finish(pend.front()); pend.erase(pend.begin()); }
  return rc;
  };
  int rc = run();
  for (int i = 0; i < kSlots; ++i) {
    const int r2 = check_cuda(cudaStreamSynchronize(e->slot[i].stream), "stream sync");
    if (rc == RPCC_OK) rc = r2;
  }
  return rc;
}
