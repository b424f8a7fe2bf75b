/*
 * rpcc_b200.h -- C ABI of librpcc_b200.so: the B200 (sm_100a) implementation of R-PCC's
 * per-frame compression hot path (project -> FPS segment -> model -> quantize -> pack,
 * plus decode and chamfer evaluation).
 *
 * This is the drop-in boundary.  The reference crosses it through pybind11 modules
 * (ops/cpp_modules/src/cpp_modules.cpp:597-636), a torch CUDAExtension
 * (ops/fps/src/fps_api.cpp:7-9) and a JIT torch extension
 * (utils/ChamferDistancePytorch/chamfer3D/chamfer_cuda.cpp:17-30).  Every entry point below
 * names the reference interface it replaces.  Signatures use plain pointers and sizes only
 * (no torch / numpy / pybind types); INTEGRATION.md shows the ctypes binding the reference
 * side would add.
 *
 * Conventions
 *  - All functions return 0 (RPCC_OK) or a negative RPCC_ERR_* code; rpcc_last_error()
 *    returns a thread-local message.  Nothing calls exit() (the reference's FPS glue does,
 *    ops/fps/src/sampling.cpp:9-21).
 *  - `*_batch` functions take DEVICE pointers, enqueue on `stream` (a cudaStream_t passed as
 *    void*; NULL = legacy default stream) and do not synchronise.  Buffers are caller-owned.
 *  - `rpcc_op_*` functions take HOST pointers, one frame, and are synchronous: they are the
 *    one-to-one replacements of the reference's pybind functions (numpy in, numpy out).
 *  - Frames of a batch are laid out frame-major: range images [B][H][W] f32, labels
 *    [B][H][W] u8 (device) / int32 (host ops, as the reference), etc.
 *  - Labels: 0 = ground, 1 = empty pixel, 2..cluster_num+1 = FPS clusters
 *    (utils/segment_utils.py:168-169).  K = cluster_num + 2 model rows.
 */
#ifndef RPCC_B200_H_
#define RPCC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define RPCC_API __attribute__((visibility("default")))
#else
#define RPCC_API
#endif

#define RPCC_OK 0
#define RPCC_ERR_ARG (-1)     /* bad argument (null pointer, size out of range) */
#define RPCC_ERR_CUDA (-2)    /* CUDA runtime error, see rpcc_last_error() */
#define RPCC_ERR_NO_DEVICE (-3)
#define RPCC_ERR_CAPACITY (-4) /* caller-provided buffer too small / batch larger than the encoder's */

#define RPCC_MAX_LABELS 256   /* labels are stored as u8 on device; K = cluster_num + 2 <= 254, i.e. --cluster_num <= 252
                                 (the reference's idx_sequence is uint16 and accepts more; tools/common.py rejects larger
                                 values with a message, DESIGN.md section 8) */
#define RPCC_TILE 1024        /* pixels per rank tile (flat raster index / 1024) */

RPCC_API const char* rpcc_last_error(void);
RPCC_API int rpcc_version(void);
/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
RPCC_API long long rpcc_launch_count(void);
RPCC_API int rpcc_device_count(void);

/* ---- a1. dataset/transformer.py:41-54 create_transform_map (host, f64 trig -> f32) ------------ */
RPCC_API int rpcc_transform_map(int H, int W, double hfov, double vmax, double vmin, float* lut_host);

/* ================================ device batch stages ======================================== */

/* a2. cpp_modules.cpp:427-467 point_cloud_to_range_image_even, B frames per launch.
 * points: packed rows of `stride` floats (3 = xyz, 4 = KITTI .bin x,y,z,intensity); for stride 4
 * the base must be 16-byte aligned.  offsets[B+1]: first row of each frame (int64, device).
 * range: [B][H][W] f32, fully overwritten (0 = empty pixel).  scratch: int32[B] (zero-depth
 * bookkeeping, SURVEY C9).  Bit-exact with the reference for finite inputs. */
RPCC_API int rpcc_project_batch(const float* points, int stride, const int64_t* offsets, int B, int H, int W,
                       float hfov, float vmax, float vmin, float* range, int32_t* scratch, void* stream);

/* Intensity owners (DESIGN.md §4, "Intensity"; beyond the reference, which drops the column).  After
 * rpcc_project_batch on the same stride-4 points (16-byte aligned rows), with its range and scratch: owner [B][H][W] u32
 * = in-frame row index of the point the reference's sequential z-buffer loop stored last into the pixel (0xFFFFFFFF:
 * empty pixel), intensity [B][H][W] f32 = that point's fourth column (0 at empty pixels). */
RPCC_API int rpcc_intensity_owner_batch(const float* points, const int64_t* offsets, int B, int H, int W, float hfov,
                                float vmax, float vmin, const float* range, const int32_t* scratch, uint32_t* owner,
                                float* intensity, void* stream);

/* a3. dataset/transformer.py:94-101 range_image_to_point_cloud: xyz[b][h][w][3] = range * lut. */
RPCC_API int rpcc_range_to_xyz_batch(const float* range, const float* lut, int B, int HW, float* xyz, void* stream);

/* a4 (first half). Deterministic ground-plane RANSAC standing in for open3d segment_plane
 * (utils/segment_utils.py:74-82,101-108; parity unpinned, see ground.cu).  Frame b is keyed by
 * (seed + frame_keys[b]); frame_keys (device, [B]) may be NULL = key 0 for every frame, in which case a
 * frame's plane depends on the frame's content alone -- not on its place in the batch, the datalist or
 * the shard.  ground: [B][4] f32, unit normal. */
RPCC_API int rpcc_ground_fit_batch(const float* range, const float* lut, int B, int H, int W, uint64_t seed,
                          const uint64_t* frame_keys, float* ground, void* stream);

/* a5. ops/fps/src/sampling_gpu.cu:24-184 furthest_point_sampling_kernel_launcher.
 * points [B][n][3] f32 -> idx [B][m] i32.  Same seeds as the reference kernel, including its
 * FMA pattern and tie rule (SURVEY A.2).  temp: [B][n] f32 scratch (the reference's `temp`;
 * contents on entry are ignored -- it is always (re)filled with 1e10). */
RPCC_API int rpcc_fps_batch(const float* points, int B, int n, int m, float* temp, int32_t* idx, void* stream);

/* a4+a5 fused (utils/segment_utils.py:133-141): non-ground mask + FPS straight from the range
 * image; never materialises xyz.  center_idx [B][m] i32 (flat pixel index), centers [B][m][3]. */
RPCC_API int rpcc_segment_fps_batch(const float* range, const float* lut, const float* ground, int B, int H, int W,
                           int m, float ground_thr, int32_t* center_idx, float* centers, void* stream);

/* utils/segment_utils.py:149-164 (segment_method 'DBSCAN'), by this project's own definition (DESIGN.md §4; parity with
 * open3d's cluster_dbscan unpinned).  Points: the non-empty pixels the FPS path masks as non-ground (ground model
 * ground [B][4], ground_thr); q is a neighbour of p when cham_d(p, q) <= (float)(eps * eps), p included; a core point
 * has >= min_points neighbours; clusters are the connected components of the cores; a non-core point with a core
 * neighbour joins the cluster of its nearest core (cham_d, then the smaller flat pixel index).  labels [B][HW] u8:
 * 0 ground, 1 empty, 2 .. cluster_num the cluster_num - 1 largest clusters (cores + borders; on equal size the smaller
 * first core pixel first) numbered in order of their first core pixel, cluster_num + 1 noise and all other clusters:
 * K stays cluster_num + 2.  Exact: neighbourhoods by a window search over the range image, a whole-image scan where
 * eps is not below the query's range or the frame holds a negative range.  Needs a 360-degree sensor; eps > 0,
 * min_points >= 1.  workspace: rpcc_dbscan_workspace_bytes(B, H, W) bytes of device memory; once the call has run,
 * its first B uint32 hold each frame's number of points that needed a whole-image scan and the next B its number of
 * clusters (before the cluster_num - 1 cut). */
RPCC_API size_t rpcc_dbscan_workspace_bytes(int B, int H, int W);
RPCC_API int rpcc_dbscan_segment_batch(const float* range, const float* lut, const float* ground, int B, int H, int W,
                              double hfov, double vmax, double vmin, double eps, int min_points, int cluster_num,
                              float ground_thr, uint8_t* labels, void* workspace, void* stream);

/* Per-frame result table (device or host copy, frame-major). */
typedef struct rpcc_frame_result {
  uint32_t sym_count;   /* int16 symbols = non-empty pixels */
  uint32_t seq_count;   /* uint16 idx_sequence entries */
  uint32_t model_rows;  /* highest label present + 1: rows of plane_param the reference writes */
  uint32_t flags;       /* bit0: exact-mean guard tripped (handled), bit1: a label >= K was seen,
                           bit3: an intensity was clamped to [0, 255] steps (rpcc_intensity_pack_batch) */
} rpcc_frame_result;

/* Bookkeeping workspace shared by assign/label_stats -> point_model -> quantize_pack (device,
 * opaque; tile histograms, label counts, exact sums, offsets).  K = number of model rows. */
RPCC_API size_t rpcc_book_bytes(int B, int H, int W, int K);

/* a4 (second half, utils/segment_utils.py:143-148,168-169) + a6 accumulation
 * (cpp_modules.cpp:471-518): per-pixel argmin over {ground, m centres} with torch's float32
 * arithmetic.  labels [B][HW] u8.  Fills `book` (K = m + 2) for the next two stages. */
RPCC_API int rpcc_assign_labels_batch(const float* range, const float* lut, const float* ground, const float* centers,
                             int B, int H, int W, int m, uint8_t* labels, void* book, void* stream);

/* Same bookkeeping for callers that bring their own labels (the standalone quantize ops).  A label >= K counts as
 * empty (label 1), as rpcc_dequantize_batch decodes it, and sets flags bit1. */
RPCC_API int rpcc_label_stats_batch(const float* range, const uint8_t* labels, int B, int H, int W, int K,
                           void* book, void* stream);

/* a6. point models + stable-order bookkeeping.  model [B][K][4] f32 rows exactly as they reach
 * the bitstream (row 0 = ground, row 1 = 0, row l = [0,0,0,mean_l]; empty cluster = NaN as the
 * reference); results [B] (sym_count, seq_count, model_rows, flags). */
RPCC_API int rpcc_point_model_batch(const float* range, const uint8_t* labels, const float* ground, void* book,
                           int B, int H, int W, int K, float* model, rpcc_frame_result* results, void* stream);

/* a6, model_method = 'plane' (utils/segment_utils.py:188-216): per-cluster RANSAC plane models.
 * rpcc_label_order_batch lists the non-empty pixels of every frame in the label-major stable order of
 * the symbol stream (order [B][order_stride] u32 flat pixel indices, first sym_count[b] valid); `book`
 * must have been through rpcc_point_model_batch.  rpcc_plane_model_batch then overwrites, in
 * model [B][K][4] (as rpcc_point_model_batch left it), the row of every cluster (label >= 2) that has
 * at least min_pixels pixels (reference: 30) and whose plane -- least-squares planes of ransac_n (4)
 * distinct points, `iterations` (10) hypotheses, inliers within dist_thr (0.1 m), refit on the inliers
 * of the best -- passes plane_angle_validation (:84-93) at angle_threshold_deg (cfgs/compressor.yaml:30).
 * Deterministic: keyed by (seed, frame_keys[b], label); frame_keys as in rpcc_ground_fit_batch (device, NULL = 0).
 * open3d's segment_plane is not reproduced
 * bit for bit (third-party, randomised; DESIGN.md "parity unpinned"). */
RPCC_API int rpcc_label_order_batch(const uint8_t* labels, void* book, int B, int H, int W, int K, uint32_t* order,
                           size_t order_stride, void* stream);
RPCC_API int rpcc_plane_model_batch(const float* range, const float* lut, const uint32_t* order, size_t order_stride,
                           void* book, int B, int H, int W, int K, int min_pixels, float dist_thr, int ransac_n,
                           int iterations, float angle_threshold_deg, uint64_t seed, const uint64_t* frame_keys,
                           float* model, void* stream);

/* a7+a8+a10. cpp_modules.cpp:248-285 intra_predict, :288-334 uniform_quantize (or :337-424 with
 * per-label steps), :521-558 extract_contour + np.packbits, fused.  step_per_label: NULL =>
 * uniform `step`; else [B][K] f32.  symbols: [B][sym_stride] i16 (first sym_count[b] valid),
 * label-major / raster-within-label.  contour_bits [B][ceil(HW/8)] u8 MSB-first;
 * seq [B][seq_stride] u16 (first seq_count[b] valid); with sym_base / seq_base non-NULL frame b's
 * streams start at symbols + sym_base[b] / seq + seq_base[b] instead.  `book` must have been
 * through rpcc_point_model_batch. */
RPCC_API int rpcc_quantize_pack_batch(const float* range, const uint8_t* labels, const float* model, const float* lut,
                             void* book, const float* step_per_label, float step, int B, int H, int W, int K,
                             int16_t* symbols, size_t sym_stride, uint8_t* contour_bits, uint16_t* seq,
                             size_t seq_stride, const uint64_t* sym_base, const uint64_t* seq_base, void* stream);

/* Exclusive scan of results[b].sym_count / seq_count into sym_base / seq_base ([B+1] u64, device;
 * entry B = totals): pass them to rpcc_quantize_pack_batch to get the frames' streams packed back
 * to back instead of strided. */
RPCC_API int rpcc_frame_offsets_batch(const rpcc_frame_result* results, int B, uint64_t* sym_base, uint64_t* seq_base,
                             void* stream);

/* The intensity section: one u8 per non-empty pixel (range != 0) in raster order, q = clamp(round half away from zero of
 * (double)intensity / step, 0, 255), NaN -> 0, frame b's bytes at out + sym_base[b] (the offsets of
 * rpcc_frame_offsets_batch: as many bytes as the frame has symbols).  A frame with a clamped pixel gets flags bit3 in
 * results (may be NULL). */
RPCC_API int rpcc_intensity_pack_batch(const float* intensity, const float* range, int B, int H, int W, double step,
                               const uint64_t* sym_base, uint8_t* out, rpcc_frame_result* results, void* stream);

/* a9. cpp_modules.cpp:28-121 extract_features_with_segment (+:10-25) and the salience rule of
 * :388-405.  key_points [B][HW] u8 (0..3); feat [B][HW] f32 curvature map or NULL;
 * salience [B][K] u8 and step_per_label [B][K] f32 (both NULL => key points only);
 * level tables are HOST arrays (<= 8 levels); kp_cnt: u32 [B][K] device scratch.
 * `book` must hold the label counts (rpcc_assign_labels_batch / rpcc_label_stats_batch). */
RPCC_API int rpcc_keypoints_salience_batch(const float* range, const uint8_t* labels, const void* book, int B, int H, int W,
                                  int K, int region, int segments, int sharp_num, int less_sharp_num, int flat_num,
                                  const int32_t* level_kp_num, const float* level_acc, int level_num,
                                  int ground_level, uint8_t* key_points, float* feat, uint8_t* salience,
                                  float* step_per_label, uint32_t* kp_cnt, void* stream);

/* a11. decode: cpp_modules.cpp:561-593 recover_map, utils/compress_utils.py:114-132
 * dequantize_residual, cpp_modules.cpp:248-285 intra_predict, tools/decompress.py:108-110,
 * dataset/transformer.py:94-101.
 * contour_bits [B][ceil(HW/8)], seq [B][seq_stride] u16 (seq_count [B] valid entries, or NULL =
 * trusted), symbols [B][sym_stride] i16 (sym_count [B] or NULL), model [B][K][4] f32,
 * steps [B][K] f64 (per-label dequantisation step: 2*accuracy, or the salience level's step).
 * Outputs: labels [B][HW] u8, range_rec [B][HW] f32, xyz [B][HW][3] f32 (may be NULL),
 * results [B]: symbols / sequence entries a well-formed stream of these labels holds (compare with
 * the section lengths), flags bit1/bit2 on malformed input.  book: rpcc_book_bytes(B,H,W,K). */
RPCC_API int rpcc_decode_batch(const uint8_t* contour_bits, const uint16_t* seq, size_t seq_stride,
                      const uint32_t* seq_count, const int16_t* symbols, size_t sym_stride,
                      const uint32_t* sym_count, const float* model, const double* steps, const float* lut,
                      int B, int H, int W, int K, uint8_t* labels, float* range_rec, float* xyz, void* book,
                      rpcc_frame_result* results, void* stream);

/* The same for streams packed back to back (what rpcc_encoder_encode_host returns and what a reader of many files
 * builds): frame b's sequence is seq[seq_base[b] .. seq_base[b+1]) and its symbols symbols[sym_base[b] .. sym_base[b+1])
 * (u64 [B+1], device). */
RPCC_API int rpcc_decode_packed_batch(const uint8_t* contour_bits, const uint16_t* seq, const uint64_t* seq_base,
                             const int16_t* symbols, const uint64_t* sym_base, const float* model, const double* steps,
                             const float* lut, int B, int H, int W, int K, uint8_t* labels, float* range_rec, float* xyz,
                             void* book, rpcc_frame_result* results, void* stream);

/* Last step of decoding (dataset/transformer.py:94-101 + save_point_cloud_to_file, dataset/dataset.py:72-81):
 * range_rec [B][HW] -> rows of (x, y, z, 0) f32 for the pixels with float32 x + y + z != 0, raster order, frames packed
 * back to back: frame b = rows[4 * row_base[b] .. 4 * row_base[b+1]) (row_base [B+1] u64, device, written here).
 * rows needs room for B*HW rows; workspace: rpcc_points_workspace_bytes(B, H, W). */
RPCC_API size_t rpcc_points_workspace_bytes(int B, int H, int W);
RPCC_API int rpcc_points_out_batch(const float* range_rec, const float* lut, int B, int H, int W, float* rows,
                          uint64_t* row_base, void* workspace, void* stream);

/* The same, with the fourth column taken from intensity [B][HW] f32 (NULL = zeros, as rpcc_points_out_batch). */
RPCC_API int rpcc_points_out_intensity_batch(const float* range_rec, const float* lut, const float* intensity, int B, int H,
                                     int W, float* rows, uint64_t* row_base, void* workspace, void* stream);
/* Inverse of rpcc_intensity_pack_batch: labels [B][HW] u8 (non-empty = label != 1) and frame b's bytes
 * in[base[b] .. base[b+1]) (u64 [B+1], device) -> intensity [B][HW] f32 = (float)((double)q * step), 0 at empty pixels
 * and at pixels past the end of a frame's bytes. */
RPCC_API int rpcc_intensity_unpack_batch(const uint8_t* labels, const uint8_t* in, const uint64_t* base, int B, int H, int W,
                                 double step, float* intensity, void* stream);

/* Second half of decoding when the labels are already known; also the batched
 * QuantizationModule.dequantize_residual (utils/compress_utils.py:114-132).  With a zero model and
 * xyz = NULL, range_rec is the dequantised residual itself.  stats_ready = 0 unless `book` already
 * holds this batch's label histograms. */
RPCC_API int rpcc_dequantize_batch(const uint8_t* labels, const int16_t* symbols, size_t sym_stride,
                          const uint32_t* sym_count, const float* model, const double* steps, const float* lut,
                          int B, int H, int W, int K, float* range_rec, float* xyz, void* book,
                          rpcc_frame_result* results, int stats_ready, void* stream);

/* a12. chamfer3D.cu:12-154 NmDistanceKernel both ways: for each point of xyz1 [n][3] the squared
 * distance to and index of its nearest neighbour in xyz2 [m][3], and vice versa.  Exact brute
 * force with the reference's FMA pattern and first-minimum tie rule.
 * scratch: (n + m) * 8 bytes of device memory.  An empty cloud on the other side yields +inf / INT_MAX. */
RPCC_API int rpcc_chamfer_batch(const float* xyz1, int n, const float* xyz2, int m, float* dist1, int32_t* idx1,
                       float* dist2, int32_t* idx2, void* scratch, void* stream);
/* utils/evaluate_metrics.py:20-22 + fscore.py:12-16 reductions: stats (device, 4 doubles) =
 * {sum sqrt(dist1), #(dist1 < threshold_sq), sum sqrt(dist2), #(dist2 < threshold_sq)}. */
RPCC_API int rpcc_chamfer_stats(const float* dist1, int n, const float* dist2, int m, float threshold_sq, double* stats,
                       void* stream);

/* ---- a12 for range images: the --eval figures (tools/compress_datalist.py:166-199, utils/evaluate_metrics.py:9-45) --- */
/* B pairs (range_ref, range_rec) of range images over the same ray table `lut` ([H][W][3]).  Per frame, metrics
 * [B][RPCC_EVAL_COLS] f64 =
 *   0 max |rec - ref|      1 sum |rec - ref| (mean = / HW)
 *   2 n1 (points of ref with x+y+z != 0)   3 sum sqrt(dist1)   4 #(dist1 < threshold_sq)   5 sum dist1
 *   6 n2 (points of rec)                    7 sum sqrt(dist2)   8 #(dist2 < threshold_sq)   9 sum dist2
 *   10 points that needed a whole-image scan   11 label mismatches (labels_ref vs labels_rec; 0 when either is NULL)
 * dist1 / dist2 = the squared nearest-neighbour distances NmDistanceKernel (chamfer3D.cu:12-154) would return for the
 * two compacted clouds, found by an exact window search in range-image space (evalq.cu); optional outputs
 * [B][HW] f32 (-1 at pixels that are not points).  Sums are accumulated in a fixed order (reproducible).
 * Needs a 360-degree sensor.  workspace: rpcc_eval_workspace_bytes(B, H, W) bytes of device memory. */
#define RPCC_EVAL_COLS 12
RPCC_API size_t rpcc_eval_workspace_bytes(int B, int H, int W);
RPCC_API int rpcc_eval_batch(const float* range_ref, const float* range_rec, const float* lut, const uint8_t* labels_ref,
                    const uint8_t* labels_rec, int B, int H, int W, double hfov, double vmax, double vmin,
                    float threshold_sq, float* dist1, float* dist2, double* metrics, void* workspace, void* stream);
/* steps [B][K] f64 for rpcc_decode_batch: `step` everywhere (salience NULL) or step + level_dacc8[salience[b][l]]
 * (QuantizationModule, utils/compress_utils.py:48; level_dacc8_dev: 8 doubles on the device). */
RPCC_API int rpcc_eval_steps_batch(const uint8_t* salience, int B, int K, double step, const double* level_dacc8_dev,
                          double* steps, void* stream);

/* ---- point-to-plane PSNR for range images (utils/evaluate_metrics.py:48-72 with its open3d normals, :133) ----------- */
/* Normals of B range images ([B][H][W] f32 over the ray table `lut`, 360-degree sensor): for every point (x+y+z != 0)
 * the PCA normal of its neighbourhood -- its `knn` nearest points in its own image, itself included, restricted to
 * those within `radius` (cham_d <= radius^2 in f32; distance ties to the smaller flat pixel index), as open3d's
 * KDTreeSearchParamHybrid(radius, max_nn) -- from the f64 two-pass covariance: the eigenvector of the smallest eigenvalue,
 * oriented so that n . p <= 0.  normals [B][HW][3] f32; (0,0,0) at pixels that are not points and where there is no normal
 * (fewer than 3 neighbours, lambda2 == 0, or lambda1 - lambda0 <= 1e-6 lambda2).  Exact k-NN by the window search of
 * rpcc_eval_batch, with a whole-image scan where the tabulated window does not settle it.  knn in [3, 32], radius > 0.
 * workspace: rpcc_normals_workspace_bytes(B, H, W) bytes of device memory; once the call has run, its first B uint32
 * hold each frame's number of points whose neighbourhood needed a whole-image scan.  Parity with open3d is unpinned
 * (DESIGN.md). */
#define RPCC_NORMAL_KNN 16
#define RPCC_NORMAL_RADIUS 1.0f
RPCC_API size_t rpcc_normals_workspace_bytes(int B, int H, int W);
RPCC_API int rpcc_normals_batch(const float* range, const float* lut, int B, int H, int W, double hfov, double vmax,
                       double vmin, int knn, float radius, float* normals, void* workspace, void* stream);
/* Point-to-plane error of B pairs (range_ref, range_rec) with their normals (rpcc_normals_batch).  For each point a of ref,
 * b = its nearest point of rec (the neighbour rpcc_eval_batch's dist1 is measured to: first minimum, smallest pixel index)
 * and err = ((a - b) . n_rec(b))^2 in f64, or the squared distance cham_d(a, b) when b has no normal; rec -> ref
 * likewise with n_ref.  metrics [B][RPCC_P2PLANE_COLS] f64 =
 *   0 n1 (points of ref)   1 sum err1   2 points of ref whose neighbour had no normal
 *   3 n2 (points of rec)   4 sum err2   5 points of rec whose neighbour had no normal
 *   6 points whose nearest-neighbour search needed a whole-image scan
 * An empty cloud on the other side gives a +inf sum.  mse = sum / n, PSNR = 10 log10(3 * 59.7^2 / mse).  Sums are
 * accumulated in a fixed order (reproducible).  workspace: rpcc_p2plane_workspace_bytes(B, H, W) bytes of device memory. */
#define RPCC_P2PLANE_COLS 7
RPCC_API size_t rpcc_p2plane_workspace_bytes(int B, int H, int W);
RPCC_API int rpcc_p2plane_batch(const float* range_ref, const float* range_rec, const float* lut, const float* normals_ref,
                       const float* normals_rec, int B, int H, int W, double hfov, double vmax, double vmin,
                       double* metrics, void* workspace, void* stream);

/* ================================ host (numpy-facing) ops ==================================== */
/* One frame, host pointers, synchronous; argument meaning follows the reference's pybind
 * functions so the reference's L3 Python can bind them one for one (INTEGRATION.md). */

/* dataset_utils_cpp.point_cloud_to_range_image_even (cpp_modules.cpp:427) */
RPCC_API int rpcc_op_point_cloud_to_range_image_even(const float* points, int64_t n, int stride, int H, int W,
                                            float hfov, float vmax, float vmin, float* range_out);
/* segment_utils_cpp.point_modeling (cpp_modules.cpp:471): out has max_label+1 floats; *K_out. */
RPCC_API int rpcc_op_point_modeling(const float* range, const int32_t* seg, int H, int W, float* out, int cap, int* K_out);
/* segment_utils_cpp.intra_predict (cpp_modules.cpp:248) */
RPCC_API int rpcc_op_intra_predict(const int32_t* seg, const float* model, int K, const float* lut, int H, int W, float* pred);
/* quantization_utils_cpp.uniform_quantize (cpp_modules.cpp:288): out cap >= H*W; *n_out. */
RPCC_API int rpcc_op_uniform_quantize(const int32_t* seg, const float* residual, int H, int W, float acc,
                             int32_t* out, int64_t* n_out);
/* feature_extractor_cpp.extract_features_with_segment (cpp_modules.cpp:28) -> (feature_map [H][W] f32
 * or NULL, key_point_map [H][W] i32); both zero where the reference leaves them unwritten (SURVEY C7). */
RPCC_API int rpcc_op_extract_features_with_segment(const float* range, const int32_t* seg, int H, int W, int region,
                                          int segments, int sharp_num, int less_sharp_num, int flat_num,
                                          float* feature_map, int32_t* key_point_map);
/* quantization_utils_cpp.nonuniform_quantize (cpp_modules.cpp:337) */
RPCC_API int rpcc_op_nonuniform_quantize(const int32_t* seg, const float* residual, const int32_t* key_point_map,
                                int H, int W, const int32_t* level_kp_num, const float* level_acc, int level_num,
                                int ground_level, int32_t* out, int64_t* n_out, int32_t* salience, int* K_out);
/* contour_utils_cpp.extract_contour (cpp_modules.cpp:521): contour [H][W] i32, seq cap H*W. */
RPCC_API int rpcc_op_extract_contour(const int32_t* seg, int H, int W, int32_t* contour, int32_t* seq, int64_t* L_out);
/* contour_utils_cpp.recover_map (cpp_modules.cpp:561) */
RPCC_API int rpcc_op_recover_map(const int32_t* contour, const int32_t* seq, int64_t L, int H, int W, int32_t* seg_out);
/* furthest_point_sampling_wrapper (ops/fps/src/sampling.cpp:24) with host arrays. */
RPCC_API int rpcc_op_furthest_point_sample(const float* points, int B, int n, int m, int32_t* idx_out);
/* PointCloudSegment.segment GPU branch given the ground model (utils/segment_utils.py:133-148,168-169).
 * seg_out [H][W] i32, center_idx_out [m] i32 (may be NULL). */
RPCC_API int rpcc_op_segment(const float* range, const float* lut, const float* ground, int H, int W, int m,
                    float ground_thr, int32_t* seg_out, int32_t* center_idx_out);
/* The same for segment_method 'DBSCAN' (rpcc_dbscan_segment_batch, one frame): seg_out [H][W] i32;
 * exhaustive_out (may be NULL): points that needed a whole-image scan; clusters_out (may be NULL): clusters found. */
RPCC_API int rpcc_op_segment_dbscan(const float* range, const float* lut, const float* ground, int H, int W, double hfov,
                           double vmax, double vmin, double eps, int min_points, int cluster_num, float ground_thr,
                           int32_t* seg_out, uint32_t* exhaustive_out, uint32_t* clusters_out);
/* chamfer_3D.forward (chamfer_cuda.cpp:17) with host arrays, B = 1. */
RPCC_API int rpcc_op_chamfer(const float* xyz1, int n, const float* xyz2, int m, float* dist1, int32_t* idx1,
                    float* dist2, int32_t* idx2);

/* PointCloudSegment.cluster_modeling (utils/segment_utils.py:172-217) for model_method 'plane' with host arrays:
 * rows_out [cap_rows][4] f32 receives the rows of labels 1 .. K-1 (the array the reference returns: label 1 =
 * [0,0,0,0], clusters = [a,b,c,d] or [0,0,0,mean]); *rows = K - 1. */
RPCC_API int rpcc_op_plane_modeling(const float* range, const int32_t* seg, const float* lut, int H, int W,
                           float angle_threshold_deg, uint64_t seed, float* rows_out, int cap_rows, int* rows);

/* PCTransformer.range_image_to_point_cloud (dataset/transformer.py:94-101) with host arrays. */
RPCC_API int rpcc_op_range_to_xyz(const float* range, const float* lut, int H, int W, float* xyz);
/* The ground-plane fit of PointCloudSegment.segment (utils/segment_utils.py:101-108), host arrays. */
RPCC_API int rpcc_op_ground_fit(const float* range, const float* lut, int H, int W, uint64_t seed, float* ground_out);
/* QuantizationModule.dequantize_residual (utils/compress_utils.py:114-132): symbols (n,) i16, seg (H,W)
 * i32, steps [K] f64 (one per label) -> residual (H,W) f32; *consumed = symbols the label map needs. */
RPCC_API int rpcc_op_dequantize(const int16_t* symbols, int64_t n, const int32_t* seg, int H, int W, const double* steps,
                       int K, float* residual_out, int64_t* consumed);
/* The intensity section of one frame: points (n rows of x, y, z, intensity) -> owner_out [H][W] u32 (may be NULL) and
 * intensity_out [H][W] f32 (rpcc_project_batch + rpcc_intensity_owner_batch); intensity image + range -> the section's
 * bytes (out, room for the non-empty pixels; *n_out bytes; *flags_out bit3 if a value was clamped; may be NULL); and the
 * section (n bytes) + label map (1 = empty) -> intensity_out [H][W] f32.  The last refuses a section whose length is not
 * the label map's number of non-empty pixels. */
RPCC_API int rpcc_op_intensity_owner(const float* points, int64_t n, int H, int W, float hfov, float vmax, float vmin,
                             uint32_t* owner_out, float* intensity_out);
RPCC_API int rpcc_op_intensity_pack(const float* intensity, const float* range, int H, int W, double step, uint8_t* out,
                            int64_t* n_out, uint32_t* flags_out);
RPCC_API int rpcc_op_intensity_unpack(const uint8_t* q, int64_t n, const int32_t* seg, int H, int W, double step,
                              float* intensity_out);

/* ================================ batched encoder / decoder =================================== */
typedef struct rpcc_encoder rpcc_encoder;

typedef struct rpcc_encoder_config {
  int H, W;
  double hfov, vmax, vmin;     /* radians, as dataset/transformer.py:32-34 computes them */
  int cluster_num;             /* cfgs/compressor.yaml:22 */
  float ground_threshold;      /* cfgs/compressor.yaml:21 */
  double step;                 /* 2 * accuracy (tools/compress.py:46) */
  int nonuniform;              /* 0 uniform, 1 non-uniform */
  int level_num;               /* non-uniform: cfgs/compressor.yaml:7-14 */
  int level_kp_num[8];
  double level_dacc[8];
  int ground_level, feature_region, segments, sharp_num, less_sharp_num, flat_num;
  int max_batch;               /* frames per call */
  int64_t max_points;          /* total point rows per call */
  int device;                  /* CUDA device ordinal */
  int model_method;            /* 0 = point (cfgs/compressor.yaml:29), 1 = plane */
  float plane_angle_threshold; /* degrees, cfgs/compressor.yaml:30 */
  int host_chunk;              /* encode_host: frames per upload/kernels/download pipeline stage;
                                  0 = one frame per SM of the device, always capped at max_batch */
  int eval;                    /* 1: every call also decodes what it wrote and fills the --eval figures
                                  (rpcc_eval_batch; tools/compress_datalist.py:166-199).  2: the same, then the normals
                                  of both clouds (rpcc_normals_batch, RPCC_NORMAL_KNN / RPCC_NORMAL_RADIUS) and
                                  rpcc_p2plane_batch; eval_metrics rows are then RPCC_EVAL_COLS + RPCC_P2PLANE_COLS wide,
                                  the first RPCC_EVAL_COLS columns as with 1 */
  float eval_threshold_sq;     /* F-score threshold on the squared distance (0.02^2, utils/evaluate_metrics.py:9) */
  int segment_method;          /* 0 = FPS (cfgs/compressor.yaml:20), 1 = DBSCAN (rpcc_dbscan_segment_batch) */
  double dbscan_eps;           /* DBSCAN: neighbourhood radius in metres (cfgs/compressor.yaml: DBSCAN_eps), > 0 */
  int dbscan_min_points;       /* DBSCAN: neighbours of a core point, itself included, >= 1 */
  double intensity_step;       /* 0: no intensity section; > 0: 2 * intensity_accuracy -- every call also packs the
                                  intensity section (stride-4 points only; rpcc_encoder_encode_host_intensity) */
} rpcc_encoder_config;

RPCC_API int rpcc_encoder_create(const rpcc_encoder_config* cfg, rpcc_encoder** out);
RPCC_API void rpcc_encoder_destroy(rpcc_encoder* enc);
/* The encoder owns rpcc_encoder_slots() independent stream slots, each with buffers for max_batch
 * frames; results of a call stay in its slot until the slot is used again. */
RPCC_API int rpcc_encoder_slots(void);
/* Device-resident inputs (bench `value`): points/offsets as rpcc_project_batch (device pointers),
 * B <= max_batch; ground_in NULL => fitted on device, else [B][4] f32 (device or pinned host).
 * frame_keys: NULL, or [B] u64 on the device -- the keys of the deterministic RANSACs (ground plane, cluster
 * planes).  With NULL every frame has key 0: its sections depend on its points alone, whatever the batch size,
 * the frame's position in a datalist, the chunking of encode_host or the number of GPUs the list is sharded over.
 * Enqueues the whole chain on the slot's stream; no synchronisation. */
RPCC_API int rpcc_encoder_encode_device(rpcc_encoder* enc, int slot, const float* points, int stride,
                               const int64_t* offsets, int B, const float* ground_in, const uint64_t* frame_keys);
/* Host inputs/outputs (bench `e2e`, and what tools/compress_datalist.py calls): any B; frames are
 * cut into chunks of host_chunk (<= max_batch) and pipelined over the slots (upload / kernels / download
 * overlap; the upload of ~1.9 MB per 64E frame over PCIe is what bounds this call, so the chunks are
 * kept small enough that the link never idles behind a kernel batch).
 *   in : points_host rows of `stride` floats, offsets_host [B+1], ground_host [B][4] or NULL (fit on device),
 *        frame_keys [B] u64 (host) or NULL as rpcc_encoder_encode_device
 *   out: results [B]; model [B][K][4] f32; contour_bits [B][ceil(HW/8)]; seq: every frame's
 *        idx_sequence back to back (sum seq_count u16, capacity seq_cap entries); symbols likewise
 *        (sum sym_count i16, capacity sym_cap); salience [B][K] u8 (non-uniform; may be NULL);
 *        eval_metrics [B][RPCC_EVAL_COLS] f64 as rpcc_eval_batch fills them (encoder created with eval = 1), or
 *        [B][RPCC_EVAL_COLS + RPCC_P2PLANE_COLS] with rpcc_p2plane_batch's columns after them (eval = 2), or NULL.
 * Pinned host buffers make the copies asynchronous.  Synchronous: returns when everything is on the host. */
RPCC_API int rpcc_encoder_encode_host(rpcc_encoder* enc, const float* points_host, int stride, const int64_t* offsets_host,
                             int B, const float* ground_host, rpcc_frame_result* results, float* model,
                             uint8_t* contour_bits, uint16_t* seq, size_t seq_cap, int16_t* symbols,
                             size_t sym_cap, uint8_t* salience, const uint64_t* frame_keys, double* eval_metrics);
/* The same with the intensity section (encoder created with intensity_step > 0): intensity receives every frame's section
 * back to back, in the frames' symbol offsets (capacity sym_cap bytes).  rpcc_encoder_encode_host refuses such an
 * encoder, and this call refuses an encoder without intensity, so that the section is never dropped silently. */
RPCC_API int rpcc_encoder_encode_host_intensity(rpcc_encoder* enc, const float* points_host, int stride,
                                       const int64_t* offsets_host, int B, const float* ground_host,
                                       rpcc_frame_result* results, float* model, uint8_t* contour_bits, uint16_t* seq,
                                       size_t seq_cap, int16_t* symbols, size_t sym_cap, uint8_t* salience,
                                       const uint64_t* frame_keys, double* eval_metrics, uint8_t* intensity);
RPCC_API int rpcc_encoder_sync(rpcc_encoder* enc);
/* Per-stage device timing with CUDA events recorded on the slots' own streams between the stages of
 * every chain call (at most 256 calls per slot are kept).  rpcc_encoder_profile(enc, 1) starts a fresh
 * recording, (enc, 0) stops it.  rpcc_encoder_stage_times synchronises and returns the summed
 * milliseconds of the 8 stages {project, ground, fps, assign, keypoints, model (+ plane models), quantize, eval}, the frames
 * they cover and the number of chain calls.  With segment_method = 1, "fps" is DBSCAN and "assign" the label statistics. */
RPCC_API int rpcc_encoder_profile(rpcc_encoder* enc, int enable);
RPCC_API int rpcc_encoder_stage_times(rpcc_encoder* enc, double* ms_out, long long* frames_out, int* calls_out);
RPCC_API void* rpcc_encoder_stream(rpcc_encoder* enc, int slot);
/* Named device buffers of a slot (tests, chaining): "range","labels","model","symbols","seq","contour",
 * "results","center_idx","centers","ground","key_points","salience","step_per_label","sym_base",
 * "seq_base","lut","points","offsets","order","eval_range","eval_labels","eval_metrics", with eval = 2 also
 * "eval_normals_ref","eval_normals_rec","eval_p2plane", with segment_method = 1 "dbscan_workspace" (its counters as
 * rpcc_dbscan_segment_batch leaves them), with intensity_step > 0 "intensity_owner" ([B][HW] u32),
 * "intensity" ([B][HW] f32) and "intensity_stream" (u8, packed at "sym_base").  NULL if unknown / not allocated. */
RPCC_API void* rpcc_encoder_device_buffer(rpcc_encoder* enc, int slot, const char* name);

/* ================================ host entropy stage / file I/O (SURVEY 8(f) rank 2) ========================== */
/* The host side of tools/compress_datalist.py:91-141 as native threads: BasicCompressor.compress_dict +
 * save_compressed_bitstream (utils/compress_utils.py:167-179,255-310) for every frame of an encode_host call, on a
 * persistent pool, straight out of the caller's pinned output buffers.  Only method "bzip2" (the reference default,
 * cfgs/compressor.yaml:2; level 9 -- the bytes CPython's bz2.compress writes); deflate / lz4 stay on the Python pool.
 * Two coders produce those bytes, the system libbz2 and rpcc_bz2_compress; every worker measures both per section and
 * uses the cheaper one (environment RPCC_BZ2_CODER = auto | libbz2 | own). */
typedef struct rpcc_packer rpcc_packer;
RPCC_API int rpcc_packer_create(int threads, const char* method, rpcc_packer** out);
RPCC_API void rpcc_packer_destroy(rpcc_packer* pk);
/* Queue the B frames of one rpcc_encoder_encode_host result (same arrays, same layout: seq / symbols back to back in
 * frame order).  The arrays must stay untouched until rpcc_packer_wait(*ticket_out) has returned.
 * paths [B] (entries may be NULL): file to write; bytes_out [B]: file size; status_out [B]; blobs: optional in-memory
 * copies, frame b at blobs + b * blob_stride (RPCC_ERR_CAPACITY if a file is longer than blob_stride). */
RPCC_API int rpcc_packer_submit(rpcc_packer* pk, int B, int K, int cbytes, int uniform, const rpcc_frame_result* results,
                       const float* model, const uint8_t* contour_bits, const uint16_t* seq, const int16_t* symbols,
                       const uint8_t* salience, const char* const* paths, uint32_t* bytes_out, int* status_out,
                       uint8_t* blobs, size_t blob_stride, long long* ticket_out);
/* The same with a sixth section: intensity (rpcc_encoder_encode_host_intensity's output, frame b's sym_count bytes back to
 * back) appended after residual_quantized; NULL writes the five-section file of rpcc_packer_submit. */
RPCC_API int rpcc_packer_submit_intensity(rpcc_packer* pk, int B, int K, int cbytes, int uniform,
                                 const rpcc_frame_result* results, const float* model, const uint8_t* contour_bits,
                                 const uint16_t* seq, const int16_t* symbols, const uint8_t* salience,
                                 const uint8_t* intensity, const char* const* paths, uint32_t* bytes_out,
                                 int* status_out, uint8_t* blobs, size_t blob_stride, long long* ticket_out);
RPCC_API int rpcc_packer_wait(rpcc_packer* pk, long long ticket);
/* bz2.compress(src) (utils/compress_utils.py:296-298: bzip2, level 9) by this library's own encoder (bz2enc.cu: the same
 * bitstream as libbz2, rotations sorted by induced sorting).  Returns RPCC_OK, RPCC_BZ2_DECLINED (1: input this encoder
 * leaves to libbz2 -- more than one block, or a block made of repetitions of a shorter string) or RPCC_ERR_CAPACITY. */
#define RPCC_BZ2_DECLINED 1
RPCC_API int rpcc_bz2_compress(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, size_t* out_len);
/* The inverse (BasicCompressor.bzip2_decompress = bz2.decompress, utils/compress_utils.py:300-302): the decoded bytes of
 * the .bz2 stream src[0..n) into dst.  Table-driven Huffman decoding, 64-bit bit buffer; both CRCs are checked.  Returns
 * RPCC_OK, RPCC_BZ2_DECLINED (a randomised block or a stream this decoder finds malformed: give it to libbz2, whose
 * verdict then counts) or RPCC_ERR_CAPACITY.  rpcc_unpack_rpcc uses it first (environment RPCC_BZ2_DECODER = own | libbz2). */
RPCC_API int rpcc_bz2_decompress(const uint8_t* src, size_t n, uint8_t* dst, size_t cap, size_t* out_len);
/* dataset/dataset.py:57-63 for a KITTI .bin (rows of x,y,z,intensity f32): the xyz columns into dst (room for
 * cap_rows rows of 3 floats, typically a slice of the pinned upload buffer); *rows_out = rows in the file. */
RPCC_API int rpcc_read_bin_xyz(const char* path, float* dst, int64_t cap_rows, int64_t* rows_out);
/* The same keeping the intensity: whole rows of 4 floats into dst (room for cap_rows rows). */
RPCC_API int rpcc_read_bin_rows(const char* path, float* dst, int64_t cap_rows, int64_t* rows_out);
/* read_compressed_bitstream + BasicCompressor.decompress_dict (utils/compress_utils.py:182-196,263-310), bzip2:
 * sections decompressed back to back into dst; sec_len [5] in file order (4 sections when uniform). */
RPCC_API int rpcc_unpack_rpcc(const uint8_t* blob, size_t n, int uniform, uint8_t* dst, size_t cap, uint32_t* sec_len);
/* The same including the intensity section after residual_quantized: sec_len [6] (the intensity last, at index 5 also
 * when uniform); a file without it is an error. */
RPCC_API int rpcc_unpack_rpcc_intensity(const uint8_t* blob, size_t n, int uniform, uint8_t* dst, size_t cap,
                                uint32_t* sec_len);

#ifdef __cplusplus
}
#endif
#endif /* RPCC_B200_H_ */
