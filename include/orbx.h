/*
 * orbx.h -- C-ABI of liborbx.so: B200-native (sm_100a) ORB extraction + brute-force Hamming matching.
 *
 * This is the drop-in boundary for the ONE hot path of BowenBZ/RGBD_VisualOdometry.  The reference has
 * no FFI/plugin layer; the operator interface the path sits behind is OpenCV's C++ one, called from the
 * front-end thread at exactly two sites (plus the same pair in a dead function):
 *
 *   orb_->detectAndCompute(frameCurr_->color_, Mat(), keypointsCurr_, descriptorsCurr_)   src/frontend.cpp:153 (dead: :422)
 *   flannMatcher_.match(mptCandidatesDescriptors, descriptorsCurr_, matches)             src/frontend.cpp:187 (dead: :439)
 *
 * with the operators constructed at src/frontend.cpp:33 (matcher) and :35-37 (ORB: number_of_features,
 * scale_factor, level_pyramid from config/default.yaml:18-20; everything else is an OpenCV default:
 * edgeThreshold 31, firstLevel 0, WTA_K 2, HARRIS_SCORE, patchSize 31, fastThreshold 20).
 * INTEGRATION.md shows the <=40-line shim that binds these entry points into FrontEnd.
 *
 * Conventions (mirroring how the reference uses the OpenCV operators):
 *   - plain pointers and sizes only; no C++ / torch / OpenCV types; the library never throws.
 *   - every function returns ORBX_OK (0) or a negative orbx_status; orbx_last_error() gives the text.
 *   - outputs are caller-allocated with an explicit capacity.  OpenCV's retainBest keeps ties, so the
 *     keypoint count can EXCEED nfeatures (e.g. 521 for nfeatures = 500); if it exceeds the capacity the
 *     call returns ORBX_E_CAPACITY with *n_out = needed and writes nothing partial to rely on.
 *   - orbx_keypoint / orbx_match are byte-identical to cv::KeyPoint (28 B) / cv::DMatch (16 B), so the shim
 *     is a memcpy; all seven KeyPoint fields are filled exactly as OpenCV fills them (util.h:52-68 hashes them all).
 *   - one context per (GPU, caller thread); a context is NOT thread-safe (the reference only ever calls
 *     these operators from the front-end thread, src/frontend.cpp:94-144).
 *   - empty image / no keypoints -> ORBX_OK with *n_out = 0; empty query or train set -> ORBX_OK, 0 matches
 *     (cv::DescriptorMatcher::match semantics).
 *   - there is NO CPU fallback: without a CUDA device orbx_create fails with ORBX_E_CUDA.
 */
#ifndef ORBX_H_
#define ORBX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORBX_MAX_LEVELS 16
#define ORBX_DESC_BYTES 32
#define ORBX_MAX_KNN 32   /* largest k of the knnMatch entry points (orbx_match_hamming_*knn) */

typedef struct orbx_ctx orbx_ctx; /* opaque */

/* == cv::KeyPoint: pt.x, pt.y, size, angle, response, octave, class_id */
typedef struct { float x, y, size, angle, response; int32_t octave, class_id; } orbx_keypoint;
/* == cv::DMatch: queryIdx, trainIdx, imgIdx, distance */
typedef struct { int32_t queryIdx, trainIdx, imgIdx; float distance; } orbx_match;

typedef enum {
    ORBX_OK = 0,
    ORBX_E_ARG = -1,         /* bad argument (null pointer, size over the context maximum, ...) */
    ORBX_E_CAPACITY = -2,    /* caller's output capacity too small; *n_out holds the needed count */
    ORBX_E_CUDA = -3,        /* CUDA runtime / driver error, or no device */
    ORBX_E_NOMEM = -4,       /* host or device allocation failed */
    ORBX_E_UNSUPPORTED = -5, /* valid OpenCV input this build does not cover (e.g. channels not 1 or 3) */
    ORBX_E_INTERNAL = -6,    /* an internal device-side bound was exceeded (never silently truncated) */
    ORBX_E_BUSY = -8,        /* orbx_submit_frame: two frames are already in flight */
    ORBX_E_ORDER = -7        /* reserved (was: introselect depth-limit fallback not reproduced; the fallback is implemented now) */
} orbx_status;

/* ---- lifecycle ----------------------------------------------------------------------------------- */

/* Replaces cv::ORB::create(nfeatures, scaleFactor, nlevels) + the matcher construction
 * (src/frontend.cpp:33-37).  max_w/max_h/max_batch size the device-resident buffers. */
int orbx_create(orbx_ctx** out, int device, int nfeatures, float scale_factor, int nlevels,
                int max_w, int max_h, int max_batch);
void orbx_destroy(orbx_ctx* ctx);
const char* orbx_last_error(const orbx_ctx* ctx);
const char* orbx_version(void);
/* Blocks until all work queued on the context's stream is done; returns any deferred device status. */
int orbx_synchronize(orbx_ctx* ctx);
/* The CUDA stream (cudaStream_t) the context launches on, for callers that time with CUDA events. */
void* orbx_stream(orbx_ctx* ctx);
/* Number of kernels this library has launched on the context since creation (bench bookkeeping). */
uint64_t orbx_launch_count(const orbx_ctx* ctx);

/* ---- ORB extraction: replaces cv::Feature2D::detectAndCompute(image, Mat(), kps, desc) ----------- */

/* One frame, HOST buffers (the literal drop-in for src/frontend.cpp:153).
 * img: h rows of `step` bytes; channels 3 = BGR 8UC3 (as cv::imread gives, app/run_vo.cpp:91), 1 = gray 8UC1.
 * kps: cap records, desc: cap*32 bytes.  *n_out = number of keypoints (order == OpenCV's). */
int orbx_detect_and_compute(orbx_ctx* ctx, const uint8_t* img, int w, int h, size_t step, int channels,
                            orbx_keypoint* kps, uint8_t* desc, int cap, int* n_out);

/* `batch` same-sized frames, HOST buffers.  imgs[i] as above; outputs are [batch][cap] / [batch][cap][32];
 * n_out[batch].  Returns ORBX_E_CAPACITY if any frame needs more than cap (n_out[] then holds the needs). */
int orbx_detect_and_compute_batch(orbx_ctx* ctx, const uint8_t* const* imgs, int batch, int w, int h, size_t step,
                                  int channels, orbx_keypoint* kps, uint8_t* desc, int cap, int* n_out);

/* Host buffers of the two calls above (and of orbx_extract_match_batch) may be pageable -- the reference's frames are
 * cv::Mat (src/frame.cpp:28) and its results std::vector / cv::Mat (frontend.h:69-70): the library then stages them through
 * its own pinned memory with a few copier threads (ORBX_STAGE_THREADS, default min(8, cores / 2)), so uploads, kernels and
 * downloads of neighbouring frame ranges still overlap.  Page-locked buffers (cudaHostAlloc, cudaHostRegister, or
 * orbx_host_register below) are copied from / into directly, which is faster still.
 * orbx_host_register page-locks a LONG-LIVED caller buffer (e.g. the ring of frame buffers of a capture loop) without the
 * caller linking CUDA; it must be unregistered before the memory is freed.  Returns ORBX_E_CUDA if the range cannot be locked. */
int orbx_host_register(orbx_ctx* ctx, void* ptr, size_t bytes);
int orbx_host_unregister(orbx_ctx* ctx, void* ptr);

/* `batch` frames already DEVICE-resident (frame i at d_imgs + i*frame_stride); outputs to device memory
 * ([batch][cap] records, [batch][cap][32] bytes, d_counts[batch]).  Asynchronous on orbx_stream(); per-frame
 * status is deferred to orbx_synchronize().  d_counts[i] may exceed cap (records beyond cap are not written). */
int orbx_detect_and_compute_device(orbx_ctx* ctx, const uint8_t* d_imgs, int batch, int w, int h, size_t step,
                                   size_t frame_stride, int channels, orbx_keypoint* d_kps, uint8_t* d_desc,
                                   int cap, int* d_counts);

/* Asynchronous form of the one-frame call for the sequential VO loop (app/run_vo.cpp:66-110, SURVEY 8(f).4): submit copies
 * the image into pinned staging and queues upload, kernels and download, returning at once, so the host can run PnP / BA
 * of frame i (or decode frame i+2) while the GPU extracts frame i+1; collect blocks until the OLDEST submitted frame is
 * done and hands out its keypoints and descriptors (same results as orbx_detect_and_compute).  At most two frames in
 * flight (ORBX_E_BUSY beyond).  The collected frame also becomes "frame 0 of the last extraction" for orbx_track_match /
 * orbx_map_upsert_from_frame -- until a later orbx_submit_frame reuses the slot that holds it (the second submit after the
 * collect): from then on those calls return ORBX_E_ARG instead of silently reading the newer frame, so call them between the
 * collect and that submit (the order INTEGRATION.md shows).  A frame whose device-side status flag is set is never handed
 * out: collect drops it and returns ORBX_E_INTERNAL, exactly as the synchronous call does. */
int orbx_submit_frame(orbx_ctx* ctx, const uint8_t* img, int w, int h, size_t step, int channels);
int orbx_collect_frame(orbx_ctx* ctx, orbx_keypoint* kps, uint8_t* desc, int cap, int* n_out);

/* ---- matching: replaces cv::DescriptorMatcher::match(query, train, matches) as exact
 *      BFMatcher(NORM_HAMMING): one DMatch per query row, ties -> lowest trainIdx, distance = (float)hamming,
 *      imgIdx = 0.  query = the map-point candidates (M x 32), train = the frame descriptors (N x 32)
 *      (src/frontend.cpp:183-187). -------------------------------------------------------------------- */

/* HOST buffers.  out: nq records.  *n_out = nq, or 0 when either set is empty. */
int orbx_match_hamming(orbx_ctx* ctx, const uint8_t* query, int nq, const uint8_t* train, int nt,
                       orbx_match* out, int* n_out);
/* knnMatch(k = 2): out holds 2*nq records, [2*i] best, [2*i+1] second best by (distance, index);
 * when nt == 1 the second record has trainIdx = -1. */
int orbx_match_hamming_knn2(orbx_ctx* ctx, const uint8_t* query, int nq, const uint8_t* train, int nt,
                            orbx_match* out, int* n_out);
/* knnMatch(query, train, k) for any 1 <= k <= ORBX_MAX_KNN, HOST buffers: out holds [nq][k] records; record r of query i
 * is its r-th nearest train row by (distance, trainIdx), exactly cv's list; records r >= nt have trainIdx = -1, distance 0.
 * *n_out = nq (0 if either set is empty).  k = 1 gives orbx_match_hamming's records, k = 2 orbx_match_hamming_knn2's.
 * k < 1 -> ORBX_E_ARG; k > ORBX_MAX_KNN or nt >= 2^20 -> ORBX_E_UNSUPPORTED. */
int orbx_match_hamming_knn(orbx_ctx* ctx, const uint8_t* query, int nq, const uint8_t* train, int nt, int k,
                           orbx_match* out, int* n_out);
/* DEVICE-resident, asynchronous, batched over `nsets` independent train sets (frames) that share one
 * query set (the map): d_train is [nsets][nt][32], d_best / d_second are [nsets][nq] (d_second may be NULL). */
int orbx_match_hamming_device(orbx_ctx* ctx, const uint8_t* d_query, int nq, const uint8_t* d_train, int nt,
                              int nsets, orbx_match* d_best, orbx_match* d_second);
/* Ragged variant: set s holds min(d_train_counts[s], train_stride_rows) valid rows at d_train + s*train_stride_rows*32
 * (exactly the [batch][cap][32] / d_counts layout orbx_detect_and_compute_device writes, so extraction feeds matching
 * without a host round trip).  A query matched against an empty set gets trainIdx = -1, distance = 0. */
int orbx_match_hamming_device_ragged(orbx_ctx* ctx, const uint8_t* d_query, int nq, const uint8_t* d_train,
                                     int train_stride_rows, const int* d_train_counts, int nsets,
                                     orbx_match* d_best, orbx_match* d_second);
/* knnMatch form of the ragged batch (layout as orbx_match_hamming_device_ragged): d_out is [nsets][nq][k], set s's records
 * of query i at d_out + (s*nq + i)*k, as orbx_match_hamming_knn; an empty set gives k records with trainIdx = -1,
 * distance 0.  nq = 0, train_stride_rows = 0 or nsets = 0 launches nothing.  k < 1, null pointers, negative sizes or
 * nsets > 65535 -> ORBX_E_ARG; k > ORBX_MAX_KNN or a stride of 2^20 rows or more -> ORBX_E_UNSUPPORTED. */
int orbx_match_hamming_device_knn(orbx_ctx* ctx, const uint8_t* d_query, int nq, const uint8_t* d_train, int train_stride_rows,
                                  const int* d_train_counts, int nsets, int k, orbx_match* d_out);
/* HOST-buffer form of the ragged batched match: one map (query) against `nsets` frames' descriptor sets
 * ([nsets][train_stride_rows][32] with train_counts[nsets]); best / second are [nsets][nq] (second may be NULL). */
int orbx_match_hamming_sets(orbx_ctx* ctx, const uint8_t* query, int nq, const uint8_t* train, int train_stride_rows,
                            const int* train_counts, int nsets, orbx_match* best, orbx_match* second);
/* BFMatcher(NORM_HAMMING, crossCheck = true).match(query, train), HOST buffers.  out: capacity nq records;
 * *n_out = number of mutual pairs, ascending queryIdx.  Empty query or train -> ORBX_OK, 0 (cv2 raises on an empty train).
 * A pair (i, j) is kept when j is query i's nearest train row and i is train row j's nearest query, the lowest index
 * winning ties in both directions.  nq >= 2^20 -> ORBX_E_UNSUPPORTED. */
int orbx_match_hamming_crosscheck(orbx_ctx* ctx, const uint8_t* query, int nq, const uint8_t* train, int nt,
                                  orbx_match* out, int* n_out);
/* DEVICE-resident, asynchronous, ragged batch (d_train / d_train_counts exactly as orbx_match_hamming_device_ragged):
 * set s's mutual pairs compacted to d_out + s*nq (ascending queryIdx), their count in d_n_out[s].  The reverse direction
 * (each train row's nearest query) comes out of the same distance tiles, with no second pass.  nq = 0 or
 * train_stride_rows = 0 zeroes d_n_out[0 .. nsets). */
int orbx_match_hamming_device_crosscheck(orbx_ctx* ctx, const uint8_t* d_query, int nq, const uint8_t* d_train,
                                         int train_stride_rows, const int* d_train_counts, int nsets,
                                         orbx_match* d_out, int* d_n_out);
/* PAIRWISE batch, DEVICE-resident, asynchronous: pair p matches query set p against train set p (per-frame candidate
 * sets, frame-to-frame, stereo or keyframe pairs), all pairs in one launch.  Query set p: min(d_query_counts[p],
 * query_stride_rows) rows at d_query + p*query_stride_rows*32 (a negative count is 0); train set p likewise with
 * d_train / train_stride_rows / d_train_counts.  These are exactly the layouts orbx_detect_and_compute_device writes, so
 * frame-to-frame matching of a batch is d_query = desc, d_train = desc + cap*32, d_query_counts = counts,
 * d_train_counts = counts + 1, both strides cap, npairs = batch - 1.  An arbitrary list of pairs is gathered into such
 * sets first.  Per pair the results equal BFMatcher(NORM_HAMMING).match (and knnMatch(k = 2) with d_second) of that
 * pair's rows: queryIdx / trainIdx index the pair's own sets, imgIdx = 0.  d_best / d_second (NULL: no second) are
 * [npairs][query_stride_rows]; record i of pair p is written for i < that pair's query count only; an empty train set
 * gives trainIdx = -1, distance = 0.  npairs = 0 or a stride of 0 launches nothing.  Null pointers, negative sizes or
 * npairs > 65535 -> ORBX_E_ARG; a stride of 2^20 rows or more -> ORBX_E_UNSUPPORTED. */
int orbx_match_hamming_device_pairwise(orbx_ctx* ctx, const uint8_t* d_query, int query_stride_rows, const int* d_query_counts,
                                       const uint8_t* d_train, int train_stride_rows, const int* d_train_counts, int npairs,
                                       orbx_match* d_best, orbx_match* d_second);
/* As above with crossCheck = true: pair p's mutual pairs compacted to d_out + p*query_stride_rows (ascending queryIdx),
 * their count in d_n_out[p].  A stride of 0 zeroes d_n_out[0 .. npairs). */
int orbx_match_hamming_device_pairwise_crosscheck(orbx_ctx* ctx, const uint8_t* d_query, int query_stride_rows,
                                                  const int* d_query_counts, const uint8_t* d_train, int train_stride_rows,
                                                  const int* d_train_counts, int npairs, orbx_match* d_out, int* d_n_out);
/* knnMatch form of the pairwise batch (layouts and count rules as orbx_match_hamming_device_pairwise): d_out is
 * [npairs][query_stride_rows][k]; the k records of query i of pair p are written for i < that pair's query count only.
 * k < 1 -> ORBX_E_ARG; k > ORBX_MAX_KNN -> ORBX_E_UNSUPPORTED; other argument rules as the pairwise call. */
int orbx_match_hamming_device_pairwise_knn(orbx_ctx* ctx, const uint8_t* d_query, int query_stride_rows, const int* d_query_counts,
                                           const uint8_t* d_train, int train_stride_rows, const int* d_train_counts, int npairs,
                                           int k, orbx_match* d_out);
/* radiusMatch(query, train, maxDistance): for every query row, every train row at Hamming distance <= maxDistance, in
 * cv::BFMatcher(NORM_HAMMING).radiusMatch's exact list order.  That order is libstdc++'s std::sort by distance alone (an
 * unstable introsort) of the rows in ascending trainIdx, NOT (distance, trainIdx): equal distances can come out in any
 * index order once a list holds more than 16 entries.  Output is CSR: list L occupies out[offsets[L] .. offsets[L + 1])
 * (offsets are 64-bit), records {queryIdx, trainIdx, 0, distance} with indices local to the set or pair.  The integer radius
 * is R = min(256, floor(max_distance)), so +inf or any value >= 256 keeps every row.  max_distance <= FLT_EPSILON or NaN
 * (cv asserts), null pointers or negative sizes -> ORBX_E_ARG; a train set (stride) of 2^20 rows or more ->
 * ORBX_E_UNSUPPORTED.  cv's crossCheck does not apply to radiusMatch: its lists are these.
 * HOST buffers: lists [nq], offsets has nq + 1 entries; *n_out = offsets[nq] = the number of records.  If that exceeds cap
 * the call returns ORBX_E_CAPACITY with *n_out = the number needed.  An empty train set gives nq empty lists (all offsets
 * 0), an empty query set none. */
int orbx_match_hamming_radius(orbx_ctx* ctx, const uint8_t* query, int nq, const uint8_t* train, int nt, float max_distance,
                              orbx_match* out, int cap, int64_t* offsets, int* n_out);
/* Ragged DEVICE batch (layout as orbx_match_hamming_device_ragged), asynchronous: list L = s*nq + i is query i against set
 * s, d_offsets has nsets*nq + 1 entries.  d_offsets is always written in full; list L's records are written only when
 * d_offsets[L + 1] <= cap (as orbx_detect_and_compute_device, records beyond cap are not written), so a caller reads
 * d_offsets[nsets*nq] and calls again with a larger buffer.  nq = 0, train_stride_rows = 0 or nsets = 0 launches nothing
 * and zeroes d_offsets; nsets > 65535 or cap < 0 -> ORBX_E_ARG. */
int orbx_match_hamming_device_radius(orbx_ctx* ctx, const uint8_t* d_query, int nq, const uint8_t* d_train, int train_stride_rows,
                                     const int* d_train_counts, int nsets, float max_distance, orbx_match* d_out, int64_t cap,
                                     int64_t* d_offsets);
/* PAIRWISE DEVICE batch (layouts and count rules as orbx_match_hamming_device_pairwise), asynchronous: list
 * L = p*query_stride_rows + i is query i of pair p against train set p; d_offsets has npairs*query_stride_rows + 1 entries.
 * Query rows past a pair's count have empty lists.  cap and d_offsets as the ragged form. */
int orbx_match_hamming_device_pairwise_radius(orbx_ctx* ctx, const uint8_t* d_query, int query_stride_rows, const int* d_query_counts,
                                              const uint8_t* d_train, int train_stride_rows, const int* d_train_counts, int npairs,
                                              float max_distance, orbx_match* d_out, int64_t cap, int64_t* d_offsets);
/* The front-end's whole per-frame pattern on HOST frames in one call (src/frontend.cpp:98-108: one detectAndCompute,
 * then match() of map-point candidates against the frame's descriptors, src/frontend.cpp:153 + :187), for a batch:
 * extraction as orbx_detect_and_compute_batch, then for each of the `nmaps` query sets (queries[j]: nq[j] x 32 host
 * rows = the map candidates) one exact Hamming match against every frame's own descriptors; best[j] receives
 * [batch][nq[j]] records (trainIdx = -1 where a frame has no keypoints).  The batch is cut into frame ranges that
 * run upload -> kernels -> download on their own streams, so the PCIe copies of one range sit under the kernels of
 * the others and the descriptors never make a host round trip between extraction and matching. */
int orbx_extract_match_batch(orbx_ctx* ctx, const uint8_t* const* imgs, int batch, int w, int h, size_t step, int channels,
                             orbx_keypoint* kps, uint8_t* desc, int cap, int* n_out, const uint8_t* const* queries,
                             const int* nq, int nmaps, orbx_match* const* best);
/* The reference's host-side post-filter (src/frontend.cpp:190-211): keep distance <= max(min*ratio, 30).
 * Pure host helper for the shim; in place compaction, returns the kept count. */
int orbx_filter_matches(orbx_match* matches, int n, float match_ratio);

/* ---- the callers either side of the matcher (SURVEY.md 8(f)): device-resident map table, candidate visibility
 *      filter, match post-filter, depth back-projection ------------------------------------------------------
 *
 * The reference gathers the candidate descriptors on the host for EVERY match call: it walks trackingMap_, tests
 * Frame::IsCouldObserveMappoint per point and push_back()s Mappoint::descriptor_ rows into a fresh cv::Mat
 * (src/frontend.cpp:169-184), then thresholds the matches on the host (:190-211).  Here the map points live in a
 * slot-addressed table in HBM keyed by the reference's map-point id (Mappoint::id_, size_t), and one call does
 * filter -> gather -> match -> threshold on the device.  Poses are T_c_w as a row-major 3 x 4 [R | t]
 * (Frame::T_c_w_, SE3::matrix3x4()); cam = {fx, fy, cx, cy} (src/camera.cpp:27-30).  Geometry is double precision in
 * the reference's operation order (parity to 1e-9 relative: the reference binary is compiled with FMA contraction). */

/* Pre-size the table (it grows on demand). */
int orbx_map_reserve(orbx_ctx* ctx, int capacity);
int orbx_map_size(const orbx_ctx* ctx);
int orbx_map_clear(orbx_ctx* ctx);
/* Insert or update `n` map points (MapManager::InsertMappoint, src/frontend.cpp:396-399; Mappoint::SetPosition after BA;
 * Mappoint::outlier_ set by the backend).  desc: n x 32 rows, pos / norm: n x 3 doubles (Mappoint::pos_, norm_), outlier:
 * n bytes.  A NULL column is left unchanged for known ids and zero for new ones.  Host buffers, borrowed for the call. */
int orbx_map_upsert(orbx_ctx* ctx, const int64_t* ids, int n, const uint8_t* desc, const double* pos, const double* norm,
                    const uint8_t* outlier);
/* As above, but the descriptor rows are copied device -> device out of frame `frame` of the last host-API extraction
 * (keypoint indices kp_index[n]): the device form of descriptorsCurr_.row(idx).clone(), src/frontend.cpp:392-394. */
int orbx_map_upsert_from_frame(orbx_ctx* ctx, const int64_t* ids, int n, int frame, const int32_t* kp_index, const double* pos,
                               const double* norm);
int orbx_map_erase(orbx_ctx* ctx, const int64_t* ids, int n);
/* FrontEnd::MatchKeyPointsInTrackingMap (src/frontend.cpp:156-215) for the tracking map `ids[m]` (in the caller's
 * iteration order): candidates = points that are not outliers and pass Frame::IsCouldObserveMappoint (src/frame.cpp:70-91:
 * in front of the camera, projects inside cols x rows, viewing angle <= pi/6); cand[] receives their positions in ids[]
 * (*n_cand of them, order kept); they are matched against the train descriptors -- host rows `train` (nt_or_frame = row
 * count) or, when train is NULL, frame `nt_or_frame` of the last host-API extraction -- and matches[] receives the
 * DMatch records with distance <= max(min_distance * match_ratio, 30) (*n_matches, queryIdx = index into cand[]).
 * An unknown id is ORBX_E_ARG.  Empty candidate or train set -> no matches (the reference dereferences end() there). */
int orbx_track_match(orbx_ctx* ctx, const int64_t* ids, int m, const double* pose_Tcw, const double* cam, int cols, int rows,
                     const uint8_t* train, int nt_or_frame, float match_ratio, int32_t* cand, int* n_cand, orbx_match* matches,
                     int* n_matches, float* min_dis, float* max_dis);
/* FrontEnd::CreateNewMappoints' geometry (src/frontend.cpp:372-389): Frame::GetDepth (src/frame.cpp:43-67: cvRound'ed
 * pixel, else its left / up / right / down neighbour, depth = d / depth_scale) and Camera::Pixel2World
 * (src/camera.cpp:56-86) for n keypoints.  depth: h rows of step_bytes, 16UC1.  pos_w: n x 3, valid: n (0 = no depth). */
int orbx_backproject(orbx_ctx* ctx, const orbx_keypoint* kps, int n, const uint16_t* depth, int w, int h, size_t step_bytes,
                     float depth_scale, const double* cam, const double* pose_Tcw, double* pos_w, uint8_t* valid);

/* ---- introspection for stage-level parity tests (not needed by the shim) ------------------------- */

/* Geometry of the pyramid the context would build for a w x h frame. */
int orbx_level_geometry(const orbx_ctx* ctx, int w, int h, int* ws, int* hs, float* scales, int* quotas);
/* Copies pyramid level `level` of frame `frame` of the LAST extraction call to host (w_l*h_l bytes, tight). */
int orbx_debug_read_level(orbx_ctx* ctx, int frame, int level, uint8_t* out, size_t out_bytes);
/* Raster-ordered, border-filtered FAST+NMS survivors of the last call: x[], y[], score[] (cap entries each);
 * *n_out = count. */
int orbx_debug_read_fast(orbx_ctx* ctx, int frame, int level, int32_t* x, int32_t* y, int32_t* score, int cap, int* n_out);
/* Average device time (ms) of each pipeline stage over the last extraction / match call, measured with CUDA
 * events on the context's stream; names[i] are static strings.  Returns the number of stages written. */
int orbx_debug_stage_times(orbx_ctx* ctx, const char** names, float* ms, int cap);
/* Pyramid, FAST and selection exist as two kernel families with identical results: warp-private kernels (pyramid / FAST:
 * TMA-fed, chosen for launches of about 26 VGA frames' worth of pixels and more; selection: one warp per (frame, level), chosen
 * for frames up to about 0.6 Mpixel) and CTA-cooperative kernels with the shorter critical path (smaller launches, e.g. the
 * one-frame calls of the VO loop; selection on large frames).  mode -1: by launch size / frame size (default), 0 / 1: always
 * the former / latter (tests run the golden vectors through both). */
int orbx_debug_force_kernels(orbx_ctx* ctx, int mode);

/* Enable (1) / disable (0) per-stage CUDA-event timing (adds event records between kernels). */
int orbx_set_profiling(orbx_ctx* ctx, int enable);

#ifdef __cplusplus
}
#endif
#endif /* ORBX_H_ */
