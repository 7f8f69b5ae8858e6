/* hvo_capi.h — C ABI of libhvofront.so, the B200-native (sm_100a) feature front-end.
 *
 * The reference (ORB-SLAM2-derived hybrid VO) has no plugin/FFI registry; its boundary for this path is the
 * public C++ class surface called by Frame/Tracking.  Each entry point below names the reference interface
 * it replaces (paths relative to the reference tree).  The C++ shim classes under
 * a-low-texture-robust-hybrid-feature-based-visual-odometry_b200/shim/ keep the reference's signatures and
 * forward here; INTEGRATION.md shows the binding a maintainer adds.
 *
 * Conventions: every call returns an int status (HVO_OK == 0); hvo_last_error() returns a thread-local
 * message for the last non-zero status; no exceptions cross the ABI; the caller owns every buffer it
 * passes; a handle owns its device buffers and one non-blocking CUDA stream; calls on different handles
 * are thread-safe, calls on one handle must be serialised by the caller (the reference's usage model:
 * one long-lived extractor per Tracking thread, src/Tracking.cc:124).  There is NO CPU fallback: without a
 * CUDA device every create call fails with HVO_ERR_CUDA.
 */
#ifndef HVO_CAPI_H
#define HVO_CAPI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HVO_OK 0
#define HVO_ERR_ARG 1      /* bad argument (null pointer, size out of range, capacity too small) */
#define HVO_ERR_CUDA 2     /* CUDA runtime / launch failure, or no device */
#define HVO_ERR_STATE 3    /* call not valid in the handle's current state */
#define HVO_ERR_OVERFLOW 4 /* an internal fixed-capacity buffer would overflow (reported, never silent) */

#define HVO_MAX_LEVELS 12

const char* hvo_last_error(void);
int hvo_device_count(int* n_out);
/* library build info, e.g. "hvofront sm_100a <date>" */
const char* hvo_version(void);
/* Profiling aid: with the timeline enabled every kernel launch site first records a timed event on its stream;
 * hvo_timeline_dump (after the work is synchronised) writes one line per mark: "ms-since-first-mark stream-id name". */
int hvo_timeline_enable(int on);
int hvo_timeline_dump(char* buf, int capacity);

/* ------------------------------------------------------------------------------------------------ ORB
 * Replaces ORB_SLAM2::ORBextractor (include/ORBextractor.h:46-110, src/ORBextractor.cc).              */

typedef struct hvo_orb hvo_orb;

/* ORBextractor::ORBextractor(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST)  ORBextractor.h:51-52 */
typedef struct hvo_orb_params {
    int nfeatures;
    float scale_factor;
    int nlevels;
    int ini_th_fast;
    int min_th_fast;
} hvo_orb_params;

/* cv::KeyPoint POD layout (28 bytes): pt.x, pt.y, size, angle, response, octave, class_id */
typedef struct hvo_keypoint {
    float x, y, size, angle, response;
    int32_t octave, class_id;
} hvo_keypoint;

/* Optional RGB-D epilogue = Frame::ComputeStereoFromRGBD (src/Frame.cc:1940-1961) fused after extraction.
 * depth is raw 16-bit (TUM: metres*5000); depth_factor = 1/DepthMapFactor (src/Tracking.cc:156-160).
 * kp_depth (mvDepth) is sampled at the DISTORTED keypoint, as the reference does (Frame.cc:1948-1951), and is always valid.
 * kp_uright (mvuRight) is kpU.pt.x - bf / d with kpU the UNDISTORTED keypoint (Frame.cc:1944, 1957).  The extract calls form it
 * only for a camera without distortion (mvKeysUn == mvKeys, Frame.cc:1703-1707).  For any other camera (TUM1.yaml, TUM2.yaml,
 * ICSL_LPVO.yaml have k1 != 0) set `distorted`: kp_uright is then filled with -1, and hvo_orb_undistort_batch_device() forms
 * mvKeysUn and mvuRight on the device right after the extraction (the frame handle does this itself when hvo_frame_params
 * carries the coefficients).  hvo_stereo_uright_from_depth() is the host form for keypoints undistorted elsewhere. */
typedef struct hvo_rgbd_params {
    float depth_factor; /* metres per raw unit, e.g. 1/5000 */
    float bf;           /* stereo baseline * fx (Camera.bf) */
    int distorted;      /* != 0: Camera.k1 != 0, kp_uright is not formed by the extract call */
} hvo_rgbd_params;

/* mvuRight of a distorted camera, host side: uright[i] = keys_un[i].x - bf / kp_depth[i] where kp_depth[i] > 0, else -1
 * (the second half of Frame::ComputeStereoFromRGBD, Frame.cc:1953-1958, on the undistorted keypoints). */
int hvo_stereo_uright_from_depth(const hvo_keypoint* keys_un, const float* kp_depth, int n, float bf, float* uright);

/* mK and mDistCoef as the reference holds them (CV_32F): DistCoef = k1, k2, p1, p2, and k3 when Camera.k3 != 0 (k3 = 0 otherwise). */
typedef struct hvo_camera {
    float fx, fy, cx, cy;
    float k1, k2, p1, p2, k3;
} hvo_camera;

/* cv::undistortPoints(xy, xy_un, mK, mDistCoef, noArray(), mK) of OpenCV 4.13, bit for bit: xy / xy_un are n (x, y) float pairs
 * (may alias).  Plain cv::undistortPoints, without the k1 == 0 shortcut of Frame::UndistortKeyPoints.  Host function, no CUDA. */
int hvo_undistort_points(const hvo_camera* cam, const float* xy, int n, float* xy_un);
/* Frame::ComputeImageBounds (src/Frame.cc:1733-1760): mnMinX = min of the undistorted corners (0,0), (0,rows); mnMaxX = max of
 * (cols,0), (cols,rows); likewise in y.  k1 == 0 gives 0, width, 0, height, as the reference tests only k1.  Host function. */
int hvo_image_bounds(const hvo_camera* cam, int width, int height, float* min_x, float* max_x, float* min_y, float* max_y);
/* Frame::UndistortKeyPoints + the mvuRight half of ComputeStereoFromRGBD on device-resident extraction results, asynchronous on the
 * handle's stream (so it follows a hvo_orb_extract_batch_device call in order).  Rows [f][i] with i < d_counts[f] of the
 * [nframes][hvo_orb_capacity] arrays are read; d_kps_un (may be NULL) receives the keypoint with x, y undistorted; d_kp_uright (may
 * be NULL, needs d_kp_depth) receives x_un - bf / d where d_kp_depth > 0, else -1.  k1 == 0: kps_un = kps, as the reference.  Rows past
 * the count are not written. */
int hvo_orb_undistort_batch_device(hvo_orb* h, const hvo_camera* cam, const hvo_keypoint* d_kps, const int32_t* d_counts, int nframes,
                                   const float* d_kp_depth, float bf, hvo_keypoint* d_kps_un, float* d_kp_uright);

/* Create an extractor for frames of width x height, up to max_batch frames per call, on CUDA `device`. */
int hvo_orb_create(const hvo_orb_params* params, int width, int height, int max_batch, int device, hvo_orb** out);
void hvo_orb_destroy(hvo_orb* h);

/* Upper bound on keypoints per frame (rows of the caller's kps / desc buffers per frame). */
int hvo_orb_capacity(const hvo_orb* h);

/* Getters of ORBextractor.h:63-83.  Each array has nlevels entries. */
int hvo_orb_get_tables(const hvo_orb* h, float* scale_factors, float* inv_scale_factors, float* level_sigma2,
                       float* inv_level_sigma2, int32_t* features_per_level);

/* ORBextractor::operator()(image, mask, keypoints, descriptors)  ORBextractor.h:59-61, .cc:1041-1103.
 * gray: host, 8-bit, `stride` bytes per row.  kps/desc: host, `capacity` rows (desc rows are 32 bytes).
 * Empty image (null / zero size) returns HVO_OK with *n_out = 0, as the reference does (.cc:1044-1045). */
int hvo_orb_extract(hvo_orb* h, const uint8_t* gray, size_t stride, hvo_keypoint* kps, uint8_t* desc, int capacity,
                    int* n_out);

/* Batched variant for offline sequences: nframes tightly packed [n][height][width] host frames; outputs are
 * [n][capacity] rows; counts[n].  depth16 (optional, [n][height][width] uint16) enables the RGB-D epilogue:
 * kp_depth / kp_uright are [n][capacity] floats (-1 where depth is invalid). */
int hvo_orb_extract_batch(hvo_orb* h, const uint8_t* gray, int nframes, hvo_keypoint* kps, uint8_t* desc,
                          int32_t* counts, const uint16_t* depth16, const hvo_rgbd_params* rgbd, float* kp_depth,
                          float* kp_uright);

/* Same, all pointers in device memory on the handle's device; asynchronous on the handle's stream. */
int hvo_orb_extract_batch_device(hvo_orb* h, const uint8_t* d_gray, int nframes, hvo_keypoint* d_kps, uint8_t* d_desc,
                                 int32_t* d_counts, const uint16_t* d_depth16, const hvo_rgbd_params* rgbd,
                                 float* d_kp_depth, float* d_kp_uright);
int hvo_orb_sync(hvo_orb* h);

/* Stream timing for benchmarks: records CUDA events on the handle's stream. */
int hvo_orb_timer_start(hvo_orb* h);
int hvo_orb_timer_stop(hvo_orb* h, float* ms_out); /* synchronises */
/* Per-stage device time of the last *_batch call made with profiling enabled (ms): pyramid, fast, octree,
 * blur, describe.  Enabling inserts events between stages; leave off for throughput runs. */
int hvo_orb_set_profiling(hvo_orb* h, int enable);
int hvo_orb_stage_times(hvo_orb* h, float* ms5);
/* Number of kernel launches issued by the last extract call. */
int hvo_orb_last_launches(const hvo_orb* h);

/* ORBextractor::mvImagePyramid (ORBextractor.h:85): copy level `level` of frame `frame` of the last call. */
int hvo_orb_level_size(const hvo_orb* h, int level, int* w, int* h_out);
int hvo_orb_get_pyramid_level(hvo_orb* h, int frame, int level, uint8_t* out, size_t out_stride);

/* Inspection of intermediates (tests): pre-quadtree FAST candidates of a level, unordered;
 * xys = [cap][3] int32 (x, y in level coordinates, score). */
int hvo_orb_get_candidates(hvo_orb* h, int frame, int level, int32_t* xys, int cap, int* n_out);

/* ---------------------------------------------------------------------------------------------- MATCH
 * Brute-force Hamming matching of 256-bit descriptors (rows of 32 bytes, ORB and LBD alike).          */

typedef struct hvo_matcher hvo_matcher;
int hvo_matcher_create(int device, hvo_matcher** out);
void hvo_matcher_destroy(hvo_matcher* m);

/* int ORBmatcher::DescriptorDistance(const cv::Mat&, const cv::Mat&)   src/ORBmatcher.cc:1676-1692
 * int LSDmatcher::DescriptorDistance(const Mat&, const Mat&)           src/LSDmatcher.cpp:1137-1153
 * (host helper: one pair is not worth a launch; the kernels below use the same 8 x popc32) */
int hvo_hamming_distance(const uint8_t* a, const uint8_t* b);

/* cv::BFMatcher(NORM_HAMMING, false).knnMatch(desc1, desc2, matches, 2) as used by LSDmatcher::matchNNR
 * (src/LSDmatcher.cpp:811-812) and FrameBFMatch (:948-949).  For query i: idx2[2i], idx2[2i+1] are the train
 * indices of the nearest and second nearest descriptor (ties: lower train index first), dist2 the integer
 * Hamming distances (cv::DMatch::distance is this integer as a float); -1 where the train set is too small.
 * q, t: host arrays of nq / nt rows of 32 bytes. */
int hvo_match_knn2(hvo_matcher* m, const uint8_t* q, int nq, const uint8_t* t, int nt, int32_t* idx2, int32_t* dist2);
/* Same with 16-byte aligned device pointers; asynchronous on the matcher's stream. */
int hvo_match_knn2_device(hvo_matcher* m, const uint8_t* d_q, int nq, const uint8_t* d_t, int nt, int32_t* d_idx2,
                          int32_t* d_dist2);
/* MapPoint::ComputeDistinctiveDescriptors (src/MapPoint.cc:240-300) and MapLine::ComputeDistinctiveDescriptors
 * (src/MapLine.cpp:331-400) for a batch of map elements: group g = the descriptors desc[offsets[g] .. offsets[g+1]) of its
 * observations (in the reference's std::map iteration order); best_idx[g] = index inside the group of the descriptor with the
 * least median distance to the others (median = sorted[int(0.5 * (N - 1))], first minimum wins), -1 for an empty group;
 * best_median (may be NULL) = that median. */
int hvo_match_distinctive(hvo_matcher* m, const uint8_t* desc, const int32_t* offsets, int ngroups, int32_t* best_idx, int32_t* best_median);
int hvo_matcher_sync(hvo_matcher* m);
int hvo_matcher_timer_start(hvo_matcher* m);
int hvo_matcher_timer_stop(hvo_matcher* m, float* ms_out);

/* ------------------------------------------------------------------------------------------------ BOW
 * Replaces Frame::ComputeBoW (src/Frame.cc:1692-1699) = DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB>::transform(features, BowVector&,
 * FeatureVector&, levelsup) (Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1137-1206, :1228-1270) for ORB-SLAM2's vocabulary type (TF-IDF
 * weights, L1 scoring), for a batch of frames.  The vocabulary tree is handed over as arrays (what ORBVocabulary::loadFromTextFile /
 * the YAML loader fill into m_nodes): node 0 is the root; node i has the children child_ids[child_start[i] .. child_start[i+1]) in the
 * reference's order (empty = leaf = word), a 32-byte descriptor, a weight and a word id (-1 for inner nodes).                          */
typedef struct hvo_bow hvo_bow;
int hvo_bow_create(int device, hvo_bow** out);
void hvo_bow_destroy(hvo_bow* h);
int hvo_bow_set_vocabulary(hvo_bow* h, int n_nodes, const int32_t* child_start, const int32_t* child_ids, const uint8_t* node_desc,
                           const double* node_weight, const int32_t* node_word, int depth_levels /* m_L */);
/* desc: the frames' descriptors concatenated (frame f = rows offsets[f] .. offsets[f+1], at most 4096 per frame).  Per feature (may be
 * NULL): word_of = word id, or -1 when the word is stopped (weight <= 0); node_of = the node passed at level m_L - levelsup (0 = root
 * when that level is <= 0 or the leaf is reached earlier, where the reference leaves the value undefined).  Per frame: the BowVector as
 * bow_counts[f] (word, value) pairs at bow_words / bow_values [offsets[f] ..], ascending word id, L1-normalised, bit-identical to the
 * reference's std::map; the FeatureVector as fv_order [offsets[f] .. + fv_counts[f]) = feature indices (inside the frame) sorted by
 * (node_of, feature): consecutive runs of equal node_of are the map's vectors. */
int hvo_bow_transform(hvo_bow* h, const uint8_t* desc, const int32_t* offsets, int nframes, int levelsup, int32_t* word_of, int32_t* node_of,
                      int32_t* bow_counts, int32_t* bow_words, double* bow_values, int32_t* fv_order, int32_t* fv_counts);
int hvo_bow_last_launches(const hvo_bow* h);

/* ------------------------------------------------------------------------------------------- PROJECTION
 * Windowed matching against one frame: the frame grid (Frame::AssignFeaturesToGrid / PosInGrid, src/Frame.cc:832-847,
 * 1680-1690), Frame::GetFeaturesInArea (src/Frame.cc:1502-1555) and the greedy best / second-best search of
 * ORBmatcher::SearchByProjection(Frame&, const vector<MapPoint*>&, th) (src/ORBmatcher.cc:45-132, mode 0) and of
 * SearchByProjection(CurrentFrame, LastFrame, th, mono) / (CurrentFrame, KF, found, th, ORBdist) (src/ORBmatcher.cc:1353-1497,
 * 1499-1628, mode 1).  The caller keeps the projection (isInFrustum, pose) and the MapPoint bookkeeping: a query is the
 * projected position, the search radius r (already multiplied by the level's scale factor), the level range handed to
 * GetFeaturesInArea, the predicted right coordinate, and whether the map point it carries has observations (so that the
 * keypoint it takes is skipped by later queries, ORBmatcher.cc:88-90).  match_idx[i] is the keypoint query i is assigned
 * to, or -1; applying `F.mvpMapPoints[match_idx[i]] = pMP_i` for i ascending reproduces the reference's final state. */
typedef struct hvo_proj_query {
    float u, v, r;                 /* window centre and half-size */
    int32_t min_level, max_level;  /* GetFeaturesInArea(minLevel, maxLevel); -1 = open */
    float ur;                      /* predicted right coordinate (checked against mvuRight > 0 with tolerance r) */
    int32_t claims;                /* != 0: the assigned keypoint counts as taken for later queries */
    int32_t reserved;
} hvo_proj_query;

typedef struct hvo_proj hvo_proj;
int hvo_proj_create(int device, hvo_proj** out);
void hvo_proj_destroy(hvo_proj* h);
/* mvKeysUn, mvuRight (or NULL), mDescriptors of the frame searched in; image bounds mnMinX.. (src/Frame.cc:1733-1760).
 * Uploads them and builds the 64 x 48 grid on the device. */
int hvo_proj_set_frame(hvo_proj* h, const hvo_keypoint* keys_un, const float* uright, const uint8_t* desc, int n, float min_x, float min_y,
                       float max_x, float max_y);
/* KeyFrame::GetFeaturesInArea (src/KeyFrame.cc:627-666) searches the grid it copied from its Frame (cells assigned with the
 * frame's float bounds, same mfGridElement*Inv) but computes the cell range of a window from its own INTEGER mnMinX / mnMinY
 * (include/KeyFrame.h:249-252: the float bounds truncated), which differs from the Frame's for distorted cameras.  After
 * hvo_proj_set_frame, this call makes every window lookup of the handle (hvo_proj_search, hvo_proj_features_in_area) use
 * (min_x, min_y) as origin, the cells unchanged; the next hvo_proj_set_frame resets it.
 * (The candidate LISTS cannot differ: cells are assigned by round(), cell ranges by floor() / ceil(), so a shift of the origin by less
 * than half a cell only adds or drops cells that hold no keypoint within r.  The call exists so that the lookup is literally the
 * reference's; KeyFrame::IsInImage with the truncated bounds, which does change results, stays on the host.) */
int hvo_proj_set_window_origin(hvo_proj* h, float min_x, float min_y);
/* inspection: cell_start [64*48 + 1] (cell = ix * 48 + iy), cell_items [n] = mGrid[ix][iy] concatenated */
int hvo_proj_get_grid(hvo_proj* h, int32_t* cell_start, int32_t* cell_items);
/* Frame::GetFeaturesInArea(x, y, r, minLevel, maxLevel): indices in the reference's order; *n_out may exceed capacity */
int hvo_proj_features_in_area(hvo_proj* h, float x, float y, float r, int min_level, int max_level, int32_t* out, int capacity, int* n_out);
/* claimed [n] or NULL: keypoints that hold a map point with observations at call time.  mode 0: accept best <= th_dist unless
 * (bestLevel == bestLevel2 && best > nnratio * second); mode 1: accept best <= th_dist.  match_dist may be NULL.
 * mode 2 = the candidate loop of ORBmatcher::Fuse(KeyFrame*, vpMapPoints, th) (src/ORBmatcher.cc:838-990): candidates of the
 * window at levels [min_level, max_level] whose reprojection error passes e2 * mvInvLevelSigma2[level] <= 5.99 (7.8 with a right
 * coordinate, error then includes ur), best only, accept best <= th_dist (TH_LOW); queries are independent (nothing is claimed,
 * claimed must be NULL); needs hvo_proj_set_level_sigma.  Replace / AddObservation stay with the caller. */
int hvo_proj_search(hvo_proj* h, const hvo_proj_query* queries, const uint8_t* qdesc, int nq, const uint8_t* claimed, int mode, int th_dist,
                    float nnratio, int32_t* match_idx, int32_t* match_dist, int* n_matches);
int hvo_proj_set_level_sigma(hvo_proj* h, const float* inv_level_sigma2, int nlevels); /* mvInvLevelSigma2 of the frame searched in */
int hvo_proj_last_rounds(const hvo_proj* h);   /* fixed-point rounds of the last search (>= 1) */
int hvo_proj_last_launches(const hvo_proj* h);
/* Candidate lists chosen by the caller (e.g. the per-node buckets of SearchByBoW, src/ORBmatcher.cc:162-293): for query i the
 * train rows cand[offsets[i] .. offsets[i+1]) in that order; best4[i] = {idx0, dist0, idx1, dist1} with the reference's
 * strict '<' updates (-1 / 256 where absent).  Invalidates the frame set by hvo_proj_set_frame. */
int hvo_proj_match_candidates(hvo_proj* h, const uint8_t* q, int nq, const uint8_t* t, int nt, const int32_t* offsets, const int32_t* cand,
                              int32_t* best4);
/* The greedy loop of ORBmatcher::SearchByBoW(KeyFrame*, Frame&, ...) (src/ORBmatcher.cc:180-251) over the same kind of lists:
 * queries = the key frame's features that hold a good map point, in the reference's visiting order (vocabulary node
 * ascending, then the node's index list); cand lists = the frame's features of the same node.  Query i skips train rows
 * taken by an earlier query of this call, and takes its best when best <= th_dist and (float)best < nnratio * (float)second.
 * match_idx[i] = frame feature or -1.  Invalidates the frame set by hvo_proj_set_frame. */
int hvo_proj_search_candidates(hvo_proj* h, const uint8_t* q, int nq, const uint8_t* t, int nt, const int32_t* offsets, const int32_t* cand,
                               int th_dist, float nnratio, int32_t* match_idx, int32_t* match_dist, int* n_matches);
/* The candidate loop of ORBmatcher::SearchForTriangulation(pKF1, pKF2, F12, vMatchedPairs, bOnlyStereo) (src/ORBmatcher.cc:668-836)
 * with CheckDistEpipolarLine (:143-160).  Queries = features of pKF1 without a map point, in (vocabulary node, index list) order, with
 * their undistorted keypoints and stereo flags; cand lists = features of pKF2 in the same node.  tflags[i]: bit 0 = pKF2 feature i
 * holds a map point, bit 1 = it has a right coordinate.  F12 row-major 3x3, (ex, ey) = epipole in pKF2, scale_factors / level_sigma2 of
 * pKF2.  match_idx[i] = pKF2 feature or -1 (the last candidate of minimum distance <= th_low that passes the gates).  The rotation
 * histogram and vMatchedPairs stay with the caller.  Invalidates the frame set by hvo_proj_set_frame. */
int hvo_proj_search_triangulation(hvo_proj* h, const uint8_t* qdesc, const hvo_keypoint* qkeys, const uint8_t* qstereo, int nq, const uint8_t* tdesc,
                                  const hvo_keypoint* tkeys, const uint8_t* tflags, int nt, const int32_t* offsets, const int32_t* cand,
                                  const float* F12, float ex, float ey, const float* scale_factors, const float* level_sigma2, int nlevels,
                                  int only_stereo, int th_low, int32_t* match_idx, int32_t* match_dist, int* n_matches);
/* ---- tracking-time projection: Frame::isInFrustum(MapPoint*, float) (src/Frame.cc:1371-1436) for a batch of map points, and the
 * whole of Tracking::SearchLocalPoints' device work (src/Tracking.cc:3251-3268): isInFrustum over the local map followed by
 * ORBmatcher::SearchByProjection(F, vpMapPoints, th) in one call, the queries never leaving the device.
 * Arithmetic is the reference's: mRcw * P + mtcw as cv::gemm evaluates it for CV_32F (float products and sums in k order, then
 * (float)(double(t) + double(c))), cv::norm / Mat::dot with double accumulation, every other operation in float.  MapPoint::PredictScale
 * (src/MapPoint.cc:400-415) = ceil(logf(maxDistance / dist) / mfLogScaleFactor) clamped to [0, nlevels): the level is found by comparing the
 * ratio with thresholds the HOST derives from its own logf by bisection over float bit patterns (hvo_predict_scale_thresholds), so the
 * level is the one the reference's libm yields, bit for bit, without a device logarithm. */
typedef struct hvo_frustum_cam {
    float Rcw[9];                      /* mRcw, row-major */
    float tcw[3];                      /* mtcw */
    float Ow[3];                       /* mOw */
    float fx, fy, cx, cy, bf;          /* Frame::fx, fy, cx, cy, mbf */
    float min_x, min_y, max_x, max_y;  /* mnMinX, mnMinY, mnMaxX, mnMaxY */
    float log_scale_factor;            /* mfLogScaleFactor */
    int32_t n_levels;                  /* mnScaleLevels */
} hvo_frustum_cam;
typedef struct hvo_map_point {
    float pos[3];     /* MapPoint::GetWorldPos() */
    float normal[3];  /* GetNormal() */
    float min_distance, max_distance; /* mfMinDistance, mfMaxDistance: the range test uses 0.8f * min and 1.2f * max
                                         (Get{Min,Max}DistanceInvariance, src/MapPoint.cc:371-381), PredictScale mfMaxDistance itself */
} hvo_map_point;
typedef struct hvo_track_point { /* what isInFrustum leaves in the MapPoint (mTrackProjX, mTrackProjY, mTrackProjXR, mnTrackScaleLevel, mTrackViewCos, mbTrackInView) */
    float u, v, ur;
    int32_t level;
    float view_cos;
    int32_t in_view;
} hvo_track_point;
/* thresholds[k], k in [0, n): the smallest float ratio with ceil(logf(ratio) / log_scale_factor) > k + lo, i.e.
 * level(ratio) = lo + #{k : ratio >= thresholds[k]} for levels in [lo, lo + n].  Host function (uses the C library's logf). */
int hvo_predict_scale_thresholds(float log_scale_factor, int lo, int n, float* thresholds);
/* out[i] for every map point; fields other than in_view are only meaningful where in_view != 0 */
int hvo_proj_frustum_points(hvo_proj* h, const hvo_frustum_cam* cam, const hvo_map_point* pts, int n, float viewing_cos_limit, hvo_track_point* out);
/* skip[i] != 0: the map point is not projected (mnLastFrameSeen == frame id, or isBad()); claims[i] != 0: it has observations.
 * pdesc [n][32] = MapPoint::GetDescriptor().  scale_factors = F.mvScaleFactors.  track (may be NULL) receives the isInFrustum
 * result; match_idx[i] = keypoint of the frame set by hvo_proj_set_frame that map point i is assigned to, or -1.  claimed as for
 * hvo_proj_search. */
int hvo_proj_search_local_map(hvo_proj* h, const hvo_frustum_cam* cam, const hvo_map_point* pts, const uint8_t* pdesc, const uint8_t* skip,
                              const uint8_t* claims, int n, float viewing_cos_limit, float th, const float* scale_factors, const uint8_t* claimed,
                              int th_dist, float nnratio, hvo_track_point* track, int32_t* match_idx, int32_t* match_dist, int* n_in_view,
                              int* n_matches);
/* ORBmatcher::SearchForInitialization(F1, F2, vbPrevMatched, vnMatches12, windowSize) (src/ORBmatcher.cc:412-497): the sequential
 * loop with its vMatchedDistance / vnMatches21 state, for the frame set by hvo_proj_set_frame as F2.  Queries = the level-0
 * keypoints of F1 in index order: window centre prev_matched[i] (x, y), F1's descriptors.  octave1[i] != 0 skips the keypoint.
 * matches12[i] = F2 keypoint or -1 BEFORE the rotation-histogram culling (:499-523, host); *n_matches likewise.  accepted12[i] = the
 * F2 keypoint query i took when it was visited (-1 if none), whether or not a later query took it over: the entries the reference
 * pushes into rotHist. */
int hvo_proj_search_initialization(hvo_proj* h, const float* prev_matched_xy, const int32_t* octave1, const uint8_t* desc1, int n1, int window_size,
                                   int th_dist, float nnratio, int32_t* matches12, int32_t* accepted12, int* n_matches);
int hvo_proj_timer_start(hvo_proj* h);
int hvo_proj_timer_stop(hvo_proj* h, float* ms_out);

/* ------------------------------------------------------------------------------------------------ LBD
 * Replaces cv::line_descriptor::BinaryDescriptor::compute(image, keylines, descriptors) as called at
 * src/LineExtractor.cpp:361-363 and src/Frame.cc:1094-1096 (vendored algorithm:
 * Thirdparty/line_descriptor/src/binary_descriptor_custom.cpp:539-687, 1026-1372).  Single octave
 * (LINE.nLevels = 1 in every shipped YAML); keylines must carry octave 0 and distinct class_id, as
 * LINEextractor::operator() and Frame::cullingLine produce them.                                       */

/* cv::line_descriptor::KeyLine POD layout (68 bytes), descriptor_custom.hpp:105-144 */
typedef struct hvo_keyline {
    float angle;
    int32_t class_id, octave;
    float pt_x, pt_y, response, size;
    float startPointX, startPointY, endPointX, endPointY;
    float sPointInOctaveX, sPointInOctaveY, ePointInOctaveX, ePointInOctaveY;
    float lineLength;
    int32_t numOfPixels;
} hvo_keyline;

typedef struct hvo_lbd hvo_lbd;
int hvo_lbd_create(int width, int height, int max_batch, int max_lines, int device, hvo_lbd** out);
void hvo_lbd_destroy(hvo_lbd* h);
/* One image: desc = n x 32 bytes.  n == 0 mirrors the reference's "keypoint list is empty" early return. */
int hvo_lbd_compute(hvo_lbd* h, const uint8_t* gray, size_t stride, const hvo_keyline* keylines, int n, uint8_t* desc);
/* Batch: gray [n][H][W], keylines [n][max_lines], counts [n], desc [n][max_lines][32]; fdesc (optional)
 * [n][max_lines][72] = the normalised float LBD before binarisation. */
int hvo_lbd_compute_batch(hvo_lbd* h, const uint8_t* gray, int nframes, const hvo_keyline* keylines, const int32_t* counts,
                          uint8_t* desc, float* fdesc);
int hvo_lbd_compute_batch_device(hvo_lbd* h, const uint8_t* d_gray, int nframes, const hvo_keyline* d_keylines,
                                 const int32_t* d_counts, uint8_t* d_desc);
/* dxImg / dyImg of BinaryDescriptor::computeSobel (:377-398) for a frame of the last call: H x W int16 each */
int hvo_lbd_get_gradients(hvo_lbd* h, int frame, int16_t* dx, int16_t* dy);
int hvo_lbd_sync(hvo_lbd* h);
int hvo_lbd_timer_start(hvo_lbd* h);
int hvo_lbd_timer_stop(hvo_lbd* h, float* ms_out);

/* ----------------------------------------------------------------------------------------------- LINE
 * Replaces ORB_SLAM2::LINEextractor (include/LineExtractor.h:187-262, src/LineExtractor.cpp:329-380):
 * line_descriptor::LSDDetector::detect (Thirdparty/line_descriptor/src/LSDDetector_custom.cpp:105-215; segments from
 * cv::createLineSegmentDetector()->detect with OpenCV's default parameters) -> response sort + truncation to
 * nLSDFeature -> LBD descriptors -> 2-D line functions.  Single octave (LINE.nLevels = 1 in every shipped YAML; the
 * float `scale` narrows to int 1 at the reference's call, LineExtractor.cpp:342).                              */

/* LINEextractor::LINEextractor(int numOctaves, float scale, unsigned nLSDFeature, double min_line_length)  LineExtractor.h:190 */
typedef struct hvo_line_params {
    int n_octaves;          /* must be 1 */
    float scale;            /* unused by the reference's single-octave path; kept for the getters */
    int n_features;         /* nLSDFeature: keep the n_features strongest responses */
    double min_line_length; /* stored only (the reference's operator() does not use it) */
} hvo_line_params;

typedef struct hvo_line hvo_line;
int hvo_line_create(const hvo_line_params* p, int width, int height, int max_batch, int device, hvo_line** out);
void hvo_line_destroy(hvo_line* h);
/* Frame::cullingLine(imGray, 5, 2.5, 15, 30) (src/Frame.cc:939, :952-1116), which Frame::ExtractLSD runs on the extractor's
 * output: merge near-collinear KeyLines (MergeTwoLines :1141-1203), rebuild the KeyLines, sort by response, LBD again
 * (:1094-1096), line functions again (:1097-1108).  enable != 0: every hvo_line_extract* call returns the culled set (the state
 * of mvKeylinesUn / mLdesc / mvKeyLineFunctions after ExtractLSD's cullingLine). */
int hvo_line_set_culling(hvo_line* h, int enable);
/* cullingLine alone, in place: keylines / linevec3 hold n rows on entry and *n_out rows on return; desc receives *n_out x 32. */
int hvo_line_cull(hvo_line* h, const uint8_t* gray, size_t stride, hvo_keyline* keylines, double* linevec3, int n, uint8_t* desc,
                  int* n_out);
/* device-resident, batched: d_keylines [n][max_lines], d_linevec3 [n][max_lines][3], d_counts [n] are read and overwritten */
int hvo_line_cull_batch_device(hvo_line* h, const uint8_t* d_gray, int nframes, hvo_keyline* d_keylines, uint8_t* d_desc,
                               double* d_linevec3, int32_t* d_counts);
int hvo_line_max_lines(const hvo_line* h);        /* rows per frame of keylines / desc / linevec3 = n_features */
int hvo_line_segment_capacity(const hvo_line* h); /* upper bound of raw LSD segments per frame */
int hvo_line_scaled_size(const hvo_line* h, int* sw, int* sh);

/* LINEextractor::operator()(image, mask, keylines, descriptors, lineVec2d)  LineExtractor.h:193 (mask: the reference
 * always passes an empty mask, Frame.cc:902).  gray: host 8-bit; keylines/desc: `capacity` >= hvo_line_max_lines()
 * rows; linevec3 (optional): rows of 3 doubles.  gray == NULL mirrors the empty-image early return. */
int hvo_line_extract(hvo_line* h, const uint8_t* gray, size_t stride, hvo_keyline* keylines, uint8_t* desc, double* linevec3,
                     int capacity, int* n_out);
/* Batch: gray [n][H][W]; keylines [n][max_lines]; desc [n][max_lines][32]; linevec3 [n][max_lines][3]; counts [n]. */
int hvo_line_extract_batch(hvo_line* h, const uint8_t* gray, int nframes, hvo_keyline* keylines, uint8_t* desc, double* linevec3,
                           int32_t* counts);
int hvo_line_extract_batch_device(hvo_line* h, const uint8_t* d_gray, int nframes, hvo_keyline* d_keylines, uint8_t* d_desc,
                                  double* d_linevec3, int32_t* d_counts);
/* cv::LineSegmentDetector::detect alone: segments4 [n][seg_capacity][4] floats (x1,y1,x2,y2), counts [n] (a count may
 * exceed seg_capacity; only the first seg_capacity segments of that frame are written). */
int hvo_line_detect_batch(hvo_line* h, const uint8_t* gray, int nframes, float* segments4, int seg_capacity, int32_t* counts);
/* Inspection (tests): the blurred + 0.8-resized image LSD works on, and the seed order (pixel indices y*sw+x). */
int hvo_line_get_scaled(hvo_line* h, int frame, uint8_t* out);
int hvo_line_get_seed_order(hvo_line* h, int frame, uint32_t* out, int cap, int* n_out);
int hvo_line_set_profiling(hvo_line* h, int enable);
int hvo_line_stage_times(hvo_line* h, float* ms4); /* prep, order, grow, keylines+LBD of the last extract call */
int hvo_line_last_launches(const hvo_line* h);
int hvo_line_sync(hvo_line* h);
int hvo_line_timer_start(hvo_line* h);
int hvo_line_timer_stop(hvo_line* h, float* ms_out);

/* ---------------------------------------------------------------------------------------------- PLANE
 * Replaces PlaneDetection::readDepthImage(depth16U, K, factor) + runPlaneDetection(H, W)
 * (src/PlaneExtractor.cpp:26-66, include/PlaneExtractor.h:36-56) and the ahc::PlaneFitter behind them
 * (include/peac/).  Results correspond to plane_num_, plane_filter.extractedPlanes[i]->normal/center and the
 * pixel membership from which plane_vertices_ is listed (ascending pixel index per plane).                */

typedef struct hvo_plane_params {
    float fx, fy, cx, cy; /* K as read by readDepthImage (K.at<float>) */
    float depth_factor;   /* kScaleFactor = 1 / DepthMapFactor */
} hvo_plane_params;

typedef struct hvo_plane hvo_plane;
/* images of up to 24576 10x10 blocks (1920x1200); larger ones are refused with HVO_ERR_ARG */
int hvo_plane_create(const hvo_plane_params* p, int width, int height, int max_batch, int device, hvo_plane** out);
void hvo_plane_destroy(hvo_plane* h);
/* depth16: host [H][W] uint16.  planes7: [max_planes][7] doubles = normal(3), center(3), N.  membership: [H*W]
 * int32 = plane id or -1.  *n_planes may exceed max_planes (only the first max_planes are written). */
int hvo_plane_detect(hvo_plane* h, const uint16_t* depth16, int32_t* n_planes, double* planes7, int max_planes,
                     int32_t* membership);
int hvo_plane_detect_batch(hvo_plane* h, const uint16_t* depth16, int nframes, int32_t* n_planes, double* planes7,
                           int max_planes, int32_t* membership);
/* Same with every pointer in device memory; asynchronous on the handle's stream.  d_planes7 is [n][max_planes][7];
 * d_membership doubles as the working membership image. */
int hvo_plane_detect_batch_device(hvo_plane* h, const uint16_t* d_depth16, int nframes, int32_t* d_n_planes, double* d_planes7,
                                  int max_planes, int32_t* d_membership);
/* Same, and also writes the final labels as one byte per pixel (plane id, 255 = no plane) into d_membership8 [n][H*W]:
 * the compact form the frame front-end copies back to the host. */
int hvo_plane_detect_batch_device_u8(hvo_plane* h, const uint16_t* d_depth16, int nframes, int32_t* d_n_planes, double* d_planes7,
                                     int max_planes, int32_t* d_membership, uint8_t* d_membership8);
int hvo_plane_last_launches(const hvo_plane* h);
/* Profiling: SM clock cycles of the graph kernel's phases for one frame of the last call: first clustering,
 * block erosion + seeds, flood fill, last merge + relabel. */
int hvo_plane_get_phase_cycles(hvo_plane* h, int frame, int64_t* out4);
/* First kernel only (initial graph nodes, AHCPlaneFitter.hpp:786-826 / AHCPlaneSeg.hpp:211-284) on device-resident
 * depth; asynchronous.  hvo_plane_get_blocks copies one frame's result: per 10x10 block 9 doubles =
 * {queued, N, center(3), normal(3), mse}. */
int hvo_plane_blocks_device(hvo_plane* h, const uint16_t* d_depth16, int nframes);
int hvo_plane_get_blocks(hvo_plane* h, int frame, double* out9);
int hvo_plane_sync(hvo_plane* h);
int hvo_plane_timer_start(hvo_plane* h);
int hvo_plane_timer_stop(hvo_plane* h, float* ms_out);

/* -------------------------------------------------------------------------------------------- NORMALS
 * Replaces the surface-normal block of Frame::ComputePlanes (src/Frame.cc:2155-2212): every 3rd pixel of the float
 * depth image -> organised cloud -> pcl::IntegralImageNormalEstimation (AVERAGE_3D_GRADIENT, MaxDepthChangeFactor
 * 0.05, NormalSmoothingSize 10) -> entries at odd (row, col) -> std::vector<SurfaceNormal> (include/SurfaceNormal.h).
 * One output entry = 8 floats: normal.xyz (NaN where PCL yields NaN), cameraPosition.xyz, FramePosition.x, .y.      */

typedef struct hvo_normals_params {
    float fx, fy, cx, cy;
    float depth_factor;            /* metres per raw depth unit */
    float max_depth_change_factor; /* ne.setMaxDepthChangeFactor(0.05f)  Frame.cc:2179 */
    float normal_smoothing_size;   /* ne.setNormalSmoothingSize(10.0f)   Frame.cc:2180 */
} hvo_normals_params;

typedef struct hvo_normals hvo_normals;
int hvo_normals_create(const hvo_normals_params* p, int width, int height, int max_batch, int device, hvo_normals** out);
void hvo_normals_destroy(hvo_normals* h);
int hvo_normals_count(const hvo_normals* h); /* entries per frame = (ceil(H/3)/2) * (ceil(W/3)/2) */
int hvo_normals_compute_batch(hvo_normals* h, const uint16_t* depth16, int nframes, float* out8);
int hvo_normals_compute_batch_device(hvo_normals* h, const uint16_t* d_depth16, int nframes, float* d_out8);
int hvo_normals_get_distance_map(hvo_normals* h, int frame, float* out); /* ceil(H/3) x ceil(W/3) floats */
int hvo_normals_sync(hvo_normals* h);
int hvo_normals_timer_start(hvo_normals* h);
int hvo_normals_timer_stop(hvo_normals* h, float* ms_out);

/* LSDmatcher::FrameBFMatchNew(ldesc1, ldesc2, LineMatches, kls1, kls2, kls2func, F, TH) (src/LSDmatcher.cpp:968-1031) with
 * mutualOverlap (:1033-1108): knn-2 of ldesc1 against ldesc2, then for the nearest neighbour only (the reference's inner loop runs
 * for j < size() - 1 = 1) the epipolar test: the query's end points are mapped through F (cv::gemm, CV_32F), intersected with the
 * train line (Mat::cross), and the overlap of the two collinear segments must exceed 0.8, with distance < TH and
 * distance < nnratio * second distance.  kls1 / kls2 = keylines of the two frames, kls2func [n2][3] doubles, F row-major 3x3 float.
 * line_matches[i] = train line or -1. */
int hvo_match_lines_epipolar(hvo_matcher* m, const uint8_t* ldesc1, const hvo_keyline* kls1, int n1, const uint8_t* ldesc2, const hvo_keyline* kls2,
                             const double* kls2func, int n2, const float* F, float th, float nnratio, int32_t* line_matches);

/* ---- windowed line matchers -------------------------------------------------------------------------------------
 * Replaces, for one frame at a time, Frame::AssignFeaturesToGridForLine (src/Frame.cc:849-872, src/lineIterator.cpp),
 * Frame::GetFeaturesInAreaForLine (src/Frame.cc:1557-1631) and the two greedy searches
 *   mode 0: LSDmatcher::SearchByProjection(Frame&, const vector<MapLine*>&, eval_orient, th)  (src/LSDmatcher.cpp:709-801)
 *   mode 1: LSDmatcher::SearchByProjection(CurrentFrame, LastFrame, th)                        (src/LSDmatcher.cpp:561-664)
 * Projection / isInFrustum / mbTrackInView / isBad stay with the caller: a query is the projected segment, the window
 * radius (RadiusByViewingCos * th, or th), the direction threshold of GetFeaturesInAreaForLine (0.998 default, 0.96 for
 * mode 1) and the data of the per-candidate gate.  match_idx[i] = frame line assigned to query i or -1; applying
 * `F.mvpMapLines[match_idx[i]] = pML_i` for i ascending reproduces the reference's final state. */
typedef struct hvo_lproj_query {
    float x1, y1, x2, y2;  /* mTrackProjX1, Y1, X2, Y2 */
    float r, cos_th;       /* window half-size; TH of GetFeaturesInAreaForLine */
    double dir[3];         /* mode 0: MapLine::GetWorldVector(); mode 1: last keyline's ePointInOctave - sPointInOctave (x, y, unused) */
    float length;          /* mode 1: lineLength of the last frame's keyline */
    int32_t claims;        /* != 0: the map line has observations, so the line it takes is skipped by later queries */
    int32_t reserved[2];
} hvo_lproj_query;

typedef struct hvo_lproj hvo_lproj;
int hvo_lproj_create(int device, hvo_lproj** out);
void hvo_lproj_destroy(hvo_lproj* h);
/* mvKeylinesUn, mvKeyLineFunctions [n][3], mLdesc [n][32], mvLines3D [n][6] = first.xyz, second.xyz (NULL when only mode 1 is
 * used) of the frame searched in (n <= 1024); image bounds mnMinX.. .  Builds the 64 x 48 line grid on the device. */
int hvo_lproj_set_frame(hvo_lproj* h, const hvo_keyline* keylines_un, const double* line_functions, const uint8_t* desc, const double* lines3d,
                        int n, float min_x, float min_y, float max_x, float max_y);
/* inspection: cell_count [64*48] (cell = ix * 48 + iy); cell_items (may be NULL) = mGridForLine[ix][iy] concatenated */
int hvo_lproj_get_grid(hvo_lproj* h, int32_t* cell_count, int32_t* cell_items, int capacity, int* n_items);
/* Frame::GetFeaturesInAreaForLine(x1, y1, x2, y2, r, -, -, TH): indices in the reference's order; *n_out may exceed capacity */
int hvo_lproj_features_in_area(hvo_lproj* h, float x1, float y1, float x2, float y2, float r, float cos_th, int32_t* out, int capacity,
                               int* n_out);
/* claimed [n] or NULL: lines that hold a map line with observations at call time.  Accept best <= 95; mode 0 also applies
 * the same-octave ratio test with nnratio (mfNNratio).  match_dist may be NULL. */
int hvo_lproj_search(hvo_lproj* h, const hvo_lproj_query* queries, const uint8_t* qdesc, int nq, const uint8_t* claimed, int mode, float nnratio,
                     int32_t* match_idx, int32_t* match_dist, int* n_matches);
/* Frame::isInFrustum(MapLine*, float) (src/Frame.cc:1438-1499) for a batch of map lines, and Tracking::SearchLocalLines' device work
 * (src/Tracking.cc:3315-3348): isInFrustum followed by LSDmatcher::SearchByProjection(F, vpMapLines, eval_orient, th) in one call.
 * The end points are narrowed to float as the reference does (Mat_<float> << P(0) ...); the mid point is
 * cv::addWeighted(SP, 0.5, EP, 0.5) - mOw; MapLine::PredictScale (src/MapLine.cpp:549-558) is NOT clamped. */
typedef struct hvo_map_line {
    double pos[6];     /* MapLine::GetWorldPos(): start xyz, end xyz */
    double normal[3];  /* GetNormal() */
    double dir[3];     /* GetWorldVector() (used by the search only) */
    float min_distance, max_distance; /* mfMinDistance, mfMaxDistance (src/MapLine.cpp:537-558), as for hvo_map_point */
} hvo_map_line;
typedef struct hvo_track_line {
    float x1, y1, x2, y2; /* mTrackProjX1, Y1, X2, Y2 */
    int32_t level;        /* mnTrackScaleLevel */
    float view_cos;
    int32_t in_view;
} hvo_track_line;
int hvo_lproj_frustum_lines(hvo_lproj* h, const hvo_frustum_cam* cam, const hvo_map_line* lines, int n, float viewing_cos_limit, hvo_track_line* out);
int hvo_lproj_search_local_map(hvo_lproj* h, const hvo_frustum_cam* cam, const hvo_map_line* lines, const uint8_t* ldesc, const uint8_t* skip,
                               const uint8_t* claims, int n, float viewing_cos_limit, float th, const uint8_t* claimed, float nnratio,
                               hvo_track_line* track, int32_t* match_idx, int32_t* match_dist, int* n_in_view, int* n_matches);
int hvo_lproj_last_rounds(const hvo_lproj* h);
int hvo_lproj_last_launches(const hvo_lproj* h);

/* ---- LPVO normals -------------------------------------------------------------------------------------------
 * Replaces Manhattan::computeNormalsLPVO (src/Manhattan.cpp:237-393, intrinsics :12-18), which Frame::ExtractMainImgPtNormals
 * runs on every frame until the Manhattan axes are initialised (src/Frame.cc:218-228): tangent vectors by central
 * differences where 0.2 <= z <= 7, seven cv::integral images, 10x10 box means every 15 px from (10, 10), normal = v x u,
 * cv::normalize.  Outputs per frame, in the reference's push_back order: pt_normals (3 doubles each), depth_normals
 * (float) and the pixel (u, v) of each sample.  Input is the raw 16-bit depth; z = (float)raw * depth_factor (the
 * reference's live caller passes the 16-bit Mat where a float Mat is read: that bug is not reproduced).  Any image size in
 * 32..8192 px.  A frame handle returns the same rows from its own call (hvo_frame_lpvo_outputs). */
typedef struct hvo_lpvo hvo_lpvo;
int hvo_lpvo_create(const hvo_plane_params* cam, int width, int height, int max_batch, int device, hvo_lpvo** out);
void hvo_lpvo_destroy(hvo_lpvo* h);
int hvo_lpvo_capacity(const hvo_lpvo* h); /* lattice samples per frame = rows of every output array per frame */
/* normals3 [n][capacity][3] double, depth [n][capacity] float, pix2 [n][capacity][2] int32, counts [n] int32 */
int hvo_lpvo_compute_batch(hvo_lpvo* h, const uint16_t* depth16, int nframes, double* normals3, float* depth, int32_t* pix2,
                           int32_t* counts);
int hvo_lpvo_compute_batch_device(hvo_lpvo* h, const uint16_t* d_depth16, int nframes, double* d_normals3, float* d_depth,
                                  int32_t* d_pix2, int32_t* d_counts);
int hvo_lpvo_sync(hvo_lpvo* h);
int hvo_lpvo_timer_start(hvo_lpvo* h);
int hvo_lpvo_timer_stop(hvo_lpvo* h, float* ms_out);

/* ---------------------------------------------------------------------------------------------- FRAME
 * The extraction part of Frame::Frame(imGray, imDepth, timeStamp, extractors, ...) (src/Frame.cc:188-233): the reference
 * runs three std::threads on one frame — ExtractORBNDepth (:874-884), ExtractLSD (:895-903), ComputePlanes
 * (:2104-2212) — and, while the Manhattan axes are not initialised (!bManhInit, :218-228), a fourth, ExtractMainImgPtNormals
 * (Manhattan::computeNormalsLPVO, :1324-1328).  hvo_frame uploads the frame (gray + raw 16-bit depth) once and runs the same
 * pipelines on CUDA streams, for a batch of frames per call; the LPVO normals run, after the surface normals on the normals
 * stream, in the calls given hvo_frame_lpvo_outputs (*_lpvo).                                                 */

#define HVO_STAGE_ORB 1
#define HVO_STAGE_LINES 2
#define HVO_STAGE_PLANES 4
#define HVO_STAGE_NORMALS 8
#define HVO_STAGE_ALL 15

typedef struct hvo_frame_params {
    hvo_orb_params orb;   /* ORBextractor.* of the settings file */
    hvo_line_params line; /* LINE.* */
    float fx, fy, cx, cy; /* Camera.* */
    float depth_factor;   /* 1 / DepthMapFactor */
    float bf;             /* Camera.bf */
    int distorted;        /* != 0: Camera.k1 != 0 (see hvo_rgbd_params): with all coefficients below 0, kp_uright is filled with -1;
                             with a non-zero coefficient the handle undistorts on the device (kps_un, kp_uright) */
    int stages;           /* HVO_STAGE_* bits */
    int max_planes;       /* rows of planes7 per frame */
    int line_cull;        /* != 0: Frame::cullingLine after the line extractor, as Frame::ExtractLSD does (src/Frame.cc:939) */
    int lanes;            /* 0 = default (2 from max_batch 2048 on, else 1).  The handle splits a batch into chunks of max_batch / lanes
                             frames that go round-robin through `lanes` sets of input / output staging (upload stream, one download
                             stream per pipeline), so uploads, kernels and downloads of different chunks overlap.  The pipelines'
                             own scratch exists once (chunk-sized): the kernels of consecutive chunks run one after the other.
                             A chunk of >= 2048 frames runs its pipelines one after the other (planes, lines, ORB, normals), each
                             alone at its saturating batch; smaller chunks run them side by side (lowest latency). */
    float k1, k2, p1, p2, k3; /* Camera.k1 .. k3 (mDistCoef, see hvo_camera); all 0 = no undistortion on the device */
} hvo_frame_params;

/* Output arrays of a batch of n frames.  Host pointers for hvo_frame_extract_batch, device pointers for
 * hvo_frame_extract_batch_device.  Row counts per frame come from hvo_frame_capacities(). */
typedef struct hvo_frame_outputs {
    hvo_keypoint* kps;     /* [n][orb_capacity]      mvKeys                                       */
    uint8_t* desc;         /* [n][orb_capacity][32]  mDescriptors                                 */
    int32_t* kp_counts;    /* [n]                    N                                            */
    float* kp_depth;       /* [n][orb_capacity]      mvDepth  (-1 invalid)   optional on the host */
    float* kp_uright;      /* [n][orb_capacity]      mvuRight (-1 invalid)   optional on the host */
    hvo_keyline* keylines; /* [n][max_lines]         mvKeylinesUn                                 */
    uint8_t* line_desc;    /* [n][max_lines][32]     mLdesc                                       */
    double* linevec3;      /* [n][max_lines][3]      mvKeyLineFunctions      optional on the host */
    int32_t* line_counts;  /* [n]                    NL                                           */
    int32_t* n_planes;     /* [n]                    plane_num_                                   */
    double* planes7;       /* [n][max_planes][7]     normal, center, N of extractedPlanes         */
    int32_t* membership;   /* [n][H*W]               plane id per pixel or -1 (-> plane_vertices_); on the host
                                                     optional when membership8 is given           */
    float* normals8;       /* [n][normals_count][8]  std::vector<SurfaceNormal>                   */
    uint8_t* membership8;  /* [n][H*W]               the same labels in one byte (255 = none)     optional */
    /* Compact forms for host callers (what goes over PCIe: 256 KB instead of 581 KB per 640x480 frame).  Optional.         */
    uint8_t* membership4;  /* [n][H*W/2]             two pixels per byte (low nibble = even pixel), 15 = none; needs
                                                     max_planes <= 15 and an even H*W.  hvo_membership4_expand() restores labels */
    float* normals3;       /* [n][normals_count][3]  the normal only (NaN = none); position and pixel of a SurfaceNormal are
                                                     functions of (m, n) and the depth: hvo_normals3_expand() restores normals8 */
    hvo_keypoint* kps_un;  /* [n][orb_capacity]      mvKeysUn (Frame::UndistortKeyPoints)   optional; only for a handle created
                                                     with distorted != 0 and a non-zero coefficient                  */
} hvo_frame_outputs;

/* Bag-of-words vectors of a batch of n frames (Frame::ComputeBoW, src/Frame.cc:1692-1699: transform(mDescriptors rows, mBowVec, mFeatVec,
 * levelsup)), for a handle with a vocabulary (hvo_frame_set_vocabulary).  Frame f's rows are those of hvo_bow_transform on the frame's
 * descriptor rows [0, kp_counts[f]), bit for bit; rows at or past a frame's count are not written.  Host pointers for the host calls,
 * device pointers for hvo_frame_extract_batch_device_bow.                                                                          */
typedef struct hvo_frame_bow_outputs {
    int32_t* bow_counts;  /* [n]                    words in mBowVec                                                               */
    int32_t* bow_words;   /* [n][orb_capacity]      ascending word ids (first bow_counts[f] rows)                                  */
    double* bow_values;   /* [n][orb_capacity]      their L1-normalised values, bit-identical to DBoW2                              */
    int32_t* fv_order;    /* [n][orb_capacity]      feature indices sorted by (node_of, feature), first fv_counts[f] rows; runs of
                                                    equal node_of are mFeatVec's vectors             optional on the host (needs node_of) */
    int32_t* fv_counts;   /* [n]                    features not stopped                             optional on the host            */
    int32_t* node_of;     /* [n][orb_capacity]      node at level m_L - levelsup (mFeatVec keys; 0 = root)  optional on the host         */
    int32_t* word_of;     /* [n][orb_capacity]      word id, or -1 where the word is stopped          optional on the host            */
} hvo_frame_bow_outputs;

/* The frame grids of a batch of n frames (Frame::AssignFeaturesToGrid / AssignFeaturesToGridForLine, src/Frame.cc:832-872, run by
 * Frame::Frame right after the extraction): mGrid / mGridForLine [64][48] as per-cell counts plus the cells' indices concatenated in
 * cell order (cell = ix * 48 + iy), a cell's indices ascending (the reference's push_back order).  The point grid is built on mvKeysUn
 * (kps_un on an undistorting handle, else kps) with Frame::PosInGrid, the line grid on the keylines the call returns (after cullingLine
 * when line_cull is set) with the reference's LineIterator walk; both with the handle's image bounds (hvo_frame_image_bounds).
 * Either pair may be NULL; a pair needs its stage (HVO_STAGE_ORB / HVO_STAGE_LINES), otherwise HVO_ERR_ARG.  uint16 entries: a point
 * grid needs orb_capacity <= 65535.  Device pointers for hvo_frame_extract_batch_device_grid, which writes no item entry past a frame's
 * total; host pointers for the host calls, which copy whole rows (entries past the total then hold unspecified values).          */
typedef struct hvo_frame_grid_outputs {
    uint16_t* grid_counts;   /* [n][3072]                mGrid[ix][iy].size()                                                          */
    uint16_t* grid_items;    /* [n][orb_capacity]        keypoint indices, first sum(grid_counts[f]) entries                           */
    uint16_t* lgrid_counts;  /* [n][3072]                mGridForLine[ix][iy].size()                                                   */
    uint16_t* lgrid_items;   /* [n][line_grid_capacity]  line indices, first sum(lgrid_counts[f]) entries.  line_grid_capacity =
                                                         64 * max_lines is exact: LineIterator advances the major axis by one cell per
                                                         step, so a line visits at most 64 in-grid cells and none twice             */
} hvo_frame_grid_outputs;

/* Manhattan::computeNormalsLPVO of a batch of n frames (src/Frame.cc:218-228, run by Frame::Frame while !bManhInit), on the frame's raw
 * depth: the rows hvo_lpvo_compute_batch returns for the same depth, bit for bit.  Rows per frame: hvo_frame_lpvo_capacity() (=
 * hvo_lpvo_capacity for the same camera and image size); frame f's first counts[f] rows are valid, in the reference's push_back order.
 * Needs HVO_STAGE_NORMALS, otherwise HVO_ERR_ARG.  Host pointers for the host calls, which copy whole rows; device pointers for
 * hvo_frame_extract_batch_device_lpvo, which needs every array and writes no row at or past a frame's count.                  */
typedef struct hvo_frame_lpvo_outputs {
    double* normals3;  /* [n][lpvo_capacity][3]   pt_normals (unit normal v x u)                                                   */
    float* depth;      /* [n][lpvo_capacity]      depth_normals                                                                    */
    int32_t* pix2;     /* [n][lpvo_capacity][2]   the sample's pixel (u, v)                                 optional on the host    */
    int32_t* counts;   /* [n]                     samples of the frame                                                             */
} hvo_frame_lpvo_outputs;

/* Host-side expanders of the compact outputs (plain C loops, no CUDA). */
/* labels4 [H*W/2] -> labels [H*W] int32 (-1 = none) */
int hvo_membership4_expand(const uint8_t* labels4, int npixels, int32_t* labels);
/* normals3 [count][3] + the frame's raw depth -> normals8 [count][8] = normal, cameraPosition, FramePosition exactly as the device
 * writes them (src/Frame.cc:2158-2171, 2191-2196): row i <-> cloud cell m = 2 (i / (cw/2)) + 1, n = 2 (i % (cw/2)) + 1, cw = ceil(W/3) */
int hvo_normals3_expand(const float* normals3, const uint16_t* depth16, int width, int height, float fx, float fy, float cx, float cy,
                        float depth_factor, float* normals8);

typedef struct hvo_frame hvo_frame;
int hvo_frame_create(const hvo_frame_params* p, int width, int height, int max_batch, int device, hvo_frame** out);
void hvo_frame_destroy(hvo_frame* h);
int hvo_frame_capacities(const hvo_frame* h, int* orb_capacity, int* max_lines, int* normals_count);
int hvo_frame_lanes(const hvo_frame* h, int* lanes, int* chunk_frames);
/* gray [n][H][W] uint8 and depth16 [n][H][W] uint16 in host memory (pinned memory makes the copies asynchronous);
 * returns when every output has been written.  n is not limited by max_batch: chunks of max_batch / lanes frames are
 * streamed through the lanes (upload of chunk k+1 and download of chunk k-1 overlap the kernels of chunk k). */
int hvo_frame_extract_batch(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out);
/* The same without the final wait: returns once everything is queued, so the uploads of the next call overlap the tail of this
 * one (host buffers must be pinned and stay untouched; results are complete after hvo_frame_sync / hvo_frame_timer_stop). */
int hvo_frame_extract_batch_async(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out);
/* Everything device-resident (n <= max_batch); asynchronous.  hvo_frame_sync / hvo_frame_timer_stop wait for all pipelines. */
int hvo_frame_extract_batch_device(hvo_frame* h, const uint8_t* d_gray, const uint16_t* d_depth16, int nframes,
                                   const hvo_frame_outputs* d_out);
/* Attach a vocabulary: the arrays of hvo_bow_set_vocabulary (validated and uploaded by it, to a vocabulary object the handle owns on its
 * device), plus levelsup (Frame::ComputeBoW passes 4).  Waits for the handle's queued work first.  Every later *_bow call given BoW
 * outputs then computes the frames' BowVector / FeatureVector on the device right after the ORB descriptors, on the ORB stream, and
 * returns them with the frame's other outputs; calls without BoW outputs compute none.  Refused (HVO_ERR_ARG) for a handle without
 * the ORB stage or with hvo_frame_capacities' orb_capacity > 4096.  n_nodes == 0 detaches the vocabulary (the other arrays may be NULL).
 * Attaching replaces the previous vocabulary; a refused or failed attach leaves the handle without one. */
int hvo_frame_set_vocabulary(hvo_frame* h, int n_nodes, const int32_t* child_start, const int32_t* child_ids, const uint8_t* node_desc,
                             const double* node_weight, const int32_t* node_word, int depth_levels, int levelsup);
/* hvo_frame_extract_batch / _async / _device with BoW outputs as well.  bow == NULL: exactly the call without _bow.  With bow != NULL
 * the handle needs a vocabulary; on the host bow_counts, bow_words and bow_values are required and fv_order needs node_of; on the
 * device every array of hvo_frame_bow_outputs is required.  Otherwise HVO_ERR_ARG. */
int hvo_frame_extract_batch_bow(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                const hvo_frame_bow_outputs* bow);
int hvo_frame_extract_batch_async_bow(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                      const hvo_frame_bow_outputs* bow);
int hvo_frame_extract_batch_device_bow(hvo_frame* h, const uint8_t* d_gray, const uint16_t* d_depth16, int nframes, const hvo_frame_outputs* d_out,
                                       const hvo_frame_bow_outputs* d_bow);
/* hvo_frame_extract_batch_bow / _async_bow / _device_bow with grid outputs as well; bow and grid may each be NULL, and grid == NULL is exactly
 * the call without _grid (it launches nothing more).  On an undistorting handle the device call needs d_out->kps_un for point grids. */
int hvo_frame_extract_batch_grid(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                 const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid);
int hvo_frame_extract_batch_async_grid(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                       const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid);
int hvo_frame_extract_batch_device_grid(hvo_frame* h, const uint8_t* d_gray, const uint16_t* d_depth16, int nframes, const hvo_frame_outputs* d_out,
                                        const hvo_frame_bow_outputs* d_bow, const hvo_frame_grid_outputs* d_grid);
/* hvo_frame_extract_batch_grid / _async_grid / _device_grid with LPVO outputs as well; bow, grid and lpvo may each be NULL, and lpvo == NULL
 * is exactly the call without _lpvo (it launches nothing more).  Every frame of a call given lpvo gets its LPVO rows: a tracker asks for
 * them in the calls of the frames it constructs while !bManhInit.  The chain runs over passes of at most 256 frames on scratch that the
 * first such call allocates (2.6 MB per frame of a pass at 640x480, 7.8 MB at 1280x720). */
int hvo_frame_extract_batch_lpvo(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                 const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid, const hvo_frame_lpvo_outputs* lpvo);
int hvo_frame_extract_batch_async_lpvo(hvo_frame* h, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                                       const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid, const hvo_frame_lpvo_outputs* lpvo);
int hvo_frame_extract_batch_device_lpvo(hvo_frame* h, const uint8_t* d_gray, const uint16_t* d_depth16, int nframes, const hvo_frame_outputs* d_out,
                                        const hvo_frame_bow_outputs* d_bow, const hvo_frame_grid_outputs* d_grid, const hvo_frame_lpvo_outputs* d_lpvo);
/* rows per frame of hvo_frame_lpvo_outputs: the LPVO lattice size, ceil((W - 11) / 15) * ceil((H - 11) / 15) (0 without the normals stage) */
int hvo_frame_lpvo_capacity(const hvo_frame* h);
/* mnMinX, mnMaxX, mnMinY, mnMaxY the grids are built with (hvo_image_bounds of the handle's camera, computed at create; (0, W, 0, H) when
 * the handle does not undistort).  Frame sets mfGridElementWidthInv = 64.f / (max_x - min_x), mfGridElementHeightInv = 48.f / (max_y - min_y). */
int hvo_frame_image_bounds(const hvo_frame* h, float* min_x, float* max_x, float* min_y, float* max_y);
/* rows per frame of lgrid_items: 64 * max_lines (0 without the line stage) */
int hvo_frame_line_grid_capacity(const hvo_frame* h);
int hvo_frame_last_launches(const hvo_frame* h);
int hvo_frame_sync(hvo_frame* h);
int hvo_frame_timer_start(hvo_frame* h);
int hvo_frame_timer_stop(hvo_frame* h, float* ms_out);

/* ---------------------------------------------------------------------------------------------- SEQUENCE (several GPUs)
 * Offline sequences (BASELINE config 5) on several GPUs of one box from ONE process: Frame construction has no cross-frame state
 * (the extractors' members are scratch: mvImagePyramid, the LBD gradient images), so the frames [0, n) of a call are partitioned
 * across the devices in contiguous ranges (hvo_seq_shard), each device gets one host thread driving one hvo_frame handle with its
 * own streams, and every device writes its own rows of the caller's output arrays: the gather is the layout.  No NCCL, no
 * collective.  gray / depth16 / outputs are HOST arrays of n frames (pinned memory makes the copies asynchronous); a device
 * processes its range as queued calls of at most frames_per_call frames.  Replaces a loop of Frame::Frame(...) extractions over a
 * recorded sequence (Examples/RGB-D/rgbd_tum.cc:86-152 without the tracking step).                                                  */
typedef struct hvo_seq hvo_seq;
int hvo_seq_create(const hvo_frame_params* p, int width, int height, const int* devices, int ndevices, int frames_per_call, hvo_seq** out);
void hvo_seq_destroy(hvo_seq* s);
int hvo_seq_devices(const hvo_seq* s);
int hvo_seq_capacities(const hvo_seq* s, int* orb_capacity, int* max_lines, int* normals_count);
/* the contiguous range of device d (of ndevices) in a call of nframes frames; sizes differ by at most one frame */
void hvo_seq_shard(int nframes, int ndevices, int d, int* first, int* count);
/* blocks until every output row has been written; a device-side fault or CUDA error of any device is returned with its device id */
int hvo_seq_extract(hvo_seq* s, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out);
/* hvo_frame_set_vocabulary on every device's handle (same arguments and rules). */
int hvo_seq_set_vocabulary(hvo_seq* s, int n_nodes, const int32_t* child_start, const int32_t* child_ids, const uint8_t* node_desc,
                           const double* node_weight, const int32_t* node_word, int depth_levels, int levelsup);
/* hvo_seq_extract with the BoW outputs of hvo_frame_extract_batch_bow (host arrays of n frames); bow == NULL: hvo_seq_extract. */
int hvo_seq_extract_bow(hvo_seq* s, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                        const hvo_frame_bow_outputs* bow);
/* hvo_seq_extract_bow with the grid outputs of hvo_frame_extract_batch_grid (host arrays of n frames); bow / grid may each be NULL. */
int hvo_seq_extract_grid(hvo_seq* s, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                         const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid);
/* hvo_seq_extract_grid with the LPVO outputs of hvo_frame_extract_batch_lpvo (host arrays of n frames); bow / grid / lpvo may each be NULL. */
int hvo_seq_extract_lpvo(hvo_seq* s, const uint8_t* gray, const uint16_t* depth16, int nframes, const hvo_frame_outputs* out,
                         const hvo_frame_bow_outputs* bow, const hvo_frame_grid_outputs* grid, const hvo_frame_lpvo_outputs* lpvo);
/* hvo_frame_image_bounds / hvo_frame_line_grid_capacity / hvo_frame_lpvo_capacity of the sequence's handles (the same on every device) */
int hvo_seq_image_bounds(const hvo_seq* s, float* min_x, float* max_x, float* min_y, float* max_y);
int hvo_seq_line_grid_capacity(const hvo_seq* s);
int hvo_seq_lpvo_capacity(const hvo_seq* s);
/* device time of the last hvo_seq_extract: CUDA events around each device's share (uploads, kernels, downloads), max over devices */
float hvo_seq_last_ms(const hvo_seq* s);

#ifdef __cplusplus
}
#endif
#endif /* HVO_CAPI_H */
