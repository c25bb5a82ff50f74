/*
 * swm_orb.h -- C ABI of the B200-native ORB front-end for SwarmMap (libswm_orb.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch/OpenCV types.  The C++
 * wrapper classes with the reference's names (swarmmap_b200/host/ORBextractor.h, ORBmatcher.h)
 * and the Python mirror (swarmmap_b200/orb.py) sit on top of exactly these entry points.
 * Every function returns 0 (SWM_OK) or a negative SWM_E_* code; nothing calls exit() or throws
 * across the boundary (the reference exits on CUDA errors, code/src/cuda/Fast_gpu.cu:346-352).
 * There is no CPU fallback: every compute entry point needs a CUDA device (sm_100a).
 *
 * Reference interfaces replaced (paths relative to /root/reference/code/):
 *   swm_orb_create/destroy      ORBextractor::ORBextractor           src/ORBextractor.cc:340-405
 *   swm_orb_extract[_batch]     ORBextractor::operator()             src/ORBextractor.cc:746-819
 *                               (ComputePyramid :821-855, ComputeKeyPointsOctTree :691-744,
 *                                GpuFast Fast_gpu.cu:284-389, IC_Angle :403-509, GpuOrb Orb_gpu.cu:67-136)
 *   swm_orb_level_ptr           public mvImagePyramid / mvImagePyramidBorder  include/ORBextractor.h:91-92
 *   swm_orb_scale_tables        GetScaleFactors() & friends          include/ORBextractor.h:64-86
 *   swm_hamming_*               ORBmatcher::DescriptorDistance       src/ORBmatcher.cc:1511-1525
 *   swm_match_init              ORBmatcher::SearchForInitialization  src/ORBmatcher.cc:375-479
 *   swm_match_window            ORBmatcher::SearchByProjection x4    src/ORBmatcher.cc:44-121,264-373,1223-1354,1356-1473
 *   swm_match_bow               ORBmatcher::SearchByBoW x2           src/ORBmatcher.cc:150-262,481-597
 *   swm_grid_build              Frame::AssignFeaturesToGrid/GetFeaturesInArea  src/Frame.cc:277-292,377-442
 *   swm_orb_stereo_match        Frame::ComputeStereoMatches          src/Frame.cc:516-690
 *   swm_frame_*                 Frame::UndistortKeyPoints / ComputeImageBounds / AssignFeaturesToGrid on the device
 *                               src/Frame.cc:454-514,277-292
 *   swm_match_triangulation, swm_window_best, swm_distinctive_descriptors
 *                               SearchForTriangulation, the search loop of Fuse x2 / SearchBySim3,
 *                               MapPoint::ComputeDistinctiveDescriptors    src/ORBmatcher.cc:599-1221, src/MapPoint.cc:361-391
 *   swm_match_*_batch           the same Search* calls for many agents in one call (src/Tracking.cc:470-472,619-626,715-737)
 *   swm_vocab_*, swm_bow_*      DBoW2 transform (Frame::ComputeBoW)  Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1151-1283
 *                               and ORBVocabulary::score (L1Scoring::score, ScoringObject.cpp)
 *   swm_kfdb_*                  KeyFrameDatabase (add / erase / clear / DetectRelocalizationCandidates /
 *                               DetectLoopCandidates)                src/KeyFrameDatabase.cc
 *   swm_db_*                    role of KeyFrameDatabase::DetectLoopCandidates + SearchByBoW(KF,KF) in
 *                               AgentMediator::CheckOverlapCandidates (src/AgentMediator.cc:140-202), recast as
 *                               brute-force Hamming top-k over a sharded descriptor database (BASELINE config 5);
 *                               across GPUs: swm_db_query_peers (peer-memory exchange) / swm_db_query_sharded (NCCL)
 */
#ifndef SWM_ORB_H
#define SWM_ORB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SWM_OK 0
#define SWM_E_INVALID (-1)   /* bad argument */
#define SWM_E_CUDA (-2)      /* CUDA runtime error; see swm_last_error */
#define SWM_E_NODEVICE (-3)  /* no CUDA device / wrong architecture: there is no CPU fallback */
#define SWM_E_CAPACITY (-4)  /* caller buffer or configured batch too small */
#define SWM_E_STATE (-5)     /* call order violation (e.g. level_ptr before the first extract) */

#define SWM_EDGE_THRESHOLD 19 /* ORBextractor.cc:78 */
#define SWM_MAX_LEVELS 16

/* Same size (28 B) and field order as cv::KeyPoint, which the reference already memcpy's raw
 * to and from the device (Fast_gpu.cu:490,507; Orb_gpu.cu:123). */
typedef struct swm_keypoint {
  float x, y;      /* pt, in level-0 pixel units (level coords * scale factor, ORBextractor.cc:808-814) */
  float size;      /* int(31 * scale[level]) (Fast_gpu.cu:462,470) */
  float angle;     /* degrees in [0,360) (Fast_gpu.cu:451-456) */
  float response;  /* FAST score */
  int32_t octave;  /* pyramid level */
  int32_t class_id; /* -1 */
} swm_keypoint;

typedef struct swm_orb_cfg {
  int32_t nfeatures;     /* ORBextractor.nFeatures */
  float scale_factor;    /* ORBextractor.scaleFactor (1.2) */
  int32_t nlevels;       /* ORBextractor.nLevels (8) */
  int32_t ini_th_fast;   /* ORBextractor.iniThFAST (20) */
  int32_t min_th_fast;   /* ORBextractor.minThFAST (7) */
  int32_t max_batch;     /* frames per launch the handle is sized for (>=1) */
  int32_t max_fast_per_level; /* FAST candidate cap per level; 0 -> 10000 (Fast.hpp:30) */
} swm_orb_cfg;

typedef struct swm_orb swm_orb; /* opaque extractor handle: owns device buffers, streams, tables */

/* ------------------------------------------------------------------ extractor */
int swm_orb_create(const swm_orb_cfg* cfg, int device, swm_orb** out);
void swm_orb_destroy(swm_orb* h);
/* Last error text of this handle (or of the failed create when h == NULL). */
const char* swm_last_error(const swm_orb* h);

/* One frame, host buffers in and out (the reference's operator() contract).  img: 8-bit gray,
 * `stride` bytes per row.  kps/desc: caller-owned, room for `cap` keypoints / cap*32 bytes.
 * *n receives the count.  An empty image (w or h == 0, or img == NULL) returns SWM_OK with *n = 0
 * (ORBextractor.cc:750-751). */
int swm_orb_extract(swm_orb* h, const uint8_t* img, int w, int h_px, int stride, swm_keypoint* kps, uint8_t* desc,
                    int cap, int* n);

/* `batch` frames of identical size, frame f at imgs + f*frame_stride; outputs for frame f at
 * kps + f*cap, desc + f*cap*32, n[f].  Host buffers (pinned memory recommended). */
int swm_orb_extract_batch(swm_orb* h, const uint8_t* imgs, int batch, int w, int h_px, int stride,
                          size_t frame_stride, swm_keypoint* kps, uint8_t* desc, int cap, int32_t* n);

/* Asynchronous form of swm_orb_extract_batch: enqueues the H2D copies, the kernels and the D2H
 * copies on the handle's stream and returns.  batch <= cfg.max_batch.  Host buffers (pinned, or
 * the copies serialise) must stay valid until swm_orb_sync(h) returns; results are defined then.
 * Two handles used alternately overlap one batch's transfers with the other's kernels. */
int swm_orb_extract_batch_async(swm_orb* h, const uint8_t* imgs, int batch, int w, int h_px, int stride,
                                size_t frame_stride, swm_keypoint* kps, uint8_t* desc, int cap, int32_t* n);
int swm_orb_sync(swm_orb* h);

/* Same, all pointers are DEVICE pointers and the work is enqueued on `stream` (a cudaStream_t
 * passed as void*; NULL = the handle's own stream).  Does not synchronise. */
int swm_orb_extract_batch_device(swm_orb* h, const uint8_t* d_imgs, int batch, int w, int h_px, int stride,
                                 size_t frame_stride, swm_keypoint* d_kps, uint8_t* d_desc, int cap, int32_t* d_n,
                                 void* stream);

/* Device pointer to pyramid level `level` of frame `frame` of the last batch.
 * which: 0 = un-blurred ROI inside the bordered plane (pointer to pixel (0,0); the 19-px
 * reflect-101 border lies at negative offsets), 1 = blurred ROI (what mvImagePyramid holds after
 * the reference's operator()). */
int swm_orb_level_ptr(swm_orb* h, int frame, int level, int which, const uint8_t** dev, int* w, int* h_px,
                      int* pitch);
int swm_orb_scale_tables(const swm_orb* h, float* scale, float* inv_scale, float* sigma2, float* inv_sigma2);
int swm_orb_level_quotas(const swm_orb* h, int32_t* quotas);
/* Capacity a caller must provide per frame so no keypoint is ever dropped. */
int swm_orb_max_keypoints(const swm_orb* h);
/* Number of kernel launches issued by the last extract call (bench.py's gpu_launches). */
int swm_orb_last_launches(const swm_orb* h);
/* Frame::ComputeStereoMatches (reference code/src/Frame.cc:516-690) on the device, from the resident results of two
 * extractors: `left` and `right` hold the last extracted batch of the left and right views of the same frames (same
 * device, batch, frame size and pyramid).  For frame f of the batch, left keypoint i gets
 * u_right[f * cap + i] = mvuRight[i] and depth[f * cap + i] = mvDepth[i] (-1 = no stereo match), bit-identical to the
 * reference's loop: best descriptor distance in the keypoint's row band (octave +-1, disparity in [-3, bf / b]), 11x11
 * SAD refinement over +-5 px in mvImagePyramid[level] as operator() leaves it (blurred in place), parabola fit, 1.5 * 1.4 * median SAD filter.  bf = mbf
 * (baseline x fx), b = mb (baseline in metres).  cap >= swm_orb_max_keypoints(left), or the cap the batch was extracted
 * with; host outputs, returns after the results are in place. */
int swm_orb_stereo_match(swm_orb* left, swm_orb* right, float bf, float b, float* u_right, float* depth, int cap);
/* Re-runs the selected stages on the data of the last *_device/_batch call (the caller brackets it with
 * CUDA events on `stream`): per-stage timing for bench.py's roofline and stage breakdown. */
int swm_orb_run_stage(swm_orb* h, int stage_mask, int batch, void* stream);
#define SWM_STAGE_PYRAMID 1 /* pyramid + border + Gaussian blur (pyr_walk_kernel x nlevels) */
#define SWM_STAGE_NMS 2     /* FAST score + tile retry + non-max suppression (fast_tile_kernel x 2) */
#define SWM_STAGE_OCTREE 4
#define SWM_STAGE_DESCRIBE 8 /* orientation + rBRIEF + output assembly */

/* Parity introspection (host copies of intermediates of frame `frame` of the last batch).
 * which: 0 = bordered un-blurred plane ((w+38)x(h+38)), 1 = blurred ROI, 2 = FAST score map (w x h). */
/* which = 2 needs swm_orb_set_debug(h, 1) before the first extract (the product keeps no score map). */
int swm_orb_set_debug(swm_orb* h, int keep_score_map);
int swm_orb_debug_plane(swm_orb* h, int frame, int level, int which, uint8_t* out, int out_stride);
/* FAST candidates after tile-retry+NMS (which = 0; ROI coords; order unspecified) or quadtree
 * selection (which = 1; final list order).  xys: (x, y, score) int32 triples. Returns count or <0. */
int swm_orb_debug_points(swm_orb* h, int frame, int level, int which, int32_t* xys, int cap);

/* ------------------------------------------------------------------ Hamming primitives */
/* Single pair on the host side of the ABI is pointless on a GPU; DescriptorDistance is served by
 * the batched forms.  a: na x 32 bytes, b: nb x 32 bytes (device pointers), out: na x nb uint16. */
int swm_hamming_matrix_device(const uint8_t* d_a, int na, const uint8_t* d_b, int nb, uint16_t* d_out, void* stream);
/* Host-buffer convenience (copies in/out). */
int swm_hamming_matrix(const uint8_t* a, int na, const uint8_t* b, int nb, uint16_t* out, int device);
/* Element-wise pairs: out[i] = dist(a[i], b[i]). */
int swm_hamming_pairs(const uint8_t* a, const uint8_t* b, int n, int32_t* out, int device);
/* MapPoint::ComputeDistinctiveDescriptors (code/src/MapPoint.cc:361-391) for a batch of MapPoints: point p owns the
 * descriptors desc[offsets[p] .. offsets[p+1]) (its observations, in the std::map<KeyFrame*, size_t> iteration order
 * the caller gathered them in; at most 1024 per point).  best_idx[p]: index inside the point of the descriptor with
 * the least median distance to the others (median = sorted[int(0.5 * (N - 1))], first minimum wins), -1 for an
 * empty point; best_median (may be NULL) that median. */
int swm_distinctive_descriptors(const uint8_t* desc, const int32_t* offsets, int npoints, int32_t* best_idx,
                                int32_t* best_median, int device);

/* ------------------------------------------------------------------ matchers (flat POD views) */
/* One frame's features as the matchers see them (host pointers). */
typedef struct swm_frame_view {
  int32_t n;
  const float* x;         /* mvKeysUn[i].pt.x */
  const float* y;
  const int32_t* octave;
  const float* angle;
  const uint8_t* desc;    /* n x 32, row-major (mDescriptors) */
  float min_x, min_y, max_x, max_y; /* Frame::mnMinX.. (Frame.cc:59-60) */
} swm_frame_view;

#define SWM_GRID_COLS 64 /* FRAME_GRID_COLS, Frame.h:38 */
#define SWM_GRID_ROWS 48 /* FRAME_GRID_ROWS, Frame.h:37 */

typedef struct swm_matcher swm_matcher; /* opaque: device scratch + stream for matcher calls */
int swm_matcher_create(int device, swm_matcher** out);
void swm_matcher_destroy(swm_matcher* m);
const char* swm_matcher_last_error(const swm_matcher* m);

/* Frame::AssignFeaturesToGrid as CSR: starts has 64*48+1 entries, cell = ix*48+iy; items (n entries
 * at most) hold keypoint indices in ascending order per cell. */
int swm_grid_build(swm_matcher* m, const swm_frame_view* f, int32_t* starts, int32_t* items);

/* M1 SearchForInitialization: prev_xy (n1 x 2 floats) is vbPrevMatched, read and updated;
 * matches12 (n1) receives F2 indices or -1; *nmatches the return value. */
int swm_match_init(swm_matcher* m, const swm_frame_view* f1, const swm_frame_view* f2, float* prev_xy,
                   int32_t* matches12, int window, float nnratio, int check_ori, int* nmatches);

/* Generic windowed projection matcher behind the four SearchByProjection overloads.  The C++
 * wrapper projects each source (MapPoint) and fills one row per source:
 *   valid[s]      0 = skipped (bad / not in view / outside image ...)
 *   u,v,radius    window centre and half-size passed to GetFeaturesInArea
 *   min_level,max_level   its level arguments (-1,-1 disables; Frame.cc:398)
 *   desc          the source descriptor (MapPoint::GetDescriptor)
 *   angle         source keypoint angle for the rotation histogram (ignored if !check_ori)
 *   blocks[s]     1 if, once assigned, the target slot is unavailable to later sources
 *                 (pMP->Observations()>0 for :67-69/:1291-1293; always 1 for :306,:1413)
 * tgt_blocked (n2, may be NULL): slots unavailable from the start.
 * ratio_mode 0: accept best <= th_dist.  ratio_mode 1: additionally reject when best and second
 * best share a level and best > nnratio*second (:110-113).
 * assignment (n2, in/out): source index written at accepted slots (later sources overwrite).
 * With check_ori the rotation histogram prunes assignments made by this call (:1320-1351). */
typedef struct swm_window_query {
  int32_t m;
  const uint8_t* desc;
  const float* u;
  const float* v;
  const float* radius;
  const int32_t* min_level;
  const int32_t* max_level;
  const uint8_t* valid;
  const float* angle;
  const uint8_t* blocks;
} swm_window_query;

int swm_match_window(swm_matcher* m, const swm_frame_view* tgt, const swm_window_query* q,
                     const uint8_t* tgt_blocked, int th_dist, int ratio_mode, float nnratio, int check_ori,
                     int32_t* assignment, int* nmatches);

/* DBoW2::FeatureVector as CSR (ascending node ids; ascending feature indices per node). */
typedef struct swm_featvec {
  int32_t n_nodes;
  const uint32_t* node_ids;
  const int32_t* offsets; /* n_nodes + 1 */
  const uint32_t* feats;
} swm_featvec;

/* M4 SearchByBoW.  mode 0: KeyFrame->Frame (:150-262): valid1 = KF feature has a good MapPoint;
 * matches (n2) = KF feature index per Frame feature or -1.  mode 1: KeyFrame<->KeyFrame
 * (:481-597): valid1/valid2 per side; matches (n1) = KF2 feature index or -1. */
int swm_match_bow(swm_matcher* m, const swm_frame_view* f1, const swm_featvec* fv1, const uint8_t* valid1,
                  const swm_frame_view* f2, const swm_featvec* fv2, const uint8_t* valid2, int mode, float nnratio,
                  int check_ori, int32_t* matches, int* nmatches);

/* Best keypoint inside a window, one independent row per query: the search loop shared by ORBmatcher::Fuse
 * (ORBmatcher.cc:824-870 and :962-999) and SearchBySim3 (:1098-1134, :1178-1214).  Candidates =
 * GetFeaturesInArea(u, v, radius, min_level, max_level) in its order (Fuse / SearchBySim3 pass nPredictedLevel - 1,
 * nPredictedLevel); with chi2 > 0 the monocular reprojection gate e2 * inv_level_sigma2[level] > chi2 -> skip
 * (:857-864, chi2 = 5.99) is applied; winner = smallest distance, the first candidate on ties ("dist < bestDist").
 * best_idx[i] = -1 and best_dist[i] = 256 when no candidate survives.  The callers' accept thresholds (TH_LOW /
 * TH_HIGH) and the MapPoint bookkeeping (Replace / AddObservation, in order) stay in the C++ wrapper. */
typedef struct swm_best_query {
  int32_t m;
  const uint8_t* desc;
  const float* u;
  const float* v;
  const float* radius;
  const int32_t* min_level;
  const int32_t* max_level;
  const uint8_t* valid;
  const float* inv_level_sigma2; /* pKF->mvInvLevelSigma2 (read when chi2 > 0) */
  int32_t nlevels;
  float chi2;                    /* <= 0: no reprojection gate */
} swm_best_query;
int swm_window_best(swm_matcher* m, const swm_frame_view* tgt, const swm_best_query* q, int32_t* best_idx,
                    int32_t* best_dist);

/* ORBmatcher::SearchForTriangulation (ORBmatcher.cc:599-749) with CheckDistEpipolarLine (:131-148), monocular
 * (mvuRight < 0, bOnlyStereo = false).  The C++ wrapper computes the epipole (:605-611) and passes F12 and pKF2's
 * level tables; valid1 / valid2 mark keypoints WITHOUT a MapPoint (:640-643, :662-666).  The reference never sets
 * vbMatched2, so every KF1 keypoint picks independently: smallest distance <= TH_LOW among the candidates of its
 * vocabulary node that pass the epipole-distance and epipolar-line tests, the last one on ties; then the rotation
 * histogram prunes.  matches12 (n1): KF2 index or -1 (vMatchedPairs = the non-negative entries in index order). */
typedef struct swm_triangulation_query {
  const float* F12;            /* 3 x 3, row-major */
  float ex, ey;                /* epipole of KF1's camera centre in KF2 */
  const float* scale_factors2; /* pKF2->mvScaleFactors */
  const float* level_sigma2;   /* pKF2->mvLevelSigma2 */
  int32_t nlevels;
} swm_triangulation_query;
int swm_match_triangulation(swm_matcher* m, const swm_frame_view* f1, const swm_featvec* fv1, const uint8_t* valid1,
                            const swm_frame_view* f2, const swm_featvec* fv2, const uint8_t* valid2,
                            const swm_triangulation_query* q, int check_ori, int32_t* matches12, int* nmatches);

/* ------------------------------------------------------------------ resident frames
 * SURVEY section 8(f) rank 1: Frame::UndistortKeyPoints (code/src/Frame.cc:454-484), ComputeImageBounds
 * (:486-514) and AssignFeaturesToGrid (:277-292, PosInGrid :427-442) on the device, so that the
 * extractor's output feeds the matchers without a host round trip.  The *_resident matchers have
 * exactly the semantics and results of their swm_frame_view forms. */
typedef struct swm_camera {
  float fx, fy, cx, cy;       /* mK */
  float k1, k2, p1, p2, k3;   /* mDistCoef (k3 = 0 when the settings file has four coefficients) */
} swm_camera;

/* bounds4 = mnMinX, mnMaxX, mnMinY, mnMaxY (Frame.cc:486-514); the four corners go through the same
 * device undistortion as the keypoints. */
int swm_camera_bounds(int device, const swm_camera* cam, int cols, int rows, float* bounds4);

typedef struct swm_frame swm_frame; /* opaque: undistorted keypoints (SoA), descriptors, grid, on one device */
int swm_frame_create(int device, swm_frame** out);
void swm_frame_destroy(swm_frame* f);
const char* swm_frame_last_error(const swm_frame* f);
int32_t swm_frame_size(const swm_frame* f);
/* Frame `index` of the extractor's most recent batch -> resident frame, on the extractor's stream:
 * cv::undistortPoints(K, D, P = K) semantics in double (bit-identical to OpenCV's scalar code), mvKeysUn =
 * mvKeys when cam is NULL or k1 == 0 (:456-460), descriptor copy, grid.  Only the 4-byte keypoint count is
 * read back. */
int swm_frame_from_extractor(swm_frame* f, swm_orb* h, int index, const swm_camera* cam, const float* bounds4);
/* The same from host arrays (e.g. a keyframe of the map); v's x / y are already undistorted. */
int swm_frame_upload(swm_frame* f, const swm_frame_view* v);
/* Reads a resident frame back (tracking needs mvKeysUn for pose optimisation); any pointer may be NULL.
 * grid_starts: 64*48+1 entries, grid_items: up to n entries (same CSR as swm_grid_build). */
int swm_frame_download(swm_frame* f, float* x, float* y, int32_t* octave, float* angle, uint8_t* desc,
                       int32_t* grid_starts, int32_t* grid_items);
/* Binary keyframe-feature slab (SURVEY section 8(f) rank 4): the wire / on-disk form of a keyframe's features in
 * place of the Boost text archive (code/src/MapUpdater.cc:192-230, code/include/KeyFrame.h:309-404).  Layout, little
 * endian: uint32 magic "SWKF", uint32 version (1), int32 n, float min_x, max_x, min_y, max_y, uint32 reserved,
 * float x[n], float y[n], int32 octave[n], float angle[n], uint8 desc[n][32] = 32 + 48 n bytes (about a quarter of
 * the text archive).  export: five device-to-host copies; import: validates the header, uploads and rebuilds the grid. */
size_t swm_frame_slab_bytes(int32_t n);
int swm_frame_export(swm_frame* f, uint8_t* buf, size_t cap, size_t* bytes);
int swm_frame_import(swm_frame* f, const uint8_t* buf, size_t bytes);

int swm_match_init_resident(swm_matcher* m, const swm_frame* f1, const swm_frame* f2, float* prev_xy, int32_t* matches12,
                            int window, float nnratio, int check_ori, int* nmatches);
int swm_match_window_resident(swm_matcher* m, const swm_frame* tgt, const swm_window_query* q,
                              const uint8_t* tgt_blocked, int th_dist, int ratio_mode, float nnratio, int check_ori,
                              int32_t* assignment, int* nmatches);
int swm_match_bow_resident(swm_matcher* m, const swm_frame* f1, const swm_featvec* fv1, const uint8_t* valid1,
                           const swm_frame* f2, const swm_featvec* fv2, const uint8_t* valid2, int mode, float nnratio,
                           int check_ori, int32_t* matches, int* nmatches);
int swm_match_triangulation_resident(swm_matcher* m, const swm_frame* f1, const swm_featvec* fv1, const uint8_t* valid1,
                                     const swm_frame* f2, const swm_featvec* fv2, const uint8_t* valid2,
                                     const swm_triangulation_query* q, int check_ori, int32_t* matches12, int* nmatches);
int swm_window_best_resident(swm_matcher* m, const swm_frame* tgt, const swm_best_query* q, int32_t* best_idx,
                             int32_t* best_dist);

/* ------------------------------------------------------------------ batched matchers (throughput form)
 * P independent matching problems per call: what a GPU serving many agents -- or a recorded stream being replayed --
 * has in flight.  All host arrays of all jobs travel in ONE upload, six launches serve the whole batch (one resolve
 * CTA per job replays that job's greedy order: code/src/ORBmatcher.cc:44-121, :150-262, :375-479, :481-597,
 * :1223-1354), ONE download brings every result back, and there is no synchronisation in the middle of the call.
 * Each job has exactly the semantics and the results of the corresponding single call above: swm_match_window,
 * swm_match_init, swm_match_bow.  A job's frames are host arrays (f1 / f2 / tgt) OR resident frames (r1 / r2 /
 * tgt_resident), never both.  nmatches is written into the job. */
typedef struct swm_window_job {
  const swm_frame_view* tgt;
  const swm_frame* tgt_resident;
  const swm_window_query* q;
  const uint8_t* tgt_blocked; /* n2, may be NULL */
  int32_t th_dist, ratio_mode;
  float nnratio;
  int32_t check_ori;
  int32_t* assignment;        /* n2, in/out */
  int32_t nmatches;           /* out */
} swm_window_job;
int swm_match_window_batch(swm_matcher* m, swm_window_job* jobs, int njobs);

typedef struct swm_init_job {
  const swm_frame_view *f1, *f2;
  const swm_frame *r1, *r2;
  float* prev_xy;             /* n1 x 2, in/out */
  int32_t* matches12;         /* n1, out */
  int32_t window;
  float nnratio;
  int32_t check_ori;
  int32_t nmatches;           /* out */
} swm_init_job;
int swm_match_init_batch(swm_matcher* m, swm_init_job* jobs, int njobs);

/* The merge-walk over the two FeatureVectors and the expansion of the shared nodes into candidate rows run on the
 * device from the two CSRs (node ids strictly ascending). */
typedef struct swm_bow_job {
  const swm_frame_view *f1, *f2;
  const swm_frame *r1, *r2;
  const swm_featvec *fv1, *fv2;
  const uint8_t *valid1, *valid2; /* valid2: mode 1 only */
  int32_t mode;
  float nnratio;
  int32_t check_ori;
  int32_t* matches;           /* mode 0: n2 entries, mode 1: n1 entries */
  int32_t nmatches;           /* out */
} swm_bow_job;
int swm_match_bow_batch(swm_matcher* m, swm_bow_job* jobs, int njobs);

/* Device time (ms, CUDA events on the matcher's stream) of the six kernels of the most recent batch call, without its
 * upload and download: what bench.py reports next to the host-clock time of the whole call. */
float swm_matcher_last_device_ms(const swm_matcher* m);

/* Resident frames for `count` frames of the extractor's most recent batch in two launches and one read-back of the
 * keypoint counts (indices == NULL: frames 0 .. count-1).  Same results as swm_frame_from_extractor per frame. */
int swm_frames_from_extractor(swm_frame** frames, int count, swm_orb* h, const int32_t* indices, const swm_camera* cam,
                              const float* bounds4);

/* ------------------------------------------------------------------ DBoW2 transform (SURVEY section 8(f) rank 2)
 * TemplatedVocabulary<FORB>::transform(features, BowVector&, FeatureVector&, levelsup)
 * (code/Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1151-1218, per feature :1242-1283) as called by
 * Frame::ComputeBoW (code/src/Frame.cc:445-452), KeyFrame::ComputeBoW (code/src/KeyFrame.cc:126-133) and the
 * server for every received keyframe (code/src/Map.cc:372-385); SwarmMap always passes levelsup = 4. */
#define SWM_BOW_MAX_FEATURES 8192
typedef struct swm_vocab swm_vocab; /* opaque: the vocabulary tree on one device */
/* blob: the file TemplatedVocabulary::loadFromBinaryFile reads (:1478-1522), e.g. ORBvoc.bin:
 * uint32 nb_nodes, uint32 size_node (41), int32 k, L, scoring, weighting; then per node id 1.. :
 * int32 parent, 32 descriptor bytes, float weight, uint8 is_leaf. */
int swm_vocab_create(int device, const uint8_t* blob, size_t bytes, swm_vocab** out);
void swm_vocab_destroy(swm_vocab* v);
const char* swm_vocab_last_error(const swm_vocab* v);
int swm_vocab_info(const swm_vocab* v, int32_t* k, int32_t* L, int32_t* n_nodes, int32_t* n_words);

/* Host output slabs for `batch` frames of capacity `cap` features each.  Frame b:
 *   BowVector      word_ids[b*cap ..], word_values[b*cap ..] (n_words[b] entries, ascending word id = std::map order)
 *   FeatureVector  node_ids[b*cap ..] (n_nodes[b] entries, ascending), node_offsets[b*(cap+1) ..] (n_nodes[b] + 1),
 *                  feats[b*cap ..] (ascending feature indices per node: FeatureVector.cpp:31-45)
 * i.e. the swm_featvec CSR the SearchByBoW entry points take. */
typedef struct swm_bow_out {
  uint32_t* word_ids;
  double* word_values;
  int32_t* n_words;
  uint32_t* node_ids;
  int32_t* node_offsets;
  uint32_t* feats;
  int32_t* n_nodes;
} swm_bow_out;
/* desc: host [batch][cap][32], n[b] valid rows per frame (<= cap <= SWM_BOW_MAX_FEATURES). */
int swm_bow_transform(swm_vocab* v, const uint8_t* desc, const int32_t* n, int batch, int cap, int levelsup,
                      const swm_bow_out* out);
/* The same for one resident frame (cap = swm_frame_size(f)); the descriptors never leave the device. */
int swm_bow_transform_frame(swm_vocab* v, const swm_frame* f, int levelsup, const swm_bow_out* out);
/* ORBVocabulary::score (TemplatedVocabulary.h, DBoW2 ScoringObject.cpp L1Scoring::score) of npairs pairs of
 * BowVectors: out[i] = score(a_i, b_i), bit-exact.  Pair i's vectors are a_words / a_values[a_offsets[i] ..
 * a_offsets[i+1]) and likewise for b; word ids strictly ascending.  L1_NORM vocabularies only (SWM_E_INVALID
 * otherwise). */
int swm_bow_score(swm_vocab* v, int npairs, const int32_t* a_offsets, const uint32_t* a_words, const double* a_values,
                  const int32_t* b_offsets, const uint32_t* b_words, const double* b_values, double* out);

/* ------------------------------------------------------------------ KeyFrameDatabase (place recognition)
 * KeyFrameDatabase::{add, erase, clear, DetectRelocalizationCandidates, DetectLoopCandidates} (ORB-SLAM2's
 * KeyFrameDatabase.cc as SwarmMap carries it; callers Tracking::Relocalization, LoopClosing::DetectLoop,
 * AgentMediator::CheckOverlapCandidates) on one device, with DBoW2's L1 score.  Results equal the reference's
 * ordered candidate lists exactly under the definitions of DESIGN.md section 2: stale reloc scores are reproduced
 * (kept per keyframe id for the database's lifetime, through erase / re-add / clear), they start at 0.0f, and every
 * query is a fresh query.  A batch of queries equals the same queries issued one after another in array order.
 *
 * A query has two phases because the reference reads the covisibility graph only for the scored keyframes:
 *   swm_kfdb_query   scores the database against nq BowVectors and returns, per query, lScoreAndMatch in list
 *                    order (keyframe ids and float scores) in the CSR scored_offsets[nq + 1] / scored_ids /
 *                    scored_scores;
 *   swm_kfdb_finish  takes each scored entry's GetBestCovisibilityKeyFrames(10) (ids, in order; CSR aligned with the
 *                    scored entries, ids not in the database are ignored) and returns the candidates per query in
 *                    the CSR cand_offsets[nq + 1] / cand_ids.
 * finish without a preceding query, or after an add / erase / clear since it, returns SWM_E_STATE.  A capacity too
 * small returns SWM_E_CAPACITY with the size needed in scored_offsets[nq] / cand_offsets[nq]; a query that fails
 * this way changes no state and can be repeated with a larger buffer. */
#define SWM_KFDB_RELOC 0 /* DetectRelocalizationCandidates(Frame*) */
#define SWM_KFDB_LOOP 1  /* DetectLoopCandidates(KeyFrame*, minScore) */
typedef struct swm_kfdb swm_kfdb; /* opaque: the database on the vocabulary's device */
/* SWM_E_INVALID unless the vocabulary's scoring type is L1_NORM (ORBvoc's). */
int swm_kfdb_create(swm_vocab* v, swm_kfdb** out);
void swm_kfdb_destroy(swm_kfdb* db);
const char* swm_kfdb_last_error(const swm_kfdb* db);
int64_t swm_kfdb_size(const swm_kfdb* db); /* live keyframes */
/* n keyframes; keyframe i: id kf_ids[i], BowVector word_ids / values[offsets[i] .. offsets[i+1]) (ascending word
 * ids).  SWM_E_INVALID (nothing added) for an id that is live already or a word id >= the vocabulary's size. */
int swm_kfdb_add(swm_kfdb* db, int n, const uint64_t* kf_ids, const int32_t* offsets, const uint32_t* word_ids,
                 const double* values);
int swm_kfdb_erase(swm_kfdb* db, int n, const uint64_t* kf_ids); /* ids that are not live are ignored */
int swm_kfdb_clear(swm_kfdb* db);
/* mode SWM_KFDB_RELOC or SWM_KFDB_LOOP; nq queries, query q = q_words / q_values[q_offsets[q] .. q_offsets[q+1]).
 * Loop mode: min_score[nq], and GetConnectedKeyFrames() of query q = conn_ids[conn_offsets[q] .. conn_offsets[q+1])
 * (conn_offsets NULL: none); both are ignored in reloc mode. */
int swm_kfdb_query(swm_kfdb* db, int mode, int nq, const int32_t* q_offsets, const uint32_t* q_words,
                   const double* q_values, const float* min_score, const int32_t* conn_offsets,
                   const uint64_t* conn_ids, int32_t* scored_offsets, uint64_t* scored_ids, float* scored_scores,
                   int32_t scored_cap);
int swm_kfdb_finish(swm_kfdb* db, const int32_t* neigh_offsets, const uint64_t* neigh_ids, int32_t* cand_offsets,
                    uint64_t* cand_ids, int32_t cand_cap);
/* Device time of the last query + finish pair, from events around each phase's device work, in ms. */
float swm_kfdb_last_device_ms(const swm_kfdb* db);

/* ------------------------------------------------------------------ place-recognition shard (config 5) */
typedef struct swm_db swm_db; /* one GPU's shard of the keyframe-descriptor database */
/* desc: ndesc x 32 bytes (host), kf_of_desc optional (NULL -> desc i belongs to kf i / desc_per_kf). */
int swm_db_create(int device, const uint8_t* desc, int64_t ndesc, int32_t desc_per_kf, int64_t first_kf_id,
                  swm_db** out);
int swm_db_create_device(int device, const uint8_t* d_desc, int64_t ndesc, int32_t desc_per_kf,
                         int64_t first_kf_id, swm_db** out);
void swm_db_destroy(swm_db* db);
/* For each of nq query descriptors (device): the k (<=2) nearest database descriptors of this
 * shard as packed 64-bit keys (dist << 48 | global_desc_index), ascending; ties -> lower index.
 * d_votes (optional, n_kf of this shard, int32): += 1 for the keyframe owning each query's best
 * match when best <= th_votes (TH_LOW). */
int swm_db_query_device(swm_db* db, const uint8_t* d_q, int nq, int k, uint64_t* d_topk, int32_t* d_votes,
                        int th_votes, void* stream);
/* Multi-GPU step after the all-gather of the per-shard (nq, k) key blocks: d_gathered is (world, nq, k); writes
 * the k smallest keys per query to d_topk and, into d_votes (optional, this shard's n_kf counters, += 1), the vote
 * of every query whose GLOBAL best match is <= th_votes and belongs to a keyframe of this shard (summed over the
 * ranks this equals the single-shard vote histogram). */
int swm_db_merge_gathered(swm_db* db, const uint64_t* d_gathered, int world, int nq, int k, uint64_t* d_topk,
                          int32_t* d_votes, int th_votes, void* stream);
/* The whole sharded query on one rank, for a C++ caller (the role of AgentMediator::CheckOverlapCandidates,
 * code/src/AgentMediator.cc:140-202 + KeyFrameDatabase.cc:74-185): local top-k, ONE ncclAllGather of the (nq, k) key
 * blocks over NVLink, merge + votes -- three enqueues on `stream`, no host synchronisation.  nccl_comm: an
 * ncclComm_t (passed as void* so that this header does not need nccl.h) of `world` ranks, one shard each; the
 * library binds ncclAllGather from the NCCL already loaded in the process (dlopen, no link-time dependency).
 * d_topk (nq x k) is identical on every rank; d_votes: this shard's keyframes, as in swm_db_merge_gathered. */
int swm_db_query_sharded(swm_db* db, void* nccl_comm, int world, const uint8_t* d_q, int nq, int k, uint64_t* d_topk,
                         int32_t* d_votes, int th_votes, void* stream);
/* The same sharded query with the exchange over PEER MEMORY (NVLink / NVSwitch) inside the merge kernel instead of an
 * NCCL collective: every rank owns a window that its peers store their (nq, k) key block into, publish a flag, and wait
 * for the others' flags -- one kernel per rank after the shard scan (db_merge_peers_kernel, csrc/match.cu).  All ranks
 * live on one node with peer access between their GPUs.
 *   swm_db_peer_window: allocate this rank's window for `world` ranks and up to nq_max (<= 8192) queries; returns its
 *     cudaIpcMemHandle_t as 64 opaque bytes (ipc_handle64, may be NULL) and / or its device address (window, may be
 *     NULL) for ranks that share the process;
 *   swm_db_peer_open: give the windows of all ranks in rank order -- either world x 64 bytes of IPC handles gathered
 *     from the other processes by whatever transport the server has (MPI, torch.distributed, a socket), or an array of
 *     device addresses when the ranks share a process; the entry of `rank` itself is ignored;
 *   swm_db_query_peers: a collective -- every rank enqueues it with the same nq and k, the same number of times;
 *     results as swm_db_query_sharded.  Three enqueues become two (scan, fused merge + exchange + merge).  A rank that
 *     never joins makes the others abort (device trap) after minutes of waiting; a rank that re-creates its window
 *     (swm_db_peer_window again) must hand the new handle to every peer before the next query. */
int swm_db_peer_window(swm_db* db, int world, int nq_max, void* ipc_handle64, void** window);
int swm_db_peer_open(swm_db* db, int rank, const void* ipc_handles, void* const* windows);
int swm_db_query_peers(swm_db* db, const uint8_t* d_q, int nq, int k, uint64_t* d_topk, int32_t* d_votes, int th_votes,
                       void* stream);
int64_t swm_db_size(const swm_db* db);
/* Measured int8 rate of the tensor pipe on `device`, in TOP/s: one CTA per SM issues `iters` back-to-back tcgen05
 * kind::i8 MMAs and nothing else (mode 0: 128 x 64 x 32 with A in TMEM, the shape the shard scan issues; mode 1:
 * 128 x 256 x 32 from shared memory).  The denominator of the shard scan's roofline in bench.py. */
int swm_i8_peak(int device, int mode, int iters, double* tops);

/* Build id string ("swm_orb <version> sm_100a <date>"). */
const char* swm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SWM_ORB_H */
