/*
 * vsg_cuda.h — C ABI of libvsg_cuda.so: the B200 (sm_100a) ORB feature front-end for vS-Graphs.
 *
 * This is the drop-in boundary for the reference's feature front-end (snt-arg/visual_sgraphs; paths
 * below are relative to that checkout).  The reference has no FFI for this path — the hot path is two
 * C++ classes compiled into liborb_slam3_ros.so — so every entry point names the reference interface
 * it replaces; the C++ classes in visual_sgraphs_b200/shim/ (VS_GRAPHS::ORBextractor / ORBmatcher,
 * same signatures as orb_slam3/include/ORBextractor.h and ORBmatcher.h) forward to these functions.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only; no C++/OpenCV/torch types.
 *   - pointers are HOST pointers unless the parameter name ends in _dev.
 *   - every function returns vsg_status (0 = ok, negative = error; vsg_last_error() has the text).
 *     There is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     VSG_ERR_CUDA.
 *   - handles are not re-entrant (like the reference's ORBextractor instance, which mutates
 *     mvImagePyramid) but distinct handles may be used concurrently from different threads; each
 *     handle owns its CUDA stream and scratch memory.  Matcher entry points take a vsg_matcher
 *     workspace handle for the same reason (reference: stack-local ORBmatcher objects used from the
 *     Tracking / LocalMapping / LoopClosing threads).
 */
#ifndef VSG_CUDA_H
#define VSG_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int vsg_status;
#define VSG_OK 0
#define VSG_ERR_INVALID (-1)   /* bad argument */
#define VSG_ERR_CUDA (-2)      /* CUDA runtime error / no device */
#define VSG_ERR_CAPACITY (-3)  /* output buffer too small */
#define VSG_EMPTY_IMAGE (-10)  /* operator() on an empty image: the reference returns -1 (ORBextractor.cc:1087) */

/* Same memory layout as cv::KeyPoint (pt.x, pt.y, size, angle, response, octave, class_id; 28 bytes),
 * the element type of the vector operator() fills (ORBextractor.h:59-61). */
typedef struct vsg_keypoint {
    float x, y;
    float size;
    float angle;
    float response;
    int32_t octave;
    int32_t class_id;
} vsg_keypoint;

/* Constructor arguments of ORBextractor (ORBextractor.h:51-52, ORBextractor.cc:411-470). */
typedef struct vsg_orb_params {
    int32_t nfeatures;
    float scale_factor;
    int32_t nlevels;
    int32_t ini_th_fast;
    int32_t min_th_fast;
} vsg_orb_params;

typedef struct vsg_extractor vsg_extractor;
typedef struct vsg_matcher vsg_matcher;

const char *vsg_last_error(void);
/* Number of visible CUDA devices (0 if none / no driver). */
int vsg_device_count(void);
/* Kernel launches issued by this library since process start (bench.py's gpu_launches). */
int64_t vsg_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Extractor — replaces VS_GRAPHS::ORBextractor (orb_slam3/include/ORBextractor.h:42-119)
 * ---------------------------------------------------------------------------------------------- */

/* ORBextractor::ORBextractor (ORBextractor.cc:411-470).  `max_batch` = frames per vsg_extract_batch
 * call the handle must be able to hold (1 for the per-frame operator()).  The oct-tree keeps a level's nodes in shared
 * memory, which bounds every level's quota (features_per_level): on a B200 a quota of more than about 3,380 features does
 * not fit (nlevels = 1 with nfeatures = 3400, for one).  Such a handle is created, but every call that needs a frame size
 * fails with VSG_ERR_INVALID before anything is launched; vsg_last_error names the level, its quota and the bytes needed. */
vsg_status vsg_extractor_create(const vsg_orb_params *params, int device, int max_batch, vsg_extractor **out);
void vsg_extractor_destroy(vsg_extractor *ex);

/* GetScaleFactors / GetInverseScaleFactors / GetScaleSigmaSquares / GetInverseScaleSigmaSquares
 * (ORBextractor.h:73-91) and mnFeaturesPerLevel (ORBextractor.cc:435-446). Any pointer may be NULL. */
vsg_status vsg_extractor_tables(const vsg_extractor *ex, float *scale, float *inv_scale, float *sigma2,
                                float *inv_sigma2, int32_t *features_per_level);

/* Upper bound of keypoints operator() can return for one frame of this size (output buffer sizing). */
int vsg_extractor_max_keypoints(vsg_extractor *ex, int width, int height);

/* ORBextractor::operator()(image, mask, keypoints, descriptors, vLappingArea)
 * (ORBextractor.cc:1083-1169).  image: 8-bit gray, `pitch` bytes per row.  The mask is ignored by the
 * reference and has no parameter here.  keypoints_out / descriptors_out (n x 32) must hold `capacity`
 * entries.  *n_out = number of keypoints, *mono_index_out = the reference's return value
 * (count of keypoints outside [lap_x0, lap_x1]).  Returns VSG_EMPTY_IMAGE for a NULL/0-sized image. */
vsg_status vsg_extract(vsg_extractor *ex, const uint8_t *image, int width, int height, int pitch, int lap_x0,
                       int lap_x1, vsg_keypoint *keypoints_out, uint8_t *descriptors_out, int capacity, int *n_out,
                       int *mono_index_out);

/* Batched operator(): `nframes` (<= max_batch) frames of identical shape, frame f at
 * images + f*frame_stride.  Outputs are [nframes][capacity] arrays; n_out / mono_index_out are
 * [nframes].  This is what BASELINE configs 1 and 4 (sequence extraction) run. */
vsg_status vsg_extract_batch(vsg_extractor *ex, const uint8_t *images, int nframes, int width, int height, int pitch,
                             size_t frame_stride, int lap_x0, int lap_x1, vsg_keypoint *keypoints_out,
                             uint8_t *descriptors_out, int capacity, int *n_out, int *mono_index_out);

/* Batched operator() on interleaved 8-bit colour frames (`channels` = 3 or 4; r_first != 0: RGB / RGBA order, else
 * BGR / BGRA): the cv::cvtColor(..., COLOR_*2GRAY) that Tracking::GrabImage{RGBD,Monocular,Stereo} runs ahead of the
 * extractor (Tracking.cc:1526-1551, 1595-1608, 1646-1660) is done on the device, bit-exact with OpenCV's 8-bit path,
 * and the gray frames feed the same pipeline.  `pitch` is the byte pitch of a colour row. */
vsg_status vsg_extract_batch_color(vsg_extractor *ex, const uint8_t *images, int nframes, int width, int height, int pitch,
                                   size_t frame_stride, int channels, int r_first, int lap_x0, int lap_x1,
                                   vsg_keypoint *keypoints_out, uint8_t *descriptors_out, int capacity, int *n_out,
                                   int *mono_index_out);

/* Same, but the frames already live in device memory (frame f at images_dev + f*frame_stride; pitch
 * and base 16-byte aligned) and the results stay on the device: keypoints_dev / descriptors_dev /
 * n_dev / mono_dev are device pointers sized as above.  Asynchronous on the handle's stream; call
 * vsg_extractor_sync before reading.  Used for the HBM-resident throughput measurement. */
vsg_status vsg_extract_batch_dev(vsg_extractor *ex, const uint8_t *images_dev, int nframes, int width, int height,
                                 int pitch, size_t frame_stride, int lap_x0, int lap_x1, vsg_keypoint *keypoints_dev,
                                 uint8_t *descriptors_dev, int capacity, int32_t *n_dev, int32_t *mono_dev);
vsg_status vsg_extractor_sync(vsg_extractor *ex);
/* The handle's CUDA stream (cudaStream_t as void*), so callers can time with events on it. */
void *vsg_extractor_stream(vsg_extractor *ex);

/* Per-stage device timing (the reference's REGISTER_TIMES hooks, Frame.cc:126-153 / Settings.h:23, made
 * per kernel group): when enabled, CUDA events bracket each stage on the handle's stream.
 * vsg_extractor_stage_ms waits for the stream, returns the accumulated milliseconds per stage and the
 * number of pipeline runs they cover, and resets the accumulators.
 * Stages: 0 pyramid (7 resize launches), 1 FAST cells, 2 oct-tree, 3 Gaussian blur, 4 slots +
 * orientation + descriptors. */
#define VSG_NUM_STAGES 5
vsg_status vsg_extractor_profile(vsg_extractor *ex, int enable);
vsg_status vsg_extractor_stage_ms(vsg_extractor *ex, double *ms_out, int64_t *runs_out);

/* mvImagePyramid (ORBextractor.h:93; consumers Frame.cc:964,1054,1069): size of / copy of level
 * `level` of frame `frame` of the last call, w x h un-bordered pixels into dst with dst_pitch. */
vsg_status vsg_pyramid_level_size(vsg_extractor *ex, int level, int *width, int *height);
vsg_status vsg_pyramid_download(vsg_extractor *ex, int frame, int level, uint8_t *dst, int dst_pitch);
/* Test/diagnostic taps (parity tests compare them with the oracle stage by stage):
 * the blurred working image of a level (ORBextractor.cc:1129-1130), */
vsg_status vsg_blurred_download(vsg_extractor *ex, int frame, int level, uint8_t *dst, int dst_pitch);
/* the FAST candidates of a level in the reference's order, n x 3 int32 (x, y relative to the 16-px
 * border as in ORBextractor.cc:866-874, score), */
vsg_status vsg_candidates_download(vsg_extractor *ex, int frame, int level, int32_t *xys, int capacity, int *n_out);
/* and the per-level keypoints after the oct-tree in list order, n x 3 int32 (x, y level coords, score). */
vsg_status vsg_level_keypoints_download(vsg_extractor *ex, int frame, int level, int32_t *xys, int capacity,
                                        int *n_out);

/* ------------------------------------------------------------------------------------------------
 * Matcher — replaces the arithmetic of VS_GRAPHS::ORBmatcher (orb_slam3/include/ORBmatcher.h:34-99)
 * on flattened arrays.  Descriptors are rows of 32 bytes.
 * ---------------------------------------------------------------------------------------------- */
vsg_status vsg_matcher_create(int device, vsg_matcher **out);
void vsg_matcher_destroy(vsg_matcher *m);
void *vsg_matcher_stream(vsg_matcher *m);
vsg_status vsg_matcher_sync(vsg_matcher *m);

/* ORBmatcher::DescriptorDistance (ORBmatcher.cc:2047-2063) for n pairs: out[i] = |a_i xor b_i|. */
vsg_status vsg_descriptor_distance(vsg_matcher *m, const uint8_t *a, const uint8_t *b, int n, int32_t *out);

/* Brute-force Hamming kNN, k = 2 — cv::BFMatcher(NORM_HAMMING).knnMatch(q, t, 2) as used at
 * Frame.cc:1200 (ties: lower train index first).  out_idx / out_dist are [nq][2]; missing neighbours
 * (nt < 2) are idx -1, dist INT32_MAX.  train_index_offset is added to the reported indices (sharded
 * train sets). */
vsg_status vsg_knn2(vsg_matcher *m, const uint8_t *query, int nq, const uint8_t *train, int nt, int train_index_offset,
                    int32_t *out_idx, int32_t *out_dist);
vsg_status vsg_knn2_dev(vsg_matcher *m, const uint8_t *query_dev, int nq, const uint8_t *train_dev, int nt,
                        int train_index_offset, int32_t *out_idx_dev, int32_t *out_dist_dev);
/* Merge `nparts` per-shard top-2 lists ([nparts][nq][2]) into one ([nq][2]) by (dist, idx)
 * lexicographic order — the step after the all-gather when the train set is sharded over GPUs. */
vsg_status vsg_knn2_merge_dev(vsg_matcher *m, const int32_t *idx_parts_dev, const int32_t *dist_parts_dev, int nparts,
                              int nq, int32_t *out_idx_dev, int32_t *out_dist_dev);

/* MapPoint::ComputeDistinctiveDescriptors (MapPoint.cc:340-417) for `npoints` map points at once: point p's observed
 * descriptors are rows ptr[p] .. ptr[p+1]-1 of `descriptors` (in the reference's vDescriptors order).  best_out[p] =
 * the row (relative to ptr[p]) with the smallest median Hamming distance to the others (median = sorted row entry
 * 0.5*(N-1), first row wins ties), or -1 for a point without descriptors (the reference leaves mDescriptor alone). */
vsg_status vsg_distinctive_descriptors(vsg_matcher *m, const uint8_t *descriptors, const int32_t *ptr, int npoints,
                                       int32_t *best_out);

/* The descriptor part of Frame::ComputeStereoFishEyeMatches (Frame.cc:1200-1208): knnMatch(k = 2) and Lowe's ratio
 * test matches[0].distance < matches[1].distance * ratio (0.7 in the reference).  match_out[i] = train index or -1;
 * dist_out (may be NULL) = best distance.  The KannalaBrandt8 triangulation gate that follows stays with the caller. */
vsg_status vsg_knn2_ratio(vsg_matcher *m, const uint8_t *query, int nq, const uint8_t *train, int nt, float ratio,
                          int32_t *match_out, int32_t *dist_out);

/* Candidate-list ("windowed") search shared by the SearchByProjection family, SearchForInitialization,
 * Fuse and SearchBySim3: for each query i, scan its candidate train rows cand[cand_ptr[i]..cand_ptr[i+1])
 * in order and return the best and second-best distances with strict '<' updates (first candidate
 * wins ties), the best candidate's train index, and the `level` attribute of best / second-best
 * (ORBmatcher.cc:77-120).  skip[j] != 0 excludes train row j (already-matched keypoints,
 * ORBmatcher.cc:88-90); may be NULL.  train_level may be NULL (levels reported as -1).
 * init_dist is the reference's initial bestDist (256 or INT_MAX, SURVEY App. C#4). */
vsg_status vsg_match_window(vsg_matcher *m, const uint8_t *query, int nq, const uint8_t *train, int nt,
                            const int32_t *cand_ptr, const int32_t *cand, const uint8_t *skip,
                            const int32_t *train_level, int init_dist, int32_t *best_idx, int32_t *best_dist,
                            int32_t *second_dist, int32_t *best_level, int32_t *second_level);

/* ------------------------------------------------------------------------------------------------
 * Search* methods on flattened views (single-camera branches, Frame::Nleft == -1).
 * The GPU does what dominates the reference's cost — Frame::GetFeaturesInArea (grid window query,
 * Frame.cc:802-868) and the Hamming distance of every candidate — for all queries of a call at once and
 * returns per-query candidate lists in the reference's order; the order-dependent bookkeeping of each
 * method (first-come claims, vMatchedDistance stealing, rotation histogram) is then replayed by host
 * code inside the library exactly as the reference's loops do (SURVEY.md Appendix C#3).
 * ---------------------------------------------------------------------------------------------- */

/* What the Search* methods read from a Frame / KeyFrame (Frame.h:254-290,363-381). */
typedef struct vsg_frame_view {
    int32_t n;                     /* N */
    const vsg_keypoint *keys;      /* mvKeysUn (pt, octave, angle are read) */
    const uint8_t *descriptors;    /* mDescriptors, n x 32 */
    const float *u_right;          /* mvuRight, NULL for monocular */
    float min_x, min_y, max_x, max_y;      /* mnMinX, mnMinY, mnMaxX, mnMaxY */
    float grid_inv_w, grid_inv_h;  /* mfGridElementWidthInv / mfGridElementHeightInv */
    int32_t grid_cols, grid_rows;  /* FRAME_GRID_COLS / FRAME_GRID_ROWS (64 / 48, Frame.h:49-50) */
    const float *scale_factors;    /* mvScaleFactors */
    int32_t n_levels;
} vsg_frame_view;

/* MapPoint fields read by SearchByProjection(Frame&, vector<MapPoint*>&) (MapPoint.h:142-177). */
typedef struct vsg_track_point {
    float proj_x, proj_y, proj_xr; /* mTrackProjX, mTrackProjY, mTrackProjXR */
    float view_cos;                /* mTrackViewCos */
    float depth;                   /* mTrackDepth */
    int32_t level;                 /* mnTrackScaleLevel */
    uint8_t in_view;               /* mbTrackInView */
    uint8_t bad;                   /* isBad() */
    uint8_t blocks;                /* Observations() > 0 */
    uint8_t pad;
} vsg_track_point;

/* A last-frame map point already projected into the current frame by the caller (ORBmatcher.cc:1690-1716:
 * the pose / camera-model arithmetic stays with the reference's Sophus / GeometricCamera classes). */
typedef struct vsg_proj_point {
    float u, v;                    /* uv = pCamera->project(Tcw * x3Dw) */
    float ur;                      /* uv(0) - mbf * invzc */
    float angle;                   /* LastFrame.mvKeysUn[i].angle */
    int32_t octave;                /* LastFrame.mvKeys[i].octave */
    uint8_t valid;                 /* pMP && !mvbOutlier[i] && invzc >= 0 && uv inside [mnMinX,mnMaxX]x[mnMinY,mnMaxY] */
    uint8_t blocks;                /* pMP->Observations() > 0 */
    uint8_t pad[2];
} vsg_proj_point;

typedef struct vsg_frame vsg_frame;
/* Uploads a frame view and builds its keypoint grid (Frame::AssignFeaturesToGrid / PosInGrid,
 * Frame.cc:521-553,870-880).  The view's arrays are copied; the handle can serve many searches. */
vsg_status vsg_frame_create(vsg_matcher *m, const vsg_frame_view *view, vsg_frame **out);
/* Every entry point that takes a vsg_frame returns only after its kernels have finished (all of them are synchronous), so a
 * frame may be destroyed as soon as the last call using it has returned — from any thread, also after its matcher is gone. */
void vsg_frame_destroy(vsg_frame *f);

/* Frame::GetFeaturesInArea for nq windows at once (x, y, r, min_level, max_level per query): CSR lists of
 * keypoint indices in the reference's order plus their Hamming distance to qdesc (nq x 32).
 * cand_ptr has nq + 1 entries; cand_idx / cand_dist hold up to `capacity` entries (VSG_ERR_CAPACITY and
 * *total_out = needed size if more). */
vsg_status vsg_area_search(vsg_matcher *m, const vsg_frame *f, int nq, const float *qx, const float *qy,
                           const float *qr, const int32_t *min_level, const int32_t *max_level,
                           const uint8_t *qdesc, int32_t *cand_ptr, int32_t *cand_idx, int32_t *cand_dist,
                           int capacity, int *total_out);

/* SearchByProjection(Frame&, const vector<MapPoint*>&, th, bFarPoints, thFarPoints) (ORBmatcher.cc:42-144).
 * occupied[i] = F.mvpMapPoints[i] && F.mvpMapPoints[i]->Observations() > 0.  assign_out[i] = index of the map
 * point the reference writes to F.mvpMapPoints[i], or -1 if untouched.  *nmatches_out = return value. */
vsg_status vsg_search_by_projection_map(vsg_matcher *m, const vsg_frame *F, const uint8_t *occupied, int n_mp,
                                        const vsg_track_point *pts, const uint8_t *mp_desc, float th, int far_points,
                                        float th_far, float nnratio, int32_t *assign_out, int *nmatches_out);

/* The same method on a two-camera frame (F.Nleft != -1, the stereo-fisheye rigs; ORBmatcher.cc:42-216 with the
 * right-camera branch :146-213).  FL / FR are the two cameras' keypoints as separate frames (FL: mvKeys and rows
 * [0, Nleft) of mDescriptors, FR: mvKeysRight and rows [Nleft, N); no u_right).  occupied and assign_out have N = Nleft +
 * Nright entries in the reference's slot order (left slots first); left_to_right / right_to_left are
 * mvLeftToRightMatch / mvRightToLeftMatch (-1 = none).  pts_left[i] holds mbTrackInView, mTrackProjX/Y, mTrackViewCos,
 * mnTrackScaleLevel plus the shared mTrackDepth / isBad / Observations() > 0; pts_right[i] the R members
 * (mbTrackInViewR, mTrackProjXR/YR in proj_x / proj_y, mTrackViewCosR, mnTrackScaleLevelR, -1 allowed). */
vsg_status vsg_search_by_projection_map_2cam(vsg_matcher *m, const vsg_frame *FL, const vsg_frame *FR, const uint8_t *occupied,
                                             const int32_t *left_to_right, const int32_t *right_to_left, int n_mp,
                                             const vsg_track_point *pts_left, const vsg_track_point *pts_right,
                                             const uint8_t *mp_desc, float th, int far_points, float th_far, float nnratio,
                                             int32_t *assign_out, int *nmatches_out);

/* The same method in two halves, for map points sharded over GPUs (BASELINE config 3; SURVEY 8e): every rank runs
 * vsg_projection_map_candidates on its contiguous shard of the map points — the window query and the Hamming distance
 * of every candidate, in the reference's candidate order (cand_ptr has n_mp + 1 entries, VSG_ERR_CAPACITY and
 * *total_out = needed size if the lists do not fit) — the lists are all-gathered in shard order, and
 * vsg_projection_map_resolve replays the order-dependent part of the loop (:76-141: claimed keypoints are skipped by
 * later map points, best / second-best with their octaves, TH_HIGH and ratio gates) over all of them.  The resolve is
 * host code and needs no device. */
vsg_status vsg_projection_map_candidates(vsg_matcher *m, const vsg_frame *F, int n_mp, const vsg_track_point *pts,
                                         const uint8_t *mp_desc, float th, int far_points, float th_far,
                                         int32_t *cand_ptr, int32_t *cand_idx, int32_t *cand_dist, int capacity,
                                         int *total_out);
vsg_status vsg_projection_map_resolve(const vsg_frame_view *F, const uint8_t *occupied, int n_mp,
                                      const vsg_track_point *pts, const int32_t *cand_ptr, const int32_t *cand_idx,
                                      const int32_t *cand_dist, float nnratio, int32_t *assign_out, int *nmatches_out);

/* ---- multi-GPU: one process per GPU, NCCL over NVLink (SURVEY 8e; the reference is a single CPU process) ----
 * Only the two matcher paths with a real exchange step use a communicator; extraction shards by frame without one.
 * vsg_comm_unique_id() is called on one rank, its 128 bytes are handed to every rank by the host application (MPI,
 * torch.distributed, a file ...), and every rank calls vsg_comm_create with the same id.  NCCL is loaded at run time
 * ("libnccl.so.2"); without it these calls return VSG_ERR_CUDA and everything else keeps working. */
#define VSG_COMM_ID_BYTES 128
typedef struct vsg_comm vsg_comm;
vsg_status vsg_comm_unique_id(uint8_t id_out[VSG_COMM_ID_BYTES]);
vsg_status vsg_comm_create(const uint8_t id[VSG_COMM_ID_BYTES], int nranks, int rank, int device, vsg_comm **out);
void vsg_comm_destroy(vsg_comm *c);
int vsg_comm_rank(const vsg_comm *c);
int vsg_comm_size(const vsg_comm *c);
int vsg_comm_nccl_version(void);   /* e.g. 22809; 0 if NCCL cannot be loaded */

/* knnMatch(k = 2) with the TRAIN descriptors sharded over the ranks (BASELINE config 5): this rank holds nt_shard rows whose
 * global index starts at train_index_offset; queries are replicated.  Local search, ncclAllGather of the per-rank top-2
 * lists, (distance, index) merge on every rank: out_* equal vsg_knn2_dev on the concatenated train set.  Device pointers,
 * asynchronous on the matcher's stream. */
vsg_status vsg_knn2_sharded(vsg_comm *comm, vsg_matcher *m, const uint8_t *query_dev, int nq, const uint8_t *train_shard_dev,
                            int nt_shard, int train_index_offset, int32_t *out_idx_dev, int32_t *out_dist_dev);

/* vsg_search_by_projection_map with the MAP POINTS sharded over the ranks (BASELINE config 3): this rank holds the
 * contiguous shard [shard_begin, shard_begin + n_local) of vpMapPoints (records + descriptors); F and occupied are
 * replicated.  All ranks run the window search of their shard concurrently; the claim state (:88-90, :130) travels down the
 * ranks as an F->n-byte token (ncclSend / ncclRecv), each rank replays its shard from it, and one ncclAllGather of the
 * per-rank assignments gives every rank assign_out / nmatches_out identical to the one-call method on the whole map
 * (assign_out holds GLOBAL map point indices).  Host pointers; synchronous. */
vsg_status vsg_search_by_projection_map_sharded(vsg_comm *comm, vsg_matcher *m, const vsg_frame *F, const uint8_t *occupied,
                                                int shard_begin, int n_local, const vsg_track_point *pts_local,
                                                const uint8_t *desc_local, float th, int far_points, float th_far, float nnratio,
                                                int32_t *assign_out, int *nmatches_out);
/* Host-only building block of the sharded method (no device, no NCCL — for tests and for callers with their own
 * transport): replays ONE shard's candidate lists (vsg_projection_map_candidates on that shard) from the claim state
 * `blocked` (in / out, F->n bytes, initially `occupied`).  assign_out entries are overwritten with shard_begin + local index
 * where this shard assigns and left alone elsewhere; *nmatches_out = this shard's assignment events. */
vsg_status vsg_projection_map_resolve_shard(const vsg_frame_view *F, uint8_t *blocked, int shard_begin, int n_local,
                                            const vsg_track_point *pts_local, const int32_t *cand_ptr, const int32_t *cand_idx,
                                            const int32_t *cand_dist, float nnratio, int32_t *assign_out, int *nmatches_out);

/* SearchByProjection(Frame& Cur, const Frame& Last, th, bMono) (ORBmatcher.cc:1667-1878).  mode: 0 = octaves
 * [o-1, o+1], 1 = forward (>= o), 2 = backward ([0, o]) (:1719-1724).  assign_out[i] = index of the last-frame
 * point written to Cur.mvpMapPoints[i], -1 untouched, -2 written and then cleared by the rotation check. */
vsg_status vsg_search_by_projection_last(vsg_matcher *m, const vsg_frame *Cur, const uint8_t *occupied, int n_last,
                                         const vsg_proj_point *pts, const uint8_t *desc, float th, int mode,
                                         int check_ori, int32_t *assign_out, int *nmatches_out);

/* The same with a two-camera current frame (CurrentFrame.Nleft != -1; ORBmatcher.cc:1667-1878 incl. the right-camera
 * search :1785-1852).  CurL / CurR as in vsg_search_by_projection_map_2cam; occupied and assign_out have Nleft + Nright
 * slots.  pts_left[i] is the last-frame point projected with the left camera (valid, u, v, the last keypoint's angle and
 * octave, blocks); pts_right[i].u / .v its projection into the right camera (mpCamera->project(Trl * x3Dc)). */
vsg_status vsg_search_by_projection_last_2cam(vsg_matcher *m, const vsg_frame *CurL, const vsg_frame *CurR,
                                              const uint8_t *occupied, int n_last, const vsg_proj_point *pts_left,
                                              const vsg_proj_point *pts_right, const uint8_t *desc, float th, int mode,
                                              int check_ori, int32_t *assign_out, int *nmatches_out);

/* SearchForInitialization(F1, F2, vbPrevMatched, vnMatches12, windowSize) (ORBmatcher.cc:643-756).
 * prev_matched: F1.n x 2 floats, updated in place like vbPrevMatched.  matches12_out: F1.n entries. */
vsg_status vsg_search_for_initialization(vsg_matcher *m, const vsg_frame_view *F1, const vsg_frame *F2,
                                         float *prev_matched, int window_size, float nnratio, int check_ori,
                                         int32_t *matches12_out, int *nmatches_out);

/* SearchByBoW(KeyFrame*, Frame&, vector<MapPoint*>&) (ORBmatcher.cc:226-428).  DBoW2::FeatureVector
 * (std::map<NodeId, vector<unsigned>>) is passed as sorted node ids + CSR lists.  kf_mp_valid[i] = the
 * keyframe's map point i exists and is not bad.  matches_f_out[j] = keyframe feature matched to frame feature j
 * (the reference stores that feature's MapPoint*), or -1. */
vsg_status vsg_search_by_bow(vsg_matcher *m, const vsg_frame_view *KF, const uint8_t *kf_mp_valid,
                             const vsg_frame_view *F, int kf_nnodes, const int32_t *kf_nodes, const int32_t *kf_ptr,
                             const int32_t *kf_idx, int f_nnodes, const int32_t *f_nodes, const int32_t *f_ptr,
                             const int32_t *f_idx, float nnratio, int check_ori, int32_t *matches_f_out,
                             int *nmatches_out);

/* The same with a two-camera frame (F.Nleft = f_nleft != -1; ORBmatcher.cc:298-322, :362-390): F (and KF, if it has a
 * second camera) list the left camera's keypoints / descriptor rows first, then the right camera's, as mDescriptors does;
 * best and second-best are kept per camera.  f_nleft == -1 is vsg_search_by_bow.  Both run vsg_search_by_bow_multi with one
 * target and share its argument rules; vsg_last_error names a rejected argument.  A view with n > 0 needs both its keys
 * and its descriptors, also when check_ori == 0. */
vsg_status vsg_search_by_bow_2cam(vsg_matcher *m, const vsg_frame_view *KF, const uint8_t *kf_mp_valid,
                                  const vsg_frame_view *F, int f_nleft, int kf_nnodes, const int32_t *kf_nodes,
                                  const int32_t *kf_ptr, const int32_t *kf_idx, int f_nnodes, const int32_t *f_nodes,
                                  const int32_t *f_ptr, const int32_t *f_idx, float nnratio, int check_ori,
                                  int32_t *matches_f_out, int *nmatches_out);

/* One side of a BoW search: a frame or keyframe view, its map-point flags (mp_valid[i] = map point i present and not bad;
 * not read for the frame of vsg_search_by_bow_multi) and its DBoW2::FeatureVector as the node ids / CSR lists the
 * single-target calls take. */
typedef struct vsg_bow_side {
    vsg_frame_view view;
    const uint8_t *mp_valid;
    int32_t nnodes;
    const int32_t *nodes, *ptr, *idx;
} vsg_bow_side;

/* Tracking::Relocalization's loop `for (i : candidates) matcher.SearchByBoW(pKF_i, mCurrentFrame, vvpMapPointMatches[i])`
 * (Tracking.cc:3687-3854) in one call: for every t < ntargets, vsg_search_by_bow_2cam(m, &KFs[t]->view, KFs[t]->mp_valid,
 * &F->view, f_nleft, <KFs[t]'s feature vector>, <F's feature vector>, nnratio, check_ori, matches_f_out + t * F->view.n,
 * &nmatches_out[t]), with one upload, one kernel launch (none if no target shares a node with F) and one download.  F is
 * shared by all targets; the same keyframe may appear more than once.  ntargets == 0 does nothing.  A null or malformed
 * target, or a feature index out of range, returns VSG_ERR_INVALID before anything is launched, and vsg_last_error names
 * the target. */
vsg_status vsg_search_by_bow_multi(vsg_matcher *m, int ntargets, const vsg_bow_side *const *KFs, const vsg_bow_side *F,
                                   int f_nleft, float nnratio, int check_ori, int32_t *matches_f_out, int *nmatches_out);

/* A map point already projected into the searched Frame / KeyFrame by the caller: the pose, Sim3 and
 * camera-model arithmetic ahead of GetFeaturesInArea (e.g. ORBmatcher.cc:444-486, 1182-1238, 1904-1929) stays
 * with the reference's Sophus / GeometricCamera classes; everything from the window query on runs here. */
typedef struct vsg_search_point {
    float u, v;                    /* uv = project(Tcw * p3Dw) */
    float ur;                      /* uv(0) - bf * invz (Fuse's stereo reprojection gate; unused elsewhere) */
    float angle;                   /* pKF->mvKeysUn[i].angle of the source observation (rotation histogram) */
    int32_t level;                 /* nPredictedLevel = pMP->PredictScale(dist, pKF) */
    uint8_t valid;                 /* the point passed every gate ahead of GetFeaturesInArea */
    uint8_t pad[3];
} vsg_search_point;

/* SearchByProjection(Frame& Cur, KeyFrame*, const set<MapPoint*>& sAlreadyFound, th, ORBdist)
 * (ORBmatcher.cc:1880-2000, relocalisation).  pts[i] = map point i of the keyframe (valid = present, not bad,
 * not already found, projection inside the frame, depth inside the scale-invariance range).
 * occupied[j] = Cur.mvpMapPoints[j] != NULL.  assign_out as in vsg_search_by_projection_last. */
vsg_status vsg_search_by_projection_reloc(vsg_matcher *m, const vsg_frame *Cur, const uint8_t *occupied, int n,
                                          const vsg_search_point *pts, const uint8_t *desc, float th, int orb_dist,
                                          int check_ori, int32_t *assign_out, int *nmatches_out);

/* SearchByProjection(KeyFrame*, Sim3f& Scw, vpPoints, vpMatched, th, ratioHamming) and the vpPointsKFs overload
 * (ORBmatcher.cc:430-528, 530-641; loop closing / merging).  matched[j] = vpMatched[j] != NULL on entry.
 * assign_out[j] = index of the point written to vpMatched[j] (and vpMatchedKF[j]), -1 untouched. */
vsg_status vsg_search_by_projection_sim3(vsg_matcher *m, const vsg_frame *KF, const uint8_t *matched, int n,
                                         const vsg_search_point *pts, const uint8_t *desc, int th,
                                         float ratio_hamming, int32_t *assign_out, int *nmatches_out);

/* The search of ORBmatcher::Fuse(KeyFrame*, vpMapPoints, th, bRight) (ORBmatcher.cc:1148-1335, variant 0: chi2
 * reprojection gates 5.99 / 7.8 against inv_level_sigma2 = pKF->mvInvLevelSigma2, initial distance 256) and of
 * Fuse(KeyFrame*, Sim3f&, vpPoints, th, vpReplacePoint) (:1337-1446, variant 1: no gate, initial INT_MAX).
 * best_idx_out[i] = the keyframe feature the reference picks for point i (bestDist <= TH_LOW), else -1.  The
 * search of a point does not depend on the map-point bookkeeping of earlier points, so the caller applies
 * Replace / AddObservation / AddMapPoint in order afterwards, re-checking isBad() / IsInKeyFrame() as the
 * reference does at the top of each iteration.  *nfused_out counts the entries >= 0.  Variant 0 is
 * vsg_fuse_search_multi with one target, variant 1 the same search without the gates; both share its argument rules,
 * so KF must live on the matcher's device. */
vsg_status vsg_fuse_search(vsg_matcher *m, const vsg_frame *KF, int n, const vsg_search_point *pts,
                           const uint8_t *desc, float th, const float *inv_level_sigma2, int variant,
                           int32_t *best_idx_out, int *nfused_out);

/* The searches of LocalMapping::SearchInNeighbors' loop `for (pKFi : vpTargetKFs) matcher.Fuse(pKFi, vpMapPointMatches)`
 * (LocalMapping.cc:764-802) in one call: vsg_fuse_search(m, KFs[t], n, pts + t * n, desc, th, inv_level_sigma2[t], 0,
 * best_idx_out + t * n, NULL) for every t < ntargets, with one upload, one kernel launch and one download whatever
 * ntargets is.  pts and best_idx_out are [ntargets][n] (point i projected into target t with that target's pose and
 * camera); desc (n x 32) is shared by all targets.  The two cameras of a two-camera keyframe are two targets.  Every
 * target must live on the matcher's device.  The caller replays the bookkeeping target by target; a map point whose
 * descriptor changes during that replay (MapPoint::Replace recomputes the survivor's) must be searched again in the
 * later targets. */
vsg_status vsg_fuse_search_multi(vsg_matcher *m, int ntargets, const vsg_frame *const *KFs,
                                 const float *const *inv_level_sigma2, int n, const vsg_search_point *pts,
                                 const uint8_t *desc, float th, int32_t *best_idx_out);

/* The searches of LoopClosing::SearchAndFuse's loop `for (pKFi, Scw : CorrectedPosesMap) matcher.Fuse(pKFi, Scw, vpMapPoints,
 * 4, vpReplacePoints)` (LoopClosing.cc:1994-2054; loop correction and map merging) in one call: vsg_fuse_search(m, KFs[t], n,
 * pts + t * n, desc, th, NULL, 1, best_idx_out + t * n, NULL) for every t < ntargets, with one upload, one kernel launch and
 * one download whatever ntargets is (none if ntargets or n is 0).  pts and best_idx_out are [ntargets][n] (point i projected
 * into target t with that target's Scw and camera); desc (n x 32) is shared by all targets.  The same keyframe may appear
 * more than once.  Argument rules as vsg_fuse_search_multi without the level tables: negative counts, a null target and a
 * target on another device than the matcher's are rejected with VSG_ERR_INVALID before anything is launched, and
 * vsg_last_error names the target.  The caller replays the bookkeeping target by target; a map point whose descriptor
 * changes during that replay (MapPoint::Replace recomputes the survivor's) must be searched again in the later targets. */
vsg_status vsg_fuse_search_sim3_multi(vsg_matcher *m, int ntargets, const vsg_frame *const *KFs, int n,
                                      const vsg_search_point *pts, const uint8_t *desc, float th, int32_t *best_idx_out);

/* SearchBySim3(pKF1, pKF2, vpMatches12, S12, th) (ORBmatcher.cc:1448-1665).  pts1[i1] (KF1.n entries): map point
 * i1 of KF1 projected into KF2 (valid = present, not already matched, not bad, depth/image/distance gates);
 * pts2[i2] likewise into KF1.  matches12_out[i1] = i2 where both directions agree, else -1. */
vsg_status vsg_search_by_sim3(vsg_matcher *m, const vsg_frame *KF1, const vsg_frame *KF2, int n1,
                              const vsg_search_point *pts1, const uint8_t *desc1, int n2,
                              const vsg_search_point *pts2, const uint8_t *desc2, float th, int32_t *matches12_out,
                              int *nfound_out);

/* SearchByBoW(KeyFrame* pKF1, KeyFrame* pKF2, vpMatches12) (ORBmatcher.cc:758-900).  mp_valid1/2[i] = map point
 * present and not bad.  matches12_out[i1] = i2 (the reference stores vpMapPoints2[i2]) or -1.  vsg_search_by_bow_kf_multi
 * with one target: the same argument rules (a view with n > 0 needs both its keys and its descriptors). */
vsg_status vsg_search_by_bow_kf(vsg_matcher *m, const vsg_frame_view *KF1, const uint8_t *mp_valid1,
                                const vsg_frame_view *KF2, const uint8_t *mp_valid2, int nnodes1,
                                const int32_t *nodes1, const int32_t *ptr1, const int32_t *idx1, int nnodes2,
                                const int32_t *nodes2, const int32_t *ptr2, const int32_t *idx2, float nnratio,
                                int check_ori, int32_t *matches12_out, int *nmatches_out);

/* LoopClosing::DetectCommonRegionsFromBoW's loop `for (j : vpCovKFi) matcherBoW.SearchByBoW(mpCurrentKF, vpCovKFi[j],
 * vvpMatchedMPs[j])` (LoopClosing.cc:573-642) in one call: for every t < ntargets, vsg_search_by_bow_kf(m, &KF1->view,
 * KF1->mp_valid, &KF2s[t]->view, KF2s[t]->mp_valid, <KF1's feature vector>, <KF2s[t]'s feature vector>, nnratio, check_ori,
 * matches12_out + t * KF1->view.n, &nmatches_out[t]), with one upload, one kernel launch (none if no target shares a node with
 * KF1) and one download.  KF1 is shared by all targets.  Argument rules as vsg_search_by_bow_multi. */
vsg_status vsg_search_by_bow_kf_multi(vsg_matcher *m, const vsg_bow_side *KF1, int ntargets, const vsg_bow_side *const *KF2s,
                                      float nnratio, int check_ori, int32_t *matches12_out, int *nmatches_out);

/* The Hamming-distance half of the BoW-guided pairings, for callers that own the per-pair geometry test — two-camera
 * SearchForTriangulation (ORBmatcher.cc:902-1146 with mpCamera2 != NULL), where the epipolar test is the caller's
 * KannalaBrandt8 camera code.  The merge walk over the two feature vectors (:966-1118): for every feature i1 of KF1 with
 * use1[i1] != 0 inside a vocabulary node both vectors share, ALL features of that node in KF2, in the reference's scan
 * order, with their descriptor distances.  q1_out[k] = i1 (walk order), its candidates are
 * cand_idx2_out / cand_dist_out[cand_ptr_out[k] .. cand_ptr_out[k + 1]).  VSG_ERR_CAPACITY with *nq_out / *total_out = the
 * needed sizes when q_capacity (+ 1 for cand_ptr_out) or capacity is too small. */
vsg_status vsg_bow_pair_distances(vsg_matcher *m, const vsg_frame_view *KF1, const uint8_t *use1, const vsg_frame_view *KF2,
                                  int nnodes1, const int32_t *nodes1, const int32_t *ptr1, const int32_t *idx1, int nnodes2,
                                  const int32_t *nodes2, const int32_t *ptr2, const int32_t *idx2, int32_t *q1_out,
                                  int32_t *cand_ptr_out, int q_capacity, int32_t *cand_idx2_out, int32_t *cand_dist_out,
                                  int capacity, int *nq_out, int *total_out);

/* SearchForTriangulation(pKF1, pKF2, vMatchedPairs, bOnlyStereo, bCoarse) (ORBmatcher.cc:902-1146), single
 * pinhole camera per keyframe (mpCamera2 == NULL).  has_mp1/2[i] = GetMapPoint(i) != NULL.  f12 = the
 * fundamental matrix of Pinhole::epipolarConstrain (Pinhole.cpp:118-141), row-major; ep = epipole of KF1 in KF2
 * (:914).  level_sigma2_2 = pKF2->mvLevelSigma2.  matches12_out[i1] = i2 or -1 (vMatchedPairs = the pairs with
 * i2 >= 0 in increasing i1).  vsg_triangulation_candidates_multi with one target, then vsg_triangulation_resolve: the
 * same argument rules (a keypoint octave of KF2 outside [0, n_levels) is rejected). */
vsg_status vsg_search_for_triangulation(vsg_matcher *m, const vsg_frame_view *KF1, const uint8_t *has_mp1,
                                        const vsg_frame_view *KF2, const uint8_t *has_mp2, int nnodes1,
                                        const int32_t *nodes1, const int32_t *ptr1, const int32_t *idx1, int nnodes2,
                                        const int32_t *nodes2, const int32_t *ptr2, const int32_t *idx2,
                                        int only_stereo, int coarse, const float *f12, const float *ep,
                                        const float *level_sigma2_2, int check_ori, int32_t *matches12_out,
                                        int *nmatches_out);

/* One neighbour of LocalMapping::CreateNewMapPoints' loop (LocalMapping.cc:406,460): keyframe 2 of
 * SearchForTriangulation, single pinhole camera.  kf2.mp_valid[i] = pKF2->GetMapPoint(i) != NULL (bad points included,
 * ORBmatcher.cc:998-1001).  f12 / ep as in vsg_search_for_triangulation; level_sigma2 = pKF2->mvLevelSigma2
 * (kf2.view.n_levels entries; may be NULL when the call is coarse). */
typedef struct vsg_triangulation_target {
    vsg_bow_side kf2;
    float f12[9];
    float ep[2];
    const float *level_sigma2;
} vsg_triangulation_target;

/* The searches of every target at once: best12_out is [ntargets][KF1->view.n].  KF1->mp_valid[i] = pKF1->GetMapPoint(i)
 * != NULL at this call.  best12_out[t][i1] = the keyframe-2 feature the reference's inner loop picks for i1 in target t,
 * -1 if none, -2 if i1 was not searched because it had a map point.  One upload, at most one launch, one download.
 * ntargets == 0 does nothing.  A null target, a malformed feature vector, a feature index out of range, a KF1 feature
 * listed twice in its feature vector, a null level_sigma2 when !coarse or a target keypoint octave outside [0, n_levels)
 * returns VSG_ERR_INVALID before anything is launched, and vsg_last_error names the target. */
vsg_status vsg_triangulation_candidates_multi(vsg_matcher *m, const vsg_bow_side *KF1, int ntargets,
                                              const vsg_triangulation_target *const *targets, int only_stereo, int coarse,
                                              int32_t *best12_out);

/* Host only, no device: SearchForTriangulation's result for one target from its row of best12, with KF1's map points as
 * they are NOW (has_mp1).  Equal to vsg_search_for_triangulation(KF1, has_mp1, KF2, …) as long as KF1 has gained, never
 * lost, map points since the candidates call.  A feature that is -2 and has no map point now returns
 * VSG_ERR_INVALID, naming the feature. */
vsg_status vsg_triangulation_resolve(const vsg_frame_view *KF1, const vsg_frame_view *KF2, const uint8_t *has_mp1,
                                     const int32_t *best12, int check_ori, int32_t *matches12_out, int *nmatches_out);

/* ------------------------------------------------------------------------------------------------
 * BoW transform — the per-feature tree walk of DBoW2::TemplatedVocabulary::transform as called by Frame::ComputeBoW /
 * KeyFrame::ComputeBoW (Frame.cc:882-889, KeyFrame.cc:99-108 -> Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1139-1265).
 * The vocabulary tree is uploaded once, flattened: node 0 is the root, the children of node i are
 * child_idx[child_ptr[i] .. child_ptr[i+1]) in the order of m_nodes[i].children (ties go to the first child), leaves
 * have no children; node_descriptors is nnodes x 32 bytes (the root's row is unused); levels = m_L.
 * vsg_bow_transform returns, per descriptor, the leaf reached (the caller maps it to word_id / weight from its own
 * vocabulary object) and the node passed at level m_L - levelsup (the FeatureVector node; 0 = root when that level is
 * <= 0 or the leaf is reached earlier).  BowVector::addWeight, FeatureVector::addFeature and the L1 normalisation are
 * O(N) double-precision bookkeeping in feature order and stay with the caller (INTEGRATION.md shows the loop).
 * ---------------------------------------------------------------------------------------------- */
typedef struct vsg_vocabulary vsg_vocabulary;
vsg_status vsg_vocabulary_create(vsg_matcher *m, int nnodes, const int32_t *child_ptr, const int32_t *child_idx,
                                 const uint8_t *node_descriptors, int levels, vsg_vocabulary **out);
void vsg_vocabulary_destroy(vsg_vocabulary *v);
vsg_status vsg_bow_transform(vsg_matcher *m, const vsg_vocabulary *voc, const uint8_t *descriptors, int n, int levelsup,
                             int32_t *leaf_node_out, int32_t *feature_node_out);

/* Frame::ComputeStereoMatches (Frame.cc:957-1127): for every left keypoint the best right keypoint in its row
 * band (octave +-1, uR in [uL - mbf/mb, uL], Hamming < TH_HIGH), then — if the distance is below
 * (TH_HIGH+TH_LOW)/2 — an 11x11 L1 patch correlation over 11 horizontal offsets on the un-blurred pyramid
 * level of both extractors, parabola sub-pixel fit, disparity gate and the final 1.5*1.4*median rejection.
 * `left` / `right` are the two extractor handles whose last call produced keys_l / keys_r (the device pyramids
 * of that call are read in place; frame_l / frame_r select the frame of a batched call).  u_right_out and
 * depth_out are mvuRight / mvDepth (n_l entries, -1 = no match). */
vsg_status vsg_stereo_match(vsg_matcher *m, vsg_extractor *left, vsg_extractor *right, int frame_l, int frame_r,
                            const vsg_keypoint *keys_l, const uint8_t *desc_l, int n_l, const vsg_keypoint *keys_r,
                            const uint8_t *desc_r, int n_r, float mb, float mbf, float *u_right_out, float *depth_out);

/* Batched ComputeStereoMatches: frames 2p / 2p+1 of the extractor's last vsg_extract_batch[_color] call are the left /
 * right image of stereo pair p (BASELINE config 2; SURVEY 8e: both images of a pair on one GPU).  Keypoints,
 * descriptors and pyramids are read where that call left them in device memory — nothing is uploaded — and the
 * median-based rejection (:1113-1126) runs on the device too.  u_right_out / depth_out are [npairs][capacity] floats
 * (capacity >= vsg_extractor_max_keypoints); entries beyond a pair's left keypoint count are -1. */
vsg_status vsg_stereo_match_batch(vsg_matcher *m, vsg_extractor *ex, int npairs, float mb, float mbf,
                                  float *u_right_out, float *depth_out, int capacity);

/* Rectification ahead of the extractor: System::TrackStereo / TrackMonocular run cv::remap(im, imToFeed, M1, M2,
 * cv::INTER_LINEAR) on every incoming image when the settings ask for it (System.cc:284-292; float maps from
 * cv::initUndistortRectifyMap, Settings.cc:571-574 — BASELINE config 2's EuRoC.yaml does).
 * vsg_extractor_set_rectify_map stores the CV_32FC1 map pair of camera `slot` (0 = left / only camera, 1 = right) in
 * OpenCV's 1/32-pixel fixed-point form on the device; width x height is the size of the rectified image (newImSize).
 * vsg_extract_batch_rectify is vsg_extract_batch on unrectified gray frames of src_width x src_height pixels: frame f is
 * remapped with the map of camera f % ncameras (ncameras = 2: left / right images interleaved, as
 * vsg_stereo_match_batch expects them) on the device, bit-exact with OpenCV's 8-bit remap (BORDER_CONSTANT, 0), and
 * extracted at the maps' size. */
vsg_status vsg_extractor_set_rectify_map(vsg_extractor *ex, int slot, const float *map_x, const float *map_y, int width,
                                         int height);
vsg_status vsg_extract_batch_rectify(vsg_extractor *ex, const uint8_t *images, int nframes, int src_width, int src_height,
                                     int pitch, size_t frame_stride, int ncameras, int lap_x0, int lap_x1,
                                     vsg_keypoint *keypoints_out, uint8_t *descriptors_out, int capacity, int *n_out,
                                     int *mono_index_out);

/* ---- per-keypoint steps of Frame's constructors right after the extractor (SURVEY 8f rank 3) ---- */

/* Frame::UndistortKeyPoints (Frame.cc:891-922) and the corner call of Frame::ComputeImageBounds (:924-955):
 * cv::undistortPoints(xy, xy, mK, mDistCoef, cv::Mat(), mK) on n (x, y) float pairs.  fx, fy, cx, cy are mK's entries and
 * dist the dist_n (0, 4, 5, 8 or 12) entries of mDistCoef (k1 k2 p1 p2 [k3 [k4 k5 k6 [s1 s2 s3 s4]]]) widened to double
 * as OpenCV does.  dist_n == 0 or dist[0] == 0 copies the input, the reference's own shortcut (:893-897).  Results are
 * bit-identical to OpenCV's (double arithmetic, five iterations).  xy_out may alias xy_in. */
vsg_status vsg_undistort_keypoints(vsg_matcher *m, int n, const float *xy_in, double fx, double fy, double cx, double cy,
                                   const double *dist, int dist_n, float *xy_out);

/* The same for the keypoints of the first nframes frames of the extractor's last vsg_extract_batch[_color] call, read where
 * that call left them in device memory: xy_out is [nframes][capacity][2] floats (capacity >=
 * vsg_extractor_max_keypoints); rows past a frame's keypoint count are (-1, -1). */
vsg_status vsg_undistort_keypoints_batch(vsg_matcher *m, vsg_extractor *ex, int nframes, double fx, double fy, double cx,
                                         double cy, const double *dist, int dist_n, float *xy_out, int capacity);

#ifdef __cplusplus
}
#endif
#endif /* VSG_CUDA_H */
