// vsg_internal.cuh — shared declarations of libvsg_cuda.so (not part of the public ABI).
//
// Geometry notes (reference orb_slam3/src/ORBextractor.cc):
//   EDGE_THRESHOLD = 19 (:71): FAST runs on [16, dim-16) (:795-798), keypoints live in [19, dim-19).
//   Device pyramid planes carry NO 19-px reflected border: nothing on the path reads it
//   (SURVEY App. A3); the shim re-creates it on the host when it materialises mvImagePyramid.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "../../include/vsg_cuda.h"

namespace vsg {

constexpr int kMaxLevels = 16;
constexpr int kEdge = 19;        // EDGE_THRESHOLD
constexpr int kBorderMin = 16;   // minBorderX/Y = EDGE_THRESHOLD - 3
constexpr int kMaxImageDim = 16384;   // packed 15/16-bit pixel coordinates (oct-tree midpoints, candidates, resize tables)
constexpr int kHalfPatch = 15;   // HALF_PATCH_SIZE
constexpr int kPatch = 31;       // PATCH_SIZE

// One pyramid level of the current image shape.
struct LevelGeom {
    int w, h;              // level size (cvRound(dim * invScale), :1176)
    int pitch;             // device row pitch in bytes (multiple of 16)
    int64_t plane_stride;  // bytes between consecutive frames of this level
    int64_t plane_offset;  // offset of frame 0 inside the pyramid / blurred buffers
    // cell grid of ComputeKeyPointsOctTree (:795-809)
    int n_cols, n_rows, w_cell, h_cell;
    int cell_begin, cell_count;  // slice of the flat cell table
    int cols_eff, rows_eff;      // the cells that survive the skip rules (:816,825) form this prefix rectangle
    uint32_t cols_rcp;           // ceil(2^32 / cols_eff): cell row = umulhi(cell index, cols_rcp)
    uint32_t wcell_rcp, hcell_rcp;   // ceil(2^32 / w_cell), ceil(2^32 / h_cell): exact quotients for coordinates below 2^16
    // oct-tree
    int quota;             // mnFeaturesPerLevel[level]
    int n_ini;             // round(width/height) root nodes (:566)
    float h_x;             // root width (:568)
    int cand_cap;          // candidate slots per frame
    int64_t cand_offset;   // first candidate slot of frame 0 (in elements); frame stride = cand_total
    int kp_cap;            // selected-keypoint slots per frame
    int kp_offset;         // first slot of this level inside a frame's level-keypoint array
    float scale;           // mvScaleFactor[level]
    float kp_size;         // (float)(int)(PATCH_SIZE * scale) (:884)
    // resize tables (device pointers) for building this level from the previous one
    int resize_tma_ok;     // every 128 x 32 tile's source window fits resize_tma_kernel's box (resize_tma.cu)
    const short4 *xtab;    // per dst x: {sx0, sx1, a0, a1}
    const short4 *ytab;    // per dst y: {sy0, sy1, b0, b1}
};

struct FrameGeom {
    int nlevels;
    int ncells;            // total cells over all levels
    int64_t cand_total;    // candidate slots per frame (all levels)
    int kp_total;          // selected keypoint slots per frame (all levels)
    int out_cap;           // output keypoint capacity per frame (== kp_total)
    LevelGeom lv[kMaxLevels];
};

// One FAST cell: the sub-image the reference hands to cv::FAST (:811-851).
struct Cell {
    short level;
    short x0, y0;          // window origin in level coordinates (iniX, iniY)
    short cw, ch;          // window size (maxX-iniX, maxY-iniY), includes FAST's 3-px rim
    short pad;
};

// FAST candidate as stored on the device: level coordinates, absolute.
struct __align__(8) Cand {
    unsigned short x, y;
    unsigned short score;  // cv::FAST response (K-1)
    unsigned short pad;
};

struct __align__(8) LevelKp {
    unsigned short x, y;   // level coordinates (already + minBorder)
    unsigned short score;
    unsigned short pad;
};

}  // namespace vsg

namespace vsg {

// Device scratch slots of a matcher (vsg_matcher::buf).  A slot's contents are only valid inside the call that wrote them
// unless its line says otherwise; a function must not call another user of a slot while it still needs that slot's contents.
enum DevSlot : int {
    kSlotKnnParts = 0,     // knn2_device (match.cu): per-chunk top-2 partials
    kSlotArg1,             // one-shot inputs: query descriptors (vsg_descriptor_distance, vsg_knn2, vsg_match_window), left
                           // keypoints (stereo.cu), descriptors (mappoint.cu, bow.cu)
    kSlotArg2,             // train descriptors (match.cu), left descriptors (stereo.cu)
    kSlotArg3,             // distances / indices (match.cu), right keypoints (stereo.cu), list offsets (mappoint.cu)
    kSlotArg4,             // distances / candidates (match.cu), right descriptors (stereo.cu)
    kSlotArg5,             // vsg_match_window: train levels and skip flags
    kSlotOut,              // one-shot results (vsg_match_window, stereo.cu, mappoint.cu, bow.cu), undistort input (frame_ops.cu);
                           // area_search_ordered: the entries in query order
    kSlotAreaQueries,      // area_search_raw / _ordered: the queries; second one-shot result (frame_ops.cu, stereo.cu)
    kSlotAreaQdesc,        // area_search_raw / _ordered: the query descriptors
    kSlotAreaCounts,       // area_search_raw / _ordered: per-query offset and count, the total
    kSlotAreaRaw,          // area_search_raw / _ordered: the entries as the kernel writes them (its size carries over as the
                           // next search's first capacity)
    kSlotAreaOrder,        // area_search_ordered: list pointers and the query of every entry
    kSlotMapShardToken,    // vsg_search_by_projection_map_sharded: claim token and per-rank records
    kSlotKnnSharded,       // vsg_knn2_sharded: own and gathered top-2 lists
    kSlotTcQuery,          // knn2_tc_device (knn_tc.cu): expanded query descriptors
    kSlotTcTrain,          // knn2_tc_device: expanded train descriptors
    kSlotTcParts,          // knn2_tc_device: per-segment top-2 partials
    kSlotBestMultiIn,      // area_best_multi: targets, queries and descriptors
    kSlotBestMultiOut,     // area_best_multi: the results
    kSlotBow,              // bow_dists, triangulation_candidates (match_methods_kf.cu): inputs, then results
    kNumDevSlots
};

// Pinned host staging slots of a matcher (vsg_matcher::hbuf): results come back without page faults.  Same rule as DevSlot.
enum HostSlot : int {
    kHostAreaCounts = 0,   // area_search_raw: offsets, counts and total (AreaLists::off / cnt); area_search_ordered: list
                           // pointers (OrderedLists::ptr) — both valid until the next area search
    kHostAreaEnt,          // area_search_raw / _ordered: the entries (AreaLists::raw, OrderedLists::ent), valid until the next
                           // area search
    kHostFrameStaging,     // vsg_frame_create: the frame's arrays on their way to the device
    kHostMapQueries,       // projection_map_search: the map points' window queries
    kHostAreaQid,          // area_search_ordered: the query of every entry (OrderedLists::qid), valid until the next area search
    kHostBestMultiOut,     // area_best_multi: the results
    kHostMapShardToken,    // vsg_search_by_projection_map_sharded: claim token and per-rank records
    kHostBestMultiIn,      // area_best_multi: targets, queries and descriptors
    kHostBow,              // bow_dists: inputs, then the distances (valid until the next BoW call); triangulation_candidates
    kNumHostSlots
};

}  // namespace vsg

// Matcher workspace: a stream plus scratch buffers that grow on demand (defined here so that match.cu and
// match_methods.cu share it).
struct vsg_matcher {
    int device = 0;
    cudaStream_t stream = nullptr;
    void *buf[vsg::kNumDevSlots] = {};
    size_t cap[vsg::kNumDevSlots] = {};
    void *hbuf[vsg::kNumHostSlots] = {};
    size_t hcap[vsg::kNumHostSlots] = {};
    std::vector<int> scratch;   // projection_map_search: query -> map point (MapSearch::q_mp), valid until the next map search
    int sm_count = 148;
};

namespace vsg {

vsg_status matcher_ensure(vsg_matcher *m, DevSlot slot, size_t bytes);
vsg_status matcher_ensure_host(vsg_matcher *m, HostSlot slot, size_t bytes);
// merge of `nparts` per-shard / per-segment top-2 lists ([nparts][nq][2]) by (distance, index) on the matcher's stream
vsg_status launch_knn2_merge_parts(vsg_matcher *m, const int32_t *idx_parts, const int32_t *dist_parts, int nparts, int nq,
                                   int32_t *out_idx, int32_t *out_dist);
// tensor-core kNN-2 (knn_tc.cu): tcgen05.mma.kind::i8 on +-1 expanded descriptors; results identical to the POPC kernel
bool knn2_tc_supported(int nq, int nt);
vsg_status knn2_tc_device(vsg_matcher *m, const uint8_t *q_dev, int nq, const uint8_t *t_dev, int nt, int offset, int *idx_dev,
                          int *dist_dev);
// bow_dists_multi_kernel (match.cu): out[segs[s].w + k] = |desc[segs[s].x] xor desc[segs[s].z + idx[segs[s].y + k]]| for the
// k-th candidate of segment s; segs holds nseg segments sorted by .w, the last one a sentinel with .w = npairs
void launch_bow_dists(vsg_matcher *m, const int4 *segs_dev, int nseg, const int *idx_dev, const uint8_t *desc_dev, int npairs,
                      uint16_t *out_dev);
// triangulation_best_kernel (match.cu): SearchForTriangulation's inner loop (ORBmatcher.cc:998-1077, pinhole) for every
// segment of every target of a call.  A segment is one (target, KF1 feature) query of a BoW merge walk; its candidates are
// idx[cand .. cand + ncand) (target-local feature indices, the reference's scan order).
struct TriSeg {
    float x1, y1;            // KF1 keypoint
    int q_row;               // KF1 descriptor row in the uploaded descriptor tables
    int cand, ncand;
    int target;
    int stereo1;             // KF1->u_right && KF1->u_right[i1] >= 0
    int pad;
};
struct TriTarget {
    float f12[9], ep[2];
    int desc0;               // first descriptor row of the target
    int key0;                // first TriKey of the target
    int lvl0;                // first level entry of the target
    int pad[2];
};
struct TriKey {
    float x, y;
    int octave;              // validated on the host: inside [0, n_levels)
    int flags;               // kTriStereo | kTriHasMp
};
constexpr int kTriStereo = 1, kTriHasMp = 2;
// out[s] = the target feature the reference ends with as bestIdx2 for segment s, or -1.  lvl[lvl0 + octave] = (scale factor,
// level sigma^2).  Nothing is launched when nseg == 0.
void launch_triangulation_best(vsg_matcher *m, const TriSeg *segs_dev, int nseg, const TriTarget *targets_dev, const int *idx_dev,
                               const uint8_t *desc_dev, const TriKey *keys_dev, const float2 *lvl_dev, int only_stereo, int coarse,
                               int *out_dev);

// Read-only view of an extractor's device pyramid of its last call (for the stereo matcher).
struct PyramidRef {
    int device;
    int nframes;
    const FrameGeom *geom;
    const uint8_t *lvl0_base;
    int lvl0_pitch;
    int64_t lvl0_stride;
    const uint8_t *pyr;
    const float *scale, *inv_scale;   // host tables, nlevels entries
    cudaStream_t stream;
    // device-resident results of the last host-pointer batch call (null after a device-resident call)
    const vsg_keypoint *kps_dev;
    const uint8_t *desc_dev;
    const int *n_dev;
    int out_cap;
};
bool extractor_pyramid(vsg_extractor *ex, PyramidRef *out);

// Programmatic dependent launch (sm_90+): a kernel launched with the attribute may be scheduled while the previous
// kernel of the stream is still draining; it must execute pdl_wait() before touching anything that kernel wrote.
// Every pipeline kernel calls pdl_launch_dependents() first thing (the next kernel's blocks can be made resident as
// soon as all of this kernel's blocks have started) and pdl_wait() ahead of its first dependent access; both are no-ops
// for ordinary launches.  Only batches of up to 8 frames are launched with the attribute (vsg_api.cu: pdl_enabled).
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
bool pdl_enabled();
void pdl_scope(int nframes);   // run_pipeline: decides per batch size (thread-local)

template <class... KArgs, class... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl,
                                 Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (pdl && pdl_enabled()) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

void set_error(const char *fmt, ...);
bool cuda_ok(cudaError_t e, const char *what);
// In functions returning vsg_status: record the CUDA error text (vsg_last_error) and return VSG_ERR_CUDA.
#define CK(call)                                          \
    do {                                                  \
        if (!cuda_ok((call), #call)) return VSG_ERR_CUDA; \
    } while (0)
void count_launch(int n = 1);

// --- kernel launchers (each file documents the reference lines it implements) ---
// pyramid_tile_kernel (pyramid.cu): the whole pyramid of a few frames in ONE launch.  A tile owns a box of every level (the
// boxes of a level partition its plane) and computes, level by level in shared memory, the slightly larger region the next
// level's region needs; both boxes are inclusive and come from the host, which built the resize tables.
struct PyrTileBox { short x0, y0, x1, y1; };
struct PyrTile {
    PyrTileBox region[kMaxLevels], owned[kMaxLevels];
    uint32_t rcp_w[kMaxLevels];      // ceil(2^32 / region width): pixel index -> row by multiply-high
};
void launch_pyramid_tiles(const FrameGeom &g, const PyrTile *tiles, int ntiles, int buf_bytes, size_t smem, const uint8_t *lvl0_base,
                          int lvl0_pitch, int64_t lvl0_stride, uint8_t *pyr, int nframes, cudaStream_t s);
bool launch_resize_level_tma(const FrameGeom &g, int level, const uint8_t *src_base, int src_pitch, int64_t src_stride, uint8_t *pyr,
                             int nframes, cudaStream_t s);
bool resize_tma_fits(const std::vector<short4> &xt, const std::vector<short4> &yt, int dw, int dh);
void launch_resize_level(const FrameGeom &g, int level, const uint8_t *src_base, int src_pitch, int64_t src_stride,
                         uint8_t *pyr, int nframes, cudaStream_t s);
// cv::cvtColor(..., COLOR_{RGB,BGR,RGBA,BGRA}2GRAY) of `nframes` device frames into 8-bit planes (src 4-byte aligned)
void launch_cvt_gray(const uint8_t *src, int src_pitch, int64_t src_stride, int channels, int r_first, uint8_t *dst,
                     int dst_pitch, int64_t dst_stride, int w, int h, int nframes, cudaStream_t s);
// Quantised rectification maps of up to two cameras (frame f of a batch uses slot f % nslots): per output pixel the
// integer source position (x | y << 16, two shorts) and the 1/32-pixel fraction (fy * 32 + fx).
struct RectifyMaps {
    const uint32_t *xy[2];
    const uint16_t *frac[2];
    int nslots;
};
void launch_remap(const uint8_t *src, int src_pitch, int64_t src_stride, int sw, int sh, const RectifyMaps &maps, int first_frame,
                  uint8_t *dst, int dst_pitch, int64_t dst_stride, int w, int h, int nframes, cudaStream_t s);
// blur_tc.cu: the blur as banded u8 GEMMs on the tensor cores; plan == nullptr: not applicable (use launch_blur)
struct BlurTcPlan;
const BlurTcPlan *plan_blur_tc(const FrameGeom &g, const uint8_t *lvl0_base, int lvl0_pitch, int64_t lvl0_stride, const uint8_t *pyr,
                               const uint8_t *blur, int nframes);
void launch_blur_tc(const BlurTcPlan *plan, uint8_t *blur, cudaStream_t s);
void launch_blur(const FrameGeom &g, const uint8_t *lvl0_base, int lvl0_pitch, int64_t lvl0_stride, const uint8_t *pyr,
                 uint8_t *blur, int nframes, cudaStream_t s);
// blur != nullptr: the Gaussian blur of the same frames runs inside the same grid (fast_blur_kernel)
vsg_status launch_fast(const FrameGeom &g, const uint8_t *lvl0_base, int lvl0_pitch, int64_t lvl0_stride, const uint8_t *pyr,
                       uint8_t *blur, Cand *cand, int *cand_count, int ini_th, int min_th, int max_cw, int max_ch, int nframes,
                       cudaStream_t s);
// octree_kernel keeps its node lists in shared memory: octree_smem_bytes(max_nodes) dynamic bytes per block, plus the
// kernel's static arrays (octree_static_smem_bytes).  Their sum must fit the device's per-block opt-in limit, so the level
// quotas a handle accepts are bounded (configure_shape checks this before anything is allocated or launched).
size_t octree_smem_bytes(int max_nodes);
vsg_status octree_static_smem_bytes(size_t *bytes);
vsg_status launch_octree(const FrameGeom &g, const Cand *cand, const int *cand_count, unsigned short *node_of,
                         LevelKp *level_kps, int *level_kp_count, int max_nodes, int nframes, cudaStream_t s);
void launch_describe(const FrameGeom &g, const uint8_t *lvl0_base, int lvl0_pitch, int64_t lvl0_stride,
                     const uint8_t *pyr, const uint8_t *blur, const LevelKp *level_kps, const int *level_kp_count,
                     int lap_x0, int lap_x1, vsg_keypoint *kps_out, uint8_t *desc_out, int out_cap, int *n_out,
                     int *mono_out, int *slot_scratch, int nframes, cudaStream_t s);

}  // namespace vsg
