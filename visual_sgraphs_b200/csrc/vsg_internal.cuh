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

// Matcher workspace: a stream plus scratch buffers that grow on demand (defined here so that match.cu and
// match_methods.cu share it).
struct vsg_matcher {
    int device = 0;
    cudaStream_t stream = nullptr;
    void *buf[20] = {};      // device scratch slots; each entry point documents the slots it owns
    size_t cap[20] = {};
    void *hbuf[9] = {};      // pinned host staging (grows on demand): results come back without page faults
    size_t hcap[9] = {};
    std::vector<char> scratch[2];   // reusable host scratch of the search methods (query lists), kept across calls
    int sm_count = 148;
};

namespace vsg {

vsg_status matcher_ensure(vsg_matcher *m, int slot, size_t bytes);
vsg_status matcher_ensure_host(vsg_matcher *m, int slot, size_t bytes);
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
