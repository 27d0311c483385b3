// match_internal.cuh — declarations shared by match_methods.cu and match_methods_kf.cu (not part of the ABI).
#pragma once
#include <vector>

#include "vsg_internal.cuh"

struct vsg_frame {
    int device = 0;        // the frame may outlive the matcher that uploaded it
    int n = 0, cols = 0, rows = 0, n_levels = 0;
    float min_x = 0, min_y = 0, inv_w = 0, inv_h = 0;
    bool has_right = false;
    // device: one stream-ordered allocation (`block`), carved into the arrays below
    void *block = nullptr;
    float2 *xy = nullptr;
    int *octave = nullptr;
    float *u_right = nullptr;
    uint8_t *desc = nullptr;
    int *cell_ptr = nullptr, *cell_idx = nullptr;
    // host copies the resolve loops read
    std::vector<vsg_keypoint> keys;
    std::vector<float> scale;
    std::vector<float> u_right_h;   // mvuRight (empty if monocular)
};

namespace vsg {

#ifndef CK
#endif

constexpr int TH_HIGH = 100, TH_LOW = 50, HISTO_LENGTH = 30;   // ORBmatcher.cc:34-36

struct FrameDev {
    int n, cols, rows;
    float min_x, min_y, inv_w, inv_h;
    const float2 *xy;
    const int *octave;
    const float *u_right;   // nullptr if monocular
    const uint4 *desc;
    const int *cell_ptr, *cell_idx;
};

struct AreaQuery {          // one GetFeaturesInArea call + the per-candidate stereo gate of the caller
    float x, y, r;
    int min_level, max_level;
    float xr, rr;           // right-image gate: skip if u_right[idx] > 0 && |xr - u_right[idx]| > rr; rr < 0 disables it
    int max_dist = 256;     // candidates farther than this are not listed: the caller proved they cannot change its result
    int desc_idx = -1;      // row of the uploaded query descriptors (-1: the query's own index)
};

// Candidate lists as the kernel left them: query q's (idx, dist) pairs are raw[off[q] .. off[q] + cnt[q]) (segments in
// arbitrary order).  The arrays live in the matcher's pinned staging and stay valid until its next search.
struct Chi2Gate {            // inverse level variances for the reprojection gates of the pose-based Fuse (:1273-1299)
    float inv_sigma2[kMaxLevels];
};

struct FuseTarget {          // one keyframe of a multi-target Fuse search: its grid / features and its level variances
    FrameDev f;
    Chi2Gate gate;
};

struct AreaLists {
    const int2 *raw = nullptr;
    const int *off = nullptr, *cnt = nullptr;
};


// Runs the area search (Frame::GetFeaturesInArea + Hamming distance, area_search_kernel) for nq queries and brings
// the lists back: ptr[nq+1] and (idx, dist) pairs in query order, each list in the reference's candidate order.
vsg_status area_search(vsg_matcher *m, const vsg_frame *f, int nq, const AreaQuery *qs, const uint8_t *qdesc,
                       std::vector<int> &ptr, std::vector<int2> &ent);
// the same without the re-pack into query order; n_qdesc rows of qdesc are uploaded (queries pick theirs by desc_idx)
// Best candidate per query on the device (window / level gates, optional chi-square gates when inv_sigma2 != nullptr): the
// whole search of the methods whose queries are independent of one another.  out[k] = (index or -1, distance or INT_MAX).
vsg_status area_best(vsg_matcher *m, const vsg_frame *f, int nq, const AreaQuery *qs, const uint8_t *qdesc, const float *inv_sigma2,
                     std::vector<int2> &out);
// area_best with the chi-square gates over the queries of several frames at once (one copy in, one launch, one copy out):
// query k searches frames[q_target[k]] with inv_sigma2[q_target[k]] and descriptor row qs[k].desc_idx of qdesc (n_qdesc rows).
vsg_status area_best_multi(vsg_matcher *m, int ntargets, const vsg_frame *const *frames, const float *const *inv_sigma2, int nq,
                           const AreaQuery *qs, const int *q_target, int n_qdesc, const uint8_t *qdesc, std::vector<int2> &out);
vsg_status area_search_raw(vsg_matcher *m, const vsg_frame *f, int nq, const AreaQuery *qs, const uint8_t *qdesc,
                           int n_qdesc, AreaLists *out);
// ---- BoW-guided pairings (SearchByBoW x 2, SearchForTriangulation; match_methods_kf.cu) ----
struct FeatVec {             // a flattened DBoW2::FeatureVector: node ids ascending, node k's features idx[ptr[k] .. ptr[k+1])
    int nnodes;
    const int32_t *nodes, *ptr, *idx;
};
// One merge walk over two FeatureVectors (e.g. ORBmatcher.cc:785-872): every feature i1 of side 1 with use1[i1] != 0 inside
// a node both vectors share is a query whose candidates are ALL features of that node on side 2.
struct BowWalk {
    const vsg_frame_view *v1;
    const uint8_t *use1;
    FeatVec a;
    const vsg_frame_view *v2;
    FeatVec b;
};
// A query of a walk: feature i1 of side 1, its candidates b.idx[jb .. je) in the reference's scan order, their distances
// dist[off .. off + je - jb).
struct BowSeg {
    int i1, jb, je, off;
};
bool featvec_ok(int nn, const int32_t *nodes, const int32_t *ptr, const int32_t *idx);
// Appends the queries of one walk to segs, output slots continuing from *npairs; rejects feature indices out of range.
vsg_status bow_walk(const BowWalk &w, std::vector<BowSeg> &segs, int64_t *npairs);
// The distances of every in-node pair of the walks: one copy in (segments, every distinct descriptor table once, every
// distinct side-2 idx array once), one launch of bow_dists_multi_kernel (none if npairs == 0), one copy out.  segs[seg_ptr[k]
// .. seg_ptr[k+1]) are walk k's.  *dist points into the matcher's pinned staging and stays valid until its next BoW call.
vsg_status bow_dists(vsg_matcher *m, int nwalks, const BowWalk *walks, const std::vector<BowSeg> &segs, const int *seg_ptr,
                     int64_t npairs, const uint16_t **dist);
// What is wrong with one side of a multi-target BoW call (nullptr: nothing); the map-point flags only if it needs them.
const char *bow_side_problem(const vsg_bow_side *s, bool needs_valid);
// ORBmatcher::ComputeThreeMaxima (ORBmatcher.cc:2002-2043)
void three_maxima(const std::vector<int> *hist, int L, int &ind1, int &ind2, int &ind3);
// rotation-histogram bin (ORBmatcher.cc:351-358)
int rot_bin(float a1, float a2);

}  // namespace vsg
