// match_internal.cuh — declarations shared by match_methods.cu and match_methods_kf.cu (not part of the ABI).
#pragma once
#include <string>
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

struct Chi2Gate {            // inverse level variances for the reprojection gates of the pose-based Fuse (:1273-1299)
    float inv_sigma2[kMaxLevels];
};

struct FuseTarget {          // one keyframe of a multi-target Fuse search: its grid / features and its level variances
    FrameDev f;
    Chi2Gate gate;
};

// Candidate lists as the kernel left them: query q's (idx, dist) pairs are raw[off[q] .. off[q] + cnt[q]) (segments in
// arbitrary order).  The arrays live in the matcher's pinned staging and stay valid until its next area search.
struct AreaLists {
    const int2 *raw = nullptr;
    const int *off = nullptr, *cnt = nullptr;
};


// Runs the area search (Frame::GetFeaturesInArea + Hamming distance, area_search_kernel) for nq queries and brings
// the lists back: ptr[nq+1] and (idx, dist) pairs in query order, each list in the reference's candidate order.
// n_qdesc rows of qdesc are uploaded (queries pick theirs by desc_idx).
vsg_status area_search(vsg_matcher *m, const vsg_frame *f, int nq, const AreaQuery *qs, const uint8_t *qdesc, int n_qdesc,
                       std::vector<int> &ptr, std::vector<int2> &ent);
// Best candidate per query on the device, over the queries of one or several frames at once (one copy in, one launch, one
// copy out): the whole search of the methods whose queries are independent of one another.  Query k searches
// frames[q_target[k]] with descriptor row qs[k].desc_idx of qdesc (n_qdesc rows), through the window / level gates and, unless
// inv_sigma2 is nullptr, the chi-square gates with inv_sigma2[q_target[k]].  out[k] = (index or -1, distance or INT_MAX).
vsg_status area_best_multi(vsg_matcher *m, int ntargets, const vsg_frame *const *frames, const float *const *inv_sigma2, int nq,
                           const AreaQuery *qs, const int *q_target, int n_qdesc, const uint8_t *qdesc, std::vector<int2> &out);
// area_search without the re-pack into query order
vsg_status area_search_raw(vsg_matcher *m, const vsg_frame *f, int nq, const AreaQuery *qs, const uint8_t *qdesc,
                           int n_qdesc, AreaLists *out);
// The nearest candidate of the list [c, ce) whose keypoint is not taken, first one on ties: (distance, index), or (256, -1).
inline int2 nearest_unclaimed(const int2 *c, const int2 *ce, const uint8_t *taken) {
    int best = 256, best_idx = -1;
    for (; c < ce; ++c) {
        if (taken[c->x]) continue;
        if (c->y < best) { best = c->y; best_idx = c->x; }
    }
    return make_int2(best, best_idx);
}
inline size_t up16(size_t x) { return (x + 15) & ~(size_t)15; }
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
// Host tables laid out back to back in one upload, each distinct one once (a frame shared by all walks, a keyframe passed
// twice): place() returns the first element of (p, n), appending it if it is not there yet.
struct TablePlacer {
    struct Table { const void *p; int n, first; };
    std::vector<Table> tabs;
    int total = 0;
    int place(const void *p, int n) {
        for (const Table &t : tabs)
            if (t.p == p && t.n == n) return t.first;
        tabs.push_back(Table{p, n, total});
        total += n;
        return tabs.back().first;
    }
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
// The target loop of the multi-target BoW calls: problem(t) says what is wrong with target t (nullptr: nothing), and
// only once every target has passed is walk(t) walked for each; walk t's segments are appended as segs[seg_ptr[t] ..
// seg_ptr[t + 1]).  Both kinds of error read "<who>: target t: <what>".
template <class Problem, class Walk>
vsg_status bow_walk_targets(const char *who, int ntargets, Problem problem, Walk walk, std::vector<BowWalk> &walks,
                            std::vector<BowSeg> &segs, std::vector<int> &seg_ptr, int64_t *npairs) {
    for (int t = 0; t < ntargets; ++t)
        if (const char *why = problem(t)) {
            set_error("%s: target %d: %s", who, t, why);
            return VSG_ERR_INVALID;
        }
    seg_ptr.assign(1, 0);
    for (int t = 0; t < ntargets; ++t) {
        walks.push_back(walk(t));
        if (bow_walk(walks.back(), segs, npairs) != VSG_OK) {
            const std::string err = vsg_last_error();
            set_error("%s: target %d: %s", who, t, err.c_str());
            return VSG_ERR_INVALID;
        }
        seg_ptr.push_back((int)segs.size());
    }
    return VSG_OK;
}
// ORBmatcher::ComputeThreeMaxima (ORBmatcher.cc:2002-2043)
void three_maxima(const std::vector<int> *hist, int L, int &ind1, int &ind2, int &ind3);
// The rotation-consistency filter (ORBmatcher.cc:2002-2043 and its callers): every entry outside the three dominant bins of
// the histogram goes to drop(), which undoes that caller's match.
template <class Drop>
void apply_rot_filter(const std::vector<int> *rot_hist, Drop drop) {
    int ind1 = -1, ind2 = -1, ind3 = -1;
    three_maxima(rot_hist, HISTO_LENGTH, ind1, ind2, ind3);
    for (int i = 0; i < HISTO_LENGTH; ++i) {
        if (i == ind1 || i == ind2 || i == ind3) continue;
        for (int idx : rot_hist[i]) drop(idx);
    }
}
// rotation-histogram bin (ORBmatcher.cc:351-358)
int rot_bin(float a1, float a2);

}  // namespace vsg
