// vsg_on_oracle.cpp — TEST ADAPTER: the matcher entry points of include/vsg_cuda.h implemented on the CPU oracle
// (oracle/oracle.h).  It exists so that the drop-in shim's host code (visual_sgraphs_b200/shim/ORBmatcher.h: flattening,
// pose arithmetic, write-back, Replace / AddObservation replay) can be run WITHOUT a GPU against the reference's own
// ORBmatcher.cc (tests/cpp/ref_matcher_test.cpp, CPU build).  Never linked into the product: libvsg_cuda.so has no CPU path.
#include <cstring>
#include <string>
#include <vector>

#include "../../include/vsg_cuda.h"
#include "../../oracle/oracle.h"

static_assert(sizeof(vsg_frame_view) == sizeof(orc_frame_view), "view layout");
static_assert(sizeof(vsg_track_point) == sizeof(orc_track_point), "track point layout");
static_assert(sizeof(vsg_proj_point) == sizeof(orc_proj_point), "proj point layout");
static_assert(sizeof(vsg_search_point) == sizeof(orc_search_point), "search point layout");
static_assert(sizeof(vsg_keypoint) == sizeof(orc_keypoint), "keypoint layout");

struct vsg_matcher { int dummy; };
struct vsg_frame {   // deep copy of the view
    std::vector<orc_keypoint> keys;
    std::vector<uint8_t> desc;
    std::vector<float> u_right, scale;
    orc_frame_view v;
};

static const orc_frame_view *V(const vsg_frame_view *v) { return reinterpret_cast<const orc_frame_view *>(v); }
static const orc_frame_view *V(const vsg_frame *f) { return &f->v; }

extern "C" {

const char *vsg_last_error(void) { return "vsg_on_oracle adapter"; }
vsg_status vsg_matcher_create(int, vsg_matcher **out) { *out = new vsg_matcher{0}; return VSG_OK; }
void vsg_matcher_destroy(vsg_matcher *m) { delete m; }

// knnMatch(k = 2): (distance, index) lexicographic top-2, missing neighbours idx -1 / dist INT32_MAX (include/vsg_cuda.h)
vsg_status vsg_knn2(vsg_matcher *, const uint8_t *query, int nq, const uint8_t *train, int nt, int offset, int32_t *out_idx, int32_t *out_dist) {
    for (int q = 0; q < nq; ++q) {
        int b0 = 0x7fffffff, b1 = 0x7fffffff, i0 = -1, i1 = -1;
        for (int t = 0; t < nt; ++t) {
            const int d = orc_descriptor_distance(query + (size_t)q * 32, train + (size_t)t * 32);
            if (d < b0) { b1 = b0; i1 = i0; b0 = d; i0 = t; }
            else if (d < b1) { b1 = d; i1 = t; }
        }
        out_idx[2 * q] = i0 >= 0 ? i0 + offset : -1; out_dist[2 * q] = b0;
        out_idx[2 * q + 1] = i1 >= 0 ? i1 + offset : -1; out_dist[2 * q + 1] = b1;
    }
    return VSG_OK;
}
vsg_status vsg_undistort_keypoints(vsg_matcher *, int n, const float *xy_in, double fx, double fy, double cx, double cy, const double *dist,
                                   int dist_n, float *xy_out) {
    orc_undistort_points(n, xy_in, fx, fy, cx, cy, dist, dist_n, xy_out);
    return VSG_OK;
}

vsg_status vsg_frame_create(vsg_matcher *, const vsg_frame_view *view, vsg_frame **out) {
    vsg_frame *f = new vsg_frame;
    const orc_frame_view *s = V(view);
    f->keys.assign(s->keys, s->keys + s->n);
    f->desc.assign(s->descriptors, s->descriptors + (size_t)s->n * 32);
    if (s->u_right) f->u_right.assign(s->u_right, s->u_right + s->n);
    f->scale.assign(s->scale_factors, s->scale_factors + s->n_levels);
    f->v = *s;
    f->v.keys = f->keys.data();
    f->v.descriptors = f->desc.data();
    f->v.u_right = s->u_right ? f->u_right.data() : nullptr;
    f->v.scale_factors = f->scale.data();
    *out = f;
    return VSG_OK;
}
void vsg_frame_destroy(vsg_frame *f) { delete f; }

vsg_status vsg_search_by_projection_map(vsg_matcher *, const vsg_frame *F, const uint8_t *occupied, int n_mp, const vsg_track_point *pts,
                                        const uint8_t *mp_desc, float th, int far_points, float th_far, float nnratio,
                                        int32_t *assign_out, int *nmatches_out) {
    *nmatches_out = orc_search_by_projection_map(V(F), occupied, n_mp, reinterpret_cast<const orc_track_point *>(pts), mp_desc, th,
                                                 far_points, th_far, nnratio, assign_out);
    return VSG_OK;
}
vsg_status vsg_search_by_projection_map_2cam(vsg_matcher *, const vsg_frame *FL, const vsg_frame *FR, const uint8_t *occupied,
                                             const int32_t *l2r, const int32_t *r2l, int n_mp, const vsg_track_point *pl,
                                             const vsg_track_point *pr, const uint8_t *mp_desc, float th, int far_points, float th_far,
                                             float nnratio, int32_t *assign_out, int *nmatches_out) {
    *nmatches_out = orc_search_by_projection_map_2cam(V(FL), V(FR), occupied, l2r, r2l, n_mp, reinterpret_cast<const orc_track_point *>(pl),
                                                      reinterpret_cast<const orc_track_point *>(pr), mp_desc, th, far_points, th_far,
                                                      nnratio, assign_out);
    return VSG_OK;
}
vsg_status vsg_search_by_projection_last(vsg_matcher *, const vsg_frame *Cur, const uint8_t *occupied, int n_last, const vsg_proj_point *pts,
                                         const uint8_t *desc, float th, int mode, int check_ori, int32_t *assign_out, int *nmatches_out) {
    *nmatches_out = orc_search_by_projection_last(V(Cur), occupied, n_last, reinterpret_cast<const orc_proj_point *>(pts), desc, th, mode,
                                                  check_ori, assign_out);
    return VSG_OK;
}
vsg_status vsg_search_by_projection_last_2cam(vsg_matcher *, const vsg_frame *CurL, const vsg_frame *CurR, const uint8_t *occupied,
                                              int n_last, const vsg_proj_point *pl, const vsg_proj_point *pr, const uint8_t *desc, float th,
                                              int mode, int check_ori, int32_t *assign_out, int *nmatches_out) {
    *nmatches_out = orc_search_by_projection_last_2cam(V(CurL), V(CurR), occupied, n_last, reinterpret_cast<const orc_proj_point *>(pl),
                                                       reinterpret_cast<const orc_proj_point *>(pr), desc, th, mode, check_ori, assign_out);
    return VSG_OK;
}
vsg_status vsg_search_for_initialization(vsg_matcher *, const vsg_frame_view *F1, const vsg_frame *F2, float *prev_matched, int window_size,
                                         float nnratio, int check_ori, int32_t *matches12_out, int *nmatches_out) {
    *nmatches_out = orc_search_for_initialization(V(F1), V(F2), prev_matched, window_size, nnratio, check_ori, matches12_out);
    return VSG_OK;
}
vsg_status vsg_search_by_bow_multi(vsg_matcher *, int ntargets, const vsg_bow_side *const *KFs, const vsg_bow_side *F, int f_nleft,
                                   float nnratio, int check_ori, int32_t *matches_f_out, int *nmatches_out) {
    for (int t = 0; t < ntargets; ++t) {
        const vsg_bow_side &a = *KFs[t];
        nmatches_out[t] = orc_search_by_bow_2cam(V(&a.view), a.mp_valid, V(&F->view), f_nleft, a.nnodes, a.nodes, a.ptr, a.idx, F->nnodes,
                                                 F->nodes, F->ptr, F->idx, nnratio, check_ori, matches_f_out + (size_t)t * F->view.n);
    }
    return VSG_OK;
}
vsg_status vsg_search_by_projection_reloc(vsg_matcher *, const vsg_frame *Cur, const uint8_t *occupied, int n, const vsg_search_point *pts,
                                          const uint8_t *desc, float th, int orb_dist, int check_ori, int32_t *assign_out,
                                          int *nmatches_out) {
    *nmatches_out = orc_search_by_projection_reloc(V(Cur), occupied, n, reinterpret_cast<const orc_search_point *>(pts), desc, th, orb_dist,
                                                   check_ori, assign_out);
    return VSG_OK;
}
vsg_status vsg_search_by_projection_sim3(vsg_matcher *, const vsg_frame *KF, const uint8_t *matched, int n, const vsg_search_point *pts,
                                         const uint8_t *desc, int th, float ratio_hamming, int32_t *assign_out, int *nmatches_out) {
    *nmatches_out = orc_search_by_projection_sim3(V(KF), matched, n, reinterpret_cast<const orc_search_point *>(pts), desc, th, ratio_hamming,
                                                  assign_out);
    return VSG_OK;
}
vsg_status vsg_fuse_search(vsg_matcher *, const vsg_frame *KF, int n, const vsg_search_point *pts, const uint8_t *desc, float th,
                           const float *inv_level_sigma2, int variant, int32_t *best_idx_out, int *nfused_out) {
    const int nf = orc_fuse_search(V(KF), n, reinterpret_cast<const orc_search_point *>(pts), desc, th, inv_level_sigma2, variant, best_idx_out);
    if (nfused_out) *nfused_out = nf;
    return VSG_OK;
}
vsg_status vsg_fuse_search_multi(vsg_matcher *, int ntargets, const vsg_frame *const *KFs, const float *const *inv_level_sigma2, int n,
                                 const vsg_search_point *pts, const uint8_t *desc, float th, int32_t *best_idx_out) {
    for (int t = 0; t < ntargets; ++t)
        orc_fuse_search(V(KFs[t]), n, reinterpret_cast<const orc_search_point *>(pts) + (size_t)t * n, desc, th, inv_level_sigma2[t], 0,
                        best_idx_out + (size_t)t * n);
    return VSG_OK;
}
vsg_status vsg_search_by_sim3(vsg_matcher *, const vsg_frame *KF1, const vsg_frame *KF2, int n1, const vsg_search_point *pts1, const uint8_t *desc1,
                              int n2, const vsg_search_point *pts2, const uint8_t *desc2, float th, int32_t *matches12_out, int *nfound_out) {
    *nfound_out = orc_search_by_sim3_n(V(KF1), V(KF2), n1, reinterpret_cast<const orc_search_point *>(pts1), desc1, n2,
                                       reinterpret_cast<const orc_search_point *>(pts2), desc2, th, matches12_out);
    return VSG_OK;
}
vsg_status vsg_search_by_bow_kf_multi(vsg_matcher *, const vsg_bow_side *KF1, int ntargets, const vsg_bow_side *const *KF2s, float nnratio,
                                      int check_ori, int32_t *matches12_out, int *nmatches_out) {
    for (int t = 0; t < ntargets; ++t) {
        const vsg_bow_side &b = *KF2s[t];
        nmatches_out[t] = orc_search_by_bow_kf(V(&KF1->view), KF1->mp_valid, V(&b.view), b.mp_valid, KF1->nnodes, KF1->nodes, KF1->ptr,
                                               KF1->idx, b.nnodes, b.nodes, b.ptr, b.idx, nnratio, check_ori,
                                               matches12_out + (size_t)t * KF1->view.n);
    }
    return VSG_OK;
}
vsg_status vsg_bow_pair_distances(vsg_matcher *, const vsg_frame_view *KF1, const uint8_t *use1, const vsg_frame_view *KF2, int nn1,
                                  const int32_t *nodes1, const int32_t *ptr1, const int32_t *idx1, int nn2, const int32_t *nodes2,
                                  const int32_t *ptr2, const int32_t *idx2, int32_t *q1_out, int32_t *cand_ptr_out, int q_capacity,
                                  int32_t *cand_idx2_out, int32_t *cand_dist_out, int capacity, int *nq_out, int *total_out) {
    std::vector<int> q1, cptr(1, 0), cand, dist;
    int ia = 0, ib = 0;
    while (ia < nn1 && ib < nn2) {                 // the merge walk of two DBoW2::FeatureVectors (ORBmatcher.cc:961-1118)
        if (nodes1[ia] == nodes2[ib]) {
            for (int k = ptr1[ia]; k < ptr1[ia + 1]; ++k) {
                const int i1 = idx1[k];
                if (!use1[i1]) continue;
                q1.push_back(i1);
                for (int j = ptr2[ib]; j < ptr2[ib + 1]; ++j) {
                    cand.push_back(idx2[j]);
                    dist.push_back(orc_descriptor_distance(KF1->descriptors + (size_t)i1 * 32, KF2->descriptors + (size_t)idx2[j] * 32));
                }
                cptr.push_back((int)cand.size());
            }
            ++ia; ++ib;
        } else if (nodes1[ia] < nodes2[ib]) {
            ++ia;
        } else {
            ++ib;
        }
    }
    *nq_out = (int)q1.size();
    *total_out = (int)cand.size();
    if ((int)q1.size() > q_capacity || (int)cand.size() > capacity) return VSG_ERR_CAPACITY;
    for (size_t k = 0; k < q1.size(); ++k) { q1_out[k] = q1[k]; cand_ptr_out[k] = cptr[k]; }
    cand_ptr_out[q1.size()] = (int)cand.size();
    for (size_t c = 0; c < cand.size(); ++c) { cand_idx2_out[c] = cand[c]; cand_dist_out[c] = dist[c]; }
    return VSG_OK;
}
vsg_status vsg_search_for_triangulation(vsg_matcher *, const vsg_frame_view *KF1, const uint8_t *has_mp1, const vsg_frame_view *KF2,
                                        const uint8_t *has_mp2, int nn1, const int32_t *nodes1, const int32_t *ptr1, const int32_t *idx1,
                                        int nn2, const int32_t *nodes2, const int32_t *ptr2, const int32_t *idx2, int only_stereo, int coarse,
                                        const float *f12, const float *ep, const float *level_sigma2_2, int check_ori,
                                        int32_t *matches12_out, int *nmatches_out) {
    *nmatches_out = orc_search_for_triangulation(V(KF1), has_mp1, V(KF2), has_mp2, nn1, nodes1, ptr1, idx1, nn2, nodes2, ptr2, idx2,
                                                 only_stereo, coarse, f12, ep, level_sigma2_2, check_ori, matches12_out);
    return VSG_OK;
}

}  // extern "C"
