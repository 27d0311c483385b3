// match_methods_kf.cu — the keyframe-side Search* / Fuse methods on flattened views (single-camera branches).
//
// Reference (snt-arg/visual_sgraphs), orb_slam3/src/ORBmatcher.cc:
//   SearchByProjection(Frame&, KeyFrame*, sAlreadyFound, th, ORBdist)            :1880-2000  (relocalisation)
//   SearchByProjection(KeyFrame*, Sim3f&, vpPoints, vpMatched, th, ratioHamming) :430-528
//   SearchByProjection(KeyFrame*, Sim3f&, vpPoints, vpPointsKFs, ...)            :530-641
//   Fuse(KeyFrame*, vpMapPoints, th, bRight)                                      :1148-1335
//   Fuse(KeyFrame*, Sim3f&, vpPoints, th, vpReplacePoint)                         :1337-1446
//   SearchBySim3(pKF1, pKF2, vpMatches12, S12, th)                                :1448-1665
//   SearchByBoW(KeyFrame*, KeyFrame*, vpMatches12)                                :758-900
//   SearchForTriangulation(pKF1, pKF2, vMatchedPairs, bOnlyStereo, bCoarse)       :902-1146
//   KeyFrame::GetFeaturesInArea                                                   orb_slam3/src/KeyFrame.cc:834-875
//   Pinhole::epipolarConstrain                                                    orb_slam3/src/CameraModels/Pinhole.cpp:118-141
//
// Same split of work as match_methods.cu: the GPU answers every window query of a call at once (grid walk +
// 256-bit Hamming distance of each candidate: area_search_kernel), or every in-node descriptor pair of a BoW
// walk (window_match_kernel); the order-dependent bookkeeping is replayed on the host over those lists.
// KeyFrame::GetFeaturesInArea is Frame::GetFeaturesInArea without the level filter; the callers' per-candidate
// level gate (kpLevel < nPredictedLevel-1 || kpLevel > nPredictedLevel) is the same filter applied later, so it
// is folded into the query (min_level = level-1, max_level = level >= 0, which always enables the check).
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "match_internal.cuh"

using namespace vsg;

namespace {

// Queries for the valid points of a projected-point list: radius = th * scale[level], levels [level+lo, level+hi]; appended
// to qs, with the point's index in q_src.
vsg_status append_queries(const vsg_frame *F, int n, const vsg_search_point *pts, float th, int lo, int hi,
                          std::vector<AreaQuery> &qs, std::vector<int> &q_src) {
    for (int i = 0; i < n; ++i) {
        const vsg_search_point &p = pts[i];
        if (!p.valid) continue;
        if (p.level < 0 || p.level >= (int)F->scale.size()) {
            set_error("search point %d: level %d out of range", i, p.level);
            return VSG_ERR_INVALID;
        }
        const float radius = th * F->scale[p.level];
        qs.push_back(AreaQuery{p.u, p.v, radius, p.level + lo, p.level + hi, 0.f, -1.f});
        q_src.push_back(i);
    }
    return VSG_OK;
}

// The same as a fresh list, with the descriptor rows of the queries gathered into qdesc.
vsg_status build_queries(const vsg_frame *F, int n, const vsg_search_point *pts, const uint8_t *desc, float th, int lo,
                         int hi, std::vector<AreaQuery> &qs, std::vector<int> &q_src, std::vector<uint8_t> &qdesc) {
    qs.clear(); q_src.clear();
    const vsg_status st = append_queries(F, n, pts, th, lo, hi, qs, q_src);
    if (st != VSG_OK) return st;
    qdesc.resize(qs.size() * 32);
    for (size_t k = 0; k < qs.size(); ++k) memcpy(&qdesc[k * 32], desc + (size_t)q_src[k] * 32, 32);
    return VSG_OK;
}

struct FeatVec {
    int nnodes;
    const int32_t *nodes, *ptr, *idx;
};

// The merge walk over two DBoW2::FeatureVectors (e.g. :785-872): for every feature of vector 1 that passes
// `use1`, inside a node both vectors share, one query whose candidates are ALL features of that node in vector 2
// (in vIndices order; per-candidate gates are applied in the replay).  Distances come from the GPU.
template <class Use1>
vsg_status bow_pair_dists(vsg_matcher *m, const vsg_frame_view *V1, const vsg_frame_view *V2, const FeatVec &a,
                          const FeatVec &b, Use1 use1, std::vector<int> &q1, std::vector<int> &cptr,
                          std::vector<int> &cand, std::vector<int> &dist) {
    q1.clear(); cand.clear(); cptr.assign(1, 0);
    int ia = 0, ib = 0;
    while (ia < a.nnodes && ib < b.nnodes) {
        if (a.nodes[ia] == b.nodes[ib]) {
            for (int k = a.ptr[ia]; k < a.ptr[ia + 1]; ++k) {
                const int i1 = a.idx[k];
                if (i1 < 0 || i1 >= V1->n) { set_error("bow: feature index out of range"); return VSG_ERR_INVALID; }
                if (!use1(i1)) continue;
                q1.push_back(i1);
                for (int j = b.ptr[ib]; j < b.ptr[ib + 1]; ++j) {
                    if (b.idx[j] < 0 || b.idx[j] >= V2->n) { set_error("bow: feature index out of range"); return VSG_ERR_INVALID; }
                    cand.push_back(b.idx[j]);
                }
                cptr.push_back((int)cand.size());
            }
            ++ia; ++ib;
        } else if (a.nodes[ia] < b.nodes[ib]) {
            while (ia < a.nnodes && a.nodes[ia] < b.nodes[ib]) ++ia;      // lower_bound
        } else {
            while (ib < b.nnodes && b.nodes[ib] < a.nodes[ia]) ++ib;
        }
    }
    const int nq = (int)q1.size(), ncand = (int)cand.size();
    dist.assign(ncand, 0);
    if (nq == 0 || ncand == 0) return VSG_OK;
    std::vector<uint8_t> qdesc((size_t)nq * 32);
    for (int k = 0; k < nq; ++k) memcpy(&qdesc[(size_t)k * 32], V1->descriptors + (size_t)q1[k] * 32, 32);
    vsg_status st;
    if ((st = matcher_ensure(m, 1, (size_t)nq * 32)) || (st = matcher_ensure(m, 2, (size_t)std::max(V2->n, 1) * 32)) ||
        (st = matcher_ensure(m, 3, (size_t)(nq + 1) * 4)) || (st = matcher_ensure(m, 4, (size_t)ncand * 4)) ||
        (st = matcher_ensure(m, 6, (size_t)ncand * 4)))
        return st;
    cudaStream_t s = m->stream;
    CK(cudaMemcpyAsync(m->buf[1], qdesc.data(), (size_t)nq * 32, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(m->buf[2], V2->descriptors, (size_t)V2->n * 32, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(m->buf[3], cptr.data(), (size_t)(nq + 1) * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(m->buf[4], cand.data(), (size_t)ncand * 4, cudaMemcpyHostToDevice, s));
    launch_window_dists(m, (const uint8_t *)m->buf[1], nq, (const uint8_t *)m->buf[2], (const int *)m->buf[3],
                        (const int *)m->buf[4], (int *)m->buf[6]);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(dist.data(), m->buf[6], (size_t)ncand * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return VSG_OK;
}

bool featvec_ok(int nn, const int32_t *nodes, const int32_t *ptr, const int32_t *idx) {
    return nn >= 0 && (nn == 0 || (nodes && ptr && idx));
}

// the rotation-consistency filter shared by the methods: everything outside the three dominant bins is dropped
template <class Drop>
void apply_rot_filter(const std::vector<int> *rot_hist, Drop drop) {
    int ind1 = -1, ind2 = -1, ind3 = -1;
    three_maxima(rot_hist, HISTO_LENGTH, ind1, ind2, ind3);
    for (int i = 0; i < HISTO_LENGTH; ++i) {
        if (i == ind1 || i == ind2 || i == ind3) continue;
        for (int idx : rot_hist[i]) drop(idx);
    }
}

}  // namespace

extern "C" {

// ORBmatcher.cc:1880-2000
vsg_status vsg_search_by_projection_reloc(vsg_matcher *m, const vsg_frame *Cur, const uint8_t *occupied, int n,
                                          const vsg_search_point *pts, const uint8_t *desc, float th, int orb_dist,
                                          int check_ori, int32_t *assign_out, int *nmatches_out) {
    if (!m || !Cur || n < 0 || !assign_out || (n > 0 && (!pts || !desc)) || (Cur->n > 0 && !occupied)) return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    std::vector<AreaQuery> qs;
    std::vector<int> q_src, ptr;
    std::vector<uint8_t> qdesc;
    std::vector<int2> ent;
    vsg_status st = build_queries(Cur, n, pts, desc, th, -1, +1, qs, q_src, qdesc);   // :1927
    if (st != VSG_OK) return st;
    if ((st = area_search(m, Cur, (int)qs.size(), qs.data(), qdesc.data(), ptr, ent)) != VSG_OK) return st;
    std::vector<uint8_t> taken(occupied, occupied + Cur->n);                          // CurrentFrame.mvpMapPoints[i2]
    for (int i = 0; i < Cur->n; ++i) assign_out[i] = -1;
    std::vector<int> rot_hist[HISTO_LENGTH];
    int nmatches = 0;
    for (size_t k = 0; k < qs.size(); ++k) {
        int best = 256, best_idx = -1;
        for (int c = ptr[k]; c < ptr[k + 1]; ++c) {
            const int i2 = ent[c].x, dist = ent[c].y;
            if (taken[i2]) continue;                                                 // :1939-1940
            if (dist < best) { best = dist; best_idx = i2; }
        }
        if (best <= orb_dist && best_idx >= 0) {                                     // :1952
            assign_out[best_idx] = q_src[k];
            taken[best_idx] = 1;
            ++nmatches;
            if (check_ori) rot_hist[rot_bin(pts[q_src[k]].angle, Cur->keys[best_idx].angle)].push_back(best_idx);
        }
    }
    if (check_ori) apply_rot_filter(rot_hist, [&](int idx) { assign_out[idx] = -2; --nmatches; });
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

// ORBmatcher.cc:430-528 and :530-641
vsg_status vsg_search_by_projection_sim3(vsg_matcher *m, const vsg_frame *KF, const uint8_t *matched, int n,
                                         const vsg_search_point *pts, const uint8_t *desc, int th,
                                         float ratio_hamming, int32_t *assign_out, int *nmatches_out) {
    if (!m || !KF || n < 0 || !assign_out || (n > 0 && (!pts || !desc)) || (KF->n > 0 && !matched)) return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    std::vector<AreaQuery> qs;
    std::vector<int> q_src, ptr;
    std::vector<uint8_t> qdesc;
    std::vector<int2> ent;
    vsg_status st = build_queries(KF, n, pts, desc, (float)th, -1, 0, qs, q_src, qdesc);   // :486, :502-503
    if (st != VSG_OK) return st;
    if ((st = area_search(m, KF, (int)qs.size(), qs.data(), qdesc.data(), ptr, ent)) != VSG_OK) return st;
    std::vector<uint8_t> taken(matched, matched + KF->n);                            // vpMatched[idx]
    for (int i = 0; i < KF->n; ++i) assign_out[i] = -1;
    int nmatches = 0;
    const float gate = TH_LOW * ratio_hamming;                                       // :520
    for (size_t k = 0; k < qs.size(); ++k) {
        int best = 256, best_idx = -1;
        for (int c = ptr[k]; c < ptr[k + 1]; ++c) {
            const int idx = ent[c].x, dist = ent[c].y;
            if (taken[idx]) continue;                                                // :497-498
            if (dist < best) { best = dist; best_idx = idx; }
        }
        if ((float)best <= gate && best_idx >= 0) {
            assign_out[best_idx] = q_src[k];
            taken[best_idx] = 1;
            ++nmatches;
        }
    }
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

// the search part of ORBmatcher.cc:1148-1335 (variant 0) and :1337-1446 (variant 1)
vsg_status vsg_fuse_search(vsg_matcher *m, const vsg_frame *KF, int n, const vsg_search_point *pts,
                           const uint8_t *desc, float th, const float *inv_level_sigma2, int variant,
                           int32_t *best_idx_out, int *nfused_out) {
    if (!m || !KF || n < 0 || (n > 0 && (!pts || !desc || !best_idx_out)) || (variant == 0 && !inv_level_sigma2) ||
        (variant != 0 && variant != 1))
        return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    std::vector<AreaQuery> qs;
    std::vector<int> q_src;
    std::vector<uint8_t> qdesc;
    vsg_status st = build_queries(KF, n, pts, desc, th, -1, 0, qs, q_src, qdesc);     // :1246, :1270-1271
    if (st != VSG_OK) return st;
    if (variant == 0)
        for (size_t k = 0; k < qs.size(); ++k) qs[k].xr = pts[q_src[k]].ur;         // the right coordinate of the chi-square gate
    // every map point's search is independent of the others: the best candidate (with the chi-square gates of :1273-1299 for
    // the pose-based variant) is picked on the device, one (index, distance) pair per point comes back
    std::vector<int2> best;
    if ((st = area_best(m, KF, (int)qs.size(), qs.data(), qdesc.data(), variant == 0 ? inv_level_sigma2 : nullptr, best)) != VSG_OK)
        return st;
    for (int i = 0; i < n; ++i) best_idx_out[i] = -1;
    int nfused = 0;
    for (size_t k = 0; k < qs.size(); ++k) {
        if (best[k].x >= 0 && best[k].y <= TH_LOW) {                                 // :1316, :1428
            best_idx_out[q_src[k]] = best[k].x;
            ++nfused;
        }
    }
    if (nfused_out) *nfused_out = nfused;
    return VSG_OK;
}

// vsg_fuse_search(..., variant 0, ...) once per target keyframe, all targets in one upload, one launch and one download:
// the searches of LocalMapping::SearchInNeighbors' loop of Fuse calls (LocalMapping.cc:764-802)
vsg_status vsg_fuse_search_multi(vsg_matcher *m, int ntargets, const vsg_frame *const *KFs, const float *const *inv_level_sigma2,
                                 int n, const vsg_search_point *pts, const uint8_t *desc, float th, int32_t *best_idx_out) {
    if (!m || ntargets < 0 || n < 0) {
        set_error("vsg_fuse_search_multi: %d targets, %d points", ntargets, n);
        return VSG_ERR_INVALID;
    }
    if (ntargets > 0 && (!KFs || !inv_level_sigma2 || (n > 0 && (!pts || !desc || !best_idx_out)))) {
        set_error("vsg_fuse_search_multi: null target table, level table, points, descriptors or output");
        return VSG_ERR_INVALID;
    }
    for (int t = 0; t < ntargets; ++t) {
        if (!KFs[t] || !inv_level_sigma2[t]) {
            set_error("vsg_fuse_search_multi: target %d: null keyframe or level table", t);
            return VSG_ERR_INVALID;
        }
        if (KFs[t]->device != m->device) {
            set_error("vsg_fuse_search_multi: target %d lives on device %d, the matcher on device %d", t, KFs[t]->device, m->device);
            return VSG_ERR_INVALID;
        }
    }
    CK(cudaSetDevice(m->device));
    std::vector<AreaQuery> qs;
    std::vector<int> q_src, q_tgt;
    for (int t = 0; t < ntargets; ++t) {
        const vsg_search_point *tp = pts + (size_t)t * n;
        const size_t first = qs.size();
        const vsg_status st = append_queries(KFs[t], n, tp, th, -1, 0, qs, q_src);      // :1246, :1270-1271
        if (st != VSG_OK) {
            const std::string why = vsg_last_error();
            set_error("vsg_fuse_search_multi: target %d: %s", t, why.c_str());
            return st;
        }
        for (size_t k = first; k < qs.size(); ++k) {
            qs[k].xr = tp[q_src[k]].ur;                                                    // the chi-square gate's right coordinate
            qs[k].desc_idx = q_src[k];                                                     // desc is shared by all targets
        }
        q_tgt.resize(qs.size(), t);
    }
    std::vector<int2> best;
    vsg_status st = area_best_multi(m, ntargets, KFs, inv_level_sigma2, (int)qs.size(), qs.data(), q_tgt.data(), n, desc, best);
    if (st != VSG_OK) return st;
    for (size_t i = 0; i < (size_t)ntargets * n; ++i) best_idx_out[i] = -1;
    for (size_t k = 0; k < qs.size(); ++k)
        if (best[k].x >= 0 && best[k].y <= TH_LOW) best_idx_out[(size_t)q_tgt[k] * n + q_src[k]] = best[k].x;   // :1316
    return VSG_OK;
}

// ORBmatcher.cc:1448-1665
vsg_status vsg_search_by_sim3(vsg_matcher *m, const vsg_frame *KF1, const vsg_frame *KF2, int n1,
                              const vsg_search_point *pts1, const uint8_t *desc1, int n2,
                              const vsg_search_point *pts2, const uint8_t *desc2, float th, int32_t *matches12_out,
                              int *nfound_out) {
    // n1 / n2 = map point slots of the keyframes; more than the searched features for two-camera keyframes (KF1 / KF2 are then
    // their left cameras): slot i of KF1 searches KF2's features, the answer is cross-checked through slot idx2 of KF2
    if (!m || !KF1 || !KF2 || n1 < KF1->n || n2 < KF2->n || (n1 > 0 && (!pts1 || !desc1 || !matches12_out)) ||
        (n2 > 0 && (!pts2 || !desc2))) {
        set_error("vsg_search_by_sim3: pts1 / pts2 need at least one entry per keyframe feature");
        return VSG_ERR_INVALID;
    }
    CK(cudaSetDevice(m->device));
    std::vector<int> match1(n1, -1), match2(n2, -1);
    for (int dir = 0; dir < 2; ++dir) {
        const vsg_frame *target = dir == 0 ? KF2 : KF1;                              // :1488-1560 then :1563-1635
        const int n = dir == 0 ? n1 : n2;
        std::vector<int> &out = dir == 0 ? match1 : match2;
        std::vector<AreaQuery> qs;
        std::vector<int> q_src;
        std::vector<uint8_t> qdesc;
        vsg_status st = build_queries(target, n, dir == 0 ? pts1 : pts2, dir == 0 ? desc1 : desc2, th, -1, 0, qs, q_src, qdesc);
        if (st != VSG_OK) return st;
        std::vector<int2> best;                                                      // independent queries: best on the device
        if ((st = area_best(m, target, (int)qs.size(), qs.data(), qdesc.data(), nullptr, best)) != VSG_OK) return st;
        for (size_t k = 0; k < qs.size(); ++k)
            if (best[k].x >= 0 && best[k].y <= TH_HIGH) out[q_src[k]] = best[k].x;   // :1556, :1631
    }
    int nfound = 0;
    for (int i1 = 0; i1 < n1; ++i1) {                                                // :1638-1652
        matches12_out[i1] = -1;
        const int idx2 = match1[i1];
        if (idx2 >= 0 && match2[idx2] == i1) { matches12_out[i1] = idx2; ++nfound; }
    }
    if (nfound_out) *nfound_out = nfound;
    return VSG_OK;
}

// ORBmatcher.cc:758-900
vsg_status vsg_search_by_bow_kf(vsg_matcher *m, const vsg_frame_view *KF1, const uint8_t *mp_valid1,
                                const vsg_frame_view *KF2, const uint8_t *mp_valid2, int nnodes1,
                                const int32_t *nodes1, const int32_t *ptr1, const int32_t *idx1, int nnodes2,
                                const int32_t *nodes2, const int32_t *ptr2, const int32_t *idx2, float nnratio,
                                int check_ori, int32_t *matches12_out, int *nmatches_out) {
    if (!m || !KF1 || !KF2 || !featvec_ok(nnodes1, nodes1, ptr1, idx1) || !featvec_ok(nnodes2, nodes2, ptr2, idx2) ||
        (KF1->n > 0 && (!mp_valid1 || !matches12_out)) || (KF2->n > 0 && !mp_valid2))
        return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    std::vector<int> q1, cptr, cand, dist;
    vsg_status st = bow_pair_dists(m, KF1, KF2, FeatVec{nnodes1, nodes1, ptr1, idx1}, FeatVec{nnodes2, nodes2, ptr2, idx2},
                                   [&](int i1) { return mp_valid1[i1] != 0; }, q1, cptr, cand, dist);
    if (st != VSG_OK) return st;
    for (int i = 0; i < KF1->n; ++i) matches12_out[i] = -1;
    std::vector<uint8_t> matched2(KF2->n, 0);
    std::vector<int> rot_hist[HISTO_LENGTH];
    int nmatches = 0;
    for (size_t k = 0; k < q1.size(); ++k) {
        const int i1 = q1[k];
        int best1 = 256, best_idx2 = -1, best2 = 256;
        for (int c = cptr[k]; c < cptr[k + 1]; ++c) {
            const int i2 = cand[c];
            if (matched2[i2] || !mp_valid2[i2]) continue;                            // :821-825
            const int d = dist[c];
            if (d < best1) { best2 = best1; best1 = d; best_idx2 = i2; }
            else if (d < best2) best2 = d;
        }
        if (best1 < TH_LOW) {                                                        // :843 (strict)
            if (static_cast<float>(best1) < nnratio * static_cast<float>(best2)) {
                matches12_out[i1] = best_idx2;
                matched2[best_idx2] = 1;
                if (check_ori) rot_hist[rot_bin(KF1->keys[i1].angle, KF2->keys[best_idx2].angle)].push_back(i1);
                ++nmatches;
            }
        }
    }
    if (check_ori) apply_rot_filter(rot_hist, [&](int i1) { matches12_out[i1] = -1; --nmatches; });
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

// The Hamming-distance half of the BoW-guided pairings for callers that own the per-pair geometry test (two-camera
// SearchForTriangulation: KannalaBrandt8::epipolarConstrain is the caller's camera code): the merge walk of :966-1118 with
// every candidate's distance from the GPU, in the reference's scan order.
vsg_status vsg_bow_pair_distances(vsg_matcher *m, const vsg_frame_view *KF1, const uint8_t *use1, const vsg_frame_view *KF2,
                                  int nnodes1, const int32_t *nodes1, const int32_t *ptr1, const int32_t *idx1, int nnodes2,
                                  const int32_t *nodes2, const int32_t *ptr2, const int32_t *idx2, int32_t *q1_out,
                                  int32_t *cand_ptr_out, int q_capacity, int32_t *cand_idx2_out, int32_t *cand_dist_out,
                                  int capacity, int *nq_out, int *total_out) {
    if (!m || !KF1 || !KF2 || !featvec_ok(nnodes1, nodes1, ptr1, idx1) || !featvec_ok(nnodes2, nodes2, ptr2, idx2) ||
        (KF1->n > 0 && !use1) || !nq_out || !total_out)
        return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    std::vector<int> q1, cptr, cand, dist;
    vsg_status st = bow_pair_dists(m, KF1, KF2, FeatVec{nnodes1, nodes1, ptr1, idx1}, FeatVec{nnodes2, nodes2, ptr2, idx2},
                                   [&](int i1) { return use1[i1] != 0; }, q1, cptr, cand, dist);
    if (st != VSG_OK) return st;
    *nq_out = (int)q1.size();
    *total_out = (int)cand.size();
    if ((int)q1.size() > q_capacity || (int)cand.size() > capacity) return VSG_ERR_CAPACITY;
    if ((!q1.empty() && (!q1_out || !cand_ptr_out)) || (!cand.empty() && (!cand_idx2_out || !cand_dist_out))) return VSG_ERR_INVALID;
    for (size_t k = 0; k < q1.size(); ++k) { q1_out[k] = q1[k]; cand_ptr_out[k] = cptr[k]; }
    if (cand_ptr_out) cand_ptr_out[q1.size()] = (int)cand.size();
    for (size_t c = 0; c < cand.size(); ++c) { cand_idx2_out[c] = cand[c]; cand_dist_out[c] = dist[c]; }
    return VSG_OK;
}

// ORBmatcher.cc:902-1146 (mpCamera2 == NULL, Pinhole::epipolarConstrain)
vsg_status vsg_search_for_triangulation(vsg_matcher *m, const vsg_frame_view *KF1, const uint8_t *has_mp1,
                                        const vsg_frame_view *KF2, const uint8_t *has_mp2, int nnodes1,
                                        const int32_t *nodes1, const int32_t *ptr1, const int32_t *idx1, int nnodes2,
                                        const int32_t *nodes2, const int32_t *ptr2, const int32_t *idx2,
                                        int only_stereo, int coarse, const float *f12, const float *ep,
                                        const float *level_sigma2_2, int check_ori, int32_t *matches12_out,
                                        int *nmatches_out) {
    if (!m || !KF1 || !KF2 || !featvec_ok(nnodes1, nodes1, ptr1, idx1) || !featvec_ok(nnodes2, nodes2, ptr2, idx2) ||
        (KF1->n > 0 && (!has_mp1 || !matches12_out)) || (KF2->n > 0 && !has_mp2) || !ep || (!coarse && (!f12 || !level_sigma2_2)) ||
        (KF2->n > 0 && !KF2->scale_factors))
        return VSG_ERR_INVALID;
    CK(cudaSetDevice(m->device));
    auto stereo1 = [&](int i) { return KF1->u_right && KF1->u_right[i] >= 0; };       // :977
    auto stereo2 = [&](int i) { return KF2->u_right && KF2->u_right[i] >= 0; };       // :1005
    std::vector<int> q1, cptr, cand, dist;
    vsg_status st = bow_pair_dists(m, KF1, KF2, FeatVec{nnodes1, nodes1, ptr1, idx1}, FeatVec{nnodes2, nodes2, ptr2, idx2},
                                   [&](int i1) { return !has_mp1[i1] && (!only_stereo || stereo1(i1)); },   // :971-981
                                   q1, cptr, cand, dist);
    if (st != VSG_OK) return st;
    for (int i = 0; i < KF1->n; ++i) matches12_out[i] = -1;
    std::vector<int> rot_hist[HISTO_LENGTH];
    int nmatches = 0;
    for (size_t k = 0; k < q1.size(); ++k) {
        const int i1 = q1[k];
        const vsg_keypoint &kp1 = KF1->keys[i1];
        const bool b_stereo1 = stereo1(i1);
        int best = TH_LOW, best_idx2 = -1;
        for (int c = cptr[k]; c < cptr[k + 1]; ++c) {
            const int i2 = cand[c];
            if (has_mp2[i2]) continue;                                               // :1001 (vbMatched2 is never set, SURVEY C#3)
            const bool b_stereo2 = stereo2(i2);
            if (only_stereo && !b_stereo2) continue;
            const int d = dist[c];
            if (d > TH_LOW || d > best) continue;                                    // :1014
            const vsg_keypoint &kp2 = KF2->keys[i2];
            if (!b_stereo1 && !b_stereo2) {                                          // :1023-1031
                const float distex = ep[0] - kp2.x, distey = ep[1] - kp2.y;
                if (distex * distex + distey * distey < 100 * KF2->scale_factors[kp2.octave]) continue;
            }
            bool ok = coarse != 0;
            if (!ok) {                                                               // Pinhole.cpp:126-140
                const float a = kp1.x * f12[0] + kp1.y * f12[3] + f12[6];
                const float b = kp1.x * f12[1] + kp1.y * f12[4] + f12[7];
                const float cc = kp1.x * f12[2] + kp1.y * f12[5] + f12[8];
                const float num = a * kp2.x + b * kp2.y + cc;
                const float den = a * a + b * b;
                if (den != 0) {
                    const float dsqr = num * num / den;
                    ok = dsqr < 3.84 * level_sigma2_2[kp2.octave];
                }
            }
            if (ok) { best_idx2 = i2; best = d; }
        }
        if (best_idx2 >= 0) {
            matches12_out[i1] = best_idx2;
            ++nmatches;
            if (check_ori) rot_hist[rot_bin(kp1.angle, KF2->keys[best_idx2].angle)].push_back(i1);
        }
    }
    if (check_ori) apply_rot_filter(rot_hist, [&](int i1) { matches12_out[i1] = -1; --nmatches; });
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

}  // extern "C"
