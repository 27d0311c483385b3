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
// 256-bit Hamming distance of each candidate: area_search_kernel), or every in-node descriptor pair of the BoW
// walks of a call (bow_dists_multi_kernel); the order-dependent bookkeeping is replayed on the host over those lists.
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

namespace vsg {

bool featvec_ok(int nn, const int32_t *nodes, const int32_t *ptr, const int32_t *idx) {
    return nn >= 0 && (nn == 0 || (nodes && ptr && (idx || ptr[nn] == 0)));
}

// The CSR lists of a FeatureVector must be well formed: the device reads side 2's idx[ptr[k] .. ptr[k+1]) from a copy of
// idx[0 .. ptr[nnodes]), so the offsets start at 0 and never decrease.  nullptr: nothing wrong.
static const char *featvec_problem(const FeatVec &v) {
    if (v.nnodes < 0) return "negative node count";
    if (v.nnodes == 0) return nullptr;
    if (!v.nodes || !v.ptr) return "null node or offset array";
    if (v.ptr[0] != 0) return "first list offset is not 0";
    for (int k = 0; k < v.nnodes; ++k)
        if (v.ptr[k + 1] < v.ptr[k]) return "list offsets decrease";
    if (v.ptr[v.nnodes] > 0 && !v.idx) return "null feature index array";
    return nullptr;
}

vsg_status bow_walk(const BowWalk &w, std::vector<BowSeg> &segs, int64_t *npairs) {
    const FeatVec &a = w.a, &b = w.b;
    for (const FeatVec *v : {&a, &b})
        if (const char *why = featvec_problem(*v)) {
            set_error("bow: malformed feature vector: %s", why);
            return VSG_ERR_INVALID;
        }
    int ia = 0, ib = 0;
    while (ia < a.nnodes && ib < b.nnodes) {
        if (a.nodes[ia] == b.nodes[ib]) {
            const int jb = b.ptr[ib], je = b.ptr[ib + 1];
            bool checked = false;                                         // side 2's node, once a query uses it
            for (int k = a.ptr[ia]; k < a.ptr[ia + 1]; ++k) {
                const int i1 = a.idx[k];
                if (i1 < 0 || i1 >= w.v1->n) {
                    set_error("bow: feature index %d out of range (%d features)", i1, w.v1->n);
                    return VSG_ERR_INVALID;
                }
                if (!w.use1[i1]) continue;
                for (int j = jb; j < je && !checked; ++j)
                    if (b.idx[j] < 0 || b.idx[j] >= w.v2->n) {
                        set_error("bow: feature index %d out of range (%d features)", b.idx[j], w.v2->n);
                        return VSG_ERR_INVALID;
                    }
                checked = true;
                segs.push_back(BowSeg{i1, jb, je, (int)std::min<int64_t>(*npairs, INT_MAX)});
                *npairs += je - jb;
            }
            ++ia; ++ib;
        } else if (a.nodes[ia] < b.nodes[ib]) {
            while (ia < a.nnodes && a.nodes[ia] < b.nodes[ib]) ++ia;      // lower_bound
        } else {
            while (ib < b.nnodes && b.nodes[ib] < a.nodes[ia]) ++ib;
        }
    }
    return VSG_OK;
}

vsg_status bow_dists(vsg_matcher *m, int nwalks, const BowWalk *walks, const std::vector<BowSeg> &segs, const int *seg_ptr,
                     int64_t npairs, const uint16_t **dist) {
    *dist = nullptr;
    if (npairs == 0) return VSG_OK;
    if (npairs > INT_MAX) {
        set_error("bow: %lld descriptor pairs in one call (at most %d)", (long long)npairs, INT_MAX);
        return VSG_ERR_INVALID;
    }
    // every distinct descriptor table and side-2 idx array once: a frame shared by all walks, a keyframe passed twice
    struct Table { const void *p; int n, first; };
    std::vector<Table> tabs, idxs;
    int rows = 0, nidx = 0;
    auto place = [](std::vector<Table> &v, const void *p, int n, int &total) {
        for (const Table &t : v)
            if (t.p == p && t.n == n) return t.first;
        v.push_back(Table{p, n, total});
        total += n;
        return v.back().first;
    };
    std::vector<int4> dsegs;
    for (int k = 0; k < nwalks; ++k) {
        const BowWalk &w = walks[k];
        int row1 = -1, row2 = -1, idx0 = -1;
        for (int q = seg_ptr[k]; q < seg_ptr[k + 1]; ++q) {
            const BowSeg &sg = segs[q];
            if (sg.je == sg.jb) continue;
            if (row1 < 0) {
                row1 = place(tabs, w.v1->descriptors, w.v1->n, rows);
                row2 = place(tabs, w.v2->descriptors, w.v2->n, rows);
                idx0 = place(idxs, w.b.idx, w.b.ptr[w.b.nnodes], nidx);
            }
            dsegs.push_back(make_int4(row1 + sg.i1, idx0 + sg.jb, row2, sg.off));
        }
    }
    dsegs.push_back(make_int4(0, 0, 0, (int)npairs));                     // sentinel
    auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
    const size_t o_seg = 0, o_desc = up16(dsegs.size() * sizeof(int4)), o_idx = o_desc + (size_t)rows * 32,
                 o_out = up16(o_idx + (size_t)nidx * sizeof(int)), total = o_out + (size_t)npairs * sizeof(uint16_t);
    vsg_status st;
    // device slot 19 and pinned host slot 8: inputs, then the distances
    if ((st = matcher_ensure(m, 19, total)) || (st = matcher_ensure_host(m, 8, total))) return st;
    uint8_t *h = (uint8_t *)m->hbuf[8], *d = (uint8_t *)m->buf[19];
    memcpy(h + o_seg, dsegs.data(), dsegs.size() * sizeof(int4));
    for (const Table &t : tabs) memcpy(h + o_desc + (size_t)t.first * 32, t.p, (size_t)t.n * 32);
    for (const Table &t : idxs) memcpy(h + o_idx + (size_t)t.first * sizeof(int), t.p, (size_t)t.n * sizeof(int));
    cudaStream_t s = m->stream;
    CK(cudaMemcpyAsync(d, h, o_out, cudaMemcpyHostToDevice, s));
    launch_bow_dists(m, (const int4 *)(d + o_seg), (int)dsegs.size(), (const int *)(d + o_idx), d + o_desc, (int)npairs,
                     (uint16_t *)(d + o_out));
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h + o_out, d + o_out, (size_t)npairs * sizeof(uint16_t), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    *dist = (const uint16_t *)(h + o_out);
    return VSG_OK;
}

const char *bow_side_problem(const vsg_bow_side *s, bool needs_valid) {
    if (!s) return "null side";
    if (s->view.n < 0) return "negative feature count";
    if (s->view.n > 0 && (!s->view.descriptors || !s->view.keys)) return "null keypoints or descriptors";
    if (needs_valid && s->view.n > 0 && !s->mp_valid) return "null map-point flags";
    if (!featvec_ok(s->nnodes, s->nodes, s->ptr, s->idx)) return "malformed feature vector";
    return nullptr;
}

// The KF-KF replay of SearchByBoW (ORBmatcher.cc:785-900) over one walk's distances: already-matched and map-point-less
// candidates skipped (:821-825), best / second best, TH_LOW (strict) and ratio gates, rotation histogram.  Returns nmatches.
static int bow_replay_kf(const vsg_frame_view *KF1, const vsg_frame_view *KF2, const uint8_t *mp_valid2, const FeatVec &b2,
                         const BowSeg *segs, int nseg, const uint16_t *dist, float nnratio, int check_ori, int32_t *matches12_out) {
    for (int i = 0; i < KF1->n; ++i) matches12_out[i] = -1;
    std::vector<uint8_t> matched2(KF2->n, 0);
    std::vector<int> rot_hist[HISTO_LENGTH];
    int nmatches = 0;
    for (int k = 0; k < nseg; ++k) {
        const BowSeg &sg = segs[k];
        const int i1 = sg.i1;
        int best1 = 256, best_idx2 = -1, best2 = 256;
        for (int j = sg.jb; j < sg.je; ++j) {
            const int i2 = b2.idx[j];
            if (matched2[i2] || !mp_valid2[i2]) continue;                            // :821-825
            const int d = dist[sg.off + j - sg.jb];
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
    return nmatches;
}

}  // namespace vsg

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
    const BowWalk w{KF1, mp_valid1, FeatVec{nnodes1, nodes1, ptr1, idx1}, KF2, FeatVec{nnodes2, nodes2, ptr2, idx2}};
    std::vector<BowSeg> segs;
    int64_t npairs = 0;
    const uint16_t *dist;
    vsg_status st = bow_walk(w, segs, &npairs);
    const int seg_ptr[2] = {0, (int)segs.size()};
    if (st != VSG_OK || (st = bow_dists(m, 1, &w, segs, seg_ptr, npairs, &dist)) != VSG_OK) return st;
    const int nmatches = bow_replay_kf(KF1, KF2, mp_valid2, w.b, segs.data(), (int)segs.size(), dist, nnratio, check_ori, matches12_out);
    if (nmatches_out) *nmatches_out = nmatches;
    return VSG_OK;
}

// vsg_search_by_bow_kf(KF1 against KF2s[t]) for every target in one upload, one launch and one download
vsg_status vsg_search_by_bow_kf_multi(vsg_matcher *m, const vsg_bow_side *KF1, int ntargets, const vsg_bow_side *const *KF2s,
                                      float nnratio, int check_ori, int32_t *matches12_out, int *nmatches_out) {
    if (!m || ntargets < 0) {
        set_error("vsg_search_by_bow_kf_multi: %d targets", ntargets);
        return VSG_ERR_INVALID;
    }
    if (ntargets == 0) return VSG_OK;
    const char *why;
    if (!KF2s || !nmatches_out || (KF1 && KF1->view.n > 0 && !matches12_out)) {
        set_error("vsg_search_by_bow_kf_multi: null target table or output");
        return VSG_ERR_INVALID;
    }
    if ((why = bow_side_problem(KF1, true))) {
        set_error("vsg_search_by_bow_kf_multi: KF1: %s", why);
        return VSG_ERR_INVALID;
    }
    for (int t = 0; t < ntargets; ++t)
        if ((why = bow_side_problem(KF2s[t], true))) {
            set_error("vsg_search_by_bow_kf_multi: target %d: %s", t, why);
            return VSG_ERR_INVALID;
        }
    CK(cudaSetDevice(m->device));
    std::vector<BowWalk> walks;
    std::vector<BowSeg> segs;
    std::vector<int> seg_ptr(1, 0);
    int64_t npairs = 0;
    for (int t = 0; t < ntargets; ++t) {
        const vsg_bow_side &b = *KF2s[t];
        walks.push_back(BowWalk{&KF1->view, KF1->mp_valid, FeatVec{KF1->nnodes, KF1->nodes, KF1->ptr, KF1->idx}, &b.view,
                                FeatVec{b.nnodes, b.nodes, b.ptr, b.idx}});
        if (bow_walk(walks.back(), segs, &npairs) != VSG_OK) {
            const std::string err = vsg_last_error();
            set_error("vsg_search_by_bow_kf_multi: target %d: %s", t, err.c_str());
            return VSG_ERR_INVALID;
        }
        seg_ptr.push_back((int)segs.size());
    }
    const uint16_t *dist;
    vsg_status st = bow_dists(m, ntargets, walks.data(), segs, seg_ptr.data(), npairs, &dist);
    if (st != VSG_OK) return st;
    for (int t = 0; t < ntargets; ++t)                                               // in target order, as the loop runs
        nmatches_out[t] = bow_replay_kf(&KF1->view, &KF2s[t]->view, KF2s[t]->mp_valid, walks[t].b, segs.data() + seg_ptr[t],
                                        seg_ptr[t + 1] - seg_ptr[t], dist, nnratio, check_ori,
                                        matches12_out + (size_t)t * KF1->view.n);
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
    const BowWalk w{KF1, use1, FeatVec{nnodes1, nodes1, ptr1, idx1}, KF2, FeatVec{nnodes2, nodes2, ptr2, idx2}};
    std::vector<BowSeg> segs;
    int64_t npairs = 0;
    const uint16_t *dist;
    vsg_status st = bow_walk(w, segs, &npairs);
    const int seg_ptr[2] = {0, (int)segs.size()};
    if (st != VSG_OK || (st = bow_dists(m, 1, &w, segs, seg_ptr, npairs, &dist)) != VSG_OK) return st;
    *nq_out = (int)segs.size();
    *total_out = (int)npairs;
    if ((int)segs.size() > q_capacity || npairs > capacity) return VSG_ERR_CAPACITY;
    if ((!segs.empty() && (!q1_out || !cand_ptr_out)) || (npairs && (!cand_idx2_out || !cand_dist_out))) return VSG_ERR_INVALID;
    for (size_t k = 0; k < segs.size(); ++k) {
        const BowSeg &sg = segs[k];
        q1_out[k] = sg.i1;
        cand_ptr_out[k] = sg.off;
        for (int j = sg.jb; j < sg.je; ++j) {
            cand_idx2_out[sg.off + j - sg.jb] = idx2[j];
            cand_dist_out[sg.off + j - sg.jb] = dist[sg.off + j - sg.jb];
        }
    }
    if (cand_ptr_out) cand_ptr_out[segs.size()] = (int)npairs;
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
    std::vector<uint8_t> use1(KF1->n);
    for (int i = 0; i < KF1->n; ++i) use1[i] = !has_mp1[i] && (!only_stereo || stereo1(i));   // :971-981
    const BowWalk w{KF1, use1.data(), FeatVec{nnodes1, nodes1, ptr1, idx1}, KF2, FeatVec{nnodes2, nodes2, ptr2, idx2}};
    std::vector<BowSeg> segs;
    int64_t npairs = 0;
    const uint16_t *dist;
    vsg_status st = bow_walk(w, segs, &npairs);
    const int seg_ptr[2] = {0, (int)segs.size()};
    if (st != VSG_OK || (st = bow_dists(m, 1, &w, segs, seg_ptr, npairs, &dist)) != VSG_OK) return st;
    for (int i = 0; i < KF1->n; ++i) matches12_out[i] = -1;
    std::vector<int> rot_hist[HISTO_LENGTH];
    int nmatches = 0;
    for (const BowSeg &sg : segs) {
        const int i1 = sg.i1;
        const vsg_keypoint &kp1 = KF1->keys[i1];
        const bool b_stereo1 = stereo1(i1);
        int best = TH_LOW, best_idx2 = -1;
        for (int j = sg.jb; j < sg.je; ++j) {
            const int i2 = idx2[j];
            if (has_mp2[i2]) continue;                                               // :1001 (vbMatched2 is never set, SURVEY C#3)
            const bool b_stereo2 = stereo2(i2);
            if (only_stereo && !b_stereo2) continue;
            const int d = dist[sg.off + j - sg.jb];
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
