"""Python mirror of the arithmetic of VS_GRAPHS::ORBmatcher (reference orb_slam3/include/ORBmatcher.h:34-99)
over the C ABI, on flattened arrays.  Used by tests and bench.py; C++ hosts use shim/ORBmatcher.h.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import PROJ_POINT_DTYPE, SEARCH_POINT_DTYPE, TRACK_POINT_DTYPE, BowSide, check, ptr
from .frame import DeviceFrame, FrameData

TH_HIGH = 100     # ORBmatcher.cc:34
TH_LOW = 50       # ORBmatcher.cc:35
HISTO_LENGTH = 30  # ORBmatcher.cc:36


def projection_map_resolve(frame_data, occupied, track_points, cand_ptr, cand_idx, cand_dist, nnratio):
    """vsg_projection_map_resolve: host code, needs no CUDA device (every rank runs it after the all-gather)."""
    L = _lib.load()
    pts = np.ascontiguousarray(track_points, TRACK_POINT_DTYPE)
    occupied = np.ascontiguousarray(occupied, np.uint8)
    cand_ptr, cand_idx, cand_dist = (np.ascontiguousarray(a, np.int32) for a in (cand_ptr, cand_idx, cand_dist))
    assign = np.zeros(frame_data.n, np.int32)
    nm = C.c_int(0)
    check(L.vsg_projection_map_resolve(C.byref(frame_data.view), ptr(occupied), len(pts), ptr(pts), ptr(cand_ptr),
                                       ptr(cand_idx), ptr(cand_dist), float(np.float32(nnratio)), ptr(assign), C.byref(nm)))
    return nm.value, assign


def projection_map_resolve_shard(frame_data, blocked, assign, shard_begin, track_points_local, cand_ptr, cand_idx, cand_dist,
                                 nnratio):
    """vsg_projection_map_resolve_shard: one shard's replay from the claim state `blocked` (updated in place, like
    `assign`).  Host code.  Returns this shard's nmatches."""
    L = _lib.load()
    pts = np.ascontiguousarray(track_points_local, TRACK_POINT_DTYPE)
    cand_ptr, cand_idx, cand_dist = (np.ascontiguousarray(a, np.int32) for a in (cand_ptr, cand_idx, cand_dist))
    assert blocked.dtype == np.uint8 and assign.dtype == np.int32 and blocked.flags.c_contiguous and assign.flags.c_contiguous
    nm = C.c_int(0)
    check(L.vsg_projection_map_resolve_shard(C.byref(frame_data.view), ptr(blocked), int(shard_begin), len(pts), ptr(pts),
                                             ptr(cand_ptr), ptr(cand_idx), ptr(cand_dist), float(np.float32(nnratio)),
                                             ptr(assign), C.byref(nm)))
    return nm.value


def _bow_side(data, mp_valid, featvec, keep):
    """A vsg_bow_side for (FrameData, map-point flags or None, (nodes, ptr, idx)); the arrays it points to go into `keep`."""
    nodes, ptr_, idx = (np.ascontiguousarray(a, np.int32) for a in featvec)
    valid = None if mp_valid is None else np.ascontiguousarray(mp_valid, np.uint8)
    keep.extend([data, nodes, ptr_, idx, valid])
    return BowSide(data.view, ptr(valid), len(nodes), ptr(nodes), ptr(ptr_), ptr(idx))


def _side_table(sides):
    """const vsg_bow_side *const[] over `sides` (the structs stay referenced by the returned table's owner)."""
    return (C.c_void_p * max(len(sides), 1))(*[C.addressof(s) for s in sides])


class ORBmatcher:
    def __init__(self, nnratio=0.6, checkOri=True, device=0):
        self._L = _lib.load()
        self._h = C.c_void_p()
        self.mfNNratio = np.float32(nnratio)
        self.mbCheckOrientation = bool(checkOri)
        check(self._L.vsg_matcher_create(device, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            self._L.vsg_matcher_destroy(self._h)
            self._h = None

    __del__ = close

    def stream(self):
        return self._L.vsg_matcher_stream(self._h)

    def sync(self):
        check(self._L.vsg_matcher_sync(self._h))

    def DescriptorDistance(self, a, b):
        """ORBmatcher.cc:2047-2063 for n pairs (rows of 32 bytes)."""
        a = np.ascontiguousarray(a, np.uint8).reshape(-1, 32)
        b = np.ascontiguousarray(b, np.uint8).reshape(-1, 32)
        assert a.shape == b.shape
        out = np.zeros(a.shape[0], np.int32)
        check(self._L.vsg_descriptor_distance(self._h, ptr(a), ptr(b), a.shape[0], ptr(out)))
        return out

    def knn2(self, query, train, train_index_offset=0):
        """Brute-force top-2 (Frame.cc:1200 semantics). Returns (idx [nq,2], dist [nq,2])."""
        query = np.ascontiguousarray(query, np.uint8).reshape(-1, 32)
        train = np.ascontiguousarray(train, np.uint8).reshape(-1, 32)
        nq, nt = query.shape[0], train.shape[0]
        idx = np.zeros((nq, 2), np.int32)
        dist = np.zeros((nq, 2), np.int32)
        check(self._L.vsg_knn2(self._h, ptr(query), nq, ptr(train), nt, train_index_offset, ptr(idx), ptr(dist)))
        return idx, dist

    def knn2_dev(self, query_dev, train_dev, idx_dev, dist_dev, train_index_offset=0):
        """torch CUDA tensors: query (nq,32) u8, train (nt,32) u8, idx/dist (nq,2) int32. Async on the matcher stream."""
        check(self._L.vsg_knn2_dev(self._h, ptr(query_dev), query_dev.shape[0], ptr(train_dev), train_dev.shape[0],
                                   train_index_offset, ptr(idx_dev), ptr(dist_dev)))

    def knn2_merge_dev(self, idx_parts_dev, dist_parts_dev, out_idx_dev, out_dist_dev):
        """Merge (nparts, nq, 2) per-shard top-2 lists into (nq, 2)."""
        nparts, nq = idx_parts_dev.shape[0], idx_parts_dev.shape[1]
        check(self._L.vsg_knn2_merge_dev(self._h, ptr(idx_parts_dev), ptr(dist_parts_dev), nparts, nq,
                                         ptr(out_idx_dev), ptr(out_dist_dev)))

    def ComputeDistinctiveDescriptors(self, descriptors, ptr_):
        """MapPoint::ComputeDistinctiveDescriptors (MapPoint.cc:340-417) for many map points: descriptors (total, 32),
        ptr_ (npoints + 1) CSR offsets. Returns best row per point (relative to its first row; -1 if it has none)."""
        descriptors = np.ascontiguousarray(descriptors, np.uint8).reshape(-1, 32)
        ptr_ = np.ascontiguousarray(ptr_, np.int32)
        best = np.zeros(len(ptr_) - 1, np.int32)
        check(self._L.vsg_distinctive_descriptors(self._h, ptr(descriptors), ptr(ptr_), len(best), ptr(best)))
        return best

    def knn2_ratio(self, query, train, ratio=0.7):
        """knnMatch(k=2) + Lowe ratio of Frame::ComputeStereoFishEyeMatches (Frame.cc:1200-1208) -> (match, dist)."""
        query = np.ascontiguousarray(query, np.uint8).reshape(-1, 32)
        train = np.ascontiguousarray(train, np.uint8).reshape(-1, 32)
        match = np.zeros(len(query), np.int32)
        dist = np.zeros(len(query), np.int32)
        check(self._L.vsg_knn2_ratio(self._h, ptr(query), len(query), ptr(train), len(train), float(ratio), ptr(match),
                                     ptr(dist)))
        return match, dist

    def match_window(self, query, train, cand_ptr, cand, skip=None, train_level=None, init_dist=256):
        """Best / second-best over per-query candidate lists (ORBmatcher.cc:77-120 idiom).
        Returns dict(best_idx, best_dist, second_dist, best_level, second_level)."""
        query = np.ascontiguousarray(query, np.uint8).reshape(-1, 32)
        train = np.ascontiguousarray(train, np.uint8).reshape(-1, 32)
        cand_ptr = np.ascontiguousarray(cand_ptr, np.int32)
        cand = np.ascontiguousarray(cand, np.int32)
        nq, nt = query.shape[0], train.shape[0]
        assert cand_ptr.shape[0] == nq + 1
        if skip is not None:
            skip = np.ascontiguousarray(skip, np.uint8)
        if train_level is not None:
            train_level = np.ascontiguousarray(train_level, np.int32)
        out = {k: np.zeros(nq, np.int32) for k in ("best_idx", "best_dist", "second_dist", "best_level", "second_level")}
        check(self._L.vsg_match_window(self._h, ptr(query), nq, ptr(train), nt, ptr(cand_ptr), ptr(cand), ptr(skip),
                                       ptr(train_level), int(init_dist), ptr(out["best_idx"]), ptr(out["best_dist"]),
                                       ptr(out["second_dist"]), ptr(out["best_level"]), ptr(out["second_level"])))
        return out

    # ---- Search* methods on flattened views (single-camera branches) ----
    def frame(self, data):
        """Upload a FrameData and build its grid (Frame::AssignFeaturesToGrid)."""
        return DeviceFrame(self, data)

    def area_search(self, frame, qx, qy, qr, min_level, max_level, qdesc):
        """Frame::GetFeaturesInArea for many windows at once -> (cand_ptr, cand_idx, cand_dist)."""
        qx, qy, qr = (np.ascontiguousarray(a, np.float32) for a in (qx, qy, qr))
        min_level, max_level = (np.ascontiguousarray(a, np.int32) for a in (min_level, max_level))
        qdesc = np.ascontiguousarray(qdesc, np.uint8).reshape(-1, 32)
        nq = len(qx)
        cand_ptr = np.zeros(nq + 1, np.int32)
        cap = max(1024, nq * 64)
        while True:
            idx, dist, total = np.zeros(cap, np.int32), np.zeros(cap, np.int32), C.c_int(0)
            st = self._L.vsg_area_search(self._h, frame._h, nq, ptr(qx), ptr(qy), ptr(qr), ptr(min_level),
                                         ptr(max_level), ptr(qdesc), ptr(cand_ptr), ptr(idx), ptr(dist), cap,
                                         C.byref(total))
            if st == _lib.VSG_ERR_CAPACITY:
                cap = total.value
                continue
            check(st)
            return cand_ptr, idx[: total.value].copy(), dist[: total.value].copy()

    def SearchByProjectionMap(self, frame, occupied, track_points, mp_desc, th=3.0, bFarPoints=False,
                              thFarPoints=50.0):
        """SearchByProjection(Frame&, vector<MapPoint*>&, th, bFarPoints, thFarPoints) (ORBmatcher.cc:42-144).
        Returns (nmatches, assign[N])."""
        pts = np.ascontiguousarray(track_points, TRACK_POINT_DTYPE)
        mp_desc = np.ascontiguousarray(mp_desc, np.uint8).reshape(-1, 32)
        occupied = np.ascontiguousarray(occupied, np.uint8)
        assign = np.zeros(frame.data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_by_projection_map(self._h, frame._h, ptr(occupied), len(pts), ptr(pts), ptr(mp_desc),
                                                   float(th), int(bFarPoints), float(thFarPoints),
                                                   float(self.mfNNratio), ptr(assign), C.byref(nm)))
        return nm.value, assign

    def SearchByProjectionMap2Cam(self, frame_l, frame_r, occupied, left_to_right, right_to_left, pts_left, pts_right,
                                  mp_desc, th=3.0, bFarPoints=False, thFarPoints=50.0):
        """The same method on a two-camera frame (F.Nleft != -1; ORBmatcher.cc:42-216 incl. the right-camera branch):
        frame_l / frame_r hold mvKeys / mvKeysRight with their descriptor rows, occupied and the returned assign have
        Nleft + Nright slots (left first).  Returns (nmatches, assign)."""
        pl = np.ascontiguousarray(pts_left, TRACK_POINT_DTYPE)
        pr = np.ascontiguousarray(pts_right, TRACK_POINT_DTYPE)
        assert len(pl) == len(pr)
        mp_desc = np.ascontiguousarray(mp_desc, np.uint8).reshape(-1, 32)
        occupied = np.ascontiguousarray(occupied, np.uint8)
        l2r = np.ascontiguousarray(left_to_right, np.int32)
        r2l = np.ascontiguousarray(right_to_left, np.int32)
        assign = np.zeros(frame_l.data.n + frame_r.data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_by_projection_map_2cam(self._h, frame_l._h, frame_r._h, ptr(occupied), ptr(l2r), ptr(r2l),
                                                        len(pl), ptr(pl), ptr(pr), ptr(mp_desc), float(th), int(bFarPoints),
                                                        float(thFarPoints), float(self.mfNNratio), ptr(assign), C.byref(nm)))
        return nm.value, assign

    def ProjectionMapCandidates(self, frame, track_points, mp_desc, th=3.0, bFarPoints=False, thFarPoints=50.0):
        """GPU half of SearchByProjection(Frame&, vector<MapPoint*>&): per-map-point candidate lists
        (cand_ptr [n+1], cand_idx, cand_dist) in the reference's order (vsg_projection_map_candidates)."""
        pts = np.ascontiguousarray(track_points, TRACK_POINT_DTYPE)
        mp_desc = np.ascontiguousarray(mp_desc, np.uint8).reshape(-1, 32)
        cand_ptr = np.zeros(len(pts) + 1, np.int32)
        cap = max(1024, len(pts) * 16)
        while True:
            idx, dist, total = np.zeros(cap, np.int32), np.zeros(cap, np.int32), C.c_int(0)
            st = self._L.vsg_projection_map_candidates(self._h, frame._h, len(pts), ptr(pts), ptr(mp_desc), float(th),
                                                       int(bFarPoints), float(thFarPoints), ptr(cand_ptr), ptr(idx),
                                                       ptr(dist), cap, C.byref(total))
            if st == _lib.VSG_ERR_CAPACITY:
                cap = total.value
                continue
            check(st)
            return cand_ptr, idx[: total.value].copy(), dist[: total.value].copy()

    def knn2_sharded(self, comm, query_dev, train_shard_dev, train_index_offset, out_idx_dev, out_dist_dev):
        """vsg_knn2_sharded: train rows sharded over the communicator's ranks (torch CUDA tensors; asynchronous)."""
        check(self._L.vsg_knn2_sharded(comm._h, self._h, ptr(query_dev), query_dev.shape[0], ptr(train_shard_dev),
                                       train_shard_dev.shape[0], int(train_index_offset), ptr(out_idx_dev), ptr(out_dist_dev)))

    def SearchByProjectionMapSharded(self, comm, frame, occupied, shard_begin, track_points_local, desc_local, th=3.0,
                                     bFarPoints=False, thFarPoints=50.0):
        """vsg_search_by_projection_map_sharded: this rank's contiguous shard of the map points; returns the
        (nmatches, assign[N]) of the one-call method on the whole map, assign holding global map point indices."""
        pts = np.ascontiguousarray(track_points_local, TRACK_POINT_DTYPE)
        desc = np.ascontiguousarray(desc_local, np.uint8).reshape(-1, 32)
        occupied = np.ascontiguousarray(occupied, np.uint8)
        assign = np.zeros(frame.data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_by_projection_map_sharded(comm._h, self._h, frame._h, ptr(occupied), int(shard_begin), len(pts),
                                                           ptr(pts), ptr(desc), float(th), int(bFarPoints), float(thFarPoints),
                                                           float(self.mfNNratio), ptr(assign), C.byref(nm)))
        return nm.value, assign

    def ProjectionMapResolve(self, frame_data, occupied, track_points, cand_ptr, cand_idx, cand_dist):
        """Host half: the order-dependent replay of ORBmatcher.cc:76-141 (vsg_projection_map_resolve)."""
        return projection_map_resolve(frame_data, occupied, track_points, cand_ptr, cand_idx, cand_dist, self.mfNNratio)

    def SearchByProjectionLast(self, cur_frame, occupied, proj_points, desc, th, mode=0):
        """SearchByProjection(Frame& Cur, const Frame& Last, th, bMono) (ORBmatcher.cc:1667-1878) with the
        projection done by the caller. Returns (nmatches, assign[N])."""
        pts = np.ascontiguousarray(proj_points, PROJ_POINT_DTYPE)
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        occupied = np.ascontiguousarray(occupied, np.uint8)
        assign = np.zeros(cur_frame.data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_by_projection_last(self._h, cur_frame._h, ptr(occupied), len(pts), ptr(pts), ptr(desc),
                                                    float(th), int(mode), int(self.mbCheckOrientation), ptr(assign),
                                                    C.byref(nm)))
        return nm.value, assign

    def SearchByProjectionLast2Cam(self, cur_l, cur_r, occupied, pts_left, pts_right, desc, th, mode=0):
        """The same with a two-camera current frame (CurrentFrame.Nleft != -1; ORBmatcher.cc:1667-1878 incl. :1785-1852):
        pts_right carries the projections into the right camera (u, v). Returns (nmatches, assign[Nleft + Nright])."""
        pl = np.ascontiguousarray(pts_left, PROJ_POINT_DTYPE)
        pr = np.ascontiguousarray(pts_right, PROJ_POINT_DTYPE)
        assert len(pl) == len(pr)
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        occupied = np.ascontiguousarray(occupied, np.uint8)
        assign = np.zeros(cur_l.data.n + cur_r.data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_by_projection_last_2cam(self._h, cur_l._h, cur_r._h, ptr(occupied), len(pl), ptr(pl), ptr(pr),
                                                         ptr(desc), float(th), int(mode), int(self.mbCheckOrientation),
                                                         ptr(assign), C.byref(nm)))
        return nm.value, assign

    def SearchForInitialization(self, f1_data, f2_frame, prev_matched, windowSize=10):
        """ORBmatcher.cc:643-756. prev_matched (n1, 2) float32 is updated in place. Returns (nmatches, matches12)."""
        assert prev_matched.dtype == np.float32 and prev_matched.flags["C_CONTIGUOUS"]
        m12 = np.zeros(f1_data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_for_initialization(self._h, C.byref(f1_data.view), f2_frame._h, ptr(prev_matched),
                                                    int(windowSize), float(self.mfNNratio),
                                                    int(self.mbCheckOrientation), ptr(m12), C.byref(nm)))
        return nm.value, m12

    def SearchByBoW(self, kf_data, kf_mp_valid, f_data, kf_featvec, f_featvec, f_nleft=-1):
        """SearchByBoW(KeyFrame*, Frame&, ...) (ORBmatcher.cc:226-428). Feature vectors are (nodes, ptr, idx)
        triples with sorted node ids; f_nleft != -1: F is a two-camera frame (left features first).
        Returns (nmatches, matches_f[F.N])."""
        kn, kp, ki = (np.ascontiguousarray(a, np.int32) for a in kf_featvec)
        fn, fp, fi = (np.ascontiguousarray(a, np.int32) for a in f_featvec)
        valid = np.ascontiguousarray(kf_mp_valid, np.uint8)
        out = np.zeros(f_data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_by_bow_2cam(self._h, C.byref(kf_data.view), ptr(valid), C.byref(f_data.view), int(f_nleft),
                                             len(kn), ptr(kn), ptr(kp), ptr(ki), len(fn), ptr(fn), ptr(fp), ptr(fi),
                                             float(self.mfNNratio), int(self.mbCheckOrientation), ptr(out), C.byref(nm)))
        return nm.value, out

    def SearchByBoWMulti(self, targets, f_data, f_featvec, f_nleft=-1):
        """SearchByBoW with one frame against many keyframes (Tracking::Relocalization's loop over its candidates) in one
        upload, one launch and one download: targets is a list of (kf_data, kf_mp_valid, kf_featvec).  Returns
        (nmatches[T], matches_f[T, F.N]), target for target what SearchByBoW returns."""
        keep = []
        sides = [_bow_side(d, v, fv, keep) for d, v, fv in targets]
        F = _bow_side(f_data, None, f_featvec, keep)
        T = len(sides)
        out = np.zeros((T, f_data.n), np.int32)
        nm = np.zeros(T, np.int32)
        check(self._L.vsg_search_by_bow_multi(self._h, T, _side_table(sides), C.byref(F), int(f_nleft), float(self.mfNNratio),
                                              int(self.mbCheckOrientation), ptr(out), ptr(nm)))
        return nm, out

    def SearchByProjectionReloc(self, cur_frame, occupied, search_points, desc, th, ORBdist):
        """SearchByProjection(Frame&, KeyFrame*, sAlreadyFound, th, ORBdist) (ORBmatcher.cc:1880-2000) with the
        projection done by the caller. Returns (nmatches, assign[N])."""
        pts = np.ascontiguousarray(search_points, SEARCH_POINT_DTYPE)
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        occupied = np.ascontiguousarray(occupied, np.uint8)
        assign = np.zeros(cur_frame.data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_by_projection_reloc(self._h, cur_frame._h, ptr(occupied), len(pts), ptr(pts), ptr(desc),
                                                     float(th), int(ORBdist), int(self.mbCheckOrientation),
                                                     ptr(assign), C.byref(nm)))
        return nm.value, assign

    def SearchByProjectionSim3(self, kf_frame, matched, search_points, desc, th, ratioHamming=1.0):
        """SearchByProjection(KeyFrame*, Sim3f&, vpPoints[, vpPointsKFs], vpMatched, th, ratioHamming)
        (ORBmatcher.cc:430-641). Returns (nmatches, assign[N])."""
        pts = np.ascontiguousarray(search_points, SEARCH_POINT_DTYPE)
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        matched = np.ascontiguousarray(matched, np.uint8)
        assign = np.zeros(kf_frame.data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_by_projection_sim3(self._h, kf_frame._h, ptr(matched), len(pts), ptr(pts), ptr(desc),
                                                    int(th), float(ratioHamming), ptr(assign), C.byref(nm)))
        return nm.value, assign

    def FuseSearch(self, kf_frame, search_points, desc, th, inv_level_sigma2=None, sim3_variant=False):
        """The search of Fuse(KeyFrame*, vpMapPoints, th) (ORBmatcher.cc:1148-1335) or, with sim3_variant, of
        Fuse(KeyFrame*, Sim3f&, ...) (:1337-1446). Returns (nFused, best_idx[n])."""
        pts = np.ascontiguousarray(search_points, SEARCH_POINT_DTYPE)
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        sig = None if inv_level_sigma2 is None else np.ascontiguousarray(inv_level_sigma2, np.float32)
        best = np.zeros(len(pts), np.int32)
        nf = C.c_int(0)
        check(self._L.vsg_fuse_search(self._h, kf_frame._h, len(pts), ptr(pts), ptr(desc), float(th), ptr(sig),
                                      int(bool(sim3_variant)), ptr(best), C.byref(nf)))
        return nf.value, best

    def fuse_search_multi(self, kf_frames, inv_level_sigma2s, search_points, desc, th=3.0):
        """FuseSearch (the pose-based variant) into every keyframe of kf_frames with one upload, one launch and one
        download: search_points is [ntargets][n] (the points projected into each target), desc (n x 32) is shared, and
        inv_level_sigma2s holds one table per target. Returns best_idx[ntargets][n]."""
        T = len(kf_frames)
        if len(inv_level_sigma2s) != T:
            raise ValueError("fuse_search_multi: %d targets but %d level tables" % (T, len(inv_level_sigma2s)))
        desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        n = len(desc)
        pts = np.ascontiguousarray(search_points, SEARCH_POINT_DTYPE).reshape(T, n)
        sigs = [np.ascontiguousarray(s, np.float32) for s in inv_level_sigma2s]
        frames = (C.c_void_p * max(T, 1))(*[f._h.value for f in kf_frames])
        sig_ptrs = (C.c_void_p * max(T, 1))(*[s.ctypes.data for s in sigs])
        best = np.zeros((T, n), np.int32)
        check(self._L.vsg_fuse_search_multi(self._h, T, frames, sig_ptrs, n, ptr(pts), ptr(desc), float(th), ptr(best)))
        return best

    def SearchBySim3(self, kf1_frame, kf2_frame, pts1, desc1, pts2, desc2, th):
        """ORBmatcher.cc:1448-1665 with both projections done by the caller. Returns (nFound, matches12[N1])."""
        pts1 = np.ascontiguousarray(pts1, SEARCH_POINT_DTYPE)
        pts2 = np.ascontiguousarray(pts2, SEARCH_POINT_DTYPE)
        desc1 = np.ascontiguousarray(desc1, np.uint8).reshape(-1, 32)
        desc2 = np.ascontiguousarray(desc2, np.uint8).reshape(-1, 32)
        m12 = np.zeros(len(pts1), np.int32)
        nf = C.c_int(0)
        check(self._L.vsg_search_by_sim3(self._h, kf1_frame._h, kf2_frame._h, len(pts1), ptr(pts1), ptr(desc1), len(pts2),
                                         ptr(pts2), ptr(desc2), float(th), ptr(m12), C.byref(nf)))
        return nf.value, m12

    def SearchByBoWKF(self, kf1_data, mp_valid1, kf2_data, mp_valid2, featvec1, featvec2):
        """SearchByBoW(KeyFrame*, KeyFrame*, vpMatches12) (ORBmatcher.cc:758-900). Returns (nmatches, matches12[N1])."""
        n1, p1, i1 = (np.ascontiguousarray(a, np.int32) for a in featvec1)
        n2, p2, i2 = (np.ascontiguousarray(a, np.int32) for a in featvec2)
        v1, v2 = np.ascontiguousarray(mp_valid1, np.uint8), np.ascontiguousarray(mp_valid2, np.uint8)
        out = np.zeros(kf1_data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_by_bow_kf(self._h, C.byref(kf1_data.view), ptr(v1), C.byref(kf2_data.view), ptr(v2),
                                           len(n1), ptr(n1), ptr(p1), ptr(i1), len(n2), ptr(n2), ptr(p2), ptr(i2),
                                           float(self.mfNNratio), int(self.mbCheckOrientation), ptr(out), C.byref(nm)))
        return nm.value, out

    def SearchByBoWKFMulti(self, kf1_data, mp_valid1, featvec1, targets):
        """SearchByBoWKF of one keyframe against many (LoopClosing::DetectCommonRegionsFromBoW's loop over the candidates
        and their covisibles) in one upload, one launch and one download: targets is a list of (kf2_data, mp_valid2,
        featvec2).  Returns (nmatches[T], matches12[T, N1]), target for target what SearchByBoWKF returns."""
        keep = []
        K1 = _bow_side(kf1_data, mp_valid1, featvec1, keep)
        sides = [_bow_side(d, v, fv, keep) for d, v, fv in targets]
        T = len(sides)
        out = np.zeros((T, kf1_data.n), np.int32)
        nm = np.zeros(T, np.int32)
        check(self._L.vsg_search_by_bow_kf_multi(self._h, C.byref(K1), T, _side_table(sides), float(self.mfNNratio),
                                                 int(self.mbCheckOrientation), ptr(out), ptr(nm)))
        return nm, out

    def SearchForTriangulation(self, kf1_data, has_mp1, kf2_data, has_mp2, featvec1, featvec2, F12, ep, level_sigma2_2,
                               bOnlyStereo=False, bCoarse=False):
        """ORBmatcher.cc:902-1146 (single pinhole camera). Returns (nmatches, matches12[N1])."""
        n1, p1, i1 = (np.ascontiguousarray(a, np.int32) for a in featvec1)
        n2, p2, i2 = (np.ascontiguousarray(a, np.int32) for a in featvec2)
        h1, h2 = np.ascontiguousarray(has_mp1, np.uint8), np.ascontiguousarray(has_mp2, np.uint8)
        F12 = np.ascontiguousarray(F12, np.float32).reshape(9)
        ep = np.ascontiguousarray(ep, np.float32).reshape(2)
        sig = np.ascontiguousarray(level_sigma2_2, np.float32)
        out = np.zeros(kf1_data.n, np.int32)
        nm = C.c_int(0)
        check(self._L.vsg_search_for_triangulation(self._h, C.byref(kf1_data.view), ptr(h1), C.byref(kf2_data.view), ptr(h2),
                                                   len(n1), ptr(n1), ptr(p1), ptr(i1), len(n2), ptr(n2), ptr(p2), ptr(i2),
                                                   int(bOnlyStereo), int(bCoarse), ptr(F12), ptr(ep), ptr(sig),
                                                   int(self.mbCheckOrientation), ptr(out), C.byref(nm)))
        return nm.value, out

    def ComputeStereoMatches(self, ex_left, ex_right, keys_l, desc_l, keys_r, desc_r, mb, mbf, frame_l=0, frame_r=0):
        """Frame::ComputeStereoMatches (Frame.cc:957-1127) on the device pyramids of the two extractors' last call.
        Returns (mvuRight, mvDepth) float32 arrays."""
        from ._lib import KEYPOINT_DTYPE
        keys_l = np.ascontiguousarray(keys_l, KEYPOINT_DTYPE)
        keys_r = np.ascontiguousarray(keys_r, KEYPOINT_DTYPE)
        desc_l = np.ascontiguousarray(desc_l, np.uint8).reshape(-1, 32)
        desc_r = np.ascontiguousarray(desc_r, np.uint8).reshape(-1, 32)
        u_right = np.zeros(len(keys_l), np.float32)
        depth = np.zeros(len(keys_l), np.float32)
        check(self._L.vsg_stereo_match(self._h, ex_left._h, ex_right._h, frame_l, frame_r, ptr(keys_l), ptr(desc_l),
                                       len(keys_l), ptr(keys_r), ptr(desc_r), len(keys_r), float(mb), float(mbf),
                                       ptr(u_right), ptr(depth)))
        return u_right, depth

    def UndistortKeyPoints(self, xy, K, dist):
        """Frame::UndistortKeyPoints (Frame.cc:891-922): cv::undistortPoints(xy, mK, mDistCoef, cv::Mat(), mK) on an
        (n, 2) float32 array; K is the 3x3 calibration matrix, dist the distortion coefficients (float32 values, as
        the reference stores them)."""
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        K = np.asarray(K, np.float64)
        dist = np.ascontiguousarray(np.asarray(dist, np.float64).ravel())
        out = np.empty_like(xy)
        check(self._L.vsg_undistort_keypoints(self._h, xy.shape[0], ptr(xy), float(K[0, 0]), float(K[1, 1]), float(K[0, 2]),
                                              float(K[1, 2]), ptr(dist), dist.size, ptr(out)))
        return out

    def UndistortKeyPointsBatch(self, ex, nframes, K, dist):
        """The same on the device-resident keypoints of the extractor's last extract_batch call: (nframes, cap, 2)."""
        cap = self._L.vsg_extractor_max_keypoints(ex._h, *ex.level_size(0))
        K = np.asarray(K, np.float64)
        dist = np.ascontiguousarray(np.asarray(dist, np.float64).ravel())
        out = np.empty((nframes, cap, 2), np.float32)
        check(self._L.vsg_undistort_keypoints_batch(self._h, ex._h, int(nframes), float(K[0, 0]), float(K[1, 1]),
                                                    float(K[0, 2]), float(K[1, 2]), ptr(dist), dist.size, ptr(out), cap))
        return out

    @staticmethod
    def ComputeStereoFromRGBD(xy, xy_un, depth, bf):
        """Frame::ComputeStereoFromRGBD (Frame.cc:1129-1150): a gather of one depth value per keypoint — host glue,
        no device work.  Returns (mvuRight, mvDepth), -1 where the depth is not positive."""
        xy = np.asarray(xy, np.float32).reshape(-1, 2)
        xy_un = np.asarray(xy_un, np.float32).reshape(-1, 2)
        depth = np.asarray(depth, np.float32)
        d = depth[xy[:, 1].astype(np.int32), xy[:, 0].astype(np.int32)]
        ok = d > 0
        safe = np.where(ok, d, np.float32(1))
        u_right = np.where(ok, xy_un[:, 0] - np.float32(bf) / safe, np.float32(-1)).astype(np.float32)
        return u_right, np.where(ok, d, np.float32(-1)).astype(np.float32)

    def ComputeStereoMatchesBatch(self, ex, npairs, mb, mbf):
        """Frame::ComputeStereoMatches for pairs (2p, 2p+1) of the extractor's last extract_batch call, on its
        device-resident results. Returns (u_right, depth) float32 arrays of shape (npairs, cap)."""
        cap = self._L.vsg_extractor_max_keypoints(ex._h, *ex.level_size(0))
        u = np.zeros((npairs, cap), np.float32)
        d = np.zeros((npairs, cap), np.float32)
        check(self._L.vsg_stereo_match_batch(self._h, ex._h, int(npairs), float(mb), float(mbf), ptr(u), ptr(d), cap))
        return u, d
