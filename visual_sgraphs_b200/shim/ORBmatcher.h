// ORBmatcher.h — drop-in for the reference's orb_slam3/include/ORBmatcher.h (snt-arg/visual_sgraphs):
// VS_GRAPHS::ORBmatcher with the same constructor, constants, static DescriptorDistance and the Search*
// methods named by the north star, forwarding to the CUDA library (include/vsg_cuda.h).
//
// The reference's methods take Frame&, KeyFrame*, MapPoint* — classes that live outside the hot path
// (they pull in Eigen, Sophus, PCL, DBoW2).  To stay source compatible without depending on those
// headers, the methods are member templates: the argument types are deduced at the reference's call
// sites (Tracking.cc:2555, 2790, 2926, 3423 ...) and only the members the reference's own
// implementation reads are touched (same names: N, Nleft, mvKeysUn, mDescriptors, mvuRight, mvpMapPoints,
// mvScaleFactors, mnMinX ..., mfGridElementWidthInv ..., mFeatVec, GetPose(), mpCamera->project(),
// MapPoint::{mbTrackInView, mTrackProjX, ..., isBad(), Observations(), GetDescriptor(), GetWorldPos()}).
// Each template flattens those members into the C ABI's view structs, calls the library and writes the
// results back exactly where the reference does.
//
// Scope: all 13 methods for single-camera frames (Frame::Nleft == -1) and for two-camera frames / keyframes (Nleft != -1,
// stereo-fisheye rigs): the methods with two-camera code of their own (SearchByProjection(Frame&, vector<MapPoint*>&),
// SearchByProjection(Frame&, const Frame&), SearchByBoW x 2, Fuse(..., bRight), SearchForTriangulation) follow it branch
// by branch; the others (relocalisation / Sim3 projections, SearchBySim3, Fuse(KF, Scw, ...)) search the left camera, as
// the reference's GetFeaturesInArea(..., bRight = false) does.  Every method is compared with the reference's own
// ORBmatcher.cc in tests/cpp/ref_matcher_test.cpp.
#ifndef VSG_SHIM_ORBMATCHER_H
#define VSG_SHIM_ORBMATCHER_H

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <set>
#include <tuple>
#include <type_traits>
#include <utility>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/vsg_cuda.h"
#include "cv_compat.h"

#ifndef FRAME_GRID_ROWS
#define FRAME_GRID_ROWS 48
#define FRAME_GRID_COLS 64
#endif

namespace VS_GRAPHS {

class ORBmatcher {
public:
    // Stateless like the reference's class (two members, ORBmatcher.h:97-98): copyable, cheap to construct on the stack per call
    // as Tracking / LocalMapping / LoopClosing do.  The CUDA stream and scratch buffers live in one workspace per calling
    // thread (below), not in the object.
    ORBmatcher(float nnratio = 0.6, bool checkOri = true) : mfNNratio(nnratio), mbCheckOrientation(checkOri) {}

    // Computes the Hamming distance between two ORB descriptors (ORBmatcher.cc:2047-2063).  Stays a cheap host
    // function: it is also called one pair at a time from MapPoint.cc:391 and Frame.cc:1032.
    static int DescriptorDistance(const cv::Mat &a, const cv::Mat &b) {
        const uint32_t *pa = a.ptr<uint32_t>(), *pb = b.ptr<uint32_t>();
        int dist = 0;
        for (int i = 0; i < 8; ++i) dist += __builtin_popcount(pa[i] ^ pb[i]);
        return dist;
    }

    // Search matches between Frame keypoints and projected MapPoints (ORBmatcher.cc:42-216). Returns #matches.
    template <class FrameT, class MapPointT>
    int SearchByProjection(FrameT &F, const std::vector<MapPointT *> &vpMapPoints, const float th = 3,
                           const bool bFarPoints = false, const float thFarPoints = 50.0f);

    // Project MapPoints tracked in the last frame into the current frame (ORBmatcher.cc:1667-1878).
    template <class FrameT>
    int SearchByProjection(FrameT &CurrentFrame, const FrameT &LastFrame, const float th, const bool bMono);

    // Brute force constrained to ORB in the same vocabulary node (ORBmatcher.cc:226-428).
    template <class KeyFrameT, class FrameT, class MapPointT>
    int SearchByBoW(KeyFrameT *pKF, FrameT &F, std::vector<MapPointT *> &vpMapPointMatches);

    // Matching for the map initialization, monocular case (ORBmatcher.cc:643-756).
    template <class FrameT>
    int SearchForInitialization(FrameT &F1, FrameT &F2, std::vector<cv::Point2f> &vbPrevMatched,
                                std::vector<int> &vnMatches12, int windowSize = 10);

    // Project MapPoints seen in a KeyFrame into the Frame; relocalisation (ORBmatcher.cc:1880-2000).
    template <class FrameT, class KeyFrameT, class MapPointT>
    int SearchByProjection(FrameT &CurrentFrame, KeyFrameT *pKF, const std::set<MapPointT *> &sAlreadyFound, const float th,
                           const int ORBdist);

    // SearchByBoW between two keyframes; loop detection (ORBmatcher.cc:758-900).
    template <class KeyFrameT, class MapPointT>
    int SearchByBoW(KeyFrameT *pKF1, KeyFrameT *pKF2, std::vector<MapPointT *> &vpMatches12);

    // Tracking::Relocalization's loop over its candidates (Tracking.cc:3687-3854) in one call: vvpMapPointMatches[i] and
    // element i of the result are what SearchByBoW(vpKFs[i], F, vvpMapPointMatches[i]) gives.  The caller skips bad
    // keyframes itself, as the loop does.
    template <class KeyFrameT, class FrameT, class MapPointT>
    std::vector<int> SearchByBoW(const std::vector<KeyFrameT *> &vpKFs, FrameT &F,
                                 std::vector<std::vector<MapPointT *>> &vvpMapPointMatches);
    // LoopClosing::DetectCommonRegionsFromBoW's loop over the candidates and their covisibles (LoopClosing.cc:573-642) in one
    // call: vvpMatches12[i] and element i of the result are what SearchByBoW(pKF1, vpKF2s[i], vvpMatches12[i]) gives.
    template <class KeyFrameT, class MapPointT>
    std::vector<int> SearchByBoW(KeyFrameT *pKF1, const std::vector<KeyFrameT *> &vpKF2s,
                                 std::vector<std::vector<MapPointT *>> &vvpMatches12);

    // Project MapPoints into a KeyFrame and search for duplicates (ORBmatcher.cc:1148-1335; bRight = false).
    template <class KeyFrameT, class MapPointT>
    int Fuse(KeyFrameT *pKF, const std::vector<MapPointT *> &vpMapPoints, const float th = 3.0, const bool bRight = false);
    // LocalMapping::SearchInNeighbors' loop (LocalMapping.cc:764-802) in one call: for each target in order, Fuse(pKFi,
    // vpMapPoints, th), then Fuse(pKFi, vpMapPoints, th, true) if pKFi->NLeft != -1.  Returns the sum of their counts.
    template <class KeyFrameT, class MapPointT>
    int Fuse(const std::vector<KeyFrameT *> &vpTargetKFs, const std::vector<MapPointT *> &vpMapPoints, const float th = 3.0);

#ifdef SOPHUS_SIM3_HPP   // the Sim3 overloads need Sophus' own SE3/Sim3 arithmetic (include sophus/sim3.hpp first, as
                         // the reference's ORBmatcher.h does)
    // Loop closing: project with a similarity transform (ORBmatcher.cc:430-528).
    template <class KeyFrameT, class MapPointT>
    int SearchByProjection(KeyFrameT *pKF, Sophus::Sim3<float> &Scw, const std::vector<MapPointT *> &vpPoints,
                           std::vector<MapPointT *> &vpMatched, int th, float ratioHamming = 1.0);
    // Place recognition (ORBmatcher.cc:530-641).
    template <class KeyFrameT, class MapPointT>
    int SearchByProjection(KeyFrameT *pKF, Sophus::Sim3<float> &Scw, const std::vector<MapPointT *> &vpPoints,
                           const std::vector<KeyFrameT *> &vpPointsKFs, std::vector<MapPointT *> &vpMatched,
                           std::vector<KeyFrameT *> &vpMatchedKF, int th, float ratioHamming = 1.0);
    // ORBmatcher.cc:1448-1665
    template <class KeyFrameT, class MapPointT>
    int SearchBySim3(KeyFrameT *pKF1, KeyFrameT *pKF2, std::vector<MapPointT *> &vpMatches12, const Sophus::Sim3f &S12,
                     const float th);
    // ORBmatcher.cc:1337-1446
    template <class KeyFrameT, class MapPointT>
    int Fuse(KeyFrameT *pKF, Sophus::Sim3f &Scw, const std::vector<MapPointT *> &vpPoints, float th,
             std::vector<MapPointT *> &vpReplacePoint);
#endif

    // Matching to triangulate new MapPoints, epipolar constraint (ORBmatcher.cc:902-1146; pinhole, mpCamera2 == NULL).
    template <class KeyFrameT>
    int SearchForTriangulation(KeyFrameT *pKF1, KeyFrameT *pKF2, std::vector<std::pair<size_t, size_t>> &vMatchedPairs,
                               const bool bOnlyStereo, const bool bCoarse = false);

    // LocalMapping::CreateNewMapPoints' loop `for (i) SearchForTriangulation(pKF1, vpKF2s[i], vMatchedPairs, bOnlyStereo,
    // bCoarse)` (LocalMapping.cc:406,460) in two halves: one device call for every neighbour up front, then, inside the loop,
    // SearchForTriangulation(search, i, vMatchedPairs), which returns exactly what the single-target call returns at that
    // moment.  The batch searches each feature of KF1 that has no map point; a resolve keeps the ones that still have none
    // and applies the rotation check.  A target is searched again by the single-target call when it is a two-camera
    // keyframe (or KF1 is one), when one of its map-point slots or either pose changed since the batch, or when a KF1
    // feature that had a map point at the batch has lost it.
    template <class KeyFrameT>
    struct TriangulationSearch;
    template <class KeyFrameT>
    TriangulationSearch<KeyFrameT> SearchForTriangulation(KeyFrameT *pKF1, const std::vector<KeyFrameT *> &vpKF2s,
                                                          const bool bOnlyStereo, const bool bCoarse);
    template <class KeyFrameT>
    int SearchForTriangulation(TriangulationSearch<KeyFrameT> &search, size_t i, std::vector<std::pair<size_t, size_t>> &vMatchedPairs);

public:
    static const int TH_LOW = 50;
    static const int TH_HIGH = 100;
    static const int HISTO_LENGTH = 30;

protected:
    float mfNNratio;
    bool mbCheckOrientation;

    template <class FrameT, class MapPointT>
    int SearchByProjectionTwoCameras(FrameT &F, const std::vector<MapPointT *> &vpMapPoints, const float th,
                                     const bool bFarPoints, const float thFarPoints);
    template <class KeyFrameT>
    int SearchForTriangulationTwoCameras(KeyFrameT *pKF1, KeyFrameT *pKF2, std::vector<std::pair<size_t, size_t>> &vMatchedPairs,
                                         const bool bOnlyStereo, const bool bCoarse);
    // ORBmatcher::ComputeThreeMaxima (ORBmatcher.cc:2002-2043) for the host-side replays
    static void ComputeThreeMaxima(std::vector<int> *histo, const int L, int &ind1, int &ind2, int &ind3) {
        int max1 = 0, max2 = 0, max3 = 0;
        for (int i = 0; i < L; i++) {
            const int s = (int)histo[i].size();
            if (s > max1) { max3 = max2; max2 = max1; max1 = s; ind3 = ind2; ind2 = ind1; ind1 = i; }
            else if (s > max2) { max3 = max2; max2 = s; ind3 = ind2; ind2 = i; }
            else if (s > max3) { max3 = s; ind3 = i; }
        }
        if (max2 < 0.1f * (float)max1) { ind2 = -1; ind3 = -1; }
        else if (max3 < 0.1f * (float)max1) { ind3 = -1; }
    }

    // ---- plumbing ----
    static void Check(vsg_status st, const char *what) {
        if (st != VSG_OK) throw std::runtime_error(std::string(what) + ": " + vsg_last_error());
    }
    // One vsg_matcher (stream + device / pinned scratch) per calling thread, created on first use and kept for the thread's
    // lifetime: the SLAM threads construct a fresh ORBmatcher for nearly every call, and a stream plus buffers per object would
    // cost more than the search.  Device: VSG_DEVICE (default 0).
    static vsg_matcher *Workspace() {
        struct Holder {
            vsg_matcher *m = nullptr;
            ~Holder() { vsg_matcher_destroy(m); }
        };
        static thread_local Holder h;
        if (!h.m) {
            const char *e = std::getenv("VSG_DEVICE");
            Check(vsg_matcher_create(e ? std::atoi(e) : 0, &h.m), "vsg_matcher_create");
        }
        return h.m;
    }

    // Flatten what the Search* methods read from a Frame / KeyFrame.
    struct Flat {
        std::vector<vsg_keypoint> keys;
        std::vector<uint8_t> desc;
        std::vector<float> scale;
        vsg_frame_view view;
    };
    // mvKeysUn, its descriptor rows and mvuRight (if any)
    template <class FrameT>
    static void Flatten(const FrameT &F, Flat &out) {
        FlattenKeys(F, F.mvKeysUn, nullptr, 0, F.mvuRight.empty() ? nullptr : F.mvuRight.data(), out);
    }
    struct CacheEntry;
    struct FrameGuard {   // RAII for an uploaded frame; a frame that lives in the thread's cache is only borrowed (and pinned)
        vsg_frame *h = nullptr;
        bool owned = true;
        CacheEntry *pin = nullptr;
        ~FrameGuard() {
            if (pin) --pin->pins;
            if (owned) vsg_frame_destroy(h);
        }
    };
    // Uploaded frames are kept per calling thread: Tracking runs up to three projection searches on the same current frame,
    // LocalMapping / LoopClosing several on the same keyframe, and what the searches read from a Frame / KeyFrame (mvKeysUn,
    // mvKeys(Right), mDescriptors, mvuRight, the grid parameters) does not change after construction.  An entry is identified
    // by the object's address and type, its mnId (Frame.h:217, KeyFrame.h:312 — a recycled address gets a new id), which of its feature
    // lists was flattened, and the size / address of its descriptor matrix.  Types without mnId, and VSG_FRAME_CACHE=0, upload
    // per call as before.  An entry borrowed by a FrameGuard is pinned: a search that holds more frames than the cache has
    // entries (the multi-target Fuse) uploads the extra ones for itself instead of evicting a frame it still reads.
    struct CacheEntry {
        const void *obj = nullptr, *desc = nullptr, *type = nullptr;
        unsigned long id = 0;
        int kind = -1, n = 0, pins = 0;
        unsigned long long stamp = 0;
        Flat flat;
        vsg_frame *h = nullptr;
    };
    struct FrameCache {
        static constexpr int kEntries = 6;
        CacheEntry e[kEntries];
        unsigned long long clock = 0, hits = 0, misses = 0;
        ~FrameCache() {
            for (CacheEntry &c : e) vsg_frame_destroy(c.h);
            if (std::getenv("VSG_FRAME_CACHE_STATS")) std::fprintf(stderr, "vsg frame cache: %llu hits, %llu uploads\n", hits, misses);
        }
    };
    static FrameCache &Cache() { static thread_local FrameCache c; return c; }
    static bool CacheEnabled() {
        static const bool on = [] { const char *e = std::getenv("VSG_FRAME_CACHE"); return !e || std::atoi(e) != 0; }();
        return on;
    }
    template <class T> static const void *TypeKey() { static const char k = 0; return &k; }   // Frame and KeyFrame count mnId separately
    template <class T> static auto FrameIdOf(const T &f, int) -> decltype((unsigned long)f.mnId) { return (unsigned long)f.mnId; }
    template <class T> static unsigned long FrameIdOf(const T &, long) { return 0; }
    template <class T> static constexpr auto HasFrameId(int) -> decltype((void)std::declval<const T &>().mnId, true) { return true; }
    template <class T> static constexpr bool HasFrameId(long) { return false; }
    // Flatten (fill) + vsg_frame_create, or the cached result of an earlier call on the same object.  `kind` names the
    // flattened feature list.  Returns the flat view to read; `guard.h` is the device frame.
    template <class FrameT, class Fill>
    static const Flat &Upload(const FrameT &F, int kind, Fill fill, Flat &local, FrameGuard &guard) {
        if (HasFrameId<FrameT>(0) && CacheEnabled()) {
            FrameCache &c = Cache();
            const void *desc = F.mDescriptors.rows > 0 ? (const void *)F.mDescriptors.ptr(0) : nullptr;
            const unsigned long id = FrameIdOf(F, 0);
            CacheEntry *slot = nullptr;
            for (CacheEntry &x : c.e) {
                if (x.h && x.obj == (const void *)&F && x.type == TypeKey<FrameT>() && x.id == id && x.kind == kind &&
                    x.n == F.mDescriptors.rows && x.desc == desc) {
                    x.stamp = ++c.clock;
                    ++c.hits;
                    ++x.pins;
                    guard.h = x.h;
                    guard.owned = false;
                    guard.pin = &x;
                    return x.flat;
                }
                if (!x.pins && (!slot || x.stamp < slot->stamp)) slot = &x;
            }
            ++c.misses;
            if (slot) {
                vsg_frame_destroy(slot->h);
                slot->h = nullptr;
                fill(slot->flat);
                Check(vsg_frame_create(Workspace(), &slot->flat.view, &slot->h), "vsg_frame_create");
                slot->obj = &F; slot->type = TypeKey<FrameT>(); slot->id = id; slot->kind = kind; slot->n = F.mDescriptors.rows; slot->desc = desc; slot->stamp = ++c.clock;
                ++slot->pins;
                guard.h = slot->h;
                guard.owned = false;
                guard.pin = slot;
                return slot->flat;
            }
        }
        fill(local);
        Check(vsg_frame_create(Workspace(), &local.view, &guard.h), "vsg_frame_create");
        return local;
    }
    template <class FV>
    static void FlattenFeatVec(const FV &fv, std::vector<int32_t> &nodes, std::vector<int32_t> &ptr, std::vector<int32_t> &idx,
                               size_t limit = (size_t)-1) {   // features >= limit are skipped (two-camera keyframes, :793-796)
        ptr.push_back(0);
        for (const auto &kv : fv) {           // DBoW2::FeatureVector = std::map<NodeId, std::vector<unsigned>>
            nodes.push_back((int32_t)kv.first);
            for (unsigned v : kv.second)
                if ((size_t)v < limit) idx.push_back((int32_t)v);
            ptr.push_back((int32_t)idx.size());
        }
    }
    // One side of a BoW search, flattened as the SearchByBoW overloads read it: both cameras of a two-camera frame /
    // keyframe or mvKeysUn, FeatureVector entries >= limit dropped, map-point flags from GetMapPointMatches() / isBad()
    // (all zero without vpMPs).  Not copyable: side points into the other members.
    struct BowSide {
        Flat flat;
        std::vector<uint8_t> valid;
        std::vector<int32_t> nodes, ptr, idx;
        vsg_bow_side side;
        BowSide() = default;
        BowSide(const BowSide &) = delete;
        BowSide &operator=(const BowSide &) = delete;
    };
    template <class FrameT, class MapPointT>
    static void FlattenBowSide(const FrameT &F, bool bothCameras, size_t limit, const std::vector<MapPointT *> *vpMPs, BowSide &o) {
        if (bothCameras) FlattenBothCameras(F, o.flat); else Flatten(F, o.flat);
        o.valid.assign(o.flat.view.n, 0);
        if (vpMPs)
            for (int i = 0; i < o.flat.view.n; ++i) o.valid[i] = (*vpMPs)[i] && !(*vpMPs)[i]->isBad();   // :262-266, :800-804
        FlattenFeatVec(F.mFeatVec, o.nodes, o.ptr, o.idx, limit);
        o.side.view = o.flat.view;
        o.side.mp_valid = o.valid.data();
        o.side.nnodes = (int32_t)o.nodes.size();
        o.side.nodes = o.nodes.data(); o.side.ptr = o.ptr.data(); o.side.idx = o.idx.data();
    }
    // SearchByBoW(KF, KF): two-camera keyframes take part with the features that have an entry in mvKeysUn (:793-796)
    template <class KeyFrameT>
    static size_t BowKFLimit(const KeyFrameT *pKF) { return pKF->NLeft != -1 ? pKF->mvKeysUn.size() : (size_t)-1; }
    template <class MapPointT>
    static void CopyDescriptor(MapPointT *pMP, std::vector<uint8_t> &desc, size_t i) {
        const cv::Mat d = pMP->GetDescriptor();
        std::memcpy(&desc[i * 32], d.ptr(0), 32);
    }
    template <class KeyFrameT>
    static void RequireSingleCameraKF(const KeyFrameT &KF) {
        if (KF.NLeft != -1)
            throw std::runtime_error("vsg ORBmatcher: two-camera keyframes (NLeft != -1) are not supported by the CUDA path");
    }
    // The gates the Sim3 / Fuse projections share between the depth test and GetFeaturesInArea
    // (e.g. ORBmatcher.cc:468-486): scale-invariance range, viewing angle, predicted level.
    template <class MapPointT, class KeyFrameT, class Vec3T>
    static bool DistanceAndNormalGates(MapPointT *pMP, KeyFrameT *pKF, const Vec3T &p3Dw, const Vec3T &Ow, bool bCheckNormal,
                                       vsg_search_point &p) {
        const float maxDistance = pMP->GetMaxDistanceInvariance();
        const float minDistance = pMP->GetMinDistanceInvariance();
        Vec3T PO = p3Dw - Ow;
        const float dist = PO.norm();
        if (dist < minDistance || dist > maxDistance) return false;
        if (bCheckNormal) {
            Vec3T Pn = pMP->GetNormal();
            if (PO.dot(Pn) < 0.5 * dist) return false;
        }
        p.level = pMP->PredictScale(dist, pKF);
        return true;
    }
    // Keys (one or two lists back to back) + descriptor rows [row0, row0 + n) of a frame / keyframe as a view.
    template <class FrameT>
    static void FlattenKeys(const FrameT &F, const std::vector<cv::KeyPoint> &keysA, const std::vector<cv::KeyPoint> *keysB,
                            int row0, const float *u_right, Flat &out) {
        static_assert(sizeof(cv::KeyPoint) == sizeof(vsg_keypoint), "cv::KeyPoint layout");
        const int nA = (int)keysA.size(), nB = keysB ? (int)keysB->size() : 0, n = nA + nB;
        out.keys.resize(n);
        if (nA) std::memcpy(out.keys.data(), keysA.data(), (size_t)nA * sizeof(vsg_keypoint));
        if (nB) std::memcpy(out.keys.data() + nA, keysB->data(), (size_t)nB * sizeof(vsg_keypoint));
        out.desc.resize((size_t)n * 32);
        for (int i = 0; i < n; ++i) std::memcpy(&out.desc[(size_t)i * 32], F.mDescriptors.ptr(row0 + i), 32);
        out.scale.assign(F.mvScaleFactors.begin(), F.mvScaleFactors.end());
        vsg_frame_view &v = out.view;
        v.n = n; v.keys = out.keys.data(); v.descriptors = out.desc.data(); v.u_right = u_right;
        v.min_x = F.mnMinX; v.min_y = F.mnMinY; v.max_x = F.mnMaxX; v.max_y = F.mnMaxY;
        v.grid_inv_w = F.mfGridElementWidthInv; v.grid_inv_h = F.mfGridElementHeightInv;
        v.grid_cols = FRAME_GRID_COLS; v.grid_rows = FRAME_GRID_ROWS;
        v.scale_factors = out.scale.data(); v.n_levels = (int)out.scale.size();
    }
    // A two-camera frame / keyframe as one feature list: mvKeys then mvKeysRight, all rows of mDescriptors (the order of
    // the indices in mFeatVec; no grid use).
    template <class FrameT>
    static void FlattenBothCameras(const FrameT &F, Flat &out) { FlattenKeys(F, F.mvKeys, &F.mvKeysRight, 0, nullptr, out); }
    // One camera of a two-camera frame / keyframe: mvKeys + descriptor rows [0, Nleft) or mvKeysRight + rows [Nleft, N),
    // the layout GetFeaturesInArea(..., bRight) works on (Frame.cc:840-848, KeyFrame.cc:834-875).
    template <class FrameT>
    static void FlattenCamera(const FrameT &F, bool bRight, int nLeft, const float *u_right, Flat &out) {
        FlattenKeys(F, bRight ? F.mvKeysRight : F.mvKeys, nullptr, bRight ? nLeft : 0, u_right, out);
    }
    template <class FrameT>
    void UploadCameras(const FrameT &F, Flat local[2], const Flat *cam[2], FrameGuard fr[2]) {
        for (int c = 0; c < 2; ++c)
            cam[c] = &Upload(F, 1 + c, [&](Flat &o) { FlattenCamera(F, c == 1, F.Nleft, nullptr, o); }, local[c], fr[c]);
    }
    // kinds: 0 = Flatten (mvKeysUn), 1 / 2 = left / right camera, 3 / 4 = left / right camera with mvuRight
    // What the methods without two-camera code of their own search on (reloc / Sim3 projections, SearchBySim3,
    // Fuse(KF, Scw, ...)): Frame::GetFeaturesInArea / KeyFrame::GetFeaturesInArea with bRight == false walk the left
    // camera's grid and keypoints (mvKeys, Frame.cc:840-848, KeyFrame.cc:862-868) and the descriptor rows [0, Nleft).
    template <class FrameT>
    static void FlattenSearched(const FrameT &F, int nLeft, Flat &out) {
        if (nLeft != -1) FlattenCamera(F, false, nLeft, nullptr, out);
        else Flatten(F, out);
    }
    // ---- Fuse(KF, vpMapPoints, th, bRight) (ORBmatcher.cc:1148-1335) in the parts the one-target and the multi-target Fuse
    // share; defined below the class ----
    template <class KeyFrameT>
    static void UploadFuseTarget(KeyFrameT *pKF, bool bRight, Flat &local, FrameGuard &fr);
    template <class KeyFrameT, class MapPointT>
    static void ProjectForFuse(KeyFrameT *pKF, bool bRight, const std::vector<MapPointT *> &vpMapPoints, vsg_search_point *pts);
    template <class KeyFrameT, class MapPointT, class OnReplace>
    static int FuseReplay(KeyFrameT *pKF, bool bRight, const std::vector<MapPointT *> &vpMapPoints, const int32_t *best,
                          OnReplace onReplace);
    // Fuse(pKF, vpMapPoints, th, bRight) for each (pKF, bRight) of targets in order, the searches in one device call; returns
    // the sum of their counts
    template <class KeyFrameT, class MapPointT>
    static int FuseTargets(const std::vector<std::pair<KeyFrameT *, bool>> &targets, const std::vector<MapPointT *> &vpMapPoints,
                           const float th);
    // ---- SearchForTriangulation (ORBmatcher.cc:902-1146) in the parts the one-target and the multi-target forms share ----
    // epipole of KF1 in KF2 and the fundamental matrix of Pinhole::epipolarConstrain (Pinhole.cpp:120-124), built with the
    // reference's own Eigen expressions (f12 is left zero when bCoarse: nothing reads it)
    template <class KeyFrameT>
    static void TriangulationGeometry(KeyFrameT *pKF1, KeyFrameT *pKF2, bool bCoarse, float f12[9], float ep[2]);
    // KF1 or a target as the C ABI reads it: mvKeysUn, mDescriptors, mFeatVec and GetMapPoint(i) != NULL (:968, :998)
    template <class KeyFrameT>
    static void FlattenTriangulationSide(KeyFrameT &KF, BowSide &o) {
        using MapPointT = typename std::remove_pointer<decltype(KF.GetMapPoint(0))>::type;
        FlattenBowSide(KF, false, (size_t)-1, static_cast<const std::vector<MapPointT *> *>(nullptr), o);
        for (int i = 0; i < o.flat.view.n; ++i) o.valid[i] = KF.GetMapPoint(i) ? 1 : 0;
    }
    template <class KeyFrameT>
    static bool TwoCameraKF(const KeyFrameT *pKF) { return pKF->NLeft != -1 || pKF->mpCamera2; }
    template <class FrameT>
    static void RequireSingleCamera(const FrameT &F) {
        if (F.Nleft != -1)
            throw std::runtime_error("vsg ORBmatcher: two-camera frames (Nleft != -1) are not supported by the CUDA path");
    }
};

// ---------------------------------------------------------------------------------------------------
// Two-camera frames (F.Nleft != -1, ORBmatcher.cc:42-216 incl. the right-camera branch :146-213): the two cameras'
// keypoints are uploaded as two frames, the library runs both window searches and replays the loop in map order.
template <class FrameT, class MapPointT>
int ORBmatcher::SearchByProjectionTwoCameras(FrameT &F, const std::vector<MapPointT *> &vpMapPoints, const float th,
                                             const bool bFarPoints, const float thFarPoints) {
    const int nL = F.Nleft, nR = (int)F.mvKeysRight.size(), N = nL + nR, nMP = (int)vpMapPoints.size();
    Flat camLocal[2];
    const Flat *cam[2];
    FrameGuard fr[2];
    UploadCameras(F, camLocal, cam, fr);
    std::vector<uint8_t> occupied(N, 0);
    for (int i = 0; i < N; ++i)
        if (F.mvpMapPoints[i] && F.mvpMapPoints[i]->Observations() > 0) occupied[i] = 1;
    std::vector<int32_t> l2r(F.mvLeftToRightMatch.begin(), F.mvLeftToRightMatch.end());
    std::vector<int32_t> r2l(F.mvRightToLeftMatch.begin(), F.mvRightToLeftMatch.end());
    l2r.resize(nL, -1);
    r2l.resize(nR, -1);
    std::vector<vsg_track_point> pl(nMP), pr(nMP);
    std::vector<uint8_t> desc((size_t)nMP * 32, 0);
    for (int i = 0; i < nMP; ++i) {
        MapPointT *pMP = vpMapPoints[i];
        std::memset(&pl[i], 0, sizeof(vsg_track_point));
        std::memset(&pr[i], 0, sizeof(vsg_track_point));
        if (!pMP->mbTrackInView && !pMP->mbTrackInViewR) continue;
        pl[i].in_view = pMP->mbTrackInView ? 1 : 0;
        pl[i].proj_x = pMP->mTrackProjX; pl[i].proj_y = pMP->mTrackProjY; pl[i].view_cos = pMP->mTrackViewCos;
        pl[i].level = pMP->mnTrackScaleLevel; pl[i].depth = pMP->mTrackDepth;
        pl[i].bad = pMP->isBad() ? 1 : 0;
        pl[i].blocks = pMP->Observations() > 0 ? 1 : 0;
        pr[i].in_view = pMP->mbTrackInViewR ? 1 : 0;
        pr[i].proj_x = pMP->mTrackProjXR; pr[i].proj_y = pMP->mTrackProjYR; pr[i].view_cos = pMP->mTrackViewCosR;
        pr[i].level = pMP->mnTrackScaleLevelR;
        const cv::Mat d = pMP->GetDescriptor();
        std::memcpy(&desc[(size_t)i * 32], d.ptr(0), 32);
    }
    std::vector<int32_t> assign(N, -1);
    int nmatches = 0;
    Check(vsg_search_by_projection_map_2cam(Workspace(), fr[0].h, fr[1].h, occupied.data(), l2r.data(), r2l.data(), nMP, pl.data(),
                                            pr.data(), desc.data(), th, bFarPoints ? 1 : 0, thFarPoints, mfNNratio, assign.data(),
                                            &nmatches),
          "vsg_search_by_projection_map_2cam");
    for (int i = 0; i < N; ++i)
        if (assign[i] >= 0) F.mvpMapPoints[i] = vpMapPoints[assign[i]];
    return nmatches;
}

template <class FrameT, class MapPointT>
int ORBmatcher::SearchByProjection(FrameT &F, const std::vector<MapPointT *> &vpMapPoints, const float th,
                                   const bool bFarPoints, const float thFarPoints) {
    if (F.Nleft != -1) return SearchByProjectionTwoCameras(F, vpMapPoints, th, bFarPoints, thFarPoints);
    Flat flatLocal;
    FrameGuard fr;
    const Flat &flat = Upload(F, 0, [&](Flat &o) { Flatten(F, o); }, flatLocal, fr);
    const int N = flat.view.n, nMP = (int)vpMapPoints.size();
    std::vector<uint8_t> occupied(N, 0);
    for (int i = 0; i < N; ++i)
        if (F.mvpMapPoints[i] && F.mvpMapPoints[i]->Observations() > 0) occupied[i] = 1;   // :88-90
    std::vector<vsg_track_point> pts(nMP);
    std::vector<uint8_t> desc((size_t)nMP * 32, 0);
    for (int i = 0; i < nMP; ++i) {
        MapPointT *pMP = vpMapPoints[i];
        vsg_track_point &p = pts[i];
        std::memset(&p, 0, sizeof(p));
        if (!pMP->mbTrackInView) continue;            // :49-50 (mbTrackInViewR belongs to the two-camera branch)
        p.in_view = 1;
        p.proj_x = pMP->mTrackProjX; p.proj_y = pMP->mTrackProjY; p.proj_xr = pMP->mTrackProjXR;
        p.view_cos = pMP->mTrackViewCos; p.depth = pMP->mTrackDepth; p.level = pMP->mnTrackScaleLevel;
        p.bad = pMP->isBad() ? 1 : 0;
        p.blocks = pMP->Observations() > 0 ? 1 : 0;
        const cv::Mat d = pMP->GetDescriptor();
        std::memcpy(&desc[(size_t)i * 32], d.ptr(0), 32);
    }
    std::vector<int32_t> assign(N, -1);
    int nmatches = 0;
    Check(vsg_search_by_projection_map(Workspace(), fr.h, occupied.data(), nMP, pts.data(), desc.data(), th,
                                       bFarPoints ? 1 : 0, thFarPoints, mfNNratio, assign.data(), &nmatches),
          "vsg_search_by_projection_map");
    for (int i = 0; i < N; ++i)
        if (assign[i] >= 0) F.mvpMapPoints[i] = vpMapPoints[assign[i]];                    // :130
    return nmatches;
}

template <class FrameT>
int ORBmatcher::SearchByProjection(FrameT &CurrentFrame, const FrameT &LastFrame, const float th, const bool bMono) {
    const bool bTwoCameras = CurrentFrame.Nleft != -1;
    Flat flatLocal, camLocal[2];
    const Flat *cam[2] = {nullptr, nullptr}, *flatp = nullptr;
    FrameGuard fr, frc[2];
    if (bTwoCameras) UploadCameras(CurrentFrame, camLocal, cam, frc);
    else flatp = &Upload(CurrentFrame, 0, [&](Flat &o) { Flatten(CurrentFrame, o); }, flatLocal, fr);
    // pose arithmetic stays with the reference's Sophus / camera classes (:1677-1716)
    const auto Tcw = CurrentFrame.GetPose();
    const auto twc = Tcw.inverse().translation();
    const auto Tlw = LastFrame.GetPose();
    const auto tlc = Tlw * twc;
    const bool bForward = tlc(2) > CurrentFrame.mb && !bMono;
    const bool bBackward = -tlc(2) > CurrentFrame.mb && !bMono;
    const int nLast = LastFrame.N, N = bTwoCameras ? cam[0]->view.n + cam[1]->view.n : flatp->view.n;
    std::vector<vsg_proj_point> pts(nLast), ptsR(bTwoCameras ? nLast : 0);
    std::vector<uint8_t> desc((size_t)nLast * 32, 0);
    for (int i = 0; i < nLast; ++i) {
        vsg_proj_point &p = pts[i];
        std::memset(&p, 0, sizeof(p));
        if (bTwoCameras) std::memset(&ptsR[i], 0, sizeof(vsg_proj_point));
        auto *pMP = LastFrame.mvpMapPoints[i];
        if (!pMP || LastFrame.mvbOutlier[i]) continue;
        const auto x3Dw = pMP->GetWorldPos();
        const auto x3Dc = Tcw * x3Dw;
        const float invzc = 1.0 / x3Dc(2);
        if (invzc < 0) continue;
        const auto uv = CurrentFrame.mpCamera->project(x3Dc);
        if (uv(0) < CurrentFrame.mnMinX || uv(0) > CurrentFrame.mnMaxX) continue;
        if (uv(1) < CurrentFrame.mnMinY || uv(1) > CurrentFrame.mnMaxY) continue;
        p.valid = 1;
        p.u = uv(0); p.v = uv(1);
        p.ur = uv(0) - CurrentFrame.mbf * invzc;                                           // :1747
        // last-frame keypoint by camera (:1711-1712, :1768-1770)
        const bool lastLeft = LastFrame.Nleft == -1 || i < LastFrame.Nleft;
        p.octave = lastLeft ? LastFrame.mvKeys[i].octave : LastFrame.mvKeysRight[i - LastFrame.Nleft].octave;
        p.angle = LastFrame.Nleft == -1 ? LastFrame.mvKeysUn[i].angle
                  : lastLeft            ? LastFrame.mvKeys[i].angle
                                        : LastFrame.mvKeysRight[i - LastFrame.Nleft].angle;
        p.blocks = pMP->Observations() > 0 ? 1 : 0;
        if (bTwoCameras) {                                                                 // :1787-1788
            const auto x3Dr = CurrentFrame.GetRelativePoseTrl() * x3Dc;
            const auto uvr = CurrentFrame.mpCamera->project(x3Dr);
            ptsR[i].u = uvr(0); ptsR[i].v = uvr(1);
        }
        const cv::Mat d = pMP->GetDescriptor();
        std::memcpy(&desc[(size_t)i * 32], d.ptr(0), 32);
    }
    std::vector<uint8_t> occupied(N, 0);
    for (int i = 0; i < N; ++i)
        if (CurrentFrame.mvpMapPoints[i] && CurrentFrame.mvpMapPoints[i]->Observations() > 0) occupied[i] = 1;
    std::vector<int32_t> assign(N, -1);
    int nmatches = 0;
    const int mode = bForward ? 1 : (bBackward ? 2 : 0);
    if (bTwoCameras)
        Check(vsg_search_by_projection_last_2cam(Workspace(), frc[0].h, frc[1].h, occupied.data(), nLast, pts.data(), ptsR.data(),
                                                 desc.data(), th, mode, mbCheckOrientation ? 1 : 0, assign.data(), &nmatches),
              "vsg_search_by_projection_last_2cam");
    else
        Check(vsg_search_by_projection_last(Workspace(), fr.h, occupied.data(), nLast, pts.data(), desc.data(), th, mode,
                                            mbCheckOrientation ? 1 : 0, assign.data(), &nmatches),
              "vsg_search_by_projection_last");
    for (int i = 0; i < N; ++i) {
        if (assign[i] >= 0) CurrentFrame.mvpMapPoints[i] = LastFrame.mvpMapPoints[assign[i]];   // :1763
        else if (assign[i] == -2) CurrentFrame.mvpMapPoints[i] = nullptr;                     // :1870
    }
    return nmatches;
}

template <class KeyFrameT, class FrameT, class MapPointT>
int ORBmatcher::SearchByBoW(KeyFrameT *pKF, FrameT &F, std::vector<MapPointT *> &vpMapPointMatches) {
    std::vector<std::vector<MapPointT *>> vvpMatches;
    const int nmatches = SearchByBoW(std::vector<KeyFrameT *>{pKF}, F, vvpMatches)[0];
    vpMapPointMatches = std::move(vvpMatches[0]);
    return nmatches;
}

template <class KeyFrameT, class FrameT, class MapPointT>
std::vector<int> ORBmatcher::SearchByBoW(const std::vector<KeyFrameT *> &vpKFs, FrameT &F,
                                         std::vector<std::vector<MapPointT *>> &vvpMapPointMatches) {
    const size_t T = vpKFs.size();
    std::vector<std::vector<MapPointT *>> vpMapPointsKF(T);
    std::vector<BowSide> kfs(T);
    std::vector<const vsg_bow_side *> table(T);
    // two-camera frames / keyframes: the left camera's keypoints followed by the right camera's, the order of
    // mDescriptors and of the indices in mFeatVec (:298-322, :341-343, :348-350)
    for (size_t t = 0; t < T; ++t) {
        vpMapPointsKF[t] = vpKFs[t]->GetMapPointMatches();
        FlattenBowSide(*vpKFs[t], vpKFs[t]->mpCamera2 != nullptr, (size_t)-1, &vpMapPointsKF[t], kfs[t]);
        table[t] = &kfs[t].side;
    }
    BowSide fr;
    FlattenBowSide(F, F.Nleft != -1, (size_t)-1, static_cast<const std::vector<MapPointT *> *>(nullptr), fr);
    const size_t n = (size_t)fr.flat.view.n;
    std::vector<int32_t> matches(T * n, -1);
    std::vector<int> counts(T, 0);
    Check(vsg_search_by_bow_multi(Workspace(), (int)T, table.data(), &fr.side, F.Nleft, mfNNratio, mbCheckOrientation ? 1 : 0,
                                  matches.data(), counts.data()), "vsg_search_by_bow_multi");
    vvpMapPointMatches.assign(T, std::vector<MapPointT *>(F.N, static_cast<MapPointT *>(nullptr)));
    for (size_t t = 0; t < T; ++t)
        for (size_t j = 0; j < n; ++j)
            if (matches[t * n + j] >= 0) vvpMapPointMatches[t][j] = vpMapPointsKF[t][matches[t * n + j]];   // :339
    return counts;
}

template <class FrameT>
int ORBmatcher::SearchForInitialization(FrameT &F1, FrameT &F2, std::vector<cv::Point2f> &vbPrevMatched,
                                        std::vector<int> &vnMatches12, int windowSize) {
    Flat f1, f2Local;
    Flatten(F1, f1);
    FrameGuard fr2;
    const Flat &f2 = Upload(F2, 0, [&](Flat &o) { Flatten(F2, o); }, f2Local, fr2);
    static_assert(sizeof(cv::Point2f) == 2 * sizeof(float), "cv::Point2f layout");
    vnMatches12 = std::vector<int>(F1.mvKeysUn.size(), -1);
    int nmatches = 0;
    Check(vsg_search_for_initialization(Workspace(), &f1.view, fr2.h, reinterpret_cast<float *>(vbPrevMatched.data()),
                                        windowSize, mfNNratio, mbCheckOrientation ? 1 : 0, vnMatches12.data(), &nmatches),
          "vsg_search_for_initialization");
    return nmatches;
}

// ---- relocalisation (ORBmatcher.cc:1880-2000) ----
template <class FrameT, class KeyFrameT, class MapPointT>
int ORBmatcher::SearchByProjection(FrameT &CurrentFrame, KeyFrameT *pKF, const std::set<MapPointT *> &sAlreadyFound,
                                   const float th, const int ORBdist) {
    Flat flatLocal;      // two-camera frames: the left camera (no code of its own, :1880-2000)
    FrameGuard fr;
    const Flat &flat = Upload(CurrentFrame, CurrentFrame.Nleft != -1 ? 1 : 0,
                              [&](Flat &o) { FlattenSearched(CurrentFrame, CurrentFrame.Nleft, o); }, flatLocal, fr);
    const auto Tcw = CurrentFrame.GetPose();
    const auto Ow = Tcw.inverse().translation();
    const std::vector<MapPointT *> vpMPs = pKF->GetMapPointMatches();
    const int n = (int)vpMPs.size(), N = flat.view.n;
    std::vector<vsg_search_point> pts(n);
    std::vector<uint8_t> desc((size_t)n * 32, 0);
    for (int i = 0; i < n; ++i) {
        vsg_search_point &p = pts[i];
        std::memset(&p, 0, sizeof(p));
        MapPointT *pMP = vpMPs[i];
        if (!pMP || pMP->isBad() || sAlreadyFound.count(pMP)) continue;               // :1898-1902
        const auto x3Dw = pMP->GetWorldPos();
        const auto x3Dc = Tcw * x3Dw;
        const auto uv = CurrentFrame.mpCamera->project(x3Dc);
        if (uv(0) < CurrentFrame.mnMinX || uv(0) > CurrentFrame.mnMaxX) continue;
        if (uv(1) < CurrentFrame.mnMinY || uv(1) > CurrentFrame.mnMaxY) continue;
        const auto PO = x3Dw - Ow;                                                     // :1915-1925
        const float dist3D = PO.norm();
        const float maxDistance = pMP->GetMaxDistanceInvariance();
        const float minDistance = pMP->GetMinDistanceInvariance();
        if (dist3D < minDistance || dist3D > maxDistance) continue;
        p.level = pMP->PredictScale(dist3D, &CurrentFrame);
        p.u = uv(0); p.v = uv(1);
        p.angle = pKF->mvKeysUn[i].angle;
        p.valid = 1;
        CopyDescriptor(pMP, desc, (size_t)i);
    }
    std::vector<uint8_t> occupied(N, 0);
    for (int i = 0; i < N; ++i) occupied[i] = CurrentFrame.mvpMapPoints[i] ? 1 : 0;   // :1939
    std::vector<int32_t> assign(N, -1);
    int nmatches = 0;
    Check(vsg_search_by_projection_reloc(Workspace(), fr.h, occupied.data(), n, pts.data(), desc.data(), th, ORBdist,
                                         mbCheckOrientation ? 1 : 0, assign.data(), &nmatches), "vsg_search_by_projection_reloc");
    for (int i = 0; i < N; ++i) {
        if (assign[i] >= 0) CurrentFrame.mvpMapPoints[i] = vpMPs[assign[i]];           // :1954
        else if (assign[i] == -2) CurrentFrame.mvpMapPoints[i] = nullptr;              // :1989
    }
    return nmatches;
}

// ---- SearchByBoW(KF, KF) (ORBmatcher.cc:758-900) ----
template <class KeyFrameT, class MapPointT>
int ORBmatcher::SearchByBoW(KeyFrameT *pKF1, KeyFrameT *pKF2, std::vector<MapPointT *> &vpMatches12) {
    std::vector<std::vector<MapPointT *>> vvpMatches;
    const int nmatches = SearchByBoW(pKF1, std::vector<KeyFrameT *>{pKF2}, vvpMatches)[0];
    vpMatches12 = std::move(vvpMatches[0]);
    return nmatches;
}

template <class KeyFrameT, class MapPointT>
std::vector<int> ORBmatcher::SearchByBoW(KeyFrameT *pKF1, const std::vector<KeyFrameT *> &vpKF2s,
                                         std::vector<std::vector<MapPointT *>> &vvpMatches12) {
    // two-camera keyframes: only the features with an entry in mvKeysUn take part (`idx >= mvKeysUn.size()` -> continue,
    // :793-796, :814-817); they are dropped from the flattened FeatureVectors
    const size_t T = vpKF2s.size();
    const std::vector<MapPointT *> vpMapPoints1 = pKF1->GetMapPointMatches();
    BowSide k1;
    FlattenBowSide(*pKF1, false, BowKFLimit(pKF1), &vpMapPoints1, k1);                 // :800-804
    std::vector<std::vector<MapPointT *>> vpMapPoints2(T);
    std::vector<BowSide> k2s(T);
    std::vector<const vsg_bow_side *> table(T);
    for (size_t t = 0; t < T; ++t) {
        vpMapPoints2[t] = vpKF2s[t]->GetMapPointMatches();
        FlattenBowSide(*vpKF2s[t], false, BowKFLimit(vpKF2s[t]), &vpMapPoints2[t], k2s[t]);   // :820-826
        table[t] = &k2s[t].side;
    }
    const size_t n = (size_t)k1.flat.view.n;
    std::vector<int32_t> m12(T * n, -1);
    std::vector<int> counts(T, 0);
    Check(vsg_search_by_bow_kf_multi(Workspace(), &k1.side, (int)T, table.data(), mfNNratio, mbCheckOrientation ? 1 : 0, m12.data(),
                                     counts.data()), "vsg_search_by_bow_kf_multi");
    vvpMatches12.assign(T, std::vector<MapPointT *>(vpMapPoints1.size(), static_cast<MapPointT *>(nullptr)));
    for (size_t t = 0; t < T; ++t)
        for (size_t i = 0; i < n; ++i)
            if (m12[t * n + i] >= 0) vvpMatches12[t][i] = vpMapPoints2[t][m12[t * n + i]];   // :847
    return counts;
}

// ---- Fuse(KF, vpMapPoints, th) (ORBmatcher.cc:1148-1335) ----
// The camera Fuse searches: two cameras -> mvKeys / mvKeysRight with their descriptor rows and grid
// (KeyFrame::GetFeaturesInArea(..., bRight)); the stereo gate reads mvuRight[idx] with the camera-local index on both sides (:1266)
template <class KeyFrameT>
void ORBmatcher::UploadFuseTarget(KeyFrameT *pKF, bool bRight, Flat &local, FrameGuard &fr) {
    const bool bTwoCameras = pKF->NLeft != -1;
    Upload(*pKF, bTwoCameras ? 3 + (bRight ? 1 : 0) : 0, [&](Flat &o) {
        if (bTwoCameras) {
            const int n = (int)(bRight ? pKF->mvKeysRight : pKF->mvKeys).size();
            FlattenCamera(*pKF, bRight, pKF->NLeft, (int)pKF->mvuRight.size() >= n && n > 0 ? pKF->mvuRight.data() : nullptr, o);
        } else {
            Flatten(*pKF, o);
        }
    }, local, fr);
}

// The projection of every map point into the camera (:1154-1244); pts[i].valid = the point reaches GetFeaturesInArea.
template <class KeyFrameT, class MapPointT>
void ORBmatcher::ProjectForFuse(KeyFrameT *pKF, bool bRight, const std::vector<MapPointT *> &vpMapPoints, vsg_search_point *pts) {
    const auto Tcw = bRight ? pKF->GetRightPose() : pKF->GetPose();                          // :1154-1165
    const auto Ow = bRight ? pKF->GetRightCameraCenter() : pKF->GetCameraCenter();
    auto *pCamera = bRight ? pKF->mpCamera2 : pKF->mpCamera;
    const float &bf = pKF->mbf;
    for (size_t i = 0; i < vpMapPoints.size(); ++i) {
        vsg_search_point &p = pts[i];
        std::memset(&p, 0, sizeof(p));
        MapPointT *pMP = vpMapPoints[i];
        if (!pMP) continue;
        // isBad() / IsInKeyFrame() change while the reference's loop runs: they are evaluated in the replay,
        // at the same point of the iteration order; the search itself does not depend on them.
        const auto p3Dw = pMP->GetWorldPos();
        const auto p3Dc = Tcw * p3Dw;
        if (p3Dc(2) < 0.0f) continue;
        const float invz = 1 / p3Dc(2);
        const auto uv = pCamera->project(p3Dc);
        if (!pKF->IsInImage(uv(0), uv(1))) continue;
        p.ur = uv(0) - bf * invz;
        if (!DistanceAndNormalGates(pMP, pKF, p3Dw, Ow, true, p)) continue;
        p.u = uv(0); p.v = uv(1);
        p.valid = 1;
    }
}

// The bookkeeping of :1173-1332 in point order, from the searched camera's best keypoints (-1: none).  onReplace(survivor)
// follows every Replace.
template <class KeyFrameT, class MapPointT, class OnReplace>
int ORBmatcher::FuseReplay(KeyFrameT *pKF, bool bRight, const std::vector<MapPointT *> &vpMapPoints, const int32_t *best,
                           OnReplace onReplace) {
    const int idxOffset = bRight ? pKF->NLeft : 0;                                            // :1295-1296
    int nFused = 0;
    for (size_t i = 0; i < vpMapPoints.size(); ++i) {
        MapPointT *pMP = vpMapPoints[i];
        if (!pMP || pMP->isBad() || pMP->IsInKeyFrame(pKF)) continue;
        if (best[i] < 0) continue;
        const int idx = best[i] + idxOffset;
        MapPointT *pMPinKF = pKF->GetMapPoint(idx);
        if (pMPinKF) {
            if (!pMPinKF->isBad()) {
                if (pMPinKF->Observations() > pMP->Observations()) { pMP->Replace(pMPinKF); onReplace(pMPinKF); }
                else { pMPinKF->Replace(pMP); onReplace(pMP); }
            }
        } else {
            pMP->AddObservation(pKF, idx);
            pKF->AddMapPoint(pMP, idx);
        }
        nFused++;
    }
    return nFused;
}

template <class KeyFrameT, class MapPointT>
int ORBmatcher::Fuse(KeyFrameT *pKF, const std::vector<MapPointT *> &vpMapPoints, const float th, const bool bRight) {
    if (bRight && pKF->NLeft == -1) throw std::runtime_error("vsg ORBmatcher::Fuse: bRight needs a two-camera keyframe");
    return FuseTargets(std::vector<std::pair<KeyFrameT *, bool>>{{pKF, bRight}}, vpMapPoints, th);
}

template <class KeyFrameT, class MapPointT>
int ORBmatcher::Fuse(const std::vector<KeyFrameT *> &vpTargetKFs, const std::vector<MapPointT *> &vpMapPoints, const float th) {
    std::vector<std::pair<KeyFrameT *, bool>> targets;                                        // (keyframe, bRight) in loop order
    for (KeyFrameT *pKF : vpTargetKFs) {
        targets.emplace_back(pKF, false);
        if (pKF->NLeft != -1) targets.emplace_back(pKF, true);
    }
    return FuseTargets(targets, vpMapPoints, th);
}

template <class KeyFrameT, class MapPointT>
int ORBmatcher::FuseTargets(const std::vector<std::pair<KeyFrameT *, bool>> &targets, const std::vector<MapPointT *> &vpMapPoints,
                            const float th) {
    const int T = (int)targets.size(), n = (int)vpMapPoints.size();
    if (T == 0) return 0;
    std::vector<Flat> local(T);
    std::vector<FrameGuard> fr(T);
    std::vector<const vsg_frame *> frames(T);
    std::vector<const float *> sigma(T);
    std::vector<vsg_search_point> pts((size_t)T * n);
    std::vector<uint8_t> searched(n, 0), desc((size_t)n * 32, 0);
    for (int t = 0; t < T; ++t) {
        KeyFrameT *pKF = targets[t].first;
        UploadFuseTarget(pKF, targets[t].second, local[t], fr[t]);
        frames[t] = fr[t].h;
        sigma[t] = pKF->mvInvLevelSigma2.data();
        ProjectForFuse(pKF, targets[t].second, vpMapPoints, &pts[(size_t)t * n]);
        for (int i = 0; i < n; ++i) searched[i] |= pts[(size_t)t * n + i].valid;
    }
    for (int i = 0; i < n; ++i)
        if (searched[i]) CopyDescriptor(vpMapPoints[i], desc, (size_t)i);
    std::vector<int32_t> best((size_t)T * n, -1);
    Check(vsg_fuse_search_multi(Workspace(), T, frames.data(), sigma.data(), n, pts.data(), desc.data(), th, best.data()),
          "vsg_fuse_search_multi");
    // Stale descriptors.  The loop searches target t with the descriptors the map points have when Fuse(target t) starts, and
    // MapPoint::Replace ends with the survivor's ComputeDistinctiveDescriptors(): a survivor that is one of vpMapPoints may
    // enter the later targets with a new descriptor and pick another keypoint there.  So after each target's replay, every
    // query that survived a Replace is compared with its uploaded row; the ones that changed are searched again, with the
    // new rows, in all later targets (one more call), before the next target is replayed.
    std::vector<std::pair<MapPointT *, int>> queryOf;                                         // map point -> its query indices
    for (int i = 0; i < n; ++i)
        if (searched[i]) queryOf.emplace_back(vpMapPoints[i], i);
    std::sort(queryOf.begin(), queryOf.end());
    std::vector<int> survivors, stale;
    auto onReplace = [&](MapPointT *pSurvivor) {
        auto it = std::lower_bound(queryOf.begin(), queryOf.end(), std::make_pair(pSurvivor, 0));
        for (; it != queryOf.end() && it->first == pSurvivor; ++it) survivors.push_back(it->second);
    };
    int nFused = 0;
    for (int t = 0; t < T; ++t) {
        nFused += FuseReplay(targets[t].first, targets[t].second, vpMapPoints, &best[(size_t)t * n], onReplace);
        if (t + 1 == T || survivors.empty()) continue;
        std::sort(survivors.begin(), survivors.end());
        survivors.erase(std::unique(survivors.begin(), survivors.end()), survivors.end());
        stale.clear();
        for (int i : survivors) {
            const cv::Mat d = vpMapPoints[i]->GetDescriptor();
            if (std::memcmp(d.ptr(0), &desc[(size_t)i * 32], 32) == 0) continue;
            std::memcpy(&desc[(size_t)i * 32], d.ptr(0), 32);
            stale.push_back(i);
        }
        survivors.clear();
        if (stale.empty()) continue;
        const int R = T - t - 1, ns = (int)stale.size();
        std::vector<vsg_search_point> rpts((size_t)R * ns);
        std::vector<uint8_t> rdesc((size_t)ns * 32);
        for (int j = 0; j < ns; ++j) {
            std::memcpy(&rdesc[(size_t)j * 32], &desc[(size_t)stale[j] * 32], 32);
            for (int r = 0; r < R; ++r) rpts[(size_t)r * ns + j] = pts[(size_t)(t + 1 + r) * n + stale[j]];
        }
        std::vector<int32_t> rbest((size_t)R * ns);
        Check(vsg_fuse_search_multi(Workspace(), R, frames.data() + t + 1, sigma.data() + t + 1, ns, rpts.data(), rdesc.data(), th,
                                    rbest.data()), "vsg_fuse_search_multi");
        for (int r = 0; r < R; ++r)
            for (int j = 0; j < ns; ++j) best[(size_t)(t + 1 + r) * n + stale[j]] = rbest[(size_t)r * ns + j];
    }
    return nFused;
}

#ifdef SOPHUS_SIM3_HPP
// ---- SearchByProjection(KF, Scw, vpPoints, vpMatched, th, ratioHamming) (ORBmatcher.cc:430-528) ----
template <class KeyFrameT, class MapPointT>
int ORBmatcher::SearchByProjection(KeyFrameT *pKF, Sophus::Sim3<float> &Scw, const std::vector<MapPointT *> &vpPoints,
                                   std::vector<MapPointT *> &vpMatched, int th, float ratioHamming) {
    std::vector<KeyFrameT *> none, none_out;
    return SearchByProjection(pKF, Scw, vpPoints, none, vpMatched, none_out, th, ratioHamming);
}

// ---- ... with vpPointsKFs / vpMatchedKF (ORBmatcher.cc:530-641; the projection is the pinhole fx, fy, cx, cy one) ----
template <class KeyFrameT, class MapPointT>
int ORBmatcher::SearchByProjection(KeyFrameT *pKF, Sophus::Sim3<float> &Scw, const std::vector<MapPointT *> &vpPoints,
                                   const std::vector<KeyFrameT *> &vpPointsKFs, std::vector<MapPointT *> &vpMatched,
                                   std::vector<KeyFrameT *> &vpMatchedKF, int th, float ratioHamming) {
    const bool bWithKFs = !vpPointsKFs.empty();
    Flat flatLocal;
    FrameGuard fr;
    const Flat &flat = Upload(*pKF, pKF->NLeft != -1 ? 1 : 0, [&](Flat &o) { FlattenSearched(*pKF, pKF->NLeft, o); }, flatLocal, fr);
    const float &fx = pKF->fx, &fy = pKF->fy, &cx = pKF->cx, &cy = pKF->cy;
    Sophus::SE3f Tcw = Sophus::SE3f(Scw.rotationMatrix(), Scw.translation() / Scw.scale());
    const auto Ow = Tcw.inverse().translation();
    std::set<MapPointT *> spAlreadyFound(vpMatched.begin(), vpMatched.end());
    spAlreadyFound.erase(static_cast<MapPointT *>(nullptr));
    const int n = (int)vpPoints.size(), N = flat.view.n;
    std::vector<vsg_search_point> pts(n);
    std::vector<uint8_t> desc((size_t)n * 32, 0);
    for (int iMP = 0; iMP < n; ++iMP) {
        vsg_search_point &p = pts[iMP];
        std::memset(&p, 0, sizeof(p));
        MapPointT *pMP = vpPoints[iMP];
        if (pMP->isBad() || spAlreadyFound.count(pMP)) continue;
        const auto p3Dw = pMP->GetWorldPos();
        const auto p3Dc = Tcw * p3Dw;
        if (p3Dc(2) < 0.0) continue;
        float u, v;
        if (bWithKFs) {                                                                     // :567-573
            const float invz = 1 / p3Dc(2);
            const float x = p3Dc(0) * invz, y = p3Dc(1) * invz;
            u = fx * x + cx; v = fy * y + cy;
        } else {                                                                            // :461
            const auto uv = pKF->mpCamera->project(p3Dc);
            u = uv(0); v = uv(1);
        }
        if (!pKF->IsInImage(u, v)) continue;
        if (!DistanceAndNormalGates(pMP, pKF, p3Dw, Ow, true, p)) continue;
        p.u = u; p.v = v;
        p.valid = 1;
        CopyDescriptor(pMP, desc, (size_t)iMP);
    }
    std::vector<uint8_t> matched(N, 0);
    for (int i = 0; i < N; ++i) matched[i] = vpMatched[i] ? 1 : 0;
    std::vector<int32_t> assign(N, -1);
    int nmatches = 0;
    Check(vsg_search_by_projection_sim3(Workspace(), fr.h, matched.data(), n, pts.data(), desc.data(), th, ratioHamming,
                                        assign.data(), &nmatches), "vsg_search_by_projection_sim3");
    for (int i = 0; i < N; ++i)
        if (assign[i] >= 0) {
            vpMatched[i] = vpPoints[assign[i]];                                              // :522 / :634
            if (bWithKFs) vpMatchedKF[i] = vpPointsKFs[assign[i]];                           // :635
        }
    return nmatches;
}

// ---- SearchBySim3 (ORBmatcher.cc:1448-1665) ----
template <class KeyFrameT, class MapPointT>
int ORBmatcher::SearchBySim3(KeyFrameT *pKF1, KeyFrameT *pKF2, std::vector<MapPointT *> &vpMatches12, const Sophus::Sim3f &S12,
                             const float th) {
    const float &fx = pKF1->fx, &fy = pKF1->fy, &cx = pKF1->cx, &cy = pKF1->cy;
    Sophus::SE3f T1w = pKF1->GetPose();
    Sophus::SE3f T2w = pKF2->GetPose();
    Sophus::Sim3f S21 = S12.inverse();
    const std::vector<MapPointT *> vpMapPoints1 = pKF1->GetMapPointMatches();
    const std::vector<MapPointT *> vpMapPoints2 = pKF2->GetMapPointMatches();
    const int N1 = (int)vpMapPoints1.size(), N2 = (int)vpMapPoints2.size();
    std::vector<bool> vbAlreadyMatched1(N1, false), vbAlreadyMatched2(N2, false);
    for (int i = 0; i < N1; i++) {                                                          // :1472-1482
        MapPointT *pMP = vpMatches12[i];
        if (pMP) {
            vbAlreadyMatched1[i] = true;
            int idx2 = std::get<0>(pMP->GetIndexInKeyFrame(pKF2));
            if (idx2 >= 0 && idx2 < N2) vbAlreadyMatched2[idx2] = true;
        }
    }
    Flat f1Local, f2Local;                         // N1 / N2 map point slots (both cameras) search the left cameras' features
    FrameGuard fr1, fr2;
    const Flat &f1 = Upload(*pKF1, pKF1->NLeft != -1 ? 1 : 0, [&](Flat &o) { FlattenSearched(*pKF1, pKF1->NLeft, o); }, f1Local, fr1);
    const Flat &f2 = Upload(*pKF2, pKF2->NLeft != -1 ? 1 : 0, [&](Flat &o) { FlattenSearched(*pKF2, pKF2->NLeft, o); }, f2Local, fr2);
    std::vector<vsg_search_point> pts1(N1), pts2(N2);
    std::vector<uint8_t> desc1((size_t)N1 * 32, 0), desc2((size_t)N2 * 32, 0);
    auto project = [&](const std::vector<MapPointT *> &vp, const std::vector<bool> &already, const Sophus::SE3f &Tw,
                       const Sophus::Sim3f &S, KeyFrameT *pTarget, std::vector<vsg_search_point> &pts, std::vector<uint8_t> &desc) {
        for (int i = 0; i < (int)vp.size(); ++i) {
            vsg_search_point &p = pts[i];
            std::memset(&p, 0, sizeof(p));
            MapPointT *pMP = vp[i];
            if (!pMP || already[i]) continue;
            if (pMP->isBad()) continue;
            const auto p3Dw = pMP->GetWorldPos();
            const auto p3Dca = Tw * p3Dw;
            const auto p3Dcb = S * p3Dca;
            if (p3Dcb(2) < 0.0) continue;
            const float invz = 1.0 / p3Dcb(2);
            const float x = p3Dcb(0) * invz, y = p3Dcb(1) * invz;
            const float u = fx * x + cx, v = fy * y + cy;
            if (!pTarget->IsInImage(u, v)) continue;
            const float maxDistance = pMP->GetMaxDistanceInvariance();
            const float minDistance = pMP->GetMinDistanceInvariance();
            const float dist3D = p3Dcb.norm();
            if (dist3D < minDistance || dist3D > maxDistance) continue;
            p.level = pMP->PredictScale(dist3D, pTarget);
            p.u = u; p.v = v;
            p.valid = 1;
            CopyDescriptor(pMP, desc, (size_t)i);
        }
    };
    project(vpMapPoints1, vbAlreadyMatched1, T1w, S21, pKF2, pts1, desc1);                  // :1488-1560
    project(vpMapPoints2, vbAlreadyMatched2, T2w, S12, pKF1, pts2, desc2);                  // :1563-1635
    std::vector<int32_t> m12(N1, -1);
    int nFound = 0;
    Check(vsg_search_by_sim3(Workspace(), fr1.h, fr2.h, N1, pts1.data(), desc1.data(), N2, pts2.data(), desc2.data(), th,
                             m12.data(), &nFound), "vsg_search_by_sim3");
    for (int i1 = 0; i1 < N1; ++i1)
        if (m12[i1] >= 0) vpMatches12[i1] = vpMapPoints2[m12[i1]];                           // :1648
    return nFound;
}

// ---- Fuse(KF, Scw, vpPoints, th, vpReplacePoint) (ORBmatcher.cc:1337-1446) ----
template <class KeyFrameT, class MapPointT>
int ORBmatcher::Fuse(KeyFrameT *pKF, Sophus::Sim3f &Scw, const std::vector<MapPointT *> &vpPoints, float th,
                     std::vector<MapPointT *> &vpReplacePoint) {
    Flat flatLocal;
    FrameGuard fr;
    const Flat &flat = Upload(*pKF, pKF->NLeft != -1 ? 1 : 0, [&](Flat &o) { FlattenSearched(*pKF, pKF->NLeft, o); }, flatLocal, fr);
    Sophus::SE3f Tcw = Sophus::SE3f(Scw.rotationMatrix(), Scw.translation() / Scw.scale());
    const auto Ow = Tcw.inverse().translation();
    const std::set<MapPointT *> spAlreadyFound = pKF->GetMapPoints();
    const int nPoints = (int)vpPoints.size();
    std::vector<vsg_search_point> pts(nPoints);
    std::vector<uint8_t> desc((size_t)nPoints * 32, 0);
    for (int iMP = 0; iMP < nPoints; ++iMP) {
        vsg_search_point &p = pts[iMP];
        std::memset(&p, 0, sizeof(p));
        MapPointT *pMP = vpPoints[iMP];
        if (spAlreadyFound.count(pMP)) continue;            // isBad() is re-checked in order below
        const auto p3Dw = pMP->GetWorldPos();
        const auto p3Dc = Tcw * p3Dw;
        if (p3Dc(2) < 0.0f) continue;
        const auto uv = pKF->mpCamera->project(p3Dc);
        if (!pKF->IsInImage(uv(0), uv(1))) continue;
        if (!DistanceAndNormalGates(pMP, pKF, p3Dw, Ow, true, p)) continue;
        p.u = uv(0); p.v = uv(1);
        p.valid = 1;
        CopyDescriptor(pMP, desc, (size_t)iMP);
    }
    std::vector<int32_t> best(nPoints, -1);
    Check(vsg_fuse_search(Workspace(), fr.h, nPoints, pts.data(), desc.data(), th, nullptr, 1, best.data(), nullptr),
          "vsg_fuse_search");
    int nFused = 0;
    for (int iMP = 0; iMP < nPoints; ++iMP) {                                               // :1353-1442 in order
        MapPointT *pMP = vpPoints[iMP];
        if (pMP->isBad() || best[iMP] < 0) continue;
        MapPointT *pMPinKF = pKF->GetMapPoint(best[iMP]);
        if (pMPinKF) {
            if (!pMPinKF->isBad()) vpReplacePoint[iMP] = pMPinKF;
        } else {
            pMP->AddObservation(pKF, best[iMP]);
            pKF->AddMapPoint(pMP, best[iMP]);
        }
        nFused++;
    }
    return nFused;
}
#endif  // SOPHUS_SIM3_HPP

// ---- SearchForTriangulation (ORBmatcher.cc:902-1146) ----
template <class KeyFrameT>
void ORBmatcher::TriangulationGeometry(KeyFrameT *pKF1, KeyFrameT *pKF2, bool bCoarse, float f12[9], float epf[2]) {
    const auto T1w = pKF1->GetPose();
    const auto T2w = pKF2->GetPose();
    const auto Tw2 = pKF2->GetPoseInverse();
    const auto Cw = pKF1->GetCameraCenter();
    const auto C2 = T2w * Cw;
    const auto ep = pKF2->mpCamera->project(C2);
    const auto T12 = T1w * Tw2;
    const auto R12 = T12.rotationMatrix();
    const auto t12 = T12.translation();
    for (int k = 0; k < 9; ++k) f12[k] = 0;
    if (!bCoarse) {
        typename std::decay<decltype(R12)>::type t12x;
        t12x << 0, -t12(2), t12(1), t12(2), 0, -t12(0), -t12(1), t12(0), 0;                 // Sophus::SO3f::hat(t12)
        const auto K1 = pKF1->mpCamera->toK_();
        const auto K2 = pKF2->mpCamera->toK_();
        const typename std::decay<decltype(R12)>::type F12 = K1.transpose().inverse() * t12x * R12 * K2.inverse();
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) f12[3 * r + c] = F12(r, c);
    }
    epf[0] = ep(0);
    epf[1] = ep(1);
}

template <class KeyFrameT>
int ORBmatcher::SearchForTriangulation(KeyFrameT *pKF1, KeyFrameT *pKF2, std::vector<std::pair<size_t, size_t>> &vMatchedPairs,
                                       const bool bOnlyStereo, const bool bCoarse) {
    if (TwoCameraKF(pKF1) || TwoCameraKF(pKF2)) return SearchForTriangulationTwoCameras(pKF1, pKF2, vMatchedPairs, bOnlyStereo, bCoarse);
    float f12[9], epf[2];
    TriangulationGeometry(pKF1, pKF2, bCoarse, f12, epf);
    BowSide k1, k2;
    FlattenTriangulationSide(*pKF1, k1);
    FlattenTriangulationSide(*pKF2, k2);
    const vsg_bow_side &s1 = k1.side, &s2 = k2.side;
    std::vector<int32_t> m12(s1.view.n, -1);
    int nmatches = 0;
    Check(vsg_search_for_triangulation(Workspace(), &s1.view, s1.mp_valid, &s2.view, s2.mp_valid, s1.nnodes, s1.nodes, s1.ptr, s1.idx,
                                       s2.nnodes, s2.nodes, s2.ptr, s2.idx, bOnlyStereo ? 1 : 0, bCoarse ? 1 : 0, f12, epf,
                                       pKF2->mvLevelSigma2.data(), mbCheckOrientation ? 1 : 0, m12.data(), &nmatches),
          "vsg_search_for_triangulation");
    vMatchedPairs.clear();
    vMatchedPairs.reserve(nmatches);
    for (size_t i = 0, iend = m12.size(); i < iend; i++) {                                  // :1136-1143
        if (m12[i] < 0) continue;
        vMatchedPairs.push_back(std::make_pair(i, (size_t)m12[i]));
    }
    return nmatches;
}

template <class KeyFrameT>
struct ORBmatcher::TriangulationSearch {
    KeyFrameT *pKF1 = nullptr;
    std::vector<KeyFrameT *> vpKF2s;
    bool bOnlyStereo = false, bCoarse = false;
    // what the batch call searched with: KF1, every target (row[t] = its row of best12, -1 if it was not batched), and
    // each target's f12 and epipole (11 floats)
    std::unique_ptr<BowSide> k1;
    std::vector<BowSide> k2;
    std::vector<int> row;
    std::vector<float> geom;
    std::vector<int32_t> best12;
};

template <class KeyFrameT>
ORBmatcher::TriangulationSearch<KeyFrameT> ORBmatcher::SearchForTriangulation(KeyFrameT *pKF1, const std::vector<KeyFrameT *> &vpKF2s,
                                                                              const bool bOnlyStereo, const bool bCoarse) {
    TriangulationSearch<KeyFrameT> s;
    const size_t T = vpKF2s.size();
    s.pKF1 = pKF1;
    s.vpKF2s = vpKF2s;
    s.bOnlyStereo = bOnlyStereo;
    s.bCoarse = bCoarse;
    s.k2 = std::vector<BowSide>(T);
    s.row.assign(T, -1);
    s.geom.assign(T * 11, 0.f);
    if (TwoCameraKF(pKF1)) return s;                                                       // all targets take the single call
    s.k1.reset(new BowSide());
    FlattenTriangulationSide(*pKF1, *s.k1);
    std::vector<vsg_triangulation_target> tgs;
    tgs.reserve(T);
    for (size_t t = 0; t < T; ++t) {
        KeyFrameT *pKF2 = vpKF2s[t];
        if (TwoCameraKF(pKF2)) continue;
        FlattenTriangulationSide(*pKF2, s.k2[t]);
        float *g = &s.geom[t * 11];
        TriangulationGeometry(pKF1, pKF2, bCoarse, g, g + 9);
        vsg_triangulation_target tg;
        tg.kf2 = s.k2[t].side;
        std::memcpy(tg.f12, g, sizeof tg.f12);
        std::memcpy(tg.ep, g + 9, sizeof tg.ep);
        tg.level_sigma2 = pKF2->mvLevelSigma2.data();
        s.row[t] = (int)tgs.size();
        tgs.push_back(tg);
    }
    std::vector<const vsg_triangulation_target *> table(tgs.size());
    for (size_t r = 0; r < tgs.size(); ++r) table[r] = &tgs[r];
    s.best12.assign(tgs.size() * (size_t)s.k1->flat.view.n, -1);
    Check(vsg_triangulation_candidates_multi(Workspace(), &s.k1->side, (int)tgs.size(), table.data(), bOnlyStereo ? 1 : 0,
                                             bCoarse ? 1 : 0, s.best12.data()), "vsg_triangulation_candidates_multi");
    return s;
}

template <class KeyFrameT>
int ORBmatcher::SearchForTriangulation(TriangulationSearch<KeyFrameT> &search, size_t i,
                                       std::vector<std::pair<size_t, size_t>> &vMatchedPairs) {
    KeyFrameT *pKF1 = search.pKF1, *pKF2 = search.vpKF2s.at(i);
    const int r = search.row[i];
    bool current = r >= 0;
    const BowSide &k2 = search.k2[i];
    for (int j = 0; current && j < k2.flat.view.n; ++j)                                    // the target's map-point slots
        current = (pKF2->GetMapPoint(j) != nullptr) == (k2.valid[j] != 0);
    if (current) {                                                                          // both poses
        float g[11];
        TriangulationGeometry(pKF1, pKF2, search.bCoarse, g, g + 9);
        current = std::memcmp(g, &search.geom[i * 11], sizeof g) == 0;
    }
    const int n1 = current ? search.k1->flat.view.n : 0;
    const int32_t *best = current ? &search.best12[(size_t)r * n1] : nullptr;
    std::vector<uint8_t> h1(n1);
    for (int j = 0; current && j < n1; ++j) {                                               // KF1's map points: gained, never lost
        h1[j] = pKF1->GetMapPoint(j) ? 1 : 0;
        current = best[j] != -2 || h1[j];
    }
    if (!current) return SearchForTriangulation(pKF1, pKF2, vMatchedPairs, search.bOnlyStereo, search.bCoarse);
    std::vector<int32_t> m12(n1, -1);
    int nmatches = 0;
    Check(vsg_triangulation_resolve(&search.k1->flat.view, &k2.flat.view, h1.data(), best, mbCheckOrientation ? 1 : 0, m12.data(),
                                    &nmatches), "vsg_triangulation_resolve");
    vMatchedPairs.clear();
    vMatchedPairs.reserve(nmatches);
    for (int j = 0; j < n1; j++)                                                            // :1136-1143
        if (m12[j] >= 0) vMatchedPairs.push_back(std::make_pair((size_t)j, (size_t)m12[j]));
    return nmatches;
}

// ---- SearchForTriangulation on two-camera keyframes (ORBmatcher.cc:902-1146 with mpCamera2 != NULL) ----
// The descriptor distances of every BoW-paired candidate come from the GPU (vsg_bow_pair_distances); the loop is replayed
// here in the reference's order because its per-pair test is the caller's camera code: which of the four camera pairs
// (left / right of either keyframe) a pair belongs to selects R12 / t12 and the two GeometricCamera objects whose
// epipolarConstrain — KannalaBrandt8's triangulation for fisheye rigs — decides (:1033-1077).
template <class KeyFrameT>
int ORBmatcher::SearchForTriangulationTwoCameras(KeyFrameT *pKF1, KeyFrameT *pKF2,
                                                 std::vector<std::pair<size_t, size_t>> &vMatchedPairs, const bool bOnlyStereo,
                                                 const bool bCoarse) {
    const auto T1w = pKF1->GetPose();
    const auto T2w = pKF2->GetPose();
    const auto Tw2 = pKF2->GetPoseInverse();
    const auto Cw = pKF1->GetCameraCenter();
    const auto C2 = T2w * Cw;
    const auto ep = pKF2->mpCamera->project(C2);
    typedef typename std::decay<decltype(T1w)>::type SE3T;
    SE3T T12, Tll, Tlr, Trl, Trr;
    typename std::decay<decltype(T12.rotationMatrix())>::type R12;
    typename std::decay<decltype(T12.translation())>::type t12;
    auto *pCamera1 = pKF1->mpCamera;
    auto *pCamera2 = pKF2->mpCamera;
    if (!pKF1->mpCamera2 && !pKF2->mpCamera2) {                                              // :922-928
        T12 = T1w * Tw2;
        R12 = T12.rotationMatrix();
        t12 = T12.translation();
    } else {                                                                                 // :929-937
        const auto Tr1w = pKF1->GetRightPose();
        const auto Twr2 = pKF2->GetRightPoseInverse();
        Tll = T1w * Tw2;
        Tlr = T1w * Twr2;
        Trl = Tr1w * Tw2;
        Trr = Tr1w * Twr2;
    }
    const auto Rll = Tll.rotationMatrix(), Rlr = Tlr.rotationMatrix(), Rrl = Trl.rotationMatrix(), Rrr = Trr.rotationMatrix();
    const auto tll = Tll.translation(), tlr = Tlr.translation(), trl = Trl.translation(), trr = Trr.translation();

    // all features of both cameras, in mDescriptors / mFeatVec index order
    Flat k1, k2;
    if (pKF1->NLeft != -1) FlattenBothCameras(*pKF1, k1); else Flatten(*pKF1, k1);
    if (pKF2->NLeft != -1) FlattenBothCameras(*pKF2, k2); else Flatten(*pKF2, k2);
    const int n1 = k1.view.n, n2 = k2.view.n;
    auto stereo1 = [&](size_t i) { return !pKF1->mpCamera2 && pKF1->mvuRight[i] >= 0; };     // :977
    auto stereo2 = [&](size_t i) { return !pKF2->mpCamera2 && pKF2->mvuRight[i] >= 0; };     // :1005
    std::vector<uint8_t> use1(n1, 0);
    for (int i = 0; i < n1; ++i) use1[i] = !pKF1->GetMapPoint(i) && (!bOnlyStereo || stereo1(i));   // :968-981
    std::vector<int32_t> nd1, p1, i1v, nd2, p2, i2v;
    FlattenFeatVec(pKF1->mFeatVec, nd1, p1, i1v);
    FlattenFeatVec(pKF2->mFeatVec, nd2, p2, i2v);
    std::vector<int32_t> q1(n1 + 1), cptr(n1 + 2), cand, dist;
    int nq = 0, total = 0;
    size_t cap = (size_t)std::max(1024, 32 * n1);
    for (int attempt = 0; attempt < 2; ++attempt) {
        cand.resize(cap);
        dist.resize(cap);
        const vsg_status st = vsg_bow_pair_distances(Workspace(), &k1.view, use1.data(), &k2.view, (int)nd1.size(), nd1.data(), p1.data(),
                                                     i1v.data(), (int)nd2.size(), nd2.data(), p2.data(), i2v.data(), q1.data(),
                                                     cptr.data(), n1 + 1, cand.data(), dist.data(), (int)cap, &nq, &total);
        if (st == VSG_ERR_CAPACITY && attempt == 0) { cap = (size_t)total + 1; continue; }
        Check(st, "vsg_bow_pair_distances");
        break;
    }
    auto key_of = [](KeyFrameT *kf, size_t idx) -> const cv::KeyPoint & {                    // :982-984, :1017-1019
        return (kf->NLeft == -1) ? kf->mvKeysUn[idx] : ((int)idx < kf->NLeft) ? kf->mvKeys[idx] : kf->mvKeysRight[idx - kf->NLeft];
    };
    int nmatches = 0;
    std::vector<int> vMatches12(pKF1->N, -1);
    std::vector<int> rotHist[HISTO_LENGTH];
    const float factor = 1.0f / HISTO_LENGTH;
    for (int k = 0; k < nq; ++k) {
        const size_t idx1 = (size_t)q1[k];
        const bool bStereo1 = stereo1(idx1);
        const cv::KeyPoint &kp1 = key_of(pKF1, idx1);
        const bool bRight1 = !(pKF1->NLeft == -1 || (int)idx1 < pKF1->NLeft);
        int bestDist = TH_LOW, bestIdx2 = -1;
        for (int c = cptr[k]; c < cptr[k + 1]; ++c) {
            const size_t idx2 = (size_t)cand[c];
            if (pKF2->GetMapPoint(idx2)) continue;                                           // :1001 (vbMatched2 is never set)
            const bool bStereo2 = stereo2(idx2);
            if (bOnlyStereo && !bStereo2) continue;
            const int d = dist[c];
            if (d > TH_LOW || d > bestDist) continue;                                        // :1014
            const cv::KeyPoint &kp2 = key_of(pKF2, idx2);
            const bool bRight2 = !(pKF2->NLeft == -1 || (int)idx2 < pKF2->NLeft);
            if (!bStereo1 && !bStereo2 && !pKF1->mpCamera2) {                                // :1023-1031
                const float distex = ep(0) - kp2.pt.x;
                const float distey = ep(1) - kp2.pt.y;
                if (distex * distex + distey * distey < 100 * pKF2->mvScaleFactors[kp2.octave]) continue;
            }
            if (pKF1->mpCamera2 && pKF2->mpCamera2) {                                        // :1033-1070
                if (bRight1 && bRight2) { R12 = Rrr; t12 = trr; T12 = Trr; pCamera1 = pKF1->mpCamera2; pCamera2 = pKF2->mpCamera2; }
                else if (bRight1 && !bRight2) { R12 = Rrl; t12 = trl; T12 = Trl; pCamera1 = pKF1->mpCamera2; pCamera2 = pKF2->mpCamera; }
                else if (!bRight1 && bRight2) { R12 = Rlr; t12 = tlr; T12 = Tlr; pCamera1 = pKF1->mpCamera; pCamera2 = pKF2->mpCamera2; }
                else { R12 = Rll; t12 = tll; T12 = Tll; pCamera1 = pKF1->mpCamera; pCamera2 = pKF2->mpCamera; }
            }
            if (bCoarse || pCamera1->epipolarConstrain(pCamera2, kp1, kp2, R12, t12, pKF1->mvLevelSigma2[kp1.octave],
                                                       pKF2->mvLevelSigma2[kp2.octave])) {
                bestIdx2 = (int)idx2;
                bestDist = d;
            }
        }
        if (bestIdx2 >= 0) {                                                                 // :1080-1100
            const cv::KeyPoint &kp2 = key_of(pKF2, (size_t)bestIdx2);
            vMatches12[idx1] = bestIdx2;
            nmatches++;
            if (mbCheckOrientation) {
                float rot = kp1.angle - kp2.angle;
                if (rot < 0.0) rot += 360.0f;
                int bin = round(rot * factor);
                if (bin == HISTO_LENGTH) bin = 0;
                rotHist[bin].push_back((int)idx1);
            }
        }
    }
    if (mbCheckOrientation) {                                                                // :1120-1137
        int ind1 = -1, ind2 = -1, ind3 = -1;
        ComputeThreeMaxima(rotHist, HISTO_LENGTH, ind1, ind2, ind3);
        for (int i = 0; i < HISTO_LENGTH; i++) {
            if (i == ind1 || i == ind2 || i == ind3) continue;
            for (size_t j = 0, jend = rotHist[i].size(); j < jend; j++) {
                vMatches12[rotHist[i][j]] = -1;
                nmatches--;
            }
        }
    }
    vMatchedPairs.clear();
    vMatchedPairs.reserve(nmatches);
    for (size_t i = 0, iend = vMatches12.size(); i < iend; i++) {
        if (vMatches12[i] < 0) continue;
        vMatchedPairs.push_back(std::make_pair(i, (size_t)vMatches12[i]));
    }
    (void)n2;
    return nmatches;
}

}  // namespace VS_GRAPHS

namespace ORB_SLAM3 {
using VS_GRAPHS::ORBmatcher;
}

#endif
