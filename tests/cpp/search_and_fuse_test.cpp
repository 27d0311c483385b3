// search_and_fuse_test.cpp — the batched VS_GRAPHS::ORBmatcher::Fuse(vpKFs, vScw, vpPoints, th) + Fuse(search, k,
// vpReplacePoint) against the loop it stands for, LoopClosing::SearchAndFuse (LoopClosing.cc:1994-2054):
//     for (k) { vector<MapPoint*> vpReplacePoints(vpPoints.size(), NULL);
//               matcher.Fuse(vpKFs[k], vScw[k], vpPoints, 4, vpReplacePoints);
//               for (i) if (MapPoint* pRep = vpReplacePoints[i]) pRep->Replace(vpPoints[i]); }
// Each world is generated twice from one seed; the loop of single-target Fuse(KF, Scw, ...) calls runs on one copy, the batch
// and its resolves (with the same Replace loop in between) on the other.  Both worlds must end identical: every keyframe's
// map-point slots, every map point's observations, bad flag, replacedBy and descriptor, and every vpReplacePoints vector and
// count.  The stand-in MapPoint::Replace moves the observations as KeyFrame::ReplaceMapPointMatch / EraseMapPointMatch do
// and recomputes the survivor's descriptor as MapPoint::ComputeDistinctiveDescriptors does (MapPoint.cc:340-417); the
// stand-in KeyFrame::GetMapPoints skips bad points.  The constructed worlds pin what a resolve must read at resolve time.
//
// Two builds: with tests/cpp/vsg_on_oracle.cpp + tests/cpp/vsg_on_oracle_sim3_multi.cpp + oracle/liborb_oracle.so (no GPU),
// and with -lvsg_cuda (B200).
//   usage: search_and_fuse_test            the checks
//          search_and_fuse_test --time     also times the loop against the batch + resolves (host projection included)
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <random>
#include <set>
#include <string>
#include <vector>

// ---- stand-ins for Eigen / Sophus (only what the shim's Sim3 Fuse uses) ----
struct Vec3 {
    float v[3];
    float operator()(int i) const { return v[i]; }
    Vec3 operator-(const Vec3 &o) const { return Vec3{{v[0] - o.v[0], v[1] - o.v[1], v[2] - o.v[2]}}; }
    Vec3 operator+(const Vec3 &o) const { return Vec3{{v[0] + o.v[0], v[1] + o.v[1], v[2] + o.v[2]}}; }
    Vec3 operator*(float s) const { return Vec3{{v[0] * s, v[1] * s, v[2] * s}}; }
    Vec3 operator/(float s) const { return Vec3{{v[0] / s, v[1] / s, v[2] / s}}; }
    float dot(const Vec3 &o) const { return v[0] * o.v[0] + v[1] * o.v[1] + v[2] * o.v[2]; }
    float norm() const { return std::sqrt(dot(*this)); }
};
struct Vec2 {
    float v[2];
    float operator()(int i) const { return v[i]; }
};
struct Mat3 {
    float m[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    Mat3 transpose() const { Mat3 t; for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) t.m[3 * r + c] = m[3 * c + r]; return t; }
    Vec3 operator*(const Vec3 &p) const {
        return Vec3{{m[0] * p.v[0] + m[1] * p.v[1] + m[2] * p.v[2], m[3] * p.v[0] + m[4] * p.v[1] + m[5] * p.v[2],
                     m[6] * p.v[0] + m[7] * p.v[1] + m[8] * p.v[2]}};
    }
    static Mat3 yaw(float a) { Mat3 R; R.m[0] = std::cos(a); R.m[2] = std::sin(a); R.m[6] = -std::sin(a); R.m[8] = std::cos(a); return R; }
};
namespace Sophus {
struct SE3f {
    Mat3 R;
    Vec3 t{{0, 0, 0}};
    SE3f() {}
    SE3f(const Mat3 &R_, const Vec3 &t_) : R(R_), t(t_) {}
    SE3f inverse() const { Mat3 Rt = R.transpose(); Vec3 nt = Rt * t; return SE3f(Rt, nt * -1.f); }
    Vec3 translation() const { return t; }
    Mat3 rotationMatrix() const { return R; }
    Vec3 operator*(const Vec3 &p) const { return R * p + t; }
};
template <class T>
struct Sim3 {   // p -> s R p + t
    Mat3 R;
    Vec3 t{{0, 0, 0}};
    T s = 1;
    Mat3 rotationMatrix() const { return R; }
    Vec3 translation() const { return t; }
    T scale() const { return s; }
    Sim3 inverse() const { Sim3 o; o.R = R.transpose(); o.s = 1 / s; o.t = (o.R * t) * (-1 / s); return o; }
};
using Sim3f = Sim3<float>;
}  // namespace Sophus
#define SOPHUS_SIM3_HPP

#include "../../visual_sgraphs_b200/shim/ORBmatcher.h"

static int g_fail = 0;
#define EXPECT(cond, ...)                                                                                                   \
    do {                                                                                                                    \
        if (!(cond)) { std::printf("FAIL %s:%d: ", __FILE__, __LINE__); std::printf(__VA_ARGS__); std::printf("\n"); ++g_fail; } \
    } while (0)

constexpr int kLevels = 8;
constexpr float kScale = 1.2f;
static unsigned long g_next_kf_id = 0;

struct Camera {
    float fx = 500, fy = 500, cx = 320, cy = 240;
    Vec2 project(const Vec3 &p) const { return Vec2{{fx * p.v[0] / p.v[2] + cx, fy * p.v[1] / p.v[2] + cy}}; }
};

struct MapPoint;
struct KeyFrame {
    int index = 0;                                   // position in its world (for comparisons across the two copies)
    unsigned long mnId = g_next_kf_id++;
    int N = 0, NLeft = -1;
    std::vector<cv::KeyPoint> mvKeys, mvKeysUn, mvKeysRight;
    cv::Mat mDescriptors;
    std::vector<float> mvuRight, mvScaleFactors;
    std::vector<MapPoint *> mvpMapPoints;
    float mnMinX = 0, mnMinY = 0, mnMaxX = 640, mnMaxY = 480;
    float mfGridElementWidthInv = 64.f / 640.f, mfGridElementHeightInv = 48.f / 480.f;
    float mfLogScaleFactor = std::log(kScale);
    int mnScaleLevels = kLevels;
    Camera cam;
    Camera *mpCamera = &cam;
    KeyFrame() {
        float s = 1.f;
        for (int l = 0; l < kLevels; ++l, s *= kScale) mvScaleFactors.push_back(s);
    }
    bool IsInImage(float x, float y) const { return x >= mnMinX && x < mnMaxX && y >= mnMinY && y < mnMaxY; }
    MapPoint *GetMapPoint(size_t i) const { return mvpMapPoints[i]; }
    void AddMapPoint(MapPoint *p, size_t i) { mvpMapPoints[i] = p; }
    std::set<MapPoint *> GetMapPoints() const;       // KeyFrame.cc: the slots' points that are not bad
};

static int hamming(const uint8_t *a, const uint8_t *b) {
    int d = 0;
    for (int i = 0; i < 32; ++i) d += __builtin_popcount((unsigned)(a[i] ^ b[i]));
    return d;
}

struct MapPoint {
    int id = 0;
    bool query = false;                              // one of vpPoints
    bool bad = false;
    MapPoint *replaced_by = nullptr;
    Vec3 pos{{0, 0, 5}}, normal{{0, 0, 1}};
    float max_dist = 10, min_dist = 0.1f;
    std::map<unsigned long, std::pair<KeyFrame *, int>> obs;   // by keyframe id: the same order in both copies of a world
    cv::Mat desc{1, 32, CV_8UC1};
    static int desc_changes;                         // descriptors of queries changed by a Replace

    bool isBad() const { return bad; }
    cv::Mat GetDescriptor() const { return desc.clone(); }
    Vec3 GetWorldPos() const { return pos; }
    Vec3 GetNormal() const { return normal; }
    float GetMaxDistanceInvariance() const { return max_dist; }
    float GetMinDistanceInvariance() const { return min_dist; }
    template <class T> int PredictScale(float dist, T *pF) const {      // MapPoint.cc:533-565
        int nScale = (int)std::ceil(std::log(max_dist / dist) / pF->mfLogScaleFactor);
        return nScale < 0 ? 0 : (nScale >= pF->mnScaleLevels ? pF->mnScaleLevels - 1 : nScale);
    }
    bool IsInKeyFrame(const KeyFrame *kf) const { return obs.count(kf->mnId) != 0; }
    void AddObservation(KeyFrame *kf, int idx) {
        if (!obs.count(kf->mnId)) obs[kf->mnId] = std::make_pair(kf, idx);
    }
    // MapPoint.cc:340-417: the observed descriptor with the smallest median distance to the others (first on ties)
    void ComputeDistinctiveDescriptors() {
        if (bad || obs.empty()) return;
        std::vector<const uint8_t *> d;
        for (auto &kv : obs) d.push_back(kv.second.first->mDescriptors.ptr(kv.second.second));
        const size_t N = d.size();
        int best_median = INT32_MAX, best_idx = 0;
        for (size_t i = 0; i < N; ++i) {
            std::vector<int> dist(N);
            for (size_t j = 0; j < N; ++j) dist[j] = hamming(d[i], d[j]);
            std::sort(dist.begin(), dist.end());
            const int median = dist[(size_t)(0.5 * (N - 1))];
            if (median < best_median) { best_median = median; best_idx = (int)i; }
        }
        if (query && !bad && std::memcmp(desc.ptr(0), d[best_idx], 32) != 0) ++desc_changes;
        std::memcpy(desc.ptr(0), d[best_idx], 32);
    }
    // MapPoint.cc:216-270: the observations move to the survivor (KeyFrame::ReplaceMapPointMatch), or are erased where it is
    // already observed (EraseMapPointMatch); the survivor recomputes its descriptor
    void Replace(MapPoint *o) {
        if (o == this) return;
        auto moved = obs;
        obs.clear();
        bad = true;
        replaced_by = o;
        for (auto &kv : moved) {
            KeyFrame *kf = kv.second.first;
            const int idx = kv.second.second;
            if (!o->IsInKeyFrame(kf)) { kf->mvpMapPoints[idx] = o; o->AddObservation(kf, idx); }
            else kf->mvpMapPoints[idx] = nullptr;
        }
        o->ComputeDistinctiveDescriptors();
    }
};
int MapPoint::desc_changes = 0;

std::set<MapPoint *> KeyFrame::GetMapPoints() const {
    std::set<MapPoint *> s;
    for (MapPoint *p : mvpMapPoints)
        if (p && !p->isBad()) s.insert(p);
    return s;
}

struct World {
    std::vector<std::unique_ptr<KeyFrame>> kfs;     // targets, then background keyframes
    std::vector<std::unique_ptr<MapPoint>> mps;     // queries, then other map points
    std::vector<KeyFrame *> targets;                // may list a keyframe twice
    std::vector<Sophus::Sim3f> scw;
    std::vector<MapPoint *> vp;
    KeyFrame *add_kf() { kfs.emplace_back(new KeyFrame()); kfs.back()->index = (int)kfs.size() - 1; return kfs.back().get(); }
    MapPoint *add_mp() { mps.emplace_back(new MapPoint()); mps.back()->id = (int)mps.size() - 1; return mps.back().get(); }
};

// keyframe rows are collected first and become mDescriptors once the keyframe is complete
struct Rows {
    std::vector<std::vector<uint8_t>> r;
    int add(const uint8_t *d) { r.emplace_back(d, d + 32); return (int)r.size() - 1; }
    void to(KeyFrame *kf) const {
        kf->mDescriptors.create((int)r.size(), 32, CV_8UC1);
        for (size_t i = 0; i < r.size(); ++i) std::memcpy(kf->mDescriptors.ptr((int)i), r[i].data(), 32);
    }
};

static void flip_bits(std::vector<uint8_t> &d, int nbits, std::mt19937 &rng) {
    for (int k = 0; k < nbits; ++k) { const unsigned b = rng() % 256; d[b / 8] ^= (uint8_t)(1u << (b % 8)); }
}
static std::vector<uint8_t> random_desc(std::mt19937 &rng) {
    std::vector<uint8_t> d(32);
    for (auto &x : d) x = (uint8_t)(rng() & 255);
    return d;
}
static float uni(std::mt19937 &rng, float a, float b) { return a + (b - a) * (float)(rng() % 1000000) / 1e6f; }
static cv::KeyPoint keypoint(float x, float y, int octave) {
    cv::KeyPoint k;
    k.pt.x = x; k.pt.y = y; k.octave = octave; k.size = 31.f; k.angle = 0.f;
    return k;
}
static Sophus::SE3f pose_of(const Sophus::Sim3f &S) { return Sophus::SE3f(S.R, S.t / S.s); }   // as the shim reads Scw
static int level_in(MapPoint *p, KeyFrame *kf, const Sophus::Sim3f &S) {
    return p->PredictScale((p->pos - pose_of(S).inverse().translation()).norm(), kf);
}

// A random world: nkf target keyframes, nq query map points and as many other map points.  Every map point is observed in
// 1-3 background keyframes with its own descriptor plus noise.  Every target gets a Sim3 pose (rotation, translation, scale)
// and keypoints near the projections of a share of the points (about kp_per_target of them, some with a near twin) with noisy
// descriptors, plus distractors.  Target 2 is a two-camera keyframe (Fuse searches its left camera), target 4 has no
// keypoints, the last target repeats target 1.  A quarter of the keypoints hold their own map point, a quarter another one:
// the queries that match those are fused by the caller's Replace.  Some queries are bad from the start, some are listed twice.
static void random_world(World &w, unsigned seed, int nkf, int nq, int kp_per_target = 0) {
    std::mt19937 rng(seed);
    const int np = 2 * nq;
    const float keep = kp_per_target > 0 ? std::min(1.f, (float)kp_per_target / np) : 0.5f;
    std::vector<std::vector<uint8_t>> ident(np);
    for (int i = 0; i < np; ++i) {
        MapPoint *p = w.add_mp();
        p->query = i < nq;
        p->pos = Vec3{{uni(rng, -3.f, 3.f), uni(rng, -2.f, 2.f), uni(rng, 4.f, 9.f)}};
        p->normal = p->pos * (1.f / p->pos.norm());
        p->max_dist = p->pos.norm() * std::pow(kScale, uni(rng, 0.5f, 7.5f));
        p->min_dist = 0.2f * p->pos.norm();
        ident[i] = random_desc(rng);
    }
    const int ndistinct = nkf > 2 ? nkf - 1 : nkf;
    for (int k = 0; k < ndistinct; ++k) w.targets.push_back(w.add_kf());
    std::vector<KeyFrame *> bg;
    std::vector<Rows> bg_rows(3);
    for (int b = 0; b < 3; ++b) bg.push_back(w.add_kf());
    for (int i = 0; i < np; ++i) {
        const int nobs = 1 + rng() % 3;
        for (int b = 0; b < nobs; ++b) {
            std::vector<uint8_t> d = ident[i];
            flip_bits(d, rng() % 24, rng);
            w.mps[i]->AddObservation(bg[b], bg_rows[b].add(d.data()));
        }
    }
    for (int b = 0; b < 3; ++b) {
        bg_rows[b].to(bg[b]);
        bg[b]->N = (int)bg_rows[b].r.size();
        bg[b]->mvpMapPoints.assign(bg[b]->N, nullptr);
    }
    for (auto &mp : w.mps)
        for (auto &kv : mp->obs) kv.second.first->mvpMapPoints[kv.second.second] = mp.get();
    for (int k = 0; k < ndistinct; ++k) {
        KeyFrame *kf = w.targets[k];
        Sophus::Sim3f S;
        S.R = Mat3::yaw(uni(rng, -0.05f, 0.05f));
        S.s = uni(rng, 0.7f, 1.4f);
        S.t = Vec3{{uni(rng, -0.3f, 0.3f), uni(rng, -0.2f, 0.2f), uni(rng, -0.3f, 0.3f)}} * S.s;
        w.scw.push_back(S);
        const Sophus::SE3f T = pose_of(S);
        const bool two = k == 2, empty = k == 4;
        Rows rows;
        std::vector<int> owner;                       // map point a keypoint was made from (-1 distractor)
        for (int c = 0; c < (two ? 2 : 1) && !empty; ++c) {
            std::vector<std::pair<cv::KeyPoint, std::pair<int, std::vector<uint8_t>>>> kps;
            for (int i = 0; i < np; ++i) {
                if (uni(rng, 0.f, 1.f) >= keep) continue;
                const Vec3 pc = T * w.mps[i]->pos;
                const Vec2 uv = kf->cam.project(pc);
                if (c == 0 && !kf->IsInImage(uv(0), uv(1))) continue;
                const int lvl = level_in(w.mps[i].get(), kf, S);
                const int twins = rng() % 4 == 0 ? 2 : 1;
                for (int t = 0; t < twins; ++t) {
                    std::vector<uint8_t> d = ident[i];
                    flip_bits(d, rng() % 40, rng);
                    const int o = std::max(0, lvl - (int)(rng() % 2));
                    const float x = c ? uni(rng, 0, 639.9f) : uv(0) + uni(rng, -0.8f, 0.8f), y = c ? uni(rng, 0, 479.9f) : uv(1) + uni(rng, -0.8f, 0.8f);
                    kps.push_back({keypoint(x, y, o), {i, d}});
                }
            }
            const int ndis = std::max(60, (int)kps.size() / 10);
            for (int j = 0; j < ndis; ++j)
                kps.push_back({keypoint(uni(rng, 0, 639.9f), uni(rng, 0, 479.9f), rng() % kLevels), {-1, random_desc(rng)}});
            std::shuffle(kps.begin(), kps.end(), rng);
            for (auto &e : kps) {
                (c ? kf->mvKeysRight : kf->mvKeys).push_back(e.first);
                rows.add(e.second.second.data());
                owner.push_back(e.second.first);
            }
        }
        kf->NLeft = two ? (int)kf->mvKeys.size() : -1;
        kf->N = (int)owner.size();
        kf->mvKeysUn = kf->mvKeys;
        rows.to(kf);
        kf->mvpMapPoints.assign(kf->N, nullptr);
        for (int j = 0; j < kf->N; ++j) {
            if (owner[j] < 0) continue;
            const unsigned r = rng() % 4;
            MapPoint *p = r == 0 ? w.mps[owner[j]].get() : r == 1 ? w.mps[rng() % np].get() : nullptr;
            if (!p || p->IsInKeyFrame(kf)) continue;
            kf->mvpMapPoints[j] = p;
            p->AddObservation(kf, j);
        }
    }
    if (nkf > 2) { w.targets.push_back(w.targets[1]); w.scw.push_back(w.scw[1]); }
    for (auto &mp : w.mps) mp->ComputeDistinctiveDescriptors();
    for (int i = 0; i < nq; ++i) {
        w.vp.push_back(w.mps[i].get());
        if (rng() % 40 == 1) w.mps[i]->bad = true;
    }
    for (size_t i = 0; i + 1 < w.vp.size(); i += 23) w.vp[i + 1] = w.vp[i];   // a map point listed twice
}

// Two query points P, Q and a keyframe pair T0, T1 with identity Sim3 poses (T1 slightly moved); set up by the callers.
struct Pair {
    MapPoint *P, *Q;
    KeyFrame *T0, *T1;
};
static Pair pair_world(World &w) {
    Pair c;
    c.P = w.add_mp(); c.Q = w.add_mp();
    c.P->query = c.Q->query = true;
    c.P->pos = Vec3{{-1.f, 0.5f, 6.f}};
    c.Q->pos = Vec3{{1.2f, -0.4f, 5.f}};
    for (MapPoint *p : {c.P, c.Q}) { p->normal = p->pos * (1.f / p->pos.norm()); p->max_dist = 2 * p->pos.norm(); p->min_dist = 0.5f; }
    c.T0 = w.add_kf(); c.T1 = w.add_kf();
    w.targets = {c.T0, c.T1};
    Sophus::Sim3f S0, S1;
    S1.t = Vec3{{0.05f, 0.f, 0.f}};
    w.scw = {S0, S1};
    return c;
}
static Vec2 uv_of(World &w, int t, MapPoint *p) { return w.targets[t]->cam.project(pose_of(w.scw[t]) * p->pos); }
static void finish(KeyFrame *k, const std::vector<cv::KeyPoint> &keys, const Rows &r) {
    k->mvKeys = k->mvKeysUn = keys;
    r.to(k);
    k->N = (int)keys.size();
    k->mvpMapPoints.assign(k->N, nullptr);
}
static void observe(MapPoint *p, KeyFrame *k, int idx) { k->mvpMapPoints[idx] = p; p->AddObservation(k, idx); }
static void observe_bg(World &w, MapPoint *p, const std::vector<uint8_t> &d) {
    KeyFrame *b = w.add_kf();
    Rows r;
    r.add(d.data());
    finish(b, {keypoint(1.f, 1.f, 0)}, r);
    observe(p, b, 0);
}

// (A) the descriptor row: in T0, P matches a keypoint holding R, and the caller's R->Replace(P) gives P R's three
// observations with descriptor B, which makes B P's descriptor (it was A).  In T1, P projects onto two keypoints with
// descriptors A and B: the loop matches P to the B keypoint, a search with the batch-time row to the A keypoint.
static void world_a(World &w) {
    std::mt19937 rng(11);
    std::vector<uint8_t> A = random_desc(rng), A2 = A, B = random_desc(rng);
    flip_bits(A2, 20, rng);
    Pair c = pair_world(w);
    MapPoint *R = w.add_mp();
    R->pos = c.P->pos;
    observe_bg(w, c.P, A); observe_bg(w, c.P, A2);
    observe_bg(w, R, B); observe_bg(w, R, B); observe_bg(w, R, B);
    const int lp0 = level_in(c.P, c.T0, w.scw[0]), lp1 = level_in(c.P, c.T1, w.scw[1]);
    const Vec2 a = uv_of(w, 0, c.P), b = uv_of(w, 1, c.P), q = uv_of(w, 1, c.Q);
    Rows r0, r1;
    r0.add(A.data()); r0.add(random_desc(rng).data());
    finish(c.T0, {keypoint(a(0) + 0.2f, a(1) - 0.1f, lp0), keypoint(100.f, 100.f, 0)}, r0);
    observe(R, c.T0, 0);
    r1.add(A.data()); r1.add(B.data()); r1.add(c.Q->desc.ptr(0));
    finish(c.T1, {keypoint(b(0) - 0.3f, b(1), lp1), keypoint(b(0) + 0.3f, b(1), lp1), keypoint(q(0), q(1), 0)}, r1);
    for (auto &mp : w.mps) mp->ComputeDistinctiveDescriptors();
    w.vp = {c.P, c.Q};
}
static bool check_a(World &l) { return l.targets[1]->mvpMapPoints[1] == l.vp[0]; }

// (B) the set of points already in the keyframe: in T0, P matches a keypoint holding R, which is also observed in T1; the
// caller's R->Replace(P) puts P into that slot of T1, so T1 must skip P (a set taken at batch time would fuse P with itself).
static void world_b(World &w) {
    std::mt19937 rng(12);
    std::vector<uint8_t> A = random_desc(rng);
    Pair c = pair_world(w);
    MapPoint *R = w.add_mp();
    R->pos = c.P->pos;
    observe_bg(w, c.P, A);
    observe_bg(w, R, A);
    const int lp0 = level_in(c.P, c.T0, w.scw[0]), lp1 = level_in(c.P, c.T1, w.scw[1]);
    const Vec2 a = uv_of(w, 0, c.P), b = uv_of(w, 1, c.P);
    Rows r0, r1;
    r0.add(A.data());
    finish(c.T0, {keypoint(a(0), a(1), lp0)}, r0);
    observe(R, c.T0, 0);
    r1.add(random_desc(rng).data()); r1.add(A.data());
    finish(c.T1, {keypoint(50.f, 50.f, 0), keypoint(b(0) + 0.2f, b(1), lp1)}, r1);
    observe(R, c.T1, 1);
    for (auto &mp : w.mps) mp->ComputeDistinctiveDescriptors();
    w.vp = {c.P, c.Q};
}
static bool check_b(World &l) { return l.targets[1]->mvpMapPoints[1] == l.vp[0] && l.vp[0]->obs.size() == 4; }

// (C) the map point in the matched slot: in T0, P matches a keypoint holding R; the caller's R->Replace(P) makes R bad and,
// since P is already observed in T1, erases R's slot of T1.  In T1, Q matches that slot: the loop adds Q there, where a
// slot read at batch time would name R as the point to replace.
static void world_c(World &w) {
    std::mt19937 rng(13);
    std::vector<uint8_t> A = random_desc(rng), D = random_desc(rng);
    Pair c = pair_world(w);
    MapPoint *R = w.add_mp();
    R->pos = c.P->pos;
    observe_bg(w, c.P, A);
    observe_bg(w, R, A);
    observe_bg(w, c.Q, D);
    const int lp0 = level_in(c.P, c.T0, w.scw[0]), lq1 = level_in(c.Q, c.T1, w.scw[1]);
    const Vec2 a = uv_of(w, 0, c.P), q = uv_of(w, 1, c.Q);
    Rows r0, r1;
    r0.add(A.data()); r0.add(random_desc(rng).data());
    finish(c.T0, {keypoint(a(0), a(1), lp0), keypoint(30.f, 30.f, 0)}, r0);
    observe(R, c.T0, 0);
    r1.add(A.data()); r1.add(D.data());
    finish(c.T1, {keypoint(600.f, 400.f, 0), keypoint(q(0) - 0.2f, q(1), lq1)}, r1);
    observe(c.P, c.T1, 0);
    observe(R, c.T1, 1);
    for (auto &mp : w.mps) mp->ComputeDistinctiveDescriptors();
    w.vp = {c.P, c.Q};
}
static bool check_c(World &l) { return l.vp[0]->obs.size() == 4 && l.targets[1]->mvpMapPoints[1] == l.vp[1]; }

// Everything Fuse and the Replace loop can change, by index, so that two copies of a world compare.
static std::vector<std::string> state(const World &w, const std::vector<int> &counts, const std::vector<std::vector<MapPoint *>> &reps) {
    std::vector<std::string> s;
    char buf[256];
    for (size_t k = 0; k < counts.size(); ++k) {
        std::string r;
        for (MapPoint *p : reps[k]) r += " " + std::to_string(p ? p->id : -1);
        std::snprintf(buf, sizeof buf, "target %zu: count %d, vpReplacePoints", k, counts[k]);
        s.push_back(buf + r);
    }
    for (auto &kf : w.kfs)
        for (size_t j = 0; j < kf->mvpMapPoints.size(); ++j) {
            std::snprintf(buf, sizeof buf, "keyframe %d slot %zu: map point %d", kf->index, j,
                          kf->mvpMapPoints[j] ? kf->mvpMapPoints[j]->id : -1);
            s.push_back(buf);
        }
    for (auto &mp : w.mps) {
        std::string o;
        for (auto &kv : mp->obs) o += " " + std::to_string(kv.second.first->index) + ":" + std::to_string(kv.second.second);
        char d[65];
        for (int i = 0; i < 32; ++i) std::snprintf(d + 2 * i, 3, "%02x", mp->desc.ptr(0)[i]);
        std::snprintf(buf, sizeof buf, "map point %d: bad %d, replacedBy %d, descriptor %s, observations", mp->id, (int)mp->bad,
                      mp->replaced_by ? mp->replaced_by->id : -1, d);
        s.push_back(buf + o);
    }
    return s;
}

static void replace_all(const std::vector<MapPoint *> &vp, const std::vector<MapPoint *> &rep) {   // LoopClosing.cc:2017-2025
    for (size_t i = 0; i < vp.size(); ++i)
        if (MapPoint *pRep = rep[i]) pRep->Replace(vp[i]);
}
static void run_loop(World &w, std::vector<int> &counts, std::vector<std::vector<MapPoint *>> &reps) {
    VS_GRAPHS::ORBmatcher matcher(0.8);
    for (size_t k = 0; k < w.targets.size(); ++k) {
        std::vector<MapPoint *> rep(w.vp.size(), nullptr);
        counts.push_back(matcher.Fuse(w.targets[k], w.scw[k], w.vp, 4.f, rep));
        replace_all(w.vp, rep);
        reps.push_back(rep);
    }
}
static void run_batch(World &w, std::vector<int> &counts, std::vector<std::vector<MapPoint *>> &reps) {
    VS_GRAPHS::ORBmatcher matcher(0.8);
    auto search = matcher.Fuse(w.targets, w.scw, w.vp, 4.f);
    for (size_t k = 0; k < w.targets.size(); ++k) {
        std::vector<MapPoint *> rep(w.vp.size(), nullptr);
        counts.push_back(matcher.Fuse(search, k, rep));
        replace_all(w.vp, rep);
        reps.push_back(rep);
    }
}

static void compare(const char *name, World &batch, World &loop, int min_fused) {
    const int changes0 = MapPoint::desc_changes;
    std::vector<int> cl, cb;
    std::vector<std::vector<MapPoint *>> rl, rb;
    run_loop(loop, cl, rl);
    const int changes = MapPoint::desc_changes - changes0;
    run_batch(batch, cb, rb);
    const std::vector<std::string> a = state(batch, cb, rb), b = state(loop, cl, rl);
    int diffs = 0;
    for (size_t i = 0; i < a.size() && i < b.size(); ++i)
        if (a[i] != b[i] && diffs++ < 5) EXPECT(false, "%s: the batch left '%.160s', the loop '%.160s'", name, a[i].c_str(), b[i].c_str());
    EXPECT(a.size() == b.size() && diffs == 0, "%s: %d differences", name, diffs);
    int nl = 0;
    for (int c : cl) nl += c;
    EXPECT(nl >= min_fused, "%s: the loop fused %d points, expected at least %d", name, nl, min_fused);
    std::printf("%s: %zu targets, %zu points, fused %d, %d query descriptors changed by Replace\n", name, loop.targets.size(),
                loop.vp.size(), nl, changes);
}

static void misuse() {
    World w;
    random_world(w, 21, 3, 100);
    VS_GRAPHS::ORBmatcher matcher;
    auto search = matcher.Fuse(w.targets, w.scw, w.vp, 4.f);
    std::vector<MapPoint *> rep(w.vp.size(), nullptr);
    auto throws = [&](auto f) { try { f(); } catch (const std::runtime_error &) { return true; } return false; };
    EXPECT(throws([&] { matcher.Fuse(search, w.targets.size(), rep); }), "a target out of range must throw");
    matcher.Fuse(search, 1, rep);
    EXPECT(throws([&] { matcher.Fuse(search, 1, rep); }), "a target resolved twice must throw");
    bool threw = false;
    std::thread other([&] { threw = throws([&] { matcher.Fuse(search, 0, rep); }); });
    other.join();
    EXPECT(threw, "a resolve on another thread must throw");
    matcher.Fuse(search, 0, rep);                    // the search is still usable on its own thread
    std::vector<Sophus::Sim3f> one(1);
    EXPECT(throws([&] { matcher.Fuse(w.targets, one, w.vp, 4.f); }), "a pose count that differs from the keyframe count must throw");
    World e;
    auto none = matcher.Fuse(e.targets, e.scw, w.vp, 4.f);   // no targets, no points
    std::vector<MapPoint *> no_points;
    auto empty = matcher.Fuse(w.targets, w.scw, no_points, 4.f);
    EXPECT(matcher.Fuse(empty, 0, no_points) == 0, "no points");
    (void)none;
}

// --time: the loop against the batch + resolves, each on a fresh copy of a world with about 1000 keypoints per target
static void timing() {
    const int ns[] = {1000, 4000, 12000}, Ts[] = {1, 10, 30, 60};
    const int reps = 7;
    std::printf("timing (stand-in world, host projection included; median of %d, microseconds)\n", reps);
    for (int n : ns)
        for (int T : Ts) {
            std::vector<double> tl, tb;
            for (int r = 0; r < reps; ++r) {
                World l, b;
                random_world(l, 1000 + r, T, n, 1000);
                random_world(b, 1000 + r, T, n, 1000);
                std::vector<int> cl, cb;
                std::vector<std::vector<MapPoint *>> rl, rb;
                auto t0 = std::chrono::steady_clock::now();
                run_loop(l, cl, rl);
                auto t1 = std::chrono::steady_clock::now();
                run_batch(b, cb, rb);
                auto t2 = std::chrono::steady_clock::now();
                EXPECT(cl == cb, "timing world n=%d T=%d: counts differ", n, T);
                tl.push_back(std::chrono::duration<double, std::micro>(t1 - t0).count());
                tb.push_back(std::chrono::duration<double, std::micro>(t2 - t1).count());
            }
            std::sort(tl.begin(), tl.end());
            std::sort(tb.begin(), tb.end());
            std::printf("TIME n=%d T=%d loop %.1f batch %.1f ratio %.2f\n", n, T, tl[reps / 2], tb[reps / 2], tl[reps / 2] / tb[reps / 2]);
        }
}

int main(int argc, char **argv) {
    struct Case { unsigned seed; int nkf, nq; };
    const Case cases[] = {{1, 1, 300}, {2, 3, 400}, {3, 6, 400}, {4, 12, 500}, {5, 25, 300}, {6, 40, 600}};
    for (const Case &c : cases) {
        World b, l;
        random_world(b, c.seed, c.nkf, c.nq);
        random_world(l, c.seed, c.nkf, c.nq);
        char name[64];
        std::snprintf(name, sizeof name, "random world %u", c.seed);
        compare(name, b, l, 10 * c.nkf);
    }
    struct Constructed { const char *name; void (*make)(World &); bool (*check)(World &); const char *what; int min_fused; };
    const Constructed cw[] = {
        {"constructed world A (descriptor)", world_a, check_a, "P takes the B keypoint of T1", 2},
        {"constructed world B (already found)", world_b, check_b, "P sits in T1's slot and is skipped there", 1},
        {"constructed world C (slot contents)", world_c, check_c, "R's slot of T1 is erased and Q added there", 2},
    };
    for (const Constructed &c : cw) {
        World b, l;
        c.make(b);
        c.make(l);
        compare(c.name, b, l, c.min_fused);
        EXPECT(c.check(l), "%s: the loop did not end with '%s' (the world does not test what it should)", c.name, c.what);
    }
    misuse();
    if (argc > 1 && std::strcmp(argv[1], "--time") == 0) timing();
    if (g_fail) { std::printf("%d failures\n", g_fail); return 1; }
    std::printf("SEARCH AND FUSE TEST OK\n");
    return 0;
}
