// fuse_multi_test.cpp — the multi-target VS_GRAPHS::ORBmatcher::Fuse(vpTargetKFs, vpMapPoints, th) against the loop of
// single-target Fuse calls it stands for (LocalMapping::SearchInNeighbors, LocalMapping.cc:764-802):
//     for (pKFi : vpTargetKFs) { matcher.Fuse(pKFi, vpMapPoints); if (pKFi->NLeft != -1) matcher.Fuse(pKFi, vpMapPoints, 3.0, true); }
// Each world is generated twice from one seed; the multi-target call runs on one copy, the loop on the other, and the two
// worlds must end identical: every keyframe's map-point slots, every map point's observations, bad flag, replacedBy and
// descriptor, and the counts.  The stand-in MapPoint::Replace recomputes the survivor's descriptor as
// MapPoint::ComputeDistinctiveDescriptors does (MapPoint.cc:340-417), so a Replace in one target can change the
// survivor's match in a later target.  The constructed world makes that happen for sure.  Needs a GPU.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <random>
#include <string>
#include <vector>

// ---- stand-ins for Eigen / Sophus (only what the shim's Fuse uses; poses are translations) ----
struct Vec3 {
    float v[3];
    float operator()(int i) const { return v[i]; }
    Vec3 operator-(const Vec3 &o) const { return Vec3{{v[0] - o.v[0], v[1] - o.v[1], v[2] - o.v[2]}}; }
    Vec3 operator+(const Vec3 &o) const { return Vec3{{v[0] + o.v[0], v[1] + o.v[1], v[2] + o.v[2]}}; }
    Vec3 operator*(float s) const { return Vec3{{v[0] * s, v[1] * s, v[2] * s}}; }
    float dot(const Vec3 &o) const { return v[0] * o.v[0] + v[1] * o.v[1] + v[2] * o.v[2]; }
    float norm() const { return std::sqrt(dot(*this)); }
};
struct Vec2 {
    float v[2];
    float operator()(int i) const { return v[i]; }
};
struct Pose {   // world -> camera: p + t
    Vec3 t{{0, 0, 0}};
    Vec3 operator*(const Vec3 &p) const { return p + t; }
    Pose inverse() const { return Pose{t * -1.f}; }
    Vec3 translation() const { return t; }
};

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
    std::vector<float> mvuRight, mvScaleFactors, mvInvLevelSigma2;
    std::vector<MapPoint *> mvpMapPoints;
    float mnMinX = 0, mnMinY = 0, mnMaxX = 640, mnMaxY = 480;
    float mfGridElementWidthInv = 64.f / 640.f, mfGridElementHeightInv = 48.f / 480.f;
    float mbf = 40.f;
    float mfLogScaleFactor = std::log(kScale);
    int mnScaleLevels = kLevels;
    Camera cam, cam2;
    Camera *mpCamera = &cam, *mpCamera2 = nullptr;
    Pose pose, right_pose;
    KeyFrame() {
        float s = 1.f;
        for (int l = 0; l < kLevels; ++l, s *= kScale) { mvScaleFactors.push_back(s); mvInvLevelSigma2.push_back(1.f / (s * s)); }
    }
    Pose GetPose() const { return pose; }
    Pose GetRightPose() const { return right_pose; }
    Vec3 GetCameraCenter() const { return pose.inverse().translation(); }
    Vec3 GetRightCameraCenter() const { return right_pose.inverse().translation(); }
    bool IsInImage(float x, float y) const { return x >= mnMinX && x < mnMaxX && y >= mnMinY && y < mnMaxY; }
    MapPoint *GetMapPoint(size_t i) const { return mvpMapPoints[i]; }
    void AddMapPoint(MapPoint *p, size_t i) { mvpMapPoints[i] = p; }
};

static int hamming(const uint8_t *a, const uint8_t *b) {
    int d = 0;
    for (int i = 0; i < 32; ++i) d += __builtin_popcount((unsigned)(a[i] ^ b[i]));
    return d;
}

struct MapPoint {
    int id = 0;
    bool query = false;                              // one of vpMapPoints
    bool bad = false;
    MapPoint *replaced_by = nullptr;
    Vec3 pos{{0, 0, 5}}, normal{{0, 0, 1}};
    float max_dist = 10, min_dist = 0.1f;
    std::map<unsigned long, std::pair<KeyFrame *, int>> obs;   // by keyframe id: the same order in both copies of a world
    cv::Mat desc{1, 32, CV_8UC1};
    static int desc_changes;                         // descriptors of queries changed by a Replace

    bool isBad() const { return bad; }
    int Observations() const { return (int)obs.size(); }
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
    // MapPoint.cc:216-270: the observations move to the survivor, which recomputes its descriptor
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

struct World {
    std::vector<std::unique_ptr<KeyFrame>> kfs;     // targets, then background keyframes
    std::vector<std::unique_ptr<MapPoint>> mps;     // queries, then other map points of the target keyframes
    std::vector<KeyFrame *> targets;
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

// A random world: nkf target keyframes (every third one a two-camera rig, every other single-camera one stereo), nq query
// map points and as many other map points.  Every map point is observed in 1-3 background keyframes with its own descriptor
// plus noise; every target camera has keypoints near the projections of half of the points (some with a near twin), with
// noisy descriptors, and distractors.  A quarter of those keypoints already hold their own map point, a quarter hold
// another one: the queries that match them get fused by Replace.
static void random_world(World &w, unsigned seed, int nkf, int nq) {
    std::mt19937 rng(seed);
    const int np = 2 * nq;
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
    for (int k = 0; k < nkf; ++k) w.targets.push_back(w.add_kf());
    std::vector<KeyFrame *> bg;
    std::vector<Rows> bg_rows(3);
    for (int b = 0; b < 3; ++b) bg.push_back(w.add_kf());
    for (int i = 0; i < np; ++i) {
        const int nobs = 1 + rng() % 3;
        for (int b = 0; b < nobs; ++b) {
            std::vector<uint8_t> d = ident[i];
            flip_bits(d, rng() % 24, rng);
            const int row = bg_rows[b].add(d.data());
            w.mps[i]->AddObservation(bg[b], row);
        }
    }
    for (int b = 0; b < 3; ++b) {
        bg_rows[b].to(bg[b]);
        bg[b]->N = (int)bg_rows[b].r.size();
        bg[b]->mvpMapPoints.assign(bg[b]->N, nullptr);
        for (auto &mp : w.mps)
            for (auto &kv : mp->obs)
                if (kv.second.first == bg[b]) bg[b]->mvpMapPoints[kv.second.second] = mp.get();
    }
    for (int k = 0; k < nkf; ++k) {
        KeyFrame *kf = w.targets[k];
        const bool two = k % 3 == 2, stereo = !two && k % 2 == 0;
        kf->pose.t = Vec3{{uni(rng, -0.3f, 0.3f), uni(rng, -0.2f, 0.2f), uni(rng, -0.3f, 0.3f)}};
        kf->right_pose.t = kf->pose.t + Vec3{{-0.1f, 0.f, 0.f}};
        if (two) kf->mpCamera2 = &kf->cam2;
        Rows rows;
        std::vector<int> owner;                       // map point a keypoint was made from (-1 distractor)
        for (int c = 0; c < (two ? 2 : 1); ++c) {
            const Pose &T = c ? kf->right_pose : kf->pose;
            std::vector<std::pair<cv::KeyPoint, std::pair<int, std::vector<uint8_t>>>> kps;
            std::vector<float> ur;
            for (int i = 0; i < np; ++i) {
                if (rng() % 2) continue;
                const Vec3 pc = T * w.mps[i]->pos;
                const Vec2 uv = kf->cam.project(pc);
                if (!kf->IsInImage(uv(0), uv(1))) continue;
                int lvl = w.mps[i]->PredictScale((w.mps[i]->pos - T.inverse().translation()).norm(), kf);
                const int twins = rng() % 4 == 0 ? 2 : 1;
                for (int t = 0; t < twins; ++t) {
                    std::vector<uint8_t> d = ident[i];
                    flip_bits(d, rng() % 40, rng);
                    const int o = std::max(0, lvl - (int)(rng() % 2));
                    kps.push_back({keypoint(uv(0) + uni(rng, -0.8f, 0.8f), uv(1) + uni(rng, -0.8f, 0.8f), o), {i, d}});
                }
            }
            for (int j = 0; j < 60; ++j)
                kps.push_back({keypoint(uni(rng, 0, 639.9f), uni(rng, 0, 479.9f), rng() % kLevels), {-1, random_desc(rng)}});
            std::shuffle(kps.begin(), kps.end(), rng);
            for (auto &e : kps) {
                (c ? kf->mvKeysRight : kf->mvKeys).push_back(e.first);
                rows.add(e.second.second.data());
                owner.push_back(e.second.first);
                if (!c) {
                    const Vec3 pc = kf->pose * (e.second.first >= 0 ? w.mps[e.second.first]->pos : Vec3{{0, 0, 5}});
                    ur.push_back(stereo && rng() % 10 < 7 ? e.first.pt.x - kf->mbf / pc(2) + uni(rng, -0.5f, 0.5f) : -1.f);
                }
            }
            if (!c) kf->mvuRight = ur;
        }
        kf->NLeft = two ? (int)kf->mvKeys.size() : -1;
        kf->N = (int)owner.size();
        kf->mvKeysUn = kf->mvKeys;
        if (two) kf->mvuRight.assign(kf->N, -1.f);
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
    for (auto &mp : w.mps) mp->ComputeDistinctiveDescriptors();
    for (int i = 0; i < nq; ++i) {
        const unsigned r = rng() % 40;
        w.vp.push_back(r == 0 ? nullptr : w.mps[i].get());
        if (r == 1) w.mps[i]->bad = true;
    }
    for (size_t i = 0; i + 1 < w.vp.size(); i += 23) w.vp[i + 1] = w.vp[i];   // duplicates: the second is skipped by IsInKeyFrame
}

// The stale-descriptor case: query P matches, in target 0, a keypoint that holds query Q.  Q has more observations, so
// P->Replace(Q): Q survives and takes P's two observations with descriptor B, which makes B its descriptor (it was A).
// In target 1 Q projects onto two keypoints, one with descriptor A and one with B: the loop matches Q to the B keypoint.
static void constructed_world(World &w) {
    std::mt19937 rng(99);
    std::vector<uint8_t> A = random_desc(rng), A2 = A, B = random_desc(rng);
    flip_bits(A2, 30, rng);
    MapPoint *P = w.add_mp(), *Q = w.add_mp();
    P->query = Q->query = true;
    P->pos = Vec3{{-1.f, 0.5f, 6.f}};
    Q->pos = Vec3{{1.2f, -0.4f, 5.f}};
    for (MapPoint *p : {P, Q}) { p->normal = p->pos * (1.f / p->pos.norm()); p->max_dist = 2 * p->pos.norm(); p->min_dist = 0.5f; }
    KeyFrame *T0 = w.add_kf(), *T1 = w.add_kf(), *bg[4] = {w.add_kf(), w.add_kf(), w.add_kf(), w.add_kf()};
    w.targets = {T0, T1};
    const std::vector<uint8_t> *bg_desc[4] = {&A, &A2, &B, &B};           // Q is observed with A and A2, P twice with B
    for (int b = 0; b < 4; ++b) {
        Rows r;
        r.add(bg_desc[b]->data());
        r.to(bg[b]);
        bg[b]->N = 1;
        MapPoint *owner = b < 2 ? Q : P;
        bg[b]->mvpMapPoints.assign(1, owner);
        owner->AddObservation(bg[b], 0);
    }
    auto level = [](MapPoint *p, KeyFrame *kf) { return p->PredictScale((p->pos - kf->GetCameraCenter()).norm(), kf); };
    // target 0: keypoint 0 at P's projection with descriptor B, holding Q (Q's third observation, descriptor B)
    {
        const Vec2 uv = T0->cam.project(T0->pose * P->pos);
        T0->mvKeys = {keypoint(uv(0) + 0.2f, uv(1) - 0.1f, level(P, T0)), keypoint(100.f, 100.f, 0)};
        Rows r;
        r.add(B.data());
        r.add(random_desc(rng).data());
        r.to(T0);
    }
    // target 1: keypoints with descriptors A and B at Q's projection (A first in the grid's scan order)
    {
        T1->pose.t = Vec3{{0.05f, 0.f, 0.f}};
        const Vec2 uv = T1->cam.project(T1->pose * Q->pos);
        const int lq = level(Q, T1);
        T1->mvKeys = {keypoint(uv(0) - 0.3f, uv(1), lq), keypoint(uv(0) + 0.3f, uv(1), lq), keypoint(500.f, 50.f, 1)};
        Rows r;
        r.add(A.data());
        r.add(B.data());
        r.add(random_desc(rng).data());
        r.to(T1);
    }
    for (KeyFrame *k : {T0, T1}) {
        k->N = (int)k->mvKeys.size();
        k->mvKeysUn = k->mvKeys;
        k->mvuRight.assign(k->N, -1.f);
        k->mvpMapPoints.assign(k->N, nullptr);
    }
    T0->mvpMapPoints[0] = Q;
    Q->AddObservation(T0, 0);
    P->ComputeDistinctiveDescriptors();
    Q->ComputeDistinctiveDescriptors();
    w.vp = {P, Q};
}

// Everything Fuse can change, by index, so that two copies of a world compare.
static std::vector<std::string> state(const World &w, int nfused) {
    std::vector<std::string> s;
    char buf[256];
    std::snprintf(buf, sizeof buf, "count %d", nfused);
    s.push_back(buf);
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

static int loop_fuse(World &w) {
    VS_GRAPHS::ORBmatcher matcher;
    int n = 0;
    for (KeyFrame *kf : w.targets) {
        n += matcher.Fuse(kf, w.vp, 3.f);
        if (kf->NLeft != -1) n += matcher.Fuse(kf, w.vp, 3.f, true);
    }
    return n;
}

static void compare(const char *name, World &multi, World &loop, int min_fused) {
    const int changes0 = MapPoint::desc_changes;
    const int nl = loop_fuse(loop);
    const int changes = MapPoint::desc_changes - changes0;
    VS_GRAPHS::ORBmatcher matcher;
    const int nm = matcher.Fuse(multi.targets, multi.vp, 3.f);
    const std::vector<std::string> a = state(multi, nm), b = state(loop, nl);
    int diffs = 0;
    for (size_t i = 0; i < a.size() && i < b.size(); ++i)
        if (a[i] != b[i] && diffs++ < 5) EXPECT(false, "%s: multi-target Fuse left '%s', the loop '%s'", name, a[i].c_str(), b[i].c_str());
    EXPECT(a.size() == b.size() && diffs == 0, "%s: %d differences", name, diffs);
    EXPECT(nl >= min_fused, "%s: the loop fused %d points, expected at least %d", name, nl, min_fused);
    std::printf("%s: %zu targets, %zu points, fused %d (loop %d), %d query descriptors changed by Replace\n", name,
                multi.targets.size(), multi.vp.size(), nm, nl, changes);
}

int main() {
    struct Case { unsigned seed; int nkf, nq; };
    const Case cases[] = {{1, 1, 300}, {2, 2, 400}, {3, 5, 400}, {4, 7, 500}, {5, 12, 300}};   // 12 keyframes: 16 cameras
    for (const Case &c : cases) {
        World m, l;
        random_world(m, c.seed, c.nkf, c.nq);
        random_world(l, c.seed, c.nkf, c.nq);
        char name[64];
        std::snprintf(name, sizeof name, "random world %u", c.seed);
        compare(name, m, l, 10 * c.nkf);
    }
    {
        World m, l;
        constructed_world(m);
        constructed_world(l);
        compare("constructed world", m, l, 2);
        // the loop itself must show the effect: Q, replaced into in target 0, takes the B keypoint of target 1
        EXPECT(l.targets[1]->mvpMapPoints[1] == l.vp[1] && l.vp[0]->isBad(), "constructed world: the loop did not move Q to "
               "the B keypoint of target 1 (the world does not test what it should)");
    }
    {   // no targets, no points
        World m;
        random_world(m, 6, 0, 50);
        VS_GRAPHS::ORBmatcher matcher;
        EXPECT(matcher.Fuse(m.targets, m.vp, 3.f) == 0, "no targets");
        std::vector<MapPoint *> none;
        World m2;
        random_world(m2, 7, 3, 50);
        EXPECT(matcher.Fuse(m2.targets, none, 3.f) == 0, "no points");
    }
    if (g_fail) { std::printf("%d failures\n", g_fail); return 1; }
    std::printf("FUSE MULTI TEST OK\n");
    return 0;
}
