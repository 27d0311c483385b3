// triangulation_multi_test.cpp — the batch form of VS_GRAPHS::ORBmatcher::SearchForTriangulation against the loop of
// single-target calls it stands for, LocalMapping::CreateNewMapPoints (LocalMapping.cc:406,460):
//     for (i) { matcher.SearchForTriangulation(mpCurrentKeyFrame, vpNeighKFs[i], vMatchedIndices, false, bCoarse); <triangulate> }
// Each world is generated twice from one seed.  One copy runs the loop, the other one batch call plus a resolve per
// neighbour.  A stand-in triangulation turns a seeded share of the returned pairs into map points of KF1 (at idx1) and of
// the neighbour (at idx2), so later searches see them.  Every pair list, every count and every map-point slot of every
// keyframe must be identical at the end.  Some worlds list a neighbour twice, hold a two-camera neighbour, change a
// neighbour's pose or erase KF1 map points between the batch call and a resolve: those searches must take the
// single-target call (the launches during the resolves show it) and still equal the loop.  Needs a GPU.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <random>
#include <vector>

// ---- stand-ins for Eigen / Sophus (only what the shim's SearchForTriangulation uses; rotations are the identity) ----
struct Vec3 {
    float v[3];
    float operator()(int i) const { return v[i]; }
    Vec3 operator+(const Vec3 &o) const { return Vec3{{v[0] + o.v[0], v[1] + o.v[1], v[2] + o.v[2]}}; }
};
struct Vec2 {
    float v[2];
    float operator()(int i) const { return v[i]; }
};
struct Mat3 {
    float m[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    int fill = 0;
    float operator()(int r, int c) const { return m[3 * r + c]; }
    Mat3 &operator<<(float x) { fill = 0; m[fill++] = x; return *this; }
    Mat3 &operator,(float x) { m[fill++] = x; return *this; }
    Mat3 transpose() const { Mat3 t; for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) t.m[3 * r + c] = m[3 * c + r]; return t; }
    Mat3 operator*(const Mat3 &o) const {
        Mat3 t;
        for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) { float a = 0; for (int k = 0; k < 3; ++k) a += m[3 * r + k] * o.m[3 * k + c]; t.m[3 * r + c] = a; }
        return t;
    }
    Vec3 operator*(const Vec3 &p) const { return Vec3{{m[0] * p.v[0] + m[1] * p.v[1] + m[2] * p.v[2], m[3] * p.v[0] + m[4] * p.v[1] + m[5] * p.v[2], m[6] * p.v[0] + m[7] * p.v[1] + m[8] * p.v[2]}}; }
    Mat3 inverse() const {
        const float *a = m;
        const float det = a[0] * (a[4] * a[8] - a[5] * a[7]) - a[1] * (a[3] * a[8] - a[5] * a[6]) + a[2] * (a[3] * a[7] - a[4] * a[6]);
        Mat3 t;
        t.m[0] = (a[4] * a[8] - a[5] * a[7]) / det; t.m[1] = (a[2] * a[7] - a[1] * a[8]) / det; t.m[2] = (a[1] * a[5] - a[2] * a[4]) / det;
        t.m[3] = (a[5] * a[6] - a[3] * a[8]) / det; t.m[4] = (a[0] * a[8] - a[2] * a[6]) / det; t.m[5] = (a[2] * a[3] - a[0] * a[5]) / det;
        t.m[6] = (a[3] * a[7] - a[4] * a[6]) / det; t.m[7] = (a[1] * a[6] - a[0] * a[7]) / det; t.m[8] = (a[0] * a[4] - a[1] * a[3]) / det;
        return t;
    }
};
struct Pose {   // world -> camera: x_c = x_w + t
    Mat3 R;
    Vec3 t{{0, 0, 0}};
    Pose inverse() const { return Pose{R, Vec3{{-t.v[0], -t.v[1], -t.v[2]}}}; }
    Vec3 translation() const { return t; }
    Mat3 rotationMatrix() const { return R; }
    Vec3 operator*(const Vec3 &p) const { return p + t; }
    Pose operator*(const Pose &o) const { return Pose{R, o.t + t}; }
};

#include "../../visual_sgraphs_b200/shim/ORBmatcher.h"

static int g_fail = 0;
#define EXPECT(cond, ...)                                                                                                   \
    do {                                                                                                                    \
        if (!(cond)) { std::printf("FAIL %s:%d: ", __FILE__, __LINE__); std::printf(__VA_ARGS__); std::printf("\n"); ++g_fail; } \
    } while (0)

constexpr int kLevels = 8;
constexpr int kNodes = 24;

struct Camera {
    float fx = 500, fy = 500, cx = 320, cy = 240;
    Vec2 project(const Vec3 &p) const { return Vec2{{fx * p.v[0] / p.v[2] + cx, fy * p.v[1] / p.v[2] + cy}}; }
    Mat3 toK_() const { Mat3 K; K << fx, 0.f, cx, 0.f, fy, cy, 0.f, 0.f, 1.f; return K; }
    // the two-camera path's per-pair test is the caller's camera code: any fixed rule will do here
    bool epipolarConstrain(Camera *, const cv::KeyPoint &kp1, const cv::KeyPoint &kp2, const Mat3 &, const Vec3 &, float, float) const {
        return std::fabs(kp1.pt.y - kp2.pt.y) < 25.f;
    }
};
struct MapPoint {
    int id;
    bool isBad() const { return false; }
};
struct KeyFrame {
    long unsigned int mnId = 0;
    int N = 0, NLeft = -1;
    std::vector<cv::KeyPoint> mvKeys, mvKeysUn, mvKeysRight;
    cv::Mat mDescriptors;
    std::vector<float> mvuRight, mvScaleFactors, mvLevelSigma2;
    float mnMinX = 0, mnMinY = 0, mnMaxX = 640, mnMaxY = 480;
    float mfGridElementWidthInv = 64.f / 640.f, mfGridElementHeightInv = 48.f / 480.f;
    std::map<unsigned, std::vector<unsigned>> mFeatVec;   // DBoW2::FeatureVector
    Pose pose, right_pose;
    Camera cam, cam2;
    Camera *mpCamera = &cam, *mpCamera2 = nullptr;
    std::vector<MapPoint *> mvpMapPoints;
    KeyFrame() {
        float s = 1.f;
        for (int l = 0; l < kLevels; ++l, s *= 1.2f) { mvScaleFactors.push_back(s); mvLevelSigma2.push_back(s * s); }
    }
    MapPoint *GetMapPoint(size_t i) const { return mvpMapPoints[i]; }
    void AddMapPoint(MapPoint *p, size_t i) { mvpMapPoints[i] = p; }
    Pose GetPose() const { return pose; }
    Pose GetPoseInverse() const { return pose.inverse(); }
    Vec3 GetCameraCenter() const { return pose.inverse().translation(); }
    Pose GetRightPose() const { return right_pose; }
    Pose GetRightPoseInverse() const { return right_pose.inverse(); }
};

struct Options {
    int nneigh = 12;
    bool stereo = false, only_stereo = false, coarse = false, check_ori = true;
    int twice = -1;              // neighbour listed again at the end of the list
    int two_camera = -1;         // neighbour with a second camera
    int pose_change_at = -1;     // that neighbour's pose moves right before its resolve
    int erase_at = -1;           // KF1 loses map points right before this neighbour's resolve
};

struct World {
    std::vector<std::unique_ptr<KeyFrame>> kfs;
    std::vector<std::unique_ptr<MapPoint>> mps;
    std::vector<KeyFrame *> neigh;
    KeyFrame *kf1 = nullptr;
    MapPoint *NewMapPoint() {
        mps.emplace_back(new MapPoint{(int)mps.size()});
        return mps.back().get();
    }
};

// A keyframe at camera translation t seeing the scene: most features are noisy projections of scene points with their
// descriptor (a few bits flipped; byte 0, which picks the vocabulary node, kept), the rest distractors.
static void observe(KeyFrame &kf, const Vec3 &t, const std::vector<Vec3> &P, const std::vector<std::vector<uint8_t>> &ident,
                    bool stereo, int nright, std::mt19937 &rng) {
    std::normal_distribution<float> noise(0.f, 0.6f);
    std::vector<cv::KeyPoint> keys;
    std::vector<std::vector<uint8_t>> desc;
    std::vector<float> ur;
    kf.pose.t = t;
    for (size_t k = 0; k < P.size(); ++k) {
        if (rng() % 10 < 4) continue;
        const Vec3 c = P[k] + t;
        if (c.v[2] < 0.5f) continue;
        const Vec2 uv = kf.cam.project(c);
        if (uv(0) < 20 || uv(0) > 620 || uv(1) < 20 || uv(1) > 460) continue;
        cv::KeyPoint kp;
        kp.pt.x = uv(0) + noise(rng);
        kp.pt.y = uv(1) + noise(rng);
        kp.octave = rng() % kLevels;
        kp.angle = std::fmod((float)(k * 37 % 360) + (float)(rng() % 6), 360.f);
        kp.size = 31.f;
        keys.push_back(kp);
        std::vector<uint8_t> d = ident[k];
        for (int b = 0, nb = rng() % 10; b < nb; ++b) { const unsigned bit = 8 + rng() % 248; d[bit / 8] ^= (uint8_t)(1u << (bit % 8)); }
        desc.push_back(d);
        ur.push_back(stereo && rng() % 2 ? uv(0) - 40.f / c.v[2] : -1.f);
    }
    for (int k = 0, nd = (int)keys.size() / 6 + nright; k < nd; ++k) {
        cv::KeyPoint kp;
        kp.pt.x = (float)(rng() % 6000) / 10.f + 20.f;
        kp.pt.y = (float)(rng() % 4400) / 10.f + 20.f;
        kp.octave = rng() % kLevels;
        kp.angle = (float)(rng() % 360);
        kp.size = 31.f;
        keys.push_back(kp);
        std::vector<uint8_t> d(32);
        for (auto &x : d) x = (uint8_t)(rng() & 255);
        desc.push_back(d);
        ur.push_back(-1.f);
    }
    const int n = (int)keys.size();
    kf.N = n;
    kf.mDescriptors.create(n, 32, CV_8UC1);
    for (int i = 0; i < n; ++i) {
        std::memcpy(kf.mDescriptors.ptr(i), desc[i].data(), 32);
        kf.mFeatVec[(unsigned)(desc[i][0] % kNodes)].push_back((unsigned)i);
    }
    if (nright) {                                          // the last nright features are a second camera's
        kf.NLeft = n - nright;
        kf.mvKeys.assign(keys.begin(), keys.begin() + kf.NLeft);
        kf.mvKeysRight.assign(keys.begin() + kf.NLeft, keys.end());
        kf.mvKeysUn = kf.mvKeys;
        kf.mpCamera2 = &kf.cam2;
        kf.right_pose.t = t + Vec3{{-0.1f, 0.f, 0.f}};
    } else {
        kf.mvKeys = kf.mvKeysUn = keys;
        kf.mvuRight = ur;                                  // -1 everywhere for a monocular keyframe, as Frame fills it
    }
    kf.mvpMapPoints.assign(n, nullptr);
}

static void make_world(World &w, unsigned seed, const Options &o) {
    std::mt19937 rng(seed);
    std::uniform_real_distribution<float> U(-1.f, 1.f);
    std::vector<Vec3> P(700);
    std::vector<std::vector<uint8_t>> ident(P.size(), std::vector<uint8_t>(32));
    for (size_t k = 0; k < P.size(); ++k) {
        P[k] = Vec3{{2.5f * U(rng), 1.8f * U(rng), 5.5f + 2.5f * U(rng)}};
        for (auto &x : ident[k]) x = (uint8_t)(rng() & 255);
    }
    for (int k = 0; k <= o.nneigh; ++k) {
        w.kfs.emplace_back(new KeyFrame());
        KeyFrame &kf = *w.kfs.back();
        kf.mnId = k;
        const Vec3 t = k == 0 ? Vec3{{0, 0, 0}} : Vec3{{0.5f * U(rng), 0.3f * U(rng), 0.2f * U(rng)}};
        observe(kf, t, P, ident, o.stereo && k % 2 == 0, k == o.two_camera ? 150 : 0, rng);
        for (int i = 0; i < kf.N; ++i)
            if (rng() % 10 < (k == 0 ? 4 : 3)) kf.mvpMapPoints[i] = w.NewMapPoint();
    }
    w.kf1 = w.kfs[0].get();
    for (int k = 1; k <= o.nneigh; ++k) w.neigh.push_back(w.kfs[k].get());
    if (o.twice >= 0) w.neigh.push_back(w.neigh[o.twice]);
}

// What happens between the searches in both forms: the stand-in triangulation of the returned pairs (a seeded share of
// them becomes map points), and the scripted changes of a world.
static void triangulate(World &w, KeyFrame *pKF2, const std::vector<std::pair<size_t, size_t>> &pairs, unsigned seed) {
    for (const auto &p : pairs) {
        const unsigned h = (unsigned)(p.first * 2654435761u) ^ (unsigned)(p.second * 40503u) ^ seed;
        if (h % 4 == 0) continue;
        MapPoint *mp = w.NewMapPoint();
        w.kf1->AddMapPoint(mp, p.first);
        pKF2->AddMapPoint(mp, p.second);
    }
}
static void before_search(World &w, const Options &o, size_t i) {
    if ((int)i == o.pose_change_at) w.neigh[i]->pose.t = w.neigh[i]->pose.t + Vec3{{0.05f, -0.02f, 0.01f}};
    if ((int)i == o.erase_at)
        for (int j = 0, erased = 0; j < w.kf1->N && erased < 15; ++j)
            if (w.kf1->mvpMapPoints[j] && w.kf1->mvpMapPoints[j]->id < w.kf1->N) { w.kf1->mvpMapPoints[j] = nullptr; ++erased; }
}

static void run(const char *name, unsigned seed, const Options &o, bool expect_fallback) {
    World wl, wb;
    make_world(wl, seed, o);
    make_world(wb, seed, o);
    VS_GRAPHS::ORBmatcher matcher(0.6f, o.check_ori);
    const size_t T = wl.neigh.size();
    std::vector<std::vector<std::pair<size_t, size_t>>> loop(T), batch(T);
    std::vector<int> nloop(T), nbatch(T);
    for (size_t i = 0; i < T; ++i) {                                                  // the reference's loop
        before_search(wl, o, i);
        nloop[i] = matcher.SearchForTriangulation(wl.kf1, wl.neigh[i], loop[i], o.only_stereo, o.coarse);
        triangulate(wl, wl.neigh[i], loop[i], seed + (unsigned)i);
    }
    auto search = matcher.SearchForTriangulation(wb.kf1, wb.neigh, o.only_stereo, o.coarse);
    const int64_t before = vsg_launch_count();
    for (size_t i = 0; i < T; ++i) {
        before_search(wb, o, i);
        nbatch[i] = matcher.SearchForTriangulation(search, i, batch[i]);
        triangulate(wb, wb.neigh[i], batch[i], seed + (unsigned)i);
    }
    const int64_t fallback_launches = vsg_launch_count() - before;
    int total = 0, diffs = 0;
    for (size_t i = 0; i < T; ++i) {
        total += nloop[i];
        EXPECT(nbatch[i] == nloop[i] && batch[i].size() == (size_t)nbatch[i], "%s: neighbour %zu: %d matches (%zu pairs), the loop %d",
               name, i, nbatch[i], batch[i].size(), nloop[i]);
        if (batch[i] != loop[i] && diffs++ < 5) EXPECT(false, "%s: neighbour %zu: the pair lists differ", name, i);
    }
    for (size_t k = 0; k < wl.kfs.size(); ++k)
        for (int j = 0; j < wl.kfs[k]->N; ++j) {
            const MapPoint *a = wl.kfs[k]->mvpMapPoints[j], *b = wb.kfs[k]->mvpMapPoints[j];
            if ((a ? a->id : -1) != (b ? b->id : -1) && diffs++ < 10) EXPECT(false, "%s: keyframe %zu, slot %d differs", name, k, j);
        }
    EXPECT(diffs == 0, "%s: %d differences", name, diffs);
    EXPECT(total >= 5 * (int)T, "%s: the loop found %d pairs over %zu neighbours", name, total, T);
    EXPECT((fallback_launches > 0) == expect_fallback, "%s: %lld launches while resolving", name, (long long)fallback_launches);
    std::printf("%s: %zu neighbours, %d pairs, %d map points, %lld launches while resolving\n", name, T, total, (int)wl.mps.size(),
                (long long)fallback_launches);
}

int main() {
    Options o;
    run("monocular, 12 neighbours", 1, o, false);
    o = Options(); o.nneigh = 30; o.check_ori = false;
    run("monocular, 30 neighbours, no rotation check", 2, o, false);
    o = Options(); o.nneigh = 10; o.stereo = true; o.coarse = true;
    run("stereo, coarse", 3, o, false);
    o = Options(); o.nneigh = 16; o.stereo = true; o.only_stereo = true;
    run("stereo, only stereo", 4, o, false);
    o = Options(); o.nneigh = 14; o.twice = 3;
    run("a neighbour listed twice", 5, o, true);
    o = Options(); o.nneigh = 10; o.two_camera = 4;
    run("a two-camera neighbour", 6, o, true);
    o = Options(); o.nneigh = 20; o.stereo = true; o.pose_change_at = 7;
    run("a pose changed before a resolve", 7, o, true);
    o = Options(); o.nneigh = 25; o.erase_at = 6;
    run("KF1 map points erased before a resolve", 8, o, true);
    if (g_fail) { std::printf("%d failures\n", g_fail); return 1; }
    std::printf("TRIANGULATION MULTI TEST OK\n");
    return 0;
}
