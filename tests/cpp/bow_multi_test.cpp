// bow_multi_test.cpp — the two multi-target VS_GRAPHS::ORBmatcher::SearchByBoW overloads against the loops of single-target
// calls they stand for:
//     Tracking::Relocalization:               for (i) nmatches[i] = matcher.SearchByBoW(vpCandidateKFs[i], mCurrentFrame, vvpMapPointMatches[i]);
//     LoopClosing::DetectCommonRegionsFromBoW: for (j) num[j] = matcherBoW.SearchByBoW(mpCurrentKF, vpCovKFi[j], vvpMatchedMPs[j]);
// Every world has single- and two-camera keyframes, a two-camera frame or a single-camera one, bad map points, a keyframe
// without map points and a keyframe listed twice.  Every returned MapPoint* and every count must be identical.  Needs a GPU.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <random>
#include <vector>

#include "../../visual_sgraphs_b200/shim/ORBmatcher.h"

static int g_fail = 0;
#define EXPECT(cond, ...)                                                                                                   \
    do {                                                                                                                    \
        if (!(cond)) { std::printf("FAIL %s:%d: ", __FILE__, __LINE__); std::printf(__VA_ARGS__); std::printf("\n"); ++g_fail; } \
    } while (0)

constexpr int kLevels = 8;
constexpr int kNodes = 24;

struct MapPoint {
    bool bad = false;
    bool isBad() const { return bad; }
};

// What SearchByBoW reads from a Frame / KeyFrame (ORBmatcher.cc:226-428, :758-900).
struct View {
    int N = 0, Nleft = -1, NLeft = -1;
    std::vector<cv::KeyPoint> mvKeys, mvKeysUn, mvKeysRight;
    cv::Mat mDescriptors;
    std::vector<float> mvuRight, mvScaleFactors;
    float mnMinX = 0, mnMinY = 0, mnMaxX = 640, mnMaxY = 480;
    float mfGridElementWidthInv = 64.f / 640.f, mfGridElementHeightInv = 48.f / 480.f;
    std::map<unsigned, std::vector<unsigned>> mFeatVec;   // DBoW2::FeatureVector
    View() {
        float s = 1.f;
        for (int l = 0; l < kLevels; ++l, s *= 1.2f) mvScaleFactors.push_back(s);
    }
};
struct Frame : View {};
struct Camera {};
struct KeyFrame : View {
    Camera cam2;
    Camera *mpCamera2 = nullptr;
    std::vector<MapPoint *> mvpMapPoints;
    std::vector<MapPoint *> GetMapPointMatches() const { return mvpMapPoints; }
};

static std::vector<uint8_t> random_desc(std::mt19937 &rng) {
    std::vector<uint8_t> d(32);
    for (auto &x : d) x = (uint8_t)(rng() & 255);
    return d;
}

// A view of n features (nright of them a second camera's): features copy one of the scene's identities with a few bits
// flipped (the first byte, which picks the vocabulary node, is kept) or are distractors; angles follow the identity plus
// a per-view rotation, so the rotation check keeps most matches.
static void fill(View &v, int nleft, int nright, const std::vector<std::vector<uint8_t>> &ident, float rot, std::mt19937 &rng) {
    const int n = nleft + nright;
    v.N = n;
    v.mDescriptors.create(n, 32, CV_8UC1);
    std::vector<cv::KeyPoint> keys(n);
    for (int i = 0; i < n; ++i) {
        std::vector<uint8_t> d;
        float angle;
        if (rng() % 5) {
            const size_t k = rng() % ident.size();
            d = ident[k];
            for (int b = 0, nb = rng() % 60; b < nb; ++b) { const unsigned bit = 8 + rng() % 248; d[bit / 8] ^= (uint8_t)(1u << (bit % 8)); }
            angle = std::fmod((float)(k * 37 % 360) + rot + (float)(rng() % 5), 360.f);
        } else {
            d = random_desc(rng);
            angle = (float)(rng() % 360);
        }
        std::memcpy(v.mDescriptors.ptr(i), d.data(), 32);
        cv::KeyPoint &kp = keys[i];
        kp.pt.x = (float)(rng() % 6400) / 10.f;
        kp.pt.y = (float)(rng() % 4800) / 10.f;
        kp.octave = rng() % kLevels;
        kp.angle = angle;
        kp.size = 31.f;
        v.mFeatVec[(unsigned)((d[0] * 7 + 3) % kNodes)].push_back((unsigned)i);
    }
    v.mvKeys.assign(keys.begin(), keys.begin() + nleft);
    v.mvKeysRight.assign(keys.begin() + nleft, keys.end());
    v.mvKeysUn = v.mvKeys;
    if (nright) { v.Nleft = v.NLeft = nleft; } else { v.mvKeysUn = keys; }
}

struct World {
    std::vector<std::unique_ptr<KeyFrame>> kfs;
    std::vector<std::unique_ptr<MapPoint>> mps;
    std::vector<KeyFrame *> targets;        // the candidate list: includes a repeated keyframe
    Frame F;
    KeyFrame *current = nullptr;            // the keyframe of the KF-KF form
};

static void make_world(World &w, unsigned seed, int nkf, bool two_camera_frame) {
    std::mt19937 rng(seed);
    std::vector<std::vector<uint8_t>> ident(500);
    for (auto &d : ident) d = random_desc(rng);
    fill(w.F, two_camera_frame ? 350 : 500, two_camera_frame ? 300 : 0, ident, 0.f, rng);
    for (int k = 0; k <= nkf; ++k) {
        w.kfs.emplace_back(new KeyFrame());
        KeyFrame *kf = w.kfs.back().get();
        const bool two = k % 3 == 1;
        fill(*kf, 300 + rng() % 200, two ? 200 + rng() % 100 : 0, ident, (float)(rng() % 20), rng);
        if (two) kf->mpCamera2 = &kf->cam2;
        kf->mvpMapPoints.assign(kf->N, nullptr);
        if (k % 4 == 3) continue;           // a keyframe without map points
        for (int i = 0; i < kf->N; ++i) {
            if (rng() % 10 == 0) continue;
            w.mps.emplace_back(new MapPoint());
            w.mps.back()->bad = rng() % 15 == 0;
            kf->mvpMapPoints[i] = w.mps.back().get();
        }
    }
    w.current = w.kfs[0].get();
    for (int k = 1; k <= nkf; ++k) w.targets.push_back(w.kfs[k].get());
    if (nkf > 1) w.targets.push_back(w.targets[1]);   // the same keyframe twice
}

static void compare(const char *name, const std::vector<int> &counts_multi, const std::vector<std::vector<MapPoint *>> &multi,
                    const std::vector<int> &counts_loop, const std::vector<std::vector<MapPoint *>> &loop, int min_total) {
    EXPECT(counts_multi.size() == counts_loop.size() && multi.size() == loop.size(), "%s: %zu / %zu targets", name,
           counts_multi.size(), counts_loop.size());
    int total = 0, diffs = 0;
    for (size_t t = 0; t < counts_loop.size() && t < counts_multi.size(); ++t) {
        total += counts_loop[t];
        EXPECT(counts_multi[t] == counts_loop[t], "%s: target %zu: %d matches, the loop %d", name, t, counts_multi[t], counts_loop[t]);
        EXPECT(multi[t].size() == loop[t].size(), "%s: target %zu: %zu slots, the loop %zu", name, t, multi[t].size(), loop[t].size());
        for (size_t i = 0; i < multi[t].size() && i < loop[t].size(); ++i)
            if (multi[t][i] != loop[t][i] && diffs++ < 5) EXPECT(false, "%s: target %zu, slot %zu differs", name, t, i);
    }
    EXPECT(diffs == 0, "%s: %d differing slots", name, diffs);
    EXPECT(total >= min_total, "%s: the loop found %d matches, expected at least %d", name, total, min_total);
    std::printf("%s: %zu targets, %d matches\n", name, counts_loop.size(), total);
}

static void run(const char *name, unsigned seed, int nkf, bool two_camera_frame, float nnratio, bool check_ori) {
    World w;
    make_world(w, seed, nkf, two_camera_frame);
    VS_GRAPHS::ORBmatcher matcher(nnratio, check_ori);
    char what[128];
    {   // SearchByBoW(KF, F) over the candidates
        std::vector<std::vector<MapPoint *>> loop(w.targets.size()), multi;
        std::vector<int> counts_loop;
        for (size_t t = 0; t < w.targets.size(); ++t) counts_loop.push_back(matcher.SearchByBoW(w.targets[t], w.F, loop[t]));
        const std::vector<int> counts = matcher.SearchByBoW(w.targets, w.F, multi);
        std::snprintf(what, sizeof what, "%s / SearchByBoW(KFs, F)", name);
        compare(what, counts, multi, counts_loop, loop, w.targets.empty() ? 0 : 20);
    }
    {   // SearchByBoW(KF, KF) over the candidates
        std::vector<std::vector<MapPoint *>> loop(w.targets.size()), multi;
        std::vector<int> counts_loop;
        for (size_t t = 0; t < w.targets.size(); ++t) counts_loop.push_back(matcher.SearchByBoW(w.current, w.targets[t], loop[t]));
        const std::vector<int> counts = matcher.SearchByBoW(w.current, w.targets, multi);
        std::snprintf(what, sizeof what, "%s / SearchByBoW(KF, KFs)", name);
        compare(what, counts, multi, counts_loop, loop, w.targets.empty() ? 0 : 20);
    }
}

int main() {
    run("one-camera frame, nnratio 0.75", 1, 6, false, 0.75f, true);
    run("two-camera frame, nnratio 0.75", 2, 7, true, 0.75f, true);
    run("one-camera frame, nnratio 0.9, no rotation check", 3, 12, false, 0.9f, false);
    run("two-camera frame, nnratio 0.9", 4, 33, true, 0.9f, true);
    run("one target", 5, 1, false, 0.75f, true);
    run("no targets", 6, 0, true, 0.75f, true);
    if (g_fail) { std::printf("%d failures\n", g_fail); return 1; }
    std::printf("BOW MULTI TEST OK\n");
    return 0;
}
