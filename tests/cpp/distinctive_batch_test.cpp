// distinctive_batch_test.cpp — the batched VS_GRAPHS::ORBmatcher::ComputeDistinctiveDescriptors(vpMPs) against the loop it
// stands for, LocalMapping's `for (pMP : vpMapPoints) pMP->ComputeDistinctiveDescriptors();` (ProcessNewKeyFrame, the update
// loop of SearchInNeighbors).  Each world is generated twice from one seed; the loop of the reference's per-point method
// (MapPoint.cc:340-417, restated below) runs on one copy, the batch on the other, and every map point's descriptor bytes
// must be equal.  The stand-in MapPoint carries the reference's tuple observation map (left index, right index; the right
// index already indexes the combined descriptor table of a two-camera keyframe) and the one method the integration adds,
// SetDistinctiveDescriptor.  Keyframes live in one array, so a map keyed on KeyFrame* iterates them in the same order in
// both copies.
//
// Two builds: with tests/cpp/vsg_on_oracle.cpp + tests/cpp/vsg_on_oracle_distinctive.cpp + oracle/liborb_oracle.so (no GPU),
// and with -lvsg_cuda (B200).
//   usage: distinctive_batch_test            the checks
//          distinctive_batch_test --time     also times the loop against the batch at 300 / 1000 / 3000 points
#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <random>
#include <string>
#include <tuple>
#include <vector>

#include "../../visual_sgraphs_b200/shim/ORBmatcher.h"

using VS_GRAPHS::ORBmatcher;

static int g_fail = 0;
#define EXPECT(cond, ...)                                                                                                   \
    do {                                                                                                                    \
        if (!(cond)) { std::printf("FAIL %s:%d: ", __FILE__, __LINE__); std::printf(__VA_ARGS__); std::printf("\n"); ++g_fail; } \
    } while (0)

struct KeyFrame {
    bool bad = false;
    int NLeft = -1;                                  // -1: one camera; else rows [NLeft, N) are the right camera's
    cv::Mat mDescriptors;
    bool isBad() const { return bad; }
};

struct MapPoint {
    bool bad = false;
    std::map<KeyFrame *, std::tuple<int, int>> mObservations;
    cv::Mat mDescriptor{1, 32, CV_8UC1};
    std::mutex mMutexFeatures;

    bool isBad() { std::unique_lock<std::mutex> lock(mMutexFeatures); return bad; }
    std::map<KeyFrame *, std::tuple<int, int>> GetObservations() {
        std::unique_lock<std::mutex> lock(mMutexFeatures);
        return mObservations;
    }
    // MapPoint.cc:340-417
    void ComputeDistinctiveDescriptors() {
        std::vector<cv::Mat> vDescriptors;
        std::map<KeyFrame *, std::tuple<int, int>> observations;
        {
            std::unique_lock<std::mutex> lock1(mMutexFeatures);
            if (bad) return;
            observations = mObservations;
        }
        if (observations.empty()) return;
        vDescriptors.reserve(observations.size());
        for (auto mit = observations.begin(), mend = observations.end(); mit != mend; mit++) {
            KeyFrame *pKF = mit->first;
            if (!pKF->isBad()) {
                std::tuple<int, int> indexes = mit->second;
                int leftIndex = std::get<0>(indexes), rightIndex = std::get<1>(indexes);
                if (leftIndex != -1) vDescriptors.push_back(pKF->mDescriptors.row(leftIndex));
                if (rightIndex != -1) vDescriptors.push_back(pKF->mDescriptors.row(rightIndex));
            }
        }
        if (vDescriptors.empty()) return;
        const size_t N = vDescriptors.size();
        std::vector<std::vector<float>> Distances(N, std::vector<float>(N));
        for (size_t i = 0; i < N; i++) {
            Distances[i][i] = 0;
            for (size_t j = i + 1; j < N; j++) {
                int distij = ORBmatcher::DescriptorDistance(vDescriptors[i], vDescriptors[j]);
                Distances[i][j] = distij;
                Distances[j][i] = distij;
            }
        }
        int BestMedian = INT_MAX;
        int BestIdx = 0;
        for (size_t i = 0; i < N; i++) {
            std::vector<int> vDists(Distances[i].begin(), Distances[i].end());
            std::sort(vDists.begin(), vDists.end());
            int median = vDists[0.5 * (N - 1)];
            if (median < BestMedian) {
                BestMedian = median;
                BestIdx = i;
            }
        }
        {
            std::unique_lock<std::mutex> lock(mMutexFeatures);
            mDescriptor = vDescriptors[BestIdx].clone();
        }
    }
    // the integration's addition to MapPoint (INTEGRATION.md §1)
    void SetDistinctiveDescriptor(const cv::Mat &descriptor) {
        std::unique_lock<std::mutex> lock(mMutexFeatures);
        mDescriptor = descriptor.clone();
    }
};

constexpr uint8_t kUntouched = 0xA5;                 // every point's descriptor before the call

struct World {
    std::vector<KeyFrame> kfs;                       // one array: pointer order == index order in both copies
    std::vector<std::unique_ptr<MapPoint>> mps;
    std::vector<MapPoint *> list;                    // what the caller passes: may hold NULL and repeats
    int rows = 0;                                    // observed rows of the listed points that are not bad (for the timing)

    void init_keyframes(int nkf, int nfeat) {
        kfs.resize(nkf);
        for (auto &kf : kfs) kf.mDescriptors = cv::Mat(nfeat, 32, CV_8UC1);
    }
    MapPoint *add_point() {
        mps.emplace_back(new MapPoint);
        std::memset(mps.back()->mDescriptor.ptr(0), kUntouched, 32);
        return mps.back().get();
    }
    void set_row(int kf, int row, const uint8_t *d) { std::memcpy(kfs[kf].mDescriptors.ptr(row), d, 32); }
};

static void perturb(std::mt19937 &rng, const uint8_t *base, int flips, uint8_t *out) {
    std::memcpy(out, base, 32);
    for (int f = 0; f < flips; ++f) {
        const int bit = (int)(rng() % 256);
        out[bit / 8] ^= (uint8_t)(1u << (bit % 8));
    }
}

// Random world: 80 keyframes (about 10 % bad, half of them two-camera), npoints points with 0..60 observations each
// (left-only, right-only or both on a two-camera keyframe), about 5 % bad points, the list shuffled with NULL entries.
// Each observed row is the point's base descriptor with a few flipped bits, so equal medians are common.
static void random_world(World &w, unsigned seed, int npoints) {
    std::mt19937 rng(seed);
    const int nkf = 80, nleft = 2000, nfeat = 2 * nleft;
    w.init_keyframes(nkf, nfeat);
    std::vector<int> next_row(nkf, 0);
    for (int k = 0; k < nkf; ++k) {
        w.kfs[k].bad = rng() % 10 == 0;
        w.kfs[k].NLeft = rng() % 2 ? nleft : -1;
    }
    std::vector<int> order(nkf);
    for (int k = 0; k < nkf; ++k) order[k] = k;
    for (int p = 0; p < npoints; ++p) {
        MapPoint *mp = w.add_point();
        mp->bad = rng() % 20 == 0;
        uint8_t base[32];
        for (auto &b : base) b = (uint8_t)rng();
        const int nobs = rng() % 4 == 0 ? (int)(rng() % 61) : (int)(rng() % 16);   // mostly short, some long
        const int maxflips = 1 + (int)(rng() % 24);
        std::shuffle(order.begin(), order.end(), rng);
        for (int o = 0; o < nobs; ++o) {
            const int k = order[o];
            KeyFrame &kf = w.kfs[k];
            int left = -1, right = -1;
            const int kind = kf.NLeft == -1 ? 0 : (int)(rng() % 3);   // 0 left only, 1 right only, 2 both
            if (next_row[k] >= nleft) continue;
            if (kind != 1) left = next_row[k];
            if (kind != 0) right = kf.NLeft + next_row[k];
            ++next_row[k];
            uint8_t d[32];
            if (left != -1) { perturb(rng, base, (int)(rng() % maxflips), d); w.set_row(k, left, d); }
            if (right != -1) { perturb(rng, base, (int)(rng() % maxflips), d); w.set_row(k, right, d); }
            mp->mObservations[&kf] = std::make_tuple(left, right);
            if (!mp->bad && !kf.bad) w.rows += (left != -1) + (right != -1);
        }
    }
    for (auto &mp : w.mps) w.list.push_back(mp.get());
    std::shuffle(w.list.begin(), w.list.end(), rng);
    for (size_t i = 0; i < w.list.size(); i += 1 + rng() % 60) w.list.insert(w.list.begin() + i, nullptr);
}

// Constructed world: each point pins one case the batch must read as the reference does.  `expect[i]` is the row (of
// keyframe 0's table) point i must end with, or -1 for "left alone".
static std::vector<int> constructed_world(World &w) {
    w.init_keyframes(8, 64);
    for (int k = 0; k < 8; ++k)
        for (int r = 0; r < 64; ++r) {
            uint8_t d[32] = {};
            d[0] = (uint8_t)k; d[1] = (uint8_t)r; d[31] = 0x5A;                     // distinct rows
            w.set_row(k, r, d);
        }
    w.kfs[1].bad = w.kfs[2].bad = true;
    w.kfs[3].NLeft = 32;                             // two-camera keyframe: rows 32..63 are the right camera's
    std::vector<int> expect;
    auto row_bits = [&](int k, int r, int lo, int nbits) {   // row r of keyframe k: bits [lo, lo + nbits) set, rest 0
        uint8_t d[32] = {};
        for (int b = lo; b < lo + nbits; ++b) d[b / 8] |= (uint8_t)(1u << (b % 8));
        w.set_row(k, r, d);
    };
    // A: every observer is bad -> left alone
    MapPoint *a = w.add_point();
    a->mObservations[&w.kfs[1]] = std::make_tuple(0, -1);
    a->mObservations[&w.kfs[2]] = std::make_tuple(1, -1);
    expect.push_back(-1);
    // B: right-only observation; without its row the answer would be keyframe 0's row 2
    MapPoint *b = w.add_point();
    row_bits(0, 2, 0, 40); row_bits(0, 3, 0, 0); row_bits(3, 40, 0, 1); row_bits(3, 41, 0, 2);
    b->mObservations[&w.kfs[0]] = std::make_tuple(2, -1);
    b->mObservations[&w.kfs[3]] = std::make_tuple(-1, 40);
    b->mObservations[&w.kfs[4]] = std::make_tuple(3, -1);
    expect.push_back(-2);                            // keyframe 3's row 40: checked below
    // C: equal medians across three rows (all 8): the first row in map order wins
    MapPoint *c = w.add_point();
    row_bits(0, 10, 0, 0); row_bits(5, 10, 0, 8); row_bits(6, 10, 8, 8);
    c->mObservations[&w.kfs[0]] = std::make_tuple(10, -1);
    c->mObservations[&w.kfs[5]] = std::make_tuple(10, -1);
    c->mObservations[&w.kfs[6]] = std::make_tuple(10, -1);
    expect.push_back(10);
    // D: even N = 4 where the entry 0.5 * (N - 1) = 1 and the entry N / 2 = 2 of the sorted rows pick different rows.
    //    Rows (bits set): R0 = [0,10), R1 = [0,11), R2 = [0,30), R3 = [0,31); distances R0: 0 1 20 21, R1: 1 0 19 20,
    //    R2: 20 19 0 1, R3: 21 20 1 0 -> entry 1: 1 1 1 1 (row 0 wins), entry 2: 20 19 19 20 (row 1 would win).
    MapPoint *d4 = w.add_point();
    row_bits(0, 20, 0, 10); row_bits(4, 20, 0, 11); row_bits(5, 20, 0, 30); row_bits(6, 20, 0, 31);
    for (int k : {0, 4, 5, 6}) d4->mObservations[&w.kfs[k]] = std::make_tuple(20, -1);
    expect.push_back(20);
    // E: odd N = 5 among the observations of two bad keyframes; rows [0,3) [0,5) [0,40) [0,41) [0,60): the sorted rows'
    //    entries 2 are 37 35 20 19 20 -> keyframe 6's row.  With the bad keyframes' rows (4 bits each) counted, N = 7 and
    //    keyframe 1's row would win.
    MapPoint *e = w.add_point();
    row_bits(0, 30, 0, 3); row_bits(4, 30, 0, 5); row_bits(5, 30, 0, 40); row_bits(6, 30, 0, 41); row_bits(7, 30, 0, 60);
    for (int k : {0, 4, 5, 6, 7}) e->mObservations[&w.kfs[k]] = std::make_tuple(30, -1);
    e->mObservations[&w.kfs[1]] = std::make_tuple(30, -1);   // bad keyframes: their rows must not count
    e->mObservations[&w.kfs[2]] = std::make_tuple(31, -1);
    row_bits(1, 30, 0, 4); row_bits(2, 31, 0, 4);
    expect.push_back(-3);                            // keyframe 6's row 30: checked below
    // F: a point listed twice gets the same answer twice; G: a bad point is left alone; H: no observations
    MapPoint *f = w.add_point();
    row_bits(0, 50, 0, 2); row_bits(5, 50, 0, 3);
    f->mObservations[&w.kfs[0]] = std::make_tuple(50, -1);
    f->mObservations[&w.kfs[5]] = std::make_tuple(50, -1);
    expect.push_back(50);
    MapPoint *g = w.add_point();
    g->bad = true;
    g->mObservations[&w.kfs[0]] = std::make_tuple(60, -1);
    expect.push_back(-1);
    w.add_point();
    expect.push_back(-1);
    w.list = {a, nullptr, b, c, f, d4, e, f, g, w.mps.back().get(), nullptr};
    return expect;
}

static bool same_descriptors(const World &x, const World &y, const char *what) {
    int bad = 0;
    for (size_t i = 0; i < x.mps.size(); ++i)
        if (std::memcmp(x.mps[i]->mDescriptor.ptr(0), y.mps[i]->mDescriptor.ptr(0), 32) != 0) {
            if (bad++ < 5) std::printf("FAIL %s: map point %zu: the batch's descriptor differs from the loop's\n", what, i);
        }
    if (bad) ++g_fail;
    return bad == 0;
}

static int changed(const World &w) {
    int n = 0;
    for (auto &mp : w.mps) n += mp->mDescriptor.ptr(0)[0] != kUntouched || mp->mDescriptor.ptr(0)[1] != kUntouched;
    return n;
}

static void run_loop(World &w) {
    for (MapPoint *p : w.list)
        if (p) p->ComputeDistinctiveDescriptors();
}

static double median_us(std::vector<double> v) {
    std::sort(v.begin(), v.end());
    return v[v.size() / 2];
}

int main(int argc, char **argv) {
    const bool timing = argc > 1 && std::string(argv[1]) == "--time";
    for (int npoints : {300, 1000, 3000}) {
        for (unsigned seed : {1u, 2u}) {
            World loop, batch;
            random_world(loop, seed * 7919u + npoints, npoints);
            random_world(batch, seed * 7919u + npoints, npoints);
            run_loop(loop);
            ORBmatcher::ComputeDistinctiveDescriptors(batch.list);
            const std::string what = "random world of " + std::to_string(npoints) + " points, seed " + std::to_string(seed);
            same_descriptors(loop, batch, what.c_str());
            EXPECT(changed(batch) > npoints / 2, "%s: only %d descriptors set", what.c_str(), changed(batch));
        }
    }
    {
        World loop, batch;
        const std::vector<int> expect = constructed_world(loop);
        constructed_world(batch);
        run_loop(loop);
        ORBmatcher::ComputeDistinctiveDescriptors(batch.list);
        same_descriptors(loop, batch, "constructed world");
        for (size_t i = 0; i < expect.size(); ++i) {
            const uint8_t *got = batch.mps[i]->mDescriptor.ptr(0);
            const uint8_t *want = expect[i] == -1 ? nullptr
                                  : expect[i] == -2 ? batch.kfs[3].mDescriptors.ptr(40)
                                  : expect[i] == -3 ? batch.kfs[6].mDescriptors.ptr(30)
                                                    : batch.kfs[0].mDescriptors.ptr(expect[i]);
            if (!want) EXPECT(got[0] == kUntouched && got[31] == kUntouched, "constructed point %zu: expected to be left alone", i);
            else EXPECT(std::memcmp(got, want, 32) == 0, "constructed point %zu: not the expected row", i);
        }
        World empty_loop, empty_batch;                // an empty vector changes nothing
        constructed_world(empty_loop);
        constructed_world(empty_batch);
        ORBmatcher::ComputeDistinctiveDescriptors(std::vector<MapPoint *>());
        EXPECT(changed(empty_batch) == 0, "empty vector: descriptors changed");
    }
    if (timing) {
        std::printf("%8s %8s %14s %14s %8s\n", "points", "rows", "loop_us", "batch_us", "speedup");
        for (int npoints : {300, 1000, 3000}) {
            World w;
            random_world(w, 99u + npoints, npoints);
            for (int r = 0; r < 3; ++r) { run_loop(w); ORBmatcher::ComputeDistinctiveDescriptors(w.list); }   // warm-up
            std::vector<double> tl, tb;
            for (int r = 0; r < 21; ++r) {           // alternate the two forms; both recompute the same answers
                auto t0 = std::chrono::steady_clock::now();
                run_loop(w);
                auto t1 = std::chrono::steady_clock::now();
                ORBmatcher::ComputeDistinctiveDescriptors(w.list);
                auto t2 = std::chrono::steady_clock::now();
                tl.push_back(std::chrono::duration<double, std::micro>(t1 - t0).count());
                tb.push_back(std::chrono::duration<double, std::micro>(t2 - t1).count());
            }
            const double l = median_us(tl), b = median_us(tb);
            std::printf("%8d %8d %14.1f %14.1f %8.2f\n", npoints, w.rows, l, b, l / b);
        }
    }
    if (g_fail) {
        std::printf("DISTINCTIVE BATCH TEST FAILED: %d checks\n", g_fail);
        return 1;
    }
    std::printf("DISTINCTIVE BATCH TEST OK\n");
    return 0;
}
