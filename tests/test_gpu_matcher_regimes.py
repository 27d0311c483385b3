"""The matcher's Search* methods against the CPU oracle across frame geometries, pyramid configurations and the
size-dependent paths of the device code (run on the B200 with -m gpu).

test_gpu_matcher_methods.py / test_gpu_matcher_kf.py check every method on one 640x480 scene with integer bounds and
an 8 x 1.2 pyramid.  The device code depends on exactly what that scene holds fixed:
  - the grid geometry: area_search_kernel / window_best_kernel find cells with floorf / ceilf((x - min_x +- r) * inv_w),
    vsg_frame_create bins keypoints with std::round and drops the ones outside the grid;
  - the level tables: windows scale with scale[level], levels [level - 1, level] (min_level = -1 at level 0), the Fuse
    chi-square gate reads inv_sigma2[octave];
  - projection_map_max_dist(nnratio), which drops candidates that cannot change SearchByProjection(Frame, MapPoints);
  - the size-dependent paths: the per-query replay below kOrderedReplayMinQueries queries and the device-ordered lists
    from there on, the one retry of both area searches when the first candidate buffer overflows, and vsg_knn2's
    automatic choice between the tensor-core kernel and the POPC kernel.
Every method runs on every configuration below and must equal the oracle exactly; the size-dependent tests also check,
through vsg_launch_count(), which path ran.
"""
import ctypes as C

import numpy as np
import pytest

from tests import match_scenarios as sc

pytestmark = pytest.mark.gpu

SHIFT = (9, 5)
# id: (size, nfeatures, scale factor, levels, grid bounds (min_x, min_y, max_x, max_y) or None for the image)
CONFIGS = {
    "default": ((640, 480), 1000, 1.2, 8, None),
    # undistorted bounds of a distorted camera: non-integer, partly negative, and narrower than the image on the right
    # and bottom, so that some keypoints round to a cell outside the grid and are dropped
    "euroc_distorted": ((752, 480), 1200, 1.2, 8, (-13.7, -9.2, 711.4, 452.8)),
    "kitti": ((1241, 376), 2000, 1.2, 8, None),
    "hd": ((1280, 720), 2000, 1.2, 8, None),
    "fine": ((640, 480), 1000, 1.1, 12, None),
    "coarse": ((640, 480), 1000, 1.5, 5, None),
    # inverse cell size exactly 0.125: planted keypoints at cell coordinate k + 0.5 (std::round and round-half-even
    # disagree), windows whose edges land exactly on cell boundaries, keypoints at exactly |dx| == r
    "exact_cells": ((512, 384), 1000, 1.2, 8, None),
}
CFG_IDS = list(CONFIGS)
ORDERED_REPLAY_MIN_QUERIES = 20000          # kOrderedReplayMinQueries (csrc/match_methods.cu)
# kernel launches (count_launch) of each path
RAW_LAUNCHES, ORDERED_LAUNCHES = 1, 3       # area_search_kernel; + scan_counts_kernel + order_segments_kernel
KNN_POPC_LAUNCHES, KNN_TC_LAUNCHES = 2, 4   # knn2_kernel + knn2_merge_kernel; 2 x expand_pm1 + knn2_tc + merge_parts


def _matcher(nnratio=0.6, check_ori=True):
    from visual_sgraphs_b200.matcher import ORBmatcher
    return ORBmatcher(nnratio, check_ori)


def _launches():
    from visual_sgraphs_b200 import _lib
    return _lib.load().vsg_launch_count()


def _same(cfg, method, **arrays):
    """Each keyword is (got, want); fails naming the configuration, the method, the array and its first differing index."""
    for name, (got, want) in arrays.items():
        got, want = np.asarray(got), np.asarray(want)
        if got.shape != want.shape:
            pytest.fail("%s / %s: %s has shape %s, the oracle's %s" % (cfg, method, name, got.shape, want.shape))
        if got.ndim == 0:
            if got != want:
                pytest.fail("%s / %s: %s is %s, the oracle's %s" % (cfg, method, name, got, want))
            continue
        bad = np.argwhere(got != want)
        if len(bad):
            i = tuple(int(k) for k in bad[0])
            pytest.fail("%s / %s: %s differs first at index %s: %s, oracle %s (%d differences)" %
                        (cfg, method, name, i if len(i) > 1 else i[0], got[i], want[i], len(bad)))


def _floor(cfg, method, what, value, floor):
    assert value > floor, "%s / %s: %s = %d, expected more than %d (the scene exercises nothing)" % (cfg, method, what, value,
                                                                                                     floor)


class Scene:
    """Two related frames of one configuration (frame B = frame A shifted by SHIFT plus noise) extracted by the oracle with
    the configuration's pyramid; FrameData carry its scale factors, bounds and size."""

    def __init__(self, oracle, cfg):
        size, nfeat, scale, nlevels, bounds = CONFIGS[cfg]
        self.cfg, self.size, self.nfeat, self.scale, self.nlevels, self.bounds = cfg, size, nfeat, scale, nlevels, bounds
        ka, da, kb, db = sc.two_frames(oracle, shift=SHIFT, size=size, nfeat=nfeat, scale=scale, nlevels=nlevels)
        ka, kb = ka.copy(), kb.copy()
        if cfg == "exact_cells":
            ka, kb = _plant_half_cells(ka, 1), _plant_half_cells(kb, 2)
        self.ka, self.da, self.kb, self.db = ka, da, kb, db
        tables = oracle.OracleExtractor(nfeat, scale, nlevels).tables()
        self.scale_factors, self.sigma2, self.inv_sigma2 = tables["scale"], tables["sigma2"], tables["inv_sigma2"]

    def frame(self, which="a", stereo_seed=None):
        keys, desc = (self.ka, self.da) if which == "a" else (self.kb, self.db)
        return sc.frame_data(keys, desc, size=self.size, stereo_seed=stereo_seed, bounds=self.bounds,
                             scale_factors=self.scale_factors)


def _plant_half_cells(keys, seed):
    """Moves a third of the keypoints to x, y = 16 j + 4: cell coordinate 2 j + 0.5 at the inverse cell size 0.125, which
    std::round (PosInGrid) puts in cell 2 j + 1 and round-half-even in cell 2 j."""
    rng = np.random.default_rng(seed)
    pick = rng.random(len(keys)) < 1 / 3
    for f in ("x", "y"):
        keys[f][pick] = (16 * np.floor(keys[f][pick] / 16) + 4).astype(np.float32)
    return keys


_SCENES = {}


@pytest.fixture(scope="module")
def scenes(oracle):
    def get(cfg):
        if cfg not in _SCENES:
            _SCENES[cfg] = Scene(oracle, cfg)
        return _SCENES[cfg]
    return get


# ---- the scene geometry itself -------------------------------------------------------------------------------------------

def test_scene_geometry(scenes):
    """The configurations hold what the tests below rely on."""
    S = scenes("euroc_distorted")
    v = S.frame().view
    px = np.floor((S.ka["x"] - np.float32(v.min_x)) * np.float32(v.grid_inv_w) + 0.5)
    py = np.floor((S.ka["y"] - np.float32(v.min_y)) * np.float32(v.grid_inv_h) + 0.5)
    outside = (px < 0) | (px >= 64) | (py < 0) | (py >= 48)
    assert 10 < outside.sum() < len(px) // 4
    E = scenes("exact_cells")
    assert E.frame().view.grid_inv_w == 0.125 and E.frame().view.grid_inv_h == 0.125
    half = (E.ka["x"] * np.float32(0.125)) % 1 == 0.5
    assert half.sum() > 200
    for cfg in ("fine", "coarse"):
        F = scenes(cfg)
        assert len(F.scale_factors) == CONFIGS[cfg][3] and F.ka["octave"].max() == CONFIGS[cfg][3] - 1


# ---- GetFeaturesInArea ----------------------------------------------------------------------------------------------------

def _area_queries(S, rng, nq=400):
    w, h = S.size
    L = S.nlevels
    qx = rng.uniform(-30, w + 30, nq).astype(np.float32)
    qy = rng.uniform(-30, h + 30, nq).astype(np.float32)
    qr = rng.uniform(1, 70, nq).astype(np.float32)
    choices = np.array([(-1, -1), (0, 0), (-1, 0), (2, 3), (1, -1), (0, 4), (L - 2, L - 1), (L - 1, L - 1), (L - 1, -1)],
                       np.int32)
    pick = rng.integers(0, len(choices), nq)
    lo, hi = choices[pick, 0].copy(), choices[pick, 1].copy()
    if S.cfg == "exact_cells":
        half = np.nonzero(((S.ka["x"] * np.float32(0.125)) % 1 == 0.5) & ((S.ka["y"] * np.float32(0.125)) % 1 == 0.5))[0]
        ex, ey, er = [], [], []
        for j in half[:80]:                       # a keypoint at exactly |dx| == r or |dy| == r: outside (strict <)
            r = float(rng.choice([3, 4, 8, 12]))
            kx, ky = float(S.ka["x"][j]), float(S.ka["y"][j])
            ex += [kx + r, kx - r, kx, kx]
            ey += [ky, ky, ky + r, ky - 0.5 * r]
            er += [r, r, r, r]
        for _ in range(120):                      # window edges x +- r, y +- r exactly on cell boundaries
            r = float(rng.integers(2, 24))
            a, b = int(rng.integers(0, 64)), int(rng.integers(0, 48))
            ex += [8 * a + r, 8 * a - r]
            ey += [8 * b - r, 8 * b + r]
            er += [r, r]
        n = len(ex)
        qx, qy, qr = (np.concatenate([v, np.array(e, np.float32)]) for v, e in ((qx, ex), (qy, ey), (qr, er)))
        lo = np.concatenate([lo, np.full(n, -1, np.int32)])
        hi = np.concatenate([hi, np.full(n, -1, np.int32)])
    return qx, qy, qr, lo, hi


def _check_area_lists(cfg, method, oracle, fd, q, ptr, idx, dist):
    qx, qy, qr, lo, hi, qdesc = q
    total = 0
    for k in range(len(qx)):
        want = oracle.get_features_in_area(fd.view, float(qx[k]), float(qy[k]), float(qr[k]), int(lo[k]), int(hi[k]))
        got = idx[ptr[k]:ptr[k + 1]]
        if not np.array_equal(got, want):
            n = min(len(got), len(want))
            at = int(np.argmax(got[:n] != want[:n])) if (got[:n] != want[:n]).any() else n
            pytest.fail("%s / %s: query %d (x %r, y %r, r %r, levels %d..%d) lists %d candidates, the oracle %d; first "
                        "difference at position %d: %s, oracle %s" %
                        (cfg, method, k, float(qx[k]), float(qy[k]), float(qr[k]), lo[k], hi[k], len(got), len(want), at,
                         got[at:at + 8].tolist(), want[at:at + 8].tolist()))
        wd = [oracle.descriptor_distance(qdesc[k], fd.descriptors[j]) for j in want]
        _same(cfg, method + " distances of query %d" % k, dist=(dist[ptr[k]:ptr[k + 1]], wd))
        total += len(want)
    return total


@pytest.mark.parametrize("cfg", CFG_IDS)
def test_area_search(oracle, scenes, cfg):
    S = scenes(cfg)
    fd = S.frame()
    rng = np.random.default_rng(8)
    qx, qy, qr, lo, hi = _area_queries(S, rng)
    qdesc = S.db[rng.integers(0, len(S.db), len(qx))]
    m = _matcher()
    ptr, idx, dist = m.area_search(m.frame(fd), qx, qy, qr, lo, hi, qdesc)
    total = _check_area_lists(cfg, "area_search", oracle, fd, (qx, qy, qr, lo, hi, qdesc), ptr, idx, dist)
    _floor(cfg, "area_search", "candidates", total, 1000)


# ---- SearchByProjection(Frame&, vector<MapPoint*>&) --------------------------------------------------------------------

def _qualifying(pts, far=False, th_far=50.0):
    q = pts["in_view"].astype(bool) & ~pts["bad"].astype(bool)
    if far:
        q &= ~(pts["depth"] > np.float32(th_far))
    return q


def _map_case(S, stereo):
    fd = S.frame(stereo_seed=5 if stereo else None)
    pts, desc, occ = sc.track_points(fd, S.kb, S.db, SHIFT, 21, stereo, nlevels=S.nlevels)
    th, far = (5.0, True) if stereo else (3.0, False)
    return fd, pts, desc, occ, th, far


@pytest.mark.parametrize("nnratio", [0.6, 0.8, 0.9, 1.0])
@pytest.mark.parametrize("stereo", [False, True])
@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_by_projection_map(oracle, scenes, cfg, stereo, nnratio):
    S = scenes(cfg)
    fd, pts, desc, occ, th, far = _map_case(S, stereo)
    searched = pts["level"][_qualifying(pts, far, 40.0)]
    assert (searched == 0).any() and (searched == S.nlevels - 1).any(), "%s: predicted levels 0 and top not both searched" % cfg
    m = _matcher(nnratio)
    nm, assign = m.SearchByProjectionMap(m.frame(fd), occ, pts, desc, th, far, 40.0)
    wnm, wassign = oracle.search_by_projection_map(fd.view, occ, pts, desc, th, far, 40.0, float(np.float32(nnratio)))
    method = "SearchByProjectionMap(%s, nnratio %g)" % ("stereo" if stereo else "mono", nnratio)
    _same(cfg, method, nmatches=(nm, wnm), assign=(assign, wassign))
    _floor(cfg, method, "nmatches", wnm, 100)


def _max_dist(nnratio):
    """projection_map_max_dist: the largest distance a candidate list keeps at this nnratio."""
    d = 101
    while d < 256 and not np.float32(nnratio) * np.float32(d) >= np.float32(100):
        d += 1
    return d - 1


@pytest.mark.parametrize("nnratio", [0.6, 0.8, 0.9, 1.0])
def test_search_by_projection_map_pruning_edges(oracle, nnratio):
    """Pairs of keypoints alone in their map point's window, at the distances where the candidate pruning decides: the best
    at TH_HIGH - 1 .. TH_HIGH + 1, the second best at the largest kept distance or one more, on the same level or not."""
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE, TRACK_POINT_DTYPE
    rng = np.random.default_rng(int(nnratio * 10))
    keep = _max_dist(nnratio)
    npairs = 15 * 11
    keys = np.zeros(2 * npairs, KEYPOINT_DTYPE)
    desc = np.zeros((2 * npairs, 32), np.uint8)
    pts = np.zeros(npairs, TRACK_POINT_DTYPE)
    qdesc = rng.integers(0, 256, (npairs, 32), dtype=np.uint8)

    def flipped(d, nbits):
        bits = np.unpackbits(d)
        bits[rng.choice(256, nbits, replace=False)] ^= 1
        return np.packbits(bits)

    for p in range(npairs):
        x, y = np.float32(20 + 40 * (p % 15)), np.float32(20 + 40 * (p // 15))
        d_best = int(rng.choice([99, 100, 100, 100, 101]))
        d_second = int(rng.choice([keep, keep, keep + 1, keep - 1])) if keep < 256 else 255
        lvl_b = 0 if rng.random() < 0.8 else 1
        first = 2 * p + int(rng.integers(0, 2))            # which of the two indices holds the best one
        second = 4 * p + 1 - first
        keys[first] = (x, y, 31, 0, 1, 0, -1)
        keys[second] = (x + np.float32(1.5), y, 31, 0, 1, lvl_b, -1)
        desc[first], desc[second] = flipped(qdesc[p], d_best), flipped(qdesc[p], d_second)
        pts[p] = (x + np.float32(0.75), y, 0, 1.0, 10.0, lvl_b, 1, 0, 1, 0)
    fd = sc.frame_data(keys, desc)
    occ = np.zeros(len(keys), np.uint8)
    m = _matcher(nnratio)
    nm, assign = m.SearchByProjectionMap(m.frame(fd), occ, pts, qdesc, 3.0)
    wnm, wassign = oracle.search_by_projection_map(fd.view, occ, pts, qdesc, 3.0, False, 50.0, float(np.float32(nnratio)))
    method = "SearchByProjectionMap(nnratio %g, max kept distance %d)" % (nnratio, keep)
    _same("planted_pairs", method, nmatches=(nm, wnm), assign=(assign, wassign))
    _floor("planted_pairs", method, "nmatches", wnm, 20)
    _floor("planted_pairs", method, "rejected by the ratio test", npairs - wnm, 5)


@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_by_projection_map_two_cameras(oracle, scenes, cfg):
    S = scenes(cfg)
    sc2 = sc.two_camera_scene(oracle, seed=11, size=S.size, nfeat=S.nfeat, scale=S.scale, nlevels=S.nlevels, bounds=S.bounds)
    m = _matcher(0.8)
    nm, assign = m.SearchByProjectionMap2Cam(m.frame(sc2["fl"]), m.frame(sc2["fr"]), sc2["occupied"], sc2["l2r"], sc2["r2l"],
                                             sc2["pl"], sc2["pr"], sc2["desc"], 3.0, False, 40.0)
    wnm, wassign = oracle.search_by_projection_map_2cam(sc2["fl"].view, sc2["fr"].view, sc2["occupied"], sc2["l2r"], sc2["r2l"],
                                                        sc2["pl"], sc2["pr"], sc2["desc"], 3.0, False, 40.0, float(np.float32(0.8)))
    _same(cfg, "SearchByProjectionMap2Cam", nmatches=(nm, wnm), assign=(assign, wassign))
    nl = sc2["fl"].n
    _floor(cfg, "SearchByProjectionMap2Cam", "left matches", (wassign[:nl] >= 0).sum(), 100)
    _floor(cfg, "SearchByProjectionMap2Cam", "right matches", (wassign[nl:] >= 0).sum(), 100)


# ---- SearchByProjection(Frame&, const Frame&) ----------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_by_projection_last(oracle, scenes, cfg, mode):
    S = scenes(cfg)
    fd = S.frame(stereo_seed=9)
    pts, desc, occ = sc.proj_points(fd, S.kb, S.db, SHIFT, 4, size=S.size)
    m = _matcher(0.9, True)
    nm, assign = m.SearchByProjectionLast(m.frame(fd), occ, pts, desc, 15.0, mode)
    wnm, wassign = oracle.search_by_projection_last(fd.view, occ, pts, desc, 15.0, mode, True)
    method = "SearchByProjectionLast(mode %d)" % mode
    _same(cfg, method, nmatches=(nm, wnm), assign=(assign, wassign))
    _floor(cfg, method, "nmatches", wnm, 50)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_by_projection_last_two_cameras(oracle, scenes, cfg, mode):
    S = scenes(cfg)
    sc2 = sc.two_camera_last_scene(oracle, seed=11, size=S.size, nfeat=S.nfeat, scale=S.scale, nlevels=S.nlevels,
                                   bounds=S.bounds)
    m = _matcher(0.9, True)
    nm, assign = m.SearchByProjectionLast2Cam(m.frame(sc2["fl"]), m.frame(sc2["fr"]), sc2["occupied"], sc2["pl"], sc2["pr"],
                                              sc2["desc"], 15.0, mode)
    wnm, wassign = oracle.search_by_projection_last_2cam(sc2["fl"].view, sc2["fr"].view, sc2["occupied"], sc2["pl"], sc2["pr"],
                                                         sc2["desc"], 15.0, mode, True)
    method = "SearchByProjectionLast2Cam(mode %d)" % mode
    _same(cfg, method, nmatches=(nm, wnm), assign=(assign, wassign))
    nl = sc2["fl"].n
    _floor(cfg, method, "left matches", (wassign[:nl] >= 0).sum(), 100)
    _floor(cfg, method, "right matches", (wassign[nl:] >= 0).sum(), 100)


# ---- SearchForInitialization, SearchByBoW(KeyFrame, Frame) ---------------------------------------------------------------

@pytest.mark.parametrize("window", [10, 60])
@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_for_initialization(oracle, scenes, cfg, window):
    S = scenes(cfg)
    f1, f2 = S.frame("a"), S.frame("b")
    m = _matcher(0.9, True)
    prev_g = np.stack([S.ka["x"], S.ka["y"]], 1).astype(np.float32).copy()
    prev_w = prev_g.copy()
    nm, m12 = m.SearchForInitialization(f1, m.frame(f2), prev_g, window)
    wnm, wm12 = oracle.search_for_initialization(f1.view, f2.view, prev_w, window, float(np.float32(0.9)), True)
    method = "SearchForInitialization(window %d)" % window
    _same(cfg, method, nmatches=(nm, wnm), matches12=(m12, wm12), prev_matched=(prev_g, prev_w))
    _floor(cfg, method, "nmatches", wnm, 30)


@pytest.mark.parametrize("two_cameras", [False, True])
@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_by_bow(oracle, scenes, cfg, two_cameras):
    S = scenes(cfg)
    kf = S.frame("b")
    if two_cameras:
        keys, desc = np.concatenate([S.ka, S.kb]), np.concatenate([S.da, S.db])
        f = sc.frame_data(keys, desc, size=S.size, bounds=S.bounds, scale_factors=S.scale_factors)
        nleft = len(S.ka)
    else:
        f, nleft = S.frame("a"), -1
    valid = (np.random.default_rng(6).random(kf.n) < 0.85).astype(np.uint8)
    kfv, ffv = sc.feature_vector(S.db, 24), sc.feature_vector(f.descriptors, 24)
    m = _matcher(0.7, True)
    nm, mf = m.SearchByBoW(kf, valid, f, kfv, ffv, f_nleft=nleft)
    wnm, wmf = oracle.search_by_bow(kf.view, valid, f.view, kfv, ffv, float(np.float32(0.7)), True, nleft)
    method = "SearchByBoW(%s)" % ("two cameras" if two_cameras else "one camera")
    _same(cfg, method, nmatches=(nm, wnm), matches=(mf, wmf))
    _floor(cfg, method, "nmatches", wnm, 20)
    if two_cameras:
        _floor(cfg, method, "right-camera matches", (wmf[nleft:] >= 0).sum(), 20)


# ---- keyframe-side methods -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_by_projection_reloc(oracle, scenes, cfg):
    S = scenes(cfg)
    fd = S.frame()
    pts = sc.search_points(S.kb, SHIFT, 3, size=S.size, nlevels=S.nlevels)
    occ = (np.random.default_rng(4).random(fd.n) < 0.1).astype(np.uint8)
    m = _matcher(0.9, True)
    nm, assign = m.SearchByProjectionReloc(m.frame(fd), occ, pts, S.db, 10.0, 100)
    wnm, wassign = oracle.search_by_projection_reloc(fd.view, occ, pts, S.db, 10.0, 100, True)
    _same(cfg, "SearchByProjectionReloc", nmatches=(nm, wnm), assign=(assign, wassign))
    _floor(cfg, "SearchByProjectionReloc", "nmatches", wnm, 100)


@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_by_projection_sim3(oracle, scenes, cfg):
    S = scenes(cfg)
    fd = S.frame()
    pts = sc.search_points(S.kb, SHIFT, 5, size=S.size, nlevels=S.nlevels)
    matched = (np.random.default_rng(6).random(fd.n) < 0.2).astype(np.uint8)
    m = _matcher()
    nm, assign = m.SearchByProjectionSim3(m.frame(fd), matched, pts, S.db, 8, 1.0)
    wnm, wassign = oracle.search_by_projection_sim3(fd.view, matched, pts, S.db, 8, float(np.float32(1.0)))
    _same(cfg, "SearchByProjectionSim3", nmatches=(nm, wnm), assign=(assign, wassign))
    _floor(cfg, "SearchByProjectionSim3", "nmatches", wnm, 50)


@pytest.mark.parametrize("variant,stereo", [(0, False), (0, True), (1, False)])
@pytest.mark.parametrize("cfg", CFG_IDS)
def test_fuse_search(oracle, scenes, cfg, variant, stereo):
    S = scenes(cfg)
    fd = S.frame(stereo_seed=8 if stereo else None)
    pts = sc.search_points(S.kb, SHIFT, 7, sigma=1.5, size=S.size, nlevels=S.nlevels)
    if stereo:
        pts["ur"] = pts["u"] - 12.0
    m = _matcher()
    nf, best = m.FuseSearch(m.frame(fd), pts, S.db, 3.0, S.inv_sigma2, sim3_variant=bool(variant))
    wnf, wbest = oracle.fuse_search(fd.view, pts, S.db, 3.0, S.inv_sigma2, variant)
    method = "FuseSearch(variant %d%s)" % (variant, ", stereo" if stereo else "")
    _same(cfg, method, nfused=(nf, wnf), best=(best, wbest))
    _floor(cfg, method, "nfused", wnf, 20 if variant == 0 else 100)


@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_by_sim3(oracle, scenes, cfg):
    S = scenes(cfg)
    f1, f2 = S.frame("a"), S.frame("b")
    pts1 = sc.search_points(S.ka, (-SHIFT[0], -SHIFT[1]), 9, size=S.size, nlevels=S.nlevels)
    pts2 = sc.search_points(S.kb, SHIFT, 10, size=S.size, nlevels=S.nlevels)
    m = _matcher()
    nf, m12 = m.SearchBySim3(m.frame(f1), m.frame(f2), pts1, S.da, pts2, S.db, 7.5)
    wnf, wm12 = oracle.search_by_sim3(f1.view, f2.view, pts1, S.da, pts2, S.db, 7.5)
    _same(cfg, "SearchBySim3", nfound=(nf, wnf), matches12=(m12, wm12))
    _floor(cfg, "SearchBySim3", "nfound", wnf, 100)


@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_by_bow_kf(oracle, scenes, cfg):
    S = scenes(cfg)
    k1, k2 = S.frame("a"), S.frame("b")
    rng = np.random.default_rng(12)
    v1 = (rng.random(k1.n) < 0.85).astype(np.uint8)
    v2 = (rng.random(k2.n) < 0.85).astype(np.uint8)
    fv1, fv2 = sc.feature_vector(S.da, 24), sc.feature_vector(S.db, 24)
    m = _matcher(0.8, True)
    nm, m12 = m.SearchByBoWKF(k1, v1, k2, v2, fv1, fv2)
    wnm, wm12 = oracle.search_by_bow_kf(k1.view, v1, k2.view, v2, fv1, fv2, float(np.float32(0.8)), True)
    _same(cfg, "SearchByBoWKF", nmatches=(nm, wnm), matches12=(m12, wm12))
    _floor(cfg, "SearchByBoWKF", "nmatches", wnm, 20)


@pytest.mark.parametrize("only_stereo,coarse", [(False, False), (True, False), (False, True)])
@pytest.mark.parametrize("cfg", CFG_IDS)
def test_search_for_triangulation(oracle, scenes, cfg, only_stereo, coarse):
    S = scenes(cfg)
    k1 = sc.frame_data(S.ka, S.da, size=S.size, stereo_seed=2, bounds=S.bounds, scale_factors=S.scale_factors)
    k2 = sc.frame_data(S.kb, S.db, size=S.size, stereo_seed=3, bounds=S.bounds, scale_factors=S.scale_factors)
    rng = np.random.default_rng(13)
    h1 = (rng.random(k1.n) < 0.3).astype(np.uint8)
    h2 = (rng.random(k2.n) < 0.3).astype(np.uint8)
    fv1, fv2 = sc.feature_vector(S.da, 24), sc.feature_vector(S.db, 24)
    f12 = sc.translation_f12(SHIFT)
    ep = np.array([0.47 * S.size[0], 0.42 * S.size[1]], np.float32)
    m = _matcher(0.6, True)
    nm, m12 = m.SearchForTriangulation(k1, h1, k2, h2, fv1, fv2, f12, ep, S.sigma2, only_stereo, coarse)
    wnm, wm12 = oracle.search_for_triangulation(k1.view, h1, k2.view, h2, fv1, fv2, only_stereo, coarse, f12, ep, S.sigma2, True)
    method = "SearchForTriangulation(only_stereo %s, coarse %s)" % (only_stereo, coarse)
    _same(cfg, method, nmatches=(nm, wnm), matches12=(m12, wm12))
    _floor(cfg, method, "nmatches", wnm, 10)


# ---- size-dependent paths ------------------------------------------------------------------------------------------------

def _large_map(S, reps, seed):
    """The frame B keypoints replicated `reps` times with noisy descriptors: a map much larger than the frame."""
    rng = np.random.default_rng(seed)
    kb2, db2 = np.concatenate([S.kb] * reps), np.concatenate([S.db] * reps)
    flip = rng.integers(0, 256, db2.shape, dtype=np.uint8) & rng.integers(0, 256, db2.shape, dtype=np.uint8) & \
        rng.integers(0, 256, db2.shape, dtype=np.uint8)
    return sc.track_points(S.frame(), kb2, db2 ^ flip, SHIFT, 33, nlevels=S.nlevels)


def _with_searched(pts, n):
    """A copy of the map in which exactly the first n of the points that reach GetFeaturesInArea still do."""
    pts = pts.copy()
    q = np.nonzero(_qualifying(pts))[0]
    assert len(q) >= n
    pts["in_view"][q[n:]] = 0
    assert _qualifying(pts).sum() == n
    return pts


def test_projection_map_replay_switch(oracle, scenes):
    """kOrderedReplayMinQueries - 1 queries take the per-query replay (one launch), kOrderedReplayMinQueries the
    device-ordered lists (three launches); both must equal the oracle."""
    S = scenes("default")
    fd = S.frame()
    pts, desc, occ = _large_map(S, 25, 2)
    m = _matcher(0.8)
    fr = m.frame(fd)
    for n, path, launches in ((ORDERED_REPLAY_MIN_QUERIES - 1, "raw", RAW_LAUNCHES),
                              (ORDERED_REPLAY_MIN_QUERIES, "ordered", ORDERED_LAUNCHES)):
        p = _with_searched(pts, n)
        before = _launches()
        nm, assign = m.SearchByProjectionMap(fr, occ, p, desc, 3.0)
        ran = _launches() - before
        method = "SearchByProjectionMap(%d queries)" % n
        assert ran == launches, "default / %s: %d kernel launches, the %s path makes %d" % (method, ran, path, launches)
        wnm, wassign = oracle.search_by_projection_map(fd.view, occ, p, desc, 3.0, False, 50.0, float(np.float32(0.8)))
        _same("default", method, nmatches=(nm, wnm), assign=(assign, wassign))
        _floor("default", method, "nmatches", wnm, 300)


def _area_search_direct(m, fr, q):
    """vsg_area_search with an output capacity that always suffices: exactly one call of the device search."""
    from visual_sgraphs_b200._lib import check, load, ptr
    qx, qy, qr, lo, hi, qdesc = q
    nq = len(qx)
    cap = nq * fr.data.n
    cand_ptr = np.zeros(nq + 1, np.int32)
    idx, dist, total = np.zeros(cap, np.int32), np.zeros(cap, np.int32), C.c_int(0)
    check(load().vsg_area_search(m._h, fr._h, nq, ptr(qx), ptr(qy), ptr(qr), ptr(lo), ptr(hi), ptr(qdesc), ptr(cand_ptr), ptr(idx),
                                 ptr(dist), cap, C.byref(total)))
    return cand_ptr, idx[:total.value], dist[:total.value]


def test_area_search_overflow_retry(oracle, scenes):
    """A fresh matcher's first buffer holds 32 candidates per query: windows over most of the frame overflow it and the
    search runs again with the exact size.  Later calls reuse the grown buffer, and a larger one grows it again."""
    S = scenes("default")
    fd = S.frame()
    rng = np.random.default_rng(17)

    def queries(nq, big):
        if big:
            qx = rng.uniform(250, 390, nq).astype(np.float32)
            qy = rng.uniform(190, 290, nq).astype(np.float32)
            qr = rng.uniform(250, 330, nq).astype(np.float32)
        else:
            qx = rng.uniform(0, 640, nq).astype(np.float32)
            qy = rng.uniform(0, 480, nq).astype(np.float32)
            qr = rng.uniform(2, 15, nq).astype(np.float32)
        lo, hi = np.full(nq, -1, np.int32), np.full(nq, -1, np.int32)
        return qx, qy, qr, lo, hi, S.db[rng.integers(0, len(S.db), nq)]

    m = _matcher()
    fr = m.frame(fd)
    # (queries, windows over most of the frame, launches): first call overflows; small call and a call that fits the grown
    # buffer run once; a call three times larger than the first overflows the grown buffer
    for step, (nq, big, launches) in enumerate(((6, True, 2), (300, False, 1), (6, True, 1), (20, True, 2), (300, False, 1))):
        q = queries(nq, big)
        before = _launches()
        ptr_, idx, dist = _area_search_direct(m, fr, q)
        ran = _launches() - before
        method = "area_search call %d (%d queries%s)" % (step, nq, ", most of the frame" if big else "")
        total = _check_area_lists("default", method, oracle, fd, q, ptr_, idx, dist)
        if big and launches == 2:
            _floor("default", method, "candidates per query", total // nq, 32)
        assert ran == launches, "default / %s: %d launches of area_search_kernel, expected %d" % (method, ran, launches)


def test_ordered_lists_overflow_retry(oracle, scenes):
    """The device-ordered path's first buffer holds 4 candidates per query: wide windows over a 20 000-point map overflow it
    (area search twice, then the two ordering kernels).  A small call in between and the same large call again reuse it."""
    S = scenes("default")
    fd = S.frame()
    pts, desc, occ = _large_map(S, 25, 5)
    big = _with_searched(pts, ORDERED_REPLAY_MIN_QUERIES + 500)
    small, sdesc, socc = sc.track_points(fd, S.kb, S.db, SHIFT, 21)
    m = _matcher(0.6)
    fr = m.frame(fd)
    for step, (p, d, th, launches) in enumerate(((big, desc, 15.0, 2 + 2), (small, sdesc, 3.0, RAW_LAUNCHES),
                                                 (big, desc, 15.0, ORDERED_LAUNCHES))):
        before = _launches()
        nm, assign = m.SearchByProjectionMap(fr, occ if p is big else socc, p, d, th)
        ran = _launches() - before
        wnm, wassign = oracle.search_by_projection_map(fd.view, occ if p is big else socc, p, d, th, False, 50.0,
                                                       float(np.float32(0.6)))
        method = "SearchByProjectionMap call %d (%d queries, th %g)" % (step, _qualifying(p).sum(), th)
        _same("default", method, nmatches=(nm, wnm), assign=(assign, wassign))
        _floor("default", method, "nmatches", wnm, 100)
        assert ran == launches, "default / %s: %d kernel launches, expected %d" % (method, ran, launches)


# ---- kNN-2: the automatic choice between the tensor-core and the POPC kernel ----------------------------------------------

def _knn_brute(q, t, rows):
    """(idx, dist) top-2 by (distance, index) of the given query rows, one row at a time over the whole train set."""
    t64 = t.view(np.uint64)
    ar = np.arange(len(t), dtype=np.int64)
    idx, dist = np.zeros((len(rows), 2), np.int64), np.zeros((len(rows), 2), np.int64)
    for k, r in enumerate(rows):
        d = np.bitwise_count(t64 ^ q[r].view(np.uint64)[None, :]).sum(1, dtype=np.int64)
        key = d * (1 << 32) + ar
        top = np.argpartition(key, 1)[:2]
        top = top[np.argsort(key[top])]
        idx[k], dist[k] = top, d[top]
    return idx, dist


@pytest.mark.parametrize("nq,nt,tc", [(255, 2**20 + 3, False), (256, 2**20 - 1, False), (256, 2**20, True),
                                      (65536, 4095, False), (65536, 4096, True), (2**17, 4095, False)])
def test_knn2_automatic_kernel_choice(monkeypatch, nq, nt, tc):
    """With VSG_KNN_TC unset the tensor-core kernel runs when nq * nt >= 2^28, nq >= 256 and nt >= 4096.  Exact duplicate
    train rows at 256 k - 1 and 256 k (the POPC kernel's chunks and the tensor-core segments are multiples of 256 rows)
    are the two nearest rows of some query: the lower index must come first, at distance 0 both."""
    monkeypatch.delenv("VSG_KNN_TC", raising=False)
    rng = np.random.default_rng(nq + nt)
    q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    ks = np.arange(1, (nt - 1) // 256 + 1)
    t[256 * ks] = t[256 * ks - 1]
    planted = min(nq - 64, len(ks))
    pk = ks[np.linspace(0, len(ks) - 1, planted).round().astype(int)]
    prow = rng.choice(nq, planted, replace=False)
    q[prow] = t[256 * pk - 1]
    m = _matcher()
    before = _launches()
    idx, dist = m.knn2(q, t)
    ran = _launches() - before
    shape = "knn2(%d x %d)" % (nq, nt)
    want = KNN_TC_LAUNCHES if tc else KNN_POPC_LAUNCHES
    assert ran == want, "%s: %d launches; the %s path makes %d" % (shape, ran, "tensor-core" if tc else "POPC", want)
    _same(shape, "planted ties", idx=(idx[prow], np.stack([256 * pk - 1, 256 * pk], 1)), dist=(dist[prow], np.zeros((planted, 2))))
    sample = np.concatenate([rng.choice(nq, 64, replace=False), prow[:8]])
    widx, wdist = _knn_brute(q, t, sample)
    _same(shape, "numpy brute force", idx=(idx[sample], widx), dist=(dist[sample], wdist))
    monkeypatch.setenv("VSG_KNN_TC", "0")
    idx0, dist0 = m.knn2(q, t)
    _same(shape, "VSG_KNN_TC=0", idx=(idx, idx0), dist=(dist, dist0))
