"""GPU parity tests for the keyframe-side matcher methods (relocalisation / Sim3 projections, Fuse, SearchBySim3,
SearchByBoW(KF, KF), SearchForTriangulation) behind the C ABI against the CPU oracle's restatement of the
reference loops.  Bit-exact: indices and counts must be identical."""
import numpy as np
import pytest

from tests import match_scenarios as sc

pytestmark = pytest.mark.gpu


def _matcher(nnratio=0.6, check_ori=True):
    from visual_sgraphs_b200.matcher import ORBmatcher
    return ORBmatcher(nnratio, check_ori)


@pytest.mark.parametrize("check_ori", [True, False])
@pytest.mark.parametrize("th,orb_dist", [(10.0, 100), (15.0, 64)])
def test_search_by_projection_reloc(oracle, check_ori, th, orb_dist):
    ka, da, kb, db = sc.two_frames(oracle)
    fd = sc.frame_data(ka, da)
    pts = sc.search_points(kb, (9, 5), 3)
    occ = (np.random.default_rng(4).random(fd.n) < 0.1).astype(np.uint8)
    m = _matcher(0.9, check_ori)
    nm, assign = m.SearchByProjectionReloc(m.frame(fd), occ, pts, db, th, orb_dist)
    wnm, wassign = oracle.search_by_projection_reloc(fd.view, occ, pts, db, th, orb_dist, check_ori)
    assert nm == wnm and np.array_equal(assign, wassign)
    assert nm > 100


@pytest.mark.parametrize("th,ratio", [(8, 1.0), (4, 1.5), (12, 0.8)])
def test_search_by_projection_sim3(oracle, th, ratio):
    ka, da, kb, db = sc.two_frames(oracle)
    fd = sc.frame_data(ka, da)
    pts = sc.search_points(kb, (9, 5), 5)
    matched = (np.random.default_rng(6).random(fd.n) < 0.2).astype(np.uint8)
    m = _matcher()
    nm, assign = m.SearchByProjectionSim3(m.frame(fd), matched, pts, db, th, ratio)
    wnm, wassign = oracle.search_by_projection_sim3(fd.view, matched, pts, db, th, float(np.float32(ratio)))
    assert nm == wnm and np.array_equal(assign, wassign)
    assert nm > 50


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("stereo", [False, True])
def test_fuse_search(oracle, variant, stereo):
    ka, da, kb, db = sc.two_frames(oracle)
    fd = sc.frame_data(ka, da, stereo_seed=8 if stereo else None)
    pts = sc.search_points(kb, (9, 5), 7, sigma=1.5)
    if stereo:   # make the right coordinate agree with the keyframe's for a share of the points
        pts["ur"] = pts["u"] - 12.0
    _, _, inv_sigma2 = sc.sigma_tables()
    m = _matcher()
    nf, best = m.FuseSearch(m.frame(fd), pts, db, 3.0, inv_sigma2, sim3_variant=bool(variant))
    wnf, wbest = oracle.fuse_search(fd.view, pts, db, 3.0, inv_sigma2, variant)
    assert nf == wnf and np.array_equal(best, wbest)
    assert nf > (20 if variant == 0 else 100)


def test_search_by_sim3(oracle):
    ka, da, kb, db = sc.two_frames(oracle)
    f1, f2 = sc.frame_data(ka, da), sc.frame_data(kb, db)
    pts1 = sc.search_points(ka, (-9, -5), 9)       # KF1's points projected into KF2
    pts2 = sc.search_points(kb, (9, 5), 10)        # KF2's points projected into KF1
    m = _matcher()
    nf, m12 = m.SearchBySim3(m.frame(f1), m.frame(f2), pts1, da, pts2, db, 7.5)
    wnf, wm12 = oracle.search_by_sim3(f1.view, f2.view, pts1, da, pts2, db, 7.5)
    assert nf == wnf and np.array_equal(m12, wm12)
    assert nf > 100


def _tie_scene():
    """A query at (320, 240) with radius 30 walks 7 x 7 grid cells (64 x 48 cells on 640 x 480), 32 per warp round.  The
    keyframe has two keypoints with the query's own descriptor: keypoint 0 in cell (29, 21), the first of round 0, and
    keypoint 1 in cell (35, 27), the 49th, in round 1; keypoint 2 is farther.  The reference's strict '<' keeps keypoint 0."""
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE, SEARCH_POINT_DTYPE

    def keys(xy):
        k = np.zeros(len(xy), KEYPOINT_DTYPE)
        k["x"], k["y"] = np.array(xy, np.float32).T
        k["size"] = 31
        return k

    d = np.random.default_rng(3).integers(0, 256, 32, dtype=np.uint8)
    kf = sc.frame_data(keys([(292, 212), (348, 268), (330, 250)]), np.stack([d, d, d ^ 0xFF]))
    q = np.zeros(1, SEARCH_POINT_DTYPE)
    q["u"], q["v"], q["valid"] = 320, 240, 1
    return kf, q, d[None].copy(), keys


@pytest.mark.parametrize("variant", [0, 1])
def test_fuse_search_tie_across_rounds(oracle, variant):
    kf, q, d, _ = _tie_scene()
    inv_sigma2 = np.full(8, 1e-4, np.float32)              # chi-square gates wide enough for the 28-px offsets
    m = _matcher()
    nf, best = m.FuseSearch(m.frame(kf), q, d, 30.0, inv_sigma2, sim3_variant=bool(variant))
    wnf, wbest = oracle.fuse_search(kf.view, q, d, 30.0, inv_sigma2, variant)
    assert nf == wnf == 1 and np.array_equal(best, wbest) and best[0] == 0


def test_search_by_sim3_tie_across_rounds(oracle):
    kf2, q, d, keys = _tie_scene()
    kf1 = sc.frame_data(keys([(100, 100)]), d)                # its one point projects onto the window; KF2's keypoint 0
    p2 = np.zeros(kf2.n, q.dtype)                             # projects back onto it
    p2[0]["u"], p2[0]["v"], p2[0]["valid"] = 100, 100, 1
    d2 = np.ascontiguousarray(kf2.descriptors)
    m = _matcher()
    nf, m12 = m.SearchBySim3(m.frame(kf1), m.frame(kf2), q, d, p2, d2, 30.0)
    wnf, wm12 = oracle.search_by_sim3(kf1.view, kf2.view, q, d, p2, d2, 30.0)
    assert nf == wnf == 1 and np.array_equal(m12, wm12) and m12[0] == 0


@pytest.mark.parametrize("check_ori", [True, False])
def test_search_by_bow_kf(oracle, check_ori):
    ka, da, kb, db = sc.two_frames(oracle, shift=(3, 2))
    k1, k2 = sc.frame_data(ka, da), sc.frame_data(kb, db)
    rng = np.random.default_rng(12)
    v1 = (rng.random(k1.n) < 0.85).astype(np.uint8)
    v2 = (rng.random(k2.n) < 0.85).astype(np.uint8)
    fv1, fv2 = sc.feature_vector(da, 24), sc.feature_vector(db, 24)
    m = _matcher(0.8, check_ori)
    nm, m12 = m.SearchByBoWKF(k1, v1, k2, v2, fv1, fv2)
    wnm, wm12 = oracle.search_by_bow_kf(k1.view, v1, k2.view, v2, fv1, fv2, float(np.float32(0.8)), check_ori)
    assert nm == wnm and np.array_equal(m12, wm12)
    assert nm > 20


@pytest.mark.parametrize("only_stereo,coarse", [(False, False), (True, False), (False, True)])
def test_search_for_triangulation(oracle, only_stereo, coarse):
    shift = (9, 1)
    ka, da, kb, db = sc.two_frames(oracle, shift=shift)
    k1, k2 = sc.frame_data(ka, da, stereo_seed=2), sc.frame_data(kb, db, stereo_seed=3)
    rng = np.random.default_rng(13)
    h1 = (rng.random(k1.n) < 0.3).astype(np.uint8)
    h2 = (rng.random(k2.n) < 0.3).astype(np.uint8)
    fv1, fv2 = sc.feature_vector(da, 24), sc.feature_vector(db, 24)
    _, sigma2, _ = sc.sigma_tables()
    f12, ep = sc.translation_f12(shift), np.array([300.0, 200.0], np.float32)
    m = _matcher(0.6, True)
    nm, m12 = m.SearchForTriangulation(k1, h1, k2, h2, fv1, fv2, f12, ep, sigma2, only_stereo, coarse)
    wnm, wm12 = oracle.search_for_triangulation(k1.view, h1, k2.view, h2, fv1, fv2, only_stereo, coarse, f12, ep, sigma2, True)
    assert nm == wnm and np.array_equal(m12, wm12)
    assert nm > 10


def test_kf_methods_empty_inputs(oracle):
    from visual_sgraphs_b200._lib import SEARCH_POINT_DTYPE
    ka, da, kb, db = sc.two_frames(oracle)
    fd = sc.frame_data(ka, da)
    m = _matcher()
    fr = m.frame(fd)
    none = np.zeros(0, SEARCH_POINT_DTYPE)
    nd = np.zeros((0, 32), np.uint8)
    nm, assign = m.SearchByProjectionReloc(fr, np.zeros(fd.n, np.uint8), none, nd, 10.0, 100)
    assert nm == 0 and (assign == -1).all()
    nm, assign = m.SearchByProjectionSim3(fr, np.zeros(fd.n, np.uint8), none, nd, 8, 1.0)
    assert nm == 0 and (assign == -1).all()
    nf, best = m.FuseSearch(fr, none, nd, 3.0, sc.sigma_tables()[2])
    assert nf == 0 and len(best) == 0
