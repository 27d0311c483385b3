"""vsg_search_by_bow_multi / vsg_search_by_bow_kf_multi (ORBmatcher.SearchByBoWMulti / SearchByBoWKFMulti) and the
multi-target shim SearchByBoW overloads, on the B200 (-m gpu).

One call matches a frame (relocalisation) or a keyframe (loop detection) against many keyframes by BoW.  For every target
t, the matches and the count must equal the single-target call on target t and the CPU oracle's search_by_bow /
search_by_bow_kf.  The targets differ in what the walk and the replay read: keypoint count (including none), a feature
vector that shares no node with the other side, all map-point flags zero, pyramid, two-camera keyframes, and the same
keyframe twice.  tests/cpp/bow_multi_test.cpp checks the shim's overloads against the loops of single-target calls.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import match_scenarios as sc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NODES = 24
# scene id: (size, nfeatures, scale factor, levels)
SCENES = {
    "default": ((640, 480), 1000, 1.2, 8),
    "fine": ((640, 480), 1000, 1.1, 12),
    "coarse": ((752, 480), 1200, 1.5, 5),
}
# target kinds: (scene, keypoints "all" / "half" / "none", map-point flags "most" / "zero", feature vector "same" / "disjoint",
# two cameras)
KINDS = [
    ("default", "all", "most", "same", False),
    ("fine", "all", "most", "same", False),
    ("coarse", "half", "most", "same", False),
    ("default", "none", "most", "same", False),
    ("default", "all", "zero", "same", False),
    ("default", "all", "most", "disjoint", False),
    ("default", "all", "most", "same", True),
    ("default", "half", "most", "same", True),
]
F32 = lambda v: float(np.float32(v))  # noqa: E731


def _matcher(nnratio, check_ori, device=0):
    from visual_sgraphs_b200.matcher import ORBmatcher
    return ORBmatcher(nnratio, check_ori, device=device)


def _launches():
    from visual_sgraphs_b200 import _lib
    return _lib.load().vsg_launch_count()


@pytest.fixture(scope="module")
def scenes(oracle):
    out = {}
    for sid, (size, nfeat, scale, nlevels) in SCENES.items():
        ka, da, kb, db = sc.two_frames(oracle, shift=(3, 2), size=size, nfeat=nfeat, scale=scale, nlevels=nlevels)
        out[sid] = (ka, da, kb, db, size, sc.scale_factors(oracle, scale, nlevels))
    return out


def _featvec(desc, disjoint=False, limit=None):
    nodes, ptr, idx = sc.feature_vector(desc, NODES)
    if limit is not None:                       # two-camera keyframe in the KF-KF form: entries past mvKeysUn dropped
        keep = [idx[ptr[k]:ptr[k + 1]] for k in range(len(nodes))]
        keep = [v[v < limit] for v in keep]
        ptr = np.concatenate([[0], np.cumsum([len(v) for v in keep])]).astype(np.int32)
        idx = np.concatenate(keep + [np.zeros(0, np.int32)]).astype(np.int32)
    if disjoint:
        nodes = nodes + 1000                    # no node in common with the other side
    return nodes.astype(np.int32), ptr, idx


def make_target(scenes, t, seed, kf_kf):
    """Target t: (FrameData, map-point flags, feature vector) as the form's single-target call takes them."""
    sid, keep, flags, fv, two = KINDS[t % len(KINDS)]
    ka, da, kb, db, size, scale = scenes[sid]
    rng = np.random.default_rng(seed)
    keys, desc = kb, db
    if keep == "half":
        pick = np.sort(rng.permutation(len(keys))[: len(keys) // 2])
        keys, desc = keys[pick], desc[pick]
    elif keep == "none":
        keys, desc = keys[:0], desc[:0]
    nleft = len(keys)
    limit = None
    if two:                                     # the second camera's features follow the first's
        keys, desc = np.concatenate([keys, ka[::3]]), np.concatenate([desc, da[::3]])
        if kf_kf:                               # KF-KF: the keyframe is its mvKeysUn (the first camera)
            limit = nleft
    featvec = _featvec(desc, fv == "disjoint", limit)
    if limit is not None:
        keys, desc = keys[:nleft], desc[:nleft]
    fd = sc.frame_data(keys, desc, size=size, scale_factors=scale)
    valid = (rng.random(fd.n) < 0.85).astype(np.uint8) if flags == "most" else np.zeros(fd.n, np.uint8)
    return fd, valid, featvec


def _targets(scenes, ntargets, kf_kf, seed0=300):
    targets = [make_target(scenes, t, seed0 + t, kf_kf) for t in range(ntargets)]
    if ntargets > 1:
        targets[-1] = targets[0]                # the same keyframe twice
    return targets


def _has_pairs(fv_a, valid_a, fv_b):
    """Does the merge walk find any (query, candidate) pair: a usable side-a feature in a node side b also lists?"""
    na, pa, ia = fv_a
    nb, pb, ib = fv_b
    for k, node in enumerate(na):
        j = np.searchsorted(nb, node)
        if j < len(nb) and nb[j] == node and pb[j + 1] > pb[j] and valid_a[ia[pa[k]:pa[k + 1]]].any():
            return True
    return False


def _frame(scenes, two_camera):
    ka, da, kb, db, size, scale = scenes["default"]
    if two_camera:
        keys, desc = np.concatenate([ka, kb[::2]]), np.concatenate([da, db[::2]])
        return sc.frame_data(keys, desc, size=size, scale_factors=scale), _featvec(desc), len(ka)
    return sc.frame_data(ka, da, size=size, scale_factors=scale), _featvec(da), -1


def _check(what, got_nm, got, singles, wants):
    for t, ((snm, sm), (wnm, wm)) in enumerate(zip(singles, wants)):
        for name, nm, m in (("the single-target call", snm, sm), ("the oracle", wnm, wm)):
            bad = np.nonzero(got[t] != m)[0]
            assert not len(bad), "%s: target %d (%s), slot %d: multi %d, %s %d (%d differences)" % (
                what, t, KINDS[t % len(KINDS)], bad[0], got[t][bad[0]], name, m[bad[0]], len(bad))
            assert got_nm[t] == nm, "%s: target %d (%s): %d matches, %s %d" % (what, t, KINDS[t % len(KINDS)], got_nm[t], name, nm)


def _floors(nm):
    """Targets without queries find nothing; the default scene's full keyframes (the searched image, shifted) find plenty."""
    for t in range(len(nm)):
        sid, keep, flags, fvk, _ = KINDS[t % len(KINDS)]
        if keep == "none" or flags == "zero" or fvk == "disjoint":
            assert nm[t] == 0
        elif keep == "all" and sid == "default":
            assert nm[t] > 20, "target %d (%s): %d matches" % (t, KINDS[t % len(KINDS)], nm[t])


RATIOS = [(0.75, True), (0.9, False), (0.9, True)]


@pytest.mark.parametrize("ntargets", [0, 1, 33])
@pytest.mark.parametrize("two_camera_frame", [False, True])
@pytest.mark.parametrize("nnratio,check_ori", RATIOS[:2])
def test_search_by_bow_multi(oracle, scenes, ntargets, two_camera_frame, nnratio, check_ori):
    f, ffv, nleft = _frame(scenes, two_camera_frame)
    targets = _targets(scenes, ntargets, False)
    m = _matcher(nnratio, check_ori)
    before = _launches()
    nm, got = m.SearchByBoWMulti(targets, f, ffv, f_nleft=nleft)
    launches = _launches() - before
    assert got.shape == (ntargets, f.n) and nm.shape == (ntargets,)
    singles = [m.SearchByBoW(kf, v, f, fv, ffv, f_nleft=nleft) for kf, v, fv in targets]
    wants = [oracle.search_by_bow(kf.view, v, f.view, fv, ffv, F32(nnratio), check_ori, nleft) for kf, v, fv in targets]
    _check("SearchByBoWMulti, %d targets" % ntargets, nm, got, singles, wants)
    assert launches == int(any(_has_pairs(fv, v, ffv) for _, v, fv in targets))
    _floors(nm)


@pytest.mark.parametrize("ntargets", [0, 1, 33])
@pytest.mark.parametrize("nnratio,check_ori", RATIOS)
def test_search_by_bow_kf_multi(oracle, scenes, ntargets, nnratio, check_ori):
    ka, da, _, _, size, scale = scenes["default"]
    k1 = sc.frame_data(ka, da, size=size, scale_factors=scale)
    v1 = (np.random.default_rng(8).random(k1.n) < 0.85).astype(np.uint8)
    fv1 = _featvec(da)
    targets = _targets(scenes, ntargets, True)
    m = _matcher(nnratio, check_ori)
    before = _launches()
    nm, got = m.SearchByBoWKFMulti(k1, v1, fv1, targets)
    launches = _launches() - before
    assert got.shape == (ntargets, k1.n) and nm.shape == (ntargets,)
    singles = [m.SearchByBoWKF(k1, v1, k2, v2, fv1, fv2) for k2, v2, fv2 in targets]
    wants = [oracle.search_by_bow_kf(k1.view, v1, k2.view, v2, fv1, fv2, F32(nnratio), check_ori) for k2, v2, fv2 in targets]
    _check("SearchByBoWKFMulti, %d targets" % ntargets, nm, got, singles, wants)
    assert launches == int(any(_has_pairs(fv1, v1, fv2) for _, _, fv2 in targets))
    _floors(nm)


def test_no_launch_without_in_node_pairs(scenes):
    """Targets without keypoints, without usable map points or without a common node: results, and no launch."""
    f, ffv, _ = _frame(scenes, False)
    targets = [make_target(scenes, t, 40 + t, False) for t in (3, 4, 5)]
    m = _matcher(0.75, True)
    before = _launches()
    nm, got = m.SearchByBoWMulti(targets, f, ffv)
    assert _launches() == before and (nm == 0).all() and (got == -1).all()
    ka, da, _, _, size, scale = scenes["default"]
    k1 = sc.frame_data(ka, da, size=size, scale_factors=scale)
    nm, got = m.SearchByBoWKFMulti(k1, np.zeros(k1.n, np.uint8), _featvec(da), [make_target(scenes, 0, 1, True)] * 3)
    assert _launches() == before and (nm == 0).all() and (got == -1).all()


def test_rejects_invalid_calls(scenes):
    from visual_sgraphs_b200 import _lib
    from visual_sgraphs_b200.matcher import _bow_side, _side_table
    L = _lib.load()
    m = _matcher(0.75, True)
    f, ffv, _ = _frame(scenes, False)
    ka, da, _, _, size, scale = scenes["default"]
    k1 = sc.frame_data(ka, da, size=size, scale_factors=scale)
    v1 = np.ones(k1.n, np.uint8)
    targets = [make_target(scenes, t, 60 + t, False) for t in (0, 1, 2, 8)]    # all with keypoints
    keep = []
    F = _bow_side(f, None, ffv, keep)
    K1 = _bow_side(k1, v1, _featvec(da), keep)
    sides = [_bow_side(d, v, fv, keep) for d, v, fv in targets]
    out = np.zeros((4, max(f.n, k1.n)), np.int32)
    nm = np.zeros(4, np.int32)
    kf_f = lambda T, tab: L.vsg_search_by_bow_multi(m._h, T, tab, C.byref(F), -1, C.c_float(0.75), 1, _lib.ptr(out),  # noqa: E731
                                                    _lib.ptr(nm))
    kf_kf = lambda T, tab: L.vsg_search_by_bow_kf_multi(m._h, C.byref(K1), T, tab, C.c_float(0.75), 1, _lib.ptr(out),  # noqa: E731
                                                        _lib.ptr(nm))
    before = _launches()
    for call in (kf_f, kf_kf):
        assert call(-1, _side_table(sides)) == _lib.VSG_ERR_INVALID and b"-1 targets" in L.vsg_last_error()
        tab = _side_table(sides)
        tab[2] = None                                     # a null target
        assert call(4, tab) == _lib.VSG_ERR_INVALID and b"target 2" in L.vsg_last_error()
        bad_idx = np.full_like(targets[3][2][2], targets[3][0].n + 5)
        bad = _bow_side(targets[3][0], targets[3][1], (targets[3][2][0], targets[3][2][1], bad_idx), keep)
        assert call(4, _side_table(sides[:3] + [bad])) == _lib.VSG_ERR_INVALID
        assert b"target 3" in L.vsg_last_error() and b"out of range" in L.vsg_last_error()
        bad_ptr = targets[3][2][1].copy()                  # list offsets that decrease: lists outside the index array
        bad_ptr[1] = bad_ptr[-1] + 10
        bad = _bow_side(targets[3][0], targets[3][1], (targets[3][2][0], bad_ptr, targets[3][2][2]), keep)
        assert call(4, _side_table(sides[:3] + [bad])) == _lib.VSG_ERR_INVALID
        assert b"target 3" in L.vsg_last_error() and b"malformed feature vector" in L.vsg_last_error()
        assert call(0, None) == _lib.VSG_OK
    assert _launches() == before                          # nothing was launched
    nm_ok, got = m.SearchByBoWMulti(targets, f, ffv)      # the matcher still works after rejected calls
    for t, (kf, v, fv) in enumerate(targets):
        snm, sm = m.SearchByBoW(kf, v, f, fv, ffv)
        assert nm_ok[t] == snm and np.array_equal(got[t], sm)
    if L.vsg_device_count() > 1:                          # a matcher of another device gives the same results
        m1 = _matcher(0.75, True, device=1)
        nm1, got1 = m1.SearchByBoWMulti(targets, f, ffv)
        assert np.array_equal(nm1, nm_ok) and np.array_equal(got1, got)
        nm1, got1 = m1.SearchByBoWKFMulti(k1, v1, _featvec(da), targets)
        nm0, got0 = m.SearchByBoWKFMulti(k1, v1, _featvec(da), targets)
        assert np.array_equal(nm1, nm0) and np.array_equal(got1, got0)


def test_cpp_multi_target_search_by_bow_equals_the_loop(tmp_path):
    pkg = os.path.join(ROOT, "visual_sgraphs_b200")
    exe = str(tmp_path / "bow_multi_test")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "bow_multi_test.cpp"),
                           "-L" + pkg, "-lvsg_cuda", "-Wl,-rpath," + pkg])
    out = subprocess.run([exe], capture_output=True, text=True)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "BOW MULTI TEST OK" in out.stdout
