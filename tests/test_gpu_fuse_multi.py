"""vsg_fuse_search_multi (ORBmatcher.fuse_search_multi) and the multi-target shim Fuse(vpTargetKFs, vpMapPoints, th), on the
B200 (-m gpu).

One call searches the same map points in many keyframes: the targets of LocalMapping::SearchInNeighbors' loop of Fuse
calls.  For every target t, best_idx[t] must equal vsg_fuse_search on target t alone and the CPU oracle's fuse_search,
index for index, with targets that differ in everything the search reads: keypoint count (including none), pyramid
(levels and scale factor), grid bounds, stereo or monocular, and the two cameras of a two-camera keyframe as two targets.
tests/cpp/fuse_multi_test.cpp then checks that the shim's multi-target Fuse leaves the same world as the loop of
single-target Fuse calls, including a map point whose descriptor a Replace changes between two targets.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import match_scenarios as sc
from visual_sgraphs_b200._lib import SEARCH_POINT_DTYPE

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIFT = (9, 5)
TH = 3.0
# scene id: (size, nfeatures, scale factor, levels, grid bounds or None for the image)
SCENES = {
    "default": ((640, 480), 1000, 1.2, 8, None),
    "fine": ((640, 480), 1000, 1.1, 12, None),
    "coarse": ((752, 480), 1200, 1.5, 5, (-13.7, -9.2, 711.4, 452.8)),
}


def _matcher():
    from visual_sgraphs_b200.matcher import ORBmatcher
    return ORBmatcher()


def _launches():
    from visual_sgraphs_b200 import _lib
    return _lib.load().vsg_launch_count()


class Scene:
    def __init__(self, oracle, sid):
        size, nfeat, scale, nlevels, bounds = SCENES[sid]
        self.size, self.nlevels, self.bounds = size, nlevels, bounds
        self.ka, self.da, self.kb, self.db = sc.two_frames(oracle, shift=SHIFT, size=size, nfeat=nfeat, scale=scale,
                                                           nlevels=nlevels)
        tables = oracle.OracleExtractor(nfeat, scale, nlevels).tables()
        self.scale_factors, self.inv_sigma2 = tables["scale"], tables["inv_sigma2"]


@pytest.fixture(scope="module")
def world(oracle):
    """The queries: the map points of every scene's frame B, back to back (desc shared by all targets)."""
    scenes = {sid: Scene(oracle, sid) for sid in SCENES}
    blocks, off = {}, 0
    for sid, S in scenes.items():
        blocks[sid] = (off, off + len(S.kb))
        off += len(S.kb)
    desc = np.concatenate([S.db for S in scenes.values()])
    return scenes, blocks, desc


# target kinds: (scene, keypoints kept: "all" / "half" / "none", stereo, bounds override, camera)
# camera "left" = frame A with the points of frame B projected by SHIFT; "right" = frame B of the same scene, the second
# camera of a two-camera keyframe, with the same points projected onto their own keypoints (no stereo gate).
KINDS = [
    ("default", "all", False, None, "left"),
    ("default", "all", False, None, "right"),
    ("fine", "all", True, None, "left"),
    ("coarse", "half", False, None, "left"),
    ("default", "none", True, None, "left"),
    ("default", "half", True, (-20.5, -11.0, 650.0, 470.5), "left"),
    ("coarse", "all", True, None, "left"),
    ("fine", "half", False, (3.0, 2.0, 630.0, 478.0), "left"),
]


def make_target(world, t, seed):
    """Target t: its FrameData, its level table and the queries projected into it ([n] search points)."""
    scenes, blocks, desc = world
    sid, keep, stereo, bounds, camera = KINDS[t % len(KINDS)]
    S = scenes[sid]
    rng = np.random.default_rng(seed)
    keys, kdesc = (S.ka, S.da) if camera == "left" else (S.kb, S.db)
    if keep == "half":
        pick = np.sort(rng.permutation(len(keys))[: len(keys) // 2])
        keys, kdesc = keys[pick], kdesc[pick]
    elif keep == "none":
        keys, kdesc = keys[:0], kdesc[:0]
    fd = sc.frame_data(keys, kdesc, size=S.size, stereo_seed=seed if stereo else None, bounds=bounds or S.bounds,
                       scale_factors=S.scale_factors)
    n = len(desc)
    pts = np.zeros(n, SEARCH_POINT_DTYPE)
    # points of other scenes: a few are searched at random places (nearly never a match), the rest are invalid here
    pts["u"] = rng.uniform(0, S.size[0], n)
    pts["v"] = rng.uniform(0, S.size[1], n)
    pts["ur"] = pts["u"] - 12.0
    pts["level"] = rng.integers(0, S.nlevels, n)
    pts["valid"] = rng.random(n) < 0.1
    b0, b1 = blocks[sid]
    own = sc.search_points(S.kb, SHIFT if camera == "left" else (0, 0), seed, sigma=1.5, size=S.size, nlevels=S.nlevels)
    if stereo:
        own["ur"] = own["u"] - 12.0
    pts[b0:b1] = own
    return fd, S.inv_sigma2, pts


def _compare(got, single, want, what):
    for t in range(len(want)):
        for name, other in (("vsg_fuse_search on the target alone", single[t]), ("the oracle", want[t])):
            bad = np.nonzero(got[t] != other)[0]
            if len(bad):
                i = int(bad[0])
                pytest.fail("%s: target %d (%s), query %d: fuse_search_multi picked keypoint %d, %s %d (%d differences)" %
                            (what, t, KINDS[t % len(KINDS)], i, got[t][i], name, other[i], len(bad)))


def _run(oracle, world, ntargets, seed0=100):
    _, _, desc = world
    targets = [make_target(world, t, seed0 + t) for t in range(ntargets)]
    m = _matcher()
    frames = [m.frame(fd) for fd, _, _ in targets]
    pts = np.stack([p for _, _, p in targets]) if targets else np.zeros((0, len(desc)), SEARCH_POINT_DTYPE)
    before = _launches()
    got = m.fuse_search_multi(frames, [s for _, s, _ in targets], pts, desc, TH)
    launches = _launches() - before
    single = [m.FuseSearch(f, p, desc, TH, s)[1] for f, (_, s, p) in zip(frames, targets)]
    want = [oracle.fuse_search(fd.view, p, desc, TH, s, 0)[1] for fd, s, p in targets]
    return got, single, want, launches


@pytest.mark.parametrize("ntargets", [0, 1, 2, 7, 31])
def test_fuse_search_multi_equals_single_target_searches(oracle, world, ntargets):
    got, single, want, launches = _run(oracle, world, ntargets)
    assert got.shape == (ntargets, len(world[2]))
    _compare(got, single, want, "%d targets" % ntargets)
    assert launches == (1 if ntargets else 0)
    for t in range(ntargets):                      # every target with keypoints finds something; the empty one nothing
        found = int((got[t] >= 0).sum())
        if KINDS[t % len(KINDS)][1] == "none":
            assert found == 0
        else:
            assert found > 20, "target %d (%s): %d points fused" % (t, KINDS[t % len(KINDS)], found)


def test_launches_do_not_grow_with_targets(oracle, world):
    n1 = _run(oracle, world, 1)[3]
    n31 = _run(oracle, world, 31)[3]
    assert n1 == n31 == 1


def test_no_points(world):
    m = _matcher()
    fd, s, _ = make_target(world, 0, 5)
    before = _launches()
    got = m.fuse_search_multi([m.frame(fd)] * 3, [s] * 3, np.zeros((3, 0), SEARCH_POINT_DTYPE), np.zeros((0, 32), np.uint8), TH)
    assert got.shape == (3, 0) and _launches() == before


def test_large_call(oracle):
    """20 000 points x 4 targets: the KITTI-sized scene's map points repeated with noise."""
    size, nfeat, scale, nlevels = (1241, 376), 2000, 1.2, 8
    ka, da, kb, db = sc.two_frames(oracle, shift=SHIFT, size=size, nfeat=nfeat, scale=scale, nlevels=nlevels)
    inv_sigma2 = oracle.OracleExtractor(nfeat, scale, nlevels).tables()["inv_sigma2"]
    reps = -(-20000 // len(kb))
    rng = np.random.default_rng(3)
    desc = np.concatenate([db ^ (rng.random(db.shape) < 0.02) * rng.integers(1, 256, db.shape, dtype=np.uint8)
                           for _ in range(reps)]).astype(np.uint8)
    n = len(desc)
    assert n >= 20000
    fds = [sc.frame_data(ka, da, size=size), sc.frame_data(ka, da, size=size, stereo_seed=4),
           sc.frame_data(ka[::2], da[::2], size=size), sc.frame_data(kb, db, size=size, stereo_seed=5)]
    pts = []
    for t in range(len(fds)):
        p = np.concatenate([sc.search_points(kb, SHIFT if t < 3 else (0, 0), 40 * t + r, sigma=1.5, size=size)
                            for r in range(reps)])
        p["ur"] = p["u"] - 12.0
        pts.append(p)
    m = _matcher()
    frames = [m.frame(fd) for fd in fds]
    got = m.fuse_search_multi(frames, [inv_sigma2] * len(fds), np.stack(pts), desc, TH)
    single = [m.FuseSearch(f, p, desc, TH, inv_sigma2)[1] for f, p in zip(frames, pts)]
    want = [oracle.fuse_search(fd.view, p, desc, TH, inv_sigma2, 0)[1] for fd, p in zip(fds, pts)]
    for t in range(len(fds)):
        for name, other in (("vsg_fuse_search on the target alone", single[t]), ("the oracle", want[t])):
            bad = np.nonzero(got[t] != other)[0]
            assert not len(bad), "large call: target %d, query %d: fuse_search_multi picked keypoint %d, %s %d" % (
                t, bad[0], got[t][bad[0]], name, other[bad[0]])
        assert (got[t] >= 0).sum() > 1000


def test_rejects_invalid_calls(world):
    from visual_sgraphs_b200 import _lib
    L = _lib.load()
    m = _matcher()
    fd, s, pts = make_target(world, 0, 7)
    desc = world[2]
    f = m.frame(fd)
    frames = (C.c_void_p * 1)(f._h.value)
    sig = (C.c_void_p * 1)(s.ctypes.data)
    best = np.zeros(len(desc), np.int32)
    call = lambda T, n, fr=frames, sg=sig, p=pts: L.vsg_fuse_search_multi(m._h, T, fr, sg, n, _lib.ptr(p), _lib.ptr(desc),
                                                                         C.c_float(TH), _lib.ptr(best))
    assert call(-1, len(desc)) == _lib.VSG_ERR_INVALID and b"-1 targets" in L.vsg_last_error()
    assert call(1, -1) == _lib.VSG_ERR_INVALID and b"-1 points" in L.vsg_last_error()
    assert call(1, len(desc), fr=(C.c_void_p * 1)(None)) == _lib.VSG_ERR_INVALID
    assert b"target 0" in L.vsg_last_error()
    assert call(1, len(desc), sg=(C.c_void_p * 1)(None)) == _lib.VSG_ERR_INVALID
    bad = pts.copy()
    bad["valid"][5], bad["level"][5] = 1, 8       # the default pyramid has 8 levels
    assert call(1, len(desc), p=bad) == _lib.VSG_ERR_INVALID
    assert b"target 0" in L.vsg_last_error() and b"level 8" in L.vsg_last_error()
    assert call(1, len(desc)) == _lib.VSG_OK      # the matcher still works after rejected calls
    if L.vsg_device_count() > 1:                  # a target uploaded by a matcher of another device
        from visual_sgraphs_b200.matcher import ORBmatcher
        m1 = ORBmatcher(device=1)
        f1 = m1.frame(fd)
        assert call(1, len(desc), fr=(C.c_void_p * 1)(f1._h.value)) == _lib.VSG_ERR_INVALID
        assert b"device 1" in L.vsg_last_error()


def test_cpp_multi_target_fuse_equals_the_loop(tmp_path):
    pkg = os.path.join(ROOT, "visual_sgraphs_b200")
    exe = str(tmp_path / "fuse_multi_test")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "fuse_multi_test.cpp"),
                           "-L" + pkg, "-lvsg_cuda", "-Wl,-rpath," + pkg])
    out = subprocess.run([exe], capture_output=True, text=True)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "FUSE MULTI TEST OK" in out.stdout
