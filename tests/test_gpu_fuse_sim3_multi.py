"""vsg_fuse_search_sim3_multi (ORBmatcher.fuse_search_sim3_multi) and the batched shim Fuse(vpKFs, vScw, vpPoints, th) +
Fuse(search, k, vpReplacePoint), on the B200 (-m gpu).

One call searches the same map points in many keyframes without the chi-square gates: the targets of
LoopClosing::SearchAndFuse's loop of Fuse(KF, Scw, ...) calls.  For every target t, best_idx[t] must equal vsg_fuse_search
(variant 1) on target t alone and the CPU oracle's fuse_search, index for index, with targets that differ in keypoint count
(including none), pyramid, grid bounds and camera, and the same frame listed twice.  tests/cpp/search_and_fuse_test.cpp then
checks that the shim's batch and resolves leave the same world as the loop of single-target calls.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import match_scenarios as sc
from tests.test_gpu_fuse_multi import KINDS, SHIFT, make_target, world  # noqa: F401  (world is a fixture)
from tests.test_gpu_matcher_kf import _tie_scene
from visual_sgraphs_b200._lib import SEARCH_POINT_DTYPE

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TH = 4.0                                   # LoopClosing::SearchAndFuse's threshold


def _matcher():
    from visual_sgraphs_b200.matcher import ORBmatcher
    return ORBmatcher()


def _launches():
    from visual_sgraphs_b200 import _lib
    return _lib.load().vsg_launch_count()


def _check(got, frames, fds, pts, desc, what, m, oracle):
    """Every target of got against vsg_fuse_search (variant 1) on that target alone and the oracle."""
    for t in range(len(frames)):
        single = m.FuseSearch(frames[t], pts[t], desc, TH, sim3_variant=True)[1]
        want = oracle.fuse_search(fds[t].view, pts[t], desc, TH, np.ones(1, np.float32), 1)[1]
        for name, other in (("vsg_fuse_search on the target alone", single), ("the oracle", want)):
            bad = np.nonzero(got[t] != other)[0]
            if len(bad):
                i = int(bad[0])
                pytest.fail("%s: target %d, query %d: fuse_search_sim3_multi picked keypoint %d, %s %d (%d differences)" %
                            (what, t, i, got[t][i], name, other[i], len(bad)))


@pytest.mark.parametrize("ntargets", [0, 1, 2, 7, 40])
def test_fuse_search_sim3_multi_equals_single_target_searches(oracle, world, ntargets):
    desc = world[2]
    targets = [make_target(world, t, 300 + t) for t in range(ntargets)]
    m = _matcher()
    fds = [fd for fd, _, _ in targets]
    frames = [m.frame(fd) for fd in fds]
    if ntargets >= 2:                          # the same frame twice, with its own projections
        frames[-1], fds[-1] = frames[0], fds[0]
        targets[-1] = (fds[0], None, make_target(world, 0, 999)[2])
    pts = np.stack([p for _, _, p in targets]) if targets else np.zeros((0, len(desc)), SEARCH_POINT_DTYPE)
    before = _launches()
    got = m.fuse_search_sim3_multi(frames, pts, desc, TH)
    assert _launches() - before == (1 if ntargets else 0)
    assert got.shape == (ntargets, len(desc))
    _check(got, frames, fds, pts, desc, "%d targets" % ntargets, m, oracle)
    for t in range(ntargets):                  # every target with keypoints finds something; the empty one nothing
        found = int((got[t] >= 0).sum())
        kind = KINDS[(0 if ntargets >= 2 and t == ntargets - 1 else t) % len(KINDS)]
        if kind[1] == "none":
            assert found == 0
        else:
            assert found > 20, "target %d (%s): %d points found" % (t, kind, found)


def test_no_points(world):
    m = _matcher()
    fd, _, _ = make_target(world, 0, 5)
    before = _launches()
    got = m.fuse_search_sim3_multi([m.frame(fd)] * 3, np.zeros((3, 0), SEARCH_POINT_DTYPE), np.zeros((0, 32), np.uint8), TH)
    assert got.shape == (3, 0) and _launches() == before


def test_loop_closure_sized_call(oracle):
    """12 000+ points x 30 targets: a covisibility group's map points searched in every corrected keyframe."""
    size, nfeat = (1241, 376), 2000
    ka, da, kb, db = sc.two_frames(oracle, shift=SHIFT, size=size, nfeat=nfeat)
    reps = -(-12000 // len(kb))
    rng = np.random.default_rng(8)
    desc = np.concatenate([db ^ (rng.random(db.shape) < 0.02) * rng.integers(1, 256, db.shape, dtype=np.uint8)
                           for _ in range(reps)]).astype(np.uint8)
    n = len(desc)
    assert n >= 12000
    variants = [sc.frame_data(ka, da, size=size), sc.frame_data(ka[::2], da[::2], size=size),
                sc.frame_data(kb, db, size=size), sc.frame_data(ka[1::3], da[1::3], size=size)]
    fds = [variants[t % len(variants)] for t in range(30)]
    pts = np.stack([np.concatenate([sc.search_points(kb, (0, 0) if t % len(variants) == 2 else SHIFT, 50 * t + r, sigma=1.5,
                                                     size=size) for r in range(reps)]) for t in range(30)])
    m = _matcher()
    frames = [m.frame(fd) for fd in fds]
    before = _launches()
    got = m.fuse_search_sim3_multi(frames, pts, desc, TH)
    assert _launches() - before == 1
    _check(got, frames, fds, pts, desc, "loop-closure-sized call", m, oracle)
    assert all((got[t] >= 0).sum() > 1000 for t in range(30))


def test_tie_across_rounds(oracle):
    """Equal distances in two warp rounds of one window, in targets 0 and 2: the first in scan order wins, as in the
    reference's strict '<'."""
    kf, q, d, keys = _tie_scene()
    near = d.copy()
    near[:, 0] ^= 0xFF                         # 8 bits away
    other = sc.frame_data(keys([(320, 240)]), near)
    m = _matcher()
    fk, fo = m.frame(kf), m.frame(other)
    got = m.fuse_search_sim3_multi([fk, fo, fk], np.stack([q, q, q]), d, 30.0)
    want = oracle.fuse_search(kf.view, q, d, 30.0, np.ones(1, np.float32), 1)[1]
    assert got[0][0] == got[2][0] == want[0] == 0
    assert got[1][0] == 0                      # the one keypoint of the other frame


def test_rejects_invalid_calls(world):
    from visual_sgraphs_b200 import _lib
    L = _lib.load()
    m = _matcher()
    fd, _, pts = make_target(world, 0, 7)
    desc = world[2]
    f = m.frame(fd)
    two = np.stack([pts, pts])
    best = np.zeros(two.shape, np.int32)
    call = lambda T, n, fr=(C.c_void_p * 2)(f._h.value, f._h.value), p=two: L.vsg_fuse_search_sim3_multi(  # noqa: E731
        m._h, T, fr, n, _lib.ptr(p), _lib.ptr(desc), C.c_float(TH), _lib.ptr(best))
    assert call(-1, len(desc)) == _lib.VSG_ERR_INVALID and b"-1 targets" in L.vsg_last_error()
    assert call(2, -1) == _lib.VSG_ERR_INVALID and b"-1 points" in L.vsg_last_error()
    assert call(2, len(desc), fr=(C.c_void_p * 2)(f._h.value, None)) == _lib.VSG_ERR_INVALID
    assert b"target 1" in L.vsg_last_error()
    bad = two.copy()
    bad[1]["valid"][5], bad[1]["level"][5] = 1, 8           # the default pyramid has 8 levels
    before = _launches()
    assert call(2, len(desc), p=bad) == _lib.VSG_ERR_INVALID
    assert b"target 1" in L.vsg_last_error() and b"level 8" in L.vsg_last_error()
    assert _launches() == before
    assert call(2, len(desc)) == _lib.VSG_OK                # the matcher still works after rejected calls
    assert np.array_equal(best[0], best[1])
    if L.vsg_device_count() > 1:                            # a target uploaded by a matcher of another device
        from visual_sgraphs_b200.matcher import ORBmatcher
        m1 = ORBmatcher(device=1)
        f1 = m1.frame(fd)
        assert call(2, len(desc), fr=(C.c_void_p * 2)(f._h.value, f1._h.value)) == _lib.VSG_ERR_INVALID
        assert b"target 1" in L.vsg_last_error() and b"device 1" in L.vsg_last_error()


def test_cpp_batched_search_and_fuse_equals_the_loop(tmp_path):
    pkg = os.path.join(ROOT, "visual_sgraphs_b200")
    exe = str(tmp_path / "search_and_fuse_test")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "search_and_fuse_test.cpp"),
                           "-L" + pkg, "-lvsg_cuda", "-Wl,-rpath," + pkg])
    out = subprocess.run([exe], capture_output=True, text=True)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "SEARCH AND FUSE TEST OK" in out.stdout
