"""vsg_distinctive_descriptors (ORBmatcher.ComputeDistinctiveDescriptors) and the shim's batched
ORBmatcher::ComputeDistinctiveDescriptors(vpMPs), on the B200 (-m gpu).

A call splits its points at 32 observed descriptors: distinctive_warp_kernel takes the short lists (one warp per point),
distinctive_kernel the long ones (one CTA per point).  Every point's row must equal the oracle's restatement of
MapPoint::ComputeDistinctiveDescriptors, in calls with only short lists, only long lists and both, and with planted ties
(the first row wins).  tests/cpp/distinctive_batch_test.cpp then checks that the shim's batch leaves the same map as the
loop of per-point calls.
"""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EDGE_COUNTS = [0, 1, 2, 3, 31, 32, 33, 64, 1024, 1025, 1500]


def _matcher():
    from visual_sgraphs_b200.matcher import ORBmatcher
    return ORBmatcher()


def _launches():
    from visual_sgraphs_b200 import _lib
    return _lib.load().vsg_launch_count()


def _rows(rng, n):
    """n observations of one map point: a base descriptor with 2-30 % of its bits flipped per row."""
    if n == 0:
        return np.zeros((0, 32), np.uint8)
    base = rng.integers(0, 256, 32, dtype=np.uint8)
    return np.stack([base ^ np.packbits(rng.random(256) < rng.uniform(0.02, 0.3)) for _ in range(n)])


def _call(descs):
    ptr = np.concatenate([[0], np.cumsum([len(d) for d in descs])]).astype(np.int32)
    allrows = np.concatenate(descs) if descs else np.zeros((0, 32), np.uint8)
    m = _matcher()
    before = _launches()
    got = m.ComputeDistinctiveDescriptors(allrows, ptr)
    return got, _launches() - before


def _check(got, descs, oracle, what):
    want = [oracle.distinctive_descriptor(d) for d in descs]
    bad = [i for i in range(len(descs)) if got[i] != want[i]]
    if bad:
        i = bad[0]
        pytest.fail("%s: point %d (%d rows): row %d, the oracle %d (%d differences)" % (what, i, len(descs[i]), got[i], want[i],
                                                                                      len(bad)))


def test_edge_and_keyframe_counts_in_one_call(oracle):
    rng = np.random.default_rng(11)
    counts = EDGE_COUNTS + rng.integers(2, 61, 1000).tolist()
    descs = [_rows(rng, n) for n in counts]
    got, launches = _call(descs)
    assert launches == 2
    _check(got, descs, oracle, "edge and keyframe counts")
    assert got[0] == -1 and got[1] == 0


@pytest.mark.parametrize("side,launches", [("short", 1), ("long", 1), ("both", 2)])
def test_sides_of_the_split(oracle, side, launches):
    rng = np.random.default_rng({"short": 1, "long": 2, "both": 3}[side])
    short = [0, 1, 2, 17, 32] + rng.integers(2, 33, 300).tolist()
    long_ = [33, 40, 64, 200, 1025] + rng.integers(33, 120, 40).tolist()
    counts = {"short": short, "long": long_, "both": long_[:20] + short + long_[20:]}[side]
    descs = [_rows(rng, n) for n in counts]
    got, n = _call(descs)
    assert n == launches
    _check(got, descs, oracle, side)


def test_planted_ties(oracle):
    """Duplicate rows and all-identical rows on both sides of the split: equal medians, the first row wins."""
    rng = np.random.default_rng(4)
    descs = []
    for n in (2, 3, 4, 5, 16, 31, 32, 33, 48, 64, 1024, 1100):
        same = np.repeat(rng.integers(0, 256, (1, 32), dtype=np.uint8), n, axis=0)     # every median 0: row 0
        descs.append(same)
        dup = _rows(rng, n)
        dup[n // 2:] = dup[: n - n // 2]                                                # each row twice (odd n: one thrice)
        descs.append(dup)
        pair = _rows(rng, n)
        pair[:] = pair[n - 1]                                                           # all rows equal to the last one
        pair[0, 0] ^= 0x0F                                                              # ... but the first, 4 bits away
        descs.append(pair)
    got, _ = _call(descs)
    _check(got, descs, oracle, "planted ties")
    assert all(got[i] == 0 for i in range(0, len(descs), 3))


def test_no_points_no_launch():
    got, launches = _call([])
    assert len(got) == 0 and launches == 0


def test_cpp_batched_distinctive_descriptors_equal_the_loop(tmp_path):
    pkg = os.path.join(ROOT, "visual_sgraphs_b200")
    exe = str(tmp_path / "distinctive_batch_test")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-o", exe,
                           os.path.join(ROOT, "tests", "cpp", "distinctive_batch_test.cpp"),
                           "-L" + pkg, "-lvsg_cuda", "-Wl,-rpath," + pkg])
    out = subprocess.run([exe], capture_output=True, text=True)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "DISTINCTIVE BATCH TEST OK" in out.stdout
