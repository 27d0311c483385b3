"""GPU parity against the REFERENCE ITSELF: the CUDA extractor behind the C ABI vs oracle/_ref/libvsg_ref.so, i.e. the
reference's ORBextractor.cc compiled unmodified (oracle/ref_build/Makefile).  The golden cases are also compared with
the reference's outputs stored in tests/golden/ (tests/golden/make_golden.py), so they run where the library is not
built; the other tests skip there.

Bars (BASELINE.json north_star): keypoint sets, order, positions, sizes, responses, octaves bit-exact; angles within
1e-3 degrees; >= 99.9 % of descriptor bits — the tests also REPORT exact equality, which holds on every frame so far.
"""
import hashlib
import json
import os

import numpy as np
import pytest

from tests.golden_cases import CASES, frame_of
from visual_sgraphs_b200.synth import synth_frame

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def live_ref():
    """The reference library where it is built, else None."""
    from oracle import ref as r
    if not r.available():
        return None
    r.lib()
    return r


@pytest.fixture(scope="module")
def ref(live_ref):
    if live_ref is None:
        pytest.skip("oracle/_ref/libvsg_ref.so is not built")
    return live_ref


def _cmp(got, want, what):
    mg, kg, dg = got
    mw, kw, dw = want
    assert mg == mw and len(kg) == len(kw), what
    for f in ("x", "y", "size", "response", "octave", "class_id"):
        assert np.array_equal(kg[f], kw[f]), (what, f)
    if not len(kw):
        return True
    da = np.abs(kg["angle"].astype(np.float64) - kw["angle"].astype(np.float64))
    assert np.minimum(da, 360 - da).max() <= 1e-3, what
    agree = 1.0 - np.unpackbits(dg ^ dw).sum() / (dw.size * 8.0)
    assert agree >= 0.999, (what, agree)
    return kg.tobytes() == kw.tobytes() and np.array_equal(dg, dw)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_golden_cases_against_the_reference(live_ref, case):
    from visual_sgraphs_b200.extractor import ORBextractor
    name, src, wh, nfeat, lap = case
    frame = frame_of(src, wh)
    ex = ORBextractor(nfeat, 1.2, 8, 20, 7)
    got = ex(frame, lap)
    gold = np.load(os.path.join(GOLD, name + ".npz"))                 # the reference's keypoints and descriptors
    meta = next(c for c in json.load(open(os.path.join(GOLD, "index.json")))["cases"] if c["name"] == name)
    assert _cmp(got, (meta["mono_index"], gold["keypoints"], gold["descriptors"]), name), \
        name + ": angles / descriptors not bit-equal"
    for level, lm in enumerate(meta["levels"]):                       # the reference's mvImagePyramid[level], as digests
        assert hashlib.sha256(np.ascontiguousarray(ex.pyramid_level(level)).tobytes()).hexdigest() == lm["level_sha"], \
            (name, level)
    if live_ref is not None:
        r = live_ref.RefExtractor(nfeat)
        assert _cmp(got, r(frame, lap), name), name + ": angles / descriptors not bit-equal"
        for level in range(8):
            assert np.array_equal(ex.pyramid_level(level), r.level(level)), (name, level)     # mvImagePyramid[level]


@pytest.mark.parametrize("seed", range(12))
def test_random_configurations_against_the_reference(ref, seed):
    from visual_sgraphs_b200.extractor import ORBextractor
    rng = np.random.default_rng(500 + seed)
    shapes = [(1241, 376), (641, 479), (322, 243), (752, 480), (517, 389), (960, 540), (400, 400), (480, 640)]
    w, h = shapes[seed % len(shapes)]
    nfeat = int(rng.integers(200, 2500))
    scale = float(np.float32(rng.choice([1.1, 1.2, 1.25, 1.3, 1.44])))
    nlevels = int(rng.integers(3, 9))
    while min(w, h) / (scale ** (nlevels - 1)) < 70:
        nlevels -= 1
    ini, mn = int(rng.integers(10, 40)), int(rng.integers(3, 10))
    frame = synth_frame(7000 + seed, w, h)
    if seed % 3 == 0:
        frame = (frame // 4 + 96).astype(np.uint8)
    lap = (0, 0) if seed % 2 else (int(w * 0.3), int(w * 0.6))
    args = (nfeat, scale, nlevels, ini, mn)
    _cmp(ORBextractor(*args)(frame, lap), ref.RefExtractor(*args)(frame, lap), "seed %d" % seed)


def test_c1_batch_of_96_frames_against_the_reference(ref):
    """The bench workload through the batched entry point: every frame's keypoints and descriptors."""
    from visual_sgraphs_b200.extractor import ORBextractor
    frames = np.stack([synth_frame(5000 + i, 640, 480) for i in range(96)])
    got = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=96).extract_batch(frames)
    r = ref.RefExtractor(1000)
    exact = 0
    for i in range(96):
        exact += bool(_cmp(got[i], r(frames[i]), "frame %d" % i))
    assert exact == 96, "%d of 96 frames bit-equal incl. angles and descriptors" % exact


def test_c4_1280x720_on_eight_frames_against_the_reference(ref):
    from visual_sgraphs_b200.extractor import ORBextractor
    frames = np.stack([synth_frame(6100 + i, 1280, 720) for i in range(8)])
    got = ORBextractor(2000, 1.2, 8, 20, 7, max_batch=8).extract_batch(frames)
    r = ref.RefExtractor(2000)
    for i in range(8):
        assert _cmp(got[i], r(frames[i]), "C4 frame %d" % i)


def test_c2_stereo_shape_and_mono_lapping_against_the_reference(ref):
    from visual_sgraphs_b200.extractor import ORBextractor
    from visual_sgraphs_b200.synth import synth_stereo_pair
    left, right = synth_stereo_pair(8100)
    ex, r = ORBextractor(1200, 1.2, 8, 20, 7), ref.RefExtractor(1200)
    for img in (left, right):
        assert _cmp(ex(img), r(img), "C2")
    mono = synth_frame(77, 640, 480)
    ex5, r5 = ORBextractor(5000, 1.2, 8, 20, 7), ref.RefExtractor(5000)      # mpIniORBextractor: 5 x features, lapping (0, 1000)
    assert _cmp(ex5(mono, (0, 1000)), r5(mono, (0, 1000)), "mono init")


def test_reference_orbmatcher_equals_shim_on_the_cuda_library(ref, tmp_path):
    """tests/cpp/ref_matcher_test.cpp linked against libvsg_cuda.so: the reference's ORBmatcher.cc (unmodified) vs the
    drop-in shim + CUDA kernels on identical worlds — all 13 Search* / Fuse methods, match for match."""
    import subprocess
    exe = ref.matcher_test_binary("gpu")
    if not exe:
        pytest.skip("oracle/_ref/ref_matcher_test_gpu was not shipped")
    a = synth_frame(11, 640, 480)
    rng = np.random.default_rng(12)
    b = np.roll(a, (5, 9), (0, 1))
    b = np.clip(b.astype(np.int16) + rng.integers(-3, 4, b.shape), 0, 255).astype(np.uint8)
    pa, pb = str(tmp_path / "a.raw"), str(tmp_path / "b.raw")
    a.tofile(pa)
    b.tofile(pb)
    out = subprocess.run([exe, pa, pb], capture_output=True, text=True, timeout=600, env=dict(os.environ, VSG_FRAME_CACHE_STATS="1"))
    assert out.returncode == 0, out.stdout[-4000:] + out.stderr[-2000:]
    assert "0 failed" in out.stdout
    import re
    m = re.search(r"vsg frame cache: (\d+) hits", out.stderr)       # the "one Track()" block reuses uploaded frames
    assert m and int(m.group(1)) >= 6, out.stderr[-500:]
