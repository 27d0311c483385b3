"""CPU-only parity PIN: the reference's own ORBextractor.cc — compiled UNMODIFIED into oracle/_ref/libvsg_ref.so
(oracle/ref_build/Makefile; OpenCV calls resolved by the cv2-pinned compat layer) — against the oracle port
(oracle/orb_oracle.cpp) and the committed golden fixtures.  Where that library is not built, only the comparison of
the oracle with the golden fixtures (the reference's stored outputs) runs; the other tests skip.

What this pins is everything the reference itself owns: constructor tables (ORBextractor.cc:411-470), the cell loop
and threshold retry (:787-900), DistributeOctTree with its std::list / push_front / std::sort order (:562-785),
IC_Angle / rBRIEF float paths compiled from the reference's expressions (:73-149), output ordering and the lapping
partition (:1113-1168), the pyramid chain and its in-place border (:1171-1195).
"""
import json
import os

import numpy as np
import pytest

from tests.golden_cases import CASES, frame_of
from visual_sgraphs_b200.synth import synth_frame

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def live_ref():
    """The reference library where it is built (or buildable from the reference's sources), else None."""
    from oracle import ref as r
    if not r.available():
        return None
    r.build()
    return r


@pytest.fixture(scope="module")
def ref(live_ref):
    if live_ref is None:
        pytest.skip("oracle/_ref/libvsg_ref.so is not built and the reference's sources are not present")
    return live_ref


def _same(a, b, what):
    ma, ka, da = a
    mb, kb, db = b
    assert ma == mb, what
    assert len(ka) == len(kb), what
    assert ka.tobytes() == kb.tobytes(), what          # x, y, size, angle, response, octave, class_id: bit-exact
    assert np.array_equal(da, db), what


def test_reference_sources_are_the_unmodified_files(ref):
    """The build recipe records the SHA-256 of the reference file it compiled; when /root/reference is present
    the digest must be that of the file as it lies there (nothing patched or copied)."""
    import hashlib
    lines = [l.split() for l in open(os.path.join(os.path.dirname(ref._LIB_PATH), "SOURCES.sha256")) if l.strip()]
    assert sorted(os.path.basename(p) for _, p in lines) == ["ORBextractor.cc", "ORBmatcher.cc"]
    if not os.path.isdir(ref._REF_ROOT):
        pytest.skip("reference tree not present (GPU box)")
    for digest, path in lines:
        assert path.startswith(ref._REF_ROOT + "/src/")
        assert digest == hashlib.sha256(open(path, "rb").read()).hexdigest(), path


def test_tables(ref, oracle):
    for args in [(1000, 1.2, 8, 20, 7), (1200, 1.2, 8, 20, 7), (2000, 1.2, 8, 20, 7), (5000, 1.2, 8, 20, 7),
                 (750, 1.1, 5, 15, 5), (333, 1.44, 4, 30, 9), (1500, 1.25, 7, 12, 3)]:
        a, b = ref.RefExtractor(*args).tables(), oracle.OracleExtractor(*args).tables()
        for k in a:
            assert a[k].tobytes() == b[k].tobytes(), (args, k)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_reference_equals_oracle_and_golden(live_ref, oracle, case):
    """The golden fixtures hold the reference's own outputs (tests/golden/make_golden.py), so the oracle is compared
    with them with or without the library; the level-by-level comparison needs the library."""
    name, src, wh, nfeat, lap = case
    frame = frame_of(src, wh)
    o = oracle.OracleExtractor(nfeat)
    got_o = o(frame, lap)
    gold = np.load(os.path.join(GOLD, name + ".npz"))
    meta = next(c for c in json.load(open(os.path.join(GOLD, "index.json")))["cases"] if c["name"] == name)
    _same(got_o, (meta["mono_index"], gold["keypoints"], gold["descriptors"]), name)
    if live_ref is None:
        return
    r = live_ref.RefExtractor(nfeat)
    _same(r(frame, lap), got_o, name)
    for level in range(8):
        assert r.level_size(level) == o.level_size(level)
        assert np.array_equal(r.level_padded(level), o.level_padded(level)), (name, level)   # incl. the 19-px frame
        kr, ko = r.level_keypoints(frame, level), o.level_keypoints(level)
        assert kr.tobytes() == ko.tobytes(), (name, level)                                   # list order + angles


@pytest.mark.parametrize("seed", range(12))
def test_random_configurations(ref, oracle, seed):
    """Same 12 parameter / shape draws as tests/test_gpu_extractor.py::test_random_configurations."""
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
    _same(ref.RefExtractor(*args)(frame, lap), oracle.OracleExtractor(*args)(frame, lap), "seed %d %s" % (seed, (args,)))


def test_two_hundred_seeded_c1_frames(ref, oracle):
    """200 frames of the bench workload (C1: 640x480, 1000 features): every keypoint field and descriptor byte."""
    r, o = ref.RefExtractor(1000), oracle.OracleExtractor(1000)
    total = 0
    for seed in range(3000, 3200):
        frame = synth_frame(seed, 640, 480)
        a, b = r(frame), o(frame)
        _same(a, b, "seed %d" % seed)
        total += len(a[1])
    assert total > 200 * 990


def test_non_contiguous_input_and_c4_shape(ref, oracle):
    big = synth_frame(41, 1400, 800)
    view = big[40:760, 60:1340]                       # 1280x720 view with a 1400-byte pitch
    _same(ref.RefExtractor(2000)(view), oracle.OracleExtractor(2000)(view), "C4 view")
    _same(ref.RefExtractor(2000)(np.ascontiguousarray(view)), oracle.OracleExtractor(2000)(view), "C4 copy vs view")


def test_distribute_octree_alone(ref, oracle):
    """DistributeOctTree on random candidate clouds incl. heavy ties in (count, UL.x) — the std::sort order case
    (SURVEY Appendix C#1) — and degenerate inputs (few points, one column, nIni = 2)."""
    rng = np.random.default_rng(11)
    r = ref.RefExtractor(1000)
    L = oracle.lib()
    for trial in range(60):
        w, h = [(608, 448), (720, 448), (1209, 344), (147, 102)][trial % 4]
        n = int(rng.choice([0, 1, 3, 17, 200, 2000, 7000]))
        grid = 1 if trial % 3 else 4                  # coarse grid -> many equal node counts
        xy = (rng.integers(0, [w // grid, h // grid], size=(n, 2)) * grid).astype(np.float32)
        resp = rng.integers(7, 60 if trial % 2 else 9, size=(n, 1)).astype(np.float32)
        xyr = np.ascontiguousarray(np.hstack([xy, resp]))
        quota = int(rng.choice([5, 60, 217, 434]))
        want = r.distribute_octree(xyr, 0, w, 0, h, quota)
        sel = np.zeros(n + 8, np.int32)
        m = L.orc_distribute_octree(xyr.ctypes.data, n, 0, w, 0, h, quota, sel.ctypes.data, len(sel))
        got = xyr[sel[:m]]
        assert got.shape == want.shape and np.array_equal(got, want), (trial, n, quota)


def test_empty_image(ref):
    mono, kps, desc = ref.RefExtractor()(np.zeros((0, 0), np.uint8))
    assert mono == -1 and len(kps) == 0


def _two_related_frames(tmp_path):
    a = synth_frame(11, 640, 480)
    rng = np.random.default_rng(12)
    b = np.roll(a, (5, 9), (0, 1))
    b = np.clip(b.astype(np.int16) + rng.integers(-3, 4, b.shape), 0, 255).astype(np.uint8)
    pa, pb = str(tmp_path / "a.raw"), str(tmp_path / "b.raw")
    a.tofile(pa)
    b.tofile(pb)
    return pa, pb


def test_reference_orbmatcher_equals_shim_on_the_oracle_port(ref, oracle, tmp_path):
    """The reference's ORBmatcher.cc (compiled unmodified against stand-in Frame / KeyFrame / MapPoint classes) vs the
    drop-in shim's host code running on the CPU oracle port (tests/cpp/vsg_on_oracle.cpp), all 13 methods incl. the
    two-camera branches the shim supports: return values, every written map-point pointer, vnMatches12 / vpMatches12 /
    vMatchedPairs / vpReplacePoint, Replace / AddObservation side effects (tests/cpp/ref_matcher_test.cpp)."""
    import subprocess
    exe = ref.matcher_test_binary("cpu")
    assert exe, "oracle/_ref/ref_matcher_test_cpu was not built"
    pa, pb = _two_related_frames(tmp_path)
    out = subprocess.run([exe, pa, pb], capture_output=True, text=True, timeout=600, env=dict(os.environ, VSG_FRAME_CACHE_STATS="1"))
    assert out.returncode == 0, out.stdout[-4000:] + out.stderr[-2000:]
    assert "0 failed" in out.stdout
    # the "one Track()" block runs three searches per frame: the shim's frame cache must have served the repeats
    import re
    m = re.search(r"vsg frame cache: (\d+) hits, (\d+) uploads", out.stderr)
    assert m and int(m.group(1)) >= 6, out.stderr[-500:]
    # ... and switching it off changes nothing
    off = subprocess.run([exe, pa, pb], capture_output=True, text=True, timeout=600, env=dict(os.environ, VSG_FRAME_CACHE="0"))
    assert off.returncode == 0 and off.stdout == out.stdout
