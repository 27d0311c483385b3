"""GPU parity tests (run on the B200 with -m gpu): the CUDA extractor behind the C ABI against the CPU
oracle, stage by stage and end to end, on the golden cases and on seeded synthetic frames.

Bars (BASELINE.json north_star): pyramid, blurred levels, FAST candidates (positions + responses),
oct-tree keypoint sets and output order bit-exact; angles within 1e-3 degrees; >= 99.9 % of
descriptor bits identical.
"""
import json
import os

import numpy as np
import pytest

from tests.golden_cases import CASES, frame_of
from visual_sgraphs_b200.synth import synth_frame, synth_sequence

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ANGLE_TOL_DEG = 1e-3
MIN_DESC_BIT_AGREEMENT = 0.999


def _extractor(nfeat, **kw):
    from visual_sgraphs_b200.extractor import ORBextractor
    return ORBextractor(nfeat, 1.2, 8, 20, 7, **kw)


def _compare_outputs(got, want, what=""):
    mono_g, k_g, d_g = got
    mono_w, k_w, d_w = want
    assert mono_g == mono_w, what
    assert len(k_g) == len(k_w), what
    for f in ("x", "y", "size", "response", "octave", "class_id"):
        assert np.array_equal(k_g[f], k_w[f]), (what, f)
    if len(k_w):
        da = np.abs(k_g["angle"].astype(np.float64) - k_w["angle"].astype(np.float64))
        da = np.minimum(da, 360.0 - da)
        assert da.max() <= ANGLE_TOL_DEG, (what, da.max())
        bits = np.unpackbits(np.bitwise_xor(d_g, d_w)).sum()
        agree = 1.0 - bits / (d_w.size * 8.0)
        assert agree >= MIN_DESC_BIT_AGREEMENT, (what, agree)
        return float(da.max()), float(agree)
    return 0.0, 1.0


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_stage_parity_on_golden_cases(oracle, case):
    name, src, wh, nfeat, lap = case
    frame = frame_of(src, wh)
    orc = oracle.OracleExtractor(nfeat)
    want = orc(frame, lap)
    ex = _extractor(nfeat)
    got = ex(frame, lap)
    for level in range(8):
        assert ex.level_size(level) == orc.level_size(level)
        assert np.array_equal(ex.pyramid_level(level), orc.level(level)), (name, "pyramid", level)
        b = orc.blurred(level)
        if b is not None:
            assert np.array_equal(ex.blurred_level(level), b), (name, "blur", level)
        assert np.array_equal(ex.candidates(level).astype(np.float32), orc.candidates(level)), (name, "fast", level)
        lk = orc.level_keypoints(level)
        want_lk = np.stack([lk["x"], lk["y"], lk["response"]], 1).astype(np.int32) if len(lk) else np.zeros((0, 3), np.int32)
        assert np.array_equal(ex.level_keypoints(level), want_lk), (name, "octree", level)
    _compare_outputs(got, want, name)
    # and against the committed fixture (generated with real OpenCV for the OpenCV-facing stages)
    gold = np.load(os.path.join(GOLD, name + ".npz"))
    meta = next(c for c in json.load(open(os.path.join(GOLD, "index.json")))["cases"] if c["name"] == name)
    assert got[0] == meta["mono_index"] and len(got[1]) == meta["n_keypoints"]
    if len(got[1]):
        _compare_outputs(got, (meta["mono_index"], gold["keypoints"], gold["descriptors"]), name + "/golden")


def test_descriptors_are_bit_exact_on_synthetic_frames(oracle):
    """Stronger than the 99.9 % bar: report (and require) exact angles and descriptors where they hold."""
    orc = oracle.OracleExtractor(1000)
    ex = _extractor(1000)
    worst_angle, worst_agree = 0.0, 1.0
    for seed in range(1000, 1006):
        frame = synth_frame(seed)
        a, g = _compare_outputs(ex(frame), orc(frame), "seed %d" % seed)
        worst_angle, worst_agree = max(worst_angle, a), min(worst_agree, g)
    print("worst angle diff %.3g deg, worst descriptor bit agreement %.6f" % (worst_angle, worst_agree))
    assert worst_angle == 0.0


def test_empty_image_returns_minus_one():
    ex = _extractor(1000)
    mono, kps, desc = ex(np.zeros((0, 0), np.uint8))
    assert mono == -1 and len(kps) == 0 and desc.shape == (0, 32)


def test_too_small_image_is_rejected():
    from visual_sgraphs_b200._lib import VsgError
    ex = _extractor(100)
    with pytest.raises(VsgError):
        ex(np.zeros((60, 60), np.uint8))


def test_non_contiguous_input_rows(oracle):
    big = np.zeros((300, 500), np.uint8)
    frame = synth_frame(3, 322, 243)
    big[20:263, 40:362] = frame
    view = big[20:263, 40:362]
    assert not view.flags["C_CONTIGUOUS"]
    _compare_outputs(_extractor(500)(view), oracle.OracleExtractor(500)(frame), "strided")


def test_shape_change_reconfigures(oracle):
    ex = _extractor(500)
    orc = oracle.OracleExtractor(500)
    for wh in ((322, 243), (640, 480), (322, 243)):
        frame = synth_frame(11, *wh)
        _compare_outputs(ex(frame), orc(frame), str(wh))


def test_batch_matches_per_frame(oracle):
    frames = synth_sequence(5, 640, 480, first_seed=2000)
    ex = _extractor(1000, max_batch=8)
    orc = oracle.OracleExtractor(1000)
    res = ex.extract_batch(frames)
    assert len(res) == 5
    for f in range(5):
        _compare_outputs(res[f], orc(frames[f]), "batch frame %d" % f)
    # per-frame taps of a batch
    orc(frames[3])
    assert np.array_equal(ex.pyramid_level(4, frame=3), orc.level(4))
    # a second, smaller batch on the same handle
    res2 = ex.extract_batch(frames[:2], lapping=(0, 1000))
    for f in range(2):
        _compare_outputs(res2[f], orc(frames[f], (0, 1000)), "batch2 frame %d" % f)


def test_device_resident_batch(oracle):
    torch = pytest.importorskip("torch")
    frames = synth_sequence(3, 640, 480, first_seed=3000)
    ex = _extractor(1000, max_batch=4)
    cap = ex.max_keypoints(640, 480)
    d_frames = torch.from_numpy(frames).cuda()
    kps = torch.zeros((3, cap, 28), dtype=torch.uint8, device="cuda")
    desc = torch.zeros((3, cap, 32), dtype=torch.uint8, device="cuda")
    n = torch.zeros(3, dtype=torch.int32, device="cuda")
    mono = torch.zeros(3, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ex.extract_batch_dev(d_frames, kps, desc, n, mono)
    ex.sync()
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE
    orc = oracle.OracleExtractor(1000)
    for f in range(3):
        nf = int(n[f])
        k = kps[f, :nf].cpu().numpy().copy().view(KEYPOINT_DTYPE).reshape(-1)
        _compare_outputs((int(mono[f]), k, desc[f, :nf].cpu().numpy()), orc(frames[f]), "dev frame %d" % f)


@pytest.mark.parametrize("wh,nfeat", [((752, 480), 1200), ((1280, 720), 2000)])
def test_other_baseline_shapes(oracle, wh, nfeat):
    frame = synth_frame(4242, *wh)
    _compare_outputs(_extractor(nfeat)(frame), oracle.OracleExtractor(nfeat)(frame), str(wh))


def test_full_size_properties_without_oracle():
    """Size-independent properties at the BASELINE batch size: determinism across repeated runs and
    invariants of the output ordering (level-major, coordinates inside the FAST-able area)."""
    frames = synth_sequence(16, 640, 480, first_seed=5000)
    ex = _extractor(1000, max_batch=16)
    r1 = ex.extract_batch(frames)
    r2 = ex.extract_batch(frames)
    scale = ex.GetScaleFactors()
    for (m1, k1, d1), (m2, k2, d2) in zip(r1, r2):
        assert m1 == m2 and k1.tobytes() == k2.tobytes() and np.array_equal(d1, d2)
        assert 990 <= len(k1) <= 1030 and m1 == len(k1)
        assert (np.diff(k1["octave"]) >= 0).all()
        lx = k1["x"] / scale[k1["octave"]]
        assert (lx >= 18.99).all()
        assert (k1["size"] == np.floor(31 * scale[k1["octave"]])).all()


@pytest.mark.parametrize("pinned", [False, True])
def test_chunked_pipeline_matches_single_stream(oracle, monkeypatch, pinned):
    """vsg_extract_batch cuts large host batches into chunks that rotate over three CUDA streams (H2D / kernels / D2H
    overlap).  Every frame must come out exactly as from a one-frame call, whatever chunk it lands in."""
    torch = pytest.importorskip("torch")
    monkeypatch.setenv("VSG_CHUNK_FRAMES", "3")          # read when the handle is created
    base = synth_sequence(4, 640, 480, first_seed=7000)
    frames = np.stack([np.roll(base[i % 4], 5 * (i // 4), 1) for i in range(11)])   # chunks of 3, 3, 3, 2
    ex = _extractor(1000, max_batch=11)
    if pinned:
        from visual_sgraphs_b200._lib import check, ptr
        cap = ex.max_keypoints(640, 480)
        t_frames = torch.from_numpy(frames).pin_memory()
        kps = torch.zeros((11, cap + 5, 28), dtype=torch.uint8).pin_memory()       # capacity > out_cap: strided D2H
        desc = torch.zeros((11, cap + 5, 32), dtype=torch.uint8).pin_memory()
        n, mono = np.zeros(11, np.int32), np.zeros(11, np.int32)
        check(ex._L.vsg_extract_batch(ex._h, ptr(t_frames), 11, 640, 480, 640, 640 * 480, 0, 0, ptr(kps), ptr(desc), cap + 5,
                                      ptr(n), ptr(mono)))
        from visual_sgraphs_b200._lib import KEYPOINT_DTYPE
        res = [(int(mono[f]), kps[f, :n[f]].numpy().copy().view(KEYPOINT_DTYPE).reshape(-1), desc[f, :n[f]].numpy().copy())
               for f in range(11)]
    else:
        res = ex.extract_batch(frames)
    single = _extractor(1000)
    orc = oracle.OracleExtractor(1000)
    for f in range(11):
        m, k, d = single(frames[f])
        assert res[f][0] == m and res[f][1].tobytes() == k.tobytes() and np.array_equal(res[f][2], d), f
    for f in (0, 4, 10):
        _compare_outputs(res[f], orc(frames[f]), "chunked frame %d" % f)
    orc(frames[7])
    assert np.array_equal(ex.pyramid_level(3, frame=7), orc.level(3))


@pytest.mark.parametrize("channels,rgb", [(3, True), (3, False), (4, True), (4, False)])
def test_colour_ingest_matches_gray_path(oracle, channels, rgb):
    """vsg_extract_batch_color: cvtColor on the device (Tracking.cc:1595-1608) then the same pipeline; must equal the
    gray path fed with the oracle's (cv2-pinned) conversion, including a width that is not a multiple of 4."""
    rng = np.random.default_rng(17 + channels + rgb)
    for w, h, nf in ((640, 480, 3), (322, 243, 2)):
        gray = synth_sequence(nf, w, h, first_seed=9100)
        col = np.empty((nf, h, w, channels), np.uint8)
        # a colour image whose luma has structure: gray plus per-channel offsets and noise
        for c in range(channels):
            col[..., c] = np.clip(gray.astype(np.int16) + rng.integers(-20, 21, gray.shape), 0, 255)
        ex = _extractor(700, max_batch=nf)
        got = ex.extract_batch_color(col, rgb=rgb)
        ref = _extractor(700)
        for f in range(nf):
            g = oracle.cvt_gray(col[f], rgb)
            m, k, d = ref(g)
            assert got[f][0] == m and got[f][1].tobytes() == k.tobytes() and np.array_equal(got[f][2], d), (w, f)
            assert np.array_equal(ex.pyramid_level(0, frame=f), g)


@pytest.mark.parametrize("seed", range(12))
def test_random_configurations(oracle, seed):
    """Randomised extractor parameters and frame shapes (incl. KITTI's 1241x376 and widths that are not multiples of
    4): every output must equal the oracle's — the constructor tables, cell grids, quotas and nIni all change."""
    rng = np.random.default_rng(500 + seed)
    shapes = [(1241, 376), (641, 479), (322, 243), (752, 480), (517, 389), (960, 540), (400, 400), (480, 640)]
    w, h = shapes[seed % len(shapes)]
    nfeat = int(rng.integers(200, 2500))
    scale = float(np.float32(rng.choice([1.1, 1.2, 1.25, 1.3, 1.44])))
    nlevels = int(rng.integers(3, 9))
    while min(w, h) / (scale ** (nlevels - 1)) < 70:       # the smallest level must still hold one 35-px cell
        nlevels -= 1
    ini, mn = int(rng.integers(10, 40)), int(rng.integers(3, 10))
    frame = synth_frame(7000 + seed, w, h)
    if seed % 3 == 0:
        frame = (frame // 4 + 96).astype(np.uint8)          # low contrast: many cells take the minThFAST retry
    lap = (0, 0) if seed % 2 else (int(w * 0.3), int(w * 0.6))
    from visual_sgraphs_b200.extractor import ORBextractor
    got = ORBextractor(nfeat, scale, nlevels, ini, mn)(frame, lap)
    want = oracle.OracleExtractor(nfeat, scale, nlevels, ini, mn)(frame, lap)
    _compare_outputs(got, want, "seed %d: %dx%d nfeat %d scale %.2f levels %d th %d/%d" % (seed, w, h, nfeat, scale, nlevels, ini, mn))


def test_error_conventions_of_the_c_abi():
    """Status codes at the boundary: bad arguments are VSG_ERR_INVALID, too-small outputs VSG_ERR_CAPACITY, an empty
    image the reference's -1 (VSG_EMPTY_IMAGE, ORBextractor.cc:1087-1088); a failed call leaves the handle usable."""
    import ctypes as C
    from visual_sgraphs_b200 import _lib
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE, ptr
    L = _lib.load()
    ex = _extractor(1000, max_batch=2)
    frame = synth_frame(77, 640, 480)
    cap = ex.max_keypoints(640, 480)
    kps, desc = np.zeros(cap, KEYPOINT_DTYPE), np.zeros((cap, 32), np.uint8)
    n, mono = C.c_int(0), C.c_int(0)
    args = lambda img, w, h, pitch, c: (ex._h, ptr(img), w, h, pitch, 0, 0, ptr(kps), ptr(desc), c, C.byref(n), C.byref(mono))
    assert L.vsg_extract(*args(None, 640, 480, 640, cap)) == _lib.VSG_EMPTY_IMAGE
    assert L.vsg_extract(*args(frame, 0, 480, 640, cap)) == _lib.VSG_EMPTY_IMAGE
    assert L.vsg_extract(*args(frame, 640, 480, 320, cap)) == _lib.VSG_ERR_INVALID          # pitch < width
    assert L.vsg_extract(*args(frame, 60, 60, 640, cap)) == _lib.VSG_ERR_INVALID            # too small for one 35-px cell
    assert b"too small" in L.vsg_last_error()
    assert L.vsg_extract(*args(frame, 640, 480, 640, 10)) == _lib.VSG_ERR_CAPACITY          # 10 slots for ~1000 keypoints
    three = np.stack([frame] * 3)
    kb, db = np.zeros((3, cap), KEYPOINT_DTYPE), np.zeros((3, cap, 32), np.uint8)
    nb, mb = np.zeros(3, np.int32), np.zeros(3, np.int32)
    assert L.vsg_extract_batch(ex._h, ptr(three), 3, 640, 480, 640, 640 * 480, 0, 0, ptr(kb), ptr(db), cap, ptr(nb),
                               ptr(mb)) == _lib.VSG_ERR_INVALID                              # 3 frames > max_batch 2
    assert L.vsg_extract_batch_color(ex._h, ptr(three), 1, 640, 480, 640 * 2, 640 * 480 * 2, 2, 1, 0, 0, ptr(kb), ptr(db),
                                     cap, ptr(nb), ptr(mb)) == _lib.VSG_ERR_INVALID          # 2 channels
    assert L.vsg_extractor_create(C.byref(_lib.OrbParams(1000, 2.5, 8, 20, 7)), 0, 1, C.byref(C.c_void_p())) == _lib.VSG_ERR_INVALID
    assert L.vsg_extractor_create(C.byref(_lib.OrbParams(1000, 1.2, 8, 20, 7)), 99, 1, C.byref(C.c_void_p())) == _lib.VSG_ERR_CUDA
    m, k, d = ex(frame)                                                                      # the handle still works
    assert m == len(k) > 900


def test_baseline_batch_size_properties(oracle):
    """The bench's batch shape (512 frames of 640x480 through the chunked host-pointer pipeline): every frame is
    independent of its position in the batch (the 32 distinct frames repeat 16 times and must repeat their results),
    the first and the last frame equal the oracle, the device-resident path gives the same bytes."""
    torch = pytest.importorskip("torch")
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE, check, ptr
    base = synth_sequence(32, 640, 480, first_seed=12000)
    frames = torch.from_numpy(np.concatenate([base] * 16)).pin_memory()
    ex = _extractor(1000, max_batch=512)
    cap = ex.max_keypoints(640, 480)
    kps = torch.zeros((512, cap, 28), dtype=torch.uint8).pin_memory()
    desc = torch.zeros((512, cap, 32), dtype=torch.uint8).pin_memory()
    n, mono = np.zeros(512, np.int32), np.zeros(512, np.int32)
    check(ex._L.vsg_extract_batch(ex._h, ptr(frames), 512, 640, 480, 640, 640 * 480, 0, 0, ptr(kps), ptr(desc), cap, ptr(n),
                                  ptr(mono)))
    kn, dn = kps.numpy(), desc.numpy()
    for f in range(32, 512):
        b = f % 32
        assert n[f] == n[b] and kn[f, :n[f]].tobytes() == kn[b, :n[b]].tobytes() and dn[f, :n[f]].tobytes() == dn[b, :n[b]].tobytes(), f
    orc = oracle.OracleExtractor(1000)
    for f in (0, 31):
        k = kn[f, :n[f]].copy().view(KEYPOINT_DTYPE).reshape(-1)
        _compare_outputs((int(mono[f]), k, dn[f, :n[f]]), orc(base[f]), "frame %d of 512" % f)
    d_frames = frames.cuda()
    kd = torch.zeros((512, cap, 28), dtype=torch.uint8, device="cuda")
    dd = torch.zeros((512, cap, 32), dtype=torch.uint8, device="cuda")
    nd = torch.zeros(512, dtype=torch.int32, device="cuda")
    md = torch.zeros(512, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ex.extract_batch_dev(d_frames, kd, dd, nd, md)
    ex.sync()
    assert np.array_equal(nd.cpu().numpy(), n)
    for f in (0, 100, 511):
        assert kd[f, :n[f]].cpu().numpy().tobytes() == kn[f, :n[f]].tobytes() and dd[f, :n[f]].cpu().numpy().tobytes() == dn[f, :n[f]].tobytes()


@pytest.mark.parametrize("wh", [(640, 480), (752, 480), (1241, 376), (320, 240)])
def test_tensor_core_blur_is_bit_identical(monkeypatch, wh):
    """VSG_BLUR_TC=1: the 7x7 Gaussian blur (ORBextractor.cc:1129-1130) runs as banded u8 GEMMs on tcgen05 (csrc/blur_tc.cu).
    Every blurred plane and every output must equal the CUDA-core blur's, borders (REFLECT_101) included."""
    from visual_sgraphs_b200.extractor import ORBextractor
    w, h = wh
    nf = 6
    frames = np.stack([synth_frame(500 + i, w, h) for i in range(nf)])
    frames[1, :, :4] = 255          # strong content on the borders
    frames[1, :, -4:] = 7
    frames[2, :4] = 200
    frames[2, -4:] = 31
    monkeypatch.setenv("VSG_BLUR_TC", "0")
    ex0 = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=nf)
    want = ex0.extract_batch(frames)
    planes0 = [[ex0.blurred_level(l, f) for l in range(8)] for f in range(nf)]
    monkeypatch.setenv("VSG_BLUR_TC", "1")
    ex1 = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=nf)
    got = ex1.extract_batch(frames)
    for f in range(nf):
        for l in range(8):
            p1 = ex1.blurred_level(l, f)
            if not np.array_equal(p1, planes0[f][l]):
                bad = np.argwhere(p1 != planes0[f][l])
                raise AssertionError("frame %d level %d: %d pixels differ, first %s (%d vs %d)" % (
                    f, l, len(bad), bad[0], p1[tuple(bad[0])], planes0[f][l][tuple(bad[0])]))
    for a, b in zip(got, want):
        assert a[0] == b[0] and a[1].tobytes() == b[1].tobytes() and np.array_equal(a[2], b[2])


def test_tensor_core_blur_falls_back_when_tma_cannot_address_the_planes(monkeypatch):
    """More than 8 levels, or a caller-owned level 0 whose pitch is not a multiple of 16 bytes: the batch takes the CUDA-core
    blur (csrc/blur_tc.cu: plan_blur_tc returns no plan) and the results do not change."""
    import torch
    from visual_sgraphs_b200.extractor import ORBextractor
    frames = np.stack([synth_frame(700 + i, 640, 480) for i in range(4)])
    outs = []
    for tc in ("0", "1"):
        monkeypatch.setenv("VSG_BLUR_TC", tc)
        outs.append(ORBextractor(1500, 1.2, 10, 20, 7, max_batch=4).extract_batch(frames))
    for a, b in zip(*outs):
        assert a[0] == b[0] and a[1].tobytes() == b[1].tobytes() and np.array_equal(a[2], b[2])
    # device-resident frames, 644 bytes per row (the device API wants 4-byte alignment; TMA wants 16)
    odd = np.stack([synth_frame(710 + i, 644, 480) for i in range(4)])
    res = []
    for tc in ("0", "1"):
        monkeypatch.setenv("VSG_BLUR_TC", tc)
        ex = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=4)
        cap = ex.max_keypoints(644, 480)
        d = torch.from_numpy(odd).cuda()
        kd = torch.zeros((4, cap, 28), dtype=torch.uint8, device="cuda")
        dd = torch.zeros((4, cap, 32), dtype=torch.uint8, device="cuda")
        nd = torch.zeros(4, dtype=torch.int32, device="cuda")
        md = torch.zeros(4, dtype=torch.int32, device="cuda")
        ex.extract_batch_dev(d, kd, dd, nd, md)
        ex.sync()
        res.append((nd.cpu().numpy(), kd.cpu().numpy(), dd.cpu().numpy()))
    assert np.array_equal(res[0][0], res[1][0])
    for f in range(4):
        n = res[0][0][f]
        assert res[0][1][f, :n].tobytes() == res[1][1][f, :n].tobytes() and res[0][2][f, :n].tobytes() == res[1][2][f, :n].tobytes()


@pytest.mark.parametrize("shape", [(640, 480, 8, 1.2), (752, 480, 8, 1.2), (1241, 376, 8, 1.2), (1280, 720, 8, 1.2), (640, 480, 5, 1.5),
                                   (800, 600, 4, 1.7), (640, 480, 12, 1.1)])
def test_one_launch_pyramid_matches_the_level_by_level_kernels(monkeypatch, shape):
    """Batches of up to VSG_PYR_TILE (4) frames build the whole pyramid in one launch (csrc/pyramid.cu: pyramid_tile_kernel,
    every level of a tile from the previous one in shared memory).  Planes and results must equal the seven resize launches'
    (ORBextractor::ComputePyramid, ORBextractor.cc:1171-1195)."""
    from visual_sgraphs_b200.extractor import ORBextractor
    w, h, nlev, sf = shape
    frames = np.stack([synth_frame(900 + i, w, h) for i in range(3)])
    monkeypatch.setenv("VSG_PYR_TILE", "0")
    ex0 = ORBextractor(1000, sf, nlev, 20, 7, max_batch=3)
    want = ex0.extract_batch(frames)
    planes0 = [[ex0.pyramid_level(l, f) for l in range(nlev)] for f in range(3)]
    monkeypatch.setenv("VSG_PYR_TILE", "4")
    ex1 = ORBextractor(1000, sf, nlev, 20, 7, max_batch=3)
    got = ex1.extract_batch(frames)
    for f in range(3):
        for l in range(nlev):
            p1 = ex1.pyramid_level(l, f)
            if not np.array_equal(p1, planes0[f][l]):
                bad = np.argwhere(p1 != planes0[f][l])
                raise AssertionError("frame %d level %d: %d pixels differ, first %s" % (f, l, len(bad), bad[0]))
    for a, b in zip(got, want):
        assert a[0] == b[0] and a[1].tobytes() == b[1].tobytes() and np.array_equal(a[2], b[2])


@pytest.mark.parametrize("shape", [(640, 480, 8, 1.2), (752, 480, 8, 1.2), (1241, 376, 8, 1.2), (1280, 720, 8, 1.2), (640, 480, 5, 1.5),
                                   (644, 484, 10, 1.1)])
def test_tma_staged_resize_matches_the_register_kernel(monkeypatch, shape):
    """VSG_RESIZE_TMA: large batches resize through resize_tma_kernel (csrc/resize_tma.cu: the tile's source window staged by one
    cp.async.bulk.tensor, every source row interpolated once).  Planes and results must equal resize_kernel's
    (ORBextractor::ComputePyramid, ORBextractor.cc:1171-1195); scale factors whose windows exceed the box fall back."""
    from visual_sgraphs_b200.extractor import ORBextractor
    w, h, nlev, sf = shape
    nf = 5
    frames = np.stack([synth_frame(950 + i, w, h) for i in range(nf)])
    monkeypatch.setenv("VSG_PYR_TILE", "0")
    monkeypatch.setenv("VSG_RESIZE_TMA", "0")
    ex0 = ORBextractor(1000, sf, nlev, 20, 7, max_batch=nf)
    want = ex0.extract_batch(frames)
    planes0 = [[ex0.pyramid_level(l, f) for l in range(nlev)] for f in range(nf)]
    monkeypatch.setenv("VSG_RESIZE_TMA", "1")
    ex1 = ORBextractor(1000, sf, nlev, 20, 7, max_batch=nf)
    got = ex1.extract_batch(frames)
    for f in range(nf):
        for l in range(nlev):
            p1 = ex1.pyramid_level(l, f)
            if not np.array_equal(p1, planes0[f][l]):
                bad = np.argwhere(p1 != planes0[f][l])
                raise AssertionError("frame %d level %d: %d pixels differ, first %s (%d vs %d)" % (
                    f, l, len(bad), bad[0], p1[tuple(bad[0])], planes0[f][l][tuple(bad[0])]))
    for a, b in zip(got, want):
        assert a[0] == b[0] and a[1].tobytes() == b[1].tobytes() and np.array_equal(a[2], b[2])
