"""Batched extraction against the CPU oracle in every batch-size regime (run on the B200 with -m gpu).

The extractor picks its kernels by the number of frames in a launch (csrc/vsg_api.cu: run_pipeline):
  <= 4 frames  the whole pyramid in one launch (pyramid_tile_kernel); >= 5: one resize launch per level
  <= 8 frames  programmatic dependent launch, octree_kernel<512>, describe_kernel<16>
  >= 9 frames  no PDL, octree_kernel<256>, describe_kernel<64>
  >= 16 frames resize_tma_kernel on the levels whose source windows fit its box, and the blur as its own tensor-core
               stage after the oct-tree (blur_tc_kernel, at most 8 levels) instead of inside the FAST grid
Host batches of at least 2 x min(VSG_CHUNK_FRAMES, 64) frames are cut into chunks that run on three streams, each at its
own frame offset in the handle's buffers.  Every configuration below runs at the batch sizes on both sides of each
boundary and once chunked, and every frame of every batch must equal the oracle's result for that frame.
"""
import re

import numpy as np
import pytest

from tests.test_gpu_extractor import _compare_outputs
from visual_sgraphs_b200.synth import synth_frame

pytestmark = pytest.mark.gpu

# id, width, height, nfeatures, scale factor, levels, iniThFAST, minThFAST, lapping area (fractions of the width or pixels),
# low-contrast frames
CONFIGS = [
    ("c1_640x480", 640, 480, 1000, 1.2, 8, 20, 7, None, False),
    ("c2_752x480", 752, 480, 1200, 1.2, 8, 20, 7, None, False),
    ("c4_1280x720", 1280, 720, 2000, 1.2, 8, 20, 7, None, False),
    ("kitti_1241x376", 1241, 376, 2000, 1.2, 8, 20, 7, None, False),        # width not a multiple of 16, several roots
    ("odd_641x479_s1.44_l5", 641, 479, 1000, 1.44, 5, 20, 7, None, False),  # odd sizes, large scale steps
    ("960x540_s1.1_l12", 960, 540, 1500, 1.1, 12, 20, 7, None, False),     # > 8 levels: CUDA-core blur at every batch size
    ("1280x720_s1.1_l16", 1280, 720, 2000, 1.1, 16, 20, 7, None, False),   # kMaxLevels
    ("single_level", 640, 480, 1000, 1.2, 1, 20, 7, None, False),          # no pyramid launch at all
    ("tiny_nfeatures", 640, 480, 10, 1.2, 8, 20, 7, None, False),          # last level's quota is 0
    ("low_contrast", 640, 480, 1000, 1.2, 8, 20, 7, None, True),           # cells take the minThFAST retry
    ("lapping_752x480", 752, 480, 1200, 1.2, 8, 20, 7, (0.3, 0.6), False),  # slot_kernel
    ("mono_init_5000", 640, 480, 5000, 1.2, 8, 20, 7, (0, 1000), False),   # monocular initialiser
]
BATCH_SIZES = (1, 4, 5, 8, 9, 15, 16, 17)
CHUNK_FRAMES, CHUNKED_BATCH = 20, 58
DISTINCT_FRAMES = 8
# the batch-size thresholds of the launchers (csrc/vsg_api.cu, octree.cu, describe.cu, resize_tma.cu, blur_tc.cu)
PYR_TILE_MAX_FRAMES, PDL_MAX_FRAMES, LARGE_BATCH_MIN_FRAMES, BLUR_TC_MAX_LEVELS = 4, 8, 16, 8


def _params(cfg):
    _, w, h, nfeat, scale, nlevels, ini, mn, lap, _ = cfg
    scale = float(np.float32(scale))
    if lap is None:
        lap = (0, 0)
    elif isinstance(lap[1], float):
        lap = (int(w * lap[0]), int(w * lap[1]))
    return w, h, (nfeat, scale, nlevels, ini, mn), lap


def _frames(cfg):
    """DISTINCT_FRAMES seeded frames; frame 1 has saturated and dark 4-px borders (REFLECT_101 of the blur, FAST at the rim)."""
    cid, w, h = cfg[:3]
    seed0 = 40000 + 100 * [c[0] for c in CONFIGS].index(cid)
    frames = np.stack([synth_frame(seed0 + i, w, h) for i in range(DISTINCT_FRAMES)])
    frames[1, :, :4] = 255
    frames[1, :, -4:] = 7
    frames[1, :4] = 200
    frames[1, -4:] = 31
    if cfg[9]:
        frames = (frames // 4 + 96).astype(np.uint8)
    return frames


_ORACLE_CACHE = {}


def _oracle_results(oracle, cfg):
    """Frames of a configuration and the oracle's outputs for each of them (computed once per configuration)."""
    if cfg[0] not in _ORACLE_CACHE:
        w, h, params, lap = _params(cfg)
        frames = _frames(cfg)
        orc = oracle.OracleExtractor(*params)
        _ORACLE_CACHE[cfg[0]] = (frames, [orc(f, lap) for f in frames])
    return _ORACLE_CACHE[cfg[0]]


def _order(nframes):
    """Distinct frame of every batch position: the distinct frames cycled in an order that depends on the batch size, so that
    each frame lands at several positions (first and last of a batch and of its chunks included)."""
    perm = np.random.default_rng(nframes).permutation(DISTINCT_FRAMES)
    return [int(perm[i % DISTINCT_FRAMES]) for i in range(nframes)]


def _chunks(nframes, chunk_frames=128):
    """Frames per chunk of a host batch: the split of vsg_api.cu's extract_batch_host."""
    min_chunk = min(chunk_frames, 64)
    if nframes < 2 * min_chunk:
        return [nframes]
    nchunks = max(2, (nframes + chunk_frames - 1) // chunk_frames)
    chunk = (nframes + nchunks - 1) // nchunks
    return [min(chunk, nframes - f0) for f0 in range(0, nframes, chunk)]


def _has_pyramid_tiles(cfg):
    """Whether configure_shape sets up the one-launch pyramid: at least two levels, and a top level of at least 2 x 12 pixels
    per side for the 12 x 12 tile grid.  (The tiles' other limits, 160 KB of shared memory and regions of at most 256 pixels
    per side, are far above what frames of up to 1280 x 720 need; the smallest top level here is about 100 pixels.)"""
    _, w, h, _, scale, nlevels = cfg[:6]
    top = scale ** (nlevels - 1)
    return nlevels >= 2 and round(w / top) >= 24 and round(h / top) >= 24


def _pipeline_launches(cfg, nf, lapping):
    """Kernel launches run_pipeline counts (count_launch) for one launch of nf frames."""
    nlevels = cfg[5]
    n = 1 if _has_pyramid_tiles(cfg) and nf <= PYR_TILE_MAX_FRAMES else nlevels - 1   # pyramid_tile_kernel / one per level
    n += 1                                                                             # FAST (with the blur below 16 frames)
    n += 1                                                                             # oct-tree
    n += 1 if nf >= LARGE_BATCH_MIN_FRAMES and nlevels <= BLUR_TC_MAX_LEVELS else 0    # blur_tc_kernel
    n += 2 if lapping != (0, 0) else 1                                                 # slot_kernel + describe
    return n


def _regime(cfg, nf):
    nlevels = cfg[5]
    small = nf <= PDL_MAX_FRAMES
    parts = ["%d frames" % nf, "PDL, octree<512>, describe<16>" if small else "octree<256>, describe<64>"]
    if nlevels > 1:
        if _has_pyramid_tiles(cfg) and nf <= PYR_TILE_MAX_FRAMES:
            parts.append("one-launch pyramid")
        else:
            parts.append("TMA resize" if nf >= LARGE_BATCH_MIN_FRAMES else "level-by-level resize")
    parts.append("tensor-core blur" if nf >= LARGE_BATCH_MIN_FRAMES and nlevels <= BLUR_TC_MAX_LEVELS else "fused FAST + blur")
    return ", ".join(parts)


def _check_output(got, want, what):
    _compare_outputs(got, want, what)
    # stronger than the bars: angles and descriptors have been bit-exact on every frame so far
    da = np.flatnonzero(got[1]["angle"] != want[1]["angle"])
    assert len(da) == 0, "%s: %d angles differ from the oracle's, first at keypoint %d" % (what, len(da), da[0])
    dd = np.flatnonzero((got[2] != want[2]).any(1))
    assert len(dd) == 0, "%s: %d descriptors differ from the oracle's, first at keypoint %d" % (what, len(dd), dd[0])


def _check_taps(ex, orc, image, frame, lap, nlevels, what):
    """Every level of batch position `frame` against the oracle's taps, in pipeline order; names the first stage that differs."""
    orc(image, lap)                         # the oracle keeps the taps of its last call only

    def level_kps(level):
        lk = orc.level_keypoints(level)
        return np.stack([lk["x"], lk["y"], lk["response"]], 1).astype(np.int32) if len(lk) else np.zeros((0, 3), np.int32)

    stages = [
        ("pyramid", lambda l: (ex.pyramid_level(l, frame=frame), orc.level(l))),
        ("blurred level", lambda l: (ex.blurred_level(l, frame=frame), orc.blurred(l))),
        ("FAST candidates", lambda l: (ex.candidates(l, frame=frame).astype(np.float32), orc.candidates(l))),
        ("oct-tree keypoints", lambda l: (ex.level_keypoints(l, frame=frame), level_kps(l))),
    ]
    for stage, get in stages:
        for level in range(nlevels):
            got, want = get(level)
            if want is None:                # the reference blurs only levels that kept keypoints
                continue
            if got.shape != want.shape or not np.array_equal(got, want):
                raise AssertionError("%s: stage '%s' diverges first, at level %d of batch frame %d (shapes %s vs %s)" % (
                    what, stage, level, frame, got.shape, want.shape))


@pytest.fixture
def default_knobs(monkeypatch):
    """The kernel choices under test are the defaults: clear the environment overrides of the thresholds."""
    for k in ("VSG_PYR_TILE", "VSG_RESIZE_TMA", "VSG_BLUR_TC", "VSG_CHUNK_FRAMES"):
        monkeypatch.delenv(k, raising=False)
    return monkeypatch


def _run_batch(oracle, cfg, nframes, chunk_frames=None):
    from visual_sgraphs_b200 import _lib
    from visual_sgraphs_b200.extractor import ORBextractor
    w, h, params, lap = _params(cfg)
    frames, want = _oracle_results(oracle, cfg)
    order = _order(nframes)
    batch = np.ascontiguousarray(frames[order])
    chunks = _chunks(nframes, chunk_frames or 128)
    ex = ORBextractor(*params, max_batch=nframes)
    L = _lib.load()
    ex.max_keypoints(w, h)                  # configure the shape outside the counted window (it launches nothing either way)
    before = L.vsg_launch_count()
    res = ex.extract_batch(batch, lapping=lap)
    launched = L.vsg_launch_count() - before
    what = "%s, %s" % (cfg[0], _regime(cfg, nframes) if len(chunks) == 1 else "%d frames in chunks of %s on three streams, each %s"
                       % (nframes, chunks, _regime(cfg, min(chunks)).split(", ", 1)[1]))
    expect = sum(_pipeline_launches(cfg, nf, lap) for nf in chunks)
    assert launched == expect, "%s: %d kernel launches, the regime implies %d" % (what, launched, expect)
    return ex, batch, order, chunks, res, want, lap, what


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
@pytest.mark.parametrize("nframes", BATCH_SIZES)
def test_every_frame_of_a_batch_matches_the_oracle(oracle, default_knobs, cfg, nframes):
    ex, batch, order, chunks, res, want, lap, what = _run_batch(oracle, cfg, nframes)
    assert chunks == [nframes]
    if nframes in (9, 17):
        _check_taps(ex, oracle.OracleExtractor(*_params(cfg)[2]), batch[-1], nframes - 1, lap, cfg[5], what)
    for f, k in enumerate(order):
        _check_output(res[f], want[k], "%s: batch frame %d (distinct frame %d)" % (what, f, k))


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_chunked_batch_matches_the_oracle(oracle, default_knobs, cfg):
    """58 frames with VSG_CHUNK_FRAMES=20: chunks of 20, 20 and 18 frames on three streams, each at its own frame offset, all
    on the large-batch kernels."""
    default_knobs.setenv("VSG_CHUNK_FRAMES", str(CHUNK_FRAMES))     # read when the handle is created
    ex, batch, order, chunks, res, want, lap, what = _run_batch(oracle, cfg, CHUNKED_BATCH, CHUNK_FRAMES)
    assert chunks == [20, 20, 18]
    assert min(chunks) >= LARGE_BATCH_MIN_FRAMES, "a chunk below the large-batch threshold makes this test vacuous"
    orc = oracle.OracleExtractor(*_params(cfg)[2])
    for last in np.cumsum(chunks) - 1:
        _check_taps(ex, orc, batch[last], int(last), lap, cfg[5], what)
    for f, k in enumerate(order):
        _check_output(res[f], want[k], "%s: batch frame %d (distinct frame %d)" % (what, f, k))


def _by_name(name):
    return next(c for c in CONFIGS if c[0] == name)


def test_device_resident_batch_matches_the_host_path(oracle, default_knobs):
    """vsg_extract_batch_dev (never chunked) at the large-batch kernels, with lapping: the same bytes as the host path."""
    torch = pytest.importorskip("torch")
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE
    from visual_sgraphs_b200.extractor import ORBextractor
    cfg = _by_name("lapping_752x480")
    w, h, params, lap = _params(cfg)
    ex, batch, order, _, res, want, _, what = _run_batch(oracle, cfg, 17)
    for f, k in enumerate(order):
        _check_output(res[f], want[k], "%s: host batch frame %d" % (what, f))
    dex = ORBextractor(*params, max_batch=17)
    cap = dex.max_keypoints(w, h)
    d_frames = torch.from_numpy(batch).cuda()
    kd = torch.zeros((17, cap, 28), dtype=torch.uint8, device="cuda")
    dd = torch.zeros((17, cap, 32), dtype=torch.uint8, device="cuda")
    nd = torch.zeros(17, dtype=torch.int32, device="cuda")
    md = torch.zeros(17, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    dex.extract_batch_dev(d_frames, kd, dd, nd, md, lapping=lap)
    dex.sync()
    n, mono, kn, dn = nd.cpu().numpy(), md.cpu().numpy(), kd.cpu().numpy(), dd.cpu().numpy()
    for f in range(17):
        m, k, d = res[f]
        got_k = kn[f, :n[f]].copy().view(KEYPOINT_DTYPE).reshape(-1)
        assert mono[f] == m and got_k.tobytes() == k.tobytes() and np.array_equal(dn[f, :n[f]], d), "device path, frame %d" % f


def test_colour_batch_matches_the_gray_path(oracle, default_knobs):
    """vsg_extract_batch_color at the large-batch kernels: cvtColor on the device, then the same pipeline as gray frames
    converted by the oracle."""
    from visual_sgraphs_b200 import _lib
    from visual_sgraphs_b200.extractor import ORBextractor
    cfg = _by_name("kitti_1241x376")
    w, h, params, lap = _params(cfg)
    frames, _ = _oracle_results(oracle, cfg)
    rng = np.random.default_rng(31)
    order = _order(17)
    col = np.empty((17, h, w, 3), np.uint8)
    for c in range(3):
        col[..., c] = np.clip(frames[order].astype(np.int16) + rng.integers(-20, 21, (17, h, w)), 0, 255)
    ex = ORBextractor(*params, max_batch=17)
    ex.max_keypoints(w, h)
    L = _lib.load()
    before = L.vsg_launch_count()
    got = ex.extract_batch_color(col, rgb=True)
    assert L.vsg_launch_count() - before == _pipeline_launches(cfg, 17, lap) + 1      # + cvt_gray_kernel
    gray = np.stack([oracle.cvt_gray(col[f], True) for f in range(17)])
    ref = ORBextractor(*params, max_batch=17).extract_batch(gray)
    orc = oracle.OracleExtractor(*params)
    for f in range(17):
        assert got[f][0] == ref[f][0] and got[f][1].tobytes() == ref[f][1].tobytes() and np.array_equal(got[f][2], ref[f][2]), f
        assert np.array_equal(ex.pyramid_level(0, frame=f), gray[f])
    for f in (0, 16):
        _check_output(got[f], orc(gray[f]), "colour batch frame %d" % f)


# ---- oct-tree quotas and shared memory ----------------------------------------------------------------------------------
# octree_kernel keeps the node lists of a level in shared memory (csrc/octree.cu: octree_smem_bytes): 68 bytes per node slot,
# slots = (max(quota, 4 nIni) + 8) rounded up to a multiple of 4, plus 64 bytes, plus the kernel's static shared arrays.


def _octree_dynamic_smem(quota, n_ini):
    cap = (max(quota, 4 * n_ini) + 8 + 3) & ~3
    return cap * 68 + 64


_SMEM_MSG = re.compile(r"level (\d+): oct-tree quota (\d+) needs (\d+) bytes of shared memory per block, the device allows (\d+)")


def _rejected(params, frame):
    from visual_sgraphs_b200 import _lib
    from visual_sgraphs_b200._lib import VSG_ERR_INVALID, VsgError
    from visual_sgraphs_b200.extractor import ORBextractor
    ex = ORBextractor(*params)
    before = _lib.load().vsg_launch_count()
    with pytest.raises(VsgError) as e:
        ex(frame)
    assert e.value.status == VSG_ERR_INVALID, str(e.value)
    m = _SMEM_MSG.search(str(e.value))
    assert m, str(e.value)
    with pytest.raises(VsgError) as again:      # the handle stays rejected, with the same error
        ex(frame)
    assert again.value.status == VSG_ERR_INVALID and str(again.value) == str(e.value)
    assert _lib.load().vsg_launch_count() == before, "a rejected configuration launched kernels"
    return tuple(int(v) for v in m.groups())


def test_octree_quota_limit_of_shared_memory(oracle):
    torch = pytest.importorskip("torch")
    from visual_sgraphs_b200.extractor import ORBextractor
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    frame = synth_frame(46000, 640, 480)
    # two levels of 7000 features: the level-0 quota (3818) alone needs more than a block may have
    params = (7000, float(np.float32(1.2)), 2, 20, 7)
    quota0 = int(oracle.OracleExtractor(*params).tables()["quota"][0])
    level, quota, need, allowed = _rejected(params, frame)
    assert (level, quota, allowed) == (0, quota0, optin)
    static = need - _octree_dynamic_smem(quota0, 1)
    assert 0 <= static < 48 * 1024, static
    # two levels of 6000 features (level-0 quota 3273) fit
    six = (6000, float(np.float32(1.2)), 2, 20, 7)
    assert _octree_dynamic_smem(int(oracle.OracleExtractor(*six).tables()["quota"][0]), 1) + static <= optin
    _check_output(ORBextractor(*six)(frame), oracle.OracleExtractor(*six)(frame), "2 levels, 6000 features")
    # one level at 640x480 (nIni = 1): the largest quota that fits is accepted and extracts exactly like the oracle, with
    # either block size of the oct-tree
    qmax = max(q for q in range(1, 8192) if _octree_dynamic_smem(q, 1) + static <= optin)
    one = (qmax, float(np.float32(1.2)), 1, 20, 7)
    want = oracle.OracleExtractor(*one)(frame)
    assert len(want[1]) > 0.9 * qmax
    _check_output(ORBextractor(*one)(frame), want, "nfeatures %d (the largest that fits), 1 frame" % qmax)
    batch = np.stack([frame] * 9)
    for f, got in enumerate(ORBextractor(*one, max_batch=9).extract_batch(batch)):
        _check_output(got, want, "nfeatures %d (the largest that fits), frame %d of 9" % (qmax, f))
    level, quota, need, allowed = _rejected((qmax + 1,) + one[1:], frame)
    assert (level, quota, need) == (0, qmax + 1, _octree_dynamic_smem(qmax + 1, 1) + static) and need > allowed == optin
    # a handle created afterwards in the same process is unaffected
    _check_output(ORBextractor(1000, float(np.float32(1.2)), 8, 20, 7)(frame), oracle.OracleExtractor(1000)(frame), "default handle")
