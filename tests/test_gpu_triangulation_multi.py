"""vsg_triangulation_candidates_multi + vsg_triangulation_resolve (ORBmatcher.SearchForTriangulationMulti /
ResolveTriangulation) and the batch form of the shim's SearchForTriangulation, on the B200 (-m gpu).

One call searches a keyframe against all its neighbours (LocalMapping::CreateNewMapPoints); a resolve per neighbour gives
SearchForTriangulation's result with KF1's map points as they are at that moment.  Every resolve must equal
vsg_search_for_triangulation on that target with the same map-point flags and the CPU oracle's search_for_triangulation.
The targets differ in keypoint count (including none), stereo or monocular, pyramid, a feature vector that shares no node
with KF1, all map-point flags set, F12 direction and an epipole among the keypoints; the same keyframe appears twice.
Planted pairs pin the tie rule, the TH_LOW bound, the epipole gate's boundary and the float / double arithmetic of the
3.84 sigma^2 gate.  tests/cpp/triangulation_multi_test.cpp checks the shim's batch form against the loop.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import match_scenarios as sc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.abspath(__file__ + "/.."))
NODES = 24
F32 = np.float32
# pyramid id: (scale factor, levels)
PYRAMIDS = {"default": (1.2, 8), "fine": (1.1, 12), "coarse": (1.5, 5)}
# target kinds: (pyramid, keypoints "all" / "half" / "none", stereo, map points "some" / "all", feature vector "same" /
# "disjoint", image shift of the F12, epipole "far" / "among")
KINDS = [
    ("default", "all", False, "some", "same", (9, 1), "far"),
    ("default", "all", True, "some", "same", (9, 1), "among"),
    ("fine", "all", False, "some", "same", (1, 9), "among"),
    ("coarse", "half", True, "some", "same", (-6, 4), "far"),
    ("default", "none", False, "some", "same", (9, 1), "far"),
    ("default", "all", False, "all", "same", (9, 1), "far"),
    ("default", "all", True, "some", "disjoint", (9, 1), "far"),
    ("default", "half", False, "some", "same", (5, -5), "among"),
]


def _matcher(check_ori=True):
    from visual_sgraphs_b200.matcher import ORBmatcher
    return ORBmatcher(0.6, check_ori)


def _launches():
    from visual_sgraphs_b200 import _lib
    return _lib.load().vsg_launch_count()


@pytest.fixture(scope="module")
def scenes(oracle):
    out = {}
    for pid, (scale, nlevels) in PYRAMIDS.items():
        ka, da, kb, db = sc.two_frames(oracle, shift=(9, 1), scale=scale, nlevels=nlevels)
        sf = np.asarray(sc.scale_factors(oracle, scale, nlevels), F32)
        out[pid] = (ka, da, kb, db, sf, (sf * sf).astype(F32))
    return out


def _featvec(desc, disjoint=False):
    nodes, ptr, idx = sc.feature_vector(desc, NODES)
    return (nodes + 1000 if disjoint else nodes).astype(np.int32), ptr, idx


def _kf1(scenes, stereo, seed=5):
    ka, da, _, _, sf, _ = scenes["default"]
    k1 = sc.frame_data(ka, da, stereo_seed=2 if stereo else None, scale_factors=sf)
    h1 = (np.random.default_rng(seed).random(k1.n) < 0.5).astype(np.uint8)
    return k1, h1, _featvec(da)


def make_target(scenes, t, seed):
    """Target t: (kf2 FrameData, has_mp2, feature vector, F12, epipole, level sigma^2)."""
    pid, keep, stereo, mps, fvk, shift, epk = KINDS[t % len(KINDS)]
    _, _, kb, db, sf, sigma2 = scenes[pid]
    rng = np.random.default_rng(seed)
    keys, desc = kb, db
    if keep == "half":
        pick = np.sort(rng.permutation(len(keys))[: len(keys) // 2])
        keys, desc = keys[pick], desc[pick]
    elif keep == "none":
        keys, desc = keys[:0], desc[:0]
    fd = sc.frame_data(keys, desc, stereo_seed=seed if stereo else None, scale_factors=sf)
    h2 = np.ones(fd.n, np.uint8) if mps == "all" else (rng.random(fd.n) < 0.3).astype(np.uint8)
    ep = np.array([320.0, 240.0] if epk == "among" else [-4000.0, 9000.0], F32)
    return fd, h2, _featvec(desc, fvk == "disjoint"), sc.translation_f12(shift), ep, sigma2


def _targets(scenes, ntargets, seed0=100):
    targets = [make_target(scenes, t, seed0 + t) for t in range(ntargets)]
    if ntargets > 1:
        targets[-1] = targets[0]                            # the same keyframe twice
    return targets


def _has_pairs(fv1, use1, fv2):
    n1, p1, i1 = fv1
    n2, p2, i2 = fv2
    for k, node in enumerate(n1):
        j = np.searchsorted(n2, node)
        if j < len(n2) and n2[j] == node and p2[j + 1] > p2[j] and use1[i1[p1[k]:p1[k + 1]]].any():
            return True
    return False


def _single_and_oracle(oracle, m, k1, h1, fv1, tg, only_stereo, coarse, check_ori):
    k2, h2, fv2, f12, ep, sig = tg
    single = m.SearchForTriangulation(k1, h1, k2, h2, fv1, fv2, f12, ep, sig, only_stereo, coarse)
    want = oracle.search_for_triangulation(k1.view, h1, k2.view, h2, fv1, fv2, only_stereo, coarse, f12, ep, sig, check_ori)
    return single, want


def _check(what, got, single, want):
    for name, (nm, m12) in (("the single-target call", single), ("the oracle", want)):
        bad = np.nonzero(got[1] != m12)[0]
        assert not len(bad), "%s: feature %d: resolve %d, %s %d (%d differences)" % (what, bad[0], got[1][bad[0]], name,
                                                                                      m12[bad[0]], len(bad))
        assert got[0] == nm, "%s: %d matches, %s %d" % (what, got[0], name, nm)


@pytest.mark.parametrize("ntargets", [0, 1, 2, 10, 30])
@pytest.mark.parametrize("only_stereo,coarse,check_ori", [(False, False, True), (True, False, False), (False, True, True)])
def test_candidates_and_resolve(oracle, scenes, ntargets, only_stereo, coarse, check_ori):
    k1, h1, fv1 = _kf1(scenes, stereo=True)
    targets = _targets(scenes, ntargets)
    m = _matcher(check_ori)
    before = _launches()
    best = m.SearchForTriangulationMulti(k1, h1, fv1, targets, only_stereo, coarse)
    launches = _launches() - before
    assert best.shape == (ntargets, k1.n)
    stereo1 = k1.u_right >= 0
    use1 = (h1 == 0) & (stereo1 if only_stereo else True)
    assert launches == int(any(_has_pairs(fv1, use1, tg[2]) for tg in targets))
    assert ((best == -2) == h1.astype(bool)[None, :]).all()
    rng = np.random.default_rng(7)
    for mode in ("unchanged", "grown"):
        h_now = h1.copy()
        for t, tg in enumerate(targets):
            before = _launches()
            got = m.ResolveTriangulation(k1, tg[0], h_now, best[t])
            assert _launches() == before                    # the resolve is host code
            single, want = _single_and_oracle(oracle, m, k1, h_now, fv1, tg, only_stereo, coarse, check_ori)
            kind = KINDS[0 if ntargets > 1 and t == ntargets - 1 else t % len(KINDS)]     # the last target is target 0 again
            _check("%d targets, target %d (%s), KF1 map points %s" % (ntargets, t, kind, mode), got, single, want)
            if mode == "grown":                             # the loop's triangulation: matched features gain map points
                h_now[got[1] >= 0] = rng.random(int((got[1] >= 0).sum())) < 0.8
                h_now |= h1
            if kind[1] == "none" or kind[3] == "all" or kind[4] == "disjoint":
                assert got[0] == 0
            elif kind[0] == "default" and kind[1] == "all" and not only_stereo and mode == "unchanged":
                assert got[0] > 10, "target %d (%s): %d matches" % (t, kind, got[0])


@pytest.mark.parametrize("coarse", [False, True])
def test_no_map_points_at_either_call(oracle, scenes, coarse):
    """KF1 without map points at the candidates call and at every resolve: every feature is searched."""
    k1, _, fv1 = _kf1(scenes, stereo=False)
    h1 = np.zeros(k1.n, np.uint8)
    targets = _targets(scenes, 10)
    m = _matcher(True)
    best = m.SearchForTriangulationMulti(k1, h1, fv1, targets, False, coarse)
    assert (best != -2).all()
    for t, tg in enumerate(targets):
        got = m.ResolveTriangulation(k1, tg[0], h1, best[t])
        _check("target %d" % t, got, *_single_and_oracle(oracle, m, k1, h1, fv1, tg, False, coarse, True))


def _planted_kf(keys_xy, desc, octave=0, nlevels=8):
    from visual_sgraphs_b200._lib import KEYPOINT_DTYPE
    n = len(keys_xy)
    k = np.zeros(n, KEYPOINT_DTYPE)
    if n:
        k["x"], k["y"] = np.asarray(keys_xy, F32).T
    k["octave"] = octave
    k["size"] = 31
    sf = np.array([1.2 ** i for i in range(nlevels)], F32)
    return sc.frame_data(k, np.asarray(desc, np.uint8).reshape(n, 32), scale_factors=sf), sf


def _flip(d, nbits, rng):
    d = d.copy()
    for b in rng.choice(256, nbits, replace=False):
        d[b // 8] ^= np.uint8(1 << (b % 8))
    return d


def test_planted_pairs(oracle):
    """Ties go to the last passing candidate, d == TH_LOW passes, the epipole gate is a strict '<' of 100 * scale."""
    rng = np.random.default_rng(21)
    D = rng.integers(0, 256, (5, 32), dtype=np.uint8)
    y = 300.0
    kf1_xy = [(100, y), (150, y), (200, y), (250, y), (260, y)]
    # KF2 in one node with KF1: per KF1 feature, its planted candidates; everything else is ~128 bits away
    kf2 = []
    kf2.append(((400, y), _flip(D[0], 3, rng)))          # 0: tie, first
    kf2.append(((410, y), _flip(D[0], 3, rng)))          # 1: tie, last: wins
    kf2.append(((420, y), _flip(D[1], 2, rng)))          # 2: tie, first: wins
    kf2.append(((430, y + 50), _flip(D[1], 2, rng)))     # 3: tie, last, off the epipolar line
    kf2.append(((440, y), _flip(D[2], 50, rng)))         # 4: d == TH_LOW: accepted
    kf2.append(((310, y), _flip(D[3], 1, rng)))          # 5: exactly 10 px from the epipole: 100 is not < 100, passes
    kf2.append(((309.99, y), _flip(D[4], 1, rng)))       # 6: just inside: rejected
    k1, sf = _planted_kf(kf1_xy, D)
    k2, _ = _planted_kf([p for p, _ in kf2], np.stack([d for _, d in kf2]))
    one = (np.array([0], np.int32), np.array([0, 5], np.int32), np.arange(5, dtype=np.int32))
    two = (np.array([0], np.int32), np.array([0, 7], np.int32), np.arange(7, dtype=np.int32))
    f12, ep, sig = sc.translation_f12((1, 0)), np.array([300.0, y], F32), (sf * sf).astype(F32)
    h1, h2 = np.zeros(5, np.uint8), np.zeros(7, np.uint8)
    m = _matcher(False)
    best = m.SearchForTriangulationMulti(k1, h1, one, [(k2, h2, two, f12, ep, sig)])
    assert list(best[0]) == [1, 2, 4, 5, -1]
    got = m.ResolveTriangulation(k1, k2, h1, best[0])
    _check("planted pairs", got, *_single_and_oracle(oracle, m, k1, h1, one, (k2, h2, two, f12, ep, sig), False, False, False))


def _line(x1, y1, f, fma):
    """Pinhole.cpp:126-128 in float32; fma: x * f[k] + y * f[k + 3] fused, as a contracting compiler would emit it."""
    out = []
    for k in range(3):
        if fma:
            s = F32(np.float64(x1) * np.float64(f[k]) + np.float64(F32(y1 * f[k + 3])))
        else:
            s = F32(F32(x1 * f[k]) + F32(y1 * f[k + 3]))
        out.append(F32(s + f[k + 6]))
    return out


def _accept(a, b, c, x2, y2, s2, double_compare=True):
    num = F32(F32(F32(a * x2) + F32(b * y2)) + c)
    den = F32(F32(a * a) + F32(b * b))
    if den == 0:
        return False
    dsqr = F32(F32(num * num) / den)
    return float(dsqr) < 3.84 * float(s2) if double_compare else dsqr < F32(F32(3.84) * s2)


def _boundary_pairs(seed, want=16):
    """A seeded float32 search for (F12, kp1, kp2, octave) whose 3.84 sigma^2 decision flips when the epipolar line is
    computed with fused multiply-adds or when the gate compares in float."""
    rng = np.random.default_rng(seed)
    sig = np.array([1.2 ** (2 * i) for i in range(8)], F32)
    found = {"fma": [], "float": []}
    for _ in range(20000):
        if min(len(v) for v in found.values()) >= want // 2:
            break
        f = np.concatenate([rng.uniform(-1e-3, 1e-3, 6), rng.uniform(-1, 1, 2), rng.uniform(-300, 300, 1)]).astype(F32)
        f[[2, 5]] = rng.uniform(-1, 1, 2)
        x1, y1 = F32(rng.uniform(20, 620)), F32(rng.uniform(20, 460))
        o = int(rng.integers(0, 8))
        a, b, c = _line(x1, y1, f, False)
        af, bf, cf = _line(x1, y1, f, True)
        if a == 0:
            continue
        y2 = F32(rng.uniform(20, 460))
        den = float(a) * float(a) + float(b) * float(b)
        x0 = (np.sqrt(3.84 * float(sig[o]) * den) * rng.choice([-1, 1]) - float(b) * float(y2) - float(c)) / float(a)
        if not 0 < x0 < 640:
            continue
        x = F32(x0)
        for _ in range(40):
            x = np.nextafter(x, F32(np.inf))
            ref = _accept(a, b, c, x, y2, sig[o])
            if ref != _accept(af, bf, cf, x, y2, sig[o]) and len(found["fma"]) < want // 2:
                found["fma"].append((f, x1, y1, x, y2, o, ref))
            elif ref != _accept(a, b, c, x, y2, sig[o], False) and len(found["float"]) < want // 2:
                found["float"].append((f, x1, y1, x, y2, o, ref))
    return found["fma"] + found["float"], sig


def test_chi_square_boundary(oracle):
    pairs, sig = _boundary_pairs(33)
    assert len(pairs) >= 12, "the search found %d boundary pairs" % len(pairs)
    rng = np.random.default_rng(34)
    n = len(pairs)
    D = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    k1, _ = _planted_kf([(p[1], p[2]) for p in pairs], D)
    h1 = np.zeros(n, np.uint8)
    fv1 = (np.arange(n, dtype=np.int32), np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32))
    targets = []
    for t, (f, _, _, x2, y2, o, _) in enumerate(pairs):     # target t: one keypoint, in KF1 feature t's node, distance 0
        k2, _ = _planted_kf([(x2, y2)], D[t:t + 1], octave=o)
        fv2 = (np.array([t], np.int32), np.array([0, 1], np.int32), np.array([0], np.int32))
        targets.append((k2, np.zeros(1, np.uint8), fv2, f, np.array([-1e4, -1e4], F32), sig))
    m = _matcher(False)
    best = m.SearchForTriangulationMulti(k1, h1, fv1, targets)
    for t, tg in enumerate(targets):
        assert best[t, t] == (0 if pairs[t][6] else -1), "boundary pair %d: %d, the reference decides %s" % (t, best[t, t], pairs[t][6])
        got = m.ResolveTriangulation(k1, tg[0], h1, best[t])
        _check("boundary pair %d" % t, got, *_single_and_oracle(oracle, m, k1, h1, fv1, tg, False, False, False))


def test_rejected_inputs(scenes):
    from visual_sgraphs_b200 import _lib
    from visual_sgraphs_b200._lib import TriangulationTarget
    from visual_sgraphs_b200.matcher import _bow_side
    L = _lib.load()
    m = _matcher(True)
    k1, h1, fv1 = _kf1(scenes, stereo=False)
    targets = _targets(scenes, 4)
    keep = []
    K1 = _bow_side(k1, h1, fv1, keep)

    def tgt(kf2, h2, fv2, f12, ep, sig):
        sig = None if sig is None else np.ascontiguousarray(sig, F32)
        keep.append(sig)
        return TriangulationTarget(_bow_side(kf2, h2, fv2, keep), (C.c_float * 9)(*f12), (C.c_float * 2)(*ep), _lib.ptr(sig))

    out = np.zeros((4, k1.n), np.int32)
    call = lambda tgs, coarse=0: L.vsg_triangulation_candidates_multi(  # noqa: E731
        m._h, C.byref(K1), len(tgs), (C.c_void_p * 4)(*[t and C.addressof(t) for t in tgs]), 0, coarse, _lib.ptr(out))
    good = [tgt(*tg) for tg in targets]
    before = _launches()
    assert call(good[:2] + [None] + good[3:]) == _lib.VSG_ERR_INVALID and b"target 2: null target" in L.vsg_last_error()
    k2, h2, (n2, p2, i2), f12, ep, sig = targets[3]
    bad_ptr = p2.copy()
    bad_ptr[1] = bad_ptr[-1] + 10
    assert call(good[:3] + [tgt(k2, h2, (n2, bad_ptr, i2), f12, ep, sig)]) == _lib.VSG_ERR_INVALID
    assert b"target 3" in L.vsg_last_error() and b"malformed feature vector" in L.vsg_last_error()
    assert call(good[:3] + [tgt(k2, h2, (n2, p2, np.full_like(i2, k2.n + 5)), f12, ep, sig)]) == _lib.VSG_ERR_INVALID
    assert b"target 3" in L.vsg_last_error() and b"out of range" in L.vsg_last_error()
    assert call(good[:1] + [tgt(*targets[1][:5], None)] + good[2:]) == _lib.VSG_ERR_INVALID
    assert b"target 1" in L.vsg_last_error() and b"level_sigma2" in L.vsg_last_error()
    assert call(good[:1] + [tgt(*targets[1][:5], None)] + good[2:], coarse=1) == _lib.VSG_OK   # coarse reads no sigma
    k_bad = sc.frame_data(k2.keys.copy(), k2.descriptors, scale_factors=k2.scale_factors)
    k_bad.keys["octave"][5] = len(k2.scale_factors)                     # the view reads this array
    before = _launches()
    assert call(good[:2] + [tgt(k_bad, h2, (n2, p2, i2), f12, ep, sig)] + good[3:]) == _lib.VSG_ERR_INVALID
    assert b"target 2: keypoint 5: octave" in L.vsg_last_error()
    assert call([]) == _lib.VSG_OK
    assert _launches() == before                            # nothing was launched
    # a -2 feature that lost its map point
    best = m.SearchForTriangulationMulti(k1, h1, fv1, targets)
    lost = h1.copy()
    i = int(np.nonzero(h1)[0][3])
    lost[i] = 0
    with pytest.raises(_lib.VsgError, match="feature %d " % i):
        m.ResolveTriangulation(k1, targets[0][0], lost, best[0])
    # the matcher still works after the rejected calls
    for t, tg in enumerate(targets):
        got = m.ResolveTriangulation(k1, tg[0], h1, best[t])
        single = m.SearchForTriangulation(k1, h1, tg[0], tg[1], fv1, tg[2], tg[3], tg[4], tg[5])
        assert got[0] == single[0] and np.array_equal(got[1], single[1])


def test_cpp_batch_equals_the_loop(tmp_path):
    pkg = os.path.join(ROOT, "visual_sgraphs_b200")
    exe = str(tmp_path / "triangulation_multi_test")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cpp", "triangulation_multi_test.cpp"),
                           "-L" + pkg, "-lvsg_cuda", "-Wl,-rpath," + pkg])
    out = subprocess.run([exe], capture_output=True, text=True)
    print(out.stdout[-3000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert "TRIANGULATION MULTI TEST OK" in out.stdout
