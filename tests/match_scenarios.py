"""Synthetic matcher scenarios shared by the CPU and GPU matcher tests: two related frames extracted by the
oracle (frame B = frame A shifted, plus noise) flattened into the view structs the Search* methods read."""
import numpy as np

from visual_sgraphs_b200._lib import PROJ_POINT_DTYPE, TRACK_POINT_DTYPE
from visual_sgraphs_b200.frame import FrameData
from visual_sgraphs_b200.synth import synth_frame

_cache = {}


def two_frames(oracle, seed=11, shift=(9, 5), size=(640, 480), nfeat=1000, scale=1.2, nlevels=8):
    key = (seed, shift, size, nfeat, scale, nlevels)
    if key not in _cache:
        a = synth_frame(seed, *size)
        rng = np.random.default_rng(seed + 1)
        b = np.roll(a, (shift[1], shift[0]), (0, 1))
        b = np.clip(b.astype(np.int16) + rng.integers(-3, 4, b.shape), 0, 255).astype(np.uint8)
        ex = oracle.OracleExtractor(nfeat, scale, nlevels)
        _, ka, da = ex(a)
        _, kb, db = ex(b)
        _cache[key] = (ka, da, kb, db)
    return _cache[key]


def scale_factors(oracle, scale=1.2, nlevels=8):
    """mvScaleFactors of an extractor with this pyramid (the table Frame copies from its ORBextractor)."""
    return oracle.OracleExtractor(1000, scale, nlevels).tables()["scale"]


def frame_data(keys, desc, size=(640, 480), stereo_seed=None, bounds=None, scale_factors=None):
    u_right = None
    if stereo_seed is not None:
        rng = np.random.default_rng(stereo_seed)
        disp = rng.uniform(2, 40, len(keys)).astype(np.float32)
        u_right = np.where(rng.random(len(keys)) < 0.7, keys["x"] - disp, -1).astype(np.float32)
    return FrameData(keys, desc, u_right=u_right, bounds=bounds, scale_factors=scale_factors, width=size[0], height=size[1])


def track_points(fd_target, kb, db, shift, seed, stereo=False, nlevels=8):
    """Map points seen in frame B, projected into frame A (the Frame being searched)."""
    rng = np.random.default_rng(seed)
    n = len(kb)
    pts = np.zeros(n, TRACK_POINT_DTYPE)
    pts["proj_x"] = kb["x"] - shift[0] + rng.normal(0, 1.5, n)
    pts["proj_y"] = kb["y"] - shift[1] + rng.normal(0, 1.5, n)
    pts["proj_xr"] = pts["proj_x"] - rng.uniform(2, 40, n) if stereo else 0
    pts["view_cos"] = rng.uniform(0.99, 1.0, n)
    pts["depth"] = rng.uniform(1, 80, n)
    pts["level"] = np.clip(kb["octave"] + rng.integers(-1, 2, n), 0, nlevels - 1)
    pts["in_view"] = rng.random(n) < 0.9
    pts["bad"] = rng.random(n) < 0.03
    pts["blocks"] = rng.random(n) < 0.9
    occupied = (rng.random(fd_target.n) < 0.1).astype(np.uint8)
    order = rng.permutation(n)            # map points are not sorted like keypoints
    return pts[order].copy(), db[order].copy(), occupied


def proj_points(fd_cur, kb, db, shift, seed, size=(640, 480)):
    rng = np.random.default_rng(seed)
    n = len(kb)
    pts = np.zeros(n, PROJ_POINT_DTYPE)
    pts["u"] = kb["x"] - shift[0] + rng.normal(0, 1.0, n)
    pts["v"] = kb["y"] - shift[1] + rng.normal(0, 1.0, n)
    pts["ur"] = pts["u"] - rng.uniform(2, 40, n)
    pts["angle"] = kb["angle"]
    pts["octave"] = kb["octave"]
    inside = (pts["u"] >= 0) & (pts["u"] <= size[0]) & (pts["v"] >= 0) & (pts["v"] <= size[1])
    pts["valid"] = inside & (rng.random(n) < 0.9)
    pts["blocks"] = rng.random(n) < 0.9
    occupied = (rng.random(fd_cur.n) < 0.05).astype(np.uint8)
    return pts, db.copy(), occupied


def feature_vector(desc, nnodes=64):
    """A stand-in for DBoW2::FeatureVector (the vocabulary blob is not in the checkout, SURVEY §8c):
    node id = a hash of the first descriptor byte; CSR lists in increasing feature index like DBoW2 builds them."""
    node = (desc[:, 0].astype(np.int32) * 7 + 3) % nnodes
    nodes = np.unique(node)
    ptr = [0]
    idx = []
    for nd in nodes:
        members = np.nonzero(node == nd)[0]
        idx.extend(members.tolist())
        ptr.append(len(idx))
    return nodes.astype(np.int32), np.array(ptr, np.int32), np.array(idx, np.int32)


def search_points(kb, shift, seed, sigma=1.0, size=(640, 480), nlevels=8):
    """Map points observed in frame B (keys kb), projected into frame A by the caller: vsg_search_point records."""
    from visual_sgraphs_b200._lib import SEARCH_POINT_DTYPE
    rng = np.random.default_rng(seed)
    n = len(kb)
    pts = np.zeros(n, SEARCH_POINT_DTYPE)
    pts["u"] = kb["x"] - shift[0] + rng.normal(0, sigma, n)
    pts["v"] = kb["y"] - shift[1] + rng.normal(0, sigma, n)
    pts["ur"] = pts["u"] - rng.uniform(2, 40, n)
    pts["angle"] = kb["angle"]
    pts["level"] = np.clip(kb["octave"] + rng.integers(-1, 2, n), 0, nlevels - 1)
    inside = (pts["u"] >= 0) & (pts["u"] < size[0]) & (pts["v"] >= 0) & (pts["v"] < size[1])
    pts["valid"] = inside & (rng.random(n) < 0.9)
    return pts


def sigma_tables():
    s = [np.float32(1.0)]
    for _ in range(7):
        s.append(np.float32(float(s[-1]) * float(np.float32(1.2))))
    scale = np.array(s, np.float32)
    sigma2 = (scale * scale).astype(np.float32)
    return scale, sigma2, (np.float32(1.0) / sigma2).astype(np.float32)


def translation_f12(shift):
    """Fundamental matrix (row-major, Pinhole::epipolarConstrain's F12) of a pure image translation by `shift`:
    the epipolar line of kp1 is the line through kp1 along the shift."""
    sx, sy = float(shift[0]), float(shift[1])
    nrm = np.hypot(sx, sy)
    nx, ny = -sy / nrm, sx / nrm
    return np.array([0, 0, -nx, 0, 0, -ny, nx, ny, 0], np.float32)


def synthetic_vocabulary(seed, k=10, levels=4, prune=0.08):
    """A stand-in for ORBvoc (the blob is not in the checkout): a k-ary tree of depth `levels` whose node descriptors
    are their parent's descriptor with random bit flips (fewer flips deeper down, like k-majority cluster centres).
    A few inner nodes are pruned to leaves so that the tree is unbalanced, like DBoW2's HKmeans can leave it.
    Returns dict(child_ptr, child_idx, node_desc, word_id, weight, levels); node 0 is the root."""
    rng = np.random.default_rng(seed)
    desc = [np.zeros(32, np.uint8)]
    children = [[]]
    depth = [0]
    frontier = [0]
    for lvl in range(1, levels + 1):
        nxt = []
        for parent in frontier:
            if lvl > 1 and rng.random() < prune:
                continue                                   # stays a leaf
            for _ in range(k):
                flips = np.packbits(rng.random(256) < (0.5 if lvl == 1 else 0.25 / lvl))
                desc.append(desc[parent] ^ flips if lvl > 1 else rng.integers(0, 256, 32, dtype=np.uint8))
                children.append([])
                depth.append(lvl)
                children[parent].append(len(desc) - 1)
                nxt.append(len(desc) - 1)
        frontier = nxt
    if len(children[1]) > 2:
        desc[children[1][2]] = desc[children[1][0]].copy()  # equal distances: the first child must win
    child_ptr, child_idx = [0], []
    for c in children:
        child_idx.extend(c)
        child_ptr.append(len(child_idx))
    n = len(desc)
    word_id = np.full(n, -1, np.int64)
    leaves = [i for i in range(n) if not children[i]]
    word_id[leaves] = np.arange(len(leaves))
    weight = np.zeros(n)
    weight[leaves] = rng.uniform(0.2, 8.0, len(leaves))
    weight[leaves[::37]] = 0.0                             # stopped words (weight 0)
    return dict(child_ptr=np.array(child_ptr, np.int32), child_idx=np.array(child_idx, np.int32),
                node_desc=np.stack(desc), word_id=word_id, weight=weight, levels=levels)


def two_camera_scene(oracle, seed=61, size=(640, 480), nfeat=800, scale=1.2, nlevels=8, bounds=None):
    """A two-camera frame (F.Nleft != -1): left / right keypoints are the two related frames of two_frames; map points are
    seen by the left camera, the right camera, or both, with their own projections and predicted levels;
    mvLeftToRightMatch / mvRightToLeftMatch pair up a third of the keypoints.  Returns a dict."""
    ka, da, kb, db = two_frames(oracle, seed=seed, size=size, nfeat=nfeat, scale=scale, nlevels=nlevels)
    sf = None if (scale, nlevels) == (1.2, 8) else scale_factors(oracle, scale, nlevels)
    fl = frame_data(ka, da, size=size, bounds=bounds, scale_factors=sf)
    fr = frame_data(kb, db, size=size, bounds=bounds, scale_factors=sf)
    rng = np.random.default_rng(seed + 7)
    nl, nr = len(ka), len(kb)
    # map points: one per left keypoint and one per right keypoint, each also projected (noisily) into the other camera
    n = nl + nr
    src_left = np.concatenate([np.arange(nl), rng.integers(0, nl, nr)])
    src_right = np.concatenate([rng.integers(0, nr, nl), np.arange(nr)])
    pl, pr = np.zeros(n, TRACK_POINT_DTYPE), np.zeros(n, TRACK_POINT_DTYPE)
    for pts, keys, src in ((pl, ka, src_left), (pr, kb, src_right)):
        pts["proj_x"] = keys["x"][src] + rng.normal(0, 1.5, n)
        pts["proj_y"] = keys["y"][src] + rng.normal(0, 1.5, n)
        pts["view_cos"] = rng.uniform(0.99, 1.0, n)
        pts["level"] = np.clip(keys["octave"][src] + rng.integers(-1, 2, n), 0, nlevels - 1)
    pl["in_view"] = rng.random(n) < 0.7
    pr["in_view"] = rng.random(n) < 0.7
    pr["level"][rng.random(n) < 0.05] = -1                   # mnTrackScaleLevelR == -1 (:149)
    pl["depth"] = rng.uniform(1, 80, n)
    pl["bad"] = rng.random(n) < 0.03
    pl["blocks"] = rng.random(n) < 0.9
    desc = np.where((np.arange(n) < nl)[:, None], da[src_left], db[src_right]).astype(np.uint8)
    flip = rng.random((n, 32)) < 0.02
    desc = desc ^ (flip * rng.integers(1, 256, (n, 32))).astype(np.uint8)
    l2r, r2l = np.full(nl, -1, np.int32), np.full(nr, -1, np.int32)
    pairs = min(nl, nr) // 3
    li, ri = rng.permutation(nl)[:pairs], rng.permutation(nr)[:pairs]
    l2r[li], r2l[ri] = ri, li
    occupied = (rng.random(nl + nr) < 0.1).astype(np.uint8)
    order = rng.permutation(n)
    return dict(fl=fl, fr=fr, pl=pl[order].copy(), pr=pr[order].copy(), desc=desc[order].copy(), l2r=l2r, r2l=r2l,
                occupied=occupied)


def two_camera_last_scene(oracle, seed=61, size=(640, 480), nfeat=800, scale=1.2, nlevels=8, bounds=None):
    """SearchByProjection(Cur, Last) with a two-camera current frame: every last-frame point comes with its projection
    into the left camera (near a left keypoint) and into the right camera (near a right keypoint or far off)."""
    ka, da, kb, db = two_frames(oracle, seed=seed, size=size, nfeat=nfeat, scale=scale, nlevels=nlevels)
    sf = None if (scale, nlevels) == (1.2, 8) else scale_factors(oracle, scale, nlevels)
    fl = frame_data(ka, da, size=size, bounds=bounds, scale_factors=sf)
    fr = frame_data(kb, db, size=size, bounds=bounds, scale_factors=sf)
    rng = np.random.default_rng(seed + 11)
    nl, nr = len(ka), len(kb)
    n = nl + nr
    src_l = np.concatenate([np.arange(nl), rng.integers(0, nl, nr)])
    src_r = np.concatenate([rng.integers(0, nr, nl), np.arange(nr)])
    pl, pr = np.zeros(n, PROJ_POINT_DTYPE), np.zeros(n, PROJ_POINT_DTYPE)
    pl["u"] = ka["x"][src_l] + rng.normal(0, 1.0, n)
    pl["v"] = ka["y"][src_l] + rng.normal(0, 1.0, n)
    pr["u"] = kb["x"][src_r] + rng.normal(0, 1.0, n)
    pr["v"] = kb["y"][src_r] + rng.normal(0, 1.0, n)
    far = rng.random(n) < 0.1                                 # the right projection may land outside the image
    pr["u"][far] += size[0] + 260
    lonely = rng.random(n) < 0.1                              # ... and the left window may be empty (skips the right search)
    pl["u"][lonely] = -200
    from_left = np.arange(n) < nl
    pl["angle"] = np.where(from_left, ka["angle"][src_l], kb["angle"][src_r])
    pl["octave"] = np.where(from_left, ka["octave"][src_l], kb["octave"][src_r])
    pl["valid"] = rng.random(n) < 0.9
    pl["blocks"] = rng.random(n) < 0.9
    desc = np.where(from_left[:, None], da[src_l], db[src_r]).astype(np.uint8)
    occupied = (rng.random(nl + nr) < 0.05).astype(np.uint8)
    order = rng.permutation(n)
    return dict(fl=fl, fr=fr, pl=pl[order].copy(), pr=pr[order].copy(), desc=desc[order].copy(), occupied=occupied)
