"""ctypes binding of libvsg_cuda.so (include/vsg_cuda.h).  No compute happens in Python.

The library is built in-tree by `make -C visual_sgraphs_b200/csrc` (or __graft_entry__.build()).
Loading fails loudly if the shared object is missing: there is no CPU fallback.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VSG_LIB_PATH") or os.path.join(_HERE, "libvsg_cuda.so")   # override: kernel-variant experiments

KEYPOINT_DTYPE = np.dtype(
    [("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"), ("octave", "<i4"),
     ("class_id", "<i4")]
)

VSG_OK = 0
VSG_ERR_INVALID = -1
VSG_ERR_CUDA = -2
VSG_ERR_CAPACITY = -3
VSG_EMPTY_IMAGE = -10


class OrbParams(C.Structure):
    _fields_ = [("nfeatures", C.c_int32), ("scale_factor", C.c_float), ("nlevels", C.c_int32),
                ("ini_th_fast", C.c_int32), ("min_th_fast", C.c_int32)]


class FrameView(C.Structure):
    """vsg_frame_view (include/vsg_cuda.h)."""
    _fields_ = [("n", C.c_int32), ("keys", C.c_void_p), ("descriptors", C.c_void_p), ("u_right", C.c_void_p),
                ("min_x", C.c_float), ("min_y", C.c_float), ("max_x", C.c_float), ("max_y", C.c_float),
                ("grid_inv_w", C.c_float), ("grid_inv_h", C.c_float), ("grid_cols", C.c_int32),
                ("grid_rows", C.c_int32), ("scale_factors", C.c_void_p), ("n_levels", C.c_int32)]


class BowSide(C.Structure):
    """vsg_bow_side (include/vsg_cuda.h): a view, its map-point flags and its flattened FeatureVector."""
    _fields_ = [("view", FrameView), ("mp_valid", C.c_void_p), ("nnodes", C.c_int32), ("nodes", C.c_void_p),
                ("ptr", C.c_void_p), ("idx", C.c_void_p)]


class TriangulationTarget(C.Structure):
    """vsg_triangulation_target (include/vsg_cuda.h): keyframe 2 of SearchForTriangulation with its F12, epipole and
    level variances."""
    _fields_ = [("kf2", BowSide), ("f12", C.c_float * 9), ("ep", C.c_float * 2), ("level_sigma2", C.c_void_p)]


TRACK_POINT_DTYPE = np.dtype([("proj_x", "<f4"), ("proj_y", "<f4"), ("proj_xr", "<f4"), ("view_cos", "<f4"),
                              ("depth", "<f4"), ("level", "<i4"), ("in_view", "u1"), ("bad", "u1"), ("blocks", "u1"),
                              ("pad", "u1")])
PROJ_POINT_DTYPE = np.dtype([("u", "<f4"), ("v", "<f4"), ("ur", "<f4"), ("angle", "<f4"), ("octave", "<i4"),
                             ("valid", "u1"), ("blocks", "u1"), ("pad", "u1", 2)])
SEARCH_POINT_DTYPE = np.dtype([("u", "<f4"), ("v", "<f4"), ("ur", "<f4"), ("angle", "<f4"), ("level", "<i4"),
                               ("valid", "u1"), ("pad", "u1", 3)])
assert TRACK_POINT_DTYPE.itemsize == 28 and PROJ_POINT_DTYPE.itemsize == 24 and SEARCH_POINT_DTYPE.itemsize == 24


class VsgError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("vsg status %d: %s" % (status, message))
        self.status = status


# every symbol include/vsg_cuda.h declares (tests/test_abi.py checks the header against this table)
_SIGNATURES = {
    "vsg_last_error": (C.c_char_p, []),
    "vsg_device_count": (C.c_int, []),
    "vsg_launch_count": (C.c_int64, []),
    "vsg_extractor_create": (C.c_int, [C.POINTER(OrbParams), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "vsg_extractor_destroy": (None, [C.c_void_p]),
    "vsg_extractor_tables": (C.c_int, [C.c_void_p] + [C.c_void_p] * 5),
    "vsg_extractor_max_keypoints": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "vsg_extract": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                              C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vsg_extract_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_int,
                                    C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "vsg_extract_batch_color": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_int,
                                          C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "vsg_extract_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_size_t,
                                        C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "vsg_extractor_sync": (C.c_int, [C.c_void_p]),
    "vsg_extractor_stream": (C.c_void_p, [C.c_void_p]),
    "vsg_extractor_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "vsg_extractor_stage_ms": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]),
    "vsg_pyramid_level_size": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vsg_pyramid_download": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "vsg_blurred_download": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "vsg_candidates_download": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "vsg_level_keypoints_download": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "vsg_matcher_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "vsg_matcher_destroy": (None, [C.c_void_p]),
    "vsg_matcher_stream": (C.c_void_p, [C.c_void_p]),
    "vsg_matcher_sync": (C.c_int, [C.c_void_p]),
    "vsg_descriptor_distance": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "vsg_knn2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vsg_knn2_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vsg_knn2_merge_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vsg_distinctive_descriptors": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "vsg_knn2_ratio": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "vsg_match_window": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 5),
    "vsg_frame_create": (C.c_int, [C.c_void_p, C.POINTER(FrameView), C.POINTER(C.c_void_p)]),
    "vsg_frame_destroy": (None, [C.c_void_p]),
    "vsg_area_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 9 + [C.c_int, C.POINTER(C.c_int)]),
    "vsg_search_by_projection_last_2cam": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float,
                                                     C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_search_by_projection_map_2cam": (C.c_int, [C.c_void_p] * 6 + [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float,
                                                    C.c_int, C.c_float, C.c_float, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_search_by_projection_map": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                               C.c_float, C.c_int, C.c_float, C.c_float, C.c_void_p,
                                               C.POINTER(C.c_int)]),
    "vsg_projection_map_candidates": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_int,
                                                C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "vsg_projection_map_resolve": (C.c_int, [C.POINTER(FrameView), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_float, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_comm_unique_id": (C.c_int, [C.c_void_p]),
    "vsg_comm_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "vsg_comm_destroy": (None, [C.c_void_p]),
    "vsg_comm_rank": (C.c_int, [C.c_void_p]),
    "vsg_comm_size": (C.c_int, [C.c_void_p]),
    "vsg_comm_nccl_version": (C.c_int, []),
    "vsg_knn2_sharded": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                   C.c_void_p]),
    "vsg_search_by_projection_map_sharded": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                                       C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_float, C.c_float,
                                                       C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_projection_map_resolve_shard": (C.c_int, [C.POINTER(FrameView), C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_search_by_projection_last": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                                C.c_float, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_search_for_initialization": (C.c_int, [C.c_void_p, C.POINTER(FrameView), C.c_void_p, C.c_void_p, C.c_int,
                                                C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_search_by_bow": (C.c_int, [C.c_void_p, C.POINTER(FrameView), C.c_void_p, C.POINTER(FrameView), C.c_int,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_search_by_bow_2cam": (C.c_int, [C.c_void_p, C.POINTER(FrameView), C.c_void_p, C.POINTER(FrameView), C.c_int, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_search_by_bow_multi": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(BowSide), C.c_int, C.c_float, C.c_int,
                                          C.c_void_p, C.c_void_p]),
    "vsg_search_by_projection_reloc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                                 C.c_float, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_search_by_projection_sim3": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                                C.c_int, C.c_float, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_fuse_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p,
                                  C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_fuse_search_multi": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                        C.c_float, C.c_void_p]),
    "vsg_fuse_search_sim3_multi": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float,
                                             C.c_void_p]),
    "vsg_search_by_sim3": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                     C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_search_by_bow_kf": (C.c_int, [C.c_void_p, C.POINTER(FrameView), C.c_void_p, C.POINTER(FrameView), C.c_void_p,
                                       C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_search_by_bow_kf_multi": (C.c_int, [C.c_void_p, C.POINTER(BowSide), C.c_int, C.c_void_p, C.c_float, C.c_int,
                                             C.c_void_p, C.c_void_p]),
    "vsg_bow_pair_distances": (C.c_int, [C.c_void_p, C.POINTER(FrameView), C.c_void_p, C.POINTER(FrameView), C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int),
                                         C.POINTER(C.c_int)]),
    "vsg_search_for_triangulation": (C.c_int, [C.c_void_p, C.POINTER(FrameView), C.c_void_p, C.POINTER(FrameView),
                                               C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_triangulation_candidates_multi": (C.c_int, [C.c_void_p, C.POINTER(BowSide), C.c_int, C.c_void_p, C.c_int, C.c_int,
                                                     C.c_void_p]),
    "vsg_triangulation_resolve": (C.c_int, [C.POINTER(FrameView), C.POINTER(FrameView), C.c_void_p, C.c_void_p, C.c_int,
                                            C.c_void_p, C.POINTER(C.c_int)]),
    "vsg_vocabulary_create": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                        C.POINTER(C.c_void_p)]),
    "vsg_vocabulary_destroy": (None, [C.c_void_p]),
    "vsg_bow_transform": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vsg_extractor_set_rectify_map": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "vsg_extract_batch_rectify": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_int,
                                            C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "vsg_undistort_keypoints": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p] + [C.c_double] * 4 + [C.c_void_p, C.c_int, C.c_void_p]),
    "vsg_undistort_keypoints_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int] + [C.c_double] * 4 +
                                      [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "vsg_stereo_match_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_int]),
    "vsg_stereo_match": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p]),
}

_lib = None


def load():
    """Loads libvsg_cuda.so; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libvsg_cuda.so is not built (%s). Run `make -C visual_sgraphs_b200/csrc` or "
                "`python -c 'import __graft_entry__ as g; g.build()'`. There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status):
    if status != VSG_OK:
        raise VsgError(status, load().vsg_last_error().decode("utf-8", "replace"))


def ptr(a):
    """void* of a numpy array, a torch tensor (data_ptr) or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    raise TypeError(type(a))
