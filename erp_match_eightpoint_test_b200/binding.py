"""ctypes binding of the C ABI declared in include/erp_b200.h.

This is the only way Python reaches the product: every call lands in
``lib/liberp_b200.so`` (hand-written sm_100a CUDA).  There is no CPU fallback and no
import of ``oracle``: if the library is missing or no B200 is visible the call raises.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ERP_B200_LIB") or os.path.join(_HERE, "lib", "liberp_b200.so")

DMATCH = np.dtype([("queryIdx", "<i4"), ("trainIdx", "<i4"), ("imgIdx", "<i4"), ("distance", "<f4")])
POSE_FLOATS = 12

METRIC_ALGEBRAIC, METRIC_SAMPSON, METRIC_ANGULAR = 0, 1, 2
ENGINE_AUTO, ENGINE_EXACT_SIMT, ENGINE_TCGEN05, ENGINE_TCGEN05_1X = 0, 1, 2, 3
OPERANDS_NONE, OPERANDS_TF32, OPERANDS_F16, OPERANDS_I8 = 0, 1, 2, 3

OK = 0
E_ARG, E_DIM, E_TOO_FEW_TRAIN, E_TOO_FEW_POINTS, E_NO_CANDIDATE, E_LIMIT = 1, 2, 3, 4, 5, 6
E_CUDA, E_NO_DEVICE, E_ARCH, E_NCCL = -1, -2, -3, -4
COMM_ID_BYTES = 128


class RansacResult(C.Structure):
    _fields_ = [("packed", C.c_uint64), ("hyp_id", C.c_uint64), ("count", C.c_int32), ("n_refit", C.c_int32),
                ("E_best", C.c_double * 9), ("E_refit", C.c_double * 9), ("pose", C.c_float * POSE_FLOATS)]


class ErpError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"erp_b200 status {status}: {message}")
        self.status = status


_lib = None

# every symbol include/erp_b200.h declares (tests check the export table against the header)
_SIGNATURES = {
    "erp_last_error": (C.c_char_p, []),
    "erp_version": (C.c_int, []),
    "erp_device_count": (C.c_int, []),
    "erp_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "erp_ctx_destroy": (None, [C.c_void_p]),
    "erp_ctx_stream": (C.c_void_p, [C.c_void_p]),
    "erp_ctx_synchronize": (C.c_int, [C.c_void_p]),
    "erp_ctx_set_engine": (C.c_int, [C.c_void_p, C.c_int]),
    "erp_ctx_device": (C.c_int, [C.c_void_p]),
    "erp_ctx_launch_count": (C.c_uint64, [C.c_void_p]),
    "erp_ctx_last_knn_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "erp_ctx_last_knn_operands": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "erp_ctx_last_knn_kernel_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "erp_ctx_last_score_kernel_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "erp_ctx_last_score_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "erp_ctx_last_stage_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "erp_gather_bearings_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int,
                                          C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "erp_knn2_match": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int,
                                 C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "erp_knn2_raw": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int,
                               C.c_void_p, C.c_void_p]),
    "erp_knn2_near_ties": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_float,
                                     C.c_void_p, C.POINTER(C.c_int)]),
    "erp_knn2_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "erp_nn1_reverse_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "erp_match_filter_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "erp_knn2_match_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p]),
    "erp_knn2_match_bin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int,
                                     C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "erp_knn2_raw_bin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int,
                                   C.c_void_p, C.c_void_p]),
    "erp_knn2_bin_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "erp_knn2_match_bin_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p,
                                         C.c_void_p]),
    "erp_pair_pose_bin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_float,
                                    C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int,
                                    C.c_float, C.c_void_p, C.POINTER(C.c_int), C.POINTER(RansacResult), C.c_void_p]),
    "erp_pair_pose_bin_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int,
                                        C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "erp_bearings_from_pixels": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "erp_bearings_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "erp_pack_float4_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "erp_eight_point_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_uint64,
                                        C.c_uint64, C.c_void_p, C.c_void_p]),
    "erp_eight_point_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_uint64,
                                            C.c_uint64, C.c_void_p, C.c_void_p]),
    "erp_philox_samples": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "erp_eight_point_estimation": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "erp_score": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "erp_score_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_uint64,
                                C.c_void_p, C.c_void_p]),
    "erp_inlier_mask": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p,
                                  C.POINTER(C.c_int)]),
    "erp_refit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "erp_ransac": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int,
                             C.c_float, C.POINTER(RansacResult), C.c_void_p]),
    "erp_ransac_pixels": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_uint64, C.c_uint64,
                                    C.c_int, C.c_int, C.c_int, C.c_float, C.POINTER(RansacResult), C.c_void_p]),
    "erp_pair_pose": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_float, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_float,
                                C.c_void_p, C.POINTER(C.c_int), C.POINTER(RansacResult), C.c_void_p]),
    "erp_pair_pose_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int,
                                    C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_float,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "erp_shard_range": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "erp_comm_unique_id": (C.c_int, [C.c_void_p]),
    "erp_comm_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "erp_comm_destroy": (C.c_int, [C.c_void_p]),
    "erp_comm_size": (C.c_int, [C.c_void_p]),
    "erp_comm_rank": (C.c_int, [C.c_void_p]),
    "erp_comm_allreduce_best_dev": (C.c_int, [C.c_void_p, C.c_void_p]),
    "erp_comm_cross_check_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "erp_pair_pose_dist_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int,
                                    C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_float,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "erp_pair_pose_dist": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_float, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_float,
                                C.c_void_p, C.POINTER(C.c_int), C.POINTER(RansacResult), C.c_void_p]),
    "erp_knn2_match_dist": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int,
                                 C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "erp_knn2_match_dist_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p]),
    "erp_group_create": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    "erp_group_destroy": (None, [C.c_void_p]),
    "erp_group_size": (C.c_int, [C.c_void_p]),
    "erp_group_ctx": (C.c_void_p, [C.c_void_p, C.c_int]),
    "erp_group_pair_pose": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_float, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_float,
                                C.c_void_p, C.POINTER(C.c_int), C.POINTER(RansacResult), C.c_void_p]),
    "erp_group_knn2_match": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_size_t, C.c_int,
                                 C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "erp_ransac_local_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64,
                                       C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "erp_ransac_finish_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64,
                                        C.c_int, C.c_int, C.c_float, C.c_void_p, C.POINTER(RansacResult)]),
    "erp_initial_guess": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "erp_find": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_int, C.c_int,
                           C.c_void_p, C.c_void_p]),
    "erp_libstdcxx_sample_table": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_uint, C.c_void_p]),
    "erp_rotate_image": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t]),
    "erp_rotate_image_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t]),
    "erp_crop_rotated_image": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_float, C.c_void_p, C.c_size_t]),
    "erp_crop_rotated_image_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_float, C.c_void_p, C.c_size_t]),
    "erp_rotate_pixels": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "erp_rotate_keypoints": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_int, C.c_int]),
    "erp_rotate_keypoints_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_int, C.c_int]),
    "erp_draw_epipole": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p, C.c_size_t]),
    "erp_draw_epipole_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p, C.c_size_t]),
}


def lib() -> C.CDLL:
    """Loads liberp_b200.so or raises: the product has no other implementation."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m erp_match_eightpoint_test_b200.build` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args
    return _lib


def _check(status: int):
    if status != OK:
        raise ErpError(status, lib().erp_last_error().decode())


def _ptr(a):
    """numpy array -> host pointer; torch tensor / int -> device pointer; None -> NULL."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if isinstance(a, int):
        return a
    return a.data_ptr()


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _f32_rows(a):
    """(n, dim) float32 descriptor rows: (array, row stride)."""
    a = _f32(a)
    return a, (a.strides[0] if a.shape[0] > 1 else 4 * a.shape[1])


def _u8_rows(a):
    """(n, nbytes) uint8 rows whose bytes within a row are contiguous (strided row views stay views): (array, row stride)."""
    a = np.asarray(a)
    if a.dtype != np.uint8 or a.ndim != 2:
        raise ValueError("binary descriptors are (n, nbytes) uint8 arrays")
    if a.strides[1] != 1 or a.strides[0] < a.shape[1]:
        a = np.ascontiguousarray(a)
    return a, (a.strides[0] if a.shape[0] > 1 else a.shape[1])


def libstdcxx_sample_table(m: int, H: int = 80, S: int | None = None, seed: int = 1) -> np.ndarray:
    S = int(m * 0.25) if S is None else S
    t = np.empty((H, S), np.int32)
    _check(lib().erp_libstdcxx_sample_table(m, H, S, seed, _ptr(t)))
    return t


_live = weakref.WeakSet()


@atexit.register
def _close_all():
    # destroy contexts while the CUDA runtime is still alive (not from __del__ at interpreter teardown)
    for c in list(_live):
        c.close()


class Context:
    """One CUDA stream + scratch on one device (include/erp_b200.h: erp_ctx)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _check(lib().erp_ctx_create(device, C.byref(self._h)))
        self.device = device
        _live.add(self)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().erp_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- context
    @property
    def stream(self) -> int:
        return int(lib().erp_ctx_stream(self._h) or 0)

    def synchronize(self):
        _check(lib().erp_ctx_synchronize(self._h))

    def set_engine(self, engine: int):
        _check(lib().erp_ctx_set_engine(self._h, engine))

    @property
    def launch_count(self) -> int:
        return int(lib().erp_ctx_launch_count(self._h))

    def last_knn_stats(self):
        """engine, rescanned, the stream-K plan of the distance kernel (segments per query row, units per CTA, grid) and, for
        float rows on a tensor engine, the largest observed |approximate - exact| / (|q|^2 + max|t|^2).  That deviation takes
        the slot of the grid in the C record, so grid is None there.  chunks / items: older names of segments / units_per_cta."""
        out = (C.c_int64 * 5)()
        _check(lib().erp_ctx_last_knn_stats(self._h, out))
        dev = self.last_knn_operands()["operands"] in (OPERANDS_TF32, OPERANDS_F16)
        return dict(engine=out[0], rescanned=out[1], segments=out[2], units_per_cta=out[3], grid=None if dev else out[4],
                    deviation=out[4] * 1e-12 if dev else 0.0, chunks=out[2], items=out[3])

    def last_knn_operands(self):
        """Operand format of the last search's tensor products (OPERANDS_*), whether the f16 range guard fired, and how many
        queries the f16 range checks sent to the exact re-scan."""
        out = (C.c_int64 * 3)()
        _check(lib().erp_ctx_last_knn_operands(self._h, out))
        return dict(operands=out[0], guard=bool(out[1]), range_rescanned=out[2])

    def last_knn_kernel_ms(self) -> float:
        ms = C.c_float(0)
        _check(lib().erp_ctx_last_knn_kernel_ms(self._h, C.byref(ms)))
        return float(ms.value)

    def last_score_kernel_ms(self):
        ms, n = C.c_float(0), C.c_int(0)
        _check(lib().erp_ctx_last_score_kernel_ms(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def last_stage_ms(self):
        """Device time of the stages of the last pair_pose* call: (match, exchange + gather, RANSAC) in ms."""
        out = (C.c_float * 3)()
        _check(lib().erp_ctx_last_stage_ms(self._h, out))
        return float(out[0]), float(out[1]), float(out[2])

    def last_score_stats(self):
        out = (C.c_int64 * 6)()
        _check(lib().erp_ctx_last_score_stats(self._h, out))
        return dict(hyps=out[0], tiles_all=out[1], tiles_total=out[2], survivors=out[3], contenders=out[4], lstar=out[5])

    # ---- matching (host buffers)
    def knn2_match(self, q, t, ratio: float = 0.3, cross_check: bool = False) -> np.ndarray:
        """feature_matcher::match_two_image (src/feature_matcher.cpp:42-59). Returns DMatch records."""
        return self._knn2_match(lib().erp_knn2_match, self._h, _f32_rows, q, t, ratio, cross_check)

    def knn2_raw(self, q, t):
        return self._knn2_raw(lib().erp_knn2_raw, _f32_rows, q, t)

    @staticmethod
    def _knn2_match(fn, handle, rows, q, t, ratio, cross_check) -> np.ndarray:
        (q, qs), (t, ts) = rows(q), rows(t)
        out = np.empty(max(q.shape[0], 1), DMATCH)
        n = C.c_int(0)
        _check(fn(handle, _ptr(q), q.shape[0], qs, _ptr(t), t.shape[0], ts, q.shape[1], ratio, int(cross_check), _ptr(out), C.byref(n)))
        return out[: n.value]          # a view of this call's own array: only the pages the records touched are resident

    def _knn2_raw(self, fn, rows, q, t):
        (q, qs), (t, ts) = rows(q), rows(t)
        idx = np.empty((q.shape[0], 2), np.int32)
        dist = np.empty((q.shape[0], 2), np.float32)
        _check(fn(self._h, _ptr(q), q.shape[0], qs, _ptr(t), t.shape[0], ts, q.shape[1], _ptr(idx), _ptr(dist)))
        return idx, dist

    def knn2_near_ties(self, q, t, rel_tol: float = 1e-6) -> np.ndarray:
        """Per-query flags of erp_knn2_near_ties: bit 0 order of the two nearest, bit 1 identity of the second."""
        (q, qs), (t, ts) = _f32_rows(q), _f32_rows(t)
        flags = np.zeros(max(q.shape[0], 1), np.uint8)
        n = C.c_int(0)
        _check(lib().erp_knn2_near_ties(self._h, _ptr(q), q.shape[0], qs, _ptr(t), t.shape[0], ts, q.shape[1], rel_tol, _ptr(flags),
                                        C.byref(n)))
        flags = flags[: q.shape[0]]
        assert int((flags != 0).sum()) == n.value
        return flags

    # ---- matching (device buffers: torch tensors or raw pointers)
    def knn2_dev(self, d_q, nq, d_t, nt, dim, d_idx2, d_dist2, d_d2=None):
        _check(lib().erp_knn2_dev(self._h, _ptr(d_q), nq, _ptr(d_t), nt, dim, _ptr(d_idx2), _ptr(d_dist2), _ptr(d_d2)))

    def nn1_reverse_dev(self, d_q, nq, d_t, nt, dim, q_offset, d_best_q, d_best_d2=None):
        _check(lib().erp_nn1_reverse_dev(self._h, _ptr(d_q), nq, _ptr(d_t), nt, dim, q_offset, _ptr(d_best_q), _ptr(d_best_d2)))

    def match_filter_dev(self, d_idx2, d_dist2, nq, ratio, d_rev, q_offset, d_out, d_n_out):
        _check(lib().erp_match_filter_dev(self._h, _ptr(d_idx2), _ptr(d_dist2), nq, ratio, _ptr(d_rev), q_offset,
                                          _ptr(d_out), _ptr(d_n_out)))

    def knn2_match_dev(self, d_q, nq, d_t, nt, dim, ratio, cross_check, d_out, d_n_out):
        _check(lib().erp_knn2_match_dev(self._h, _ptr(d_q), nq, _ptr(d_t), nt, dim, ratio, int(cross_check),
                                        _ptr(d_out), _ptr(d_n_out)))

    # ---- binary descriptors (Hamming distance; include/erp_b200.h "binary descriptors")
    def knn2_match_bin(self, q, t, ratio: float = 0.3, cross_check: bool = False) -> np.ndarray:
        """match_two_image with cv::BFMatcher(NORM_HAMMING): (n, nbytes) uint8 rows -> DMatch records."""
        return self._knn2_match(lib().erp_knn2_match_bin, self._h, _u8_rows, q, t, ratio, cross_check)

    def knn2_raw_bin(self, q, t):
        return self._knn2_raw(lib().erp_knn2_raw_bin, _u8_rows, q, t)

    def knn2_bin_dev(self, d_q, nq, d_t, nt, nbytes, d_idx2, d_dist2, d_d2=None):
        _check(lib().erp_knn2_bin_dev(self._h, _ptr(d_q), nq, _ptr(d_t), nt, nbytes, _ptr(d_idx2), _ptr(d_dist2), _ptr(d_d2)))

    def knn2_match_bin_dev(self, d_q, nq, d_t, nt, nbytes, ratio, cross_check, d_out, d_n_out):
        _check(lib().erp_knn2_match_bin_dev(self._h, _ptr(d_q), nq, _ptr(d_t), nt, nbytes, ratio, int(cross_check),
                                            _ptr(d_out), _ptr(d_n_out)))

    def pair_pose_bin(self, q, t, left_xy, right_xy, W, H_img, ratio=0.8, cross_check=False, seed=1, H=10000, S=8,
                      metric=METRIC_ALGEBRAIC, tau=0.002):
        """erp_pair_pose_bin: binary descriptors + all keypoints of both views -> (match records, RANSAC result with mask)."""
        return self._pair_pose(lib().erp_pair_pose_bin, self._h, _u8_rows, q, t, left_xy, right_xy, W, H_img, ratio, cross_check, seed,
                               H, S, metric, tau)

    def pair_pose_bin_dev(self, d_q, nq, d_t, nt, nbytes, ratio, cross_check, d_left_xy, d_right_xy, kp_stride, W, H_img, seed, H,
                          S, metric, tau, d_matches, d_n, d_mask, d_result):
        """erp_pair_pose_bin_dev: enqueue only."""
        _check(lib().erp_pair_pose_bin_dev(self._h, _ptr(d_q), nq, _ptr(d_t), nt, nbytes, ratio, int(cross_check), _ptr(d_left_xy),
                                           _ptr(d_right_xy), kp_stride, W, H_img, seed, H, S, metric, tau, _ptr(d_matches), _ptr(d_n),
                                           _ptr(d_mask), _ptr(d_result)))

    # ---- geometry
    def bearings(self, xy, W: int, H: int) -> np.ndarray:
        """Pixel -> bearing of eight_point::find (src/eight_point.cpp:163-186). xy: (n,2) float32."""
        xy = _f32(xy)
        out = np.empty((xy.shape[0], 3), np.float64)
        _check(lib().erp_bearings_from_pixels(self._h, _ptr(xy), 8, xy.shape[0], W, H, _ptr(out)))
        return out

    def bearings_dev(self, d_xy, stride, n, W, H, d_out3, d_out4=None):
        _check(lib().erp_bearings_dev(self._h, _ptr(d_xy), stride, n, W, H, _ptr(d_out3), _ptr(d_out4)))

    def gather_bearings_dev(self, d_matches, n, d_left_xy, d_right_xy, stride, q_offset, W, H, d_l3, d_r3, d_l4, d_r4):
        _check(lib().erp_gather_bearings_dev(self._h, _ptr(d_matches), n, _ptr(d_left_xy), _ptr(d_right_xy), stride, q_offset,
                                             W, H, _ptr(d_l3), _ptr(d_r3), _ptr(d_l4), _ptr(d_r4)))

    def pack_float4_dev(self, d_v3, n, d_v4):
        _check(lib().erp_pack_float4_dev(self._h, _ptr(d_v3), n, _ptr(d_v4)))

    def eight_point_batch(self, l3, r3, samples=None, H=None, S=8, seed=0, hyp_offset=0, want_pose=True):
        l3, r3 = _f64(l3), _f64(r3)
        if samples is not None:
            samples = np.ascontiguousarray(samples, np.int32)
            H, S = samples.shape
        E = np.empty((H, 9), np.float64)
        pose = np.empty((H, POSE_FLOATS), np.float32) if want_pose else None
        _check(lib().erp_eight_point_batch(self._h, _ptr(l3), _ptr(r3), l3.shape[0], _ptr(samples), H, S, seed, hyp_offset,
                                           _ptr(E), _ptr(pose)))
        return E.reshape(H, 3, 3), pose

    def philox_samples(self, seed, hyp_offset, H, S, m) -> np.ndarray:
        out = np.empty((H, S), np.int32)
        _check(lib().erp_philox_samples(self._h, seed, hyp_offset, H, S, m, _ptr(out)))
        return out

    def eight_point_estimation(self, l3, r3):
        """eight_point::eight_point_estimation (src/eight_point.cpp:16-85) on all given points."""
        l3, r3 = _f64(l3), _f64(r3)
        E = np.empty(9)
        R1, R2, T = np.empty(3, np.float32), np.empty(3, np.float32), np.empty(3, np.float32)
        v1, v2 = C.c_int(0), C.c_int(0)
        _check(lib().erp_eight_point_estimation(self._h, _ptr(l3), _ptr(r3), l3.shape[0], _ptr(E), _ptr(R1), _ptr(R2), _ptr(T),
                                                C.byref(v1), C.byref(v2)))
        return dict(E=E.reshape(3, 3), R1=R1, R2=R2, T=T, R1_valid=bool(v1.value), R2_valid=bool(v2.value))

    # ---- scoring / RANSAC
    def score(self, E, l3, r3, metric=METRIC_ALGEBRAIC, tau=0.002) -> np.ndarray:
        E = _f64(E).reshape(-1, 9)
        l3, r3 = _f64(l3), _f64(r3)
        counts = np.empty(E.shape[0], np.int32)
        _check(lib().erp_score(self._h, _ptr(E), E.shape[0], _ptr(l3), _ptr(r3), l3.shape[0], metric, tau, _ptr(counts)))
        return counts

    def score_dev(self, d_E, H, d_l4, d_r4, m, metric, tau, hyp_offset, d_counts, d_best=None):
        _check(lib().erp_score_dev(self._h, _ptr(d_E), H, _ptr(d_l4), _ptr(d_r4), m, metric, tau, hyp_offset,
                                   _ptr(d_counts), _ptr(d_best)))

    def inlier_mask(self, E, l3, r3, metric=METRIC_ALGEBRAIC, tau=0.002):
        l3, r3 = _f64(l3), _f64(r3)
        mask = np.empty(l3.shape[0], np.uint8)
        n = C.c_int(0)
        _check(lib().erp_inlier_mask(self._h, _ptr(_f64(E).reshape(9)), _ptr(l3), _ptr(r3), l3.shape[0], metric, tau,
                                     _ptr(mask), C.byref(n)))
        return mask, n.value

    def refit(self, l3, r3, mask=None):
        l3, r3 = _f64(l3), _f64(r3)
        if mask is not None:
            mask = np.ascontiguousarray(mask, np.uint8)
        E = np.empty(9)
        pose = np.empty(POSE_FLOATS, np.float32)
        _check(lib().erp_refit(self._h, _ptr(l3), _ptr(r3), l3.shape[0], _ptr(mask), _ptr(E), _ptr(pose)))
        return E.reshape(3, 3), pose

    @staticmethod
    def _result(res: RansacResult) -> dict:
        return dict(packed=int(res.packed), hyp=int(res.hyp_id), count=int(res.count), n_refit=int(res.n_refit),
                    E=np.array(res.E_best).reshape(3, 3), E_refit=np.array(res.E_refit).reshape(3, 3),
                    pose=np.array(res.pose, np.float32))

    def ransac(self, l3, r3, seed, hyp_offset, H, S=8, metric=METRIC_ALGEBRAIC, tau=0.002):
        l3, r3 = _f64(l3), _f64(r3)
        res = RansacResult()
        mask = np.empty(l3.shape[0], np.uint8)
        _check(lib().erp_ransac(self._h, _ptr(l3), _ptr(r3), l3.shape[0], seed, hyp_offset, H, S, metric, tau,
                                C.byref(res), _ptr(mask)))
        out = self._result(res)
        out["mask"] = mask
        return out

    def ransac_pixels(self, left_xy, right_xy, W, H_img, seed, hyp_offset, H, S=8, metric=METRIC_ALGEBRAIC, tau=0.002):
        """erp_ransac_pixels: matched keypoints (n x 2 float32 pixel pairs) -> pose; the bearings stay on the device."""
        left_xy, right_xy = _f32(left_xy), _f32(right_xy)
        res = RansacResult()
        mask = np.empty(left_xy.shape[0], np.uint8)
        _check(lib().erp_ransac_pixels(self._h, W, H_img, _ptr(left_xy), _ptr(right_xy), left_xy.strides[0], left_xy.shape[0],
                                       seed, hyp_offset, H, S, metric, tau, C.byref(res), _ptr(mask)))
        out = self._result(res)
        out["mask"] = mask
        return out

    def pair_pose(self, q, t, left_xy, right_xy, W, H_img, ratio=0.3, cross_check=False, seed=1, H=10000, S=8,
                  metric=METRIC_ALGEBRAIC, tau=0.002):
        """erp_pair_pose: descriptors + all keypoints of both views -> (match records, RANSAC result with mask)."""
        return self._pair_pose(lib().erp_pair_pose, self._h, _f32_rows, q, t, left_xy, right_xy, W, H_img, ratio, cross_check, seed, H, S,
                               metric, tau)

    def pair_pose_dev(self, d_q, nq, d_t, nt, dim, ratio, cross_check, d_left_xy, d_right_xy, kp_stride, W, H_img, seed, H, S,
                      metric, tau, d_matches, d_n, d_mask, d_result, dist=False):
        """erp_pair_pose_dev / erp_pair_pose_dist_dev (dist=True: d_q is this rank's shard, nq the TOTAL): enqueue only."""
        fn = lib().erp_pair_pose_dist_dev if dist else lib().erp_pair_pose_dev
        _check(fn(self._h, _ptr(d_q), nq, _ptr(d_t), nt, dim, ratio, int(cross_check), _ptr(d_left_xy), _ptr(d_right_xy), kp_stride,
                  W, H_img, seed, H, S, metric, tau, _ptr(d_matches), _ptr(d_n), _ptr(d_mask), _ptr(d_result)))

    # ---- multi-GPU: one process per GPU (the caller distributes the id, e.g. with torch.distributed)
    def comm_init(self, nranks: int, rank: int, unique_id: bytes):
        buf = (C.c_char * COMM_ID_BYTES).from_buffer_copy(unique_id)
        _check(lib().erp_comm_init(self._h, nranks, rank, buf))

    def comm_destroy(self):
        _check(lib().erp_comm_destroy(self._h))

    @property
    def comm_size(self) -> int:
        return int(lib().erp_comm_size(self._h))

    @property
    def comm_rank(self) -> int:
        return int(lib().erp_comm_rank(self._h))

    def comm_allreduce_best_dev(self, d_packed):
        _check(lib().erp_comm_allreduce_best_dev(self._h, _ptr(d_packed)))

    def comm_cross_check_dev(self, d_best_q, d_best_d2, nt):
        _check(lib().erp_comm_cross_check_dev(self._h, _ptr(d_best_q), _ptr(d_best_d2), nt))

    def pair_pose_dist(self, q, t, left_xy, right_xy, W, H_img, ratio=0.3, cross_check=False, seed=1, H=10000, S=8,
                       metric=METRIC_ALGEBRAIC, tau=0.002):
        """erp_pair_pose_dist: collective over the context's clique, host buffers (every rank passes the same arrays)."""
        return self._pair_pose(lib().erp_pair_pose_dist, self._h, _f32_rows, q, t, left_xy, right_xy, W, H_img, ratio, cross_check, seed, H, S,
                               metric, tau)

    def knn2_match_dist(self, q, t, ratio: float = 0.3, cross_check: bool = False) -> np.ndarray:
        """This rank's part of the query-sharded match list (global query ids)."""
        return self._knn2_match(lib().erp_knn2_match_dist, self._h, _f32_rows, q, t, ratio, cross_check)

    def knn2_match_dist_dev(self, d_q_shard, nq_total, d_t, nt, dim, ratio, cross_check, d_out, d_n_out):
        _check(lib().erp_knn2_match_dist_dev(self._h, _ptr(d_q_shard), nq_total, _ptr(d_t), nt, dim, ratio, int(cross_check),
                                             _ptr(d_out), _ptr(d_n_out)))

    @classmethod
    def _pair_pose(cls, fn, handle, rows, q, t, left_xy, right_xy, W, H_img, ratio, cross_check, seed, H, S, metric, tau):
        (q, qs), (t, ts) = rows(q), rows(t)
        left_xy, right_xy = _f32(left_xy), _f32(right_xy)
        out = np.empty(q.shape[0], DMATCH)
        n = C.c_int(0)
        res = RansacResult()
        mask = np.empty(q.shape[0], np.uint8)
        _check(fn(handle, _ptr(q), q.shape[0], qs, _ptr(t), t.shape[0], ts, q.shape[1],
                  ratio, int(cross_check), _ptr(left_xy), _ptr(right_xy), left_xy.strides[0], W, H_img,
                  seed, H, S, metric, tau, _ptr(out), C.byref(n), C.byref(res), _ptr(mask)))
        r = cls._result(res)
        r["mask"] = mask[:n.value]
        return out[:n.value], r

    def ransac_local_dev(self, d_l3, d_r3, d_l4, d_r4, m, seed, hyp_offset, H, S, metric, tau, d_packed):
        _check(lib().erp_ransac_local_dev(self._h, _ptr(d_l3), _ptr(d_r3), _ptr(d_l4), _ptr(d_r4), m, seed, hyp_offset, H, S,
                                          metric, tau, _ptr(d_packed)))

    def ransac_finish_dev(self, d_l3, d_r3, d_l4, d_r4, m, seed, packed, S, metric, tau, d_mask=None) -> dict:
        res = RansacResult()
        _check(lib().erp_ransac_finish_dev(self._h, _ptr(d_l3), _ptr(d_r3), _ptr(d_l4), _ptr(d_r4), m, seed, packed, S,
                                           metric, tau, _ptr(d_mask), C.byref(res)))
        return self._result(res)

    # ---- rows next to the hot path (SURVEY 8f)
    def rotate_image(self, im, R) -> np.ndarray:
        """erp_rotation::rotate_image (src/erp_rotation.cpp:94-122) on an (H, W, 3) uint8 image."""
        im = np.ascontiguousarray(im, np.uint8)
        out = np.empty_like(im)
        _check(lib().erp_rotate_image(self._h, _ptr(im), im.shape[1], im.shape[0], im.strides[0], _ptr(_f64(R).reshape(9)),
                                      _ptr(out), out.strides[0]))
        return out

    def rotate_image_dev(self, d_im, W, H, R, d_out):
        _check(lib().erp_rotate_image_dev(self._h, _ptr(d_im), W, H, W * 3, _ptr(_f64(R).reshape(9)), _ptr(d_out), W * 3))

    def crop_rotated_image(self, im, pitch_deg: float) -> np.ndarray:
        """spherical_surf::crop_rotated_image (src/spherical_surf.cpp:16-48)."""
        im = np.ascontiguousarray(im, np.uint8)
        out = np.empty((im.shape[0] // 4, im.shape[1], 3), np.uint8)
        _check(lib().erp_crop_rotated_image(self._h, _ptr(im), im.shape[1], im.shape[0], im.strides[0], pitch_deg,
                                            _ptr(out), out.strides[0]))
        return out

    def rotate_pixels(self, rc, R, W, H) -> np.ndarray:
        rc = np.ascontiguousarray(rc, np.int32)
        out = np.empty_like(rc)
        _check(lib().erp_rotate_pixels(self._h, _ptr(rc), rc.shape[0], _ptr(_f64(R).reshape(9)), W, H, _ptr(out)))
        return out

    def rotate_keypoints(self, xy, pitch_inv_deg: float, W, H) -> np.ndarray:
        """spherical_surf::rotate_keypoint (src/spherical_surf.cpp:50-63); returns the rotated copy."""
        xy = np.array(xy, np.float32, copy=True, order="C")
        _check(lib().erp_rotate_keypoints(self._h, _ptr(xy), 8, xy.shape[0], pitch_inv_deg, W, H))
        return xy

    def draw_epipole(self, E, left_xy, right_xy, im_w, im_h, out_w, out_h) -> np.ndarray:
        """epipolar_tool::draw_epipole (src/epipolar_tool.cpp:84-128) for <= 7 selected correspondences."""
        left_xy, right_xy = _f32(left_xy), _f32(right_xy)
        out = np.empty((out_h, out_w, 3), np.uint8)
        _check(lib().erp_draw_epipole(self._h, _ptr(_f64(E).reshape(9)), _ptr(left_xy), _ptr(right_xy), 8, left_xy.shape[0],
                                      im_w, im_h, out_w, out_h, _ptr(out), out.strides[0]))
        return out

    # ---- reference mode
    def initial_guess(self, l3, r3, samples=None, H=80, S=None):
        """eight_point::initial_guess (src/eight_point.cpp:87-150)."""
        l3, r3 = _f64(l3), _f64(r3)
        m = l3.shape[0]
        if samples is not None:
            samples = np.ascontiguousarray(samples, np.int32)
            H, S = samples.shape
        elif S is None:
            S = int(m * 0.25)
        R, T = np.empty(3, np.float32), np.empty(3, np.float32)
        cR, cT = np.empty((2 * H, 3), np.float32), np.empty((2 * H, 3), np.float32)
        nc, ch = C.c_int(0), C.c_int(-1)
        _check(lib().erp_initial_guess(self._h, _ptr(l3), _ptr(r3), m, _ptr(samples), H, S, _ptr(R), _ptr(T), _ptr(cR), _ptr(cT),
                                       C.byref(nc), C.byref(ch)))
        return dict(R=R, T=T, cand_R=cR[: nc.value].copy(), cand_T=cT[: nc.value].copy(), chosen=ch.value)

    def find(self, W, H, left_xy, right_xy, match_size=None, samples=None, n_hyp=0, S=0):
        """eight_point::find (src/eight_point.cpp:152-192). left_xy/right_xy: (n,2) float32 KeyPoint.pt."""
        left_xy, right_xy = _f32(left_xy), _f32(right_xy)
        match_size = left_xy.shape[0] if match_size is None else match_size
        if samples is not None:
            samples = np.ascontiguousarray(samples, np.int32)
            n_hyp, S = samples.shape
        R, T = np.empty(3, np.float32), np.empty(3, np.float32)
        _check(lib().erp_find(self._h, W, H, _ptr(left_xy), _ptr(right_xy), 8, match_size, _ptr(samples), n_hyp, S,
                              _ptr(R), _ptr(T)))
        return R, T


def shard_range(n: int, rank: int, nranks: int) -> tuple[int, int]:
    lo, hi = C.c_int(0), C.c_int(0)
    _check(lib().erp_shard_range(n, rank, nranks, C.byref(lo), C.byref(hi)))
    return lo.value, hi.value


def comm_unique_id() -> bytes:
    """ncclUniqueId of a new clique (rank 0 calls this and broadcasts the bytes)."""
    buf = (C.c_char * COMM_ID_BYTES)()
    _check(lib().erp_comm_unique_id(buf))
    return bytes(buf)


class Group:
    """One process, several GPUs (include/erp_b200.h: erp_group): the calls fan out inside the library."""

    def __init__(self, devices):
        devices = list(devices)
        arr = (C.c_int * len(devices))(*devices)
        self._h = C.c_void_p()
        _check(lib().erp_group_create(arr, len(devices), C.byref(self._h)))
        self.devices = devices
        _live.add(self)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().erp_group_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __len__(self):
        return int(lib().erp_group_size(self._h))

    def set_engine(self, engine: int):
        for r in range(len(self)):
            _check(lib().erp_ctx_set_engine(lib().erp_group_ctx(self._h, r), engine))

    def stage_ms(self, rank: int = 0):
        out = (C.c_float * 3)()
        _check(lib().erp_ctx_last_stage_ms(lib().erp_group_ctx(self._h, rank), out))
        return float(out[0]), float(out[1]), float(out[2])

    def pair_pose(self, q, t, left_xy, right_xy, W, H_img, ratio=0.3, cross_check=False, seed=1, H=10000, S=8,
                  metric=METRIC_ALGEBRAIC, tau=0.002):
        return Context._pair_pose(lib().erp_group_pair_pose, self._h, _f32_rows, q, t, left_xy, right_xy, W, H_img, ratio, cross_check,
                                  seed, H, S, metric, tau)

    def knn2_match(self, q, t, ratio: float = 0.3, cross_check: bool = False) -> np.ndarray:
        return Context._knn2_match(lib().erp_group_knn2_match, self._h, _f32_rows, q, t, ratio, cross_check)
