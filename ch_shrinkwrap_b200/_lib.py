"""ctypes binding of libnanowrap.so (include/nanowrap.h).  No torch, no CPU fallback: if the CUDA
library is missing or no GPU is usable, the product path raises."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint8, c_uint64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('NANOWRAP_LIB', os.path.join(_HERE, 'libnanowrap.so'))   # override is for kernel-variant experiments

NW_OK, NW_ERR_CUDA, NW_ERR_ARG, NW_ERR_NAN, NW_ERR_COMM = 0, 1, 2, 3, 4

_f, _d, _i = POINTER(c_float), POINTER(c_double), POINTER(c_int32)

# name -> (restype, argtypes); mirrors include/nanowrap.h one to one
SIGNATURES = {
    'nw_version': (c_int, []),
    'nw_create': (c_int, [c_int, POINTER(c_void_p)]),
    'nw_destroy': (None, [c_void_p]),
    'nw_last_error': (c_char_p, [c_void_p]),
    'nw_comm_unique_id': (c_int, [c_char_p]),
    'nw_comm_init': (c_int, [c_void_p, c_int, c_int, c_char_p]),
    'nw_set_points': (c_int, [c_void_p, c_void_p, c_int, c_int64, _f, c_float, _f]),
    'nw_set_topology': (c_int, [c_void_p, _f, _f, _i, _i, POINTER(c_uint8), c_int, c_int]),
    'nw_set_topology_halfedge': (c_int, [c_void_p, _f, _f, _i, _i, _i, c_int, POINTER(c_uint8), c_int, c_int]),
    'nw_set_topology_records': (c_int, [c_void_p, c_void_p, _i, c_void_p, c_int, c_int, c_int, c_int]),
    'nw_set_positions': (c_int, [c_void_p, _f]),
    'nw_get_positions': (c_int, [c_void_p, _f]),
    'nw_get_positions_strided': (c_int, [c_void_p, c_void_p, c_int, c_int]),
    'nw_search': (c_int, [c_void_p, c_float, c_int, c_int, _d, c_int, _f, _d, _d, _d, _d, _d, POINTER(c_int)]),
    'nw_set_regulariser': (c_int, [c_void_p, c_int]),
    'nw_compute_weights': (c_int, [c_void_p]),
    'nw_get_weights': (c_int, [c_void_p, _i, _f, _d, _i]),
    'nw_apply_A': (c_int, [c_void_p, _f, _f]),
    'nw_apply_AH': (c_int, [c_void_p, _f, _f]),
    'nw_point_influence': (c_int, [c_void_p, _f]),
    'nw_ncc': (c_int, [c_void_p, _d]),
    'nw_get_res': (c_int, [c_void_p, _f]),
    'nw_get_S': (c_int, [c_void_p, _f]),
    'nw_l_func': (c_int, [c_void_p, _f, _f]),
    'nw_lh_func': (c_int, [c_void_p, _f, _f]),
    'nw_lw_func': (c_int, [c_void_p, _f, _f, _f]),
    'nw_lhw_func': (c_int, [c_void_p, _f, _f, _f]),
    'nw_vertex_area_weights': (c_int, [c_void_p, _f, _f]),
    'nw_curvature_grad': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_float,
                                  _f, _f, _f, _f, _f, _f, _f, _f, _f, _f, _f, c_float, c_float, c_float, _f, _d, c_uint64]),
    'nw_neck_candidates': (c_int, [c_void_p, c_float, c_float, _i, POINTER(c_int)]),
    'nw_set_point_targets': (c_int, [c_void_p, c_void_p, c_int, c_int64]),
    'nw_points_from_mesh': (c_int, [c_void_p, _f, _i, c_int, c_int, c_double, _d, c_int64, POINTER(c_int64)]),
    'nw_holepunch_pair_candidate_faces': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, _i, c_int, _i]),
    'nw_surface_distance': (c_int, [c_void_p, c_void_p, c_int, c_int64, _d, _i, _d, _d]),
    'nw_surface_signed_distance': (c_int, [c_void_p, c_void_p, c_int, c_int64, _d, _i, _d, _d]),
    'nw_self_intersections': (c_int, [c_void_p, _i, c_int64, POINTER(c_int64), POINTER(c_int64)]),
    'nw_bench_kernel': (c_int, [c_void_p, c_char_p, c_int, _f]),
    'nw_sync': (c_int, [c_void_p]),
    'nw_reset_seeds': (c_int, [c_void_p]),
    'nw_set_profile': (c_int, [c_void_p, c_int]),
    'nw_get_stage_trace': (c_int, [c_void_p, _i, _f, c_int, POINTER(c_int)]),
    'nw_get_profile': (c_int, [c_void_p, _d, POINTER(c_int64), _d]),
    'nw_get_traversal_stats': (c_int, [c_void_p, POINTER(c_uint64)]),
    'nw_debug_tree': (c_int, [c_void_p, c_int, _f, POINTER(c_int), POINTER(c_int)]),
    'nw_launch_count': (c_int64, [c_void_p]),
}

_lib = None


def load():
    """Load libnanowrap.so; raises (never falls back) if it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                'libnanowrap.so is not built (%s). Run `python -m ch_shrinkwrap_b200.build`; '
                'there is no CPU fallback for the NanoWrap hot path.' % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def fptr(a):
    return None if a is None else a.ctypes.data_as(_f)


def dptr(a):
    return None if a is None else a.ctypes.data_as(_d)


def iptr(a):
    return None if a is None else a.ctypes.data_as(_i)


def as_f32(a):
    """C-contiguous float32 view/copy.  The reference's C helpers raise RuntimeError on
    non-contiguous input (conj_grad_utils.c:130-149); here we make the copy instead."""
    return np.ascontiguousarray(a, dtype=np.float32)


class Handle:
    """Owns one nw_ctx (one GPU, one stream)."""

    def __init__(self, device=0):
        self.lib = load()
        h = c_void_p()
        rc = self.lib.nw_create(int(device), ctypes.byref(h))
        if rc != NW_OK or not h:
            raise RuntimeError('nw_create(device=%d) failed with code %d: no usable CUDA device; '
                               'the NanoWrap hot path has no CPU fallback' % (device, rc))
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, 'h', None):
            self.lib.nw_destroy(self.h)
            self.h = None

    __del__ = close

    def check(self, rc):
        if rc == NW_OK:
            return
        msg = (self.lib.nw_last_error(self.h) or b'').decode('utf-8', 'replace')
        if rc == NW_ERR_NAN:
            raise AssertionError(msg)          # mirrors the reference's NaN asserts
        if rc == NW_ERR_ARG:
            raise ValueError(msg)
        raise RuntimeError('libnanowrap error %d: %s' % (rc, msg))

    def call(self, name, *args):
        self.check(getattr(self.lib, name)(self.h, *args))
