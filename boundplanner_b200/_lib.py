"""ctypes binding of libbpgeo.so (C ABI declared in include/bpgeo.h).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a) and
loaded from this package directory.  There is no CPU fallback: a missing
library, or a machine without a CUDA device, is a hard error.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbpgeo.so")

BP_MAX_ROWS = 48
ABI_VERSION = 6

STATUS_OK = 0
STATUS_ELLIPSE_VIOLATION = 1
STATUS_ROW_OVERFLOW = 2
STATUS_MVIE_NO_INTERIOR = 3
STATUS_MVIE_NOT_CONVERGED = 4
STATUS_ROW_CAP = 5
STATUS_NOT_A_POLYTOPE = 6

_c = ctypes
_vp, _i, _d, _sz = _c.c_void_p, _c.c_int, _c.c_double, _c.c_size_t
_dp = _c.POINTER(_c.c_double)

class BpTail(ctypes.Structure):
    """bp_tail of include/bpgeo.h (pair tests in the tail of the set build)"""
    _fields_ = [("S_glob", _c.c_int), ("words", _c.c_int), ("A", _vp), ("b", _vp), ("m", _vp), ("aabb", _vp),
                ("count", _vp), ("log", _vp), ("bits", _vp), ("epoch", _vp), ("off_count", _sz), ("off_log", _sz),
                ("off_bits", _sz), ("tol", _c.c_double)]


# name -> (restype, argtypes); every symbol include/bpgeo.h declares
SIGNATURES = {
    "bpgeo_abi_version": (_i, []),
    "bp_last_error_string": (_c.c_char_p, []),
    "bp_scene_create": (_i, [_dp, _i, _d, _c.POINTER(_vp)]),
    "bp_scene_create_batch": (_i, [_dp, _c.POINTER(_c.c_int), _i, _d, _c.POINTER(_vp)]),
    "bp_scene_create_polytopes": (_i, [_dp, _c.POINTER(_c.c_int), _dp, _c.POINTER(_c.c_int), _i, _i, _c.POINTER(_vp)]),
    "bp_scene_create_polytopes_batch": (_i, [_dp, _c.POINTER(_c.c_int), _dp, _c.POINTER(_c.c_int),
                                             _c.POINTER(_c.c_int), _i, _i, _c.POINTER(_vp)]),
    "bp_scene_update": (_i, [_vp, _dp, _i, _d, _vp]),
    "bp_scene_update_batch": (_i, [_vp, _dp, _c.POINTER(_c.c_int), _i, _d, _vp]),
    "bp_scene_update_polytopes_batch": (_i, [_vp, _dp, _c.POINTER(_c.c_int), _dp, _c.POINTER(_c.c_int),
                                             _c.POINTER(_c.c_int), _i, _i, _vp]),
    "bp_scene_destroy": (_i, [_vp]),
    "bp_scene_size": (_i, [_vp]),
    "bp_closest_points": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "bp_closest_points_line": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "bp_polyhedron": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "bp_mvie": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bp_mvie_fixed_r": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bp_build_sets_around_line": (_i, [_vp, _vp, _vp, _i, _dp, _dp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _i, _vp]),
    "bp_build_sets_workspace_bytes": (_sz, [_i]),
    "bp_build_sets_point": (_i, [_vp, _vp, _i, _dp, _dp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                 _i, _vp, _sz, _vp]),
    "bp_build_sets_point_ms": (_i, [_vp, _vp, _vp, _i, _dp, _dp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                    _vp, _i, _vp, _sz, _vp]),
    "bp_build_sets_point_x": (_i, [_vp, _vp, _vp, _i, _dp, _dp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                   _vp, _i, _vp, _vp, _i, _i, _sz, _sz, _sz, _sz, _vp, _sz, _vp]),
    "bp_step_begin": (_i, [_c.POINTER(BpTail), _i, _vp]),
    "bp_build_sets_point_tail": (_i, [_vp, _vp, _vp, _i, _dp, _dp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                      _vp, _i, _vp, _vp, _i, _i, _sz, _sz, _sz, _sz, _c.POINTER(BpTail), _vp, _sz,
                                      _vp]),
    "bp_build_sets_line_ms": (_i, [_vp, _vp, _vp, _vp, _i, _dp, _dp, _i, _d, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp,
                                   _vp, _vp, _sz, _vp]),
    "bp_pairs_feasible_list": (_i, [_vp, _vp, _vp, _i, _i, _d, _vp, _i, _vp, _vp, _vp, _sz, _vp]),
    "bp_build_sets_line": (_i, [_vp, _vp, _vp, _i, _dp, _dp, _i, _d, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                _vp, _sz, _vp]),
    "bp_pair_workspace_bytes": (_sz, [_i, _i]),
    "bp_set_aabb": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp]),
    "bp_pair_feasible": (_i, [_vp, _vp, _vp, _i, _i, _d, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "bp_pair_feasible_stages": (_i, [_vp, _vp, _vp, _i, _i, _d, _i, _i, _vp, _vp, _vp, _sz, _vp,
                                    _c.POINTER(_c.c_float)]),
    "bp_reduce_ineqs": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bp_check_fit": (_i, [_vp, _vp, _vp, _i, _i, _vp, _i, _vp, _vp, _dp, _i, _d, _vp, _vp, _vp]),
    "bp_project_points": (_i, [_vp, _vp, _vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "bp_sample_filter": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "bp_dedupe_distance": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bp_shortest_paths": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "bp_scatter_sets_peers": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _i, _sz, _sz, _sz, _sz, _vp]),
    "bp_scatter_rows_peers": (_i, [_vp, _i, _i, _i, _vp, _i, _sz, _vp]),
    "bp_fk_iiwa14": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "bp_sample_filter_tables": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "bp_dedupe_distance_tables": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bp_polytope_vertices": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "bp_debug_counters": (_i, [_c.POINTER(_c.c_ulonglong), _i, _i]),
    "bp_fk_iiwa14_kin": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "bp_probe_fp64": (_i, [_i, _i, _i, _i, _vp, _vp]),
    # native lock-step planner driver: (scene batch, Q[, query -> scene map], &handle) / (handle, &bp_plan_in, &bp_plan_out, stream)
    "bp_plan_create": (_i, [_vp, _i, _c.POINTER(_vp)]),
    "bp_plan_create_mapped": (_i, [_vp, _i, _c.POINTER(_c.c_int), _c.POINTER(_vp)]),
    "bp_plan_run": (_i, [_vp, _vp, _vp, _vp]),
    "bp_plan_destroy": (_i, [_vp]),
}

_lib = None


class BpGeoError(RuntimeError):
    pass


def load():
    """Load libbpgeo.so (once) and bind every declared symbol."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BpGeoError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  boundplanner_b200 has no CPU fallback."
        )
    # BPGEO_LIB: an alternative build of the same library (tools/prof_phases.py loads the -DBPGEO_PROFILE one)
    lib = ctypes.CDLL(os.environ.get("BPGEO_LIB", LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.bpgeo_abi_version() != ABI_VERSION:
        raise BpGeoError("libbpgeo.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().bp_last_error_string()
        raise BpGeoError(msg.decode() if msg else f"libbpgeo error {rc}")
