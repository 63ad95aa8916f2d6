"""ctypes binding of ``libheadland_b200.so`` (``include/headland_b200.h``).

PyTorch is used for device memory and streams only; every pointer handed to the
library is a raw ``data_ptr()``.  Nothing here computes on the CPU.
"""
import ctypes as C
import os
import threading

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libheadland_b200.so"

ABI_VERSION = 5
HL_MAX_PRIMS = 16
HL_CAPSULE_VERTS = 66
HL_RS_CANDIDATES = 46
HL_RS_MAX_SEGS = 5

CHECK_OBSTACLES = 1
CHECK_BOUNDARY = 2
CHECK_AUX = 4
CHECK_LANE = 8

STATUS_NAMES = {0: "ok", 1: "start_goal_blocked", 2: "open_empty", 3: "max_nodes",
                4: "capacity", 5: "rs_assert"}


class HeadlandError(RuntimeError):
    pass


class HlEnvHost(C.Structure):
    _fields_ = [
        ("n_obs", C.c_int32), ("obs_xy", C.POINTER(C.c_double)),
        ("n_field", C.c_int32), ("field_xy", C.POINTER(C.c_double)),
        ("n_seg", C.c_int32), ("seg_xy", C.POINTER(C.c_double)),
        ("seg_poly", C.POINTER(C.c_double)), ("seg_len", C.POINTER(C.c_double)),
        ("n_crit", C.c_int32), ("crit_xy", C.POINTER(C.c_double)),
        ("n_guide", C.c_int32), ("guide", C.POINTER(C.c_double)),
        ("default_search_length", C.c_double),
        ("body_ext", C.c_double * 4),
        ("n_aux", C.c_int32), ("aux_ext", C.POINTER(C.c_double)),
    ]


class HlSearchParams(C.Structure):
    _fields_ = [
        ("plan_resolution", C.c_double), ("yaw_resolution", C.c_double),
        ("maxc", C.c_double), ("max_steer", C.c_double), ("wheel_base", C.c_double),
        ("n_prims", C.c_int32),
        ("prim_steer", C.c_double * HL_MAX_PRIMS), ("prim_dir", C.c_double * HL_MAX_PRIMS),
        ("prim_yaw_step", C.c_double * HL_MAX_PRIMS), ("prim_curv", C.c_double * HL_MAX_PRIMS),
        ("prim_steer_eff", C.c_double * HL_MAX_PRIMS),
        ("steps_default", C.c_int32), ("steps_large", C.c_int32),
        ("steer_cost", C.c_double), ("delta_steer_cost", C.c_double),
        ("direction_change_cost", C.c_double), ("reverse_cost", C.c_double),
        ("hybrid_cost", C.c_double), ("min_length_to_goal", C.c_double),
        ("max_nodes", C.c_int32), ("max_path_poses", C.c_int32),
        ("motion_type", C.c_int32), ("dubins_capacity", C.c_int32),
    ]


class HlGridField(C.Structure):
    _fields_ = [
        ("occ_offset", C.c_int64), ("out_offset", C.c_int64),
        ("w", C.c_int32), ("h", C.c_int32), ("gi", C.c_int32), ("gj", C.c_int32),
    ]


class HlRasterGrid(C.Structure):
    _fields_ = [
        ("out_offset", C.c_int64), ("env_id", C.c_int32),
        ("w", C.c_int32), ("h", C.c_int32), ("i0", C.c_int32), ("j0", C.c_int32),
    ]


SCENARIO_DTYPE = np.dtype([("env_id", "<i4"), ("reserved", "<i4"),
                           ("start", "<f8", (3,)), ("goal", "<f8", (3,))])
RESULT_DTYPE = np.dtype([("status", "<i4"), ("counter", "<i4"), ("n_expanded", "<i4"),
                         ("arrival", "<i4"), ("path_len", "<i4"), ("rs_word", "<i4"),
                         ("path_offset", "<i8"), ("goal_cost", "<f8"),
                         ("n_pose_checks", "<i8"), ("n_exact", "<i8"), ("keys_offset", "<i8"),
                         ("cycles", "<i8"), ("n_pose_checks_ref", "<i8")])
RSWORD_DTYPE = np.dtype([("cand", "<i4"), ("n_seg", "<i4"), ("npts", "<i4"), ("collide", "<i4"),
                         ("L", "<f8"), ("cost", "<f8"), ("len", "<f8", (HL_RS_MAX_SEGS,)),
                         ("nlen", "<f8", (HL_RS_MAX_SEGS,))])
assert SCENARIO_DTYPE.itemsize == 56 and RESULT_DTYPE.itemsize == 80 and RSWORD_DTYPE.itemsize == 112

EXPORTS = [
    "hl_last_error", "hl_abi_version", "hl_ctx_create", "hl_ctx_destroy", "hl_ctx_sm_count", "hl_ctx_device",
    "hl_ctx_set_astar_variant", "hl_env_upload", "hl_env_free", "hl_env_count", "hl_env_device", "hl_collision_check", "hl_path_reduce",
    "hl_rs_all_paths", "hl_rs_sample", "hl_hybrid_astar_batch", "hl_hybrid_astar_workspace_bytes", "hl_astar_phase_cycles",
    "hl_distance_field", "hl_distance_field_batch", "hl_grid_pack", "hl_grid_footprint_check", "hl_grid_footprint_check_at", "hl_env_rasterize",
    "hl_measure_fp32_peak", "hl_ypark_paths", "hl_arc_paths", "hl_ref_path_count", "hl_ref_path_fill",
    "hl_dubins_count", "hl_dubins_knots", "hl_dubins_fill", "hl_min_boundary_distance", "hl_corridor_hits",
]



class _Missing:
    def __init__(self, name):
        self._name = name
        self.argtypes = None
        self.restype = None

    def __call__(self, *a, **k):
        raise HeadlandError(f"libheadland_b200.so does not export {self._name}: rebuild the library")


class _Tolerant:
    """CDLL proxy: a symbol absent from an out-of-date build raises HeadlandError
    when CALLED instead of breaking the import of every other entry point."""

    def __init__(self, cdll):
        self._cdll = cdll
        self._missing = {}

    def __getattr__(self, name):
        try:
            return getattr(self._cdll, name)
        except AttributeError:
            return self._missing.setdefault(name, _Missing(name))


_lib = None
_lock = threading.RLock()      # re-entrant: check() -> last_error() -> load_library() under get_ctx's lock
_ctxs = {}


def library_path():
    return os.path.join(HERE, _LIB_NAME)


def load_library():
    """dlopen the in-tree library; fail loudly if it has not been built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if not os.path.exists(path):
            raise HeadlandError(
                f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)")
        lib = _Tolerant(C.CDLL(path))
        vp, i32, i64, u32, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_double
        lib.hl_last_error.restype = C.c_char_p
        lib.hl_abi_version.restype = C.c_int
        lib.hl_ctx_create.argtypes = [C.POINTER(vp), C.c_int]
        lib.hl_ctx_destroy.argtypes = [vp]
        lib.hl_ctx_destroy.restype = None
        lib.hl_ctx_sm_count.argtypes = [vp]
        lib.hl_ctx_device.argtypes = [vp]
        lib.hl_ctx_set_astar_variant.argtypes = [vp, C.c_int]
        lib.hl_env_device.argtypes = [vp]
        lib.hl_env_upload.argtypes = [vp, C.POINTER(HlEnvHost), i32, C.POINTER(vp)]
        lib.hl_env_free.argtypes = [vp]
        lib.hl_env_free.restype = None
        lib.hl_env_count.argtypes = [vp]
        lib.hl_env_count.restype = i32
        lib.hl_collision_check.argtypes = [vp, vp, vp, vp, vp, i64, u32, vp, vp, vp]
        lib.hl_path_reduce.argtypes = [vp, vp, vp, i64, vp, vp]
        lib.hl_rs_all_paths.argtypes = [vp, vp, vp, vp, i64, dbl, dbl, dbl, u32, vp, vp, vp, vp]
        lib.hl_rs_sample.argtypes = [vp, vp, vp, i64, dbl, dbl, vp, vp, vp, vp, vp, vp, vp]
        lib.hl_hybrid_astar_batch.argtypes = [vp, vp, vp, i32, C.POINTER(HlSearchParams), vp, vp, i64, vp,
                                              vp, vp, vp, vp, vp, i64, vp, vp]
        lib.hl_hybrid_astar_workspace_bytes.argtypes = [vp, C.POINTER(HlSearchParams)]
        lib.hl_hybrid_astar_workspace_bytes.restype = i64
        lib.hl_astar_phase_cycles.argtypes = [vp, C.POINTER(C.c_uint64), i32, i32]
        lib.hl_distance_field.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, C.POINTER(i32), vp]
        lib.hl_distance_field_batch.argtypes = [vp, vp, i64, C.POINTER(HlGridField), i32, i32, vp, i64, C.POINTER(i32), vp]
        lib.hl_grid_pack.argtypes = [vp, vp, i32, i32, vp, vp]
        lib.hl_grid_footprint_check.argtypes = [vp, vp, i32, i32, dbl, vp, i64, C.POINTER(dbl), vp, vp]
        lib.hl_grid_footprint_check_at.argtypes = [vp, vp, i32, i32, i32, i32, dbl, vp, i64, C.POINTER(dbl), vp, vp]
        lib.hl_env_rasterize.argtypes = [vp, vp, C.POINTER(HlRasterGrid), i32, dbl, u32, vp, i64, vp, vp]
        lib.hl_measure_fp32_peak.argtypes = [vp, C.POINTER(dbl)]
        lib.hl_ypark_paths.argtypes = [vp, vp, vp, i64, dbl, vp, vp]
        lib.hl_arc_paths.argtypes = [vp, vp, vp, i64, dbl, vp, vp]
        lib.hl_ref_path_count.argtypes = [vp, vp, vp, vp, vp, i64, dbl, vp, vp, vp]
        lib.hl_ref_path_fill.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, dbl, dbl, dbl, vp, vp, vp]
        lib.hl_dubins_count.argtypes = [vp, vp, i64, dbl, dbl, dbl, i32, vp, vp, vp, vp]
        lib.hl_dubins_knots.argtypes = [vp, vp, i64, dbl, dbl, dbl, i32, vp, vp, vp, vp, vp, vp]
        lib.hl_min_boundary_distance.argtypes = [vp, vp, vp, vp, vp, i64, i32, vp, vp]
        lib.hl_corridor_hits.argtypes = [vp, vp, vp, vp, vp, i64, dbl, vp, vp]
        lib.hl_dubins_fill.argtypes = [vp, i64, dbl, vp, vp, vp, vp, vp, vp]
        if lib.hl_abi_version() != ABI_VERSION:
            raise HeadlandError("libheadland_b200.so ABI version mismatch")
        _lib = lib
        return lib


def last_error():
    return load_library().hl_last_error().decode("utf-8", "replace")


def check(rc, what):
    if rc != 0:
        raise HeadlandError(f"{what}: {last_error()}")


def have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def get_ctx(device=None):
    """One hl_ctx per CUDA device, created on first use.  Raises without a GPU."""
    import torch
    lib = load_library()
    if not torch.cuda.is_available():
        raise HeadlandError("no CUDA device: headland_trajectory_planning_b200 has no CPU fallback")
    if device is None:
        device = torch.cuda.current_device()
    device = int(device)
    with _lock:
        if device in _ctxs:
            return _ctxs[device]
        h = C.c_void_p()
        rc = lib.hl_ctx_create(C.byref(h), device)
        msg = lib.hl_last_error().decode("utf-8", "replace") if rc != 0 else ""
        if rc == 0:
            _ctxs[device] = h
    if rc != 0:                           # raised outside the lock
        raise HeadlandError(f"hl_ctx_create: {msg}")
    return h


ASTAR_VARIANTS = {"spec": 0, "warp": 1, "level": 2}


def apply_astar_variant(ctx):
    """A/B switch of the search kernel (``HL_ASTAR_VARIANT`` = spec | warp | level).  The C library reads the
    variable once, at context creation; the Python binding forwards later changes (the tests flip it per case)."""
    v = os.environ.get("HL_ASTAR_VARIANT", "spec")
    check(load_library().hl_ctx_set_astar_variant(ctx, ASTAR_VARIANTS.get(v, 0)), "hl_ctx_set_astar_variant")


def ptr(t):
    """Raw device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous()
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dptr(a):
    """ctypes double* of a C-contiguous float64 numpy array (kept alive by the caller)."""
    return a.ctypes.data_as(C.POINTER(C.c_double))
