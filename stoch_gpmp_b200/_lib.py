"""ctypes binding of include/stoch_gpmp_b200.h (libsgpmp.so, built in-tree by stoch_gpmp_b200.build).

There is deliberately no fallback: if the library is missing or a call fails, this raises.
"""
import ctypes as C
import os
import shutil

from . import build as _build

SGPMP_F32, SGPMP_F64 = 0, 1
OK, ERR_INVALID_ARG, ERR_UNSUPPORTED, ERR_CUDA, ERR_NO_DEVICE = 0, 1, 2, 3, 4
TABLE_STRIDE = 16
MAX_FRAMES = 16
MAX_SPHERES = 16
FIELD_RBF, FIELD_SDF, FIELD_SDF_CLAMPED, FIELD_OCCUPANCY = 0, 1, 2, 3
GPMP_INVERSE, GPMP_CHOLESKY = 0, 1
MAX_INTERP = 8
MAX_LINK_POINTS = 48
NUM_TERMS = 7
TERM_NAMES = ("start", "gp", "goal", "coll", "is", "self", "ee")
ABI_VERSION = 7
MAX_TIME_INTERP = 32


class Shape(C.Structure):
    _fields_ = [("B", C.c_int32), ("G", C.c_int32), ("K", C.c_int32), ("S", C.c_int32), ("T", C.c_int32),
                ("n_dof", C.c_int32), ("dtype", C.c_int32), ("sample_gid0", C.c_int32), ("problem_gid0", C.c_int64)]


class CostDesc(C.Structure):
    _fields_ = [
        ("dt", C.c_double), ("sigma_start", C.c_double), ("sigma_gp", C.c_double),
        ("sigma_goal_prior", C.c_double), ("temperature", C.c_double),
        ("start", C.c_void_p), ("goals", C.c_void_p),
        ("occ_map", C.c_void_p), ("map_of_problem", C.c_void_p),
        ("n_maps", C.c_int32), ("map_h", C.c_int32), ("map_w", C.c_int32),
        ("origin_xi", C.c_int32), ("origin_yi", C.c_int32), ("reserved0", C.c_int32),
        ("map_inv_cell", C.c_double), ("map_sigma_coll", C.c_double),
        ("spheres", C.c_void_p), ("n_spheres", C.c_int32), ("spheres_per_problem", C.c_int32),
        ("sphere_sigma_coll", C.c_double),
        ("n_frames", C.c_int32), ("include_base", C.c_int32),
        ("chain_R", (C.c_double * 9) * MAX_FRAMES), ("chain_p", (C.c_double * 3) * MAX_FRAMES),
        ("chain_joint", C.c_int32 * MAX_FRAMES),
        ("self_margin", C.c_double), ("self_sigma_coll", C.c_double),
        ("occ_map_u8", C.c_void_p),
        ("sphere_field_type", C.c_int32), ("reserved1", C.c_int32),
        ("sphere_interp_n", C.c_int32), ("sphere_interp_lo", C.c_int32), ("sphere_interp_hi", C.c_int32),
        ("self_interp_n", C.c_int32), ("self_interp_lo", C.c_int32), ("self_interp_hi", C.c_int32),
        ("sphere_interp_alpha", C.c_double * MAX_INTERP), ("self_interp_alpha", C.c_double * MAX_INTERP),
        ("ee_sigma_goal", C.c_double), ("ee_target_R", C.c_double * 9), ("ee_target_p", C.c_double * 3),
        ("ee_w_pos", C.c_double), ("ee_w_rot", C.c_double), ("ee_square", C.c_int32), ("reserved2", C.c_int32),
    ]


# name -> (restype, argtypes); every symbol include/stoch_gpmp_b200.h declares
_vp, _i32, _i64, _u32, _u64, _dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_double
_SP, _DP = C.POINTER(Shape), C.POINTER(CostDesc)
SIGNATURES = {
    "sgpmp_abi_version": (C.c_int, []),
    "sgpmp_last_error": (C.c_char_p, []),
    "sgpmp_dof_supported": (C.c_int, [_i32]),
    "sgpmp_launch_count": (_i64, []),
    "sgpmp_prior_factor": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "sgpmp_prior_dense_L": (C.c_int, [_i32, _i32, _vp, _i32, _vp, _vp]),
    "sgpmp_sample": (C.c_int, [_SP, _vp, _vp, _vp, _u64, _u32, _vp, _vp, _vp]),
    "sgpmp_cost": (C.c_int, [_SP, _DP, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sgpmp_fk_link_positions": (C.c_int, [_DP, _i32, _i32, _i32, _vp, _vp, _vp]),
    "sgpmp_select_plans": (C.c_int, [_SP, _DP, _i32, _dbl, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sgpmp_update": (C.c_int, [_SP, _dbl, _dbl, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sgpmp_iterate": (C.c_int, [_SP, _DP, _vp, _dbl, _i32, _vp, _u64, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sgpmp_iterate_lowlat": (C.c_int, [_SP, _DP, _vp, _dbl, _i32, _vp, _u64, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sgpmp_local_stats": (C.c_int, [_SP, _dbl, _vp, _vp, _vp, _vp]),
    "sgpmp_apply_stats": (C.c_int, [_SP, _vp, _dbl, _vp, _vp, _vp, _vp]),
    "sgpmp_iterate_stats": (C.c_int, [_SP, _DP, _vp, _u64, _u32, _vp, _vp, _vp, _vp]),
    "sgpmp_merge_apply_stats": (C.c_int, [_SP, _vp, _dbl, _vp, _i32, _vp, _vp, _vp]),
    "sgpmp_nccl_load": (C.c_int, [C.c_char_p]),
    "sgpmp_comm_unique_id": (C.c_int, [_vp]),
    "sgpmp_comm_init": (C.c_int, [_vp, _i32, _i32, C.POINTER(C.c_void_p)]),
    "sgpmp_comm_destroy": (C.c_int, [_vp]),
    "sgpmp_allreduce_stats": (C.c_int, [_vp, _SP, _vp, _vp, _vp]),
    "sgpmp_iterate_split_particles": (C.c_int, [_SP, _DP, _vp, _dbl, _i32, _u64, _u32, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "sgpmp_gpmp_workspace_bytes": (_i64, [_SP, _i32]),
    "sgpmp_gpmp_step": (C.c_int, [_SP, _DP, _vp, _vp, _dbl, _i32, _i32, _dbl, _i32, _vp, _vp, _vp, _vp, _i64, _vp, _vp]),
    "sgpmp_sample_dense_tc": (C.c_int, [_SP, _vp, _vp, _vp, _vp, _vp]),
    "sgpmp_weighted_cov": (C.c_int, [_SP, _vp, _vp, _vp, _vp, _i32, _vp]),
    "sgpmp_probe": (C.c_int, [_i32, _i32, _i32, _vp, _vp]),
}

_lib = None


class SgpmpError(RuntimeError):
    pass


def lib_path():
    # $SGPMP_LIB: an alternative build of the same ABI (kernel-tuning experiments, scratch/variants.py)
    return os.environ.get("SGPMP_LIB") or _build.LIB


def load():
    """Load libsgpmp.so (once).  Raises ImportError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError(
            "stoch_gpmp_b200: CUDA library %s is missing — build it with `python -m stoch_gpmp_b200.build` "
            "(needs nvcc; there is no CPU fallback)" % path)
    if path == _build.LIB and os.path.isdir(_build.CSRC) and not _build.is_fresh():
        # ADVICE r1: a library older than csrc/ would silently validate old kernels
        if shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc"):
            _build.build()
        else:
            raise ImportError("stoch_gpmp_b200: %s is older than the sources under csrc/ and nvcc is not available to rebuild it" % path)
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.sgpmp_abi_version() != ABI_VERSION:
        raise ImportError("stoch_gpmp_b200: %s has ABI %d, binding expects %d — rebuild"
                          % (path, lib.sgpmp_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(rc, what=""):
    """Translate a status code into the exception class the reference would raise."""
    if rc == OK:
        return
    msg = load().sgpmp_last_error().decode(errors="replace")
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError("%s: %s" % (what, msg))
    if rc == ERR_INVALID_ARG:
        raise ValueError("%s: %s" % (what, msg))
    raise SgpmpError("%s: status %d: %s" % (what, rc, msg))


def launch_count():
    return int(load().sgpmp_launch_count())
