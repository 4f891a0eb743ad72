"""ctypes loader for libgymchess_b200.so (the C ABI declared in include/gymchess_b200.h).

There is NO CPU fallback: if the shared library is missing, or no CUDA device is visible when a
compute entry point is called, this raises.  `build()` compiles the library in-tree with nvcc for
sm_100a (also used by __graft_entry__.build()).
"""
import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
# GYMCHESS_B200_LIB selects another build of the same library (used to A/B kernel variants on the GPU box)
SO_PATH = os.environ.get("GYMCHESS_B200_LIB") or os.path.join(_PKG, "libgymchess_b200.so")
_CSRC = os.path.join(_PKG, "csrc")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


class GcbError(RuntimeError):
    pass


def sources():
    return [os.path.join(_CSRC, f) for f in ("gcb_kernels.cu", "chess_core.cuh", "env_core.cuh")] + [
        os.path.join(_ROOT, "include", "gymchess_b200.h")
    ]


# test-support builds of the same sources (tests/test_memory_safety.py): index checks compiled in; the self-test build
# re-introduces a known out-of-bounds access to prove that the checks see that class of bug
VARIANTS = {"checked": ["-DGCB_CHECKED"], "checked_selftest": ["-DGCB_CHECKED", "-DGCB_SELFTEST_OOB"]}


def variant_path(name):
    return os.path.join(_PKG, "libgymchess_b200_%s.so" % name)


def build(force=False, verbose=False, variant=None):
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> gym_chess_b200/libgymchess_b200.so (or a VARIANTS build)"""
    srcs = sources()
    out = SO_PATH if variant is None else variant_path(variant)
    if not force and os.path.exists(out) and os.path.getmtime(out) >= max(os.path.getmtime(s) for s in srcs):
        return out
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (VARIANTS[variant] if variant else []) + (["-Xptxas", "-v"] if verbose else []) + ["-o", out, srcs[0]]
    subprocess.check_call(cmd)
    return out


def build_all(force=True):
    """the product library and the test-support variants, compiled side by side (three nvcc runs in parallel)"""
    nvcc = os.environ.get("NVCC", "nvcc")
    srcs = sources()
    jobs = []
    for variant in [None] + list(VARIANTS):
        out = SO_PATH if variant is None else variant_path(variant)
        if not force and os.path.exists(out) and os.path.getmtime(out) >= max(os.path.getmtime(x) for x in srcs):
            continue
        cmd = [nvcc] + NVCC_FLAGS + (VARIANTS[variant] if variant else []) + ["-o", out, srcs[0]]
        jobs.append((cmd, subprocess.Popen(cmd)))
    for cmd, proc in jobs:
        if proc.wait() != 0:
            raise subprocess.CalledProcessError(proc.returncode, cmd)
    return SO_PATH


class Positions(C.Structure):
    _fields_ = [("bb01", C.c_void_p), ("bb23", C.c_void_p), ("player", C.c_void_p), ("rights", C.c_void_p)]


class EnvConfig(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int32),
        ("env_id_offset", C.c_uint32),
        ("seed", C.c_uint64),
        ("opponent", C.c_int32),
        ("agent_black", C.c_int32),
        ("auto_reset", C.c_int32),
        ("piece_slots", C.c_int32),
        ("history_cap", C.c_int32),
        ("moves_max", C.c_int32),
        ("n_templates", C.c_int32),
        ("template_boards", C.c_void_p),
        ("device", C.c_int32),
    ]


vp, i32 = C.c_void_p, C.c_int
# every symbol include/gymchess_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "gcb_last_error": (C.c_char_p, []),
    "gcb_version": (i32, []),
    "gcb_launch_count": (C.c_uint64, []),
    "gcb_device_count": (i32, []),
    "gcb_pack": (i32, [i32, vp, vp, vp, Positions, vp]),
    "gcb_unpack": (i32, [i32, Positions, vp, vp, vp, vp]),
    "gcb_get_possible_moves": (i32, [i32, Positions, i32, i32, vp, i32, vp, vp, vp]),
    "gcb_next_state": (i32, [i32, Positions, vp, Positions, vp, vp, vp, vp]),
    "gcb_update_state": (i32, [i32, Positions, vp, vp, vp]),
    "gcb_host_get_possible_moves": (i32, [i32, vp, vp, vp, i32, i32, vp, i32, vp, vp]),
    "gcb_host_next_state": (i32, [i32] + [vp] * 9),
    "gcb_host_update_state": (i32, [i32] + [vp] * 4),
    "gcb_env_create": (i32, [C.POINTER(EnvConfig), C.POINTER(vp)]),
    "gcb_env_destroy": (i32, [vp]),
    "gcb_env_reset": (i32, [vp, vp, vp]),
    "gcb_env_import": (i32, [vp, vp, vp, vp, vp, vp, vp]),
    "gcb_env_clone": (i32, [vp, vp, vp, vp]),
    "gcb_env_step": (i32, [vp, vp, vp, vp, vp, vp]),
    "gcb_env_step_index": (i32, [vp, vp, vp, vp, vp, vp]),
    "gcb_env_bot_ply": (i32, [vp, vp, vp, vp, vp, vp]),
    "gcb_env_step_sampled": (i32, [vp, i32, vp, vp, vp, vp, vp, vp]),
    "gcb_env_step_host": (i32, [vp, vp, vp, vp, vp, vp]),
    "gcb_env_step_index_host": (i32, [vp, vp, vp, vp, vp, vp]),
    "gcb_env_step_host_async": (i32, [vp, vp, vp, vp, vp, vp]),
    "gcb_env_step_index_host_async": (i32, [vp, vp, vp, vp, vp, vp]),
    "gcb_env_wait": (i32, [vp, vp]),
    "gcb_env_step_packed": (i32, [vp, vp, vp, vp]),
    "gcb_env_step_index_packed": (i32, [vp, vp, vp, vp]),
    "gcb_env_export": (i32, [vp, vp, vp, vp]),
    "gcb_env_legal_mask": (i32, [vp, vp, vp]),
    "gcb_env_legal_bitmask": (i32, [vp, vp, i32, vp]),
    "gcb_env_step_mask_output": (i32, [vp, vp, i32]),
    "gcb_env_legal_actions": (i32, [vp, vp, i32, vp, vp]),
    "gcb_env_sample_policy": (i32, [vp, vp, i32, C.c_int64, C.c_float, vp, vp, vp, vp]),
    "gcb_env_encode": (i32, [vp, vp, i32, vp, vp]),
    "gcb_env_piece_slots": (i32, [vp, C.POINTER(vp), C.POINTER(C.c_int32)]),
    "gcb_env_positions": (i32, [vp, C.POINTER(Positions)]),
    "gcb_env_snapshot_bytes": (i32, [vp, C.POINTER(C.c_uint64)]),
    "gcb_env_snapshot": (i32, [vp, vp, C.POINTER(C.c_uint64), vp]),
    "gcb_env_restore": (i32, [vp, vp, C.c_uint64, vp]),
    "gcb_env_stats": (i32, [vp, vp, vp]),
    "gcb_env_stats_reset": (i32, [vp, vp]),
    "gcb_env_stats_ptr": (i32, [vp, C.POINTER(vp), vp]),
    "gcb_env_check_guards": (i32, [vp, C.POINTER(C.c_uint64)]),
    "gcb_debug_violations": (i32, [C.POINTER(C.c_uint64), i32]),
    "gcb_build_is_checked": (i32, []),
}

_lib = None


def lib():
    """Load the shared library (raises if it has not been built: there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise GcbError(
                "gym_chess_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU fallback." % SO_PATH
            )
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError here = the .so does not match the header
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise GcbError("libgymchess_b200 error %d: %s" % (rc, lib().gcb_last_error().decode()))


def require_gpu():
    if lib().gcb_device_count() <= 0:
        raise GcbError("gym_chess_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
