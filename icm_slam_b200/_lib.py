"""ctypes binding of libicmslam.so (include/icmslam.h).  There is no CPU fallback: if the shared
library is missing or the CUDA device cannot be opened, calls raise."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libicmslam.so")
SRC_DIR = os.path.join(_HERE, "csrc")
INCLUDE_DIR = os.path.join(os.path.dirname(_HERE), "include")

HOST, DEVICE = 0, 1
SCHED = {"sequential": 0, "redblack": 1}
SOLVER = {"nm": 0, "newton": 1}
VIEW = {"running": 0, "full": 1, "prev": 2}

OK = 0
EMPTY_FIRST_SCAN = 1
ERR_LABEL_CAP = -2
ERR_EMPTY_LAST = -3
ERR_EMPTY_MAP = -4


class IcmConfig(C.Structure):
    _fields_ = [("deltat", C.c_double), ("q1", C.c_double), ("q2", C.c_double), ("r1", C.c_double), ("r2", C.c_double),
                ("r3", C.c_double), ("cte_odom", C.c_double), ("cota", C.c_double), ("dist_thr", C.c_double),
                ("rango_laser_max", C.c_double), ("radio", C.c_double), ("L", C.c_int32), ("device", C.c_int32)]


class SweepOpts(C.Structure):
    _fields_ = [("schedule", C.c_int32), ("solver", C.c_int32), ("map_view", C.c_int32), ("newton_maxit", C.c_int32),
                ("newton_tol", C.c_double), ("fused", C.c_int32), ("reserved", C.c_int32)]


def sources():
    return sorted(os.path.join(SRC_DIR, f) for f in os.listdir(SRC_DIR) if f.endswith((".cu", ".cuh"))) + [
        os.path.join(INCLUDE_DIR, "icmslam.h")]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/icmslam.cu for sm_100a into icm_slam_b200/lib/libicmslam.so (in tree, so the
    built file travels to the GPU box)."""
    os.makedirs(os.path.dirname(LIB_PATH), exist_ok=True)
    stale = force or not os.path.isfile(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in sources())
    if stale:
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
               "-shared", "-o", LIB_PATH, os.path.join(SRC_DIR, "icmslam.cu")]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    return LIB_PATH


_lib = None
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


def lib():
    """Loads the shared library; raises if it was not built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError("libicmslam.so is not built (%s missing); run `python -c 'import __graft_entry__ as g; g.build()'`. "
                           "There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    L.icmslam_abi_version.restype = C.c_int
    L.icmslam_strerror.restype = C.c_char_p
    L.icmslam_strerror.argtypes = [C.c_int]
    L.icmslam_last_error.restype = C.c_char_p
    L.icmslam_last_error.argtypes = [vp]
    L.icmslam_create.argtypes = [C.POINTER(IcmConfig), C.POINTER(vp)]
    L.icmslam_destroy.argtypes = [vp]
    L.icmslam_set_stream.argtypes = [vp, vp]
    L.icmslam_synchronize.argtypes = [vp]
    L.icmslam_load.argtypes = [vp, vp, i32, i32, i64, vp, i64, vp, i64, vp, vp, i32, i32]
    L.icmslam_extract.argtypes = [vp]
    L.icmslam_extraction_size.argtypes = [vp, C.POINTER(i64), _ip, _ip]
    L.icmslam_get_extraction.argtypes = [vp, vp, vp, vp, vp, vp, i32]
    L.icmslam_set_landmarks_actuales.argtypes = [vp, i32]
    L.icmslam_get_landmarks_actuales.argtypes = [vp, _ip]
    L.icmslam_get_counts.argtypes = [vp, vp, i32, i32]
    L.icmslam_set_counts.argtypes = [vp, vp, i32, i32]
    L.icmslam_sweep.argtypes = [vp, vp, i32, i64, vp, i64, vp, vp, i32, i64, vp, C.POINTER(SweepOpts), i32]
    L.icmslam_set_map.argtypes = [vp, vp, i32, i64, i32]
    L.icmslam_get_map.argtypes = [vp, vp, i32, i64, _ip, i32]
    L.icmslam_iterate.argtypes = [vp, vp, i64, vp, i32, C.POINTER(SweepOpts), i32]
    L.icmslam_set_poses.argtypes = [vp, vp, i64, i32]
    L.icmslam_get_poses.argtypes = [vp, vp, i64, i32]
    L.icmslam_set_segment.argtypes = [vp, i32, i32, i32, i32]
    L.icmslam_set_batch.argtypes = [vp, i32, vp, i64, i32]
    L.icmslam_set_batch_lengths.argtypes = [vp, vp, i32, vp, i64]
    L.icmslam_device_ptr.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(i64)]
    L.icmslam_seg_begin.argtypes = [vp, vp, C.POINTER(SweepOpts)]
    L.icmslam_seg_exchange.argtypes = [vp, vp, i32, i32]
    L.icmslam_seg_halo.argtypes = [vp, vp, i32, i32]
    L.icmslam_get_trace.argtypes = [vp, vp, vp]
    L.icmslam_pose_eval.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp, C.POINTER(dbl), C.POINTER(i32),
                                    C.POINTER(SweepOpts)]
    L.icmslam_p2p_export.argtypes = [vp, vp, i64]
    L.icmslam_p2p_import.argtypes = [vp, i32, i32, vp, i64]
    L.icmslam_seg_finish.argtypes = [vp]
    L.icmslam_fcluster.argtypes = [vp, vp, i32, dbl, vp, _ip]
    L.icmslam_pass0.argtypes = [vp, vp, vp, i64, vp, i32, i64, _ip, i32]
    L.icmslam_append.argtypes = [vp, vp, i32, i64, vp, i64, vp, i64, i32]
    L.icmslam_pass0_begin.argtypes = [vp, vp]
    L.icmslam_pass0_advance.argtypes = [vp, _ip]
    L.icmslam_pass0_finish.argtypes = [vp, vp, i64, vp, i32, i64, _ip, i32]
    L.icmslam_get_kernel_ms.argtypes = [vp, vp]
    L.icmslam_get_launch_count.argtypes = [vp, C.POINTER(i64)]
    L.icmslam_get_transfer_bytes.argtypes = [vp, C.POINTER(i64), C.POINTER(i64)]
    L.icmslam_get_associations.argtypes = [vp, vp, i32]
    L.icmslam_get_raw_map.argtypes = [vp, vp, i32, i64, vp, _ip, i32]
    L.icmslam_get_sweep_stats.argtypes = [vp, C.POINTER(i64), i32]
    L.icmslam_filter_map.argtypes = [vp, vp, i64, vp, i32, vp, i32, i64, vp, _ip, i32]
    L.icmslam_calc_cambio.argtypes = [vp, vp, i32, i64, vp, i32, i64, vp, i32]
    L.icmslam_filtrar_obs.argtypes = [vp, vp, i32, i32, i64, dbl, i32, vp, i64, i32]
    L.icmslam_associate.argtypes = [vp, vp, i32, i64, vp, vp, i32, vp, i32, i64, vp, i32]
    L.icmslam_iterate_until.argtypes = [vp, vp, i32, dbl, C.POINTER(SweepOpts), vp, _ip]
    L.icmslam_batch_iterate_until.argtypes = [vp, i32, dbl, dbl, i32, C.POINTER(SweepOpts), vp, _ip, _ip]
    for name in EXPORTS:
        getattr(L, name)  # fail loudly if the header and the library disagree
        if name not in ("icmslam_strerror", "icmslam_last_error"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


EXPORTS = [
    "icmslam_create", "icmslam_destroy", "icmslam_abi_version", "icmslam_strerror", "icmslam_last_error",
    "icmslam_set_stream", "icmslam_synchronize", "icmslam_load", "icmslam_extract", "icmslam_extraction_size",
    "icmslam_get_extraction", "icmslam_set_landmarks_actuales", "icmslam_get_landmarks_actuales", "icmslam_get_counts",
    "icmslam_sweep", "icmslam_get_associations", "icmslam_get_raw_map", "icmslam_get_sweep_stats", "icmslam_filter_map",
    "icmslam_calc_cambio", "icmslam_filtrar_obs", "icmslam_set_map", "icmslam_get_map", "icmslam_iterate",
    "icmslam_get_kernel_ms", "icmslam_get_launch_count", "icmslam_get_transfer_bytes", "icmslam_set_poses", "icmslam_get_poses", "icmslam_set_segment", "icmslam_device_ptr", "icmslam_seg_begin",
    "icmslam_seg_exchange", "icmslam_seg_halo", "icmslam_p2p_export", "icmslam_p2p_import", "icmslam_get_trace", "icmslam_pose_eval", "icmslam_seg_finish", "icmslam_fcluster", "icmslam_pass0", "icmslam_associate", "icmslam_iterate_until", "icmslam_set_counts", "icmslam_set_batch",
    "icmslam_batch_iterate_until", "icmslam_set_batch_lengths", "icmslam_append", "icmslam_pass0_begin", "icmslam_pass0_advance",
    "icmslam_pass0_finish",
]


class IcmSlamError(RuntimeError):
    def __init__(self, status, detail=""):
        self.status = status
        msg = lib().icmslam_strerror(status).decode()
        super().__init__("libicmslam: %s (%d)%s" % (msg, status, (": " + detail) if detail else ""))


def check(status, handle=None):
    """Maps C status codes onto the exceptions the reference raises at the same points."""
    if status in (OK, EMPTY_FIRST_SCAN):
        return status
    if status in (ERR_LABEL_CAP, ERR_EMPTY_LAST):
        raise IndexError(lib().icmslam_strerror(status).decode())
    if status == ERR_EMPTY_MAP:
        raise ValueError(lib().icmslam_strerror(status).decode())
    detail = lib().icmslam_last_error(handle).decode() if handle else ""
    raise IcmSlamError(status, detail)
