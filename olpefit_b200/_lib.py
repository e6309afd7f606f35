"""ctypes binding of liblapf.so (include/lapf.h).  There is no CPU fallback: if the library is
missing or a compute call runs without an sm_100 device, a LapfError is raised."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

MAX_PARAMS = 19


class LapfError(RuntimeError):
    pass


class Problem(C.Structure):
    _fields_ = [("nbody", C.c_int32), ("ny", C.c_int32), ("nx", C.c_int32), ("n_frames", C.c_int32),
                ("floor_index", C.c_int32), ("flags", C.c_int32),
                ("data", C.c_void_p), ("weight", C.c_void_p), ("origin", C.c_void_p),
                ("outside", C.c_void_p)]


class Config(C.Structure):
    _fields_ = [("problem", Problem), ("n_walkers", C.c_int64), ("id_base", C.c_int64),
                ("id_stride", C.c_int64), ("seed", C.c_uint64), ("frame_of", C.c_void_p),
                ("init_params", C.c_void_p), ("widths", C.POINTER(C.c_double)),
                ("burn_in", C.c_int64), ("thin", C.c_int32), ("team_warps", C.c_int32)]


# every symbol include/lapf.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "lapf_abi_version": (C.c_int, []),
    "lapf_last_error": (C.c_char_p, []),
    "lapf_num_params": (C.c_int, [C.c_int]),
    "lapf_default_widths": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "lapf_model_chi2": (C.c_int, [C.POINTER(Problem), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p]),
    "lapf_sampler_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p), C.c_void_p]),
    "lapf_sampler_destroy": (C.c_int, [C.c_void_p]),
    "lapf_sampler_selftest": (C.c_int, [C.c_void_p, C.c_void_p]),
    "lapf_sampler_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "lapf_sampler_checkpoint_bytes": (C.c_int64, [C.c_void_p]),
    "lapf_sampler_save": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "lapf_sampler_load": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "lapf_sampler_set_widths": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "lapf_sampler_rows_for": (C.c_int64, [C.c_void_p, C.c_int64]),
    "lapf_sampler_run": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    "lapf_sampler_set_chain_format": (C.c_int, [C.c_void_p, C.c_int32]),
    "lapf_sampler_chain_bytes": (C.c_int64, [C.c_void_p, C.c_int64]),
    "lapf_sampler_start": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_sampler_sketch_enable": (C.c_int, [C.c_void_p, C.c_int32, C.c_double, C.c_double, C.c_void_p, C.c_void_p]),
    "lapf_sampler_sketch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_sampler_batchmeans_enable": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "lapf_sampler_batchmeans": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_sampler_draws_enable": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "lapf_sampler_draws": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_sampler_set_frame_widths": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_void_p]),
    "lapf_sampler_frame_widths": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_sampler_frame_counts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_sampler_adapt_widths": (C.c_int, [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]),
    "lapf_sampler_set_priors": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_void_p]),
    "lapf_sampler_priors": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_frame_outside": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                     C.c_int32, C.c_double, C.c_double, C.c_void_p, C.c_void_p]),
    "lapf_sampler_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_sampler_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_sampler_count": (C.c_int64, [C.c_void_p]),
    "lapf_sampler_launches": (C.c_int64, [C.c_void_p]),
    "lapf_chain_drain": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "lapf_write_chain_csv": (C.c_int, [C.c_char_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int32]),
    "lapf_frame_prep": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                  C.c_int32, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_philox_draws": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int32, C.c_int32, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "lapf_measure_peaks": (C.c_int, [C.POINTER(C.c_double)]),
}

_lib = None


def lib_path() -> str:
    return _build.LIB


def load():
    """Load liblapf.so (building it in-tree first if the sources are newer and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("LAPF_LIB") or lib_path()      # LAPF_LIB: an experimental build of the same sources
    if path == lib_path() and _build.is_stale():
        try:
            _build.build()
        except Exception as exc:  # no nvcc on this box: use what is there, or fail loudly
            if not os.path.exists(path):
                raise LapfError("liblapf.so is missing and cannot be built (%s). "
                                "There is no CPU fallback." % exc) from exc
    try:
        lib = C.CDLL(path)
    except OSError as exc:
        raise LapfError("cannot load %s: %s. There is no CPU fallback." % (path, exc)) from exc
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.lapf_abi_version() != 2:
        raise LapfError("liblapf ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int):
    if rc < 0:
        msg = load().lapf_last_error().decode("utf-8", "replace")
        if rc == -5:                                  # LAPF_ERR_SELFTEST: say which toolchain built this binary
            msg += "\n" + (_build.build_info() or "(no build record beside the library)")
        raise LapfError("liblapf error %d: %s" % (rc, msg))
    return rc
