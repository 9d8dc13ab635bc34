"""ctypes binding of libame.so (include/ame.h).  Fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libame.so")

AME_F_WARMTH, AME_F_WIDTH, AME_F_MULTIBAND, AME_F_NORMALIZE, AME_F_LIMITER, AME_F_TRUE_PEAK = 1, 2, 4, 8, 16, 32
AME_F_MEASURE_OUTPUT = 64
AME_N_KERNELS = 12
AME_EQ_BYPASS, AME_EQ_SHELF_BOOST, AME_EQ_SHELF_CUT, AME_EQ_PEAK = 0, 1, 2, 3
AME_ABI_VERSION = 5


class Biquad(C.Structure):
    _fields_ = [("b0", C.c_double), ("b1", C.c_double), ("b2", C.c_double), ("a1", C.c_double), ("a2", C.c_double)]


class EqStage(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_sections", C.c_int32), ("g", C.c_double), ("gm1", C.c_double),
                ("s", Biquad * 4)]


class CompBand(C.Structure):
    _fields_ = [("thresh_rms", C.c_double), ("coef", C.c_double), ("attack_frames", C.c_double),
                ("release_frames", C.c_double), ("look_frames", C.c_int32), ("table", C.c_int32)]


class TrackParams(C.Structure):
    _fields_ = [("offset_frames", C.c_int64), ("n_frames", C.c_int64), ("halo_frames", C.c_int64), ("sample_rate", C.c_int32),
                ("chunk_frames", C.c_int32), ("flags", C.c_uint32), ("warm_lut", C.c_int32),
                ("wl_b0", C.c_double), ("wl_b1", C.c_double), ("wl_a1", C.c_double), ("wl_gm1", C.c_double),
                ("wh_b0", C.c_double), ("wh_b1", C.c_double), ("wh_a1", C.c_double), ("wh_gm1", C.c_double),
                ("eq", EqStage * 4), ("width", C.c_float), ("pad0_", C.c_float),
                ("xlp", Biquad * 2), ("xhp", Biquad * 2), ("comp", CompBand * 3), ("kw", Biquad * 2),
                ("target_lufs", C.c_double), ("warm_eq", C.c_int32), ("warm_xover", C.c_int32),
                ("warm_kw", C.c_int32), ("lim_frames", C.c_int32), ("lim_limit", C.c_double), ("lim_level", C.c_double),
                ("lim_fs_release", C.c_double), ("lim_release_frames", C.c_int32), ("lim_thr_i", C.c_int32)]


class TrackResult(C.Structure):
    _fields_ = [("input_i", C.c_double), ("measured_i_2dp", C.c_double), ("gain", C.c_double),
                ("rel_threshold", C.c_double), ("n_blocks", C.c_int64), ("normalized", C.c_int32),
                ("sample_peak", C.c_int32), ("input_lra", C.c_double), ("input_thresh", C.c_double),
                ("true_peak", C.c_double)]


class Loudness(C.Structure):
    _fields_ = [("integrated", C.c_double), ("thresh", C.c_double), ("lra", C.c_double), ("true_peak", C.c_double),
                ("max_momentary", C.c_double), ("max_short_term", C.c_double), ("n_blocks", C.c_int64),
                ("sample_peak", C.c_int32), ("measured", C.c_int32)]


class PlanOptions(C.Structure):
    _fields_ = [("eq_tile_frames", C.c_int32), ("xover_tile_frames", C.c_int32), ("kw_tile_subblocks", C.c_int32),
                ("host_io", C.c_int32), ("n_waves", C.c_int32), ("chain_warps", C.c_int32), ("n_slots", C.c_int32),
                ("precision", C.c_int32)]


class AmeError(RuntimeError):
    pass


_lib = None

# name -> (restype, argtypes); every symbol include/ame.h declares
SYMBOLS = {
    "ame_abi_version": (C.c_int, []),
    "ame_sizeof_track_params": (C.c_size_t, []),
    "ame_sizeof_track_result": (C.c_size_t, []),
    "ame_sizeof_plan_options": (C.c_size_t, []),
    "ame_sizeof_loudness": (C.c_size_t, []),
    "ame_last_error": (C.c_char_p, []),
    "ame_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "ame_release_cached_memory": (C.c_int, [C.c_int]),
    "ame_plan_create": (C.c_int, [C.c_int, C.POINTER(TrackParams), C.c_int32, C.POINTER(PlanOptions), C.POINTER(C.c_void_p)]),
    "ame_plan_destroy": (None, [C.c_void_p]),
    "ame_plan_set_warm_luts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "ame_plan_total_frames": (C.c_int64, [C.c_void_p]),
    "ame_plan_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "ame_plan_launch_count": (C.c_int64, [C.c_void_p]),
    "ame_plan_wave_count": (C.c_int32, [C.c_void_p]),
    "ame_plan_slot_count": (C.c_int32, [C.c_void_p]),
    "ame_plan_limiter_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "ame_plan_set_limiter_guess": (C.c_int, [C.c_void_p, C.c_int32]),
    "ame_plan_chain_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                      C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "ame_plan_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "ame_plan_kernel_times": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "ame_kernel_name": (C.c_char_p, [C.c_int]),
    "ame_plan_wave_timeline": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.c_int]),
    "ame_plan_kernel_timeline": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_float), C.c_int]),
    "ame_master_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(TrackResult), C.c_void_p]),
    "ame_master_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(TrackResult)]),
    "ame_plan_output_loudness": (C.c_int, [C.c_void_p, C.POINTER(Loudness), C.c_void_p]),
    "ame_measure_loudness": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Loudness), C.c_void_p]),
    "ame_measure_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ame_normalize_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(TrackResult), C.c_void_p]),
    "ame_shard_halo_exchange": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p]),
    "ame_hist_allreduce": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ame_stage_eq": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ame_stage_band_split": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ame_stage_compress": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ame_stage_loudness_hist": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ame_stage_apply_gain": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(TrackResult), C.c_void_p]),
    "ame_stage_limiter": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ame_plan_tap_pre": (C.c_void_p, [C.c_void_p]),
    "ame_plan_tap_bands": (C.c_void_p, [C.c_void_p]),
    "ame_plan_tap_subblock_energy": (C.c_void_p, [C.c_void_p]),
    "ame_plan_mb_frames": (C.c_int64, [C.c_void_p]),
    "ame_plan_mb_offset": (C.c_int64, [C.c_void_p, C.c_int32]),
    "ame_plan_subblock_offset": (C.c_int64, [C.c_void_p, C.c_int32]),
    "ame_plan_read_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
}


def load():
    """Load libame.so (built by build.py / __graft_entry__.build()).  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AmeError(f"{LIB_PATH} is missing: run `python -m audio_mastering_engine_b200.build` "
                           "(nvcc, sm_100a). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if (lib.ame_sizeof_track_params() != C.sizeof(TrackParams) or lib.ame_sizeof_track_result() != C.sizeof(TrackResult)
                or lib.ame_sizeof_plan_options() != C.sizeof(PlanOptions) or lib.ame_sizeof_loudness() != C.sizeof(Loudness)):
            raise AmeError("ctypes structs are out of sync with include/ame.h")
        if lib.ame_abi_version() != AME_ABI_VERSION:
            raise AmeError(f"libame.so has ABI version {lib.ame_abi_version()}, this package needs {AME_ABI_VERSION}: "
                           "rebuild with `python -m audio_mastering_engine_b200.build --force`")
        _lib = lib
    return _lib


def check(rc: int):
    if rc != 0:
        raise AmeError(f"libame error {rc}: {load().ame_last_error().decode(errors='replace')}")
