"""ctypes binding of libb2f.so (include/b2f.h).  No fallback: if the library is missing or a
compute call finds no GPU, the error is raised, never swallowed."""
from __future__ import annotations

import ctypes as C
import os

B2F_MAX_IF = 32
B2F_MAX_DM = 64
_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2F_LIB") or os.path.join(_HERE, "libb2f.so")   # B2F_LIB: an alternative build (A/B kernel experiments)

POL_P0, POL_P1, POL_I, POL_I2, POL_COHERENCE, POL_IQUV, POL_PPQQ = range(7)
K_VALIDATE, K_COLUMN, K_EPS, K_ROW, K_STATS, K_QUANT, K_DECODE, K_DEDISP = range(8)
KERNEL_NAMES = ["validate", "column", "eps", "row", "stats", "quant", "decode", "dedisp", "fused", "tsum"]

EINVAL, ECUDA, ENOMEM, ESTATE, EUNSUPPORTED = -1, -2, -3, -4, -5
DECODE_STATIC, DECODE_JA98 = 0, 1
RESCALE_CONSTANT, RESCALE_RUNNING = 0, 1
RAW_VDIF, RAW_MARK5B = 0, 1


class Params(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("nif", C.c_int32), ("nchan", C.c_int32),
        ("freq_res", C.c_int32), ("tscrunch", C.c_int32), ("pol_mode", C.c_int32), ("out_nbit", C.c_int32),
        ("in_nbit", C.c_int32), ("frame_bytes", C.c_int32), ("header_bytes", C.c_int32),
        ("frame_time_mode", C.c_int32), ("mask_faults", C.c_int32), ("keep_bandpass", C.c_int32),
        ("splice_pol_major", C.c_int32), ("chunk_units", C.c_int32), ("rescale_interval_s", C.c_double),
        ("bw_mhz", C.c_double * B2F_MAX_IF), ("freq_mhz", C.c_double * B2F_MAX_IF),
        ("if_order", C.c_int32 * B2F_MAX_IF), ("dm", C.c_double), ("coherent", C.c_int32),
        ("profile", C.c_int32), ("stream", C.c_void_p),
        ("raw_word_bits", C.c_int32), ("raw_bits", (C.c_uint8 * 4) * B2F_MAX_IF),
        ("decode_mode", C.c_int32), ("in8_offset_mode", C.c_int32), ("fft_normalised", C.c_int32),
        ("rescale_mode", C.c_int32), ("digi_sigma", C.c_double),
        ("raw_format", C.c_int32), ("reserved0", C.c_int32),
        ("ndm", C.c_int32), ("dm_trials", C.c_double * B2F_MAX_DM),
        ("remove_delays", C.c_int32), ("delay_ref_mhz", C.c_double),
    ]


class Geometry(C.Structure):
    _fields_ = [
        ("unit_frames", C.c_int64), ("unit_blocks", C.c_int64), ("chunk_frames", C.c_int64),
        ("chunk_rows", C.c_int64), ("block_samples", C.c_int64), ("samples_per_frame", C.c_int64),
        ("row_bytes", C.c_int64), ("nprod", C.c_int32), ("freq_res", C.c_int32), ("tsamp_s", C.c_double),
        ("interval_rows", C.c_int64), ("nfilt_pos", C.c_int32), ("nfilt_neg", C.c_int32),
        ("ndm", C.c_int32), ("trial_row_bytes", C.c_int64),
    ]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "frames_ok", "frames_invalid", "frames_with_fill", "fill_words", "frames_dropped",
        "frames_misplaced", "frames_badhdr", "slots_missing", "rows_produced", "rows_emitted",
        "blocks_dirty", "kernel_launches", "rescale_frozen", "rescale_preset")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class FilHeaderC(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("source_name", C.c_char_p), ("rawdatafile", C.c_char_p),
        ("telescope_id", C.c_int32), ("machine_id", C.c_int32), ("src_raj", C.c_double), ("src_dej", C.c_double),
        ("tstart_mjd", C.c_double), ("tsamp_s", C.c_double), ("nbits", C.c_int32), ("fch1_mhz", C.c_double),
        ("foff_mhz", C.c_double), ("nchans", C.c_int32), ("nifs", C.c_int32), ("refdm", C.c_double),
        ("write_refdm", C.c_int32),
    ]


class ScanIO(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("start_s", C.c_double), ("nsec", C.c_double), ("source_name", C.c_char_p),
        ("rawdatafile", C.c_char_p), ("telescope_id", C.c_int32), ("machine_id", C.c_int32),
        ("src_raj", C.c_double), ("src_dej", C.c_double), ("refdm", C.c_double), ("write_refdm", C.c_int32),
        ("ring", C.c_int32), ("readers_per_file", C.c_int32), ("part_index", C.c_int32), ("part_count", C.c_int32),
        ("stats_only", C.c_int32), ("trial_out_paths", C.POINTER(C.c_char_p)),
    ]


class ScanResult(C.Structure):
    _fields_ = [
        ("frames_per_if", C.c_int64), ("rows", C.c_int64), ("bytes_in", C.c_int64), ("bytes_out", C.c_int64),
        ("tstart_mjd", C.c_double), ("seconds_of_data", C.c_double), ("wall_s", C.c_double),
        ("setup_s", C.c_double), ("wait_read_s", C.c_double), ("wait_gpu_s", C.c_double), ("write_s", C.c_double),
        ("counters", Counters),
    ]


#: every symbol include/b2f.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "b2f_version": (C.c_int, []),
    "b2f_last_error": (C.c_char_p, []),
    "b2f_device_count": (C.c_int, []),
    "b2f_plan_create": (C.c_int, [C.POINTER(Params), C.POINTER(C.c_void_p)]),
    "b2f_plan_destroy": (C.c_int, [C.c_void_p]),
    "b2f_get_geometry": (C.c_int, [C.c_void_p, C.POINTER(Geometry)]),
    "b2f_push": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int64, C.c_int]),
    "b2f_flush": (C.c_int, [C.c_void_p]),
    "b2f_pull": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.POINTER(C.c_int64)]),
    "b2f_pull_strided": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.POINTER(C.c_int64)]),
    "b2f_sync": (C.c_int, [C.c_void_p]),
    "b2f_reset": (C.c_int, [C.c_void_p]),
    "b2f_get_counters": (C.c_int, [C.c_void_p, C.POINTER(Counters)]),
    "b2f_get_rescale": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2f_set_rescale": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2f_kernel_time": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "b2f_reset_timers": (C.c_int, [C.c_void_p]),
    "b2f_decode": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                             C.c_void_p, C.c_int, C.c_int, C.POINTER(Counters)]),
    "b2f_fp32_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
    "b2f_mark": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "b2f_wait": (C.c_int, [C.c_void_p, C.c_int64]),
    "b2f_get_params": (C.c_int, [C.c_void_p, C.POINTER(Params)]),
    "b2f_channeliser_path": (C.c_int, [C.c_void_p]),
    "b2f_get_delays": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b2f_sigproc_header": (C.c_int, [C.POINTER(FilHeaderC), C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "b2f_run_scan": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.c_char_p, C.POINTER(ScanIO),
                               C.POINTER(ScanResult)]),
    "b2f_release_host_cache": (C.c_int, []),
    "b2f_run_file": (C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p, C.POINTER(ScanIO), C.POINTER(ScanResult)]),
    "b2f_debug_copy": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
}

_lib = None


class B2FError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libb2f error {code}: {message}")
        self.code = code
        self.message = message


def lib() -> C.CDLL:
    """Load libb2f.so (built in-tree by `make -C frb-baseband_b200/csrc` / __graft_entry__.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OSError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise B2FError(rc, lib().b2f_last_error().decode(errors="replace"))
