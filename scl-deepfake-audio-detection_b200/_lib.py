"""ctypes binding of ``lib/librawboost_b200.so`` (C ABI: ``include/rawboost_b200.h``).

Fails loudly: a missing library raises ``RawBoostLibraryError`` -- nothing here falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# RAWBOOST_B200_LIB selects another build of the same ABI (kernel-variant experiments); default is the in-tree build.
LIB_PATH = os.environ.get("RAWBOOST_B200_LIB") or os.path.join(HERE, "lib", "librawboost_b200.so")

RB_ABI_VERSION = 1

#: every symbol ``include/rawboost_b200.h`` declares (checked by the CPU test-suite against the header)
SYMBOLS = (
    "rb_error_string", "rb_abi_version", "rb_workspace_bytes", "rb_workspace_bytes_for", "rb_filter_fir", "rb_normwav", "rb_lnl", "rb_isd",
    "rb_ssi", "rb_process", "rb_ctx_create", "rb_ctx_destroy", "rb_process_host", "rb_ctx_last_traffic",
    "rb_probe_fp32", "rb_launch_count", "rb_profile_enable", "rb_profile_read", "rb_planner_create", "rb_planner_destroy",
    "rb_planner_draw", "rb_devplan_bytes", "rb_devplan_draw", "rb_process_host_seeded",
    "rb_ctx_set_chunk", "rb_submit_host_seeded", "rb_ctx_wait", "rb_ctx_trace", "rb_ctx_timeline", "rb_multiview_assemble",
    "rb_multiview_assemble_ex", "rb_submit_seeded_ex", "rb_reverb_workspace_bytes", "rb_reverb",
    "rb_items_workspace_bytes", "rb_items_draw", "rb_items_run", "rb_items_stream_draw", "rb_items_stream_run",
    "rb_submit_seeded_packed", "rb_items_run_packed", "rb_items_stream_run_packed", "rb_set_tap_trim",
    "rb_tap_support",
)
RB_IO_HOST_F32, RB_IO_HOST_PCM16, RB_IO_DEVICE_F32 = 0, 1, 2
RB_CORPUS_F32, RB_CORPUS_PCM16 = 0, 1


class RawBoostLibraryError(RuntimeError):
    """The CUDA library is missing / not loadable, or one of its entry points returned an error."""


class RbPlan(C.Structure):
    """``struct rb_plan`` -- field order and types must match the header."""
    _fields_ = [
        ("n_f", C.c_int32),
        ("lnl_taps", C.c_void_p),
        ("lnl_tap_off", C.c_void_p),
        ("isd_off", C.c_void_p),
        ("isd_idx", C.c_void_p),
        ("isd_fr", C.c_void_p),
        ("g_sd", C.c_float),
        ("ssi_noise", C.c_void_p),
        ("ssi_taps", C.c_void_p),
        ("ssi_tap_off", C.c_void_p),
        ("ssi_snr_db", C.c_void_p),
    ]


class RbArgs(C.Structure):
    """``struct rb_args``: the reference's RawBoost knobs (main.py:258-298) plus the sample rate."""
    _fields_ = [("N_f", C.c_int32), ("nBands", C.c_int32)] + [(n, C.c_double) for n in (
        "minF", "maxF", "minBW", "maxBW", "minCoeff", "maxCoeff", "minG", "maxG", "minBiasLinNonLin", "maxBiasLinNonLin",
        "P", "g_sd", "SNRmin", "SNRmax", "fs")]


class RbCorpus(C.Structure):
    """``struct rb_corpus``: a packed corpus (rows from 16-byte chunk boundaries) for the ``_packed`` item entries."""
    _fields_ = [("samples", C.c_void_p), ("kind", C.c_int32), ("rows", C.c_int32), ("chunks", C.c_int64), ("start", C.c_void_p),
                ("len", C.c_void_p)]


class RbRngState(C.Structure):
    """``struct rb_rng_state``: numpy's legacy MT19937 state."""
    _fields_ = [("key", C.c_uint32 * 624), ("pos", C.c_int32), ("has_gauss", C.c_int32), ("cached_gaussian", C.c_double)]


def args_struct(args, sr) -> RbArgs:
    """``rb_args`` from the reference's argparse namespace (main.py:258-298) and the sample rate."""
    s = RbArgs()
    s.N_f, s.nBands = int(args.N_f), int(args.nBands)
    for name in ("minF", "maxF", "minBW", "maxBW", "minCoeff", "maxCoeff", "minG", "maxG", "minBiasLinNonLin", "maxBiasLinNonLin",
                 "P", "g_sd", "SNRmin", "SNRmax"):
        setattr(s, name, float(getattr(args, name)))
    s.fs = float(sr)
    return s


_lib = None


def build_hint() -> str:
    return ("build it with `python -c \"import __graft_entry__ as g; g.build()\"` "
            "or `scl-deepfake-audio-detection_b200/csrc/build.sh`")


def load() -> C.CDLL:
    """Load the shared library once and declare the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RawBoostLibraryError(f"{LIB_PATH} not found; {build_hint()}. There is no CPU fallback.")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise RawBoostLibraryError(f"cannot load {LIB_PATH}: {e}") from e
    vp, i32, sz = C.c_void_p, C.c_int, C.c_size_t
    lib.rb_error_string.restype = C.c_char_p
    lib.rb_error_string.argtypes = [i32]
    lib.rb_abi_version.restype = i32
    lib.rb_abi_version.argtypes = []
    lib.rb_workspace_bytes.restype = sz
    lib.rb_workspace_bytes.argtypes = [i32, i32]
    lib.rb_workspace_bytes_for.restype = sz
    lib.rb_workspace_bytes_for.argtypes = [i32, i32, i32]
    lib.rb_filter_fir.restype = i32
    lib.rb_filter_fir.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp]
    lib.rb_normwav.restype = i32
    lib.rb_normwav.argtypes = [vp, vp, i32, i32, i32, vp, vp, sz, vp]
    for name in ("rb_lnl", "rb_isd", "rb_ssi"):
        fn = getattr(lib, name)
        fn.restype = i32
        fn.argtypes = [vp, vp, i32, i32, C.POINTER(RbPlan), vp, vp, sz, vp]
    lib.rb_process.restype = i32
    lib.rb_process.argtypes = [i32, vp, vp, i32, i32, C.POINTER(RbPlan), vp, vp, sz, vp]
    lib.rb_ctx_create.restype = i32
    lib.rb_ctx_create.argtypes = [C.POINTER(vp), i32]
    lib.rb_ctx_destroy.restype = i32
    lib.rb_ctx_destroy.argtypes = [vp]
    lib.rb_process_host.restype = i32
    lib.rb_process_host.argtypes = [vp, i32, vp, vp, i32, i32, C.POINTER(RbPlan), vp]
    lib.rb_ctx_last_traffic.restype = i32
    lib.rb_ctx_last_traffic.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.rb_probe_fp32.restype = i32
    lib.rb_probe_fp32.argtypes = [i32, i32, vp, C.POINTER(C.c_double), vp]
    lib.rb_launch_count.restype = C.c_uint64
    lib.rb_launch_count.argtypes = []
    lib.rb_profile_enable.restype = i32
    lib.rb_profile_enable.argtypes = [i32]
    lib.rb_profile_read.restype = i32
    lib.rb_profile_read.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_uint64), i32]
    lib.rb_set_tap_trim.restype = i32
    lib.rb_set_tap_trim.argtypes = [i32]
    lib.rb_tap_support.restype = i32
    lib.rb_tap_support.argtypes = [vp, vp, i32, vp, vp]
    lib.rb_planner_create.restype = i32
    lib.rb_planner_create.argtypes = [C.POINTER(vp), i32, i32]
    lib.rb_planner_destroy.restype = i32
    lib.rb_planner_destroy.argtypes = [vp]
    lib.rb_planner_draw.restype = i32
    lib.rb_planner_draw.argtypes = [vp, C.POINTER(RbArgs), i32, i32, i32, vp, vp, C.POINTER(RbRngState), C.POINTER(RbPlan)]
    lib.rb_multiview_assemble.restype = i32
    lib.rb_multiview_assemble.argtypes = [vp, vp, i32, i32, i32, vp, i32, i32, i32, vp, vp, vp]
    lib.rb_multiview_assemble_ex.restype = i32
    lib.rb_multiview_assemble_ex.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, i32, i32, i32, vp, vp, vp, vp, vp]
    lib.rb_submit_seeded_ex.restype = i32
    lib.rb_submit_seeded_ex.argtypes = [vp, i32, C.POINTER(RbArgs), vp, i32, vp, vp, i32, i32, vp, i32, vp, i32, C.POINTER(C.c_uint64)]
    lib.rb_submit_seeded_packed.restype = i32
    lib.rb_submit_seeded_packed.argtypes = [vp, i32, C.POINTER(RbArgs), vp, i32, vp, vp, i32, i32, vp, i32, vp, i32,
                                            C.POINTER(C.c_uint64)]
    lib.rb_reverb_workspace_bytes.restype = sz
    lib.rb_reverb_workspace_bytes.argtypes = [i32, i32]
    lib.rb_reverb.restype = i32
    lib.rb_reverb.argtypes = [vp, vp, i32, i32, vp, vp, vp, i32, vp, vp, sz, vp]
    lib.rb_submit_host_seeded.restype = i32
    lib.rb_submit_host_seeded.argtypes = [vp, i32, C.POINTER(RbArgs), vp, vp, vp, i32, i32, vp, C.POINTER(C.c_uint64)]
    lib.rb_ctx_wait.restype = i32
    lib.rb_ctx_wait.argtypes = [vp, C.c_uint64]
    lib.rb_ctx_trace.restype = i32
    lib.rb_ctx_trace.argtypes = [vp, i32]
    lib.rb_ctx_timeline.restype = i32
    lib.rb_ctx_timeline.argtypes = [vp, C.POINTER(C.c_double), i32]
    lib.rb_ctx_set_chunk.restype = i32
    lib.rb_ctx_set_chunk.argtypes = [vp, i32]
    lib.rb_process_host_seeded.restype = i32
    lib.rb_process_host_seeded.argtypes = [vp, i32, C.POINTER(RbArgs), vp, vp, vp, i32, i32, vp]
    lib.rb_devplan_bytes.restype = sz
    lib.rb_devplan_bytes.argtypes = [C.POINTER(RbArgs), i32, i32, i32]
    lib.rb_devplan_draw.restype = i32
    lib.rb_devplan_draw.argtypes = [C.POINTER(RbArgs), i32, i32, i32, vp, vp, vp, sz, C.POINTER(RbPlan), vp]
    lib.rb_items_workspace_bytes.restype = sz
    lib.rb_items_workspace_bytes.argtypes = [C.POINTER(RbArgs), i32, i32, i32, i32, i32]
    lib.rb_items_draw.restype = i32
    lib.rb_items_draw.argtypes = [C.POINTER(RbArgs), i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, sz,
                                  C.POINTER(RbPlan), vp]
    lib.rb_items_run.restype = i32
    lib.rb_items_run.argtypes = [C.POINTER(RbArgs), i32, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.rb_items_stream_draw.restype = i32
    lib.rb_items_stream_draw.argtypes = [C.POINTER(RbArgs), i32, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, sz,
                                         C.POINTER(RbPlan), vp]
    lib.rb_items_stream_run.restype = i32
    lib.rb_items_stream_run.argtypes = [C.POINTER(RbArgs), i32, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp,
                                        vp, vp, sz, vp]
    lib.rb_items_run_packed.restype = i32
    lib.rb_items_run_packed.argtypes = [C.POINTER(RbArgs), i32, i32, i32, i32, i32, i32, i32, i32, C.POINTER(RbCorpus), vp, vp, vp, vp,
                                        vp, vp, vp, sz, vp]
    lib.rb_items_stream_run_packed.restype = i32
    lib.rb_items_stream_run_packed.argtypes = [C.POINTER(RbArgs), i32, vp, i32, i32, i32, i32, i32, i32, i32, i32, C.POINTER(RbCorpus),
                                               vp, vp, vp, vp, vp, vp, vp, sz, vp]
    if lib.rb_abi_version() != RB_ABI_VERSION:
        raise RawBoostLibraryError(f"ABI mismatch: library {lib.rb_abi_version()}, binding {RB_ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(code: int, what: str = "") -> None:
    """Raise on a non-zero return code of any entry point."""
    if code != 0:
        msg = load().rb_error_string(code).decode()
        raise RawBoostLibraryError(f"{what or 'rawboost_b200'} failed with code {code}: {msg}")
