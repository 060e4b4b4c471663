"""ctypes binding of libkokoro_align_b200.so (C ABI: include/kokoro_align_b200.h).

The shared object is built in-tree with nvcc for sm_100a by ``build()`` (also called from
``__graft_entry__.build``).  There is no CPU fallback: if the library is missing and cannot
be built, or no CUDA device is present, the compute entry points raise.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
SO_PATH = os.path.join(_HERE, "libkokoro_align_b200.so")
SOURCES = [os.path.join(_HERE, "csrc", f) for f in
           ("kab_api.cu", "kab_common.cuh", "kab_warp.cuh", "kab_band.cuh", "kab_bandp.cuh", "kab_bandq.cuh", "kab_bandr.cuh", "kab_btpar.cuh", "kab_wide.cuh", "kab_segstats.cuh", "kab_spans.cuh", "kab_compact.cuh", "kab_generic.cuh", "kab_softmax.cuh", "kab_pool.h", "kab_text.h", "kab_debug.h")]
HEADER = os.path.join(_ROOT, "include", "kokoro_align_b200.h")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]

KAB_OK, KAB_E_CUDA, KAB_E_BAD_ARG, KAB_E_NOMEM, KAB_E_UNSUPPORTED = 0, -1, -2, -3, -4
ST_OK, ST_DEAD_BAND, ST_BAD_LABEL, ST_NONFINITE = 0, 1, 2, 3

EXPORTS = ["kab_version", "kab_error_string", "kab_last_cuda_error", "kab_device_count",
           "kab_plan_create", "kab_plan_create_ctc", "kab_plan_create_ctc_long", "kab_plan_create_ctc_band", "kab_plan_get_info", "kab_plan_destroy", "kab_plan_run_device",
           "kab_plan_run_host", "kab_plan_run_host_logits", "kab_plan_run_host_segments", "kab_plan_segment_stats_device", "kab_log_softmax_device", "kab_log_softmax_pack_device", "kab_merge_tokens_device", "kab_word_spans_device", "kab_ctc_best_path", "kab_encode_transcript", "kab_merge_repeated", "kab_pool_trim", "kab_host_alloc", "kab_host_free"]


class PlanInfo(ctypes.Structure):
    _fields_ = [("n_lattices", ctypes.c_int64), ("n_class", ctypes.c_int64 * 4),
                ("total_frames", ctypes.c_int64), ("cells_eval", ctypes.c_int64),
                ("cells_nominal", ctypes.c_int64), ("workspace_bytes", ctypes.c_int64),
                ("backptr_bytes", ctypes.c_int64), ("algorithmic_bytes", ctypes.c_int64),
                ("kernel_launches", ctypes.c_int32), ("device", ctypes.c_int32),
                ("band_kernel", ctypes.c_int32), ("band_cluster", ctypes.c_int32)]

BAND_KERNELS = {0: None, 1: "kab_band_kernel", 2: "kab_bandp_kernel", 3: "kab_bandq_kernel", 4: "kab_bandr_kernel",
                5: "kab_bandr_kernel for the longest lattices + kab_band_kernel"}


class SegmentRecord(ctypes.Structure):
    """kab_segment_record"""
    _fields_ = [("text_start", ctypes.c_int32), ("text_end", ctypes.c_int32), ("non_blanks", ctypes.c_int32),
                ("non_blanks_score", ctypes.c_float), ("all_score", ctypes.c_float), ("status", ctypes.c_int32)]


class TokenSpanRec(ctypes.Structure):
    """kab_token_span"""
    _fields_ = [("token", ctypes.c_int32), ("start", ctypes.c_int32), ("end", ctypes.c_int32),
                ("score", ctypes.c_float)]


class WordSpanRec(ctypes.Structure):
    """kab_word_span"""
    _fields_ = [("start", ctypes.c_int32), ("end", ctypes.c_int32), ("first_token", ctypes.c_int32),
                ("score", ctypes.c_float)]


class KabError(RuntimeError):
    pass


def needs_build():
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    return any(os.path.exists(s) and os.path.getmtime(s) > t for s in SOURCES + [HEADER])


def build(force=False, verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> libkokoro_align_b200.so (in-tree)."""
    if not force and not needs_build():
        return SO_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO_PATH, SOURCES[0]]
    subprocess.check_call(cmd)
    return SO_PATH


_lib = None


def lib():
    """Load the C-ABI library (building it first when the sources are newer and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    so = os.environ.get("KAB_LIBRARY")  # development: an alternative build of the same C ABI
    if not so:
        so = SO_PATH
        if needs_build():
            try:
                build()
            except (OSError, subprocess.CalledProcessError) as e:
                if not os.path.exists(SO_PATH):
                    raise KabError(f"libkokoro_align_b200.so is missing and could not be built: {e}") from e
    L = ctypes.CDLL(so)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    L.kab_version.restype = ctypes.c_int
    L.kab_error_string.restype = ctypes.c_char_p
    L.kab_error_string.argtypes = [ctypes.c_int]
    L.kab_last_cuda_error.restype = ctypes.c_char_p
    L.kab_device_count.argtypes = [ctypes.POINTER(ctypes.c_int)]
    L.kab_plan_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int, i64, vp, vp, vp, i32, i32, i32]
    L.kab_plan_create_ctc.argtypes = [ctypes.POINTER(vp), ctypes.c_int, i64, vp, vp, vp, i32, i32]
    L.kab_plan_create_ctc_long.argtypes = [ctypes.POINTER(vp), ctypes.c_int, i64, vp, vp, vp, i32, i32]
    L.kab_plan_create_ctc_band.argtypes = [ctypes.POINTER(vp), ctypes.c_int, i64, vp, vp, vp, i32, i32, i32]
    L.kab_plan_get_info.argtypes = [vp, ctypes.POINTER(PlanInfo)]
    L.kab_plan_destroy.argtypes = [vp]
    L.kab_plan_run_device.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.kab_plan_run_host.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.kab_plan_run_host_logits.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.kab_log_softmax_device.argtypes = [vp, vp, i64, i32, vp]
    L.kab_log_softmax_pack_device.argtypes = [vp, i64, i64, i32, vp, vp, i64, vp]
    L.kab_plan_segment_stats_device.argtypes = [vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp]
    L.kab_plan_run_host_segments.argtypes = [vp, vp, i32, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.kab_merge_tokens_device.argtypes = [i64, vp, vp, vp, i32, vp, vp, vp]
    L.kab_word_spans_device.argtypes = [i64, vp, vp, vp, vp, vp, vp, vp, vp]
    L.kab_ctc_best_path.argtypes = [vp, i64, i32, vp, i64, i32, i32, vp, vp, vp, vp, vp]
    L.kab_encode_transcript.argtypes = [vp, i64, vp, vp, ctypes.POINTER(i64)]
    L.kab_merge_repeated.argtypes = [vp, i64, vp, ctypes.POINTER(i64)]
    L.kab_host_alloc.argtypes = [ctypes.POINTER(vp), ctypes.c_size_t]
    L.kab_host_free.argtypes = [vp]
    for name in EXPORTS:
        if name not in ("kab_error_string", "kab_last_cuda_error"):
            getattr(L, name).restype = ctypes.c_int
    _lib = L
    return L


def check(rc):
    if rc == KAB_OK:
        return
    L = lib()
    msg = L.kab_error_string(rc).decode()
    if rc == KAB_E_CUDA:
        msg += ": " + L.kab_last_cuda_error().decode()
    raise KabError(f"kokoro_align_b200 error {rc}: {msg}")
