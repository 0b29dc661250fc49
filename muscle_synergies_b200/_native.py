"""ctypes binding of libms_b200.so (the C ABI declared in include/ms_b200.h).

There is no CPU fallback: if the shared library is missing or cannot be loaded this module
raises, and so does everything that needs it.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libms_b200.so")

MS_TILE_BYTES = 49152
MS_MAX_ROW_BYTES = 8192
MS_MAX_BLANK_ROWS = 8
MS_MAX_SECTIONS = 4

MS_SCAN_HAS_HIGH_BYTES = 1
MS_SCAN_BLANK_OVERFLOW = 2
MS_SCAN_HAS_CR = 4

MS_ERR_NONE = 0xFFFFFFFFFFFFFFFF
MS_ERR_KIND_BAD_FLOAT = 1
MS_ERR_KIND_NON_ASCII = 2
MS_ERR_KIND_ROW_TOO_LONG = 3


class ScanSummary(ctypes.Structure):
    _fields_ = [
        ("n_bytes", ctypes.c_int64),
        ("n_rows", ctypes.c_int64),
        ("n_terminators", ctypes.c_int64),
        ("n_quotes", ctypes.c_int64),
        ("n_blank_rows", ctypes.c_int64),
        ("flags", ctypes.c_uint32),
        ("n_reported", ctypes.c_uint32),
        ("blank_row", ctypes.c_int64 * MS_MAX_BLANK_ROWS),
        ("blank_end", ctypes.c_int64 * MS_MAX_BLANK_ROWS),
    ]


class Section(ctypes.Structure):
    _fields_ = [
        ("row_begin", ctypes.c_int64),
        ("row_end", ctypes.c_int64),
        ("num_cols", ctypes.c_int32),
        ("n_keep", ctypes.c_int32),
        ("d_out", ctypes.c_void_p),
        ("stride", ctypes.c_int64),
    ]


MS_LOAD_PEEK = 8192
MS_LOAD_HAVE_HEADER0 = 1
MS_LOAD_HAVE_DESC0 = 4
MS_LOAD_HAVE_ROWS0 = 16
MS_LOAD_FLAG_NAMES = {1: "ROW_TOO_LONG", 2: "DENSE_ROWS", 4: "MANY_BLANKS", 8: "TAIL_ROWS", 16: "OVERFLOW",
                      32: "BAD_HEADER", 64: "HIGH_BYTES"}


class LoadPlan(ctypes.Structure):
    _fields_ = [
        ("d_arena", ctypes.c_void_p),
        ("arena_elems", ctypes.c_int64),
        ("cap_rows", ctypes.c_int64 * 2),
        ("tile_bytes", ctypes.c_int32),
        ("overhang_bytes", ctypes.c_int32),
    ]


class LoadResult(ctypes.Structure):
    _fields_ = [
        ("status", ctypes.c_uint64),
        ("flags", ctypes.c_uint32),
        ("have", ctypes.c_uint32),
        ("n_blank_rows", ctypes.c_uint32),
        ("reserved", ctypes.c_uint32),
        ("tail_rows", ctypes.c_int64),
        ("n_quotes", ctypes.c_int64),
        ("header_offset", ctypes.c_int64 * 2),
        ("peek_bytes", ctypes.c_int64 * 2),
        ("blank_end", ctypes.c_int64 * 2),
        ("data_rows", ctypes.c_int64 * 2),
        ("num_cols", ctypes.c_int32 * 2),
        ("n_keep", ctypes.c_int32 * 2),
        ("stride", ctypes.c_int64 * 2),
        ("out_offset", ctypes.c_int64 * 2),
    ]


class WindowPlan(ctypes.Structure):
    _fields_ = [
        ("divisor", ctypes.c_int64),
        ("n_rows", ctypes.c_int64),
        ("n_channels", ctypes.c_int32),
        ("cycles", ctypes.c_int32),
        ("d_starts", ctypes.c_void_p),
        ("d_stops", ctypes.c_void_p),
        ("d_offsets", ctypes.c_void_p),
    ]


MS_MAX_WINDOW_PLANS = 4


class NativeError(RuntimeError):
    pass


_lib = None


def _declare(L):
    vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32
    sigs = {
        "ms_workspace_bytes": (i64, [i64]),
        "ms_workspace_masks_offset": (i64, [i64]),
        "ms_scan": (ctypes.c_int, [vp, i64, vp, i64, vp, vp]),
        "ms_scan_quoted": (ctypes.c_int, [vp, i64, vp, i64, vp, vp]),
        "ms_peek_after_blank": (ctypes.c_int, [vp, i64, vp, i32, vp, i32, vp, vp]),
        "ms_parse": (ctypes.c_int, [vp, i64, vp, ctypes.POINTER(Section), i32, vp, vp]),
        "ms_transitions_workspace_bytes": (i64, [i64]),
        "ms_find_transitions": (ctypes.c_int, [vp, vp, i64, i32, i32, vp, vp, vp, vp, vp]),
        "ms_segment_trial": (ctypes.c_int, [vp, vp, i64, i32, i32, vp, vp, vp, vp, ctypes.POINTER(WindowPlan), i32, vp]),
        "ms_cut_windows": (ctypes.c_int, [vp, i64, i32, vp, vp, vp, i32, vp, i64, vp]),
        "ms_plan_phase_windows": (ctypes.c_int, [vp, vp, i32, i32, i64, i64, i32, vp, vp, vp, vp]),
        "ms_channel_means": (ctypes.c_int, [vp, i64, i32, i64, vp, vp]),
        "ms_rms_envelope": (ctypes.c_int, [vp, i64, i32, i64, vp, i32, vp, i64, vp]),
        "ms_sosfilt_workspace_bytes": (ctypes.c_size_t, [i64, i32, i64, i32]),
        "ms_sosfilt": (ctypes.c_int, [vp, i64, i32, i64, ctypes.POINTER(ctypes.c_double), i32,
                                      ctypes.POINTER(ctypes.c_double), i64, i32, vp, i32, vp, i64, vp, vp]),
        "ms_time_normalize_windows": (ctypes.c_int, [vp, i64, i32, vp, vp, i32, i32, i32, vp, vp]),
        "ms_nmf_resident_max_rows": (i32, [i32, i32]),
        "ms_nmf_mu_batched": (ctypes.c_int, [vp, i32, i32, ctypes.POINTER(i32), ctypes.POINTER(i32), i32, vp, vp, i32,
                                             ctypes.c_float, i32, vp, vp, vp, vp, vp]),
        "ms_host_copy_stream": (ctypes.c_int, [vp, vp, i64]),
        "ms_nmf_plan": (i32, [i32, i32, ctypes.POINTER(i32), ctypes.POINTER(i32), i32, vp]),
        "ms_nmf_mu_batched_planned": (ctypes.c_int, [vp, i32, i32, vp, i32, i32, vp, vp, i32, ctypes.c_float, i32, vp, vp, vp, vp]),
        "ms_nmf_stream_workspace_bytes": (i64, [i32, i32]),
        "ms_nmf_mu_stream": (ctypes.c_int, [vp, i64, i32, ctypes.POINTER(i32), ctypes.POINTER(i32), i32, vp, vp, i32,
                                            ctypes.c_float, i32, vp, vp, vp, vp, vp]),
        "ms_nmf_cd_resident_max_rows": (i32, [i32, i32]),
        "ms_nmf_cd_batched_planned": (ctypes.c_int, [vp, i32, i32, vp, i32, i32, vp, vp, i32, ctypes.c_double, vp, vp, vp, vp]),
        "ms_nmf_cd_stream_workspace_bytes": (i64, [i32, i32]),
        "ms_nmf_cd_stream": (ctypes.c_int, [vp, i64, i32, vp, i32, i32, vp, vp, i32, ctypes.c_double, vp, vp, vp, vp, vp]),
        "ms_nndsvd_workspace_bytes": (i64, [i32, i32]),
        "ms_nndsvd_init": (ctypes.c_int, [vp, i64, i32, i32, vp, i32, i32, i32, vp, vp, vp, vp, vp]),
        "ms_nmf_fixed_h_resident_max_rows": (i32, [i32, i32]),
        "ms_nmf_fixed_h_workspace_bytes": (i64, [i64, i32, i32, i32]),
        "ms_nmf_fixed_h": (ctypes.c_int, [vp, i64, i32, i64, i64, vp, i32, i32, vp, vp, i32, i32, ctypes.c_double, i32, vp,
                                          vp, vp, vp, vp]),
        "ms_nmf_beta_resident_max_rows": (i32, [i32, i32]),
        "ms_nmf_beta_workspace_bytes": (i64, [i64, i32, i32, i32]),
        "ms_nmf_beta": (ctypes.c_int, [vp, i64, i32, i64, i64, vp, i32, i32, vp, vp, ctypes.c_double, i32, i32,
                                       ctypes.c_double, i32, vp, vp, vp, vp, vp]),
        "ms_synergy_match_workspace_bytes": (i64, [i32]),
        "ms_synergy_match": (ctypes.c_int, [vp, i32, vp, i32, i32, vp, i64, vp, vp, vp, vp, i64, vp]),
        "ms_parse_long_workspace_bytes": (i64, [i64]),
        "ms_parse_long": (ctypes.c_int, [vp, i64, vp, ctypes.POINTER(Section), i32, i64, vp, vp, vp]),
        "ms_load_workspace_bytes": (i64, [i64, i32]),
        "ms_load_fused": (ctypes.c_int, [vp, i64, ctypes.POINTER(LoadPlan), vp, i64, vp, vp, vp]),
        "ms_copy_rows_to_host": (ctypes.c_int, [vp, i64, vp, i64, i64, i64, vp]),
        "ms_last_cuda_error": (ctypes.c_char_p, []),
        "ms_version": (ctypes.c_char_p, []),
        "ms_launch_count": (i64, []),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(L, name)  # AttributeError here = the library does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    return sigs


def lib():
    """Returns the loaded library; raises NativeError when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). muscle_synergies_b200 has no CPU fallback."
        )
    L = ctypes.CDLL(LIB_PATH)
    _declare(L)
    _lib = L
    return L


def check(code: int, what: str):
    if code != 0:
        names = {-1: "MS_E_INVALID", -2: "MS_E_CUDA", -3: "MS_E_WORKSPACE", -4: "MS_E_NO_DEVICE"}
        detail = lib().ms_last_cuda_error().decode() if code == -2 else ""
        raise NativeError(f"{what} failed: {names.get(code, code)} {detail}".strip())


def on_tensor_device(fn):
    """Runs `fn` with the CUDA device of its first tensor argument (or of the `.tensor` of a DeviceData) current.
    The C entry points launch on the runtime's current device: a tensor on cuda:1 handed to them while cuda:0 is
    current would fail (invalid resource handle) or touch the wrong device's memory."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        import torch

        dev = None
        for a in list(args) + list(kwargs.values()):
            t = a if isinstance(a, torch.Tensor) else getattr(a, "__dict__", {}).get("_block") and a.tensor
            if isinstance(t, torch.Tensor) and t.is_cuda:
                dev = t.device
                break
        if dev is None:
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)

    return wrapper


def launch_count() -> int:
    return int(lib().ms_launch_count())
