"""ctypes binding of libetude_b200.so (the C ABI declared in include/etude_b200.h).

There is no CPU fallback and no alternative backend: if the shared library is missing or cannot be loaded the
import of any compute entry point raises, and ``etude_create`` itself fails on a machine without an sm_100 GPU.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libetude_b200.so")
_lib = None

c_i64p = ctypes.POINTER(ctypes.c_int64)
c_vp = ctypes.c_void_p


class Note(ctypes.Structure):
    """etude_note_t"""
    _fields_ = [("pitch", ctypes.c_int32), ("velocity", ctypes.c_int32), ("onset", ctypes.c_double),
                ("offset", ctypes.c_double)]


class PcmSong(ctypes.Structure):
    """etude_pcm_song_t"""
    _fields_ = [("byte_offset", ctypes.c_int64), ("n_frames", ctypes.c_int64), ("frame_stride", ctypes.c_int64),
                ("channel_stride", ctypes.c_int64), ("dst_offset", ctypes.c_int64), ("channels", ctypes.c_int32),
                ("sample_rate", ctypes.c_int32), ("format", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class EtudeError(RuntimeError):
    pass


# name -> (restype, argtypes): every symbol the two public headers declare (tests/test_boundary.py checks this
# table against the headers and against the built library).
SIGNATURES = {
    "etude_last_error": (ctypes.c_char_p, []),
    "etude_version": (ctypes.c_char_p, []),
    "etude_create": (ctypes.c_int, [ctypes.c_int, c_vp, ctypes.c_size_t, ctypes.POINTER(c_vp)]),
    "etude_destroy": (None, [c_vp]),
    "etude_workspace_bytes": (ctypes.c_size_t, [c_vp, ctypes.c_int]),
    "etude_feature_rows": (ctypes.c_int64, [ctypes.c_int64]),
    "etude_logmel": (ctypes.c_int, [c_vp, c_vp, c_i64p, c_i64p, ctypes.c_int, c_vp, c_i64p, c_vp]),
    "etude_logmel_layout": (ctypes.c_int, [c_vp, c_vp, c_i64p, c_i64p, ctypes.c_int, c_vp, c_i64p, c_i64p, ctypes.c_int, ctypes.c_float,
                                           ctypes.c_int, c_vp]),
    "etude_resampled_length": (ctypes.c_int64, [ctypes.c_int64, ctypes.c_int, ctypes.c_int]),
    "etude_ingest": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, ctypes.c_int64, ctypes.c_int, ctypes.c_int, c_vp, c_vp]),
    "etude_ingest_reserve": (ctypes.c_int, [c_vp, ctypes.POINTER(ctypes.c_int), ctypes.c_int, ctypes.c_int]),
    "etude_ingest_pcm": (ctypes.c_int, [c_vp, c_vp, ctypes.POINTER(PcmSong), ctypes.c_int, ctypes.c_int, c_vp, c_vp]),
    "etude_forward_windows": (ctypes.c_int, [c_vp, c_vp, c_i64p, c_i64p, ctypes.c_int, ctypes.POINTER(c_vp),
                                             ctypes.POINTER(c_vp), c_vp, c_vp, c_vp, c_vp, ctypes.c_size_t, c_vp]),
    "etude_n_frame": (ctypes.c_int, [c_vp]),
    "etude_max_windows": (ctypes.c_int, [c_vp]),
    "etude_forward_windows_stride": (ctypes.c_int, [c_vp, c_vp, c_i64p, c_i64p, ctypes.c_int, ctypes.POINTER(c_vp), ctypes.POINTER(c_vp),
                                                    ctypes.c_int, ctypes.c_int, c_vp, ctypes.c_size_t, c_vp]),
    "etude_encode_windows": (ctypes.c_int, [c_vp, c_vp, c_i64p, ctypes.c_int, c_vp, c_vp, ctypes.c_size_t, c_vp]),
    "etude_decode_windows": (ctypes.c_int, [c_vp, c_vp, c_i64p, ctypes.c_int, ctypes.POINTER(c_vp), ctypes.POINTER(c_vp), c_vp, c_vp, c_vp,
                                            c_vp, ctypes.c_size_t, c_vp]),
    "etude_notes": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64p, c_i64p, ctypes.c_int, ctypes.c_int,
                                   ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_int,
                                   ctypes.c_int, ctypes.POINTER(ctypes.POINTER(Note)), c_i64p, c_vp]),
    "etude_notes_begin": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64p, c_i64p, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_int,
                                         ctypes.c_int, c_i64p, c_vp]),
    "etude_notes_fetch": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int64, c_vp]),
    "etude_notes_reserve": (ctypes.c_int, [c_vp, ctypes.c_int64, ctypes.c_int]),
    "etude_profile_classes": (ctypes.c_int, []),
    "etude_profile_class_name": (ctypes.c_char_p, [ctypes.c_int]),
    "etude_profile_reset": (ctypes.c_int, [c_vp, ctypes.c_int]),
    "etude_profile_read": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp]),
    "etude_profile_timeline": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, ctypes.c_int]),
    "etude_k_gemm": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_vp, c_vp,
                                    ctypes.c_int, c_vp, c_vp, c_vp, c_vp]),
    "etude_k_attn_qkv": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int, c_vp, c_vp]),
    "etude_k_chain": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int64, c_vp,
                                     ctypes.c_int, c_vp]),
    "etude_k_embed": (ctypes.c_int, [c_vp, c_vp, c_i64p, ctypes.c_int, c_vp, ctypes.c_int, c_vp]),
    "etude_k_heads": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, c_i64p, ctypes.c_int, ctypes.c_int,
                                     ctypes.POINTER(c_vp), c_vp, c_vp]),
    "etude_k_transpose_time": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, c_vp, c_vp]),
    "etude_k_attention": (ctypes.c_int, [c_vp, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_vp, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_vp, c_vp,
                                         c_vp]),
}

# test-only entry points of libetude_b200_dev.so (include/etude_b200_dev.h); never bound against the product library
DEV_SIGNATURES = {
    "etude_debug_mma_bench": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_i64p]),
    "etude_debug_mma_mix": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_i64p]),
    "etude_debug_tmem_bench": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_i64p]),
    "etude_debug_chain_trace": (ctypes.c_int, [ctypes.c_int, c_i64p, ctypes.c_int]),
    "etude_debug_pairmma": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp]),
    "etude_debug_pairmma_bench": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_i64p]),
    "etude_debug_attn_qkv_cta1": (ctypes.c_int, [c_vp, c_vp, c_vp, ctypes.c_int, c_vp, c_vp]),
}
DEV_LIB_PATH = os.path.join(_HERE, "libetude_b200_dev.so")
_dev = None


def load_dev():
    """The test-only superset build (micro-benchmarks, kernel timelines, generic GEMM epilogues).  tests/ only."""
    global _dev
    if _dev is None:
        if not os.path.exists(DEV_LIB_PATH):
            raise EtudeError(f"{DEV_LIB_PATH} is missing: build it with `python etude_b200/build.py`")
        lib = ctypes.CDLL(DEV_LIB_PATH)
        for name, (res, args) in {**SIGNATURES, **DEV_SIGNATURES}.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _dev = lib
    return _dev


def load():
    """Loads the library (building nothing: run ``python etude_b200/build.py`` or ``__graft_entry__.build()``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EtudeError(f"{LIB_PATH} is missing: build it with `python etude_b200/build.py` "
                             "(nvcc, sm_100a).  etude_b200 has no CPU or PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, what, lib=None):
    if rc != 0:
        raise EtudeError(f"{what}: {(lib or load()).etude_last_error().decode()}")


def i64_array(values):
    arr = (ctypes.c_int64 * len(values))(*[int(v) for v in values])
    return arr
