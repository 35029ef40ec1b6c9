"""ctypes binding of libdctts_b200.so (include/dctts.h).

There is deliberately no fallback: if the shared library has not been built
(`python -m dc_tts_b200.build`) importing this module raises ImportError, and if no
sm_100 GPU is present `dctts_create` fails -- the product path never computes on the CPU.
"""
import ctypes as C
import os

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libdctts_b200.so")


class HParams(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "vocab_size", "e", "d", "c", "n_mels", "n_fft", "max_N", "max_T", "attention_win_size", "r")]


Handle = C.c_void_p
_p, _i32, _i64 = C.c_void_p, C.c_int32, C.c_int64

# name -> (restype, argtypes); mirrors include/dctts.h one to one
SIGNATURES = {
    "dctts_create": (C.c_int, [C.POINTER(HParams), C.c_int, C.POINTER(Handle)]),
    "dctts_destroy": (C.c_int, [Handle]),
    "dctts_last_error": (C.c_char_p, [Handle]),
    "dctts_version": (C.c_char_p, []),
    "dctts_set_param": (C.c_int, [Handle, C.c_char_p, _p, C.POINTER(_i64), _i32]),
    "dctts_commit_params": (C.c_int, [Handle]),
    "dctts_num_params": (_i64, [Handle]),
    "dctts_embed": (C.c_int, [Handle, C.c_char_p, _p, _i32, _i32, _p, _p]),
    "dctts_normalize": (C.c_int, [Handle, C.c_char_p, _p, _i64, _i32, _p, _p]),
    "dctts_conv1d": (C.c_int, [Handle, C.c_char_p, _p, _i32, _i32, _i32, _i32, _i32, _p, _p]),
    "dctts_hc": (C.c_int, [Handle, C.c_char_p, _p, _i32, _i32, _i32, _i32, _p, _p]),
    "dctts_conv1d_transpose": (C.c_int, [Handle, C.c_char_p, _p, _i32, _i32, _p, _p]),
    "dctts_textenc": (C.c_int, [Handle, _p, _i32, _p, _p, _p]),
    "dctts_audioenc": (C.c_int, [Handle, _p, _i32, _i32, _p, _p]),
    "dctts_attention": (C.c_int, [Handle, _p, _p, _p, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p]),
    "dctts_audiodec": (C.c_int, [Handle, _p, _i32, _i32, _p, _p, _p]),
    "dctts_ssrn": (C.c_int, [Handle, _p, _i32, _i32, _p, _p, _p]),
    "dctts_text2mel_forward": (C.c_int, [Handle, _p, _p, _p, _i32, _p, _p, _p, _p]),
    "dctts_text2mel_generate": (C.c_int, [Handle, _p, _i32, _i32, _p, _p, _p, _p, _p]),
    "dctts_synthesize_host": (C.c_int, [Handle, _p, _i32, _p, _p]),
    "dctts_bench_block": (C.c_int, [Handle, C.c_char_p, _i32, _i32, _i32, _i32, C.POINTER(C.c_float),
                                    C.POINTER(_i32), _p]),
    "dctts_set_vocoder_params": (C.c_int, [Handle, _i32, _i32, C.c_float, C.c_float, C.c_float, C.c_float, _i32]),
    "dctts_spectrogram2wav": (C.c_int, [Handle, _p, _i32, _i32, _i32, _p, _p, _p]),
    "dctts_get_spectrograms": (C.c_int, [Handle, _p, _i64, _i32, _p, _p, _i32, C.POINTER(_i32), C.POINTER(_i32), _p]),
    "dctts_train_init": (C.c_int, [Handle, _i32, C.c_float]),
    "dctts_train_step": (C.c_int, [Handle, _p, _p, _i32, _i64, C.c_uint32, C.c_float, _i32, C.POINTER(C.c_float), _p]),
    "dctts_train_apply": (C.c_int, [Handle, _i64, C.c_float, _p]),
    "dctts_train_init_ssrn": (C.c_int, [Handle, _i32, _i32, C.c_float]),
    "dctts_train_step_ssrn": (C.c_int, [Handle, _p, _p, _i32, _i64, C.c_uint32, C.c_float, _i32, C.POINTER(C.c_float), _p]),
    "dctts_train_step_shaped": (C.c_int, [Handle, _p, _i32, _p, _i32, _i32, _i64, C.c_uint32, C.c_float, _i32,
                                          C.POINTER(C.c_float), _p]),
    "dctts_train_step_ssrn_shaped": (C.c_int, [Handle, _p, _p, _i32, _i32, _i64, C.c_uint32, C.c_float, _i32,
                                               C.POINTER(C.c_float), _p]),
    "dctts_train_reserve": (C.c_int, [Handle, _i32, _i32]),
    "dctts_train_grads": (C.c_int, [Handle, C.POINTER(_p), C.POINTER(_i64)]),
    "dctts_train_tensor": (C.c_int, [Handle, C.c_char_p, _i32, _p, _i64]),
    "dctts_train_set_tensor": (C.c_int, [Handle, C.c_char_p, _i32, _p, _i64]),
    "dctts_reserve": (C.c_int, [Handle, _i32]),
    "dctts_launch_count": (_i64, [Handle]),
    "dctts_crc32c": (C.c_uint32, [C.c_uint32, _p, _i64]),
    "dctts_set_tensor_path": (C.c_int, [Handle, _i32]),
    "dctts_set_option": (C.c_int, [Handle, C.c_char_p, _i32]),
    "dctts_get_option": (C.c_int, [Handle, C.c_char_p, C.POINTER(_i32)]),
    "dctts_decode_stats": (C.c_int, [Handle, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "dctts_decode_profile": (C.c_int, [Handle, C.POINTER(_i64), _i32]),
    "dctts_malloc": (C.c_int, [Handle, C.POINTER(_p), _i64]),
    "dctts_free": (C.c_int, [Handle, _p]),
    "dctts_memcpy_h2d": (C.c_int, [Handle, _p, _p, _i64, _p]),
    "dctts_memcpy_d2h": (C.c_int, [Handle, _p, _p, _i64, _p]),
    "dctts_malloc_host": (C.c_int, [Handle, C.POINTER(_p), _i64]),
    "dctts_free_host": (C.c_int, [Handle, _p]),
    "dctts_stream_sync": (C.c_int, [Handle, _p]),
}

_lib = None


def load():
    """Load the shared library and attach the prototypes (cached)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s is missing: build it with `python -m dc_tts_b200.build` "
            "(dc_tts_b200 has no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if the .so does not export it
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib
