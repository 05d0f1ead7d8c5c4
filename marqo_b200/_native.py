"""ctypes binding of include/marqo_b200.h.  There is no fallback: a missing library is an ImportError-class
failure at first use, and every non-zero status becomes an exception carrying b200_last_error()."""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

_LIB_NAME = "libmarqo_b200.so"
_lib = None
_lock = threading.Lock()

OK, ERR_INVALID_ARG, ERR_NO_DEVICE, ERR_CUDA, ERR_OOM, ERR_UNSUPPORTED, ERR_INTERNAL, ERR_MISSING_WEIGHT = range(8)

METRIC_PRENORMALIZED_ANGULAR, METRIC_ANGULAR, METRIC_DOTPRODUCT, METRIC_EUCLIDEAN = range(4)
ARCH_CLIP, ARCH_BERT, ARCH_MPNET = 0, 1, 2
ACT_GELU, ACT_QUICKGELU = 0, 1
POOL_MEAN, POOL_CLS = 0, 1
MAX_ATTRIBUTE_COLUMNS = 64
MAX_MODIFIER_TERMS = 16


class NativeError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"marqo_b200 native error {code}: {message}")
        self.code = code
        self.message = message


class NativeLibraryMissing(ImportError):
    pass


class TowerDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("width", "layers", "heads", "mlp", "ctx", "vocab", "image_size", "patch")]


class ModelDesc(C.Structure):
    _fields_ = [
        ("arch", C.c_int32), ("embed_dim", C.c_int32), ("act", C.c_int32), ("pool", C.c_int32),
        ("type_vocab", C.c_int32), ("max_batch", C.c_int32),
        ("image_mean", C.c_float * 3), ("image_std", C.c_float * 3),
        ("vision", TowerDesc), ("text", TowerDesc),
    ]


class SearchOpts(C.Structure):
    """b200_search_opts (include/marqo_b200.h)."""
    _fields_ = [
        ("mult_cols", C.c_void_p), ("mult_w", C.c_void_p), ("n_mult", C.c_int32),
        ("add_cols", C.c_void_p), ("add_w", C.c_void_p), ("n_add", C.c_int32),
        ("filter_bits", C.c_void_p), ("filter_docs", C.c_int64), ("filter_tag", C.c_uint64),
    ]


EXCHANGE_HANDLE_BYTES = 64

_P = C.c_void_p
_SIGNATURES = {
    "b200_abi_version": (C.c_int, []),
    "b200_last_error": (C.c_char_p, []),
    "b200_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "b200_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(_P)]),
    "b200_host_free": (C.c_int, [_P]),
    "b200_index_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int64, C.POINTER(_P)]),
    "b200_index_destroy": (C.c_int, [_P]),
    "b200_index_add": (C.c_int, [_P, _P, _P, C.c_int64]),
    "b200_index_add_device": (C.c_int, [_P, _P, _P, C.c_int64]),
    "b200_index_add_device_docs": (C.c_int, [_P, _P, _P, C.c_int64]),
    "b200_index_delete_doc": (C.c_int, [_P, C.c_int32]),
    "b200_index_delete_rows": (C.c_int, [_P, _P, C.c_int64]),
    "b200_index_compact": (C.c_int, [_P, _P, C.POINTER(C.c_int64)]),
    "b200_index_get_rows": (C.c_int, [_P, _P, C.c_int64, _P]),
    "b200_index_search_ex": (C.c_int, [_P, _P, C.c_int, C.c_int, C.POINTER(SearchOpts), _P, _P, _P]),
    "b200_index_search_stats": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                          C.POINTER(C.c_int64)]),
    "b200_index_set_attributes_multi": (C.c_int, [_P, _P, _P, _P, C.c_int64]),
    "b200_exchange_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_P), _P]),
    "b200_exchange_open": (C.c_int, [_P, _P]),
    "b200_exchange_destroy": (C.c_int, [_P]),
    "b200_index_search_exchange": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, _P, _P, _P, _P, C.c_int]),
    "b200_index_num_rows": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "b200_index_info": (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "b200_index_get_row": (C.c_int, [_P, C.c_int64, _P]),
    "b200_index_search": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P]),
    "b200_index_search_device": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, C.c_int]),
    "b200_index_set_attributes": (C.c_int, [_P, C.c_int, _P, _P, C.c_int64]),
    "b200_index_search_modified": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, C.c_int, _P, _P, C.c_int, _P, _P, _P]),
    "b200_index_set_stream": (C.c_int, [_P, _P, C.c_int]),
    "b200_index_last_timing": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "b200_index_set_doc_offset": (C.c_int, [_P, C.c_int32]),
    "b200_topk_merge_device": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_int]),
    "b200_topk_merge": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P]),
    "b200_index_save": (C.c_int, [_P, C.c_char_p]),
    "b200_index_load": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(_P)]),
    "b200_model_create": (C.c_int, [C.c_int, C.POINTER(ModelDesc), C.POINTER(_P)]),
    "b200_model_destroy": (C.c_int, [_P]),
    "b200_model_load_tensor": (C.c_int, [_P, C.c_char_p, _P, C.c_int64]),
    "b200_model_finalize": (C.c_int, [_P]),
    "b200_model_encode_images_u8": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "b200_model_encode_images_f32": (C.c_int, [_P, _P, C.c_int, C.c_int, _P]),
    "b200_model_encode_tokens": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "b200_model_encode_images_u8_device": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int]),
    "b200_model_encode_tokens_device": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int]),
    "b200_model_set_stream": (C.c_int, [_P, _P, C.c_int]),
    "b200_model_set_profiling": (C.c_int, [_P, C.c_int]),
    "b200_model_profile": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "b200_model_last_timing": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "b200_debug_gemm": (C.c_int, [C.c_int, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "b200_debug_patch_embed": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, _P, _P, C.c_int, _P]),
    "b200_debug_attention": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "b200_debug_attention_relbias": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "b200_debug_relative_position_buckets": (C.c_int, [C.c_int, _P]),
    "b200_debug_attention_time": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "b200_debug_layernorm": (C.c_int, [C.c_int, _P, _P, _P, C.c_float, C.c_int, C.c_int, _P]),
    "b200_debug_resize": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "b200_jpeg_info": (C.c_int, [_P, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "b200_jpeg_decode_batch": (C.c_int, [C.c_int, _P, _P, C.c_int, _P, _P, _P, _P]),
    "b200_debug_jpeg_decode_host": (C.c_int, [_P, C.c_size_t, _P, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "b200_tokenizer_create_wordpiece": (C.c_int, [C.c_char_p, C.c_size_t, C.c_int, C.POINTER(_P)]),
    "b200_tokenizer_create_wordpiece_special": (C.c_int, [C.c_char_p, C.c_size_t, C.c_int, C.c_char_p, C.c_char_p,
                                                          C.c_char_p, C.c_char_p, C.POINTER(_P)]),
    "b200_tokenizer_create_clip_bpe": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(_P)]),
    "b200_tokenizer_destroy": (C.c_int, [_P]),
    "b200_tokenizer_vocab_size": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "b200_tokenizer_encode": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, _P, _P, C.POINTER(C.c_int)]),
    "b200_fuse_vectors": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "b200_interpolate_vectors": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, C.POINTER(C.c_int)]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib_path() -> Path:
    env = os.environ.get("MARQO_B200_LIB")
    return Path(env) if env else Path(__file__).resolve().parent / _LIB_NAME


def load() -> C.CDLL:
    """Load libmarqo_b200.so once.  Raises NativeLibraryMissing if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = lib_path()
        if not path.exists():
            raise NativeLibraryMissing(
                f"{path} not found: the CUDA extension has not been built (run `python -m marqo_b200.build`). "
                "marqo_b200 has no CPU fallback.")
        lib = C.CDLL(str(path))
        for name, (restype, argtypes) in _SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here == header/library drift
            fn.restype = restype
            fn.argtypes = argtypes
        if lib.b200_abi_version() != 1:
            raise NativeLibraryMissing(f"{path}: ABI version {lib.b200_abi_version()} != 1")
        _lib = lib
        return lib


def check(status: int) -> None:
    if status != OK:
        msg = load().b200_last_error()
        raise NativeError(status, msg.decode("utf-8", "replace") if msg else "")


def device_count() -> int:
    n = C.c_int(0)
    check(load().b200_device_count(C.byref(n)))
    return n.value
