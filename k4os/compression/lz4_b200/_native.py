"""ctypes binding of libk4lz4.so (include/k4lz4.h).  Fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libk4lz4.so")

OK = 0
E_NODEVICE, E_CUDA, E_ARG, E_NOMEM = -100, -101, -102, -103
R_DELEGATE = -2
R_CORRUPT = -1000
MEM_HOST, MEM_DEVICE = 0, 1
ALL_DEVICES = -1

# every symbol include/k4lz4.h declares (tests/test_abi.py checks the .so exports them all)
SYMBOLS = [
    "k4lz4_codec_version", "k4lz4_device_count", "k4lz4_last_error", "k4lz4_max_output_size",
    "k4lz4_encode", "k4lz4_decode", "k4lz4_encode_batch", "k4lz4_decode_batch",
    "k4lz4_pickle_bound", "k4lz4_pickle_batch", "k4lz4_unpickled_size_batch",
    "k4lz4_unpickle_batch", "k4lz4_synth_host", "k4lz4_synth_device", "k4lz4_launch_count",
    "k4lz4_copy_blocks_device", "k4lz4_decode_stats",
    "k4lz4_decode_dict", "k4lz4_partial_decode", "k4lz4_decode_dict_batch", "k4lz4_partial_decode_batch",
    "k4lz4_pickle_writer_bound", "k4lz4_pickle_writer_batch", "k4lz4_encode_x32", "k4lz4_encode_batch_x32",
    "k4lz4_xxh32", "k4lz4_xxh32_batch", "k4lz4_encode_stats",
]


class NativeLibraryMissing(RuntimeError):
    pass


class K4Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libk4lz4 error {code}: {msg}")
        self.code = code


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise NativeLibraryMissing(
            f"{SO_PATH} not found: build it with `python -m k4os.compression.lz4_b200.build` "
            "(or __graft_entry__.build()). There is no CPU fallback by design.")
    L = C.CDLL(SO_PATH)
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    L.k4lz4_codec_version.restype = i32
    L.k4lz4_device_count.restype = i32
    L.k4lz4_last_error.restype = C.c_char_p
    L.k4lz4_launch_count.restype = i64
    L.k4lz4_max_output_size.argtypes = [i32]; L.k4lz4_max_output_size.restype = i32
    L.k4lz4_pickle_bound.argtypes = [i32]; L.k4lz4_pickle_bound.restype = i32
    L.k4lz4_encode.argtypes = [vp, i32, vp, i32, i32]; L.k4lz4_encode.restype = i32
    L.k4lz4_decode.argtypes = [vp, i32, vp, i32]; L.k4lz4_decode.restype = i32
    L.k4lz4_encode_batch.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, i32]
    L.k4lz4_encode_batch.restype = i32
    L.k4lz4_decode_batch.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, i32]
    L.k4lz4_decode_batch.restype = i32
    L.k4lz4_pickle_batch.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, i32]
    L.k4lz4_pickle_batch.restype = i32
    L.k4lz4_unpickled_size_batch.argtypes = [vp, vp, vp, vp, i32, i32, vp, i32]
    L.k4lz4_unpickled_size_batch.restype = i32
    L.k4lz4_unpickle_batch.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, i32]
    L.k4lz4_unpickle_batch.restype = i32
    L.k4lz4_synth_host.argtypes = [vp, i64, i32, i32, u64, i64]; L.k4lz4_synth_host.restype = i32
    L.k4lz4_synth_device.argtypes = [vp, i64, i32, i32, u64, i64, vp, i32]
    L.k4lz4_synth_device.restype = i32
    L.k4lz4_copy_blocks_device.argtypes = [vp, vp, vp, vp, vp, i32, vp, i32]
    L.k4lz4_copy_blocks_device.restype = i32
    L.k4lz4_decode_stats.argtypes = [i32, vp, i32]; L.k4lz4_decode_stats.restype = i32
    L.k4lz4_encode_stats.argtypes = [i32, vp, i32]; L.k4lz4_encode_stats.restype = i32
    L.k4lz4_decode_dict.argtypes = [vp, i32, vp, i32, vp, i32]; L.k4lz4_decode_dict.restype = i32
    L.k4lz4_partial_decode.argtypes = [vp, i32, vp, i32]; L.k4lz4_partial_decode.restype = i32
    L.k4lz4_decode_dict_batch.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, i32]
    L.k4lz4_decode_dict_batch.restype = i32
    L.k4lz4_partial_decode_batch.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, i32]
    L.k4lz4_partial_decode_batch.restype = i32
    L.k4lz4_encode_x32.argtypes = [vp, i32, vp, i32, i32]; L.k4lz4_encode_x32.restype = i32
    L.k4lz4_encode_batch_x32.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, i32]
    L.k4lz4_encode_batch_x32.restype = i32
    L.k4lz4_xxh32.argtypes = [vp, i64, C.c_uint32]; L.k4lz4_xxh32.restype = C.c_uint32
    L.k4lz4_xxh32_batch.argtypes = [vp, vp, vp, C.c_uint32, vp, i32, i32, vp, i32]; L.k4lz4_xxh32_batch.restype = i32
    L.k4lz4_pickle_writer_bound.argtypes = [i32]; L.k4lz4_pickle_writer_bound.restype = i32
    L.k4lz4_pickle_writer_batch.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, i32]
    L.k4lz4_pickle_writer_batch.restype = i32
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != OK:
        raise K4Error(rc, lib().k4lz4_last_error().decode("utf-8", "replace"))
