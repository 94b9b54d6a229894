"""Batched entry points (the path that is actually fast) over the C ABI.

Two families:
* ``*_host``   -- numpy / bytes in host memory (``memKind = K4LZ4_MEM_HOST``): the call a
  host-language binding makes; copies H2D/D2H inside.
* ``*_device`` -- raw device pointers (``memKind = K4LZ4_MEM_DEVICE``), e.g. from
  ``torch.Tensor.data_ptr()``; only enqueues kernels on the given CUDA stream.
No torch types cross the ABI; torch is used by callers purely as a device allocator.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np

import ctypes as C

from . import _native as N


def _i64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.int64)


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.int32)


# ---- flat host API: caller supplies base buffers + offset/length arrays ------------------------

def encode_batch_flat_host(src: np.ndarray, src_off, src_len, dst: np.ndarray, dst_off, dst_cap,
                           level: int = 0, device: int = 0) -> np.ndarray:
    src_off, dst_off, src_len, dst_cap = _i64(src_off), _i64(dst_off), _i32(src_len), _i32(dst_cap)
    n = int(src_len.shape[0])
    out = np.full(n, -1, dtype=np.int32)
    N.check(N.lib().k4lz4_encode_batch(src.ctypes.data, src_off.ctypes.data, src_len.ctypes.data,
                                       dst.ctypes.data, dst_off.ctypes.data, dst_cap.ctypes.data,
                                       out.ctypes.data, n, int(level), N.MEM_HOST, None, int(device)))
    return out


def decode_batch_flat_host(src: np.ndarray, src_off, src_len, dst: np.ndarray, dst_off, dst_cap,
                           device: int = 0) -> np.ndarray:
    src_off, dst_off, src_len, dst_cap = _i64(src_off), _i64(dst_off), _i32(src_len), _i32(dst_cap)
    n = int(src_len.shape[0])
    out = np.full(n, -1, dtype=np.int32)
    N.check(N.lib().k4lz4_decode_batch(src.ctypes.data, src_off.ctypes.data, src_len.ctypes.data,
                                       dst.ctypes.data, dst_off.ctypes.data, dst_cap.ctypes.data,
                                       out.ctypes.data, n, N.MEM_HOST, None, int(device)))
    return out


# ---- list-of-buffers host API (convenience for tests and small batches) ------------------------

def _pack(bufs: Sequence) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    arrs = [b if isinstance(b, np.ndarray) else np.frombuffer(b, dtype=np.uint8) for b in bufs]
    lens = np.array([a.shape[0] for a in arrs], dtype=np.int32)
    offs = np.zeros(len(arrs), dtype=np.int64)
    if len(arrs):
        offs[1:] = np.cumsum(lens[:-1], dtype=np.int64)
    base = np.concatenate(arrs) if len(arrs) and int(lens.sum()) else np.zeros(1, dtype=np.uint8)
    if base.dtype != np.uint8:
        base = base.astype(np.uint8)
    return np.ascontiguousarray(base), offs, lens


def encode_batch_host(blocks: Sequence, caps: Sequence[int] | None = None, level: int = 0,
                      device: int = 0):
    """-> (list[bytes], outLen int32[n]); caps default to MaximumOutputSize(len)."""
    src, so, sl = _pack(blocks)
    if caps is None:
        caps = [N.lib().k4lz4_max_output_size(int(x)) for x in sl]
    dc = _i32(caps)
    do = np.zeros(len(dc), dtype=np.int64)
    if len(dc):
        do[1:] = np.cumsum(np.maximum(dc[:-1], 0), dtype=np.int64)
    dst = np.full(int(np.maximum(dc, 0).sum()) + 1, 0xCD, dtype=np.uint8)
    out = encode_batch_flat_host(src, so, sl, dst, do, dc, level, device)
    res = [dst[do[i]:do[i] + out[i]].tobytes() if out[i] > 0 else b"" for i in range(len(dc))]
    return res, out


def decode_batch_host(blocks: Sequence, caps: Sequence[int], device: int = 0):
    """-> (list[bytes], outLen int32[n])."""
    src, so, sl = _pack(blocks)
    dc = _i32(caps)
    do = np.zeros(len(dc), dtype=np.int64)
    if len(dc):
        do[1:] = np.cumsum(np.maximum(dc[:-1], 0), dtype=np.int64)
    dst = np.full(int(np.maximum(dc, 0).sum()) + 1, 0xCD, dtype=np.uint8)
    out = decode_batch_flat_host(src, so, sl, dst, do, dc, device)
    res = [dst[do[i]:do[i] + out[i]].tobytes() if out[i] > 0 else b"" for i in range(len(dc))]
    return res, out


def pickle_batch_host(messages: Sequence, level: int = 0, device: int = 0):
    """LZ4Pickler.Pickle over a batch -> (list[bytes], outLen int32[n])."""
    src, so, sl = _pack(messages)
    n = len(sl)
    bound = np.where(sl > 0, sl.astype(np.int64) + 1, 0)
    do = np.zeros(n, dtype=np.int64)
    if n:
        do[1:] = np.cumsum(bound[:-1])
    dst = np.full(int(bound.sum()) + 1, 0xCD, dtype=np.uint8)
    out = np.full(n, -1, dtype=np.int32)
    N.check(N.lib().k4lz4_pickle_batch(src.ctypes.data, so.ctypes.data, sl.ctypes.data,
                                       dst.ctypes.data, do.ctypes.data, out.ctypes.data,
                                       n, int(level), N.MEM_HOST, None, int(device)))
    res = [dst[do[i]:do[i] + out[i]].tobytes() if out[i] > 0 else b"" for i in range(n)]
    return res, out


def pickle_writer_batch_host(messages: Sequence, level: int = 0, device: int = 0):
    """LZ4Pickler.Pickle<TBufferWriter> over a batch -> (list[bytes], outLen int32[n]): what the
    reference would have advanced each writer by (LZ4Pickler.pickle.cs:113-148)."""
    src, so, sl = _pack(messages)
    n = len(sl)
    L = N.lib()
    bound = np.array([L.k4lz4_pickle_writer_bound(int(v)) for v in sl], dtype=np.int64)
    do = np.zeros(n, dtype=np.int64)
    if n:
        do[1:] = np.cumsum(bound[:-1])
    dst = np.full(int(bound.sum()) + 1, 0xCD, dtype=np.uint8)
    out = np.full(n, -1, dtype=np.int32)
    N.check(L.k4lz4_pickle_writer_batch(src.ctypes.data, so.ctypes.data, sl.ctypes.data,
                                        dst.ctypes.data, do.ctypes.data, out.ctypes.data,
                                        n, int(level), N.MEM_HOST, None, int(device)))
    res = [dst[do[i]:do[i] + out[i]].tobytes() if out[i] > 0 else b"" for i in range(n)]
    return res, out


def unpickled_size_batch_host(pickles: Sequence, device: int = 0) -> np.ndarray:
    src, so, sl = _pack(pickles)
    n = len(sl)
    out = np.full(n, -1, dtype=np.int32)
    N.check(N.lib().k4lz4_unpickled_size_batch(src.ctypes.data, so.ctypes.data, sl.ctypes.data,
                                               out.ctypes.data, n, N.MEM_HOST, None, int(device)))
    return out


def unpickle_batch_host(pickles: Sequence, outputs: Sequence[np.ndarray] | None = None,
                        device: int = 0):
    """With ``outputs`` (writable uint8 arrays, one per message): fills them, returns outLen.
    Without: sizes are taken from UnpickledSize and (list[bytes], outLen) is returned."""
    src, so, sl = _pack(pickles)
    n = len(sl)
    if outputs is None:
        sizes = unpickled_size_batch_host(pickles, device)
        dl = np.where(sizes > 0, sizes, 0).astype(np.int32)
    else:
        dl = np.array([o.shape[0] for o in outputs], dtype=np.int32)
    do = np.zeros(n, dtype=np.int64)
    if n:
        do[1:] = np.cumsum(dl[:-1], dtype=np.int64)
    dst = np.full(int(dl.sum()) + 1, 0xCD, dtype=np.uint8)
    out = np.full(n, -1, dtype=np.int32)
    N.check(N.lib().k4lz4_unpickle_batch(src.ctypes.data, so.ctypes.data, sl.ctypes.data,
                                         dst.ctypes.data, do.ctypes.data, dl.ctypes.data,
                                         out.ctypes.data, n, N.MEM_HOST, None, int(device)))
    if outputs is None:
        res = [dst[do[i]:do[i] + out[i]].tobytes() if out[i] > 0 else b"" for i in range(n)]
        # a message whose header was corrupt reports R_CORRUPT in `sizes`; keep that verdict
        out = np.where(sizes == N.R_CORRUPT, N.R_CORRUPT, out).astype(np.int32)
        return res, out
    for i, o in enumerate(outputs):
        if out[i] > 0:
            o[:out[i]] = dst[do[i]:do[i] + out[i]]
    return out


# ---- device-pointer API ----------------------------------------------------------------------------

def encode_batch_device(src_ptr: int, src_off_ptr: int, src_len_ptr: int, dst_ptr: int,
                        dst_off_ptr: int, dst_cap_ptr: int, out_len_ptr: int, n: int,
                        level: int = 0, stream: int = 0, device: int = -1) -> None:
    N.check(N.lib().k4lz4_encode_batch(src_ptr, src_off_ptr, src_len_ptr, dst_ptr, dst_off_ptr,
                                       dst_cap_ptr, out_len_ptr, int(n), int(level), N.MEM_DEVICE,
                                       stream or None, int(device)))


def decode_batch_device(src_ptr: int, src_off_ptr: int, src_len_ptr: int, dst_ptr: int,
                        dst_off_ptr: int, dst_cap_ptr: int, out_len_ptr: int, n: int,
                        stream: int = 0, device: int = -1) -> None:
    N.check(N.lib().k4lz4_decode_batch(src_ptr, src_off_ptr, src_len_ptr, dst_ptr, dst_off_ptr,
                                       dst_cap_ptr, out_len_ptr, int(n), N.MEM_DEVICE,
                                       stream or None, int(device)))


def pickle_batch_device(src_ptr, src_off_ptr, src_len_ptr, dst_ptr, dst_off_ptr, out_len_ptr, n,
                        level: int = 0, stream: int = 0, device: int = -1) -> None:
    N.check(N.lib().k4lz4_pickle_batch(src_ptr, src_off_ptr, src_len_ptr, dst_ptr, dst_off_ptr,
                                       out_len_ptr, int(n), int(level), N.MEM_DEVICE,
                                       stream or None, int(device)))


def unpickle_batch_device(src_ptr, src_off_ptr, src_len_ptr, dst_ptr, dst_off_ptr, dst_len_ptr,
                          out_len_ptr, n, stream: int = 0, device: int = -1) -> None:
    N.check(N.lib().k4lz4_unpickle_batch(src_ptr, src_off_ptr, src_len_ptr, dst_ptr, dst_off_ptr,
                                         dst_len_ptr, out_len_ptr, int(n), N.MEM_DEVICE,
                                         stream or None, int(device)))


def unpickled_size_batch_device(src_ptr, src_off_ptr, src_len_ptr, out_size_ptr, n,
                                stream: int = 0, device: int = -1) -> None:
    N.check(N.lib().k4lz4_unpickled_size_batch(src_ptr, src_off_ptr, src_len_ptr, out_size_ptr,
                                               int(n), N.MEM_DEVICE, stream or None, int(device)))


# ---- synthetic workloads -------------------------------------------------------------------------------

def synth_host(n_blocks: int, block_size: int, match_permille: int, seed: int = 1234,
               first_block: int = 0) -> np.ndarray:
    buf = np.empty(int(n_blocks) * int(block_size), dtype=np.uint8)
    N.check(N.lib().k4lz4_synth_host(buf.ctypes.data, int(n_blocks), int(block_size),
                                     int(match_permille), int(seed), int(first_block)))
    return buf


def synth_device(ptr: int, n_blocks: int, block_size: int, match_permille: int, seed: int = 1234,
                 first_block: int = 0, stream: int = 0, device: int = -1) -> None:
    N.check(N.lib().k4lz4_synth_device(ptr, int(n_blocks), int(block_size), int(match_permille),
                                       int(seed), int(first_block), stream or None, int(device)))


def copy_blocks_device(src_ptr: int, src_off_ptr: int, dst_ptr: int, dst_off_ptr: int, len_ptr: int,
                       n: int, stream: int = 0, device: int = -1) -> None:
    N.check(N.lib().k4lz4_copy_blocks_device(src_ptr, src_off_ptr, dst_ptr, dst_off_ptr, len_ptr,
                                             int(n), stream or None, int(device)))


def decode_stats(device: int = 0, reset: bool = False) -> dict:
    """Decoder path counters (k4lz4_decode_stats): which engine decoded how many blocks."""
    v = (C.c_uint64 * 4)()
    N.check(N.lib().k4lz4_decode_stats(device, C.addressof(v), int(reset)))
    return {"tile": int(v[0]), "tile_big": int(v[1]), "generic": int(v[2]), "repair_walks": int(v[3])}


def encode_stats(device: int = 0, reset: bool = False) -> dict:
    """Encoder path counters (k4lz4_encode_stats): which warps encoded how many blocks."""
    v = (C.c_uint64 * 3)()
    N.check(N.lib().k4lz4_encode_stats(device, C.addressof(v), int(reset)))
    return {"shared": int(v[0]), "global": int(v[1]), "u32": int(v[2])}


def decode_dict_batch_host(blocks: Sequence, caps: Sequence[int], dicts: Sequence, device: int = 0):
    """LZ4Codec.Decode(source, target, dictionary) over a batch (k4lz4_decode_dict_batch, host memory).
    Returns (list of bytes, int32 results)."""
    src, so, sl = _pack(blocks)
    dic, do, dl = _pack(dicts)
    n = len(sl)
    caps = _i32(caps)
    doff = np.zeros(n, dtype=np.int64)
    if n > 1:
        doff[1:] = np.cumsum(np.maximum(caps[:-1], 0).astype(np.int64))
    dst = np.zeros(int(np.maximum(caps, 0).sum()) + 16, dtype=np.uint8)
    out = np.zeros(n, dtype=np.int32)
    N.check(N.lib().k4lz4_decode_dict_batch(src.ctypes.data, so.ctypes.data, sl.ctypes.data, dst.ctypes.data,
                                            doff.ctypes.data, caps.ctypes.data, dic.ctypes.data, do.ctypes.data,
                                            dl.ctypes.data, out.ctypes.data, n, N.MEM_HOST, None, int(device)))
    return [dst[doff[i]:doff[i] + max(int(out[i]), 0)].tobytes() for i in range(n)], out


def partial_decode_batch_host(blocks: Sequence, targets: Sequence[int], device: int = 0):
    """LZ4Codec.PartialDecode over a batch (k4lz4_partial_decode_batch, host memory)."""
    src, so, sl = _pack(blocks)
    n = len(sl)
    tg = _i32(targets)
    doff = np.zeros(n, dtype=np.int64)
    if n > 1:
        doff[1:] = np.cumsum(np.maximum(tg[:-1], 0).astype(np.int64))
    dst = np.zeros(int(np.maximum(tg, 0).sum()) + 16, dtype=np.uint8)
    out = np.zeros(n, dtype=np.int32)
    N.check(N.lib().k4lz4_partial_decode_batch(src.ctypes.data, so.ctypes.data, sl.ctypes.data, dst.ctypes.data,
                                               doff.ctypes.data, tg.ctypes.data, out.ctypes.data, n,
                                               N.MEM_HOST, None, int(device)))
    return [dst[doff[i]:doff[i] + max(int(out[i]), 0)].tobytes() for i in range(n)], out
