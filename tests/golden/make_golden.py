"""Generates the committed golden fixtures from a checkout of the reference (K4os.Compression.LZ4, whose
orig/ holds the upstream lz4 C sources):

    python tests/golden/make_golden.py <reference checkout>

1. issue64_block0.{lz4,bin}: the reference's own golden DECODE vector -- block #0 of
   <reference>/assets/issue64/input.dat (a "bv41" container: 12-byte header at byte 20,
   14 505 compressed bytes -> 65 536 bytes == output.dat[0:65536]); exercised by the
   reference's Issue64.cs:16-55.  issue64_block1.{lz4,bin}: block #1 of the same file (366 -> 3 034
   bytes), which only decodes with block #0's output as external dictionary.
2. encode_rows.json: known-answer rows for LZ4Codec.Encode at L00_FAST in the style of the
   reference's ChecksumBlockTests.cs:185-216 (exact length, Adler-32 of the compressed bytes,
   first 60 compressed bytes base64) over the deterministic inputs of tests/inputs.py,
   produced -- like the reference's own rows (playground/SharedSources/app.cpp:94-97) -- by the
   upstream C engine orig/lib/lz4.c compiled as-is (oracle/_ref/libk4ref.so), including
   limited-output capacities and the expected return codes.
3. ref_engine.npz: that engine's results (return value, CRC-32 of the output) on every case set of
   tests/inputs.py -- encode, decode of malformed streams, dictionary and partial decode, XXH32, the
   data generator, and upstream lz4frame.c's frames -- which the tests compare the oracle and the
   frame writer with.  Needs libk4lz4.so built (the synth inputs), no GPU.
4. hc_blocks.npz: blocks written by upstream LZ4_compress_HC (orig/lib/lz4hc.c) at levels 3, 9 and 12 --
   fewer literals, longer matches and larger offsets than the fast encoder writes -- with the
   (kind, size, seed, level) and CRC-32 of their raw data, which tests regenerate (inputs.hc_raw).
"""
import base64
import ctypes
import hashlib
import json
import os
import struct
import subprocess
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from tests import inputs  # noqa: E402


def main(ref_dir):
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "REF=" + os.path.abspath(ref_dir)], check=True)
    R = oracle.Ref()
    # 1. issue64
    blob = open(os.path.join(ref_dir, "assets/issue64/input.dat"), "rb").read()
    expect = open(os.path.join(ref_dir, "assets/issue64/output.dat"), "rb").read()
    assert blob[20:24] == b"bv41"
    usize, csize = struct.unpack("<II", blob[24:32])
    comp = blob[32:32 + csize]
    r, out = R.decode(comp, usize)
    assert r == usize == 65536 and out == expect[:usize]
    open(os.path.join(HERE, "issue64_block0.lz4"), "wb").write(comp)
    open(os.path.join(HERE, "issue64_block0.bin"), "wb").write(expect[:usize])
    # block #1 needs block #0's output as its dictionary (Issue64.cs:39-49)
    pos1 = 32 + csize
    assert blob[pos1:pos1 + 4] == b"bv41"
    usize1, csize1 = struct.unpack("<II", blob[pos1 + 4:pos1 + 12])
    comp1 = blob[pos1 + 12:pos1 + 12 + csize1]
    r1, out1 = R.decode_dict(comp1, usize1, expect[:usize])
    assert r1 == usize1 == 3034 and csize1 == 366 and out1 == expect[usize:usize + usize1]
    assert blob[pos1 + 12 + csize1:pos1 + 16 + csize1] == b"bv4$"
    open(os.path.join(HERE, "issue64_block1.lz4"), "wb").write(comp1)
    open(os.path.join(HERE, "issue64_block1.bin"), "wb").write(out1)

    # 2. encode rows
    rows = []
    sizes = inputs.THRESHOLD_SIZES + inputs.BIG_SIZES
    for kind in inputs.KINDS:
        for n in sizes:
            if kind.startswith("synth") and n < 13:
                continue
            seed = 0xAA if kind == "repeat" else (n * 7 + 1) & 0xFFFF
            data = inputs.gen(kind, n, seed)
            r, c = R.encode(data)
            row = {"kind": kind, "size": n, "seed": seed, "len": r,
                   "adler32": zlib.adler32(c) & 0xFFFFFFFF,
                   "sha256": hashlib.sha256(c).hexdigest(),
                   "head60": base64.b64encode(c[:60]).decode()}
            caps = sorted({c_ for c_ in (n, 1024, r, r - 1, r + 1, max(r // 2, 1), n + n // 255 + 15)
                           if c_ > 0})
            row["limited"] = [[cap, R.encode(data, cap)[0]] for cap in caps]
            rows.append(row)
    json.dump({"engine": "orig/lib/lz4.c LZ4_compress_fast(src,dst,n,cap,1)",
               "lz4_version": R.version(), "rows": rows},
              open(os.path.join(HERE, "encode_rows.json"), "w"), indent=0)
    print(len(rows), "encode rows; issue64 ok")

    # 3. the reference engine's results on the case sets of tests/inputs.py
    P = oracle.Port()
    sets = {}
    for name, rows_of in inputs.ENGINE_SETS.items():
        sets[name] = np.array(rows_of(P, R)[1], dtype=np.int64)

    def upstream_frame(d, bc, cc):
        f = R.frame_compress(d, bc, cc)
        assert R.frame_decompress(f, len(d) + 16) == d
        return f
    sets["frame"] = np.array(inputs.frame_rows(P, upstream_frame)[1], dtype=np.int64)
    np.savez_compressed(inputs.REF_RESULTS, **sets)
    print({k: len(v) for k, v in sets.items()}, "reference results")

    # 4. HC blocks
    hc = R._lib.LZ4_compress_HC
    hc.restype = ctypes.c_int
    hc.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    cols = {k: [] for k in ("kind", "size", "seed", "level", "crc")}
    streams = []
    for kind, size, seed in inputs.HC_INPUTS:
        raw = np.frombuffer(inputs.hc_raw(P, kind, size, seed), dtype=np.uint8)
        for level in (3, 9, 12):
            dst = np.zeros(size + size // 255 + 16, dtype=np.uint8)
            r = hc(raw.ctypes.data, dst.ctypes.data, size, dst.size, level)
            assert r > 0 and P.decode(dst[:r], size) == (size, raw.tobytes()), (kind, size, level)
            streams.append(dst[:r])
            for k, v in zip(cols, (kind, size, seed, level, zlib.crc32(raw))):
                cols[k].append(v)
    off = np.concatenate([[0], np.cumsum([len(s) for s in streams])])
    np.savez_compressed(inputs.HC_BLOCKS, streams=np.concatenate(streams), stream_off=off.astype(np.int64),
                        **{k: np.array(v, dtype=None if k == "kind" else np.int64) for k, v in cols.items()})
    print(len(streams), "HC blocks,", os.path.getsize(inputs.HC_BLOCKS), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
