"""Deterministic test inputs shared by tests/ and tests/golden/make_golden.py.

Modelled on the reference's own test inputs (src/K4os.Compression.LZ4.Tests/
BlockRoundtripTests.cs:63-112: single bytes, repeated bytes incl. 64 KiB of 0xAA, repeated
Lorem text, seeded random bytes) plus sizes around every threshold of the engine
(SURVEY.md section 7 step 1c) and blocks of the library's own synthetic generator.
Everything is reproducible from (kind, size, seed) with numpy only.

The reference engine's results on the case sets below (return value and CRC-32 of the bytes of
every call) are stored in golden/ref_engine.npz; `RefResults` compares an engine's results with them.
"""
from __future__ import annotations

import os
import zlib

import numpy as np

REF_RESULTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_engine.npz")

LOREM = (
    b"Sed ut perspiciatis unde omnis iste natus error sit voluptatem accusantium doloremque "
    b"laudantium, totam rem aperiam, eaque ipsa quae ab illo inventore veritatis et quasi "
    b"architecto beatae vitae dicta sunt explicabo. Nemo enim ipsam voluptatem quia voluptas "
    b"sit aspernatur aut odit aut fugit, sed quia consequuntur magni dolores eos qui ratione "
    b"voluptatem sequi nesciunt. Neque porro quisquam est, qui dolorem ipsum quia dolor sit amet. "
)

THRESHOLD_SIZES = [1, 2, 3, 4, 5, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 31, 32, 33, 63, 64, 65,
                   100, 254, 255, 256, 270, 271, 1005, 1006, 1023, 1024, 1025, 4095, 4096, 4097,
                   32767, 65535, 65536]
BIG_SIZES = [65546, 65547, 65548, 100000, 0x123456 // 8]


def gen(kind: str, size: int, seed: int = 0) -> bytes:
    """kind in: random, repeat, lorem, text2, lowent, synth545, synth435, runs."""
    if size == 0:
        return b""
    if kind == "random":
        return np.random.default_rng(seed).integers(0, 256, size, dtype=np.uint8).tobytes()
    if kind == "repeat":
        return bytes([seed & 0xFF]) * size
    if kind == "lorem":
        return (LOREM * (size // len(LOREM) + 1))[:size]
    if kind == "lowent":      # 2-bit symbols: dense accidental matches, many overlapping copies
        return np.random.default_rng(seed).integers(0, 4, size, dtype=np.uint8).tobytes()
    if kind == "text2":       # word soup: realistic short matches at short distances
        rng = np.random.default_rng(seed)
        words = [bytes(rng.integers(97, 123, int(rng.integers(2, 9)), dtype=np.uint8)) for _ in range(200)]
        out = bytearray()
        while len(out) < size:
            out += words[int(rng.integers(0, 200))] + b" "
        return bytes(out[:size])
    if kind == "runs":        # long runs of one byte separated by noise: long LSIC lengths, offset 1
        rng = np.random.default_rng(seed)
        out = bytearray()
        while len(out) < size:
            out += bytes([int(rng.integers(0, 256))]) * int(rng.integers(1, 3000))
            out += rng.integers(0, 256, int(rng.integers(0, 40)), dtype=np.uint8).tobytes()
        return bytes(out[:size])
    if kind.startswith("synth"):
        from k4os.compression.lz4_b200.batch import synth_host
        mp = int(kind[5:])
        nb = (size + 65535) // 65536
        return synth_host(nb, 65536, mp, seed=1234, first_block=seed).tobytes()[:size]
    raise ValueError(kind)


KINDS = ["random", "repeat", "lorem", "lowent", "text2", "runs", "synth525", "synth435"]


def corpus(sizes=None, kinds=None):
    """Yields (name, bytes) over the cross product, small enough to run in seconds."""
    sizes = THRESHOLD_SIZES if sizes is None else sizes
    kinds = KINDS if kinds is None else kinds
    for k in kinds:
        for n in sizes:
            yield f"{k}-{n}", gen(k, n, seed=(n * 7 + 1) & 0xFFFF if k != "repeat" else 0xAA)


def mutate(stream: bytes, rng: np.random.Generator) -> bytes:
    """One random corruption of a compressed stream (for malformed-input parity)."""
    c = bytearray(stream)
    k = int(rng.integers(0, 5))
    if k == 0 and len(c):
        for _ in range(int(rng.integers(1, 4))):
            c[int(rng.integers(0, len(c)))] = int(rng.integers(0, 256))
    elif k == 1 and len(c) > 1:
        c = c[:int(rng.integers(1, len(c)))]
    elif k == 2:
        c += rng.integers(0, 256, int(rng.integers(1, 9)), dtype=np.uint8).tobytes()
    elif k == 3 and len(c):
        c[int(rng.integers(0, len(c)))] = [0xFF, 0xF0, 0x0F, 0x00][int(rng.integers(0, 4))]
    elif len(c) > 4:
        i = int(rng.integers(0, len(c) - 2))
        c[i + 1] = 0; c[i + 2] = 0          # plant a zero offset somewhere
    return bytes(c)


def uses_zero_offset(stream: bytes) -> bool:
    """True iff the token chain of `stream` contains a match with offset 0 (or cannot be walked).

    The reference accepts such a match -- `match == op >= dst` passes LL64.dec.cs:338 -- and copies
    whatever the destination buffer held before, so the CONTENT of the decoded block is unspecified
    (only the returned length is contractual).  Content comparisons skip exactly these streams; a
    plain `b"\x00\x00" in stream` test would also skip every stream with two zero literals."""
    c = bytes(stream)
    n = len(c)
    p = 0
    try:
        while p < n:
            t = c[p]; p += 1
            lit = t >> 4
            if lit == 15:
                while True:
                    s = c[p]; p += 1; lit += s
                    if s != 255:
                        break
            p += lit
            if p + 2 > n:
                return False
            if c[p] == 0 and c[p + 1] == 0:
                return True
            p += 2
            if (t & 15) == 15:
                while True:
                    s = c[p]; p += 1
                    if s != 255:
                        break
        return False
    except IndexError:
        return True


# ---- case sets whose reference-engine results are stored (golden/make_golden.py) ----------------

def result_row(ret: int, out: bytes = b"") -> tuple[int, int]:
    """What is kept of one engine call: its return value and the CRC-32 of the bytes it produced."""
    return int(ret), zlib.crc32(bytes(out))


class RefResults:
    """The reference engine's recorded results, one (return value, CRC-32) row per call."""

    def __init__(self, path: str = REF_RESULTS):
        with np.load(path) as z:
            self._sets = {k: z[k] for k in z.files}

    def check(self, name: str, labels: list, rows: list) -> None:
        want = self._sets[name]
        got = np.array(rows, dtype=np.int64).reshape(-1, 2)
        n = min(len(got), len(want))
        bad = np.flatnonzero((got[:n] != want[:n]).any(axis=1))
        assert bad.size == 0, (f"{name}: {bad.size} of {n} calls differ from the reference engine; first at "
                               f"{labels[bad[0]]}: got {got[bad[0]].tolist()}, reference {want[bad[0]].tolist()}")
        assert len(got) == len(want), (name, len(got), len(want))


def _decoded(r: int, out: bytes, stream: bytes) -> tuple[int, int]:
    """A decode call's row; the bytes count only where they are specified (not for offset-0 matches)."""
    return result_row(r, out if r > 0 and not uses_zero_offset(stream) else b"")


def corpus_rows(port, eng):
    """Encode of the corpus, then decode of each result at capacities around its size."""
    labels, rows = [], []
    for name, data in corpus(sizes=THRESHOLD_SIZES + BIG_SIZES):
        r, c = eng.encode(data)
        labels.append(name); rows.append(result_row(r, c))
        n = len(data)
        for cap in sorted({n, n + 1, n - 1, 2 * n, max(n - 13, 0)}):
            labels.append((name, cap)); rows.append(result_row(*eng.decode(c, cap)))
    return labels, rows


def malformed_rows(port, eng):
    """Decode of oracle-encoded streams with one random corruption each."""
    rng = np.random.default_rng(7)
    labels, rows = [], []
    for it in range(6000):
        n = int(rng.choice([20, 50, 100, 300, 1000, 5000]))
        kind = ["text2", "lowent", "runs", "random", "lorem"][it % 5]
        c = mutate(port.encode(gen(kind, n, it))[1], rng)
        cap = int(rng.choice([n, n, n + 5, n - 1, 2 * n, n + 64, 0, 1]))
        labels.append((it, kind, n, cap)); rows.append(_decoded(*eng.decode(c, cap), c))
    return labels, rows


def dictionary_rows(port, eng):
    """Decode with an external dictionary of streams whose offsets were mutated to reach into it."""
    rng = np.random.default_rng(5)
    labels, rows = [], []
    for it in range(3000):
        n = int(rng.choice([40, 200, 1000, 5000]))
        kind = ["text2", "lowent", "runs", "lorem", "random"][it % 5]
        c = bytearray(port.encode(gen(kind, n, it))[1])
        dic = gen("text2", int(rng.choice([1, 7, 64, 300, 4096, 70000])), it + 1)
        if it % 3 and len(c) > 8:       # enlarge some offsets so that matches start inside the dictionary
            for _ in range(3):
                i = int(rng.integers(1, len(c) - 2))
                c[i] = int(rng.integers(0, 256))
        cap = int(rng.choice([n, n + 9, n - 1, 2 * n]))
        labels.append((it, kind, n, cap)); rows.append(_decoded(*eng.decode_dict(bytes(c), cap, dic), bytes(c)))
    return labels, rows


def partial_decode_cases(port):
    """(label, data, stream, target, mutated stream): well-formed streams of `data` and one corruption of each."""
    rng = np.random.default_rng(9)
    for it in range(3000):
        n = int(rng.choice([30, 100, 1000, 5000, 70000]))
        kind = ["text2", "lowent", "runs", "lorem", "random"][it % 5]
        data = gen(kind, n, it)
        c = port.encode(data)[1]
        target = int(rng.choice([0, 1, 5, 12, 13, n // 3, n // 2, n - 1, n, n + 1, 2 * n]))
        yield (it, kind, n, target), data, c, target, mutate(c, rng)


def partial_rows(port, eng):
    """Partial decode of well-formed streams."""
    labels, rows = [], []
    for label, _, c, target, _ in partial_decode_cases(port):
        labels.append(label); rows.append(result_row(*eng.partial_decode(c, target)))
    return labels, rows


def datagen_rows(port, eng):
    """The synthetic-data generator (RDG_genBuffer) at several sizes and probabilities."""
    labels, rows = [], []
    for size, mp, lp, seed in [(1 << 20, 0.63, 0.0, 1234), (1 << 20, 0.55, 0.0, 1234), (300001, 0.3, 0.0, 7),
                               (65536, 0.9, 0.25, 99), (1, 0.63, 0.0, 1), (0, 0.63, 0.0, 1)]:
        labels.append((size, mp, lp, seed)); rows.append(result_row(size, eng.datagen(size, mp, lp, seed).tobytes()))
    return labels, rows


def xxh32_rows(port, eng):
    """XXH32, the checksum of the LZ4 Frame container, around its 16-byte stripes."""
    rng = np.random.default_rng(2)
    labels, rows = [], []
    for n in [0, 1, 3, 4, 15, 16, 17, 31, 32, 33, 100, 65536, 100001]:
        a = rng.integers(0, 256, n, dtype=np.uint8)
        for seed in (0, 1, 0xDEADBEEF):
            labels.append((n, seed)); rows.append(result_row(eng.xxh32(a, seed)))
    return labels, rows


def frame_datas(port) -> list[bytes]:
    """Frame contents: empty, one byte, one short block, several blocks, an incompressible block, datagen."""
    return [b"", b"a", gen("text2", 1000, 1), gen("synth525", 3 * 65536 + 777, 2),
            gen("random", 65536 + 5, 3), port.datagen(5 * 65536, 0.63).tobytes()]


def frame_rows(port, write_frame):
    """Frames of independent 64 KiB blocks, `write_frame(data, block_checksum, content_checksum) -> bytes`."""
    labels, rows = [], []
    for d in frame_datas(port):
        for bc in (False, True):
            for cc in (False, True):
                f = write_frame(d, bc, cc)
                labels.append((len(d), bc, cc)); rows.append(result_row(len(f), f))
    return labels, rows


def fuzz_encode_rows(port, eng, count: int = 600):
    """Encode of arbitrary byte strings -- uniform bytes, short units repeated, small alphabets -- into the
    bound and into capacities around the compressed size."""
    rng = np.random.default_rng(17)
    labels, rows = [], []
    for i in range(count):
        k = i % 3
        if k == 0:
            data = rng.integers(0, 256, int(rng.integers(0, 601)), dtype=np.uint8).tobytes()
        elif k == 1:
            unit = rng.integers(0, 256, int(rng.integers(1, 41)), dtype=np.uint8).tobytes()
            data = (unit * int(rng.integers(1, 301)))[:5000]
        else:
            hi = int(rng.choice([2, 4, 16, 256]))
            data = rng.integers(0, hi, int(rng.integers(0, 3001)), dtype=np.uint8).tobytes()
        slack = int(rng.integers(0, 41))
        full = eng.encode(data)
        labels.append((i, len(data))); rows.append(result_row(*full))
        n = len(data)
        if full[0] > 0:
            assert eng.decode(full[1], n) == (n, data)
        for cap in sorted({max(full[0] - slack, 1), n, 1024, full[0] + slack}):
            if n == 0 or cap <= 0:
                continue
            labels.append((i, n, cap)); rows.append(result_row(*eng.encode(data, cap)))
    return labels, rows


def fuzz_decode_rows(port, eng, count: int = 1200):
    """Decode of arbitrary byte strings -- uniform bytes, and bytes drawn mostly from the values that steer
    the token parse (0x00, 0x0F, 0xF0, 0xFF, small offsets)."""
    rng = np.random.default_rng(19)
    palette = np.array([0x00, 0x01, 0x04, 0x0F, 0x10, 0x1F, 0xF0, 0xFF], dtype=np.uint8)
    labels, rows = [], []
    for i in range(count):
        n = int(rng.integers(0, 301))
        if i % 2:
            s = rng.integers(0, 256, n, dtype=np.uint8)
        else:
            s = np.where(rng.random(n) < 0.6, rng.choice(palette, n), rng.integers(0, 256, n)).astype(np.uint8)
        stream, cap = s.tobytes(), int(rng.integers(0, 701))
        labels.append((i, n, cap)); rows.append(_decoded(*eng.decode(stream, cap), stream))
    return labels, rows


# ---- blocks written by upstream LZ4_compress_HC (golden/hc_blocks.npz) ------------------------------

HC_BLOCKS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hc_blocks.npz")
HC_INPUTS = [(kind, size, seed) for seed, (kind, size) in enumerate(
    [(k, n) for k in ("text2", "lowent", "runs", "datagen63") for n in (65536, 5000, 300, 40)], start=101)]


def hc_raw(port, kind: str, size: int, seed: int) -> bytes:
    """The raw data of an HC block: `gen`, or the reference data generator at match probability 0.63."""
    if kind == "datagen63":
        return port.datagen(size, 0.63, 0.0, seed).tobytes()
    return gen(kind, size, seed)


def hc_blocks(port):
    """-> [(kind, size, level, stream, raw)] of golden/hc_blocks.npz, raw data regenerated and CRC-checked."""
    with np.load(HC_BLOCKS) as z:
        f = {k: z[k] for k in z.files}
    out = []
    for i in range(len(f["kind"])):
        kind, size, seed = str(f["kind"][i]), int(f["size"][i]), int(f["seed"][i])
        raw = hc_raw(port, kind, size, seed)
        assert zlib.crc32(raw) == int(f["crc"][i]), (kind, size, seed)
        stream = f["streams"][f["stream_off"][i]:f["stream_off"][i + 1]].tobytes()
        out.append((kind, size, int(f["level"][i]), stream, raw))
    return out


# every set above that an engine computes alone, by the name its results are stored under
ENGINE_SETS = {"corpus": corpus_rows, "malformed": malformed_rows, "dictionary": dictionary_rows,
               "partial": partial_rows, "datagen": datagen_rows, "xxh32": xxh32_rows,
               "fuzz_encode": fuzz_encode_rows, "fuzz_decode": fuzz_decode_rows}
