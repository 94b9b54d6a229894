"""The block decoder on composed LZ4 streams aimed at the tile decoder's scheduling, limits and alignment.

Every block here is built from an explicit plan (tests/compose.py), so its raw data is known exactly and
independently of any decoder.  The CPU tests prove each plan family against the restatement of the
reference decoder (oracle.Port).  The GPU tests decode each family as one batch through
batch.decode_batch_device, compare return codes and bytes with the plan and with Port, check that the
bytes around every destination slot stay 0xCD, and assert which engine decoded how many blocks
(decode_stats: small-stage tile kernel, big-stage tile kernel, exact generic decoder): the tile path
declines whatever it is unsure of and the generic decoder then still gets the right answer, so only the
counters show a block that left the tile path.

Constants of csrc/decode_tile.cuh the plans aim at: steps of 512 sequences (16 warps of 32), parse
segments of 80 stream bytes on the small stage and 128 on the big one, the small stage takes a block when
`shift + n + 16 <= 40960` (shift = source address mod 16), at most 16 384 sequences, 65 535 stream bytes
and 65 536 output bytes, and the descriptors (4 bytes per sequence, growing down from the end of the
64 KiB + 32 tile) leave the jump table intact while `shift + n + 4 + 4 N <= 65568`.
"""
from __future__ import annotations

import collections
import functools
from typing import NamedTuple

import numpy as np
import pytest

from tests import compose as K
from tests import inputs

STEP, SEG_SMALL, SEG_BIG = 512, 80, 128
STAGE_SMALL, DT_NMAX, DT_MAX_SRC, TILE = 40960, 16384, 65535, 65536

# LZ4Codec.Decode of the plans that break one end rule, at capacity = decoded size (oracle.Port).  A zero
# offset passes the reference's bounds test and copies whatever the destination held: only the length counts.
BROKEN_CODES = {"mflimit": -1, "lastliterals": -1, "offset_zero": 58, "offset_far": -1, "trailing_match": -1}


class Case(NamedTuple):
    stream: bytes
    cap: int
    want: int                 # expected return code
    raw: bytes | None         # expected output when the block decodes (None: compare with Port only)
    path: str                 # engine expected to decode it: "tile", "tile_big" or "generic"
    shift: int = 0            # source address mod 16
    dshift: int = 0           # destination address mod 16


def route(n: int, O: int, N: int, cap: int, shift: int = 0) -> str:
    """The engine that decodes a block that is valid at `cap`: the tile path whenever its limits allow."""
    if n > DT_MAX_SRC or O > TILE or N > DT_NMAX or O > cap:
        return "generic"
    return "tile_big" if shift + n + 16 > STAGE_SMALL else "tile"


def clean_case(seqs, tail, cap=None, shift=0, dshift=0, path=None) -> Case:
    assert K.clean(seqs, tail)
    b = K.compose(seqs, tail)
    O = len(b.raw)
    cap = O if cap is None else cap
    if path is None:
        path = route(len(b.stream), O, len(b.tokens), cap, shift)
    ok = cap >= O
    return Case(b.stream, cap, O if ok else -1, b.raw if ok else None, path, shift, dshift)


def pad_stream(seqs, lit, n: int) -> bytes:
    return K.pad_to_stream_size(seqs, lit, n)


# ---- plan families ---------------------------------------------------------------------------------------

def _fill(lit, count, pos=0):
    return K.far_fillers(lit, count, pos)


def _out(seqs):
    return sum(len(l) + m for l, _, m in seqs)


@functools.lru_cache(maxsize=None)
def near_family():
    """Near-match scheduling: dependency chains, sources straddling a step start, matches that read their own
    literals, and every copy branch for overlapping matches, near and far."""
    lit = K.Bytes(1)
    cases = []
    # chains 1..512 deep starting at lane 0 / lane 31 of a warp, in step 0 (no step before) and step 1
    for depth in (1, 31, 32, 33, 511, 512):
        for lane in (0, 31):
            for step in (0, 1):
                for length, overlap in ((4, 0), (33, 0), (7, 3), (40, 0), (20, 12)):
                    if depth * length > 30000:
                        continue
                    pre = _fill(lit, step * STEP + lane)
                    seqs = pre + K.chain(lit, depth, length, overlap)
                    cases.append(clean_case(seqs, K.tail_for(seqs, lit, 9), shift=len(cases) % 16))
    # long chains whose copies take the warp paths: periodic (offset < 160) and sliced (>= 160)
    for depth, length, overlap in ((120, 200, 140), (60, 400, 200), (100, 129, 1)):
        seqs = _fill(lit, STEP + 5) + K.chain(lit, depth, length, overlap)
        cases.append(clean_case(seqs, K.tail_for(seqs, lit)))
    # sources straddling the step start Sr: sequence 512 (lit 0, d == Sr) is a far match; sequence 513 reads a
    # window that ends at Sr + e, i.e. its last byte is Sr - 1 (e = 0, far) or Sr (e = 1, near), then a chain
    for lane in (1, 2, 40, 200):
        for L0, L1 in ((8, 8), (4, 20), (16, 5), (30, 30)):
            for e in (-1, 0, 1, 2, 3):
                pre = _fill(lit, STEP)
                Sr = _out(pre)
                seqs = pre + [(b"", Sr, L0)]                       # d == Sr, reads output [0, L0)
                seqs += _fill(lit, lane - 1, Sr + L0)               # more far matches in the same step
                d = _out(seqs)
                seqs += [(b"", d - (Sr + e - L1), L1)]              # source [Sr + e - L1, Sr + e)
                seqs += K.chain(lit, 40, 6)[1:]                     # continues from that output
                cases.append(clean_case(seqs, K.tail_for(seqs, lit), shift=(lane + e) % 16))
    # matches that read only their own literals, in step 0 and in a later step
    for step in (0, 2):
        seqs = _fill(lit, step * STEP + 3)
        for L in (1, 2, 5, 20, 33, 64):
            for off in sorted({1, 2, L // 2 or 1, L}):
                for ml in (4, 31, 40, 300):
                    seqs.append((lit(L), off, ml))
        cases.append(clean_case(seqs, K.tail_for(seqs, lit)))
    # every offset x length: far (first sequence of step 1 with no literals, so d == Sr) and near (3 literals after)
    offsets = (1, 2, 3, 4, 5, 7, 8, 15, 16, 31, 32, 33, 63, 64, 127, 159, 160, 161, 255, 256)
    lengths = (4, 5, 31, 32, 33, 64, 127, 128, 129, 1000, 20000)
    for off in offsets:
        for ml in lengths:
            seqs = _fill(lit, STEP)
            seqs += [(b"", off, ml), (lit(3), off, ml), (lit(1), off, 4)]
            cases.append(clean_case(seqs, K.tail_for(seqs, lit), shift=(off + ml) % 16, dshift=off % 16))
    return cases


def _long_run_block(lit, k, seg, delta, big, shift):
    """A literal run covering k whole segments, placed so that the next token sits at segment start + delta."""
    seqs = _fill(lit, 7)
    run = k * seg + 3
    for _ in range(4):
        b = K.compose(seqs + [(lit(run), 4, 6)], b"")
        p = b.tokens[-1]                                         # the token after the run
        fix = (delta - p) % seg
        if fix == 0:
            break
        run += fix
    seqs.append((lit(run), 4, 6))
    assert K.compose(seqs, b"").tokens[-1] % seg == delta % seg
    seqs += _fill(lit, 30, _out(seqs))
    seqs.append((lit(2 * seg + 1), 9, 30))                        # a second, shorter run
    if big:                                                       # pad until the big stage takes it
        n = len(K.compose(seqs, b"").stream)
        while n < STAGE_SMALL + 200:
            seqs.append((lit(int(lit.rng.integers(60, 400))), 1 + int(lit.rng.integers(0, 64)), 8))
            n += K.sequence_bytes(len(seqs[-1][0]), 8)
    return clean_case(seqs, K.tail_for(seqs, lit), shift=shift)


@functools.lru_cache(maxsize=None)
def parse_family():
    """Parse and repair: literal runs covering 1..70 segments, the next token at segment start -1/0/+1, on the
    small stage (80-byte segments) and padded onto the big stage (128-byte segments)."""
    lit = K.Bytes(2)
    cases = []
    for big, seg in ((False, SEG_SMALL), (True, SEG_BIG)):
        for k in (1, 2, 31, 32, 33, 64, 70):
            for delta in (-1, 0, 1):
                cases.append(_long_run_block(lit, k, seg, delta, big, shift=(k + delta) % 16))
    for c in cases:
        assert c.path == ("tile_big" if len(c.stream) + c.shift + 16 > STAGE_SMALL else "tile")
    return cases


def _literal_heavy(lit, n, shift=0, lits=200):
    """A clean block of exactly n stream bytes, mostly literals with short matches between them."""
    seqs, size = [], 1
    while size < n - 3 * lits:
        seqs.append((lit(lits), 1 + int(lit.rng.integers(0, lits)), 4 + int(lit.rng.integers(0, 30))))
        size += K.sequence_bytes(lits, seqs[-1][2])
    return seqs, pad_stream(seqs, lit, n)


@functools.lru_cache(maxsize=None)
def limits_family():
    lit = K.Bytes(3)
    cases = []
    # The sequence limit.  A valid block of N sequences decodes to at least 4 (N - 1) + 1 + 5 bytes: every match is
    # >= 4 bytes, the first sequence needs a literal, and a sequence with a match needs 8 stream bytes after its
    # literals, which short last matches leave to >= 5 terminal literals.  So 16 383 sequences reach 65 536 bytes
    # (with room behind them: the last match starts 9 bytes before the end) and 16 384 do not; the same block
    # with 16 384 sequences and no terminal literals is rejected, and 16 385 sequences are valid beyond the tile.
    rng = np.random.default_rng(3)
    seqs, pos = [(lit(3), 3, 4)], 7
    for _ in range(DT_NMAX - 3):
        seqs.append((b"", int(rng.integers(1, min(pos, 300) + 1)), 4))
        pos += 4
    b = K.compose(seqs, lit(5))
    assert len(b.tokens) == DT_NMAX - 1 and len(b.raw) == TILE
    for cap, dshift in ((70000, 0), (65539, 15), (65538, 9)):
        ok = cap >= TILE + 3
        cases.append(Case(b.stream, cap, TILE if ok else -1, b.raw if ok else None, "tile_big" if ok else "generic",
                          dshift % 4, dshift))
    b = K.compose([(lit(4), 4, 4)] + [(b"", 4, 4)] * (DT_NMAX - 2), b"")
    assert len(b.tokens) == DT_NMAX and len(b.raw) == TILE
    cases.append(Case(b.stream, 70000, -1, None, "generic"))
    b = K.compose([(lit(4), 4, 4)] + [(b"", 4, 4)] * (DT_NMAX - 1), lit(5))
    assert len(b.tokens) == DT_NMAX + 1
    cases.append(Case(b.stream, 70000, len(b.raw), b.raw, "generic"))
    # A terminal with fewer than 4 literals is never valid: a long last match must end its length bytes 5 stream
    # bytes before the end.  The zero-literal terminal at 65 536 (whose output position the tile clamps to 16
    # bits) is rejected; 4 terminal literals are valid once the capacity leaves 5 bytes behind the last match.
    for t, cap, want in ((0, 70000, -1), (4, TILE, -1), (4, TILE + 4, TILE), (4, 70000, TILE)):
        b = K.compose([(lit(100), 100, 30000), (lit(36 - t), 7000, TILE - 30136)], lit(t))
        assert len(b.raw) == TILE
        cases.append(Case(b.stream, cap, want, b.raw if want > 0 else None, "tile" if want > 0 else "generic"))
    # both sides of the jump-table switch shift + n + 4 + 4N = 65 568, small and big stage, two shifts
    for N, L in ((8000, 1), (5000, 5)):
        for shift in (0, 13):
            for side in (0, 1):
                seqs = [(lit(L), L, 4)] + [(lit(L), 5 + L, 4) for _ in range(N - 2)]
                n = 65564 - shift - 4 * N + side
                c = clean_case(seqs, pad_stream(seqs, lit, n), shift=shift)
                assert len(K.compose(seqs, b"").tokens) == N and len(c.stream) == n
                cases.append(c)
    # both sides of the small/big stage boundary for every source shift
    for shift in range(16):
        for side in (0, 1):
            seqs, tail = _literal_heavy(lit, STAGE_SMALL - 16 - shift + side)
            c = clean_case(seqs, tail, shift=shift)
            assert c.path == ("tile_big" if side else "tile")
            cases.append(c)
    # the largest stream the tile path takes, and one byte more
    for n, shift in ((DT_MAX_SRC, 0), (DT_MAX_SRC, 1), (DT_MAX_SRC, 15), (DT_MAX_SRC + 1, 0), (DT_MAX_SRC + 1, 7)):
        seqs = [(lit(30000), 1, 4), (lit(30000), 30000, 100)]
        c = clean_case(seqs, pad_stream(seqs, lit, n), shift=shift)
        assert len(c.raw) <= TILE and c.path == ("tile_big" if n == DT_MAX_SRC else "generic")
        cases.append(c)
    # capacities around the decoded size, short and long blocks
    for seqs in ([(lit(10), 3, 40), (lit(5), 20, 7)], _fill(lit, 900)):
        tail = K.tail_for(seqs, lit)
        O = K.decoded_size(seqs, tail)
        for k in (-1, 0, 1, 4, 5, 12, 13):
            cases.append(clean_case(seqs, tail, cap=O + k, path="generic" if k < 0 else None))
    # 65 537 bytes: too big for the tile
    seqs = [(lit(50), 50, 40000)]
    tail = lit(TILE + 1 - 40050)
    cases.append(clean_case(seqs, tail))
    cases.append(clean_case(seqs, tail, cap=TILE))
    # plans that break one end rule: the tile path declines them, the exact decoder gives Port's code
    for rule in K.BROKEN_RULES:
        seqs, tail = K.broken(rule, lit)
        b = K.compose(seqs, tail)
        raw = b.raw if BROKEN_CODES[rule] > 0 and b.raw is not None else None
        cases.append(Case(b.stream, len(b.raw) if b.raw else K.decoded_size(seqs, tail), BROKEN_CODES[rule], raw, "generic"))
    return cases


def align_blocks():
    """Small and odd block sizes: n < 16, O < 16, O = 16 / 17 / 31, and one block of several steps."""
    lit = K.Bytes(4)
    plans = [([], lit(5)), ([(lit(1), 1, 4)], lit(8)), ([(lit(2), 2, 6)], lit(8)), ([(lit(3), 1, 6)], lit(8)),
             ([(lit(5), 3, 10), (lit(2), 7, 4)], lit(10))]
    seqs = _fill(lit, 1100) + K.chain(lit, 40, 9, 2)
    plans.append((seqs, K.tail_for(seqs, lit)))
    return plans


@functools.lru_cache(maxsize=None)
def align_family():
    cases = []
    for i, (seqs, tail) in enumerate(align_blocks()):
        for s in range(16):
            for d in range(16):
                cases.append(clean_case(seqs, tail, cap=None if (s + d + i) % 3 else K.decoded_size(seqs, tail) + 7,
                                        shift=s, dshift=d))
    O = [len(compose_raw) for compose_raw in (K.compose(s, t).raw for s, t in align_blocks())]
    assert O[:5] == [5, 13, 16, 17, 31] and len(K.compose(*align_blocks()[0]).stream) < 16
    return cases


def _big_plan(lit, rng):
    """A clean plan whose stream needs the big stage, several steps long, with chains between its matches."""
    seqs, pos = [], 0
    target = int(rng.integers(STAGE_SMALL + 100, 55000))
    n = 0
    while n < target:
        L = int(rng.integers(20, 90))
        ml = int(rng.integers(4, 13))
        start = pos + L
        off = int(rng.integers(1, min(start, 65535) + 1)) if rng.random() < 0.7 else max(1, min(ml, start))
        seqs.append((lit(L), off, ml))
        pos = start + ml
        n += K.sequence_bytes(L, ml)
    return seqs


@functools.lru_cache(maxsize=None)
def reuse_family(count: int):
    """Big-stage blocks, interleaved: clean; invalid only in the last sequence (its offset reaches before the
    block), so the tile is abandoned after the earlier steps ran; rejected at the scan (decoded size > cap)."""
    lit = K.Bytes(5)
    rng = np.random.default_rng(5)
    cases = []
    for i in range(count):
        seqs = _big_plan(lit, rng)
        tail = K.tail_for(seqs, lit)
        if i % 3 == 0:
            c = clean_case(seqs, tail, shift=i % 16, dshift=(3 * i) % 16)
            assert c.path == "tile_big"
        elif i % 3 == 1:
            l, _, ml = seqs[-1]
            seqs[-1] = (l, _out(seqs[:-1]) + len(l) + 1, ml)
            b = K.compose(seqs, tail)
            c = Case(b.stream, K.decoded_size(seqs, tail), -1, None, "generic", i % 16, (3 * i) % 16)
        else:
            c = clean_case(seqs, tail, cap=K.decoded_size(seqs, tail) - 1, path="generic", shift=i % 16)
        assert len(K.compose(seqs, tail).tokens) > STEP and len(c.stream) + c.shift + 16 > STAGE_SMALL
        cases.append(c)
    return cases


@functools.lru_cache(maxsize=None)
def random_family(count: int = 20000, seed: int = 2024):
    """Seeded random clean plans: most decode to at most 64 KiB (sizes skewed towards short blocks, one in 64
    allowed the whole 64 KiB), one in 1000 to 64 KiB .. 4 MiB."""
    lit = K.Bytes(seed)
    rng = np.random.default_rng(seed)
    cases = []
    for i in range(count):
        if i % 1000 == 999:
            limit = int(np.exp(rng.uniform(np.log(TILE + 1), np.log(4 << 20))))
            seqs, tail = K.random_plan(rng, lit, limit, stop=0.0)
        else:
            limit = TILE if i % 64 == 0 else int(5 * (TILE / 5) ** (rng.random() ** 2))
            seqs, tail = K.random_plan(rng, lit, limit)
        O = K.decoded_size(seqs, tail)
        cap = O if i % 4 else O + int(rng.integers(1, 100))
        cases.append(clean_case(seqs, tail, cap=cap, shift=i % 16, dshift=(i // 16) % 16))
    return cases


@functools.lru_cache(maxsize=None)
def hc_family():
    import oracle
    return [Case(s, size, size, raw, route(len(s), size, 0, size)) for _, size, _, s, raw in inputs.hc_blocks(oracle.Port())]


FAMILIES = {"near": near_family, "parse": parse_family, "limits": limits_family, "align": align_family,
            "reuse": lambda: reuse_family(60), "random": lambda: random_family(3000), "hc": hc_family}


# ---- CPU: the composer against the restatement ---------------------------------------------------------------

def test_compose_expands_overlapping_matches():
    b = K.compose([(b"ab", 2, 7), (b"", 1, 4), (b"xyz", 5, 6)], b"12345")
    assert b.raw == b"ab" + b"abababa" + b"aaaa" + b"xyz" + b"aaxyza" + b"12345"
    assert b.tokens[0] == 0 and b.outs == [0, 9, 13, 22]
    assert b.stream[:3] == bytes([0x23]) + b"ab" and b.stream[3:5] == b"\x02\x00"
    long = K.compose([(b"q" * 300, 1, 300)], b"")
    assert long.stream[:3] == bytes([0xFF, 255, 30]) and long.raw == b"q" * 600


@pytest.mark.parametrize("name", sorted(FAMILIES))
def test_family_decodes_with_port(port, name):
    for i, c in enumerate(FAMILIES[name]()):
        r, out = port.decode(c.stream, c.cap)
        assert r == c.want, (name, i, r, c.want)
        if c.raw is not None:
            assert out == c.raw, (name, i)


@pytest.mark.parametrize("rule", K.BROKEN_RULES)
def test_broken_plans_break_one_rule(port, rule):
    lit = K.Bytes(9)
    seqs, tail = K.broken(rule, lit)
    assert not K.clean(seqs, tail)
    b = K.compose(seqs, tail)
    assert port.decode(b.stream, K.decoded_size(seqs, tail))[0] == BROKEN_CODES[rule]
    # the same plan with the rule repaired is clean and decodes to its raw bytes
    if rule in ("mflimit", "lastliterals", "trailing_match"):
        fixed = tail + lit(12)
        assert K.clean(seqs, fixed)
        assert port.decode(K.compose(seqs, fixed).stream, K.decoded_size(seqs, fixed)) == \
            (K.decoded_size(seqs, fixed), K.compose(seqs, fixed).raw)


def test_random_plans_are_clean_and_heavy_tailed():
    cases = random_family(3000)
    sizes = np.array([len(c.raw) for c in cases])
    assert sizes.max() > TILE and (sizes <= TILE).mean() > 0.99 and (sizes < 256).sum() > 1000
    assert collections.Counter(c.path for c in cases)["tile"] > 2000


def test_hc_fixture_regenerates():
    blocks = hc_family()
    assert len(blocks) == 48
    assert sum(len(c.stream) for c in blocks) < 400_000


# ---- GPU -----------------------------------------------------------------------------------------------------

GUARD = 48


@pytest.fixture(scope="module")
def k4(native):
    import k4os.compression.lz4_b200 as k
    if native.k4lz4_device_count() <= 0:
        pytest.fail("no CUDA device: the GPU tests need one")
    return k


def gpu_decode(k4, cases):
    """One batch through decode_batch_device: each source at its shift, each destination slot at its shift
    between 0xCD guards.  -> (outputs, return codes, path counters); asserts that no byte outside the decoded
    output was written (outside the whole slot for a block that fails)."""
    import torch
    nb = len(cases)
    soff, pos = [], 0
    for c in cases:
        pos = (pos + 15) // 16 * 16 + c.shift
        soff.append(pos)
        pos += len(c.stream) + 1
    src = np.zeros(pos + 16, dtype=np.uint8)
    for c, o in zip(cases, soff):
        src[o:o + len(c.stream)] = np.frombuffer(c.stream, dtype=np.uint8)
    doff, pos = [], 0
    for c in cases:
        pos = (pos + GUARD + 15) // 16 * 16 + c.dshift
        doff.append(pos)
        pos += c.cap
    total = pos + GUARD
    dev = torch.device("cuda", 0)

    def t(a, dt):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
    d_src = t(src, np.uint8)
    d_soff, d_slen = t(soff, np.int64), t([len(c.stream) for c in cases], np.int32)
    d_doff, d_cap = t(doff, np.int64), t([c.cap for c in cases], np.int32)
    d_dst = torch.full((total,), 0xCD, dtype=torch.uint8, device=dev)
    d_out = torch.full((nb,), -7, dtype=torch.int32, device=dev)
    k4.batch.decode_stats(0, reset=True)
    k4.batch.decode_batch_device(d_src.data_ptr(), d_soff.data_ptr(), d_slen.data_ptr(), d_dst.data_ptr(),
                                 d_doff.data_ptr(), d_cap.data_ptr(), d_out.data_ptr(), nb,
                                 torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    stats = k4.batch.decode_stats(0, reset=True)
    dst, rets = d_dst.cpu().numpy(), d_out.cpu().numpy()
    may = np.zeros(total, dtype=bool)
    for i, c in enumerate(cases):
        r = int(rets[i])
        may[doff[i]:doff[i] + (r if r > 0 else c.cap)] = True
    bad = np.flatnonzero(~may & (dst != 0xCD))
    assert bad.size == 0, f"{bad.size} bytes written outside the decoded output, first at {bad[0]}"
    outs = [dst[doff[i]:doff[i] + int(rets[i])].tobytes() if rets[i] > 0 else b"" for i in range(nb)]
    return outs, rets, stats


def check_batch(k4, port, cases):
    outs, rets, st = gpu_decode(k4, cases)
    for i, c in enumerate(cases):
        r, ref = port.decode(c.stream, c.cap)
        assert (int(rets[i]), r) == (c.want, c.want), (i, c.path, len(c.stream), c.cap, int(rets[i]), r, c.want)
        if c.raw is not None:
            assert outs[i] == c.raw, (i, c.path, len(c.stream), c.cap)
        elif r > 0 and not inputs.uses_zero_offset(c.stream):
            assert outs[i] == ref, i
    want = collections.Counter(c.path for c in cases)
    got = {k: st[k] for k in ("tile", "tile_big", "generic")}
    assert got == {k: want.get(k, 0) for k in got}, (got, dict(want))


@pytest.mark.gpu
def test_near_match_scheduling_gpu(k4, port):
    check_batch(k4, port, near_family())


@pytest.mark.gpu
def test_parse_and_repair_gpu(k4, port):
    check_batch(k4, port, parse_family())


@pytest.mark.gpu
def test_limits_gpu(k4, port):
    check_batch(k4, port, limits_family())


@pytest.mark.gpu
def test_alignment_and_sentinels_gpu(k4, port):
    check_batch(k4, port, align_family())


@pytest.mark.gpu
def test_persistent_big_stage_reuse_gpu(k4, port):
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    check_batch(k4, port, reuse_family(3 * sms + 2))          # every CTA of the persistent kernel decodes several


@pytest.mark.gpu
def test_random_composed_streams_gpu(k4, port):
    cases = random_family(20000)
    assert sum(len(c.raw) > TILE for c in cases) >= 20
    check_batch(k4, port, cases)


@pytest.mark.gpu
def test_hc_blocks_gpu(k4, port):
    check_batch(k4, port, hc_family())


# ---- GPU: the recorded results of the reference engine ------------------------------------------------------

class GpuEngine:
    """The GPU as an engine of tests/inputs.py's case sets, answered in batches.  A recording pass runs a row
    function with the restatement answering (its control flow may depend on results), a batched pass computes
    every recorded call on the GPU, and the replay pass runs the row function again with the GPU's answers;
    a call that differs from the recorded one fails the replay."""

    def __init__(self, k4, port):
        self.k4, self.port = k4, port
        self.calls, self.answers, self.recording = [], None, True

    def _call(self, kind, *args):
        if self.recording:
            self.calls.append((kind, args))
            return getattr(self.port, kind)(*args)
        i = self.at
        self.at += 1
        assert self.calls[i] == (kind, args), (i, kind)
        return self.answers[i]

    def encode(self, data, cap=None):
        return self._call("encode", bytes(data), cap)

    def decode(self, src, cap):
        return self._call("decode", bytes(src), int(cap))

    def decode_dict(self, src, cap, dictionary):
        return self._call("decode_dict", bytes(src), int(cap), bytes(dictionary))

    def partial_decode(self, src, target):
        return self._call("partial_decode", bytes(src), int(target))

    def run(self):
        B, MOS = self.k4.batch, self.k4.LZ4Codec.MaximumOutputSize
        self.answers = [None] * len(self.calls)
        by_kind = collections.defaultdict(list)
        for i, (kind, _) in enumerate(self.calls):
            by_kind[kind].append(i)
        for kind, idx in by_kind.items():
            a = [self.calls[i][1] for i in idx]
            if kind == "encode":
                res, lens = B.encode_batch_host([x[0] for x in a], [MOS(len(x[0])) if x[1] is None else x[1] for x in a])
            elif kind == "decode":
                res, lens = B.decode_batch_host([x[0] for x in a], [x[1] for x in a])
            elif kind == "decode_dict":
                res, lens = B.decode_dict_batch_host([x[0] for x in a], [x[1] for x in a], [x[2] for x in a])
            else:
                res, lens = B.partial_decode_batch_host([x[0] for x in a], [x[1] for x in a])
            for i, r, b in zip(idx, lens, res):
                self.answers[i] = (int(r), b if r > 0 else b"")
        self.recording, self.at = False, 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["corpus", "malformed", "dictionary", "partial", "fuzz_encode", "fuzz_decode"])
def test_gpu_matches_recorded_reference_results(k4, port, ref, name, monkeypatch):
    rows_of = inputs.ENGINE_SETS[name]
    monkeypatch.setattr(inputs, "gen", functools.lru_cache(maxsize=None)(inputs.gen))   # both passes, one generation
    eng = GpuEngine(k4, port)
    rows_of(port, eng)
    eng.run()
    ref.check(name, *rows_of(port, eng))
    assert eng.at == len(eng.calls)
