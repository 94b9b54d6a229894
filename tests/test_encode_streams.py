"""The block encoders on inputs aimed at the warp-batched match search, its limits and both table kinds.

Every aimed block is built with tests/encplan.py and run through its traced restatement of the L00_FAST
loop.  The CPU tests prove that the model gives oracle.Port's bytes and that each family reaches what it
was built for (the aim: probe indices, batch lanes, catch-up lengths and bounds, forwarding sources,
match ends, failing capacity checks).  The GPU tests encode each family through
batch.encode_batch_device, compare return codes and bytes with Port, check that the 0xCD bytes behind
every destination slot stay untouched, and read encode_stats to see which warps did the work:

* a small batch (at most SMs x 8 blocks) runs on the shared-memory-table warps alone;
* the family repeated and shuffled into at least 4 x SMs x 8 blocks also runs on the global-table warps
  (32-bit slots holding a 16-bit tag beside the position), which take blocks in a race.

Constants of csrc/encode_tile.cuh the inputs aim at: 32 probes per batch, the post-match probe on lane 0,
the catch-up in rounds of 8 then 32 lanes, LZ4_count in rounds of 8 then 32 lanes of 4 bytes, and the
u16-table encoder for blocks below 65 547 bytes (the u32-table engine above).
"""
from __future__ import annotations

import ctypes as C
import functools
from typing import NamedTuple

import numpy as np
import pytest

from tests import encplan as E
from tests import inputs

SM_WARPS = 8                 # ENC_SM_WARPS: shared-memory-table warps per SM
# Global-table blocks a mixed batch must show, per 1000 blocks below 65 547 bytes: half the smallest share measured
# on one NVIDIA B200 (148 SMs, 1000 W power limit), 63 % (3 241 of 5 112; the other families 68 %).
MIXED_GLOBAL_FLOOR = 310


class Case(NamedTuple):
    data: bytes
    cap: int | None = None   # None: MaximumOutputSize (not limited)
    shift: int = 0           # source address mod 16
    dshift: int = 0          # destination address mod 16


def mos(n: int) -> int:
    return n + n // 255 + 16


def first(data) -> E.Hit:
    return E.encode(data).hits[0]


# ---- builders ---------------------------------------------------------------------------------------------

def next_probe(x: int, base: int) -> tuple[int, int]:
    """(q, position) of the first probe at or after x of a run that began at `base`."""
    q = 0
    while base + E.advance(q) < x:
        q += 1
    return q, base + E.advance(q)


@functools.lru_cache(maxsize=None)
def probe_family():
    """First hits at chosen search-probe indices, in runs with and without a post probe, and runs that end."""
    out = []
    qs = list(range(0, 71)) + list(range(95, 101)) + list(range(127, 132))
    k = 2
    while E.advance(64 * k + 1) + 120 < 65000:
        qs.append(64 * k + 1)                            # the probe after the step grows to k + 1
        k += 1
    for i, q in enumerate(sorted(set(qs))):
        P = E.first_run_probe(q)
        b = E.Block(P + 140, 100 + i)
        if q < 8:                                        # a prefix of period q + 1: probe q repeats position 0
            b.a[0:q + 9] = (b.a[0:q + 1] * 9)[:q + 9]
        else:
            b.copy(P, 0 if i % 2 else E.first_run_probe(q - 5 if q < 64 else 3), 8)
        out.append(b.bytes())
    # runs that begin with a post probe: first match ends at e, then the hit at search probe q of the next run
    for q in list(range(0, 40)) + [62, 63, 64, 65, 66, 94, 95, 96]:
        def build(seed, q=q):
            b = E.Block(E.advance(q) + 200, 300 + 1000 * seed + q)
            b.copy(21, 0, 8)                             # probe 20 of the first run hits position 0
            e = first(b.bytes()).end
            b.copy(e + 1 + E.advance(q), 11 if q % 2 else 14 + (q % 3), 6)   # a source stored by the first run
            return b.bytes()
        out.append(aimed(build, lambda r, q=q: len(r.hits) > 1 and r.hits[1].q == q and r.hits[1].post_run))
    # post probes that hit: through the table, and through put(ip-2) (the post probe's hash equals hash(ip-2))
    for s in range(6):
        b = E.Block(400, 400 + s)
        b.copy(21, 0, 8)
        e = first(b.bytes()).end
        if s % 2:
            b.a[e:e + 4] = bytes([b.a[e - 2], b.a[e - 1]]) * 2
        else:
            b.copy(e, 11 + s, 6)
        out.append(b.bytes())
    # the last probe that executes, and the first that does not: a hit there or the run's end
    for n in list(range(13, 80)) + [200, 1000, 5000]:
        for side in (0, 1):
            b = E.Block(n, 500 + n)
            pr = 0
            while 1 + E.advance(pr + 1) <= n - 11:
                pr += 1
            P = E.first_run_probe(pr - 1 + side)
            if pr >= 1 and P + 4 <= n:
                b.copy(P, 0, 4)
            out.append(b.bytes())
    return out


def forward_family():
    return _forward_items()[0]


@functools.lru_cache(maxsize=None)
def _forward_items():
    """Same-hash groups inside one batch: forwarding from the nearest earlier lane, the commit of the lanes up to
    the hit, the post probe and the lanes that see put(ip-2), and equal-hash / equal-tag pairs.
    -> (blocks, groups): groups[k] = (block index, positions of the group's lanes, nearest-lane case)."""
    out, groups = [], []
    rng = np.random.default_rng(7)
    # batch 7 of the first run: probes 224..255, 4 bytes apart (step 4), so every lane's 4 bytes are its own
    B7 = 224
    pos = [E.first_run_probe(B7 + ln) for ln in range(32)]
    assert all(pos[i + 1] - pos[i] == 4 for i in range(31))
    for g in (2, 3, 4):
        for near in (True, False):
            for f in (g - 1, 9, 20, 31):
                lanes = sorted({f - 5 * (g - 1 - j) for j in range(g)})
                if lanes[0] < 0:
                    continue
                b = E.Block(pos[-1] + 200, int(rng.integers(1 << 30)))
                V = E.value_with_hash(int(rng.integers(8192)), int(rng.integers(1 << 19)))
                vals = [E.same_hash_other_tag(V, 1 + j) for j in range(g)]
                vals[-1] = V
                if near:
                    vals[-2] = V                                  # the nearest earlier lane holds V
                else:
                    vals[0] = V                                   # only the farthest one does
                for ln, v in zip(lanes, vals):
                    b.put(pos[ln], v)
                if g == 4:
                    b.put(pos[f] + 8, E.same_hash_same_tag(V))    # a later lane, equal hash and tag
                groups.append((len(out), [pos[ln] for ln in lanes], near))
                out.append(b.bytes())
    # a lane before the hit shares its hash only with a lane after the hit (discarded); a later probe with the
    # earlier lane's value then finds that lane's position only if it was committed
    for j, f in ((2, 10), (0, 5), (9, 30), (20, 21)):
        b = E.Block(pos[-1] + 200, 900 + j)
        X = E.value_with_hash(int(rng.integers(8192)), int(rng.integers(1 << 19)))
        b.put(15, E.same_hash_other_tag(X))                       # source bytes + 4: X' with X's hash
        b.put(pos[j], X)
        b.copy(pos[f], 11, 12)                                    # hit at f; lane f + 1 lies in the match: X'
        e = E.encode(b.bytes()).hits[0].end
        b.put(e, X)                                               # the post probe looks X up
        out.append(b.bytes())
    # post runs: hash(ip-2) == hash(post probe) with a hit through put(ip-2); a search lane of batch 0 that sees
    # put(ip-2); a lane at or before the hit that shares hash(ip-2) (it, not put(ip-2), survives); put(ip-2)
    # read back from the table in a later batch (the tag stored with it must be its own)
    for s in range(4):
        for kind in ("post", "lane", "same2", "later", "tagpair"):
            b = E.Block(700, 1000 + 10 * s + len(kind))
            b.copy(21 + s, 0, 8 + s)
            e = first(b.bytes()).end
            g2 = b.gram(e - 2)
            if kind == "post":
                b.a[e:e + 4] = bytes([b.a[e - 2], b.a[e - 1]]) * 2
            elif kind == "lane":
                b.put(e + 4 + 4 * s, g2)                          # lane 4 + 4s (search probe 3 + 4s)
            elif kind == "same2":
                b.put(e + 8, E.same_hash_other_tag(g2))           # lane 8 takes hash(ip-2)
                b.copy(e + 16, 11, 6)                             # hit at lane 16
                e2 = E.encode(b.bytes()).hits[1].end
                b.put(e2, g2)                                     # the next post probe looks g2 up
            elif kind == "later":
                b.put(e + 1 + E.advance(40 + s), g2)              # batch 1 of the run reads put(ip-2) back
            else:
                b.put(e + 1 + E.advance(40 + s), E.same_hash_same_tag(g2))   # passes the tag filter, must not hit
                b.put(e + 1 + E.advance(50 + s), g2)
            out.append(b.bytes())
    return out, groups


def aimed(build, ok, tries: int = 12) -> bytes:
    """The first of `build(seed)` whose trace passes `ok` (a later probe can overwrite a table slot the aim needs
    by a hash collision; another filler then avoids it)."""
    for seed in range(tries):
        d = build(seed)
        r = E.encode(d)
        if ok(r):
            return d
    raise AssertionError("no seed reached the aim")


@functools.lru_cache(maxsize=None)
def catch_family():
    """Catch-up lengths 0..43 stopped by a byte and by m reaching 0, and lengths up to 40 stopped by `anchor`.
    The copy starts c bytes before a probe of a zone whose step exceeds c, so no probe lands inside it before."""
    out = []
    for c in range(0, 45):
        q = 64 * (c + 1) + 2                         # the step before probe q is c + 2
        P = E.first_run_probe(q)
        if P + 80 > 65540:
            continue
        k = max(3, (c + 16) // (c + 2) + 1)
        S = E.first_run_probe(q - k)                 # a source stored shortly before, c + 16 bytes or more away

        def build(seed, c=c, P=P, S=S, m0=False):
            b = E.Block(P + 80, 2000 + 100 * seed + 2 * c + m0)
            if m0:
                b.copy(P - c, 0, c + 12)             # the hit sees position c; the catch-up walks back to 0
            else:
                b.copy(P - c, S - c, c + 12)
            return b.bytes()
        out.append(aimed(build, lambda r, c=c: bool(r.hits) and (r.hits[0].catch, r.hits[0].stop) == (c, "byte")))
        out.append(aimed(functools.partial(build, m0=True),
                         lambda r, c=c: bool(r.hits) and (r.hits[0].catch, r.hits[0].stop) == (c, "m0")))
    # the catch-up reaches the previous match's end: the source lies in a sparse zone of the first run
    for c in (1, 2, 5, 8, 9, 20, 33, 40):
        qs = 64 * (c + 2) + 2
        Ss = E.first_run_probe(qs)
        P1 = E.first_run_probe(qs + 3)

        def build(seed, c=c, Ss=Ss, P1=P1):
            b = E.Block(P1 + 200, 2200 + 100 * seed + c)
            b.copy(P1, 0, 8)
            e = E.encode(b.bytes()).hits[0].end if E.encode(b.bytes()).hits else P1 + 8
            b.copy(e, Ss - c, c + 8)                 # the post probe and search probes 0..c-2 miss; c - 1 hits
            b.a[Ss - c - 1] = b.a[e - 1]             # only `anchor` stops the catch-up: the bytes before agree too
            return b.bytes()
        out.append(aimed(build, lambda r, c=c: len(r.hits) > 1 and (r.hits[1].catch, r.hits[1].stop) == (c, "anchor")))
    return out


@functools.lru_cache(maxsize=None)
def count_family():
    """Match ends at matchlimit - 2 .. matchlimit, match and literal lengths around the length-field boundaries,
    and last-literal runs of 5, 14, 15, 270, 525 and 8000+."""
    out = []
    # the last match runs into the end of the block: ends at mlim - k (a byte differs) or is clipped at mlim
    for n in (40, 41, 42, 43, 60, 77, 100, 1000, 4099):
        for k in (2, 1, 0):
            b = E.Block(n, 3000 + n + k)
            P = 21
            mlim = n - 5
            ln = n - P if k == 0 else mlim - k - P
            b.copy(P, 0, ln)
            if k:
                b.a[P + ln] = b.a[ln] ^ 0x5A
            out.append(b.bytes())
    # match lengths (mc = length - 4) around 15, 270, 525 and above 32 x 255 + 15
    for mc in (13, 14, 15, 16, 17, 268, 269, 270, 271, 272, 523, 524, 525, 526, 527, 8175, 8176, 9000, 20000):
        ml = mc + 4
        b = E.Block(2 * ml + 160, 3100 + mc)
        P = ml + 100
        b.copy(P, 0, ml)
        out.append(b.bytes())
    # literal runs of the same lengths: a copy starting exactly at x in the first run
    for lit in (13, 14, 15, 16, 17, 268, 269, 270, 271, 272, 523, 524, 525, 526, 527, 8175, 8176, 9000):
        q, P = next_probe(lit, 1)
        b = E.Block(P + 100, 3200 + lit)
        b.copy(lit, 2, (P - lit) + 8)
        out.append(b.bytes())
    # last-literal runs
    for run in (5, 6, 11, 12, 14, 15, 16, 270, 525, 8000, 9001):
        b = E.Block(200 + run, 3300 + run)
        b.copy(100, 0, 100)
        b.a[200] = b.a[100] ^ 0x33
        out.append(b.bytes())
    return out


FILLS = ("zeros", "p1", "p2", "p3", "p4", "unique")


def fill(kind: str, n: int, seed: int = 0) -> bytes:
    if kind == "zeros":
        return bytes(n)
    if kind == "unique":
        return E.unique_filler(n, seed)
    p = int(kind[1])
    pat = bytes([0xA7, 0x13, 0x5C, 0xE1][:p])
    return (pat * (n // p + 1))[:n]


@functools.lru_cache(maxsize=None)
def size_family():
    out = [fill(k, n, n) for n in range(0, 201) for k in FILLS]
    out += [fill(k, n, 7) for n in range(65535, 65549) for k in FILLS]
    return out


# ---- CPU: the model against Port, and the aims -------------------------------------------------------------

def traces(blocks):
    return [E.encode(d) for d in blocks]


def assert_model_matches_port(port, blocks):
    for i, d in enumerate(blocks):
        if len(d) >= E.LIMIT_64K:
            continue
        r = E.encode(d)
        assert (r.ret, r.data) == port.encode(d), (i, len(d))


def all_hits(blocks):
    return [h for r in traces(blocks) for h in r.hits]


def test_model_matches_port_on_corpus(port):
    items = [d for _, d in inputs.corpus() if len(d) < E.LIMIT_64K]
    assert len(items) > 200
    assert_model_matches_port(port, items)


def test_builders():
    v = E.value_with_hash(1234, 99)
    assert E.hash13(v) == 1234
    w, t = E.same_hash_other_tag(v), E.same_hash_same_tag(v)
    assert E.hash13(w) == E.hash13(t) == 1234 and E.tag16(w) != E.tag16(v) and E.tag16(t) == E.tag16(v)
    assert len({w, t, v}) == 3
    f = E.unique_filler(70000, 3)
    grams = {f[i:i + 4] for i in range(len(f) - 3)}
    assert len(grams) == len(f) - 3
    assert [E.advance(q) for q in (0, 1, 64, 65, 66, 129, 130)] == [0, 1, 64, 65, 67, 193, 196]


def test_probe_family_aim(port):
    blocks = probe_family()
    assert_model_matches_port(port, blocks)
    hits = all_hits(blocks)
    first_run = {h.q for h in hits if not h.post_run and not h.post}
    want = set(range(0, 71)) | set(range(95, 101)) | set(range(127, 132)) | {65, 129, 193, 257, 321}
    assert want <= first_run, sorted(want - first_run)
    assert max(first_run) >= 64 * 38                        # up to a step of about 40
    assert {h.lane for h in hits if not h.post_run} == set(range(32))
    assert {h.lane for h in hits if h.post_run} == set(range(32))
    assert {h.lane for h in hits if h.post_run and h.batch == 1} >= set(range(8))
    post = [h for h in hits if h.post]
    assert {h.src for h in post} == {"table", "put2"}
    assert {h.src for h in hits} == {"table", "lane", "put2"}
    ends = [r.end for r in traces(blocks) if r.end is not None]
    assert {e.lane for e in ends if not e.post_run} == set(range(32))
    assert any(e.post_run for e in ends)


def test_forward_family_aim(port):
    blocks = forward_family()
    assert_model_matches_port(port, blocks)
    hits = all_hits(blocks)
    grp = [h for h in hits if h.src == "lane"]
    for g in (2, 3):                                         # the nearest earlier lane matches, the farthest not
        assert any(h.before == g and h.near_ok and not h.far_ok for h in grp), g
    assert any(h.before == 1 for h in grp)
    # the reverse case never hits through the lane: its hit, if any, comes later from the table
    assert any(h.straddle for h in hits)
    assert any(h.after > 0 for h in hits)
    assert any(h.post and h.src == "put2" and h.h2_post for h in hits)
    assert any(not h.post and h.src == "put2" for h in hits)
    assert any(h.same2 for h in hits)
    assert any(h.src == "table" and h.store == "put2" for h in hits)


def test_forward_groups_layout():
    """The group blocks hold what they were built for: lanes of one batch sharing a hash, the hit lane last.  In the
    nearest-lane case the lane before it holds the hit lane's 4 bytes; in the reverse case only the farthest lane
    does, so the hit lane's probe runs and misses (forwarding from the farthest lane would make it hit)."""
    blocks, groups = _forward_items()
    batch7 = {E.first_run_probe(q) for q in range(224, 256)}
    reverse = set()
    for k, lanes, near in groups:
        d = blocks[k]
        g = [int.from_bytes(d[p:p + 4], "little") for p in lanes]
        assert len({E.hash13(v) for v in g}) == 1, k
        assert set(lanes) <= batch7, k
        hits = E.encode(d).hits
        probed = [h.ip + h.catch for h in hits]
        assert all(p >= lanes[-1] for p in probed[:1]), k     # no hit before the group: its probes all run
        if near:
            assert g[-2] == g[-1] and hits and probed[0] == lanes[-1] and hits[0].src == "lane", k
        elif len(lanes) >= 3:
            reverse.add(len(lanes))
            assert g[0] == g[-1] and all(v != g[-1] for v in g[1:-1]), k
            assert lanes[-1] not in probed, k                  # the hit lane's probe missed
    assert reverse == {3, 4}


def test_catch_family_aim(port):
    blocks = catch_family()
    assert_model_matches_port(port, blocks)
    hits = all_hits(blocks)
    got = {h.catch for h in hits if h.stop == "byte"}
    assert set(range(0, 42)) <= got, sorted(set(range(42)) - got)
    assert {h.catch for h in hits if h.stop == "m0"} >= set(range(0, 42))
    assert any(h.stop == "anchor" and h.catch >= 8 for h in hits)
    assert {h.catch for h in hits if h.stop == "anchor"} >= {1, 2, 5, 8, 9}
    # Only `anchor` stops these: the byte before the anchor agrees too.  A bound one byte looser (ip >= anchor + lane)
    # would take the match start to anchor - 1, a literal run of -1 (2^32 - 1 as the encoder's uint32): with an
    # unlimited capacity it would copy that many literals, far past the slot.
    anchored = [(d, h) for d, r in zip(blocks, traces(blocks)) for h in r.hits if h.stop == "anchor" and h.catch]
    assert len(anchored) >= 8
    assert all(h.lit == 0 and d[h.ip - 1] == d[h.m - 1] for d, h in anchored)


def test_count_family_aim(port):
    blocks = count_family()
    assert_model_matches_port(port, blocks)
    rs = traces(blocks)
    hits = [h for r in rs for h in r.hits]
    ends = {(len(d) - 5) - h.end for d, r in zip(blocks, rs) for h in r.hits}
    assert {0, 1, 2} <= ends
    assert any(h.clip for h in hits)
    mcs = {h.ml - 4 for h in hits}
    assert {14, 15, 16, 269, 270, 271, 524, 525, 526} <= mcs and max(mcs) > 32 * 255 + 15
    lits = {h.lit for h in hits}
    assert {14, 15, 16, 269, 270, 271, 524, 525, 526} <= lits and max(lits) > 32 * 255 + 15
    last = {len(d) - (r.hits[-1].end if r.hits else 0) for d, r in zip(blocks, rs)}
    assert {5, 14, 15, 270, 525} <= last and max(last) >= 8000


def test_size_family(port):
    blocks = size_family()
    assert len(blocks) == 201 * 6 + 14 * 6
    assert_model_matches_port(port, [d for d in blocks if len(d) <= 200])


@functools.lru_cache(maxsize=None)
def u32_family():
    """Blocks of 70 000 .. 300 000 bytes (the u32-table engine) with copies at distances 65 534 .. 65 537: a
    short repeat right before the source and the copy restarts the search at step 1 there."""
    out = []
    for i, (n, D) in enumerate([(70000, 65534), (70000, 65535), (90000, 65536), (131072, 65537),
                                (200000, 65535), (300000, 65534), (150000, 65535), (120000, 65537)]):
        b = E.Block(n, 4000 + i)
        S = 1000 + 97 * i
        for k, x in enumerate((S, S + D)):
            b.a[x - 200:x] = bytes([0x11 * (k + 1)]) * 200   # a match ending at x: the next run probes x, x + 1, ...
        b.copy(S + D, S, 64)
        out.append(b.bytes())
    return out


def offsets(stream: bytes) -> list:
    """The match offsets of an LZ4 block."""
    i, out = 0, []
    while i < len(stream):
        t = stream[i]
        i += 1
        L = t >> 4
        if L == 15:
            while stream[i] == 255:
                L += 255
                i += 1
            L += stream[i]
            i += 1
        i += L
        if i >= len(stream):
            break
        out.append(stream[i] | stream[i + 1] << 8)
        i += 2
        if t & 15 == 15:
            while stream[i] == 255:
                i += 1
            i += 1
    return out


def test_u32_family_aim(port):
    for d in u32_family():
        for x32 in (False, True):
            r, c = port.encode(d, enforce32=x32)
            assert r > 0
    found = {o for d in u32_family() for x32 in (False, True) for o in offsets(port.encode(d, enforce32=x32)[1])}
    assert {65534, 65535} <= found


def limit_blocks():
    """Blocks whose capacities are swept: aimed blocks from each family."""
    pf, ff, cf, kf = probe_family(), forward_family(), catch_family(), count_family()
    return [pf[5], pf[70], pf[100], ff[3], ff[30], cf[10], cf[41], kf[3], kf[20], kf[35], kf[-3], kf[-1]]


@functools.lru_cache(maxsize=None)
def limit_cases():
    cases = []
    for d in limit_blocks():
        r = E.encode(d).ret
        for cap in range(max(0, r - 300), mos(len(d)) + 1):
            cases.append(Case(d, cap))
    for d in set(probe_family() + forward_family() + catch_family() + count_family()):
        cases.append(Case(d, mos(len(d)) - 1))
    return cases


def sequences(stream: bytes):
    """The (literal length, mc) of every sequence of an LZ4 block (mc = match length - 4), and the last literal run."""
    i, seqs = 0, []
    while True:
        t = stream[i]
        i += 1
        L = t >> 4
        if L == 15:
            while stream[i] == 255:
                L += 255
                i += 1
            L += stream[i]
            i += 1
        i += L
        if i >= len(stream):
            return seqs, L
        i += 2
        mc = t & 15
        if mc == 15:
            while stream[i] == 255:
                mc += 255
                i += 1
            mc += stream[i]
            i += 1
        seqs.append((L, mc))


def failing_check(stream: bytes, cap: int) -> tuple[int, list]:
    """Which limited-output check fails first when the block whose unlimited output is `stream` is encoded at `cap`
    (a limited capacity only adds checks: the sequences stay the same): 1 literals, 2 match, 3 last literals,
    0 none, 12 a zero-literal sequence, where a post-match hit skips check 1 but then fails check 2 anyway.
    Also -> the capacities at which each check switches."""
    seqs, run = sequences(stream)
    op, fail, edges = 0, 0, []
    for lit, mc in seqs:
        t1 = op + 1 + lit + 8 + lit // 255
        hdr = 1 if lit < 15 else 2 + (lit - 15) // 255
        after = op + hdr + lit + 2
        t2 = after + 6 + (mc + 240) // 255
        edges += [t1, t2]
        if not fail and t1 > cap:
            fail = 1 if lit else 12
        if not fail and t2 > cap:
            fail = 2
        op = after + ((mc - 15) // 255 + 1 if mc >= 15 else 0)
    t3 = op + run + 1 + (run + 240) // 255
    edges.append(t3)
    if not fail and t3 > cap:
        fail = 3
    return fail, edges


@functools.lru_cache(maxsize=None)
def u32_limit_cases(x32: bool):
    """The u32 family at the capacities on both sides of every check of encode_generic.cuh, and at
    MaximumOutputSize - 1."""
    import oracle
    port, cases = oracle.Port(), []
    for d in u32_family():
        r, c = port.encode(d, enforce32=x32)
        edges = failing_check(c, r)[1]
        caps = sorted({t + k for t in edges for k in (-1, 0)} | {mos(len(d)) - 1})
        cases += [Case(d, cap) for cap in caps if 0 <= cap < mos(len(d))]
    return cases


def test_limit_sweep_aim(port):
    fails = set()
    for c in limit_cases():
        fails.add(E.encode(c.data, c.cap).fail)
    assert {1, 2, 3} <= fails
    # the check that the stream predicts is the one the model's encoder fails at
    for d in limit_blocks():
        c = E.encode(d).data
        caps = set(range(max(0, len(c) - 300), mos(len(d)))) | {t + k for t in failing_check(c, 0)[1] for k in (-1, 0)}
        for cap in sorted(caps):
            want, got = E.encode(d, cap).fail, failing_check(c, cap)[0]
            assert want == got or (got == 12 and want in (1, 2)), (cap, want, got)
    for x32 in (False, True):
        u32 = set()
        for cs in u32_limit_cases(x32):
            r, c = port.encode(cs.data, enforce32=x32)
            f = failing_check(c, cs.cap)[0]
            assert (f == 0) == (port.encode(cs.data, cs.cap, enforce32=x32)[0] > 0), (len(cs.data), cs.cap)
            u32.add(f)
        assert {1, 2, 3} <= u32, (x32, u32)


@functools.lru_cache(maxsize=None)
def pickle_messages():
    """Messages whose compressed length (capacity as the pickler gives it) is n - 2 .. n + 1, messages of 1 000 ..
    1 024 bytes (the 1 024-byte scratch makes the encoder limited) and of 65 546 / 65 547 bytes."""
    import oracle
    port = oracle.Port()
    out, seen = [], set()
    for n in (64, 300, 1000, 1024, 1100, 5000, 65546):
        for L in range(0, min(n - 40, 400)):
            b = E.Block(n, 5000 + n)
            if L:
                b.copy(n - L - 20, 10, L)
            d = b.bytes()
            k = port.encode(d)[0] - n
            if k in (-2, -1, 0, 1) and (n, k) not in seen:
                seen.add((n, k))
                out.append(d)
            if len([s for s in seen if s[0] == n]) == 4:
                break
    out += [(E.unique_filler(n, n)[:n // 2] * 3)[:n] for n in range(1000, 1025)]
    out += [E.unique_filler(n, n) for n in range(1000, 1025, 8)]
    out += [fill("p3", 65546), fill("p3", 65547), E.unique_filler(65546, 1), E.unique_filler(65547, 1)]
    return out


def test_pickle_messages_aim(port):
    ks = {(len(d), port.encode(d)[0] - len(d)) for d in pickle_messages()}
    assert {k for n, k in ks} >= {-2, -1, 0, 1}
    assert {n for n, _ in ks} >= set(range(1000, 1025)) | {65546, 65547}


def align_blocks():
    return [probe_family()[40], forward_family()[5], count_family()[12]]


def test_align_blocks_aim():
    hs = [E.encode(d).hits for d in align_blocks()]
    assert all(hs)


# ---- GPU ------------------------------------------------------------------------------------------------------

GAP = 64


@pytest.fixture(scope="module")
def k4(native):
    import k4os.compression.lz4_b200 as k
    if native.k4lz4_device_count() <= 0:
        pytest.fail("no CUDA device: the GPU tests need one")
    return k


def _dev(a, dt):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(torch.device("cuda", 0))


def gpu_encode(k4, cases, x32=False):
    """One launch through encode_batch_device (or its x32 entry): each source at its shift, each destination slot
    at its shift with a GAP of 0xCD behind it.  -> (return codes, outputs, encode_stats); asserts that nothing at
    or past the returned length (the capacity, for a block that fails) was written."""
    import torch
    nb = len(cases)
    soff, pos = [], 0
    for c in cases:
        pos = (pos + 15) // 16 * 16 + c.shift
        soff.append(pos)
        pos += len(c.data) + 1
    src = np.zeros(pos + 16, dtype=np.uint8)
    for c, o in zip(cases, soff):
        src[o:o + len(c.data)] = np.frombuffer(c.data, dtype=np.uint8)
    caps = [mos(len(c.data)) if c.cap is None else c.cap for c in cases]
    doff, pos = [], 0
    for c, cap in zip(cases, caps):
        pos = (pos + 15) // 16 * 16 + c.dshift
        doff.append(pos)
        pos += max(cap, 0) + GAP
    total = pos + 16
    d_src, d_soff = _dev(src, np.uint8), _dev(soff, np.int64)
    d_slen, d_doff, d_cap = _dev([len(c.data) for c in cases], np.int32), _dev(doff, np.int64), _dev(caps, np.int32)
    d_dst = torch.full((total,), 0xCD, dtype=torch.uint8, device="cuda:0")
    d_out = torch.full((nb,), -7, dtype=torch.int32, device="cuda:0")
    k4.batch.encode_stats(0, reset=True)
    st = torch.cuda.current_stream().cuda_stream
    args = (d_src.data_ptr(), d_soff.data_ptr(), d_slen.data_ptr(), d_dst.data_ptr(), d_doff.data_ptr(),
            d_cap.data_ptr(), d_out.data_ptr(), nb)
    if x32:
        L = k4._native.lib()
        k4._native.check(L.k4lz4_encode_batch_x32(*args, 0, k4._native.MEM_DEVICE, C.c_void_p(st), -1))
    else:
        k4.batch.encode_batch_device(*args, 0, st)
    torch.cuda.synchronize()
    stats = k4.batch.encode_stats(0, reset=True)
    dst, rets = d_dst.cpu().numpy(), d_out.cpu().numpy()
    may = np.zeros(total, dtype=bool)
    for i, cap in enumerate(caps):
        r = int(rets[i])
        may[doff[i]:doff[i] + (r if r > 0 else max(cap, 0))] = True
    bad = np.flatnonzero(~may & (dst != 0xCD))
    assert bad.size == 0, f"{bad.size} bytes written past the output, first at {bad[0]}"
    outs = [dst[doff[i]:doff[i] + int(rets[i])].tobytes() if rets[i] > 0 else b"" for i in range(nb)]
    return rets, outs, stats


@functools.lru_cache(maxsize=None)
def _port_encode(d: bytes, cap, x32: bool):
    import oracle
    return oracle.Port().encode(d, cap, enforce32=x32)


def check(k4, cases, x32=False):
    rets, outs, st = gpu_encode(k4, cases, x32)
    for i, c in enumerate(cases):
        r, ref = _port_encode(c.data, c.cap, x32)
        assert (int(rets[i]), outs[i]) == (r, ref), (i, len(c.data), c.cap, int(rets[i]), r)
    return st


def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def check_both_kernels(k4, blocks, x32=False):
    """The family as small batches (shared-memory-table warps only), then repeated and shuffled into at least
    4 x SMs x 8 blocks (global-table warps too).  `blocks`: bytes, or Cases with their own capacities and shifts.
    The u32-table engine runs in either warp kind and has one counter for both."""
    cases = [d if isinstance(d, Case) else Case(d, shift=i % 16, dshift=(7 * i) % 16) for i, d in enumerate(blocks)]
    wave = sms() * SM_WARPS
    for lo in range(0, len(cases), wave):
        part = cases[lo:lo + wave]
        st = check(k4, part, x32)
        n16 = sum(0 < len(c.data) < E.LIMIT_64K for c in part)
        assert st == {"shared": n16, "global": 0, "u32": sum(len(c.data) >= E.LIMIT_64K for c in part)}, st
    R = -(-4 * wave // len(cases))
    rng = np.random.default_rng(len(cases))
    mixed = [cases[i % len(cases)] for i in rng.permutation(R * len(cases))]
    st = check(k4, mixed, x32)
    n16 = sum(0 < len(c.data) < E.LIMIT_64K for c in mixed)
    print(f"mixed batch of {len(mixed)}: {st}")
    assert st["shared"] + st["global"] == n16, st
    assert st["u32"] == sum(len(c.data) >= E.LIMIT_64K for c in mixed), st
    assert st["global"] * 1000 >= MIXED_GLOBAL_FLOOR * n16, st


@pytest.mark.gpu
def test_probe_schedule_gpu(k4):
    check_both_kernels(k4, probe_family())


@pytest.mark.gpu
def test_forwarding_and_commit_gpu(k4):
    check_both_kernels(k4, forward_family())


@pytest.mark.gpu
def test_catch_up_gpu(k4):
    check_both_kernels(k4, catch_family())


@pytest.mark.gpu
def test_count_end_and_fields_gpu(k4):
    check_both_kernels(k4, count_family())


@pytest.mark.gpu
def test_sizes_gpu(k4):
    check_both_kernels(k4, size_family())


@pytest.mark.gpu
def test_u32_engine_gpu(k4):
    for x32 in (False, True):
        check_both_kernels(k4, u32_family(), x32)


@pytest.mark.gpu
def test_output_limits_gpu(k4):
    check_both_kernels(k4, [c._replace(dshift=i % 16) for i, c in enumerate(limit_cases())])
    for x32 in (False, True):
        check(k4, [c._replace(shift=i % 16) for i, c in enumerate(u32_limit_cases(x32))], x32)


def _pickle_device(k4, msgs, writer):
    import torch
    N = k4._native
    L = N.lib()
    bound = [(L.k4lz4_pickle_writer_bound(len(m)) if writer else len(m) + 1) for m in msgs]
    soff = np.concatenate([[0], np.cumsum([len(m) for m in msgs])[:-1]]).astype(np.int64)
    src = np.frombuffer(b"".join(msgs) + b"\0" * 16, dtype=np.uint8).copy()
    doff, pos = [], 0
    for b in bound:
        doff.append(pos)
        pos += b + GAP
    d_dst = torch.full((pos + 16,), 0xCD, dtype=torch.uint8, device="cuda:0")
    d_out = torch.full((len(msgs),), -7, dtype=torch.int32, device="cuda:0")
    d_src, d_soff, d_slen, d_doff = _dev(src, np.uint8), _dev(soff, np.int64), \
        _dev([len(m) for m in msgs], np.int32), _dev(doff, np.int64)
    fn = L.k4lz4_pickle_writer_batch if writer else L.k4lz4_pickle_batch
    N.check(fn(d_src.data_ptr(), d_soff.data_ptr(), d_slen.data_ptr(), d_dst.data_ptr(), d_doff.data_ptr(),
               d_out.data_ptr(), len(msgs), 0, N.MEM_DEVICE, C.c_void_p(torch.cuda.current_stream().cuda_stream), -1))
    torch.cuda.synchronize()
    dst, rets = d_dst.cpu().numpy(), d_out.cpu().numpy()
    outs = []
    for i, b in enumerate(bound):
        r = int(rets[i])
        assert (dst[doff[i] + r:doff[i] + b + GAP] == 0xCD).all(), i
        outs.append(dst[doff[i]:doff[i] + r].tobytes())
    return outs


@pytest.mark.gpu
def test_pickler_gpu(k4, port):
    msgs = pickle_messages()
    assert _pickle_device(k4, msgs, False) == [port.pickle(m) for m in msgs]
    assert _pickle_device(k4, msgs, True) == [port.pickle_writer(m) for m in msgs]


@pytest.mark.gpu
def test_alignment_gpu(k4):
    check_both_kernels(k4, [Case(d, shift=s, dshift=t) for d in align_blocks() for s in range(16) for t in range(16)])
