"""A traced restatement of the L00_FAST block encoder for blocks below 65 547 bytes, and input builders
aimed at the warp-batched match search of csrc/encode_tile.cuh.

`encode` follows the reference's serial loop (the u16 table, hash4 with 13 bits, the skip schedule
`step = cnt++ >> 6`) and returns the compressed bytes with a trace of every sequence: where the hit lay in
its search run and in the 32-lane probe batch that evaluates it on the GPU, which store supplied its
candidate, and what stopped the catch-up and the match count.  The tests use the trace to prove that
an aimed input really reaches the state it was built for; oracle.Port stays the authority for the bytes.

The GPU evaluates a search run 32 probes at a time.  After a match, the probe at the match end (the "post"
probe) rides as lane 0 of the next batch and search probes start at lane 1, so search probe q sits on lane
(q + 1) mod 32; a run that begins without a post probe has probe q on lane q mod 32.
"""
from __future__ import annotations

import functools
from typing import NamedTuple

import numpy as np

MINMATCH, MFLIMIT, LASTLITERALS, MINLENGTH, LIMIT_64K = 4, 12, 5, 13, 65547
PRIME = 2654435761
INV = pow(PRIME, -1, 1 << 32)            # v = p * INV has v * PRIME == p (mod 2^32)
M32 = 0xFFFFFFFF


def product(v: int) -> int:
    return (v * PRIME) & M32


def hash13(v: int) -> int:
    return product(v) >> 19


def tag16(v: int) -> int:
    """The 16-bit tag the global-table warps keep beside each position (TAGMODE 2): product bits 3..18."""
    return (product(v) >> 3) & 0xFFFF


def value_of(p: int) -> int:
    """The 4-byte value (little-endian) whose product with the hash prime is p."""
    return (p * INV) & M32


@functools.lru_cache(maxsize=None)
def _advances(limit: int = 70000):
    adv, pos, cnt, step = [0], 0, 64, 1
    while pos <= limit:
        pos += step
        step = cnt >> 6
        cnt += 1
        adv.append(pos)
    return adv


def advance(q: int) -> int:
    """Distance of search probe q from probe 0 of its run."""
    return _advances()[q]


def lane_of(q: int, post_run: bool) -> tuple[int, int]:
    """(batch, lane) of search probe q in a run that began with (post_run) or without a post probe."""
    k = q + (1 if post_run else 0)
    return k // 32, k % 32


class Hit(NamedTuple):
    ip: int                  # position of the match after the catch-up
    m: int                   # position of its source
    lit: int                 # literal run before it
    ml: int                  # match length (>= 4)
    post: bool               # found by the post-match probe (a zero-literal sequence)
    q: int                   # search-probe index of the hit within its run (-1 for a post hit)
    post_run: bool           # the run began with a post probe
    batch: int               # batch of the run the hit lies in
    lane: int                # lane of the hit in that batch
    src: str                 # how the GPU sees the candidate: "table", "lane" (nearest earlier lane) or "put2"
    store: str               # who stored it: "zero" (cleared table), "init", "probe", "post" or "put2"
    catch: int               # catch-up length
    stop: str                # what ended the catch-up: "anchor", "m0", "byte" or "post" (no catch-up)
    clip: bool               # LZ4_count stopped at matchlimit
    end: int                 # ip + ml: where the match ends
    before: int              # valid lanes before the hit lane with the hit's hash
    after: int               # valid lanes after the hit lane with the hit's hash
    far_ok: bool             # the farthest earlier same-hash lane holds the hit's 4 bytes
    near_ok: bool            # the nearest one does
    h2_post: bool            # hash(ip_post - 2) == hash(post probe) in this batch (batch 0 of a post run)
    same2: bool              # a valid lane at or before the hit shares hash(ip_post - 2)
    straddle: bool           # a lane at or before the hit shares its hash with a lane after it


class RunEnd(NamedTuple):
    post_run: bool
    probes: int              # search probes executed before the run met the end
    batch: int
    lane: int                # the first lane whose probe does not execute


class Result(NamedTuple):
    ret: int
    data: bytes
    hits: list
    end: RunEnd | None
    fail: int = 0            # which limited-output check failed: 1 literals, 2 match, 3 last literals


def _grams(d: bytes):
    a = np.frombuffer(d, dtype=np.uint8).astype(np.uint64)
    if a.size < 4:
        return [], []
    g = a[:-3] | (a[1:-2] << 8) | (a[2:-1] << 16) | (a[3:] << 24)
    h = ((g * np.uint64(PRIME)) & np.uint64(M32)) >> np.uint64(19)
    return g.astype(np.int64).tolist(), h.astype(np.int64).tolist()


def _common(d: bytes, a: int, b: int, lim: int) -> int:
    k = 0
    while a + k < lim:
        w = min(64, lim - a - k)
        if d[a + k:a + k + w] == d[b + k:b + k + w]:
            k += w
            continue
        while d[a + k] == d[b + k]:
            k += 1
        return k
    return k


def _run_header(out: bytearray, run: int) -> None:
    if run >= 15:
        out.append(0xF0)
        rest = run - 15
        while rest >= 255:
            out.append(255)
            rest -= 255
        out.append(rest)
    else:
        out.append(run << 4)


def encode(data: bytes, cap: int | None = None) -> Result:
    """LZ4Codec.Encode at L00_FAST of a block below 65 547 bytes -> (return code, bytes, trace)."""
    d = bytes(data)
    n = len(d)
    assert n < LIMIT_64K
    if n == 0:
        return Result(0, b"", [], None)
    bound = n + n // 255 + 16
    cap = bound if cap is None else cap
    limited = cap < bound
    G, H = _grams(d)
    table = [0] * 8192
    who = [("zero", -1, -1)] * 8192          # (kind, episode, batch) of the last store to each slot
    out = bytearray()
    hits, end = [], None
    anchor = 0

    def fail(check):
        return Result(-1, b"", hits, end, check)

    if n >= MINLENGTH:
        mfl1, mlim = n - MFLIMIT + 1, n - LASTLITERALS
        table[H[0]] = 0
        who[H[0]] = ("init", -1, -1)
        ip, episode, post_ip = 1, 0, None     # post_ip: position of the post probe that opens this episode
        while True:
            post_run = post_ip is not None
            hit = None
            if post_run:
                ip_post = post_ip
                h2 = H[ip_post - 2]
                table[h2] = ip_post - 2
                who[h2] = ("put2", episode, 0)
                h = H[ip_post]
                m, w = table[h], who[h]
                table[h] = ip_post
                who[h] = ("post", episode, 0)
                if G[m] == G[ip_post]:
                    hit = (ip_post, m, w, -1, 0, 0)
                base = ip_post + 1
            else:
                base = ip
            if hit is None:
                q = 0
                while True:
                    cur = base + advance(q)
                    if base + advance(q + 1) > mfl1:
                        b, ln = lane_of(q, post_run)
                        end = RunEnd(post_run, q, b, ln)
                        break
                    h = H[cur]
                    m, w = table[h], who[h]
                    b, ln = lane_of(q, post_run)
                    table[h] = cur
                    who[h] = ("probe", episode, b)
                    if G[m] == G[cur]:
                        hit = (cur, m, w, q, b, ln)
                        break
                    q += 1
            if hit is None:
                break
            cur, m, w, q, b, ln = hit
            kind, wep, wb = w
            if kind in ("probe", "post") and wep == episode and wb == b:
                src = "lane"
            elif kind == "put2" and wep == episode and b == 0:
                src = "put2"
            else:
                src = "table"
            lanes = _batch_lanes(H, G, base, post_run, post_ip, b, mfl1)
            ip, catch = cur, 0
            if q < 0:
                stop = "post"
            else:
                while True:
                    if not ip > anchor:
                        stop = "anchor"
                        break
                    if not m > 0:
                        stop = "m0"
                        break
                    if d[ip - 1] != d[m - 1]:
                        stop = "byte"
                        break
                    ip, m, catch = ip - 1, m - 1, catch + 1
            lit = ip - anchor
            if q >= 0:
                if limited and len(out) + 1 + lit + 8 + lit // 255 > cap:
                    return fail(1)
                tok = len(out)
                _run_header(out, lit)
                out += d[anchor:ip]
            else:
                tok = len(out)
                out.append(0)
            out += bytes([(ip - m) & 0xFF, (ip - m) >> 8])
            mc = _common(d, ip + MINMATCH, m + MINMATCH, mlim)
            clip = ip + MINMATCH + mc == mlim
            if limited and len(out) + 6 + (mc + 240) // 255 > cap:
                return fail(2)
            if mc >= 15:
                out[tok] += 15
                rest = mc - 15
                out += b"\xff" * (rest // 255)
                out.append(rest % 255)
            else:
                out[tok] += mc
            hf = H[cur]
            same = [i for i, (p, v, hh, g) in enumerate(lanes) if v and hh == hf]
            earlier = [i for i in same if i < ln]
            h2l = H[post_ip - 2] if post_run and b == 0 else None
            upto = [i for i in range(ln + 1) if lanes[i][1]]
            hits.append(Hit(
                ip=ip, m=m, lit=lit, ml=mc + MINMATCH, post=q < 0, q=q, post_run=post_run, batch=b, lane=ln,
                src=src, store=kind, catch=catch, stop=stop, clip=clip, end=ip + MINMATCH + mc,
                before=len(earlier), after=len([i for i in same if i > ln]),
                far_ok=bool(earlier) and lanes[earlier[0]][3] == G[cur],
                near_ok=bool(earlier) and lanes[earlier[-1]][3] == G[cur],
                h2_post=h2l is not None and lanes[0][2] == h2l,
                same2=h2l is not None and any(lanes[i][2] == h2l for i in upto),
                straddle=any(lanes[j][1] and lanes[j][2] == lanes[i][2] for i in upto for j in range(ln + 1, 32))))
            ip = ip + MINMATCH + mc
            anchor = ip
            if ip >= mfl1:
                end = None
                break
            episode += 1
            post_ip = ip
    run = n - anchor
    if limited and len(out) + run + 1 + (run + 255 - 15) // 255 > cap:
        return fail(3)
    _run_header(out, run)
    out += d[anchor:]
    return Result(len(out), bytes(out), hits, end)


def _batch_lanes(H, G, base, post_run, post_ip, b, mfl1):
    """(position, valid, hash, value) of the 32 lanes of batch b of a run."""
    lanes = []
    for ln in range(32):
        if post_run and b == 0 and ln == 0:
            p = post_ip
            lanes.append((p, True, H[p], G[p]))
            continue
        q = 32 * b + ln - (1 if post_run else 0)
        p = base + advance(q)
        ok = base + advance(q + 1) <= mfl1
        lanes.append((p, ok, H[p] if ok else -1, G[p] if ok else -1))
    return lanes


# ---- input builders ---------------------------------------------------------------------------------------

class Block:
    """A block under construction: unique-4-gram filler by default, with values and copies placed into it."""

    def __init__(self, n: int, seed: int):
        self.a = bytearray(unique_filler(n, seed))

    def put(self, pos: int, v: int) -> None:
        self.a[pos:pos + 4] = int(v).to_bytes(4, "little")

    def copy(self, dst: int, src: int, length: int) -> None:
        self.a[dst:dst + length] = self.a[src:src + length]

    def gram(self, pos: int) -> int:
        return int.from_bytes(self.a[pos:pos + 4], "little")

    def bytes(self) -> bytes:
        return bytes(self.a)


@functools.lru_cache(maxsize=None)
def _filler(n: int, seed: int) -> bytes:
    rng = np.random.default_rng(seed)
    pool = rng.integers(0, 256, n + 1024, dtype=np.uint8).tolist()
    out, seen, k = bytearray(), set(), 0
    for i in range(n):
        while True:
            c = pool[k % len(pool)]
            k += 1
            if i < 3:
                break
            g = bytes(out[-3:]) + bytes([c])
            if g not in seen:
                seen.add(g)
                break
            pool[k % len(pool)] = (pool[k % len(pool)] + 97) & 0xFF
        out.append(c)
    return bytes(out)


def unique_filler(n: int, seed: int = 0) -> bytes:
    """n bytes in which no 4-byte value occurs twice."""
    return _filler(n, seed)


def value_with_hash(h: int, low: int) -> int:
    """A 4-byte value whose 13-bit hash is h; `low` (19 bits) picks which one: bits 0-2 leave the 16-bit tag alone."""
    return value_of(((h & 0x1FFF) << 19) | (low & 0x7FFFF))


def same_hash_other_tag(v: int, k: int = 1) -> int:
    """A value with v's hash and a different 16-bit tag."""
    p = product(v)
    return value_of((p & ~0x7FFF8) | ((((p >> 3) + 0x9E5 * k) & 0xFFFF) << 3))


def same_hash_same_tag(v: int, k: int = 1) -> int:
    """A different value with v's hash and v's tag: the products differ only in bits 0-2."""
    p = product(v)
    return value_of((p & ~7) | ((p + k) & 7))


def first_run_probe(q: int) -> int:
    """Position of search probe q of the block's first run (it starts at position 1)."""
    return 1 + advance(q)
