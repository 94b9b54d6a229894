"""Composes LZ4 blocks from explicit plans, with the raw data each plan defines.

A plan is a list of sequences `(literals, offset, match_length)` plus the terminal literal run.
`compose` writes the block bytes and, independently of any decoder, the raw bytes: each match is
expanded by the copy rule of the format (byte k of a match is the byte `offset` positions before
it), so overlapping copies are right by construction.  The tests use the raw bytes as the exact
expected output of a decoder, and the recorded token positions to aim sequences at the decoder's
segment and step boundaries.

A plan is "clean" when it follows the end rules of the block format: the last match starts at
least 12 bytes before the end of the block (MFLIMIT) and the last 5 bytes are literals
(LASTLITERALS); every offset is between 1 and the number of bytes already produced.  `broken`
builds plans that break exactly one of those rules.
"""
from __future__ import annotations

from typing import NamedTuple

import numpy as np

MINMATCH, MFLIMIT, LASTLITERALS, MAX_OFFSET = 4, 12, 5, 65535


class Block(NamedTuple):
    stream: bytes
    raw: bytes | None        # None when an offset is 0 or reaches before the first output byte
    tokens: list             # stream position of every token, the terminal's last
    outs: list               # output position where every sequence begins, the terminal's last


def _length(out: bytearray, v: int) -> None:
    """The extension bytes of a length whose 4-bit field holds 15: 255-bytes, then the rest."""
    while v >= 255:
        out.append(255)
        v -= 255
    out.append(v)


def compose(seqs, tail: bytes) -> Block:
    stream, raw = bytearray(), bytearray()
    tokens, outs = [], []
    valid = True
    for lit, off, ml in seqs:
        assert ml >= MINMATCH and 0 <= off <= MAX_OFFSET, (ml, off)
        tokens.append(len(stream)); outs.append(len(raw))
        L, M = len(lit), ml - MINMATCH
        stream.append((min(L, 15) << 4) | min(M, 15))
        if L >= 15:
            _length(stream, L - 15)
        stream += lit
        stream += bytes([off & 0xFF, off >> 8])
        if M >= 15:
            _length(stream, M - 15)
        raw += lit
        if off == 0 or off > len(raw):
            valid = False
        if valid:
            # byte by byte this is `raw.append(raw[-off])`: byte k of the match is byte k mod off of
            # the `off` bytes before the match, so the match is that window repeated
            window = raw[len(raw) - off:]
            raw += (window * (ml // off + 1))[:ml]
        else:
            raw += bytes(ml)              # keeps the output positions right
    tokens.append(len(stream)); outs.append(len(raw))
    stream.append(min(len(tail), 15) << 4)
    if len(tail) >= 15:
        _length(stream, len(tail) - 15)
    stream += tail
    raw += tail
    return Block(bytes(stream), bytes(raw) if valid else None, tokens, outs)


def sequence_bytes(lit_len: int, ml: int) -> int:
    """Stream bytes of one sequence (ml = 0: the terminal one)."""
    ext = lambda v: 0 if v < 15 else (v - 15) // 255 + 1
    return 1 + ext(lit_len) + lit_len + (2 + ext(ml - MINMATCH) if ml else 0)


def decoded_size(seqs, tail: bytes) -> int:
    return sum(len(l) + m for l, _, m in seqs) + len(tail)


def clean(seqs, tail: bytes) -> bool:
    pos = 0
    for lit, off, ml in seqs:
        pos += len(lit)
        if not 1 <= off <= pos:
            return False
        pos += ml
    if not seqs:
        return True
    last_start = pos - seqs[-1][2]
    return len(tail) >= LASTLITERALS and pos + len(tail) - last_start >= MFLIMIT


# ---- plan builders -------------------------------------------------------------------------------------

class Bytes:
    """Literal bytes: slices of one seeded pool (byte values 1..255, so a stale zero never passes)."""

    def __init__(self, seed: int, size: int = 1 << 22):
        self.pool = np.random.default_rng(seed).integers(1, 256, size, dtype=np.uint8).tobytes()
        self.rng = np.random.default_rng(seed + 1)
        self.at = 0

    def __call__(self, n: int) -> bytes:
        assert n <= len(self.pool)
        self.at = (self.at + 7919) % len(self.pool)               # a new window each call, no rng call
        s = self.at % (len(self.pool) - n + 1)
        return self.pool[s:s + n]


def tail_for(seqs, lit: Bytes, at_least: int = LASTLITERALS) -> bytes:
    """The shortest terminal literal run (>= at_least) that makes `seqs` clean."""
    if not seqs:
        return lit(max(at_least, 1))
    need = max(at_least, MFLIMIT - seqs[-1][2], LASTLITERALS)
    return lit(need)


def pad_to_stream_size(seqs, lit: Bytes, n: int, first: int = LASTLITERALS) -> bytes:
    """A terminal literal run (>= `first` bytes) that makes the clean block exactly `n` stream bytes."""
    base = len(compose(seqs, b"").stream) - 1
    for t in range(max(first, MFLIMIT - seqs[-1][2] if seqs else 1), n):
        size = base + 1 + (0 if t < 15 else (t - 15) // 255 + 1) + t
        if size == n:
            return lit(t)
        if size > n:
            break
    raise ValueError(f"no terminal run gives a stream of {n} bytes")


def chain(lit: Bytes, depth: int, length: int, overlap: int = 0):
    """`depth` matches in a row, each reading the output of the one before it.  The first copies its
    own literals; every later one has no literals and copies the previous match (offset = length)
    or, with `overlap` > 0, the previous match's last bytes and its own (offset = length - overlap)."""
    off = length - overlap
    seqs = [(lit(off), off, length)]
    seqs += [(b"", off, length)] * (depth - 1)
    return seqs


def far_fillers(lit: Bytes, count: int, pos: int, ml: int = 4):
    """`count` sequences of 4 literals and a match of `ml` bytes from output byte 0 onwards
    (the block must begin with at least `ml` literals).  `pos` is the output position where they start."""
    seqs = []
    for _ in range(count):
        pos += 4
        seqs.append((lit(4), pos, ml))
        pos += ml
    return seqs


def broken(rule: str, lit: Bytes):
    """A plan that breaks exactly one rule: 'mflimit' (the last match starts 11 bytes before the end),
    'lastliterals' (the block ends with 4 literals), 'offset_zero', 'offset_far' (the offset reaches one byte
    before the first output byte), 'trailing_match' (the block ends with a match: no terminal literals)."""
    head = [(lit(20), 7, 9), (lit(3), 20, 6)]
    if rule == "mflimit":
        return head + [(lit(2), 4, 6)], lit(5)
    if rule == "lastliterals":
        return head + [(lit(2), 4, 8)], lit(4)
    if rule == "offset_zero":
        return head + [(lit(2), 0, 6)], lit(12)
    if rule == "offset_far":
        return head + [(lit(2), 20 + 9 + 3 + 6 + 2 + 1, 6)], lit(12)
    if rule == "trailing_match":
        return head + [(lit(2), 4, 12)], b""
    raise ValueError(rule)


BROKEN_RULES = ("mflimit", "lastliterals", "offset_zero", "offset_far", "trailing_match")


def random_plan(rng: np.random.Generator, lit: Bytes, limit: int, stop: float = 0.002):
    """A seeded random clean plan that decodes to at most `limit` bytes.  Heavy tails everywhere: a third of
    the sequences have no literals, literal runs reach thousands of bytes, match lengths 4..20 000, offsets
    1..65 535, and a quarter of the matches read the previous match's output (dependency chains).  After each
    sequence the plan ends with probability `stop`."""
    seqs, pos, prev_ml = [], 0, 0
    while True:
        k = 256                                   # random draws in batches: one numpy call per column
        Ls = np.minimum(rng.pareto(1.1, k) * 3 + 1, 6000).astype(np.int64)
        Ls[rng.random(k) < 0.35] = 0
        mls = MINMATCH + np.minimum(rng.pareto(1.0, k) * 2, 20000 - MINMATCH).astype(np.int64)
        kinds, near = rng.random(k), rng.integers(-3, 4, k)
        short, wide = rng.integers(1, 160, k), rng.integers(1, MAX_OFFSET + 1, k)
        tailed = np.minimum(rng.pareto(0.8, k) * 8 + 1, MAX_OFFSET).astype(np.int64)
        ends = rng.random(k) < stop
        for L, ml, kd, dn, sh, wd, tl, end in zip(Ls.tolist(), mls.tolist(), kinds.tolist(), near.tolist(),
                                                   short.tolist(), wide.tolist(), tailed.tolist(), ends.tolist()):
            if pos + L == 0:
                L = 1
            if pos + L + ml + max(LASTLITERALS, MFLIMIT - ml) > limit:
                return seqs, _random_tail(rng, seqs, lit, limit - pos)
            start = pos + L
            if kd < 0.25 and prev_ml:
                off = prev_ml + dn                                      # the previous match's output
            elif kd < 0.45:
                off = sh                                                # short periods
            elif kd < 0.7:
                off = wd
            else:
                off = tl
            off = max(1, min(off, start, MAX_OFFSET))
            seqs.append((lit(L), off, ml))
            pos = start + ml
            prev_ml = ml
            if end:
                return seqs, _random_tail(rng, seqs, lit, limit - pos)


def _random_tail(rng, seqs, lit: Bytes, room: int) -> bytes:
    return tail_for(seqs, lit, min(int(rng.integers(LASTLITERALS, 40)), room))
