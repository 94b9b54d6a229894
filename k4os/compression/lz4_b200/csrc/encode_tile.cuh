// encode_tile.cuh -- bit-exact LZ4 L00_FAST encoder for blocks below the 64 KiB table limit
// (n < 65 547: the reference's byU16 case, LL64.fast.cs:526,548), one warp per block with the whole
// block staged in shared memory.
//
// The reference's match search is a serial chain per probe (hash -> slot load -> slot store ->
// 4-byte compare, LL64.fast.cs:158-234).  Inside one search run the probe POSITIONS do not depend on
// the data (step = searchMatchNb++ >> 6, :159-170), only the table contents do -- and the only table
// writes between two probes of a run are the run's own earlier probes.  So a warp evaluates 32
// consecutive probes at once: every lane hashes its position, loads the slot, and `__match_any_sync`
// on the hash substitutes the position of the nearest earlier lane with the same hash (= the store
// the serial code would have done in between).  The first hitting lane wins; lanes up to it commit
// their slot stores (last writer per hash), later lanes are discarded -- exactly the serial history.
// The probe right after a match (put ip-2, test ip, LL64.fast.cs:394-466) rides as lane 0 of the
// next batch.  Common-prefix counting and the backward catch-up are lane-parallel; the block
// (TMA bulk load) and the 16 KiB u16 table live in shared memory, so the chain never waits on HBM.
//
// Reference: /root/reference/src/K4os.Compression.LZ4/Engine/x64/LL64.fast.cs:35-576,
// Engine/LL.tools.cs:38-51, Engine/x64/LL64.tools.cs:87-133; step numbers = SURVEY.md App. A.
#pragma once
#include "common.cuh"
#include "encode_generic.cuh"

namespace k4 {


__device__ __forceinline__ uint32_t lds_u32u(const uint8_t* p) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
    return __funnelshift_r(w[0], w[1], (uint32_t)(a & 3) * 8);
}

// Distance of search probe q from probe 0 of its run.  The reference advances by `step`, then
// sets step = searchMatchNb++ >> 6 with searchMatchNb starting at 64 (LL64.fast.cs:159-170): the
// first advance is 1, advance i >= 1 is (63 + i) >> 6, so the first 65 advances are 1, the next 64 are 2, ...
// Experiment switches of the match path (tools/build_variant.py; defaults = the shipped build):
//   K4_ENC_OVL  issue the first LZ4_count round together with the backward catch-up (one memory round trip instead of two)
//   K4_ENC_PF   bit 0: lanes whose tag agrees also prefetch the sectors around their candidate (count / catch-up then hit L1);
//               bit 1: prefetch the input ahead of the probes
#ifndef K4_ENC_OVL
#define K4_ENC_OVL 1
#endif
#ifndef K4_ENC_PF
#define K4_ENC_PF 0
#endif
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" :: "l"(p)); }

__device__ __forceinline__ uint32_t probe_advance(uint32_t q) {
    if (q <= 64u) return q;                       // the common case: a run shorter than 65 probes
    if (q == 0) return 0;
    const uint32_t c = 63u + q, k = c >> 6;
    return 1u + 32u * k * (k - 1u) + (c - 64u * k) * k;
}

// The encoder proper.  STAGED: the block sits in shared memory at `sin` (sin[p] == src[p]);
// otherwise positions are read from global memory through L1 (more blocks in flight per SM).
// Returns the engine's value: bytes written, 0 when the reference's limitedOutput checks fail.
// TAGMODE: 0 = plain u16 slots; 1 = u16 slots + one filter byte per slot behind the table, both loaded per probe;
// 2 = 32-bit slots (position | 16-bit tag << 16); 3 = as 1, but the position is loaded only when the tag agrees.
template <bool STAGED, bool HARD = true, bool GTAB = false, int TAGMODE = (K4_ENC_TAGS ? 1 : 0)>
__device__ int encode_spec_warp(const uint8_t* __restrict__ src, const uint8_t* sin, const uint32_t n,
                                uint8_t* __restrict__ dst, const int cap, const int hardCap, uint16_t* table) {
    const int lane = lane_id();
    const int64_t hard = hardCap;       // physical write bound (pickler, see pickle.cuh); 0x7fffffff otherwise
#define RD32(p) (STAGED ? lds_u32u(sin + (p)) : ldg_u32u(src + (p)))
    // GTAB: the table lives in global memory; its accesses go to L2 (.cg) so that the little L1 left
    // beside 224 KiB of shared memory keeps the input windows of all warps of the SM
#ifndef K4_ENC_GTAB_L1
#define K4_ENC_GTAB_L1 0
#endif
#define TGET(h) ((GTAB && !K4_ENC_GTAB_L1) ? (uint32_t)__ldcg(table + (h)) : (uint32_t)table[(h)])
    // Tag filter.  Next to every 16-bit slot sits a tag: bits below the hash of the same product whose
    // bits 19..31 are the hash, taken from the 4 bytes AT the stored position.  Equal 4-byte values
    // have equal tags, so a probe only has to fetch its candidate's bytes (a scattered global load into
    // the 64 KiB window, 32 of them per batch otherwise) when the tags agree -- one probe in 256 (65 536)
    // by chance, plus the true hits.  The decision `hit` is unchanged.
    constexpr bool TAGS = TAGMODE != 0;
    constexpr uint32_t TAG_SHIFT = TAGMODE == 2 ? 3u : 11u, TAG_MASK = TAGMODE == 2 ? 0xFFFFu : 0xFFu;
    uint8_t* const tags = reinterpret_cast<uint8_t*>(table) + ENC_TABLE_BYTES;
    uint32_t* const table32 = reinterpret_cast<uint32_t*>(table);
    auto tagGet = [&](uint32_t h) -> uint32_t {
        return (GTAB && !K4_ENC_GTAB_L1) ? (uint32_t)__ldcg(tags + h) : (uint32_t)tags[h];
    };
    auto slotPut = [&](uint32_t h, uint32_t pos, uint32_t tg) {
        if (TAGMODE == 2) {
            if (GTAB) __stcg(table32 + h, pos | (tg << 16)); else table32[h] = pos | (tg << 16);
        } else {
            if (GTAB && !K4_ENC_GTAB_L1) __stcg(table + h, (uint16_t)pos); else table[h] = (uint16_t)pos;
            if (TAGS) { if (GTAB && !K4_ENC_GTAB_L1) __stcg(tags + h, (uint8_t)tg); else tags[h] = (uint8_t)tg; }
        }
    };
#define RD8(p) (STAGED ? (uint32_t)sin[(p)] : (uint32_t)__ldg(src + (p)))
    {   // LZ4_initStream: zero the table (LL.tools.cs:235-239); every slot then "holds" position 0
        const uint32_t t0 = (TAGS && n >= 4) ? (((RD32(0) * 2654435761u) >> TAG_SHIFT) & TAG_MASK) : 0u;
        const uint32_t fillT = TAGMODE == 2 ? (t0 << 16) : 0u;
        uint4* t = reinterpret_cast<uint4*>(table);
        constexpr int TBYTES = TAGMODE == 2 ? 2 * ENC_TABLE_BYTES : ENC_TABLE_BYTES;
        for (int i = lane; i < TBYTES / 16; i += 32) {
            if (GTAB) __stcg(t + i, make_uint4(fillT, fillT, fillT, fillT)); else t[i] = make_uint4(fillT, fillT, fillT, fillT);
        }
        if (TAGMODE == 1 || TAGMODE == 3) {
            const uint32_t b4 = t0 * 0x01010101u;
            uint4* g = reinterpret_cast<uint4*>(tags);
            for (int i = lane; i < (ENC_TABLE_BYTES / 2) / 16; i += 32) {
                if (GTAB) __stcg(g + i, make_uint4(b4, b4, b4, b4)); else g[i] = make_uint4(b4, b4, b4, b4);
            }
        }
        __syncwarp();
    }
    const bool limited = !(cap >= max_output_size((int)n));                           // LL64.fast.cs:524
    const int64_t olimit = cap;
    uint32_t ip = 0, anchor = 0, op = 0;

    if (n >= (uint32_t)MINLENGTH) {                                               // :117
        const uint32_t mfl1 = n - MFLIMIT + 1, mlim = n - LASTLITERALS;           // :70-71
        if (lane == 0) { const uint32_t p0 = RD32(0) * 2654435761u; slotPut(p0 >> 19, 0u, (p0 >> TAG_SHIFT) & TAG_MASK); }   // :120
        __syncwarp();
        ip = 1;
        bool post = false;              // lane 0 of the next batch is the post-match probe at ip
        uint32_t q0 = 0;                // first search-probe index of the next batch
        uint32_t base = 1;              // position of search probe 0 of the current run
        for (;;) {
            // ---- one batch of up to 32 probes (App. A step 3, and step 8 as lane 0) -----------------
            uint32_t h2 = 0xFFFFFFFFu, tag2 = 0;
            if (post) { const uint32_t p2 = RD32(ip - 2) * 2654435761u; h2 = p2 >> 19; tag2 = (p2 >> TAG_SHIFT) & TAG_MASK; }   // put(ip-2), :394
            const bool isPost = post && lane == 0;
            const uint32_t q = q0 + (uint32_t)lane - (post ? 1u : 0u);            // search-probe index (lanes >= 1 if post)
            const uint32_t pos = isPost ? ip : base + probe_advance(q);
            // a search probe executes only if the NEXT probe position stays <= mflimitPlusOne (:172)
            const bool valid = isPost || (base + probe_advance(q + 1) <= mfl1);
            const uint32_t v = valid ? RD32(pos) : 0u;
            const uint32_t prod = v * 2654435761u;
            const uint32_t h = valid ? prod >> 19 : (0x10000u + (uint32_t)lane);
            const uint32_t tg = (prod >> TAG_SHIFT) & TAG_MASK;
            uint32_t cand = 0u, ctag = tg;                                        // TAGMODE 0: no filter, every candidate is fetched
            bool lazyPos = false;                                                 // TAGMODE 3: position not loaded yet
            if (TAGMODE == 2) {
                const uint32_t e32 = valid ? ((GTAB && !K4_ENC_GTAB_L1) ? __ldcg(table32 + h) : table32[h]) : 0xFFFF0000u;
                cand = e32 & 0xFFFFu; ctag = e32 >> 16;
                if (!valid) ctag = 0x10000u;
            } else if (TAGMODE == 3) {
                ctag = valid ? tagGet(h) : 0x100u;
                lazyPos = true;
            } else {
                cand = valid ? TGET(h) : 0u;
                if (TAGMODE == 1) ctag = valid ? tagGet(h) : 0x100u;
            }
            if (h == h2) { cand = ip - 2; ctag = TAGS ? tag2 : tg; lazyPos = false; }   // sees the put(ip-2)
            const unsigned peers = __match_any_sync(FULL, h);
            const unsigned earlier = peers & ((1u << lane) - 1u);
            const int fromLane = earlier ? 31 - __clz(earlier) : lane;
            const uint32_t fwdPos = __shfl_sync(FULL, pos, fromLane);
            const uint32_t fwdTag = __shfl_sync(FULL, tg, fromLane);
            if (earlier) { cand = fwdPos; ctag = TAGS ? fwdTag : tg; lazyPos = false; }   // sees the nearest earlier store
            bool hit = false;
            if (valid && ctag == tg) {                                            // :228 (byU16: no distance test)
                if (TAGMODE == 3 && lazyPos) cand = TGET(h);
                hit = RD32(cand) == v;
                if (TAGS && !STAGED && (K4_ENC_PF & 1)) {                          // few lanes get here: the tag filter
                    prefetch_l1(src + (cand + 32u < n ? cand + 32u : n - 1u));
                    if (cand >= 8u) prefetch_l1(src + cand - 8u);
                }
            }
            if (!STAGED && (K4_ENC_PF & 2) && lane == 0) prefetch_l1(src + (pos + 384u < n ? pos + 384u : n - 1u));
            const unsigned hits = __ballot_sync(FULL, hit);
            const unsigned ends = __ballot_sync(FULL, !valid);
            const int f = hits ? __ffs(hits) - 1 : 32;
            const int e = ends ? __ffs(ends) - 1 : 32;
            if (e < f) break;                                                     // ran into the end: last literals
            // commit the slot stores of probes 0..f in serial order: last writer per hash wins
            {
                const unsigned upto = (f >= 31) ? 0xffffffffu : ((2u << f) - 1u);
                const unsigned later = peers & ~((2u << lane) - 1u) & upto;       // lanes in (lane, f] with my hash
                const bool doStore = valid && ((1u << lane) & upto) && !(lane < 31 ? later : 0u);
                if (post) {
                    const unsigned same2 = __ballot_sync(FULL, valid && h == h2) & upto;
                    if (lane == 0 && !same2) {                                    // nobody overwrote the put(ip-2)
                        slotPut(h2, ip - 2, tag2);
                    }
                }
                if (doStore) slotPut(h, pos, tg);
                __syncwarp();
            }
            if (f == 32) {                                                        // 32 misses: keep searching
                if (post) { post = false; base = ip + 1; q0 = 31; }
                else q0 += 32;
                continue;
            }
            const bool zeroLit = post && f == 0;                                  // :459-463
            uint32_t m = __shfl_sync(FULL, cand, f);
            ip = __shfl_sync(FULL, pos, f);
            // LZ4_count does not depend on the catch-up: [ip-c, ip+4) is known equal, so counting from the hit's
            // ip+4 and adding c gives the reference's value (ip+4 <= mflimit+4 < matchlimit).  Its first round of
            // loads is issued before the catch-up loop so that both wait for memory at the same time.
            const uint32_t a0h = ip + MINMATCH, b0h = m + MINMATCH;
            uint32_t x1 = 0u;
            if (K4_ENC_OVL) {
                const uint32_t a = a0h + 4u * lane;
                if (lane < 8 && (int)mlim - (int)a > 0) x1 = RD32(a) ^ RD32(b0h + 4u * lane);
            }
            uint32_t caught = 0;
            if (!zeroLit) {                                                       // step 4: catch-up, :237-242
                // eight lanes first: a catch-up is rarely longer, and lanes that do not take part issue no load
                for (int width = 8;; width = 32) {
                    const bool part = lane < width;
                    const bool ok = !part || ((ip > anchor + lane) && (m > (uint32_t)lane) &&
                                              (RD8(ip - 1 - lane) == RD8(m - 1 - lane)));
                    const unsigned bad = __ballot_sync(FULL, !ok);
                    const int c = bad ? __ffs(bad) - 1 : width;
                    ip -= c; m -= c; caught += (uint32_t)c;
                    if (bad) break;
                }
            }
            // ---- step 5/6: literal run, offset, match length -----------------------------------------
            const uint32_t lit = ip - anchor;
            if (!zeroLit && limited && (int64_t)op + 1 + lit + 8 + lit / 255 > olimit) return 0;   // :246-251
            uint32_t mc = caught;
            {   // LZ4_count(ip+4, m+4, matchlimit), 4 bytes per lane, :328; the first round looks at 32 bytes
                // (eight lanes: half of all matches end there and the other lanes' lines are not fetched)
                uint32_t a0 = a0h, b0 = b0h;
                for (int width = 8;; width = 32) {
                    const uint32_t a = a0 + 4u * lane, bb = b0 + 4u * lane;
                    const bool part = lane < width;
                    const int room = (int)mlim - (int)a;                          // bytes of this lane below matchlimit
                    const uint32_t x = (K4_ENC_OVL && width == 8) ? x1 : ((part && room > 0) ? (RD32(a) ^ RD32(bb)) : 0u);
                    int eq = x ? ((__ffs(x) - 1) >> 3) : 4;
                    if (eq > room) eq = room < 0 ? 0 : room;
                    if (!part) eq = 4;
                    const unsigned stop = __ballot_sync(FULL, eq < 4);
                    if (stop) {
                        const int s = __ffs(stop) - 1;
                        mc += 4u * s + (uint32_t)__shfl_sync(FULL, eq, s);
                        break;
                    }
                    mc += 4u * width; a0 += 4u * width; b0 += 4u * width;
                }
            }
            const uint32_t hdr = run_header_size(lit);
            const uint32_t afterOff = op + hdr + lit + 2;
            if (limited && (int64_t)afterOff + 6 + (mc + 240) / 255 > olimit) return 0;   // :332-362
            if (HARD && (int64_t)afterOff + (mc >= 15 ? (mc - 15) / 255 + 1 : 0) > hard) return 0;
            // emit: token, literal length bytes, literals, offset, match length bytes
            {
                const uint32_t mlTok = mc >= 15 ? 15u : mc;
                if (lane == 0) {
                    if (lit >= 15) {
                        uint32_t o = op, rest = lit - 15;
                        dst[o++] = (uint8_t)(0xF0 | mlTok);
                        for (; rest >= 255; rest -= 255) dst[o++] = 255;
                        dst[o] = (uint8_t)rest;
                    } else dst[op] = (uint8_t)((lit << 4) | mlTok);
                    dst[afterOff - 2] = (uint8_t)(ip - m);
                    dst[afterOff - 1] = (uint8_t)((ip - m) >> 8);
                }
                for (uint32_t i = lane; i < lit; i += 32) dst[op + hdr + i] = RD8(anchor + i);
                op = afterOff;
                if (mc >= 15) {                                                   // :365-379
                    const uint32_t rest = mc - 15, nff = rest / 255;
                    for (uint32_t i = lane; i < nff; i += 32) dst[op + i] = 0xFF;
                    if (lane == 0) dst[op + nff] = (uint8_t)(rest % 255);
                    op += nff + 1;
                }
            }
            ip += mc + MINMATCH;
            anchor = ip;                                                          // :388
            if (ip >= mfl1) break;                                                // :391
            post = true; q0 = 0; base = ip + 1;                                   // step 8 rides with the next batch
        }
    }
    {   // ---- step 9: last literals, :469-503 -----------------------------------------------------------
        const uint32_t run = n - anchor;
        if (limited && (int64_t)op + run + 1 + (run + 255 - 15) / 255 > olimit) return 0;
        const uint32_t hdr = run_header_size(run);
        if (HARD && (int64_t)op + hdr + run > hard) return 0;
        if (lane == 0) write_run_header(dst, op, run);
        op += hdr;
        for (uint32_t i = lane; i < run; i += 32) dst[op + i] = RD8(anchor + i);
        op += run;
        return (int)op;
    }
#undef RD32
#undef TGET
#undef RD8
}

// Encoder path counters (k4lz4_encode_stats): blocks of n > 0 encoded by [0] the shared-memory-table warps,
// [1] the global-table warps (both with encode_spec_warp), [2] the u32-table engine (encode_block_warp, either
// warp kind).  Diagnostics only: the tests read them to see which warps did the work.
__device__ unsigned long long g_encode_stats[3];

// Persistent encoder, one warp per block at a time, one warp per CTA (a CTA leaves as soon as ITS warp
// runs out of blocks, so the CTAs of the next launch on another stream move in without a gap).  Blocks
// are handed out by a device counter.  Input and output stay in global memory.  Two kernels pull from
// the same counter and run concurrently: `encode_spec_kernel` keeps its 16 KiB hash table in shared
// memory (ENC_SM_WARPS of them fill an SM), `encode_spec_gtab_kernel` keeps it in an L2-resident
// workspace -- slower per block, but those warps use issue slots and registers the others leave idle.
template <bool GTAB>
__device__ __forceinline__ void encode_persistent_warp(
        const uint8_t* __restrict__ srcBase, const int64_t* __restrict__ srcOff,
        const int32_t* __restrict__ srcLen, uint8_t* __restrict__ dstBase,
        const int64_t* __restrict__ dstOff, const int32_t* __restrict__ dstCap,
        int32_t* __restrict__ outLen, const int nBlocks, int level,
        uint32_t* __restrict__ nextBlock, uint16_t* const table, const int reserve) {
    const int lane = lane_id();
    const bool enforce32 = (level & ENC_FLAG_X32) != 0;   // LL.Enforce32 (LL.tools.cs:29): hash4 for the byU32 table
    level &= 0xFF;
    for (;;) {
        int b = 0;
        if (lane == 0) {
            // the slower global-table warps leave the last `reserve` blocks to the shared-memory warps
            if (GTAB && (int)*(volatile uint32_t*)nextBlock >= nBlocks - reserve) b = nBlocks;
            else b = (int)atomicAdd(nextBlock, 1u);
        }
        b = __shfl_sync(FULL, b, 0);
        if (b >= nBlocks) return;
        const int n_ = srcLen[b];
        const uint8_t* __restrict__ src = srcBase + srcOff[b];
        uint8_t* __restrict__ dst = dstBase + dstOff[b];
        const int cap = dstCap[b];
        if (n_ <= 0) { if (lane == 0) outLen[b] = 0; continue; }
        if (level >= 3) { if (lane == 0) outLen[b] = -2; continue; }
        int r;
        if (n_ >= LIMIT_64K) r = encode_block_warp(src, n_, dst, cap, 0x7fffffff, table, enforce32);
        else r = encode_spec_warp<false, false, GTAB, GTAB ? ENC_GTAG : (K4_ENC_TAGS ? 1 : 0)>(src, nullptr, (uint32_t)n_, dst, cap, 0x7fffffff, table);
        if (lane == 0) {
            outLen[b] = r <= 0 ? -1 : r;
            atomicAdd(&g_encode_stats[n_ >= LIMIT_64K ? 2 : (GTAB ? 1 : 0)], 1ull);
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(32)
encode_spec_kernel(const uint8_t* __restrict__ srcBase, const int64_t* __restrict__ srcOff,
                   const int32_t* __restrict__ srcLen, uint8_t* __restrict__ dstBase,
                   const int64_t* __restrict__ dstOff, const int32_t* __restrict__ dstCap,
                   int32_t* __restrict__ outLen, int nBlocks, int level, uint32_t* __restrict__ nextBlock) {
    extern __shared__ __align__(128) uint8_t smem_encs[];
    encode_persistent_warp<false>(srcBase, srcOff, srcLen, dstBase, dstOff, dstCap, outLen, nBlocks, level,
                                  nextBlock, reinterpret_cast<uint16_t*>(smem_encs), 0);
}

__global__ void __launch_bounds__(32)
encode_spec_gtab_kernel(const uint8_t* __restrict__ srcBase, const int64_t* __restrict__ srcOff,
                        const int32_t* __restrict__ srcLen, uint8_t* __restrict__ dstBase,
                        const int64_t* __restrict__ dstOff, const int32_t* __restrict__ dstCap,
                        int32_t* __restrict__ outLen, int nBlocks, int level, uint32_t* __restrict__ nextBlock,
                        uint8_t* __restrict__ gtab, int reserve) {
    encode_persistent_warp<true>(srcBase, srcOff, srcLen, dstBase, dstOff, dstCap, outLen, nBlocks, level, nextBlock,
                                 reinterpret_cast<uint16_t*>(gtab + (size_t)blockIdx.x * ENC_GSLOT_BYTES), reserve);
}

}  // namespace k4
