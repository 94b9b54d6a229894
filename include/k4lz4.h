/*
 * k4lz4.h -- C ABI of libk4lz4: a B200-native (sm_100a CUDA) LZ4 *block* codec that is a
 * drop-in for ONE hot path of K4os.Compression.LZ4:
 *     LZ4Codec.Encode(..., LZ4Level.L00_FAST)   LZ4Codec.Decode(...)   LZ4Pickler.Pickle/Unpickle
 * over batches of independent blocks.  Plain C: pointers and sizes only.
 *
 * The reference (pure managed C#) has no FFI seam of its own; the seam sits directly under
 * its public block API.  Each entry point below names the reference call it replaces
 * (paths relative to /root/reference/src/K4os.Compression.LZ4/).  INTEGRATION.md shows the
 * [DllImport] stubs a maintainer adds.
 *
 * Conventions shared by every call
 *   - return values of the per-block functions and the per-block outLen[] entries are
 *     EXACTLY what the reference's LZ4Codec / LZ4Pickler would have returned for that block
 *     (bytes written, 0 for empty input, -1 when it does not fit / is malformed);
 *   - K4LZ4_E_* (<= -100) are library-level failures (no device, CUDA error, bad argument)
 *     and never collide with codec results; k4lz4_last_error() gives the message;
 *   - bytes of a destination block at index >= its returned length are never written
 *     (SpanTests.cs:36-37, PartialDecompressionTests.cs:33-35);
 *   - the library never falls back to a CPU codec: without a usable CUDA device every
 *     compute entry point returns K4LZ4_E_NODEVICE.
 */
#ifndef K4LZ4_H
#define K4LZ4_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define K4LZ4_API __declspec(dllexport)
#else
#define K4LZ4_API __attribute__((visibility("default")))
#endif

/* library-level error codes (never produced by the codec itself) */
#define K4LZ4_OK              0
#define K4LZ4_E_NODEVICE   (-100)  /* no CUDA device / driver: the product path refuses to run */
#define K4LZ4_E_CUDA       (-101)  /* a CUDA runtime call failed; see k4lz4_last_error()        */
#define K4LZ4_E_ARG        (-102)  /* null pointer / negative count / unknown memKind           */
#define K4LZ4_E_NOMEM      (-103)  /* device or pinned-host allocation failed                   */

/* per-block result that is not a reference value: "this level is not handled natively"
 * (HC/OPT levels >= 3 keep delegating to the managed engine, LZ4Codec.cs:48-50) */
#define K4LZ4_R_DELEGATE   (-2)
/* per-message result standing for the reference's InvalidDataException
 * (LZ4Pickler.unpickle.cs:131-135,142-143,115-117,126-128) */
#define K4LZ4_R_CORRUPT    (-1000)

/* memKind */
#define K4LZ4_MEM_HOST     0   /* every pointer is host memory; the call is synchronous      */
#define K4LZ4_MEM_DEVICE   1   /* every pointer (incl. offset/length arrays) is device memory
                                  of `device`; the call only enqueues work on `cudaStream`   */

/* ---- information -------------------------------------------------------------------- */

/* LZ4Codec.Version (LZ4Codec.cs:13) -- the lz4 version whose token streams are reproduced. */
K4LZ4_API int32_t k4lz4_codec_version(void);
/* Number of usable CUDA devices (0 => every compute call returns K4LZ4_E_NODEVICE). */
K4LZ4_API int32_t k4lz4_device_count(void);
/* Message of the last library-level failure on the calling thread ("" if none). */
K4LZ4_API const char *k4lz4_last_error(void);

/* ---- single block: mirrors of the reference's pointer overloads ------------------------ */

/* LZ4Codec.MaximumOutputSize(int) -- LZ4Codec.cs:30-31, Engine/LL.tools.cs:38-40. */
K4LZ4_API int32_t k4lz4_max_output_size(int32_t length);

/* LZ4Codec.Encode(byte*,int,byte*,int,LZ4Level) -- LZ4Codec.cs:40-52; replaces the call to
 * LLxx.LZ4_compress_fast (Engine/LLxx.cs:65-75).  Host pointers.  level < 3 is encoded as
 * L00_FAST (acceleration 1); level >= 3 returns K4LZ4_R_DELEGATE. */
K4LZ4_API int32_t k4lz4_encode(const uint8_t *src, int32_t srcLen,
                               uint8_t *dst, int32_t dstCap, int32_t level);

/* LZ4Codec.Decode(byte*,int,byte*,int) -- LZ4Codec.cs:104-115; replaces the call to
 * LLxx.LZ4_decompress_safe (Engine/LLxx.cs:17-26).  Host pointers. */
K4LZ4_API int32_t k4lz4_decode(const uint8_t *src, int32_t srcLen,
                               uint8_t *dst, int32_t dstCap);

/* ---- batches of independent blocks (the fast path) ------------------------------------- */

/*
 * Block i reads srcBase[srcOff[i] .. +srcLen[i]) and writes dstBase[dstOff[i] .. +dstCap[i]).
 * outLen[i] receives exactly what k4lz4_encode / k4lz4_decode would return for block i with
 * the same dstCap[i].  Function result: K4LZ4_OK or K4LZ4_E_*.
 *
 * memKind == K4LZ4_MEM_DEVICE: all seven pointers live on `device`; work is enqueued on
 *   `cudaStream` (a cudaStream_t; NULL = default stream) and the call returns without
 *   synchronising.
 * memKind == K4LZ4_MEM_HOST: pointers are host memory; `device` >= 0 runs on that GPU,
 *   `device` == K4LZ4_ALL_DEVICES splits the block list contiguously (balanced by bytes) over
 *   every visible GPU, one host thread + stream per GPU, no inter-GPU traffic.  Synchronous.
 */
#define K4LZ4_ALL_DEVICES  (-1)

K4LZ4_API int32_t k4lz4_encode_batch(const uint8_t *srcBase, const int64_t *srcOff, const int32_t *srcLen,
                                     uint8_t *dstBase, const int64_t *dstOff, const int32_t *dstCap,
                                     int32_t *outLen, int32_t nBlocks, int32_t level,
                                     int32_t memKind, void *cudaStream, int32_t device);

/* The same two calls with the reference's global LL.Enforce32 switch set (Engine/LL.tools.cs:29-36,
 * LZ4Codec.cs:21-25): the 32-bit engine LL32.  Its output differs from LL64's only for inputs of
 * >= 65 547 bytes (4 096-entry u32 table with hash4 instead of hash5, LL64.tools.cs:135-143 vs
 * LL32); below that both engines emit identical bytes and these calls equal the plain ones. */
K4LZ4_API int32_t k4lz4_encode_x32(const uint8_t *src, int32_t srcLen, uint8_t *dst, int32_t dstCap, int32_t level);
K4LZ4_API int32_t k4lz4_encode_batch_x32(const uint8_t *srcBase, const int64_t *srcOff, const int32_t *srcLen,
                                         uint8_t *dstBase, const int64_t *dstOff, const int32_t *dstCap,
                                         int32_t *outLen, int32_t nBlocks, int32_t level,
                                         int32_t memKind, void *cudaStream, int32_t device);

K4LZ4_API int32_t k4lz4_decode_batch(const uint8_t *srcBase, const int64_t *srcOff, const int32_t *srcLen,
                                     uint8_t *dstBase, const int64_t *dstOff, const int32_t *dstCap,
                                     int32_t *outLen, int32_t nBlocks,
                                     int32_t memKind, void *cudaStream, int32_t device);

/* ---- decode with an external dictionary, partial decode (SURVEY 8f rows 3 and 4) ------------ */

/* LZ4Codec.Decode(byte*,int,byte*,int,byte*,int) -- LZ4Codec.cs:144-157; replaces the call to
 * LLxx.LZ4_decompress_safe_usingDict (Engine/LLxx.cs:42-52, Engine/x64/LL64.dec.cs:523-546).
 * Matches may reach back into `dict` (the bytes logically preceding the block).  Host pointers. */
K4LZ4_API int32_t k4lz4_decode_dict(const uint8_t *src, int32_t srcLen, uint8_t *dst, int32_t dstCap,
                                    const uint8_t *dict, int32_t dictLen);

/* LZ4Codec.PartialDecode(byte*,int,byte*,int) -- LZ4Codec.cs:123-134; replaces the call to
 * LLxx.LZ4_decompress_safe_partial (Engine/LLxx.cs:29-39): decoding stops at targetLen bytes. */
K4LZ4_API int32_t k4lz4_partial_decode(const uint8_t *src, int32_t srcLen, uint8_t *dst, int32_t targetLen);

/* Batched forms; block i uses dictBase[dictOff[i] .. +dictLen[i]) (dictBase may be NULL: no
 * dictionaries).  Same memKind / stream / device conventions as k4lz4_decode_batch, except that
 * memKind == K4LZ4_MEM_HOST runs on one GPU (`device`, K4LZ4_ALL_DEVICES = GPU 0).  These are the
 * exact warp-per-block engine (decode_generic.cuh), not the tile kernel. */
K4LZ4_API int32_t k4lz4_decode_dict_batch(const uint8_t *srcBase, const int64_t *srcOff, const int32_t *srcLen,
                                          uint8_t *dstBase, const int64_t *dstOff, const int32_t *dstCap,
                                          const uint8_t *dictBase, const int64_t *dictOff, const int32_t *dictLen,
                                          int32_t *outLen, int32_t nBlocks,
                                          int32_t memKind, void *cudaStream, int32_t device);
K4LZ4_API int32_t k4lz4_partial_decode_batch(const uint8_t *srcBase, const int64_t *srcOff, const int32_t *srcLen,
                                             uint8_t *dstBase, const int64_t *dstOff, const int32_t *targetLen,
                                             int32_t *outLen, int32_t nBlocks,
                                             int32_t memKind, void *cudaStream, int32_t device);

/* ---- XXH32: the checksum of the LZ4 Frame container (SURVEY 8f row 2) ------------------------ */

/* XXH32 of one buffer on the host (frame header byte, serial content checksum) --
 * Streams/Frames/LZ4FrameWriter.cs:100,162-181 via K4os.Hash.xxHash; orig/lib/xxhash.c. */
K4LZ4_API uint32_t k4lz4_xxh32(const uint8_t *data, int64_t length, uint32_t seed);
/* XXH32 of every block of a batch on the GPU (per-block checksums, LZ4FrameWriter.cs:169-175):
 * out[i] = XXH32(base[off[i] .. +len[i]), seed). */
K4LZ4_API int32_t k4lz4_xxh32_batch(const uint8_t *base, const int64_t *off, const int32_t *len, uint32_t seed,
                                    uint32_t *out, int32_t nBlocks,
                                    int32_t memKind, void *cudaStream, int32_t device);

/* ---- LZ4Pickler, byte[] variant, batched ----------------------------------------------- */

/* Upper bound of Pickle() output for an n-byte message: n + 1 (0 for n == 0). */
K4LZ4_API int32_t k4lz4_pickle_bound(int32_t length);

/* LZ4Pickler.Pickle(ReadOnlySpan<byte>, LZ4Level) -- LZ4Pickler.pickle.cs:51-106.
 * Message i -> dstBase[dstOff[i] ..), which must hold k4lz4_pickle_bound(srcLen[i]) bytes;
 * outLen[i] = pickle length (0 for an empty message).  The scratch-capacity rule of the
 * reference (1024 if n <= 1024 else n, pickle.cs:57-67) is applied internally. */
K4LZ4_API int32_t k4lz4_pickle_batch(const uint8_t *srcBase, const int64_t *srcOff, const int32_t *srcLen,
                                     uint8_t *dstBase, const int64_t *dstOff,
                                     int32_t *outLen, int32_t nMessages, int32_t level,
                                     int32_t memKind, void *cudaStream, int32_t device);

/* LZ4Pickler.Pickle<TBufferWriter>(ReadOnlySpan<byte>, writer, level) -- LZ4Pickler.pickle.cs:113-148.
 * Different bytes than the byte[] variant: the header width is chosen from the full length before
 * encoding (:129,161-165) and the payload is encoded with capacity n (:130-133).  Message i ->
 * dstBase[dstOff[i] ..), which must hold k4lz4_pickle_writer_bound(srcLen[i]) bytes (what the
 * reference asks its writer for); outLen[i] = bytes the reference would Advance() the writer by. */
K4LZ4_API int32_t k4lz4_pickle_writer_bound(int32_t length);
K4LZ4_API int32_t k4lz4_pickle_writer_batch(const uint8_t *srcBase, const int64_t *srcOff, const int32_t *srcLen,
                                            uint8_t *dstBase, const int64_t *dstOff,
                                            int32_t *outLen, int32_t nMessages, int32_t level,
                                            int32_t memKind, void *cudaStream, int32_t device);

/* LZ4Pickler.UnpickledSize(ReadOnlySpan<byte>) -- LZ4Pickler.unpickle.cs:83-92,131-148.
 * outSize[i] = unpickled size, or K4LZ4_R_CORRUPT where the reference throws. */
K4LZ4_API int32_t k4lz4_unpickled_size_batch(const uint8_t *srcBase, const int64_t *srcOff,
                                             const int32_t *srcLen, int32_t *outSize,
                                             int32_t nMessages,
                                             int32_t memKind, void *cudaStream, int32_t device);

/* LZ4Pickler.Unpickle(ReadOnlySpan<byte>, Span<byte>) -- LZ4Pickler.unpickle.cs:99-129.
 * dstLen[i] must equal the unpickled size (else K4LZ4_R_CORRUPT, unpickle.cs:115-117);
 * outLen[i] = bytes produced or K4LZ4_R_CORRUPT. */
K4LZ4_API int32_t k4lz4_unpickle_batch(const uint8_t *srcBase, const int64_t *srcOff, const int32_t *srcLen,
                                       uint8_t *dstBase, const int64_t *dstOff, const int32_t *dstLen,
                                       int32_t *outLen, int32_t nMessages,
                                       int32_t memKind, void *cudaStream, int32_t device);

/* ---- synthetic workload generator (bench / tests; not part of the reference surface) ---- */

/*
 * Fills nBlocks blocks of blockSize bytes (block i at base + i*blockSize) with LZ-friendly
 * synthetic data: each block independently, a seeded mix of skewed-alphabet literal runs and
 * back-references within the block.  matchPermille steers compressibility (0 = noise only).
 * The host and device variants produce identical bytes for identical arguments.
 */
K4LZ4_API int32_t k4lz4_synth_host(uint8_t *base, int64_t nBlocks, int32_t blockSize,
                                   int32_t matchPermille, uint64_t seed, int64_t firstBlock);
K4LZ4_API int32_t k4lz4_synth_device(uint8_t *base, int64_t nBlocks, int32_t blockSize,
                                     int32_t matchPermille, uint64_t seed, int64_t firstBlock,
                                     void *cudaStream, int32_t device);

/*
 * Batched variable-length copy on the device: block i moves len[i] bytes from
 * srcBase[srcOff[i]..) to dstBase[dstOff[i]..)  (len[i] <= 0 copies nothing).  Used to pack the
 * padded output slots of an encode batch into a dense stream (and by the host path before
 * its single D2H).  Device pointers only; enqueues on `cudaStream`.
 */
K4LZ4_API int32_t k4lz4_copy_blocks_device(const uint8_t *srcBase, const int64_t *srcOff,
                                           uint8_t *dstBase, const int64_t *dstOff,
                                           const int32_t *len, int32_t nBlocks,
                                           void *cudaStream, int32_t device);

/* Counters for bench.py: number of kernels this library has launched since load. */
K4LZ4_API int64_t k4lz4_launch_count(void);

/* Decoder path counters of `device` since the last reset: out4[0] blocks decoded by the
 * shared-memory tile kernel (two CTAs per SM), [1] by its big-stage variant, [2] by the exact
 * warp-per-block decoder (malformed / oversized / unusual blocks), [3] parse repair walks.
 * Synchronises the device.  Diagnostics only (tests assert that clean data stays on the tile path). */
K4LZ4_API int32_t k4lz4_decode_stats(int32_t device, uint64_t *out4, int32_t reset);

/* Encoder path counters of `device` since the last reset, blocks of n > 0 the batched encoder ran:
 * out3[0] encoded by the shared-memory-table warps, [1] by the global-table warps (both below
 * 65 547 bytes), [2] by the u32-table engine (65 547 bytes and more, either warp kind).
 * Synchronises the device.  Diagnostics only. */
K4LZ4_API int32_t k4lz4_encode_stats(int32_t device, uint64_t *out3, int32_t reset);

#ifdef __cplusplus
}
#endif
#endif /* K4LZ4_H */
