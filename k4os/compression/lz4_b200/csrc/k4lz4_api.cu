// k4lz4_api.cu -- the C ABI of libk4lz4 (include/k4lz4.h): argument handling, the
// device-resident launch path, the host-buffer staging path (chunked, double-buffered,
// NCCL-free multi-GPU split of the block list) and the synthetic workload generator.
//
// There is deliberately NO CPU codec in this library: without a usable CUDA device every
// compute entry point fails with K4LZ4_E_NODEVICE.
#include "../../../../include/k4lz4.h"

#include <cuda_runtime.h>
#if defined(__linux__)
#include <sched.h>
#endif

#include <algorithm>
#include <cctype>
#include <cstdlib>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "decode_generic.cuh"
#include "decode_tile.cuh"
#include "encode_generic.cuh"
#include "encode_tile.cuh"
#include "pickle.cuh"
#include "synth.cuh"
#include "copy_blocks.cuh"
#include "xxh32.cuh"

namespace {

std::atomic<int64_t> g_launches{0};
thread_local std::string t_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    t_err = buf;
    return code;
}

#define CU_TRY(expr)                                                                         \
    do {                                                                                     \
        cudaError_t e__ = (expr);                                                            \
        if (e__ != cudaSuccess)                                                              \
            return fail(K4LZ4_E_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__));      \
    } while (0)

int device_count_cached() {
    static int n = [] {
        int c = 0;
        cudaError_t e = cudaGetDeviceCount(&c);
        if (e != cudaSuccess) { (void)cudaGetLastError(); return 0; }
        return c;
    }();
    return n;
}

// ---- kernel launchers (device pointers) ---------------------------------------------------

enum Op { OP_ENCODE = 0, OP_DECODE = 1, OP_PICKLE = 2, OP_UNPICKLE = 3, OP_USIZE = 4, OP_PICKLEW = 5 };

std::once_flag g_attr_once[64];

void set_func_attrs(int dev) {
    if (dev < 0 || dev >= 64) return;
    std::call_once(g_attr_once[dev], [] {
        cudaFuncSetAttribute(k4::pickle_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             k4::ENC_WARPS_PER_CTA * k4::ENC_SLOT_BYTES);
        // both encoder kernels ask for the same shared-memory / L1 split (they share SMs): just enough for the
        // shared-memory tables (+1 KiB the hardware reserves per CTA), the rest stays L1 for the input windows
        const int carve = (k4::ENC_SM_WARPS * (k4::ENC_SLOT_BYTES + 1024) * 100 + 228 * 1024 - 1) / (228 * 1024);
        cudaFuncSetAttribute(k4::encode_spec_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve > 100 ? 100 : carve);
        cudaFuncSetAttribute(k4::encode_spec_gtab_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve > 100 ? 100 : carve);
    });
}

// Enqueues the block encoder: a shared-memory-table kernel on `st` and, when the batch is big enough for
// it to pay, a global-memory-table kernel on a helper stream that runs beside it (fork / join by events).
// Both are persistent and pull blocks from one device counter.  The workspace (counter + the global
// tables) comes from the private stream-ordered pool.
cudaError_t encode_launch(const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen,
                          uint8_t* dstBase, const int64_t* dstOff, const int32_t* dstCap,
                          int32_t* outLen, int n, int level, cudaStream_t st, int* launches) {
    int dev = 0;
    cudaGetDevice(&dev);
    k4::DecodeDev* D = k4::decode_dev(dev);
    if (!D || D->err != cudaSuccess) return D ? D->err : cudaErrorInvalidDevice;
    const int wave = D->sms * k4::ENC_SM_WARPS;
    const int gridS = n < wave ? n : wave;
    // The global-table warps need longer per block than the shared-memory warps: a batch that the latter
    // finish in one round goes to them alone.
    const bool useG = k4::ENC_GM_WARPS > 0 && n > wave;
    const int gridG = useG ? D->sms * k4::ENC_GM_WARPS : 0;
    const size_t tabBytes = (size_t)gridG * k4::ENC_GSLOT_BYTES;
    uint8_t* ws = nullptr;
    cudaError_t e = cudaMallocFromPoolAsync((void**)&ws, 256 + tabBytes, D->pool, st);
    if (e != cudaSuccess) return e;
    uint32_t* counter = reinterpret_cast<uint32_t*>(ws);
    e = cudaMemsetAsync(ws, 0, 4, st);
    cudaEvent_t fork = nullptr, join = nullptr;
    if (e == cudaSuccess && useG) {
        // ONE side stream per device: the global-table kernels of consecutive chunks run one after the other, so an
        // SM never holds more than ENC_GM_WARPS of them (CTAs of a queued launch would otherwise fill the SM's spare
        // CTA slots and crowd out the mix; measured slower)
        cudaStream_t hs = D->helper;
        e = cudaEventCreateWithFlags(&fork, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&join, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventRecord(fork, st);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(hs, fork, 0);
        if (e == cudaSuccess) {
            k4::encode_spec_gtab_kernel<<<gridG, 32, 0, hs>>>(srcBase, srcOff, srcLen, dstBase, dstOff, dstCap, outLen,
                                                             n, level, counter, ws + 256, wave);
            e = cudaGetLastError();
            if (launches) (*launches)++;
        }
        if (e == cudaSuccess) e = cudaEventRecord(join, hs);
    }
    if (e == cudaSuccess && gridS > 0) {
        k4::encode_spec_kernel<<<gridS, 32, k4::ENC_SLOT_BYTES, st>>>(srcBase, srcOff, srcLen, dstBase, dstOff, dstCap,
                                                                      outLen, n, level, counter);
        e = cudaGetLastError();
        if (launches) (*launches)++;
    }
    if (join && e == cudaSuccess) e = cudaStreamWaitEvent(st, join, 0);
    if (fork) cudaEventDestroy(fork);
    if (join) cudaEventDestroy(join);
    cudaFreeAsync(ws, st);
    return e;
}

struct DevArgs {
    const uint8_t* srcBase; const int64_t* srcOff; const int32_t* srcLen;
    uint8_t* dstBase; const int64_t* dstOff; const int32_t* dstCap;
    int32_t* outLen; int n; int level;
};

cudaError_t launch_op(Op op, const DevArgs& a, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    int dev = 0;
    cudaGetDevice(&dev);
    set_func_attrs(dev);
    switch (op) {
    case OP_ENCODE: {
        int nl = 0;
        const cudaError_t ee = encode_launch(a.srcBase, a.srcOff, a.srcLen, a.dstBase, a.dstOff, a.dstCap,
                                             a.outLen, a.n, a.level, st, &nl);
        g_launches += nl;
        if (ee != cudaSuccess) { (void)cudaGetLastError(); return ee; }
        break;
    }
    case OP_DECODE: {
        cudaError_t de = cudaSuccess;
        const int nl = k4::decode_launch(a.srcBase, a.srcOff, a.srcLen, a.dstBase, a.dstOff,
                                         a.dstCap, a.outLen, a.n, st, &de);
        if (nl < 0) { (void)cudaGetLastError(); return de != cudaSuccess ? de : cudaErrorUnknown; }
        g_launches += nl;
        break;
    }
    case OP_PICKLE:
    case OP_PICKLEW: {
        const int ctas = (a.n + k4::ENC_WARPS_PER_CTA - 1) / k4::ENC_WARPS_PER_CTA;
        k4::pickle_kernel<<<ctas, k4::ENC_WARPS_PER_CTA * 32,
                            k4::ENC_WARPS_PER_CTA * k4::ENC_SLOT_BYTES, st>>>(
            a.srcBase, a.srcOff, a.srcLen, a.dstBase, a.dstOff, a.outLen, a.n, a.level, op == OP_PICKLEW ? 1 : 0);
        g_launches++;
        break;
    }
    case OP_UNPICKLE: {
        const int ctas = (a.n + 3) / 4;
        k4::unpickle_kernel<<<ctas, 128, 0, st>>>(a.srcBase, a.srcOff, a.srcLen, a.dstBase, a.dstOff,
                                                  a.dstCap, a.outLen, a.n);
        g_launches++;
        break;
    }
    case OP_USIZE: {
        const int ctas = (a.n + 255) / 256;
        k4::unpickled_size_kernel<<<ctas, 256, 0, st>>>(a.srcBase, a.srcOff, a.srcLen, a.outLen, a.n);
        g_launches++;
        break;
    }
    }
    return cudaGetLastError();
}

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (dev >= 0) {
            cudaGetDevice(&prev);
            if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess; else prev = -1;
        }
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int run_device(Op op, const DevArgs& a, void* stream, int device) {
    if (device_count_cached() <= 0) return fail(K4LZ4_E_NODEVICE, "no CUDA device available");
    if (a.n < 0) return fail(K4LZ4_E_ARG, "negative block count");
    if (a.n == 0) return K4LZ4_OK;
    if (!a.srcBase || !a.srcOff || !a.srcLen || !a.outLen) return fail(K4LZ4_E_ARG, "null pointer argument");
    if (op != OP_USIZE && (!a.dstBase || !a.dstOff)) return fail(K4LZ4_E_ARG, "null pointer argument");
    if ((op == OP_ENCODE || op == OP_DECODE || op == OP_UNPICKLE) && !a.dstCap)
        return fail(K4LZ4_E_ARG, "null pointer argument");
    DeviceGuard g(device);
    if (!g.ok) return fail(K4LZ4_E_CUDA, "cudaSetDevice(%d) failed", device);
    CU_TRY(launch_op(op, a, (cudaStream_t)stream));
    return K4LZ4_OK;
}

// ---- host-buffer path ----------------------------------------------------------------------

struct DBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 4 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { e = cudaMalloc(&p, n); want = n; }
        if (e == cudaSuccess) cap = want; else p = nullptr;
        return e;
    }
};
struct HBuf {   // pinned host
    void* p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 4 + 4096;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e != cudaSuccess) { e = cudaHostAlloc(&p, n, cudaHostAllocDefault); want = n; }
        if (e == cudaSuccess) cap = want; else p = nullptr;
        return e;
    }
};

struct Slot {          // one in-flight chunk
    cudaStream_t stream = nullptr;
    DBuf dSrc, dDst, dMeta, dPack, dPackOff;
    HBuf hSrc, hDst, hMeta, hPackOff;
    const int64_t* dDstOffArr = nullptr;   // device copies of the chunk's dst offsets / results (inside dMeta)
    const int32_t* dOutLenArr = nullptr;
    bool compact = false;             // stage 2 gathered the produced bytes on the device first
    std::vector<int64_t> compactOff;  // ... and this is where block k starts in the staging buffer
    // description of the chunk that is in flight
    int64_t b0 = 0, b1 = 0;           // block range
    int64_t dLo = 0;                  // dst extent origin (direct mode) or 0 (packed mode)
    bool dstPacked = false;
    std::vector<int64_t> packedDstOff;
    int64_t dstBytes = 0;             // device-side extent of the destination region of the chunk
    bool direct = false;              // stage 2 copied straight into the caller's buffer
    int state = 0;                    // 0 idle, 3 inputs on their way, 1 kernel + outLen enqueued, 2 data D2H enqueued
    DevArgs launch{};                 // the chunk's kernel arguments (state 3 -> 1)
};

constexpr int ENC_BIG_WAVES = 6;        // encode chunks in the middle of a batch: this many waves of blocks
constexpr int NSLOT = 4;                // chunks in flight per device (see run_host_slice)

struct DevCtx {
    int dev = -1;
    std::mutex mu;
    Slot slot[NSLOT];
    bool init = false;
};

DevCtx* get_ctx(int dev) {
    static std::mutex m;
    static std::vector<std::unique_ptr<DevCtx>> ctxs;
    std::lock_guard<std::mutex> lk(m);
    if ((int)ctxs.size() <= dev) ctxs.resize(dev + 1);
    if (!ctxs[dev]) { ctxs[dev].reset(new DevCtx()); ctxs[dev]->dev = dev; }
    return ctxs[dev].get();
}

struct HostArgs {
    const uint8_t* srcBase; const int64_t* srcOff; const int32_t* srcLen;
    uint8_t* dstBase; const int64_t* dstOff; const int32_t* dstCap;
    int32_t* outLen; int level;
};

inline int64_t dst_room(Op op, const HostArgs& a, int64_t i) {
    switch (op) {
    case OP_PICKLE: return a.srcLen[i] <= 0 ? 0 : (int64_t)a.srcLen[i] + 1;
    case OP_PICKLEW: return a.srcLen[i] <= 0 ? 0 : (int64_t)a.srcLen[i] + 1 + k4::pickle_diff_width(a.srcLen[i]);
    case OP_USIZE: return 0;
    case OP_ENCODE: {      // a capacity beyond compressBound(srcLen) behaves like compressBound (notLimited)
        const int64_t cap = a.dstCap[i] < 0 ? 0 : a.dstCap[i];
        const int64_t bound = a.srcLen[i] > 0 ? k4::max_output_size(a.srcLen[i]) : 0;
        return cap < bound ? cap : bound;
    }
    default: return a.dstCap[i] < 0 ? 0 : a.dstCap[i];
    }
}
inline int64_t src_size(const HostArgs& a, int64_t i) { return a.srcLen[i] < 0 ? 0 : a.srcLen[i]; }

void parallel_for_blocks(int64_t b0, int64_t b1, int64_t bytesHint, const std::function<void(int64_t, int64_t)>& fn);
int launch_chunk(Op op, Slot& s);

constexpr int64_t CHUNK_BYTES = 192ll << 20;   // src + dst payload per in-flight chunk

// Copies every produced byte of chunk [b0,b1) from the pinned staging buffer into the
// caller's destination; bytes at index >= outLen[i] are never touched.
void scatter_chunk(Op op, const HostArgs& a, Slot& s) {
    if (op == OP_USIZE) return;
    const uint8_t* stage = (const uint8_t*)s.hDst.p;
    int64_t total = 0;
    for (int64_t i = s.b0; i < s.b1; i++) total += std::max<int32_t>(a.outLen[i], 0);
    parallel_for_blocks(s.b0, s.b1, total, [&](int64_t lo, int64_t hi) {
        for (int64_t i = lo; i < hi; i++) {
            const int32_t r = a.outLen[i];
            if (r <= 0) continue;
            const int64_t off = s.compact ? s.compactOff[i - s.b0]
                                : (s.dstPacked ? s.packedDstOff[i - s.b0] : a.dstOff[i] - s.dLo);
            memcpy(a.dstBase + a.dstOff[i], stage + off, (size_t)r);
        }
    });
}

// stage 2: the kernel of the chunk has finished -> per-block results to the caller, then the
// data D2H.  When every block filled its whole slot and the slots are contiguous (the decode
// case) the bytes go straight into the caller's buffer in one copy; otherwise through the pinned
// staging buffer and a host-side scatter (stage 3) that leaves bytes >= outLen[i] untouched.
int stage2_slot(Op op, const HostArgs& a, Slot& s) {
    if (s.state == 3) { int rc = launch_chunk(op, s); if (rc != K4LZ4_OK) return rc; }
    if (s.state != 1) return K4LZ4_OK;
    CU_TRY(cudaStreamSynchronize(s.stream));
    memcpy(a.outLen + s.b0, (const int32_t*)s.hMeta.p, sizeof(int32_t) * (size_t)(s.b1 - s.b0));
    s.state = 2;
    s.direct = false;
    s.compact = false;
    if (op == OP_USIZE || s.dstBytes <= 0) return K4LZ4_OK;
    bool full = !s.dstPacked;
    int64_t sum = 0;
    for (int64_t i = s.b0; i < s.b1 && full; i++) {
        const int64_t room = dst_room(op, a, i);
        full = (int64_t)a.outLen[i] == room;
        sum += room;
    }
    full = full && sum == s.dstBytes;                 // slots tile the extent exactly: no gaps
    if (full) {
        s.direct = true;
        CU_TRY(cudaMemcpyAsync(a.dstBase + s.dLo, s.dDst.p, (size_t)s.dstBytes, cudaMemcpyDeviceToHost, s.stream));
    } else {
        // variable-length results (encode, pickle, short decodes): gather the produced bytes on the
        // device (copy_blocks_kernel) so that only they cross PCIe, not the slots' slack
        const int64_t nb = s.b1 - s.b0;
        s.compactOff.resize((size_t)nb);
        int64_t total = 0;
        for (int64_t k = 0; k < nb; k++) {
            s.compactOff[(size_t)k] = total;
            const int32_t r = a.outLen[s.b0 + k];
            if (r > 0) total += ((int64_t)r + 15) & ~int64_t(15);
        }
        s.compact = true;
        s.dstBytes = total;
        if (total == 0) return K4LZ4_OK;
        CU_TRY(s.hPackOff.ensure((size_t)nb * 8));
        CU_TRY(s.dPackOff.ensure((size_t)nb * 8));
        CU_TRY(s.dPack.ensure((size_t)total + 16));
        CU_TRY(s.hDst.ensure((size_t)total + 16));
        memcpy(s.hPackOff.p, s.compactOff.data(), (size_t)nb * 8);
        CU_TRY(cudaMemcpyAsync(s.dPackOff.p, s.hPackOff.p, (size_t)nb * 8, cudaMemcpyHostToDevice, s.stream));
        k4::copy_blocks_kernel<<<(unsigned)nb, 256, 0, s.stream>>>(
            (const uint8_t*)s.dDst.p, s.dDstOffArr, (uint8_t*)s.dPack.p, (const int64_t*)s.dPackOff.p,
            s.dOutLenArr, (int)nb);
        g_launches++;
        CU_TRY(cudaGetLastError());
        CU_TRY(cudaMemcpyAsync(s.hDst.p, s.dPack.p, (size_t)total, cudaMemcpyDeviceToHost, s.stream));
    }
    return K4LZ4_OK;
}

// stage 3: data has landed
int stage3_slot(Op op, const HostArgs& a, Slot& s) {
    if (s.state == 1 || s.state == 3) { int rc = stage2_slot(op, a, s); if (rc != K4LZ4_OK) return rc; }
    if (s.state != 2) return K4LZ4_OK;
    s.state = 0;
    CU_TRY(cudaStreamSynchronize(s.stream));
    if (!s.direct) scatter_chunk(op, a, s);
    return K4LZ4_OK;
}

// stage 1a: stage the chunk's inputs and block table on the device (asynchronous copies on the slot's stream)
int enqueue_chunk(Op op, const HostArgs& a, Slot& s, int64_t b0, int64_t b1) {
    const int64_t nb = b1 - b0;
    s.b0 = b0; s.b1 = b1;
    // extents
    int64_t sLo = INT64_MAX, sHi = INT64_MIN, dLo = INT64_MAX, dHi = INT64_MIN, sSum = 0, dSum = 0;
    for (int64_t i = b0; i < b1; i++) {
        const int64_t sl = src_size(a, i), dl = dst_room(op, a, i);
        if (sl > 0) { sLo = std::min(sLo, a.srcOff[i]); sHi = std::max(sHi, a.srcOff[i] + sl); sSum += sl; }
        if (dl > 0) { dLo = std::min(dLo, a.dstOff[i]); dHi = std::max(dHi, a.dstOff[i] + dl); dSum += dl; }
    }
    if (sSum == 0) { sLo = 0; sHi = 0; }
    if (dSum == 0) { dLo = 0; dHi = 0; }
    const bool srcPacked = (sHi - sLo) > sSum + sSum / 4 + 65536;
    const bool dstPacked = (dHi - dLo) > dSum + dSum / 4 + 65536;
    s.dstPacked = dstPacked;
    s.dLo = dLo;

    // meta layout (device): srcOff[nb] dstOff[nb] (int64) | srcLen[nb] dstCap[nb] outLen[nb] (int32)
    const size_t metaBytes = (size_t)nb * (8 + 8 + 4 + 4 + 4);
    CU_TRY(s.dMeta.ensure(metaBytes));
    CU_TRY(s.hMeta.ensure(metaBytes));
    int64_t* hSrcOff = (int64_t*)s.hMeta.p;
    int64_t* hDstOff = hSrcOff + nb;
    int32_t* hSrcLen = (int32_t*)(hDstOff + nb);
    int32_t* hDstCap = hSrcLen + nb;
    // (outLen comes back into the front of hMeta after the kernel; see below)
    int64_t* dSrcOff = (int64_t*)s.dMeta.p;
    int64_t* dDstOff = dSrcOff + nb;
    int32_t* dSrcLen = (int32_t*)(dDstOff + nb);
    int32_t* dDstCap = dSrcLen + nb;
    int32_t* dOutLen = dDstCap + nb;

    const int64_t srcBytes = srcPacked ? sSum : (sHi - sLo);
    const int64_t dstBytes = dstPacked ? dSum : (dHi - dLo);
    CU_TRY(s.dSrc.ensure((size_t)srcBytes + 16));
    if (op != OP_USIZE) CU_TRY(s.dDst.ensure((size_t)dstBytes + 16));
    s.dstBytes = (op == OP_USIZE) ? 0 : dstBytes;
    if (dstPacked) s.packedDstOff.resize((size_t)nb);

    int64_t sp = 0, dp = 0;
    if (srcPacked) CU_TRY(s.hSrc.ensure((size_t)sSum + 16));
    for (int64_t i = b0; i < b1; i++) {
        const int64_t k = i - b0;
        const int64_t sl = src_size(a, i), dl = dst_room(op, a, i);
        hSrcLen[k] = a.srcLen[i];
        hDstCap[k] = (op == OP_PICKLE || op == OP_PICKLEW || op == OP_USIZE) ? 0 : (op == OP_ENCODE ? (int32_t)dl : a.dstCap[i]);
        if (srcPacked) {
            hSrcOff[k] = sp;
            if (sl > 0) memcpy((uint8_t*)s.hSrc.p + sp, a.srcBase + a.srcOff[i], (size_t)sl);
            sp += sl;
        } else {
            hSrcOff[k] = sl > 0 ? a.srcOff[i] - sLo : 0;
        }
        if (dstPacked) { hDstOff[k] = dp; s.packedDstOff[(size_t)k] = dp; dp += dl; }
        else hDstOff[k] = dl > 0 ? a.dstOff[i] - dLo : 0;
    }

    cudaStream_t st = s.stream;
    if (srcBytes > 0)
        CU_TRY(cudaMemcpyAsync(s.dSrc.p, srcPacked ? (const void*)s.hSrc.p : (const void*)(a.srcBase + sLo),
                               (size_t)srcBytes, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(s.dMeta.p, s.hMeta.p, (size_t)nb * 24, cudaMemcpyHostToDevice, st));
    s.launch = DevArgs{(const uint8_t*)s.dSrc.p, dSrcOff, dSrcLen, (uint8_t*)s.dDst.p, dDstOff, dDstCap,
                       dOutLen, (int)nb, a.level};
    s.dDstOffArr = dDstOff;
    s.dOutLenArr = dOutLen;
    s.state = 3;
    return K4LZ4_OK;
}

// stage 1b: the kernel of a chunk whose inputs are on their way (same stream), then its per-block results
int launch_chunk(Op op, Slot& s) {
    if (s.state != 3) return K4LZ4_OK;
    CU_TRY(launch_op(op, s.launch, s.stream));
    // outLen lands at the front of hMeta (offset arrays there are no longer needed once the
    // H2D of the chunk has been issued *and completed*; stream order guarantees that)
    CU_TRY(cudaMemcpyAsync(s.hMeta.p, s.launch.outLen, (size_t)s.launch.n * 4, cudaMemcpyDeviceToHost, s.stream));
    s.state = 1;
    return K4LZ4_OK;
}

// blocks the encoder finishes in about one shared-memory-warp block time on `dev` (a global-table warp counts half)
int64_t enc_wave_blocks(int dev) {
    static int sms[64] = {0};
    if (dev < 0 || dev >= 64) return 1;
    if (!sms[dev]) { int v = 0; if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) v = 0; sms[dev] = v > 0 ? v : -1; }
    return sms[dev] > 0 ? (int64_t)sms[dev] * (k4::ENC_SM_WARPS + (k4::ENC_GM_WARPS + 1) / 2) : 1;
}

// One device, blocks [b0, b1): chunked + double-buffered (H2D/kernel/D2H of chunk c overlap
// the host-side scatter of chunk c-1 and the copies of chunk c+1 on the other stream).
int run_host_slice(Op op, const HostArgs& a, int64_t b0, int64_t b1, int dev) {
    if (b1 <= b0) return K4LZ4_OK;
    DevCtx* ctx = get_ctx(dev);
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard g(dev);
    if (!g.ok) return fail(K4LZ4_E_CUDA, "cudaSetDevice(%d) failed", dev);
    if (!ctx->init) {
        for (auto& s : ctx->slot) CU_TRY(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        ctx->init = true;
    }
    int rc = K4LZ4_OK;
    // Chunk boundaries.  Encode: a warp works on one block for milliseconds; consecutive chunks' kernels
    // overlap (one-warp CTAs leave individually and the next launch, on another stream, moves in), so a
    // chunk only has to be long enough to hide its copies and the host's work behind the previous kernel:
    // ENC_BIG_WAVES waves in the middle of a batch, one and two waves at both ends so that the pipeline
    // fills and drains fast.
    auto chunk_end = [&](int64_t i, int c) {
        int64_t bytes = 0, j = i;
        int64_t limit = CHUNK_BYTES, maxBlocks = INT64_MAX;
        if (op == OP_ENCODE) {
            const int64_t W = enc_wave_blocks(dev), rem = b1 - i;
            limit = 2560ll << 20;
            if (c == 0) maxBlocks = W;
            else if (c == 1) maxBlocks = 2 * W;
            else if (2 * rem <= 3 * W) maxBlocks = rem;
            else if (2 * rem <= 7 * W) maxBlocks = std::min<int64_t>(2 * W, rem - W);
            else maxBlocks = std::max<int64_t>(std::min<int64_t>(ENC_BIG_WAVES * W, rem - 3 * W), W);
        } else if (op == OP_PICKLE || op == OP_PICKLEW) {
            limit = 4 * CHUNK_BYTES;
        }
        while (j < b1 && j - i < maxBlocks && (j == i || bytes + src_size(a, j) + dst_room(op, a, j) <= limit)) {
            bytes += src_size(a, j) + dst_room(op, a, j);
            j++;
        }
        return j;
    };
    // Four chunks in flight, copies issued two chunks ahead, kernels one:
    //   inputs(c+1) -> wait kernel(c-1), its results, gather + data D2H (stage 2) -> kernel(c+1) -> scatter(c-2)
    // so while kernel c runs, chunk c+1 is queued behind it with its inputs already on the device, the data
    // of chunk c-1 crosses PCIe and the host scatters chunk c-2: the GPU never waits for PCIe or for the host.
    // No more than two kernels are queued at any time (a third one would crowd the SMs with the CTAs of
    // three launches; measured slower).
    auto slot_of = [&](int c) -> Slot& { return ctx->slot[((c % NSLOT) + NSLOT) % NSLOT]; };
    int64_t next = b0;                                     // first block not yet staged
    int staged = 0;                                        // chunks whose inputs have been issued
    auto stage_next = [&]() -> int {
        if (next >= b1) return K4LZ4_OK;
        Slot& s = slot_of(staged);
        int r = stage3_slot(op, a, s);                     // chunk staged-4: long done
        if (r != K4LZ4_OK) return r;
        const int64_t j = chunk_end(next, staged);
        r = enqueue_chunk(op, a, s, next, j);
        next = j; staged++;
        return r;
    };
    rc = stage_next();
    if (rc == K4LZ4_OK) rc = launch_chunk(op, slot_of(0));
    for (int c = 0; rc == K4LZ4_OK && c < staged; c++) {
        if ((rc = stage_next()) != K4LZ4_OK) break;                                       // inputs of chunk c+1
        if (c >= 1 && (rc = stage2_slot(op, a, slot_of(c - 1))) != K4LZ4_OK) break;       // kernel c-1 done
        if (c + 1 < staged && (rc = launch_chunk(op, slot_of(c + 1))) != K4LZ4_OK) break; // kernel c+1 queued
        if (c >= 2 && (rc = stage3_slot(op, a, slot_of(c - 2))) != K4LZ4_OK) break;       // scatter c-2
    }
    if (rc != K4LZ4_OK) { for (auto& s : ctx->slot) s.state = 0; cudaDeviceSynchronize(); return rc; }
    // drain in issue order: results + data D2H of everything still on the device first, then the scatters
    for (int k = staged - NSLOT; k < staged && rc == K4LZ4_OK; k++) if (k >= 0) rc = stage2_slot(op, a, slot_of(k));
    for (int k = staged - NSLOT; k < staged && rc == K4LZ4_OK; k++) if (k >= 0) rc = stage3_slot(op, a, slot_of(k));
    if (rc != K4LZ4_OK) { for (auto& s : ctx->slot) s.state = 0; cudaDeviceSynchronize(); }
    return rc;
}

void parallel_for_blocks(int64_t b0, int64_t b1, int64_t bytesHint,
                         const std::function<void(int64_t, int64_t)>& fn) {
    unsigned hw = std::thread::hardware_concurrency();
    int T = (int)std::min<unsigned>(hw ? hw : 1, 16);
    if (bytesHint < (8 << 20) || b1 - b0 < 2 * T) T = 1;
    if (T <= 1) { fn(b0, b1); return; }
    std::vector<std::thread> th;
    for (int t = 0; t < T; t++) {
        int64_t lo = b0 + (b1 - b0) * t / T, hi = b0 + (b1 - b0) * (t + 1) / T;
        th.emplace_back([=, &fn] { fn(lo, hi); });
    }
    for (auto& t : th) t.join();
}

// Best effort: run the calling thread on the CPUs of the NUMA node GPU `dev` is attached to, so that
// the pinned staging buffers it allocates (first touch) and its memcpy traffic stay node-local.
// (HGX boards hang GPUs 0-3 and 4-7 off different sockets; staging through the far socket halves the
// aggregate PCIe rate of an all-devices call.)
void bind_thread_near_gpu(int dev) {
#if defined(__linux__)
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), dev) != cudaSuccess) { (void)cudaGetLastError(); return; }
    for (char* c = bus; *c; c++) *c = (char)tolower(*c);
    char path[128];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    if (!f) return;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    if (node < 0) return;
    snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f) return;
    char list[4096] = {0};
    const size_t got = fread(list, 1, sizeof(list) - 1, f);
    fclose(f);
    if (got == 0) return;
    cpu_set_t want, have;
    CPU_ZERO(&want);
    if (sched_getaffinity(0, sizeof(have), &have) != 0) return;
    int any = 0;
    for (char* p = list; *p;) {
        char* e;
        long lo = strtol(p, &e, 10), hi = lo;
        if (e == p) break;
        if (*e == '-') { p = e + 1; hi = strtol(p, &e, 10); }
        for (long c = lo; c <= hi && c < CPU_SETSIZE; c++) if (CPU_ISSET((int)c, &have)) { CPU_SET((int)c, &want); any = 1; }
        p = (*e == ',') ? e + 1 : e;
        if (*e != ',' ) break;
    }
    if (any) sched_setaffinity(0, sizeof(want), &want);
#else
    (void)dev;
#endif
}

int run_host(Op op, const HostArgs& a, int64_t n, int device) {
    const int ndev = device_count_cached();
    if (ndev <= 0) return fail(K4LZ4_E_NODEVICE, "no CUDA device available");
    if (n < 0) return fail(K4LZ4_E_ARG, "negative block count");
    if (n == 0) return K4LZ4_OK;
    if (!a.srcBase || !a.srcOff || !a.srcLen || !a.outLen) return fail(K4LZ4_E_ARG, "null pointer argument");
    if (op != OP_USIZE && (!a.dstBase || !a.dstOff)) return fail(K4LZ4_E_ARG, "null pointer argument");
    if ((op == OP_ENCODE || op == OP_DECODE || op == OP_UNPICKLE) && !a.dstCap)
        return fail(K4LZ4_E_ARG, "null pointer argument");
    if (device >= ndev) return fail(K4LZ4_E_ARG, "device %d out of range (%d visible)", device, ndev);
    if (device >= 0 || ndev == 1) return run_host_slice(op, a, 0, n, device >= 0 ? device : 0);

    // K4LZ4_ALL_DEVICES: contiguous split balanced by bytes, one host thread per GPU
    std::vector<int64_t> cut(ndev + 1, n);
    cut[0] = 0;
    int64_t total = 0;
    for (int64_t i = 0; i < n; i++) total += src_size(a, i) + dst_room(op, a, i) + 64;
    int64_t acc = 0; int g = 1;
    for (int64_t i = 0; i < n && g < ndev; i++) {
        acc += src_size(a, i) + dst_room(op, a, i) + 64;
        while (g < ndev && acc >= total * g / ndev) cut[g++] = i + 1;
    }
    std::vector<int> rcs(ndev, K4LZ4_OK);
    std::vector<std::string> errs(ndev);
    std::vector<std::thread> th;
    for (int d = 0; d < ndev; d++)
        th.emplace_back([&, d] {
            bind_thread_near_gpu(d);
            rcs[d] = run_host_slice(op, a, cut[d], cut[d + 1], d);
            if (rcs[d] != K4LZ4_OK) errs[d] = t_err;
        });
    for (auto& t : th) t.join();
    for (int d = 0; d < ndev; d++) if (rcs[d] != K4LZ4_OK) { t_err = errs[d]; return rcs[d]; }
    return K4LZ4_OK;
}

int run(Op op, const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen, uint8_t* dstBase,
        const int64_t* dstOff, const int32_t* dstCap, int32_t* outLen, int64_t n, int level,
        int memKind, void* stream, int device) {
    if (memKind == K4LZ4_MEM_DEVICE) {
        if (n > INT32_MAX) return fail(K4LZ4_E_ARG, "too many blocks");
        DevArgs d{srcBase, srcOff, srcLen, dstBase, dstOff, dstCap, outLen, (int)n, level};
        return run_device(op, d, stream, device);
    }
    if (memKind == K4LZ4_MEM_HOST) {
        HostArgs h{srcBase, srcOff, srcLen, dstBase, dstOff, dstCap, outLen, level};
        return run_host(op, h, n, device);
    }
    return fail(K4LZ4_E_ARG, "unknown memKind %d", memKind);
}

// ---- dictionary / partial decode (SURVEY 8f rows 3 and 4): exactness first, simple staging ------

struct GeneralArgs {
    const uint8_t* srcBase; const int64_t* srcOff; const int32_t* srcLen;
    uint8_t* dstBase; const int64_t* dstOff; const int32_t* dstCap;
    const uint8_t* dictBase; const int64_t* dictOff; const int32_t* dictLen;   // all three may be null
    int32_t* outLen; int64_t n; bool partial;
};

cudaError_t launch_general(const GeneralArgs& g, cudaStream_t st) {
    if (g.n <= 0) return cudaSuccess;
    const long long ctas = (g.n + 3) / 4;
    k4::decode_general_kernel<<<(unsigned)ctas, 128, 0, st>>>(g.srcBase, g.srcOff, g.srcLen, g.dstBase, g.dstOff,
                                                              g.dstCap, g.dictBase, g.dictOff, g.dictLen, g.outLen,
                                                              (int)g.n, g.partial ? 1 : 0);
    g_launches++;
    return cudaGetLastError();
}

struct DevMem {
    void* p = nullptr;
    ~DevMem() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t n) { return cudaMalloc(&p, n ? n : 1); }
};

// host pointers: pack the blocks of a chunk, one H2D per array, one kernel, one D2H, exact scatter
int run_general_host(const GeneralArgs& g, int device) {
    const int ndev = device_count_cached();
    if (ndev <= 0) return fail(K4LZ4_E_NODEVICE, "no CUDA device available");
    if (g.n < 0) return fail(K4LZ4_E_ARG, "negative block count");
    if (g.n == 0) return K4LZ4_OK;
    if (!g.srcBase || !g.srcOff || !g.srcLen || !g.dstBase || !g.dstOff || !g.dstCap || !g.outLen)
        return fail(K4LZ4_E_ARG, "null pointer argument");
    if (g.dictBase && (!g.dictOff || !g.dictLen)) return fail(K4LZ4_E_ARG, "null pointer argument");
    const int dev = device >= 0 ? device : 0;
    if (dev >= ndev) return fail(K4LZ4_E_ARG, "device %d out of range (%d visible)", dev, ndev);
    DeviceGuard guard(dev);
    if (!guard.ok) return fail(K4LZ4_E_CUDA, "cudaSetDevice(%d) failed", dev);
    const int64_t CH = 256ll << 20;
    int64_t i = 0;
    while (i < g.n) {
        int64_t j = i, bytes = 0;
        while (j < g.n) {
            const int64_t add = std::max<int64_t>(g.srcLen[j], 0) + std::max<int64_t>(g.dstCap[j], 0) +
                                (g.dictBase ? std::max<int64_t>(g.dictLen[j], 0) : 0);
            if (j > i && bytes + add > CH) break;
            bytes += add; j++;
        }
        const int64_t nb = j - i;
        std::vector<int64_t> so(nb), doff(nb), dio(nb);
        std::vector<int32_t> sl(nb), dc(nb), dl(nb), res(nb);
        int64_t sTot = 0, dTot = 0, diTot = 0;
        for (int64_t k = 0; k < nb; k++) {
            sl[k] = g.srcLen[i + k]; dc[k] = g.dstCap[i + k] < 0 ? 0 : g.dstCap[i + k];
            dl[k] = g.dictBase ? std::max<int32_t>(g.dictLen[i + k], 0) : 0;
            so[k] = sTot; doff[k] = dTot; dio[k] = diTot;
            sTot += std::max<int32_t>(sl[k], 0); dTot += dc[k]; diTot += dl[k];
        }
        std::vector<uint8_t> hs((size_t)sTot + 16), hd((size_t)diTot + 16), ho((size_t)dTot + 16);
        for (int64_t k = 0; k < nb; k++) {
            if (sl[k] > 0) memcpy(hs.data() + so[k], g.srcBase + g.srcOff[i + k], (size_t)sl[k]);
            if (dl[k] > 0) memcpy(hd.data() + dio[k], g.dictBase + g.dictOff[i + k], (size_t)dl[k]);
        }
        DevMem dS, dD, dO, dM;
        CU_TRY(dS.alloc((size_t)sTot + 16)); CU_TRY(dD.alloc((size_t)diTot + 16)); CU_TRY(dO.alloc((size_t)dTot + 16));
        CU_TRY(dM.alloc((size_t)nb * (8 * 3 + 4 * 4)));
        int64_t* mSo = (int64_t*)dM.p; int64_t* mDo = mSo + nb; int64_t* mDio = mDo + nb;
        int32_t* mSl = (int32_t*)(mDio + nb); int32_t* mDc = mSl + nb; int32_t* mDl = mDc + nb; int32_t* mRes = mDl + nb;
        CU_TRY(cudaMemcpy(dS.p, hs.data(), (size_t)sTot, cudaMemcpyHostToDevice));
        if (diTot) CU_TRY(cudaMemcpy(dD.p, hd.data(), (size_t)diTot, cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(mSo, so.data(), (size_t)nb * 8, cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(mDo, doff.data(), (size_t)nb * 8, cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(mDio, dio.data(), (size_t)nb * 8, cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(mSl, sl.data(), (size_t)nb * 4, cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(mDc, dc.data(), (size_t)nb * 4, cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(mDl, dl.data(), (size_t)nb * 4, cudaMemcpyHostToDevice));
        GeneralArgs d{(const uint8_t*)dS.p, mSo, mSl, (uint8_t*)dO.p, mDo, mDc,
                      g.dictBase ? (const uint8_t*)dD.p : nullptr, mDio, mDl, mRes, nb, g.partial};
        CU_TRY(launch_general(d, nullptr));
        CU_TRY(cudaMemcpy(res.data(), mRes, (size_t)nb * 4, cudaMemcpyDeviceToHost));
        if (dTot) CU_TRY(cudaMemcpy(ho.data(), dO.p, (size_t)dTot, cudaMemcpyDeviceToHost));
        for (int64_t k = 0; k < nb; k++) {
            g.outLen[i + k] = res[k];
            if (res[k] > 0) memcpy(g.dstBase + g.dstOff[i + k], ho.data() + doff[k], (size_t)res[k]);
        }
        i = j;
    }
    return K4LZ4_OK;
}

int run_general(const GeneralArgs& g, int memKind, void* stream, int device) {
    if (memKind == K4LZ4_MEM_HOST) return run_general_host(g, device);
    if (memKind != K4LZ4_MEM_DEVICE) return fail(K4LZ4_E_ARG, "unknown memKind %d", memKind);
    if (device_count_cached() <= 0) return fail(K4LZ4_E_NODEVICE, "no CUDA device available");
    if (g.n < 0 || g.n > INT32_MAX) return fail(K4LZ4_E_ARG, "bad block count");
    if (g.n == 0) return K4LZ4_OK;
    if (!g.srcBase || !g.srcOff || !g.srcLen || !g.dstBase || !g.dstOff || !g.dstCap || !g.outLen)
        return fail(K4LZ4_E_ARG, "null pointer argument");
    if (g.dictBase && (!g.dictOff || !g.dictLen)) return fail(K4LZ4_E_ARG, "null pointer argument");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(K4LZ4_E_CUDA, "cudaSetDevice(%d) failed", device);
    CU_TRY(launch_general(g, (cudaStream_t)stream));
    return K4LZ4_OK;
}

}  // namespace

// ---- exported C ABI ------------------------------------------------------------------------

extern "C" {

int32_t k4lz4_codec_version(void) { return 192; }
int32_t k4lz4_device_count(void) { return device_count_cached(); }
const char* k4lz4_last_error(void) { return t_err.c_str(); }
int64_t k4lz4_launch_count(void) { return g_launches.load(); }

int32_t k4lz4_decode_stats(int32_t device, uint64_t* out4, int32_t reset) {
    if (device_count_cached() <= 0) return fail(K4LZ4_E_NODEVICE, "no CUDA device available");
    if (!out4) return fail(K4LZ4_E_ARG, "null pointer argument");
    DeviceGuard g(device);
    if (!g.ok) return fail(K4LZ4_E_CUDA, "cudaSetDevice(%d) failed", device);
    unsigned long long v[4] = {0, 0, 0, 0};
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpyFromSymbol(v, k4::g_decode_stats, sizeof(v)));
    for (int i = 0; i < 4; i++) out4[i] = v[i];
    if (reset) { unsigned long long z[4] = {0, 0, 0, 0}; CU_TRY(cudaMemcpyToSymbol(k4::g_decode_stats, z, sizeof(z))); }
    return K4LZ4_OK;
}

int32_t k4lz4_encode_stats(int32_t device, uint64_t* out3, int32_t reset) {
    if (device_count_cached() <= 0) return fail(K4LZ4_E_NODEVICE, "no CUDA device available");
    if (!out3) return fail(K4LZ4_E_ARG, "null pointer argument");
    DeviceGuard g(device);
    if (!g.ok) return fail(K4LZ4_E_CUDA, "cudaSetDevice(%d) failed", device);
    unsigned long long v[3] = {0, 0, 0};
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpyFromSymbol(v, k4::g_encode_stats, sizeof(v)));
    for (int i = 0; i < 3; i++) out3[i] = v[i];
    if (reset) { unsigned long long z[3] = {0, 0, 0}; CU_TRY(cudaMemcpyToSymbol(k4::g_encode_stats, z, sizeof(z))); }
    return K4LZ4_OK;
}

#ifdef K4_DT_PROFILE
// tools-only build: per-phase cycle sums of the tile decoder (scratch/, never shipped)
__attribute__((visibility("default"))) int32_t k4lz4_debug_prof(uint64_t* out32, int32_t reset) {
    unsigned long long v[32];
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpyFromSymbol(v, k4::g_decode_prof, sizeof(v)));
    for (int i = 0; i < 32; i++) out32[i] = v[i];
    if (reset) { unsigned long long z[32] = {0}; CU_TRY(cudaMemcpyToSymbol(k4::g_decode_prof, z, sizeof(z))); }
    return K4LZ4_OK;
}
#endif

int32_t k4lz4_max_output_size(int32_t length) { return k4::max_output_size(length); }
int32_t k4lz4_pickle_bound(int32_t length) { return length <= 0 ? 0 : length + 1; }

int32_t k4lz4_encode(const uint8_t* src, int32_t srcLen, uint8_t* dst, int32_t dstCap, int32_t level) {
    if (srcLen <= 0) return 0;                       // LZ4Codec.cs:45-46
    if (level >= 3) return K4LZ4_R_DELEGATE;
    if (!src || (!dst && dstCap > 0)) return fail(K4LZ4_E_ARG, "null pointer argument");
    if (dstCap <= 0) return -1;                      // nothing fits in an empty target
    int64_t so = 0, dof = 0; int32_t out = -1;
    int rc = run(OP_ENCODE, src, &so, &srcLen, dst, &dof, &dstCap, &out, 1, level, K4LZ4_MEM_HOST, nullptr, 0);
    return rc != K4LZ4_OK ? rc : out;
}

int32_t k4lz4_decode(const uint8_t* src, int32_t srcLen, uint8_t* dst, int32_t dstCap) {
    if (srcLen <= 0) return 0;                       // LZ4Codec.cs:108-109
    if (!src || (!dst && dstCap > 0)) return fail(K4LZ4_E_ARG, "null pointer argument");
    if (dstCap <= 0) return -1;                      // LL64.dec.cs:162-168 gives 0 or -1 => -1
    int64_t so = 0, dof = 0; int32_t out = -1;
    int rc = run(OP_DECODE, src, &so, &srcLen, dst, &dof, &dstCap, &out, 1, 0, K4LZ4_MEM_HOST, nullptr, 0);
    return rc != K4LZ4_OK ? rc : out;
}

int32_t k4lz4_decode_dict(const uint8_t* src, int32_t srcLen, uint8_t* dst, int32_t dstCap,
                          const uint8_t* dict, int32_t dictLen) {
    if (srcLen <= 0) return 0;                       // LZ4Codec.cs:150-151
    if (!src || (!dst && dstCap > 0) || (!dict && dictLen > 0)) return fail(K4LZ4_E_ARG, "null pointer argument");
    if (dstCap <= 0) return -1;
    int64_t zero = 0; int32_t out = -1;
    GeneralArgs g{src, &zero, &srcLen, dst, &zero, &dstCap, dictLen > 0 ? dict : nullptr, &zero, &dictLen, &out, 1, false};
    const int rc = run_general(g, K4LZ4_MEM_HOST, nullptr, 0);
    return rc != K4LZ4_OK ? rc : out;
}

int32_t k4lz4_partial_decode(const uint8_t* src, int32_t srcLen, uint8_t* dst, int32_t targetLen) {
    if (srcLen <= 0) return 0;                       // LZ4Codec.cs:129-130
    if (!src || (!dst && targetLen > 0)) return fail(K4LZ4_E_ARG, "null pointer argument");
    if (targetLen <= 0) return -1;                   // engine returns 0 -> -1 (LZ4Codec.cs:135)
    int64_t zero = 0; int32_t out = -1;
    GeneralArgs g{src, &zero, &srcLen, dst, &zero, &targetLen, nullptr, nullptr, nullptr, &out, 1, true};
    const int rc = run_general(g, K4LZ4_MEM_HOST, nullptr, 0);
    return rc != K4LZ4_OK ? rc : out;
}

int32_t k4lz4_decode_dict_batch(const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen,
                                uint8_t* dstBase, const int64_t* dstOff, const int32_t* dstCap,
                                const uint8_t* dictBase, const int64_t* dictOff, const int32_t* dictLen,
                                int32_t* outLen, int32_t nBlocks, int32_t memKind, void* cudaStream,
                                int32_t device) {
    GeneralArgs g{srcBase, srcOff, srcLen, dstBase, dstOff, dstCap, dictBase, dictOff, dictLen, outLen, nBlocks, false};
    return run_general(g, memKind, cudaStream, device);
}

int32_t k4lz4_partial_decode_batch(const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen,
                                   uint8_t* dstBase, const int64_t* dstOff, const int32_t* targetLen,
                                   int32_t* outLen, int32_t nBlocks, int32_t memKind, void* cudaStream,
                                   int32_t device) {
    GeneralArgs g{srcBase, srcOff, srcLen, dstBase, dstOff, targetLen, nullptr, nullptr, nullptr, outLen, nBlocks, true};
    return run_general(g, memKind, cudaStream, device);
}

int32_t k4lz4_encode_x32(const uint8_t* src, int32_t srcLen, uint8_t* dst, int32_t dstCap, int32_t level) {
    if (srcLen <= 0) return 0;
    if (level >= 3) return K4LZ4_R_DELEGATE;
    if (!src || (!dst && dstCap > 0)) return fail(K4LZ4_E_ARG, "null pointer argument");
    if (dstCap <= 0) return -1;
    int64_t so = 0, dof = 0; int32_t out = -1;
    int rc = run(OP_ENCODE, src, &so, &srcLen, dst, &dof, &dstCap, &out, 1, level | k4::ENC_FLAG_X32, K4LZ4_MEM_HOST, nullptr, 0);
    return rc != K4LZ4_OK ? rc : out;
}

int32_t k4lz4_encode_batch_x32(const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen,
                               uint8_t* dstBase, const int64_t* dstOff, const int32_t* dstCap,
                               int32_t* outLen, int32_t nBlocks, int32_t level, int32_t memKind,
                               void* cudaStream, int32_t device) {
    if (level < 0 || level > 0xFF) return fail(K4LZ4_E_ARG, "bad level");
    return run(OP_ENCODE, srcBase, srcOff, srcLen, dstBase, dstOff, dstCap, outLen, nBlocks, level | k4::ENC_FLAG_X32,
               memKind, cudaStream, device);
}

int32_t k4lz4_encode_batch(const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen,
                           uint8_t* dstBase, const int64_t* dstOff, const int32_t* dstCap,
                           int32_t* outLen, int32_t nBlocks, int32_t level, int32_t memKind,
                           void* cudaStream, int32_t device) {
    if (level < 0 || level > 0xFF) return fail(K4LZ4_E_ARG, "bad level");
    return run(OP_ENCODE, srcBase, srcOff, srcLen, dstBase, dstOff, dstCap, outLen, nBlocks, level,
               memKind, cudaStream, device);
}

int32_t k4lz4_decode_batch(const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen,
                           uint8_t* dstBase, const int64_t* dstOff, const int32_t* dstCap,
                           int32_t* outLen, int32_t nBlocks, int32_t memKind, void* cudaStream,
                           int32_t device) {
    return run(OP_DECODE, srcBase, srcOff, srcLen, dstBase, dstOff, dstCap, outLen, nBlocks, 0,
               memKind, cudaStream, device);
}

int32_t k4lz4_pickle_batch(const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen,
                           uint8_t* dstBase, const int64_t* dstOff, int32_t* outLen,
                           int32_t nMessages, int32_t level, int32_t memKind, void* cudaStream,
                           int32_t device) {
    return run(OP_PICKLE, srcBase, srcOff, srcLen, dstBase, dstOff, nullptr, outLen, nMessages, level,
               memKind, cudaStream, device);
}

int32_t k4lz4_pickle_writer_bound(int32_t length) { return length <= 0 ? 0 : length + 1 + k4::pickle_diff_width(length); }

int32_t k4lz4_pickle_writer_batch(const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen,
                                  uint8_t* dstBase, const int64_t* dstOff, int32_t* outLen,
                                  int32_t nMessages, int32_t level, int32_t memKind, void* cudaStream,
                                  int32_t device) {
    return run(OP_PICKLEW, srcBase, srcOff, srcLen, dstBase, dstOff, nullptr, outLen, nMessages, level,
               memKind, cudaStream, device);
}

int32_t k4lz4_unpickled_size_batch(const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen,
                                   int32_t* outSize, int32_t nMessages, int32_t memKind,
                                   void* cudaStream, int32_t device) {
    return run(OP_USIZE, srcBase, srcOff, srcLen, nullptr, nullptr, nullptr, outSize, nMessages, 0,
               memKind, cudaStream, device);
}

int32_t k4lz4_unpickle_batch(const uint8_t* srcBase, const int64_t* srcOff, const int32_t* srcLen,
                             uint8_t* dstBase, const int64_t* dstOff, const int32_t* dstLen,
                             int32_t* outLen, int32_t nMessages, int32_t memKind, void* cudaStream,
                             int32_t device) {
    return run(OP_UNPICKLE, srcBase, srcOff, srcLen, dstBase, dstOff, dstLen, outLen, nMessages, 0,
               memKind, cudaStream, device);
}

uint32_t k4lz4_xxh32(const uint8_t* data, int64_t length, uint32_t seed) {
    return k4::xxh32_host(data, length > 0 && data ? (size_t)length : 0, seed);
}

int32_t k4lz4_xxh32_batch(const uint8_t* base, const int64_t* off, const int32_t* len, uint32_t seed,
                          uint32_t* out, int32_t nBlocks, int32_t memKind, void* cudaStream, int32_t device) {
    if (device_count_cached() <= 0) return fail(K4LZ4_E_NODEVICE, "no CUDA device available");
    if (nBlocks < 0 || !base || !off || !len || !out) return fail(K4LZ4_E_ARG, "bad xxh32 arguments");
    if (nBlocks == 0) return K4LZ4_OK;
    DeviceGuard g(memKind == K4LZ4_MEM_HOST && device < 0 ? 0 : device);
    if (!g.ok) return fail(K4LZ4_E_CUDA, "cudaSetDevice(%d) failed", device);
    const unsigned ctas = (unsigned)(((int64_t)nBlocks * 4 + 127) / 128);
    if (memKind == K4LZ4_MEM_DEVICE) {
        k4::xxh32_batch_kernel<<<ctas, 128, 0, (cudaStream_t)cudaStream>>>(base, off, len, seed, out, nBlocks);
        g_launches++;
        CU_TRY(cudaGetLastError());
        return K4LZ4_OK;
    }
    if (memKind != K4LZ4_MEM_HOST) return fail(K4LZ4_E_ARG, "unknown memKind %d", memKind);
    // host memory: pack, one H2D, one kernel, one D2H (checksums are a side channel of the frame writer)
    std::vector<int64_t> po((size_t)nBlocks);
    int64_t tot = 0;
    for (int i = 0; i < nBlocks; i++) { po[(size_t)i] = tot; tot += len[i] > 0 ? len[i] : 0; }
    std::vector<uint8_t> pk((size_t)tot + 16);
    for (int i = 0; i < nBlocks; i++) if (len[i] > 0) memcpy(pk.data() + po[(size_t)i], base + off[i], (size_t)len[i]);
    DevMem dB, dM;
    CU_TRY(dB.alloc((size_t)tot + 16));
    CU_TRY(dM.alloc((size_t)nBlocks * 16));
    int64_t* dOff = (int64_t*)dM.p; int32_t* dLen = (int32_t*)(dOff + nBlocks); uint32_t* dOut = (uint32_t*)(dLen + nBlocks);
    CU_TRY(cudaMemcpy(dB.p, pk.data(), (size_t)tot, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(dOff, po.data(), (size_t)nBlocks * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(dLen, len, (size_t)nBlocks * 4, cudaMemcpyHostToDevice));
    k4::xxh32_batch_kernel<<<ctas, 128>>>((const uint8_t*)dB.p, dOff, dLen, seed, dOut, nBlocks);
    g_launches++;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpy(out, dOut, (size_t)nBlocks * 4, cudaMemcpyDeviceToHost));
    return K4LZ4_OK;
}

int32_t k4lz4_synth_host(uint8_t* base, int64_t nBlocks, int32_t blockSize, int32_t matchPermille,
                         uint64_t seed, int64_t firstBlock) {
    if (!base || nBlocks < 0 || blockSize <= 0) return fail(K4LZ4_E_ARG, "bad synth arguments");
    unsigned hw = std::thread::hardware_concurrency();
    int T = (int)std::min<int64_t>(std::min<unsigned>(hw ? hw : 1, 64), std::max<int64_t>(nBlocks, 1));
    std::vector<std::thread> th;
    for (int t = 0; t < T; t++)
        th.emplace_back([=] {
            for (int64_t b = nBlocks * t / T; b < nBlocks * (t + 1) / T; b++)
                k4::synth_block(base + b * (int64_t)blockSize, blockSize, (uint32_t)matchPermille, seed,
                                (uint64_t)(firstBlock + b));
        });
    for (auto& t : th) t.join();
    return K4LZ4_OK;
}

int32_t k4lz4_synth_device(uint8_t* base, int64_t nBlocks, int32_t blockSize, int32_t matchPermille,
                           uint64_t seed, int64_t firstBlock, void* cudaStream, int32_t device) {
    if (device_count_cached() <= 0) return fail(K4LZ4_E_NODEVICE, "no CUDA device available");
    if (!base || nBlocks < 0 || blockSize <= 0) return fail(K4LZ4_E_ARG, "bad synth arguments");
    if (nBlocks == 0) return K4LZ4_OK;
    DeviceGuard g(device);
    if (!g.ok) return fail(K4LZ4_E_CUDA, "cudaSetDevice(%d) failed", device);
    const int threads = 64;
    const long long ctas = (nBlocks + threads - 1) / threads;
    k4::synth_kernel<<<(unsigned)ctas, threads, 0, (cudaStream_t)cudaStream>>>(
        base, nBlocks, blockSize, (uint32_t)matchPermille, seed, firstBlock);
    g_launches++;
    CU_TRY(cudaGetLastError());
    return K4LZ4_OK;
}

int32_t k4lz4_copy_blocks_device(const uint8_t* srcBase, const int64_t* srcOff, uint8_t* dstBase,
                                 const int64_t* dstOff, const int32_t* len, int32_t nBlocks,
                                 void* cudaStream, int32_t device) {
    if (device_count_cached() <= 0) return fail(K4LZ4_E_NODEVICE, "no CUDA device available");
    if (nBlocks < 0 || !srcBase || !srcOff || !dstBase || !dstOff || !len)
        return fail(K4LZ4_E_ARG, "bad copy_blocks arguments");
    if (nBlocks == 0) return K4LZ4_OK;
    DeviceGuard g(device);
    if (!g.ok) return fail(K4LZ4_E_CUDA, "cudaSetDevice(%d) failed", device);
    k4::copy_blocks_kernel<<<nBlocks, 256, 0, (cudaStream_t)cudaStream>>>(srcBase, srcOff, dstBase,
                                                                         dstOff, len, nBlocks);
    g_launches++;
    CU_TRY(cudaGetLastError());
    return K4LZ4_OK;
}

}  // extern "C"
