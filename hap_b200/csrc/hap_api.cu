// hap_b200/csrc/hap_api.cu -- the C-ABI of libhap_b200.so: the six entry points of include/hap.h
// (same signatures and behaviour as /root/reference/source/hap.h:76-152) and the extensions of
// include/hap_b200.h.  Host code here only validates arguments, walks section headers, moves
// buffers and launches kernels; all compression, decompression, block coding and frame assembly
// runs in the kernels of this directory.  There is no CPU implementation of any of those steps in
// this library: without a CUDA device the compute entry points return HapResult_Internal_Error.
#include "../../include/hap_b200.h"

#include "bc_decode.cuh"
#include "bc_encode.cuh"
#include "hap_assemble.cuh"
#include "hap_host.h"
#include "hap_mov.h"
#include "hap_parse.cuh"
#include "snappy_decode.cuh"
#include "snappy_encode.cuh"

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

using namespace hapb200;

namespace {

std::atomic<unsigned long long> g_launches{0};
// Options (HapB200SetOption).  g_use_index: the decoder uses a frame's embedded fragment index when it has one
// (hap_index.h).  g_write_index: the encoder writes that section into Complex texture sections.
std::atomic<int> g_use_index{1};
std::atomic<int> g_write_index{0};
std::atomic<int> g_write_offsets{0};
std::atomic<int> g_chroma_refine{0};   // HAPB200_OPTION_CHROMA_REFINE

// Optional per-stage device timing (HapB200SetStageTiming): CUDA events around every kernel, on the
// stream the kernel is launched on.  Off by default; bench.py turns it on for its roofline pass only.
enum Stage { kStBcEncode = 0, kStSnappyEncode, kStPlan, kStPlace, kStParse, kStSnappyDecode, kStCollect, kStBcDecode, kStSnappyIndex, kStWindows, kStCount };
struct StageTimer {
    std::mutex mu;
    bool on = false;
    struct Rec { int stage; cudaEvent_t a, b; };
    std::vector<Rec> recs;
    double ms[kStCount] = {0};
    unsigned long long n[kStCount] = {0};
};
StageTimer g_timer;

struct StageScope {
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t st;
    int stage;
    bool live;
    StageScope(int stage_, cudaStream_t st_) : st(st_), stage(stage_), live(g_timer.on)
    {
        if (live) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, st); }
    }
    ~StageScope()
    {
        if (!live) return;
        cudaEventRecord(b, st);
        std::lock_guard<std::mutex> l(g_timer.mu);
        g_timer.recs.push_back({stage, a, b});
    }
};

#define HAP_KLAUNCH(stage, kernel, grid, block, smem, stream, ...)         \
    do {                                                                   \
        StageScope hap_scope_(stage, stream);                              \
        HAP_LAUNCH(kernel, grid, block, smem, stream, __VA_ARGS__);        \
        g_launches.fetch_add(1, std::memory_order_relaxed);                \
    } while (0)

// ---- devices ------------------------------------------------------------------------------------------------------------
// The library can drive every GPU of the box from one process (or one GPU per process under torchrun -- both work):
//   * a call that has a DEVICE pointer among its buffers runs on that pointer's device;
//   * a call with host pointers only runs on the process's default device: the device that was current in the thread that
//     made the library's first call, or the one named by HapB200SetDevice (a new host thread starts on device 0, so "the
//     calling thread's current device" would send the worker threads of a process that drives GPU 3 to GPU 0);
//   * the caller's current device is restored when the call returns.
// Per-device state (SM count, kernel attributes, memory-pool threshold) is set up on a device's first use.
constexpr int kMaxDevices = 64;
struct DeviceState {
    std::once_flag once;
    bool ready = false;
    int sm_count = 148;
    int k5_ctas_per_sm = 0;   // resident CTAs of the fragment compressor (K5) per SM
};
DeviceState g_dev[kMaxDevices];
std::atomic<int> g_default_device{-1};
std::mutex g_legacy_mu;   // serialises the calls that run on the legacy default stream (those with a device pointer among their buffers)
thread_local int t_device = 0;   // device of the library call running on this thread

void device_init(int dev)
{
    DeviceState &d = g_dev[dev];
    if (cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || d.sm_count <= 0) { cudaGetLastError(); d.sm_count = 148; }
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        unsigned long long keep = ~0ull;  // keep freed scratch in the pool: steady-state calls never hit the OS
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    // (function attributes are per device: set them on each device's first use)
    bool ok = cudaFuncSetAttribute(snappy_execute_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ExecSmem)) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(snappy_index_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IndexSmem)) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(snappy_encode_fragments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)sizeof(EncodeSmem)) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(snappy_encode_fragments_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                    (int)cudaSharedmemCarveoutMaxShared) == cudaSuccess;
    // K5 is built for kEncCtasPerSm resident CTAs (registers, shared memory); a device that fits fewer is not set up
    ok = ok && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&d.k5_ctas_per_sm, snappy_encode_fragments_kernel, kEncThreads,
                                                             sizeof(EncodeSmem)) == cudaSuccess;
    ok = ok && d.k5_ctas_per_sm >= kEncCtasPerSm;
    if (!ok) { cudaGetLastError(); return; }
    d.ready = true;
}

int pointer_device(const void *p)   // device ordinal of a device / managed pointer, -1 for host memory
{
    cudaPointerAttributes a;
    if (!p || cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return -1; }
    return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) ? a.device : -1;
}

// One per entry point.  `hints`: the call's buffers; the first device pointer among them decides the device.
struct DeviceGuard {
    int saved = -1;
    bool ok = false;
    DeviceGuard(std::initializer_list<const void *> hints)
    {
        static std::once_flag env_once;
        std::call_once(env_once, [] {
            // process-wide defaults of the two options (HapB200SetOption overrides them)
            if (const char *e = getenv("HAPB200_WRITE_INDEX")) g_write_index.store(atoi(e) != 0);
            if (const char *e = getenv("HAPB200_USE_INDEX")) g_use_index.store(atoi(e) != 0);
            if (const char *e = getenv("HAPB200_WRITE_OFFSET_TABLE")) g_write_offsets.store(atoi(e) != 0);
            if (const char *e = getenv("HAPB200_CHROMA_REFINE")) g_chroma_refine.store(atoi(e) != 0);
        });
        if (cudaGetDevice(&saved) != cudaSuccess) { cudaGetLastError(); saved = -1; return; }
        int want = -1;
        for (const void *h : hints) {
            want = pointer_device(h);
            if (want >= 0) break;
        }
        if (want < 0) {
            int expected = -1;
            g_default_device.compare_exchange_strong(expected, saved);   // first call: this thread's device becomes the default
            want = g_default_device.load();
        }
        if (want < 0 || want >= kMaxDevices) return;
        if (want != saved && cudaSetDevice(want) != cudaSuccess) { cudaGetLastError(); return; }
        std::call_once(g_dev[want].once, device_init, want);
        t_device = want;
        ok = g_dev[want].ready;
    }
    ~DeviceGuard()
    {
        int cur = -1;
        if (saved >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != saved) cudaSetDevice(saved);
        cudaGetLastError();
    }
};
#define HAP_ENTER(...)                                     \
    DeviceGuard hap_device_guard_({__VA_ARGS__});          \
    if (!hap_device_guard_.ok) return HapResult_Internal_Error

inline int sm_count() { return g_dev[t_device].sm_count; }
const cudaStream_t kLegacyStream = cudaStreamLegacy;
// NULL-stream calls and the host-pointer entry points that touch caller-owned device buffers run on the LEGACY default
// stream: it orders itself against every blocking stream of the process, so buffers a caller produced on its own (blocking)
// stream -- torch's current stream, cudaMemset, ... -- are complete before our kernels touch them.

// Stream of one host-pointer call.  When every buffer of the call is host memory nothing outside the call can
// be ordered against it, so it takes a private non-blocking stream from a pool and concurrent calls from
// different host threads overlap their copies and kernels (the reference is re-entrant, hap.c has no globals).
// With any device pointer among the arguments the call uses the legacy default stream under a mutex, which
// orders it after whatever produced those buffers on the caller's (blocking) streams.
// A pooled stream brings its own memory pool: scratch freed by one host-pointer call is handed to the next call
// on the SAME stream.  With the device's default pool, memory freed on one stream and re-used on another makes the
// second stream wait for the first, which chained concurrent calls from different host threads one behind the other.
struct PooledStream {
    cudaStream_t st = nullptr;
    cudaMemPool_t mem = nullptr;
};
thread_local cudaMemPool_t g_call_mem = nullptr;   // pool of the host-pointer call running on this thread, if any

struct CallStream {
    cudaStream_t st = nullptr;
    bool pooled = false;
    PooledStream ps;
    std::unique_lock<std::mutex> serial;
    static std::mutex &pool_mu() { static std::mutex m; return m; }
    static std::vector<PooledStream> &pool() { static std::vector<PooledStream> v[kMaxDevices]; return v[t_device]; }
    int device = 0;
    explicit CallStream(bool all_host)
    {
        device = t_device;
        if (all_host) {
            {
                std::lock_guard<std::mutex> l(pool_mu());
                if (!pool().empty()) { ps = pool().back(); pool().pop_back(); }
            }
            if (!ps.st) {
                if (cudaStreamCreateWithFlags(&ps.st, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); ps.st = nullptr; }
                int dev = 0;
                cudaMemPoolProps props;
                memset(&props, 0, sizeof props);
                props.allocType = cudaMemAllocationTypePinned;
                props.handleTypes = cudaMemHandleTypeNone;
                props.location.type = cudaMemLocationTypeDevice;
                if (ps.st && cudaGetDevice(&dev) == cudaSuccess) {
                    props.location.id = dev;
                    if (cudaMemPoolCreate(&ps.mem, &props) == cudaSuccess) {
                        unsigned long long keep = ~0ull;
                        cudaMemPoolSetAttribute(ps.mem, cudaMemPoolAttrReleaseThreshold, &keep);
                    } else {
                        cudaGetLastError();
                        ps.mem = nullptr;   // fall back to the default pool
                    }
                }
            }
            st = ps.st;
            pooled = st != nullptr;
            if (pooled) g_call_mem = ps.mem;
        }
        if (!pooled) {
            serial = std::unique_lock<std::mutex>(g_legacy_mu);
            st = kLegacyStream;
        }
    }
    ~CallStream()
    {
        if (pooled) {
            g_call_mem = nullptr;
            std::lock_guard<std::mutex> l(pool_mu());
            static_cast<void>(device);
            pool().push_back(ps);   // (t_device is still this call's device: the guard outlives the stream)
        }
    }
};

bool is_device_pointer(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// stream-ordered scratch
struct DevBuf {
    void *p = nullptr;
    cudaStream_t s;
    explicit DevBuf(cudaStream_t st) : s(st) {}
    bool alloc(size_t n)
    {
        n = (n + 31) & ~(size_t)15;   // whole 16-byte cells + one: kernels read their inputs in aligned 16-byte cells
        if (g_call_mem) return cudaMallocFromPoolAsync(&p, n, g_call_mem, s) == cudaSuccess;
        return cudaMallocAsync(&p, n, s) == cudaSuccess;
    }
    ~DevBuf() { if (p) cudaFreeAsync(p, s); }
    template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

inline uint64_t align16(uint64_t v) { return (v + 15) & ~15ull; }

// ---- codec tables ------------------------------------------------------------------------------
struct CodecInfo {
    uint32_t textures;
    uint32_t fmt[2];
    uint32_t block_bytes[2];
    int bc_kind;
};
bool codec_info(unsigned codec, CodecInfo &c)
{
    switch (codec) {
    case HapB200Codec_Hap1: c = {1, {HapFmt_RGB_DXT1, 0}, {8, 0}, kBcDxt1}; return true;
    case HapB200Codec_Hap5: c = {1, {HapFmt_RGBA_DXT5, 0}, {16, 0}, kBcDxt5}; return true;
    case HapB200Codec_HapY: c = {1, {HapFmt_YCoCg_DXT5, 0}, {16, 0}, kBcYCoCg}; return true;
    case HapB200Codec_HapM: c = {2, {HapFmt_YCoCg_DXT5, HapFmt_A_RGTC1}, {16, 8}, kBcYCoCgPlusAlpha}; return true;
    case HapB200Codec_HapA: c = {1, {HapFmt_A_RGTC1, 0}, {8, 0}, kBcRgtc1}; return true;
    default: return false;
    }
}

// ---- device pipelines (all asynchronous on `st`) -------------------------------------------------

// textures of `frames` frames (device, described by G.s[i].in_offset/in_stride relative to `base`) ->
// frames at out + f*out_stride, lengths in used[f]
uint32_t launch_encode(const uint8_t *base, const FrameGeom &G, uint32_t frames, uint8_t *out, uint64_t out_stride,
                       unsigned long long *used, cudaStream_t st)
{
    const uint64_t nfrag = (uint64_t)frames * G.frags_per_frame;
    if (nfrag == 0 || nfrag >= (1ull << 31)) return HapResult_Bad_Arguments;
    DevBuf scratch(st), fsize(st), fdst(st), fidx(st), fent(st);
    bool any_compress = false;
    for (uint32_t i = 0; i < G.sections; i++) any_compress = any_compress || G.s[i].compress;
    const uint32_t write_index = any_compress && g_write_index.load() ? 1u : 0u;
    if (!scratch.alloc(any_compress ? nfrag * kFragCap : 16) || !fsize.alloc(nfrag * 4) || !fdst.alloc(nfrag * 4) || !fidx.alloc(nfrag * 4) ||
        !fent.alloc(write_index ? nfrag * kFragEntryStride : 16)) {
        cudaGetLastError();
        return HapResult_Internal_Error;
    }
    // every resident CTA slot of the device strides over the fragments (two CTAs of 512 threads per SM)
    const uint64_t k5_slots = (uint64_t)g_dev[t_device].k5_ctas_per_sm * (uint64_t)sm_count();
    const unsigned k5_grid = (unsigned)(nfrag < k5_slots ? nfrag : k5_slots);
    HAP_KLAUNCH(kStSnappyEncode, snappy_encode_fragments_kernel, dim3(k5_grid), dim3(kEncThreads), sizeof(EncodeSmem), st, base, G,
                (uint32_t)nfrag, scratch.as<uint8_t>(), fsize.as<uint32_t>(), write_index ? fent.as<uint8_t>() : (uint8_t *)nullptr);
    HAP_KLAUNCH(kStPlan, hap_plan_frames_kernel, dim3(frames), dim3(kPlanThreads), 0, st, G, base, fsize.as<uint32_t>(),
                fdst.as<uint32_t>(), fidx.as<uint32_t>(), (write_index ? kPlanWriteIndex : 0u) | (g_write_offsets.load() ? kPlanWriteOffsets : 0u), out,
                out_stride, used);
    HAP_KLAUNCH(kStPlace, hap_place_fragments_kernel, dim3((unsigned)nfrag), dim3(kPlaceThreads), 0, st, G, base,
                scratch.as<uint8_t>(), fsize.as<uint32_t>(), fdst.as<uint32_t>(), fidx.as<uint32_t>(),
                write_index ? fent.as<uint8_t>() : (const uint8_t *)nullptr, out, out_stride);
    return cudaGetLastError() == cudaSuccess ? HapResult_No_Error : HapResult_Internal_Error;
}

uint32_t launch_block_encode(const uint8_t *rgba, uint32_t frames, uint64_t frame_stride, uint32_t width, uint32_t height,
                             uint64_t row_bytes, const CodecInfo &ci, uint8_t *blocks, uint64_t blocks_stride,
                             uint64_t second_offset, cudaStream_t st)
{
    BcGeom g;
    g.blocks_x = width / 4;
    g.blocks_y = height / 4;
    g.row_bytes = (uint32_t)row_bytes;
    const uint64_t inv = 0x100000000ull / g.blocks_x;          // 2^32 when the image is one block wide
    g.inv_blocks_x = inv > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)inv;
    g.frame_bytes = frame_stride;
    g.out_stride = blocks_stride;
    g.second_offset = second_offset;
    dim3 grid((g.blocks_x * g.blocks_y + kBcThreads - 1) / kBcThreads, frames);
    const bool refine = g_chroma_refine.load() != 0;
    switch (ci.bc_kind) {
    case kBcDxt1: HAP_KLAUNCH(kStBcEncode, bc_encode_kernel<kBcDxt1>, grid, dim3(kBcThreads), 0, st, rgba, g, blocks); break;
    case kBcDxt5: HAP_KLAUNCH(kStBcEncode, bc_encode_kernel<kBcDxt5>, grid, dim3(kBcThreads), 0, st, rgba, g, blocks); break;
    case kBcYCoCg:
        if (refine) HAP_KLAUNCH(kStBcEncode, (bc_encode_kernel<kBcYCoCg, true>), grid, dim3(kBcThreads), 0, st, rgba, g, blocks);
        else HAP_KLAUNCH(kStBcEncode, bc_encode_kernel<kBcYCoCg>, grid, dim3(kBcThreads), 0, st, rgba, g, blocks);
        break;
    case kBcRgtc1: HAP_KLAUNCH(kStBcEncode, bc_encode_kernel<kBcRgtc1>, grid, dim3(kBcThreads), 0, st, rgba, g, blocks); break;
    default:
        if (refine) HAP_KLAUNCH(kStBcEncode, (bc_encode_kernel<kBcYCoCgPlusAlpha, true>), grid, dim3(kBcThreads), 0, st, rgba, g, blocks);
        else HAP_KLAUNCH(kStBcEncode, bc_encode_kernel<kBcYCoCgPlusAlpha>, grid, dim3(kBcThreads), 0, st, rgba, g, blocks);
        break;
    }
    return cudaGetLastError() == cudaSuccess ? HapResult_No_Error : HapResult_Internal_Error;
}

uint32_t launch_block_decode(const uint8_t *blocks, const uint8_t *alpha, uint32_t frames, uint64_t blocks_stride,
                             uint64_t alpha_stride, uint32_t width, uint32_t height, const CodecInfo &ci, uint8_t *rgba,
                             uint64_t frame_stride, uint64_t row_bytes, cudaStream_t st, const uint32_t *frame_results = nullptr)
{
    BcDecodeGeom g;
    g.blocks_x = width / 4;
    g.blocks_y = height / 4;
    g.row_bytes = (uint32_t)row_bytes;
    g.merge_alpha = ci.textures == 2;
    g.in_stride = blocks_stride;
    g.alpha_stride = alpha_stride;
    g.frame_bytes = frame_stride;
    dim3 grid((g.blocks_x * g.blocks_y + kBcThreads - 1) / kBcThreads, frames);
    switch (ci.bc_kind) {
    case kBcDxt1: HAP_KLAUNCH(kStBcDecode, bc_decode_kernel<kBcDxt1>, grid, dim3(kBcThreads), 0, st, blocks, alpha, g, rgba, frame_results); break;
    case kBcDxt5: HAP_KLAUNCH(kStBcDecode, bc_decode_kernel<kBcDxt5>, grid, dim3(kBcThreads), 0, st, blocks, alpha, g, rgba, frame_results); break;
    case kBcRgtc1: HAP_KLAUNCH(kStBcDecode, bc_decode_kernel<kBcRgtc1>, grid, dim3(kBcThreads), 0, st, blocks, alpha, g, rgba, frame_results); break;
    default: HAP_KLAUNCH(kStBcDecode, bc_decode_kernel<kBcYCoCg>, grid, dim3(kBcThreads), 0, st, blocks, alpha, g, rgba, frame_results); break;
    }
    return cudaGetLastError() == cudaSuccess ? HapResult_No_Error : HapResult_Internal_Error;
}

// Decode-side options (HapB200SetOption): 1 = use a frame's embedded fragment index when it has one (hap_index.h)

// Everything after the jobs exist (device array): windows, on-the-fly index, execute, repair of chunks whose embedded
// index did not hold up.  in_bound / out_bound: upper bounds of the jobs' total compressed / decoded bytes (they size the
// window list; a list that turns out too short makes the affected chunks report Internal_Error, never overruns).
// The decode of a list of chunk jobs: first pass (windows -> on-the-fly index for chunks without one -> execute) and the repair
// pass for chunks whose embedded index did not describe their stream (decoded again as if they had none).  Batch calls queue
// both passes (the second finds nothing to do on honest frames); HapDecode, which reads the statuses on the host anyway, only
// launches the repair pass when a chunk asks for it.
struct DecodePasses {
    DevBuf wins, entries, done, ctl;
    ChunkJob *jobs = nullptr;
    uint32_t njobs = 0, win_cap = 0, entry_slots = 0;
    cudaStream_t st;
    explicit DecodePasses(cudaStream_t s) : wins(s), entries(s), done(s), ctl(s), st(s) {}

    uint32_t first(ChunkJob *j, uint32_t n, uint64_t in_bound, uint64_t out_bound)
    {
        jobs = j; njobs = n;
        // windows: up to kIdxParts per 16 KiB of stream from the index kernel (twice: a chunk may be indexed again by the repair
        // pass), one per fragment of an indexed chunk, one per 64 KiB of a verbatim chunk
        const uint64_t slots64 = 2 * (in_bound / kIdxWin + njobs) + 16;
        const uint64_t cap64 = kIdxParts * slots64 + out_bound / kIndexFragBytes + 2ull * njobs + 16;
        if (cap64 >= (1ull << 31)) return HapResult_Bad_Arguments;
        win_cap = (uint32_t)cap64; entry_slots = (uint32_t)slots64;
        if (!wins.alloc((size_t)win_cap * sizeof(DecWin)) || !entries.alloc((size_t)entry_slots * kIdxThreads) || !done.alloc((size_t)win_cap * 4) ||
            !ctl.alloc(sizeof(DecodeCtl) + 16)) {
            cudaGetLastError();
            return HapResult_Internal_Error;
        }
        if (cudaMemsetAsync(ctl.p, 0, sizeof(DecodeCtl) + 16, st) != cudaSuccess || cudaMemsetAsync(done.p, 0, (size_t)win_cap * 4, st) != cudaSuccess) {
            cudaGetLastError();
            return HapResult_Internal_Error;
        }
        DecodeCtl *c = ctl.as<DecodeCtl>();
        const unsigned ex_grid = (unsigned)sm_count() * (unsigned)HAPB200_EX_MIN_BLOCKS;
        HAP_KLAUNCH(kStWindows, hap_build_windows_kernel, dim3((njobs + 127) / 128), dim3(128), 0, st, jobs, njobs, (uint32_t)g_use_index.load(),
                    wins.as<DecWin>(), win_cap, c);
        HAP_KLAUNCH(kStSnappyIndex, snappy_index_kernel, dim3(njobs), dim3(kIdxThreads), sizeof(IndexSmem), st, jobs, (int)njobs, 0u,
                    wins.as<DecWin>(), win_cap, entries.as<uint8_t>(), entry_slots, c);
        HAP_KLAUNCH(kStSnappyDecode, snappy_execute_kernel, dim3(ex_grid), dim3(kExThreads), sizeof(ExecSmem), st, jobs, njobs, 0u, wins.as<DecWin>(), c,
                    done.as<uint32_t>());
        return cudaGetLastError() == cudaSuccess ? HapResult_No_Error : HapResult_Internal_Error;
    }

    // chunks whose embedded index did not describe their stream: decode them again as if they had none
    uint32_t repair()
    {
        DecodeCtl *c = ctl.as<DecodeCtl>();
        uint32_t *any_left = reinterpret_cast<uint32_t *>(ctl.as<uint8_t>() + sizeof(DecodeCtl));
        const unsigned ex_grid = (unsigned)sm_count() * (unsigned)HAPB200_EX_MIN_BLOCKS;
        HAP_KLAUNCH(kStWindows, hap_requeue_mismatched_kernel, dim3((njobs + 127) / 128), dim3(128), 0, st, jobs, njobs, any_left);
        HAP_KLAUNCH(kStSnappyIndex, snappy_index_kernel, dim3(njobs), dim3(kIdxThreads), sizeof(IndexSmem), st, jobs, (int)njobs, 1u,
                    wins.as<DecWin>(), win_cap, entries.as<uint8_t>(), entry_slots, c);
        HAP_KLAUNCH(kStSnappyDecode, snappy_execute_kernel, dim3(ex_grid), dim3(kExThreads), sizeof(ExecSmem), st, jobs, njobs, 1u, wins.as<DecWin>(),
                    c, done.as<uint32_t>());
        return cudaGetLastError() == cudaSuccess ? HapResult_No_Error : HapResult_Internal_Error;
    }
};

uint32_t launch_decode_jobs(ChunkJob *jobs, uint32_t njobs, uint64_t in_bound, uint64_t out_bound, cudaStream_t st, bool may_have_index = true)
{
    DecodePasses P(st);
    uint32_t r = P.first(jobs, njobs, in_bound, out_bound);
    if (r == HapResult_No_Error && g_use_index.load() && may_have_index) r = P.repair();
    return r;
}

// device frames -> texture `index` of each; jobs scratch is allocated here
uint32_t launch_decode_batch(const uint8_t *in, uint32_t frames, uint64_t in_stride, const unsigned long long *in_bytes,
                             uint32_t index, uint32_t max_chunks, uint8_t *out, uint64_t out_stride, uint64_t out_capacity,
                             unsigned long long *used, uint32_t *formats, uint32_t *results, cudaStream_t st)
{
    const uint64_t njobs = (uint64_t)frames * max_chunks;
    if (njobs == 0 || njobs >= (1ull << 31)) return HapResult_Bad_Arguments;
    DevBuf jobs(st), whole(st);
    if (!jobs.alloc(njobs * sizeof(ChunkJob)) || !whole.alloc((size_t)frames * 4)) { cudaGetLastError(); return HapResult_Internal_Error; }
    HAP_KLAUNCH(kStParse, hap_parse_frames_kernel, dim3((frames + 127) / 128), dim3(128), 0, st, in, in_stride, in_bytes, frames, index,
                max_chunks, out, out_stride, out_capacity, jobs.as<ChunkJob>(), used, formats, results, whole.as<uint32_t>());
    uint32_t r = launch_decode_jobs(jobs.as<ChunkJob>(), (uint32_t)njobs, (uint64_t)frames * in_stride, (uint64_t)frames * out_capacity, st);
    if (r != HapResult_No_Error) return r;
    HAP_KLAUNCH(kStCollect, hap_collect_status_kernel, dim3((frames + 127) / 128), dim3(128), 0, st, jobs.as<ChunkJob>(), frames,
                max_chunks, whole.as<uint32_t>(), results, used);
    return cudaGetLastError() == cudaSuccess ? HapResult_No_Error : HapResult_Internal_Error;
}

// host-side view of a frame whose bytes may live on the device.  Header walks read a few hundred bytes at data-dependent
// places (section headers, the Decode Instructions tables, five bytes at the head of every chunk, the trailing index header), so
// a device frame is mirrored LAZILY: `p` points at a zero-page-backed image of the whole frame and need(off, len) fetches the
// 4 KiB pages under [off, off+len) that are not there yet.  A 4K Hap Q frame costs ~10 small copies instead of 5 MB.
struct HeaderView {
    static constexpr uint64_t kPage = 4096;
    uint8_t *mirror = nullptr;
    const uint8_t *dev = nullptr;
    const uint8_t *p = nullptr;
    uint64_t bytes = 0;
    std::vector<bool> have;
    bool ok = true;
    HeaderView(const void *frame, unsigned long n) : bytes(n)
    {
        if (!is_device_pointer(frame)) { p = (const uint8_t *)frame; return; }
        dev = (const uint8_t *)frame;
        mirror = (uint8_t *)calloc(n ? n : 1, 1);     // untouched pages stay uncommitted
        if (!mirror) { ok = false; return; }
        p = mirror;
        have.assign((size_t)((n + kPage - 1) / kPage), false);
        need(0, kPage);
    }
    ~HeaderView() { free(mirror); }
    HeaderView(const HeaderView &) = delete;
    HeaderView &operator=(const HeaderView &) = delete;
    // make [off, off+len) of the frame readable through p (clamped to the frame); false after a failed copy
    bool need(uint64_t off, uint64_t len)
    {
        if (!dev || !ok || off >= bytes || len == 0) return ok;
        if (len > bytes - off) len = bytes - off;
        uint64_t a = off / kPage;
        const uint64_t b = (off + len - 1) / kPage;
        while (a <= b) {
            if (have[(size_t)a]) { a++; continue; }
            uint64_t e = a;
            while (e <= b && !have[(size_t)e]) have[(size_t)e++] = true;
            const uint64_t lo = a * kPage, hi = e * kPage < bytes ? e * kPage : bytes;
            if (cudaMemcpy(mirror + lo, dev + lo, hi - lo, cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); ok = false; return false; }
            a = e;
        }
        return true;
    }
    // the texture section `index` (hap.c:932-991), fetching the inner section headers a two-texture frame needs
    uint32_t locate(uint32_t index, Located &loc)
    {
        Section top;
        if (dev && read_section_header(p, (uint32_t)bytes, top) == HapResult_No_Error && top.type == kSecMultipleImages) {
            uint64_t off = top.hdr;
            for (uint32_t i = 0; i < index; i++) {
                Section s;
                need(off, 8);
                if (off >= bytes || read_section_header(p + off, (uint32_t)(bytes - off), s) != HapResult_No_Error) break;
                off += (uint64_t)s.hdr + s.len;
            }
            need(off, 8);
        }
        if (!ok) return HapResult_Internal_Error;
        return locate_texture(p, (uint32_t)bytes, index, loc);
    }
    // the Decode Instructions container at the head of texture section `loc` (hap.c:644-730)
    void need_tables(const Located &loc)
    {
        if (!dev) return;
        need(loc.offset, 8);
        Section di;
        if (loc.offset < bytes && read_section_header(p + loc.offset, loc.len, di) == HapResult_No_Error)
            need(loc.offset, (uint64_t)di.hdr + di.len);
    }
    // the trailing fragment index section's header and record-offset table (hap_index.h)
    void need_index_header()
    {
        if (!dev) return;
        Section top;
        if (read_section_header(p, (uint32_t)bytes, top) != HapResult_No_Error) return;
        const uint64_t end = (uint64_t)top.hdr + top.len;
        need(end, 8 + kIndexHeaderBytes);
        FragmentIndex ix;
        if (locate_fragment_index(p, (uint32_t)bytes, ix)) need(ix.body, (uint64_t)kIndexHeaderBytes + 4ull * ((uint64_t)ix.chunks[0] + ix.chunks[1]));
    }
};

struct WorkState {
    std::atomic<unsigned> claimed{0};
};
void work_function(void *p, unsigned int)
{
    // every chunk was submitted to the GPU before the callback ran (hap.h contract: the callee calls
    // this once per chunk, from any threads, and returns when all calls returned)
    reinterpret_cast<WorkState *>(p)->claimed.fetch_add(1, std::memory_order_relaxed);
}

}  // namespace

// ---- delivery rings: helpers ----
namespace {
struct OnDevice {      // the calling thread's device for the duration of one ring call
    int saved = -1;
    bool ok = false;
    explicit OnDevice(int device)
    {
        if (device < 0 || device >= kMaxDevices || cudaGetDevice(&saved) != cudaSuccess) { cudaGetLastError(); return; }
        ok = device == saved || cudaSetDevice(device) == cudaSuccess;
        if (ok) { std::call_once(g_dev[device].once, device_init, device); ok = g_dev[device].ready; }
        if (!ok) cudaGetLastError();
    }
    ~OnDevice()
    {
        int cur = -1;
        if (saved >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != saved) cudaSetDevice(saved);
        cudaGetLastError();
    }
};
__global__ void ring_publish_kernel(unsigned int *flag, unsigned int value)
{
    // the kernels queued before this one have completed, their stores to the peer are performed; the fence orders this
    // thread's view, the release store makes the flag the last thing the consumer can see
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}
__global__ void ring_wait_kernel(const unsigned int *flag, unsigned int value, unsigned long long timeout_ns)
{
    unsigned int v;
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int)(v - value) >= 0) break;
        hap_nanosleep(500);
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (timeout_ns && t1 - t0 > timeout_ns) break;     // a producer that died must not hang the consumer's GPU for ever
    }
}
}  // namespace


// =====================================================================================================
extern "C" {

const char *HapB200Version(void) { return "hap-b200 0.1 (sm_100a)"; }
unsigned long long HapB200KernelLaunchCount(void) { return g_launches.load(); }

// The device host-pointer calls run on (device-pointer calls run where their buffers live).  -1: forget it; the next
// host-pointer call takes its thread's current device.
int HapB200SetDevice(int device)
{
    if (device < -1 || device >= kMaxDevices) return -1;
    g_default_device.store(device);
    return 0;
}
int HapB200GetDevice(void) { return g_default_device.load(); }

// ---- delivery rings (include/hap_b200.h) ---------------------------------------------------------------------------
unsigned int HapB200RingCreate(int device, unsigned long bytes, void **ring, void *handle)
{
    if (!ring || bytes == 0) return HapResult_Bad_Arguments;
    OnDevice on(device);
    if (!on.ok) return HapResult_Internal_Error;
    void *p = nullptr;
    // plain cudaMalloc: memory of a stream-ordered pool cannot be exported
    if (cudaMalloc(&p, bytes) != cudaSuccess || cudaMemset(p, 0, bytes) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
        cudaGetLastError();
        if (p) cudaFree(p);
        return HapResult_Internal_Error;
    }
    if (handle) {
        static_assert(sizeof(cudaIpcMemHandle_t) == HAPB200_RING_HANDLE_BYTES, "handle size");
        cudaIpcMemHandle_t h;
        if (cudaIpcGetMemHandle(&h, p) != cudaSuccess) { cudaGetLastError(); cudaFree(p); return HapResult_Internal_Error; }
        memcpy(handle, &h, sizeof h);
    }
    *ring = p;
    return HapResult_No_Error;
}

unsigned int HapB200RingDestroy(int device, void *ring)
{
    if (!ring) return HapResult_Bad_Arguments;
    OnDevice on(device);
    if (!on.ok) return HapResult_Internal_Error;
    cudaDeviceSynchronize();
    const bool ok = cudaFree(ring) == cudaSuccess;
    cudaGetLastError();
    return ok ? HapResult_No_Error : HapResult_Internal_Error;
}

unsigned int HapB200RingOpen(int device, const void *handle, void **ring)
{
    if (!handle || !ring) return HapResult_Bad_Arguments;
    OnDevice on(device);
    if (!on.ok) return HapResult_Internal_Error;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    void *p = nullptr;
    if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
    *ring = p;
    return HapResult_No_Error;
}

unsigned int HapB200RingClose(int device, void *ring)
{
    if (!ring) return HapResult_Bad_Arguments;
    OnDevice on(device);
    if (!on.ok) return HapResult_Internal_Error;
    cudaDeviceSynchronize();
    const bool ok = cudaIpcCloseMemHandle(ring) == cudaSuccess;
    cudaGetLastError();
    return ok ? HapResult_No_Error : HapResult_Internal_Error;
}

unsigned int HapB200RingAttach(int device, int ringDevice)
{
    if (ringDevice < 0 || ringDevice >= kMaxDevices) return HapResult_Bad_Arguments;
    if (device == ringDevice) return HapResult_No_Error;
    OnDevice on(device);
    if (!on.ok) return HapResult_Internal_Error;
    int can = 0;
    if (cudaDeviceCanAccessPeer(&can, device, ringDevice) != cudaSuccess || !can) { cudaGetLastError(); return HapResult_Internal_Error; }
    const cudaError_t e = cudaDeviceEnablePeerAccess(ringDevice, 0);
    cudaGetLastError();
    return (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) ? HapResult_No_Error : HapResult_Internal_Error;
}

unsigned int HapB200RingPublish(int device, void *flag, unsigned int value, void *stream)
{
    if (!flag || ((uintptr_t)flag & 3)) return HapResult_Bad_Arguments;
    OnDevice on(device);
    if (!on.ok) return HapResult_Internal_Error;
    cudaStream_t st = stream ? (cudaStream_t)stream : kLegacyStream;
    ring_publish_kernel<<<1, 1, 0, st>>>((unsigned int *)flag, value);
    g_launches.fetch_add(1);
    return cudaGetLastError() == cudaSuccess ? HapResult_No_Error : HapResult_Internal_Error;
}

unsigned int HapB200RingWait(int device, const void *flag, unsigned int value, unsigned int timeoutMs, void *stream)
{
    if (!flag || ((uintptr_t)flag & 3)) return HapResult_Bad_Arguments;
    OnDevice on(device);
    if (!on.ok) return HapResult_Internal_Error;
    cudaStream_t st = stream ? (cudaStream_t)stream : kLegacyStream;
    if (timeoutMs == 0) {
        // No timeout asked for: a stream memory operation of the driver (cuStreamWaitValue32, "flag - value >= 0" compared as
        // signed), which holds the stream WITHOUT occupying an SM.  (A polling kernel resident on one SM keeps the encoder's
        // one-CTA-per-SM fragment kernel from getting that SM: measured, a third more time per step.)
        typedef int (*WaitValue32)(cudaStream_t, unsigned long long, unsigned int, unsigned int);
        static WaitValue32 wait_value = [] {
            void *fn = nullptr;
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) { cudaGetLastError(); fn = nullptr; }
            return (WaitValue32)fn;
        }();
        if (wait_value && wait_value(st, (unsigned long long)(uintptr_t)flag, value, 0u /* CU_STREAM_WAIT_VALUE_GEQ */) == 0) return HapResult_No_Error;
        // (driver without stream memory operations: the polling kernel below, waiting for ever)
    }
    ring_wait_kernel<<<1, 1, 0, st>>>((const unsigned int *)flag, value, 1000000ull * timeoutMs);
    g_launches.fetch_add(1);
    return cudaGetLastError() == cudaSuccess ? HapResult_No_Error : HapResult_Internal_Error;
}

// Options.  HAPB200_OPTION_USE_INDEX (1): decoder uses a frame's embedded fragment index (default 1).
// HAPB200_OPTION_WRITE_INDEX (2): encoder writes the fragment index section (default: see g_write_index).
int HapB200SetOption(int option, int value)
{
    if (option == 1) { g_use_index.store(value != 0); return 0; }
    if (option == 2) { g_write_index.store(value != 0); return 0; }
    if (option == 3) { g_write_offsets.store(value != 0); return 0; }
    if (option == 4) { g_chroma_refine.store(value != 0); return 0; }
    return -1;
}

void HapB200SetStageTiming(int enabled)
{
    std::lock_guard<std::mutex> l(g_timer.mu);
    g_timer.on = enabled != 0;
}

// Synchronises the device, folds the recorded events into per-stage totals and returns them:
// ms[i], launches[i] for i < n (stage order: bc_encode, snappy_encode, plan, place, parse, snappy_decode,
// collect, bc_decode).  Totals are reset by the call.
int HapB200StageTimes(double *ms, unsigned long long *launches, int n)
{
    cudaDeviceSynchronize();
    std::lock_guard<std::mutex> l(g_timer.mu);
    for (auto &r : g_timer.recs) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) { g_timer.ms[r.stage] += t; g_timer.n[r.stage]++; }
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    g_timer.recs.clear();
    for (int i = 0; i < n && i < kStCount; i++) { ms[i] = g_timer.ms[i]; launches[i] = g_timer.n[i]; }
    for (int i = 0; i < kStCount; i++) { g_timer.ms[i] = 0; g_timer.n[i] = 0; }
    cudaGetLastError();
    return kStCount;
}

// hap.c:324-353
unsigned long HapMaxEncodedLength(unsigned int count, unsigned long *lengths, unsigned int *textureFormats,
                                  unsigned int *chunkCounts)
{
    if (count == 0 || count > 2 || !lengths || !textureFormats || !chunkCounts) return 0;
    unsigned long total = 8;
    for (unsigned i = 0; i < count; i++) {
        if (chunkCounts[i] == 0) return 0;
        total += (unsigned long)max_encoded_length_one(lengths[i], textureFormats[i], HapCompressorSnappy, chunkCounts[i]);
    }
    return total;
}

// hap.c:1042-1087
unsigned int HapGetFrameTextureCount(const void *inputBuffer, unsigned long inputBufferBytes, unsigned int *outputTextureCount)
{
    HeaderView hv(inputBuffer, inputBufferBytes);
    if (!hv.ok) return HapResult_Internal_Error;
    const uint8_t *in = hv.p;
    Section top;
    uint32_t r = read_section_header(in, (uint32_t)inputBufferBytes, top);
    if (r != HapResult_No_Error) return r;
    if (top.type != kSecMultipleImages) { *outputTextureCount = 1; return HapResult_No_Error; }
    uint32_t off = top.hdr;
    *outputTextureCount = 0;
    while (off < top.len) {  // hap.c:1064 compares against the body length, as here
        Section s;
        if (!hv.need(off, 8)) return HapResult_Internal_Error;
        r = read_section_header(in + off, (uint32_t)(inputBufferBytes - off), s);
        if (r != HapResult_No_Error) return r;
        off += s.hdr + s.len;
        *outputTextureCount += 1;
    }
    return HapResult_No_Error;
}

// hap.c:1089-1126
unsigned int HapGetFrameTextureFormat(const void *inputBuffer, unsigned long inputBufferBytes, unsigned int index,
                                      unsigned int *outputBufferTextureFormat)
{
    if (!inputBuffer || index > 1 || !outputBufferTextureFormat) return HapResult_Bad_Arguments;
    HeaderView hv(inputBuffer, inputBufferBytes);
    if (!hv.ok) return HapResult_Internal_Error;
    Located loc;
    uint32_t r = hv.locate(index, loc);
    if (r != HapResult_No_Error) return r;
    *outputBufferTextureFormat = format_from_nibble(loc.type & 0xF);
    return *outputBufferTextureFormat ? HapResult_No_Error : HapResult_Bad_Frame;
}

// hap.c:1128-1188
unsigned int HapGetFrameTextureChunkCount(const void *inputBuffer, unsigned long inputBufferBytes, unsigned int index,
                                          int *chunk_count)
{
    *chunk_count = 0;  // before validation, like hap.c:1134
    if (!inputBuffer || index > 1) return HapResult_Bad_Arguments;
    HeaderView hv(inputBuffer, inputBufferBytes);
    if (!hv.ok) return HapResult_Internal_Error;
    Located loc;
    uint32_t r = hv.locate(index, loc);
    if (r != HapResult_No_Error) return r;
    const uint32_t compressor = (loc.type >> 4) & 0xF;
    if (compressor == kHapComplex) {
        ChunkTables t;
        t.count = 0;
        hv.need_tables(loc);
        if (!hv.ok) return HapResult_Internal_Error;
        r = parse_decode_instructions(hv.p + loc.offset, loc.len, t);
        *chunk_count = t.count;
        return r;
    }
    if (compressor == kHapChunkSnappy || compressor == kHapChunkRaw) { *chunk_count = 1; return HapResult_No_Error; }
    return HapResult_Bad_Frame;
}

// hap.c:506-604 + :355-504
unsigned int HapEncode(unsigned int count, const void **inputBuffers, unsigned long *inputBuffersBytes,
                       unsigned int *textureFormats, unsigned int *compressors, unsigned int *chunkCounts,
                       void *outputBuffer, unsigned long outputBufferBytes, unsigned long *outputBufferBytesUsed)
{
    if (count == 0 || count > 2 || !inputBuffers || !inputBuffersBytes || !textureFormats || !compressors || !chunkCounts ||
        !outputBuffer || outputBufferBytes == 0 || !outputBufferBytesUsed)
        return HapResult_Bad_Arguments;
    for (unsigned i = 0; i < count; i++)
        if (chunkCounts[i] == 0) return HapResult_Bad_Arguments;
    if (count == 2 && textureFormats[0] != HapFmt_YCoCg_DXT5 && textureFormats[1] != HapFmt_YCoCg_DXT5 &&
        textureFormats[0] != HapFmt_A_RGTC1 && textureFormats[1] != HapFmt_A_RGTC1)
        return HapResult_Bad_Arguments;  // hap.c:551-559 (SURVEY.md Q5)

    TextureArgs ta[2];
    for (unsigned i = 0; i < count; i++) ta[i] = TextureArgs{inputBuffersBytes[i], textureFormats[i], compressors[i], chunkCounts[i]};
    // hap.c:563-576: outer header from the worst case, with the REQUESTED chunk counts (SURVEY.md Q6)
    uint64_t outer = 0;
    if (count == 2) {
        uint64_t worst = 0;
        for (unsigned i = 0; i < 2; i++) worst += ta[i].bytes + decode_instructions_length(ta[i].chunks) + 4;
        outer = worst > kU24Max ? 8 : 4;
    }
    // Errors surface in texture order: the reference encodes texture 0 completely before it looks at
    // texture 1 (hap.c:580-596).  The capacity test of texture 1 is made against what section 0 really
    // used (hap.c:589), which is only known after compression: checked further down.
    if (!inputBuffers[0] || validate_texture_args(ta[0]) != HapResult_No_Error) return HapResult_Bad_Arguments;
    if (outputBufferBytes < outer ||
        outputBufferBytes - outer < max_encoded_length_one(ta[0].bytes, ta[0].format, ta[0].compressor, ta[0].chunks))
        return HapResult_Buffer_Too_Small;
    if (count == 2 && (!inputBuffers[1] || validate_texture_args(ta[1]) != HapResult_No_Error)) return HapResult_Bad_Arguments;
    FrameGeom G;
    {
        uint32_t gr = build_frame_geom(count, ta, G);
        if (gr != HapResult_No_Error) return gr;
    }

    bool all_host_verbatim = !is_device_pointer(outputBuffer);
    for (unsigned i = 0; i < count; i++)
        all_host_verbatim = all_host_verbatim && ta[i].compressor == HapCompressorNone && !is_device_pointer(inputBuffers[i]);
    if (all_host_verbatim) {
        // hap.c:490-501 for every texture: headers plus a copy, nothing to compute and nothing for a GPU to do
        uint8_t *o = (uint8_t *)outputBuffer;
        uint64_t pos = outer;
        for (unsigned i = 0; i < count; i++) {
            const uint32_t hdr = G.s[i].top_hdr;
            if (i == 1 && (outputBufferBytes < pos ||
                           outputBufferBytes - pos < max_encoded_length_one(ta[1].bytes, ta[1].format, ta[1].compressor, ta[1].chunks)))
                return HapResult_Buffer_Too_Small;
            uint8_t h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            const uint32_t len = (uint32_t)ta[i].bytes;
            if (hdr == 4) { h[0] = (uint8_t)len; h[1] = (uint8_t)(len >> 8); h[2] = (uint8_t)(len >> 16); }
            else { h[4] = (uint8_t)len; h[5] = (uint8_t)(len >> 8); h[6] = (uint8_t)(len >> 16); h[7] = (uint8_t)(len >> 24); }
            h[3] = (uint8_t)((kHapChunkRaw << 4) | G.s[i].fmt_nibble);
            memcpy(o + pos, h, hdr);
            memcpy(o + pos + hdr, inputBuffers[i], ta[i].bytes);
            pos += hdr + ta[i].bytes;
        }
        if (count == 2) {
            const uint32_t len = (uint32_t)(pos - outer);
            uint8_t h[8] = {0, 0, 0, (uint8_t)kSecMultipleImages, 0, 0, 0, 0};
            if (outer == 4) { h[0] = (uint8_t)len; h[1] = (uint8_t)(len >> 8); h[2] = (uint8_t)(len >> 16); }
            else { h[4] = (uint8_t)len; h[5] = (uint8_t)(len >> 8); h[6] = (uint8_t)(len >> 16); h[7] = (uint8_t)(len >> 24); }
            memcpy(o, h, outer);
        }
        *outputBufferBytesUsed = (unsigned long)pos;
        return HapResult_No_Error;
    }

    HAP_ENTER(outputBuffer, inputBuffers[0], count == 2 ? inputBuffers[1] : nullptr);
    bool enc_all_host = !is_device_pointer(outputBuffer);
    for (unsigned i = 0; i < count; i++) enc_all_host = enc_all_host && !is_device_pointer(inputBuffers[i]);
    CallStream call(enc_all_host);
    cudaStream_t st = call.st;

    // worst-case frame in device scratch; textures staged into 16-byte aligned device memory
    unsigned long lens[2] = {ta[0].bytes, count == 2 ? ta[1].bytes : 0};
    unsigned fmts[2] = {ta[0].format, ta[1].format}, chunks[2] = {ta[0].chunks, ta[1].chunks};
    const unsigned long cap = HapMaxEncodedLength(count, lens, fmts, chunks);
    DevBuf tex(st), frame(st), used(st);
    const uint64_t off1 = align16(ta[0].bytes);
    const uint64_t tex_bytes = off1 + (count == 2 ? align16(ta[1].bytes) : 0) + 16;
    if (!tex.alloc(tex_bytes) || !frame.alloc(cap) || !used.alloc(sizeof(unsigned long long) * 4)) { cudaGetLastError(); return HapResult_Internal_Error; }
    for (unsigned i = 0; i < count; i++) {
        uint8_t *d = tex.as<uint8_t>() + (i ? off1 : 0);
        cudaMemcpyKind kind = is_device_pointer(inputBuffers[i]) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        if (cudaMemcpyAsync(d, inputBuffers[i], ta[i].bytes, kind, st) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
        G.s[i].in_offset = i ? off1 : 0;
        G.s[i].in_stride = 0;
    }
    uint32_t r = launch_encode(tex.as<uint8_t>(), G, 1, frame.as<uint8_t>(), cap, used.as<unsigned long long>(), st);
    if (r != HapResult_No_Error) return r;
    unsigned long long total = 0;
    if (cudaMemcpyAsync(&total, used.p, sizeof total, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
    if (total > outputBufferBytes) return HapResult_Buffer_Too_Small;
    if (count == 2) {
        // hap.c:589: capacity left for texture 1 = outputBufferBytes - (outer header + actual section 0)
        Section s0;
        uint8_t head[16];
        if (cudaMemcpy(head, frame.as<uint8_t>() + outer, 8, cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
        if (read_section_header(head, 0xFFFFFFFFu, s0) == HapResult_No_Error) {
            uint64_t before = outer + s0.hdr + s0.len;
            if (outputBufferBytes < before ||
                outputBufferBytes - before < max_encoded_length_one(ta[1].bytes, ta[1].format, ta[1].compressor, ta[1].chunks))
                return HapResult_Buffer_Too_Small;
        }
    }
    cudaMemcpyKind okind = is_device_pointer(outputBuffer) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    if (cudaMemcpyAsync(outputBuffer, frame.p, total, okind, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) {
        cudaGetLastError();
        return HapResult_Internal_Error;
    }
    *outputBufferBytesUsed = (unsigned long)total;
    return HapResult_No_Error;
}

// hap.c:993-1040 + :732-930
unsigned int HapDecode(const void *inputBuffer, unsigned long inputBufferBytes, unsigned int index,
                       HapDecodeCallback callback, void *info, void *outputBuffer, unsigned long outputBufferBytes,
                       unsigned long *outputBufferBytesUsed, unsigned int *outputBufferTextureFormat)
{
    if (!inputBuffer || index > 1 || !callback || !outputBuffer || !outputBufferTextureFormat) return HapResult_Bad_Arguments;
    const bool in_dev = is_device_pointer(inputBuffer), out_dev = is_device_pointer(outputBuffer);
    HeaderView hv(inputBuffer, inputBufferBytes);
    if (!hv.ok) return HapResult_Internal_Error;
    const uint8_t *frame = hv.p;
    Located loc;
    uint32_t r = hv.locate(index, loc);
    if (r != HapResult_No_Error) return r;
    const uint8_t *sec = frame + loc.offset;
    const uint32_t compressor = (loc.type >> 4) & 0xF;
    *outputBufferTextureFormat = format_from_nibble(loc.type & 0xF);
    if (*outputBufferTextureFormat == 0) return HapResult_Bad_Frame;

    struct HostJob { uint32_t src_off, src_bytes, dst_off, dst_bytes, compressor, index_off, index_bytes; };
    std::vector<HostJob> hj;
    uint32_t hv_index_body = 0, hv_index_len = 0;
    uint64_t produced = 0;
    bool whole = false;
    if (compressor == kHapComplex) {
        ChunkTables t;
        t.count = 0;
        hv.need_tables(loc);
        if (!hv.ok) return HapResult_Internal_Error;
        r = parse_decode_instructions(sec, loc.len, t);
        if (r != HapResult_No_Error) return r;
        hv.need_index_header();
        FragmentIndex ix;
        const bool have_ix = locate_fragment_index(frame, (uint32_t)inputBufferBytes, ix);
        if (have_ix) { hv_index_body = ix.body; hv_index_len = ix.len; }
        if (t.count > 0) {
            uint64_t in_run = 0, out_run = 0;
            hj.resize((size_t)t.count);
            for (int i = 0; i < t.count; i++) {
                const uint32_t cc = sec[t.compressors + i];
                const uint32_t sz = rd_le32(sec + t.sizes + 4 * i);
                const uint64_t start = t.data + (t.offsets != 0xFFFFFFFFu ? (uint64_t)rd_le32(sec + t.offsets + 4 * i) : in_run);
                in_run += sz;
                if (start + sz > loc.len) return HapResult_Bad_Frame;  // SURVEY.md Q9: the reference reads out of bounds here
                if (cc == kHapChunkSnappy && !hv.need(loc.offset + start, 5)) return HapResult_Internal_Error;
                uint32_t usz = sz;
                if (cc == kHapChunkSnappy && !snappy_preamble(sec + start, sz, usz)) return HapResult_Bad_Frame;  // hap.c:817-829
                hj[i] = HostJob{(uint32_t)start, sz, 0, usz, (cc == kHapChunkSnappy || cc == kHapChunkRaw) ? cc : 0xFFu, 0, 0};
                if (cc == kHapChunkSnappy && have_ix) fragment_index_record(frame, ix, index, (uint32_t)t.count, (uint32_t)i, hj[i].index_off, hj[i].index_bytes);
                if (out_run > 0xFFFFFFFFull) return HapResult_Buffer_Too_Small;
                hj[i].dst_off = (uint32_t)out_run;
                out_run += usz;
            }
            if (out_run > outputBufferBytes) return HapResult_Buffer_Too_Small;  // hap.c:840-843
            produced = out_run;
        }
    } else if (compressor == kHapChunkSnappy) {
        uint32_t usz = 0;
        if (!hv.need(loc.offset, 5)) return HapResult_Internal_Error;
        if (!snappy_preamble(sec, loc.len, usz)) return HapResult_Internal_Error;  // hap.c:890-894
        if (usz > outputBufferBytes) return HapResult_Buffer_Too_Small;
        hj.push_back(HostJob{0, loc.len, 0, usz, kHapChunkSnappy, 0, 0});
        produced = usz;
        whole = true;
    } else if (compressor == kHapChunkRaw) {
        if (loc.len > outputBufferBytes) return HapResult_Buffer_Too_Small;
        // hap.c:905-916: a verbatim texture is a copy; nothing to compute
        if (!in_dev && !out_dev) {
            memcpy(outputBuffer, sec, loc.len);
        } else {
            HAP_ENTER(inputBuffer, outputBuffer);
            const uint8_t *src = in_dev ? (const uint8_t *)inputBuffer + loc.offset : sec;
            if (cudaMemcpy(outputBuffer, src, loc.len, cudaMemcpyDefault) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
        }
        if (outputBufferBytesUsed) *outputBufferBytesUsed = loc.len;
        return HapResult_No_Error;
    } else {
        return HapResult_Bad_Frame;
    }

    if (!hj.empty()) {
        HAP_ENTER(inputBuffer, outputBuffer);
        CallStream call(!in_dev && !out_dev);
        cudaStream_t st = call.st;
        DevBuf din(st), dout(st), djobs(st);
        const uint8_t *dsec;
        const uint8_t *dindex = nullptr;    // device address of byte 0 of the fragment index body (hap_index.h), when the frame has one
        bool any_index = false;
        for (auto &h : hj) any_index = any_index || h.index_bytes != 0;
        if (in_dev) {
            dsec = (const uint8_t *)inputBuffer + loc.offset;
            if (any_index) dindex = (const uint8_t *)inputBuffer + hv_index_body;
        } else {
            // the texture section, and behind it (16-byte aligned) the body of the frame's trailing index section
            const uint64_t ioff = align16(loc.len);
            if (!din.alloc(ioff + (any_index ? hv_index_len : 0)) || cudaMemcpyAsync(din.p, sec, loc.len, cudaMemcpyHostToDevice, st) != cudaSuccess ||
                (any_index && cudaMemcpyAsync(din.as<uint8_t>() + ioff, frame + hv_index_body, hv_index_len, cudaMemcpyHostToDevice, st) != cudaSuccess)) {
                cudaGetLastError();
                return HapResult_Internal_Error;
            }
            dsec = din.as<uint8_t>();
            if (any_index) dindex = din.as<uint8_t>() + ioff;
        }
        uint8_t *ddst;
        if (out_dev) ddst = (uint8_t *)outputBuffer;
        else {
            if (!dout.alloc(produced)) { cudaGetLastError(); return HapResult_Internal_Error; }
            ddst = dout.as<uint8_t>();
        }
        std::vector<ChunkJob> jobs(hj.size());
        uint64_t in_sum = 0;
        for (size_t i = 0; i < hj.size(); i++) {
            jobs[i].src = dsec + hj[i].src_off;
            jobs[i].dst = ddst + hj[i].dst_off;
            jobs[i].src_bytes = hj[i].src_bytes;
            jobs[i].dst_bytes = hj[i].dst_bytes;
            jobs[i].compressor = hj[i].compressor;
            jobs[i].status = HapResult_Internal_Error;
            jobs[i].index = hj[i].index_bytes ? dindex + (hj[i].index_off - hv_index_body) : nullptr;
            jobs[i].index_bytes = hj[i].index_bytes;
            jobs[i].mode = kJobUndecided;
            jobs[i].win_base = 0;
            jobs[i].win_count = 0;
            in_sum += hj[i].src_bytes;
        }
        if (!djobs.alloc(jobs.size() * sizeof(ChunkJob)) ||
            cudaMemcpyAsync(djobs.p, jobs.data(), jobs.size() * sizeof(ChunkJob), cudaMemcpyHostToDevice, st) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
        DecodePasses passes(st);
        r = passes.first(djobs.as<ChunkJob>(), (uint32_t)jobs.size(), in_sum, produced);
        if (r != HapResult_No_Error) return r;
        if (compressor == kHapComplex && jobs.size() > 1) {
            WorkState ws;
            callback(work_function, &ws, (unsigned)jobs.size(), info);  // hap.c:861
        }
        if (cudaMemcpyAsync(jobs.data(), djobs.p, jobs.size() * sizeof(ChunkJob), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
        bool mismatch = false;     // a chunk whose embedded index failed the execute kernel's checks: the repair pass, then the statuses again
        for (size_t i = 0; i < jobs.size(); i++) mismatch = mismatch || jobs[i].status == kStatusIndexMismatch;
        if (mismatch) {
            r = passes.repair();
            if (r != HapResult_No_Error) return r;
            if (cudaMemcpyAsync(jobs.data(), djobs.p, jobs.size() * sizeof(ChunkJob), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
        }
        for (size_t i = 0; i < jobs.size(); i++)
            if (jobs[i].status != HapResult_No_Error) return whole ? (uint32_t)HapResult_Internal_Error : jobs[i].status;  // hap.c:867-875, :899-903
        if (!out_dev && produced) {
            if (cudaMemcpyAsync(outputBuffer, ddst, produced, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
        }
    }
    if (outputBufferBytesUsed) *outputBufferBytesUsed = (unsigned long)produced;
    return HapResult_No_Error;
}

// ---- extensions ----------------------------------------------------------------------------------

unsigned long HapB200TextureBytes(unsigned int width, unsigned int height, unsigned int codec, unsigned int index)
{
    CodecInfo ci;
    if (!codec_info(codec, ci) || index >= ci.textures || width % 4 || height % 4) return 0;
    return (unsigned long)(width / 4) * (height / 4) * ci.block_bytes[index];
}

unsigned long HapB200MaxEncodedLengthRGBA(unsigned int width, unsigned int height, unsigned int codec, unsigned int chunkCount)
{
    CodecInfo ci;
    if (!codec_info(codec, ci)) return 0;
    unsigned long lens[2] = {HapB200TextureBytes(width, height, codec, 0), HapB200TextureBytes(width, height, codec, 1)};
    unsigned fmts[2] = {ci.fmt[0], ci.fmt[1]}, chunks[2] = {chunkCount, chunkCount};
    if (lens[0] == 0) return 0;
    return HapMaxEncodedLength(ci.textures, lens, fmts, chunks);
}

unsigned int HapB200BlockEncodeBatch(const void *rgba, unsigned int frames, unsigned long frameStride, unsigned int width,
                                     unsigned int height, unsigned long rowBytes, unsigned int codec, void *blocks,
                                     unsigned long blocksStride, void *stream)
{
    CodecInfo ci;
    if (!rgba || !blocks || frames == 0 || !codec_info(codec, ci) || width == 0 || height == 0 || width % 4 || height % 4 ||
        rowBytes < 4ul * width || rowBytes % 16 || ((uintptr_t)rgba | (uintptr_t)blocks | frameStride | blocksStride) % 16)
        return HapResult_Bad_Arguments;
    HAP_ENTER(rgba, blocks);
    cudaStream_t st = stream ? (cudaStream_t)stream : kLegacyStream;
    uint32_t r = launch_block_encode((const uint8_t *)rgba, frames, frameStride, width, height, rowBytes, ci, (uint8_t *)blocks,
                                     blocksStride, HapB200TextureBytes(width, height, codec, 0), st);
    if (r == HapResult_No_Error && !stream && cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); r = HapResult_Internal_Error; }
    return r;
}

unsigned int HapB200BlockDecodeBatch(const void *blocks, unsigned int frames, unsigned long blocksStride, unsigned int width,
                                     unsigned int height, unsigned int codec, void *rgba, unsigned long frameStride,
                                     unsigned long rowBytes, void *stream)
{
    CodecInfo ci;
    if (!rgba || !blocks || frames == 0 || !codec_info(codec, ci) || width == 0 || height == 0 || width % 4 || height % 4 ||
        rowBytes < 4ul * width || rowBytes % 16 || ((uintptr_t)rgba | (uintptr_t)blocks | frameStride | blocksStride) % 16)
        return HapResult_Bad_Arguments;
    HAP_ENTER(blocks, rgba);
    cudaStream_t st = stream ? (cudaStream_t)stream : kLegacyStream;
    const uint8_t *b = (const uint8_t *)blocks;
    uint32_t r = launch_block_decode(b, b + HapB200TextureBytes(width, height, codec, 0), frames, blocksStride, blocksStride, width,
                                     height, ci, (uint8_t *)rgba, frameStride, rowBytes, st);
    if (r == HapResult_No_Error && !stream && cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); r = HapResult_Internal_Error; }
    return r;
}

unsigned int HapB200EncodeBatch(unsigned int count, const void **textures, unsigned long *textureStrides,
                                unsigned long *textureBytes, unsigned int *textureFormats, unsigned int *compressors,
                                unsigned int *chunkCounts, unsigned int frames, void *out, unsigned long outStride,
                                unsigned long long *used, void *stream)
{
    if (count == 0 || count > 2 || !textures || !textureStrides || !textureBytes || !textureFormats || !compressors ||
        !chunkCounts || frames == 0 || !out || !used)
        return HapResult_Bad_Arguments;
    TextureArgs ta[2];
    for (unsigned i = 0; i < count; i++) {
        if (chunkCounts[i] == 0 || !textures[i] || ((uintptr_t)textures[i] | textureStrides[i]) % 16) return HapResult_Bad_Arguments;
        ta[i] = TextureArgs{textureBytes[i], textureFormats[i], compressors[i], chunkCounts[i]};
        if (validate_texture_args(ta[i]) != HapResult_No_Error) return HapResult_Bad_Arguments;
    }
    if (count == 2 && textureFormats[0] != HapFmt_YCoCg_DXT5 && textureFormats[1] != HapFmt_YCoCg_DXT5 &&
        textureFormats[0] != HapFmt_A_RGTC1 && textureFormats[1] != HapFmt_A_RGTC1)
        return HapResult_Bad_Arguments;
    if (outStride < HapMaxEncodedLength(count, textureBytes, textureFormats, chunkCounts)) return HapResult_Buffer_Too_Small;
    FrameGeom G;
    uint32_t r = build_frame_geom(count, ta, G);
    if (r != HapResult_No_Error) return r;
    HAP_ENTER(out, textures[0]);
    cudaStream_t st = stream ? (cudaStream_t)stream : kLegacyStream;
    const uint8_t *base = (const uint8_t *)textures[0];
    for (unsigned i = 0; i < count; i++) {
        G.s[i].in_offset = (uint64_t)((const uint8_t *)textures[i] - base);  // wraps for i = 1 when below base; 64-bit add undoes it
        G.s[i].in_stride = textureStrides[i];
    }
    r = launch_encode(base, G, frames, (uint8_t *)out, outStride, used, st);
    if (r == HapResult_No_Error && !stream && cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); r = HapResult_Internal_Error; }
    return r;
}

unsigned int HapB200EncodeRGBABatch(const void *rgba, unsigned int frames, unsigned long frameStride, unsigned int width,
                                    unsigned int height, unsigned long rowBytes, unsigned int codec, unsigned int compressor,
                                    unsigned int chunkCount, void *out, unsigned long outStride, unsigned long long *used,
                                    void *stream)
{
    CodecInfo ci;
    if (!rgba || !out || !used || frames == 0 || chunkCount == 0 || !codec_info(codec, ci) || width == 0 || height == 0 ||
        width % 4 || height % 4 || rowBytes < 4ul * width || rowBytes % 16 || ((uintptr_t)rgba | frameStride) % 16 ||
        (compressor != HapCompressorNone && compressor != HapCompressorSnappy))
        return HapResult_Bad_Arguments;
    if (outStride < HapB200MaxEncodedLengthRGBA(width, height, codec, chunkCount)) return HapResult_Buffer_Too_Small;
    HAP_ENTER(rgba, out);
    cudaStream_t st = stream ? (cudaStream_t)stream : kLegacyStream;
    const uint64_t t0 = HapB200TextureBytes(width, height, codec, 0), t1 = HapB200TextureBytes(width, height, codec, 1);
    const uint64_t dxt_stride = align16(t0) + align16(t1);
    DevBuf dxt(st);
    if (!dxt.alloc(dxt_stride * frames + 16)) { cudaGetLastError(); return HapResult_Internal_Error; }
    uint32_t r = launch_block_encode((const uint8_t *)rgba, frames, frameStride, width, height, rowBytes, ci, dxt.as<uint8_t>(),
                                     dxt_stride, align16(t0), st);
    if (r != HapResult_No_Error) return r;
    TextureArgs ta[2] = {{t0, ci.fmt[0], compressor, chunkCount}, {t1, ci.fmt[1], compressor, chunkCount}};
    FrameGeom G;
    r = build_frame_geom(ci.textures, ta, G);
    if (r != HapResult_No_Error) return r;
    for (unsigned i = 0; i < ci.textures; i++) {
        G.s[i].in_offset = i ? align16(t0) : 0;
        G.s[i].in_stride = dxt_stride;
    }
    r = launch_encode(dxt.as<uint8_t>(), G, frames, (uint8_t *)out, outStride, used, st);
    if (r == HapResult_No_Error && !stream && cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); r = HapResult_Internal_Error; }
    return r;
}

unsigned int HapB200EncodeRGBA(const void *rgba, unsigned int width, unsigned int height, unsigned long rowBytes,
                               unsigned int codec, unsigned int compressor, unsigned int chunkCount, void *outputBuffer,
                               unsigned long outputBufferBytes, unsigned long *outputBufferBytesUsed)
{
    CodecInfo ci;
    if (!rgba || !outputBuffer || !outputBufferBytesUsed || chunkCount == 0 || !codec_info(codec, ci) || width == 0 ||
        height == 0 || width % 4 || height % 4 || rowBytes < 4ul * width ||
        (compressor != HapCompressorNone && compressor != HapCompressorSnappy))
        return HapResult_Bad_Arguments;
    const unsigned long cap = HapB200MaxEncodedLengthRGBA(width, height, codec, chunkCount);
    if (outputBufferBytes < cap) return HapResult_Buffer_Too_Small;
    HAP_ENTER(rgba, outputBuffer);
    CallStream call(!is_device_pointer(rgba) && !is_device_pointer(outputBuffer));
    cudaStream_t st = call.st;
    DevBuf img(st), frame(st), used(st);
    const uint64_t tight = 4ull * width;
    if (!img.alloc(tight * height) || !frame.alloc(cap) || !used.alloc(32)) { cudaGetLastError(); return HapResult_Internal_Error; }
    if (cudaMemcpy2DAsync(img.p, tight, rgba, rowBytes, tight, height, cudaMemcpyDefault, st) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
    uint32_t r = HapB200EncodeRGBABatch(img.p, 1, align16(tight * height), width, height, tight, codec, compressor, chunkCount,
                                        frame.p, cap, used.as<unsigned long long>(), st);
    if (r != HapResult_No_Error) return r;
    unsigned long long total = 0;
    if (cudaMemcpyAsync(&total, used.p, sizeof total, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess ||
        total > outputBufferBytes || cudaMemcpyAsync(outputBuffer, frame.p, total, cudaMemcpyDefault, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }
    *outputBufferBytesUsed = (unsigned long)total;
    return HapResult_No_Error;
}

unsigned int HapB200DecodeBatch(const void *in, unsigned int frames, unsigned long inStride, const unsigned long long *inBytes,
                                unsigned int index, unsigned int maxChunks, void *out, unsigned long outStride,
                                unsigned long long *used, unsigned int *formats, unsigned int *results, void *stream)
{
    if (!in || !inBytes || !out || !used || !formats || !results || frames == 0 || maxChunks == 0 || index > 1)
        return HapResult_Bad_Arguments;
    HAP_ENTER(in, out);
    cudaStream_t st = stream ? (cudaStream_t)stream : kLegacyStream;
    uint32_t r = launch_decode_batch((const uint8_t *)in, frames, inStride, inBytes, index, maxChunks, (uint8_t *)out, outStride, outStride,
                                     used, formats, results, st);
    if (r == HapResult_No_Error && !stream && cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); r = HapResult_Internal_Error; }
    return r;
}

unsigned int HapB200DecodeRGBABatch(const void *in, unsigned int frames, unsigned long inStride, const unsigned long long *inBytes,
                                    unsigned int maxChunks, unsigned int codec, unsigned int width, unsigned int height, void *rgba,
                                    unsigned long frameStride, unsigned long rowBytes, unsigned int *results, void *stream)
{
    CodecInfo ci;
    if (!in || !inBytes || !rgba || !results || frames == 0 || maxChunks == 0 || !codec_info(codec, ci) || width == 0 ||
        height == 0 || width % 4 || height % 4 || rowBytes < 4ul * width || rowBytes % 16 || ((uintptr_t)rgba | frameStride) % 16)
        return HapResult_Bad_Arguments;
    HAP_ENTER(in, rgba);
    cudaStream_t st = stream ? (cudaStream_t)stream : kLegacyStream;
    const uint64_t t0 = HapB200TextureBytes(width, height, codec, 0), t1 = HapB200TextureBytes(width, height, codec, 1);
    const uint64_t dxt_stride = align16(t0) + align16(t1);
    DevBuf dxt(st), used(st), formats(st), res1(st);
    if (!dxt.alloc(dxt_stride * frames + 16) || !used.alloc(8ull * frames) || !formats.alloc(4ull * frames) || !res1.alloc(4ull * frames)) {
        cudaGetLastError();
        return HapResult_Internal_Error;
    }
    uint32_t r = HapResult_No_Error;
    for (uint32_t ti = 0; ti < ci.textures && r == HapResult_No_Error; ti++) {
        uint32_t *res = ti == 0 ? results : res1.as<uint32_t>();
        // the decoded size must equal the texture size: offer exactly that much room per frame (the slot stride is
        // wider: both textures of a frame share a slot, so a texture that over-declares its size must not reach its
        // neighbour or the next frame's slot)
        r = launch_decode_batch((const uint8_t *)in, frames, inStride, inBytes, ti, maxChunks, dxt.as<uint8_t>() + (ti ? align16(t0) : 0),
                                dxt_stride, ti ? t1 : t0, used.as<unsigned long long>(), formats.as<uint32_t>(), res, st);
        if (r != HapResult_No_Error) break;
        HAP_KLAUNCH(kStCollect, hap_check_texture_kernel, dim3((frames + 127) / 128), dim3(128), 0, st, frames, used.as<unsigned long long>(),
                    formats.as<uint32_t>(), res, (unsigned long long)(ti ? t1 : t0), ci.fmt[ti], results);
    }
    if (r == HapResult_No_Error)
        r = launch_block_decode(dxt.as<uint8_t>(), dxt.as<uint8_t>() + align16(t0), frames, dxt_stride, dxt_stride, width, height, ci,
                                (uint8_t *)rgba, frameStride, rowBytes, st, results);
    if (r == HapResult_No_Error && !stream && cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); r = HapResult_Internal_Error; }
    return r;
}

unsigned int HapB200DecodeRGBA(const void *inputBuffer, unsigned long inputBufferBytes, unsigned int width, unsigned int height,
                               void *rgba, unsigned long rowBytes)
{
    if (!inputBuffer || !rgba || width == 0 || height == 0 || width % 4 || height % 4 || rowBytes < 4ul * width)
        return HapResult_Bad_Arguments;
    unsigned count = 0, f0 = 0, f1 = 0;
    uint32_t r = HapGetFrameTextureCount(inputBuffer, inputBufferBytes, &count);
    if (r != HapResult_No_Error) return r;
    r = HapGetFrameTextureFormat(inputBuffer, inputBufferBytes, 0, &f0);
    if (r != HapResult_No_Error) return r;
    unsigned codec;
    if (count == 2) {
        r = HapGetFrameTextureFormat(inputBuffer, inputBufferBytes, 1, &f1);
        if (r != HapResult_No_Error) return r;
        if (f0 != HapFmt_YCoCg_DXT5 || f1 != HapFmt_A_RGTC1) return HapResult_Bad_Frame;
        codec = HapB200Codec_HapM;
    } else if (count == 1) {
        codec = f0 == HapFmt_RGB_DXT1 ? HapB200Codec_Hap1 : f0 == HapFmt_RGBA_DXT5 ? HapB200Codec_Hap5 :
                f0 == HapFmt_YCoCg_DXT5 ? HapB200Codec_HapY : f0 == HapFmt_A_RGTC1 ? HapB200Codec_HapA : 99u;
    } else {
        return HapResult_Bad_Frame;
    }
    CodecInfo ci;
    if (!codec_info(codec, ci)) return HapResult_Bad_Frame;  // BPTC frames carry no RGBA decoder here
    HAP_ENTER(inputBuffer, rgba);
    const uint64_t t0 = HapB200TextureBytes(width, height, codec, 0), t1 = HapB200TextureBytes(width, height, codec, 1);
    const uint64_t tight = 4ull * width;
    // scratch from the device's stream-ordered pool on the legacy stream (the nested HapDecode calls below write it on
    // that stream, or on a pooled stream they synchronise before returning): no cudaMalloc/cudaFree, no device-wide sync
    DevBuf dxtb(kLegacyStream), imgb(kLegacyStream);
    if (!dxtb.alloc(align16(t0) + align16(t1) + 16) || !imgb.alloc(tight * height)) { cudaGetLastError(); return HapResult_Internal_Error; }
    void *dxt = dxtb.p, *img = imgb.p;
    if (cudaStreamSynchronize(kLegacyStream) != cudaSuccess) { cudaGetLastError(); return HapResult_Internal_Error; }   // the allocations are real now
    auto serial = [](HapDecodeWorkFunction fn, void *p, unsigned n, void *) { for (unsigned i = 0; i < n; i++) fn(p, i); };
    unsigned long used = 0;
    unsigned fmt = 0;
    r = HapDecode(inputBuffer, inputBufferBytes, 0, serial, nullptr, dxt, t0, &used, &fmt);
    if (r == HapResult_No_Error && used != t0) r = HapResult_Bad_Frame;
    if (r == HapResult_No_Error && count == 2) {
        r = HapDecode(inputBuffer, inputBufferBytes, 1, serial, nullptr, (uint8_t *)dxt + align16(t0), t1, &used, &fmt);
        if (r == HapResult_No_Error && used != t1) r = HapResult_Bad_Frame;
    }
    if (r == HapResult_No_Error) {
        CallStream call(false);  // dxt / img are device buffers filled on the legacy stream by HapDecode above
        cudaStream_t st = call.st;
        r = launch_block_decode((const uint8_t *)dxt, (const uint8_t *)dxt + align16(t0), 1, 0, 0, width, height, ci, (uint8_t *)img,
                                0, tight, st);
        if (r == HapResult_No_Error &&
            (cudaMemcpy2DAsync(rgba, rowBytes, img, tight, tight, height, cudaMemcpyDefault, st) != cudaSuccess ||
             cudaStreamSynchronize(st) != cudaSuccess)) { cudaGetLastError(); r = HapResult_Internal_Error; }
    }
    return r;
}

// ---- include/hap_mov.h: QuickTime sample tables around Hap frames (host code only) -------------------------

unsigned int HapB200MovFourCCForFrame(const void *frame, unsigned long frameBytes, unsigned int *fourcc)
{
    if (!frame || !fourcc) return HapResult_Bad_Arguments;
    unsigned int count = 0, f0 = 0, f1 = 0;
    if (HapGetFrameTextureCount(frame, frameBytes, &count) != HapResult_No_Error || count < 1 || count > 2) return HapResult_Bad_Frame;
    if (HapGetFrameTextureFormat(frame, frameBytes, 0, &f0) != HapResult_No_Error) return HapResult_Bad_Frame;
    if (count == 2 && HapGetFrameTextureFormat(frame, frameBytes, 1, &f1) != HapResult_No_Error) return HapResult_Bad_Frame;
    // HapVideoDRAFT.md:132-142
    char c = 0;
    if (count == 1) {
        switch (f0) {
        case HapTextureFormat_RGB_DXT1: c = '1'; break;
        case HapTextureFormat_RGBA_DXT5: c = '5'; break;
        case HapTextureFormat_YCoCg_DXT5: c = 'Y'; break;
        case HapTextureFormat_A_RGTC1: c = 'A'; break;
        case HapTextureFormat_RGBA_BPTC_UNORM: c = '7'; break;
        case HapTextureFormat_RGB_BPTC_UNSIGNED_FLOAT:
        case HapTextureFormat_RGB_BPTC_SIGNED_FLOAT: c = 'H'; break;
        default: break;
        }
    } else if ((f0 == HapTextureFormat_YCoCg_DXT5 && f1 == HapTextureFormat_A_RGTC1) ||
               (f1 == HapTextureFormat_YCoCg_DXT5 && f0 == HapTextureFormat_A_RGTC1)) {
        c = 'M';
    }
    if (!c) return HapResult_Bad_Frame;
    *fourcc = HAPB200_FOURCC('H', 'a', 'p', c);
    return HapResult_No_Error;
}

HapB200Mov *HapB200MovOpen(const char *path) { return hapmov::open_read(path); }

unsigned int HapB200MovInfo(const HapB200Mov *mov, unsigned int *fourcc, unsigned int *width, unsigned int *height,
                            unsigned long *frameCount, unsigned int *timescale, unsigned long *duration)
{
    if (!mov) return HapResult_Bad_Arguments;
    if (fourcc) *fourcc = mov->fourcc;
    if (width) *width = mov->width;
    if (height) *height = mov->height;
    if (frameCount) *frameCount = (unsigned long)mov->size.size();
    if (timescale) *timescale = mov->timescale;
    if (duration) *duration = (unsigned long)mov->duration;
    return HapResult_No_Error;
}

unsigned long HapB200MovFrameBytes(const HapB200Mov *mov, unsigned long index)
{
    return (mov && index < mov->size.size()) ? mov->size[index] : 0;
}

unsigned int HapB200MovReadFrame(HapB200Mov *mov, unsigned long index, void *buffer, unsigned long bufferBytes,
                                 unsigned long *bytesUsed, unsigned int *durationTicks)
{
    if (!mov || mov->writing || !buffer || index >= mov->size.size()) return HapResult_Bad_Arguments;
    const unsigned long n = mov->size[index];
    if (n > bufferBytes) return HapResult_Buffer_Too_Small;
    if (fseeko(mov->f, (off_t)mov->offset[index], SEEK_SET) != 0 || fread(buffer, 1, n, mov->f) != n) return HapResult_Internal_Error;
    if (bytesUsed) *bytesUsed = n;
    if (durationTicks) *durationTicks = mov->ticks[index];
    return HapResult_No_Error;
}

HapB200Mov *HapB200MovCreate(const char *path, unsigned int fourcc, unsigned int width, unsigned int height, unsigned int timescale)
{
    return hapmov::create(path, fourcc, width, height, timescale);
}

unsigned int HapB200MovWriteFrame(HapB200Mov *mov, const void *frame, unsigned long frameBytes, unsigned int durationTicks)
{
    return hapmov::write_frame(mov, frame, frameBytes, durationTicks);
}

unsigned int HapB200MovClose(HapB200Mov *mov)
{
    if (!mov) return HapResult_No_Error;
    unsigned int r = HapResult_No_Error;
    if (mov->writing) r = hapmov::finish(mov);
    if (mov->f && fclose(mov->f) != 0 && r == HapResult_No_Error) r = HapResult_Internal_Error;
    delete mov;
    return r;
}

}  // extern "C"
