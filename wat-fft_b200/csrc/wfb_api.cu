// wfb_api.cu -- C ABI (include/watfft_b200.h) over the sm_100a kernels of wfb_kernels.cuh.
//
// Plans own: reference-exact twiddle tables (host-built, uploaded once), device buffers laid out
// [batch][row], optional pinned host staging buffers that the JS side wraps as ArrayBuffers, and a
// stream.  There is no CPU path anywhere in this file: without an sm_100 device every call fails.
#include "../../include/watfft_b200.h"
#include "wfb_registry.h"
#include "wfb_twiddle.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <map>
#include <mutex>
#include <set>
#include <utility>
#include <string>
#include <vector>

namespace wfb {

static thread_local char g_cuda_err[256] = "";
static std::atomic<unsigned long long> g_launches{0};

static int cuda_fail(cudaError_t e, const char *what) {
    snprintf(g_cuda_err, sizeof g_cuda_err, "%s: %s", what, cudaGetErrorString(e));
    return WFB_ERR_CUDA;
}
#define CK(call)                                                 \
    do {                                                         \
        cudaError_t e_ = (call);                                 \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call);      \
    } while (0)

// ----------------------------------------------------------------------------------------
// kernel launch helpers (one launch counter and one attribute cache for the whole library)
// ----------------------------------------------------------------------------------------
static std::mutex g_mu;

// Per-launch tile counters of the persistent kernels: a ring of {claims, departures} pairs per device, zeroed once
// when the ring is created.  Every kernel leaves its pair at zero again (claim_epilogue), so nothing has to be cleared
// between launches; a pair would only be reused while still live if 4096 persistent launches were outstanding at once.
static cudaError_t next_counter(unsigned long long **out) {
    enum { RING = 4096 };
    static std::map<int, unsigned long long *> rings;
    static std::map<int, unsigned> heads;
    int dev = 0;
    cudaGetDevice(&dev);
    unsigned long long *ring;
    unsigned idx;
    {
        std::lock_guard<std::mutex> lock(g_mu);
        auto it = rings.find(dev);
        if (it == rings.end()) {
            unsigned long long *r = nullptr;
            cudaError_t e = cudaMalloc(&r, 2 * RING * sizeof(unsigned long long));
            if (e != cudaSuccess) return e;
            // plan streams are non-blocking (they do not order against the legacy stream): finish the clear here
            if ((e = cudaMemset(r, 0, 2 * RING * sizeof(unsigned long long))) != cudaSuccess) return e;
            if ((e = cudaDeviceSynchronize()) != cudaSuccess) return e;
            it = rings.emplace(dev, r).first;
            heads[dev] = 0;
        }
        ring = it->second;
        idx = heads[dev]++ % RING;
    }
    *out = ring + 2 * idx;
    return cudaSuccess;
}

cudaError_t launch(const void *kernel, size_t smem, size_t smem_attr, int threads, long work_items, void *params,
                   unsigned long long **ctr, cudaStream_t s) {
    if (!kernel) return cudaErrorInvalidDeviceFunction;
    static std::set<std::pair<int, const void *>> configured;
    static std::map<std::pair<std::pair<int, const void *>, size_t>, int> resident;    // (device, kernel, smem) -> CTAs on the GPU
    int dev = 0, ctas = 0;
    cudaGetDevice(&dev);
    {
        std::lock_guard<std::mutex> lock(g_mu);
        const auto fk = std::make_pair(dev, kernel);
        if (!configured.count(fk)) {
            // the dynamic-smem attribute is per (device, function); set it once for each pair
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_attr);
            if (e != cudaSuccess) return e;
            // NOTE: forcing cudaSharedmemCarveoutMaxShared was measured (gpurun sweep9) to LOSE 5-15 %: it shrinks
            // L1, which the twiddle tables and the direct-load kernels live in.  The driver's default split stays.
            configured.insert(fk);
        }
        auto it = resident.find(std::make_pair(fk, smem));
        if (it == resident.end()) {
            int per_sm = 0, sms = 0;
            cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem);
            if (e != cudaSuccess) return e;
            if (per_sm < 1) return cudaErrorInvalidConfiguration;      // not even one CTA fits an SM
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            it = resident.emplace(std::make_pair(fk, smem), per_sm * sms).first;
        }
        ctas = it->second;
    }
    long grid = work_items;
    if (ctr) {
        cudaError_t e = next_counter(ctr);
        if (e != cudaSuccess) return e;
        grid = std::min<long>(work_items, ctas);
    }
    void *args[] = {params};
    cudaError_t e = cudaLaunchKernel(kernel, dim3((unsigned)grid), dim3(threads), args, smem, s);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return e != cudaSuccess ? e : cudaGetLastError();
}

// ----------------------------------------------------------------------------------------
// Small-allocation pools.  cudaHostAlloc / cudaMalloc cost 0.1-1 ms each, and the reference's call shape is one small
// context per transform size (createFFT(size), index.js:69-91): a batch-1 plan needs two 4-KB host views, a few KB of
// tables and a completion flag.  Those come out of 4-MiB slabs (pinned + device-mapped + portable host memory; device
// memory per GPU) with per-size free lists; only allocations above SMALL_MAX go to the driver directly.
// ----------------------------------------------------------------------------------------
struct SmallPool {
    enum : size_t { SLAB = 4u << 20, SMALL_MAX = 512u << 10 };      // (a module-sized host arena is 4-8 WASM pages = 256-512 KiB)
    bool host;
    int device;
    char *cur = nullptr;
    size_t left = 0;
    std::map<size_t, std::vector<void *>> free_lists;
    static size_t round(size_t b) { return (b + 255) / 256 * 256; }
    cudaError_t alloc(size_t bytes, void **out) {          // caller holds g_mu
        const size_t r = round(bytes);
        auto it = free_lists.find(r);
        if (it != free_lists.end() && !it->second.empty()) { *out = it->second.back(); it->second.pop_back(); return cudaSuccess; }
        if (left < r) {
            void *slab = nullptr;
            cudaError_t e = host ? cudaHostAlloc(&slab, SLAB, cudaHostAllocMapped | cudaHostAllocPortable) : cudaMalloc(&slab, SLAB);
            if (e != cudaSuccess) return e;
            cur = (char *)slab; left = SLAB;              // (the tail of the previous slab stays unused)
        }
        *out = cur; cur += r; left -= r;
        return cudaSuccess;
    }
    void release(void *p, size_t bytes) { free_lists[round(bytes)].push_back(p); }
};
static SmallPool g_host_pool{true, -1};
static std::map<int, SmallPool> g_dev_pools;

static cudaError_t host_alloc(size_t bytes, void **out) {
    if (bytes > SmallPool::SMALL_MAX) return cudaHostAlloc(out, bytes, cudaHostAllocMapped | cudaHostAllocPortable);
    std::lock_guard<std::mutex> lock(g_mu);
    return g_host_pool.alloc(bytes, out);
}
static void host_free(void *p, size_t bytes) {
    if (!p) return;
    if (bytes > SmallPool::SMALL_MAX) { cudaFreeHost(p); return; }
    std::lock_guard<std::mutex> lock(g_mu);
    g_host_pool.release(p, bytes);
}
static cudaError_t dev_alloc(int device, size_t bytes, void **out) {
    if (bytes > SmallPool::SMALL_MAX) return cudaMalloc(out, bytes);
    std::lock_guard<std::mutex> lock(g_mu);
    auto it = g_dev_pools.find(device);
    if (it == g_dev_pools.end()) it = g_dev_pools.emplace(device, SmallPool{false, device}).first;
    return it->second.alloc(bytes, out);
}
static void dev_free(int device, void *p, size_t bytes) {
    if (!p) return;
    if (bytes > SmallPool::SMALL_MAX) { cudaFree(p); return; }
    std::lock_guard<std::mutex> lock(g_mu);
    g_dev_pools.find(device)->second.release(p, bytes);
}

static bool is_pow2(long n) { return n > 0 && (n & (n - 1)) == 0; }
static int ilog2(long n) { int k = 0; while ((1L << k) < n) k++; return k; }

}  // namespace wfb

using namespace wfb;

// ----------------------------------------------------------------------------------------
// plan object
// ----------------------------------------------------------------------------------------
// one kernel variant of a plan and its twiddle tables, built and uploaded on the variant's first launch (ensure_tables)
struct PlanVariant {
    const Variant *v;
    void *d_tables = nullptr;          // the one allocation d_tw / d_rtw point into; null until the tables are uploaded
    size_t tables_bytes = 0;
    void *d_tw[2] = {};                // stage tables by direction (WFB_FORWARD, WFB_INVERSE)
    void *d_rtw = nullptr;             // W_n^k of the real transforms (table format depends on the lane type)
    std::vector<unsigned char> h_tw0[2];   // head of each stage table for KParams::tw0 (scalar-lane variants)
};

struct wfb_plan {
    int kind, precision, layout, n, device, flags;
    long batch;
    int core_n;
    size_t elem;                       // sizeof(real)
    std::vector<PlanVariant> variants; // every registered variant of this (precision, core size, kind), best first
    int variant;                       // forward-direction kernel variant
    int variant_inv;                   // inverse-direction kernel variant
    // buffers: C2C -> plane 0 / plane 1; R2C -> time / spectrum
    void *d_buf[2];
    void *h_buf[2];
    size_t bytes[2];
    bool host_alias;                   // R2C batch == 1: both host views share one allocation
    void *hd_buf[2];                   // device-side addresses of the (mapped) host buffers: the zero-copy path
    int mapped_variant;                // direct-load kernel the zero-copy path launches
    long mapped_max_bytes;             // zero-copy below this many payload bytes (in + out)
    long stage_chunk_bytes;            // staging pipeline: bytes of the widest plane per chunk
    int stage_streams;                 // ... and the number of streams the chunks cycle over
    bool stage_ramp;                   // short chunks at both ends of the pipeline (see exec_impl)
    int last_path;                     // WFB_PATH_* of the latest wfb_exec
    // completion flag of the zero-copy path: the kernel's last act is a store of `token` to this word of mapped host
    // memory (after a system-scope fence behind its data stores); wfb_exec polls it instead of calling into the driver
    volatile unsigned *h_flag;
    unsigned *hd_flag, *d_done_ctr;
    unsigned token;
    cudaStream_t stream;
    // staging pipeline: chunks of rows cycle over these streams so the H2D copy of chunk c+1, the
    // kernel of chunk c and the D2H copy of chunk c-1 overlap (PCIe is full duplex)
    enum { NPIPE = 6 };
    cudaStream_t pipe[NPIPE];
    cudaEvent_t pipe_done[NPIPE], start_ev;
    bool pipe_ready;                   // streams / events above exist (created by the first pipelined exec)
};

static int check_device_uncached(int device);
// cudaGetDeviceProperties costs milliseconds; a plan is created per transform size, so the verdict is cached per device
static int check_device(int device) {
    static std::map<int, int> ok;
    {
        std::lock_guard<std::mutex> lock(g_mu);
        auto it = ok.find(device);
        if (it != ok.end()) return it->second;
    }
    const int rc = check_device_uncached(device);
    if (rc == WFB_OK) { std::lock_guard<std::mutex> lock(g_mu); ok[device] = rc; }
    return rc;
}
static int check_device_uncached(int device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) {
        snprintf(g_cuda_err, sizeof g_cuda_err, "no usable CUDA device (%s)", e == cudaSuccess ? "index out of range" : cudaGetErrorString(e));
        return WFB_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return WFB_ERR_NO_DEVICE;
    if (prop.major != 10) {   // kernels are built for sm_100a only
        snprintf(g_cuda_err, sizeof g_cuda_err, "device %d is sm_%d%d, need sm_100 (B200)", device, prop.major, prop.minor);
        return WFB_ERR_NO_DEVICE;
    }
    return WFB_OK;
}

extern "C" {

int wfb_device_count(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) return 0;
    return count;
}

int wfb_require_b200(int device) { return check_device(device); }

const char *wfb_strerror(int code) {
    switch (code) {
        case WFB_OK: return "ok";
        case WFB_ERR_NO_DEVICE: return "no B200 (sm_100) device available; this engine has no CPU fallback";
        case WFB_ERR_BAD_SIZE: return "transform size must be a power of two within the supported range";
        case WFB_ERR_BAD_ARG: return "bad argument";
        case WFB_ERR_UNSUPPORTED: return "unsupported (kind, precision, layout) combination";
        case WFB_ERR_ALLOC: return "allocation failed";
        case WFB_ERR_CUDA: return "CUDA error (see wfb_last_cuda_error)";
        case WFB_ERR_NO_HOST_BUFFERS: return "plan was created without host staging buffers";
        default: return "unknown error";
    }
}

const char *wfb_last_cuda_error(void) { return g_cuda_err; }

int wfb_size_range(int kind, int precision, int layout, int *min_n, int *max_n) {
    int lo, hi;
    if (kind == WFB_C2C) {
        if (precision == WFB_F32 && (layout == WFB_SPLIT || layout == WFB_INTERLEAVED)) { lo = 4; hi = 8192; }
        else if (precision == WFB_F64 && layout == WFB_INTERLEAVED) { lo = 4; hi = 8192; }
        else return WFB_ERR_UNSUPPORTED;
    } else if (kind == WFB_R2C) {
        // rfft_split itself requires n >= 32 (fft_split_native_f32.wat:1562); n = 8 and 16 are accepted because
        // the public createRFFTf32 context does (it is backed by fft_real_f32_dual, benchmarks/shared/
        // wat-surfaces.mjs:133-141): same I/O contract, tolerance-based parity against that module
        if (precision == WFB_F32) { lo = 8; hi = 16384; }
        else if (precision == WFB_F64) { lo = 8; hi = 16384; }
        else return WFB_ERR_UNSUPPORTED;
    } else return WFB_ERR_UNSUPPORTED;
    if (min_n) *min_n = lo;
    if (max_n) *max_n = hi;
    return WFB_OK;
}

int wfb_reference_twiddles(int flavour, int n, int count, void *re, void *im) {
    if (!re || !im || n <= 0 || count < 0) return WFB_ERR_BAD_ARG;
    if (flavour == TW_F64) {
        std::vector<double> r, i;
        base_twiddles<double>(TW_F64, n, count, r, i);
        memcpy(re, r.data(), sizeof(double) * count); memcpy(im, i.data(), sizeof(double) * count);
    } else if (flavour == TW_F32_SPLIT || flavour == TW_F32_DUAL) {
        std::vector<float> r, i;
        base_twiddles<float>(flavour, n, count, r, i);
        memcpy(re, r.data(), sizeof(float) * count); memcpy(im, i.data(), sizeof(float) * count);
    } else return WFB_ERR_BAD_ARG;
    return WFB_OK;
}

}  // extern "C"

// Base-table flavour of an f32 scalar-lane core whose reference table is `reference`.  Kernels that DERIVE w2 = w1^2,
// w3 = w1*w2 in registers (f32 scalar lanes, core >= WFB_DERIVE_MIN_N: derive_tw in wfb_kernels.cuh) square and cube
// whatever error w1 carries.  The reference's f32 table is a 6-term Taylor series good to ~5e-7; derived from it, w3 is off
// by 1.5e-6 and N = 4096 misses the reference's own absolute threshold (tests/fft_f32_dual.test.js:83-86: 2.6e-4 against
// 2.0e-4).  So those kernels get CORRECTLY ROUNDED w1 (error 6e-8): the derived factors are then more accurate than the
// reference's looked-up ones, and the f32 contract is tolerance-based.
static int scalar_f32_flavour(int m, int reference) { return m >= WFB_DERIVE_MIN_N ? TW_EXACT : reference; }

// rfft_split's fused radix-8 opening uses exact W_8 constants for group 1 of the l = 2 stage
// (fft_split_native_f32.wat:1199-1371): patched into the forward stage table `fwd` of an f32 r2c core
static void w8_opening(int m, const std::vector<int> &radices, std::vector<float> &fwd) {
    if (!((ilog2(m) & 1) && m >= 32 && radices.size() >= 2 && radices[0] == 2 && radices[1] == 4)) return;
    const float c = float(0.7071067811865476);
    const size_t off = 2 * 1;               // skip the radix-2 stage's single entry (re,im)
    const int l = 2;
    const float w[3][2] = {{c, -c}, {0.0f, -1.0f}, {-c, -c}};
    for (int mm = 0; mm < 3; mm++) { fwd[off + 2 * (mm * l + 1)] = w[mm][0]; fwd[off + 2 * (mm * l + 1) + 1] = w[mm][1]; }
}

static size_t up256(size_t b) { return (b + 255) / 256 * 256; }

// builds forward / inverse stage tables for one variant and uploads them
template <typename R>
static int upload_tables(wfb_plan *pl, PlanVariant &pv) {
    const Variant &v = *pv.v;
    const int m = v.core_n;
    int flavour;
    if (sizeof(R) == 8) flavour = (m == 16 || m <= 4) ? TW_EXACT : TW_F64;
    else {
        flavour = (pl->kind == WFB_C2C && pl->layout == WFB_INTERLEAVED) ? (m <= 16 ? TW_EXACT : TW_F32_DUAL) : TW_F32_SPLIT;
        if (v.lanes == 1) flavour = scalar_f32_flavour(m, flavour);
    }
    std::vector<R> bre, bim, fwd, inv;
    base_twiddles<R>(flavour, m, m, bre, bim);
    stage_tables<R>(v.radices, m, bre, bim, false, fwd);
    stage_tables<R>(v.radices, m, bre, bim, true, inv);
    if constexpr (sizeof(R) == 4) if (pl->kind == WFB_R2C) w8_opening(m, v.radices, fwd);
    if (fwd.empty()) { fwd.assign(2, R(0)); inv.assign(2, R(0)); }
    // packed-lane kernels read entries as (re, re, im, im)
    auto widen = [&](std::vector<R> &t) {
        if (v.lanes != 2) return;
        std::vector<R> o;
        o.reserve(t.size() * 2);
        for (size_t i = 0; i + 1 < t.size(); i += 2) { o.push_back(t[i]); o.push_back(t[i]); o.push_back(t[i + 1]); o.push_back(t[i + 1]); }
        t.swap(o);
    };
    if (v.lanes == 1) {
        auto head = [](const std::vector<R> &t, std::vector<unsigned char> &h) {
            h.assign(KParams::TW0_BYTES, 0);
            memcpy(h.data(), t.data(), std::min<size_t>(t.size() * sizeof(R), KParams::TW0_BYTES));
        };
        head(fwd, pv.h_tw0[WFB_FORWARD]); head(inv, pv.h_tw0[WFB_INVERSE]);
    }
    widen(fwd); widen(inv);
    std::vector<R> packed;
    if (pl->kind == WFB_R2C) {
        // W_n^k, k = 0..M (fft_split_native_f32.wat:1167-1191; fft_real_combined.wat:931-948)
        int rf = sizeof(R) == 8 ? ((pl->n == 8 || pl->n == 32) ? TW_EXACT : TW_F64) : TW_F32_SPLIT;
        std::vector<R> rre, rim;
        base_twiddles<R>(rf, pl->n, m + 1, rre, rim);
        for (int k = 0; k <= m; k++) { packed.push_back(rre[k]); packed.push_back(rim[k]); }
        widen(packed);
    }
    // one allocation and one copy per variant: [forward | inverse | W_n^k], each 256-byte aligned
    const size_t bf = up256(fwd.size() * sizeof(R)), bi = up256(inv.size() * sizeof(R)), br = up256(packed.size() * sizeof(R));
    std::vector<unsigned char> blob(bf + bi + br, 0);
    memcpy(blob.data(), fwd.data(), fwd.size() * sizeof(R));
    memcpy(blob.data() + bf, inv.data(), inv.size() * sizeof(R));
    if (!packed.empty()) memcpy(blob.data() + bf + bi, packed.data(), packed.size() * sizeof(R));
    void *d = nullptr;
    CK(dev_alloc(pl->device, blob.size(), &d));
    // stream-ordered on the plan's stream and completed here: launches on ANY stream may follow (plan streams are
    // non-blocking, so the legacy-stream cudaMemcpy would not order against them)
    cudaError_t e = cudaMemcpyAsync(d, blob.data(), blob.size(), cudaMemcpyHostToDevice, pl->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(pl->stream);
    if (e != cudaSuccess) { dev_free(pl->device, d, blob.size()); return cuda_fail(e, "twiddle table upload"); }
    pv.d_tables = d;
    pv.tables_bytes = blob.size();
    pv.d_tw[WFB_FORWARD] = d;
    pv.d_tw[WFB_INVERSE] = (unsigned char *)d + bf;
    pv.d_rtw = packed.empty() ? nullptr : (unsigned char *)d + bf + bi;
    return WFB_OK;
}

// Twiddle tables are per kernel variant (stage grouping and lane packing differ); only the variants that are actually
// launched get theirs: the plan's defaults at creation (this is the reference's precompute_* call), the others on
// their first launch.
static int ensure_tables(wfb_plan *pl, int vi) {
    PlanVariant &pv = pl->variants[vi];
    if (pv.d_tables) return WFB_OK;
    return pl->precision == WFB_F64 ? upload_tables<double>(pl, pv) : upload_tables<float>(pl, pv);
}

static int ensure_device_buffers(wfb_plan *pl) {
    if (pl->flags & WFB_PLAN_NO_DEVICE_BUFFERS) return WFB_OK;
    for (int i = 0; i < 2; i++)
        if (pl->bytes[i] && !pl->d_buf[i]) {
            if (dev_alloc(pl->device, pl->bytes[i], &pl->d_buf[i]) != cudaSuccess) { cudaGetLastError(); return WFB_ERR_ALLOC; }
        }
    return WFB_OK;
}

static int ensure_pipeline(wfb_plan *pl) {
    if (pl->pipe_ready) return WFB_OK;
    for (int i = 0; i < wfb_plan::NPIPE; i++) {
        CK(cudaStreamCreateWithFlags(&pl->pipe[i], cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&pl->pipe_done[i], cudaEventDisableTiming));
    }
    CK(cudaEventCreateWithFlags(&pl->start_ev, cudaEventDisableTiming));
    pl->pipe_ready = true;
    return WFB_OK;
}

static size_t payload_bytes(const wfb_plan *pl) {
    const size_t e = pl->elem, n = (size_t)pl->n, b = (size_t)pl->batch;
    if (pl->kind == WFB_C2C) return 2 * (2 * e * n) * b;          // one read + one write of n complex values
    return (e * n + e * (n + 2)) * b;                               // n reals one way, n/2+1 bins the other
}

// true when wfb_exec(H2D | D2H) runs the zero-copy path: the kernel reads and writes the mapped host buffers directly
static bool use_mapped(const wfb_plan *pl) {
    return pl->hd_buf[0] && pl->mapped_variant >= 0 && (long)payload_bytes(pl) <= pl->mapped_max_bytes;
}

static long env_long(const char *name, long dflt) { const char *e = getenv(name); return e ? atol(e) : dflt; }

static int plan_init(wfb_plan *pl) {
    CK(cudaSetDevice(pl->device));
    CK(cudaStreamCreateWithFlags(&pl->stream, cudaStreamNonBlocking));
    const size_t e = pl->elem, n = (size_t)pl->n, b = (size_t)pl->batch;
    if (pl->kind == WFB_C2C) {
        if (pl->layout == WFB_SPLIT) { pl->bytes[0] = pl->bytes[1] = e * n * b; }
        else { pl->bytes[0] = 2 * e * n * b; pl->bytes[1] = 0; }
    } else {
        pl->bytes[WFB_BUF_TIME] = e * n * b;
        pl->bytes[WFB_BUF_SPECTRUM] = e * (n + 2) * b;
    }
    // staging knobs (wfb_plan_set_option overrides the environment defaults)
    pl->mapped_max_bytes = env_long("WFB_MAPPED_MAX_KB", 256) << 10;
    pl->stage_chunk_bytes = std::max(1L, env_long("WFB_STAGE_CHUNK_MB", 32)) << 20;
    pl->stage_streams = (int)std::min<long>(wfb_plan::NPIPE, std::max(1L, env_long("WFB_STAGE_STREAMS", 3)));
    pl->stage_ramp = env_long("WFB_STAGE_RAMP", 1) != 0;
    // the zero-copy path launches the direct-load kernel (no TMA pipeline to fill, no tile counter): lowest alignment need
    pl->mapped_variant = -1;
    for (size_t i = 0; i < pl->variants.size(); i++)
        if (pl->variants[i].v->direct && pl->variants[i].v->lanes == 1) { pl->mapped_variant = (int)i; break; }
    if (!(pl->flags & WFB_PLAN_NO_HOST_BUFFERS)) {
        // mapped + portable: the kernels can address these buffers directly (hd_buf), which is what the small-batch path does
        if (pl->kind == WFB_R2C && pl->batch == 1) {
            // the reference's input and output views are the same bytes (index.js:136-141)
            if (host_alloc(pl->bytes[1], &pl->h_buf[1]) != cudaSuccess) { cudaGetLastError(); return WFB_ERR_ALLOC; }
            memset(pl->h_buf[1], 0, pl->bytes[1]);
            pl->h_buf[0] = pl->h_buf[1];
            pl->host_alias = true;
        } else {
            for (int i = 0; i < 2; i++)
                if (pl->bytes[i]) {
                    if (host_alloc(pl->bytes[i], &pl->h_buf[i]) != cudaSuccess) { cudaGetLastError(); return WFB_ERR_ALLOC; }
                    memset(pl->h_buf[i], 0, pl->bytes[i]);
                }
        }
        for (int i = 0; i < 2; i++)
            if (pl->h_buf[i] && cudaHostGetDevicePointer(&pl->hd_buf[i], pl->h_buf[i], 0) != cudaSuccess) { cudaGetLastError(); pl->hd_buf[0] = pl->hd_buf[1] = nullptr; break; }
    }
    // completion flag (host word) + CTA counter (device word) of the zero-copy path (also used by wfb_exec_host on
    // plans without host buffers of their own)
    void *f = nullptr, *c = nullptr;
    if (host_alloc(256, &f) == cudaSuccess && dev_alloc(pl->device, 256, &c) == cudaSuccess) {
        pl->h_flag = (volatile unsigned *)f;
        *pl->h_flag = 0;
        pl->d_done_ctr = (unsigned *)c;
        if (cudaHostGetDevicePointer((void **)&pl->hd_flag, f, 0) != cudaSuccess ||
            cudaMemsetAsync(c, 0, 256, pl->stream) != cudaSuccess || cudaStreamSynchronize(pl->stream) != cudaSuccess) {
            cudaGetLastError();
            pl->hd_flag = nullptr;
        }
    } else {
        cudaGetLastError();
        if (f) host_free(f, 256);
        if (c) dev_free(pl->device, c, 256);
    }
    int rc;
    if (use_mapped(pl)) {
        // small plan: exec never leaves the mapped buffers; device buffers and the other variants' tables are made on demand
        if ((rc = ensure_tables(pl, pl->mapped_variant))) return rc;
    } else {
        if ((rc = ensure_tables(pl, pl->variant)) || (rc = ensure_tables(pl, pl->variant_inv))) return rc;
        if ((rc = ensure_device_buffers(pl))) return rc;
    }
    return WFB_OK;
}

extern "C" {

wfb_plan *wfb_plan_create_ex(int kind, int precision, int layout, int n, long batch, int device, int flags, int *err) {
    int dummy;
    if (!err) err = &dummy;
    int lo, hi;
    *err = wfb_size_range(kind, precision, layout, &lo, &hi);
    if (*err) return nullptr;
    if (!is_pow2(n) || n < lo || n > hi) { *err = WFB_ERR_BAD_SIZE; return nullptr; }
    if (batch < 1) { *err = WFB_ERR_BAD_ARG; return nullptr; }
    *err = check_device(device);
    if (*err) return nullptr;

    wfb_plan *pl = new wfb_plan();
    pl->kind = kind; pl->precision = precision; pl->layout = (kind == WFB_C2C) ? layout : WFB_INTERLEAVED;
    pl->n = n; pl->batch = batch; pl->device = device; pl->flags = flags;
    pl->core_n = (kind == WFB_R2C) ? n / 2 : n;
    pl->elem = precision == WFB_F64 ? 8 : 4;
    pl->variant = 0;
    pl->variant_inv = 0;
    std::vector<const std::vector<Variant> *> families;
    if (precision == WFB_F64) families = {&variants_f64_pipe(), &variants_f64()};
    else families = {&variants_f32_tile(), &variants_f32_pipe(), &variants_f32_real_pipe(), &variants_f32_x2(), &variants_f32_direct()};
    for (const auto *fam : families)
        for (const Variant &v : *fam)
            if (v.core_n == pl->core_n && v.ops[kind == WFB_C2C ? OP_IL_FWD : OP_R2C].kernel) pl->variants.push_back({&v});
    const bool il = kind == WFB_C2C && layout == WFB_INTERLEAVED;
    std::stable_sort(pl->variants.begin(), pl->variants.end(), [il](const PlanVariant &a, const PlanVariant &b) {
        return (il ? a.v->priority_il : a.v->priority) > (il ? b.v->priority_il : b.v->priority);
    });
    for (size_t i = 0; i < pl->variants.size(); i++)
        if (!il && pl->variants[i].v->priority_inv > pl->variants[pl->variant_inv].v->priority_inv) pl->variant_inv = (int)i;
    if (pl->variants.empty()) { *err = WFB_ERR_BAD_SIZE; delete pl; return nullptr; }
    *err = plan_init(pl);
    if (*err) { wfb_plan_destroy(pl); return nullptr; }
    return pl;
}

wfb_plan *wfb_plan_create(int kind, int precision, int layout, int n, long batch, int device, int *err) {
    return wfb_plan_create_ex(kind, precision, layout, n, batch, device, 0, err);
}

void wfb_plan_destroy(wfb_plan *pl) {
    if (!pl) return;
    cudaSetDevice(pl->device);
    if (pl->stream) { cudaStreamSynchronize(pl->stream); cudaStreamDestroy(pl->stream); }
    for (int i = 0; i < wfb_plan::NPIPE; i++) {
        if (pl->pipe[i]) { cudaStreamSynchronize(pl->pipe[i]); cudaStreamDestroy(pl->pipe[i]); }
        if (pl->pipe_done[i]) cudaEventDestroy(pl->pipe_done[i]);
    }
    if (pl->start_ev) cudaEventDestroy(pl->start_ev);
    for (const PlanVariant &pv : pl->variants) dev_free(pl->device, pv.d_tables, pv.tables_bytes);
    for (int i = 0; i < 2; i++) dev_free(pl->device, pl->d_buf[i], pl->bytes[i]);
    if (pl->host_alias) host_free(pl->h_buf[1], pl->bytes[1]);
    else for (int i = 0; i < 2; i++) host_free(pl->h_buf[i], pl->bytes[i]);
    if (pl->h_flag) host_free((void *)pl->h_flag, 256);
    if (pl->d_done_ctr) dev_free(pl->device, pl->d_done_ctr, 256);
    delete pl;
}

void *wfb_host_buffer(wfb_plan *pl, int which) { return (pl && which >= 0 && which < 2) ? pl->h_buf[which] : nullptr; }
void *wfb_device_buffer(wfb_plan *pl, int which) {
    if (!pl || which < 0 || which >= 2) return nullptr;
    if (!pl->d_buf[which] && pl->bytes[which]) {          // small plans allocate their device buffers on demand
        cudaSetDevice(pl->device);
        if (ensure_device_buffers(pl) != WFB_OK) return nullptr;
    }
    return pl->d_buf[which];
}
size_t wfb_host_bytes(wfb_plan *pl, int which) { return (pl && which >= 0 && which < 2) ? pl->bytes[which] : 0; }
// C2C contexts are in place: the input view is the output view (index.js:78-83)
void *wfb_host_in(wfb_plan *pl, int plane) { return wfb_host_buffer(pl, plane); }
void *wfb_host_out(wfb_plan *pl, int plane) { return wfb_host_buffer(pl, plane); }
void *wfb_plan_stream(wfb_plan *pl) { return pl ? (void *)pl->stream : nullptr; }

int wfb_plan_variant_count(wfb_plan *pl) { return pl ? (int)pl->variants.size() : 0; }
int wfb_plan_set_variant(wfb_plan *pl, int v) {
    if (!pl || v < 0 || v >= (int)pl->variants.size()) return WFB_ERR_BAD_ARG;
    pl->variant = v;
    pl->variant_inv = v;
    pl->mapped_max_bytes = 0;      // an explicitly chosen kernel is the kernel that runs: no zero-copy detour
    return WFB_OK;
}
int wfb_plan_current_variant(wfb_plan *pl, int direction) {
    if (!pl || (direction != WFB_FORWARD && direction != WFB_INVERSE)) return WFB_ERR_BAD_ARG;
    return direction == WFB_INVERSE ? pl->variant_inv : pl->variant;
}
const char *wfb_plan_variant_name(wfb_plan *pl, int v) {
    if (!pl || v < 0 || v >= (int)pl->variants.size()) return "";
    return pl->variants[v].v->name;
}
size_t wfb_plan_algorithmic_bytes(wfb_plan *pl) { return pl ? payload_bytes(pl) : 0; }

int wfb_plan_set_option(wfb_plan *pl, int option, long value) {
    if (!pl || value < 0) return WFB_ERR_BAD_ARG;
    switch (option) {
        case WFB_OPT_MAPPED_MAX_BYTES: pl->mapped_max_bytes = value; return WFB_OK;
        case WFB_OPT_STAGE_CHUNK_BYTES: if (value < 4096) return WFB_ERR_BAD_ARG; pl->stage_chunk_bytes = value; return WFB_OK;
        case WFB_OPT_STAGE_STREAMS: if (value < 1 || value > wfb_plan::NPIPE) return WFB_ERR_BAD_ARG; pl->stage_streams = (int)value; return WFB_OK;
        case WFB_OPT_STAGE_RAMP: pl->stage_ramp = value != 0; return WFB_OK;
        default: return WFB_ERR_BAD_ARG;
    }
}
long wfb_plan_get_option(wfb_plan *pl, int option) {
    if (!pl) return -1;
    switch (option) {
        case WFB_OPT_MAPPED_MAX_BYTES: return pl->mapped_max_bytes;
        case WFB_OPT_STAGE_CHUNK_BYTES: return pl->stage_chunk_bytes;
        case WFB_OPT_STAGE_STREAMS: return pl->stage_streams;
        case WFB_OPT_STAGE_RAMP: return pl->stage_ramp ? 1 : 0;
        default: return -1;
    }
}
int wfb_plan_last_path(wfb_plan *pl) { return pl ? pl->last_path : WFB_ERR_BAD_ARG; }
unsigned long long wfb_kernel_launch_count(void) { return g_launches.load(); }

// launches the current variant over `rows` rows starting at the given plane pointers
static int launch_rows(wfb_plan *pl, int direction, const void *in0, const void *in1, void *out0, void *out1,
                       long rows, cudaStream_t s, int force_variant = -1, bool signal = false) {
    int vi = force_variant >= 0 ? force_variant : (direction == WFB_INVERSE ? pl->variant_inv : pl->variant);
    // The TMA / 128-bit kernels need 16-byte aligned planes (cudaMalloc gives 256).  Caller-supplied
    // pointers that are less aligned are served by the first variant whose requirement they meet.
    // The second plane pointers only exist for split c2c; elsewhere whatever the caller left there is ignored.
    const bool two_planes = pl->kind == WFB_C2C && pl->layout == WFB_SPLIT;
    if (!two_planes) { in1 = nullptr; out1 = nullptr; }
    const uintptr_t bits = (uintptr_t)in0 | (uintptr_t)in1 | (uintptr_t)out0 | (uintptr_t)out1;
    auto need = [&](const Variant *v) {
        // direct kernels read split planes with scalar loads
        return (v->align < 16 && pl->kind == WFB_C2C && pl->layout == WFB_SPLIT) ? (int)pl->elem : v->align;
    };
    if (bits & (uintptr_t)(need(pl->variants[vi].v) - 1)) {
        int alt = -1;
        for (size_t i = 0; i < pl->variants.size() && alt < 0; i++)
            if (!(bits & (uintptr_t)(need(pl->variants[i].v) - 1))) alt = (int)i;
        if (alt < 0) return WFB_ERR_BAD_ARG;
        vi = alt;
    }
    if (int rc = ensure_tables(pl, vi)) return rc;
    const PlanVariant &pv = pl->variants[vi];
    KParams p;
    p.in0 = in0; p.in1 = in1; p.out0 = out0; p.out1 = out1;
    p.tw = pv.d_tw[direction];
    p.rtw = pv.d_rtw;
    p.batch = rows;
    p.scale = 1.0 / (double)pl->n;
    p.ctr = nullptr;
    p.done_flag = signal ? pl->hd_flag : nullptr;
    p.done_ctr = pl->d_done_ctr;
    p.done_token = pl->token;
    if (!pv.h_tw0[direction].empty()) memcpy(p.tw0, pv.h_tw0[direction].data(), KParams::TW0_BYTES);
    const int op = (pl->kind == WFB_R2C ? OP_R2C : pl->layout == WFB_SPLIT ? OP_SPLIT_FWD : OP_IL_FWD) + direction;
    cudaError_t e = launch_op(*pv.v, op, p, rows, s);
    if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
    return WFB_OK;
}

int wfb_exec_device(wfb_plan *pl, int direction, const void *const d_in[2], void *const d_out[2], void *stream) {
    if (!pl || !d_in || !d_out || (direction != WFB_FORWARD && direction != WFB_INVERSE)) return WFB_ERR_BAD_ARG;
    CK(cudaSetDevice(pl->device));
    cudaStream_t s = stream ? (cudaStream_t)stream : pl->stream;
    if (pl->kind == WFB_C2C) {
        if (!d_in[0] || !d_out[0] || (pl->layout == WFB_SPLIT && (!d_in[1] || !d_out[1]))) return WFB_ERR_BAD_ARG;
    } else {
        if (!d_in[0] || !d_out[0]) return WFB_ERR_BAD_ARG;
        if (pl->batch > 1 && d_in[0] == d_out[0]) return WFB_ERR_BAD_ARG;   // strides differ: rows would overlap
    }
    return launch_rows(pl, direction, d_in[0], d_in[1], d_out[0], d_out[1], pl->batch, s);
}

int wfb_sync(wfb_plan *pl) {
    if (!pl) return WFB_ERR_BAD_ARG;
    CK(cudaSetDevice(pl->device));
    CK(cudaStreamSynchronize(pl->stream));
    return WFB_OK;
}

}  // extern "C"

// Host arenas handed out by wfb_host_alloc: base -> (bytes, device-side address).  wfb_exec_host accepts only pointers
// inside one of them (pinned + device-mapped memory is what both of its paths need).
struct Arena { size_t bytes; char *dev; };
static std::map<uintptr_t, Arena> g_arenas;
static bool arena_lookup(const void *p, size_t need, void **dev_alias) {
    std::lock_guard<std::mutex> lock(g_mu);
    auto it = g_arenas.upper_bound((uintptr_t)p);
    if (it == g_arenas.begin()) return false;
    --it;
    const uintptr_t off = (uintptr_t)p - it->first;
    if (off + need > it->second.bytes) return false;
    *dev_alias = it->second.dev + off;
    return true;
}

// Rows per pipeline chunk of wfb_exec: `chunk_bytes` of the widest plane, whole kernel tiles (tiles hold up to 256 rows)
// and 16-byte aligned chunk starts for the (n+2)-wide spectrum rows (an even number of rows).
static long stage_chunk_rows(long chunk_bytes, size_t widest_row_bytes) {
    long chunk = (long)(chunk_bytes / (long)widest_row_bytes);
    if (chunk >= 512) chunk &= ~255L; else if (chunk >= 2) chunk &= ~1L;
    return chunk < 1 ? 1 : chunk;
}
// Chunk schedule of the pipelined path (batch > 2 * chunk).  The first H2D copy has no D2H running beside it and the last
// D2H no H2D: those two ends are the part of the call that cannot overlap, so with `ramp` the schedule goes up through
// short chunks (1/8, 1/4, 1/2 of the steady-state size) and down again.  Every chunk but the last keeps the alignment
// rules of stage_chunk_rows; the rows of the chunks add up to `batch`.
static std::vector<long> stage_schedule(long batch, long chunk, bool ramp_on) {
    std::vector<long> sched;
    auto aligned = [](long c) { if (c >= 512) c &= ~255L; else if (c >= 2) c &= ~1L; return c < 1 ? 1L : c; };
    const long ramp[3] = {aligned(chunk / 8), aligned(chunk / 4), aligned(chunk / 2)};
    const long ends = 2 * (ramp[0] + ramp[1] + ramp[2]);
    if (ramp_on && chunk >= 16 && batch >= ends + 2 * chunk) {
        long mid = batch - ends;
        for (int i = 0; i < 3; i++) sched.push_back(ramp[i]);
        for (; mid >= chunk; mid -= chunk) sched.push_back(chunk);
        const long rem = mid >= 2 ? (mid & ~1L) : 0;      // an even remainder keeps the next chunk start aligned
        if (rem) sched.push_back(rem);
        for (int i = 2; i >= 0; i--) sched.push_back(ramp[i]);
        sched.back() += mid - rem;                         // (an odd batch's last row)
    } else {
        for (long r0 = 0; r0 < batch; r0 += chunk) sched.push_back(batch - r0 < chunk ? batch - r0 : chunk);
    }
    return sched;
}

// wfb_exec / wfb_exec_host: `hs`, `hd` = host addresses of the planes read and written (indexed like src[] / dst[] below),
// `as`, `ad` = the device-side addresses of the same bytes (zero-copy path; null when the memory is not mapped)
static int exec_impl(wfb_plan *pl, int direction, int flags, void *const hs_in[2], void *const hd_in[2], void *const as_in[2], void *const ad_in[2]) {
    if (pl->flags & WFB_PLAN_NO_DEVICE_BUFFERS) return WFB_ERR_BAD_ARG;
    CK(cudaSetDevice(pl->device));
    // buffer ids and per-row byte strides of the planes read and written
    int src[2] = {-1, -1}, dst[2] = {-1, -1};
    size_t src_row[2] = {0, 0}, dst_row[2] = {0, 0};
    const size_t e = pl->elem, n = (size_t)pl->n;
    if (pl->kind == WFB_C2C) {
        src[0] = dst[0] = 0;
        src_row[0] = dst_row[0] = (pl->layout == WFB_SPLIT ? 1 : 2) * e * n;
        if (pl->layout == WFB_SPLIT) { src[1] = dst[1] = 1; src_row[1] = dst_row[1] = e * n; }
    } else {
        const int a = direction == WFB_FORWARD ? WFB_BUF_TIME : WFB_BUF_SPECTRUM;
        src[0] = a; dst[0] = 1 - a;
        src_row[0] = e * (a == WFB_BUF_TIME ? n : n + 2);
        dst_row[0] = e * (a == WFB_BUF_TIME ? n + 2 : n);
    }
    // host / alias pointers per plane slot: the plan's own buffers unless the caller supplied some
    void *hs[2] = {nullptr, nullptr}, *hd[2] = {nullptr, nullptr}, *as[2] = {nullptr, nullptr}, *ad[2] = {nullptr, nullptr};
    for (int i = 0; i < 2; i++) {
        if (src[i] >= 0) { hs[i] = hs_in ? hs_in[i] : pl->h_buf[src[i]]; as[i] = hs_in ? as_in[i] : pl->hd_buf[src[i]]; }
        if (dst[i] >= 0) { hd[i] = hd_in ? hd_in[i] : pl->h_buf[dst[i]]; ad[i] = hd_in ? ad_in[i] : pl->hd_buf[dst[i]]; }
    }
    const bool h2d = flags & WFB_STAGE_H2D, d2h = flags & WFB_STAGE_D2H;

    // ---- zero-copy path (small payloads; the reference's own call shape is batch = 1, index.js:84-89): ONE launch of
    // the direct-load kernel on the mapped host buffers -- the loads and stores cross PCIe themselves, so there is no
    // copy node in front of or behind the kernel and nothing to wait for but the kernel.  In place is safe: every CTA of
    // the direct kernels has all its rows in registers (behind a barrier for multi-pass plans) before its first store.
    const bool mapped_ok = as[0] && ad[0] && pl->mapped_variant >= 0 && (long)payload_bytes(pl) <= pl->mapped_max_bytes;
    if (h2d && d2h && mapped_ok) {
        const bool flagged = (flags & WFB_SYNC) && pl->hd_flag;
        if (flagged) pl->token++;
        int rc = launch_rows(pl, direction, as[0], as[1], ad[0], ad[1], pl->batch, pl->stream, pl->mapped_variant, flagged);
        if (rc) return rc;
        pl->last_path = WFB_PATH_MAPPED;
        if (flagged) {
            // the results are in host memory when the token is: no driver call on the way back.  The stream is consulted
            // only if the token is late (a faulting kernel never writes it).
            const unsigned want = pl->token;
            auto t0 = std::chrono::steady_clock::now();
            for (unsigned spins = 0; *pl->h_flag != want; spins++) {
                __builtin_ia32_pause();
                if ((spins & 0xFFF) == 0xFFF && std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(2)) {
                    CK(cudaStreamSynchronize(pl->stream));       // also surfaces a kernel fault as an error code
                    break;
                }
            }
            std::atomic_thread_fence(std::memory_order_acquire);
        } else if (flags & WFB_SYNC) {
            CK(cudaStreamSynchronize(pl->stream));
        }
        return WFB_OK;
    }

    if (int rc = ensure_device_buffers(pl)) return rc;
    // rows per pipeline chunk: stage_chunk_bytes of the widest plane, so each copy is long enough to run at
    // full PCIe rate while there are enough chunks to overlap the two directions
    size_t widest = src_row[0] > dst_row[0] ? src_row[0] : dst_row[0];
    const int nstreams = pl->stage_streams;
    const long chunk = stage_chunk_rows(pl->stage_chunk_bytes, widest);
    const bool pipelined = (h2d || d2h) && pl->batch > 2 * chunk;
    if (!pipelined) {
        pl->last_path = WFB_PATH_STAGED;
        if (h2d)
            for (int i = 0; i < 2; i++)
                if (src[i] >= 0) CK(cudaMemcpyAsync(pl->d_buf[src[i]], hs[i], pl->bytes[src[i]], cudaMemcpyHostToDevice, pl->stream));
        int rc = launch_rows(pl, direction, pl->d_buf[src[0]], src[1] >= 0 ? pl->d_buf[src[1]] : nullptr,
                             pl->d_buf[dst[0]], dst[1] >= 0 ? pl->d_buf[dst[1]] : nullptr, pl->batch, pl->stream);
        if (rc) return rc;
        if (d2h)
            for (int i = 0; i < 2; i++)
                if (dst[i] >= 0) CK(cudaMemcpyAsync(hd[i], pl->d_buf[dst[i]], pl->bytes[dst[i]], cudaMemcpyDeviceToHost, pl->stream));
    } else {
        pl->last_path = WFB_PATH_PIPELINED;
        if (int rc = ensure_pipeline(pl)) return rc;
        // the kernels of every chunk share one variant: its tables must exist before the first stream uses them
        if (int rc = ensure_tables(pl, direction == WFB_INVERSE ? pl->variant_inv : pl->variant)) return rc;
        // order the pipeline after whatever is already queued on the plan's stream
        CK(cudaEventRecord(pl->start_ev, pl->stream));
        for (int i = 0; i < nstreams; i++) CK(cudaStreamWaitEvent(pl->pipe[i], pl->start_ev, 0));
        const std::vector<long> sched = stage_schedule(pl->batch, chunk, pl->stage_ramp);
        long r0 = 0;
        for (size_t c = 0; c < sched.size(); r0 += sched[c], c++) {
            const long rows = sched[c];
            cudaStream_t s = pl->pipe[c % nstreams];
            char *di[2] = {nullptr, nullptr}, *dout[2] = {nullptr, nullptr};
            for (int i = 0; i < 2; i++) {
                if (src[i] >= 0) {
                    di[i] = (char *)pl->d_buf[src[i]] + (size_t)r0 * src_row[i];
                    if (h2d) CK(cudaMemcpyAsync(di[i], (char *)hs[i] + (size_t)r0 * src_row[i], (size_t)rows * src_row[i], cudaMemcpyHostToDevice, s));
                }
                if (dst[i] >= 0) dout[i] = (char *)pl->d_buf[dst[i]] + (size_t)r0 * dst_row[i];
            }
            int rc = launch_rows(pl, direction, di[0], di[1], dout[0], dout[1], rows, s);
            if (rc) return rc;
            if (d2h)
                for (int i = 0; i < 2; i++)
                    if (dst[i] >= 0) CK(cudaMemcpyAsync((char *)hd[i] + (size_t)r0 * dst_row[i], dout[i], (size_t)rows * dst_row[i], cudaMemcpyDeviceToHost, s));
        }
        for (int i = 0; i < nstreams; i++) {
            CK(cudaEventRecord(pl->pipe_done[i], pl->pipe[i]));
            CK(cudaStreamWaitEvent(pl->stream, pl->pipe_done[i], 0));
        }
    }
    if (flags & WFB_SYNC) CK(cudaStreamSynchronize(pl->stream));
    return WFB_OK;
}

extern "C" {

int wfb_stage_schedule(long batch, size_t widest_row_bytes, long chunk_bytes, int ramp, long *rows_out, int capacity) {
    if (batch < 1 || widest_row_bytes < 1 || chunk_bytes < 1 || capacity < 0 || (capacity > 0 && !rows_out)) return WFB_ERR_BAD_ARG;
    const long chunk = stage_chunk_rows(chunk_bytes, widest_row_bytes);
    if (batch <= 2 * chunk) return 0;                      // not pipelined: one copy in, one launch, one copy out
    const std::vector<long> sched = stage_schedule(batch, chunk, ramp != 0);
    for (size_t i = 0; i < sched.size() && (int)i < capacity; i++) rows_out[i] = sched[i];
    return (int)sched.size();
}

int wfb_exec(wfb_plan *pl, int direction, int flags) {
    if (!pl || (direction != WFB_FORWARD && direction != WFB_INVERSE)) return WFB_ERR_BAD_ARG;
    if ((flags & (WFB_STAGE_H2D | WFB_STAGE_D2H)) && !pl->h_buf[0] && !pl->h_buf[1]) return WFB_ERR_NO_HOST_BUFFERS;
    return exec_impl(pl, direction, flags, nullptr, nullptr, nullptr, nullptr);
}

void *wfb_host_alloc(size_t bytes) {
    if (bytes == 0) return nullptr;
    void *p = nullptr, *d = nullptr;
    if (host_alloc(bytes, &p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    memset(p, 0, bytes);
    if (cudaHostGetDevicePointer(&d, p, 0) != cudaSuccess) { cudaGetLastError(); host_free(p, bytes); return nullptr; }
    std::lock_guard<std::mutex> lock(g_mu);
    g_arenas[(uintptr_t)p] = Arena{bytes, (char *)d};
    return p;
}

void wfb_host_free(void *p) {
    if (!p) return;
    size_t bytes = 0;
    {
        std::lock_guard<std::mutex> lock(g_mu);
        auto it = g_arenas.find((uintptr_t)p);
        if (it == g_arenas.end()) return;
        bytes = it->second.bytes;
        g_arenas.erase(it);
    }
    host_free(p, bytes);
}

int wfb_exec_host(wfb_plan *pl, int direction, const void *const h_in[2], void *const h_out[2], int flags) {
    if (!pl || !h_in || !h_out || (direction != WFB_FORWARD && direction != WFB_INVERSE)) return WFB_ERR_BAD_ARG;
    const bool two = pl->kind == WFB_C2C && pl->layout == WFB_SPLIT;
    size_t in_bytes[2], out_bytes[2];
    if (pl->kind == WFB_C2C) { in_bytes[0] = out_bytes[0] = pl->bytes[0]; in_bytes[1] = out_bytes[1] = pl->bytes[1]; }
    else {
        const int a = direction == WFB_FORWARD ? WFB_BUF_TIME : WFB_BUF_SPECTRUM;
        in_bytes[0] = pl->bytes[a]; out_bytes[0] = pl->bytes[1 - a]; in_bytes[1] = out_bytes[1] = 0;
    }
    void *hs[2] = {nullptr, nullptr}, *hd[2] = {nullptr, nullptr}, *as[2] = {nullptr, nullptr}, *ad[2] = {nullptr, nullptr};
    for (int i = 0; i < (two ? 2 : 1); i++) {
        if (!h_in[i] || !h_out[i]) return WFB_ERR_BAD_ARG;
        if (!arena_lookup(h_in[i], in_bytes[i], &as[i]) || !arena_lookup(h_out[i], out_bytes[i], &ad[i])) return WFB_ERR_BAD_ARG;
        hs[i] = const_cast<void *>(h_in[i]); hd[i] = h_out[i];
    }
    // in place needs rows of equal stride on both sides (C2C always; R2C only at batch = 1, where a row is the whole buffer)
    if (pl->kind == WFB_R2C && pl->batch > 1 && h_in[0] == h_out[0]) return WFB_ERR_BAD_ARG;
    return exec_impl(pl, direction, flags | WFB_STAGE_H2D | WFB_STAGE_D2H, hs, hd, as, ad);
}

}  // extern "C"

extern "C" {

// Pinned-copy ceiling of the link wfb_exec stages over: plain cudaMemcpyAsync between a pinned host buffer and the
// device, each direction alone and both at once (one stream each), CUDA-event timed.  bench.py runs it on every rank
// at the same moment, so the figure is the CONCURRENT ceiling of the box, the roofline of the e2e number.
struct wfb_pcie_probe_state {
    int device; size_t bytes;
    void *h[2], *d[2];
    cudaStream_t st[2];
    cudaEvent_t ev[4];
};

void wfb_pcie_probe_close(wfb_pcie_probe_state *ps) {
    if (!ps) return;
    cudaSetDevice(ps->device);
    for (int i = 0; i < 2; i++) { if (ps->h[i]) cudaFreeHost(ps->h[i]); if (ps->d[i]) cudaFree(ps->d[i]); if (ps->st[i]) cudaStreamDestroy(ps->st[i]); }
    for (int i = 0; i < 4; i++) if (ps->ev[i]) cudaEventDestroy(ps->ev[i]);
    delete ps;
}

int wfb_pcie_probe_open(int device, size_t bytes, wfb_pcie_probe_state **out) {
    if (!out || bytes < 4096) return WFB_ERR_BAD_ARG;
    *out = nullptr;
    int rc = check_device(device);
    if (rc) return rc;
    CK(cudaSetDevice(device));
    wfb_pcie_probe_state *ps = new wfb_pcie_probe_state();
    memset(ps, 0, sizeof *ps);
    ps->device = device; ps->bytes = bytes;
#define CKP(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { wfb_pcie_probe_close(ps); return cuda_fail(e_, #call); } } while (0)
    for (int i = 0; i < 2; i++) {
        CKP(cudaHostAlloc(&ps->h[i], bytes, cudaHostAllocMapped | cudaHostAllocPortable));
        memset(ps->h[i], 0, bytes);
        CKP(cudaMalloc(&ps->d[i], bytes));
        CKP(cudaStreamCreateWithFlags(&ps->st[i], cudaStreamNonBlocking));
    }
    for (int i = 0; i < 4; i++) CKP(cudaEventCreate(&ps->ev[i]));
    // one untimed copy each way: first-touch costs of the mappings stay out of the timed phases
    CKP(cudaMemcpyAsync(ps->d[0], ps->h[0], bytes, cudaMemcpyHostToDevice, ps->st[0]));
    CKP(cudaMemcpyAsync(ps->h[1], ps->d[1], bytes, cudaMemcpyDeviceToHost, ps->st[1]));
    CKP(cudaStreamSynchronize(ps->st[0]));
    CKP(cudaStreamSynchronize(ps->st[1]));
#undef CKP
    *out = ps;
    return WFB_OK;
}

int wfb_pcie_probe_run(wfb_pcie_probe_state *ps, int directions, int iters, double seconds[2]) {
    if (!ps || !seconds || iters < 1 || !(directions & 3)) return WFB_ERR_BAD_ARG;
    const bool up = directions & 1, down = directions & 2;
    CK(cudaSetDevice(ps->device));
    if (up) CK(cudaEventRecord(ps->ev[0], ps->st[0]));
    if (down) CK(cudaEventRecord(ps->ev[2], ps->st[1]));
    for (int i = 0; i < iters; i++) {
        if (up) CK(cudaMemcpyAsync(ps->d[0], ps->h[0], ps->bytes, cudaMemcpyHostToDevice, ps->st[0]));
        if (down) CK(cudaMemcpyAsync(ps->h[1], ps->d[1], ps->bytes, cudaMemcpyDeviceToHost, ps->st[1]));
    }
    if (up) CK(cudaEventRecord(ps->ev[1], ps->st[0]));
    if (down) CK(cudaEventRecord(ps->ev[3], ps->st[1]));
    CK(cudaStreamSynchronize(ps->st[0]));
    CK(cudaStreamSynchronize(ps->st[1]));
    float ms;
    seconds[0] = seconds[1] = 0.0;
    if (up) { CK(cudaEventElapsedTime(&ms, ps->ev[0], ps->ev[1])); seconds[0] = ms * 1e-3; }
    if (down) { CK(cudaEventElapsedTime(&ms, ps->ev[2], ps->ev[3])); seconds[1] = ms * 1e-3; }
    return WFB_OK;
}

int wfb_pcie_probe(int device, size_t bytes, int iters, double gbs[4]) {
    if (!gbs || bytes < 4096 || iters < 1) return WFB_ERR_BAD_ARG;
    wfb_pcie_probe_state *ps = nullptr;
    int rc = wfb_pcie_probe_open(device, bytes, &ps);
    if (rc) return rc;
    double a[2], b[2], c[2];
    if ((rc = wfb_pcie_probe_run(ps, 1, iters, a)) || (rc = wfb_pcie_probe_run(ps, 2, iters, b)) || (rc = wfb_pcie_probe_run(ps, 3, iters, c))) {
        wfb_pcie_probe_close(ps);
        return rc;
    }
    const double gb = (double)bytes * iters / 1e9;
    gbs[0] = gb / a[0]; gbs[1] = gb / b[1]; gbs[2] = gb / c[0]; gbs[3] = gb / c[1];
    wfb_pcie_probe_close(ps);
    return WFB_OK;
}

}  // extern "C"


// ----------------------------------------------------------------------------------------
// batched STFT front-end
// ----------------------------------------------------------------------------------------
struct wfb_stft {
    int fft_size, wsize, hop, mode, window, device, flags;
    long num_samples, frames, batch;   // frames per signal; batch signals of num_samples each
    const StftVariant *variant;
    void *d_tables;                    // the one allocation d_tw / d_tw_span / d_rtw / d_window point into
    void *d_tw, *d_tw_span, *d_rtw, *d_window, *d_samples, *d_out;
    void *h_samples, *h_out;
    size_t in_bytes, out_bytes;        // whole batch
    float db_floor, inv_range;
    // filterbank handles (mode STFT_MODE_FILTERBANK): the filters' bands {first bin, bins, weight offset, 0} and packed
    // weights (host copies; device copies in d_tables), the power and L
    int num_filters, power;
    float log_scale, log_offset, log_floor;
    std::vector<int> fb_band;
    std::vector<float> fb_w;
    void *d_fb_band, *d_fb_w;
    cudaStream_t stream;
    // inverse (wfb_stft_exec_inverse*): built on the first inverse call, so a forward-only handle never pays for it
    const IstftVariant *inv_variant;
    void *d_tw_inv;                    // conjugated stage tables of the inverse kernel's core plan
    cudaEvent_t inv_ready;             // recorded behind their upload: later calls on other streams wait for it
};

// WINDOW_FUNCTIONS of playground/src/spectrogram.js:1-25, evaluated in double like the JS, stored as f32
static double window_value(int type, int i, int n) {
    const double x = 2.0 * M_PI * i / (n - 1);
    switch (type) {
        case WFB_WINDOW_HAMMING: return 0.54 - 0.46 * cos(x);
        case WFB_WINDOW_BLACKMAN: return 0.42 - 0.5 * cos(x) + 0.08 * cos(2 * x);
        case WFB_WINDOW_BLACKMAN_HARRIS: return 0.35875 - 0.48829 * cos(x) + 0.14128 * cos(2 * x) - 0.01168 * cos(3 * x);
        case WFB_WINDOW_RECTANGULAR: return 1.0;
        default: return 0.5 * (1.0 - cos(x));
    }
}

static int stft_init(wfb_stft *st) {
    CK(cudaSetDevice(st->device));
    CK(cudaStreamCreateWithFlags(&st->stream, cudaStreamNonBlocking));
    const int n = st->fft_size, m = n / 2;
    const StftVariant &v = *st->variant;
    std::vector<float> bre, bim, fwd, fwd_span, rre, rim, packed, win(st->wsize);
    base_twiddles<float>(scalar_f32_flavour(m, TW_F32_SPLIT), m, m, bre, bim);
    auto tables = [&](const std::vector<int> &radices, std::vector<float> &t) {
        stage_tables<float>(radices, m, bre, bim, false, t);
        w8_opening(m, radices, t);
    };
    tables(v.radices, fwd);
    if (!v.span_radices.empty() && v.span_radices != v.radices) tables(v.span_radices, fwd_span);   // the span kernel's core plan groups the stages differently
    base_twiddles<float>(TW_F32_SPLIT, n, m + 1, rre, rim);
    for (int k = 0; k <= m; k++) { packed.push_back(rre[k]); packed.push_back(rim[k]); }
    for (int i = 0; i < st->wsize; i++) win[i] = (float)window_value(st->window, i, st->wsize);
    // one allocation and one copy: [forward | span forward | W_n^k | window | filter bands | filter weights], each
    // 256-byte aligned (the last two are empty but for filterbank handles)
    const std::pair<const void *, size_t> sec[6] = {
        {fwd.data(), fwd.size() * sizeof(float)}, {fwd_span.data(), fwd_span.size() * sizeof(float)},
        {packed.data(), packed.size() * sizeof(float)}, {win.data(), win.size() * sizeof(float)},
        {st->fb_band.data(), st->fb_band.size() * sizeof(int)}, {st->fb_w.data(), st->fb_w.size() * sizeof(float)}};
    size_t off[7] = {0};
    for (int i = 0; i < 6; i++) off[i + 1] = off[i] + up256(sec[i].second);
    std::vector<unsigned char> blob(off[6], 0);
    for (int i = 0; i < 6; i++) if (sec[i].second) memcpy(blob.data() + off[i], sec[i].first, sec[i].second);
    CK(cudaMalloc(&st->d_tables, blob.size()));
    // stream-ordered on the handle's stream and completed here: launches on ANY stream may follow
    CK(cudaMemcpyAsync(st->d_tables, blob.data(), blob.size(), cudaMemcpyHostToDevice, st->stream));
    CK(cudaStreamSynchronize(st->stream));
    unsigned char *d = (unsigned char *)st->d_tables;
    st->d_tw = d;
    st->d_tw_span = fwd_span.empty() ? nullptr : d + off[1];
    st->d_rtw = d + off[2];
    st->d_window = d + off[3];
    st->d_fb_band = st->fb_band.empty() ? nullptr : d + off[4];
    st->d_fb_w = st->fb_w.empty() ? nullptr : d + off[5];
    if (!(st->flags & WFB_PLAN_NO_DEVICE_BUFFERS)) {
        if (cudaMalloc(&st->d_samples, st->in_bytes) != cudaSuccess) { cudaGetLastError(); return WFB_ERR_ALLOC; }
        if (cudaMalloc(&st->d_out, st->out_bytes) != cudaSuccess) { cudaGetLastError(); return WFB_ERR_ALLOC; }
    }
    if (!(st->flags & WFB_PLAN_NO_HOST_BUFFERS)) {
        if (cudaHostAlloc(&st->h_samples, st->in_bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return WFB_ERR_ALLOC; }
        if (cudaHostAlloc(&st->h_out, st->out_bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return WFB_ERR_ALLOC; }
        memset(st->h_samples, 0, st->in_bytes);
        memset(st->h_out, 0, st->out_bytes);
    }
    return WFB_OK;
}

// The STFT kernel for these pointers (STFT_DIRECT, STFT_SPAN or STFT_PIPE).  The bulk-copy kernels (span, pipe) copy
// frames or tile spans into shared memory, so frame starts and sizes must be 16-byte aligned in every signal.
static int stft_route(const wfb_stft *st, const float *d_samples, const void *d_out) {
    const StftVariant &v = *st->variant;
    const bool rows16 = ((uintptr_t)d_samples % 16) == 0 && (st->batch == 1 || st->num_samples % 4 == 0);
    const bool bulk = st->hop % 4 == 0 && st->wsize % 4 == 0 && rows16;
    // span kernel: whole tiles of overlapping frames as one bulk copy in, and one bulk store out; very large hops make
    // the span too large for shared memory
    const char *span_env = getenv("WFB_STFT_SPAN");             // (read per call: tests and A/B runs flip it)
    const bool span_on = span_env ? atoi(span_env) != 0 : v.span_default;      // WFB_STFT_SPAN=1 forces, =0 forbids
    if (span_on && v.launch[STFT_SPAN] && bulk && ((uintptr_t)d_out % 16) == 0 &&
        v.span_fixed_bytes + stft_span_bytes(v.span_frames, st->hop, st->wsize) <= STFT_SPAN_SMEM_MAX)
        return STFT_SPAN;
    const char *pipe_env = getenv("WFB_STFT_PIPE_MIN_N");       // (read per call, like WFB_STFT_SPAN)
    const int pipe_min = pipe_env ? atoi(pipe_env) : 8192;
    return st->fft_size >= pipe_min && bulk ? STFT_PIPE : STFT_DIRECT;
}

extern "C" {

wfb_stft *wfb_stft_create(int fft_size, int zero_padding, int hop, int window_type, long num_samples, int mode,
                          float gain_db, float range_db, int device, int flags, int *err) {
    return wfb_stft_create_ex(fft_size, zero_padding, hop, window_type, num_samples, 1, mode, gain_db, range_db, device, flags, err);
}

}  // extern "C"

// The geometry checks and the handle of every mode, before its tables are built: the caller has checked fft_size and its
// mode's own arguments.  row_floats: output floats per frame.
static wfb_stft *stft_new(int fft_size, int zero_padding, int hop, int window_type, long num_samples, long batch, int mode,
                          size_t row_floats, int device, int flags, int *err) {
    if (zero_padding < 1 || !is_pow2(zero_padding) || zero_padding > fft_size / 2 || hop < 1 ||
        window_type < 0 || window_type > WFB_WINDOW_RECTANGULAR) { *err = WFB_ERR_BAD_ARG; return nullptr; }
    const int wsize = fft_size / zero_padding;
    if (num_samples < wsize) { *err = WFB_ERR_BAD_ARG; return nullptr; }      // "Audio too short" (spectrogram.js:299-301)
    // the whole batch's input and output must be addressable: batch * num_samples floats, batch * frames * row values
    const size_t frames = (size_t)((num_samples - wsize) / hop + 1);
    const size_t row_bytes = row_floats * sizeof(float);
    size_t in_bytes, out_bytes;
    if (batch < 1 || __builtin_mul_overflow((size_t)num_samples, sizeof(float), &in_bytes) ||
        __builtin_mul_overflow(in_bytes, (size_t)batch, &in_bytes) || __builtin_mul_overflow(frames, row_bytes, &out_bytes) ||
        __builtin_mul_overflow(out_bytes, (size_t)batch, &out_bytes)) { *err = WFB_ERR_BAD_ARG; return nullptr; }
    *err = check_device(device);
    if (*err) return nullptr;
    wfb_stft *st = new wfb_stft();
    st->fft_size = fft_size; st->wsize = wsize; st->hop = hop; st->device = device; st->flags = flags;
    st->mode = mode;
    st->window = window_type;
    st->num_samples = num_samples;
    st->frames = (long)frames;
    st->batch = batch;
    st->in_bytes = in_bytes;
    st->out_bytes = out_bytes;
    for (const StftVariant &v : variants_stft()) if (v.core_n == fft_size / 2) st->variant = &v;
    if (!st->variant) { *err = WFB_ERR_BAD_SIZE; delete st; return nullptr; }
    for (const IstftVariant &v : variants_istft()) if (v.core_n == fft_size / 2) st->inv_variant = &v;
    return st;
}

static wfb_stft *stft_ready(wfb_stft *st, int *err) {
    *err = stft_init(st);
    if (*err) { wfb_stft_destroy(st); return nullptr; }
    return st;
}

extern "C" {

wfb_stft *wfb_stft_create_ex(int fft_size, int zero_padding, int hop, int window_type, long num_samples, long batch, int mode,
                             float gain_db, float range_db, int device, int flags, int *err) {
    int dummy;
    if (!err) err = &dummy;
    if (!is_pow2(fft_size) || fft_size < 64 || fft_size > 8192) { *err = WFB_ERR_BAD_SIZE; return nullptr; }
    if ((mode != WFB_STFT_DB && mode != WFB_STFT_COMPLEX) || !(range_db > 0.0f)) { *err = WFB_ERR_BAD_ARG; return nullptr; }
    const size_t row_floats = (size_t)(fft_size / 2 + 1) * (mode == WFB_STFT_COMPLEX ? 2 : 1);
    wfb_stft *st = stft_new(fft_size, zero_padding, hop, window_type, num_samples, batch, mode, row_floats, device, flags, err);
    if (!st) return nullptr;
    st->db_floor = gain_db - range_db;
    st->inv_range = 1.0f / range_db;
    return stft_ready(st, err);
}

wfb_stft *wfb_stft_create_filterbank(int fft_size, int zero_padding, int hop, int window_type, long num_samples, long batch,
                                     int num_filters, const float *filters, int power, float log_scale, float log_offset,
                                     float log_floor, int device, int flags, int *err) {
    int dummy;
    if (!err) err = &dummy;
    if (!is_pow2(fft_size) || fft_size < 64 || fft_size > 8192) { *err = WFB_ERR_BAD_SIZE; return nullptr; }
    const int bins = fft_size / 2 + 1;
    const bool log_ok = std::isfinite(log_scale) &&
        (log_scale == 0.0f || (std::isfinite(log_floor) && log_floor > 0.0f && std::isfinite(log_offset) && log_offset >= 0.0f));
    if (num_filters < 1 || num_filters > bins || !filters || (power != 1 && power != 2) || !log_ok) {
        *err = WFB_ERR_BAD_ARG;
        return nullptr;
    }
    for (size_t i = 0; i < (size_t)num_filters * bins; i++)
        if (!std::isfinite(filters[i])) { *err = WFB_ERR_BAD_ARG; return nullptr; }
    wfb_stft *st = stft_new(fft_size, zero_padding, hop, window_type, num_samples, batch, STFT_MODE_FILTERBANK,
                            (size_t)num_filters, device, flags, err);
    if (!st) return nullptr;
    st->num_filters = num_filters;
    st->power = power;
    st->log_scale = log_scale; st->log_offset = log_offset; st->log_floor = log_floor;
    // each filter's band runs from its first to its last non-zero weight (zeros inside it stay); all zero: 0 bins
    for (int m = 0; m < num_filters; m++) {
        const float *f = filters + (size_t)m * bins;
        int lo = 0, hi = bins - 1;
        while (lo < bins && f[lo] == 0.0f) lo++;
        while (hi >= lo && f[hi] == 0.0f) hi--;
        const int count = lo < bins ? hi - lo + 1 : 0;
        st->fb_band.insert(st->fb_band.end(), {count ? lo : 0, count, (int)st->fb_w.size(), 0});
        st->fb_w.insert(st->fb_w.end(), f + lo, f + lo + count);
    }
    return stft_ready(st, err);
}

void wfb_stft_destroy(wfb_stft *st) {
    if (!st) return;
    cudaSetDevice(st->device);
    if (st->stream) { cudaStreamSynchronize(st->stream); cudaStreamDestroy(st->stream); }
    void *d[] = {st->d_tables, st->d_samples, st->d_out, st->d_tw_inv};
    for (void *p : d) if (p) cudaFree(p);
    if (st->inv_ready) cudaEventDestroy(st->inv_ready);
    if (st->h_samples) cudaFreeHost(st->h_samples);
    if (st->h_out) cudaFreeHost(st->h_out);
    delete st;
}

long wfb_stft_frames(wfb_stft *st) { return st ? st->frames : 0; }
long wfb_stft_batch(wfb_stft *st) { return st ? st->batch : 0; }
int wfb_stft_bins(wfb_stft *st) { return st ? st->fft_size / 2 + 1 : 0; }
int wfb_stft_filters(wfb_stft *st) { return st ? st->num_filters : 0; }
void *wfb_stft_host_samples(wfb_stft *st) { return st ? st->h_samples : nullptr; }
void *wfb_stft_host_output(wfb_stft *st) { return st ? st->h_out : nullptr; }
size_t wfb_stft_output_bytes(wfb_stft *st) { return st ? st->out_bytes : 0; }
size_t wfb_stft_algorithmic_bytes(wfb_stft *st) { return st ? st->in_bytes + st->out_bytes : 0; }

int wfb_stft_exec_device(wfb_stft *st, const float *d_samples, void *d_out, void *stream) {
    if (!st || !d_samples || !d_out) return WFB_ERR_BAD_ARG;
    CK(cudaSetDevice(st->device));
    StftParams sp;
    sp.samples = d_samples; sp.window = (const float *)st->d_window; sp.out = d_out;
    sp.tw = st->d_tw; sp.rtw = st->d_rtw;
    sp.frames = st->frames; sp.batch = st->batch; sp.num_samples = st->num_samples; sp.hop = st->hop; sp.wsize = st->wsize; sp.mode = st->mode;
    sp.db_floor = st->db_floor; sp.inv_range = st->inv_range; sp.inv_half_n = 2.0f / (float)st->fft_size;
    sp.ctr = nullptr;
    sp.span_bytes = 0;
    sp.tiles = 0; sp.tps = sp.tps_magic = 0; sp.tps_shift = 0;      // (set by the persistent kernels' launchers)
    sp.fb_band = (const int4 *)st->d_fb_band; sp.fb_w = (const float *)st->d_fb_w;
    sp.fb_n = st->num_filters; sp.fb_power = st->power;
    sp.fb_scale = st->log_scale; sp.fb_offset = st->log_offset; sp.fb_floor = st->log_floor;
    // a caller's pointer may be any float address (scalar loads then); the rows of a batch keep the base's alignment only
    // when num_samples is a multiple of 2 (8 bytes) or 4 (16 bytes, the bulk-copy kernels: stft_route)
    sp.aligned8 = ((uintptr_t)d_samples % 8) == 0 && (st->batch == 1 || st->num_samples % 2 == 0);
    // fast dB path: v = lg_a * log2(|2 X|^2) + lg_b  ==  (10 log10(|X|^2 c^2) - floor) / range,  c = 2 / fft_size
    sp.lg_a = 3.0102999566398120f * st->inv_range;
    sp.lg_b = sp.lg_a * (2.0f * log2f(sp.inv_half_n) - 2.0f) - st->db_floor * st->inv_range;
    const int route = stft_route(st, d_samples, d_out);
    if (route == STFT_SPAN && st->d_tw_span) sp.tw = st->d_tw_span;
    cudaError_t e = st->variant->launch[route](sp, stream ? (cudaStream_t)stream : st->stream);
    if (e != cudaSuccess) return cuda_fail(e, "stft launch");
    return WFB_OK;
}

int wfb_stft_exec(wfb_stft *st, int flags) {
    if (!st || !st->d_samples) return WFB_ERR_BAD_ARG;
    if ((flags & (WFB_STAGE_H2D | WFB_STAGE_D2H)) && !st->h_samples) return WFB_ERR_NO_HOST_BUFFERS;
    CK(cudaSetDevice(st->device));
    if (flags & WFB_STAGE_H2D) CK(cudaMemcpyAsync(st->d_samples, st->h_samples, st->in_bytes, cudaMemcpyHostToDevice, st->stream));
    int rc = wfb_stft_exec_device(st, (const float *)st->d_samples, st->d_out, nullptr);
    if (rc) return rc;
    if (flags & WFB_STAGE_D2H) CK(cudaMemcpyAsync(st->h_out, st->d_out, st->out_bytes, cudaMemcpyDeviceToHost, st->stream));
    if (flags & WFB_SYNC) CK(cudaStreamSynchronize(st->stream));
    return WFB_OK;
}

// Inverse stage tables of the inverse kernel's core plan (the c2r convention: the forward base table conjugated, no
// W_8 opening constants), uploaded on `cs` ahead of the launch that follows; calls on any other stream wait for the upload.
static int stft_inverse_tables(wfb_stft *st, cudaStream_t cs) {
    if (st->d_tw_inv) {
        CK(cudaStreamWaitEvent(cs, st->inv_ready, 0));
        return WFB_OK;
    }
    const int m = st->fft_size / 2;
    std::vector<float> bre, bim, inv;
    base_twiddles<float>(scalar_f32_flavour(m, TW_F32_SPLIT), m, m, bre, bim);
    stage_tables<float>(st->inv_variant->radices, m, bre, bim, true, inv);
    if (inv.empty()) inv.assign(2, 0.0f);
    void *d = nullptr;
    CK(cudaMalloc(&d, inv.size() * sizeof(float)));
    cudaError_t e = cudaMemcpyAsync(d, inv.data(), inv.size() * sizeof(float), cudaMemcpyHostToDevice, cs);
    if (e == cudaSuccess && !st->inv_ready) e = cudaEventCreateWithFlags(&st->inv_ready, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventRecord(st->inv_ready, cs);
    if (e != cudaSuccess) { cudaFree(d); return cuda_fail(e, "stft inverse tables"); }
    st->d_tw_inv = d;
    return WFB_OK;
}

int wfb_stft_exec_inverse_device(wfb_stft *st, const void *d_spectra, float *d_samples, void *stream) {
    if (!st || !d_spectra || !d_samples) return WFB_ERR_BAD_ARG;
    if (st->mode != WFB_STFT_COMPLEX) return WFB_ERR_UNSUPPORTED;      // dB magnitudes have no inverse
    if (((uintptr_t)d_spectra % 8) != 0) return WFB_ERR_BAD_ARG;
    const uintptr_t s0 = (uintptr_t)d_spectra, s1 = s0 + st->out_bytes;
    const uintptr_t x0 = (uintptr_t)d_samples, x1 = x0 + st->in_bytes;
    if (s0 < x1 && x0 < s1) return WFB_ERR_BAD_ARG;
    if (!st->inv_variant) return WFB_ERR_BAD_SIZE;
    CK(cudaSetDevice(st->device));
    cudaStream_t cs = stream ? (cudaStream_t)stream : st->stream;
    int rc = stft_inverse_tables(st, cs);
    if (rc) return rc;
    const IstftVariant &v = *st->inv_variant;
    const int X = v.frames_per_round;
    // a CTA owns P hops of output and recomputes the halo = ceil(W/H) - 1 frames before them: P + halo is a whole number
    // of rounds and P >= 10 halo (<= 10 % recomputed frames), and at least 16 frames
    const long H = st->hop, W = st->wsize, halo = (W + H - 1) / H - 1;
    const long rounds = std::max((11 * halo + X - 1) / X, (16L + X - 1) / X);
    IstftParams ip;
    ip.spectra = (const float2 *)d_spectra; ip.out = d_samples; ip.window = (const float *)st->d_window;
    ip.tw = st->d_tw_inv; ip.rtw = st->d_rtw;
    ip.frames = st->frames; ip.num_samples = st->num_samples;
    ip.tile_frames = rounds * X - halo;
    ip.tiles = (st->num_samples + ip.tile_frames * H - 1) / (ip.tile_frames * H);
    ip.hop = st->hop; ip.wsize = st->wsize; ip.halo = (int)halo;
    ip.inv_hop = 1.0f / (float)st->hop;
    cudaError_t e = v.launch(ip, ip.tiles * st->batch, cs);
    if (e != cudaSuccess) return cuda_fail(e, "stft inverse launch");
    return WFB_OK;
}

int wfb_stft_exec_inverse(wfb_stft *st, int flags) {
    if (!st || !st->d_samples) return WFB_ERR_BAD_ARG;
    if (st->mode != WFB_STFT_COMPLEX) return WFB_ERR_UNSUPPORTED;
    if ((flags & (WFB_STAGE_H2D | WFB_STAGE_D2H)) && !st->h_out) return WFB_ERR_NO_HOST_BUFFERS;
    CK(cudaSetDevice(st->device));
    if (flags & WFB_STAGE_H2D) CK(cudaMemcpyAsync(st->d_out, st->h_out, st->out_bytes, cudaMemcpyHostToDevice, st->stream));
    int rc = wfb_stft_exec_inverse_device(st, st->d_out, (float *)st->d_samples, nullptr);
    if (rc) return rc;
    if (flags & WFB_STAGE_D2H) CK(cudaMemcpyAsync(st->h_samples, st->d_samples, st->in_bytes, cudaMemcpyDeviceToHost, st->stream));
    if (flags & WFB_SYNC) CK(cudaStreamSynchronize(st->stream));
    return WFB_OK;
}

}  // extern "C"
