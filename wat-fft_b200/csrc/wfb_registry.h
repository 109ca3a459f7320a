// wfb_registry.h -- kernel-variant registry shared by the variant translation units and the API.
//
// Each wfb_variants_*.cu instantiates a family of kernels and returns one descriptor (Variant) per entry.  A Variant
// describes its launches as data: per operation (c2c split / interleaved x forward / inverse, r2c, c2r) the kernel,
// threads per CTA, batch rows per work item and dynamic shared memory; launch_op turns one of them into a launch.  A
// plan (wfb_api.cu) holds every registered variant of its (precision, core size, kind), ordered by priority: the first
// is the default, the others stay selectable (wfb_plan_set_variant) for tuning and parity tests.
#pragma once
#include "wfb_kernels.cuh"

#include <array>
#include <vector>

namespace wfb {

// the operations of a variant; c2c and real operations are (base + direction), direction WFB_FORWARD = 0 / WFB_INVERSE = 1
enum { OP_SPLIT_FWD, OP_SPLIT_INV, OP_IL_FWD, OP_IL_INV, OP_R2C, OP_C2R, NOPS };
// one operation's launch: `kernel` null = the variant does not do it; a work item is one CTA of a grid kernel or one
// tile of a persistent one
struct OpLaunch {
    const void *kernel;
    int threads;
    int rows_per_item;
    size_t smem;
};
typedef std::array<OpLaunch, NOPS> OpLaunches;

struct Variant {
    const char *name;
    int core_n;        // complex points of the core transform (n for C2C, n/2 for R2C)
    int lanes;         // batch rows per thread group: 2 for the packed-FP32 (f32x2) kernels
    int priority;      // larger = preferred default (set from measurements, profiles/)
    int priority_inv;  // same for the inverse direction (c2r / ifft)
    int priority_il;   // same for interleaved c2c layouts
    int align;         // required alignment (bytes) of every plane pointer: 16 for the TMA / float4 kernels,
                       // one complex value for the direct kernels (one scalar when the layout is split)
    std::vector<int> radices;
    OpLaunches ops;
    bool persistent;   // grid = resident CTAs claiming tiles from a counter (KParams::ctr)
    bool direct;       // plain global loads/stores, one launch-sized grid (no TMA pipeline, no tile counter): the zero-copy path's kernel
};

// Every kernel launch of the library (wfb_api.cu: one launch counter, one attribute and occupancy cache).  `params` is
// the kernel's one parameter struct; `smem_attr` is the dynamic shared-memory limit set once per (device, kernel).  With
// `ctr` (the struct's tile-counter field) the launch is persistent: it gets a zeroed counter and at most as many CTAs
// as are resident on the whole GPU; otherwise the grid is `work_items` CTAs.
cudaError_t launch(const void *kernel, size_t smem, size_t smem_attr, int threads, long work_items, void *params,
                   unsigned long long **ctr, cudaStream_t s);
template <class P> cudaError_t launch_grid(const void *kernel, size_t smem, int threads, long ctas, const P &p, cudaStream_t s) {
    return launch(kernel, smem, smem, threads, ctas, (void *)&p, nullptr, s);
}
template <class P> cudaError_t launch_persistent(const void *kernel, size_t smem, int threads, long work_items, const P &p, cudaStream_t s) {
    P q = p;
    return launch(kernel, smem, smem, threads, work_items, &q, &q.ctr, s);
}
// operation `op` of `v` over `rows` batch rows (a persistent kernel's counter goes to p.ctr); a variant without that
// operation gives cudaErrorInvalidDeviceFunction
inline cudaError_t launch_op(const Variant &v, int op, KParams &p, long rows, cudaStream_t s) {
    const OpLaunch &l = v.ops[op];
    if (!l.kernel) return cudaErrorInvalidDeviceFunction;
    return launch(l.kernel, l.smem, l.smem, l.threads, (rows + l.rows_per_item - 1) / l.rows_per_item, &p,
                  v.persistent ? &p.ctr : nullptr, s);
}

const std::vector<Variant> &variants_f32_direct();
const std::vector<Variant> &variants_f32_x2();
const std::vector<Variant> &variants_f32_tile();
const std::vector<Variant> &variants_f32_pipe();
const std::vector<Variant> &variants_f64();
const std::vector<Variant> &variants_f32_real_pipe();
const std::vector<Variant> &variants_f64_pipe();

template <class PL> std::vector<int> plan_radices() {
    std::vector<int> r;
    for (int p = 0; p < PL::npass(); p++)
        for (int q = 0; q < pass_nsub(PL::code(p)); q++) r.push_back(pass_radix(PL::code(p), q));
    return r;
}

// the descriptor every family's make() returns; priority_inv and priority_il default (-1) to `priority`
template <class PL> Variant make_variant(const char *name, int priority, int priority_inv, int priority_il, int lanes, int align,
                                         bool persistent, const OpLaunches &ops, bool direct = false) {
    return Variant{name, PL::N, lanes, priority, priority_inv < 0 ? priority : priority_inv, priority_il < 0 ? priority : priority_il,
                   align, plan_radices<PL>(), ops, persistent, direct};
}
// the c2c records of a family: k(io, inverse) is the kernel instantiation; SPLIT = false leaves the split layout without one
template <bool SPLIT, class K> void c2c_ops(OpLaunches &ops, int threads, int rows_per_item, size_t smem, K k) {
    using std::integral_constant;
    if constexpr (SPLIT) {
        ops[OP_SPLIT_FWD] = {k(integral_constant<int, IO_SPLIT>{}, std::false_type{}), threads, rows_per_item, smem};
        ops[OP_SPLIT_INV] = {k(integral_constant<int, IO_SPLIT>{}, std::true_type{}), threads, rows_per_item, smem};
    }
    ops[OP_IL_FWD] = {k(integral_constant<int, IO_INTERLEAVED>{}, std::false_type{}), threads, rows_per_item, smem};
    ops[OP_IL_INV] = {k(integral_constant<int, IO_INTERLEAVED>{}, std::true_type{}), threads, rows_per_item, smem};
}

constexpr int PADQ = 16;   // one pad slot per 16 complex values: conflict-free for every plan (tools/bank_sim.py)

// one transform (or lane pair) per thread group, X groups per CTA, direct global loads/stores
template <typename R, class PL, int X, int MINB, bool SPLIT_IO> struct Launchers {
    static constexpr size_t smem = sizeof(cx<R>) * (size_t)padded_size<PADQ>(PL::N) * X;
    static constexpr int LANES = RT<R>::LANES;
    static Variant make(const char *name, int priority, int priority_inv = -1, int priority_il = -1) {
        OpLaunches ops{};
        c2c_ops<SPLIT_IO>(ops, PL::T * X, X * LANES, smem, [](auto io, auto inv) {
            return (const void *)k_c2c<R, PL, X, PADQ, decltype(io)::value, decltype(inv)::value, MINB>;
        });
        ops[OP_R2C] = {(const void *)k_r2c<R, PL, X, PADQ, MINB>, PL::T * X, X * LANES, smem};
        ops[OP_C2R] = {(const void *)k_c2r<R, PL, X, PADQ, MINB>, PL::T * X, X * LANES, smem};
        return make_variant<PL>(name, priority, priority_inv, priority_il, LANES, 2 * (int)sizeof(typename RT<R>::scalar), false, ops, true);
    }
};

// persistent TMA-pipelined c2c: grid = resident CTAs, each loops over tiles of X*LANES rows
template <typename R, class PL, int X, int MINB, int RC = 0, int PQ = PADQ, bool TS = false, bool HT = false> struct PipeLaunchers {
    static constexpr size_t smem = 2 * pipe_buf_bytes<R, PL, PQ, X>() + 64;
    static constexpr int LANES = RT<R>::LANES;
    static Variant make(const char *name, int priority, int priority_inv = -1, int priority_il = -1) {
        OpLaunches ops{};
        c2c_ops<true>(ops, PL::T * X, X * LANES, smem, [](auto io, auto inv) {
            return (const void *)k_c2c_pipe<R, PL, X, PQ, decltype(io)::value, decltype(inv)::value, MINB, RC, TS, HT>;
        });
        return make_variant<PL>(name, priority, priority_inv, priority_il, LANES, 16, true, ops);
    }
};

// register-prefetch persistent c2c (k_c2c_rpf): one transform per CTA iteration
template <typename R, class PL, int MINB, bool TS, int PQ = PADQ> struct RegPipeLaunchers {
    static constexpr size_t smem = (TS ? 2 : 1) * pipe_buf_bytes<R, PL, PQ, 1>() + 64;
    static Variant make(const char *name, int priority, int priority_inv = -1, int priority_il = -1) {
        OpLaunches ops{};
        c2c_ops<true>(ops, PL::T, 1, smem, [](auto io, auto inv) {
            return (const void *)k_c2c_rpf<R, PL, PQ, decltype(io)::value, decltype(inv)::value, MINB, TS>;
        });
        // TS: bulk stores need 16-byte aligned rows; the loads are plain element loads either way
        return make_variant<PL>(name, priority, priority_inv, priority_il, 1, TS ? 16 : 2 * (int)sizeof(typename RT<R>::scalar), true, ops);
    }
};

// persistent TMA-pipelined r2c / c2r (scalar lanes)
// XI: rows per tile of the c2r direction (1 = single-row tiles with shifted bulk copies, see k_real_pipe)
template <typename R, class PL, int X, int MINB, bool RC = false, int PQ = PADQ, bool TS = false, int XI = X, bool HT = false> struct RealPipeLaunchers {
    static constexpr size_t smem_f = 2 * real_pipe_buf_bytes<R, PL, PQ, X, false>() + 64;
    static constexpr size_t smem_i = 2 * real_pipe_buf_bytes<R, PL, PQ, XI, true>() + 64;
    static Variant make(const char *name, int priority, int priority_inv = -1, int priority_il = -1) {
        OpLaunches ops{};
        ops[OP_R2C] = {(const void *)k_real_pipe<R, PL, X, PQ, false, MINB, RC, TS, HT>, PL::T * X, X, smem_f};
        ops[OP_C2R] = {(const void *)k_real_pipe<R, PL, XI, PQ, true, MINB, false, TS, HT>, PL::T * XI, XI, smem_i};
        return make_variant<PL>(name, priority, priority_inv, priority_il, 1, 16, true, ops);
    }
};

// thread-per-row tile kernels (N <= 64)
template <class PL, int X, int MINB> struct TileLaunchers {
    static constexpr size_t smem = sizeof(float) * 2 * (size_t)(PL::N + 2) * X;
    static Variant make(const char *name, int priority, int priority_inv = -1, int priority_il = -1) {
        OpLaunches ops{};
        c2c_ops<true>(ops, X, X, smem, [](auto io, auto inv) {
            return (const void *)k_c2c_tile<float, PL, X, decltype(io)::value, decltype(inv)::value, MINB>;
        });
        return make_variant<PL>(name, priority, priority_inv, priority_il, 1, 16, false, ops);
    }
};

// persistent, fully TMA-fed thread-per-row c2c (N <= 64); the f64 kernels are interleaved only
template <class PL, int X, int MINB, typename R = float> struct TilePipeLaunchers {
    static constexpr bool F64 = sizeof(R) == 8;
    static constexpr size_t smem_i = 2 * tpipe_buf_bytes<R, PL, X, IO_INTERLEAVED>() + 64;
    static constexpr size_t smem_s = F64 ? 0 : 2 * tpipe_buf_bytes<float, PL, X, IO_SPLIT>() + 64;
    static constexpr size_t smem = smem_s > smem_i ? smem_s : smem_i;
    static Variant make(const char *name, int priority, int priority_inv = -1, int priority_il = -1) {
        OpLaunches ops{};
        c2c_ops<!F64>(ops, X, X, smem, [](auto io, auto inv) {
            return (const void *)k_c2c_tpipe<R, PL, X, decltype(io)::value, decltype(inv)::value, MINB>;
        });
        return make_variant<PL>(name, priority, priority_inv, priority_il, 1, 16, true, ops);
    }
};

// persistent, fully TMA-fed thread-per-row r2c / c2r (N = 64, 128)
template <class PL, int X, int MINB, typename R = float> struct RealTilePipeLaunchers {
    static constexpr size_t smem = 2 * rtpipe_buf_bytes<R, PL, X>() + 64;
    static Variant make(const char *name, int priority, int priority_inv = -1, int priority_il = -1) {
        OpLaunches ops{};
        ops[OP_R2C] = {(const void *)k_real_tpipe<R, PL, X, false, MINB>, X, X, smem};
        ops[OP_C2R] = {(const void *)k_real_tpipe<R, PL, X, true, MINB>, X, X, smem};
        return make_variant<PL>(name, priority, priority_inv, priority_il, 1, 16, true, ops);
    }
};

// thread-per-row tile kernels for the real transforms (core M <= 64)
template <class PL, int X, int MINB> struct RealTileLaunchers {
    static constexpr size_t smem = sizeof(float) * (size_t)(2 * PL::N + 4) * X;
    static Variant make(const char *name, int priority, int priority_inv = -1, int priority_il = -1) {
        OpLaunches ops{};
        ops[OP_R2C] = {(const void *)k_r2c_tile<PL, X, MINB>, X, X, smem};
        ops[OP_C2R] = {(const void *)k_c2r_tile<PL, X, MINB>, X, X, smem};
        return make_variant<PL>(name, priority, priority_inv, priority_il, 1, 16, false, ops);
    }
};

// fused STFT (frame gather + window + r2c + magnitude/dB): three kernels, picked per call by stft_route (wfb_api.cu)
enum { STFT_DIRECT = 0, STFT_SPAN = 1, STFT_PIPE = 2 };
typedef cudaError_t (*stft_launch_fn)(const StftParams &sp, cudaStream_t s);
struct StftVariant {
    const char *name; int core_n; std::vector<int> radices;
    stft_launch_fn launch[3];          // by route (STFT_DIRECT, STFT_SPAN, STFT_PIPE); no span kernel below N = 256
    std::vector<int> span_radices;     // stage structure of the span kernel's core plan (its own twiddle table when it differs)
    int span_frames = 0;               // span kernel: frames per tile ...
    size_t span_fixed_bytes = 0;       // ... and its shared memory besides the span stage
    bool span_default = false;         // measured faster than the direct kernel at hop = N/4 (profiles/): used unless WFB_STFT_SPAN says otherwise
};
const std::vector<StftVariant> &variants_stft();
constexpr size_t STFT_SPAN_SMEM_MAX = 200 * 1024;      // the span kernel's shared-memory limit; larger spans take another kernel
// the span stage of k_stft_span: the samples of `frames` overlapping frames, in whole 128-byte lines
inline size_t stft_span_bytes(int frames, int hop, int wsize) {
    return ((size_t)((long)(frames - 1) * hop + wsize) * sizeof(float) + 127) / 128 * 128;
}
// kernel flavour: fast dB / exact dB / complex / filterbank output.  The fast form drops the +1e-10 of magnitudeToDb,
// which lowers a value by 20 log10(1 + 1e-10 / (|X| c)) dB, the most at the floor (gain - range): it runs only where that
// is at most 1e-6 of the [0, 1] output there (floors down to about -99 dB at range 80)
inline int stft_flavour(const StftParams &sp) {
    if (sp.mode == STFT_MODE_COMPLEX) return STFT_K_COMPLEX;
    if (sp.mode == STFT_MODE_FILTERBANK) return STFT_K_FB;
    const double worst = 20.0 * log10(1.0 + 1e-10 * pow(10.0, -(double)sp.db_floor / 20.0)) * (double)sp.inv_range;
    return worst > 1e-6 ? STFT_K_EXACT : STFT_K_FAST;
}
// the instantiation k(KM, PAD) of an STFT kernel for a flavour; the unpadded fast-dB case (window = FFT size, the
// spectrogram default) has its own instantiation without the per-element bound check; the others exist padded only
template <class K> const void *stft_kernel(int flavour, bool pad, K k) {
    using std::integral_constant;
    switch (flavour) {
        case STFT_K_FAST: return pad ? k(integral_constant<int, STFT_K_FAST>{}, std::true_type{}) : k(integral_constant<int, STFT_K_FAST>{}, std::false_type{});
        case STFT_K_EXACT: return k(integral_constant<int, STFT_K_EXACT>{}, std::true_type{});
        case STFT_K_FB: return k(integral_constant<int, STFT_K_FB>{}, std::true_type{});
        default: return k(integral_constant<int, STFT_K_COMPLEX>{}, std::true_type{});
    }
}
template <class PL, int X, int MINB, int PQ = PADQ> struct StftLaunchers {
    static constexpr size_t smem = sizeof(cx<float>) * (size_t)padded_size<PQ>(PL::N) * X;
    static cudaError_t direct(const StftParams &sp, cudaStream_t s) {
        const void *k = stft_kernel(stft_flavour(sp), sp.wsize < 2 * PL::N, [](auto km, auto pad) {
            return (const void *)k_stft<PL, X, PQ, MINB, decltype(km)::value, decltype(pad)::value>;
        });
        return launch_grid(k, smem, PL::T * X, (sp.frames * sp.batch + X - 1) / X, sp, s);
    }
    // pipelined variant: XP frames per CTA (>= one warp of threads)
    static constexpr int XP = (PL::T * X >= 128) ? X : 128 / PL::T;
    static constexpr size_t smem_pipe = 2 * real_pipe_buf_bytes<float, PL, PQ, XP, false>() + 64;
    static cudaError_t pipe(const StftParams &sp0, cudaStream_t s) {
        StftParams sp = sp0;
        sp.tps = (unsigned)((sp.frames + XP - 1) / XP);
        sp.tiles = (long)sp.tps * sp.batch;
        stft_tile_magic(sp);
        const void *k = stft_kernel(stft_flavour(sp), sp.wsize < 2 * PL::N, [](auto km, auto pad) {
            return (const void *)k_stft_pipe<PL, XP, PQ, MINB, decltype(km)::value, decltype(pad)::value>;
        });
        return launch_persistent(k, smem_pipe, PL::T * XP, sp.tiles, sp, s);
    }
    static StftVariant make(const char *name) { return StftVariant{name, PL::N, plan_radices<PL>(), {&direct, nullptr, &pipe}}; }
};

// span-staged persistent STFT (k_stft_span): SPL = core plan (may differ from the direct kernel's: the one-exchange plans
// the plain r2c kernels use), XS frames per tile.  Shared memory: the work area, the span stage, mbarriers/slots, window.
template <class PL, int X, int MINB, class SPL, int XS, int SMINB, int SPQ, bool DEFAULT> struct StftSpanLaunchers {
    static constexpr size_t fixed = stft_work_bytes<SPL, SPQ, XS>() + 128 + sizeof(float2) * SPL::N;
    static cudaError_t span(const StftParams &sp0, cudaStream_t s) {
        StftParams sp = sp0;
        const size_t stage = stft_span_bytes(XS, sp.hop, sp.wsize);
        sp.span_bytes = (int)stage;
        sp.tps = (unsigned)((sp.frames + XS - 1) / XS);
        sp.tiles = (long)sp.tps * sp.batch;
        stft_tile_magic(sp);
        const void *k = stft_kernel(stft_flavour(sp), sp.wsize < 2 * SPL::N, [](auto km, auto pad) {
            return (const void *)k_stft_span<SPL, XS, SPQ, SMINB, decltype(km)::value, decltype(pad)::value>;
        });
        return launch(k, fixed + stage, STFT_SPAN_SMEM_MAX, SPL::T * XS, sp.tiles, &sp, &sp.ctr, s);
    }
    static StftVariant make(const char *name) {
        static_assert(SPL::N == PL::N, "same core size");
        using D = StftLaunchers<PL, X, MINB>;
        return StftVariant{name, PL::N, plan_radices<PL>(), {&D::direct, &span, &D::pipe}, plan_radices<SPL>(), XS, fixed, DEFAULT};
    }
};

// fused inverse STFT (c2r + window + overlap-add, k_istft): one per FFT size, on the core plan of that size's STFT span
// kernel (the direct kernel's where there is none); X frames per round
typedef cudaError_t (*istft_launch_fn)(const IstftParams &ip, long tiles, cudaStream_t s);
struct IstftVariant {
    const char *name; int core_n; std::vector<int> radices; istft_launch_fn launch; int frames_per_round;
};
const std::vector<IstftVariant> &variants_istft();
template <class PL, int X, int PQ, int MINB> struct IstftLaunchers {
    static constexpr size_t smem = istft_smem_bytes<PL, PQ, X>();
    static cudaError_t launch(const IstftParams &ip, long tiles, cudaStream_t s) {
        return launch_grid((const void *)k_istft<PL, X, PQ, MINB>, smem, PL::T * X, tiles, ip, s);
    }
    static IstftVariant make(const char *name) { return IstftVariant{name, PL::N, plan_radices<PL>(), &launch, X}; }
};

#define XROWS(T) ((T) >= 256 ? 1 : 256 / (T))

// f32 core plans: the reference's split-core stage structure (radix-4, leading radix-2 for odd log2)
using F32_4 = Plan<4, 1, 0x4>;
using F32_8 = Plan<8, 1, 0x222>;
using F32_16 = Plan<16, 1, 0x44>;
using F32_32 = Plan<32, 2, 0x2, 0x44>;
using F32_64 = Plan<64, 4, 0x4, 0x44>;
using F32_128 = Plan<128, 8, 0x24, 0x44>;
using F32_256 = Plan<256, 16, 0x44, 0x44>;
using F32_512 = Plan<512, 32, 0x2, 0x44, 0x44>;
using F32_1024 = Plan<1024, 64, 0x4, 0x44, 0x44>;
using F32_2048 = Plan<2048, 128, 0x24, 0x44, 0x44>;
using F32_4096 = Plan<4096, 256, 0x44, 0x44, 0x44>;
using F32_8192 = Plan<8192, 512, 0x2, 0x44, 0x44, 0x44>;
// experimental: 32 values per thread (two register blocks per pass), half the threads per transform
using P32_4096_T128 = Plan<4096, 128, 0x44, 0x44, 0x44>;
using P32_2048_T64 = Plan<2048, 64, 0x24, 0x44, 0x44>;
// 64 values per thread: two passes, ONE shared-memory exchange (pad slot per 64 values: tools/bank_sim.py)
using P64_4096 = Plan<4096, 64, 0x444, 0x444>;
using P64_2048 = Plan<2048, 32, 0x244, 0x444>;
using P64_1024 = Plan<1024, 16, 0x44, 0x444>;
// 32 values per thread: two passes, one exchange; a 1024-point transform is ONE warp (no block barriers).
// f32 only (tolerance-based parity lets the stage radices be regrouped as 2,4,4 | 2,4,4).
using P32_1024 = Plan<1024, 32, 0x244, 0x244>;    // pad slot per 32 values
using P32_512 = Plan<512, 16, 0x244, 0x44>;
using P32_8192 = Plan<8192, 256, 0x244, 0x44, 0x44>;   // the same seven stages as F32_8192 in three passes instead of four
// thread-per-row plans for the tile kernels (whole transform in registers)
using T32_32 = Plan<32, 1, 0x244>;
using T32_64 = Plan<64, 1, 0x444>;
// f64 core plans: radix-4 for N = 4^p, radix-2 otherwise (fft_combined.wat:727-732)
using F64_4 = Plan<4, 1, 0x4>;
using F64_8 = Plan<8, 1, 0x222>;
using F64_16 = Plan<16, 1, 0x44>;
using F64_32 = Plan<32, 2, 0x2, 0x2222>;
using T64_32 = Plan<32, 1, 0x22222>;              // thread-per-row (same radix-2 stage sequence)
using F64_64 = Plan<64, 4, 0x4, 0x44>;
using F64_128 = Plan<128, 8, 0x222, 0x2222>;
using F64_256 = Plan<256, 16, 0x44, 0x44>;
using F64_512 = Plan<512, 32, 0x2, 0x2222, 0x2222>;
using F64_1024 = Plan<1024, 64, 0x4, 0x44, 0x44>;
using D32_512 = Plan<512, 16, 0x22222, 0x2222>;      // 32 values per thread: the same nine radix-2 stages, one exchange
using F64_2048 = Plan<2048, 128, 0x222, 0x2222, 0x2222>;
using F64_4096 = Plan<4096, 256, 0x44, 0x44, 0x44>;
using F64_8192 = Plan<8192, 512, 0x2, 0x2222, 0x2222, 0x2222>;

}  // namespace wfb
