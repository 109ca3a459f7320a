// wfb_kernels.cuh -- hand-written sm_100a batched FFT kernels (single HBM pass per transform).
//
// One engine serves the four transforms of the hot path.  Arithmetic follows the reference's
// Stockham autosort DIT stages -- radix-4 with an optional leading radix-2 for the f32 split core
// (modules/fft_split_native_f32.wat:748-888, :710-743), radix-4 for N = 4^p else radix-2 for f64
// (modules/fft_combined.wat:361-474, :486-716) -- so every product `table entry x operand` and
// every add/sub pairing is the one the reference forms (required for the f64 parity bound,
// SURVEY.md F4).  What is B200-specific is the execution: instead of log4(N) passes over memory,
// consecutive reference stages are fused into register-resident "passes" of combined radix up to
// 16 (each thread holds E = N/T complex values), with one padded shared-memory exchange between
// passes, coalesced global loads in the first pass and coalesced global stores in the last, so
// each transform crosses HBM exactly once in each direction.
//
// Index algebra (s = stride, l = groups, N = r*l*s for a stage of radix r):
//   stage reads   r*j*s + t + m*s   (group j < l, lane t < s, input m < r)
//   stage writes  j*s + t + q*N/r   (output q < r)
//   twiddle for input m: W_N^(m*j*N/(r*l))  = stage_table[(m-1)*l + j]
// A pass fusing stages of radices r1..rg (Rp = r1*...*rg) entered with l groups and leaving
// stride s' = N/(l*Rp) gives thread-block b = j*s' + t' the Rp inputs  Rp*s'*j + t' + k*s'
// and the Rp outputs  b + k'*(N/Rp),  k' = mixed-radix digit reversal of the register slot k.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include <utility>

namespace wfb {

// Compile-time loop: the body receives std::integral_constant<int, I>, so every index derived from it
// is a constant expression.  (A plain `#pragma unroll` loop left the plan's helper functions to be
// evaluated at run time: ncu showed 2.4x the expected instruction count.)
template <int... Is, class F>
__device__ __forceinline__ void static_for_impl(std::integer_sequence<int, Is...>, F &&f) {
    (f(std::integral_constant<int, Is>{}), ...);
}
template <int N, class F> __device__ __forceinline__ void static_for(F &&f) {
    static_for_impl(std::make_integer_sequence<int, N>{}, static_cast<F &&>(f));
}
#define CIDX(name, tag) constexpr int name = decltype(tag)::value

// ----------------------------------------------------------------------------------------
// compile-time plan description
// ----------------------------------------------------------------------------------------
// A pass is encoded as hex digits, most significant = first stage: 0x44 = radix-4 then radix-4.
__host__ __device__ constexpr int pass_nsub(int code) { int n = 0; while (code) { n++; code >>= 4; } return n; }
__host__ __device__ constexpr int pass_radix(int code, int q) { return (code >> (4 * (pass_nsub(code) - 1 - q))) & 0xF; }
__host__ __device__ constexpr int pass_rp(int code) { int r = 1; while (code) { r *= (code & 0xF); code >>= 4; } return r; }

template <int N_, int T_, int P0, int P1 = 0, int P2 = 0, int P3 = 0, int P4 = 0, int P5 = 0>
struct Plan {
    static constexpr int N = N_;          // complex points per transform
    static constexpr int T = T_;          // threads per transform
    static constexpr int E = N_ / T_;     // complex values held per thread
    static constexpr int MAXP = 6;
    __host__ __device__ static constexpr int code(int p) {
        return p == 0 ? P0 : p == 1 ? P1 : p == 2 ? P2 : p == 3 ? P3 : p == 4 ? P4 : p == 5 ? P5 : 0;
    }
    __host__ __device__ static constexpr int npass() { int n = 0; for (int p = 0; p < MAXP; p++) if (code(p)) n++; return n; }
    // groups on entry to pass p
    __host__ __device__ static constexpr int l_in(int p) { int l = 1; for (int i = 0; i < p; i++) l *= pass_rp(code(i)); return l; }
    // offset (in complex entries) of the table of sub-stage q of pass p
    __host__ __device__ static constexpr int tw_off(int p, int q) {
        int off = 0, l = 1;
        for (int i = 0; i < MAXP; i++) {
            int c = code(i);
            for (int k = 0; k < pass_nsub(c); k++) {
                if (i == p && k == q) return off;
                int r = pass_radix(c, k);
                off += (r - 1) * l;
                l *= r;
            }
        }
        return off;
    }
    __host__ __device__ static constexpr int tw_total() { return tw_off(MAXP, 0); }
    __host__ __device__ static constexpr bool valid() {
        int prod = 1;
        for (int p = 0; p < MAXP; p++) if (code(p)) { prod *= pass_rp(code(p)); if (E % pass_rp(code(p))) return false; }
        return prod == N && N % T == 0;
    }
};

// ----------------------------------------------------------------------------------------
// arithmetic types.  Three "real" types run through the same engine:
//   float   one f32 transform per thread group
//   double  one f64 transform per thread group
//   f32x2   TWO f32 transforms (adjacent batch rows) in the two lanes of Blackwell's packed-FP32
//           instructions (FADD2 / FMUL2 / FFMA2, sm_100+): one issue slot does the work of two.
//           The engine is issue-bound, not FP32-pipe-bound (ncu: fma pipe 30 %, issue 70 %), so
//           halving the instruction count per transform is what moves it toward the HBM roofline.
// ----------------------------------------------------------------------------------------
struct f32x2 { float2 v; };

__device__ __forceinline__ float radd(float a, float b) { return a + b; }
__device__ __forceinline__ float rsub(float a, float b) { return a - b; }
__device__ __forceinline__ float rmul(float a, float b) { return a * b; }
__device__ __forceinline__ float rfma(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ float rneg(float a) { return -a; }
__device__ __forceinline__ double radd(double a, double b) { return a + b; }
__device__ __forceinline__ double rsub(double a, double b) { return a - b; }
__device__ __forceinline__ double rmul(double a, double b) { return a * b; }
__device__ __forceinline__ double rfma(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ double rneg(double a) { return -a; }
__device__ __forceinline__ f32x2 radd(f32x2 a, f32x2 b) { return {__fadd2_rn(a.v, b.v)}; }
__device__ __forceinline__ f32x2 rsub(f32x2 a, f32x2 b) { return {__ffma2_rn(b.v, make_float2(-1.f, -1.f), a.v)}; }
__device__ __forceinline__ f32x2 rmul(f32x2 a, f32x2 b) { return {__fmul2_rn(a.v, b.v)}; }
__device__ __forceinline__ f32x2 rfma(f32x2 a, f32x2 b, f32x2 c) { return {__ffma2_rn(a.v, b.v, c.v)}; }
__device__ __forceinline__ f32x2 rneg(f32x2 a) { return {__fmul2_rn(a.v, make_float2(-1.f, -1.f))}; }

template <typename R> struct RT;
template <> struct RT<float> {
    using scalar = float; using twel = float2;
    static constexpr int LANES = 1;
    static __device__ __forceinline__ float splat(float s) { return s; }
};
template <> struct RT<double> {
    using scalar = double; using twel = double2;
    static constexpr int LANES = 1;
    static __device__ __forceinline__ double splat(double s) { return s; }
};
template <> struct RT<f32x2> {
    using scalar = float; using twel = float4;      // table entry (re, re, im, im)
    static constexpr int LANES = 2;
    static __device__ __forceinline__ f32x2 splat(float s) { return {make_float2(s, s)}; }
};

// complex value / twiddle of lane type R
template <typename R> struct alignas(2 * sizeof(R)) cx { R x, y; };
template <typename R> struct twd { R x, y, ny; };        // (re, im, -im)
template <typename R> __device__ __forceinline__ cx<R> mk(R a, R b) { cx<R> v; v.x = a; v.y = b; return v; }
template <typename R> __device__ __forceinline__ cx<R> cadd(cx<R> a, cx<R> b) { return mk<R>(radd(a.x, b.x), radd(a.y, b.y)); }
template <typename R> __device__ __forceinline__ cx<R> csub(cx<R> a, cx<R> b) { return mk<R>(rsub(a.x, b.x), rsub(a.y, b.y)); }
// (wr*vr - wi*vi, wr*vi + wi*vr): the reference's product (fft_split_native_f32.wat:826-837,
// fft_combined.wat:417-419) with the second term of each component fused (FMA)
template <typename R> __device__ __forceinline__ cx<R> cmul(twd<R> w, cx<R> v) {
    return mk<R>(rfma(w.ny, v.y, rmul(w.x, v.x)), rfma(w.y, v.x, rmul(w.x, v.y)));
}
__device__ __forceinline__ twd<float> ld_tw(const float2 *p) { float2 t = __ldg(p); return {t.x, t.y, -t.y}; }
__device__ __forceinline__ twd<double> ld_tw(const double2 *p) { double2 t = __ldg(p); return {t.x, t.y, -t.y}; }
__device__ __forceinline__ twd<f32x2> ld_tw(const float4 *p) {
    float4 t = __ldg(p);
    f32x2 re = {make_float2(t.x, t.y)}, im = {make_float2(t.z, t.w)};
    return {re, im, rneg(im)};
}

// Where a pass finds the twiddles that do not depend on the thread (pass 0: every group index is 0).
// Entries below LIMIT come from a copy of the table's head inside the kernel parameter block: the values
// reach the FFMA/FMUL instructions through the constant bank / uniform registers -- no LSU/MIO slot, no
// scoreboard wait.  The rest (and everything for packed lanes, whose FFMA2 takes register pairs) comes from the
// global stage table through the read-only data path (LDG.CONSTANT).  A radix-64 opening has 63 entries,
// twice what the 63 uniform registers hold: measured, any constant share there is a loss (limit 0).
template <typename R, int LIMIT> struct HTw {
    const typename RT<R>::twel *c;     // parameter-block copy (unused when LIMIT == 0)
    const typename RT<R>::twel *g;     // global table
    template <int I> __device__ __forceinline__ twd<R> at() const {
        if constexpr (I < LIMIT) { const typename RT<R>::twel t = c[I]; return {t.x, t.y, -t.y}; }
        else return ld_tw(g + I);
    }
};
template <typename R> using GTw = HTw<R, 0>;

// shared-memory slot of logical element p (units of one complex value).  One pad slot per PADQ
// elements keeps both the contiguous writes (tid + e*T) and the strided gathers of the later
// passes (Rp*s'*j + t' + k*s') conflict-free; verified by tools/bank_sim.py for every plan.
template <int PADQ> __host__ __device__ constexpr int pad_idx(int p) { return PADQ ? p + (p / PADQ) : p; }
template <int PADQ> __host__ __device__ constexpr int padded_size(int n) { return PADQ ? n + (n / PADQ) : n; }
// pad_idx(base + off) == pad_idx(base) + pad_off(off) whenever `base mod PADQ + off mod PADQ < PADQ`
// is guaranteed by construction (see exchange()); lets every smem access use an immediate offset.
template <int PADQ> __host__ __device__ constexpr int pad_off(int off) { return PADQ ? off + off / PADQ : off; }

// mixed-radix helpers over the sub-stages of one pass
// hi enumerates the already-transformed (more significant) digits before sub-stage q.
__host__ __device__ constexpr int hi_count(int code, int q) { int h = 1; for (int a = 0; a < q; a++) h *= pass_radix(code, a); return h; }
// c(hi): output-group offset contributed by those digits = sum m'_a * prod_{h<a} r_h
__host__ __device__ constexpr int hi_to_c(int code, int q, int hi) {
    int c = 0, w = hi_count(code, q);
    int mult = 1;
    for (int a = 0; a < q; a++) {
        int r = pass_radix(code, a);
        w /= r;
        int d = (hi / w) % r;
        c += d * mult;
        mult *= r;
    }
    return c;
}
// final register slot k -> output digit-reversed index k'
__host__ __device__ constexpr int slot_to_out(int code, int k) {
    int g = pass_nsub(code), w = pass_rp(code), mult = 1, out = 0;
    for (int a = 0; a < g; a++) {
        int r = pass_radix(code, a);
        w /= r;
        int d = (k / w) % r;
        out += d * mult;
        mult *= r;
    }
    return out;
}
// after pass P, register slot s = i + NB*k holds logical element  tid + out_elem(s)*T
template <class PL, int P> __host__ __device__ constexpr int out_elem(int slot) {
    constexpr int NB = PL::E / pass_rp(PL::code(P));
    return (slot % NB) + NB * slot_to_out(PL::code(P), slot / NB);
}

// inverse of out_elem: the register slot that holds logical element tid + e*T after pass P
template <class PL, int P> __host__ __device__ constexpr int slot_of_elem(int e) {
    for (int q = 0; q < PL::E; q++) if (out_elem<PL, P>(q) == e) return q;
    return -1;
}

// First half of a twiddled radix-4 butterfly: t0 = A + w2*C, t1 = A - w2*C, t2 = w1*B + w3*D,
// t3 = w1*B - w3*D  (fft_split_native_f32.wat:826-848).  Generic form: three products, four add/subs.
template <typename R>
__device__ __forceinline__ void twiddled_r4(const cx<R> &A, const cx<R> &B, const cx<R> &C, const cx<R> &D,
                                            const twd<R> &w1, const twd<R> &w2, const twd<R> &w3,
                                            cx<R> &t0, cx<R> &t1, cx<R> &t2, cx<R> &t3) {
    const cx<R> wb = cmul<R>(w1, B), wc = cmul<R>(w2, C), wd = cmul<R>(w3, D);
    t0 = cadd<R>(A, wc); t1 = csub<R>(A, wc);
    t2 = cadd<R>(wb, wd); t3 = csub<R>(wb, wd);
}
// Scalar lanes (f32 and f64): FMA-fused form, 16 instead of 20 instructions (negated operands are free
// SASS modifiers): t0 and t2 as FMA chains, then t1 = 2A - t0 and t3 = 2*(w1*B) - t2.  Same table
// entries on the same operands; only the rounding points move (f64 parity stays ~1 % of its bound).
#define WFB_FUSED_R4(T)                                                                                      \
    __device__ __forceinline__ void twiddled_r4(const cx<T> &A, const cx<T> &B, const cx<T> &C, const cx<T> &D, \
                                                const twd<T> &w1, const twd<T> &w2, const twd<T> &w3,         \
                                                cx<T> &t0, cx<T> &t1, cx<T> &t2, cx<T> &t3) {                 \
        const cx<T> wb = cmul<T>(w1, B);                                                                     \
        t0 = mk<T>(rfma(w2.ny, C.y, rfma(w2.x, C.x, A.x)), rfma(w2.y, C.x, rfma(w2.x, C.y, A.y)));           \
        t2 = mk<T>(rfma(w3.ny, D.y, rfma(w3.x, D.x, wb.x)), rfma(w3.y, D.x, rfma(w3.x, D.y, wb.y)));         \
        t1 = mk<T>(rfma(T(2), A.x, -t0.x), rfma(T(2), A.y, -t0.y));                                          \
        t3 = mk<T>(rfma(T(2), wb.x, -t2.x), rfma(T(2), wb.y, -t2.y));                                        \
    }
WFB_FUSED_R4(float)
WFB_FUSED_R4(double)
#undef WFB_FUSED_R4

// Large f32 cores (N >= 2048) are bound by the L1/shared-memory data pipe (ncu: 81-91 % busy, a quarter of it
// twiddle loads), so for the per-thread twiddles of a radix-4 stage only w1 is loaded and w2 = w1^2, w3 = w1*w2
// are formed in registers (8 FP instructions for two 8-byte loads).  The reference LOOKS UP all three
// (fft_split_native_f32.wat:225-252), each carrying the Taylor error of its own angle (5e-7); the derived ones
// carry 2-3x the error of w1 instead.  Measured against the oracle: 12-21 % of the parity bound instead of
// 2-8 %; c2c N = 4096 goes from 92 % to 102 % of the measured HBM peak.  f64 keeps the tables (its parity
// bound is 1e4 times tighter than the twiddle error), and so do all smaller f32 sizes.
#ifndef WFB_DERIVE_MIN_N
#define WFB_DERIVE_MIN_N 2048
#endif
template <typename R, class PL> __host__ __device__ constexpr bool derive_tw() {
    return sizeof(typename RT<R>::scalar) == 4 && RT<R>::LANES == 1 && PL::N >= WFB_DERIVE_MIN_N;
}

// ----------------------------------------------------------------------------------------
// one fused pass over the E register-resident values of a thread
// ----------------------------------------------------------------------------------------
// Last-pass twiddles held in registers across the tiles of a persistent kernel ("hoisting").  In the last pass every
// thread multiplies by table entries only it uses (group index = thread index): 15 complex values per 16-point block
// that are the same for every transform the thread ever processes.  Re-loading them per tile is a third of the L1 data
// pipe traffic of the f64 real kernels (ncu, profiles/r02_ncu_full.md: r2c f64 N = 2048 at 84 % L1 pipe, a quarter of the
// wavefronts twiddle LDG.128s); the f64 CTAs are small (64-256 threads, 1-4 per SM), so the registers are there.
//   hoist_count: entries per thread;  hoist_index: register of (block i, sub-stage q, digit prefix hi, input m >= 1)
template <typename R, class PL, int P> __host__ __device__ constexpr int hoist_per_block() {
    int n = 0;
    for (int q = 0; q < pass_nsub(PL::code(P)); q++) n += hi_count(PL::code(P), q) * (pass_radix(PL::code(P), q) - 1);
    return n;
}
template <typename R, class PL, int P> __host__ __device__ constexpr int hoist_count() {
    return hoist_per_block<R, PL, P>() * (PL::E / pass_rp(PL::code(P)));
}
template <typename R, class PL, int P> __host__ __device__ constexpr int hoist_index(int i, int q, int hi, int m) {
    int base = 0;
    for (int a = 0; a < q; a++) base += hi_count(PL::code(P), a) * (pass_radix(PL::code(P), a) - 1);
    return i * hoist_per_block<R, PL, P>() + base + hi * (pass_radix(PL::code(P), q) - 1) + (m - 1);
}
struct NoHoist { static constexpr bool ON = false; };
template <typename R> struct Hoisted {
    static constexpr bool ON = true;
    const typename RT<R>::twel *regs;
    template <int I> __device__ __forceinline__ twd<R> at() const { const typename RT<R>::twel t = regs[I]; return {t.x, t.y, -t.y}; }
};

template <typename R, class PL, int P, int I, int Q, int HI, int RADIX, class HS>
__device__ __forceinline__ void hoisted_get(const HS &hs, twd<R> &w1, twd<R> &w2, twd<R> &w3) {
    if constexpr (HS::ON) {
        w1 = hs.template at<hoist_index<R, PL, P>(I, Q, HI, 1)>();
        if constexpr (RADIX == 4) { w2 = hs.template at<hoist_index<R, PL, P>(I, Q, HI, 2)>(); w3 = hs.template at<hoist_index<R, PL, P>(I, Q, HI, 3)>(); }
    }
}

template <typename R, class PL, int P, bool INV, class U, class HS = NoHoist>
__device__ __forceinline__ void run_pass(cx<R> (&x)[PL::E], const typename RT<R>::twel *__restrict__ tw, const U &tw0, int tid, const HS &hs = HS()) {
    constexpr int CODE = PL::code(P);
    constexpr int RP = pass_rp(CODE);
    constexpr int NB = PL::E / RP;                 // register blocks per thread
    constexpr int L_IN = PL::l_in(P);
    constexpr int SP = PL::N / (L_IN * RP);        // stride on exit (s')
    constexpr int G = pass_nsub(CODE);
    // group index of block i: j = (tid + i*T) / SP
    constexpr bool SPLITJ = (PL::T % SP == 0);
    const int j0 = (L_IN == 1) ? 0 : tid / SP;
    static_for<NB>([&](auto I_) {
        CIDX(i, I_);
        const int j = (L_IN == 1) ? 0 : (SPLITJ ? j0 + i * (PL::T / SP) : (tid + i * PL::T) / SP);
        const typename RT<R>::twel *twj = tw + j;
        static_for<G>([&](auto Q_) {
            CIDX(q, Q_);
            constexpr int r = pass_radix(CODE, q);
            constexpr int H = hi_count(CODE, q);
            constexpr int w = RP / (H * r);            // slot stride of this digit
            constexpr int lq = L_IN * H;               // groups of this stage
            constexpr int off = PL::tw_off(P, q);
            static_for<H>([&](auto HI_) {
                CIDX(hi, HI_);
                constexpr int c = hi_to_c(CODE, q, hi);
                constexpr bool unit = (L_IN == 1 && c == 0);     // group 0: W^0 = 1
                twd<R> w1, w2, w3;
                if constexpr (!unit && L_IN == 1) {           // thread-independent: constant operands
                    w1 = tw0.template at<off + c>();
                    if constexpr (r == 4) { w2 = tw0.template at<off + lq + c>(); w3 = tw0.template at<off + 2 * lq + c>(); }
                } else if constexpr (!unit && HS::ON) {
                    static_assert(!HS::ON || !derive_tw<R, PL>(), "hoisting keeps table entries, not derived ones");
                    hoisted_get<R, PL, P, i, q, hi, r>(hs, w1, w2, w3);
                } else if constexpr (!unit) {
                    w1 = ld_tw(twj + (off + L_IN * c));
                    if constexpr (r == 4) {
                        if constexpr (derive_tw<R, PL>()) {
                            w2.x = rfma(w1.x, w1.x, rneg(rmul(w1.y, w1.y))); w2.y = rmul(radd(w1.x, w1.x), w1.y); w2.ny = rneg(w2.y);
                            w3.x = rfma(w1.x, w2.x, rneg(rmul(w1.y, w2.y))); w3.y = rfma(w1.x, w2.y, rmul(w1.y, w2.x)); w3.ny = rneg(w3.y);
                        } else {
                            w2 = ld_tw(twj + (off + lq + L_IN * c));
                            w3 = ld_tw(twj + (off + 2 * lq + L_IN * c));
                        }
                    }
                }
                static_for<w>([&](auto LO_) {
                    CIDX(lo, LO_);
                    constexpr int k0 = hi * (w * r) + lo;
                    if constexpr (r == 2) {
                        cx<R> &A = x[i + NB * k0], &B = x[i + NB * (k0 + w)];
                        cx<R> wb = B;
                        if constexpr (!unit) wb = cmul<R>(w1, B);
                        const cx<R> a = A;
                        A = cadd<R>(a, wb);
                        B = csub<R>(a, wb);
                    } else {
                        cx<R> &A = x[i + NB * k0], &B = x[i + NB * (k0 + w)];
                        cx<R> &C = x[i + NB * (k0 + 2 * w)], &D = x[i + NB * (k0 + 3 * w)];
                        cx<R> t0, t1, t2, t3;
                        if constexpr (unit) {
                            t0 = cadd<R>(A, C); t1 = csub<R>(A, C);
                            t2 = cadd<R>(B, D); t3 = csub<R>(B, D);
                        } else {
                            twiddled_r4(A, B, C, D, w1, w2, w3, t0, t1, t2, t3);
                        }
                        A = cadd<R>(t0, t2);
                        C = csub<R>(t0, t2);
                        // forward: out1 = t1 - i*t3, out3 = t1 + i*t3; the inverse swaps them
                        // (fft_split_native_f32.wat:785-788)
                        const cx<R> m1 = mk<R>(radd(t1.x, t3.y), rsub(t1.y, t3.x));
                        const cx<R> m3 = mk<R>(rsub(t1.x, t3.y), radd(t1.y, t3.x));
                        B = INV ? m3 : m1;
                        D = INV ? m1 : m3;
                    }
                });
            });
        });
    });
}

// fills the hoisted registers of pass P: the very table entries run_pass would load, in hoist_index order
template <typename R, class PL, int P>
__device__ __forceinline__ void hoist_load(typename RT<R>::twel (&hw)[hoist_count<R, PL, P>()], const typename RT<R>::twel *__restrict__ tw, int tid) {
    constexpr int CODE = PL::code(P);
    constexpr int RP = pass_rp(CODE);
    constexpr int NB = PL::E / RP;
    constexpr int L_IN = PL::l_in(P);
    constexpr int SP = PL::N / (L_IN * RP);
    static_assert(L_IN > 1, "pass 0 has no thread-dependent twiddles");
    static_for<NB>([&](auto I_) {
        CIDX(i, I_);
        const int j = (tid + i * PL::T) / SP;
        static_for<pass_nsub(CODE)>([&](auto Q_) {
            CIDX(q, Q_);
            constexpr int r = pass_radix(CODE, q);
            constexpr int H = hi_count(CODE, q);
            constexpr int lq = L_IN * H;
            constexpr int off = PL::tw_off(P, q);
            static_for<H>([&](auto HI_) {
                CIDX(hi, HI_);
                constexpr int c = hi_to_c(CODE, q, hi);
                static_for<r - 1>([&](auto M_) {
                    CIDX(m0, M_);
                    hw[hoist_index<R, PL, P>(i, q, hi, m0 + 1)] = __ldg(tw + j + (off + m0 * lq + L_IN * c));
                });
            });
        });
    });
}

// ----------------------------------------------------------------------------------------
// barriers scoped to the threads of one transform (pair)
// ----------------------------------------------------------------------------------------
template <int T, int X> __device__ __forceinline__ void sync_transform(int xi) {
    if constexpr (T <= 32) {
        __syncwarp();
    } else if constexpr (X == 1) {
        __syncthreads();
    } else {
        asm volatile("bar.sync %0, %1;" ::"r"(xi + 1), "n"(T) : "memory");
    }
}

// registers -> smem in the natural layout of pass P's outputs (element tid + e*T at pad(tid)+pad_off(e*T))
template <typename R, class PL, int P, int PADQ>
__device__ __forceinline__ void spill_outputs(const cx<R> (&x)[PL::E], cx<R> *sm, int tid) {
    static_assert(PL::T % PADQ == 0 || PADQ % PL::T == 0, "pad algebra needs T | PADQ or PADQ | T");
    cx<R> *base = sm + pad_idx<PADQ>(tid);
    static_for<PL::E>([&](auto S_) {
        CIDX(slot, S_);
        constexpr int e = out_elem<PL, P>(slot);
        base[pad_off<PADQ>(e * PL::T)] = x[slot];
    });
}

// smem -> registers in the gather layout of pass P's inputs
template <typename R, class PL, int P, int PADQ>
__device__ __forceinline__ void fill_inputs(cx<R> (&x)[PL::E], const cx<R> *sm, int tid) {
    constexpr int RP = pass_rp(PL::code(P));
    constexpr int NB = PL::E / RP;
    constexpr int SP = PL::N / (PL::l_in(P) * RP);
    constexpr bool FAST = (SP % PADQ == 0) || (PADQ % SP == 0 && (RP * SP) % PADQ == 0);
    static_for<NB>([&](auto I_) {
        CIDX(i, I_);
        const int b = tid + i * PL::T;
        const int j = b / SP, t = b % SP;
        const int base = RP * SP * j + t;
        if constexpr (FAST) {
            const cx<R> *bp = sm + pad_idx<PADQ>(base);
            static_for<RP>([&](auto K_) { CIDX(k, K_); x[i + NB * k] = bp[pad_off<PADQ>(k * SP)]; });
        } else {
            static_for<RP>([&](auto K_) { CIDX(k, K_); x[i + NB * k] = sm[pad_idx<PADQ>(base + k * SP)]; });
        }
    });
}

// all passes; on entry x holds pass 0's inputs (element tid + e*T in slot e), on exit the last
// pass's outputs.  `smem_dirty`: other threads may still be reading smem when we get here.
template <typename R, class PL, int PADQ, int X, bool INV, int P = 0, class U, class HS = NoHoist>
__device__ __forceinline__ void run_all(cx<R> (&x)[PL::E], const typename RT<R>::twel *__restrict__ tw, const U &tw0, cx<R> *sm,
                                        int tid, int xi, bool smem_dirty, const HS &hs = HS()) {
    if constexpr (HS::ON && P + 1 == PL::npass() && P > 0) run_pass<R, PL, P, INV>(x, tw, tw0, tid, hs);   // hoisted: the last pass
    else run_pass<R, PL, P, INV>(x, tw, tw0, tid);
    if constexpr (P + 1 < PL::npass()) {
        if (smem_dirty || P > 0) sync_transform<PL::T, X>(xi);
        spill_outputs<R, PL, P, PADQ>(x, sm, tid);
        sync_transform<PL::T, X>(xi);
        fill_inputs<R, PL, P + 1, PADQ>(x, sm, tid);
        run_all<R, PL, PADQ, X, INV, P + 1>(x, tw, tw0, sm, tid, xi, true, hs);
    }
}

// ----------------------------------------------------------------------------------------
// kernel parameters
// ----------------------------------------------------------------------------------------
struct KParams {
    const void *in0, *in1;     // input planes
    void *out0, *out1;         // output planes
    const void *tw;            // stage tables for this direction
    const void *rtw;           // W_Nreal^k, k = 0..M, for the real transforms
    long batch;
    double scale;              // applied on store (1/N for the inverse c2c)
    unsigned long long *ctr;   // persistent kernels: this launch's counter pair {tile claims, departed CTAs}, zero on entry AND on exit
    // zero-copy path (direct kernels on mapped host buffers): when done_flag is set, the last CTA to finish stores
    // done_token there -- a word of mapped HOST memory the caller polls -- behind a system-scope fence
    unsigned *done_flag, *done_ctr;
    unsigned done_token;
    // the first TW0_BYTES of the stage table `tw` (scalar-lane variants): pass 0's thread-independent twiddles,
    // read as constant-bank operands (see CTw)
    enum { TW0_BYTES = 1008 };                         // 63 entries of a radix-64 opening pass in f64
    alignas(16) unsigned char tw0[TW0_BYTES];
};
#ifndef WFB_CTW_LIMIT64
#define WFB_CTW_LIMIT64 0
#endif
// pass-0 twiddle source of a kernel with lane type R and plan PL
template <typename R, class PL> struct UTw {
    static constexpr int ENTRIES = PL::tw_off(1, 0);   // table entries of pass 0
    // thread-per-row plans (T == 1) have no other warp to hide a load behind: constants pay there even at 63 entries
    static constexpr int LIMIT = RT<R>::LANES != 1 ? 0 : ((ENTRIES <= 31 || PL::T == 1) ? ENTRIES : WFB_CTW_LIMIT64);
    static_assert(LIMIT * sizeof(typename RT<R>::twel) <= KParams::TW0_BYTES, "tw0 capacity");
    static __device__ __forceinline__ HTw<R, LIMIT> make(const KParams &p, const typename RT<R>::twel *tw) {
        return {reinterpret_cast<const typename RT<R>::twel *>(p.tw0), tw};
    }
};

enum IoMode { IO_SPLIT = 0, IO_INTERLEAVED = 1 };

// Completion signal of the zero-copy path.  Every thread fences its own stores to the mapped host buffers at system
// scope, the CTA meets at a barrier, and the last CTA of the grid (device-memory counter, left at zero again) publishes
// the token: a host thread that reads the token then reads the results (PCIe posted writes keep their order).
// All threads of the CTA must call this (no early return before it).
__device__ __forceinline__ void signal_done(const KParams &p) {
    if (p.done_flag == nullptr) return;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        bool last = true;
        if (gridDim.x > 1) {
            last = atomicAdd(p.done_ctr, 1u) == gridDim.x - 1;
            if (last) *p.done_ctr = 0u;
        }
        if (last) {
            __threadfence_system();
            *reinterpret_cast<volatile unsigned *>(p.done_flag) = p.done_token;
        }
    }
}

// streaming global accesses: every payload byte is touched exactly once
template <typename V> __device__ __forceinline__ V ld_stream(const V *p) { return __ldcs(p); }
template <typename V> __device__ __forceinline__ void st_stream(V *p, V v) { __stcs(p, v); }

// Global <-> register movement of one complex element for each lane type.  `rs` is the row stride
// in elements of the pointed-to type; lane 1 of f32x2 is the NEXT batch row (clamped onto lane 0's
// row when the batch is odd and this is the last group: loaded twice, stored once).
template <typename R> struct GIO;
template <> struct GIO<float> {
    static __device__ __forceinline__ cx<float> ld_split(const float *re, const float *im, long, bool) { return mk<float>(ld_stream(re), ld_stream(im)); }
    static __device__ __forceinline__ cx<float> ld_il(const float2 *z, long, bool) { float2 v = ld_stream(z); return mk<float>(v.x, v.y); }
    static __device__ __forceinline__ void st_split(float *re, float *im, long, bool, cx<float> v) { st_stream(re, v.x); st_stream(im, v.y); }
    static __device__ __forceinline__ void st_il(float2 *z, long, bool, cx<float> v) { st_stream(z, make_float2(v.x, v.y)); }
    static __device__ __forceinline__ float re0(cx<float> v) { return v.x; }
};
template <> struct GIO<double> {
    static __device__ __forceinline__ cx<double> ld_split(const double *re, const double *im, long, bool) { return mk<double>(ld_stream(re), ld_stream(im)); }
    static __device__ __forceinline__ cx<double> ld_il(const double2 *z, long, bool) { double2 v = ld_stream(z); return mk<double>(v.x, v.y); }
    static __device__ __forceinline__ void st_split(double *re, double *im, long, bool, cx<double> v) { st_stream(re, v.x); st_stream(im, v.y); }
    static __device__ __forceinline__ void st_il(double2 *z, long, bool, cx<double> v) { st_stream(z, make_double2(v.x, v.y)); }
};
template <> struct GIO<f32x2> {
    static __device__ __forceinline__ cx<f32x2> ld_split(const float *re, const float *im, long rs, bool) {
        f32x2 a = {make_float2(ld_stream(re), ld_stream(re + rs))};
        f32x2 b = {make_float2(ld_stream(im), ld_stream(im + rs))};
        return mk<f32x2>(a, b);
    }
    static __device__ __forceinline__ cx<f32x2> ld_il(const float2 *z, long rs, bool) {
        float2 a = ld_stream(z), b = ld_stream(z + rs);
        return mk<f32x2>({make_float2(a.x, b.x)}, {make_float2(a.y, b.y)});
    }
    static __device__ __forceinline__ void st_split(float *re, float *im, long rs, bool two, cx<f32x2> v) {
        st_stream(re, v.x.v.x); st_stream(im, v.y.v.x);
        if (two) { st_stream(re + rs, v.x.v.y); st_stream(im + rs, v.y.v.y); }
    }
    static __device__ __forceinline__ void st_il(float2 *z, long rs, bool two, cx<f32x2> v) {
        st_stream(z, make_float2(v.x.v.x, v.y.v.x));
        if (two) st_stream(z + rs, make_float2(v.x.v.y, v.y.v.y));
    }
};
template <typename R> struct VecOf;
template <> struct VecOf<float> { using s = float; using v2 = float2; };
template <> struct VecOf<double> { using s = double; using v2 = double2; };
template <> struct VecOf<f32x2> { using s = float; using v2 = float2; };

// per-thread-group row bookkeeping
template <typename R, int T, int X> struct Rows {
    int xi, tid;
    long row;          // first row of this group
    bool active, two;  // any row valid / second lane's row valid
    long lane1;        // element offset multiplier of lane 1's row (0 when clamped)
    __device__ __forceinline__ Rows(long batch) {
        xi = threadIdx.x / T; tid = threadIdx.x % T;
        row = ((long)blockIdx.x * X + xi) * RT<R>::LANES;
        active = row < batch;
        two = RT<R>::LANES == 2 && row + 1 < batch;
        lane1 = two ? 1 : 0;
    }
};

// ----------------------------------------------------------------------------------------
// Transform 1 and 3 (f32) / 4 (f64): batched c2c, split or interleaved I/O
// ----------------------------------------------------------------------------------------
template <typename R, class PL, int X, int PADQ, int IO, bool INV, int MINB>
__global__ void __launch_bounds__(PL::T *X, MINB) k_c2c(const __grid_constant__ KParams p) {
    static_assert(PL::valid(), "plan does not factor N");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using S = typename VecOf<R>::s;
    using V2 = typename VecOf<R>::v2;
    constexpr int LAST = PL::npass() - 1;
    const Rows<R, PL::T, X> g(p.batch);
    const int tid = g.tid;
    cx<R> *sm = reinterpret_cast<cx<R> *>(smem_raw) + (size_t)g.xi * padded_size<PADQ>(PL::N);
    const typename RT<R>::twel *tw = reinterpret_cast<const typename RT<R>::twel *>(p.tw);
    cx<R> x[PL::E];
    const long rs = g.lane1 * PL::N;

    if (g.active) {
        if constexpr (IO == IO_SPLIT) {
            const S *re = reinterpret_cast<const S *>(p.in0) + g.row * PL::N + tid;
            const S *im = reinterpret_cast<const S *>(p.in1) + g.row * PL::N + tid;
            static_for<PL::E>([&](auto E_) { CIDX(e, E_); x[e] = GIO<R>::ld_split(re + e * PL::T, im + e * PL::T, rs, g.two); });
        } else {
            const V2 *z = reinterpret_cast<const V2 *>(p.in0) + g.row * PL::N + tid;
            static_for<PL::E>([&](auto E_) { CIDX(e, E_); x[e] = GIO<R>::ld_il(z + e * PL::T, rs, g.two); });
        }
    } else {
        static_for<PL::E>([&](auto E_) { CIDX(e, E_); x[e] = mk<R>(RT<R>::splat(0), RT<R>::splat(0)); });
    }

    run_all<R, PL, PADQ, X, INV>(x, tw, UTw<R, PL>::make(p, tw), sm, tid, g.xi, false);

    if (g.active) {
        const R sc = RT<R>::splat((S)p.scale);
        if constexpr (IO == IO_SPLIT) {
            S *re = reinterpret_cast<S *>(p.out0) + g.row * PL::N + tid;
            S *im = reinterpret_cast<S *>(p.out1) + g.row * PL::N + tid;
            static_for<PL::E>([&](auto S_) {
                CIDX(slot, S_);
                constexpr int e = out_elem<PL, LAST>(slot);
                cx<R> v = x[slot];
                if (INV) v = mk<R>(rmul(v.x, sc), rmul(v.y, sc));
                GIO<R>::st_split(re + e * PL::T, im + e * PL::T, rs, g.two, v);
            });
        } else {
            V2 *z = reinterpret_cast<V2 *>(p.out0) + g.row * PL::N + tid;
            static_for<PL::E>([&](auto S_) {
                CIDX(slot, S_);
                constexpr int e = out_elem<PL, LAST>(slot);
                cx<R> v = x[slot];
                if (INV) v = mk<R>(rmul(v.x, sc), rmul(v.y, sc));
                GIO<R>::st_il(z + e * PL::T, rs, g.two, v);
            });
        }
    }
    signal_done(p);
}

// ----------------------------------------------------------------------------------------
// Transform 2 (f32) / 4-real (f64): batched r2c.  PL describes the M = N/2 point complex core.
// The even/odd deinterleave is the float2 view of the packed input (fused into the first-stage
// loads, cf. $stage_r4_first_fused :1376-1459); the Hermitian post-process runs out of shared
// memory straight into the coalesced spectrum store (cf. $rfft_postprocess_split :1471-1559,
// fft_real_combined.wat:455-592).
// ----------------------------------------------------------------------------------------
template <typename R> struct RealPost {
    // f32 flavour (float and f32x2): one twiddle W^k serves both X[k] and X[M-k]
    static __device__ __forceinline__ void pair(cx<R> z, cx<R> zm, twd<R> w, twd<R>, cx<R> &xk, cx<R> &xm) {
        const R half = RT<R>::splat(0.5f);
        const R gr = radd(z.x, zm.x), gi = rsub(z.y, zm.y), hr = radd(z.y, zm.y), hi = rsub(zm.x, z.x);
        const R tr = rfma(w.ny, hi, rmul(w.x, hr)), ti = rfma(w.y, hr, rmul(w.x, hi));
        xk = mk<R>(rmul(half, radd(gr, tr)), rmul(half, radd(gi, ti)));
        xm = mk<R>(rmul(half, rsub(gr, tr)), rmul(half, rsub(ti, gi)));
    }
    // X[M/2]: the reference's last vector iteration stores the mirrored form last (:1527-1545);
    // the M = 32 fused ending stores conj(Z[M/2]) (:2710)
    static __device__ __forceinline__ cx<R> middle(cx<R> z, twd<R> w, int m) {
        if (m == 32) return mk<R>(z.x, rneg(z.y));
        cx<R> a, b;
        pair(z, z, w, w, a, b);
        return b;
    }
};
// f64 flavour: T[k] and T[M-k] are separately tabulated (fft_real_combined.wat:502-503,533-534)
template <> struct RealPost<double> {
    using C = cx<double>;
    static __device__ __forceinline__ C one(C z, C zm, twd<double> w) {
        double sr = z.x + zm.x, si = z.y - zm.y, dr = z.x - zm.x, di = z.y + zm.y;
        double wdr = w.y * dr + w.x * di, wdi = w.y * di - w.x * dr;
        return mk<double>(0.5 * (sr + wdr), 0.5 * (si + wdi));
    }
    static __device__ __forceinline__ void pair(C z, C zm, twd<double> w, twd<double> wm, C &xk, C &xm) {
        xk = one(z, zm, w);
        xm = one(zm, z, wm);
    }
    static __device__ __forceinline__ C middle(C z, twd<double> w, int) {
        // sum = (2 re, 0), diff = (0, 2 im)  (fft_real_combined.wat:1031-1050)
        double sr = 2.0 * z.x, si = 0.0, dr = 0.0, di = 2.0 * z.y;
        double wdr = w.y * dr + w.x * di, wdi = w.y * di - w.x * dr;
        return mk<double>(0.5 * (sr + wdr), 0.5 * (si + wdi));
    }
};

// Second twiddle of a bin pair (k, M-k) in the f64 post-process.  The reference tabulates T[k] and T[M-k] separately
// (fft_real_combined.wat:502-503,533-534), but its range reduction folds the angle of T[M-k] onto the argument of T[k]
// (-PI - x for the sine, PI + x with sign -1 for the cosine, fft_combined.wat:43-106), so the two entries are mirror images:
// T[M-k] = (-T[k].re, T[k].im) to within ONE rounding of the folded argument -- measured over every table N = 8..16384:
// max |difference| = 3.3e-16 (tests/test_cabi.py::test_f64_rfft_table_mirror_symmetry), five orders below the
// 6.5e-11 Taylor error both carry and 1e-3 of the parity bound.  Forming it in registers removes one 16-byte load per
// bin pair: in the f64 r2c kernels those loads were as many bytes through the L1 data pipe as a whole pass over the data
// (the c2r direction, which needs only T[k], ran 5-13 % faster for that reason).  k = M/2 pairs with itself and keeps its
// own table entry (RealPost<double>::middle).  -DWFB_F64_MIRROR_TW=0 restores the second load.
#ifndef WFB_F64_MIRROR_TW
#define WFB_F64_MIRROR_TW 1
#endif
template <typename R>
__device__ __forceinline__ twd<R> ld_tw_mirror(const typename RT<R>::twel *rtw, int k, int m, const twd<R> &w) {
    if constexpr (sizeof(typename RT<R>::scalar) == 8 && WFB_F64_MIRROR_TW) return twd<R>{rneg(w.x), w.y, w.ny};
    else if constexpr (sizeof(typename RT<R>::scalar) == 8) return ld_tw(rtw + (m - k));
    else return w;                                     // f32: one twiddle serves both bins (RealPost<R>::pair)
}

template <typename R, class PL, int X, int PADQ, int MINB>
__global__ void __launch_bounds__(PL::T *X, MINB) k_r2c(const __grid_constant__ KParams p) {
    static_assert(PL::valid(), "plan does not factor N");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using V2 = typename VecOf<R>::v2;
    constexpr int M = PL::N;
    constexpr int LAST = PL::npass() - 1;
    const Rows<R, PL::T, X> g(p.batch);
    const int tid = g.tid;
    cx<R> *sm = reinterpret_cast<cx<R> *>(smem_raw) + (size_t)g.xi * padded_size<PADQ>(M);
    const typename RT<R>::twel *tw = reinterpret_cast<const typename RT<R>::twel *>(p.tw);
    const typename RT<R>::twel *rtw = reinterpret_cast<const typename RT<R>::twel *>(p.rtw);
    cx<R> x[PL::E];

    if (g.active) {
        const V2 *z = reinterpret_cast<const V2 *>(p.in0) + g.row * M + tid;   // z[j] = x[2j] + i x[2j+1]
        static_for<PL::E>([&](auto E_) { CIDX(e, E_); x[e] = GIO<R>::ld_il(z + e * PL::T, g.lane1 * M, g.two); });
    } else {
        static_for<PL::E>([&](auto E_) { CIDX(e, E_); x[e] = mk<R>(RT<R>::splat(0), RT<R>::splat(0)); });
    }

    run_all<R, PL, PADQ, X, false>(x, tw, UTw<R, PL>::make(p, tw), sm, tid, g.xi, false);

    // Z -> shared memory in natural order
    if (PL::npass() > 1) sync_transform<PL::T, X>(g.xi);
    spill_outputs<R, PL, LAST, PADQ>(x, sm, tid);
    sync_transform<PL::T, X>(g.xi);
    if (g.active) {
    V2 *out = reinterpret_cast<V2 *>(p.out0) + g.row * (M + 1);
    const long rs = g.lane1 * (M + 1);
    // pairs (k, M-k), k = tid + i*T over 0 .. M/2-1; k = 0 is DC/Nyquist; thread 0 adds k = M/2
    constexpr int HALF = M / 2;
    constexpr int PER = (HALF + PL::T - 1) / PL::T;
    const R zero = RT<R>::splat(0);
    static_for<PER>([&](auto I_) {
        CIDX(i, I_);
        const int k = tid + i * PL::T;
        if (k < HALF) {
            if (i == 0 && k == 0) {
                const cx<R> z0 = sm[0];
                GIO<R>::st_il(out, rs, g.two, mk<R>(radd(z0.x, z0.y), zero));
                GIO<R>::st_il(out + M, rs, g.two, mk<R>(rsub(z0.x, z0.y), zero));
                const cx<R> zh = sm[pad_idx<PADQ>(HALF)];
                GIO<R>::st_il(out + HALF, rs, g.two, RealPost<R>::middle(zh, ld_tw(rtw + HALF), M));
            } else {
                const cx<R> z = sm[pad_idx<PADQ>(k)], zm = sm[pad_idx<PADQ>(M - k)];
                cx<R> xk, xm;
                const twd<R> wk = ld_tw(rtw + k);
                RealPost<R>::pair(z, zm, wk, ld_tw_mirror<R>(rtw, k, M, wk), xk, xm);
                GIO<R>::st_il(out + k, rs, g.two, xk);
                GIO<R>::st_il(out + (M - k), rs, g.two, xm);
            }
        }
    });
    }
    signal_done(p);
}

// ----------------------------------------------------------------------------------------
// c2r: Hermitian pre-process (scale 0.5/M folded in, $irfft_preprocess_split :1656-1748) fused
// into the loads, inverse M-point core, re-interleave on store ($stage_r4_s1_inv_fused :1756-1932).
// The f64 variant has no reference counterpart (extension, parity unpinned) and uses the same
// formulas in double.
// ----------------------------------------------------------------------------------------
template <typename R, class PL, int X, int PADQ, int MINB>
__global__ void __launch_bounds__(PL::T *X, MINB) k_c2r(const __grid_constant__ KParams p) {
    static_assert(PL::valid(), "plan does not factor N");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using S = typename VecOf<R>::s;
    using V2 = typename VecOf<R>::v2;
    constexpr int M = PL::N;
    constexpr int LAST = PL::npass() - 1;
    const Rows<R, PL::T, X> g(p.batch);
    const int tid = g.tid;
    cx<R> *sm = reinterpret_cast<cx<R> *>(smem_raw) + (size_t)g.xi * padded_size<PADQ>(M);
    const typename RT<R>::twel *tw = reinterpret_cast<const typename RT<R>::twel *>(p.tw);
    const typename RT<R>::twel *rtw = reinterpret_cast<const typename RT<R>::twel *>(p.rtw);
    cx<R> x[PL::E];

    constexpr int HALF = M / 2;
    constexpr int PER = (HALF + PL::T - 1) / PL::T;
    const R sc = RT<R>::splat(S(0.5) / S(M));
    if (g.active) {
        const V2 *in = reinterpret_cast<const V2 *>(p.in0) + g.row * (M + 1);
        const long rs = g.lane1 * (M + 1);
        static_for<PER>([&](auto I_) {
            CIDX(i, I_);
            const int k = tid + i * PL::T;
            if (k < HALF) {
                if (i == 0 && k == 0) {
                    // real parts only (:1679-1684)
                    const cx<R> a0 = GIO<R>::ld_il(in, rs, g.two), am = GIO<R>::ld_il(in + M, rs, g.two);
                    sm[0] = mk<R>(rmul(radd(a0.x, am.x), sc), rmul(rsub(a0.x, am.x), sc));
                }
                const int kk = (k == 0) ? HALF : k;     // thread 0's slot k = 0 also covers the self-paired k = M/2
                const cx<R> a = GIO<R>::ld_il(in + kk, rs, g.two), b = GIO<R>::ld_il(in + (M - kk), rs, g.two);
                const twd<R> w = ld_tw(rtw + kk);
                const R gr = radd(a.x, b.x), gi = rsub(a.y, b.y), ur = rsub(a.x, b.x), ui = radd(a.y, b.y);
                // hr = wr*ur + wi*ui, hi = wr*ui - wi*ur   (conj(W) * u)
                const R hr = rfma(w.y, ui, rmul(w.x, ur)), hi = rfma(w.ny, ur, rmul(w.x, ui));
                // forward store first, mirrored second: at k = M/2 the mirrored form survives (:1722-1740)
                sm[pad_idx<PADQ>(kk)] = mk<R>(rmul(sc, rsub(gr, hi)), rmul(sc, radd(gi, hr)));
                sm[pad_idx<PADQ>(M - kk)] = mk<R>(rmul(sc, radd(gr, hi)), rmul(sc, rsub(hr, gi)));
            }
        });
    }
    sync_transform<PL::T, X>(g.xi);
    {
        const cx<R> *base = sm + pad_idx<PADQ>(tid);
        static_for<PL::E>([&](auto E_) { CIDX(e, E_); x[e] = base[pad_off<PADQ>(e * PL::T)]; });
    }

    run_all<R, PL, PADQ, X, true>(x, tw, UTw<R, PL>::make(p, tw), sm, tid, g.xi, true);

    if (g.active) {
        V2 *z = reinterpret_cast<V2 *>(p.out0) + g.row * M + tid;
        static_for<PL::E>([&](auto S_) {
            CIDX(slot, S_);
            constexpr int e = out_elem<PL, LAST>(slot);
            GIO<R>::st_il(z + e * PL::T, g.lane1 * M, g.two, x[slot]);
        });
    }
    signal_done(p);
}


// ----------------------------------------------------------------------------------------
// Small-N c2c (N <= 64): one thread per transform, whole transform in registers (single pass, no
// exchange), X rows per CTA staged through shared memory so that EVERY global access is a
// coalesced 128-bit load/store of a dense [X][N] tile (a thread-per-row kernel reading global
// memory directly touches 32 different 64-byte segments per instruction: ncu showed 25 % of the
// HBM roofline at N = 16).  Row stride in smem is N + 2 complex values (N*8 + 16 bytes): the
// per-row LDS.128/STS.128 of 8 consecutive threads then fall in 8 distinct 16-byte bank groups.
// ----------------------------------------------------------------------------------------
template <typename R, class PL, int X, int IO, bool INV, int MINB>
__global__ void __launch_bounds__(X, MINB) k_c2c_tile(const __grid_constant__ KParams p) {
    static_assert(PL::valid() && PL::T == 1 && PL::npass() == 1 && RT<R>::LANES == 1, "tile kernel: one thread per row");
    static_assert(sizeof(R) == 4, "tile kernel is f32");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int N = PL::N;
    constexpr int RS = N + 2;                           // row stride, complex values
    float *smf = reinterpret_cast<float *>(smem_raw);
    const int t = threadIdx.x;
    const long row0 = (long)blockIdx.x * X;
    const int rows = (p.batch - row0 < X) ? (int)(p.batch - row0) : X;
    const typename RT<R>::twel *tw = reinterpret_cast<const typename RT<R>::twel *>(p.tw);

    // ---- stage in: dense tile -> padded interleaved rows
    if constexpr (IO == IO_SPLIT) {
        constexpr int CPR = N / 4;                      // float4 chunks per row per plane
        const float4 *re = reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(p.in0) + row0 * N);
        const float4 *im = reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(p.in1) + row0 * N);
#pragma unroll
        for (int f = t; f < X * CPR; f += X) {
            const int r = f / CPR, c = f % CPR;
            if (r < rows) {
                const float4 a = ld_stream(re + f), b = ld_stream(im + f);
                float4 *dst = reinterpret_cast<float4 *>(smf + r * 2 * RS + 8 * c);
                dst[0] = make_float4(a.x, b.x, a.y, b.y);
                dst[1] = make_float4(a.z, b.z, a.w, b.w);
            }
        }
    } else {
        constexpr int CPR = N / 2;                      // 16-byte chunks (2 complex) per row
        const float4 *z = reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(p.in0) + row0 * 2 * N);
#pragma unroll
        for (int f = t; f < X * CPR; f += X) {
            const int r = f / CPR, c = f % CPR;
            if (r < rows) *reinterpret_cast<float4 *>(smf + r * 2 * RS + 4 * c) = ld_stream(z + f);
        }
    }
    __syncthreads();

    // ---- each thread: its own row -> registers -> transform -> back to its row
    cx<R> x[N];
    float4 *rowp = reinterpret_cast<float4 *>(smf + t * 2 * RS);
    static_for<N / 2>([&](auto H_) {
        CIDX(h, H_);
        const float4 v = rowp[h];
        x[2 * h] = mk<R>(v.x, v.y);
        x[2 * h + 1] = mk<R>(v.z, v.w);
    });
    run_pass<R, PL, 0, INV>(x, tw, UTw<R, PL>::make(p, tw), 0);
    {
        const float sc = (float)p.scale;
        // register slot s holds element out_elem(s); emit adjacent element pairs as one STS.128
        static_for<N>([&](auto S_) {
            CIDX(sa, S_);
            constexpr int ea = out_elem<PL, 0>(sa);
            if constexpr (ea % 2 == 0) {
                // find the slot holding element ea + 1
                constexpr int sb = []() { for (int q = 0; q < N; q++) if (out_elem<PL, 0>(q) == ea + 1) return q; return -1; }();
                float4 v = make_float4(x[sa].x, x[sa].y, x[sb].x, x[sb].y);
                if (INV) v = make_float4(v.x * sc, v.y * sc, v.z * sc, v.w * sc);
                rowp[ea / 2] = v;
            }
        });
    }
    __syncthreads();

    // ---- stage out
    if constexpr (IO == IO_SPLIT) {
        constexpr int CPR = N / 4;
        float4 *re = reinterpret_cast<float4 *>(reinterpret_cast<float *>(p.out0) + row0 * N);
        float4 *im = reinterpret_cast<float4 *>(reinterpret_cast<float *>(p.out1) + row0 * N);
#pragma unroll
        for (int f = t; f < X * CPR; f += X) {
            const int r = f / CPR, c = f % CPR;
            if (r < rows) {
                const float4 *src = reinterpret_cast<const float4 *>(smf + r * 2 * RS + 8 * c);
                const float4 u = src[0], v = src[1];
                st_stream(re + f, make_float4(u.x, u.z, v.x, v.z));
                st_stream(im + f, make_float4(u.y, u.w, v.y, v.w));
            }
        }
    } else {
        constexpr int CPR = N / 2;
        float4 *z = reinterpret_cast<float4 *>(reinterpret_cast<float *>(p.out0) + row0 * 2 * N);
#pragma unroll
        for (int f = t; f < X * CPR; f += X) {
            const int r = f / CPR, c = f % CPR;
            if (r < rows) st_stream(z + f, *reinterpret_cast<const float4 *>(smf + r * 2 * RS + 4 * c));
        }
    }
}


// ----------------------------------------------------------------------------------------
// TMA-pipelined persistent c2c (large N).  Each CTA owns T threads and loops over its transforms;
// an elected thread streams the NEXT transform's rows into shared memory with cp.async.bulk (the
// TMA engine; SASS UBLKCP) while the CTA computes the current one, completion signalled on an
// mbarrier.  The global->smem traffic therefore never occupies registers or LSU issue slots and
// there is always one transform per resident CTA in flight -- the one-CTA-one-transform kernel
// above alternates load and compute phases and left ~30 % of the HBM roofline idle at N = 4096.
// The two stage buffers double as the exchange scratch of the transform being computed.
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// smem -> global bulk copy (TMA store), tracked by the issuing thread's bulk groups
__device__ __forceinline__ void tma_store_1d(void *dst_gmem, const void *src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all of this thread's committed bulk stores have finished READING their shared-memory source
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// Dynamic tile scheduling for the persistent kernels.  Tiles are claimed from a global counter, so they are
// handed out in monotonic order and the CTAs of the whole GPU work on one tight, advancing window of the
// arrays -- like the hardware CTA scheduler does for a one-tile-per-CTA launch.  A static `tile += gridDim.x`
// schedule lets CTAs drift apart; tools/microbench/copy_pipe.cu measures 6.05 TB/s (static) vs 6.85 TB/s
// (dynamic) for the same TMA-pipelined copy.  Called by warp 0; the claim for the NEXT tile is made when
// its prefetch is issued, one iteration ahead, and published to the CTA through `slot[stage]`.
// EARLY: the claim itself is software-pipelined -- the atomic whose result is consumed here was fired one claim
// earlier (`pending`, thread 0), so the issuing warp never waits for the round trip to L2.  In the one-warp CTAs
// of the thread-per-row kernels that wait stalls the whole CTA once per tile (power-capped: +3..5 % at N = 32..128).
// For the large transforms it is a loss (r2c N = 4096: -4.6 %): a claim made a whole tile early widens the window
// of rows the GPU works on at any moment, the very thing the dynamic schedule is there to keep tight.
template <bool EARLY> __device__ __forceinline__ long claim_prime(unsigned long long *ctr) {
    return (EARLY && threadIdx.x == 0) ? (long)atomicAdd(ctr, 1ULL) : 0L;
}
template <bool EARLY, class IssueFn>
__device__ __forceinline__ void claim_and_issue(unsigned long long *ctr, long &pending, long tiles, long *slot, int st, IssueFn &&issue) {
    if (threadIdx.x < 32) {
        long tn = 0;
        if constexpr (EARLY) {
            tn = pending;
            if (threadIdx.x == 0) { pending = (long)atomicAdd(ctr, 1ULL); slot[st] = tn; }
        } else {
            if (threadIdx.x == 0) { tn = (long)atomicAdd(ctr, 1ULL); slot[st] = tn; }
        }
        tn = __shfl_sync(0xffffffffu, tn, 0);
        if (tn < tiles) issue(tn, st);
    }
}

// Epilogue of every persistent kernel: the last CTA to leave puts the launch's counter pair {claims, departures} back to
// zero, so the host never has to clear a slot between launches (a cudaMemsetAsync in front of every kernel cost one more
// stream-order dependency per launch).  Each CTA's claims have returned before it reports its departure; the fences order
// them against the reset by the CTA that sees gridDim.x - 1 earlier departures.
__device__ __forceinline__ void claim_epilogue(unsigned long long *ctr) {
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned long long gone = atomicAdd(ctr + 1, 1ULL);
        if (gone == gridDim.x - 1) {
            __threadfence();
            ctr[0] = 0ULL;
            ctr[1] = 0ULL;
        }
    }
}

template <typename R, class PL, int PADQ, int X> __host__ __device__ constexpr size_t pipe_buf_bytes() {
    size_t a = sizeof(cx<R>) * (size_t)padded_size<PADQ>(PL::N) * X;
    return (a + 127) / 128 * 128;
}

// TS ("TMA stores"): the results go back into the tile's stage buffer (same layout as the input) and leave as bulk
// stores issued after the next loop-top barrier, instead of per-thread STG; the stage is refilled once those
// stores have drained (cp.async.bulk.wait_group.read), which the issuing lanes check after the row loads of the
// following tile.
template <typename R, class PL, int X, int PADQ, int IO, bool INV, int MINB, int RC = 0, bool TS = false, bool HT = false>
__global__ void __launch_bounds__(PL::T *X, MINB) k_c2c_pipe(const __grid_constant__ KParams p) {
    static_assert(PL::valid(), "plan does not factor N");
    static_assert(!TS || RT<R>::LANES == 1, "TMA stores: scalar lanes");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using S = typename VecOf<R>::s;
    using V2 = typename VecOf<R>::v2;
    constexpr int LANES = RT<R>::LANES;
    constexpr int N = PL::N;
    constexpr int LAST = PL::npass() - 1;
    constexpr int ROWS = X * LANES;                 // rows per CTA iteration
    // RC > 0 ("row copies"): the tile arrives as groups of RC consecutive rows, one bulk copy per group and plane, with
    // N/16 elements of padding behind every group, and the 32/T thread groups of a warp work on rows of 32/T DIFFERENT
    // groups: the rows a warp reads side by side then start T banks apart (a dense tile puts every row on bank 0: ncu
    // showed 4-way conflicts and mio_throttle as the top stall at N = 128).  RC = 1 is one copy per row; larger groups
    // mean fewer copies -- each one costs the issuing warp ~9 instructions of elect / R2UR / branch per lane, while the
    // CTA's other warps wait at the barrier (ncu r02, N = 128 with RC = 1: barrier 39 % of the stall samples, a fifth
    // of the instructions in those loops).
    constexpr int RG = RC > 0 ? RC : 1;             // rows per copy group
    constexpr int NGR = ROWS / RG;                  // groups per tile
    constexpr int GSTR = RG * N + (PL::T < 32 ? PL::T : N / 16);   // smem group stride, elements (RC only): groups T banks apart
    constexpr int PSTR = RC ? NGR * GSTR : ROWS * N;   // plane stride (split layout), elements
    static_assert(!RC || (ROWS % RG == 0 && NGR >= 32 / PL::T && LANES == 1), "a warp's thread groups must land in distinct copy groups");
    static_assert(!RC || (size_t)(IO == IO_SPLIT ? 2 : 1) * NGR * GSTR * (IO == IO_SPLIT ? 1 : 2) * sizeof(typename VecOf<R>::s) <= pipe_buf_bytes<R, PL, PADQ, X>(),
                  "the padded groups must fit the stage buffer (sized for the scratch)");
    static_assert(!RC || (N >= 64 && PL::T * X >= 32), "row copies need 16-byte aligned padded groups and a full issuing warp");
    constexpr size_t BUF = pipe_buf_bytes<R, PL, PADQ, X>();
    uint64_t *mbar = reinterpret_cast<uint64_t *>(smem_raw + 2 * BUF);
    const int xi = threadIdx.x / PL::T, tid = threadIdx.x % PL::T;
    // row of the tile this thread group works on, and where that row sits in the stage buffer (elements)
    const int xr = RC ? (xi % NGR) * RG + xi / NGR : xi;
    const int roff = RC ? (xr / RG) * GSTR + (xr % RG) * N : xi * LANES * N;
    const typename RT<R>::twel *tw = reinterpret_cast<const typename RT<R>::twel *>(p.tw);
    const long tiles = (p.batch + ROWS - 1) / ROWS;

    if (threadIdx.x == 0) {
        mbar_init(mbar + 0, 1);
        mbar_init(mbar + 1, 1);
        fence_proxy_async();
    }
    __syncthreads();

    // stream a tile's rows into stage st: thread 0 (dense tile: one copy per plane) or warp 0
    // (row copies: one copy per group and plane, spread over the lanes)
    auto issue = [&](long tile, int st) {
        const long row = tile * ROWS;
        const int rows = (p.batch - row < ROWS) ? (int)(p.batch - row) : ROWS;
        unsigned char *dst = smem_raw + st * BUF;
        constexpr int PLANES = (IO == IO_SPLIT) ? 2 : 1;
        constexpr uint32_t ROWB = (uint32_t)((IO == IO_SPLIT ? 1 : 2) * N * sizeof(S));     // bytes per row per plane
        constexpr uint32_t ESB = (uint32_t)((IO == IO_SPLIT ? 1 : 2) * sizeof(S));         // bytes per element per plane
        if constexpr (TS) { bulk_wait_read_all(); __syncwarp(); }   // the stores out of this stage have drained
        if constexpr (!RC) {
            if (threadIdx.x == 0) {
                mbar_expect_tx(mbar + st, PLANES * rows * ROWB);
                tma_load_1d(dst, reinterpret_cast<const unsigned char *>(p.in0) + row * ROWB, rows * ROWB, mbar + st);
                if constexpr (PLANES == 2)
                    tma_load_1d(dst + PSTR * ESB, reinterpret_cast<const unsigned char *>(p.in1) + row * ROWB, rows * ROWB, mbar + st);
            }
        } else {
            if (threadIdx.x < 32) {
                if (threadIdx.x == 0) mbar_expect_tx(mbar + st, PLANES * rows * ROWB);
                __syncwarp();
                const int groups = (rows + RG - 1) / RG;
                for (int c = threadIdx.x; c < PLANES * groups; c += 32) {
                    const int pl = c / groups, g = c - pl * groups;
                    const int nr = rows - g * RG < RG ? rows - g * RG : RG;
                    const unsigned char *src = reinterpret_cast<const unsigned char *>(pl ? p.in1 : p.in0) + (row + (long)g * RG) * ROWB;
                    tma_load_1d(dst + (size_t)(pl * PSTR + g * GSTR) * ESB, src, nr * ROWB, mbar + st);
                }
            }
        }
    };

    // TS: bulk-store the finished tile sitting in stage st (warp 0; same copy granularity as the loads)
    auto store_tile = [&](long tile, int st) {
        const long row = tile * ROWS;
        const int rows = (p.batch - row < ROWS) ? (int)(p.batch - row) : ROWS;
        const unsigned char *src = smem_raw + st * BUF;
        constexpr int PLANES = (IO == IO_SPLIT) ? 2 : 1;
        constexpr uint32_t ROWB = (uint32_t)((IO == IO_SPLIT ? 1 : 2) * N * sizeof(S));
        constexpr uint32_t ESB = (uint32_t)((IO == IO_SPLIT ? 1 : 2) * sizeof(S));
        if (threadIdx.x < 32) {
            if constexpr (!RC) {
                if (threadIdx.x == 0) {
                    tma_store_1d(reinterpret_cast<unsigned char *>(p.out0) + row * ROWB, src, rows * ROWB);
                    if constexpr (PLANES == 2)
                        tma_store_1d(reinterpret_cast<unsigned char *>(p.out1) + row * ROWB, src + PSTR * ESB, rows * ROWB);
                }
            } else {
                const int groups = (rows + RG - 1) / RG;
                for (int c = threadIdx.x; c < PLANES * groups; c += 32) {
                    const int pl = c / groups, g = c - pl * groups;
                    const int nr = rows - g * RG < RG ? rows - g * RG : RG;
                    unsigned char *dst = reinterpret_cast<unsigned char *>(pl ? p.out1 : p.out0) + (row + (long)g * RG) * ROWB;
                    tma_store_1d(dst, src + (size_t)(pl * PSTR + g * GSTR) * ESB, nr * ROWB);
                }
            }
            bulk_commit();
        }
    };

    static_assert(PL::T * X >= 32, "tile claims are made by a full warp");
    long *slot = reinterpret_cast<long *>(smem_raw + 2 * BUF + 32);   // tile claimed for each stage
    long pending = claim_prime<(PL::N <= 256)>(p.ctr);
    claim_and_issue<(PL::N <= 256)>(p.ctr, pending, tiles, slot, 0, issue);
    cx<R> x[PL::E];
    // HT: the last pass's thread-invariant twiddles live in registers for the whole kernel (see hoist_load).  For the f32
    // kernels this measured neutral at N = 4096 and 3-6 % slower below (profiles/r01_sweep.md); the f64 kernels are bound by
    // the L1 data pipe these loads go through, and their small CTAs have the registers to spare.
    typename RT<R>::twel hw[HT ? hoist_count<R, PL, (LAST > 0 ? LAST : 1)>() : 1];
    if constexpr (HT) { static_assert(LAST > 0, "hoisting needs a multi-pass plan"); hoist_load<R, PL, LAST>(hw, tw, tid); }
    const auto hsrc = [&]() { if constexpr (HT) return Hoisted<R>{hw}; else return NoHoist{}; }();
    for (int it = 0;; it++) {
        const int st = it & 1;
        fence_proxy_async();      // our generic-proxy accesses to the other stage precede its refill
        __syncthreads();          // ... and everyone is done using it as scratch
        if constexpr (TS) { if (it > 0) store_tile(slot[st ^ 1], st ^ 1); }   // last iteration's results (all written: barrier above)
        const long tile = slot[st];
        if (tile >= tiles) break;
        if constexpr (!TS) claim_and_issue<(PL::N <= 256)>(p.ctr, pending, tiles, slot, st ^ 1, issue);
        mbar_wait(mbar + st, (it >> 1) & 1);

        const long row = tile * ROWS + (long)xr * LANES;
        const bool active = row < p.batch;
        const bool two = LANES == 2 && row + 1 < p.batch;
        unsigned char *buf = smem_raw + st * BUF;
        if constexpr (IO == IO_SPLIT) {
            constexpr int RSTR = N;                 // next row of a lane pair (packed lanes: dense tiles only)
            const S *re = reinterpret_cast<const S *>(buf) + roff + tid;
            const S *im = re + PSTR;
            static_for<PL::E>([&](auto E_) {
                CIDX(e, E_);
                if constexpr (LANES == 2) {
                    x[e].x.v = make_float2(re[e * PL::T], re[RSTR + e * PL::T]);
                    x[e].y.v = make_float2(im[e * PL::T], im[RSTR + e * PL::T]);
                } else {
                    x[e] = mk<R>(re[e * PL::T], im[e * PL::T]);
                }
            });
        } else {
            constexpr int RSTR = N;
            const V2 *z = reinterpret_cast<const V2 *>(buf) + roff + tid;
            static_for<PL::E>([&](auto E_) {
                CIDX(e, E_);
                if constexpr (LANES == 2) {
                    const V2 a = z[e * PL::T], b = z[RSTR + e * PL::T];
                    x[e].x.v = make_float2(a.x, b.x);
                    x[e].y.v = make_float2(a.y, b.y);
                } else {
                    const V2 a = z[e * PL::T];
                    x[e] = mk<R>(a.x, a.y);
                }
            });
        }
        // the dense input tile and the padded per-group scratch regions alias: every group must
        // have its inputs in registers before any group spills
        if constexpr (PL::npass() > 1 || TS) __syncthreads();
        // TS: slot[st ^ 1] still names the tile just stored; the claim overwrites it only now, after the barrier
        if constexpr (TS) claim_and_issue<(PL::N <= 256)>(p.ctr, pending, tiles, slot, st ^ 1, issue);
        cx<R> *scratch = reinterpret_cast<cx<R> *>(buf) + (size_t)xi * padded_size<PADQ>(N);
        run_all<R, PL, PADQ, X, INV>(x, tw, UTw<R, PL>::make(p, tw), scratch, tid, xi, false, hsrc);

        if constexpr (TS) {
            // results -> the tile's rows in the stage buffer (they alias every group's scratch)
            if constexpr (PL::npass() > 1) __syncthreads();
            const R sc = RT<R>::splat((S)p.scale);
            if constexpr (IO == IO_SPLIT) {
                S *re = reinterpret_cast<S *>(buf) + roff + tid;
                S *im = re + PSTR;
                static_for<PL::E>([&](auto S_) {
                    CIDX(slot_, S_);
                    constexpr int e = out_elem<PL, LAST>(slot_);
                    cx<R> v = x[slot_];
                    if (INV) v = mk<R>(rmul(v.x, sc), rmul(v.y, sc));
                    re[e * PL::T] = v.x; im[e * PL::T] = v.y;
                });
            } else {
                V2 *z = reinterpret_cast<V2 *>(buf) + roff + tid;
                static_for<PL::E>([&](auto S_) {
                    CIDX(slot_, S_);
                    constexpr int e = out_elem<PL, LAST>(slot_);
                    cx<R> v = x[slot_];
                    if (INV) v = mk<R>(rmul(v.x, sc), rmul(v.y, sc));
                    V2 o; o.x = v.x; o.y = v.y;
                    z[e * PL::T] = o;
                });
            }
        } else if (active) {
            const long rs = two ? N : 0;
            const R sc = RT<R>::splat((S)p.scale);
            if constexpr (IO == IO_SPLIT) {
                S *re = reinterpret_cast<S *>(p.out0) + row * N + tid;
                S *im = reinterpret_cast<S *>(p.out1) + row * N + tid;
                static_for<PL::E>([&](auto S_) {
                    CIDX(slot, S_);
                    constexpr int e = out_elem<PL, LAST>(slot);
                    cx<R> v = x[slot];
                    if (INV) v = mk<R>(rmul(v.x, sc), rmul(v.y, sc));
                    GIO<R>::st_split(re + e * PL::T, im + e * PL::T, rs, two, v);
                });
            } else {
                V2 *z = reinterpret_cast<V2 *>(p.out0) + row * N + tid;
                static_for<PL::E>([&](auto S_) {
                    CIDX(slot, S_);
                    constexpr int e = out_elem<PL, LAST>(slot);
                    cx<R> v = x[slot];
                    if (INV) v = mk<R>(rmul(v.x, sc), rmul(v.y, sc));
                    GIO<R>::st_il(z + e * PL::T, rs, two, v);
                });
            }
        }
    }
    if constexpr (TS) { if (threadIdx.x < 32) bulk_wait_read_all(); }   // shared memory must outlive the stores that read it
    claim_epilogue(p.ctr);
}


// ----------------------------------------------------------------------------------------
// Register-prefetch persistent c2c (large N, scalar lanes, one transform per CTA iteration).
// ncu on the TMA-pipelined kernels above (profiles/r02_ncu_full.md) shows the shared-memory SRAM as their co-critical
// unit, and 15-20 % of its wavefronts are LSU accesses replayed because the copy engine was using the banks: a
// three-pass transform costs EIGHT passes over its tile there (bulk copy in, LDS, two exchanges, STS, bulk copy out).
// This kernel takes the input off that SRAM: every thread loads the NEXT transform's E values straight from global
// memory into a second register set (coalesced 128-byte LDGs, issued before the current transform's first pass and
// consumed a whole transform later, so their latency is covered without a stage buffer), and the current transform
// runs out of the first set.  The loop body is instantiated twice with the two register sets swapped (no copies).
// TS: results leave through one of two alternating shared-memory tiles as bulk stores (as in k_c2c_pipe); otherwise
// as per-thread streaming stores.
// ----------------------------------------------------------------------------------------
template <int N_> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N_) : "memory"); }

template <typename R, class PL, int PADQ, int IO, bool INV, int MINB, bool TS>
__global__ void __launch_bounds__(PL::T, MINB) k_c2c_rpf(const __grid_constant__ KParams p) {
    static_assert(PL::valid() && RT<R>::LANES == 1 && PL::T >= 32 && PL::npass() > 1, "multi-pass scalar-lane plans");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using S = typename VecOf<R>::s;
    using V2 = typename VecOf<R>::v2;
    constexpr int N = PL::N, T = PL::T, E = PL::E;
    constexpr int LAST = PL::npass() - 1;
    constexpr size_t BUF = pipe_buf_bytes<R, PL, PADQ, 1>();
    constexpr int NBUF = TS ? 2 : 1;
    long *slot = reinterpret_cast<long *>(smem_raw + NBUF * BUF);        // tile claimed for iteration parity 0 / 1
    const int tid = threadIdx.x;
    const typename RT<R>::twel *tw = reinterpret_cast<const typename RT<R>::twel *>(p.tw);
    const long tiles = p.batch;
    const auto tw0 = UTw<R, PL>::make(p, tw);
    const R sc = RT<R>::splat((S)p.scale);

    auto load = [&](long row, cx<R> (&v)[E]) {
        if constexpr (IO == IO_SPLIT) {
            const S *re = reinterpret_cast<const S *>(p.in0) + row * N + tid;
            const S *im = reinterpret_cast<const S *>(p.in1) + row * N + tid;
            static_for<E>([&](auto E_) { CIDX(e, E_); v[e] = mk<R>(ld_stream(re + e * T), ld_stream(im + e * T)); });
        } else {
            const V2 *z = reinterpret_cast<const V2 *>(p.in0) + row * N + tid;
            static_for<E>([&](auto E_) { CIDX(e, E_); const V2 a = ld_stream(z + e * T); v[e] = mk<R>(a.x, a.y); });
        }
    };
    auto store_tile = [&](long row, int st) {                              // thread 0: the finished tile in buffer st
        const unsigned char *src = smem_raw + st * BUF;
        constexpr uint32_t ROWB = (uint32_t)((IO == IO_SPLIT ? 1 : 2) * N * sizeof(S));
        tma_store_1d(reinterpret_cast<unsigned char *>(p.out0) + row * ROWB, src, ROWB);
        if constexpr (IO == IO_SPLIT) tma_store_1d(reinterpret_cast<unsigned char *>(p.out1) + row * ROWB, src + ROWB, ROWB);
        bulk_commit();
    };

    if (tid == 0) slot[0] = (long)atomicAdd(p.ctr, 1ULL);
    __syncthreads();
    long tile = slot[0], prev = -1;
    int it = 0;
    cx<R> ra[E], rb[E];
    if (tile < tiles) load(tile, ra);

    // one iteration: x holds `tile` (loads possibly still in flight), nx receives the next tile
    auto iter = [&](cx<R> (&x)[E], cx<R> (&nx)[E]) -> bool {
        const int st = TS ? (it & 1) : 0;
        if (tid == 0) {
            slot[(it + 1) & 1] = (long)atomicAdd(p.ctr, 1ULL);
            // TS: the store issued one iteration ago (tile it-2, out of buffer st) has had a whole transform to drain
            if constexpr (TS) bulk_wait_read<0>();
        }
        if constexpr (TS) fence_proxy_async();        // our result writes (generic proxy) precede the bulk store below
        __syncthreads();                              // slot published; last tile's results complete; scratch free
        if constexpr (TS) { if (prev >= 0 && tid == 0) store_tile(prev, st ^ 1); }
        if (tile >= tiles) return false;
        const long next = slot[(it + 1) & 1];
        if (next < tiles) load(next, nx);
        unsigned char *buf = smem_raw + st * BUF;
        run_all<R, PL, PADQ, 1, INV>(x, tw, tw0, reinterpret_cast<cx<R> *>(buf), tid, 0, false);
        if constexpr (TS) {
            __syncthreads();                          // the result rows alias the scratch everyone just read
            if constexpr (IO == IO_SPLIT) {
                S *re = reinterpret_cast<S *>(buf) + tid;
                S *im = re + N;
                static_for<E>([&](auto S_) {
                    CIDX(slot_, S_);
                    constexpr int e = out_elem<PL, LAST>(slot_);
                    cx<R> v = x[slot_];
                    if (INV) v = mk<R>(rmul(v.x, sc), rmul(v.y, sc));
                    re[e * T] = v.x; im[e * T] = v.y;
                });
            } else {
                V2 *z = reinterpret_cast<V2 *>(buf) + tid;
                static_for<E>([&](auto S_) {
                    CIDX(slot_, S_);
                    constexpr int e = out_elem<PL, LAST>(slot_);
                    cx<R> v = x[slot_];
                    if (INV) v = mk<R>(rmul(v.x, sc), rmul(v.y, sc));
                    V2 o; o.x = v.x; o.y = v.y;
                    z[e * T] = o;
                });
            }
        } else {
            if constexpr (IO == IO_SPLIT) {
                S *re = reinterpret_cast<S *>(p.out0) + tile * N + tid;
                S *im = reinterpret_cast<S *>(p.out1) + tile * N + tid;
                static_for<E>([&](auto S_) {
                    CIDX(slot_, S_);
                    constexpr int e = out_elem<PL, LAST>(slot_);
                    cx<R> v = x[slot_];
                    if (INV) v = mk<R>(rmul(v.x, sc), rmul(v.y, sc));
                    GIO<R>::st_split(re + e * T, im + e * T, 0, false, v);
                });
            } else {
                V2 *z = reinterpret_cast<V2 *>(p.out0) + tile * N + tid;
                static_for<E>([&](auto S_) {
                    CIDX(slot_, S_);
                    constexpr int e = out_elem<PL, LAST>(slot_);
                    cx<R> v = x[slot_];
                    if (INV) v = mk<R>(rmul(v.x, sc), rmul(v.y, sc));
                    GIO<R>::st_il(z + e * T, 0, false, v);
                });
            }
        }
        prev = tile; tile = next; it++;
        return true;
    };
    for (;;) {
        if (!iter(ra, rb)) break;
        if (!iter(rb, ra)) break;
    }
    if constexpr (TS) { if (tid == 0) bulk_wait_read<0>(); }             // shared memory must outlive the stores that read it
    claim_epilogue(p.ctr);
}


// ----------------------------------------------------------------------------------------
// Persistent, fully TMA-fed thread-per-row c2c (N <= 64, f32).  Same arithmetic as k_c2c_tile, but no thread
// ever touches global memory: rows arrive by bulk copy, are transformed in place by their thread, and leave by
// bulk store.  Against k_c2c_tile this drops the cooperative staging loops -- a third of the LSU instructions
// and half the shared-memory traffic per row, which is what the kernel is short of once the SM clock sits at
// the power cap.
//   * The copy engine retires roughly one bulk operation per 14 clocks per SM (measured: 256-byte row copies
//     cap the kernel at 78 % of the HBM peak, 512-byte ones do not), so G consecutive rows travel as ONE
//     512-byte copy per plane.  A group lands as [G rows re | G rows im | 16 bytes pad] (interleaved: [G rows |
//     pad]); thread t owns row G*(t mod X/G) + t/(X/G) of the tile, so 8 consecutive lanes sit in 8 consecutive
//     groups, whose stride is an odd number of 16-byte bank groups: LDS.128/STS.128 are conflict-free.
//   * Two stages; the stage being refilled is the one whose bulk stores were issued last, so the issuing lanes
//     drain their own store group (cp.async.bulk.wait_group.read) right before the refill -- after the row
//     loads of the current tile, which gives the store engine that time for free.
// ----------------------------------------------------------------------------------------
// Bytes per bulk copy.  Every copy is issued by one lane through a uniform-datapath instruction (UBLKCP), which the
// compiler wraps in an elect / R2UR / branch sequence of ~9 instructions per lane and copy: at 512 bytes the N = 64
// split kernel spent 64 copies x 9 = 30 % of its instructions (ncu r01: R2UR 15 %, PLOP3 13 %) issuing them, all
// serialised in the one warp that also does the arithmetic.  Wider groups mean fewer copies where the row is wide
// enough for the arithmetic to matter: N = 64 split moves 1024 bytes per copy with 32-row tiles (+2.3 % under the
// power cap) and 2048 bytes with 64-row tiles (two warps per CTA, the default: another +1 %); N = 16, 32 and the
// interleaved rows keep 512 (no change or -0.7 % with more).  A tile always has at least 8 groups (the lane <-> row
// mapping below needs them).  -DWFB_TPIPE_GROUP_BYTES=n forces one size everywhere (A/B builds).
#ifndef WFB_TPIPE_WIDE_GROUP_BYTES
#define WFB_TPIPE_WIDE_GROUP_BYTES 2048
#endif
template <typename R, class PL, int IO, int X> __host__ __device__ constexpr int tpipe_group() {
    const int row_bytes = (IO == IO_SPLIT ? 1 : 2) * (int)sizeof(R) * PL::N;   // bytes of one row in one plane
#ifdef WFB_TPIPE_GROUP_BYTES
    const int group_bytes = WFB_TPIPE_GROUP_BYTES;
#else
    const int group_bytes = (IO == IO_SPLIT && sizeof(R) == 4 && PL::N >= 64) ? WFB_TPIPE_WIDE_GROUP_BYTES : 512;
#endif
    const int g = row_bytes >= group_bytes ? 1 : group_bytes / row_bytes;
    return g > X / 8 ? X / 8 : g;                      // at least 8 groups per tile (lane <-> row mapping below)
}
template <typename R, class PL, int X, int IO> __host__ __device__ constexpr size_t tpipe_buf_bytes() {
    constexpr int G = tpipe_group<R, PL, IO, X>();
    return ((size_t)(G * 2 * sizeof(R) * PL::N + 16) * (X / G) + 127) / 128 * 128;
}

template <typename R, class PL, int X, int IO, bool INV, int MINB>
__global__ void __launch_bounds__(X, MINB) k_c2c_tpipe(const __grid_constant__ KParams p) {
    static_assert(PL::valid() && PL::T == 1 && PL::npass() == 1 && X % 32 == 0, "tile kernel: one thread per row, whole warps");
    static_assert(RT<R>::LANES == 1 && (sizeof(R) == 4 || IO == IO_INTERLEAVED), "f32 (both layouts) or f64 interleaved");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int N = PL::N;
    constexpr int ES = (int)sizeof(R);                 // bytes of a real
    constexpr int G = tpipe_group<R, PL, IO, X>();     // rows per bulk copy
    constexpr int NG = X / G;                          // groups per tile
    static_assert(X % G == 0 && NG % 8 == 0, "8 consecutive lanes must sit in 8 consecutive groups");
    constexpr int GSTR = G * 2 * ES * N + 16;          // group stride, bytes (odd multiple of 16)
    constexpr int PLANE = (IO == IO_SPLIT ? 1 : 2) * ES * N;   // bytes of one row in one plane
    constexpr size_t BUF = tpipe_buf_bytes<R, PL, X, IO>();
    uint64_t *mbar = reinterpret_cast<uint64_t *>(smem_raw + 2 * BUF);
    long *slot = reinterpret_cast<long *>(smem_raw + 2 * BUF + 32);
    const int t = threadIdx.x;
    const int gj = t % NG, gb = t / NG;                // my group, my row within it
    const long tiles = (p.batch + X - 1) / X;
    const typename RT<R>::twel *tw = reinterpret_cast<const typename RT<R>::twel *>(p.tw);
    auto cta_sync = [&]() { if constexpr (X == 32) __syncwarp(); else __syncthreads(); };

    if (t == 0) {
        mbar_init(mbar + 0, 1);
        mbar_init(mbar + 1, 1);
        fence_proxy_async();
    }
    cta_sync();

    auto tile_rows = [&](long tile) { const long row = tile * X; return (p.batch - row < X) ? (int)(p.batch - row) : X; };
    auto issue = [&](long tile, int st) {              // warp 0, all lanes
        const int rows = tile_rows(tile);
        unsigned char *buf = smem_raw + st * BUF;
        bulk_wait_read_all();                          // this lane's stores out of this stage have left shared memory
        if (t == 0) mbar_expect_tx(mbar + st, (uint32_t)(rows * 2 * ES * N));
        __syncwarp();
        for (int g = t; g * G < rows; g += 32) {
            const long row = tile * X + (long)g * G;
            const int nr = rows - g * G < G ? rows - g * G : G;
            unsigned char *dst = buf + (size_t)g * GSTR;
            if constexpr (IO == IO_SPLIT) {
                tma_load_1d(dst, reinterpret_cast<const R *>(p.in0) + row * N, (uint32_t)(nr * PLANE), mbar + st);
                tma_load_1d(dst + G * PLANE, reinterpret_cast<const R *>(p.in1) + row * N, (uint32_t)(nr * PLANE), mbar + st);
            } else {
                tma_load_1d(dst, reinterpret_cast<const R *>(p.in0) + row * 2 * N, (uint32_t)(nr * PLANE), mbar + st);
            }
        }
    };

    long pending = claim_prime<true>(p.ctr);
    claim_and_issue<true>(p.ctr, pending, tiles, slot, 0, issue);
    unsigned phasebits = 0;
    cx<R> x[N];
    for (int it = 0;; it++) {
        const int st = it & 1;
        cta_sync();                                    // slot[st] is published; last iteration's stores are issued
        const long tile = slot[st];
        if (tile >= tiles) break;
        unsigned char *buf = smem_raw + st * BUF;
        const int rows = tile_rows(tile);
        mbar_wait(mbar + st, (phasebits >> st) & 1u);
        phasebits ^= 1u << st;

        unsigned char *grp = buf + (size_t)gj * GSTR;
        float4 *rowp = reinterpret_cast<float4 *>(grp + gb * PLANE);               // re row (or the interleaved row)
        float4 *rowq = reinterpret_cast<float4 *>(grp + (G + gb) * PLANE);         // im row (split only)
        if constexpr (IO == IO_SPLIT) {
            static_for<N / 4>([&](auto H_) {
                CIDX(h, H_);
                const float4 a = rowp[h], b = rowq[h];
                x[4 * h] = mk<R>(a.x, b.x); x[4 * h + 1] = mk<R>(a.y, b.y);
                x[4 * h + 2] = mk<R>(a.z, b.z); x[4 * h + 3] = mk<R>(a.w, b.w);
            });
        } else if constexpr (sizeof(R) == 8) {
            const double2 *rowd = reinterpret_cast<const double2 *>(rowp);
            static_for<N>([&](auto H_) { CIDX(h, H_); const double2 v = rowd[h]; x[h] = mk<R>(v.x, v.y); });
        } else {
            static_for<N / 2>([&](auto H_) {
                CIDX(h, H_);
                const float4 v = rowp[h];
                x[2 * h] = mk<R>(v.x, v.y); x[2 * h + 1] = mk<R>(v.z, v.w);
            });
        }
        claim_and_issue<true>(p.ctr, pending, tiles, slot, st ^ 1, issue);       // refill the other stage while this tile computes

        run_pass<R, PL, 0, INV>(x, tw, UTw<R, PL>::make(p, tw), 0);

        const R sc = INV ? (R)p.scale : R(1);
        if constexpr (IO == IO_SPLIT) {
            static_for<N / 4>([&](auto H_) {
                CIDX(h, H_);
                constexpr int s0 = slot_of_elem<PL, 0>(4 * h), s1 = slot_of_elem<PL, 0>(4 * h + 1);
                constexpr int s2 = slot_of_elem<PL, 0>(4 * h + 2), s3 = slot_of_elem<PL, 0>(4 * h + 3);
                float4 a = make_float4(x[s0].x, x[s1].x, x[s2].x, x[s3].x), b = make_float4(x[s0].y, x[s1].y, x[s2].y, x[s3].y);
                if (INV) { a = make_float4(a.x * sc, a.y * sc, a.z * sc, a.w * sc); b = make_float4(b.x * sc, b.y * sc, b.z * sc, b.w * sc); }
                rowp[h] = a; rowq[h] = b;
            });
        } else if constexpr (sizeof(R) == 8) {
            double2 *rowd = reinterpret_cast<double2 *>(rowp);
            static_for<N>([&](auto H_) {
                CIDX(h, H_);
                constexpr int s0 = slot_of_elem<PL, 0>(h);
                double2 v = make_double2(x[s0].x, x[s0].y);
                if (INV) v = make_double2(v.x * sc, v.y * sc);
                rowd[h] = v;
            });
        } else {
            static_for<N / 2>([&](auto H_) {
                CIDX(h, H_);
                constexpr int s0 = slot_of_elem<PL, 0>(2 * h), s1 = slot_of_elem<PL, 0>(2 * h + 1);
                float4 v = make_float4(x[s0].x, x[s0].y, x[s1].x, x[s1].y);
                if (INV) v = make_float4(v.x * sc, v.y * sc, v.z * sc, v.w * sc);
                rowp[h] = v;
            });
        }
        fence_proxy_async();                           // generic-proxy writes -> visible to the bulk-copy engine
        cta_sync();
        if (t < 32) {
            for (int g = t; g * G < rows; g += 32) {
                const long row = tile * X + (long)g * G;
                const int nr = rows - g * G < G ? rows - g * G : G;
                const unsigned char *src = buf + (size_t)g * GSTR;
                if constexpr (IO == IO_SPLIT) {
                    tma_store_1d(reinterpret_cast<R *>(p.out0) + row * N, src, (uint32_t)(nr * PLANE));
                    tma_store_1d(reinterpret_cast<R *>(p.out1) + row * N, src + G * PLANE, (uint32_t)(nr * PLANE));
                } else {
                    tma_store_1d(reinterpret_cast<R *>(p.out0) + row * 2 * N, src, (uint32_t)(nr * PLANE));
                }
            }
            bulk_commit();
        }
    }
    if (t < 32) bulk_wait_read_all();                  // shared memory must outlive the stores that read it
    claim_epilogue(p.ctr);
}


// ----------------------------------------------------------------------------------------
// TMA-pipelined persistent r2c / c2r (scalar lanes).  Same pipeline as k_c2c_pipe: the next tile
// of X rows is streamed into shared memory while the current one is transformed.
//   r2c: rows of N reals are read as M = N/2 complex values; the Hermitian post-process runs out
//        of the group's scratch into coalesced 8-byte stores of the (M+1)-bin rows.
//   c2r: rows are (M+1) complex values (8-byte aligned only), so tiles hold an even number of rows
//        (16-byte aligned starts and sizes); an odd-sized last tile is copied by the threads.
// ----------------------------------------------------------------------------------------
template <typename R, class PL, int PADQ, int X, bool C2R> __host__ __device__ constexpr size_t real_pipe_buf_bytes() {
    size_t scratch = sizeof(cx<R>) * (size_t)padded_size<PADQ>(PL::N) * X;
    size_t raw = sizeof(cx<R>) * (size_t)(C2R ? PL::N + 1 : PL::N) * X;
    size_t a = scratch > raw ? scratch : raw;
    return (a + 127) / 128 * 128;
}

// TS ("TMA stores", as in k_c2c_pipe): results are assembled as a dense tile in the stage buffer and leave as ONE
// bulk store after the next loop-top barrier.  r2c: each row's (M+1) bins; the mirrored halves are parked in the
// row's own slots [1, M/2], and the thread that reads park[k] is the one that overwrites it with X[k], so the
// post-process is in place.  c2r: the M complex (= N real) outputs of each row.
#ifndef WFB_REAL_DENSE
#define WFB_REAL_DENSE 0           // 1: the dense side of every tile as one block (A/B builds; see GROUPED below)
#endif
template <typename R, class PL, int X, int PADQ, bool C2R, int MINB, bool RC = false, bool TS = false, bool HT = false>
__global__ void __launch_bounds__(PL::T *X, MINB) k_real_pipe(const __grid_constant__ KParams p) {
    static_assert(PL::valid() && RT<R>::LANES == 1, "scalar lanes only");
    static_assert(!C2R || X % 2 == 0 || X == 1 || sizeof(R) == 8, "f32 c2r tiles: an even number of rows (16-byte alignment), or single rows");
    // c2r with ONE row per tile (N >= 4096: a row is the 16 KB tile): rows are (M+1) bins = 8 bytes more than a multiple
    // of 16, so the copy of row r covers (M+2) bins starting at bin -(r & 1) of the row -- 16-byte aligned start and size;
    // the extra bin belongs to a neighbouring row and is ignored.  (The very last row of an odd batch has no bin after
    // it: it takes the cooperative-copy path.)
    constexpr bool SHIFT = C2R && X == 1 && sizeof(R) == 4;     // (f64 rows are 16-byte multiples already)
    static_assert(!RC || (!C2R && PL::N >= 32 && PL::T * X >= 32), "row copies: r2c only (c2r rows are 8-byte aligned)");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using S = typename VecOf<R>::s;
    using V2 = typename VecOf<R>::v2;
    constexpr int M = PL::N;
    constexpr int LAST = PL::npass() - 1;
    constexpr int IN_ROW = C2R ? M + 1 : M;          // row lengths in complex values
    constexpr int RSTR = RC ? M + M / 16 : IN_ROW;   // smem row stride (RC: rows T banks apart, see k_c2c_pipe)
    static_assert(!RC || RSTR <= padded_size<PADQ>(M), "padded rows must fit the stage buffer (sized for the scratch)");
    constexpr size_t BUF = real_pipe_buf_bytes<R, PL, PADQ, X, C2R>();
    uint64_t *mbar = reinterpret_cast<uint64_t *>(smem_raw + 2 * BUF);
    const int xi = threadIdx.x / PL::T, tid = threadIdx.x % PL::T;
    // r2c with bulk stores and thread groups narrower than a shared-memory phase (T < 16 lanes of 8 bytes, < 8 of 16):
    // the GP = phase/T groups that share a phase take rows T apart -- the dense result rows have an odd stride
    // ((M+1) bins), so rows h, h+T, ... land in disjoint bank ranges, while adjacent rows would overlap in all but one
    // bank (ncu: 2-way conflicts on every park/result access at N = 256).  Row of the tile this group works on:
    constexpr int PHL = 128 / (int)sizeof(typename VecOf<R>::v2);     // lanes per phase
    // GROUPED: the DENSE side of such a tile (the r2c input rows, the c2r result rows: stride M bins, a multiple of 32
    // banks) would put the two thread groups of a phase on the same banks whatever rows they take (ncu r02, N = 256:
    // 33 / 40 % of the shared-memory wavefronts replayed, pipe at 90 / 94 %).  With exactly two groups per phase the dense
    // side therefore moves in groups of T rows, one bulk copy each, with 64 bytes of padding behind every group: rows a
    // and a + T then sit 16 banks apart.  The c2r direction uses the same row mapping (its (M+1)-bin input rows are the
    // odd-stride side there).
    constexpr bool GROUPED = TS && !RC && X > 1 && PL::T < PHL && PHL / PL::T == 2 && X % PHL == 0 && !WFB_REAL_DENSE;
    constexpr bool ROWMAP = (!C2R || GROUPED) && TS && PL::T < PHL && X % PHL == 0;
    const int xr = ROWMAP ? ((xi / (PHL / PL::T)) / PL::T) * PHL + (xi / (PHL / PL::T)) % PL::T + PL::T * (xi % (PHL / PL::T)) : xi;
    constexpr int GPAD = 64 / (int)sizeof(typename VecOf<R>::v2);                  // padding behind a dense-side group, bins
    constexpr int GSTR = PL::T * M + GPAD;                                           // dense-side group stride, bins
    constexpr int NGRP = X / PL::T;                                                  // dense-side groups per tile
    static_assert(!GROUPED || (size_t)NGRP * GSTR * sizeof(typename VecOf<R>::v2) <= real_pipe_buf_bytes<R, PL, PADQ, X, C2R>(),
                  "the padded dense side must fit the stage buffer (sized for the scratch)");
    const int doff = GROUPED ? (xr / PL::T) * GSTR + (xr % PL::T) * M : xr * M;      // my dense-side row, bins
    const typename RT<R>::twel *tw = reinterpret_cast<const typename RT<R>::twel *>(p.tw);
    const typename RT<R>::twel *rtw = reinterpret_cast<const typename RT<R>::twel *>(p.rtw);
    const long tiles = (p.batch + X - 1) / X;
    const V2 *gin = reinterpret_cast<const V2 *>(p.in0);
    constexpr int OUT_ROW = C2R ? M : M + 1;         // row lengths of the result tile, complex values
    V2 *gout = reinterpret_cast<V2 *>(p.out0);

    if (threadIdx.x == 0) {
        mbar_init(mbar + 0, 1);
        mbar_init(mbar + 1, 1);
        fence_proxy_async();
    }
    __syncthreads();

    auto tile_rows = [&](long tile) { const long row = tile * X; return (p.batch - row < X) ? (int)(p.batch - row) : X; };
    auto tma_ok = [&](long tile) { return !C2R || sizeof(R) == 8 || (SHIFT ? ((tile & 1) || tile + 1 < p.batch) : (tile_rows(tile) % 2 == 0)); };
    auto issue = [&](long tile, int st) {
        if constexpr (TS) { bulk_wait_read_all(); __syncwarp(); }   // the stores out of this stage have drained
        if (!tma_ok(tile)) return;
        const int rows = tile_rows(tile);
        if constexpr (SHIFT) {
            if (threadIdx.x == 0) {
                const uint32_t bytes = (uint32_t)((M + 2) * sizeof(V2));
                mbar_expect_tx(mbar + st, bytes);
                tma_load_1d(smem_raw + st * BUF, gin + tile * IN_ROW - (tile & 1), bytes, mbar + st);
            }
        } else if constexpr (GROUPED && !C2R) {
            if (threadIdx.x == 0) {                   // the dense time-domain side: one copy per group of T rows
                mbar_expect_tx(mbar + st, (uint32_t)(rows * M * sizeof(V2)));
                for (int g = 0; g * PL::T < rows; g++) {
                    const int nr = rows - g * PL::T < PL::T ? rows - g * PL::T : PL::T;
                    tma_load_1d(smem_raw + st * BUF + (size_t)g * GSTR * sizeof(V2), gin + (tile * X + (long)g * PL::T) * M,
                                (uint32_t)(nr * M * sizeof(V2)), mbar + st);
                }
            }
        } else if constexpr (!RC) {
            if (threadIdx.x == 0) {
                const uint32_t bytes = (uint32_t)(rows * IN_ROW * sizeof(V2));
                mbar_expect_tx(mbar + st, bytes);
                tma_load_1d(smem_raw + st * BUF, gin + tile * X * IN_ROW, bytes, mbar + st);
            }
        } else {
            if (threadIdx.x < 32) {
                if (threadIdx.x == 0) mbar_expect_tx(mbar + st, (uint32_t)(rows * IN_ROW * sizeof(V2)));
                __syncwarp();
                for (int r = threadIdx.x; r < rows; r += 32)
                    tma_load_1d(smem_raw + st * BUF + (size_t)r * RSTR * sizeof(V2), gin + (tile * X + r) * IN_ROW,
                                (uint32_t)(IN_ROW * sizeof(V2)), mbar + st);
            }
        }
    };

    // TS: the finished tile in stage st leaves as one bulk store (odd-sized last r2c tile: plain stores by warp 0)
    // r2c with ONE row per tile (f32, N >= 4096): a row of (M+1) bins is 8 bytes more than a multiple of 16 and odd rows
    // start 8 bytes off.  The row is assembled at element offset (row & 1) of the stage, M of its bins leave as one
    // aligned bulk store (bins 0..M-1 of an even row, 1..M of an odd one) and the remaining bin as a plain store.
    constexpr bool ROW1 = !C2R && TS && X == 1 && sizeof(R) == 4;
    auto store_tile = [&](long tile, int st) {
        if (threadIdx.x >= 32) return;
        const int count = tile_rows(tile) * OUT_ROW;
        const V2 *src = reinterpret_cast<const V2 *>(smem_raw + st * BUF);
        V2 *dst = gout + tile * X * OUT_ROW;
        if constexpr (GROUPED && C2R) {
            if (threadIdx.x == 0) {                   // the dense time-domain side: one store per group of T rows
                const int rows = tile_rows(tile);
                for (int g = 0; g * PL::T < rows; g++) {
                    const int nr = rows - g * PL::T < PL::T ? rows - g * PL::T : PL::T;
                    tma_store_1d(dst + (size_t)g * PL::T * M, src + (size_t)g * GSTR, (uint32_t)(nr * M * sizeof(V2)));
                }
                bulk_commit();
            }
        } else if constexpr (ROW1) {
            if (threadIdx.x == 0) {
                const int sh = (int)(tile & 1);
                tma_store_1d(dst + sh, src + 2 * sh, (uint32_t)(M * sizeof(V2)));
                bulk_commit();
                st_stream(dst + (sh ? 0 : M), src[sh ? 1 : M]);
            }
        } else if ((count * sizeof(V2)) % 16 == 0) {
            if (threadIdx.x == 0) { tma_store_1d(dst, src, (uint32_t)(count * sizeof(V2))); bulk_commit(); }
        } else {
            for (int i = threadIdx.x; i < count; i += 32) st_stream(dst + i, src[i]);
        }
    };

    static_assert(PL::T * X >= 32, "tile claims are made by a full warp");
    long *slot = reinterpret_cast<long *>(smem_raw + 2 * BUF + 32);   // tile claimed for each stage
    long pending = claim_prime<false>(p.ctr);
    claim_and_issue<false>(p.ctr, pending, tiles, slot, 0, issue);
    cx<R> x[PL::E];
    typename RT<R>::twel hw[HT ? hoist_count<R, PL, (LAST > 0 ? LAST : 1)>() : 1];      // HT: see k_c2c_pipe
    if constexpr (HT) { static_assert(LAST > 0, "hoisting needs a multi-pass plan"); hoist_load<R, PL, LAST>(hw, tw, tid); }
    const auto hsrc = [&]() { if constexpr (HT) return Hoisted<R>{hw}; else return NoHoist{}; }();
    unsigned phasebits = 0;                            // mbarrier phase parity per stage (bit st)
    for (int it = 0;; it++) {
        const int st = it & 1;
        fence_proxy_async();
        __syncthreads();
        if constexpr (TS) { if (it > 0) store_tile(slot[st ^ 1], st ^ 1); }   // last iteration's results (all written: barrier above)
        const long tile = slot[st];
        if (tile >= tiles) break;
        if constexpr (!TS) claim_and_issue<false>(p.ctr, pending, tiles, slot, st ^ 1, issue);
        unsigned char *buf = smem_raw + st * BUF;
        if (tma_ok(tile)) {
            mbar_wait(mbar + st, (phasebits >> st) & 1u);
            phasebits ^= 1u << st;
        } else {                                       // odd-sized last c2r tile: plain cooperative copy
            const int count = tile_rows(tile) * IN_ROW;
            V2 *dst = reinterpret_cast<V2 *>(buf);
            for (int i = threadIdx.x; i < count; i += PL::T * X) dst[i] = ld_stream(gin + tile * X * IN_ROW + i);
            __syncthreads();
        }
        const long row = tile * X + xr;
        const bool active = row < p.batch;
        cx<R> *scratch = reinterpret_cast<cx<R> *>(buf) + (size_t)xi * padded_size<PADQ>(M);
        const V2 *raw = reinterpret_cast<const V2 *>(buf) + ((GROUPED && !C2R) ? (size_t)doff : (size_t)xr * RSTR) + ((SHIFT && tma_ok(tile)) ? (int)(tile & 1) : 0);

        if constexpr (!C2R) {
            // ---------------- r2c
            static_for<PL::E>([&](auto E_) { CIDX(e, E_); const V2 a = raw[tid + e * PL::T]; x[e] = mk<R>(a.x, a.y); });
            __syncthreads();                           // dense tile and padded scratch alias
            if constexpr (TS) claim_and_issue<false>(p.ctr, pending, tiles, slot, st ^ 1, issue);   // (slot[st ^ 1] was read before the barrier)
            run_all<R, PL, PADQ, X, false>(x, tw, UTw<R, PL>::make(p, tw), scratch, tid, xi, false, hsrc);
            // TS: the result rows are dense ([X][M+1]) and alias the other groups' scratch
            cx<R> *park = TS ? reinterpret_cast<cx<R> *>(buf) + (size_t)xr * (M + 1) + (ROW1 ? (int)(tile & 1) : 0) : scratch;
            if (PL::npass() > 1) { if constexpr (TS && X > 1) __syncthreads(); else sync_transform<PL::T, X>(xi); }
            // Hermitian post-process: bin k = tid + i*T (k < M/2) pairs the thread's OWN register value Z[k] with
            // Z[M-k], which another thread of the group owns.  Only the upper half (elements >= M/2) travels
            // through shared memory: half a spill and half a re-read instead of a full spill and two full reads.
            // Z[k'] is parked at UNPADDED index M - k' (1..M/2), i.e. at the bin index of the thread that reads it:
            // readers tid, tid+1, ... hit consecutive words, and so do writers (thread 0 lands on column T of the
            // row the others fill at columns 1..T-1).
            static_for<PL::E>([&](auto S_) {
                CIDX(slot, S_);
                constexpr int e = out_elem<PL, LAST>(slot);
                if constexpr (e >= PL::E / 2) park[M - e * PL::T - tid] = x[slot];
            });
            sync_transform<PL::T, X>(xi);
            if (active || TS) {
                V2 *out = TS ? reinterpret_cast<V2 *>(park) : reinterpret_cast<V2 *>(p.out0) + row * (M + 1);
                constexpr int HALF = M / 2;
                constexpr int PER = PL::E / 2;
                static_assert(PER * PL::T == HALF, "bins per thread");
                const R zero = RT<R>::splat(0);
                auto put = [&](V2 *q, cx<R> v) { if constexpr (TS) { V2 o; o.x = v.x; o.y = v.y; *q = o; } else GIO<R>::st_il(q, 0, false, v); };
                static_for<PER>([&](auto I_) {
                    CIDX(i, I_);
                    const int k = tid + i * PL::T;
                    const cx<R> z = x[slot_of_elem<PL, LAST>(i)];
                    if (i == 0 && k == 0) {
                        put(out, mk<R>(radd(z.x, z.y), zero));
                        put(out + M, mk<R>(rsub(z.x, z.y), zero));
                        const cx<R> zh = park[HALF];
                        put(out + HALF, RealPost<R>::middle(zh, ld_tw(rtw + HALF), M));
                    } else {
                        const cx<R> zm = park[k];
                        cx<R> xk, xm;
                        const twd<R> wk = ld_tw(rtw + k);
                RealPost<R>::pair(z, zm, wk, ld_tw_mirror<R>(rtw, k, M, wk), xk, xm);
                        put(out + k, xk);
                        put(out + (M - k), xm);
                    }
                });
            }
        } else {
            // ---------------- c2r: Hermitian pre-process into registers, then through the scratch
            constexpr int HALF = M / 2;
            constexpr int PER = PL::E / 2;
            static_assert(PER * PL::T == HALF, "bins per thread");
            // Z[k] for k = tid + i*T < M/2 is this thread's own pass-0 input e = i: it stays in its register.
            // Only the mirrored halves Z[M-k] travel through the scratch to the threads that own them.
            const R sc = RT<R>::splat(S(0.5) / S(M));
            cx<R> zb[PER];
            static_for<PER>([&](auto I_) {
                CIDX(i, I_);
                const int k = tid + i * PL::T;
                const int kk = (i == 0 && k == 0) ? HALF : k;
                const V2 a = raw[kk], b = raw[M - kk];
                const twd<R> w = ld_tw(rtw + kk);
                const R gr = radd(a.x, b.x), gi = rsub(a.y, b.y), ur = rsub(a.x, b.x), ui = radd(a.y, b.y);
                const R hr = rfma(w.y, ui, rmul(w.x, ur)), hi = rfma(w.ny, ur, rmul(w.x, ui));
                x[i] = mk<R>(rmul(sc, rsub(gr, hi)), rmul(sc, radd(gi, hr)));
                zb[i] = mk<R>(rmul(sc, radd(gr, hi)), rmul(sc, rsub(hr, gi)));
                if (i == 0 && k == 0) {
                    const V2 a0 = raw[0], am = raw[M];              // real parts only (:1679-1684)
                    x[0] = mk<R>(rmul(radd(a0.x, am.x), sc), rmul(rsub(a0.x, am.x), sc));
                }
            });
            __syncthreads();                           // every group has consumed its raw rows
            if constexpr (TS) claim_and_issue<false>(p.ctr, pending, tiles, slot, st ^ 1, issue);
            static_for<PER>([&](auto I_) {
                CIDX(i, I_);
                const int k = tid + i * PL::T;
                const int kk = (i == 0 && k == 0) ? HALF : k;       // Z[M/2]: the mirrored form survives (:1722-1740)
                scratch[kk] = zb[i];                   // Z[M - kk] parked at unpadded index kk (conflict-free both ways)
            });
            sync_transform<PL::T, X>(xi);
            static_for<PER>([&](auto E_) { CIDX(e, E_); x[PER + e] = scratch[M - (PER + e) * PL::T - tid]; });
            run_all<R, PL, PADQ, X, true>(x, tw, UTw<R, PL>::make(p, tw), scratch, tid, xi, true, hsrc);
            if constexpr (TS) {
                if constexpr (X > 1) __syncthreads(); else sync_transform<PL::T, X>(xi);   // result rows alias the scratch
                V2 *z = reinterpret_cast<V2 *>(buf) + (GROUPED ? (size_t)doff : (size_t)xi * M) + tid;
                static_for<PL::E>([&](auto S_) {
                    CIDX(slot_, S_);
                    constexpr int e = out_elem<PL, LAST>(slot_);
                    V2 o; o.x = x[slot_].x; o.y = x[slot_].y;
                    z[e * PL::T] = o;
                });
            } else if (active) {
                V2 *z = reinterpret_cast<V2 *>(p.out0) + row * M + tid;
                static_for<PL::E>([&](auto S_) {
                    CIDX(slot, S_);
                    constexpr int e = out_elem<PL, LAST>(slot);
                    GIO<R>::st_il(z + e * PL::T, 0, false, x[slot]);
                });
            }
        }
    }
    if constexpr (TS) { if (threadIdx.x < 32) bulk_wait_read_all(); }   // shared memory must outlive the stores that read it
    claim_epilogue(p.ctr);
}


// ----------------------------------------------------------------------------------------
// Small-N real transforms (N <= 128, core M = N/2 <= 64): thread-per-row tile kernels, the real
// counterparts of k_c2c_tile.  The Hermitian post/pre-process happens entirely in registers (the
// thread owns every Z[k] of its row).  Spectrum rows are (M+1) complex values = an ODD number of
// 8-byte words, so the dense [rows][M+1] tile is already bank-conflict-free for per-thread row
// access and is copied to/from global memory as one contiguous, 16-byte aligned block.
// ----------------------------------------------------------------------------------------

template <class PL, int X, int MINB>
__global__ void __launch_bounds__(X, MINB) k_r2c_tile(const __grid_constant__ KParams p) {
    static_assert(PL::valid() && PL::T == 1 && PL::npass() == 1 && X % 2 == 0, "tile kernel: one thread per row");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using R = float;
    constexpr int M = PL::N, N = 2 * M;
    constexpr int RSI = N + 4;                         // input row stride (floats): N*4 + 16 bytes
    float *smf = reinterpret_cast<float *>(smem_raw);
    float2 *smc = reinterpret_cast<float2 *>(smem_raw);
    const int t = threadIdx.x;
    const long row0 = (long)blockIdx.x * X;
    const int rows = (p.batch - row0 < X) ? (int)(p.batch - row0) : X;
    const float2 *tw = reinterpret_cast<const float2 *>(p.tw);
    const float2 *rtw = reinterpret_cast<const float2 *>(p.rtw);

    {   // stage in: dense [rows][N] reals -> padded rows
        constexpr int CPR = N / 4;
        const float4 *src = reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(p.in0) + row0 * N);
#pragma unroll
        for (int f = t; f < X * CPR; f += X) {
            const int r = f / CPR, c = f % CPR;
            if (r < rows) *reinterpret_cast<float4 *>(smf + r * RSI + 4 * c) = ld_stream(src + f);
        }
    }
    __syncthreads();

    cx<R> x[M];
    {
        const float4 *rowp = reinterpret_cast<const float4 *>(smf + t * RSI);
        static_for<M / 2>([&](auto H_) {
            CIDX(h, H_);
            const float4 v = rowp[h];
            x[2 * h] = mk<R>(v.x, v.y);                // z[j] = x[2j] + i x[2j+1]
            x[2 * h + 1] = mk<R>(v.z, v.w);
        });
    }
    run_pass<R, PL, 0, false>(x, tw, UTw<R, PL>::make(p, tw), 0);
    __syncthreads();                                   // input rows and output rows alias

    {   // Hermitian post-process in registers -> dense output row t ((M+1) float2, odd stride)
        float2 *orow = smc + (size_t)t * (M + 1);
        constexpr int HALF = M / 2;
        const cx<R> z0 = x[slot_of_elem<PL, 0>(0)];
        orow[0] = make_float2(z0.x + z0.y, 0.0f);
        orow[M] = make_float2(z0.x - z0.y, 0.0f);
        const cx<R> zh = x[slot_of_elem<PL, 0>(HALF)];
        const cx<R> xh = RealPost<R>::middle(zh, ld_tw(rtw + HALF), M);
        orow[HALF] = make_float2(xh.x, xh.y);
        static_for<HALF - 1>([&](auto K_) {
            CIDX(k0, K_);
            constexpr int k = k0 + 1;
            const cx<R> z = x[slot_of_elem<PL, 0>(k)], zm = x[slot_of_elem<PL, 0>(M - k)];
            cx<R> xk, xm;
            const twd<R> w = ld_tw(rtw + k);
            RealPost<R>::pair(z, zm, w, w, xk, xm);
            orow[k] = make_float2(xk.x, xk.y);
            orow[M - k] = make_float2(xm.x, xm.y);
        });
    }
    __syncthreads();

    {   // stage out: rows*(M+1) float2, contiguous and 16-byte aligned (X even)
        float2 *dst = reinterpret_cast<float2 *>(p.out0) + row0 * (M + 1);
        const int count = rows * (M + 1);
        const int pairs = count / 2;
        for (int f = t; f < pairs; f += X)
            st_stream(reinterpret_cast<float4 *>(dst) + f, reinterpret_cast<const float4 *>(smc)[f]);
        if ((count & 1) && t == 0) st_stream(dst + (count - 1), smc[count - 1]);
    }
}

template <class PL, int X, int MINB>
__global__ void __launch_bounds__(X, MINB) k_c2r_tile(const __grid_constant__ KParams p) {
    static_assert(PL::valid() && PL::T == 1 && PL::npass() == 1 && X % 2 == 0, "tile kernel: one thread per row");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using R = float;
    constexpr int M = PL::N, N = 2 * M;
    constexpr int RSO = N + 4;                         // output row stride (floats)
    float *smf = reinterpret_cast<float *>(smem_raw);
    float2 *smc = reinterpret_cast<float2 *>(smem_raw);
    const int t = threadIdx.x;
    const long row0 = (long)blockIdx.x * X;
    const int rows = (p.batch - row0 < X) ? (int)(p.batch - row0) : X;
    const float2 *tw = reinterpret_cast<const float2 *>(p.tw);
    const float2 *rtw = reinterpret_cast<const float2 *>(p.rtw);

    {   // stage in: dense [rows][M+1] float2 block
        const float2 *src = reinterpret_cast<const float2 *>(p.in0) + row0 * (M + 1);
        const int count = rows * (M + 1);
        const int pairs = count / 2;
        for (int f = t; f < pairs; f += X)
            reinterpret_cast<float4 *>(smc)[f] = ld_stream(reinterpret_cast<const float4 *>(src) + f);
        if ((count & 1) && t == 0) smc[count - 1] = ld_stream(src + (count - 1));
    }
    __syncthreads();

    cx<R> x[M];
    {   // Hermitian pre-process in registers (scale 0.5/M folded in, :1674)
        const float2 *irow = smc + (size_t)t * (M + 1);
        constexpr int HALF = M / 2;
        const float sc = 0.5f / float(M);
        const float2 a0 = irow[0], am = irow[M];       // real parts only (:1679-1684)
        x[0] = mk<R>((a0.x + am.x) * sc, (a0.x - am.x) * sc);
        static_for<HALF>([&](auto K_) {
            CIDX(k0, K_);
            constexpr int k = k0 + 1;                  // 1 .. M/2 (k = M/2 is self-paired)
            const float2 a = irow[k], b = irow[M - k];
            const twd<R> w = ld_tw(rtw + k);
            const float gr = a.x + b.x, gi = a.y - b.y, ur = a.x - b.x, ui = a.y + b.y;
            const float hr = fmaf(w.y, ui, w.x * ur), hi = fmaf(w.ny, ur, w.x * ui);
            // forward form first, mirrored second: at k = M/2 the mirrored form survives (:1722-1740)
            x[k] = mk<R>(sc * (gr - hi), sc * (gi + hr));
            x[M - k] = mk<R>(sc * (gr + hi), sc * (hr - gi));
        });
    }
    run_pass<R, PL, 0, true>(x, tw, UTw<R, PL>::make(p, tw), 0);
    __syncthreads();                                   // input rows and output rows alias

    {   // time-domain row: z[j] = (x[2j], x[2j+1]); adjacent complex pairs as one STS.128
        float4 *rowp = reinterpret_cast<float4 *>(smf + t * RSO);
        static_for<M>([&](auto S_) {
            CIDX(sa, S_);
            constexpr int ea = out_elem<PL, 0>(sa);
            if constexpr (ea % 2 == 0) {
                constexpr int sb = slot_of_elem<PL, 0>(ea + 1);
                rowp[ea / 2] = make_float4(x[sa].x, x[sa].y, x[sb].x, x[sb].y);
            }
        });
    }
    __syncthreads();

    {   // stage out: dense [rows][N] reals
        constexpr int CPR = N / 4;
        float4 *dst = reinterpret_cast<float4 *>(reinterpret_cast<float *>(p.out0) + row0 * N);
#pragma unroll
        for (int f = t; f < X * CPR; f += X) {
            const int r = f / CPR, c = f % CPR;
            if (r < rows) st_stream(dst + f, *reinterpret_cast<const float4 *>(smf + r * RSO + 4 * c));
        }
    }
}


// ----------------------------------------------------------------------------------------
// Persistent, fully TMA-fed thread-per-row r2c / c2r (N = 64, 128; core M = N/2), the real counterparts of
// k_c2c_tpipe.  The time-domain side uses the grouped, padded rows of k_c2c_tpipe (512-byte bulk copies); the
// spectrum side is the dense [rows][M+1] tile of k_r2c_tile, which is one contiguous block in global memory and
// moves as ONE bulk copy.  Both sides live in the same stage buffer (the thread owns its row in registers in
// between).  Thread <-> row: within every 8G lanes, row = base + G*(lane % 8) + lane / 8, so 8 consecutive lanes
// sit in 8 consecutive groups (LDS.128 on the padded side) and 16 consecutive lanes cover 16 consecutive rows
// (LDS.64 on the dense side, odd row stride): both sides are conflict-free.  A ragged last tile (fewer than X
// rows) moves its spectrum rows with plain loads/stores (bulk copies need 16-byte sizes).
// ----------------------------------------------------------------------------------------
// bytes per bulk copy of the time-domain rows: as in k_c2c_tpipe every copy costs its issuing lane ~9 instructions, so
// wider groups where the mapping allows them (r2c f32 N = 128 power-capped: 0.989 -> 1.017 with 1024 instead of 512;
// the other sizes unchanged within 0.5 %)
#ifndef WFB_RTPIPE_GROUP_BYTES
#define WFB_RTPIPE_GROUP_BYTES 1024
#endif
template <typename R, class PL> __host__ __device__ constexpr int rtpipe_group() {
    const int row_bytes = 2 * (int)sizeof(R) * PL::N;                  // a time-domain row: N = 2M reals
    const int g = row_bytes >= WFB_RTPIPE_GROUP_BYTES ? 1 : WFB_RTPIPE_GROUP_BYTES / row_bytes;
    const int cap = sizeof(R) == 8 ? 8 : 2;                            // the lane <-> row mapping of k_real_tpipe
    return g > cap ? cap : g;
}
template <typename R, class PL, int X> __host__ __device__ constexpr size_t rtpipe_buf_bytes() {
    constexpr int G = rtpipe_group<R, PL>();
    size_t padded = (size_t)(G * 2 * sizeof(R) * PL::N + 16) * (X / G), dense = (size_t)X * (PL::N + 1) * 2 * sizeof(R);
    return ((padded > dense ? padded : dense) + 127) / 128 * 128;
}

template <typename R, class PL, int X, bool C2R, int MINB>
__global__ void __launch_bounds__(X, MINB) k_real_tpipe(const __grid_constant__ KParams p) {
    static_assert(PL::valid() && PL::T == 1 && PL::npass() == 1 && X % 32 == 0, "tile kernel: one thread per row, whole warps");
    static_assert(RT<R>::LANES == 1, "scalar lanes");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using V2 = typename VecOf<R>::v2;                  // one complex value as stored (float2 / double2)
    constexpr int M = PL::N, N = 2 * M, HALF = M / 2;
    constexpr int ES = (int)sizeof(R);
    constexpr int G = rtpipe_group<R, PL>();           // time-domain rows per bulk copy
    static_assert((G <= 2 || (sizeof(R) == 8 && G <= 8)) && X % (8 * G) == 0, "thread <-> row mapping: f32 G = 1, 2; f64 G = 1..8");
    constexpr int ROWT = ES * N;                       // bytes of a time-domain row
    constexpr int GSTR = G * ROWT + 16;                // group stride, bytes (odd multiple of 16)
    constexpr int SPECB = (M + 1) * 2 * ES;            // bytes of a spectrum row
    constexpr size_t BUF = rtpipe_buf_bytes<R, PL, X>();
    uint64_t *mbar = reinterpret_cast<uint64_t *>(smem_raw + 2 * BUF);
    long *slot = reinterpret_cast<long *>(smem_raw + 2 * BUF + 32);
    const int t = threadIdx.x;
    // my row of the tile.  f32 (8-byte bins: 16 lanes per shared-memory phase on the dense side): within 8G lanes,
    // row = G*(lane % 8) + lane / 8.  f64 (16-byte bins: 8 lanes per phase on BOTH sides): the 8 lanes of a phase
    // must sit in 8 distinct groups AND in 8 rows distinct mod 8: lane j of phase ph takes row
    // G*j + (j / (8/G) + ph) mod G of its group -- for G = 2: rows 0,2,4,6,9,11,13,15 / 1,3,5,7,8,10,12,14.
    const int lane8 = t % (8 * G), j8 = lane8 % 8;
    const int myrow = t - lane8 + (ES == 8 ? G * j8 + (j8 / (8 / G) + lane8 / 8) % G : G * j8 + lane8 / 8);
    const long tiles = (p.batch + X - 1) / X;
    const typename RT<R>::twel *tw = reinterpret_cast<const typename RT<R>::twel *>(p.tw);
    const typename RT<R>::twel *rtw = reinterpret_cast<const typename RT<R>::twel *>(p.rtw);
    R *time_g = C2R ? reinterpret_cast<R *>(p.out0) : const_cast<R *>(reinterpret_cast<const R *>(p.in0));
    V2 *spec_g = C2R ? const_cast<V2 *>(reinterpret_cast<const V2 *>(p.in0)) : reinterpret_cast<V2 *>(p.out0);
    auto cta_sync = [&]() { if constexpr (X == 32) __syncwarp(); else __syncthreads(); };
    auto bulk_ok = [&](int rows) { return (rows * SPECB) % 16 == 0; };      // bulk copies move multiples of 16 bytes

    if (t == 0) {
        mbar_init(mbar + 0, 1);
        mbar_init(mbar + 1, 1);
        fence_proxy_async();
    }
    cta_sync();

    auto tile_rows = [&](long tile) { const long row = tile * X; return (p.batch - row < X) ? (int)(p.batch - row) : X; };
    auto issue = [&](long tile, int st) {              // warp 0, all lanes
        const int rows = tile_rows(tile);
        unsigned char *buf = smem_raw + st * BUF;
        bulk_wait_read_all();                          // stores out of this stage have left shared memory ...
        __syncwarp();                                  // ... for every lane of the issuing warp
        if constexpr (!C2R) {
            if (t == 0) mbar_expect_tx(mbar + st, (uint32_t)(rows * ROWT));
            __syncwarp();
            for (int g = t; g * G < rows; g += 32) {
                const int nr = rows - g * G < G ? rows - g * G : G;
                tma_load_1d(buf + (size_t)g * GSTR, time_g + (tile * X + (long)g * G) * N, (uint32_t)(nr * ROWT), mbar + st);
            }
        } else if (bulk_ok(rows)) {                    // otherwise the threads copy the tile (see the main loop)
            if (t == 0) {
                mbar_expect_tx(mbar + st, (uint32_t)(rows * SPECB));
                tma_load_1d(buf, spec_g + tile * X * (M + 1), (uint32_t)(rows * SPECB), mbar + st);
            }
        }
    };

    long pending = claim_prime<true>(p.ctr);
    claim_and_issue<true>(p.ctr, pending, tiles, slot, 0, issue);
    unsigned phasebits = 0;
    cx<R> x[M];
    for (int it = 0;; it++) {
        const int st = it & 1;
        cta_sync();                                    // slot[st] is published; last iteration's stores are issued
        const long tile = slot[st];
        if (tile >= tiles) break;
        unsigned char *buf = smem_raw + st * BUF;
        const int rows = tile_rows(tile);
        V2 *dense = reinterpret_cast<V2 *>(buf);
        V2 *drow = dense + (size_t)myrow * (M + 1);                                       // my spectrum row
        unsigned char *trow = buf + (size_t)(myrow / G) * GSTR + (myrow % G) * ROWT;      // my time row
        if (!C2R || bulk_ok(rows)) {
            mbar_wait(mbar + st, (phasebits >> st) & 1u);
            phasebits ^= 1u << st;
        } else {
            const V2 *src = spec_g + tile * X * (M + 1);
            for (int f = t; f < rows * (M + 1); f += X) dense[f] = ld_stream(src + f);
            cta_sync();
        }

        if constexpr (!C2R) {
            if constexpr (ES == 8) {                   // z[j] = x[2j] + i x[2j+1]: one LDS.128 per complex value
                const double2 *tr = reinterpret_cast<const double2 *>(trow);
                static_for<M>([&](auto H_) { CIDX(h, H_); const double2 v = tr[h]; x[h] = mk<R>(v.x, v.y); });
            } else {
                const float4 *tr = reinterpret_cast<const float4 *>(trow);
                static_for<M / 2>([&](auto H_) {
                    CIDX(h, H_);
                    const float4 v = tr[h];
                    x[2 * h] = mk<R>(v.x, v.y);
                    x[2 * h + 1] = mk<R>(v.z, v.w);
                });
            }
            claim_and_issue<true>(p.ctr, pending, tiles, slot, st ^ 1, issue);
            run_pass<R, PL, 0, false>(x, tw, UTw<R, PL>::make(p, tw), 0);
            cta_sync();                                // time rows and spectrum rows alias
            auto put = [&](int k, cx<R> v) { V2 o; o.x = v.x; o.y = v.y; drow[k] = o; };
            const cx<R> z0 = x[slot_of_elem<PL, 0>(0)];
            put(0, mk<R>(radd(z0.x, z0.y), R(0)));
            put(M, mk<R>(rsub(z0.x, z0.y), R(0)));
            put(HALF, RealPost<R>::middle(x[slot_of_elem<PL, 0>(HALF)], ld_tw(rtw + HALF), M));
            static_for<HALF - 1>([&](auto K_) {
                CIDX(k0, K_);
                constexpr int k = k0 + 1;
                const cx<R> z = x[slot_of_elem<PL, 0>(k)], zm = x[slot_of_elem<PL, 0>(M - k)];
                cx<R> xk, xm;
                const twd<R> wk = ld_tw(rtw + k);
                RealPost<R>::pair(z, zm, wk, ld_tw_mirror<R>(rtw, k, M, wk), xk, xm);     // (f32 ignores the second entry)
                put(k, xk);
                put(M - k, xm);
            });
            if (bulk_ok(rows)) {
                fence_proxy_async();
                cta_sync();
                if (t == 0) { tma_store_1d(spec_g + tile * X * (M + 1), buf, (uint32_t)(rows * SPECB)); bulk_commit(); }
            } else {
                cta_sync();
                V2 *dst = spec_g + tile * X * (M + 1);
                for (int f = t; f < rows * (M + 1); f += X) st_stream(dst + f, dense[f]);
            }
        } else {
            {   // Hermitian pre-process in registers (scale 0.5/M folded in, :1674)
                const R sc = R(0.5) / R(M);
                const V2 a0 = drow[0], am = drow[M];          // real parts only (:1679-1684)
                x[0] = mk<R>(rmul(radd(a0.x, am.x), sc), rmul(rsub(a0.x, am.x), sc));
                static_for<HALF>([&](auto K_) {
                    CIDX(k0, K_);
                    constexpr int k = k0 + 1;                 // 1 .. M/2 (k = M/2 is self-paired)
                    const V2 a = drow[k], b = drow[M - k];
                    const twd<R> w = ld_tw(rtw + k);
                    const R gr = radd(a.x, b.x), gi = rsub(a.y, b.y), ur = rsub(a.x, b.x), ui = radd(a.y, b.y);
                    const R hr = rfma(w.y, ui, rmul(w.x, ur)), hi = rfma(w.ny, ur, rmul(w.x, ui));
                    // forward form first, mirrored second: at k = M/2 the mirrored form survives (:1722-1740)
                    x[k] = mk<R>(rmul(sc, rsub(gr, hi)), rmul(sc, radd(gi, hr)));
                    x[M - k] = mk<R>(rmul(sc, radd(gr, hi)), rmul(sc, rsub(hr, gi)));
                });
            }
            claim_and_issue<true>(p.ctr, pending, tiles, slot, st ^ 1, issue);
            run_pass<R, PL, 0, true>(x, tw, UTw<R, PL>::make(p, tw), 0);
            cta_sync();                                // spectrum rows and time rows alias
            if constexpr (ES == 8) {
                double2 *tr = reinterpret_cast<double2 *>(trow);
                static_for<M>([&](auto H_) { CIDX(h, H_); constexpr int s0 = slot_of_elem<PL, 0>(h); tr[h] = make_double2(x[s0].x, x[s0].y); });
            } else {
                float4 *tr = reinterpret_cast<float4 *>(trow);
                static_for<M / 2>([&](auto H_) {
                    CIDX(h, H_);
                    constexpr int s0 = slot_of_elem<PL, 0>(2 * h), s1 = slot_of_elem<PL, 0>(2 * h + 1);
                    tr[h] = make_float4(x[s0].x, x[s0].y, x[s1].x, x[s1].y);
                });
            }
            fence_proxy_async();
            cta_sync();
            if (t < 32) {
                for (int g = t; g * G < rows; g += 32) {
                    const int nr = rows - g * G < G ? rows - g * G : G;
                    tma_store_1d(time_g + (tile * X + (long)g * G) * N, buf + (size_t)g * GSTR, (uint32_t)(nr * ROWT));
                }
                bulk_commit();
            }
        }
    }
    if (t < 32) bulk_wait_read_all();                  // shared memory must outlive the stores that read it
    claim_epilogue(p.ctr);
}


// Hermitian step, shared-memory half: park the upper half of the core's outputs (elements >= M/2) at the UNPADDED
// index M - k', i.e. at the bin index of the thread that pairs it with its own register value Z[k] (see k_real_pipe).
template <typename R, class PL, int LAST>
__device__ __forceinline__ void park_upper_half(const cx<R> (&x)[PL::E], cx<R> *park, int tid) {
    static_for<PL::E>([&](auto S_) {
        CIDX(slot, S_);
        constexpr int e = out_elem<PL, LAST>(slot);
        if constexpr (e >= PL::E / 2) park[PL::N - e * PL::T - tid] = x[slot];
    });
}

// ----------------------------------------------------------------------------------------
// Batched STFT front-end (SURVEY 8f-1): the reference's only batched caller is the spectrogram loop
// of playground/src/spectrogram.js:281-360 -- per frame: slice `window` samples at `frame*hop`,
// multiply by the window function, zero-pad to the FFT size, r2c, then |X| -> dB -> [0,1].
// Here the frame gather + window multiply + zero padding are fused into the r2c load stage and the
// magnitude/dB/normalise step into its store stage, so a spectrogram is ONE kernel: the overlapping
// frames are read once from HBM (L2 serves the overlap) and only (N/2+1) floats per frame are written.
// PL describes the M = N/2 point complex core, exactly as in k_r2c.
// ----------------------------------------------------------------------------------------
struct StftParams {
    const float *samples;      // [batch][num_samples]
    const float *window;       // [wsize] window function values (f32), host-built
    void *out;                 // MODE_DB: float [batch][frames][M+1];  MODE_COMPLEX: float2 [batch][frames][M+1]
    const void *tw, *rtw;      // stage tables / W_N^k of the r2c core
    long frames;               // per signal: no frame reads samples of another signal
    long batch, num_samples;   // signals, and the sample stride between them
    long tiles;                // persistent kernels: tiles of X frames in all, tps per signal: tile t = (t / tps, t % tps)
    unsigned tps, tps_magic;   // t / tps = (umulhi(t, tps_magic) + t) >> tps_shift for t < 2^31 (stft_tile_signal)
    int tps_shift;
    int hop, wsize, mode;
    float db_floor;            // gain - range
    float inv_range;           // 1 / range
    float inv_half_n;          // 1 / (N/2)
    unsigned long long *ctr;   // pipelined kernel: zeroed tile counter of this launch
    float lg_a, lg_b;          // fast dB path: value = lg_a * log2(|2 X|^2) + lg_b (host-folded constants)
    int aligned8;              // every signal's `samples` row is 8-byte aligned: even hops may use 64-bit loads
    int span_bytes;            // span kernel: shared-memory bytes of one span stage (multiple of 128)
    // MODE_FILTERBANK: out is float [batch][frames][fb_n], out = L(sum_k F[m][k] |X[k]|^fb_power), F band-sparse:
    const int4 *fb_band;       // per filter {first bin, bins, offset into fb_w, 0}; an all-zero filter has 0 bins
    const float *fb_w;         // the bands' weights, packed
    int fb_n, fb_power;        // filters (1 <= fb_n <= M+1); 1 (|X|) or 2 (|X|^2)
    float fb_scale, fb_offset, fb_floor;   // L(v) = v if fb_scale == 0, else fb_scale log2(max(v + fb_offset, fb_floor))
};
enum { STFT_MODE_DB = 0, STFT_MODE_COMPLEX = 1, STFT_MODE_FILTERBANK = 2 };
// tile -> (signal, tile within the signal) without a division.  Tiles stay below 2^31: each writes at least one row of
// N/2 + 1 >= 33 floats, and 2^31 such rows are more than device memory holds.
inline void stft_tile_magic(StftParams &sp) {
    int l = 0;
    while ((1ull << l) < sp.tps) l++;
    sp.tps_magic = (unsigned)((((1ull << l) - sp.tps) << 32) / sp.tps + 1);      // round-up reciprocal (Granlund-Montgomery)
    sp.tps_shift = l;
}
__device__ __forceinline__ unsigned stft_tile_signal(long tile, const StftParams &sp) {
    const unsigned t = (unsigned)tile;
    return (__umulhi(t, sp.tps_magic) + t) >> sp.tps_shift;
}
// kernel flavours (template parameter KM): the dB output has a fast path that needs no square root and folds every
// constant of computeMagnitude / magnitudeToDb / the gain-range normalisation into one FFMA after the MUFU.LG2:
//   10 log10(|X|^2 c^2) = 20 log10(|X| c + 1e-10) - 20 log10(1 + 1e-10 / (|X| c)): below by 1e-6 dB at -61 dB, 8.7e-5 dB
//   at -100 dB and ten times more per 20 dB deeper.  Everything below the floor (gain - range) clamps to 0 either way, so the error
//   that counts is the one at the floor; stft_flavour takes the fast form only where it is at most 1e-6 of the
//   normalised output there, and the exact form below that.
// STFT_K_FB (filterbank) writes the per-bin power |X|^p, takes the filter product over it and stores fb_n values per frame.
enum { STFT_K_FAST = 0, STFT_K_EXACT = 1, STFT_K_COMPLEX = 2, STFT_K_FB = 3 };
template <int KM> using stft_value_t = typename std::conditional<KM == STFT_K_COMPLEX, float2, float>::type;   // one output bin

__device__ __forceinline__ float stft_db(float re, float im, const StftParams &sp) {
    // computeMagnitude + magnitudeToDb + normalisation (spectrogram.js:78-96, :343-352)
    // 20*log10(v) = 6.0206*log2(v): one MUFU.LG2 instead of the ~25-instruction log10f (|error| < 1e-5 dB)
    const float mag = sqrtf(re * re + im * im);
    const float db = 6.0205999132796239f * __log2f(mag * sp.inv_half_n + 1e-10f);
    const float v = (db - sp.db_floor) * sp.inv_range;
    return fminf(1.0f, fmaxf(0.0f, v));
}
// fast path on the UNHALVED bin value 2 X[k] (the 1/2 of the Hermitian step is folded into lg_b as well)
__device__ __forceinline__ float stft_db_fast(cx<float> x2, const StftParams &sp) {
    const float v = fmaf(__log2f(fmaf(x2.x, x2.x, x2.y * x2.y)), sp.lg_a, sp.lg_b);   // log2(0) = -inf clamps to 0
    return fminf(1.0f, fmaxf(0.0f, v));
}

// Hermitian post-process + output conversion shared by the STFT kernels.  `park` holds the upper half of the core's
// outputs (park_upper_half); Z[k] for k < M/2 is the thread's own register value.  Each output value v goes to
// out(i, s, bin, v), i = the compile-time block of bin k = tid + i*T:  s = 0: bin k,  s = 1: bin M - k,  s = 2: bin M/2
// (thread 0, i = 0 only, where bins k and M - k are 0 and M).  V is float (dB flavours) or float2 (complex).
template <class PL, int LAST, int KM, class Out>
__device__ __forceinline__ void stft_values(const cx<float> (&x)[PL::E], const cx<float> *park, const float2 *rtw, int tid,
                                            const StftParams &sp, Out &&out) {
    using R = float;
    using V = stft_value_t<KM>;
    constexpr int M = PL::N, HALF = M / 2, PER = PL::E / 2;
    static_assert(PER * PL::T == HALF, "bins per thread");
    auto conv = [&](int k, cx<R> v) -> V {                               // exact forms (and the three special bins)
        if constexpr (KM == STFT_K_COMPLEX) return make_float2(v.x, v.y);
        else if constexpr (KM == STFT_K_FB) {                            // |X|^2 or |X|; no bin is zeroed
            const float p = fmaf(v.x, v.x, v.y * v.y);
            return sp.fb_power == 2 ? p : sqrtf(p);
        }
        else return k < 3 ? 0.0f : stft_db(v.x, v.y, sp);               // DC and near-DC bins zeroed (:338-342)
    };
    static_for<PER>([&](auto I_) {
        CIDX(i, I_);
        const int k = tid + i * PL::T;
        const cx<R> z = x[slot_of_elem<PL, LAST>(i)];                   // Z[k]: this thread's own output
        if (i == 0 && k == 0) {
            out(I_, 0, 0, conv(0, mk<R>(z.x + z.y, 0.0f)));
            out(I_, 1, M, conv(M, mk<R>(z.x - z.y, 0.0f)));
            out(I_, 2, HALF, conv(HALF, RealPost<R>::middle(park[HALF], ld_tw(rtw + HALF), M)));
        } else {
            const cx<R> zm = park[k];
            const twd<R> w = ld_tw(rtw + k);
            if constexpr (KM == STFT_K_FAST) {
                // 2 X[k] and 2 X[M-k]: RealPost::pair without its four multiplications by 1/2
                const R gr = z.x + zm.x, gi = z.y - zm.y, hr = z.y + zm.y, hi = zm.x - z.x;
                const R tr = fmaf(w.ny, hi, w.x * hr), ti = fmaf(w.y, hr, w.x * hi);
                float vk = stft_db_fast(mk<R>(gr + tr, gi + ti), sp);
                const float vm = stft_db_fast(mk<R>(gr - tr, ti - gi), sp);
                if constexpr (i * PL::T < 3) vk = k < 3 ? 0.0f : vk;    // only the first block(s) hold bins below 3
                out(I_, 0, k, vk);
                out(I_, 1, M - k, vm);
            } else {
                cx<R> xk, xm;
                RealPost<R>::pair(z, zm, w, w, xk, xm);
                out(I_, 0, k, conv(k, xk));
                out(I_, 1, M - k, conv(M - k, xm));
            }
        }
    });
}

// Filterbank stage (STFT_K_FB).  The per-bin powers of a frame arrive in registers from stft_values; the group writes them
// as one row of M+1 floats to shared memory and, after a group barrier, each thread computes filters m = tid, tid + T, ...:
// one f32 FMA chain over the filter's band in increasing bin order, then L.  The same arithmetic on every route, so results
// are bitwise repeatable and a batch row equals its single-signal run.
template <class PL, int LAST> struct StftFbValues {
    static constexpr int PER = PL::E / 2;
    float vk[PER], vm[PER], vh = 0.0f;
    __device__ __forceinline__ void take(const cx<float> (&x)[PL::E], const cx<float> *park, const float2 *rtw, int tid,
                                         const StftParams &sp) {
        stft_values<PL, LAST, STFT_K_FB>(x, park, rtw, tid, sp, [&](auto I_, int s, int, float v) {
            CIDX(i, I_);
            (s == 0 ? vk[i] : s == 1 ? vm[i] : vh) = v;
        });
    }
    __device__ __forceinline__ void to_row(float *row, int tid) const {
        static_for<PER>([&](auto I_) {
            CIDX(i, I_);
            const int k = tid + i * PL::T;
            row[k] = vk[i];
            row[PL::N - k] = vm[i];
            if (i == 0 && k == 0) row[PL::N / 2] = vh;
        });
    }
};
__device__ __forceinline__ float stft_fb_log(float v, const StftParams &sp) {
    return sp.fb_scale == 0.0f ? v : sp.fb_scale * __log2f(fmaxf(v + sp.fb_offset, sp.fb_floor));
}
// filters m = tid, tid + T, ...: one f32 FMA chain over the band in increasing bin order (float4 loads of weights and
// powers, and a snake order of filters over threads, were measured slower or no faster: DESIGN §8)
template <int T, class Out>
__device__ __forceinline__ void stft_fb_filters(const float *row, int tid, const StftParams &sp, Out &&out) {
    for (int m = tid; m < sp.fb_n; m += T) {
        const int4 b = __ldg(sp.fb_band + m);
        const float *w = sp.fb_w + b.z;
        const float *p = row + b.x;
        float acc = 0.0f;
        for (int j = 0; j < b.y; j++) acc = fmaf(__ldg(w + j), p[j], acc);
        out(m, stft_fb_log(acc, sp));
    }
}
// direct and pipe kernels: `scratch` is the group's scratch row holding the parked upper half; the results leave from
// registers.  Every group takes both barriers (groups narrower than a warp share one); only an active one stores.
template <class PL, int LAST, int X>
__device__ __forceinline__ void stft_fb_frame(const cx<float> (&x)[PL::E], cx<float> *scratch, const float2 *rtw, int tid, int xi,
                                              const StftParams &sp, long frame, bool active) {
    StftFbValues<PL, LAST> v;
    v.take(x, scratch, rtw, tid, sp);
    sync_transform<PL::T, X>(xi);                                        // the group has read its parked half
    float *row = reinterpret_cast<float *>(scratch);
    v.to_row(row, tid);
    sync_transform<PL::T, X>(xi);
    if (!active) return;
    float *orow = reinterpret_cast<float *>(sp.out) + frame * sp.fb_n;
    stft_fb_filters<PL::T>(row, tid, sp, [&](int m, float o) { st_stream(orow + m, o); });
}

// KM: output flavour (STFT_K_*); PAD: window shorter than the FFT size (zero padding)
template <class PL, int X, int PADQ, int MINB, int KM, bool PAD>
__global__ void __launch_bounds__(PL::T *X, MINB) k_stft(const __grid_constant__ StftParams sp) {
    static_assert(PL::valid(), "plan does not factor N");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using R = float;
    constexpr int M = PL::N;
    constexpr int LAST = PL::npass() - 1;
    const int xi = threadIdx.x / PL::T, tid = threadIdx.x % PL::T;
    const long frame = (long)blockIdx.x * X + xi;                       // output row: frame f of signal sig
    const bool active = frame < sp.frames * sp.batch;
    const long sig = frame / sp.frames, f = frame - sig * sp.frames;
    cx<R> *sm = reinterpret_cast<cx<R> *>(smem_raw) + (size_t)xi * padded_size<PADQ>(M);
    const float2 *tw = reinterpret_cast<const float2 *>(sp.tw);
    const float2 *rtw = reinterpret_cast<const float2 *>(sp.rtw);
    cx<R> x[PL::E];

    {   // gather + window + zero-pad: z[p] = (s[off+2p] w[2p], s[off+2p+1] w[2p+1])
        const float *s = sp.samples + (active ? sig * sp.num_samples + f * (long)sp.hop : 0);
        const bool vec = sp.aligned8 && ((sp.hop | sp.wsize) & 1) == 0;    // aligned base, even hop: frame starts are 8-byte aligned
        static_for<PL::E>([&](auto E_) {
            CIDX(e, E_);
            const int i0 = 2 * (tid + e * PL::T);
            float a = 0.0f, b = 0.0f;
            if (vec) {
                if (!PAD || i0 < sp.wsize) {           // (an inactive group reads frame 0 and stores nothing)
                    const float2 v = __ldg(reinterpret_cast<const float2 *>(s + i0));
                    const float2 w = __ldg(reinterpret_cast<const float2 *>(sp.window + i0));
                    a = v.x * w.x; b = v.y * w.y;
                }
            } else {
                if (active && i0 < sp.wsize) a = __ldg(s + i0) * __ldg(sp.window + i0);
                if (active && i0 + 1 < sp.wsize) b = __ldg(s + i0 + 1) * __ldg(sp.window + i0 + 1);
            }
            x[e] = mk<R>(a, b);
        });
    }
    run_all<R, PL, PADQ, X, false>(x, tw, GTw<R>{nullptr, tw}, sm, tid, xi, false);
    if (PL::npass() > 1) sync_transform<PL::T, X>(xi);
    park_upper_half<R, PL, LAST>(x, sm, tid);
    sync_transform<PL::T, X>(xi);
    if constexpr (KM == STFT_K_FB) {
        stft_fb_frame<PL, LAST, X>(x, sm, rtw, tid, xi, sp, frame, active);
        return;
    }
    if (!active) return;

    using V = stft_value_t<KM>;
    V *orow = reinterpret_cast<V *>(sp.out) + frame * (M + 1);
    stft_values<PL, LAST, KM>(x, sm, rtw, tid, sp, [&](auto, int, int bin, V v) { st_stream(orow + bin, v); });
}


// TMA-pipelined STFT: frames are rows at `hop` stride in the sample array, so when hop is a
// multiple of 4 samples (16-byte aligned frame starts) each frame is one bulk copy into a padded
// smem row, prefetched one tile ahead exactly like k_real_pipe's row-copy mode.
template <class PL, int X, int PADQ, int MINB, int KM, bool PAD>
__global__ void __launch_bounds__(PL::T *X, MINB) k_stft_pipe(const __grid_constant__ StftParams sp) {
    static_assert(PL::valid() && PL::T * X >= 32, "needs a full issuing warp");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using R = float;
    constexpr int M = PL::N;
    constexpr int LAST = PL::npass() - 1;
    constexpr int RSTR = M + M / 16;                   // smem row stride (float2): rows T banks apart
    static_assert(RSTR <= padded_size<PADQ>(M), "the padded frame rows must fit the stage buffer (sized for the scratch)");
    constexpr size_t BUF = real_pipe_buf_bytes<R, PL, PADQ, X, false>();
    uint64_t *mbar = reinterpret_cast<uint64_t *>(smem_raw + 2 * BUF);
    const int xi = threadIdx.x / PL::T, tid = threadIdx.x % PL::T;
    const float2 *tw = reinterpret_cast<const float2 *>(sp.tw);
    const float2 *rtw = reinterpret_cast<const float2 *>(sp.rtw);
    const long tiles = sp.tiles;

    if (threadIdx.x == 0) {
        mbar_init(mbar + 0, 1);
        mbar_init(mbar + 1, 1);
        fence_proxy_async();
    }
    __syncthreads();

    auto issue = [&](long tile, int st) {
        if (threadIdx.x < 32) {
            const unsigned sig = stft_tile_signal(tile, sp);
            const long f0 = (long)((unsigned)tile - sig * sp.tps) * X;
            const int rows = (sp.frames - f0 < X) ? (int)(sp.frames - f0) : X;
            const uint32_t rowb = (uint32_t)(sp.wsize * sizeof(float));
            const float *s = sp.samples + (long)sig * sp.num_samples;
            if (threadIdx.x == 0) mbar_expect_tx(mbar + st, rows * rowb);
            __syncwarp();
            for (int r = threadIdx.x; r < rows; r += 32)
                tma_load_1d(smem_raw + st * BUF + (size_t)r * RSTR * sizeof(float2), s + (f0 + r) * (long)sp.hop, rowb, mbar + st);
        }
    };

    long *slot = reinterpret_cast<long *>(smem_raw + 2 * BUF + 32);   // tile claimed for each stage
    long pending = claim_prime<false>(sp.ctr);
    claim_and_issue<false>(sp.ctr, pending, tiles, slot, 0, issue);
    cx<R> x[PL::E];
    const float2 *win = reinterpret_cast<const float2 *>(sp.window);
    for (int it = 0;; it++) {
        const int st = it & 1;
        fence_proxy_async();
        __syncthreads();
        const long tile = slot[st];
        if (tile >= tiles) break;
        claim_and_issue<false>(sp.ctr, pending, tiles, slot, st ^ 1, issue);
        mbar_wait(mbar + st, (it >> 1) & 1);
        unsigned char *buf = smem_raw + st * BUF;
        const unsigned sig = stft_tile_signal(tile, sp);
        const long f = (long)((unsigned)tile - sig * sp.tps) * X + xi;
        const bool active = f < sp.frames;
        const long frame = (long)sig * sp.frames + f;                   // output row
        cx<R> *scratch = reinterpret_cast<cx<R> *>(buf) + (size_t)xi * padded_size<PADQ>(M);
        const float2 *raw = reinterpret_cast<const float2 *>(buf) + (size_t)xi * RSTR;

        static_for<PL::E>([&](auto E_) {               // window multiply + zero padding on the way to registers
            CIDX(e, E_);
            const int pidx = tid + e * PL::T;
            float a = 0.0f, b = 0.0f;
            if (!PAD || 2 * pidx < sp.wsize) {         // (rows beyond the last frame hold stale data and store nothing)
                const float2 v = raw[pidx], w = __ldg(win + pidx);
                a = v.x * w.x; b = v.y * w.y;
            }
            x[e] = mk<R>(a, b);
        });
        __syncthreads();                               // raw rows and padded scratch alias
        run_all<R, PL, PADQ, X, false>(x, tw, GTw<R>{nullptr, tw}, scratch, tid, xi, false);
        if (PL::npass() > 1) sync_transform<PL::T, X>(xi);
        park_upper_half<R, PL, LAST>(x, scratch, tid);
        sync_transform<PL::T, X>(xi);
        if constexpr (KM == STFT_K_FB) stft_fb_frame<PL, LAST, X>(x, scratch, rtw, tid, xi, sp, frame, active);
        else if (active) {
            using V = stft_value_t<KM>;
            V *orow = reinterpret_cast<V *>(sp.out) + frame * (M + 1);
            stft_values<PL, LAST, KM>(x, scratch, rtw, tid, sp, [&](auto, int, int bin, V v) { st_stream(orow + bin, v); });
        }
    }
    claim_epilogue(sp.ctr);
}


// ----------------------------------------------------------------------------------------
// Span-staged persistent STFT (the default when hop and window are multiples of 4 samples).
//   * The X frames of a tile overlap, so their samples are ONE contiguous span of (X-1)*hop + window floats: it arrives
//     as ONE bulk copy (prefetched while the previous tile is computed) and every frame is formed out of shared memory.  The
//     direct kernel above re-loads every sample window/hop times through the L1 data pipe, its top-utilised unit.
//   * The window function sits in shared memory for the whole kernel (the direct kernel re-loads it from global memory
//     for every frame, through the tagged L1 path).
//   * The dB (or complex) rows of a tile are contiguous in the output: they are assembled in shared memory and leave as
//     one bulk store.  Rows are (M+1) floats, so a tile starts at any multiple of 4 bytes: the tile is assembled at the
//     same 16-byte phase as its destination, the aligned interior goes out as a bulk store and the <= 3 floats at either
//     end as plain stores.
// Shared memory: [work: X padded scratch rows, reused for the result tile][span][mbarrier, slots][window].
// ----------------------------------------------------------------------------------------
template <class PL, int PADQ, int X> __host__ __device__ constexpr size_t stft_work_bytes() {
    size_t a = sizeof(cx<float>) * (size_t)padded_size<PADQ>(PL::N) * X + 16;      // + the output phase offset
    size_t b = sizeof(float) * 2 * (size_t)(PL::N + 1) * X + 16;                   // complex result tile
    return ((a > b ? a : b) + 127) / 128 * 128;
}

template <class PL, int X, int PADQ, int MINB, int KM, bool PAD>
__global__ void __launch_bounds__(PL::T *X, MINB) k_stft_span(const __grid_constant__ StftParams sp) {
    static_assert(PL::valid() && PL::T * X >= 32, "needs a full issuing warp");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    using R = float;
    using V = stft_value_t<KM>;
    constexpr int M = PL::N, T = PL::T, E = PL::E, PER = E / 2, HALF = M / 2;
    constexpr int LAST = PL::npass() - 1;
    constexpr size_t WORK = stft_work_bytes<PL, PADQ, X>();
    const uint32_t span_cap = (uint32_t)sp.span_bytes;                   // bytes of the span buffer (multiple of 128)
    unsigned char *work = smem_raw;
    unsigned char *span = smem_raw + WORK;
    uint64_t *mbar = reinterpret_cast<uint64_t *>(smem_raw + WORK + (size_t)span_cap);
    long *slot = reinterpret_cast<long *>(mbar + 4);
    const int xi = threadIdx.x / T, tid = threadIdx.x % T;
    const float2 *tw = reinterpret_cast<const float2 *>(sp.tw);
    const float2 *rtw = reinterpret_cast<const float2 *>(sp.rtw);
    const long tiles = sp.tiles;
    constexpr int VW = (int)(sizeof(V) / sizeof(float));                 // floats per output bin
    float *gout = reinterpret_cast<float *>(sp.out);

    if (threadIdx.x == 0) {
        mbar_init(mbar, 1);
        fence_proxy_async();
    }
    // the window function, once per CTA, in shared memory behind the span stages (zero beyond the window): the frames are
    // formed with two conflict-free LDS.64 per value pair.  (Holding each thread's window values in registers for the whole
    // kernel was measured first: 64 more registers on the 32-value plans, 8 warps per SM, 8 % slower than the direct kernel.)
    float2 *winsm = reinterpret_cast<float2 *>(smem_raw + WORK + (size_t)span_cap + 128);
    {
        const float2 *w2 = reinterpret_cast<const float2 *>(sp.window);
        for (int pidx = threadIdx.x; pidx < M; pidx += T * X)
            winsm[pidx] = (!PAD || 2 * pidx < sp.wsize) ? __ldg(w2 + pidx) : make_float2(0.0f, 0.0f);
    }
    __syncthreads();

    // a tile's place, worked out once by the issuing thread and kept per stage in shared memory (not in registers, which
    // the 32-value plans have none to spare for): {first output row, first frame within its signal}
    long *geom = slot + 2;
    auto tile_rows = [&](long f0) { return (sp.frames - f0 < X) ? (int)(sp.frames - f0) : X; };
    // ONE span buffer: a tile's samples are consumed (into registers) at the very start of its iteration, so the next
    // tile's span is fetched into the same bytes while this tile is computed.  A span ends at its signal's last frame.
    auto issue = [&](long tile, int st) {
        if (threadIdx.x == 0) {
            const unsigned sig = stft_tile_signal(tile, sp);
            const unsigned f0 = ((unsigned)tile - sig * sp.tps) * X;     // (frames of one signal are far below 2^31)
            geom[2 * st] = (long)sig * sp.frames + f0;
            geom[2 * st + 1] = f0;
            const uint32_t bytes = (uint32_t)((tile_rows(f0) - 1) * sp.hop + sp.wsize) * sizeof(float);
            mbar_expect_tx(mbar, bytes);
            tma_load_1d(span, sp.samples + (long)sig * sp.num_samples + (long)f0 * sp.hop, bytes, mbar);
        }
    };
    // the result tile of stage `st` sits in `work` at the 16-byte phase of its destination
    // floats per output row: M+1 bins of VW floats, or one per filter
    auto row_floats = [&]() -> int { if constexpr (KM == STFT_K_FB) return sp.fb_n; else return (M + 1) * VW; };
    auto out_phase = [&](int st) { return (int)((geom[2 * st] * (long)row_floats()) & 3); };      // in floats
    auto store_tile = [&](int st) {
        if (threadIdx.x >= 32) return;
        const long o0 = geom[2 * st] * (long)row_floats();               // first float of the tile in the output
        const int total = tile_rows(geom[2 * st + 1]) * row_floats(), ph = out_phase(st);
        int head = (4 - ph) & 3;                                         // floats up to the next 16-byte boundary
        if constexpr (KM == STFT_K_FB) head = min(head, total);          // (rows of 1-3 filters: a tile may be shorter)
        const int interior = (total - head) & ~3;
        const float *src = reinterpret_cast<const float *>(work) + ph;
        if (threadIdx.x == 0 && interior > 0) {
            tma_store_1d(gout + o0 + head, src + head, (uint32_t)(interior * sizeof(float)));
            bulk_commit();
        }
        if ((int)threadIdx.x < head) st_stream(gout + o0 + threadIdx.x, src[threadIdx.x]);
        const int tail0 = head + interior;
        if ((int)threadIdx.x < total - tail0) st_stream(gout + o0 + tail0 + threadIdx.x, src[tail0 + threadIdx.x]);
    };

    long pending = claim_prime<false>(sp.ctr);
    claim_and_issue<false>(sp.ctr, pending, tiles, slot, 0, issue);
    cx<R> x[E];
    unsigned phasebits = 0;
    for (int it = 0;; it++) {
        const int st = it & 1;
        fence_proxy_async();       // the result tile written below (generic proxy) precedes its bulk store
        __syncthreads();           // slot[st] is published; the result tile of the last iteration is complete
        if (it > 0) store_tile(st ^ 1);                                  // (before the next claim rewrites its geometry)
        const long tile = slot[st];
        if (tile >= tiles) break;
        mbar_wait(mbar, phasebits);
        phasebits ^= 1u;
        // hop is a multiple of 4 samples: every frame starts on a 16-byte boundary of the span
        const float2 *raw = reinterpret_cast<const float2 *>(span) + (size_t)xi * (sp.hop >> 1);
        static_for<E>([&](auto E_) {
            CIDX(e, E_);
            const int pidx = tid + e * T;
            float2 v = make_float2(0.0f, 0.0f);
            if (!PAD || 2 * pidx < sp.wsize) v = raw[pidx];              // (frames past the last one read stale data and are dropped)
            const float2 w = winsm[pidx];
            x[e] = mk<R>(v.x * w.x, v.y * w.y);
        });
        if (threadIdx.x == 0) bulk_wait_read_all();                     // the last result tile has left `work` ...
        fence_proxy_async();                                             // (our reads of the span precede its refill by the copy engine)
        __syncthreads();                                                 // ... before anyone uses it as scratch; all span reads done
        claim_and_issue<false>(sp.ctr, pending, tiles, slot, st ^ 1, issue);   // next tile's span, while this tile is computed
        cx<R> *scratch = reinterpret_cast<cx<R> *>(work) + (size_t)xi * padded_size<PADQ>(M);
        run_all<R, PL, PADQ, X, false>(x, tw, GTw<R>{nullptr, tw}, scratch, tid, xi, false);
        if (PL::npass() > 1) sync_transform<T, X>(xi);
        park_upper_half<R, PL, LAST>(x, scratch, tid);
        sync_transform<T, X>(xi);
        if constexpr (KM == STFT_K_FB) {
            // result tile: X rows of fb_n floats at the output's phase; each group's power row of M+1 floats behind it
            // (fb_n <= M+1, so both fit the complex tile's bytes)
            StftFbValues<PL, LAST> v;
            v.take(x, scratch, rtw, tid, sp);
            __syncthreads();                                             // every group has read its parked half
            float *row = reinterpret_cast<float *>(work) + 4 + (size_t)X * sp.fb_n + (size_t)xi * (M + 1);
            v.to_row(row, tid);
            sync_transform<T, X>(xi);
            if (geom[2 * st + 1] + xi < sp.frames) {
                float *orow = reinterpret_cast<float *>(work) + out_phase(st) + (size_t)xi * sp.fb_n;
                stft_fb_filters<T>(row, tid, sp, [&](int m, float o) { orow[m] = o; });
            }
            continue;
        }
        V vk[PER], vm[PER], vh = V();
        stft_values<PL, LAST, KM>(x, scratch, rtw, tid, sp, [&](auto I_, int s, int, V v) {
            CIDX(i, I_);
            (s == 0 ? vk[i] : s == 1 ? vm[i] : vh) = v;
        });
        __syncthreads();                                                 // every group has read its parked half: `work` becomes the result tile
        if (geom[2 * st + 1] + xi < sp.frames) {                         // (frames of the tile's signal)
            V *orow = reinterpret_cast<V *>(reinterpret_cast<float *>(work) + out_phase(st)) + (size_t)xi * (M + 1);
            static_for<PER>([&](auto I_) {
                CIDX(i, I_);
                const int k = tid + i * T;
                orow[k] = vk[i];
                orow[M - k] = vm[i];
                if (i == 0 && k == 0) orow[HALF] = vh;
            });
        }
    }
    if (threadIdx.x == 0) bulk_wait_read_all();                         // shared memory must outlive the store that reads it
    claim_epilogue(sp.ctr);
}

// ----------------------------------------------------------------------------------------
// Inverse STFT (extension, no reference counterpart): the weighted overlap-add / least-squares estimate of a signal from
// the complex spectra the STFT_MODE_COMPLEX kernels write,
//   y_f = c2r(X_f) (1/N, real parts of DC and Nyquist),   x[t] = sum_f w[t-fH] y_f[t-fH] / sum_f w[t-fH]^2
// (0 where the denominator is below 1e-11, i.e. where no frame carries weight), in ONE kernel: c2r pre-process, inverse
// core, window multiply and overlap-add fused, every spectrum read once and every sample written once.
//   * A CTA owns the output samples of `tile_frames` hops, [a, b), and nothing else writes them.  It recomputes the
//     ceil(W/H) - 1 earlier frames that reach into [a, b) (the halo) instead of exchanging seams with its neighbours.
//   * Frames are computed X at a time (a round), one per thread group, and land windowed in shared memory.  One thread
//     per output sample then adds the round's contributions to what earlier rounds left in a carry buffer (increasing
//     frame order throughout, so the result does not depend on the tiling) and, for the samples no later frame can
//     reach, divides by the window-square sum formed from the window in shared memory and stores.
// Shared memory: [X scratch rows, reused as the windowed frames][2 carry buffers of N floats][window, M float2].
// ----------------------------------------------------------------------------------------
struct IstftParams {
    const float2 *spectra;     // [batch][frames][M+1] complex bins
    float *out;                // [batch][num_samples]
    const float *window;       // [wsize] window function values (f32), host-built
    const void *tw, *rtw;      // inverse stage tables / W_N^k of the c2r core
    long frames, num_samples;  // per signal
    long tile_frames;          // hops of output one CTA owns
    long tiles;                // CTAs per signal: block b owns tile b % tiles of signal b / tiles
    int hop, wsize, halo;      // halo = ceil(wsize / hop) - 1
    float inv_hop;             // 1 / hop (for small quotients, corrected exactly)
};

template <class PL, int PADQ, int X> __host__ __device__ constexpr size_t istft_smem_bytes() {
    return sizeof(float) * 2 * (size_t)padded_size<PADQ>(PL::N) * X + sizeof(float) * 4 * (size_t)PL::N + sizeof(float2) * (size_t)PL::N;
}

template <class PL, int X, int PADQ, int MINB>
__global__ void __launch_bounds__(PL::T *X, MINB) k_istft(const __grid_constant__ IstftParams ip) {
    static_assert(PL::valid(), "plan does not factor N");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using R = float;
    constexpr int M = PL::N, T = PL::T, E = PL::E, HALF = M / 2, PER = (HALF + T - 1) / T, NT = T * X;
    constexpr int LAST = PL::npass() - 1;
    constexpr int SROW = 2 * padded_size<PADQ>(M);                      // floats per group row (scratch, then frame)
    float *work = reinterpret_cast<float *>(smem_raw);
    float *carry = work + (size_t)X * SROW;                              // two buffers of 2M >= wsize floats
    float2 *winsm = reinterpret_cast<float2 *>(carry + 4 * M);
    const float *winf = reinterpret_cast<const float *>(winsm);
    const int xi = threadIdx.x / T, tid = threadIdx.x % T;
    const float2 *tw = reinterpret_cast<const float2 *>(ip.tw);
    const float2 *rtw = reinterpret_cast<const float2 *>(ip.rtw);
    const int H = ip.hop, W = ip.wsize;
    {
        const float2 *w2 = reinterpret_cast<const float2 *>(ip.window);
        for (int p = threadIdx.x; p < M; p += NT) winsm[p] = 2 * p < W ? __ldg(w2 + p) : make_float2(0.0f, 0.0f);
    }
    const long sig = blockIdx.x / ip.tiles;
    const long k0 = (blockIdx.x - sig * ip.tiles) * ip.tile_frames;      // first frame this CTA owns
    const float2 *spectra = ip.spectra + sig * ip.frames * (M + 1);
    float *out = ip.out + sig * ip.num_samples;
    const long a = k0 * H, b = min(a + ip.tile_frames * H, ip.num_samples);
    // sample offset u (from the round's first frame start) = q*H + r, stepped by NT without dividing
    const int tq = threadIdx.x / H, tr = threadIdx.x % H, sq = NT / H, sr = NT % H;
    const long ucov = max((long)(X - 1) * H + W, (long)X * H);          // reach of a round's frames (or its hops)
    const R sc = 0.5f / (float)M;
    int cur = 0;
    __syncthreads();
    for (long g = max(0L, k0 - ip.halo); g * H < b; g += X) {
        if (g < ip.frames) {                                             // (CTA-uniform) the round has frames
            const long f = g + xi;
            cx<R> *sm = reinterpret_cast<cx<R> *>(work + (size_t)xi * SROW);
            if (f < ip.frames && f * H < b) {
                // Hermitian pre-process of k_c2r (scale 0.5/M folded in, real parts only at DC and Nyquist)
                const float2 *in = spectra + f * (M + 1);
                static_for<PER>([&](auto I_) {
                    CIDX(i, I_);
                    const int k = tid + i * T;
                    if (k < HALF) {
                        if (i == 0 && k == 0) {
                            const float2 a0 = __ldg(in), am = __ldg(in + M);
                            sm[0] = mk<R>((a0.x + am.x) * sc, (a0.x - am.x) * sc);
                        }
                        const int kk = (k == 0) ? HALF : k;
                        const float2 va = __ldg(in + kk), vb = __ldg(in + (M - kk));
                        const twd<R> w = ld_tw(rtw + kk);
                        const R gr = va.x + vb.x, gi = va.y - vb.y, ur = va.x - vb.x, ui = va.y + vb.y;
                        const R hr = fmaf(w.y, ui, w.x * ur), hi = fmaf(w.ny, ur, w.x * ui);
                        sm[pad_idx<PADQ>(kk)] = mk<R>(sc * (gr - hi), sc * (gi + hr));
                        sm[pad_idx<PADQ>(M - kk)] = mk<R>(sc * (gr + hi), sc * (hr - gi));
                    }
                });
            }
            sync_transform<T, X>(xi);
            cx<R> x[E];
            {
                const cx<R> *base = sm + pad_idx<PADQ>(tid);
                static_for<E>([&](auto E_) { CIDX(e, E_); x[e] = base[pad_off<PADQ>(e * T)]; });
            }
            run_all<R, PL, PADQ, X, true>(x, tw, GTw<R>{nullptr, tw}, sm, tid, xi, true);
            sync_transform<T, X>(xi);                                    // the group's last reads of its scratch are done
            float2 *frame = reinterpret_cast<float2 *>(sm);              // y[2p], y[2p+1] times the window (0 past it)
            static_for<E>([&](auto S_) {
                CIDX(slot, S_);
                const int p = tid + out_elem<PL, LAST>(slot) * T;
                const float2 w = winsm[p];
                frame[p] = make_float2(x[slot].x * w.x, x[slot].y * w.y);
            });
        }
        __syncthreads();
        // overlap-add: this round's frames g .. g + flast reach [gH, gH + ucov); samples below (g + X) H are final
        const long gH = g * H;
        const int flast = (int)max(-1L, min((long)X - 1, ip.frames - 1 - g));
        const float *cin = carry + cur * 2 * M;
        float *cout = carry + (cur ^ 1) * 2 * M;
        const bool carried = g > max(0L, k0 - ip.halo);                  // an earlier round of this CTA left sums
        const long u0 = gH < a ? a - gH : 0, uend = min(ucov, b - gH);
        int q = (int)((gH < a ? k0 - g : 0) + tq), r = tr;              // u0 is a multiple of H
        for (long u = u0 + threadIdx.x; u < uend; u += NT) {
            float num = (carried && u < W - H) ? cin[u] : 0.0f;
            int dmax = -1;                                               // frames q - d with d*H + r < W cover u
            if (r < W) {
                const int span = W - 1 - r;
                dmax = __float2int_rz((float)span * ip.inv_hop);
                if (dmax * H > span) dmax--;
                else if ((dmax + 1) * H <= span) dmax++;
            }
            for (int d = min(dmax, q); d >= max(0, q - flast); d--) num += work[(q - d) * SROW + d * H + r];
            if (q < X) {
                const long fg = g + q;                                   // frames fg - d, every one that exists
                float den = 0.0f;
                const int dlo = (int)min(max(0L, fg - (ip.frames - 1)), (long)dmax + 1);
                for (int d = (int)min((long)dmax, fg); d >= dlo; d--) { const float w = winf[d * H + r]; den = fmaf(w, w, den); }
                st_stream(out + gH + u, den >= 1e-11f ? num / den : 0.0f);
            } else {
                cout[u - (long)X * H] = num;
            }
            r += sr; q += sq;
            if (r >= H) { r -= H; q++; }
        }
        cur ^= 1;
        __syncthreads();
    }
}

}  // namespace wfb
