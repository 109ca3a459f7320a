/*
 * watfft_oracle.c -- CPU restatement of the wat-fft transform path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product (wat-fft_b200/) may
 * include, link or call this file; only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs use it, and only as the
 * checker or the reported CPU baseline.
 *
 * Parity status: PINNED.  tests/test_oracle_pinning.py compares every entry
 * point below against oracle/_ref/libwatref.so (the reference's own WAT
 * modules transpiled to C by oracle/wat2c.py and compiled without FMA) and
 * against the fixtures committed under tests/golden/ (generated from libwatref
 * by tests/golden/make_fixtures.py); tests/test_reference_suites.py checks the
 * reference's inline golden vectors (tests/golden_reference.test.js:32-214).
 *
 * All citations are file:line under the reference repo (EmNudge/wat-fft).
 * Build with -ffp-contract=off: WebAssembly has no fused multiply-add.
 *
 * One engine serves every transform: a Stockham autosort DIT pipeline of
 * radix-4 / radix-2 stages in which stage (radix r, l groups, stride
 * s = n/(r*l)) reads group j, lane t at  r*j*s + t + m*s  (m < r), multiplies
 * input m by the table twiddle  W_n^(m*j*n/(r*l)), and writes output q to
 * j*s + t + q*n/r:
 *   modules/fft_split_native_f32.wat:748-888 ($stage_r4_generic),
 *   :710-743 ($stage_r2_lead), modules/fft_combined.wat:361-474
 *   ($fft_radix4_general), :486-716 ($fft_stockham_general),
 *   modules/fft_stockham_f32_dual.wat:549-869 ($fft_general).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>

#define WFO_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------ */
/* Reference trig: Taylor series with range reduction (Appendix B).   */
/* f32: modules/fft_split_native_f32.wat:68-143                       */
/* f64: modules/fft_combined.wat:43-106                               */
/* ------------------------------------------------------------------ */
static const float PI_F = 3.14159265358979323846f;
static const float HALF_PI_F = 1.5707963267948966f;
static const double PI_D = 3.14159265358979323846;
static const double HALF_PI_D = 1.5707963267948966;

WFO_API float wfo_sin_f32(float x) {
    if (x < -PI_F) x = x + 2.0f * PI_F;
    if (x > PI_F) x = x - 2.0f * PI_F;
    if (x > HALF_PI_F) x = PI_F - x;
    if (x < -HALF_PI_F) x = -PI_F - x;
    float x2 = x * x, sum = x, term = x;
    static const float d[5] = {-6.0f, -20.0f, -42.0f, -72.0f, -110.0f};
    for (int i = 0; i < 5; i++) { term = term * (x2 / d[i]); sum = sum + term; }
    return sum;
}

WFO_API float wfo_cos_f32(float x) {
    float sign = 1.0f;
    if (x < -PI_F) x = x + 2.0f * PI_F;
    if (x > PI_F) x = x - 2.0f * PI_F;
    if (x > HALF_PI_F) { x = PI_F - x; sign = -1.0f; }
    if (x < -HALF_PI_F) { x = PI_F + x; sign = -1.0f; }
    float x2 = x * x, sum = 1.0f, term = 1.0f;
    static const float d[5] = {-2.0f, -12.0f, -30.0f, -56.0f, -90.0f};
    for (int i = 0; i < 5; i++) { term = term * (x2 / d[i]); sum = sum + term; }
    return sum * sign;
}

WFO_API double wfo_sin_f64(double x) {
    if (x < -PI_D) x = x + 2.0 * PI_D;
    if (x > PI_D) x = x - 2.0 * PI_D;
    if (x > HALF_PI_D) x = PI_D - x;
    if (x < -HALF_PI_D) x = -PI_D - x;
    double x2 = x * x, sum = x, term = x;
    static const double d[7] = {-6.0, -20.0, -42.0, -72.0, -110.0, -156.0, -210.0};
    for (int i = 0; i < 7; i++) { term = term * (x2 / d[i]); sum = sum + term; }
    return sum;
}

WFO_API double wfo_cos_f64(double x) {
    double sign = 1.0;
    if (x < -PI_D) x = x + 2.0 * PI_D;
    if (x > PI_D) x = x - 2.0 * PI_D;
    if (x > HALF_PI_D) { x = PI_D - x; sign = -1.0; }
    if (x < -HALF_PI_D) { x = PI_D + x; sign = -1.0; }
    double x2 = x * x, sum = 1.0, term = 1.0;
    static const double d[7] = {-2.0, -12.0, -30.0, -56.0, -90.0, -132.0, -182.0};
    for (int i = 0; i < 7; i++) { term = term * (x2 / d[i]); sum = sum + term; }
    return sum * sign;
}

/* ------------------------------------------------------------------ */
/* Base twiddle tables W_n^k, k < count.                               */
/* ------------------------------------------------------------------ */
/* split module: angle = f32(-6.283185307)/f32(n) * f32(k)   (fft_split_native_f32.wat:159,167) */
WFO_API void wfo_twiddles_f32_split(int n, int count, float *re, float *im) {
    float step = -6.283185307f / (float)(uint32_t)n;
    for (int k = 0; k < count; k++) {
        float a = step * (float)(uint32_t)k;
        re[k] = wfo_cos_f32(a);
        im[k] = wfo_sin_f32(a);
    }
}
/* dual module: angle = f32(k) * ((-2*PI)/n)   (fft_stockham_f32_dual.wat:129-141) */
WFO_API void wfo_twiddles_f32_dual(int n, int count, float *re, float *im) {
    float step = (-2.0f * PI_F) / (float)(uint32_t)n;
    for (int k = 0; k < count; k++) {
        float a = (float)(uint32_t)k * step;
        re[k] = wfo_cos_f32(a);
        im[k] = wfo_sin_f32(a);
    }
}
/* f64 modules: angle = f64(k) * ((-2*PI)/n)   (fft_combined.wat:114-124) */
WFO_API void wfo_twiddles_f64(int n, int count, double *re, double *im) {
    double step = (-2.0 * PI_D) / (double)(uint32_t)n;
    for (int k = 0; k < count; k++) {
        double a = (double)(uint32_t)k * step;
        re[k] = wfo_cos_f64(a);
        im[k] = wfo_sin_f64(a);
    }
}
/* Hard-coded codelet constants (fft_combined.wat:175-356, fft_real_combined.wat:166-445,
 * fft_stockham_f32_dual.wat:166-534): correctly rounded cos/sin of multiples of 2*pi/n. */
static void exact_twiddles_f64(int n, int count, double *re, double *im) {
    for (int k = 0; k < count; k++) {
        double a = -2.0 * M_PI * (double)k / (double)n;
        double c = cos(a), s = sin(a);
        if ((4 * k) % n == 0) {                        /* multiples of pi/2 */
            int m = (4 * k) / n % 4;
            c = (m == 0) ? 1.0 : (m == 2) ? -1.0 : 0.0;
            s = (m == 1) ? -1.0 : (m == 3) ? 1.0 : 0.0;
        } else if ((8 * k) % n == 0) {                 /* odd multiples of pi/4 */
            double h = 0.7071067811865476;
            c = (c > 0) ? h : -h;
            s = (s > 0) ? h : -h;
        }
        re[k] = c; im[k] = s;
    }
}

/* ------------------------------------------------------------------ */
/* Generic engine, instantiated for float and double.                  */
/* ------------------------------------------------------------------ */
#define DEFINE_ENGINE(SUF, REAL)                                                           \
/* cmul as the reference forms it: (wr*xr - wi*xi, wr*xi + wi*xr)                          \
 * (fft_split_native_f32.wat:826-837; fft_combined.wat:417-419 is the same values). */     \
static void stage_##SUF(int n, int r, int l, const REAL *sr, const REAL *si,               \
                        REAL *dr, REAL *di, const REAL *tr, const REAL *ti, int inv) {     \
    int s = n / (r * l);                                                                   \
    int step = n / (r * l);                                                                \
    int nq = n / r;                                                                        \
    REAL isg = inv ? (REAL)-1.0 : (REAL)1.0;                                               \
    for (int j = 0; j < l; j++) {                                                          \
        REAL wr[4], wi[4];                                                                 \
        for (int m = 1; m < r; m++) {                                                      \
            int idx = (m * j * step) % n;                                                  \
            wr[m] = tr[idx];                                                               \
            wi[m] = isg * ti[idx]; /* conjugated tables for the inverse (:230-252) */      \
        }                                                                                  \
        for (int t = 0; t < s; t++) {                                                      \
            int in0 = r * j * s + t;                                                       \
            int q = j * s + t;                                                             \
            if (r == 2) {                                                                  \
                REAL ar = sr[in0], ai = si[in0];                                           \
                REAL br = sr[in0 + s], bi = si[in0 + s];                                   \
                REAL wbr = wr[1] * br - wi[1] * bi;                                        \
                REAL wbi = wr[1] * bi + wi[1] * br;                                        \
                dr[q] = ar + wbr;       di[q] = ai + wbi;                                  \
                dr[q + nq] = ar - wbr;  di[q + nq] = ai - wbi;                             \
            } else {                                                                       \
                REAL ar = sr[in0], ai = si[in0];                                           \
                REAL br = sr[in0 + s], bi = si[in0 + s];                                   \
                REAL cr = sr[in0 + 2 * s], ci = si[in0 + 2 * s];                           \
                REAL xr = sr[in0 + 3 * s], xi = si[in0 + 3 * s];                           \
                REAL wcr = wr[2] * cr - wi[2] * ci, wci = wr[2] * ci + wi[2] * cr;         \
                REAL wbr = wr[1] * br - wi[1] * bi, wbi = wr[1] * bi + wi[1] * br;         \
                REAL wdr = wr[3] * xr - wi[3] * xi, wdi = wr[3] * xi + wi[3] * xr;         \
                REAL t0r = ar + wcr, t0i = ai + wci;                                       \
                REAL t1r = ar - wcr, t1i = ai - wci;                                       \
                REAL t2r = wbr + wdr, t2i = wbi + wdi;                                     \
                REAL t3r = wbr - wdr, t3i = wbi - wdi;                                     \
                /* the -i rotation flips for the inverse: middle blocks swap (:785-788) */ \
                int oa = inv ? 3 * nq : nq, ob = inv ? nq : 3 * nq;                        \
                dr[q] = t0r + t2r;           di[q] = t0i + t2i;                            \
                dr[q + oa] = t1r + t3i;      di[q + oa] = t1i - t3r;                       \
                dr[q + 2 * nq] = t0r - t2r;  di[q + 2 * nq] = t0i - t2i;                   \
                dr[q + ob] = t1r - t3i;      di[q + ob] = t1i + t3r;                       \
            }                                                                              \
        }                                                                                  \
    }                                                                                      \
}                                                                                          \
/* runs the stage list over split work planes; result returned in (re, im) */             \
static void pipeline_##SUF(int n, const int *radices, int nst, REAL *re, REAL *im,         \
                           const REAL *tr, const REAL *ti, int inv) {                      \
    REAL *br = (REAL *)malloc(sizeof(REAL) * 2 * (size_t)n), *bi = br + n;                 \
    REAL *sr = re, *si = im, *dr = br, *di = bi;                                           \
    int l = 1;                                                                             \
    for (int i = 0; i < nst; i++) {                                                        \
        stage_##SUF(n, radices[i], l, sr, si, dr, di, tr, ti, inv);                        \
        l *= radices[i];                                                                   \
        REAL *t = sr; sr = dr; dr = t; t = si; si = di; di = t;                            \
    }                                                                                      \
    if (sr != re) { memcpy(re, sr, sizeof(REAL) * n); memcpy(im, si, sizeof(REAL) * n); }  \
    free(br);                                                                              \
}

DEFINE_ENGINE(f32, float)
DEFINE_ENGINE(f64, double)

static int ilog2(int n) { int k = 0; while ((1 << k) < n) k++; return k; }
static int is_pow4(int n) { return (ilog2(n) & 1) == 0; }

/* stage lists */
/* split f32: n=4 codelet == one twiddle-free radix-4 (:273-329); n=8 radix-2 Stockham
 * (:2027-2115); n>=16 radix-4 core with a leading radix-2 when log2 n is odd (:1100-1158). */
static int plan_split_f32(int n, int *rad) {
    int k = 0;
    if (n == 8) { rad[0] = rad[1] = rad[2] = 2; return 3; }
    if (ilog2(n) & 1) rad[k++] = 2;
    for (int m = (ilog2(n) & 1) ? n / 2 : n; m > 1; m /= 4) rad[k++] = 4;
    return k;
}
/* f64: radix-4 when n is a power of 4, else radix-2 (fft_combined.wat:727-732) */
static int plan_f64(int n, int *rad) {
    int k = 0;
    if (is_pow4(n)) { for (int m = n; m > 1; m /= 4) rad[k++] = 4; }
    else { for (int m = n; m > 1; m /= 2) rad[k++] = 2; }
    return k;
}
/* interleaved f32 dual: radix-2 throughout (fft_stockham_f32_dual.wat:549-869);
 * n=4 codelet is a twiddle-free radix-4 (:166-200). */
static int plan_dual_f32(int n, int *rad) {
    int k = 0;
    if (n == 4) { rad[0] = 4; return 1; }
    for (int m = n; m > 1; m /= 2) rad[k++] = 2;
    return k;
}

/* ------------------------------------------------------------------ */
/* Transform 1: c2c f32 split  (fft_split :2001-2116, ifft_split :2124-2190) */
/* ------------------------------------------------------------------ */
WFO_API void wfo_fft_split_f32(int n, float *re, float *im, int inverse) {
    int rad[16], nst = plan_split_f32(n, rad);
    float *tr = (float *)malloc(sizeof(float) * 2 * (size_t)n), *ti = tr + n;
    wfo_twiddles_f32_split(n, n, tr, ti);
    pipeline_f32(n, rad, nst, re, im, tr, ti, inverse);
    if (inverse) {
        float sc = 1.0f / (float)(uint32_t)n;                 /* :2137-2149 */
        for (int i = 0; i < n; i++) { re[i] = re[i] * sc; im[i] = im[i] * sc; }
    }
    free(tr);
}

/* ------------------------------------------------------------------ */
/* Transform 2: r2c / c2r f32  (rfft_split :1578-1639, irfft_split :1945-1999) */
/* in: n reals; out: n/2+1 interleaved bins (n+2 floats).  n >= 32.            */
/* ------------------------------------------------------------------ */
/* Second half of $stage_r8_first_fused (:1199-1371): the radix-4 stage with l = 2 that follows the
 * twiddle-free radix-2 when log2(M) is odd.  Group 0 has unit twiddles; group 1 uses W_8^1, W_8^2 = -i
 * and W_8^3 as EXACT constants with the shuffle-free forms c*(Dr+Di, Di-Dr), (Di, -Dr) and
 * c*(Di-Dr, -(Dr+Di)), c = f32(0.7071067811865476) -- not the Taylor table the c2c path reads. */
static void stage_r4_l2_exact_f32(int n, const float *sr, const float *si, float *dr, float *di) {
    const float c = 0.7071067811865476f;
    int s = n / 8, nq = n / 4;
    for (int j = 0; j < 2; j++) {
        for (int t = 0; t < s; t++) {
            int in0 = 4 * j * s + t, q = j * s + t;
            float ar = sr[in0], ai = si[in0];
            float br = sr[in0 + s], bi = si[in0 + s];
            float cr = sr[in0 + 2 * s], ci = si[in0 + 2 * s];
            float xr = sr[in0 + 3 * s], xi = si[in0 + 3 * s];
            float t0r, t0i, t1r, t1i, t2r, t2i, t3r, t3i;
            if (j == 0) {
                t0r = ar + cr; t0i = ai + ci; t1r = ar - cr; t1i = ai - ci;
                t2r = br + xr; t2i = bi + xi; t3r = br - xr; t3i = bi - xi;
            } else {
                t0r = ar + ci; t0i = ai - cr; t1r = ar - ci; t1i = ai + cr;   /* a -/+ i*c */
                float wbr = c * (br + bi), wbi = c * (bi - br);
                float wdr = c * (xi - xr), wdi = -(c * (xr + xi));
                t2r = wbr + wdr; t2i = wbi + wdi; t3r = wbr - wdr; t3i = wbi - wdi;
            }
            dr[q] = t0r + t2r;           di[q] = t0i + t2i;
            dr[q + nq] = t1r + t3i;      di[q + nq] = t1i - t3r;
            dr[q + 2 * nq] = t0r - t2r;  di[q + 2 * nq] = t0i - t2i;
            dr[q + 3 * nq] = t1r - t3i;  di[q + 3 * nq] = t1i + t3r;
        }
    }
}

WFO_API void wfo_rfft_split_f32(int n, const float *x, float *out) {
    int m = n / 2, rad[16], nst = plan_split_f32(m, rad);
    float *zr = (float *)malloc(sizeof(float) * 4 * (size_t)m), *zi = zr + m, *tr = zi + m, *ti = tr + m;
    float *wr = (float *)malloc(sizeof(float) * 2 * (size_t)(m / 2 + 4)), *wi = wr + (m / 2 + 4);
    wfo_twiddles_f32_split(m, m, tr, ti);                     /* :1167-1191 */
    wfo_twiddles_f32_split(n, m / 2 + 4, wr, wi);             /* W_N^k, k = 0..N/4+3 */
    for (int j = 0; j < m; j++) { zr[j] = x[2 * j]; zi[j] = x[2 * j + 1]; }   /* :1376-1459 */
    if (rad[0] == 2 && m >= 32) {
        /* odd log2(M): fused radix-8 opening with exact W_8 constants (:1599-1607) */
        float *br = (float *)malloc(sizeof(float) * 2 * (size_t)m), *bi = br + m;
        stage_f32(m, 2, 1, zr, zi, br, bi, tr, ti, 0);
        stage_r4_l2_exact_f32(m, br, bi, zr, zi);
        free(br);
        /* remaining stages start at l = 8 */
        float *cr = (float *)malloc(sizeof(float) * 2 * (size_t)m), *ci = cr + m;
        float *sr = zr, *si = zi, *dr = cr, *di = ci;
        int l = 8;
        for (int i = 2; i < nst; i++) {
            stage_f32(m, rad[i], l, sr, si, dr, di, tr, ti, 0);
            l *= rad[i];
            float *t = sr; sr = dr; dr = t; t = si; si = di; di = t;
        }
        if (sr != zr) { memcpy(zr, sr, sizeof(float) * m); memcpy(zi, si, sizeof(float) * m); }
        free(cr);
    } else {
        pipeline_f32(m, rad, nst, zr, zi, tr, ti, 0);
    }
    /* $rfft_postprocess_split :1471-1559 */
    float z0r = zr[0], z0i = zi[0];
    out[0] = z0r + z0i; out[1] = 0.0f;
    for (int k = 1; k <= m / 2; k++) {
        float ar = zr[k], ai = zi[k], mr = zr[m - k], mi = zi[m - k];
        float gr = ar + mr, gi = ai - mi, hr = ai + mi, hi = mr - ar;
        float t_r = wr[k] * hr - wi[k] * hi;
        float t_i = wr[k] * hi + wi[k] * hr;
        float xr = 0.5f * (gr + t_r), xi = 0.5f * (gi + t_i);
        float yr = 0.5f * (gr - t_r), yi = 0.5f * (t_i - gi);
        /* X[M/2] is stored twice by the reference's last vector iteration (:1527-1545): the
         * forward block first, then the mirrored block, so the MIRRORED form 0.5*(G - T) is
         * what survives at k = M/2 (the two differ by the Taylor error of W_N^(N/4)). */
        out[2 * k] = xr; out[2 * k + 1] = xi;
        out[2 * (m - k)] = yr; out[2 * (m - k) + 1] = yi;
        /* M = 32 runs the fused ending $stage_r4_s1_rfft_fused (:2220-2714), which stores
         * X[M/2] = conj(Z[M/2]) directly (:2210, :2710) */
        if (m == 32 && k == m / 2) { out[2 * k] = ar; out[2 * k + 1] = -ai; }
    }
    out[2 * m] = z0r - z0i; out[2 * m + 1] = 0.0f;
    free(zr); free(wr);
}

WFO_API void wfo_irfft_split_f32(int n, const float *spec, float *x) {
    int m = n / 2, rad[16], nst = plan_split_f32(m, rad);
    float *zr = (float *)malloc(sizeof(float) * 4 * (size_t)m), *zi = zr + m, *tr = zi + m, *ti = tr + m;
    float *wr = (float *)malloc(sizeof(float) * 2 * (size_t)(m / 2 + 4)), *wi = wr + (m / 2 + 4);
    wfo_twiddles_f32_split(m, m, tr, ti);
    wfo_twiddles_f32_split(n, m / 2 + 4, wr, wi);
    /* $irfft_preprocess_split :1656-1748; scale 0.5/M folded in (:1674) */
    float sc = 0.5f / (float)(uint32_t)m;
    float x0 = spec[0], xm = spec[2 * m];      /* real parts only (:1679-1684) */
    zr[0] = (x0 + xm) * sc; zi[0] = (x0 - xm) * sc;
    for (int k = 1; k <= m / 2; k++) {
        float ar = spec[2 * k], ai = spec[2 * k + 1];
        float br = spec[2 * (m - k)], bi = spec[2 * (m - k) + 1];
        float gr = ar + br, gi = ai - bi, ur = ar - br, ui = ai + bi;
        float hr = wr[k] * ur + wi[k] * ui;
        float hi = wr[k] * ui - wi[k] * ur;
        /* same double store at k = M/2 (:1722-1740): forward first, mirrored survives */
        zr[k] = sc * (gr - hi); zi[k] = sc * (gi + hr);
        zr[m - k] = sc * (gr + hi); zi[m - k] = sc * (hr - gi);
    }
    pipeline_f32(m, rad, nst, zr, zi, tr, ti, 1);
    for (int j = 0; j < m; j++) { x[2 * j] = zr[j]; x[2 * j + 1] = zi[j]; }   /* :1756-1932 */
    free(zr); free(wr);
}

/* ------------------------------------------------------------------ */
/* Transform 3: c2c f32 interleaved (fft_stockham_f32_dual.wat fft :1314, ifft :1329) */
/* ------------------------------------------------------------------ */
WFO_API void wfo_fft_interleaved_f32(int n, float *data, int inverse) {
    int rad[16], nst = plan_dual_f32(n, rad);
    float *re = (float *)calloc(4 * (size_t)n, sizeof(float)), *im = re + n, *tr = im + n, *ti = tr + n;
    if (n <= 16) {  /* codelets with hard-coded constants (:166-534) */
        double er[16], ei[16];
        exact_twiddles_f64(n, n, er, ei);
        for (int k = 0; k < n; k++) { tr[k] = (float)er[k]; ti[k] = (float)ei[k]; }
    } else {
        wfo_twiddles_f32_dual(n, n, tr, ti);
    }
    for (int i = 0; i < n; i++) { re[i] = data[2 * i]; im[i] = data[2 * i + 1]; }
    pipeline_f32(n, rad, nst, re, im, tr, ti, inverse);
    float sc = inverse ? 1.0f / (float)(uint32_t)n : 1.0f;    /* folded into the r=1 stage (:645-681) */
    for (int i = 0; i < n; i++) { data[2 * i] = re[i] * sc; data[2 * i + 1] = im[i] * sc; }
    free(re);
}

/* ------------------------------------------------------------------ */
/* Transform 4: c2c f64 (fft_combined.wat fft :727, ifft :823) and     */
/* r2c f64 forward (fft_real_combined.wat rfft :953-1052)              */
/* ------------------------------------------------------------------ */
static void c2c_f64_core(int n, double *re, double *im, int inverse) {
    int rad[32], nst = plan_f64(n, rad);
    double *tr = (double *)malloc(sizeof(double) * 2 * (size_t)n), *ti = tr + n;
    /* precompute_twiddles is skipped for n <= 4 and the n=16 codelet carries exact constants
     * (fft_combined.wat:113, :175-356) */
    if (n == 16 || n <= 4) exact_twiddles_f64(n, n, tr, ti);
    else wfo_twiddles_f64(n, n, tr, ti);
    /* ifft = conj -> fft -> conj * 1/N (:823-830): identical arithmetic to running the
     * engine with conjugated twiddles and the +/-i rotation flipped. */
    pipeline_f64(n, rad, nst, re, im, tr, ti, inverse);
    free(tr);
}

WFO_API void wfo_fft_f64(int n, double *data, int inverse) {
    double *re = (double *)malloc(sizeof(double) * 2 * (size_t)n), *im = re + n;
    for (int i = 0; i < n; i++) { re[i] = data[2 * i]; im[i] = data[2 * i + 1]; }
    c2c_f64_core(n, re, im, inverse);
    double sc = inverse ? 1.0 / (double)(uint32_t)n : 1.0;
    for (int i = 0; i < n; i++) { data[2 * i] = re[i] * sc; data[2 * i + 1] = im[i] * sc; }
    free(re);
}

/* in: n reals at data[0..n); out: n/2+1 interleaved bins at data[0..n+2) (in place, like the module) */
WFO_API void wfo_rfft_f64(int n, double *data) {
    int m = n / 2;
    double *re = (double *)malloc(sizeof(double) * 4 * (size_t)(m + 1)), *im = re + (m + 1);
    double *wr = im + (m + 1), *wi = wr + (m + 1);
    for (int j = 0; j < m; j++) { re[j] = data[2 * j]; im[j] = data[2 * j + 1]; }
    c2c_f64_core(m, re, im, 0);
    /* codelet sizes carry exact constants (rfft_8 :166, rfft_32 :250) */
    if (n == 8 || n == 32) exact_twiddles_f64(n, m + 1, wr, wi);
    else wfo_twiddles_f64(n, m + 1, wr, wi);                  /* :931-948, k = 0..M */
    double z0r = re[0], z0i = im[0];
    data[0] = z0r + z0i; data[1] = 0.0;
    data[2 * m] = z0r - z0i; data[2 * m + 1] = 0.0;
    for (int k = 1; k < m / 2; k++) {                         /* :982-1030 / :489-560 */
        int mk = m - k;
        double sr = re[k] + re[mk], si = im[k] - im[mk];
        double dr = re[k] - re[mk], di = im[k] + im[mk];
        double wdr = wi[k] * dr + wr[k] * di;
        double wdi = wi[k] * di - wr[k] * dr;
        double s2r = re[mk] + re[k], s2i = im[mk] - im[k];
        double d2r = re[mk] - re[k], d2i = im[mk] + im[k];
        double wd2r = wi[mk] * d2r + wr[mk] * d2i;
        double wd2i = wi[mk] * d2i - wr[mk] * d2r;
        data[2 * k] = 0.5 * (sr + wdr);      data[2 * k + 1] = 0.5 * (si + wdi);
        data[2 * mk] = 0.5 * (s2r + wd2r);   data[2 * mk + 1] = 0.5 * (s2i + wd2i);
    }
    if ((m & 1) == 0 && m > 2) {                              /* middle element :1031-1050 */
        int k = m / 2;
        double sr = 2.0 * re[k], si = 0.0, dr = 0.0, di = 2.0 * im[k];
        double wdr = wi[k] * dr + wr[k] * di;
        double wdi = wi[k] * di - wr[k] * dr;
        data[2 * k] = 0.5 * (sr + wdr); data[2 * k + 1] = 0.5 * (si + wdi);
    }
    free(re);
}

/* f64 c2r: the reference has NO implementation (fft_real_combined.wat exports only
 * precompute_rfft_twiddles and rfft; index.js:145-147 calls a missing export).
 * PARITY UNPINNED: defined here as the exact algebraic inverse of wfo_rfft_f64's
 * formulas, in the order of the f32 pre-process ($irfft_preprocess_split :1656-1748),
 * and gated against the f64 DFT.  The k = M/2 bin pairs with itself: the forward form
 * is stored first and the mirrored one survives, like wfo_irfft_split_f32 and every
 * c2r kernel.  (The two differ by 2*wr[M/2]*Im X[M/2], and the Taylor table's
 * wr[M/2] = cos(pi/2) is ~1e-11, not 0.) */
WFO_API void wfo_irfft_f64(int n, const double *spec, double *x) {
    int m = n / 2;
    double *re = (double *)malloc(sizeof(double) * 4 * (size_t)(m + 1)), *im = re + (m + 1);
    double *wr = im + (m + 1), *wi = wr + (m + 1);
    if (n == 8 || n == 32) exact_twiddles_f64(n, m + 1, wr, wi);
    else wfo_twiddles_f64(n, m + 1, wr, wi);
    double sc = 0.5 / (double)(uint32_t)m;
    re[0] = (spec[0] + spec[2 * m]) * sc; im[0] = (spec[0] - spec[2 * m]) * sc;
    for (int k = 1; k <= m / 2; k++) {
        double ar = spec[2 * k], ai = spec[2 * k + 1];
        double br = spec[2 * (m - k)], bi = spec[2 * (m - k) + 1];
        double gr = ar + br, gi = ai - bi, ur = ar - br, ui = ai + bi;
        double hr = wr[k] * ur + wi[k] * ui;
        double hi = wr[k] * ui - wi[k] * ur;
        re[k] = sc * (gr - hi); im[k] = sc * (gi + hr);
        re[m - k] = sc * (gr + hi); im[m - k] = sc * (hr - gi);
    }
    c2c_f64_core(m, re, im, 1);
    for (int j = 0; j < m; j++) { x[2 * j] = re[j]; x[2 * j + 1] = im[j]; }
    free(re);
}

/* ------------------------------------------------------------------ */
/* Ground truth: O(N^2) f64 DFT (tests/dft-reference.js:14-88)         */
/* ------------------------------------------------------------------ */
WFO_API void wfo_dft_f64(int n, const double *re, const double *im, double *ore, double *oim, int inverse) {
    double sgn = inverse ? 2.0 : -2.0;
    for (int k = 0; k < n; k++) {
        double sr = 0.0, si = 0.0;
        for (int j = 0; j < n; j++) {
            double a = (sgn * M_PI * (double)(((int64_t)j * k) % n)) / (double)n;
            double c = cos(a), s = sin(a);
            sr += re[j] * c - im[j] * s;
            si += re[j] * s + im[j] * c;
        }
        if (inverse) { sr /= n; si /= n; }
        ore[k] = sr; oim[k] = si;
    }
}

/* ------------------------------------------------------------------ */
/* Batched driver used by bench.py's cpu_baseline "port" leg: each row */
/* is transformed independently, like one WASM instance per transform. */
/* ------------------------------------------------------------------ */
WFO_API void wfo_fft_split_f32_batch(int n, int batch, float *re, float *im, int inverse) {
    for (int b = 0; b < batch; b++)
        wfo_fft_split_f32(n, re + (size_t)b * n, im + (size_t)b * n, inverse);
}
