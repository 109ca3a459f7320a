/*
 * watfft_b200.h -- C ABI of the B200-native batched FFT engine.
 *
 * This is the drop-in boundary for wat-fft's transform path: the entry points
 * below are what the N-API addon (wat-fft_b200/napi/watfft_napi.cc), the JS
 * loader (wat-fft_b200/js/index.js) and the pytest/ctypes harness bind.  Plain
 * pointers and sizes only; no C++/torch types cross it; no exceptions or
 * longjmp cross it (int error codes + wfb_strerror).
 *
 * What each call replaces in the reference (file:line under EmNudge/wat-fft):
 *
 *   wfb_plan_create   <- loadWasm()+instantiate (index.js:13-18) followed by the module's
 *                        precompute export: precompute_twiddles_split / precompute_rfft_twiddles_split
 *                        (modules/fft_split_native_f32.wat:151, :1167), precompute_twiddles
 *                        (modules/fft_stockham_f32_dual.wat:117, modules/fft_combined.wat:111),
 *                        precompute_rfft_twiddles (modules/fft_real_combined.wat:931).
 *   wfb_host_in/out   <- `new Float32Array(exports.memory.buffer, off, len)` views
 *                        (index.js:78-83, :107-112, :136-141, :165-170; REAL_OFFSET/IMAG_OFFSET
 *                        of modules/fft_split_native_f32.wat:60-61).
 *   wfb_exec(FORWARD) <- exports.fft_split / rfft_split (fft_split_native_f32.wat:2001, :1578),
 *                        exports.fft (fft_stockham_f32_dual.wat:1314, fft_combined.wat:727),
 *                        exports.rfft (fft_real_combined.wat:953).
 *   wfb_exec(INVERSE) <- exports.ifft_split / irfft_split (fft_split_native_f32.wat:2124, :1945),
 *                        exports.ifft (fft_stockham_f32_dual.wat:1329, fft_combined.wat:823).
 *                        f64 c2r has no reference implementation (index.js:145-147 calls a
 *                        missing export); it is provided as an extension.
 *   wfb_plan_destroy  <- garbage collection of the WebAssembly.Instance (new obligation).
 *
 * Batched buffer layout (reduces to the reference's memory map at batch = 1):
 *   C2C SPLIT        plane 0 = re[batch][n], plane 1 = im[batch][n]            (in place)
 *   C2C INTERLEAVED  plane 0 = [batch][2n]  (re,im pairs)                      (in place)
 *   R2C              time plane  = [batch][n] reals,
 *                    spectrum    = [batch][n+2]  (n/2+1 interleaved bins)
 *                    FORWARD reads time, writes spectrum; INVERSE the opposite.
 *                    At batch = 1 the two host views alias (same bytes, like index.js:136-141).
 * All transforms are unnormalised forward / 1/n-normalised inverse, natural bin order.
 *
 * Threading: a plan is not re-entrant; distinct plans are independent and may be driven from
 * distinct host threads.  Each plan binds one device and one stream.
 * There is NO CPU fallback: every entry point fails with WFB_ERR_NO_DEVICE when no sm_100
 * device is present.
 */
#ifndef WATFFT_B200_H
#define WATFFT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define WFB_API __declspec(dllexport)
#else
#define WFB_API __attribute__((visibility("default")))
#endif

typedef struct wfb_plan wfb_plan;

enum { WFB_C2C = 0, WFB_R2C = 1 };                 /* kind */
enum { WFB_F32 = 0, WFB_F64 = 1 };                 /* precision */
enum { WFB_SPLIT = 0, WFB_INTERLEAVED = 1 };       /* layout (C2C only) */
enum { WFB_FORWARD = 0, WFB_INVERSE = 1 };         /* direction */
enum { WFB_STAGE_H2D = 1, WFB_STAGE_D2H = 2, WFB_SYNC = 4, WFB_EXEC_DEFAULT = 7 };   /* exec flags */
enum { WFB_BUF_TIME = 0, WFB_BUF_SPECTRUM = 1 };   /* R2C buffer ids for wfb_*_buffer */

enum {
    WFB_OK = 0,
    WFB_ERR_NO_DEVICE = -1,     /* no CUDA device, or device is not sm_100 (B200) */
    WFB_ERR_BAD_SIZE = -2,      /* n not a power of two or outside the supported range */
    WFB_ERR_BAD_ARG = -3,
    WFB_ERR_UNSUPPORTED = -4,   /* (kind, precision, layout) combination not provided */
    WFB_ERR_ALLOC = -5,
    WFB_ERR_CUDA = -6,          /* see wfb_last_cuda_error() */
    WFB_ERR_NO_HOST_BUFFERS = -7
};

/* ---- device discovery ------------------------------------------------ */
WFB_API int wfb_device_count(void);
/* 0 when `device` is an sm_100 part; WFB_ERR_NO_DEVICE otherwise (the JS factory throws on it). */
WFB_API int wfb_require_b200(int device);
WFB_API const char *wfb_strerror(int code);
WFB_API const char *wfb_last_cuda_error(void);

/* ---- supported sizes -------------------------------------------------- */
/* Writes the inclusive [min_n, max_n] range for a combination; returns WFB_OK or WFB_ERR_UNSUPPORTED.
 * Works without a GPU (pure host logic). */
WFB_API int wfb_size_range(int kind, int precision, int layout, int *min_n, int *max_n);

/* ---- plans ------------------------------------------------------------- */
/* flags for wfb_plan_create_ex */
enum { WFB_PLAN_NO_HOST_BUFFERS = 1,    /* device-resident use only (bench / multi-GPU driver) */
       WFB_PLAN_NO_DEVICE_BUFFERS = 2   /* caller supplies device pointers to wfb_exec_device */ };

WFB_API wfb_plan *wfb_plan_create(int kind, int precision, int layout, int n, long batch, int device, int *err);
WFB_API wfb_plan *wfb_plan_create_ex(int kind, int precision, int layout, int n, long batch, int device,
                                     int flags, int *err);
WFB_API void wfb_plan_destroy(wfb_plan *plan);

/* Pinned host staging buffers, stable for the lifetime of the plan.
 *   C2C: plane 0 (re or interleaved), plane 1 (im; NULL for INTERLEAVED); in == out.
 *   R2C: wfb_host_in(plan, dir-agnostic plane) -- use wfb_host_buffer(plan, WFB_BUF_TIME|WFB_BUF_SPECTRUM). */
WFB_API void *wfb_host_in(wfb_plan *plan, int plane);
WFB_API void *wfb_host_out(wfb_plan *plan, int plane);
WFB_API void *wfb_host_buffer(wfb_plan *plan, int which);
WFB_API size_t wfb_host_bytes(wfb_plan *plan, int which);
WFB_API void *wfb_device_buffer(wfb_plan *plan, int which);

/* Runs `direction` over the plan's own buffers.  flags = WFB_EXEC_DEFAULT reproduces the reference's
 * synchronous forward()/inverse(): H2D of the input view, kernel, D2H of the output view, sync. */
WFB_API int wfb_exec(wfb_plan *plan, int direction, int flags);

/* Device-pointer entry (bench harness, multi-GPU driver).  d_in/d_out hold two plane pointers
 * (second unused unless C2C SPLIT).  `stream` is a cudaStream_t (NULL = the plan's stream).  The plan's stream is
 * NON-BLOCKING: it does not order against the legacy default stream, so a caller that produced the inputs on another
 * stream passes that stream here, or synchronises first.
 * In-place (d_in == d_out) is allowed for C2C and for R2C at batch = 1. */
WFB_API int wfb_exec_device(wfb_plan *plan, int direction, const void *const d_in[2], void *const d_out[2],
                            void *stream);
WFB_API int wfb_sync(wfb_plan *plan);

/* ---- module-shaped host memory (the exports facade) -----------------------------------------------------------------
 * The reference's raw exports work on ONE linear memory per instance: callers write inputs into `exports.memory.buffer`
 * at the module's offsets, call fft_split(n) / fft(n) / rfft(n), and read the results from the same bytes
 * (tests/fft_split_native.test.js:78-114; memory maps in modules/fft_split_native_f32.wat:7-18).  wfb_host_alloc returns
 * such a memory: pinned, device-mapped host bytes (zeroed) that the JS side wraps as `memory.buffer`; wfb_exec_host runs a
 * plan on plane pointers INSIDE memories obtained from wfb_host_alloc (anything else is WFB_ERR_BAD_ARG).  Small
 * payloads (WFB_OPT_MAPPED_MAX_BYTES) are transformed in place by one kernel that reads and writes those bytes directly --
 * no copy in either direction, like the WASM module working on its linear memory; larger ones are staged through the
 * plan's device buffers.  h_in/h_out: two plane pointers (second unused unless C2C SPLIT); in == out is allowed for C2C
 * and for R2C at batch = 1.  H2D/D2H staging is implied; flags adds WFB_SYNC (or not). */
WFB_API void *wfb_host_alloc(size_t bytes);
WFB_API void wfb_host_free(void *memory);
WFB_API int wfb_exec_host(wfb_plan *plan, int direction, const void *const h_in[2], void *const h_out[2], int flags);
WFB_API void *wfb_plan_stream(wfb_plan *plan);

/* ---- introspection / tuning ------------------------------------------- */
/* Kernel variants compiled for this plan's (kind, precision, n); variant 0 is the default.
 * wfb_plan_set_variant pins BOTH directions to that kernel and switches the zero-copy small-batch path off for the
 * plan (WFB_OPT_MAPPED_MAX_BYTES = 0), so that wfb_exec runs exactly the kernel that was asked for. */
WFB_API int wfb_plan_variant_count(wfb_plan *plan);
WFB_API int wfb_plan_set_variant(wfb_plan *plan, int variant);
WFB_API const char *wfb_plan_variant_name(wfb_plan *plan, int variant);
/* Index of the variant wfb_exec(plan, direction, ...) launches (the two directions may default to different kernels). */
WFB_API int wfb_plan_current_variant(wfb_plan *plan, int direction);
/* Algorithmic bytes one exec moves (one read + one write of the payload; twiddles excluded). */
WFB_API size_t wfb_plan_algorithmic_bytes(wfb_plan *plan);

/* Staging knobs of wfb_exec (defaults from the environment: WFB_MAPPED_MAX_KB, WFB_STAGE_CHUNK_MB, WFB_STAGE_STREAMS,
 * WFB_STAGE_RAMP).
 *   WFB_OPT_MAPPED_MAX_BYTES   payloads (input + output bytes) up to this size skip the copies: ONE kernel launch reads
 *                              and writes the pinned, device-mapped host buffers directly.  This is the path of the
 *                              reference's own call shape, batch = 1 (index.js:84-89).  0 disables it.
 *   WFB_OPT_STAGE_CHUNK_BYTES  bytes of the widest plane per chunk of the H2D / kernel / D2H pipeline
 *   WFB_OPT_STAGE_STREAMS      streams the chunks cycle over (1..6)
 *   WFB_OPT_STAGE_RAMP         1 (default): the pipeline starts and ends with short chunks (1/8, 1/4, 1/2 of the
 *                              steady-state size), shortening the two copies that have nothing to overlap with */
enum { WFB_OPT_MAPPED_MAX_BYTES = 0, WFB_OPT_STAGE_CHUNK_BYTES = 1, WFB_OPT_STAGE_STREAMS = 2, WFB_OPT_STAGE_RAMP = 3 };
WFB_API int wfb_plan_set_option(wfb_plan *plan, int option, long value);
WFB_API long wfb_plan_get_option(wfb_plan *plan, int option);
/* The chunk schedule wfb_exec uses for a batch (pure host logic, no GPU needed): rows per chunk of the H2D / kernel / D2H
 * pipeline for `batch` rows whose widest plane has `widest_row_bytes` per row, with WFB_OPT_STAGE_CHUNK_BYTES =
 * chunk_bytes and WFB_OPT_STAGE_RAMP = ramp.  Writes up to `capacity` entries and returns the number of chunks (0 when the
 * batch is small enough for one staged copy; a negative error code for bad arguments). */
WFB_API int wfb_stage_schedule(long batch, size_t widest_row_bytes, long chunk_bytes, int ramp, long *rows_out, int capacity);
/* Which path the latest wfb_exec took. */
enum { WFB_PATH_NONE = 0, WFB_PATH_STAGED = 1, WFB_PATH_PIPELINED = 2, WFB_PATH_MAPPED = 3 };
WFB_API int wfb_plan_last_path(wfb_plan *plan);

/* Pinned-copy ceiling of the host link of `device`: gbs[0] = H2D alone, gbs[1] = D2H alone, gbs[2], gbs[3] = H2D and
 * D2H running at the same time (GB/s each; `bytes` per copy, `iters` copies per direction).  The denominator of the
 * end-to-end (host-buffer) throughput: wfb_exec cannot move a transform faster than its bytes cross this link. */
WFB_API int wfb_pcie_probe(int device, size_t bytes, int iters, double gbs[4]);
/* The same probe in phases, for callers that drive several GPUs (one process or thread each) and want every GPU in the
 * same phase at the same moment -- open (allocates, one untimed copy each way), then per phase: barrier across the
 * ranks, run.  directions: 1 = H2D, 2 = D2H, 3 = both at once; seconds[0] / seconds[1] = device time of the H2D / D2H
 * train of `iters` copies of `bytes` (0 for a direction not run). */
typedef struct wfb_pcie_probe_state wfb_pcie_probe_state;
WFB_API int wfb_pcie_probe_open(int device, size_t bytes, wfb_pcie_probe_state **out);
WFB_API int wfb_pcie_probe_run(wfb_pcie_probe_state *probe, int directions, int iters, double seconds[2]);
WFB_API void wfb_pcie_probe_close(wfb_pcie_probe_state *probe);
/* Number of kernels this library has launched in this process (bench.py's gpu_launches). */
WFB_API unsigned long long wfb_kernel_launch_count(void);

/* Host-side reference-exact twiddle generation (no GPU needed): fills re/im[count] with the
 * W_n^k table the reference's precompute export would build.  flavour: 0 = f32 split module,
 * 1 = f32 interleaved module, 2 = f64 modules.  re/im are float* for 0/1, double* for 2. */
WFB_API int wfb_reference_twiddles(int flavour, int n, int count, void *re, void *im);

/* ---- batched STFT front-end (the reference's batched caller) ------------------------------
 * Replaces the per-frame JavaScript loop of playground/src/spectrogram.js:281-360
 * (slice -> applyWindow :27-38 -> zeroPad :40-45 -> context.run() -> computeMagnitude :47-58 ->
 * magnitudeToDb :60-62 -> gain/range normalisation :335-352) by ONE kernel launch over all frames:
 * frame gather, window multiply and zero padding are fused into the r2c load stage, |X| -> dB ->
 * [0,1] into its store stage.
 *   frames = floor((num_samples - window) / hop) + 1,  window = fft_size / zero_padding,
 *   bins   = fft_size/2 + 1.
 * Output, mode WFB_STFT_DB: float [frames][bins] in [0,1] (bins 0..2 forced to 0, :338-342);
 *         mode WFB_STFT_COMPLEX: float [frames][bins][2] (the raw spectra of the windowed frames).
 * Batches: wfb_stft_create_ex takes `batch` >= 1 equal-length signals in one handle, one launch for all of them.
 *   Input float [batch][num_samples], contiguous; output float [batch][frames][bins] (dB) or
 *   float [batch][frames][bins][2] (complex); `frames` (wfb_stft_frames) stays the count of ONE signal.  Every signal's
 *   rows are exactly what a single-signal handle computes for it: no frame reads samples of another signal, and the
 *   dB normalisation uses the fixed gain/range only.  wfb_stft_create is wfb_stft_create_ex with batch = 1.
 *   wfb_stft_output_bytes, wfb_stft_algorithmic_bytes and the pinned buffers cover the whole batch.  WFB_ERR_BAD_ARG
 *   for batch < 1 or a batch whose bytes overflow size_t.
 *   Alignment: the bulk-copy kernels (by default N = 1024, 2048 and 8192) need 16-byte aligned frame starts in every
 *   signal, the direct kernel's 64-bit loads 8-byte aligned ones.  With batch > 1 they are taken only when num_samples
 *   is a multiple of 4 (respectively 2) floats; otherwise the same results come from the direct kernel with narrower
 *   loads, as for an unaligned d_samples. */
typedef struct wfb_stft wfb_stft;
enum { WFB_WINDOW_HANN = 0, WFB_WINDOW_HAMMING = 1, WFB_WINDOW_BLACKMAN = 2, WFB_WINDOW_BLACKMAN_HARRIS = 3,
       WFB_WINDOW_RECTANGULAR = 4 };
enum { WFB_STFT_DB = 0, WFB_STFT_COMPLEX = 1 };
WFB_API wfb_stft *wfb_stft_create(int fft_size, int zero_padding, int hop, int window_type, long num_samples,
                                  int mode, float gain_db, float range_db, int device, int flags, int *err);
WFB_API wfb_stft *wfb_stft_create_ex(int fft_size, int zero_padding, int hop, int window_type, long num_samples,
                                     long batch, int mode, float gain_db, float range_db, int device, int flags, int *err);
/* Filterbank spectrogram (mel and the like; an extension: the reference has none), still ONE kernel launch:
 *   out[b][f][m] = L( sum_k F[m][k] * |X_bf[k]|^power ),
 * X_bf the raw (unnormalised) spectrum of frame f of signal b exactly as WFB_STFT_COMPLEX writes it, F a dense host
 * matrix float [num_filters][fft_size/2+1] (copied at creation; stored band-sparse on the device: each filter from its
 * first to its last non-zero bin), L(v) = v when log_scale == 0, else log_scale * log2(max(v + log_offset, log_floor))
 * (log_scale = ln 2 gives ln, log10(2) log10, 10 log10(2) dB of a power).  No bin is zeroed.
 * Output float [batch][frames][num_filters].  Each filter is one f32 FMA chain over its band in increasing bin order, so
 * results are bitwise repeatable and a batch row is bit-for-bit the single-signal result on the same kernel.
 * Geometry (fft_size, zero_padding, hop, window_type, num_samples, batch) as wfb_stft_create_ex, with num_filters floats
 * per output row in the overflow checks.  WFB_ERR_BAD_ARG also when num_filters is not in [1, fft_size/2+1], filters is
 * NULL or holds a non-finite value, power is not 1 or 2, log_scale is not finite, or log_scale != 0 and log_floor is not
 * a finite value > 0 or log_offset not a finite value >= 0.  The exec, buffer and size calls work unchanged;
 * wfb_stft_exec_inverse* returns WFB_ERR_UNSUPPORTED. */
WFB_API wfb_stft *wfb_stft_create_filterbank(int fft_size, int zero_padding, int hop, int window_type, long num_samples,
                                             long batch, int num_filters, const float *filters, int power, float log_scale,
                                             float log_offset, float log_floor, int device, int flags, int *err);
WFB_API void wfb_stft_destroy(wfb_stft *st);
WFB_API long wfb_stft_frames(wfb_stft *st);             /* per signal */
WFB_API long wfb_stft_batch(wfb_stft *st);
WFB_API int wfb_stft_bins(wfb_stft *st);
WFB_API int wfb_stft_filters(wfb_stft *st);             /* num_filters; 0 for a dB or complex handle */
WFB_API void *wfb_stft_host_samples(wfb_stft *st);      /* pinned, batch x num_samples floats */
WFB_API void *wfb_stft_host_output(wfb_stft *st);       /* pinned, wfb_stft_output_bytes() */
WFB_API size_t wfb_stft_output_bytes(wfb_stft *st);
WFB_API int wfb_stft_exec(wfb_stft *st, int flags);     /* flags as wfb_exec */
WFB_API int wfb_stft_exec_device(wfb_stft *st, const float *d_samples, void *d_out, void *stream);
/* Algorithmic bytes of one exec: every sample read once + the output written once. */
WFB_API size_t wfb_stft_algorithmic_bytes(wfb_stft *st);
/* Inverse of a WFB_STFT_COMPLEX spectrogram (an extension: the reference has no inverse).  Weighted overlap-add, the
 * least-squares estimate (what torch.istft(..., center=False) computes):
 *   y_f = the c2r of row f (1/N normalised, real parts of DC and Nyquist only), its first `window` samples used;
 *   num[t] = sum_f w[t-f*hop] y_f[t-f*hop],  D[t] = sum_f w[t-f*hop]^2  over the frames with 0 <= t-f*hop < window;
 *   x[t] = num[t] / D[t] where D[t] >= 1e-11, else 0  (window edges that are 0, gaps when hop > window), and 0 on
 *   [(frames-1)*hop + window, num_samples).
 * Unmodified spectra give back the signal wherever D >= 1e-11, to f32 rounding.  Every sum runs in increasing f, so the
 * result is bitwise repeatable.  WFB_ERR_UNSUPPORTED for a WFB_STFT_DB handle (magnitudes in dB cannot be inverted).
 * The inverse's twiddle tables are built by the first inverse call, not at creation.
 * wfb_stft_exec_inverse runs over the handle's own buffers: H2D of wfb_stft_host_output, kernel, D2H of
 * wfb_stft_host_samples, sync (flags as wfb_exec).  wfb_stft_exec_inverse_device reads batch x frames x bins complex
 * values at d_spectra (8-byte aligned) and writes batch x num_samples floats at d_samples (any float address); the two
 * must not overlap.  Each signal of a batch is reconstructed from its own frames only, exactly as by a single-signal
 * handle.  The stream contract is wfb_exec_device's. */
WFB_API int wfb_stft_exec_inverse(wfb_stft *st, int flags);
WFB_API int wfb_stft_exec_inverse_device(wfb_stft *st, const void *d_spectra, float *d_samples, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* WATFFT_B200_H */
