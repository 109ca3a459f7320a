#!/usr/bin/env python3
"""bench.py -- benchmark of the B200 batched-FFT hot path (every BASELINE.json config in one record).

HEADLINE (BASELINE.json configs[1], the configuration the metric is quoted on): batched complex f32
split-format fft_split + ifft_split at N = 16, 32, ..., 4096, batch sized to 1 GiB of input per launch per
GPU (B = 2^30 / 8N).  One STEP = forward then inverse at each of the 9 sizes = 18 kernel launches, each
reading 1 GiB and writing 1 GiB (all far larger than the 126 MB L2, so no flush is needed between
iterations).  Inputs are synthetic (uniform [-1,1)), resident in HBM when the timed region starts.  N > 1
GPUs: the batch is sharded, every rank runs the same per-GPU workload on its own device with no data-path
collective (weak scaling).

Printed JSON (one line, rank 0).  Besides the contract's keys:
  configs      every other BASELINE config, device-resident, CUDA-event timed per kernel:
               configs[0] (c2c f32 split N=1024, batch 1: forward() latency through the API + plan creation),
               configs[2] (r2c/c2r f32 N=64..4096), configs[3] (f64 c2c + r2c N=256..4096), the interleaved f32
               transform, the fused STFT, and at N>1 configs[4] (c2c N=4096, 262144 rows strong-scaled over the ranks)
  e2e          the headline workload through createFFTf32Split().forward()/inverse() on pinned HOST buffers
               (H2D + kernel + D2H in the timed region), random inputs with a sampled oracle check, next to the
               CONCURRENT pinned-copy ceiling of the link measured in the same run (pcie_peak_GBs, frac), plus r2c and
               STFT companions (fewer PCIe bytes per transform)
  roofline     the headline kernel with the largest share of the step
  cpu_baseline the reference's own modules (transpiled, oracle/_ref) on all host cores: persistent thread pool,
               instance + precompute once per size outside the timed region, memcpy-in + transform per row

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SIZES = [16, 32, 64, 128, 256, 512, 1024, 2048, 4096]
REAL_SIZES = [64, 128, 256, 512, 1024, 2048, 4096]
F64_SIZES = [256, 512, 1024, 2048, 4096]
STFT_SIZES = [256, 512, 1024, 2048, 4096]
GIB = 1 << 30
METRIC = "batched FFT transforms/s (c2c f32 split fft+ifft, N=16-4096, 1 GiB/launch/GPU)"
UNIT = "transforms/s"
CPU_SAMPLE_DIV = 4          # the CPU legs process 1/4 of every batch per step (256 MiB of input per launch)


def workload_config(n_gpus):
    return {
        "workload": "configs[1]: batched complex f32 split fft_split+ifft_split, N=16..4096 (9 sizes), "
                    "batch = 2^30/(8N) per GPU (1 GiB input per launch)",
        "sizes": SIZES,
        "input_bytes_per_launch_per_gpu": GIB,
        "launches_per_step": 2 * len(SIZES),
        "cache": "inputs (1 GiB per launch) larger than L2 (126 MB); no flush needed",
        "parallelism": f"batch-sharded x{n_gpus}, no data-path collective",
    }


def peaks():
    try:
        p = json.load(open(ROOT / "MEASURED_PEAKS.json"))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# --------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        # nvidia-smi numbers the physical GPUs; a CUDA_VISIBLE_DEVICES list of plain indices maps the CUDA ordinal onto them
        vis = [v.strip() for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip()]
        if index < len(vis) and vis[index].isdigit():
            index = int(vis[index])
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        rows = [l.strip().split(", ") for l in open(self.tmp.name) if l.strip()]
        os.unlink(self.tmp.name)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for name, v in zip(names, r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if sm:
            busy = [s for s in sm if s > 0.5 * max(mx)] or sm
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       power_w_max=max(pw) if pw else None)
        return out


# --------------------------------------------------------------------------------------------
# the reference arm / CPU baseline: the reference's own modules (oracle/_ref/libwatref.so) on the host cores
# --------------------------------------------------------------------------------------------
class CpuReference:
    """Times the transpiled reference modules with a persistent pool of pthreads (one private module memory each).
    Per size the instance + precompute happen once, untimed (benchmarks/lib/wat-contexts.js:110-131); a timed sample is
    `memcpy(row) -> transform(n)` over the sample rows (:125-129).  Rows are views of ONE random buffer that is larger
    than the caches (256 MiB), the same way the GPU leg reuses its 1 GiB buffers for every size."""

    def __init__(self, threads=None):
        sys.path.insert(0, str(ROOT / "oracle"))
        import numpy as np
        import oracle as om
        om.build()
        self.np, self.om = np, om
        self.kind = "reference" if om.WatRef.available() else "port"
        self.cores = threads or os.cpu_count() or 1
        rng = np.random.default_rng(1234)
        self.words = (GIB // CPU_SAMPLE_DIV) // 4
        self.buf32 = rng.uniform(-1, 1, self.words + 4096).astype(np.float32)
        self.buf64 = None
        if self.kind == "reference":
            self.ref = om.WatRef()
            self.pool = om.WatRefPool(self.ref, self.cores)
        else:                                   # no transpiled reference on this box: the single-thread C port
            self.port = om.Oracle()
            self.cores = 1

    def describe(self):
        if self.kind == "reference":
            return ("transpiled reference WAT modules (oracle/_ref/libwatref.so), persistent pool of "
                    f"{self.cores} pthreads pinned one per core, one module memory per thread, precompute once per size "
                    "outside the timed region, memcpy-in + transform per row")
        return "single-thread C port (oracle/watfft_oracle.c)"

    # (module, precompute, export, words per row in, bytes/elem, second-plane offset or None)
    def _spec(self, transform, n, inverse):
        IM = self.om.SPLIT_IMAG_OFFSET
        if transform == "c2c_split":
            return ("fft_split_native_f32", "precompute_twiddles_split", "ifft_split" if inverse else "fft_split", n, 4, IM)
        if transform == "c2c_il":
            return ("fft_stockham_f32_dual", "precompute_twiddles", "ifft" if inverse else "fft", 2 * n, 4, None)
        if transform == "real_f32":
            return ("fft_split_native_f32", "precompute_rfft_twiddles_split", "irfft_split" if inverse else "rfft_split",
                    n + 2 if inverse else n, 4, None)
        if transform == "c2c_f64":
            return ("fft_combined", "precompute_twiddles", "ifft" if inverse else "fft", 2 * n, 8, None)
        if transform == "r2c_f64":
            return ("fft_real_combined", "precompute_rfft_twiddles", "rfft", n, 8, None)
        raise ValueError(transform)

    def samples(self, transform, n, inverse=False, rows=None, count=3, min_s=0.15, pool=None):
        """`count` timed samples of >= min_s seconds each; returns (rows per sample pass, [seconds per pass])."""
        np = self.np
        module, pre, export, row_words, esz, im_off = self._spec(transform, n, inverse)
        if esz == 8 and self.buf64 is None:
            self.buf64 = self.buf32[: self.words // 2].astype(np.float64)
        src = self.buf64 if esz == 8 else self.buf32
        planes = 2 if im_off is not None else 1
        if rows is None:
            rows = (len(src) // planes) // row_words
        a = src[: rows * row_words].reshape(rows, row_words)
        b = src[rows * row_words: 2 * rows * row_words].reshape(rows, row_words) if planes == 2 else None
        if self.kind != "reference":
            assert transform == "c2c_split"
            out = []
            for _ in range(count):
                t0 = time.perf_counter()
                r2, i2 = a.copy(), b.copy()
                self.port.lib.wfo_fft_split_f32_batch(n, rows, r2.ctypes.data_as(self.om._c_f32p),
                                                      i2.ctypes.data_as(self.om._c_f32p), int(inverse))
                out.append(time.perf_counter() - t0)
            return rows, out
        pool = pool or self.pool
        pool.prepare(module, pre, n)
        run = lambda reps: pool.run(module, export, n, a, 0, b, im_off or 0, reps=reps)
        t1 = run(1)                                   # warm-up pass, also calibrates the repeat count
        reps = max(1, int(math.ceil(min_s / max(t1, 1e-6))))
        return rows, [run(reps) / reps for _ in range(count)]

    def rate(self, transform, n, inverse=False, **kw):
        rows, ts = self.samples(transform, n, inverse, **kw)
        return rows / statistics.median(ts)

    def headline(self, steps, warmup, min_s=0.0):
        """The headline mix: per size, `steps` timed passes of fft_split and of ifft_split over 1/CPU_SAMPLE_DIV of the
        batch; step k = the sum over sizes and directions of pass k.  Returns (value, per_step_s list, per_n dict)."""
        t = [[0.0] * len(SIZES) * 2 for _ in range(steps)]
        per_n, transforms = {}, 0
        for i, n in enumerate(SIZES):
            for d in (0, 1):
                rows, ts = self.samples("c2c_split", n, bool(d), count=steps + max(1, min(warmup, 2)), min_s=min_s)
                ts = ts[-steps:]
                for k in range(steps):
                    t[k][2 * i + d] = ts[k]
                per_n.setdefault(str(n), {})["inv" if d else "fwd"] = round(rows / statistics.median(ts) / 1e6, 3)
                transforms += rows
        per_step = [sum(r) for r in t]
        return transforms / statistics.median(per_step), per_step, per_n, transforms

    def anchor(self):
        """One thread, one resident N=1024 input, one transform per call: the shape of the reference's own published
        numbers (BASELINE.md section 1: 1.05 M/s on an M5 Pro under V8) and of BASELINE configs[0]."""
        if self.kind != "reference":
            return None
        p1 = self.om.WatRefPool(self.ref, 1)
        try:
            rows, ts = self.samples("c2c_split", 1024, rows=1, count=3, min_s=0.15, pool=p1)
            return 1.0 / statistics.median(ts)
        finally:
            p1.close()

    def thread_scaling(self, n=1024):
        if self.kind != "reference":
            return None
        out = {}
        for th in sorted({1, max(1, self.cores // 4), max(1, self.cores // 2), self.cores}):
            p = self.om.WatRefPool(self.ref, th)
            try:
                out[str(th)] = round(self.rate("c2c_split", n, count=2, min_s=0.1, pool=p) / 1e6, 3)
            finally:
                p.close()
        return out

    def stft_rate(self, n, hop, min_s=0.15):
        """frames/s of the spectrogram loop (playground/src/spectrogram.js:299-353, C port) around the module's rfft_split."""
        np = self.np
        x = self.buf32[: min(self.words, 1 << 24)]
        w = self.om.window_function("hann", n)
        frames = (len(x) - n) // hop + 1
        out = np.empty(frames * (n // 2 + 1), np.float32)
        self.pool.prepare("fft_split_native_f32", "precompute_rfft_twiddles_split", n)
        t1 = self.pool.run_stft(x, n, hop, w, 0.0, 80.0, out)
        reps = max(1, int(math.ceil(min_s / max(t1, 1e-6))))
        return frames / (self.pool.run_stft(x, n, hop, w, 0.0, 80.0, out, reps=reps) / reps)

    def baseline_block(self, steps=5, warmup=1):
        value, per_step, per_n, transforms = self.headline(steps, warmup)
        bytes_in = 2 * len(SIZES) * (GIB // CPU_SAMPLE_DIV)
        blk = {"value": value, "unit": UNIT, "cores": self.cores, "kind": self.kind,
               "sample": f"1/{CPU_SAMPLE_DIV} of each batch (N=16..4096, fwd+inv; {transforms} transforms, "
                         f"{bytes_in >> 20} MiB copied in per step; median of {steps} steps), " + self.describe(),
               "per_n_Mtransforms_s": per_n,
               "input_stream_GBs": round(bytes_in / statistics.median(per_step) / 1e9, 2)}
        if self.kind == "reference":
            a = self.anchor()
            blk["anchor_1thread_n1024"] = {"Mtransforms_s": round(a / 1e6, 4), "us_per_call": round(1e6 / a, 3),
                                           "published_M5Pro_V8_Mtransforms_s": 1.05,
                                           "note": "one thread, resident input, memcpy + fft_split per call (BASELINE.md section 1 shape)"}
            blk["thread_scaling_n1024_Mtransforms_s"] = self.thread_scaling()
        return blk

    def close(self):
        if self.kind == "reference":
            self.pool.close()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cpu = CpuReference()
    steps = max(1, args.steps)
    value, per_step, per_n, transforms = cpu.headline(steps, args.warmup)
    bytes_in = 2 * len(SIZES) * (GIB // CPU_SAMPLE_DIV)
    sample = (f"1/{CPU_SAMPLE_DIV} of each batch per step (N=16..4096, fwd+inv; {transforms} transforms, {bytes_in >> 20} MiB "
              f"copied in per step), " + cpu.describe())
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": statistics.median(per_step) * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cpu.cores, "kind": cpu.kind, "sample": sample,
                         "per_n_Mtransforms_s": per_n},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    cpu.close()
    emit(line)
    return 0


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
DUMP_FLOATS = 1 << 18       # floats per dumped array (1 MiB): 9 sizes x 4 planes = 36 MiB in all


def dump_outputs(out_dir, steps, step, seed_input, a, b):
    """--dump-outputs: writes what the last of the `steps` timed headline steps returned at each size -- the forward
    spectrum and the inverse's result, split re/im planes, a fixed seeded sample of rows of each -- as
    <out_dir>/<name>.npy (float32).  The timed steps start from the seeded input and the kernels are deterministic, so
    replaying steps - 1 steps and capturing the next one reproduces the last timed step; the replay is checked bit for
    bit against the state the timed steps left (at the largest size, whose outputs the step does not overwrite)."""
    import numpy as np
    import torch
    pick = np.random.default_rng(20250)
    rows = {}
    for n in SIZES:
        batch = GIB // (8 * n)
        rows[n] = torch.as_tensor(np.sort(pick.choice(batch, min(batch, DUMP_FLOATS // n), replace=False)),
                                  device=a[0].device)

    def take(n, planes):
        return [p.view(-1, n).index_select(0, rows[n]).cpu().numpy() for p in planes]

    out = {}

    def capture(n, direction, re, im):
        out[f"c2c_f32_split_n{n}_{direction}_re"], out[f"c2c_f32_split_n{n}_{direction}_im"] = take(n, (re, im))

    n = SIZES[-1]
    timed = take(n, b) + take(n, a)
    seed_input()
    for _ in range(steps - 1):
        step()
    step(capture=capture)
    replayed = [out[f"c2c_f32_split_n{n}_{d}_{p}"] for d in ("forward", "inverse") for p in ("re", "im")]
    assert all(np.array_equal(x, y) for x, y in zip(timed, replayed)), "replayed last step differs from the timed one"
    assert sum(x.nbytes for x in out.values()) <= 64 * 10**6
    os.makedirs(out_dir, exist_ok=True)
    for name, x in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), x)


def run_ours(args):
    import ctypes
    import numpy as np
    import torch
    import watfft_b200 as wf
    C = wf._cabi
    lib = C.lib()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # Rank -> GPU.  When the box shows more GPUs than there are ranks, the ranks take GPUs spread over the whole box
    # (rank i -> GPU i * visible/world) instead of the first `world`: the host bridges of an 8-GPU board serve half the
    # GPUs each, and on this pool GPUs 0..3 together get no more host bandwidth than GPU 0 alone
    # (profiles/r02_pcie.md), which decides the end-to-end number.  WFB_BENCH_DEVICE_ORDER=seq restores rank i -> GPU i.
    visible = torch.cuda.device_count()
    from watfft_b200.sharding import rank_device
    local = rank_device(local_rank, world, visible, os.environ.get("WFB_BENCH_DEVICE_ORDER", "spread"))
    spread = rank_device(world - 1, world, visible, os.environ.get("WFB_BENCH_DEVICE_ORDER", "spread")) != world - 1
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout; keep stdout to the single JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", os.devnull)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    n_gpus = world
    rc = lib.wfb_require_b200(local)
    if rc != 0:
        raise SystemExit("bench.py: " + lib.wfb_strerror(rc).decode() + " -- " + lib.wfb_last_cuda_error().decode())
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    assert sptr != 0
    peak, peak_src = peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return float(v)
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device memory: ONE arena, carved per workload.  Region A = 1 GiB input, region B = 1 GiB (+ slack for the
    # two extra floats per spectrum row) output; every size of every transform reuses them.
    SLACK = 64 << 20
    arena = torch.empty(2 * GIB + 2 * SLACK, dtype=torch.uint8, device=dev)
    a_ptr = arena.data_ptr()
    b_ptr = a_ptr + GIB + SLACK
    A32 = arena[: GIB].view(torch.float32)
    g = torch.Generator(device=dev)

    def seed_input():
        g.manual_seed(1234 + rank)
        A32.uniform_(-1, 1, generator=g)
    seed_input()
    nfloat = GIB // 8
    a_re, a_im = A32[:nfloat], A32[nfloat:]
    Bv = arena[GIB + SLACK: 2 * GIB + SLACK].view(torch.float32)
    b_re, b_im = Bv[:nfloat], Bv[nfloat:]
    ref_re = a_re[: 1 << 20].clone()
    ref_im = a_im[: 1 << 20].clone()
    flags = C.PLAN_NO_HOST_BUFFERS | C.PLAN_NO_DEVICE_BUFFERS
    plans = {n: wf.Plan(C.C2C, C.F32, C.SPLIT, n, GIB // (8 * n), local, flags) for n in SIZES}
    A = (a_re.data_ptr(), a_im.data_ptr())
    B = (b_re.data_ptr(), b_im.data_ptr())

    def step(events=None, capture=None):
        for i, n in enumerate(SIZES):
            if events is not None:
                events[2 * i].record(stream)
            plans[n].exec_device(C.FORWARD, A, B, sptr)       # A -> B
            if capture is not None:
                capture(n, "forward", b_re, b_im)
            if events is not None:
                events[2 * i + 1].record(stream)
            plans[n].exec_device(C.INVERSE, B, A, sptr)       # B -> A (round trip restores the data)
            if capture is not None:
                capture(n, "inverse", a_re, a_im)
        if events is not None:
            events[2 * len(SIZES)].record(stream)

    # ---- headline: warm-up, then EXACTLY K timed steps.
    # Every rank keeps its GPU under load for a fixed 0.75 s right up to the start barrier, so that the timed region
    # sees the same sustained (power-capped) clocks at every N.  (Round 1 waited at a barrier with idle GPUs at N > 1:
    # the boards dropped out of the power cap and the 120 ms timed region ran at burst clocks, 5.5 % faster per GPU
    # than the N = 1 run, which had no such pause.)
    sampler = ClockSampler(local) if rank == 0 else None     # nvidia-smi needs ~0.3 s to start sampling
    warm = max(3, args.warmup)
    for _ in range(warm):
        step()
    barrier()
    t_w = time.perf_counter()
    while time.perf_counter() - t_w < 0.75:
        step()
        torch.cuda.synchronize()
    # the warm-up made a wall-clock-dependent number of round trips over A: the timed steps start again from the seeded
    # input, so that they compute the same values in every run with the same arguments
    seed_input()
    launches0 = lib.wfb_kernel_launch_count()
    K = args.steps
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2 * len(SIZES) + 1)] for _ in range(K)]
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin.record(stream)
    for k in range(K):
        step(evs[k])
    t_end.record(stream)
    barrier()
    launches = lib.wfb_kernel_launch_count() - launches0
    assert launches == K * 2 * len(SIZES), launches
    elapsed_ms = t_begin.elapsed_time(t_end)
    clocks = sampler.stop() if sampler else None
    # the round trips must have restored the input: proof the timed launches did the work.  f32 rounding
    # accumulates over the fft->ifft round trips since the input was seeded (those of the timed steps), so the bound
    # scales with their number ...
    trips = len(SIZES) * K
    drift = float((a_re[: 1 << 20] - ref_re).abs().max())
    assert drift < max(1e-3, 4e-6 * trips), f"round-trip drift {drift} after {trips} round trips"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, K, step, seed_input, (a_re, a_im), (b_re, b_im))
    # ... and one fresh step on pristine data must come back within the reference's own round-trip tolerance
    a_re[: 1 << 20] = ref_re
    a_im[: 1 << 20] = ref_im
    step()
    torch.cuda.synchronize()
    fresh = max(float((a_re[: 1 << 20] - ref_re).abs().max()), float((a_im[: 1 << 20] - ref_im).abs().max()))
    assert fresh < 1e-4, f"fresh-step round-trip error {fresh}"
    elapsed_ms = max_over_ranks(elapsed_ms)

    transforms_per_step_gpu = 2 * sum(GIB // (8 * n) for n in SIZES)
    ms_per_step = elapsed_ms / K
    value = n_gpus * transforms_per_step_gpu / (ms_per_step * 1e-3)
    bytes_per_launch = 2 * GIB
    agg_gbs = n_gpus * 2 * len(SIZES) * bytes_per_launch / (ms_per_step * 1e-3) / 1e9
    step_ms = [evs[k][0].elapsed_time(evs[k][2 * len(SIZES)]) for k in range(K)]

    # per-kernel launch durations (rank-local), averaged over the K timed steps
    per_kernel = []
    for i, n in enumerate(SIZES):
        for d, nm in ((0, "fwd"), (1, "inv")):
            ms = statistics.fmean(evs[k][2 * i + d].elapsed_time(evs[k][2 * i + d + 1]) for k in range(K))
            per_kernel.append({"kernel": f"k_c2c<f32,N={n},split,{nm}>", "variant": plans[n].current_variant(d), "n": n, "dir": nm, "ms": ms,
                               "GBs": bytes_per_launch / ms / 1e6, "Mtransforms_s": (GIB // (8 * n)) / ms / 1e3})
    dom = max(per_kernel, key=lambda r: r["ms"])
    traffic = None
    try:
        prof = json.load(open(ROOT / "profiles" / "traffic.json"))
        traffic = prof.get(dom["kernel"])
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom["kernel"], "variant": dom["variant"], "achieved": dom["GBs"], "peak": peak, "unit": "GB/s",
                "frac": dom["GBs"] / peak, "traffic": traffic,
                "traffic_source": "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one committed ncu --set full "
                                  "capture of this kernel (not re-measured in this run)",
                "peak_source": peak_src,
                "peak_note": "the measured peak is torch's copy_ rate; a TMA-pipelined copy (tools/microbench/copy_pipe.cu) reaches 6.85 TB/s on the same board, so fractions slightly above 1.0 are possible",
                "algorithmic_bytes_per_launch": bytes_per_launch,
                "share_of_step": dom["ms"] / ms_per_step,
                "aggregate_GBs_per_gpu": agg_gbs / n_gpus, "aggregate_frac": agg_gbs / n_gpus / peak}
    for r in per_kernel:
        r["frac"] = round(r["GBs"] / peak, 3)
        r["ms"] = round(r["ms"], 4); r["GBs"] = round(r["GBs"], 1); r["Mtransforms_s"] = round(r["Mtransforms_s"], 2)
    for p in plans.values():
        p.destroy()

    # ---- the other BASELINE configs, device-resident, CUDA events around `reps` back-to-back launches each
    def time_launch(fn, reps=5, warmups=2):
        for _ in range(warmups):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / reps

    def row(name, n, ms, nbytes, units, variant, unit_name="Mtransforms_s"):
        return {"kernel": name, "n": n, "variant": variant, "ms": round(ms, 4), "GBs": round(nbytes / ms / 1e6, 1),
                "frac": round(nbytes / ms / 1e6 / peak, 3), unit_name: round(units / ms / 1e3, 2)}

    configs = {}
    r2c_rate = {}
    A1, B1 = (a_ptr, None), (b_ptr, None)
    rows_ = []
    for n in REAL_SIZES:                                      # configs[2]: rfft_split / irfft_split, B = 2^30/(4N)
        b = GIB // (4 * n)
        p = wf.Plan(C.R2C, C.F32, C.INTERLEAVED, n, b, local, flags)
        nb = p.algorithmic_bytes()
        ms = time_launch(lambda: p.exec_device(C.FORWARD, A1, B1, sptr))
        rows_.append(row(f"r2c<f32,N={n}>", n, ms, nb, b, p.current_variant(0)))
        r2c_rate[n] = rows_[-1]["Mtransforms_s"]
        ms = time_launch(lambda: p.exec_device(C.INVERSE, B1, A1, sptr))
        rows_.append(row(f"c2r<f32,N={n}>", n, ms, nb, b, p.current_variant(1)))
        p.destroy()
    configs["configs[2] r2c/c2r f32 (rfft_split/irfft_split), batch 2^30/(4N)"] = rows_
    rows_ = []
    for n in F64_SIZES:                                       # configs[3]: fft_combined / fft_real_combined, B = 2^30/(16N)
        b = GIB // (16 * n)
        p = wf.Plan(C.C2C, C.F64, C.INTERLEAVED, n, b, local, flags)
        nb = p.algorithmic_bytes()
        ms = time_launch(lambda: p.exec_device(C.FORWARD, A1, B1, sptr))
        rows_.append(row(f"c2c<f64,N={n},fwd>", n, ms, nb, b, p.current_variant(0)))
        ms = time_launch(lambda: p.exec_device(C.INVERSE, B1, A1, sptr))
        rows_.append(row(f"c2c<f64,N={n},inv>", n, ms, nb, b, p.current_variant(1)))
        p.destroy()
        p = wf.Plan(C.R2C, C.F64, C.INTERLEAVED, n, b, local, flags)
        nb = p.algorithmic_bytes()
        ms = time_launch(lambda: p.exec_device(C.FORWARD, A1, B1, sptr))
        rows_.append(row(f"r2c<f64,N={n}>", n, ms, nb, b, p.current_variant(0)))
        ms = time_launch(lambda: p.exec_device(C.INVERSE, B1, A1, sptr))
        rows_.append(row(f"c2r<f64,N={n}> (extension: the reference has no f64 inverse)", n, ms, nb, b, p.current_variant(1)))
        p.destroy()
    configs["configs[3] f64 c2c (fft_combined) + r2c (fft_real_combined), batch 2^30/(16N)"] = rows_
    rows_ = []
    for n in SIZES:                                           # transform 3: fft_stockham_f32_dual, interleaved
        b = GIB // (8 * n)
        p = wf.Plan(C.C2C, C.F32, C.INTERLEAVED, n, b, local, flags)
        nb = p.algorithmic_bytes()
        ms = time_launch(lambda: p.exec_device(C.FORWARD, A1, B1, sptr))
        rows_.append(row(f"c2c<f32,N={n},interleaved,fwd>", n, ms, nb, b, p.current_variant(0)))
        ms = time_launch(lambda: p.exec_device(C.INVERSE, B1, A1, sptr))
        rows_.append(row(f"c2c<f32,N={n},interleaved,inv>", n, ms, nb, b, p.current_variant(1)))
        p.destroy()
    configs["interleaved c2c f32 (fft_stockham_f32_dual), batch 2^30/(8N)"] = rows_
    rows_ = []
    stft_samples = 1 << 26                                    # 256 MiB of samples; hop N/4 -> ~512 MiB of dB output
    for n in STFT_SIZES:
        sp = wf.Spectrogram(stft_samples, n, n // 4, "hann", flags=flags, device=local)
        nb = sp.algorithmic_bytes()
        ms = time_launch(lambda: sp.run_device(a_ptr, b_ptr, sptr))
        r = row(f"stft<f32,N={n},hop=N/4,hann,dB>", n, ms, nb, sp.numFrames, "fused", "Mframes_s")
        # the spectrogram's HBM bytes are a third of its r2c work (frames overlap 4x, half the bins' bytes leave): its
        # yardstick is the plain r2c kernel's rows/s at the same N, measured a few lines up
        plain = r2c_rate.get(n)
        if plain:
            r["r2c_Mrows_s"] = plain
            r["frames_per_r2c_row"] = round(r["Mframes_s"] / plain, 3)
        rows_.append(r)
        sp.dispose()
    configs["STFT front-end (playground/src/spectrogram.js loop fused), 2^26 samples, hop N/4"] = rows_
    del A32, a_re, a_im, Bv, b_re, b_im, arena
    torch.cuda.empty_cache()
    if world > 1:                                             # configs[4]: c2c N=4096, 8 GiB total, STRONG-scaled over the ranks
        from watfft_b200.sharding import partition
        total = 262144
        lo, hi = partition(total, world, rank)
        p = wf.Plan(C.C2C, C.F32, C.SPLIT, 4096, hi - lo, local, flags)
        pre = torch.empty((hi - lo) * 4096, dtype=torch.float32, device=dev).uniform_(-1, 1, generator=g)
        pim = torch.empty((hi - lo) * 4096, dtype=torch.float32, device=dev).uniform_(-1, 1, generator=g)
        P = (pre.data_ptr(), pim.data_ptr())
        fn = lambda: (p.exec_device(C.FORWARD, P, P, sptr), p.exec_device(C.INVERSE, P, P, sptr))   # in place, like the contexts
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        reps = 5
        for _ in range(reps):
            fn()
        e1.record(stream)
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1) / reps)
        configs["configs[4] c2c f32 split N=4096, 262144 rows (8 GiB) sharded over the ranks, fft+ifft in place"] = {
            "scaling": "strong", "ranks": world, "rows_per_rank": hi - lo, "ms_fft_plus_ifft": round(ms, 4),
            "Mtransforms_s_total": round(2 * total / ms / 1e3, 2),
            "GBs_per_gpu": round(2 * (hi - lo) * 4096 * 16 / ms / 1e6, 1),
            "frac": round(2 * (hi - lo) * 4096 * 16 / ms / 1e6 / peak, 3)}
        p.destroy()
        del pre, pim
        torch.cuda.empty_cache()

    # ---- configs[0]: c2c f32 split N=1024, batch 1 -- the reference's own call shape (index.js:84-89)
    sys.path.insert(0, str(ROOT / "oracle"))
    import oracle as om
    om.build()
    orc = om.Oracle()
    lat = {}
    if rank == 0:
        t_create = []
        for _ in range(5):
            t0 = time.perf_counter()
            c = wf.createFFTf32Split(1024)
            t_create.append((time.perf_counter() - t0) * 1e3)
            c.dispose()
        ctx = wf.createFFTf32Split(1024)
        re_in, im_in = om.bench_complex_inputs(1024)          # mulberry32, seed = N (benchmarks/lib/wat-contexts.js:34-50)
        re_in, im_in = re_in.astype(np.float32), im_in.astype(np.float32)

        def one_call():
            ctx.getRealBuffer()[:] = re_in                      # input staging is charged, like bench() (:125-129)
            ctx.getImagBuffer()[:] = im_in
            ctx.forward()

        def lat_us(iters=2000):
            for _ in range(200):
                one_call()
            ts = []
            for _ in range(iters):
                t0 = time.perf_counter_ns()
                one_call()
                ts.append(time.perf_counter_ns() - t0)
            ts.sort()
            return ts[len(ts) // 2] / 1e3, ts[len(ts) // 10] / 1e3, ts[(len(ts) * 99) // 100] / 1e3
        med, p10, p99 = lat_us()
        path = ctx.plan.last_path()
        o_re, o_im = orc.fft_split_f32(re_in, im_in)
        err = float(np.max(np.abs(np.r_[ctx.getRealBuffer() - o_re, ctx.getImagBuffer() - o_im])) /
                    np.linalg.norm(np.r_[re_in, im_in]))
        assert err <= 2e-6 * 10, f"configs[0] parity: {err}"
        truth = om.dft(re_in.astype(np.float64) + 1j * im_in.astype(np.float64))
        err_dft = float(np.max(np.abs((ctx.getRealBuffer() + 1j * ctx.getImagBuffer()) - truth)) / np.linalg.norm(np.r_[re_in, im_in]))
        ctx.plan.set_option(C.OPT_MAPPED_MAX_BYTES, 0)          # the copy path, for comparison
        med_staged, _, _ = lat_us(500)
        ctx.dispose()
        lat = {"workload": "configs[0]: c2c f32 split N=1024, batch 1, createFFTf32Split(1024).forward() incl. writing the input views",
               "latency_us": round(med, 2), "latency_us_p10": round(p10, 2), "latency_us_p99": round(p99, 2),
               "path": {C.PATH_MAPPED: "zero-copy (one kernel on the mapped host buffers, one sync)", C.PATH_STAGED: "staged copies",
                        C.PATH_PIPELINED: "pipelined copies"}.get(path, str(path)),
               "latency_us_copy_path": round(med_staged, 2),
               "plan_create_ms": round(statistics.median(t_create), 3),
               "max_err_over_norm_vs_oracle": err, "max_err_over_norm_vs_f64_dft": err_dft,
               "Mtransforms_s": round(1.0 / med, 4),
               "measured_through": "the Python mirror of the context API (ctypes call + two numpy view writes per call included)"}
        # the same call sequence from C (tools/native/abi_latency.c): what the N-API shim sees, no host-language overhead
        try:
            exe = ROOT / "tools" / "native" / "abi_latency"
            out = subprocess.run([str(exe), "1024", "1", "5000"], capture_output=True, text=True, timeout=120)
            lat["native_c_abi"] = json.loads(out.stdout.strip().splitlines()[-1])
        except Exception as ex:                                 # the tool is optional evidence, never a reason to fail the bench
            lat["native_c_abi"] = {"unavailable": repr(ex)}

    # ---- pinned-copy ceiling of the host link (the roofline of the e2e number).  Every rank runs each phase -- H2D alone,
    # D2H alone, both at once -- at the SAME moment: a barrier in front of every phase (round 1's probe let the ranks drift
    # through the phases on their own and over-stated the multi-GPU ceiling).  Per phase and direction: the slowest rank's
    # rate and the sum of the ranks' rates.  The e2e time is a max over ranks, so `world x slowest` is the ceiling it can reach.
    probe = ctypes.c_void_p()
    PROBE_BYTES, PROBE_ITERS = 256 << 20, 8
    C.check(lib.wfb_pcie_probe_open(local, PROBE_BYTES, ctypes.byref(probe)))
    sec = (ctypes.c_double * 2)()
    pcie = {}
    for name, dirs in (("alone_h2d", 1), ("alone_d2h", 2), ("duplex", 3)):
        barrier()
        C.check(lib.wfb_pcie_probe_run(probe, dirs, PROBE_ITERS, sec))
        for bit, key, t in ((1, "h2d", sec[0]), (2, "d2h", sec[1])):
            if not dirs & bit:
                continue
            rate = PROBE_ITERS * PROBE_BYTES / t / 1e9
            if world > 1:
                tt = torch.tensor([rate, -rate], device=dev, dtype=torch.float64)
                tsum = tt.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
                tmax = tt.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
                lo, total = -float(tmax[1]), float(tsum[0])
            else:
                lo = total = rate
            pcie[("duplex_" if dirs == 3 else "alone_") + key] = {"slowest_rank": round(lo, 2), "sum": round(total, 2)}
    lib.wfb_pcie_probe_close(probe)
    barrier()

    # ---- e2e: the headline workload through the public context API with pinned HOST buffers --------
    rng = np.random.default_rng(99 + rank)
    block = rng.uniform(-1, 1, 1 << 24).astype(np.float32)     # 64 MiB of random values, tiled over the host buffers

    def fill(view):
        for off in range(0, view.size, block.size):
            m = min(block.size, view.size - off)
            view[off: off + m] = block[:m]

    e2e_ms = 0.0
    h2d = d2h = 0
    e2e_iters = max(1, min(K, 2))
    e2e_per_n = {}
    worst = 0.0
    for n in SIZES:
        b = GIB // (8 * n)
        ctx = wf.createFFTf32Split(n, batch=b, device=local)
        re, im = ctx.getRealBuffer(), ctx.getImagBuffer()
        fill(re); fill(im[::-1])                            # (the reversed view decorrelates the planes)
        pick = sorted({0, 1, b // 2, b - 1})
        keep = {r: (re[r * n:(r + 1) * n].copy(), im[r * n:(r + 1) * n].copy()) for r in pick}
        ctx.forward()                                       # warm-up (also pages in the pinned buffers) + parity sample
        for r in pick:
            o_re, o_im = orc.fft_split_f32(*keep[r])
            e = float(np.max(np.abs(np.r_[re[r * n:(r + 1) * n] - o_re, im[r * n:(r + 1) * n] - o_im])) / np.linalg.norm(np.r_[keep[r][0], keep[r][1]]))
            worst = max(worst, e / (2e-6 * math.log2(n)))
            assert e <= 2e-6 * math.log2(n), f"e2e parity N={n} row {r}: {e}"
        ctx.inverse()
        for r in pick:
            assert float(np.max(np.abs(np.r_[re[r * n:(r + 1) * n] - keep[r][0], im[r * n:(r + 1) * n] - keep[r][1]]))) < 1e-4
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_iters):
            ctx.forward()                                   # H2D 1 GiB, kernel, D2H 1 GiB, sync
            ctx.inverse()
        torch.cuda.synchronize()
        dt = max_over_ranks((time.perf_counter() - t0) / e2e_iters)
        e2e_ms += dt * 1e3
        e2e_per_n[str(n)] = round(dt * 1e3, 2)
        h2d += 2 * GIB
        d2h += 2 * GIB
        for r in pick:                                      # the timed calls round-tripped the data as well
            assert float(np.max(np.abs(re[r * n:(r + 1) * n] - keep[r][0]))) < 1e-3
        ctx.dispose()
    e2e_value = n_gpus * transforms_per_step_gpu / (e2e_ms * 1e-3)
    e2e_dir_gbs = h2d / (e2e_ms * 1e-3) / 1e9                 # per GPU, per direction (both run at once)

    # companions with fewer PCIe bytes per transform: r2c f32 and the fused STFT, N = 1024 and 4096
    comp = {}
    for n in (1024, 4096):
        b = GIB // (4 * n)
        ctx = wf.createRFFTf32(n, batch=b, device=local)
        x = ctx.getInputBuffer()
        fill(x)
        keep0 = x[:n].copy()
        ctx.forward()
        e = float(np.max(np.abs(ctx.getOutputBuffer()[: n + 2] - orc.rfft_split_f32(keep0))) / np.linalg.norm(keep0))
        assert e <= 2e-6 * math.log2(n), f"e2e r2c parity N={n}: {e}"
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_iters):
            ctx.forward()
        dt = max_over_ranks((time.perf_counter() - t0) / e2e_iters)
        comp[f"r2c_f32_N{n}"] = {"api": "createRFFTf32(n, batch).forward()", "batch_per_gpu": b, "ms": round(dt * 1e3, 2),
                                 "Mtransforms_s": round(n_gpus * b / dt / 1e6, 2),
                                 "h2d_bytes": n_gpus * b * n * 4, "d2h_bytes": n_gpus * b * (n + 2) * 4}
        ctx.dispose()
        ns = 1 << 26
        sp = wf.Spectrogram(ns, n, n // 4, "hann", device=local)
        fill(sp.getInputBuffer())
        sp.run()
        small = om.spectrogram_reference(sp.getInputBuffer()[: n + 3 * (n // 4)], n, n // 4, rfft=orc.rfft_split_f32)
        assert float(np.max(np.abs(sp.getOutputBuffer()[:4] - small))) < 2e-4
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_iters):
            sp.run()
        dt = max_over_ranks((time.perf_counter() - t0) / e2e_iters)
        comp[f"stft_N{n}_hop{n // 4}"] = {"api": "Spectrogram(samples, n, n/4).run()", "frames_per_gpu": sp.numFrames, "ms": round(dt * 1e3, 2),
                                          "Mframes_s": round(n_gpus * sp.numFrames / dt / 1e6, 2),
                                          "h2d_bytes": n_gpus * ns * 4, "d2h_bytes": n_gpus * sp.numFrames * sp.numBins * 4}
        sp.dispose()

    # ---- configs[4] end to end from ONE process: 262144 rows of N=4096 (8 GiB) in pinned host memory, cut into grains that
    # the GPUs pull (watfft_b200.sharding.ShardedSplitFFT, schedule="dynamic"); rank 0 drives the very GPUs the ranks used,
    # the other ranks wait at the barrier below with idle devices
    sharded = None
    if world > 1 and rank == 0 and not args.no_sharded_e2e:
        try:
            from watfft_b200.sharding import ShardedSplitFFT
            devs = [rank_device(i, world, visible, os.environ.get("WFB_BENCH_DEVICE_ORDER", "spread")) for i in range(world)]
            total, n4 = 262144, 4096
            sh = ShardedSplitFFT(n4, total, devs, schedule="dynamic", grain_bytes=32 << 20, workers_per_device=2)
            fill(sh.real.reshape(-1)); fill(sh.imag.reshape(-1)[::-1])
            pick = sorted({0, 1, total // 2, total - 1})
            keep = {r: (sh.real[r].copy(), sh.imag[r].copy()) for r in pick}
            sh.run(); sh.run(inverse=True)                     # warm-up: contexts, tables, first touch
            t0 = time.perf_counter(); sh.run(); t_f = time.perf_counter() - t0
            counts = list(sh.last_counts)
            for r in pick:
                o_re, o_im = orc.fft_split_f32(*keep[r])
                e = float(np.max(np.abs(np.r_[sh.real[r] - o_re, sh.imag[r] - o_im])) / np.linalg.norm(np.r_[keep[r][0], keep[r][1]]))
                assert e <= 2e-6 * 12, f"sharded e2e parity row {r}: {e}"
            t0 = time.perf_counter(); sh.run(inverse=True); t_i = time.perf_counter() - t0
            for r in pick:
                assert float(np.max(np.abs(sh.real[r] - keep[r][0]))) < 1e-3
            nbytes = total * n4 * 8
            sharded = {"workload": "configs[4]: c2c f32 split N=4096, 262144 rows (8 GiB) in pinned host memory, ONE process, the GPUs pull 32 MiB grains "
                                   "(ShardedSplitFFT schedule=dynamic, 2 host threads per GPU), forward then inverse, in place",
                       "devices": devs, "ms_forward": round(t_f * 1e3, 1), "ms_inverse": round(t_i * 1e3, 1),
                       "Mtransforms_s": round(2 * total / (t_f + t_i) / 1e6, 2),
                       "GBs_per_direction_total": round(2 * nbytes / (t_f + t_i) / 1e9, 2),
                       "frac_of_duplex_sum": round(2 * nbytes / (t_f + t_i) / 1e9 / max(1e-9, min(pcie["duplex_h2d"]["sum"], pcie["duplex_d2h"]["sum"])), 3),
                       "grains_per_device_forward": counts,
                       "parity": "rows 0, 1, B/2, B-1 against the oracle after forward, against the input after inverse"}
            sh.dispose()
        except AssertionError:
            raise
        except Exception as ex:                             # an allocation failure here must not cost the run its headline
            sharded = {"error": repr(ex)}
    if world > 1 and not args.no_sharded_e2e:
        # the other ranks wait on the rendezvous store (host side): an NCCL barrier would park a spinning kernel on the
        # GPUs rank 0 is driving
        try:
            store = dist.distributed_c10d._get_default_store()
            if rank == 0:
                store.set("wfb_sharded_done", "1")
            else:
                store.wait(["wfb_sharded_done"])
        except Exception:
            pass
    barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    devices = {"visible": visible, "rank0_device": local, "order": "spread (rank i -> GPU i*visible/world)" if spread else "rank i -> GPU i"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": warm, "devices": devices,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(n_gpus),
        "achieved_GBs": agg_gbs,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * n_gpus, "d2h_bytes_per_step": d2h * n_gpus,
                "ms_per_step": e2e_ms, "ms_per_n": e2e_per_n,
                "api": "createFFTf32Split(n, batch).forward()/inverse() on pinned host buffers, random inputs",
                "parity": f"rows 0, 1, B/2, B-1 of every size checked against the oracle after forward() (worst = {worst:.3f} of the "
                          "2e-6*log2(N) bound) and against the input after inverse()",
                "GBs_per_direction_per_gpu": round(e2e_dir_gbs, 2),
                "pcie_peak_GBs": dict({"what": f"plain cudaMemcpyAsync, {PROBE_ITERS} x {PROBE_BYTES >> 20} MiB pinned copies per direction, CUDA-event timed, "
                                               "every rank in the same phase at the same time (barrier per phase); GB/s per direction: the slowest "
                                               "rank's rate and the sum over the ranks"}, **pcie),
                "frac": round(e2e_dir_gbs * n_gpus / max(1e-9, min(pcie["duplex_h2d"]["sum"], pcie["duplex_d2h"]["sum"])), 3),
                "frac_of_slowest_rank_ceiling": round(e2e_dir_gbs / max(1e-9, min(pcie["duplex_h2d"]["slowest_rank"], pcie["duplex_d2h"]["slowest_rank"])), 3),
                "frac_note": "achieved bytes per direction / the slower direction of the concurrent duplex pinned-copy ceiling: `frac` against the sum "
                             "over ranks, `frac_of_slowest_rank_ceiling` against n_gpus x the slowest rank (the e2e time is a max over ranks, and the "
                             "host fabric does not share its bandwidth evenly).  Every transform crosses the link once each way, so this is the "
                             "roofline of the e2e number; tools/microbench/pcie_peak.cu measures the same ceiling from one C process "
                             "(profiles/r02_pcie.md)",
                "companions": comp},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "per_step_ms": {"first": round(step_ms[0], 4), "median": round(statistics.median(step_ms), 4), "last": round(step_ms[-1], 4),
                        "note": "rank 0; every rank holds its GPU under load for 0.75 s right up to the start barrier (sustained clocks at every N)"},
        "per_kernel": per_kernel,
        "configs": configs,
        "latency": lat,
    }
    if sharded:
        line["e2e"]["one_process_sharded"] = sharded
    if n_gpus == 1 and not args.no_cpu_baseline:
        cpu = CpuReference()
        line["cpu_baseline"] = cpu.baseline_block(steps=5, warmup=1)
        if cpu.kind == "reference":
            extra = {}
            extra["r2c_f32"] = {str(n): round(cpu.rate("real_f32", n, count=2, min_s=0.1) / 1e6, 3) for n in REAL_SIZES}
            extra["c2r_f32"] = {str(n): round(cpu.rate("real_f32", n, True, count=2, min_s=0.1) / 1e6, 3) for n in REAL_SIZES}
            extra["c2c_f64_fwd"] = {str(n): round(cpu.rate("c2c_f64", n, count=2, min_s=0.1) / 1e6, 3) for n in F64_SIZES}
            extra["r2c_f64"] = {str(n): round(cpu.rate("r2c_f64", n, count=2, min_s=0.1) / 1e6, 3) for n in F64_SIZES}
            extra["c2c_f32_interleaved_fwd"] = {str(n): round(cpu.rate("c2c_il", n, count=2, min_s=0.1) / 1e6, 3) for n in SIZES}
            extra["stft_hopN4_Mframes_s"] = {str(n): round(cpu.stft_rate(n, n // 4, min_s=0.1) / 1e6, 3) for n in STFT_SIZES}
            line["cpu_baseline"]["other_transforms_Mtransforms_s"] = extra
            if lat:
                lat["cpu_reference_us_per_call"] = line["cpu_baseline"]["anchor_1thread_n1024"]["us_per_call"]
        cpu.close()
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


_REAL_STDOUT = None


def quiet_stdout():
    """stdout carries exactly ONE JSON line: libraries that chat on fd 1 (NCCL prints its version banner there on
    the first collective, whatever NCCL_DEBUG_FILE says) are sent to stderr for the rest of the run."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded-e2e", action="store_true", help="skip the one-process configs[4] end-to-end leg (N > 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a seeded sample of what the last timed headline step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU headline path (--impl ours)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not (args.impl == "ours" and args.gpus > 1 and world == 1):      # (the torchrun re-launch prints through its ranks)
        quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29541", __file__, "--gpus", str(args.gpus),
               "--steps", str(args.steps), "--warmup", str(args.warmup)]
        if args.dump_outputs:
            cmd += ["--dump-outputs", args.dump_outputs]
        return subprocess.call(cmd)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
