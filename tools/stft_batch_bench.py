"""Batched STFT / inverse STFT throughput on one GPU: B equal-length clips in one launch (Spectrogram(batch=B)), against
(b) the same clips as a loop of per-clip launches on one reused single-signal handle and (c) one long signal with the
same total frame count (the rate the kernels reach when nothing bounds their tiles).

Workloads: clips of 16 000 and 160 000 samples, N in {256, 512, 1024, 2048}, hop N/4, hann, 2^26 samples in all (more
than L2: the 256 MiB input alone is twice its size), everything device-resident, CUDA events around --iters launches
(--loop-iters passes of the per-clip loop) after --warmup.  A seeded sample of (a)'s rows is checked bit for bit
against per-clip runs.  One end-to-end row: Spectrogram(batch=B).run() from its pinned host buffers (H2D, kernel, D2H,
sync), host clock.  Prints one JSON line and writes it to DIR/stft_batch_bench.json, with the card name, power limit
and SM clock read in the same run.

    python tools/stft_batch_bench.py --out DIR [--iters 20] [--loop-iters 3] [--warmup 3]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, sm, smax = [s.strip() for s in q[0].split(",")]
    return {"gpu": name, "power_limit": power, "sm_clock": sm, "sm_clock_max": smax}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for stft_batch_bench.json")
    ap.add_argument("--samples", type=int, default=1 << 26)
    ap.add_argument("--clips", default="16000,160000", help="clip lengths in samples")
    ap.add_argument("--sizes", default="256,512,1024,2048")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--loop-iters", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--check-rows", type=int, default=8, help="clips of (a) checked bit for bit against per-clip runs")
    a = ap.parse_args()

    import torch
    import watfft_b200 as wf
    C = wf._cabi
    flags = C.PLAN_NO_HOST_BUFFERS | C.PLAN_NO_DEVICE_BUFFERS
    # a stream of our own: the legacy default stream's handle is 0, which the library reads as "the handle's stream"
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream

    def time_launch(fn, iters):
        for _ in range(a.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(iters):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / iters

    gen = torch.Generator(device="cuda").manual_seed(0)
    rng = np.random.default_rng(0)
    rows, mismatches = [], 0
    for clip in [int(s) for s in a.clips.split(",")]:
        batch = a.samples // clip
        x = torch.rand(batch * clip, dtype=torch.float32, device="cuda", generator=gen) * 2 - 1
        for n in [int(s) for s in a.sizes.split(",")]:
            hop, bins = n // 4, n // 2 + 1
            row = {"clip": clip, "batch": batch, "n": n, "hop": hop}
            for mode in ("db", "complex"):
                vw = 2 if mode == "complex" else 1
                bat = wf.Spectrogram(clip, n, hop, "hann", mode=mode, flags=flags, batch=batch)
                one = wf.Spectrogram(clip, n, hop, "hann", mode=mode, flags=flags)
                frames = bat.numFrames
                total = batch * frames
                lng = wf.Spectrogram((total - 1) * hop + n, n, hop, "hann", mode=mode, flags=flags)
                assert lng.numFrames == total
                xl = torch.rand((total - 1) * hop + n, dtype=torch.float32, device="cuda", generator=gen) * 2 - 1
                out = torch.empty(total * bins * vw, dtype=torch.float32, device="cuda")
                rowf = frames * bins * vw                                  # floats per clip of output
                torch.cuda.synchronize()

                def loop_fwd():
                    for b in range(batch):
                        one.run_device(x.data_ptr() + 4 * b * clip, out.data_ptr() + 4 * b * rowf, sptr)

                ta = time_launch(lambda: bat.run_device(x.data_ptr(), out.data_ptr(), sptr), a.iters)
                tb = time_launch(loop_fwd, a.loop_iters)
                tc = time_launch(lambda: lng.run_device(xl.data_ptr(), out.data_ptr(), sptr), a.iters)
                # (a)'s rows against per-clip runs into their own (16-byte aligned) buffers: the same kernel either way
                bat.run_device(x.data_ptr(), out.data_ptr(), sptr)
                tmp = torch.empty(rowf, dtype=torch.float32, device="cuda")
                for b in sorted(set(rng.integers(0, batch, a.check_rows).tolist()) | {0, batch - 1}):
                    one.run_device(x.data_ptr() + 4 * b * clip, tmp.data_ptr(), sptr)
                    if not torch.equal(tmp.view(torch.int32), out[b * rowf:(b + 1) * rowf].view(torch.int32)):
                        mismatches += 1
                key = "fwd_" + mode
                row[key] = {"frames": total, "a_ms": round(ta, 4), "b_ms": round(tb, 3), "c_ms": round(tc, 4),
                            "a_Mframes_s": round(total / ta / 1e3, 2), "b_Mframes_s": round(total / tb / 1e3, 2),
                            "c_Mframes_s": round(total / tc / 1e3, 2), "a_over_c": round(tc / ta, 3),
                            "a_over_b": round(tb / ta, 2)}
                if mode == "complex":
                    spec = out                                             # the forward's complex frames
                    back = torch.empty(batch * clip, dtype=torch.float32, device="cuda")
                    backl = torch.empty_like(xl)

                    def loop_inv():
                        for b in range(batch):
                            one.inverse_device(spec.data_ptr() + 4 * b * rowf, back.data_ptr() + 4 * b * clip, sptr)

                    ta = time_launch(lambda: bat.inverse_device(spec.data_ptr(), back.data_ptr(), sptr), a.iters)
                    tb = time_launch(loop_inv, a.loop_iters)
                    tc = time_launch(lambda: lng.inverse_device(spec.data_ptr(), backl.data_ptr(), sptr), a.iters)
                    bat.inverse_device(spec.data_ptr(), back.data_ptr(), sptr)
                    tmp = torch.empty(clip, dtype=torch.float32, device="cuda")
                    for b in sorted(set(rng.integers(0, batch, a.check_rows).tolist()) | {0, batch - 1}):
                        one.inverse_device(spec.data_ptr() + 4 * b * rowf, tmp.data_ptr(), sptr)
                        if not torch.equal(tmp.view(torch.int32), back[b * clip:(b + 1) * clip].view(torch.int32)):
                            mismatches += 1
                    row["inv"] = {"frames": total, "a_ms": round(ta, 4), "b_ms": round(tb, 3), "c_ms": round(tc, 4),
                                  "a_Mframes_s": round(total / ta / 1e3, 2), "b_Mframes_s": round(total / tb / 1e3, 2),
                                  "c_Mframes_s": round(total / tc / 1e3, 2), "a_over_c": round(tc / ta, 3),
                                  "a_over_b": round(tb / ta, 2)}
                    del back, backl
                for s in (bat, one, lng):
                    s.dispose()
                del xl, out
                torch.cuda.empty_cache()
            rows.append(row)
        del x

    # end to end from pinned host memory: one batched run() of 16 000-sample clips at N = 1024
    clip, n = 16000, 1024
    batch = a.samples // clip
    sp = wf.Spectrogram(clip, n, n // 4, "hann", batch=batch)
    sp.getInputBuffer()[:] = rng.uniform(-1, 1, (batch, clip)).astype(np.float32)
    for _ in range(a.warmup):
        sp.run()
    t0 = time.perf_counter()
    for _ in range(a.iters):
        sp.run()
    dt = (time.perf_counter() - t0) / a.iters
    pcie = 4 * batch * clip + 4 * batch * sp.numFrames * sp.numBins
    e2e = {"api": "Spectrogram(batch=B).run()", "clip": clip, "batch": batch, "n": n, "hop": n // 4,
           "ms": round(dt * 1e3, 3), "Mframes_s": round(batch * sp.numFrames / dt / 1e6, 2),
           "pcie_GBs": round(pcie / dt / 1e9, 2)}
    sp.dispose()

    res = {"bench": "stft_batch", "samples": a.samples, "window": "hann", "hop": "N/4", **card(),
           "bitwise_mismatches": mismatches, "rows": rows, "end_to_end": e2e}
    line = json.dumps(res)
    print(line)
    outdir = Path(a.out)
    outdir.mkdir(parents=True, exist_ok=True)
    (outdir / "stft_batch_bench.json").write_text(line + "\n")
    if mismatches:
        sys.exit(f"{mismatches} sampled rows differ from per-clip runs")


if __name__ == "__main__":
    main()
