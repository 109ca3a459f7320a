"""Inverse STFT throughput on one GPU: the fused kernel (Spectrogram.inverse_device, k_istft) against the plain c2r
kernel at the same N and against the path a user has without it (the library's batched c2r into [F][N], then torch
fold for the overlap-add and the division by the window-square sum).

Workload: 2^26 samples, hann, hop = N/4, N in {256 .. 4096}, everything device-resident, CUDA events around
--iters launches after --warmup.  Algorithmic bytes of the fused inverse: F*(N+2)*4 read + num_samples*4 written.
Prints one JSON line and writes it to DIR/istft_bench.json, with the card name, power limit and SM clock read in the
same run.

    python tools/istft_bench.py --out DIR [--iters 20] [--warmup 3]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, sm, smax = [s.strip() for s in q[0].split(",")]
    return {"gpu": name, "power_limit": power, "sm_clock": sm, "sm_clock_max": smax}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for istft_bench.json")
    ap.add_argument("--samples", type=int, default=1 << 26)
    ap.add_argument("--sizes", default="256,512,1024,2048,4096")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()

    import torch
    import watfft_b200 as wf
    C = wf._cabi
    stream = torch.cuda.current_stream()
    sptr = stream.cuda_stream

    def time_launch(fn):
        for _ in range(a.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(a.iters):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / a.iters

    # the copy rate of this run: torch copy_ of 1 GiB (read + write)
    src = torch.empty(1 << 28, dtype=torch.float32, device="cuda").uniform_()
    dst = torch.empty_like(src)
    copy_ms = time_launch(lambda: dst.copy_(src))
    copy_gbs = 2 * src.numel() * 4 / copy_ms / 1e6
    del src, dst

    ns = a.samples
    rows = []
    gen = torch.Generator(device="cuda").manual_seed(0)
    for n in [int(s) for s in a.sizes.split(",")]:
        hop, bins = n // 4, n // 2 + 1
        sp = wf.Spectrogram(ns, n, hop, "hann", mode="complex", flags=C.PLAN_NO_HOST_BUFFERS)
        frames = sp.numFrames
        spec = torch.randn((frames, bins, 2), dtype=torch.float32, device="cuda", generator=gen)
        out = torch.empty(ns, dtype=torch.float32, device="cuda")
        fused_ms = time_launch(lambda: sp.inverse_device(spec.data_ptr(), out.data_ptr(), sptr))
        nbytes = frames * (n + 2) * 4 + ns * 4

        # plain c2r: the same frames as a batch of rows, [F][N+2] -> [F][N]
        plan = wf.Plan(C.R2C, C.F32, C.INTERLEAVED, n, frames, 0, C.PLAN_NO_HOST_BUFFERS | C.PLAN_NO_DEVICE_BUFFERS)
        y = torch.empty((frames, n), dtype=torch.float32, device="cuda")
        c2r_ms = time_launch(lambda: plan.exec_device(C.INVERSE, (spec.data_ptr(), None), (y.data_ptr(), None), sptr))

        # composed: batched c2r, window, fold (overlap-add), division by the fold of the squared window
        w = torch.hann_window(n, periodic=False, dtype=torch.float64).float().cuda()
        den = torch.nn.functional.fold((w * w).expand(frames, n).T.unsqueeze(0), (1, (frames - 1) * hop + n),
                                       (1, n), stride=(1, hop)).flatten()

        def composed():
            plan.exec_device(C.INVERSE, (spec.data_ptr(), None), (y.data_ptr(), None), sptr)
            num = torch.nn.functional.fold((y * w).T.unsqueeze(0), (1, (frames - 1) * hop + n), (1, n),
                                           stride=(1, hop)).flatten()
            out[: num.numel()] = torch.where(den >= 1e-11, num / den, torch.zeros_like(num))
            out[num.numel():] = 0
        composed_ms = time_launch(composed)
        # the fused result against the composed one (same contract, different rounding order)
        sp.inverse_device(spec.data_ptr(), out.data_ptr(), sptr)
        fused = out.clone()
        composed()
        diff = float((fused - out).abs().max())
        rows.append({"n": n, "hop": hop, "frames": frames, "fused_ms": round(fused_ms, 4),
                     "Mframes_s": round(frames / fused_ms / 1e3, 2), "GBs": round(nbytes / fused_ms / 1e6, 1),
                     "copy_frac": round(nbytes / fused_ms / 1e6 / copy_gbs, 3),
                     "c2r_ms": round(c2r_ms, 4), "c2r_Mrows_s": round(frames / c2r_ms / 1e3, 2),
                     "frames_per_c2r_row": round(c2r_ms / fused_ms, 3),
                     "composed_ms": round(composed_ms, 4), "speedup_vs_composed": round(composed_ms / fused_ms, 2),
                     "max_abs_diff_vs_composed": diff})
        del plan, y, spec, out
        sp.dispose()
        torch.cuda.empty_cache()
    res = {"bench": "istft", "samples": ns, "window": "hann", "hop": "N/4", "copy_GBs": round(copy_gbs, 1), **card(),
           "rows": rows}
    line = json.dumps(res)
    print(line)
    outdir = Path(a.out)
    outdir.mkdir(parents=True, exist_ok=True)
    (outdir / "istft_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
