"""Filterbank (mel) spectrogram throughput on one GPU, device-resident: Spectrogram(mode="filterbank") against the dB
spectrogram of the same geometry (the same route and kernel family) and against the torch path a user would write
otherwise: torch.stft(center=False) with the library's f32 window, then abs()**2 @ F.T, then the log.

Workloads: N in {512, 1024, 2048}, hop N/4, hann; 2^26 samples as one signal, and 4194 clips of 16 000 samples (both
more than L2: the 256 MiB input alone is twice its size); 80 and 128 mel filters (htk, 16 kHz); power 2; linear and
log10 output (log10(max(v, 1e-10))).  CUDA events around --iters launches after --warmup, on a stream of our own.
Beside each row: the max difference between the library's and the torch path's outputs (relative to the largest
value for linear output, absolute for log10).  Prints one JSON line and writes it to DIR/stft_fb_bench.json, with the
card name, power limit and SM clock read in the same run.

    python tools/stft_fb_bench.py --out DIR [--iters 20] [--warmup 3]
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))
sys.path.insert(0, str(ROOT / "tools"))

from stft_batch_bench import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for stft_fb_bench.json")
    ap.add_argument("--samples", type=int, default=1 << 26, help="samples of the one-signal workload")
    ap.add_argument("--clips", type=int, default=4194)
    ap.add_argument("--clip", type=int, default=16000)
    ap.add_argument("--sizes", default="512,1024,2048")
    ap.add_argument("--mels", default="80,128")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()

    import torch
    import oracle as om
    import watfft_b200 as wf
    C = wf._cabi
    flags = C.PLAN_NO_HOST_BUFFERS | C.PLAN_NO_DEVICE_BUFFERS
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
    rows = []
    for workload, batch, ns in (("long", None, a.samples), ("clips", a.clips, a.clip)):
        nb = batch or 1
        x = torch.rand(nb * ns, dtype=torch.float32, device="cuda", generator=gen) * 2 - 1
        for n in [int(s) for s in a.sizes.split(",")]:
            hop = n // 4
            db = wf.Spectrogram(ns, n, hop, "hann", flags=flags, batch=batch)
            frames = db.numFrames
            total = nb * frames
            out_db = torch.empty(total * db.numBins, dtype=torch.float32, device="cuda")
            t_db = time_launch(lambda: db.run_device(x.data_ptr(), out_db.data_ptr(), sptr), a.iters)
            db.dispose()
            del out_db
            win = torch.from_numpy(om.window_function("hann", n).astype(np.float32)).cuda()
            xt = x.view(nb, ns)
            for nm in [int(s) for s in a.mels.split(",")]:
                F = wf.mel_filterbank(n, 16000, nm)
                Ft = torch.from_numpy(F).cuda()
                for log in (None, "log10"):
                    sp = wf.Spectrogram(ns, n, hop, "hann", mode="filterbank", filters=F, power=2, log=log, flags=flags,
                                        batch=batch)
                    out = torch.empty(total * nm, dtype=torch.float32, device="cuda")
                    t_fb = time_launch(lambda: sp.run_device(x.data_ptr(), out.data_ptr(), sptr), a.iters)
                    sp.dispose()

                    def torch_path():
                        s = torch.stft(xt, n, hop_length=hop, win_length=n, window=win, center=False,
                                       return_complex=True)
                        v = s.abs().pow(2).transpose(1, 2) @ Ft.T
                        return torch.log10(torch.clamp(v, min=1e-10)) if log else v

                    t_torch = time_launch(torch_path, max(3, a.iters // 4))
                    ref = torch_path().reshape(-1)
                    torch.cuda.synchronize()
                    d = (out - ref).abs().max().item()
                    diff = d if log else d / ref.abs().max().item()
                    rows.append({"workload": workload, "batch": nb, "num_samples": ns, "n": n, "hop": hop,
                                 "n_mels": nm, "log": log or "linear", "frames": total,
                                 "fb_ms": round(t_fb, 4), "fb_Mframes_s": round(total / t_fb / 1e3, 2),
                                 "db_Mframes_s": round(total / t_db / 1e3, 2), "fb_over_db": round(t_db / t_fb, 3),
                                 "torch_ms": round(t_torch, 3), "torch_Mframes_s": round(total / t_torch / 1e3, 2),
                                 "fb_over_torch": round(t_torch / t_fb, 1),
                                 ("max_abs_diff" if log else "max_rel_diff"): float(f"{diff:.3g}")})
                    del out, ref
                    torch.cuda.empty_cache()
        del x

    res = {"bench": "stft_fb", "window": "hann", "hop": "N/4", "power": 2, "mel": "htk, 16 kHz", **card(), "rows": rows}
    line = json.dumps(res)
    print(line)
    outdir = Path(a.out)
    outdir.mkdir(parents=True, exist_ok=True)
    (outdir / "stft_fb_bench.json").write_text(line + "\n")


if __name__ == "__main__":
    main()
