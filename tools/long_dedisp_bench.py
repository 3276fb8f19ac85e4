#!/usr/bin/env python3
"""Coherent dedispersion with transforms longer than 4096 points (b2f_kl.cu), one JSON line per case.

8 IF x 32 MHz (2-bit, alternating sidebands from 1254 MHz, 8-bit Stokes I, resident on the device) at nchan 8 / DM 349
(freq_res 65536), nchan 16 / DM 560 (32768) and nchan 32 / DM 1000 (16384), each at 4 us output resolution, plus a trial
plan at nchan 32 with 8 trials up to DM 1000.  Each line gives the wall time of one step (device events around reset,
pushes, pulls and a synchronise), the factor over real time, b2f_kernel_time per kernel id, and the FP32 work by the
5 N log2 N count (one M-point forward transform per block, one L-point backward transform per channel, polarisation and
trial) over the step time, as a share of the FP32 FMA peak measured in the same run.  The card's name and power limit are
read in the same run.  `--out FILE` also appends the lines to FILE."""
import argparse
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

import bench  # noqa: E402
from dm_trials_bench import card, run  # noqa: E402
from frb_baseband_b200.plan import fp32_peak_tflops  # noqa: E402

CASES = {
    "nchan8-dm349": dict(nchan=8, D=16, dms=349.0),
    "nchan16-dm560": dict(nchan=16, D=8, dms=560.0),
    "nchan32-dm1000": dict(nchan=32, D=4, dms=1000.0),
    "nchan32-8trials-dm1000": dict(nchan=32, D=4, dms=[1000.0 * (k + 1) / 8 for k in range(8)]),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", nargs="*", default=list(CASES), choices=list(CASES))
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    gpu = card()
    peak = fp32_peak_tflops(0)
    nif, bw = 8, 32.0
    fps = int(round(2 * bw * 1e6 / 16000))
    bench.FPS = fps
    nframes = int(a.seconds * fps)
    vd = [bench.make_device_vdif(torch, dev, nframes, 700 + i) for i in range(nif)]
    lines = []
    for name in a.case:
        c = CASES[name]
        g = dict(nif=nif, bw=bw, nchan=c["nchan"], D=c["D"], seconds=a.seconds)
        ms, kt, info = run(dev, g, vd, nframes, c["dms"], steps=a.steps, warmup=a.warmup)
        L, R = info["freq_res"], 2 * c["nchan"]
        M = R * L
        step = (L - 2 * info["nfilt"]) * R
        blocks = nif * (nframes * 16000 - M) // step
        flop = blocks * 5.0 * M * (math.log2(M) + info["ndm"] * math.log2(L))
        line = {"case": name, "gpu": gpu, "seconds_of_data": a.seconds, "nif": nif, "nchan": c["nchan"], "tscrunch": c["D"], **info,
                "ms_per_step": round(ms, 2), "x_real_time": round(a.seconds / (ms * 1e-3), 1),
                "kernel_ms": {k: round(v, 3) for k, v in kt.items()},
                "fp32_flop": flop, "fp32_tflops": round(flop / (ms * 1e-3) / 1e12, 3), "fp32_peak_tflops": round(peak, 1),
                "fp32_share_of_peak": round(flop / (ms * 1e-3) / 1e12 / peak, 4)}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        with open(a.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
