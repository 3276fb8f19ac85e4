#!/usr/bin/env python3
"""Coherent dedispersion at K trial DMs in one plan against K single-DM plans run back to back, one JSON line per case.

C4 geometry (8 IF x 32 MHz, 2-bit, nchan 128, tscrunch 16, 8-bit Stokes I, 20 s resident on the device) with K in
{1, 2, 4, 8, 16, 32} trials spread evenly up to DM 560 (the largest trial sets nfilt, as C4's single DM does), and the P1
geometry (nchan 1024 -> -F1024:2048, tscrunch 2, generic kernels, 10 s) with K in {1, 4}.  Each line gives the wall time
of one step (device events around reset, pushes, pulls and a synchronise), the factor over real time, and
b2f_kernel_time per kernel, for the trial plan and summed over the K single-DM plans.  The card's name and power limit
are read in the same run.  `--out FILE` also appends the lines to FILE."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from frb_baseband_b200 import _lib  # noqa: E402
from frb_baseband_b200.plan import Plan, PlanConfig  # noqa: E402

GEOMETRIES = {
    "C4": dict(nif=8, bw=32.0, nchan=128, D=16, seconds=20.0, dm_max=560.0, ks=[1, 2, 4, 8, 16, 32]),
    "P1": dict(nif=8, bw=32.0, nchan=1024, D=2, seconds=10.0, dm_max=560.0, ks=[1, 4]),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def run(dev, g, vd, nframes, dms, *, steps, warmup):
    """Time one plan (trial DMs if len(dms) > 1 or trials=True) over the resident input: ms per step, kernel ms per step."""
    nif = g["nif"]
    bws = [g["bw"] if i % 2 == 0 else -g["bw"] for i in range(1, nif + 1)]
    freqs = [1254.0 + (i - 1) * g["bw"] for i in range(1, nif + 1)]
    trials = dms if isinstance(dms, list) else None
    pl = Plan(PlanConfig(nchan=g["nchan"], bw_mhz=bws, freq_mhz=freqs, tscrunch=g["D"], out_nbit=8, pol_mode=_lib.POL_I,
                         dm=0.0 if trials else float(dms), coherent=True, dm_trials=trials,
                         stream=torch.cuda.current_stream(dev).cuda_stream, profile=True))
    cf = int(pl.chunk_frames)
    cap = int(g["seconds"] / pl.tsamp_s) + 2 * int(pl.chunk_rows)
    out = torch.empty((cap, int(pl.row_bytes)), dtype=torch.uint8, device=dev)
    chunks = [(f0, min(cf, nframes - f0)) for f0 in range(0, nframes, cf)]

    def step():
        pl.reset()
        got = 0
        for f0, n in chunks:
            pl.push([v[f0].data_ptr() for v in vd], nframes=n, on_device=True)
            got += pl.pull_device(out[got].data_ptr(), cap - got)
        pl.flush()
        got += pl.pull_device(out[got].data_ptr(), cap - got)
        return got

    for _ in range(warmup):
        rows = step()
    pl.sync()
    torch.cuda.synchronize()
    pl.reset_timers()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        rows = step()
    pl.sync()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    kt = {k: v[0] / steps for k, v in pl.kernel_times().items() if v[1]}
    info = dict(rows=rows, ndm=int(pl.ndm), freq_res=int(pl.geometry.freq_res), nfilt=int(pl.geometry.nfilt_pos))
    pl.close()
    del out
    torch.cuda.empty_cache()
    return ms, kt, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--geometry", nargs="*", default=list(GEOMETRIES), choices=list(GEOMETRIES))
    ap.add_argument("--ks", type=int, nargs="*", default=None, help="trial counts (default: the geometry's)")
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    gpu = card()
    lines = []
    for name in a.geometry:
        g = GEOMETRIES[name]
        fps = int(round(2 * g["bw"] * 1e6 / 16000))
        bench.FPS = fps
        nframes = int(g["seconds"] * fps)
        vd = [bench.make_device_vdif(torch, dev, nframes, 500 + i) for i in range(g["nif"])]
        for K in a.ks or g["ks"]:
            dms = [g["dm_max"] * (k + 1) / K for k in range(K)]
            ms, kt, info = run(dev, g, vd, nframes, dms, steps=a.steps, warmup=a.warmup)
            s_ms, s_kt = 0.0, {}
            for d in dms:                                   # K single-DM plans, back to back
                m1, k1, i1 = run(dev, g, vd, nframes, d, steps=a.steps, warmup=a.warmup)
                s_ms += m1
                for k, v in k1.items():
                    s_kt[k] = s_kt.get(k, 0.0) + v
            single_top = run(dev, g, vd, nframes, dms[-1], steps=a.steps, warmup=a.warmup)[1].get("dedisp", 0.0)
            line = {"geometry": name, "K": K, "gpu": gpu, "seconds_of_data": g["seconds"], **info,
                    "trial_plan_ms": round(ms, 2), "trial_plan_rt": round(g["seconds"] / (ms * 1e-3), 1),
                    "single_plans_ms": round(s_ms, 2), "single_plans_rt": round(g["seconds"] / (s_ms * 1e-3), 1),
                    "speedup": round(s_ms / ms, 3),
                    "dedisp_ms_per_trial": round(kt.get("dedisp", 0.0) / K, 3), "single_dedisp_ms_at_dm_max": round(single_top, 3),
                    "trial_kernel_ms": {k: round(v, 3) for k, v in kt.items()},
                    "single_plans_kernel_ms": {k: round(v, 3) for k, v in s_kt.items()}}
            print(json.dumps(line), flush=True)
            lines.append(line)
        del vd
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
