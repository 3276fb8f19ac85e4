#!/usr/bin/env python3
"""digifil -K (inter-channel dispersion delays removed after detection) against the same plan without it, one JSON line
per case.

8 IF x 32 MHz (2-bit, alternating sidebands from 1254 MHz, 8-bit Stokes I, resident on the device): the C4 geometry
(nchan 128, tscrunch 16, coherent dedispersion at DM 560, 20 s) without and with -K, the P1 geometry (nchan 1024,
tscrunch 2, 10 s) incoherent-only at DM 560 with -K, and 8 coherent trials up to DM 560 with -K.  Each line gives the wall
time of one step (device events around reset, pushes, pulls and a synchronise), the factor over real time, b2f_kernel_time
per kernel, and for -K the time of kd_delay_sum (reported as "tsum") with the bytes it must move -- every channel sample
of the delay ring read once, every output row written once -- over that time, against the 7.7 TB/s of the B200 data
sheet.  The hold is given twice: the d_max part, d_max |BW| 4 B nprod nif ndm, and the device memory the -K plan takes
beyond the plain one.  The card's name and power limit are read in the same run.  `--out FILE` appends the lines."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

import bench  # noqa: E402
from dm_trials_bench import card  # noqa: E402
from frb_baseband_b200 import _lib  # noqa: E402
from frb_baseband_b200.plan import Plan, PlanConfig  # noqa: E402

HBM_TBS = 7.7
CASES = {
    "C4": dict(nchan=128, D=16, seconds=20.0, dm=560.0, coherent=True, K=False),
    "C4-K": dict(nchan=128, D=16, seconds=20.0, dm=560.0, coherent=True, K=True),
    "P1-incoherent-K": dict(nchan=1024, D=2, seconds=10.0, dm=560.0, coherent=False, K=True),
    "C4-8trials-K": dict(nchan=128, D=16, seconds=20.0, dm=[560.0 * (k + 1) / 8 for k in range(8)], coherent=True, K=True),
}


def plan_of(c, dev, nif, bw):
    bws = [bw if i % 2 == 0 else -bw for i in range(1, nif + 1)]
    freqs = [1254.0 + (i - 1) * bw for i in range(1, nif + 1)]
    trials = c["dm"] if isinstance(c["dm"], list) else None
    return Plan(PlanConfig(nchan=c["nchan"], bw_mhz=bws, freq_mhz=freqs, tscrunch=c["D"], out_nbit=8, pol_mode=_lib.POL_I,
                           dm=0.0 if trials else c["dm"], coherent=c["coherent"], dm_trials=trials, remove_delays=c["K"],
                           stream=torch.cuda.current_stream(dev).cuda_stream, profile=True))


def run(dev, c, vd, nframes, nif, bw, steps, warmup):
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    pl = plan_of(c, dev, nif, bw)
    plan_bytes = free0 - torch.cuda.mem_get_info()[0]
    cf = int(pl.chunk_frames)
    cap = int(c["seconds"] / pl.tsamp_s) + 2 * int(pl.chunk_rows)
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
    d = pl.delays()
    info = dict(rows=rows, ndm=int(pl.ndm), freq_res=int(pl.geometry.freq_res), nfilt=int(pl.geometry.nfilt_pos),
                d_max=int(d.max()), nslot=int(pl.ndm) * nif, ncol=int(pl.nprod) * c["nchan"], plan_device_bytes=int(plan_bytes))
    pl.close()
    del out
    torch.cuda.empty_cache()
    return ms, kt, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", nargs="*", default=list(CASES), choices=list(CASES))
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    gpu = card()
    nif, bw = 8, 32.0
    bench.FPS = int(round(2 * bw * 1e6 / 16000))
    nframes = int(max(CASES[n]["seconds"] for n in a.case) * bench.FPS)
    vd = [bench.make_device_vdif(torch, dev, nframes, 900 + i) for i in range(nif)]
    lines = []
    for name in a.case:
        c = CASES[name]
        nfr = int(c["seconds"] * bench.FPS)
        ms, kt, info = run(dev, c, vd, nfr, nif, bw, a.steps, a.warmup)
        line = {"case": name, "gpu": gpu, "seconds_of_data": c["seconds"], "nif": nif, "nchan": c["nchan"], "tscrunch": c["D"],
                "dm": c["dm"], "coherent": c["coherent"], "remove_delays": c["K"], **info,
                "ms_per_step": round(ms, 2), "x_real_time": round(c["seconds"] / (ms * 1e-3), 1),
                "kernel_ms": {k: round(v, 3) for k, v in kt.items()}}
        if c["K"]:
            torch.cuda.synchronize()
            free0 = torch.cuda.mem_get_info()[0]
            pl = plan_of(dict(c, K=False), dev, nif, bw)
            plain_bytes = free0 - torch.cuda.mem_get_info()[0]
            pl.close()
            # kd_delay_sum: each channel sample of the ring read once, each output row written once (float32)
            moved = 4.0 * info["nslot"] * info["ncol"] * (info["rows"] * c["D"] + info["rows"])
            t = kt.get("tsum", 0.0)
            line.update({"kd_delay_sum_ms": round(t, 3), "kd_delay_sum_bytes": moved,
                         "kd_delay_sum_tb_per_s": round(moved / (t * 1e-3) / 1e12, 3) if t else None,
                         "kd_delay_sum_share_of_7p7_tbs": round(moved / (t * 1e-3) / 1e12 / HBM_TBS, 3) if t else None,
                         "hold_dmax_bytes": 4 * info["d_max"] * info["ncol"] * info["nslot"],
                         "extra_device_bytes_over_plain_plan": info["plan_device_bytes"] - plain_bytes})
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        with open(a.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
