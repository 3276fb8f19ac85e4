#!/usr/bin/env python3
"""bench.py -- baseband -> filterbank throughput on B200 (BASELINE.json metric).

Workload (config C2): Effelsberg-style 8 dual-pol IFs x 32 MHz (16 BBC channels, 2 Gbps),
2-bit VDIF, 60 s, Stokes I, 128 channels per IF, freq_res 512 (digifil -F128:512), tscrunch 16
(64 us), 8-bit spliced filterbank.  One step = one pass of the whole hot path (validate ->
decode -> channelise -> detect -> integrate -> rescale -> requantise -> splice) over the full
60 s scan.  `value` is measured with the VDIF already in HBM; `e2e` pushes the same scan from
pinned host memory through the C ABI and reads the finished rows back to the host.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--seconds S] [--impl reference] [--dump-outputs DIR]

N > 1: launched under torch.distributed.run, one rank per GPU; every rank processes its own
8-IF band (weak scaling: N x 8 subbands) and the finished 8-bit tiles are gathered over NCCL
into rank 0's band-ordered rows -- the one exchange the path has (base2fil.sh:422).

--dump-outputs DIR (one GPU): after the timed steps, write what the last of them delivered as float32
.npy files (see dump_outputs).  The input is generated from fixed seeds, so two builds run with the
same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FRAME_BYTES, PAYLOAD = 8032, 8000
FREQ_LSB0 = 1254.0
METRIC = "input baseband GB/s (VDIF bytes, headers included) per B200, 2 Gbps 16x32 MHz 2-bit -> 8-bit Stokes I"

#: BASELINE.json `configs`, in its order.  C2 is the configuration the metric is quoted on and the default.
CONFIGS = {
    "C1": dict(nif=4, bw=16.0, nchan=32, tscrunch=32, seconds=10.0, pol="I", out_nbit=8,
               what="C1: 4 IF x 16 MHz dual-pol 2-bit VDIF (512 Mbps; the reading of '8 subbands (512 Mbps)' that "
                    "base2fil.sh:251 gives), 10 s, nchan 32, freq_res 512, tscrunch 32 (64 us), 8-bit Stokes I"),
    "C2": dict(nif=8, bw=32.0, nchan=128, tscrunch=16, seconds=60.0, pol="I", out_nbit=8,
               what="C2: 8 IF x 32 MHz dual-pol 2-bit VDIF (2 Gbps), {sec:.0f} s, nchan 128, freq_res 512 (digifil -F128:512), "
                    "tscrunch 16, 8-bit Stokes I spliced to 1024 channels"),
    "C3": dict(nif=8, bw=32.0, nchan=128, tscrunch=16, seconds=60.0, pol="coherence", out_nbit=-32,
               what="C3: the C2 input to PP, QQ, Re PQ*, Im PQ* (digifil -d4), 32-bit float output, {sec:.0f} s"),
    "C4": dict(nif=8, bw=32.0, nchan=128, tscrunch=16, seconds=60.0, pol="I", out_nbit=8, dm=560.0,
               what="C4: C2 + coherent in-channel dedispersion at DM 560 (overlap-save), {sec:.0f} s"),
    "C5": dict(nif=16, bw=32.0, nchan=128, tscrunch=16, seconds=3600.0, sample_seconds=30.0, pol="I", out_nbit=8,
               what="C5: 16 IF x 32 MHz 2-bit (4 Gbps) streaming Stokes I; bounded sample of {sec:.0f} s of the 3600 s scan "
                    "(the scan is 120 such stretches; nothing carries over between them but the frozen rescale)"),
    # not a BASELINE.json configuration: the shape the reference's own job policy asks for at DM 560 (submit_job.py:58-76 ->
    # 8192 band channels over 8 IFs, DownSamp int(64 us / 32 us) = 2) -- the generic path with compile-time geometry
    "P1": dict(nif=8, bw=32.0, nchan=1024, tscrunch=2, seconds=20.0, pol="I", out_nbit=8,
               what="P1: the C2 input at the reference policy's channelisation for DM 560: nchan 1024 per IF, freq_res 2048 "
                    "(digifil -F1024:2048, process_vdif.py:162), tscrunch 2, 8-bit Stokes I spliced to 8192 channels, {sec:.0f} s"),
}
# module-level geometry of the selected configuration (set by select_config; tools/ import these)
NIF, BW, NCHAN, FREQ_RES, TSCRUNCH = 8, 32.0, 128, 512, 16
FPS = 4000                                  # frames per second per IF
BYTES_PER_DATA_SEC = NIF * FPS * FRAME_BYTES   # 257.024 MB of VDIF per second of sky


def select_config(name: str) -> dict:
    global NIF, BW, NCHAN, FREQ_RES, TSCRUNCH, FPS, BYTES_PER_DATA_SEC
    c = CONFIGS[name]
    NIF, BW, NCHAN, TSCRUNCH = c["nif"], c["bw"], c["nchan"], c["tscrunch"]
    FREQ_RES = 512 if NCHAN <= 128 else 2 * NCHAN          # process_vdif.py:162
    FPS = int(round(2 * BW * 1e6 / 16000))
    BYTES_PER_DATA_SEC = NIF * FPS * FRAME_BYTES
    return c


def if_plan():
    """base2fil.sh:54,65,254,407-414: IF i centred at freqLSB_0+(i-1)*bw, odd LSB / even USB"""
    bws, freqs = [], []
    for i in range(1, NIF + 1):
        freqs.append(FREQ_LSB0 + (i - 1) * BW)
        bws.append(BW if i % 2 == 0 else -BW)
    return bws, freqs


# --------------------------------------------------------------------------------------------
# synthetic input on the device (BASELINE.md section 5 recipe, torch Philox instead of PCG64:
# 15.4 GB cannot be generated with NumPy in bench time)
# --------------------------------------------------------------------------------------------
def make_device_vdif(torch, dev, nframes: int, seed: int):
    """uint8 tensor [nframes, 8032]: Gaussian sigma=1 per pol, thresholds +-0.9674, offset binary."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    out = torch.empty((nframes, FRAME_BYTES), dtype=torch.uint8, device=dev)
    step = 2048
    for f0 in range(0, nframes, step):
        n = min(step, nframes - f0)
        x = torch.randn((n, PAYLOAD, 2, 2), generator=g, device=dev)        # [frame, byte, t-in-byte, pol]
        c = ((x >= -0.9674).to(torch.uint8) + (x >= 0).to(torch.uint8) + (x >= 0.9674).to(torch.uint8))
        b = c[..., 0, 0] | (c[..., 0, 1] << 2) | (c[..., 1, 0] << 4) | (c[..., 1, 1] << 6)
        out[f0:f0 + n, 32:] = b
        idx = torch.arange(f0, f0 + n, device=dev, dtype=torch.int64)
        hdr = torch.zeros((n, 8), dtype=torch.int32, device=dev)
        hdr[:, 0] = (idx // FPS).to(torch.int32)
        hdr[:, 1] = ((idx % FPS) | (40 << 24)).to(torch.int32)
        hdr[:, 2] = (FRAME_BYTES // 8) | (1 << 24)
        hdr[:, 3] = 0x4566 | (1 << 26)
        out[f0:f0 + n, :32] = hdr.view(torch.uint8).reshape(n, 32)
    return out


#: size limit of the rows --dump-outputs writes as float32; longer outputs are dumped as a seeded sample of whole rows
DUMP_ROW_BYTES = 48 << 20


def dump_outputs(path: str, torch, plan, out_dev, rows: int):
    """The outputs of the last timed step as float32 .npy files in `path`:
    rows.npy         the spliced output rows in their sample values ([n, channels x products]); all `rows` of them, or n of
                     them chosen with a fixed seed when all would exceed DUMP_ROW_BYTES
    row_index.npy    which rows those are (float64), so that a build producing a different row count shows up
    rescale_mean.npy, rescale_scale.npy   the requantiser's statistics the step measured ([nif, products, nchan])"""
    os.makedirs(path, exist_ok=True)
    elems = plan.view_rows(np.empty((0, int(plan.row_bytes)), np.uint8)).shape[1]
    n = min(rows, max(1, DUMP_ROW_BYTES // (4 * elems)))
    idx = np.arange(rows) if n == rows else np.sort(np.random.default_rng(20121102).choice(rows, n, replace=False))
    sample = out_dev[torch.from_numpy(idx).to(out_dev.device)].cpu().numpy()
    mean, scale = plan.rescale()
    for name, a in (("rows", plan.view_rows(sample)), ("row_index", idx.astype(np.float64)),
                    ("rescale_mean", mean), ("rescale_scale", scale)):
        np.save(os.path.join(path, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.rows:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------
# CPU arm: the oracle port, one worker process per IF (base2fil.sh:60-66,219)
# --------------------------------------------------------------------------------------------
def _cpu_worker(args):
    seed, nframes, fc, sbw, nthr, cfg = args
    os.environ["OMP_NUM_THREADS"] = "1"
    import contextlib
    from frb_baseband_b200 import synth
    from oracle import digifil_oracle as o
    v = synth.make_vdif(nframes, seed=seed, bw_mhz=abs(sbw))
    try:                      # digifil -threads K (process_vdif.py --nthreads): FFT batches over K threads
        import scipy.fft
        pool = scipy.fft.set_workers(nthr)
    except Exception:
        pool = contextlib.nullcontext()
    dm, nfilt = cfg.get("dm", 0.0), None
    if dm > 0:             # overlap-save discard, the library's rule: 0.55 x the smearing of the lowest channel, whole output samples
        D = cfg["tscrunch"]
        nf = int(np.ceil(0.55 * o.smearing_samples(fc, sbw, cfg["nchan"], dm)))
        nf = max(D, (nf + D - 1) // D * D)
        nfilt = (nf, nf)
    t0 = time.perf_counter()
    with pool:
        r = o.digifil(v, freq_mhz=fc, bw_mhz=sbw, nchan=cfg["nchan"], freq_res=FREQ_RES, tscrunch_factor=cfg["tscrunch"],
                      pol_mode=cfg["pol"], out_nbit=cfg["out_nbit"], dm=dm, coherent=dm > 0, nfilt=nfilt, dtype=np.float32)
    return time.perf_counter() - t0, r["data"].shape[0]


def cpu_arm(cfg: dict, sample_seconds: float, steps: int = 1, warmup: int = 0):
    """Time the oracle (CPU restatement of digifil+splice) on the host's cores: `warmup` untimed passes, then the median
    of `steps` timed ones."""
    import multiprocessing as mp
    from frb_baseband_b200 import synth
    cores = len(os.sched_getaffinity(0))
    workers = min(NIF, cores)
    nthr = max(1, cores // workers)        # all host cores: one process per IF, digifil_nthreads = cores / nif
    unit = 1024 if BW >= 32 else 256       # frames holding whole FFT blocks
    nframes = int(round(sample_seconds * FPS / unit)) * unit or unit
    bws, freqs = if_plan()
    jobs = [(synth.config_seed(2, i + 1), nframes, freqs[i], bws[i], nthr, cfg) for i in range(NIF)]
    ctx = mp.get_context("spawn")      # the parent may hold a CUDA context: never fork it
    times = []
    with ctx.Pool(workers) as pool:
        for k in range(warmup + steps):
            res = pool.map(_cpu_worker, jobs)
            # splice: concatenate per-IF rows, highest frequency first (trivial next to digifil)
            wall = max(r[0] for r in res) if workers >= NIF else sum(r[0] for r in res) / workers
            if k >= warmup:
                times.append(max(wall, 1e-9))
    t = float(np.median(times))
    data_sec = nframes / FPS
    return {"value": NIF * nframes * FRAME_BYTES / t / 1e9, "unit": "GB/s", "cores": workers * nthr, "kind": "port",
            "sample": f"{data_sec:.3f} s of all {NIF} IFs of the workload, one oracle process per IF with {nthr} FFT "
                      f"thread(s) each (NumPy/SciPy-pocketfft float32 restatement of digifil+splice, NOT DSPSR/FFTW "
                      f"digifil itself: ratios against it would shrink by a small integer factor against the real thing)",
            "rt_factor": data_sec / t, "seconds_per_step": t}


def parity_check(torch, vd0, cfg: dict, bw_signed: float, freq: float, device: int):
    """The bench's own input through the same kernels vs the oracle: the first frames of one IF, float output
    (digifil -b-32 -I0), so a timed kernel that wrote garbage cannot score."""
    from frb_baseband_b200 import _lib
    from frb_baseband_b200.plan import Plan, PlanConfig
    from oracle import digifil_oracle as o
    nfr = 1024 if BW >= 32 else 512
    v = vd0[:nfr].cpu().numpy().reshape(-1)
    dm = cfg.get("dm", 0.0)
    mode = {"I": _lib.POL_I, "coherence": _lib.POL_COHERENCE, "IQUV": _lib.POL_IQUV}[cfg["pol"]]
    with Plan(PlanConfig(nchan=cfg["nchan"], bw_mhz=[bw_signed], freq_mhz=[freq], tscrunch=cfg["tscrunch"], pol_mode=mode,
                         out_nbit=-32, keep_bandpass=True, dm=dm, coherent=dm > 0, device=device)) as pl:
        path = pl.path
        nfilt = (int(pl.geometry.nfilt_pos), int(pl.geometry.nfilt_neg))
        pl.push([v])
        pl.flush()
        rows = pl.pull().view(np.float32).astype(np.float64)
    ref = o.digifil(v, freq_mhz=freq, bw_mhz=bw_signed, nchan=cfg["nchan"], tscrunch_factor=cfg["tscrunch"], pol_mode=cfg["pol"],
                    out_nbit=-32, keep_bandpass=True, dm=dm, coherent=dm > 0, nfilt=nfilt if dm > 0 else None)["data"].astype(np.float64)
    n = min(rows.shape[0], ref.shape[0])
    ref = ref[:n]
    got = rows[:n].reshape(ref.shape)
    rms = np.sqrt((ref ** 2).mean(axis=(0, 2), keepdims=True))
    err = float((np.abs(got - ref) / np.maximum(np.abs(ref), rms)).max()) if n else float("nan")
    return {"max_rel": err, "tol": 1e-5, "ok": bool(n > 0 and err <= 1e-5), "rows": int(n), "frames": nfr,
            "channeliser_path": path, "what": "first frames of IF 1 of the timed input, float path vs the NumPy oracle"}


# --------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS), help="BASELINE.json configuration (default: C2, the headline)")
    ap.add_argument("--seconds", type=float, default=None, help="seconds of sky data per step (default: the configuration's)")
    ap.add_argument("--impl", default="b2f", choices=["b2f", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg of a multi-GPU run")
    ap.add_argument("--chunk-units", type=int, default=4, help="frames per push in units of whole-block frame groups (0 = library default)")
    ap.add_argument("--nccl-gather", action="store_true", help="splice with an NCCL gather instead of peer stores")
    ap.add_argument("--cpu-sample", type=float, default=1.024, help="seconds of data for the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR as float32 .npy files (one GPU only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = select_config(args.config)
    seconds = args.seconds if args.seconds else cfg.get("sample_seconds", cfg["seconds"])
    workload = cfg["what"].format(sec=seconds)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (world > 1 or args.impl != "b2f"):
        ap.error("--dump-outputs dumps the b2f path of a one-GPU run")

    if args.impl == "reference":
        if rank != 0:
            return 0
        W = max(args.warmup, 0)
        r = cpu_arm(cfg, args.cpu_sample, steps=args.steps, warmup=min(W, 1))
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "GB/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["seconds_per_step"] * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "rt_factor": r["rt_factor"],
                "config": {"workload": workload + "; bounded sample per step: " + r["sample"]},
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": r["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from frb_baseband_b200 import _lib
    from frb_baseband_b200.plan import Plan, PlanConfig, fp32_peak_tflops
    from frb_baseband_b200.dist import PeerSplice, gather_splice, rank_if_plan

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the b2f path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    nframes = int(round(seconds * FPS))
    unit = 1024 if BW >= 32 else 256
    nframes -= nframes % unit
    _, bws, freqs = rank_if_plan(NIF * world, world, rank, FREQ_LSB0, BW)   # rank r owns the next NIF subbands up
    stream = torch.cuda.current_stream(dev)
    mode = {"I": _lib.POL_I, "coherence": _lib.POL_COHERENCE, "IQUV": _lib.POL_IQUV}[cfg["pol"]]
    dm = cfg.get("dm", 0.0)
    out_nbit = cfg["out_nbit"]

    def make_plan(bws_, freqs_, chunk_units):
        return Plan(PlanConfig(nchan=NCHAN, bw_mhz=bws_, freq_mhz=freqs_, tscrunch=TSCRUNCH, out_nbit=out_nbit, freq_res=FREQ_RES,
                               pol_mode=mode, dm=dm, coherent=dm > 0, device=local_rank, profile=True, stream=stream.cuda_stream,
                               chunk_units=chunk_units))

    generic = FREQ_RES != 512             # pushes of the generic path are plain frame counts (library default 1024), not block units
    pl = make_plan(bws, freqs, 0 if (dm > 0 or generic) else args.chunk_units)
    cf = int(pl.chunk_frames)
    row_bytes = int(pl.row_bytes)
    rows_total = int(seconds / pl.tsamp_s) + 8          # only an upper bound
    vd = [make_device_vdif(torch, dev, nframes, 20121102 + 2000 + 100 * rank + i) for i in range(NIF)]
    out_dev = torch.empty((rows_total + int(pl.chunk_rows), row_bytes), dtype=torch.uint8, device=dev)
    cap_rows = out_dev.shape[0]
    gathered = None
    peer = None
    if world > 1 and not args.nccl_gather:
        try:       # splice by peer stores over NVLink from the requantise kernel itself
            peer = PeerSplice(cap_rows, row_bytes, world, rank, dev)
        except Exception as ex:
            if rank == 0:
                print(f"peer splice unavailable ({ex!r}); falling back to an NCCL gather", file=sys.stderr)
    if world > 1 and peer is None and rank == 0:
        gathered = torch.empty((world, cap_rows, row_bytes), dtype=torch.uint8, device=dev)

    def make_step(plan, vds, out, peer_):
        cfr = int(plan.chunk_frames)
        chunks_ = [(f0, min(cfr, nframes - f0)) for f0 in range(0, nframes, cfr)]
        cap = out.shape[0]

        def step():
            plan.reset()
            got = 0
            for f0, n in chunks_:
                plan.push([v[f0].data_ptr() for v in vds], nframes=n, on_device=True)
                if peer_ is not None:
                    got += plan.pull_strided(peer_.dst(got), cap - got, peer_.pitch)
                else:
                    got += plan.pull_device(out[got].data_ptr(), cap - got)
            plan.flush()
            if peer_ is not None:
                got += plan.pull_strided(peer_.dst(got), cap - got, peer_.pitch)
            else:
                got += plan.pull_device(out[got].data_ptr(), cap - got)
                if world > 1 and plan is pl:   # fallback: gather every rank's tile into rank 0's band-ordered rows
                    gather_splice(out, world, rank, dst=0, out=gathered)
            return got
        return step, chunks_

    step_device, chunks = make_step(pl, vd, out_dev, peer)

    def timed(plan, fn, steps, warmup):
        for _ in range(warmup):
            fn()
        plan.sync(); torch.cuda.synchronize(dev)
        plan.reset_timers()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        l0 = plan.counters()["kernel_launches"]
        e0.record(stream)
        for _ in range(steps):
            rows = fn()
        plan.sync()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        t1 = time.time()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        launches = plan.counters()["kernel_launches"] - l0
        return ms / steps, rows, launches, (t0, t1)

    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    ms_step, rows, launches, (t0, t1) = timed(pl, step_device, args.steps, max(args.warmup, 3))
    clocks = sampler.stop(t0, t1)
    ktimes = pl.kernel_times()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, torch, pl, out_dev, int(rows))
    data_sec = nframes / FPS
    in_bytes = NIF * nframes * FRAME_BYTES
    value = world * in_bytes / (ms_step * 1e-3) / 1e9

    # ---- strong scaling: the SAME band cut over the ranks (base2fil.sh:60-66 runs one process per IF; here 1/N of the
    # IFs per GPU), pushes N times longer so that a launch still holds as many FFT blocks as the grid needs
    strong = None
    if world > 1 and not args.no_strong and NIF % world == 0:
        per = NIF // world
        sl = slice(rank * per, (rank + 1) * per)
        _, bws1, freqs1 = rank_if_plan(NIF, 1, 0, FREQ_LSB0, BW)
        pls = make_plan(bws1[sl], freqs1[sl], 0 if (dm > 0 or generic) else args.chunk_units * world)
        outs = torch.empty((cap_rows, int(pls.row_bytes)), dtype=torch.uint8, device=dev)
        peers = None
        if peer is not None:
            try:
                peers = PeerSplice(cap_rows, int(pls.row_bytes), world, rank, dev)
            except Exception:
                peers = None
        step_s, _ = make_step(pls, vd[:per], outs, peers)
        ms_s, rows_s, _, _ = timed(pls, step_s, args.steps, 2)
        strong = {"ifs_per_gpu": per, "ms_per_step": ms_s, "value": in_bytes / (ms_s * 1e-3) / 1e9, "unit": "GB/s",
                  "rt_factor": data_sec / (ms_s * 1e-3), "efficiency_vs_this_runs_weak_per_gpu_rate": ms_step / (world * ms_s),
                  "chunk_frames": int(pls.chunk_frames), "rows_per_step": int(rows_s),
                  "note": "the configuration's own band (not N bands): every GPU takes nif/N subbands, splice by peer stores"}
        pls.close()
        del outs

    # ---- e2e: pinned host VDIF -> C ABI -> rows back in pinned host memory
    e2e = None
    if not args.no_e2e:
        hold_frames = min(nframes, 12 * FPS)            # pinned host copy of 12 s, cycled through the scan
        hold_frames -= hold_frames % cf
        hold_frames = max(hold_frames, cf)
        host = [torch.empty((hold_frames, FRAME_BYTES), dtype=torch.uint8, pin_memory=True) for _ in range(NIF)]
        for i in range(NIF):
            host[i].copy_(vd[i][:hold_frames])
        torch.cuda.synchronize(dev)
        out_host = torch.empty((cap_rows, row_bytes), dtype=torch.uint8, pin_memory=True)
        hptr = [h.data_ptr() for h in host]
        import ctypes as C

        def step_host():
            pl.reset()
            got = 0
            for f0, n in chunks:
                h0 = f0 % hold_frames
                if h0 + n > hold_frames:
                    n = hold_frames - h0
                ptrs = (C.c_void_p * NIF)(*[p + h0 * FRAME_BYTES for p in hptr])
                _lib.check(_lib.lib().b2f_push(pl._h, ptrs, n, 0))
                got += pl.pull_async(out_host[got].data_ptr(), cap_rows - got)
            pl.flush()
            got += pl.pull_async(out_host[got].data_ptr(), cap_rows - got)
            pl.sync()
            return got

        ms_e2e, rows_e, _, _ = timed(pl, step_host, args.steps, 1)
        h2d = sum(n for _, n in chunks) * NIF * FRAME_BYTES
        # the ceiling of that number: a bare pinned-host -> device copy of the same buffers (PCIe), nothing else
        scratch = torch.empty_like(vd[0][:hold_frames])
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        scratch.copy_(host[0], non_blocking=True)
        torch.cuda.synchronize(dev)
        c0.record(stream)
        for i in range(NIF):
            scratch.copy_(host[i], non_blocking=True)
        c1.record(stream)
        torch.cuda.synchronize(dev)
        h2d_copy = NIF * hold_frames * FRAME_BYTES / (c0.elapsed_time(c1) * 1e-3) / 1e9
        del scratch
        e2e = {"value": world * in_bytes / (ms_e2e * 1e-3) / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(rows_e * row_bytes), "ms_per_step": ms_e2e,
               "rt_factor": world * data_sec / (ms_e2e * 1e-3),
               "h2d_copy_GBps_per_gpu": h2d_copy, "frac_of_h2d_copy": in_bytes / (ms_e2e * 1e-3) / 1e9 / h2d_copy,
               "note": "pinned host VDIF pushed chunk by chunk through b2f_push, rows pulled to pinned host memory; "
                       "12 s of host-resident VDIF cycled to cover the scan"}

    # ---- roofline of the dominant kernel.  The path is FP32-FFT bound (AI ~245 FLOP/B, SURVEY 8d): `roofline` is that
    # view; `roofline_hbm` is the algorithmic-bytes view the spec also asks for (small by construction).
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    fused = ktimes.get("fused", (0.0, 0))[1] > 0
    R, L = 2 * NCHAN, FREQ_RES
    blocks_per_step = NIF * (nframes * 16000 // (R * L))
    col_flops = blocks_per_step * 2.0 * R * 5 * L * np.log2(L)   # FFT_L + IFFT_L per column, 5 N log2 N
    row_flops = blocks_per_step * L * 5.0 * R * np.log2(R)
    if fused:
        dom, dom_name = ktimes["fused"], f"kf_fused<{R},{cfg['pol']}> (decode + column pass + row pass + detection, one persistent kernel)"
        dom_flops = col_flops + row_flops
    elif pl.path == 1:
        dom, dom_name = ktimes["column"], f"kf_fused<{R},I> column half (decode + FFT_512 . diag . IFFT_512 per column pair, warp-autonomous)"
        dom_flops = col_flops
    elif generic:
        dom, dom_name = ktimes["column"], f"kgt_column_pass<{int(np.log2(L))}> (decode + FFT_{L} . diag . IFFT_{L} per column, compile-time geometry)"
        dom_flops = col_flops
    else:
        dom, dom_name = ktimes["column"], "ka_column_pass (decode + column pass)"
        dom_flops = col_flops
    dom_ms, dom_n = dom
    dom_launch_ms = dom_ms / max(dom_n, 1)
    launches_per_step = max(dom_n, 1) / args.steps
    fp32_peak = fp32_peak_tflops(local_rank)
    traffic = None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = None if generic else prof.get("kf_fused_dram_bytes_per_launch" if fused else
                           ("kf_column_half_dram_bytes_per_launch" if pl.path == 1 else "ka_column_pass_dram_bytes_per_launch"))
    except Exception:
        pass
    ach = dom_flops / launches_per_step / (dom_launch_ms * 1e-3) / 1e12
    roofline = {"kernel": dom_name, "bound": "fp32", "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach / fp32_peak,
                "traffic": traffic, "traffic_source": "ncu --set full of tools/prof_run.py (same push size), profiles/traffic.json",
                "peak_source": "measured live: FP32 FMA loop (b2f_fp32_peak); MEASURED_PEAKS.json holds no FP32 CUDA-core figure "
                               "(nominal 148 SM x 128 lanes x 2 x 1.965 GHz = 74.4)",
                "avg_launch_ms": dom_launch_ms, "share_of_step": dom_ms / args.steps / ms_step,
                "convention": "5 N log2 N per complex FFT (SURVEY 8d)",
                "whole_step": {"achieved": (col_flops + row_flops) / (ms_step * 1e-3) / 1e12,
                               "frac": (col_flops + row_flops) / (ms_step * 1e-3) / 1e12 / fp32_peak}}
    alg_bytes_step = in_bytes + rows * row_bytes
    ach_b = alg_bytes_step / launches_per_step / (dom_launch_ms * 1e-3) / 1e9
    roofline_hbm = {"kernel": dom_name, "bound": "hbm", "achieved": ach_b, "peak": hbm_peak, "unit": "GB/s", "frac": ach_b / hbm_peak,
                    "peak_source": peak_src, "note": "algorithmic bytes (VDIF in + rows out) / dominant kernel time: not the binding roofline"}

    par = None
    if rank == 0:
        try:
            par = parity_check(torch, vd[0], cfg, bws[0], freqs[0], local_rank)
        except Exception as ex:
            par = {"ok": False, "error": repr(ex)}

    line = {
        "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "rt_factor": world * data_sec / (ms_step * 1e-3),
        "config": {"workload": workload, "name": args.config, "nif_per_gpu": NIF, "chunk_frames": cf,
                   "channeliser_path": "generic kernels with compile-time geometry (kgt_column_pass + kgt_row_pass)" if generic else {0: "round-1 kernels (ka_column_pass + kb_row_pass)", 1: "round-2 kernels (warp-autonomous column kernel + tile row pass)", 2: "round-2 fused kernel, L2 ring"}.get(pl.path),
                   "l2": "inputs (%.1f GB/step) larger than L2" % (in_bytes / 1e9),
                   "parallelism": (f"subband groups x{world} (weak: every GPU its own {NIF}-IF band), " + ("splice by NVLink peer stores from the requantise kernel" if peer is not None else "NCCL gather of 8-bit tiles")) if world > 1 else "1 GPU"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": roofline, "roofline_hbm": roofline_hbm, "parity_check": par,
        "kernel_ms_per_step": {k: v[0] / args.steps for k, v in ktimes.items() if v[1]},
        "rows_per_step": int(rows),
    }
    if strong is not None:
        line["strong"] = strong
    if rank == 0 and world == 1:
        try:
            line["cpu_baseline"] = {k: v for k, v in cpu_arm(cfg, args.cpu_sample).items() if k != "seconds_per_step"}
        except Exception as ex:      # never lose the GPU number to a host-side hiccup
            line["cpu_baseline"] = {"error": repr(ex)}
    if rank == 0:
        print(json.dumps(line))
    pl.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
