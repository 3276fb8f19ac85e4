"""What bench.py times, against the float64 oracle.

bench.py's timed leg drives a plan unlike the parity tests: profiling on, on the caller's torch stream, device pointers in,
pull_device out, b2f_reset before every step.  Its e2e leg pushes pinned host memory and pulls with pull_async; its strong
leg pulls with pull_strided into a buffer whose pitch is several tiles wide.  Each case here builds the input and plan of
one configuration exactly as bench.main does, over a short scan (two whole pushes and a ragged one), runs each leg and
checks its rows: the first and last tile against the oracle, every other tile against a plan of that IF alone.

The values the replica shares with bench.py are kept below as plain data; test_bench_legs_host.py checks them against
bench.py's source, so a change in how bench.py drives the plan fails there by name."""
import ctypes as C
import types

import numpy as np
import pytest

import bench
from oracle import digifil_oracle as o
from frb_baseband_b200 import _lib
from helpers import run_plan
from test_gpu_multi_if import COH, I, expected_tiles, oracle_floats, tile_error, tile_of

pytestmark = pytest.mark.gpu

#: the PlanConfig keywords of bench.make_plan
PLAN_KEYWORDS = ("nchan", "bw_mhz", "freq_mhz", "tscrunch", "out_nbit", "freq_res", "pol_mode", "dm", "coherent", "device",
                 "profile", "stream", "chunk_units")
#: bench.main's push size (the third argument of make_plan for the timed plan; `args.chunk_units * world` for the strong leg)
CHUNK_UNITS_RULE = "0 if dm > 0 or generic else args.chunk_units"
STRONG_CHUNK_UNITS_RULE = "0 if dm > 0 or generic else args.chunk_units * world"
#: seed of IF i's synthetic VDIF on rank `rank` (bench.make_device_vdif)
SEED_RULE = "20121102 + 2000 + 100 * rank + i"
#: the plan calls of one step, in order: make_step's (peer splice: pull_strided, else pull_device) and step_host's
DEVICE_STEP_CALLS = ("reset", "push(on_device=True)", "pull_strided", "pull_device", "flush", "pull_strided", "pull_device")
HOST_STEP_CALLS = ("reset", "b2f_push(..., 0)", "pull_async", "flush", "pull_async", "sync")
BENCH_CHUNK_UNITS = 4           # bench.py --chunk-units default

CONFIGS = ["C1", "C2", "C3", "C4", "C5", "P1"]
FB = bench.FRAME_BYTES


@pytest.fixture
def config():
    """bench.select_config sets module globals: put bench back to its default configuration afterwards."""
    yield
    bench.select_config("C2")


def pol_mode(cfg):
    return {"I": _lib.POL_I, "coherence": _lib.POL_COHERENCE, "IQUV": _lib.POL_IQUV}[cfg["pol"]]


def chunk_units(cfg, world=1):
    env = dict(dm=cfg.get("dm", 0.0), generic=bench.FREQ_RES != 512, args=types.SimpleNamespace(chunk_units=BENCH_CHUNK_UNITS),
               world=world)
    return eval(STRONG_CHUNK_UNITS_RULE if world > 1 else CHUNK_UNITS_RULE, {}, env)


def make_plan(torch, cfg, bws, freqs, units):
    from frb_baseband_b200.plan import Plan, PlanConfig
    dm = cfg.get("dm", 0.0)
    kw = dict(nchan=bench.NCHAN, bw_mhz=bws, freq_mhz=freqs, tscrunch=bench.TSCRUNCH, out_nbit=cfg["out_nbit"], freq_res=bench.FREQ_RES,
              pol_mode=pol_mode(cfg), dm=dm, coherent=dm > 0, device=0, profile=True,
              stream=torch.cuda.current_stream(0).cuda_stream, chunk_units=units)
    assert tuple(kw) == PLAN_KEYWORDS
    return Plan(PlanConfig(**kw))


def device_step(pl, vds, nframes, out):
    """bench.make_step's step() without a peer splice: reset, device pushes, pull_device after each and after the flush."""
    cf = int(pl.chunk_frames)
    cap = out.shape[0]
    pl.reset()
    got = 0
    for f0 in range(0, nframes, cf):
        n = min(cf, nframes - f0)
        pl.push([v[f0].data_ptr() for v in vds], nframes=n, on_device=True)
        got += pl.pull_device(out[got].data_ptr(), cap - got)
    pl.flush()
    got += pl.pull_device(out[got].data_ptr(), cap - got)
    return got


def strided_step(pl, vds, nframes, dst, pitch, cap):
    """make_step with a peer splice: rows go to dst(row) = base + row * pitch + column."""
    cf = int(pl.chunk_frames)
    pl.reset()
    got = 0
    for f0 in range(0, nframes, cf):
        n = min(cf, nframes - f0)
        pl.push([v[f0].data_ptr() for v in vds], nframes=n, on_device=True)
        got += pl.pull_strided(dst(got), cap - got, pitch)
    pl.flush()
    got += pl.pull_strided(dst(got), cap - got, pitch)
    return got


def host_step(pl, host, hold_frames, nframes, out_host):
    """bench.main's step_host: pinned host frames cycled through the hold, b2f_push(..., 0), pull_async, sync."""
    cf = int(pl.chunk_frames)
    cap = out_host.shape[0]
    hptr = [h.data_ptr() for h in host]
    pl.reset()
    got = 0
    for f0 in range(0, nframes, cf):
        n = min(cf, nframes - f0)
        h0 = f0 % hold_frames
        if h0 + n > hold_frames:
            n = hold_frames - h0
        ptrs = (C.c_void_p * len(host))(*[p + h0 * FB for p in hptr])
        _lib.check(_lib.lib().b2f_push(pl._h, ptrs, n, 0))
        got += pl.pull_async(out_host[got].data_ptr(), cap - got)
    pl.flush()
    got += pl.pull_async(out_host[got].data_ptr(), cap - got)
    pl.sync()
    return got


def pushed_frames(nframes, cf, hold_frames):
    """The frame indices step_host pushes, in order: a ragged scan re-sends the start of the hold."""
    idx = []
    for f0 in range(0, nframes, cf):
        n = min(cf, nframes - f0)
        h0 = f0 % hold_frames
        n = min(n, hold_frames - h0)
        idx.extend(range(h0, h0 + n))
    return np.asarray(idx)


def oracle_rows(cfg, v, bw, freq, nfilt):
    """The oracle's float rows [t, nprod, chan] of one IF."""
    dm = cfg.get("dm", 0.0)
    pol = {"I": I, "coherence": COH}[cfg["pol"]]
    return oracle_floats([v], [bw], [freq], nchan=bench.NCHAN, D=bench.TSCRUNCH, pol=pol, freq_res=bench.FREQ_RES, dm=dm,
                         nfilt=nfilt if dm > 0 else (0, 0))[0]


def oracle_tile(cfg, fl, bw):
    """What the plan should write into the tile of one IF: 8-bit via the oracle's rescale_stats / digitise over all rows (bench's
    10 s interval is longer than the scan), or for float output without keep_bandpass (x - mean) * scale."""
    if cfg["out_nbit"] == -32:
        mean, scale = o.rescale_stats(fl, fl.shape[0])
        y = (fl - mean) * scale
        return y[:, :, ::-1] if bw > 0 else y
    return expected_tiles([fl], [bw], out_nbit=cfg["out_nbit"], nint=fl.shape[0])[0]


def check_tile(name, cfg, rows, s, nif, want, what):
    nprod = want.shape[1]
    elems = rows.view(np.float32) if cfg["out_nbit"] == -32 else rows
    g = tile_of(elems, s, nif, nprod, bench.NCHAN, False)
    assert g.shape == want.shape, (what, g.shape, want.shape)
    if cfg["out_nbit"] == -32:          # test_requantised_output's criterion for float output in sigma units
        err = np.abs(g.astype(np.float64) - want).max()
        assert err <= 1e-3, f"{name} {what}: tile {s} off by {err:.2e} sigma"
    else:
        msg = tile_error(g, want, cfg["out_nbit"], None)
        assert msg is None, f"{name} {what}: tile {s}: {msg}"


def scan_frames(cf, unit):
    """A multiple of bench's frame unit holding two whole pushes and a ragged one; when the push is one unit (the generic
    path's 1024 frames) every multiple is whole pushes, and the scan is three of them."""
    n = (2 * cf // unit + 1) * unit
    return n if n < 3 * cf else 3 * cf


@pytest.mark.parametrize("name", CONFIGS)
def test_bench_legs_against_the_oracle(gpu, config, name):
    import torch
    from frb_baseband_b200.dist import rank_if_plan
    from frb_baseband_b200.plan import Plan, PlanConfig
    cfg = bench.select_config(name)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    nif = bench.NIF
    unit = 1024 if bench.BW >= 32 else 256
    _, bws, freqs = rank_if_plan(nif, 1, 0, bench.FREQ_LSB0, bench.BW)
    dm = cfg.get("dm", 0.0)

    pl = make_plan(torch, cfg, bws, freqs, chunk_units(cfg))
    cf, rb, path = int(pl.chunk_frames), int(pl.row_bytes), pl.path
    nfilt = (int(pl.geometry.nfilt_pos), int(pl.geometry.nfilt_neg))
    nframes = scan_frames(cf, unit)
    assert nframes % unit == 0 and nframes >= 2 * cf
    vd = [bench.make_device_vdif(torch, dev, nframes, eval(SEED_RULE, {}, dict(rank=0, i=i))) for i in range(nif)]
    cap = int(nframes / bench.FPS / pl.tsamp_s) + 8 + int(pl.chunk_rows)
    out = torch.empty((cap, rb), dtype=torch.uint8, device=dev)

    # ---- the timed leg: three steps, byte-identical
    steps = []
    for _ in range(3):
        got = device_step(pl, vd, nframes, out)
        pl.sync()
        steps.append(out[:got].cpu().numpy().copy())
    assert all(np.array_equal(s, steps[0]) for s in steps[1:]), f"{name}: the timed steps differ from each other"
    rows = steps[-1]
    assert len(rows) > 0
    host_vd = [v.cpu().numpy().reshape(-1) for v in vd]
    order = pl.if_order
    assert bws[order[0]] > 0 and bws[order[-1]] < 0 and order[-1] == 0          # highest IF (USB) first, IF 1 (LSB) last
    fl = {}
    for s in (0, nif - 1):
        i = order[s]
        fl[i] = oracle_rows(cfg, host_vd[i], bws[i], freqs[i], nfilt)
        check_tile(name, cfg, rows, s, nif, oracle_tile(cfg, fl[i][:len(rows)], bws[i]), "timed leg")
    for s in range(1, nif - 1):
        i = order[s]
        # dedispersion takes its overlap from the lowest channel of the plan: IF 1 rides along so that nfilt is the band's
        pick = [0, i] if dm > 0 else [i]
        one, info = run_plan([host_vd[k] for k in pick], nchan=bench.NCHAN, bw=[bws[k] for k in pick], freq=[freqs[k] for k in pick],
                             tscrunch=bench.TSCRUNCH, pol_mode=pol_mode(cfg), out_nbit=cfg["out_nbit"], freq_res=bench.FREQ_RES,
                             chunk_units=chunk_units(cfg), dm=dm, coherent=dm > 0)
        one = np.ascontiguousarray(one).view(np.uint8).reshape(len(one), -1)
        assert (int(info["geometry"].nfilt_pos), int(info["geometry"].nfilt_neg)) == nfilt
        if info["path"] != path:        # another channeliser: equal within the oracle's tolerance, not byte for byte
            check_tile(name, cfg, rows, s, nif, oracle_tile(cfg, oracle_rows(cfg, host_vd[i], bws[i], freqs[i], nfilt)[:len(rows)], bws[i]),
                       f"timed leg (one-IF plan on path {info['path']})")
            continue
        tb = rb // nif
        col = info["if_order"].index(1) if dm > 0 else 0
        assert np.array_equal(rows[:, s * tb:(s + 1) * tb], one[:, col * tb:(col + 1) * tb]), f"{name}: tile {s} (IF {i + 1})"

    # ---- the e2e leg: pinned host frames cycled through a hold of whole pushes
    hold = min(nframes, 12 * bench.FPS)
    hold -= hold % cf
    hold = max(hold, cf)
    host = [torch.empty((hold, FB), dtype=torch.uint8, pin_memory=True) for _ in range(nif)]
    for i in range(nif):
        host[i].copy_(vd[i][:hold])
    torch.cuda.synchronize(dev)
    out_host = torch.empty((cap, rb), dtype=torch.uint8, pin_memory=True)
    got = host_step(pl, host, hold, nframes, out_host)
    e2e = out_host[:got].numpy().copy()
    c1 = pl.counters()
    idx = pushed_frames(nframes, cf, hold)
    resent = int((idx != np.arange(len(idx))).sum())
    assert (resent > 0) == (nframes > hold)
    assert c1["frames_misplaced"] == nif * resent, f"{name}: {c1['frames_misplaced']} frames misplaced, {nif * resent} re-sent"
    if resent:
        seq = [v[torch.from_numpy(idx).to(dev)].contiguous() for v in vd]
        got = device_step(pl, seq, len(idx), out)
        pl.sync()
        again = out[:got].cpu().numpy()
        assert np.array_equal(e2e, again), f"{name}: the e2e rows differ from a device push of the same frames"
        for s in (0, nif - 1):
            i = order[s]
            if dm > 0 or bench.FREQ_RES != 512:
                f2 = oracle_rows(cfg, host_vd[i].reshape(-1, FB)[idx].reshape(-1), bws[i], freqs[i], nfilt)
            else:
                # whole FFT blocks per push and no carry: the rows of the re-sent frames are the first rows of the scan
                def rows_of(frames):
                    return frames * 16000 // (2 * bench.NCHAN * 512) * 512 // bench.TSCRUNCH
                f2 = np.concatenate([fl[i][:rows_of(hold)], fl[i][:rows_of(len(idx) - hold)]])
            check_tile(name, cfg, e2e, s, nif, oracle_tile(cfg, f2[:len(e2e)], bws[i]), "e2e leg")
        del seq
    else:
        assert np.array_equal(e2e, rows), f"{name}: the e2e rows differ from the timed rows"
    del host, out_host

    # ---- the strong leg on one GPU: w plans of nif / w consecutive IFs, pulled side by side into one pitched buffer
    for w in {"C2": (2, 8), "C4": (2,), "P1": (2,)}.get(name, ()):
        per = nif // w
        plans = [make_plan(torch, cfg, bws[r * per:(r + 1) * per], freqs[r * per:(r + 1) * per], chunk_units(cfg, w)) for r in range(w)]
        tb = int(plans[0].row_bytes)
        assert tb * w == rb
        margin = 16
        pitch = w * tb + margin
        buf = torch.full((cap, pitch), 0x5A, dtype=torch.uint8, device=dev)
        n_r = []
        for r, p in enumerate(plans):
            col = (w - 1 - r) * tb               # PeerSplice.dst: highest frequencies leftmost
            base = buf.data_ptr() + col
            n_r.append(strided_step(p, vd[r * per:(r + 1) * per], nframes, lambda row: base + row * pitch, pitch, cap))
            p.sync()
        b = buf.cpu().numpy()
        same = [(int(p.geometry.nfilt_pos), int(p.geometry.nfilt_neg)) == nfilt for p in plans]
        for p in plans:
            p.close()
        assert (b[:, w * tb:] == 0x5A).all(), f"{name} strong x{w}: the margin right of the tiles was written"
        for r in range(w):
            col = (w - 1 - r) * tb
            assert (b[n_r[r]:, col:col + tb] == 0x5A).all(), f"{name} strong x{w}: rank {r} wrote past its rows"
            if not same[r]:
                # the dedispersion overlap of a plan follows its own lowest channel: a plan of higher IFs discards less, its
                # rows start at another time and cannot be the full plan's
                continue
            assert n_r[r] == len(rows), (name, w, r, n_r[r], len(rows))
            assert np.array_equal(b[:len(rows), col:col + tb], rows[:, col:col + tb]), f"{name} strong x{w}: rank {r}'s tile"
        assert same[0]
    pl.close()
    del out

    # ---- bench's own parity check on the same input
    par = bench.parity_check(torch, vd[0], cfg, bws[0], freqs[0], 0)
    assert par["ok"], par
