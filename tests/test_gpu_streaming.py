"""Every way of driving a plan gives the rows of the plain host-push, full-drain scan, on every kernel family.

The parity tests push host memory and pull everything into host memory after every push.  Callers do more than that: they
push device pointers, pull into device memory, into pinned memory behind tickets, into a strided buffer, on their own
stream; they pull fewer rows than are held, let rows pile up until a push is refused, and reuse one plan for several scans.
Each of those touches bookkeeping the plain loop never reaches (partial pulls and the compaction of held rows, a refused
push, the carried state of every family across b2f_reset).  Each family's plain scan (helpers.run_plan) is checked once
against the float64 oracle; every other pattern must then reproduce it byte for byte, with the same counters."""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest

from frb_baseband_b200 import _lib, synth
from frb_baseband_b200.plan import B2FError, Plan, PlanConfig
from helpers import run_plan
from test_gpu_multi_if import COH, I, NAME, cached, check_splice, expected_tiles, oracle_floats
from test_gpu_dm_trials import slices, trial_floats
from test_gpu_remove_delays import k_floats

pytestmark = pytest.mark.gpu

FB = 8032

#: name: nchan, |bw|, tscrunch, pol, out_nbit, push size (chunk_units), rescale interval as a fraction of one push's rows
#: (0 = keep_bandpass), full pushes and ragged frames of the scan (-1: half a push), other PlanConfig fields, B2F_PATH, the
#: channeliser path the plan must report, stream seed.  An interval shorter than a push and at least three pushes make the
#: held rows outgrow the buffer while some are still held (see test_partial_pulls_and_compaction).
FAMILIES = {
    "round1-nchan32": dict(nchan=32, bw=16.0, D=32, pol=COH, nbit=8, chunk=1, ifrac=0.3, full=4, ragged=100, path=0, seed=10100),
    "round2-nchan128": dict(nchan=128, bw=32.0, D=16, pol=I, nbit=8, chunk=1, ifrac=0.3, full=3, ragged=600, path=1, seed=10200),
    "round2-fused": dict(nchan=128, bw=32.0, D=16, pol=I, nbit=8, chunk=1, ifrac=0.3, full=3, ragged=600, path=2, seed=10200,
                         env="fused"),
    "tuned-dedisp": dict(nchan=128, bw=32.0, D=16, pol=COH, nbit=8, chunk=2, ifrac=0.3, full=3, ragged=-1, path=0, seed=10300,
                         kw=dict(dm=300.0, coherent=True)),
    "generic-compile-time": dict(nchan=512, bw=32.0, D=4, pol=COH, nbit=-32, chunk=200, ifrac=0, full=3, ragged=130, path=0,
                                 seed=10400),
    "generic-runtime-dedisp": dict(nchan=64, bw=32.0, D=8, pol=COH, nbit=8, chunk=150, ifrac=0.3, full=3, ragged=70, path=0,
                                   seed=10500, kw=dict(freq_res=256, dm=100.0, coherent=True)),
    "long-transforms": dict(nchan=16, bw=32.0, D=2, pol=I, nbit=16, chunk=90, ifrac=0.3, full=10, ragged=40, path=0, seed=10600,
                            kw=dict(dm=560.0, coherent=True)),
    "trials": dict(nchan=128, bw=32.0, D=16, pol=I, nbit=8, chunk=2, ifrac=0.3, full=3, ragged=-1, path=0, seed=10700,
                   kw=dict(dm_trials=[0.0, 150.0, 300.0], coherent=True)),
    "remove-delays": dict(nchan=128, bw=32.0, D=16, pol=I, nbit=8, chunk=1, ifrac=0.3, full=3, ragged=512, path=1, seed=10800,
                          kw=dict(dm=300.0, remove_delays=True)),
    "tscrunch24-dedisp": dict(nchan=128, bw=32.0, D=24, pol=I, nbit=8, chunk=2, ifrac=0.3, full=3, ragged=-1, path=0, seed=10900,
                              kw=dict(dm=300.0, coherent=True)),
    "tscrunch100": dict(nchan=128, bw=32.0, D=100, pol=I, nbit=8, chunk=1, ifrac=0.3, full=3, ragged=600, path=1, seed=11000),
    "running-rescale": dict(nchan=128, bw=32.0, D=16, pol=I, nbit=8, chunk=1, ifrac=0.3, full=3, ragged=600, path=1, seed=10200,
                            kw=dict(rescale_mode=_lib.RESCALE_RUNNING)),
}

#: counters a scan must reproduce (kernel_launches accumulates over the life of the plan)
SCAN_COUNTERS = ("frames_ok", "frames_invalid", "frames_with_fill", "fill_words", "frames_dropped", "frames_misplaced",
                 "frames_badhdr", "slots_missing", "rows_produced", "rows_emitted", "blocks_dirty", "rescale_frozen")


@contextlib.contextmanager
def path_env(f):
    """B2F_PATH is read when a plan is created."""
    old = os.environ.get("B2F_PATH")
    if f.get("env"):
        os.environ["B2F_PATH"] = f["env"]
    else:
        os.environ.pop("B2F_PATH", None)
    try:
        yield
    finally:
        if old is None:
            os.environ.pop("B2F_PATH", None)
        else:
            os.environ["B2F_PATH"] = old


def band(f):
    """2 IFs 1 |bw| apart: LSB below, USB above."""
    b = f["bw"]
    return [-b, b], [1254.0, 1254.0 + b]


def plan_cfg(f, interval, **over):
    bws, freqs = band(f)
    kw = dict(nchan=f["nchan"], bw_mhz=bws, freq_mhz=freqs, tscrunch=f["D"], pol_mode=f["pol"], out_nbit=f["nbit"],
              keep_bandpass=not interval, chunk_units=f["chunk"], rescale_interval_s=interval or 10.0, **f.get("kw", {}))
    kw.update(over)
    return PlanConfig(**kw)


def new_plan(name, **over):
    f = FAMILIES[name]
    with path_env(f):
        return Plan(plan_cfg(f, geometry(name)["interval"], **over))


def make_streams(f, nframes, seed):
    """One stream per IF with a tone, polarisation correlation and faults of its own (as test_gpu_multi_if.streams)."""
    mix = [{"invalid_frac": 0.01}, {"fill_frac": 0.01}]
    return [synth.make_vdif(nframes, seed=seed + 7 * i, bw_mhz=f["bw"], tone_frac=0.05 + (0.13 + 0.19 * i) % 0.9,
                            tone_amp=0.3 + 0.1 * i, rho=0.1 + 0.07 * i, **mix[i]) for i in range(2)]


def geometry(name):
    """chunk_frames, frames of the scan (`full` whole pushes and a ragged one; ragged -1: half a push) and rescale interval
    (s) of a family.  For remove_delays, as many pushes as make the delay ring wrap at least twice."""
    def make():
        f = FAMILIES[name]
        with path_env(f), Plan(plan_cfg(f, 0)) as pl:
            g = pl.geometry
            cf, cr, tsamp, dmax = int(pl.chunk_frames), int(g.chunk_rows), float(pl.tsamp_s), int(pl.delays().max())
            spf, M, L = int(g.samples_per_frame), int(g.block_samples), int(g.freq_res)
        full = f["full"]
        if f.get("kw", {}).get("remove_delays"):
            # ring rows dl_cap = d_max + D - 1 + 2 P with P <= chunk_rows * D channel samples per push; each pass of the ring
            # writes at most dl_cap of them, so a scan of more than 2 dl_cap channel samples wraps it at least twice
            D = f["D"]
            cap = dmax + D - 1 + 2 * cr * D
            while full * cf * spf // M * L <= 2 * cap + D:
                full += 1
        ragged = cf // 2 if f["ragged"] < 0 else f["ragged"]
        assert 0 < ragged < cf
        return dict(cf=cf, nframes=full * cf + ragged, interval=round(f["ifrac"] * cr * tsamp, 6))
    return cached(("stream-geometry", name), make)


def chunks(name):
    cf, n = geometry(name)["cf"], geometry(name)["nframes"]
    return [(f0, min(cf, n - f0)) for f0 in range(0, n, cf)]


def streams_of(name, other=False):
    f = FAMILIES[name]
    n = geometry(name)["nframes"]
    seed = f["seed"] + (5000 if other else 0)
    return cached(("stream-vd", f["bw"], n, seed), lambda: make_streams(f, n, seed))


def as_bytes(rows):
    rows = np.ascontiguousarray(rows)
    return rows.view(np.uint8).reshape(rows.shape[0], -1)


def scan_counters(c):
    return {k: c[k] for k in SCAN_COUNTERS}


def reference(name):
    """The plain scan: host pushes, every row pulled into host memory after every push."""
    def make():
        f = FAMILIES[name]
        bws, freqs = band(f)
        interval = geometry(name)["interval"]
        kw = dict(nchan=f["nchan"], bw=bws, freq=freqs, tscrunch=f["D"], pol_mode=f["pol"], out_nbit=f["nbit"],
                  keep_bandpass=not interval, interval=interval or 10.0, chunk_units=f["chunk"], **f.get("kw", {}))
        with path_env(f):
            rows, info = run_plan(streams_of(name), **kw)
        assert info["path"] == f["path"], (name, info["path"])
        assert info["chunk_frames"] == geometry(name)["cf"]
        assert len(rows) > 0
        return as_bytes(rows), info
    return cached(("stream-ref", name), make)


def cap_rows(name):
    ref, info = reference(name)
    return len(ref) + int(info["geometry"].interval_rows) + 2 * int(info["geometry"].chunk_rows)


def assert_same_scan(name, what, rows, counters):
    ref, info = reference(name)
    assert rows.shape == ref.shape, f"{name} / {what}: {rows.shape} rows, the plain scan {ref.shape}"
    if not np.array_equal(rows, ref):
        bad = np.argwhere((rows != ref).any(axis=1))[:, 0]
        pytest.fail(f"{name} / {what}: {len(bad)} of {len(ref)} rows differ from the plain scan, the first at row {bad[0]}")
    assert scan_counters(counters) == scan_counters(info["counters"]), f"{name} / {what}"


# ---------------------------------------------------------------- drivers
def host_scan(pl, vd, chunk_list):
    """run_plan's loop on an existing plan: host pushes, full drains."""
    out = []

    def drain():
        while True:
            r = pl.pull()
            if not len(r):
                return
            out.append(r.copy())
    for f0, n in chunk_list:
        pl.push([v[f0 * FB:(f0 + n) * FB] for v in vd])
        drain()
    pl.flush()
    drain()
    return np.concatenate(out) if out else np.empty((0, int(pl.row_bytes)), np.uint8)


def device_scan(pl, vd, chunk_list, cap):
    """Device pointers in, pull_device out."""
    import torch
    dv = [torch.from_numpy(v).to("cuda") for v in vd]
    out = torch.empty((cap, int(pl.row_bytes)), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    got = 0

    def drain():
        nonlocal got
        while True:
            n = pl.pull_device(out[got].data_ptr(), cap - got)
            if not n:
                return
            got += n
    for f0, n in chunk_list:
        pl.push([d.data_ptr() + f0 * FB for d in dv], nframes=n, on_device=True)
        drain()
    pl.flush()
    drain()
    pl.sync()
    rows = out[:got].cpu().numpy()
    del dv
    return rows


# ---------------------------------------------------------------- the plain scan against the oracle
def oracle_tiles(name):
    f = FAMILIES[name]
    bws, freqs = band(f)
    vd = streams_of(name)
    ref, info = reference(name)
    g = info["geometry"]
    nint, running = int(g.interval_rows), f.get("kw", {}).get("rescale_mode") == _lib.RESCALE_RUNNING
    kw = f.get("kw", {})
    nf = (int(g.nfilt_pos), int(g.nfilt_neg))
    # the float rows do not depend on the channeliser path or the rescale mode: families that differ only there share them
    key = ("stream-floats", f["seed"], geometry(name)["nframes"], f["nchan"], f["D"], f["pol"],
           repr(sorted((k, v) for k, v in kw.items() if k != "rescale_mode")))
    if "dm_trials" in kw:
        fl = cached(key, lambda: [trial_floats(vd, bws, freqs, nchan=f["nchan"], D=f["D"], pol=f["pol"], dm=d, nfilt=nf,
                                               freq_res=int(g.freq_res)) for d in kw["dm_trials"]])
        return [expected_tiles(x, bws, out_nbit=f["nbit"], nint=nint) for x in fl]
    if kw.get("remove_delays"):
        fl = cached(key, lambda: k_floats(vd, bws, freqs, nchan=f["nchan"], D=f["D"], pol=f["pol"], dm=kw["dm"], coherent=False))
    else:
        fl = cached(key, lambda: oracle_floats(vd, bws, freqs, nchan=f["nchan"], D=f["D"], pol=f["pol"], freq_res=int(g.freq_res),
                                               dm=kw.get("dm", 0.0), nfilt=nf))
    return [expected_tiles(fl, bws, out_nbit=f["nbit"], nint=nint, running=running)]


@pytest.mark.parametrize("name", list(FAMILIES))
def test_plain_scan_matches_the_oracle(gpu, name):
    """The reference every other pattern is compared with is itself right: within the project's tolerances of the oracle."""
    f = FAMILIES[name]
    ref, info = reference(name)
    g = info["geometry"]
    if name == "long-transforms":
        assert int(g.freq_res) >= 8192
    if name == "generic-runtime-dedisp":
        assert int(g.freq_res) == 256 and int(g.nfilt_pos) > 0
    if name == "generic-compile-time":
        assert int(g.freq_res) == 1024
    if f["ifrac"]:
        assert 0 < int(g.interval_rows) < int(g.chunk_rows)
    view = {8: np.uint8, 16: np.uint16, -32: np.float32}[f["nbit"]]
    rows = ref.view(view)
    exp = oracle_tiles(name)
    parts = slices(rows, len(exp)) if len(exp) > 1 else [rows]
    for k, (part, e) in enumerate(zip(parts, exp)):
        check_splice(np.ascontiguousarray(part), e, info["if_order"], pol=f["pol"], nchan=f["nchan"], out_nbit=f["nbit"],
                     pol_major=False, what=f"{name} slice {k}")


# ---------------------------------------------------------------- 1: device push, device pull
@pytest.mark.parametrize("name", list(FAMILIES))
def test_device_push_device_pull(gpu, name):
    f = FAMILIES[name]
    with new_plan(name) as pl:
        rows = device_scan(pl, streams_of(name), chunks(name), cap_rows(name))
        assert_same_scan(name, "device push + pull_device", rows, pl.counters())


# ---------------------------------------------------------------- 2: pinned pipeline with tickets (b2f_run_scan's pattern)
@pytest.mark.parametrize("name", list(FAMILIES))
def test_pinned_pipeline_with_tickets(gpu, name):
    """Pinned host pushes; every pull_async goes to one of two pinned buffers and is followed by a ticket; a buffer is read
    only after wait() on the ticket of the pull that filled it, two pulls later; sync() at the end."""
    import torch
    f = FAMILIES[name]
    vd = streams_of(name)
    host = [torch.from_numpy(v).pin_memory() for v in vd]
    with new_plan(name) as pl:
        g = pl.geometry
        cap = int(g.interval_rows) + 2 * int(g.chunk_rows)          # the most rows a plan ever holds
        bufs = [torch.empty((cap, int(pl.row_bytes)), dtype=torch.uint8).pin_memory() for _ in range(2)]
        pulls, tickets, out = [], [], []

        def collect(k):
            n = pulls[k]
            out.append(bufs[k % 2][:n].numpy().copy())

        def drain():
            while True:
                k = len(pulls)
                if k >= 2:
                    pl.wait(tickets[k - 2])
                    collect(k - 2)
                n = pl.pull_async(bufs[k % 2].data_ptr(), cap)
                pulls.append(n)
                tickets.append(pl.mark())
                if not n:
                    return
        for f0, n in chunks(name):
            ptrs = (C.c_void_p * 2)(*[h.data_ptr() + f0 * FB for h in host])
            _lib.check(_lib.lib().b2f_push(pl._h, ptrs, n, 0))
            drain()
        pl.flush()
        drain()
        pl.sync()
        for k in range(max(0, len(pulls) - 2), len(pulls)):
            collect(k)
        while len(tickets) < 10:
            tickets.append(pl.mark())
        with pytest.raises(B2FError) as ex:
            pl.wait(tickets[-10])
        assert ex.value.code == _lib.ESTATE
        pl.wait(tickets[-8])
        rows = np.concatenate(out)
        assert_same_scan(name, "pinned pull_async with tickets", rows, pl.counters())


# ---------------------------------------------------------------- 3: partial pulls, backlog held, compaction
class Mirror:
    """The plan's row buffer bookkeeping (b2f_push / pull_impl) followed from the outside: where the held rows sit, and
    whether a push moves them to the front and in how many pieces."""

    def __init__(self, pl):
        g = pl.geometry
        self.cap = int(g.interval_rows) + 2 * int(g.chunk_rows)    # F_cap_rows
        self.off = self.held = 0
        self.compactions = []

    def pushed(self, rows):
        if self.off + self.held + rows > self.cap and self.off > 0 and self.held + rows <= self.cap:
            self.compactions.append(-(-self.held // self.off))      # pieces of at most `off` rows
            self.off = 0
        self.held += rows

    def pulled(self, n):
        self.held -= n
        self.off = self.off + n if self.held else 0


@pytest.mark.parametrize("name", list(FAMILIES))
def test_partial_pulls_and_compaction(gpu, name):
    """Pulls of 1, 7 and 61 rows in turn, only after every second push (and before a push that would not fit), so rows stay
    held at an offset and a later push moves them to the front of the buffer in several pieces."""
    f = FAMILIES[name]
    sizes = [1, 7, 61]
    vd = streams_of(name)
    with new_plan(name) as pl:
        m = Mirror(pl)
        cr = int(pl.geometry.chunk_rows)
        out, k, produced = [], 0, 0

        def pull_one():
            nonlocal k
            want = sizes[k % 3]
            k += 1
            r = pl.pull(want)
            assert len(r) <= want
            m.pulled(len(r))
            out.append(r.copy())
            c = pl.counters()
            assert c["rows_emitted"] == sum(len(x) for x in out) and c["rows_produced"] - c["rows_emitted"] == m.held
            return len(r)
        for j, (f0, n) in enumerate(chunks(name)):
            while m.held + cr > m.cap:          # this push could be refused: make room, a piece at a time
                assert pull_one() > 0
            pl.push([v[f0 * FB:(f0 + n) * FB] for v in vd])
            c = pl.counters()["rows_produced"]
            m.pushed(c - produced)
            produced = c
            if j % 2:
                pull_one()
        pl.flush()
        while m.held:
            assert pull_one() > 0
        assert pull_one() == 0
        assert max(m.compactions, default=0) >= 2, f"{name}: no push moved held rows in more than one piece {m.compactions}"
        assert_same_scan(name, "partial pulls", np.concatenate(out), pl.counters())


# ---------------------------------------------------------------- 4: backlog until refused, then retry
@pytest.mark.parametrize("name", list(FAMILIES))
def test_refused_push_is_retried(gpu, name):
    """Push without pulling until b2f_push refuses (B2F_ESTATE, row buffer full), pull everything, push the refused chunk
    again: the refusal must leave nothing behind (delay ring, kernel rows pending integration, carried samples)."""
    f = FAMILIES[name]
    vd = streams_of(name)
    with new_plan(name) as pl:
        out, refused = [], 0

        def drain():
            while True:
                r = pl.pull()
                if not len(r):
                    return
                out.append(r.copy())
        for f0, n in chunks(name):
            part = [v[f0 * FB:(f0 + n) * FB] for v in vd]
            try:
                pl.push(part)
            except B2FError as ex:
                assert ex.code == _lib.ESTATE, ex
                refused += 1
                before = pl.counters()
                drain()
                assert pl.counters()["rows_emitted"] > before["rows_emitted"]
                pl.push(part)
        pl.flush()
        drain()
        assert refused > 0, f"{name}: no push was refused"
        assert_same_scan(name, f"{refused} refused pushes retried", np.concatenate(out), pl.counters())


# ---------------------------------------------------------------- 5: strided pull on one plan
@pytest.mark.parametrize("name", [n for n in FAMILIES if "dm_trials" not in FAMILIES[n].get("kw", {})])
def test_strided_pull_keeps_the_padding(gpu, name):
    """pull_strided at a pitch of one row plus the store width into a canary-filled device buffer: the rows land at their
    pitch and the padding is untouched.  A misaligned pitch or pointer is refused before any row is consumed."""
    import torch
    f = FAMILIES[name]
    align = {8: 4, 16: 8, -32: 16}[f["nbit"]]
    vd = streams_of(name)
    cap = cap_rows(name)
    with new_plan(name) as pl:
        rb = int(pl.row_bytes)
        pitch = rb + align
        buf = torch.full((cap, pitch), 0xA5, dtype=torch.uint8, device="cuda")
        got, probed = 0, False

        def drain():
            nonlocal got, probed
            while True:
                if not probed and pl.counters()["rows_produced"] > pl.counters()["rows_emitted"] + 1:
                    probed = True
                    for p, pt in ((buf[got].data_ptr(), pitch + 1), (buf[got].data_ptr() + 1, pitch), (buf[got].data_ptr(), rb - align)):
                        e0 = pl.counters()["rows_emitted"]
                        with pytest.raises(B2FError) as ex:
                            pl.pull_strided(p, cap - got, pt)
                        assert ex.value.code == _lib.EINVAL and pl.counters()["rows_emitted"] == e0
                n = pl.pull_strided(buf[got].data_ptr(), cap - got, pitch)
                if not n:
                    return
                got += n
        for f0, n in chunks(name):
            pl.push([v[f0 * FB:(f0 + n) * FB] for v in vd])
            drain()
        pl.flush()
        drain()
        pl.sync()
        assert probed
        b = buf.cpu().numpy()
        assert (b[:, rb:] == 0xA5).all(), f"{name}: {(b[:, rb:] != 0xA5).sum()} padding bytes written"
        assert (b[got:] == 0xA5).all(), f"{name}: rows written past the {got} pulled"
        assert_same_scan(name, "pull_strided", np.ascontiguousarray(b[:got, :rb]), pl.counters())


# ---------------------------------------------------------------- 6: caller's stream, profiling on
@pytest.mark.parametrize("name", list(FAMILIES))
def test_external_stream_with_profile(gpu, name):
    import torch
    f = FAMILIES[name]
    s = torch.cuda.Stream()
    with new_plan(name, stream=s.cuda_stream, profile=True) as pl:
        rows = device_scan(pl, streams_of(name), chunks(name), cap_rows(name))
        t = pl.kernel_times()
        assert t["quant"][1] > 0 and t["quant"][0] > 0
        assert_same_scan(name, "external stream, profile", rows, pl.counters())
    torch.cuda.synchronize()


# ---------------------------------------------------------------- 7: reset hygiene
@pytest.mark.parametrize("name", list(FAMILIES))
def test_reset_mid_scan(gpu, name):
    """b2f_reset after an unfinished scan (no flush): every push but the last, a piece of the next, and a partial pull, so
    that carried samples, kernel rows pending integration, the delay ring, held rows and a half-emitted interval are all
    live -- then the whole scan must give the rows and counters of a fresh plan."""
    f = FAMILIES[name]
    vd = streams_of(name)
    cl = chunks(name)
    with new_plan(name) as pl:
        for f0, n in cl[:-1]:
            pl.push([v[f0 * FB:(f0 + n) * FB] for v in vd])
            while len(pl.pull()):
                pass
        f0 = cl[-1][0]
        pl.push([v[f0 * FB:(f0 + 37) * FB] for v in vd])
        pl.pull(7)
        c = pl.counters()
        assert c["rows_emitted"] > 0
        if name == "tscrunch100":
            # kernel rows of 4 samples each (the power-of-two part of 100), 25 of them per row: the 37-frame push leaves some
            g = pl.geometry
            blocks = sum(n * int(g.samples_per_frame) // int(g.block_samples) for _, n in cl[:-1] + [(0, 37)])
            assert blocks * 512 // 4 % 25
        pl.reset()
        rows = host_scan(pl, vd, cl)
        assert_same_scan(name, "reset mid-scan", rows, pl.counters())


@pytest.mark.parametrize("name", list(FAMILIES))
def test_reset_after_another_scan(gpu, name):
    """One plan, a scan of other data to the end, b2f_reset, then the scan: the first scan's statistics, carry, pending
    rows and ring must all be gone."""
    f = FAMILIES[name]
    with new_plan(name) as pl:
        host_scan(pl, streams_of(name, other=True), chunks(name))
        pl.reset()
        rows = host_scan(pl, streams_of(name), chunks(name))
        assert_same_scan(name, "reset after another scan", rows, pl.counters())
        if name == "remove-delays":
            g = pl.geometry
            D, dmax = FAMILIES[name]["D"], int(pl.delays().max())
            assert len(rows) * D + dmax > 2 * (dmax + D - 1 + 2 * int(g.chunk_rows) * D)     # the ring wrapped at least twice
