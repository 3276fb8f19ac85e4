"""digifil -K on the GPU: inter-channel dispersion delays removed after detection, against the float64 oracle.

The plan's row kernels write channel samples into a ring and kd_delay_sum adds tscrunch of them at each channel's delay.  At
-t 1 a -K plan's rows are the plain plan's rows shifted per channel, byte for byte, on every kernel family; with integration,
other products, several IFs, requantised output, trials and other inputs they match delay_oracle.digifil_k with the
band's reference at REL_TOL.  The row count is floor((K0 - d_max) / D) whatever the push size, DM 0 runs exactly as the plain
plan, and the file runner, its time parts, process_vdif and IF-sharded plans give the rows of one streaming run."""
import os
import struct
import threading

import numpy as np
import pytest

import delay_oracle as dl
from oracle import digifil_oracle as o
from frb_baseband_b200 import _lib, dist, process_vdif, synth
from frb_baseband_b200.plan import Plan, PlanConfig
from helpers import run_plan
from test_gpu_multi_if import BW, COH, I, IQUV, NAME, band, cached, check_splice, expected_tiles, streams

pytestmark = pytest.mark.gpu

NFR = 640                                  # 0.16 s at 32 MHz: about twice the 78 ms sweep at DM 300 over two 32 MHz IFs


def top_centre(freqs, nchan):
    return max(freqs) + BW / 2 - BW / (2 * nchan)


def nfilt_of(nchan, bws, freqs, D, dm, **kw):
    with Plan(PlanConfig(nchan=nchan, bw_mhz=bws, freq_mhz=freqs, tscrunch=D, coherent=True, dm=dm, **kw)) as pl:
        return (int(pl.geometry.nfilt_pos), int(pl.geometry.nfilt_neg)), int(pl.geometry.freq_res)


def k_floats(vd, bws, freqs, *, nchan, D, pol, dm, coherent, nfilt=(0, 0), freq_res=None, in_nbit=2, decode_mode="static", ref=None):
    """dl.digifil_k per IF at the band's reference (the plan's top channel centre), cut to the shortest IF."""
    ref = top_centre(freqs, nchan) if ref is None else ref
    out = []
    for v, b, f in zip(vd, bws, freqs):
        r = dl.digifil_k(v, freq_mhz=f, bw_mhz=b, nchan=nchan, dm=dm, tscrunch_factor=D, delay_ref_mhz=ref, freq_res=freq_res,
                         pol_mode=NAME[pol], in_nbit=in_nbit, coherent=coherent, nfilt=nfilt, decode_mode=decode_mode)
        out.append(np.asarray(r["float"], np.float64))
    n = min(d.shape[0] for d in out)
    return [d[:n] for d in out]


def tiles_natural(rows, info, bws, nprod, nchan):
    """Float rows -> [IF, t, nprod, chan] in plan IF order and natural channel order (USB tiles flipped back)."""
    nif = len(bws)
    e = rows.reshape(rows.shape[0], nif, nprod, nchan)
    out = np.empty((nif,) + e.shape[:1] + e.shape[2:], e.dtype)
    for s, i in enumerate(info["if_order"]):
        out[i] = e[:, s, :, ::-1] if bws[i] > 0 else e[:, s]
    return out


# ---------------------------------------------------------------- delay table
def test_delay_table(gpu):
    bws, freqs = band(3)
    with Plan(PlanConfig(nchan=128, bw_mhz=bws, freq_mhz=freqs, dm=300.0, remove_delays=True)) as pl:
        d = pl.delays()
        ref = top_centre(freqs, 128)
        assert d.shape == (1, 3, 128)
        for i in range(3):
            assert np.array_equal(d[0, i], dl.channel_delays(freqs[i], bws[i], 128, 300.0, ref))
    with Plan(PlanConfig(nchan=128, bw_mhz=bws, freq_mhz=freqs, dm=300.0, remove_delays=True, delay_ref_mhz=1500.0)) as pl:
        assert all(np.array_equal(pl.delays()[0, i], dl.channel_delays(freqs[i], bws[i], 128, 300.0, 1500.0)) for i in range(3))
    trials = [100.0, 300.0, 560.0]
    with Plan(PlanConfig(nchan=128, bw_mhz=bws, freq_mhz=freqs, coherent=True, dm_trials=trials, remove_delays=True)) as pl:
        d = pl.delays()
        assert d.shape == (3, 3, 128)
        for k, dm in enumerate(trials):
            for i in range(3):
                assert np.array_equal(d[k, i], dl.channel_delays(freqs[i], bws[i], 128, dm, ref)), (dm, i)
    with Plan(PlanConfig(nchan=128, bw_mhz=bws, freq_mhz=freqs, dm=300.0)) as pl:
        assert not pl.delays().any()


# ---------------------------------------------------------------- exact shift at -t 1
SHIFT = {
    "round2-nchan128-incoherent": dict(nchan=128, nif=2, dm=300.0, coherent=False, path=1),
    "tuned-dedispersion": dict(nchan=128, nif=2, dm=300.0, coherent=True, path=0),
    "generic-nchan1024": dict(nchan=1024, nif=2, dm=300.0, coherent=False, path=0),
    "long-nchan16": dict(nchan=16, nif=1, dm=560.0, coherent=True, path=0, usb=True),
}


@pytest.mark.parametrize("name", list(SHIFT))
def test_exact_shift_at_tscrunch_1(gpu, name):
    c = SHIFT[name]
    bws, freqs = ([BW], [1286.0]) if c.get("usb") else band(c["nif"])
    vd = cached(("kshift", c["nif"]), lambda: streams(c["nif"], NFR, 8800 + c["nif"]))
    kw = dict(nchan=c["nchan"], bw=bws, freq=freqs, out_nbit=-32, keep_bandpass=True, dm=c["dm"], coherent=c["coherent"])
    plain, pi = run_plan(vd, **kw)
    krows, ki = run_plan(vd, remove_delays=True, **kw)
    assert pi["path"] == ki["path"] == c["path"]
    g0, g1 = pi["geometry"], ki["geometry"]
    assert (g0.freq_res, g0.nfilt_pos, g0.chunk_frames) == (g1.freq_res, g1.nfilt_pos, g1.chunk_frames)
    with Plan(PlanConfig(nchan=c["nchan"], bw_mhz=bws, freq_mhz=freqs, dm=c["dm"], coherent=c["coherent"], remove_delays=True)) as pl:
        d = pl.delays()[0]
    nif, nchan = len(bws), c["nchan"]
    a = tiles_natural(plain, pi, bws, 1, nchan)
    b = tiles_natural(krows, ki, bws, 1, nchan)
    assert b.shape[1] == a.shape[1] - d.max() > 0, (b.shape, a.shape, d.max())
    want = np.empty_like(b)
    for i in range(nif):
        for ch in range(nchan):
            want[i, :, :, ch] = a[i, d[i, ch]: d[i, ch] + b.shape[1], :, ch]
    assert np.array_equal(b.view(np.uint32), want.view(np.uint32)), name


# ---------------------------------------------------------------- against the oracle
ORACLE = {
    "t16-coherent": dict(nchan=128, nif=2, pol=I, D=16, dm=300.0, coherent=True),
    "t24-coherent": dict(nchan=128, nif=2, pol=I, D=24, dm=300.0, coherent=True),
    "coherence-incoherent": dict(nchan=64, nif=2, pol=COH, D=8, dm=300.0, coherent=False, freq_res=256),
    "iquv-3if": dict(nchan=128, nif=3, pol=IQUV, D=4, dm=200.0, coherent=True),
    "iquv-3if-polmajor": dict(nchan=128, nif=3, pol=IQUV, D=4, dm=200.0, coherent=True, pol_major=True),
    "ja98": dict(nchan=128, nif=2, pol=I, D=16, dm=300.0, coherent=False, decode="ja98"),
    "8bit-input": dict(nchan=256, nif=2, pol=I, D=8, dm=300.0, coherent=True, in_nbit=8),
}


def _oracle_case(name):
    c = ORACLE[name]

    def make():
        bws, freqs = band(c["nif"])
        nbit = c.get("in_nbit", 2)
        nfr = NFR * 4 if nbit == 8 else NFR                # 8-bit frames hold a quarter of the samples
        vd = streams(c["nif"], nfr, 8900 + c["nchan"] + 13 * nbit + c["nif"], nbit=nbit, faults=None if nbit == 8 else [{}] * c["nif"])
        nf, L = nfilt_of(c["nchan"], bws, freqs, c["D"], c["dm"], **({"freq_res": c["freq_res"]} if "freq_res" in c else {})) \
            if c["coherent"] else ((0, 0), c.get("freq_res"))
        fl = k_floats(vd, bws, freqs, nchan=c["nchan"], D=c["D"], pol=c["pol"], dm=c["dm"], coherent=c["coherent"], nfilt=nf,
                      freq_res=L, in_nbit=nbit, decode_mode=c.get("decode", "static"))
        return vd, bws, freqs, fl
    return cached(("koracle", name.replace("-polmajor", "")), make)


def _oracle_kw(c, bws, freqs):
    kw = dict(nchan=c["nchan"], bw=bws, freq=freqs, tscrunch=c["D"], pol_mode=c["pol"], in_nbit=c.get("in_nbit", 2), dm=c["dm"],
              coherent=c["coherent"], remove_delays=True, splice_pol_major=c.get("pol_major", False))
    if "freq_res" in c:
        kw["freq_res"] = c["freq_res"]
    if c.get("decode") == "ja98":
        kw["decode_mode"] = _lib.DECODE_JA98
    return kw


@pytest.mark.parametrize("name", list(ORACLE))
def test_against_the_oracle(gpu, name):
    c = ORACLE[name]
    vd, bws, freqs, fl = _oracle_case(name)
    rows, info = run_plan(vd, out_nbit=-32, keep_bandpass=True, **_oracle_kw(c, bws, freqs))
    assert rows.shape[0] > 0
    check_splice(rows, expected_tiles(fl, bws, out_nbit=-32), info["if_order"], pol=c["pol"], nchan=c["nchan"], out_nbit=-32,
                 pol_major=c.get("pol_major", False), what=name)


@pytest.mark.parametrize("running", [False, True])
def test_requantised_output(gpu, running):
    """8-bit rows: digifil -c statistics of the first interval of delayed rows, or every interval with its own (+-1 LSB)."""
    c = ORACLE["t16-coherent"]
    vd, bws, freqs, fl = _oracle_case("t16-coherent")
    kw = _oracle_kw(c, bws, freqs)
    if running:
        kw["rescale_mode"] = _lib.RESCALE_RUNNING
    rows, info = run_plan(vd, out_nbit=8, interval=0.02, **kw)
    nint = int(info["geometry"].interval_rows)
    check_splice(rows, expected_tiles(fl, bws, out_nbit=8, nint=nint, running=running), info["if_order"], pol=I, nchan=128, out_nbit=8,
                 pol_major=False, what=f"8-bit, running={running}")


# ---------------------------------------------------------------- trials
def test_trials_against_the_oracle_and_single_dm(gpu):
    trials = [100.0, 300.0, 560.0]
    bws, freqs = band(2)
    vd = cached(("kshift", 2), lambda: streams(2, NFR, 8802))
    nf, L = nfilt_of(128, bws, freqs, 16, trials[-1])
    kw = dict(nchan=128, bw=bws, freq=freqs, tscrunch=16, coherent=True, remove_delays=True, out_nbit=-32, keep_bandpass=True)
    rows, info = run_plan(vd, dm_trials=trials, **kw)
    assert info["geometry"].ndm == 3
    from test_gpu_dm_trials import slices
    parts = slices(rows, 3)
    for k, dm in enumerate(trials):
        fl = k_floats(vd, bws, freqs, nchan=128, D=16, pol=I, dm=dm, coherent=True, nfilt=nf, freq_res=L)
        n = parts[k].shape[0]
        assert fl[0].shape[0] >= n
        check_splice(parts[k], expected_tiles([f[:n] for f in fl], bws, out_nbit=-32), info["if_order"], pol=I, nchan=128, out_nbit=-32,
                     pol_major=False, what=f"trial DM {dm}")
    one, _ = run_plan(vd, dm=trials[-1], **kw)
    assert one.shape[0] == parts[-1].shape[0]
    assert np.array_equal(parts[-1].view(np.uint8), one.view(np.uint8).reshape(one.shape[0], -1))


# ---------------------------------------------------------------- a dispersed pulse
def test_dispersed_pulse_is_aligned(gpu):
    """A pulse dispersed at DM 300 over an LSB and a USB IF (2-bit, with noise): after coherent dedispersion and -K every
    channel of the spliced band peaks in the same row (+-1); without -K the peaks follow the delay table."""
    from test_remove_delays_host import KBW, KF0, KN, KDM, _pulse
    rng = np.random.default_rng(11)
    vd, bws, freqs = [], [], []
    for i, fc, bw in sorted(o.if_plan(2, KF0, KBW)):
        x = _pulse(fc, bw)
        x = (x / x.std() + rng.standard_normal(x.shape)) / np.sqrt(2.0)
        spf = 8000 * 8 // 4
        vd.append(synth.make_vdif(KN // spf, seed=i, bw_mhz=KBW, x=x[:, : KN // spf * spf]))
        bws.append(bw)
        freqs.append(fc)
    kw = dict(nchan=128, bw=bws, freq=freqs, out_nbit=-32, keep_bandpass=True, dm=KDM, coherent=True)
    peaks = {}
    for remove in (False, True):
        rows, info = run_plan(vd, remove_delays=remove, **kw)
        t = tiles_natural(rows, info, bws, 1, 128)[:, :, 0, :]
        peaks[remove] = t.argmax(axis=1).reshape(-1)
    p = peaks[True]
    assert p.max() - p.min() <= 1, (p.min(), p.max())
    ref = dist.band_reference_mhz(2, KF0, KBW, 128)
    d = np.concatenate([dl.channel_delays(f, b, 128, KDM, ref) for f, b in zip(freqs, bws)])
    q = peaks[False] - d
    assert q.max() - q.min() <= 1 and abs(int(np.median(q)) - int(np.median(p))) <= 1


# ---------------------------------------------------------------- DM 0, push size
def test_dm0_runs_as_the_plain_plan(gpu):
    bws, freqs = band(2)
    vd = cached(("kshift", 2), lambda: streams(2, NFR, 8802))
    kw = dict(nchan=128, bw=bws, freq=freqs, tscrunch=16, out_nbit=8, interval=0.05, profile=True)
    a, ai = run_plan(vd, **kw)
    b, bi = run_plan(vd, remove_delays=True, **kw)
    assert np.array_equal(a, b)
    assert {k: v[1] for k, v in ai["times"].items()} == {k: v[1] for k, v in bi["times"].items()}
    assert ai["counters"]["kernel_launches"] == bi["counters"]["kernel_launches"]


def test_push_size_and_row_count(gpu):
    """Generic nchan 64 (pushes of chunk_units frames): 1- and 4-frame pushes, far shorter than d_max, and the default push
    give the same bytes, and floor((K0 - d_max) / D) rows."""
    bws, freqs = band(2)
    vd = cached(("kshift", 2), lambda: streams(2, NFR, 8802))
    kw = dict(nchan=64, freq_res=256, bw=bws, freq=freqs, tscrunch=8, pol_mode=COH, out_nbit=8, interval=0.02, dm=300.0)
    outs = [run_plan(vd, chunk_units=cu, remove_delays=True, **kw)[0] for cu in (1, 4, 0)]
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
    k0 = run_plan(vd, **dict(kw, tscrunch=1, out_nbit=-32, keep_bandpass=True))[0].shape[0]
    with Plan(PlanConfig(nchan=64, freq_res=256, bw_mhz=bws, freq_mhz=freqs, dm=300.0, remove_delays=True)) as pl:
        dmax = int(pl.delays().max())
    assert dmax > 4 * 16000 // 128 * 8                     # more than 8 pushes of 4 frames
    assert outs[0].shape[0] == (k0 - dmax) // 8 > 0


# ---------------------------------------------------------------- runner
def _write(tmp_path, vd, stem="if"):
    paths = []
    for i, v in enumerate(vd):
        p = tmp_path / f"{stem}{i}.vdif"
        v.tofile(p)
        paths.append(str(p))
    return paths


def _body(path):
    data = open(path, "rb").read()
    return data[data.index(b"HEADER_END") + len(b"HEADER_END"):]


R_KW = dict(nchan=128, tscrunch=16, coherent=True, dm=300.0, remove_delays=True, rescale_interval_s=0.05)


def test_run_scan_fifo_and_time_parts(gpu, tmp_path):
    bws, freqs = band(2)
    vd = streams(2, 2 * NFR, 9300)
    paths = _write(tmp_path, vd)
    whole = tmp_path / "whole.fil"
    cfg = PlanConfig(bw_mhz=bws, freq_mhz=freqs, **R_KW)
    with Plan(cfg) as pl:
        r = pl.run_scan(paths, str(whole), source_name="S")
    rows, _ = run_plan(vd, nchan=128, bw=bws, freq=freqs, tscrunch=16, coherent=True, dm=300.0, remove_delays=True, interval=0.05)
    assert r["rows"] == rows.shape[0] > 0 and _body(whole) == rows.tobytes()
    # a FIFO reader gets the same bytes
    fifo = tmp_path / "out.fifo"
    os.mkfifo(fifo)
    got = []
    th = threading.Thread(target=lambda: got.append(open(fifo, "rb").read()))
    th.start()
    with Plan(cfg) as pl:
        pl.run_scan(paths, str(fifo), source_name="S")
    th.join()
    assert got[0] == open(whole, "rb").read()
    for n in (2, 3):
        out = tmp_path / f"parts{n}.fil"
        with Plan(cfg) as pl:
            pl.run_scan(paths, None, stats_only=True)
            pl.set_rescale(*pl.rescale())
            total = sum(pl.run_scan(paths, str(out), source_name="S", part=(k, n))["rows"] for k in reversed(range(n)))
        assert total == r["rows"]
        assert open(out, "rb").read() == open(whole, "rb").read(), f"{n} parts differ from the single run"


def test_run_file_and_process_vdif(gpu, tmp_path):
    v = streams(1, NFR, 9400, faults=[{}])[0]
    src = tmp_path / "scan_if1.vdif"
    v.tofile(src)
    cfg = PlanConfig(bw_mhz=[-BW], freq_mhz=[1254.0], **R_KW)
    fil = tmp_path / "one.fil"
    with Plan(cfg) as pl:
        lib = _lib.lib()
        io = _lib.ScanIO()
        io.struct_size = _lib.C.sizeof(io)
        io.nsec = -1.0
        _lib.check(lib.b2f_run_file(pl._h, str(src).encode(), str(fil).encode(), _lib.C.byref(io), None))
        dmax = int(pl.delays().max())
    rows, _ = run_plan([v], nchan=128, bw=[-BW], freq=[1254.0], tscrunch=16, coherent=True, dm=300.0, remove_delays=True, interval=0.05)
    assert _body(fil) == rows.tobytes()
    # process_vdif --remove_delays: refdm = the DM, floor((K0 - d_max) / 16) rows
    out = tmp_path / "out"
    out.mkdir()
    assert process_vdif.main(["FRB1", str(src), "-l", "-f", "1254", "-b", str(BW), "--ra", "00:00:00", "--dec", "00:00:00",
                              "--nchan", "128", "--tscrunch", "16", "--start", "0", "--nsec", "0.15", "--keepBP", "--nbit", "8",
                              "--coherent_dm", "300", "--remove_delays", "--fil_out_dir", str(out)]) == 0
    data = open(out / "scan_if1.vdif_pol2.fil", "rb").read()
    i = data.index(b"refdm") + 5
    assert struct.unpack("<d", data[i:i + 8])[0] == 300.0
    nf, L = nfilt_of(128, [-BW], [1254.0], 16, 300.0)
    keep = L - 2 * nf[0]
    T = 600 * 16000                                        # 0.15 s of samples
    k0 = ((T - 256 * L) // (keep * 256) + 1) * keep
    assert len(_body(out / "scan_if1.vdif_pol2.fil")) == (k0 - dmax) // 16 * 128


# ---------------------------------------------------------------- IF sharding, memory
def test_if_sharded_plans_reproduce_the_full_plan(gpu):
    """Two plans of two IFs each, aligned to the whole band's fch1 (dist.band_reference_mhz), write the tiles of the 4-IF plan
    (incoherent dedispersion: a coherent plan's overlap follows its own lowest IF)."""
    bws, freqs = band(4)
    vd = streams(4, NFR, 9600, faults=[{}] * 4)
    kw = dict(nchan=128, tscrunch=4, out_nbit=-32, keep_bandpass=True, dm=150.0, remove_delays=True)
    full, fi = run_plan(vd, bw=bws, freq=freqs, **kw)
    ft = tiles_natural(full, fi, bws, 1, 128)
    ref = dist.band_reference_mhz(4, freqs[0], BW, 128)
    for lo in (0, 2):
        part, pi = run_plan(vd[lo:lo + 2], bw=bws[lo:lo + 2], freq=freqs[lo:lo + 2], delay_ref_mhz=ref, **kw)
        pt = tiles_natural(part, pi, bws[lo:lo + 2], 1, 128)
        assert pt.shape[1] >= ft.shape[1]
        assert np.array_equal(pt[:, : ft.shape[1]].view(np.uint32), ft[lo:lo + 2].view(np.uint32)), lo


def test_oversized_hold_is_refused(gpu):
    """32 IFs from 400 MHz at DM 5000, IQUV: about 2 TB of delay hold."""
    nif = 32
    with pytest.raises(_lib.B2FError) as e:
        Plan(PlanConfig(nchan=128, bw_mhz=[BW] * nif, freq_mhz=[400.0 + BW * i for i in range(nif)], pol_mode=IQUV, dm=5000.0,
                        remove_delays=True))
    assert e.value.code == _lib.ENOMEM and "bytes" in e.value.message, e.value.message
