"""Coherent dedispersion at several trial DMs in one pass, against the oracle and against single-DM plans.

A trial plan computes the spectrum of every overlap-save block once and applies one chirp per trial DM.  Each trial's slice
of a row must be what the oracle gives at that DM with the plan's nfilt (the nfilt of the largest trial), and the largest
trial must equal a single-DM plan at that DM byte for byte: the per-trial arithmetic is that of the single-DM kernels."""
import os
import struct

import numpy as np
import pytest

from oracle import digifil_oracle as o
from frb_baseband_b200 import _lib, process_vdif
from frb_baseband_b200.plan import Plan, PlanConfig
from helpers import run_plan
from test_gpu_multi_if import BW, COH, I, NAME, band, cached, check_splice, expected_tiles, streams

pytestmark = pytest.mark.gpu


def _nfilt(nchan, D, dms, bws, freqs, **kw):
    with Plan(PlanConfig(nchan=nchan, bw_mhz=bws, freq_mhz=freqs, tscrunch=D, coherent=True, dm_trials=list(dms), **kw)) as pl:
        return int(pl.geometry.nfilt_pos), int(pl.geometry.nfilt_neg), int(pl.geometry.freq_res)


def trial_floats(vd, bws, freqs, *, nchan, D, pol, dm, nfilt, freq_res, in_nbit=2):
    """Oracle floats per IF at one trial DM with the trial plan's nfilt.  o.digifil does not dedisperse at DM 0, so that
    trial is built from o.filterbank_dedisp with a unit chirp."""
    out = []
    for v, b, f in zip(vd, bws, freqs):
        if dm > 0:
            r = o.digifil(v, freq_mhz=f, bw_mhz=b, nchan=nchan, freq_res=freq_res, tscrunch_factor=D, pol_mode=NAME[pol],
                          in_nbit=in_nbit, out_nbit=-32, keep_bandpass=True, return_float=True, dm=dm, coherent=True, nfilt=nfilt)
            d = np.asarray(r["float"], np.float64)
        else:
            x = o.decode_vdif(v, nbit=in_nbit, header_bytes=32, frame_bytes=8032)
            H = np.ones((nchan, freq_res), np.complex128)
            yP = o.filterbank_dedisp(x[0], nchan, freq_res, H, nfilt[0], nfilt[1])
            yQ = o.filterbank_dedisp(x[1], nchan, freq_res, H, nfilt[0], nfilt[1])
            d = o.tscrunch(o.detect(yP, yQ, NAME[pol]), D)
        out.append(d)
    n = min(d.shape[0] for d in out)
    return [d[:n] for d in out]


def slices(rows, ndm):
    """[t, ndm * trial elems] (or bytes) -> list of per-trial [t, trial elems]."""
    return [s for s in np.split(rows.reshape(rows.shape[0], -1), ndm, axis=1)]


# ---------------------------------------------------------------- 1: tuned path (nchan 128, 512 points)
T_DMS = [0.0, 150.0, 300.0, 560.0]
T_KW = dict(nchan=128, tscrunch=16, pol_mode=COH, chunk_units=4, coherent=True)


def _case_t():
    bws, freqs = band(2)
    vd = streams(2, 700, 7100)
    nf = _nfilt(128, 16, T_DMS, bws, freqs)
    fl = [trial_floats(vd, bws, freqs, nchan=128, D=16, pol=COH, dm=d, nfilt=nf[:2], freq_res=512) for d in T_DMS]
    return vd, bws, freqs, nf, fl


def test_tuned_trials_against_the_oracle(gpu):
    """One LSB and one USB IF, trials 0 / 150 / 300 / 560: float output of every trial, then 8-bit output against the oracle's
    own rescale_stats / digitise."""
    vd, bws, freqs, nf, fl = cached("t", _case_t)
    rows, info = run_plan(vd, bw=bws, freq=freqs, out_nbit=-32, keep_bandpass=True, dm_trials=T_DMS, **T_KW)
    g = info["geometry"]
    assert info["path"] == 0 and g.freq_res == 512 and g.ndm == 4 and (int(g.nfilt_pos), int(g.nfilt_neg)) == nf[:2]
    assert g.row_bytes == 4 * g.trial_row_bytes == 4 * 2 * 4 * 128 * 4
    for k, part in enumerate(slices(rows, 4)):
        check_splice(part, expected_tiles(fl[k], bws, out_nbit=-32), info["if_order"], pol=COH, nchan=128, out_nbit=-32,
                     pol_major=False, what=f"tuned trial DM {T_DMS[k]}")
    nint = int(np.floor(0.05 / (16 * 128 / (BW * 1e6)) + 0.5))
    rows8, info8 = run_plan(vd, bw=bws, freq=freqs, out_nbit=8, interval=0.05, dm_trials=T_DMS, **T_KW)
    assert info8["rescale"][0].shape == (4, 2, 4, 128)
    for k, part in enumerate(slices(rows8, 4)):
        check_splice(part, expected_tiles(fl[k], bws, out_nbit=8, nint=nint), info8["if_order"], pol=COH, nchan=128, out_nbit=8,
                     pol_major=False, what=f"tuned trial DM {T_DMS[k]}, 8-bit")


def test_tuned_trials_match_single_dm_plans(gpu):
    """The largest trial is a single-DM plan at its DM, byte for byte; a trial's slice does not depend on the other trials."""
    vd, bws, freqs, _, _ = cached("t", _case_t)
    rows, _ = run_plan(vd, bw=bws, freq=freqs, out_nbit=8, interval=0.05, dm_trials=T_DMS, **T_KW)
    one, _ = run_plan(vd, bw=bws, freq=freqs, out_nbit=8, interval=0.05, dm=T_DMS[-1], **T_KW)
    parts = slices(rows, 4)
    assert np.array_equal(parts[-1], one)
    two, _ = run_plan(vd, bw=bws, freq=freqs, out_nbit=8, interval=0.05, dm_trials=[T_DMS[1], T_DMS[-1]], **T_KW)
    p2 = slices(two, 2)
    assert np.array_equal(p2[0], parts[1]) and np.array_equal(p2[1], parts[-1])


# ---------------------------------------------------------------- 2: generic path
G_CASES = {
    # nchan 512 -> -F512:1024 on the compile-time generic kernels; nchan 128 at DM 2000 needs L 4096: run-time kernels
    "nchan512-L1024": dict(nchan=512, D=4, dms=[0.0, 280.0, 560.0], nframes=300, chunk=100, L=1024, pol=COH),
    "nchan128-L4096": dict(nchan=128, D=16, dms=[0.0, 1000.0, 2000.0], nframes=330, chunk=120, L=4096, pol=I),
}


def _case_g(c):
    def make():
        bws, freqs = band(2)
        vd = streams(2, c["nframes"], 7200 + c["nchan"])
        nf = _nfilt(c["nchan"], c["D"], c["dms"], bws, freqs)
        fl = [trial_floats(vd, bws, freqs, nchan=c["nchan"], D=c["D"], pol=c["pol"], dm=d, nfilt=nf[:2], freq_res=c["L"])
              for d in c["dms"]]
        return vd, bws, freqs, nf, fl
    return make


@pytest.mark.parametrize("name", list(G_CASES))
def test_generic_trials_against_the_oracle_and_single_dm(gpu, name):
    c = G_CASES[name]
    vd, bws, freqs, nf, fl = cached(("g", name), _case_g(c))
    kw = dict(nchan=c["nchan"], bw=bws, freq=freqs, tscrunch=c["D"], pol_mode=c["pol"], out_nbit=-32, keep_bandpass=True,
              chunk_units=c["chunk"], coherent=True)
    rows, info = run_plan(vd, dm_trials=c["dms"], **kw)
    g = info["geometry"]
    assert info["path"] == 0 and g.freq_res == c["L"] and g.ndm == 3 and (int(g.nfilt_pos), int(g.nfilt_neg)) == nf[:2]
    parts = slices(rows, 3)
    for k, part in enumerate(parts):
        check_splice(part, expected_tiles(fl[k], bws, out_nbit=-32), info["if_order"], pol=c["pol"], nchan=c["nchan"],
                     out_nbit=-32, pol_major=False, what=f"generic {name} trial DM {c['dms'][k]}")
    one, _ = run_plan(vd, dm=c["dms"][-1], **kw)
    assert np.array_equal(parts[-1].view(np.uint8), one.view(np.uint8))


# ---------------------------------------------------------------- 4: modes
MODES = {
    "coherence-pol-major": dict(pol_mode=COH, splice_pol_major=True, tscrunch=16, out_nbit=8),
    "tscrunch-24": dict(pol_mode=I, tscrunch=24, out_nbit=16),
    "running-rescale": dict(pol_mode=I, tscrunch=16, out_nbit=8, rescale_mode=_lib.RESCALE_RUNNING),
    "8bit-input": dict(pol_mode=I, tscrunch=16, out_nbit=8, in_nbit=8),
}


@pytest.mark.parametrize("mode", list(MODES))
def test_trial_modes(gpu, mode):
    """Product-major splice inside each trial, kd_sum_rows over every (trial, IF) slot, the running rescale per trial and 8-bit
    input: the largest trial equals the single-DM plan byte for byte and the DM-0 trial matches the oracle."""
    m = dict(MODES[mode])
    nbit = m.get("in_nbit", 2)
    bws, freqs = band(2)
    nframes = 700 if nbit == 2 else 2400
    vd = cached(("m", nbit), lambda: streams(2, nframes, 7300 + nbit, nbit=nbit))
    dms = [0.0, 200.0, 560.0]
    kw = dict(nchan=128, bw=bws, freq=freqs, interval=0.04, coherent=True, chunk_units=4, **m)
    rows, info = run_plan(vd, dm_trials=dms, **kw)
    one, _ = run_plan(vd, dm=dms[-1], **kw)
    parts = slices(rows.view(np.uint8), 3)
    assert np.array_equal(parts[-1], one.view(np.uint8).reshape(one.shape[0], -1))
    g = info["geometry"]
    D = m["tscrunch"]
    fl = trial_floats(vd, bws, freqs, nchan=128, D=D, pol=m["pol_mode"], dm=0.0, nfilt=(int(g.nfilt_pos), int(g.nfilt_neg)),
                      freq_res=512, in_nbit=nbit)
    nint = int(g.interval_rows)
    running = m.get("rescale_mode") == _lib.RESCALE_RUNNING
    view = np.uint16 if m["out_nbit"] == 16 else np.uint8
    check_splice(parts[0].view(view), expected_tiles(fl, bws, out_nbit=m["out_nbit"], nint=nint, running=running), info["if_order"],
                 pol=m["pol_mode"], nchan=128, out_nbit=m["out_nbit"], pol_major=m.get("splice_pol_major", False),
                 what=f"{mode}, DM 0 trial")


# ---------------------------------------------------------------- 5: runner
def _write(tmp_path, vd):
    paths = []
    for i, v in enumerate(vd):
        p = tmp_path / f"if{i}.vdif"
        v.tofile(p)
        paths.append(str(p))
    return paths


def _refdm(head):
    i = head.index(b"refdm") + 5
    return struct.unpack("<d", head[i:i + 8])[0]


def test_run_scan_writes_one_file_per_trial(gpu, tmp_path):
    vd, bws, freqs, _, _ = cached("t", _case_t)
    paths = _write(tmp_path, vd)
    cfg = PlanConfig(nchan=128, bw_mhz=bws, freq_mhz=freqs, tscrunch=16, pol_mode=COH, out_nbit=8, rescale_interval_s=0.05,
                     coherent=True, dm_trials=T_DMS)
    outs = [str(tmp_path / f"t{k}.fil") for k in range(4)]
    with Plan(cfg) as pl:
        res = pl.run_scan(paths, outs)
    rows, _ = run_plan(vd, bw=bws, freq=freqs, out_nbit=8, interval=0.05, dm_trials=T_DMS, nchan=128, tscrunch=16, pol_mode=COH,
                       coherent=True)
    with Plan(cfg) as pl:
        per_trial = pl.trial_rows(rows)
    assert res["rows"] == rows.shape[0]
    for k, f in enumerate(outs):
        data = open(f, "rb").read()
        hn = data.index(b"HEADER_END") + len(b"HEADER_END")
        assert _refdm(data[:hn]) == T_DMS[k]
        assert data[hn:] == per_trial[k].tobytes(), f"trial {k}"


def test_process_vdif_coherent_numdms(gpu, tmp_path):
    v = streams(1, 400, 7400)[0]
    src = tmp_path / "scan_if1.vdif"
    v.tofile(src)
    out = tmp_path / "out"
    out.mkdir()
    rc = process_vdif.main(["FRB1", str(src), "-l", "-f", "1254", "-b", str(BW), "--ra", "00:00:00", "--dec", "00:00:00",
                            "--nchan", "128", "--tscrunch", "16", "--start", "0", "--nsec", "0.08", "--keepBP",
                            "--coherent_dm", "100", "--coherent_numdms", "3", "--coherent_dmstep", "50", "--fil_out_dir", str(out)])
    assert rc == 0
    names = sorted(os.listdir(out))
    assert names == [f"scan_if1.vdif_pol2_DM{d:.2f}.fil" for d in (100.0, 150.0, 200.0)]
    for n, d in zip(names, (100.0, 150.0, 200.0)):
        assert _refdm(open(out / n, "rb").read(1024)) == d


# ---------------------------------------------------------------- 6: refusals
def test_trial_plan_refusals(gpu, tmp_path):
    vd, bws, freqs, _, _ = cached("t", _case_t)
    paths = _write(tmp_path, vd)
    cfg = PlanConfig(nchan=128, bw_mhz=bws, freq_mhz=freqs, tscrunch=16, pol_mode=COH, out_nbit=8, keep_bandpass=True,
                     coherent=True, dm_trials=[100.0, 200.0])
    with Plan(cfg) as pl:
        with pytest.raises(_lib.B2FError) as e:
            pl.pull_strided(0, 16, 2 * pl.row_bytes)
        assert e.value.code == _lib.EUNSUPPORTED
        with pytest.raises(_lib.B2FError) as e:
            pl.run_scan(paths, [str(tmp_path / "a.fil"), str(tmp_path / "b.fil")], part=(0, 2))
        assert e.value.code == _lib.EUNSUPPORTED
        fifo = tmp_path / "b.fifo"
        os.mkfifo(fifo)
        with pytest.raises(_lib.B2FError) as e:
            pl.run_scan(paths, [str(tmp_path / "a.fil"), str(fifo)])
        assert e.value.code == _lib.EINVAL and "FIFO" in e.value.message
        with pytest.raises(_lib.B2FError) as e:            # one path for a trial plan
            pl.run_scan(paths, str(tmp_path / "a.fil"))
        assert e.value.code == _lib.EINVAL
        # stats_only measures every trial's first interval and writes nothing
        pl.set_rescale(None)
        pl.run_scan(paths, None, stats_only=True)
        mean, scale = pl.rescale()
        assert mean.shape == (2, 2, 4, 128)
