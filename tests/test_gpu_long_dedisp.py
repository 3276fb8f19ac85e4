"""Coherent dedispersion with overlap-save transforms of 8192..65536 points (nchan 8..64), against the oracle in float64.

Each case runs o.digifil with the plan's own nfilt and freq_res and checks that the plan chose a transform longer than 4096
points.  Pushes are shorter than a block, so blocks straddle pushes (and, with several IFs, the batches straddle IFs)."""
import numpy as np
import pytest

from oracle import digifil_oracle as o
from frb_baseband_b200 import _lib
from frb_baseband_b200.plan import Plan, PlanConfig
from helpers import run_plan
from test_gpu_multi_if import BW, COH, I, IQUV, PPQQ, NAME, band, cached, check_splice, expected_tiles, oracle_floats, streams

pytestmark = pytest.mark.gpu


def geometry(nchan, bws, freqs, D, **kw):
    with Plan(PlanConfig(nchan=nchan, bw_mhz=bws, freq_mhz=freqs, tscrunch=D, coherent=True, **kw)) as pl:
        g = pl.geometry
        return (int(g.nfilt_pos), int(g.nfilt_neg)), int(g.freq_res)


# name: nchan, DM, freq_res expected, IFs (first IF LSB, alternating), pol, D, frames, push, in_nbit, extra plan / oracle args
CASES = {
    "nchan8-dm349-I": dict(nchan=8, dm=349.0, L=65536, nif=1, pol=I, D=1, nframes=200, chunk=70),
    "nchan16-dm560-coh-usb": dict(nchan=16, dm=560.0, L=32768, nif=1, pol=COH, D=2, nframes=200, chunk=90, usb=True),
    "nchan32-dm1000-iquv-3if": dict(nchan=32, dm=1000.0, L=16384, nif=3, pol=IQUV, D=4, nframes=200, chunk=40),
    "nchan64-fr8192-ppqq": dict(nchan=64, dm=200.0, L=8192, nif=1, pol=PPQQ, D=8, nframes=160, chunk=50, freq_res=8192),
    "8bit-faults": dict(nchan=32, dm=300.0, L=8192, nif=2, pol=I, D=4, nframes=400, chunk=130, freq_res=8192, in_nbit=8),
    "1bit": dict(nchan=16, dm=349.0, L=32768, nif=1, pol=I, D=2, nframes=120, chunk=50, in_nbit=1),
    "ja98": dict(nchan=16, dm=349.0, L=32768, nif=2, pol=COH, D=16, nframes=200, chunk=70, decode="ja98"),
    "tscrunch24": dict(nchan=32, dm=1000.0, L=16384, nif=1, pol=I, D=24, nframes=200, chunk=60),
}


def _case(name):
    c = CASES[name]

    def make():
        if c.get("usb"):
            bws, freqs = [BW], [1286.0]
        else:
            bws, freqs = band(c["nif"])
        nbit = c.get("in_nbit", 2)
        faults = None if nbit == 8 else [{}] * c["nif"]
        vd = streams(c["nif"], c["nframes"], 9100 + c["nchan"] + 13 * nbit, nbit=nbit, faults=faults)
        kw = {"freq_res": c["freq_res"]} if "freq_res" in c else {}
        nf, L = geometry(c["nchan"], bws, freqs, c["D"], dm=c["dm"], **kw)
        fl = oracle_floats(vd, bws, freqs, nchan=c["nchan"], D=c["D"], pol=c["pol"], freq_res=L, in_nbit=nbit, dm=c["dm"], nfilt=nf,
                           decode_mode=c.get("decode", "static"))
        return vd, bws, freqs, nf, L, fl
    return cached(("long", name), make)


def _plan_kw(c, bws, freqs):
    kw = dict(nchan=c["nchan"], bw=bws, freq=freqs, tscrunch=c["D"], pol_mode=c["pol"], in_nbit=c.get("in_nbit", 2),
              chunk_units=c["chunk"], coherent=True)
    if "freq_res" in c:
        kw["freq_res"] = c["freq_res"]
    if c.get("decode") == "ja98":
        kw["decode_mode"] = _lib.DECODE_JA98
    return kw


@pytest.mark.parametrize("name", list(CASES))
def test_long_dedispersion_against_the_oracle(gpu, name):
    c = CASES[name]
    vd, bws, freqs, nf, L, fl = _case(name)
    assert L == c["L"] > 4096
    rows, info = run_plan(vd, out_nbit=-32, keep_bandpass=True, dm=c["dm"], **_plan_kw(c, bws, freqs))
    g = info["geometry"]
    assert int(g.freq_res) == c["L"] and (int(g.nfilt_pos), int(g.nfilt_neg)) == nf
    if c.get("in_nbit") == 8:
        assert info["counters"]["frames_invalid"] > 0
    check_splice(rows, expected_tiles(fl, bws, out_nbit=-32), info["if_order"], pol=c["pol"], nchan=c["nchan"], out_nbit=-32,
                 pol_major=False, what=name)


@pytest.mark.parametrize("out_nbit,running", [(8, False), (2, False), (8, True), (2, True)])
def test_long_dedispersion_integer_output(gpu, out_nbit, running):
    """Requantised output, digifil -c statistics of the first interval or a running rescale, against the oracle's own
    rescale_stats / digitise on its floats."""
    c = CASES["nchan16-dm560-coh-usb"]
    vd, bws, freqs, nf, L, fl = _case("nchan16-dm560-coh-usb")
    interval = 0.004
    kw = _plan_kw(c, bws, freqs)
    if running:
        kw["rescale_mode"] = _lib.RESCALE_RUNNING
    rows, info = run_plan(vd, out_nbit=out_nbit, interval=interval, dm=c["dm"], **kw)
    nint = int(info["geometry"].interval_rows)
    check_splice(rows, expected_tiles(fl, bws, out_nbit=out_nbit, nint=nint, running=running), info["if_order"], pol=c["pol"],
                 nchan=c["nchan"], out_nbit=out_nbit, pol_major=False, what=f"{out_nbit}-bit, running={running}")


TRIALS = [100.0, 300.0, 560.0]


def test_long_trials_against_the_oracle_and_single_dm(gpu):
    """Trials at nchan 16 share the forward transforms; each slice matches the oracle at its DM with the plan's nfilt and
    freq_res (those of the largest trial), and the largest trial equals a single-DM plan byte for byte."""
    from test_gpu_dm_trials import slices, trial_floats
    c = CASES["nchan16-dm560-coh-usb"]
    vd, bws, freqs, nf, L, _ = _case("nchan16-dm560-coh-usb")
    kw = _plan_kw(c, bws, freqs)
    rows, info = run_plan(vd, out_nbit=-32, keep_bandpass=True, dm_trials=TRIALS, **kw)
    g = info["geometry"]
    assert int(g.freq_res) == L == 32768 and (int(g.nfilt_pos), int(g.nfilt_neg)) == nf and g.ndm == 3
    parts = slices(rows, 3)
    for k, part in enumerate(parts):
        fl = trial_floats(vd, bws, freqs, nchan=16, D=c["D"], pol=c["pol"], dm=TRIALS[k], nfilt=nf, freq_res=L)
        check_splice(part, expected_tiles(fl, bws, out_nbit=-32), info["if_order"], pol=c["pol"], nchan=16, out_nbit=-32,
                     pol_major=False, what=f"trial DM {TRIALS[k]}")
    one, _ = run_plan(vd, out_nbit=-32, keep_bandpass=True, dm=TRIALS[-1], **kw)
    assert np.array_equal(parts[-1].view(np.uint8), one.view(np.uint8).reshape(one.shape[0], -1))


def test_long_ja98_refuses_unaligned_blocks(gpu):
    """JA98 levels are per window of 512 samples: nchan 8 at DM 349 with tscrunch 1 gives blocks that do not start on
    multiples of 512 samples, which stays refused on the long path too."""
    with pytest.raises(_lib.B2FError) as e:
        Plan(PlanConfig(nchan=8, bw_mhz=[-BW], freq_mhz=[1254.0], coherent=True, dm=349.0, decode_mode=_lib.DECODE_JA98))
    assert e.value.code == _lib.EUNSUPPORTED and "512" in e.value.message


def test_long_run_scan_file_and_time_parts(gpu, tmp_path):
    """b2f_run_scan file -> file equals the streaming calls, and 2 or 3 time parts give the same file byte for byte."""
    bws, freqs = [-BW], [1254.0]
    nfr = 3600
    v = streams(1, nfr, 9500, faults=[{}])[0]
    path = tmp_path / "if1.vdif"
    v.tofile(path)
    kw = dict(nchan=16, bw_mhz=bws, freq_mhz=freqs, tscrunch=128, coherent=True, dm=560.0, rescale_interval_s=0.1)
    whole = tmp_path / "whole.fil"
    with Plan(PlanConfig(**kw)) as pl:
        assert int(pl.geometry.freq_res) == 32768
        r = pl.run_scan([str(path)], str(whole), source_name="S")
        assert r["rows"] > 0
    ref = open(whole, "rb").read()
    rows, _ = run_plan([v], nchan=16, bw=bws, freq=freqs, tscrunch=128, coherent=True, dm=560.0, interval=0.1)
    hn = ref.index(b"HEADER_END") + len(b"HEADER_END")
    assert ref[hn:] == rows.tobytes()
    for n in (2, 3):
        out = tmp_path / f"parts{n}.fil"
        with Plan(PlanConfig(**kw)) as pl:
            pl.run_scan([str(path)], None, stats_only=True)
            pl.set_rescale(*pl.rescale())
            got = sum(pl.run_scan([str(path)], str(out), source_name="S", part=(k, n))["rows"] for k in reversed(range(n)))
        assert got == r["rows"]
        assert open(out, "rb").read() == ref, f"{n} parts differ from the single run"
