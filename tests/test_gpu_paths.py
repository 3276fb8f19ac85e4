"""The three channeliser paths (round-1 kernels, the round-2 kernels as two launches, the fused kernel with the
L2 ring) against the oracle on the same inputs, and against each other.  B2F_PATH selects the path at plan creation."""
import numpy as np
import pytest

from oracle import digifil_oracle as o
from frb_baseband_b200 import _lib, synth
from frb_baseband_b200.plan import Plan, PlanConfig
from helpers import REL_TOL, assert_rel, run_plan

pytestmark = pytest.mark.gpu

PATHS = {"legacy": 0, "split": 1, "fused": 2}


def _rows(monkeypatch, path, vdifs, **kw):
    monkeypatch.setenv("B2F_PATH", path)
    rows, info = run_plan(vdifs, **kw)
    return rows, info


@pytest.mark.parametrize("nchan,bw,D,nfr", [(128, 32.0, 16, 2048 + 512), (32, 16.0, 32, 700), (64, 32.0, 1, 600),
                                            (128, 32.0, 512, 2048), (8, 16.0, 4, 200), (256, 32.0, 8, 1024),
                                            (16, 16.0, 64, 400), (128, 32.0, 4, 1024), (128, 32.0, 2, 600),
                                            (128, 32.0, 64, 1024), (128, 32.0, 1, 600)])
def test_paths_match_oracle_float(gpu, monkeypatch, nchan, bw, D, nfr):
    """-b-32 -I0 rows of every path within 1e-5 of the oracle (faulty frames included)."""
    v = synth.make_vdif(nfr, seed=900 + nchan, bw_mhz=bw, tone_frac=0.27, invalid_frac=0.004, fill_frac=0.004)
    ref = o.digifil(v, freq_mhz=1400.0, bw_mhz=-bw, nchan=nchan, tscrunch_factor=D, out_nbit=-32, keep_bandpass=True)
    ref = ref["data"].astype(np.float64)
    for name, code in PATHS.items():
        monkeypatch.setenv("B2F_PATH", name)
        with Plan(PlanConfig(nchan=nchan, bw_mhz=[-bw])) as probe:
            assert probe.path == code, f"B2F_PATH={name} gave path {probe.path}"
        rows, info = _rows(monkeypatch, name, [v], nchan=nchan, bw=[-bw], tscrunch=D, out_nbit=-32, keep_bandpass=True)
        assert_rel(rows.reshape(ref.shape[0], 1, nchan), ref, REL_TOL, f"{name} nchan {nchan} D {D}")
        c = info["counters"]
        assert c["frames_ok"] + c["frames_invalid"] + c["frames_with_fill"] == nfr, (name, c)


@pytest.mark.parametrize("path", ["fused", "split"])
@pytest.mark.parametrize("mode,name", [(_lib.POL_COHERENCE, "coherence"), (_lib.POL_IQUV, "IQUV")])
def test_round2_pol_modes_equal_round1(gpu, monkeypatch, mode, name, path):
    """The four-product modes of the round-2 kernels against the round-1 kernels (which test_pol_modes pins to the oracle).
    The round-2 kernels are built for Stokes I, coherence products and IQUV; the other products run on the round-1 kernels
    whatever B2F_PATH says."""
    nchan, bw, D = 128, 32.0, 16
    monkeypatch.setenv("B2F_PATH", path)
    with Plan(PlanConfig(nchan=nchan, bw_mhz=[bw], pol_mode=mode)) as probe:
        assert probe.path == PATHS[path]
    with Plan(PlanConfig(nchan=nchan, bw_mhz=[bw], pol_mode=_lib.POL_PPQQ)) as probe:
        assert probe.path in (0, PATHS[path])
    v = synth.make_vdif(1024, seed=77, bw_mhz=bw, tone_frac=0.2, rho=0.4)
    kw = dict(nchan=nchan, bw=[bw], tscrunch=D, pol_mode=mode, out_nbit=-32, keep_bandpass=True)
    leg, _ = _rows(monkeypatch, "legacy", [v], **kw)
    fus, info = _rows(monkeypatch, path, [v], **kw)
    nprod = info["nprod"]
    assert_rel(fus.reshape(-1, nprod, nchan), leg.reshape(-1, nprod, nchan).astype(np.float64), 2e-6, name)


def test_fused_many_rounds_multi_if_8bit(gpu, monkeypatch):
    """C2 geometry, 8 IFs, two pushes (dozens of ring rounds per launch):
    8-bit rows of the fused kernel within 1 LSB of the round-1 kernels and identical between two runs (the
    inter-warp ordering through the ring is deterministic in its results)."""
    nchan, bw, D, nif = 128, 32.0, 16, 8
    vs = [synth.make_vdif(3 * 1024, seed=500 + i, bw_mhz=bw, tone_frac=0.1 * (i + 1)) for i in range(nif)]
    bws = [bw if i % 2 else -bw for i in range(nif)]
    kw = dict(nchan=nchan, bw=bws, tscrunch=D, interval=0.4)
    leg, _ = _rows(monkeypatch, "legacy", vs, **kw)
    f1, _ = _rows(monkeypatch, "fused", vs, **kw)
    f2, _ = _rows(monkeypatch, "fused", vs, **kw)
    assert f1.shape == leg.shape
    assert np.array_equal(f1, f2)
    d = np.abs(f1.astype(int) - leg.astype(int))
    assert d.max() <= 1 and (d != 0).mean() < 1e-3
