"""digifil -K (inter-channel dispersion delays removed after detection): what is decided on the host (no device needed).

The oracle's delay stage aligns a dispersed pulse across a spliced two-IF band; the delay table is the cold-plasma law at
channel-sample resolution; every refusal of a -K plan is a B2F_EINVAL raised before libb2f looks for a GPU; process_vdif
parses --remove_delays and hands it to run_digifil."""
import ctypes as C
import inspect

import numpy as np
import pytest

import delay_oracle as dl
from oracle import digifil_oracle as o
from frb_baseband_b200 import _lib, dist, process_vdif, synth
from frb_baseband_b200.plan import Plan, PlanConfig

# ---------------------------------------------------------------- oracle known-answer test
KBW, KF0, KNCHAN, KDM = 16.0, 1208.0, 128, 300.0          # IF 1 LSB at 1208 MHz, IF 2 USB at 1224 MHz: 1200..1232 MHz
KN = 1 << 21                                               # 65.5 ms per IF at 32 MS/s
KT0 = 0.005                                                # arrival at the top of the band, s


def _pulse(fc, bw):
    """An impulse dispersed at KDM as one IF samples it (LSB: the spectrally inverted view, as test_oracle_kat builds it).
    It reaches sky frequency f at KT0 + D DM (f^-2 - f_top^-2), f_top the band's top edge."""
    k = np.arange(KN // 2 + 1)
    fbb = k * (2 * abs(bw)) / KN                           # MHz above the IF's lower edge
    fsky = fc - abs(bw) / 2 + fbb
    f_top = KF0 + KBW + KBW / 2
    shift = o.DISPERSION_CONSTANT * KDM / f_top ** 2 - KT0   # s: moves the arrival at f_top to KT0
    phi = 2 * np.pi * o.DISPERSION_CONSTANT * KDM * 1e6 / fsky + 2 * np.pi * fbb * 1e6 * shift
    x = np.fft.irfft(np.exp(1j * phi), KN)
    if bw < 0:
        x = x * (-1.0) ** np.arange(KN)
    return np.stack([x, x])


def _pulse_rows(remove):
    """Float rows [t, nchan] per IF of the two-IF band, coherently dedispersed, with or without -K at the band's reference."""
    ref = dist.band_reference_mhz(2, KF0, KBW, KNCHAN)
    vd = synth.make_vdif(4, seed=1, bw_mhz=KBW)
    nf = int(np.ceil(0.55 * o.smearing_samples(KF0, -KBW, KNCHAN, KDM)))
    out = {}
    for i, fc, bw in o.if_plan(2, KF0, KBW):
        kw = dict(freq_mhz=fc, bw_mhz=bw, nchan=KNCHAN, freq_res=512, dm=KDM, coherent=True, nfilt=(nf, nf), x=_pulse(fc, bw))
        if remove:
            r = dl.digifil_k(vd, delay_ref_mhz=ref, **kw)
        else:
            r = o.digifil(vd, out_nbit=-32, keep_bandpass=True, return_float=True, **kw)
        out[i] = r["float"][:, 0, :]
    n = min(v.shape[0] for v in out.values())
    return [out[1][:n], out[2][:n]], ref


def test_dispersed_pulse_is_aligned_across_the_spliced_band():
    (lo, hi), ref = _pulse_rows(True)
    peaks = np.concatenate([lo.argmax(axis=0), hi.argmax(axis=0)])
    assert peaks.max() - peaks.min() <= 1, (peaks.min(), peaks.max())
    assert 0 < peaks.min()
    # without -K the peaks follow the delay table of each IF against the band's reference
    (lo0, hi0), _ = _pulse_rows(False)
    d = np.concatenate([dl.channel_delays(KF0, -KBW, KNCHAN, KDM, ref), dl.channel_delays(KF0 + KBW, KBW, KNCHAN, KDM, ref)])
    p0 = np.concatenate([lo0.argmax(axis=0), hi0.argmax(axis=0)])
    assert d.max() > 4000                                  # 44 ms of sweep across the band
    assert (p0 - d).max() - (p0 - d).min() <= 1
    assert abs(int(np.median(p0 - d)) - int(np.median(peaks))) <= 1


def test_rows_of_the_delay_stage():
    """out[r][p][c] = sum_{k<D} det[r D + k + d_c][p][c]; floor((K0 - d_max) / D) rows."""
    rng = np.random.default_rng(5)
    det = rng.standard_normal((1000, 2, 8))
    dly = np.array([0, 3, 7, 11, 20, 21, 40, 99])
    out = dl.remove_delays_stage(det, dly, 16)
    assert out.shape == ((1000 - 99) // 16, 2, 8)
    for r in (0, 5, out.shape[0] - 1):
        for c in range(8):
            assert np.allclose(out[r, :, c], det[r * 16 + dly[c]: r * 16 + dly[c] + 16, :, c].sum(axis=0))


def test_base2fil_aligns_every_if_to_the_band():
    """base2fil passes the band's top channel centre to every IF: splice's shortest input leaves the rows of the IF with the
    largest delay, the same count a GPU plan of the whole band gives."""
    nif, bw, nchan, dm = 3, 16.0, 64, 50.0
    vd = {i: synth.make_vdif(300, seed=40 + i, bw_mhz=bw) for i in range(1, nif + 1)}
    out = dl.base2fil_k(vd, nif=nif, freq_lsb0=1300.0, bw=bw, nchan=nchan, dm=dm)
    ref = dist.band_reference_mhz(nif, 1300.0, bw, nchan)
    assert out["fch1"] == pytest.approx(ref)
    dmax = max(dl.channel_delays(fc, sbw, nchan, dm, ref).max() for _, fc, sbw in o.if_plan(nif, 1300.0, bw))
    k0 = 300 * 16000 // (2 * nchan * 512) * 512           # channel samples: whole blocks of 2 nchan 512 samples
    assert dmax > 0 and out["data"].shape[0] == k0 - dmax


# ---------------------------------------------------------------- delay table
def test_delay_table_by_hand():
    """An LSB IF at 1254 MHz, 32 MHz, 4 channels of 8 MHz (tsamp0 0.125 us): centres 1266, 1258, 1250, 1242 MHz."""
    K = 1.0 / 2.41e-4
    dm, tsamp0 = 100.0, 4 / 32e6
    want = [0, round(K * dm * (1 / 1258 ** 2 - 1 / 1266 ** 2) / tsamp0), round(K * dm * (1 / 1250 ** 2 - 1 / 1266 ** 2) / tsamp0),
            round(K * dm * (1 / 1242 ** 2 - 1 / 1266 ** 2) / tsamp0)]
    assert want[3] == 80817                                # 10.1 ms
    assert list(dl.channel_delays(1254.0, -32.0, 4, dm)) == want
    # USB: the same sky channels in the opposite order; an explicit reference 34 MHz higher adds to every channel
    assert list(dl.channel_delays(1254.0, 32.0, 4, dm)) == want[::-1]
    far = dl.channel_delays(1254.0, -32.0, 4, dm, 1300.0)
    assert far[0] == round(K * dm * (1 / 1266 ** 2 - 1 / 1300 ** 2) / tsamp0) > 0 and np.all(np.diff(far) > 0)
    assert not dl.channel_delays(1254.0, -32.0, 4, 0.0).any()


def test_band_reference_is_the_spliced_fch1():
    for nif, f0, bw, nchan in ((8, 1254.0, 32.0, 128), (3, 1300.0, 16.0, 64), (1, 1400.0, 8.0, 1024)):
        top = max(fc for _, fc, _ in o.if_plan(nif, f0, bw))
        assert dist.band_reference_mhz(nif, f0, bw, nchan) == top + bw / 2 - bw / (2 * nchan)


# ---------------------------------------------------------------- refusals before the device
def _cfg(**kw):
    base = dict(nchan=128, bw_mhz=[-32.0, 32.0], freq_mhz=[1254.0, 1286.0], dm=300.0, remove_delays=True)
    base.update(kw)
    return PlanConfig(**base)


@pytest.mark.parametrize("kw,what", [
    (dict(delay_ref_mhz=1300.0), "at least"),              # top channel centre is 1301.875 MHz
    (dict(delay_ref_mhz=float("nan")), "delay_ref_mhz"),
    (dict(delay_ref_mhz=float("inf")), "delay_ref_mhz"),
    (dict(dm=-1.0), "dm >= 0"),
    (dict(dm=float("nan")), "finite dm"),
    (dict(freq_mhz=[10.0, 42.0]), "above 0 MHz"),
    (dict(remove_delays=False, delay_ref_mhz=1400.0), "needs remove_delays"),
], ids=["ref-below-top", "ref-nan", "ref-inf", "dm-negative", "dm-nan", "channel-below-0", "ref-without-K"])
def test_refusals_come_before_the_device(kw, what):
    with pytest.raises(_lib.B2FError) as e:
        Plan(_cfg(**kw))
    assert e.value.code == _lib.EINVAL and what in e.value.message, e.value.message


def test_remove_delays_flag_values():
    p = _lib.Params()
    p.struct_size = C.sizeof(p)
    p.nif, p.nchan, p.pol_mode, p.out_nbit, p.in_nbit, p.frame_bytes, p.header_bytes = 1, 128, _lib.POL_I, 8, 2, 8032, 32
    p.bw_mhz[0], p.freq_mhz[0], p.dm, p.remove_delays = 32.0, 1400.0, 100.0, 2
    h = C.c_void_p()
    assert _lib.lib().b2f_plan_create(C.byref(p), C.byref(h)) == _lib.EINVAL
    assert b"remove_delays must be 0 or 1" in _lib.lib().b2f_last_error()


def test_valid_plans_reach_the_device_check():
    if _lib.lib().b2f_device_count() > 0:
        pytest.skip("GPU present: the plan would be created")
    for kw in (dict(), dict(delay_ref_mhz=1400.0), dict(dm=0.0), dict(coherent=True), dict(dm=0.0, coherent=True, dm_trials=[0.0, 300.0])):
        with pytest.raises(_lib.B2FError) as e:
            Plan(_cfg(**kw))
        assert e.value.code == _lib.ECUDA, kw


# ---------------------------------------------------------------- process_vdif
def test_process_vdif_remove_delays_flag(tmp_path, monkeypatch):
    a = process_vdif.options(["FRB1", "/data/x.vdif", "-u", "--coherent_dm", "300", "--remove_delays"])
    assert a.remove_delays and a.coherent_dm == 300.0
    assert not process_vdif.options(["FRB1", "/data/x.vdif", "-u"]).remove_delays
    sig = inspect.signature(process_vdif.run_digifil)
    assert list(sig.parameters)[-1] == "remove_delays" and sig.parameters["remove_delays"].default is False
    seen = {}
    monkeypatch.setattr(process_vdif, "run_digifil", lambda *args, **kw: seen.update(kw) or "x.fil")
    for extra, trials in (([], None), (["--coherent_numdms", "3", "--coherent_dmstep", "100"], [300.0, 400.0, 500.0])):
        seen.clear()
        process_vdif.main(["FRB1", str(tmp_path / "x.vdif"), "-u", "--ra", "0", "--dec", "0", "--coherent_dm", "300",
                           "--remove_delays"] + extra)
        assert seen["remove_delays"] is True and seen["dm"] == 300.0 and seen["dm_trials"] == trials
