"""Coherent dedispersion at several trial DMs: what is decided on the host (no device needed).

Every refusal of a trial plan is a B2F_EINVAL raised before libb2f looks for a GPU; the search policy spaces the trials so
that no DM up to the ceiling keeps more smearing than the time resolution; process_vdif parses the trial flags and names
one file per trial."""
import ctypes as C
import math

import pytest

from frb_baseband_b200 import _lib, job_policy, process_vdif
from frb_baseband_b200.plan import Plan, PlanConfig


def _cfg(**kw):
    base = dict(nchan=128, bw_mhz=[-32.0, 32.0], freq_mhz=[1254.0, 1286.0], coherent=True, dm_trials=[0.0, 150.0, 300.0])
    base.update(kw)
    return PlanConfig(**base)


@pytest.mark.parametrize("kw,what", [
    (dict(coherent=False), "coherent = 1"),
    (dict(dm=100.0), "dm must be 0"),
    (dict(dm_trials=[0.0, 150.0, 150.0]), "strictly increasing"),
    (dict(dm_trials=[300.0, 150.0]), "strictly increasing"),
    (dict(dm_trials=[-1.0, 150.0]), ">= 0"),
    (dict(dm_trials=[0.0, float("nan")]), "finite"),
    (dict(dm_trials=[0.0, float("inf")]), "finite"),
    (dict(dm_trials=[0.0]), "largest trial DM must be > 0"),
], ids=["not-coherent", "dm-set", "repeated", "decreasing", "negative", "nan", "inf", "only-zero"])
def test_trial_refusals_come_before_the_device(kw, what):
    with pytest.raises(_lib.B2FError) as e:
        Plan(_cfg(**kw))
    assert e.value.code == _lib.EINVAL and what in e.value.message, e.value.message


def test_too_many_trials():
    with pytest.raises(_lib.B2FError) as e:
        Plan(_cfg(dm_trials=[float(k) for k in range(_lib.B2F_MAX_DM + 1)]))
    assert e.value.code == _lib.EINVAL
    # the C side refuses an ndm beyond the array as well
    p = _lib.Params()
    p.struct_size = C.sizeof(p)
    p.ndm = _lib.B2F_MAX_DM + 1
    p.nif, p.nchan, p.pol_mode, p.out_nbit, p.in_nbit = 1, 128, _lib.POL_I, 8, 2
    h = C.c_void_p()
    assert _lib.lib().b2f_plan_create(C.byref(p), C.byref(h)) == _lib.EINVAL
    assert b"ndm" in _lib.lib().b2f_last_error()


def test_trial_refusals_of_the_largest_trial():
    """The geometry follows the largest trial, so today's refusals of a single DM apply to it."""
    with pytest.raises(_lib.B2FError) as e:          # smearing beyond 4096 channel samples at nchan 128
        Plan(_cfg(dm_trials=[0.0, 100000.0]))
    assert e.value.code == _lib.EUNSUPPORTED and "smearing" in e.value.message


def test_valid_trials_reach_the_device_check():
    if _lib.lib().b2f_device_count() > 0:
        pytest.skip("GPU present: the plan would be created")
    with pytest.raises(_lib.B2FError) as e:
        Plan(_cfg())
    assert e.value.code == _lib.ECUDA


# ---------------------------------------------------------------- policy
def _smear_us(ddm, chbw, f_min_ghz):
    return job_policy.K_SMEAR_US * ddm * chbw / f_min_ghz ** 3


def test_coherent_search_plan_c2_band():
    """8 IF x 32 MHz from 1238 MHz, nchan 128 (0.25 MHz channels), 64 us: 13 trials about 117 apart cover DM 0..1500."""
    p = job_policy.coherent_search_plan(None, 1238.0 + 32.0, 32.0, 8)
    assert p.coherent and p.nchan_if == 128 and p.tscrunch == 16 and p.t_res_us == 64 and p.dm == job_policy.UNKNOWN_DM
    t = p.dm_trials
    assert len(t) == 13
    step = t[1] - t[0]
    assert step == pytest.approx(117.0, abs=0.5)
    assert t[0] == pytest.approx(step / 2) and all(b - a == pytest.approx(step) for a, b in zip(t, t[1:]))
    assert t[-1] + step / 2 >= 1500 and t[-1] - step / 2 < 1500
    # every DM of [0, 1500] lies within half a step of a trial, and half a step leaves at most t_res of smearing
    for k, d in enumerate(t):
        assert _smear_us(step / 2, 0.25, 1.238) <= p.t_res_us * (1 + 1e-12)
        assert d - step / 2 == pytest.approx(k * step)
    # gpu_plan and search_plan are what they were
    assert job_policy.gpu_plan(560.0, 1270.0, 32.0, 8).dm_trials == ()
    assert job_policy.search_plan(None, 1270.0, 32.0, 8).dm_trials == ()


def test_coherent_search_plan_limits():
    p = job_policy.coherent_search_plan(100.0, 1270.0, 32.0, 8)
    assert len(p.dm_trials) == 1 and p.dm_trials[0] == pytest.approx(58.5, abs=0.5)
    with pytest.raises(ValueError):                  # 2 us resolution: hundreds of trials to DM 1500
        job_policy.coherent_search_plan(None, 1270.0, 32.0, 8, log2_t_res_us=1)
    n = math.ceil(1500 / (2 * 16 * 1.238 ** 3 / (8.3 * 0.25)))
    assert len(job_policy.coherent_search_plan(None, 1270.0, 32.0, 8, log2_t_res_us=4).dm_trials) == n <= 64


# ---------------------------------------------------------------- process_vdif
def test_process_vdif_trial_flags_and_names():
    a = process_vdif.options(["FRB1", "/data/x.vdif", "-u", "--coherent_dm", "100", "--coherent_numdms", "3",
                              "--coherent_dmstep", "50.5", "--fil_out_dir", "/out"])
    trials = process_vdif.coherent_trials(a.coherent_dm, a.coherent_numdms, a.coherent_dmstep)
    assert trials == [100.0, 150.5, 201.0]
    names = process_vdif.trial_output_paths("/data/x.vdif_pol2.hdr", a.fil_out_dir, trials)
    assert names == ["/out/x.vdif_pol2_DM100.00.fil", "/out/x.vdif_pol2_DM150.50.fil", "/out/x.vdif_pol2_DM201.00.fil"]
    assert process_vdif.trial_output_paths("/data/x.vdif_pol2.hdr", None, [0.0])[0] == "/data/x.vdif_pol2_DM0.00.fil"
    # one trial is today's single-DM run
    a1 = process_vdif.options(["FRB1", "/data/x.vdif", "-u", "--coherent_dm", "100"])
    assert a1.coherent_numdms == 1 and process_vdif.coherent_trials(a1.coherent_dm, 1, 0.0) is None
    with pytest.raises(process_vdif.InputError):
        process_vdif.coherent_trials(100.0, 3, 0.0)
    with pytest.raises(process_vdif.InputError):
        process_vdif.coherent_trials(100.0, 0, 10.0)


def test_process_vdif_trials_keep_existing_files(tmp_path):
    hdr = tmp_path / "x.vdif_pol2.hdr"
    hdr.write_text("")
    (tmp_path / "x.vdif_pol2_DM150.00.fil").write_bytes(b"old")
    with pytest.raises(process_vdif.InputError) as e:
        process_vdif.run_digifil(str(hdr), dm_trials=[100.0, 150.0])
    assert "exists already" in e.value.message
    with pytest.raises(process_vdif.InputError) as e:
        process_vdif.main(["FRB1", str(tmp_path / "x.vdif"), "-u", "--ra", "0", "--dec", "0", "--coherent_numdms", "2",
                           "--coherent_dmstep", "10", "--do_prepdata"])
    assert "prepdata" in e.value.message
