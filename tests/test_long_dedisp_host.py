"""Coherent dedispersion with overlap-save transforms of 8192..65536 points: what is decided on the host (no device needed).

Few wide channels give the finest time resolution but the most smearing per channel.  With dedispersion, nchan 8..64 may
use transforms of up to 2^20 / (2 nchan) points; everything else is refused as before, with a message that names the cap."""
import pytest

from frb_baseband_b200 import _lib, job_policy
from frb_baseband_b200.plan import Plan, PlanConfig

BAND = dict(bw_mhz=[-32.0], freq_mhz=[1254.0])


def _no_gpu():
    if _lib.lib().b2f_device_count() > 0:
        pytest.skip("GPU present: the plan would be created")


@pytest.mark.parametrize("kw", [
    dict(nchan=8, dm=349.0), dict(nchan=8, dm=560.0),
    dict(nchan=16, dm=349.0), dict(nchan=16, dm=560.0),
    dict(nchan=32, dm=1000.0), dict(nchan=32, dm=3000.0),
    dict(nchan=64, dm=6000.0), dict(nchan=64, dm=100.0, freq_res=8192),
    dict(nchan=8, dm=100.0, freq_res=65536), dict(nchan=16, dm_trials=[100.0, 300.0, 560.0]),
], ids=lambda kw: "-".join(f"{k}{v}" for k, v in kw.items()))
def test_long_shapes_reach_the_device_check(kw):
    _no_gpu()
    with pytest.raises(_lib.B2FError) as e:
        Plan(PlanConfig(coherent=True, **BAND, **kw))
    assert e.value.code == _lib.ECUDA, e.value.message


@pytest.mark.parametrize("kw,cap", [
    (dict(nchan=8, dm=1000.0, coherent=True), 65536),           # smearing beyond the cap of nchan 8
    (dict(nchan=64, dm=7000.0, coherent=True), 8192),
    (dict(nchan=128, freq_res=8192, dm=100.0, coherent=True), 4096),
    (dict(nchan=8, freq_res=8192), 65536),                        # no dedispersion
    (dict(nchan=8, freq_res=8192, dm=100.0), 65536),              # a DM without coherent = 1
    (dict(nchan=32, freq_res=32768, dm=100.0, coherent=True), 16384),
], ids=["nchan8-dm1000", "nchan64-dm7000", "nchan128-fr8192", "no-dm", "incoherent", "nchan32-fr32768"])
def test_refusals_name_the_cap(kw, cap):
    with pytest.raises(_lib.B2FError) as e:
        Plan(PlanConfig(**BAND, **kw))
    assert e.value.code == _lib.EUNSUPPORTED and f"{cap} " in e.value.message and f"nchan {kw['nchan']}" in e.value.message, e.value.message


def test_nchan32_search_ladder_passes_validation():
    """8 IF x 32 MHz at 1.25 GHz, nchan 32: the ladder to DM 1500 has 52 trials and needs 16384 points."""
    _no_gpu()
    p = job_policy.coherent_search_plan(1500.0, 1238.0 + 32.0, 32.0, 8, nchan_if=32)
    assert len(p.dm_trials) == 52 and 1500 < p.dm_trials[-1] < 1510
    bws = [-32.0 if i % 2 == 0 else 32.0 for i in range(8)]
    freqs = [1254.0 + 32.0 * i for i in range(8)]
    with pytest.raises(_lib.B2FError) as e:
        Plan(PlanConfig(nchan=32, bw_mhz=bws, freq_mhz=freqs, tscrunch=p.tscrunch, coherent=True, dm_trials=list(p.dm_trials)))
    assert e.value.code == _lib.ECUDA, e.value.message
    with pytest.raises(ValueError):                  # nchan 16: more than 64 trials
        job_policy.coherent_search_plan(1500.0, 1238.0 + 32.0, 32.0, 8, nchan_if=16)
