"""Channelisation policy: how many channels per IF and which tscrunch a scan gets, from the DM.

Host-side mirror of the chooser in /root/reference/submit_job.py:51-111 (SURVEY.md section 8 row N4).
The rule is the reference's: pick the channel width whose intra-channel dispersion smearing
8.3 us * DM * RBW[MHz] / f[GHz]^3 equals the wanted time resolution at the bottom of the band, round
the channel count up to a power of two (capped at 2^13 over the whole band), then integrate channel
samples up to the wanted time resolution.

`gpu_plan` is the B200 addition: with in-channel coherent dedispersion (b2f_params.coherent) the
smearing term vanishes, so the channel count is set by what the search downstream wants rather than
by the DM.  `coherent_search_plan` is its search form for an unknown DM: a ladder of trial DMs, each
coherently dedispersed (b2f_params.ndm / dm_trials), spaced so that the smearing left inside a channel
never exceeds the time resolution.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

K_SMEAR_US = 8.3            # submit_job.py:60 (us per MHz per pc/cc at 1 GHz)
MAX_BAND_CHANNELS = 2 ** 13   # submit_job.py:63
UNKNOWN_DM = 1500.0         # submit_job.py:52-54: Heimdall's search ceiling when the source has no DM
MAX_TRIAL_DMS = 64          # B2F_MAX_DM of include/b2f.h
FLAG_DIR = "/data1/franz/fetch/Standard/"   # submit_job.py:38


@dataclass
class ChannelPlan:
    nchan_band: int | float     # channels over all IFs (power of two)
    nchan_if: int               # --nchan for process_vdif / b2f_params.nchan
    tscrunch: int               # --tscrunch / b2f_params.tscrunch
    t_res_us: float             # time resolution after tscrunch
    f_min_mhz: int
    f_max_mhz: int
    coherent: bool = False
    dm: float = 0.0
    dm_trials: tuple = ()       # coherent trial DMs (coherent_search_plan), ascending

    def flag_file(self, telescope: str, flag_dir: str = FLAG_DIR) -> str:
        """RFI flag file FETCH is pointed at: submit_job.py:117"""
        return f"{flag_dir}{telescope}.flag_{self.f_min_mhz}-{self.f_max_mhz}MHz_{self.nchan_band}chan"


def _pow2_at_least(x: float) -> int:
    """smallest 2^i (i = 1..13) that is >= x; 2^13 when x is larger (submit_job.py:71-75)"""
    for i in range(1, 14):
        if x <= 2 ** i:
            return 2 ** i
    return 2 ** 13


def _channels_for(t_res_us: float, f_min_ghz: float, dm: float, band_mhz: float) -> float:
    rbw = t_res_us * f_min_ghz ** 3 / (K_SMEAR_US * dm)      # MHz
    return band_mhz / rbw


def _finish(nchan_band, nchan_if: int, t_res_us: float, f_min_ghz: float, if_mhz: float, band_mhz: float,
            **kw) -> ChannelPlan:
    # submit_job.py:106-111.  Nyquist sample 1/(2 IF) us; one channel sample = 2 nchan of them.
    t_samp = 1 / (2 * if_mhz) * 2 * nchan_if
    f_min = int(f_min_ghz * 1000)
    return ChannelPlan(nchan_band=nchan_band, nchan_if=nchan_if, tscrunch=int(t_res_us / t_samp), t_res_us=t_res_us,
                       f_min_mhz=f_min, f_max_mhz=int(f_min + band_mhz), **kw)


def search_plan(dm: float | None, fref_mhz: float, if_mhz: float, nif: int, *, log2_t_res_us: int = 6) -> ChannelPlan:
    """FRB search branch (submit_job.py:58-76)."""
    dm = UNKNOWN_DM if dm is None else dm
    f_min_ghz = (fref_mhz - if_mhz) / 1000
    band = float(nif) * if_mhz
    t_res = 2 ** log2_t_res_us
    n = _channels_for(t_res, f_min_ghz, dm, band)
    if n > MAX_BAND_CHANNELS:
        # smearing left in the widest allowed channel; if it is >= 100 us halve the time resolution instead
        smear_at_cap = band / MAX_BAND_CHANNELS * K_SMEAR_US * dm / f_min_ghz ** 3
        if smear_at_cap >= 100:
            t_res *= 2
            n = _channels_for(t_res, f_min_ghz, dm, band)
    nband = _pow2_at_least(n)
    return _finish(nband, int(nband / float(nif)), t_res, f_min_ghz, if_mhz, band, dm=dm)


def pulsar_plan(dm: float, period_s: float, fref_mhz: float, if_mhz: float, nif: int, *, log2_t_res_us: int = 6,
                nbins: int = 512, min_chan_if: int = 32) -> ChannelPlan:
    """Pulsar branch (submit_job.py:77-104): time resolution = period / 512 bins, rounded down to a power
    of two microseconds but never below 2^log2_t_res_us."""
    f_min_ghz = (fref_mhz - if_mhz) / 1000
    band = float(nif) * if_mhz
    t_res = period_s * 1e6 / nbins
    i = log2_t_res_us
    while True:
        p = 2 ** i
        if t_res == p:
            break
        if t_res < p:
            t_res = p / 2
            break
        i += 1
    nband = _pow2_at_least(_channels_for(t_res, f_min_ghz, dm, band))
    nif_f = float(nif)
    nchan_if = int(nband / nif_f)
    if nchan_if < min_chan_if:
        nchan_if = min_chan_if
        nband = nchan_if * nif_f      # a float in the reference too; it ends up in the flag-file name
    return _finish(nband, nchan_if, t_res, f_min_ghz, if_mhz, band, dm=dm)


def gpu_plan(dm: float | None, fref_mhz: float, if_mhz: float, nif: int, *, log2_t_res_us: int = 6,
             nchan_if: int = 128) -> ChannelPlan:
    """B200 policy: remove the intra-channel smearing exactly (coherent dedispersion inside the channels) and
    keep a fixed, search-friendly channel count.  With an unknown DM there is nothing to remove: fall back to
    the reference's rule."""
    if dm is None:
        return search_plan(dm, fref_mhz, if_mhz, nif, log2_t_res_us=log2_t_res_us)
    f_min_ghz = (fref_mhz - if_mhz) / 1000
    band = float(nif) * if_mhz
    return _finish(nchan_if * nif, nchan_if, 2 ** log2_t_res_us, f_min_ghz, if_mhz, band, coherent=True, dm=dm)


def coherent_search_plan(dm_max: float | None, fref_mhz: float, if_mhz: float, nif: int, *, log2_t_res_us: int = 6,
                         nchan_if: int = 128) -> ChannelPlan:
    """Search for an unknown DM with coherent dedispersion at a ladder of trial DMs, all in one pass over the baseband.

    A channel dedispersed at DM d keeps 8.3 us * |DM - d| * chbw / f_min^3 of smearing at the bottom of the band.  Trials
    `step` apart with step = 2 t_res f_min^3 / (8.3 chbw), at step/2 + k step, leave at most t_res for every DM in
    [0, dm_max].  More than MAX_TRIAL_DMS trials is a ValueError: use fewer channels' worth of time resolution or a lower
    dm_max.  With few wide channels the largest trial may need overlap-save transforms longer than 4096 points; libb2f
    takes up to 2^20 / (2 nchan) of them (nchan_if=32 at 1.25 GHz: 52 trials to DM 1500 on 16384 points), while nchan_if=16
    needs more than 64 trials to DM 1500 and stays a ValueError here."""
    dm_max = UNKNOWN_DM if dm_max is None else float(dm_max)
    if not dm_max > 0:
        raise ValueError(f"dm_max = {dm_max}: must be > 0")
    f_min_ghz = (fref_mhz - if_mhz) / 1000
    band = float(nif) * if_mhz
    t_res = 2 ** log2_t_res_us
    chbw = if_mhz / nchan_if
    step = 2 * t_res * f_min_ghz ** 3 / (K_SMEAR_US * chbw)
    n = max(1, math.ceil(dm_max / step - 1e-9))
    if n > MAX_TRIAL_DMS:
        raise ValueError(f"{n} trial DMs {step:.1f} apart are needed up to DM {dm_max} at {t_res} us, at most {MAX_TRIAL_DMS} fit one plan")
    trials = tuple(step / 2 + k * step for k in range(n))
    return _finish(nchan_if * nif, nchan_if, t_res, f_min_ghz, if_mhz, band, coherent=True, dm=dm_max, dm_trials=trials)


def create_config_argv(plan: ChannelPlan, *, vex: str, source: str, telescope: str, scan: str, config_file: str,
                       total_slots: int = 37, search: bool = True, flag_dir: str = FLAG_DIR) -> list[str]:
    """argv of the create_config.py call the reference issues once (submit_job.py:118; the reference then
    appends the string to itself by accident, `:119-122`, which we do not repeat)."""
    argv = ["create_config.py", "-i", vex, "-s", source, "-t", telescope, "-N", str(total_slots),
            "-d", str(plan.tscrunch), "-n", str(plan.nchan_if), "-S", scan, "-F", plan.flag_file(telescope, flag_dir),
            "--online", "-o", config_file]
    argv += ["--search"] if search else ["--pol", "4"]
    return argv
