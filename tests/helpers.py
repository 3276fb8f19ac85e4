"""Shared helpers for the parity tests."""
import numpy as np

from frb_baseband_b200 import synth
from frb_baseband_b200 import _lib
from frb_baseband_b200.plan import Plan, PlanConfig

#: float spectra tolerance stated by BASELINE.json's north_star
REL_TOL = 1e-5


def assert_rel(gpu, ref, tol=REL_TOL, what="", power=None):
    """|gpu-ref| <= tol * max(|ref|, rms(ref) per product).  Detected powers are sums of
    squares so |ref| is the natural scale; cross products may pass through zero, where the rms
    of the same product is used instead.  `power` (same shape as one product, [row][chan]): the
    total power PP + QQ of every sample -- the scale of a difference or cross product (Q = PP - QQ,
    Re/Im PQ*) in a channel that holds a strong line, where the product is a small difference of
    two large numbers and its rms over all channels says nothing about the rounding to expect."""
    gpu = np.asarray(gpu, np.float64)
    ref = np.asarray(ref, np.float64)
    assert gpu.shape == ref.shape, (gpu.shape, ref.shape)
    rms = np.sqrt((ref ** 2).mean(axis=(0, 2), keepdims=True)) if ref.ndim == 3 else np.sqrt((ref ** 2).mean())
    den = np.maximum(np.abs(ref), rms)
    if power is not None:
        den = np.maximum(den, np.asarray(power, np.float64)[:, None, :] if ref.ndim == 3 else power)
    err = np.abs(gpu - ref) / np.where(den > 0, den, 1.0)
    assert err.max() <= tol, f"{what}: max rel err {err.max():.3e} > {tol} at {np.unravel_index(err.argmax(), err.shape)}"
    return err.max()


def run_plan(vdifs, *, nchan, bw, tscrunch=1, pol_mode=_lib.POL_I, out_nbit=8, in_nbit=2, keep_bandpass=False,
             freq=None, interval=10.0, chunk_units=0, splice_pol_major=False, profile=False, **cfg_kw):
    """Push a list of per-IF VDIF arrays through a Plan chunk by chunk; return (rows, plan info).  `chunk_units`
    sets the push size (PlanConfig.chunk_units, 0 = the library default); other PlanConfig fields go in `cfg_kw`.
    Every pull is repeated until it returns nothing: the running rescale mode hands out one interval per pull."""
    cfg = PlanConfig(nchan=nchan, bw_mhz=list(bw), freq_mhz=freq, tscrunch=tscrunch, pol_mode=pol_mode,
                     out_nbit=out_nbit, in_nbit=in_nbit, keep_bandpass=keep_bandpass, chunk_units=chunk_units,
                     rescale_interval_s=interval, splice_pol_major=splice_pol_major, profile=profile, **cfg_kw)
    out = []

    def drain(pl):
        while True:
            r = pl.pull()
            if not len(r):
                return
            out.append(r.copy())

    with Plan(cfg) as pl:
        fb = cfg.frame_bytes
        nfr = min(v.size // fb for v in vdifs)
        cf = pl.chunk_frames
        for f0 in range(0, nfr, cf):
            n = min(cf, nfr - f0)
            pl.push([v[f0 * fb:(f0 + n) * fb] for v in vdifs])
            drain(pl)
        pl.flush()
        drain(pl)
        info = {"counters": pl.counters(), "rescale": pl.rescale(), "geometry": pl.geometry, "path": pl.path,
                "chunk_frames": int(cf), "nprod": pl.nprod, "if_order": pl.if_order,
                "times": pl.kernel_times() if profile else None}
        rows = pl.view_rows(np.concatenate(out)) if out else np.empty((0, pl.row_bytes), np.uint8)
    return rows, info
