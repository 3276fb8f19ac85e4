"""digifil -K in the oracle's terms: the inter-channel dispersion delay stage that DSPSR's SampleDelay applies after detection
(recalled, not pinned -- SURVEY Appendix A), on top of oracle.digifil_oracle.

Order, as in DSPSR: Detection -> SampleDelay -> TScrunch -> Rescale.  `digifil_k` takes the oracle's detected floats at
tscrunch 1 and applies the delay stage and the integration; `base2fil_k` aligns every IF of a scan to the centre of the
band's highest channel and splices, so that splice's shortest-input rule leaves the rows of the IF with the largest delay."""
import numpy as np

from oracle import digifil_oracle as o


def channel_delays(freq_mhz: float, bw_mhz: float, nchan: int, dm: float, ref_mhz: float | None = None) -> np.ndarray:
    """Delay of each channel in channel samples of tsamp0 = nchan/|BW| us, natural channel order.

    Channel c has the sky centre o.chirp uses, f_c = FREQ - BW/2 + (c+0.5)*BW/N (BW signed), and
        d_c = llround(D * DM * (f_c^-2 - f_ref^-2) / tsamp0)
    with D = o.DISPERSION_CONSTANT.  f_ref defaults to the centre of this IF's highest channel."""
    chbw = bw_mhz / nchan
    fc = freq_mhz - bw_mhz / 2 + (np.arange(nchan) + 0.5) * chbw
    if ref_mhz is None:
        ref_mhz = freq_mhz + abs(bw_mhz) / 2 - abs(bw_mhz) / (2 * nchan)
    tsamp0 = nchan / (abs(bw_mhz) * 1e6)
    t = o.DISPERSION_CONSTANT * dm * (fc ** -2.0 - float(ref_mhz) ** -2.0) / tsamp0
    return np.array([int(np.floor(abs(v) + 0.5)) * (1 if v >= 0 else -1) for v in t], dtype=np.int64)   # C llround


def remove_delays_stage(d: np.ndarray, delays: np.ndarray, D: int) -> np.ndarray:
    """SampleDelay + TScrunch on detected d[t, prod, chan]: out[r][p][c] = sum_{k<D} d[r D + k + delays[c]][p][c].  There is
    no look-behind: floor((K0 - max delay) / D) rows, the tail dropped."""
    D = max(1, D)
    n = max(0, (d.shape[0] - int(delays.max())) // D)
    out = np.empty((n,) + d.shape[1:], dtype=d.dtype)
    for c, dc in enumerate(delays):
        out[:, :, c] = d[dc: dc + n * D, :, c].reshape(n, D, d.shape[1]).sum(axis=1)
    return out


def digifil_k(vdif, *, freq_mhz: float, bw_mhz: float, nchan: int, dm: float, tscrunch_factor: int = 1,
              delay_ref_mhz: float | None = None, **kw) -> dict:
    """digifil -D dm -K (with coherent=True also -F nchan:D): float rows [t, nprod, chan] in natural channel order under 'float',
    detected, delayed and integrated, without rescaling (digifil -I0).  Other keywords go to o.digifil."""
    r = o.digifil(vdif, freq_mhz=freq_mhz, bw_mhz=bw_mhz, nchan=nchan, dm=dm, tscrunch_factor=1, out_nbit=-32, keep_bandpass=True,
                  return_float=True, **kw)
    d = remove_delays_stage(np.asarray(r["float"], np.float64), channel_delays(freq_mhz, bw_mhz, nchan, dm, delay_ref_mhz),
                            tscrunch_factor)
    out = dict(r)
    out["float"] = d
    out["tsamp_s"] = r["tsamp_s"] * max(1, tscrunch_factor)
    out["data"] = (d[:, :, ::-1] if bw_mhz > 0 else d).astype(np.float32)      # file order: USB flipped, foff < 0
    return out


def base2fil_k(vdifs: dict, *, nif: int, freq_lsb0: float, bw: float, nchan: int, dm: float, **kw) -> dict:
    """All IFs of a scan with -K aligned to the centre of the band's highest channel, then splice."""
    top = max(fc for _, fc, _ in o.if_plan(nif, freq_lsb0, bw))
    ref = top + abs(bw) / 2 - abs(bw) / (2 * nchan)
    return o.splice([digifil_k(vdifs[i], freq_mhz=fc, bw_mhz=sbw, nchan=nchan, dm=dm, delay_ref_mhz=ref, **kw)
                     for i, fc, sbw in o.if_plan(nif, freq_lsb0, bw)])
