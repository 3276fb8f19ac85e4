"""Scans of several IFs against the oracle run once per IF, on every channeliser path.

Every real scan has several IFs (base2fil hands over 4 to 16 subbands), and much of the code is per IF or spans IFs:
block indices that run over all IFs of a push (`ifi = gb / nblk`), batches of blocks that straddle IF boundaries, a chirp
table, a carry, word masks and JA98 levels per IF, statistics per (IF, product, channel), and the splice of the IF tiles
in `if_order`, in either layout.  Each IF here carries a visibly different signal (own seed, tone position, correlation
and fault mix), and a tile that fails names the IF whose reference it matches best."""
import numpy as np
import pytest

from oracle import digifil_oracle as o
from frb_baseband_b200 import _lib, synth
from frb_baseband_b200.plan import Plan, PlanConfig
from helpers import REL_TOL, assert_rel, run_plan

pytestmark = pytest.mark.gpu

BW = 32.0
FB = 8032
I, COH, IQUV, PPQQ = _lib.POL_I, _lib.POL_COHERENCE, _lib.POL_IQUV, _lib.POL_PPQQ
NAME = {I: "I", COH: "coherence", IQUV: "IQUV", PPQQ: "PPQQ"}

_cache = {}


def cached(key, make):
    """Streams and oracle spectra are shared by the parameter sets of one case: the oracle runs once per IF and case."""
    if key not in _cache:
        _cache[key] = make()
    return _cache[key]


def band(nif, f0=1254.0):
    """Subbands 32 MHz apart, alternating sidebands like base2fil's plan (first IF LSB): (signed bw, centre freq)."""
    return [BW if i % 2 else -BW for i in range(nif)], [f0 + BW * i for i in range(nif)]


def streams(nif, nframes, seed, *, nbit=2, faults=None):
    """One VDIF stream per IF.  `faults`: per IF dict of make_vdif fault fractions; default a different mix per IF."""
    mix = [{}, {"invalid_frac": 0.01}, {"fill_frac": 0.01}, {"invalid_frac": 0.01, "fill_frac": 0.01}]
    out = []
    for i in range(nif):
        f = faults[i] if faults is not None else mix[i % 4]
        out.append(synth.make_vdif(nframes, seed=seed + 7 * i, bw_mhz=BW, nbit=nbit, tone_frac=0.05 + (0.13 + 0.19 * i) % 0.9,
                                   tone_amp=0.3 + 0.1 * (i % 3), rho=0.1 + 0.07 * (i % 8), **f))
    return out


def oracle_floats(vd, bws, freqs, *, nchan, D, pol, freq_res=None, in_nbit=2, dm=0.0, nfilt=(0, 0), decode_mode="static"):
    """o.digifil in float64 once per IF with that IF's signed bw and centre: detected, integrated spectra [t, nprod, chan]
    in natural channel order, cut to the shortest IF."""
    out = []
    for v, b, f in zip(vd, bws, freqs):
        r = o.digifil(v, freq_mhz=f, bw_mhz=b, nchan=nchan, freq_res=freq_res, tscrunch_factor=D, pol_mode=NAME[pol], in_nbit=in_nbit,
                      out_nbit=-32, keep_bandpass=True, return_float=True, dm=dm, coherent=dm > 0, nfilt=nfilt, decode_mode=decode_mode)
        out.append(np.asarray(r["float"], np.float64))
    n = min(d.shape[0] for d in out)
    return [d[:n] for d in out]


def unpack2(b):
    """2-bit output bytes [t, n] -> codes [t, 4 n] in element order (element 4 j + a sits at bits 2a of byte j)."""
    return np.stack([(b >> s) & 3 for s in (0, 2, 4, 6)], -1).reshape(b.shape[0], -1)


def expected_tiles(floats, bws, *, out_nbit, nint=0, running=False):
    """What the plan writes into each IF's tile, [t, nprod, chan] per IF in file order (USB channels reversed): the oracle's
    floats, or for integer output the oracle's own rescale_stats / digitise applied to them (digifil -c: the first `nint`
    rows; running: every interval of `nint` rows with its own statistics)."""
    out = []
    for d, b in zip(floats, bws):
        if out_nbit == -32:
            y = d
        else:
            y = np.empty_like(d)
            for r0 in range(0, d.shape[0], nint if running else d.shape[0]):
                r1 = r0 + nint if running else d.shape[0]
                mean, scale = o.rescale_stats(d[r0:r1], nint)
                y[r0:r1] = (d[r0:r1] - mean) * scale
        if b > 0:
            y = y[:, :, ::-1]
        if out_nbit == -32:
            out.append(y)
        elif out_nbit == 2:
            out.append(unpack2(o.digitise(y.reshape(y.shape[0], -1), 2)).reshape(y.shape))
        else:
            out.append(o.digitise(y, out_nbit))
    return out


def tile_of(elems, s, nif, nprod, nchan, pol_major):
    """Tile s [t, nprod, chan] of spliced rows: [tile][prod][chan], or [prod][tile][chan] with splice_pol_major."""
    t = elems.shape[0]
    if pol_major:
        return elems.reshape(t, nprod, nif, nchan)[:, :, s]
    return elems.reshape(t, nif, nprod, nchan)[:, s]


def tile_error(g, e, out_nbit, power):
    """None if tile g matches the reference e within the project's tolerances, else what is wrong."""
    if out_nbit == -32:
        try:
            assert_rel(g, e, REL_TOL, power=power)
        except AssertionError as ex:
            return str(ex).lstrip(": ")
        return None
    d = np.abs(g.astype(np.int64) - e.astype(np.int64))
    lim = 2e-2 if out_nbit == 16 else 1e-3      # a 16-bit LSB is 1/256 of an 8-bit one (test_requantised_output)
    if d.max() <= 1 and (d != 0).mean() <= lim:
        return None
    return f"max diff {d.max()} LSB, {(d != 0).mean():.2e} of samples off"


def check_splice(rows, expected, if_order, *, pol, nchan, out_nbit, pol_major, what):
    """Every output tile s against the reference of IF if_order[s]; a failing tile names the IF it resembles most."""
    nif, nprod = len(expected), expected[0].shape[1]
    elems = unpack2(rows) if out_nbit == 2 else rows
    assert elems.shape == (expected[0].shape[0], nif * nprod * nchan), (what, elems.shape, expected[0].shape)
    fails = []
    for s, want in enumerate(if_order):
        g = tile_of(elems, s, nif, nprod, nchan, pol_major)
        e = expected[want]
        # total power per sample: the scale of the difference / cross products in the channel of a tone
        power = (e[:, 0] + e[:, 1] if pol == COH else e[:, 0]) if out_nbit == -32 and pol in (COH, IQUV) else None
        msg = tile_error(g, e, out_nbit, power)
        if msg:
            gf = g.astype(np.float64)
            dist = [np.abs(gf - x).mean() / max(np.abs(x.astype(np.float64)).mean(), 1e-30) for x in expected]
            best = int(np.argmin(dist))
            who = f"holds IF {best}" if best != want else "is closest to its own IF"
            fails.append(f"{what}: tile {s} should hold IF {want} and {who} (mean rel. distance to IF 0..{nif - 1}: "
                         + ", ".join(f"{x:.2e}" for x in dist) + f"): {msg}")
    assert not fails, "\n".join(fails)


# ---------------------------------------------------------------- a: generic, compile-time geometry (-F512:1024)
def _case_a():
    nif, nframes = 3, 1300
    vd = streams(nif, nframes, 6100)
    bws, freqs = band(nif)
    return vd, bws, freqs, oracle_floats(vd, bws, freqs, nchan=512, D=4, pol=COH)


A_KW = dict(nchan=512, tscrunch=4, pol_mode=COH, out_nbit=-32, keep_bandpass=True, chunk_units=400)


@pytest.mark.parametrize("pol_major", [False, True])
def test_generic_compile_time_geometry_three_ifs(gpu, pol_major):
    """nchan 512 (-F512:1024, the CLI default): 3 IFs of alternating sidebands, coherence products, pushes of 400 frames
    that end inside FFT blocks (the carry of every IF), both splice layouts."""
    vd, bws, freqs, fl = cached("a", _case_a)
    rows, info = run_plan(vd, bw=bws, freq=freqs, splice_pol_major=pol_major, **A_KW)
    assert info["path"] == 0 and info["geometry"].freq_res == 1024 and info["chunk_frames"] == 400
    assert info["if_order"] == [2, 1, 0]
    check_splice(rows, expected_tiles(fl, bws, out_nbit=-32), info["if_order"], pol=COH, nchan=512, out_nbit=-32,
                 pol_major=pol_major, what=f"generic nchan 512, pol_major {pol_major}")


# ---------------------------------------------------------------- b: generic, run-time kernels (freq_res 256)
B_NINT_S = 0.12


def _case_b():
    nif, nframes = 4, 700
    vd = streams(nif, nframes, 6200)
    bws, freqs = band(nif)
    return vd, bws, freqs, oracle_floats(vd, bws, freqs, nchan=64, D=8, pol=IQUV, freq_res=256)


B_KW = dict(nchan=64, freq_res=256, tscrunch=8, pol_mode=IQUV, out_nbit=8, interval=B_NINT_S, chunk_units=200)


def _b_nint():
    return int(np.floor(B_NINT_S / (8 * 64 / (BW * 1e6)) + 0.5))


@pytest.mark.parametrize("pol_major", [False, True])
def test_generic_runtime_kernels_iquv_8bit(gpu, pol_major):
    """nchan 64 with freq_res 256 (run-time generic kernels), 4 IFs, IQUV to 8 bits with a rescale interval of about 2.4
    pushes, both splice layouts; mean and scale of every IF, product and channel against the oracle's rescale_stats."""
    vd, bws, freqs, fl = cached("b", _case_b)
    rows, info = run_plan(vd, bw=bws, freq=freqs, splice_pol_major=pol_major, **B_KW)
    assert info["path"] == 0 and info["geometry"].freq_res == 256 and info["chunk_frames"] == 200
    nint = _b_nint()
    assert int(info["geometry"].interval_rows) == nint and nint > int(info["geometry"].chunk_rows) * 2
    check_splice(rows, expected_tiles(fl, bws, out_nbit=8, nint=nint), info["if_order"], pol=IQUV, nchan=64, out_nbit=8,
                 pol_major=pol_major, what=f"run-time generic IQUV 8-bit, pol_major {pol_major}")
    mean, scale = info["rescale"]                       # [IF][product][channel], natural channel order
    ref = [o.rescale_stats(d, nint) for d in fl]
    for i, (m, s) in enumerate(ref):
        # cross products have means near zero: their error is measured against the product's sigma
        bad_m = np.abs(mean[i] - m) > 2e-5 * (np.abs(m) + 1.0 / s)
        bad_s = np.abs(scale[i] - s) > 1e-4 * s
        if bad_m.any() or bad_s.any():
            near = int(np.argmin([np.abs(scale[i] / r[1] - 1).mean() for r in ref]))
            pytest.fail(f"IF {i}: {bad_m.sum()} means and {bad_s.sum()} scales off (first at product/channel "
                        f"{np.argwhere(bad_m | bad_s)[0].tolist()}); the scales are closest to those of IF {near}")


# ---------------------------------------------------------------- c: generic with forced batches
@pytest.mark.parametrize("shape", ["compile-time", "run-time"])
def test_generic_forced_batches_bit_identical(gpu, monkeypatch, shape):
    """B2F_BATCH_BLOCKS=5 (5 divides neither a push's blocks nor one IF's): batches start at b0 > 0 and straddle IF
    boundaries.  Within the oracle's tolerance, and bit-identical to one batch per push -- every block is computed by the
    same code whichever launch it falls in, so batching must not change a bit."""
    if shape == "compile-time":
        (vd, bws, freqs, fl), kw, nchan, pol, nbit, nint = cached("a", _case_a), A_KW, 512, COH, -32, 0
    else:
        (vd, bws, freqs, fl), kw, nchan, pol, nbit, nint = cached("b", _case_b), B_KW, 64, IQUV, 8, _b_nint()
    whole, _ = run_plan(vd, bw=bws, freq=freqs, **kw)
    monkeypatch.setenv("B2F_BATCH_BLOCKS", "5")
    rows, info = run_plan(vd, bw=bws, freq=freqs, **kw)
    check_splice(rows, expected_tiles(fl, bws, out_nbit=nbit, nint=nint), info["if_order"], pol=pol, nchan=nchan, out_nbit=nbit,
                 pol_major=False, what=f"{shape} generic, batches of 5 blocks")
    assert np.array_equal(rows, whole), f"batches of 5 blocks change {(rows != whole).mean():.2e} of the output"


# ---------------------------------------------------------------- d: policy geometry at the library's own push size
D_NIF = 11


def _case_d():
    plan = sorted(o.if_plan(D_NIF, 1254.0, BW))             # by IF number: stream i - 1 is IF i
    bws, freqs = [p[2] for p in plan], [p[1] for p in plan]
    vd = streams(D_NIF, 1100, 6400)
    return vd, bws, freqs, oracle_floats(vd, bws, freqs, nchan=1024, D=2, pol=I)


@pytest.mark.parametrize("out_nbit", [-32, 8])
def test_policy_geometry_default_batches(gpu, out_nbit):
    """nchan 1024 (-F1024:2048), D 2, default pushes of 1024 frames, 1100 frames (two pushes, the last ragged), base2fil's
    frequency plan.  The generic kernels' default batch is 1 GiB of intermediate = 32 blocks of 2048 x 2048; a push holds 3
    blocks per IF, so with 11 IFs the first push runs in two batches, the second starting inside IF 10 -- no override."""
    vd, bws, freqs, fl = cached("d", _case_d)
    kw = dict(keep_bandpass=True) if out_nbit == -32 else dict(interval=0.1)
    rows, info = run_plan(vd, nchan=1024, bw=bws, freq=freqs, tscrunch=2, out_nbit=out_nbit, **kw)
    g = info["geometry"]
    assert info["path"] == 0 and g.freq_res == 2048 and info["chunk_frames"] == 1024
    blocks = 1024 * int(g.samples_per_frame) // int(g.block_samples)
    batch = (1 << 30) // (2048 * 2048 * 8)
    assert D_NIF * blocks > batch and batch % blocks, (blocks, batch)
    assert info["if_order"] == list(range(D_NIF))[::-1]
    nint = int(np.floor(0.1 / (2 * 1024 / (BW * 1e6)) + 0.5))
    check_splice(rows, expected_tiles(fl, bws, out_nbit=out_nbit, nint=nint), info["if_order"], pol=I, nchan=1024,
                 out_nbit=out_nbit, pol_major=False, what=f"nchan 1024, {D_NIF} IFs, out_nbit {out_nbit}")


# ---------------------------------------------------------------- e / f: coherent dedispersion
DM = 560.0


def _plan_nfilt(nchan, D, dm, bws, freqs):
    with Plan(PlanConfig(nchan=nchan, bw_mhz=bws, freq_mhz=freqs, tscrunch=D, dm=dm, coherent=True)) as pl:
        return int(pl.geometry.nfilt_pos), int(pl.geometry.nfilt_neg)


def _case_e():
    nif = 4
    bws, freqs = band(nif)
    vd = streams(nif, 700, 6500)
    nf = _plan_nfilt(128, 16, DM, bws, freqs)
    return vd, bws, freqs, nf, oracle_floats(vd, bws, freqs, nchan=128, D=16, pol=COH, dm=DM, nfilt=nf)


@pytest.mark.parametrize("batch", [None, "7"])
def test_tuned_dedispersion_four_ifs(gpu, monkeypatch, batch):
    """digifil -D 560 -F128:D for 4 IFs at 1254 / 1286 / 1318 / 1350 MHz, alternating sidebands: the chirp of every IF from its
    own centre and sideband, nfilt from the lowest channel of all IFs, the halo carried per IF over pushes of 512 frames
    (the last ragged); also in batches of 7 blocks that straddle IFs."""
    vd, bws, freqs, nf, fl = cached("e", _case_e)
    if batch:
        monkeypatch.setenv("B2F_BATCH_BLOCKS", batch)
    rows, info = run_plan(vd, nchan=128, bw=bws, freq=freqs, tscrunch=16, pol_mode=COH, out_nbit=-32, keep_bandpass=True,
                          chunk_units=4, dm=DM, coherent=True)
    g = info["geometry"]
    assert info["path"] == 0 and g.freq_res == 512 and (int(g.nfilt_pos), int(g.nfilt_neg)) == nf
    assert 700 > info["chunk_frames"] and 700 % info["chunk_frames"]
    # the lowest IF alone needs as much overlap as all four; the highest alone needs less
    assert _plan_nfilt(128, 16, DM, [bws[0]], [freqs[0]]) == nf and _plan_nfilt(128, 16, DM, [bws[-1]], [freqs[-1]])[0] < nf[0]
    check_splice(rows, expected_tiles(fl, bws, out_nbit=-32), info["if_order"], pol=COH, nchan=128, out_nbit=-32,
                 pol_major=False, what=f"tuned dedispersion, batch {batch}")


def _case_f(nchan, D, dm, nframes, pol):
    def make():
        bws, freqs = band(2)
        vd = streams(2, nframes, 6600 + nchan)
        nf = _plan_nfilt(nchan, D, dm, bws, freqs)
        return vd, bws, freqs, nf, oracle_floats(vd, bws, freqs, nchan=nchan, D=D, pol=pol, dm=dm, nfilt=nf,
                                                 freq_res=1024 if nchan == 512 else 4096)
    return make


@pytest.mark.parametrize("nchan,D,dm,nframes,chunk,L,pol", [(512, 4, 560.0, 300, 100, 1024, COH), (128, 16, 2000.0, 330, 120, 4096, I)],
                         ids=["nchan512-L1024", "nchan128-L4096"])
def test_generic_dedispersion_two_ifs(gpu, nchan, D, dm, nframes, chunk, L, pol):
    """kx_dedisp_generic behind the generic kernels for 2 IFs of opposite sidebands: nchan 512 (L 1024) and nchan 128 at
    DM 2000, whose smearing needs L 4096."""
    vd, bws, freqs, nf, fl = cached(("f", nchan), _case_f(nchan, D, dm, nframes, pol))
    rows, info = run_plan(vd, nchan=nchan, bw=bws, freq=freqs, tscrunch=D, pol_mode=pol, out_nbit=-32, keep_bandpass=True,
                          chunk_units=chunk, dm=dm, coherent=True)
    g = info["geometry"]
    assert info["path"] == 0 and g.freq_res == L and (int(g.nfilt_pos), int(g.nfilt_neg)) == nf and info["chunk_frames"] == chunk
    check_splice(rows, expected_tiles(fl, bws, out_nbit=-32), info["if_order"], pol=pol, nchan=nchan, out_nbit=-32,
                 pol_major=False, what=f"generic dedispersion nchan {nchan} L {L}")


# ---------------------------------------------------------------- g / h: 8-bit and 1-bit input
def _fault_counts(vd, nframes):
    inv = fill_words = fill_frames = 0
    for v in vd:
        fr = v.reshape(-1, FB)[:nframes]
        bad = (fr[:, 3] >> 7).astype(bool)
        words = np.ascontiguousarray(fr[:, 32:]).view("<u4") == 0x11223344
        inv += int(bad.sum())
        fill_words += int(words[~bad].sum())
        fill_frames += int((words.any(axis=1) & ~bad).sum())
    return inv, fill_words, fill_frames


@pytest.mark.parametrize("nchan,D,chunk,nframes", [(128, 16, 0, 0), (512, 4, 400, 1300)])
def test_8bit_input_faults_per_if(gpu, nchan, D, chunk, nframes):
    """8-bit VDIF, 3 IFs: clean / invalid frames / fill words, on the round-1 tuned kernels (nchan 128, one push) and the
    generic ones (nchan 512, carried samples and word masks): the masks and dirty-block flags of each IF, and the fault
    counters summed over the IFs."""
    bws, freqs = band(3)
    if not nframes:
        with Plan(PlanConfig(nchan=nchan, bw_mhz=bws, freq_mhz=freqs, in_nbit=8)) as pl:
            nframes = int(pl.chunk_frames)

    def make():
        vd = streams(3, nframes, 6700 + nchan, nbit=8, faults=[{}, {"invalid_frac": 0.02}, {"fill_frac": 0.03}])
        return vd, oracle_floats(vd, bws, freqs, nchan=nchan, D=D, pol=I, in_nbit=8)
    vd, fl = cached(("g", nchan), make)
    rows, info = run_plan(vd, nchan=nchan, bw=bws, freq=freqs, tscrunch=D, in_nbit=8, out_nbit=-32, keep_bandpass=True, chunk_units=chunk)
    assert info["path"] == 0
    c = info["counters"]
    inv, fw, ff = _fault_counts(vd, nframes)
    assert inv > 0 and fw > 0
    assert (c["frames_invalid"], c["fill_words"], c["frames_with_fill"]) == (inv, fw, ff)
    assert c["frames_ok"] + c["frames_invalid"] + c["frames_with_fill"] == 3 * nframes
    check_splice(rows, expected_tiles(fl, bws, out_nbit=-32), info["if_order"], pol=I, nchan=nchan, out_nbit=-32, pol_major=False,
                 what=f"8-bit input nchan {nchan}")


@pytest.mark.parametrize("nchan,D,chunk,nframes", [(64, 16, 0, 0), (512, 4, 60, 170)])
def test_1bit_input_two_ifs(gpu, nchan, D, chunk, nframes):
    """1-bit VDIF, 2 IFs: the tuned kernels (nchan 64, one push) and the generic ones (nchan 512, carried samples)."""
    bws, freqs = band(2)
    if not nframes:
        with Plan(PlanConfig(nchan=nchan, bw_mhz=bws, freq_mhz=freqs, in_nbit=1)) as pl:
            nframes = min(int(pl.chunk_frames), 160)

    def make():
        vd = streams(2, nframes, 6800 + nchan, nbit=1, faults=[{"fill_frac": 0.04}, {"invalid_frac": 0.03}])
        return vd, oracle_floats(vd, bws, freqs, nchan=nchan, D=D, pol=I, in_nbit=1)
    vd, fl = cached(("h", nchan), make)
    rows, info = run_plan(vd, nchan=nchan, bw=bws, freq=freqs, tscrunch=D, in_nbit=1, out_nbit=-32, keep_bandpass=True, chunk_units=chunk)
    assert info["path"] == 0 and int(info["geometry"].samples_per_frame) == 32000
    check_splice(rows, expected_tiles(fl, bws, out_nbit=-32), info["if_order"], pol=I, nchan=nchan, out_nbit=-32, pol_major=False,
                 what=f"1-bit input nchan {nchan}")


# ---------------------------------------------------------------- i: JA98 decode
@pytest.mark.parametrize("nchan,nif,D,chunk,nframes,path", [(128, 3, 16, 0, 1024, 1), (512, 2, 4, 100, 300, 0)])
def test_ja98_levels_per_if(gpu, nchan, nif, D, chunk, nframes, path):
    """decode_mode JA98 with several IFs: the round-2 column kernel (nchan 128, path 1) and the generic kernels with levels
    per window of the de-framed stream of each IF (nchan 512)."""
    bws, freqs = band(nif)

    def make():
        vd = streams(nif, nframes, 6900 + nchan)
        return vd, oracle_floats(vd, bws, freqs, nchan=nchan, D=D, pol=I, decode_mode="ja98")
    vd, fl = cached(("i", nchan), make)
    rows, info = run_plan(vd, nchan=nchan, bw=bws, freq=freqs, tscrunch=D, out_nbit=-32, keep_bandpass=True, chunk_units=chunk,
                          decode_mode=_lib.DECODE_JA98)
    assert info["path"] == path
    check_splice(rows, expected_tiles(fl, bws, out_nbit=-32), info["if_order"], pol=I, nchan=nchan, out_nbit=-32, pol_major=False,
                 what=f"JA98 nchan {nchan}")


# ---------------------------------------------------------------- j: multi-product integer output
@pytest.mark.parametrize("out_nbit", [8, 16, 2])
@pytest.mark.parametrize("pol,path", [(COH, 1), (IQUV, 1), (PPQQ, 0)], ids=["coherence", "IQUV", "PPQQ"])
def test_multi_product_integer_output(gpu, pol, path, out_nbit):
    """nchan 128, 4 IFs: coherence and IQUV on the round-2 kernels, PPQQ on the round-1 ones, to 8, 16 and 2 bits -- the
    statistics, quantisation and flip of every IF and product (IQUV spliced product-major)."""
    nif, D, interval = 4, 16, 0.1
    bws, freqs = band(nif)

    def make():
        vd = streams(nif, 1024, 7000)
        return vd, oracle_floats(vd, bws, freqs, nchan=128, D=D, pol=COH)
    vd, coh = cached("j", make)
    # the other products are linear in the oracle's integrated coherence products (PP, QQ, Re PQ*, Im PQ*)
    fl = [{COH: c, IQUV: np.stack([c[:, 0] + c[:, 1], 2 * c[:, 2], 2 * c[:, 3], c[:, 0] - c[:, 1]], 1), PPQQ: c[:, :2]}[pol] for c in coh]
    pol_major = pol == IQUV
    rows, info = run_plan(vd, nchan=128, bw=bws, freq=freqs, tscrunch=D, pol_mode=pol, out_nbit=out_nbit, interval=interval,
                          splice_pol_major=pol_major)
    assert info["path"] == path
    nint = int(np.floor(interval / (D * 128 / (BW * 1e6)) + 0.5))
    check_splice(rows, expected_tiles(fl, bws, out_nbit=out_nbit, nint=nint), info["if_order"], pol=pol, nchan=128, out_nbit=out_nbit,
                 pol_major=pol_major, what=f"{NAME[pol]} to {out_nbit} bits")


# ---------------------------------------------------------------- k: splice order and running rescale
K_ORDER = [0, 2, 1]


def _case_k():
    bws, freqs = band(3)
    with Plan(PlanConfig(nchan=32, bw_mhz=bws, freq_mhz=freqs, chunk_units=1)) as pl:
        nframes = 3 * int(pl.chunk_frames) + 37
    vd = streams(3, nframes, 7100)
    return vd, bws, freqs, oracle_floats(vd, bws, freqs, nchan=32, D=32, pol=COH)


@pytest.mark.parametrize("pol_major", [False, True])
def test_if_order_and_running_rescale(gpu, pol_major):
    """An if_order that is not sorted by frequency either way (tile 0 <- IF 0, 1 <- 2, 2 <- 1) and rescale_mode running:
    every 0.06 s interval of every IF scaled with its own statistics, intervals straddling pushes; both splice layouts."""
    vd, bws, freqs, fl = cached("k", _case_k)
    interval = 0.06
    rows, info = run_plan(vd, nchan=32, bw=bws, freq=freqs, tscrunch=32, pol_mode=COH, out_nbit=8, interval=interval, chunk_units=1,
                          if_order=K_ORDER, rescale_mode=_lib.RESCALE_RUNNING, splice_pol_major=pol_major)
    assert info["path"] == 0 and info["if_order"] == K_ORDER
    nint = int(np.floor(interval / (32 * 32 / (BW * 1e6)) + 0.5))
    assert nint < 5 * int(info["geometry"].chunk_rows) and int(info["geometry"].chunk_rows) % nint    # boundaries inside pushes
    check_splice(rows, expected_tiles(fl, bws, out_nbit=8, nint=nint, running=True), K_ORDER, pol=COH, nchan=32, out_nbit=8,
                 pol_major=pol_major, what=f"if_order {K_ORDER}, running rescale, pol_major {pol_major}")
