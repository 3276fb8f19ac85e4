"""Every kernel instantiation the plan can dispatch to, against the float64 oracle.

libb2f picks its kernels with `switch` statements over the row length R = 2 nchan, the detection product, the input bit
depth and single DM or trials; each arm is its own compiled kernel with its own loop bounds, shared-memory layout and
mirror-bin arithmetic.  CASES below names one plan per row: its shape, input, product and override.  `expected_arms`
mirrors the selection of b2f_plan_create / push_dedisp and says which instantiations a case reaches; MATRIX is that map
written out (instantiation key -> case ids) and test_dispatch_matrix_host.py checks it against the arms parsed from the
sources, so an arm without a case fails without a GPU.

Each case compares the plan's float rows (-b-32 -I0) with the oracle at REL_TOL, and checks the facts that show which arm
ran: the path, freq_res, nfilt, ndm and the launch counts of kernel_times().  The oracle channelises each input once in
float64, one polarisation at a time, and derives every product with o.detect / o.tscrunch; cases that share an input are
adjacent, so the channelisation is computed once for all of them."""
import numpy as np
import pytest

from oracle import digifil_oracle as o
from frb_baseband_b200 import _lib
from frb_baseband_b200.plan import Plan, PlanConfig
from helpers import assert_rel, run_plan
from test_gpu_multi_if import BW, COH, I, IQUV, PPQQ, check_splice, expected_tiles, streams

pytestmark = pytest.mark.gpu

P0, P1, I2 = _lib.POL_P0, _lib.POL_P1, _lib.POL_I2
MODE = {P0: "P0", P1: "P1", I: "I", I2: "I2", PPQQ: "PPQQ", COH: "coherence", IQUV: "IQUV"}
ALL = [P0, P1, I, I2, PPQQ, COH, IQUV]
KF_MODES = ("I", "coherence", "IQUV")          # the round-2 kernels are built for these (Makefile: B2F_KF_MAIN_MODES)
ENV = ("B2F_PATH", "B2F_GENERIC", "B2F_BATCH_BLOCKS")
TIMED = ("column", "eps", "row", "dedisp", "fused", "tsum")


# ---------------------------------------------------------------- the case table
def dm_for(nchan, nfilt, f0=1254.0):
    """The DM whose plan nfilt (before rounding to tscrunch) is `nfilt`: 0.55 x the smearing across the lowest channel."""
    return (nfilt - 0.5) / 0.55 / o.smearing_samples(f0, BW, nchan, 1.0)


CASES = {}


def _case(cid, fam, nchan, L, *, pol=I, D=1, nif=2, usb=False, nframes, push=0, nbit=2, decode="static", freq_res=0, dm=0.0,
          trials=None, env=None, same_as=None, keep_min=0, seed):
    assert cid not in CASES
    CASES[cid] = dict(fam=fam, nchan=nchan, L=L, pol=pol, D=D, nif=nif, usb=usb, nframes=nframes, push=push, nbit=nbit,
                      decode=decode, freq_res=freq_res, dm=dm, trials=trials, env=env or {}, same_as=same_as, keep_min=keep_min,
                      seed=seed)


NF_T = {8: 150, 16: 150, 32: 300, 64: 600, 128: 600, 256: 650}      # 2-bit frames of the 512-point shapes
NF_8 = {8: 300, 16: 300, 32: 400, 64: 600, 128: 600, 256: 1300}               # 8-bit frames (4000 samples each)
D_T = {8: 4, 16: 4, 32: 4, 64: 16, 128: 16, 256: 16}
NF_D = {8: 120, 16: 120, 32: 150, 64: 200, 128: 300, 256: 300}      # tuned dedispersion
D_D = {8: 4, 16: 4, 32: 4, 64: 8, 128: 16, 256: 16}

for n in (8, 16, 32, 64, 128, 256):
    R = 2 * n
    st = dict(nframes=NF_T[n], seed=40000 + n)
    if n != 128:
        # A: round-1 tuned channeliser, every product
        for p in ALL:
            _case(f"A-n{n}-{MODE[p]}", "A", n, 512, pol=p, D=D_T[n], **st)
    else:
        for p in ALL:
            _case(f"A-n{n}-{MODE[p]}-legacy", "A", n, 512, pol=p, D=D_T[n], env={"B2F_PATH": "legacy"}, **st)
    # C: round-2 kernels.  Static levels with B2F_PATH=split / fused at D = 2048 / R > 1024 / R (the fused kernel then sums
    # partial rows in kt_sum_partials); JA98 with no override at D <= 1024 / R (the fused kernel writes its rows itself).
    for p in (I, COH, IQUV):
        if n != 128:
            _case(f"C-n{n}-{MODE[p]}-split", "C", n, 512, pol=p, D=2048 // R, env={"B2F_PATH": "split"}, **st)
        _case(f"C-n{n}-{MODE[p]}-fused", "C", n, 512, pol=p, D=2048 // R, env={"B2F_PATH": "fused"}, **st)
    # B: JA98 with a product the fused kernel is not built for selects the round-1 column kernel with stream levels
    for p in (P0, PPQQ, I2):
        _case(f"B-n{n}-ja98-{MODE[p]}", "B", n, 512, pol=p, D=D_T[n], decode="ja98", **st)
    for p in (I, COH, IQUV):
        _case(f"C-n{n}-ja98-{MODE[p]}", "C", n, 512, pol=p, D=max(1, 512 // R), decode="ja98",
              env={"B2F_PATH": "fused"} if n == 128 else None, **st)
    # B: 8-bit input on the round-1 column kernel
    for p in (I, COH):
        _case(f"B-n{n}-8bit-{MODE[p]}", "B", n, 512, pol=p, D=D_T[n], nbit=8, nframes=NF_8[n], seed=41000 + n)
    # D: tuned dedispersion with 2 nfilt ~ 0.6 x 512; trials [d/3, 2d/3, d], the largest equal to the single-DM plan
    d = dm_for(n, 154)
    sd = dict(nframes=NF_D[n], seed=42000 + n, D=D_D[n])
    _case(f"D-n{n}-I", "D", n, 512, pol=I, dm=d, **sd)
    _case(f"D-n{n}-coherence", "D", n, 512, pol=COH, dm=d, **sd)
    _case(f"D-n{n}-trials", "D", n, 512, pol=I, trials=[d / 3, 2 * d / 3, d], same_as=f"D-n{n}-I", **sd)
    # JA98 levels count windows of 512 samples from each push's first carried sample: blocks must start on multiples of
    # 512 samples, i.e. keep = 512 - 2 nfilt a multiple of 512 / R, which a tscrunch of at least 256 / R guarantees
    _case(f"D-n{n}-ja98-coherence", "D", n, 512, pol=COH, dm=d, decode="ja98", **{**sd, "D": max(D_D[n], 256 // R)})
    _case(f"D-n{n}-8bit-I", "D", n, 512, pol=I, dm=d, nbit=8, nframes=2 * NF_D[n], seed=43000 + n, D=D_D[n])

# E: generic run-time kernels at nchan 2048 (kg_row_pass<8>): freq_res 1024, freq_res 4096 with B2F_GENERIC=runtime (it
# shares the input of F's nchan 2048), and dedispersion at the default 4096 (kgt column, kg_row_pass<8> volt, kx)
for p in (I, COH, IQUV, PPQQ):
    _case(f"E-n2048-fr1024-{MODE[p]}", "E", 2048, 1024, pol=p, D=2, nframes=600, push=250, freq_res=1024, seed=44000)
# ... and at nchan 64 / freq_res 256 for 8-bit and JA98 input (kg_column_pass<8>, <22>; kg_row_pass<4>)
for nb, dec in ((8, "static"), (2, "ja98")):
    _case(f"E-n64-fr256-{'8bit' if nb == 8 else 'ja98'}-coherence", "E", 64, 256, pol=COH, D=4, nbit=nb, decode=dec, nframes=300 if nb == 8 else 120,
          push=70 if nb == 8 else 25, freq_res=256, seed=44064)
# F: compile-time generic kernels at LG 10..13 (nchan 512..4096), every product; 8-bit and JA98 input
F_ST = {512: dict(nif=2, nframes=300, push=100, seed=45512), 1024: dict(nif=2, nframes=600, push=250, seed=46024),
        2048: dict(nif=1, usb=True, nframes=2150, push=400, seed=45000), 4096: dict(nif=1, usb=True, nframes=4300, push=400, seed=48000)}
for n in (512, 1024, 2048, 4096):
    for p in ALL:
        _case(f"F-n{n}-{MODE[p]}", "F", n, 2 * n, pol=p, D=2, **F_ST[n])
    if n == 2048:
        for p in (I, COH):
            _case(f"E-n2048-runtime-{MODE[p]}", "E", n, 2 * n, pol=p, D=2, env={"B2F_GENERIC": "runtime"}, **F_ST[n])
    _case(f"F-n{n}-ja98-I", "F", n, 2 * n, pol=I, D=2, decode="ja98", **F_ST[n])
    _case(f"F-n{n}-8bit-I", "F", n, 2 * n, pol=I, D=2, nbit=8, nif=1, nframes=max(300, n * 2 + 200) if n < 4096 else 16800,
          push=max(100, n // 2) if n < 4096 else 4000, seed=47000 + n)
d = dm_for(2048, 512)
E_DD = dict(D=4, nif=1, nframes=1900, push=500, seed=46000)
_case("E-n2048-dedisp-I", "E", 2048, 4096, pol=I, dm=d, **E_DD)
_case("E-n2048-dedisp-IQUV", "E", 2048, 4096, pol=IQUV, dm=d, **E_DD)
_case("E-n2048-dedisp-trials", "E", 2048, 4096, pol=I, trials=[d / 2, d], same_as="E-n2048-dedisp-I", **E_DD)

# G: long transforms.  nchan 64 / 8192 points with 3 IFs, every product; batches of 1 and 5 blocks (5 straddles IFs and
# pushes of ~4.5 blocks per IF) byte-identical to the default batch; nchan 8 and 16 at 8192 points; trials at nchan 8 and 64
d = dm_for(64, 2048)
G64 = dict(nif=3, nframes=400, push=150, freq_res=8192, D=8, seed=50000)
for p in ALL:
    _case(f"G-n64-{MODE[p]}", "G", 64, 8192, pol=p, dm=d, **G64)
for b in (1, 5):
    _case(f"G-n64-batch{b}-coherence", "G", 64, 8192, pol=COH, dm=d, env={"B2F_BATCH_BLOCKS": str(b)}, same_as="G-n64-coherence", **G64)
_case("G-n64-trials", "G", 64, 8192, pol=COH, trials=[d / 2, d], same_as="G-n64-coherence", **G64)
d8, d16 = dm_for(8, 2048), dm_for(16, 2048)
G8 = dict(nif=2, nframes=120, push=25, freq_res=8192, D=4, seed=51000)
_case("G-n8-fr8192-coherence", "G", 8, 8192, pol=COH, dm=d8, **G8)
_case("G-n8-trials", "G", 8, 8192, pol=COH, trials=[d8 / 2, d8], same_as="G-n8-fr8192-coherence", **G8)
_case("G-n16-fr8192-IQUV", "G", 16, 8192, pol=IQUV, dm=d16, nif=2, nframes=120, push=25, freq_res=8192, D=4, seed=52000)

# H: the largest DM each back end accepts at one shape (bisection over plan creation); the long path at the largest DM that
# keeps L / 16 samples of each block, to bound the oracle's work
_case("H-tuned-n8", "H", 8, 512, pol=COH, D=32, nif=2, nframes=40, freq_res=512, dm="edge", seed=53008)
_case("H-tuned-n256", "H", 256, 512, pol=I, D=64, nif=2, nframes=200, freq_res=512, dm="edge", seed=53256)
_case("H-generic-n128", "H", 128, 4096, pol=I, D=128, nif=1, nframes=200, push=70, freq_res=4096, dm="edge", seed=54000)
_case("H-long-n8", "H", 8, 65536, pol=I, D=64, nif=1, nframes=150, push=40, freq_res=65536, dm="edge", keep_min=65536 // 16, seed=55008)
_case("H-long-n64", "H", 64, 8192, pol=COH, D=64, nif=1, nframes=150, push=40, freq_res=8192, dm="edge", keep_min=8192 // 16, seed=55064)


# ---------------------------------------------------------------- which arms a case reaches
def kernel_D(D_user, L, dedisp):
    D = D_user & -D_user
    while D > L:
        D >>= 1
    while dedisp and D > 128:
        D >>= 1
    return D


def expected_arms(c, L, env=None):
    """Mirror of the kernel selection in b2f_plan_create / push_dedisp / push_fused for case `c` at freq_res L under the
    override variables `env`: {"path": channeliser path, "arms": instantiation keys, "launched": kernel_times() ids that
    must count launches (the others of TIMED must not)}."""
    env = c["env"] if env is None else env
    R, N, mode = 2 * c["nchan"], c["nchan"], MODE[c["pol"]]
    ja98 = c["decode"] == "ja98"
    dedisp = bool(c["dm"]) or bool(c["trials"])
    nbit = 22 if ja98 else (8 if c["nbit"] == 8 else 2)            # 1-bit input arrives as the 2-bit index bytes
    generic = not (L == 512 and R <= 512)
    longfft = L > 4096 and L != R
    D = kernel_D(c["D"], L, dedisp)
    if longfft:
        return dict(path=0, arms={("kl_pass", "stream"), ("kl_pass", "f"), ("kl_pass", "unmix"), ("kl_detect", mode)},
                    launched={"column", "row", "dedisp"})
    if generic:
        lg = L.bit_length() - 1
        kgt = L == R and L >= 1024 and not (env.get("B2F_GENERIC") == "runtime" and L <= 4096)
        cpt = 8 if N > 1024 else 4
        arms = {("kgt_col", lg, nbit) if kgt else ("kg_col", nbit)}
        if dedisp:
            arms |= {("kg_row", cpt, "volt"), ("kx",)}
        else:
            arms.add(("kgt_row", lg, mode) if kgt else ("kg_row", cpt, "detect"))
        return dict(path=0, arms=arms, launched={"column", "eps", "row"} | ({"dedisp"} if dedisp else set()))
    if dedisp:
        return dict(path=0, arms={("ka", nbit, R, "fwd"), ("kb", R, "spectrum"), ("kc_trials" if c["trials"] else "kc_back", R)},
                    launched={"column", "row", "dedisp"})
    eligible = c["nbit"] == 2                                      # 2-bit split streams, positional frames, 8032-byte frames
    want = 1 if R == 256 else (2 if ja98 else 0)
    want = {"legacy": 0, "split": 1, "fused": 2}.get(env.get("B2F_PATH"), want)
    path = want if eligible and mode in KF_MODES else 0            # the round-2 kernels exist for KF_MODES only
    kf = "kfj" if ja98 else "kf"
    if path == 0:
        return dict(path=0, arms={("ka", nbit, R, "full"), ("kb", R, mode)}, launched={"column", "eps", "row"})
    if path == 1:
        return dict(path=1, arms={(kf, R, "I"), ("kt", mode) if R == 256 else ("kr", R, mode)}, launched={"column", "eps", "row"})
    return dict(path=2, arms={(kf, R, mode)}, launched={"fused"} | ({"tsum"} if min(D, 1024 // R) < D else set()))


def derive_matrix():
    m = {}
    for cid, c in CASES.items():
        for k in expected_arms(c, c["L"])["arms"]:
            m.setdefault(k, []).append(cid)
    return m


# instantiation key -> the cases that reach it (derive_matrix() written out; test_dispatch_matrix_host.py keeps the two
# equal and checks every arm of the sources against the keys)
MATRIX = {
    ("ka", 2, 16, "fwd"): ["D-n8-I", "D-n8-coherence", "D-n8-trials", "H-tuned-n8"],
    ("ka", 2, 16, "full"): ["A-n8-P0", "A-n8-P1", "A-n8-I", "A-n8-I2", "A-n8-PPQQ", "A-n8-coherence", "A-n8-IQUV"],
    ("ka", 2, 32, "fwd"): ["D-n16-I", "D-n16-coherence", "D-n16-trials"],
    ("ka", 2, 32, "full"): ["A-n16-P0", "A-n16-P1", "A-n16-I", "A-n16-I2", "A-n16-PPQQ", "A-n16-coherence", "A-n16-IQUV"],
    ("ka", 2, 64, "fwd"): ["D-n32-I", "D-n32-coherence", "D-n32-trials"],
    ("ka", 2, 64, "full"): ["A-n32-P0", "A-n32-P1", "A-n32-I", "A-n32-I2", "A-n32-PPQQ", "A-n32-coherence", "A-n32-IQUV"],
    ("ka", 2, 128, "fwd"): ["D-n64-I", "D-n64-coherence", "D-n64-trials"],
    ("ka", 2, 128, "full"): ["A-n64-P0", "A-n64-P1", "A-n64-I", "A-n64-I2", "A-n64-PPQQ", "A-n64-coherence", "A-n64-IQUV"],
    ("ka", 2, 256, "fwd"): ["D-n128-I", "D-n128-coherence", "D-n128-trials"],
    ("ka", 2, 256, "full"): ["A-n128-P0-legacy", "A-n128-P1-legacy", "A-n128-I-legacy", "A-n128-I2-legacy", "A-n128-PPQQ-legacy",
        "A-n128-coherence-legacy", "A-n128-IQUV-legacy"],
    ("ka", 2, 512, "fwd"): ["D-n256-I", "D-n256-coherence", "D-n256-trials", "H-tuned-n256"],
    ("ka", 2, 512, "full"): ["A-n256-P0", "A-n256-P1", "A-n256-I", "A-n256-I2", "A-n256-PPQQ", "A-n256-coherence", "A-n256-IQUV"],
    ("ka", 8, 16, "fwd"): ["D-n8-8bit-I"],
    ("ka", 8, 16, "full"): ["B-n8-8bit-I", "B-n8-8bit-coherence"],
    ("ka", 8, 32, "fwd"): ["D-n16-8bit-I"],
    ("ka", 8, 32, "full"): ["B-n16-8bit-I", "B-n16-8bit-coherence"],
    ("ka", 8, 64, "fwd"): ["D-n32-8bit-I"],
    ("ka", 8, 64, "full"): ["B-n32-8bit-I", "B-n32-8bit-coherence"],
    ("ka", 8, 128, "fwd"): ["D-n64-8bit-I"],
    ("ka", 8, 128, "full"): ["B-n64-8bit-I", "B-n64-8bit-coherence"],
    ("ka", 8, 256, "fwd"): ["D-n128-8bit-I"],
    ("ka", 8, 256, "full"): ["B-n128-8bit-I", "B-n128-8bit-coherence"],
    ("ka", 8, 512, "fwd"): ["D-n256-8bit-I"],
    ("ka", 8, 512, "full"): ["B-n256-8bit-I", "B-n256-8bit-coherence"],
    ("ka", 22, 16, "fwd"): ["D-n8-ja98-coherence"],
    ("ka", 22, 16, "full"): ["B-n8-ja98-P0", "B-n8-ja98-PPQQ", "B-n8-ja98-I2"],
    ("ka", 22, 32, "fwd"): ["D-n16-ja98-coherence"],
    ("ka", 22, 32, "full"): ["B-n16-ja98-P0", "B-n16-ja98-PPQQ", "B-n16-ja98-I2"],
    ("ka", 22, 64, "fwd"): ["D-n32-ja98-coherence"],
    ("ka", 22, 64, "full"): ["B-n32-ja98-P0", "B-n32-ja98-PPQQ", "B-n32-ja98-I2"],
    ("ka", 22, 128, "fwd"): ["D-n64-ja98-coherence"],
    ("ka", 22, 128, "full"): ["B-n64-ja98-P0", "B-n64-ja98-PPQQ", "B-n64-ja98-I2"],
    ("ka", 22, 256, "fwd"): ["D-n128-ja98-coherence"],
    ("ka", 22, 256, "full"): ["B-n128-ja98-P0", "B-n128-ja98-PPQQ", "B-n128-ja98-I2"],
    ("ka", 22, 512, "fwd"): ["D-n256-ja98-coherence"],
    ("ka", 22, 512, "full"): ["B-n256-ja98-P0", "B-n256-ja98-PPQQ", "B-n256-ja98-I2"],
    ("kb", 16, "I"): ["A-n8-I", "B-n8-8bit-I"],
    ("kb", 16, "I2"): ["A-n8-I2", "B-n8-ja98-I2"],
    ("kb", 16, "P0"): ["A-n8-P0", "B-n8-ja98-P0"],
    ("kb", 16, "P1"): ["A-n8-P1"],
    ("kb", 16, "IQUV"): ["A-n8-IQUV"],
    ("kb", 16, "PPQQ"): ["A-n8-PPQQ", "B-n8-ja98-PPQQ"],
    ("kb", 16, "coherence"): ["A-n8-coherence", "B-n8-8bit-coherence"],
    ("kb", 16, "spectrum"): ["D-n8-I", "D-n8-coherence", "D-n8-trials", "D-n8-ja98-coherence", "D-n8-8bit-I", "H-tuned-n8"],
    ("kb", 32, "I"): ["A-n16-I", "B-n16-8bit-I"],
    ("kb", 32, "I2"): ["A-n16-I2", "B-n16-ja98-I2"],
    ("kb", 32, "P0"): ["A-n16-P0", "B-n16-ja98-P0"],
    ("kb", 32, "P1"): ["A-n16-P1"],
    ("kb", 32, "IQUV"): ["A-n16-IQUV"],
    ("kb", 32, "PPQQ"): ["A-n16-PPQQ", "B-n16-ja98-PPQQ"],
    ("kb", 32, "coherence"): ["A-n16-coherence", "B-n16-8bit-coherence"],
    ("kb", 32, "spectrum"): ["D-n16-I", "D-n16-coherence", "D-n16-trials", "D-n16-ja98-coherence", "D-n16-8bit-I"],
    ("kb", 64, "I"): ["A-n32-I", "B-n32-8bit-I"],
    ("kb", 64, "I2"): ["A-n32-I2", "B-n32-ja98-I2"],
    ("kb", 64, "P0"): ["A-n32-P0", "B-n32-ja98-P0"],
    ("kb", 64, "P1"): ["A-n32-P1"],
    ("kb", 64, "IQUV"): ["A-n32-IQUV"],
    ("kb", 64, "PPQQ"): ["A-n32-PPQQ", "B-n32-ja98-PPQQ"],
    ("kb", 64, "coherence"): ["A-n32-coherence", "B-n32-8bit-coherence"],
    ("kb", 64, "spectrum"): ["D-n32-I", "D-n32-coherence", "D-n32-trials", "D-n32-ja98-coherence", "D-n32-8bit-I"],
    ("kb", 128, "I"): ["A-n64-I", "B-n64-8bit-I"],
    ("kb", 128, "I2"): ["A-n64-I2", "B-n64-ja98-I2"],
    ("kb", 128, "P0"): ["A-n64-P0", "B-n64-ja98-P0"],
    ("kb", 128, "P1"): ["A-n64-P1"],
    ("kb", 128, "IQUV"): ["A-n64-IQUV"],
    ("kb", 128, "PPQQ"): ["A-n64-PPQQ", "B-n64-ja98-PPQQ"],
    ("kb", 128, "coherence"): ["A-n64-coherence", "B-n64-8bit-coherence"],
    ("kb", 128, "spectrum"): ["D-n64-I", "D-n64-coherence", "D-n64-trials", "D-n64-ja98-coherence", "D-n64-8bit-I"],
    ("kb", 256, "I"): ["A-n128-I-legacy", "B-n128-8bit-I"],
    ("kb", 256, "I2"): ["A-n128-I2-legacy", "B-n128-ja98-I2"],
    ("kb", 256, "P0"): ["A-n128-P0-legacy", "B-n128-ja98-P0"],
    ("kb", 256, "P1"): ["A-n128-P1-legacy"],
    ("kb", 256, "IQUV"): ["A-n128-IQUV-legacy"],
    ("kb", 256, "PPQQ"): ["A-n128-PPQQ-legacy", "B-n128-ja98-PPQQ"],
    ("kb", 256, "coherence"): ["A-n128-coherence-legacy", "B-n128-8bit-coherence"],
    ("kb", 256, "spectrum"): ["D-n128-I", "D-n128-coherence", "D-n128-trials", "D-n128-ja98-coherence", "D-n128-8bit-I"],
    ("kb", 512, "I"): ["A-n256-I", "B-n256-8bit-I"],
    ("kb", 512, "I2"): ["A-n256-I2", "B-n256-ja98-I2"],
    ("kb", 512, "P0"): ["A-n256-P0", "B-n256-ja98-P0"],
    ("kb", 512, "P1"): ["A-n256-P1"],
    ("kb", 512, "IQUV"): ["A-n256-IQUV"],
    ("kb", 512, "PPQQ"): ["A-n256-PPQQ", "B-n256-ja98-PPQQ"],
    ("kb", 512, "coherence"): ["A-n256-coherence", "B-n256-8bit-coherence"],
    ("kb", 512, "spectrum"): ["D-n256-I", "D-n256-coherence", "D-n256-trials", "D-n256-ja98-coherence", "D-n256-8bit-I",
        "H-tuned-n256"],
    ("kc_back", 16): ["D-n8-I", "D-n8-coherence", "D-n8-ja98-coherence", "D-n8-8bit-I", "H-tuned-n8"],
    ("kc_back", 32): ["D-n16-I", "D-n16-coherence", "D-n16-ja98-coherence", "D-n16-8bit-I"],
    ("kc_back", 64): ["D-n32-I", "D-n32-coherence", "D-n32-ja98-coherence", "D-n32-8bit-I"],
    ("kc_back", 128): ["D-n64-I", "D-n64-coherence", "D-n64-ja98-coherence", "D-n64-8bit-I"],
    ("kc_back", 256): ["D-n128-I", "D-n128-coherence", "D-n128-ja98-coherence", "D-n128-8bit-I"],
    ("kc_back", 512): ["D-n256-I", "D-n256-coherence", "D-n256-ja98-coherence", "D-n256-8bit-I", "H-tuned-n256"],
    ("kc_trials", 16): ["D-n8-trials"],
    ("kc_trials", 32): ["D-n16-trials"],
    ("kc_trials", 64): ["D-n32-trials"],
    ("kc_trials", 128): ["D-n64-trials"],
    ("kc_trials", 256): ["D-n128-trials"],
    ("kc_trials", 512): ["D-n256-trials"],
    ("kf", 16, "I"): ["C-n8-I-split", "C-n8-I-fused", "C-n8-coherence-split", "C-n8-IQUV-split"],
    ("kf", 16, "IQUV"): ["C-n8-IQUV-fused"],
    ("kf", 16, "coherence"): ["C-n8-coherence-fused"],
    ("kf", 32, "I"): ["C-n16-I-split", "C-n16-I-fused", "C-n16-coherence-split", "C-n16-IQUV-split"],
    ("kf", 32, "IQUV"): ["C-n16-IQUV-fused"],
    ("kf", 32, "coherence"): ["C-n16-coherence-fused"],
    ("kf", 64, "I"): ["C-n32-I-split", "C-n32-I-fused", "C-n32-coherence-split", "C-n32-IQUV-split"],
    ("kf", 64, "IQUV"): ["C-n32-IQUV-fused"],
    ("kf", 64, "coherence"): ["C-n32-coherence-fused"],
    ("kf", 128, "I"): ["C-n64-I-split", "C-n64-I-fused", "C-n64-coherence-split", "C-n64-IQUV-split"],
    ("kf", 128, "IQUV"): ["C-n64-IQUV-fused"],
    ("kf", 128, "coherence"): ["C-n64-coherence-fused"],
    ("kf", 256, "I"): ["C-n128-I-fused"],
    ("kf", 256, "IQUV"): ["C-n128-IQUV-fused"],
    ("kf", 256, "coherence"): ["C-n128-coherence-fused"],
    ("kf", 512, "I"): ["C-n256-I-split", "C-n256-I-fused", "C-n256-coherence-split", "C-n256-IQUV-split"],
    ("kf", 512, "IQUV"): ["C-n256-IQUV-fused"],
    ("kf", 512, "coherence"): ["C-n256-coherence-fused"],
    ("kfj", 16, "I"): ["C-n8-ja98-I"],
    ("kfj", 16, "IQUV"): ["C-n8-ja98-IQUV"],
    ("kfj", 16, "coherence"): ["C-n8-ja98-coherence"],
    ("kfj", 32, "I"): ["C-n16-ja98-I"],
    ("kfj", 32, "IQUV"): ["C-n16-ja98-IQUV"],
    ("kfj", 32, "coherence"): ["C-n16-ja98-coherence"],
    ("kfj", 64, "I"): ["C-n32-ja98-I"],
    ("kfj", 64, "IQUV"): ["C-n32-ja98-IQUV"],
    ("kfj", 64, "coherence"): ["C-n32-ja98-coherence"],
    ("kfj", 128, "I"): ["C-n64-ja98-I"],
    ("kfj", 128, "IQUV"): ["C-n64-ja98-IQUV"],
    ("kfj", 128, "coherence"): ["C-n64-ja98-coherence"],
    ("kfj", 256, "I"): ["C-n128-ja98-I"],
    ("kfj", 256, "IQUV"): ["C-n128-ja98-IQUV"],
    ("kfj", 256, "coherence"): ["C-n128-ja98-coherence"],
    ("kfj", 512, "I"): ["C-n256-ja98-I"],
    ("kfj", 512, "IQUV"): ["C-n256-ja98-IQUV"],
    ("kfj", 512, "coherence"): ["C-n256-ja98-coherence"],
    ("kg_col", 2): ["E-n2048-fr1024-I", "E-n2048-fr1024-coherence", "E-n2048-fr1024-IQUV", "E-n2048-fr1024-PPQQ",
        "E-n2048-runtime-I", "E-n2048-runtime-coherence", "H-generic-n128"],
    ("kg_col", 8): ["E-n64-fr256-8bit-coherence"],
    ("kg_col", 22): ["E-n64-fr256-ja98-coherence"],
    ("kg_row", 4, "volt"): ["H-generic-n128"],
    ("kg_row", 4, "detect"): ["E-n64-fr256-8bit-coherence", "E-n64-fr256-ja98-coherence"],
    ("kg_row", 8, "volt"): ["E-n2048-dedisp-I", "E-n2048-dedisp-IQUV", "E-n2048-dedisp-trials"],
    ("kg_row", 8, "detect"): ["E-n2048-fr1024-I", "E-n2048-fr1024-coherence", "E-n2048-fr1024-IQUV", "E-n2048-fr1024-PPQQ",
        "E-n2048-runtime-I", "E-n2048-runtime-coherence"],
    ("kgt_col", 10, 2): ["F-n512-P0", "F-n512-P1", "F-n512-I", "F-n512-I2", "F-n512-PPQQ", "F-n512-coherence", "F-n512-IQUV"],
    ("kgt_col", 10, 8): ["F-n512-8bit-I"],
    ("kgt_col", 10, 22): ["F-n512-ja98-I"],
    ("kgt_col", 11, 2): ["F-n1024-P0", "F-n1024-P1", "F-n1024-I", "F-n1024-I2", "F-n1024-PPQQ", "F-n1024-coherence",
        "F-n1024-IQUV"],
    ("kgt_col", 11, 8): ["F-n1024-8bit-I"],
    ("kgt_col", 11, 22): ["F-n1024-ja98-I"],
    ("kgt_col", 12, 2): ["F-n2048-P0", "F-n2048-P1", "F-n2048-I", "F-n2048-I2", "F-n2048-PPQQ", "F-n2048-coherence",
        "F-n2048-IQUV", "E-n2048-dedisp-I", "E-n2048-dedisp-IQUV", "E-n2048-dedisp-trials"],
    ("kgt_col", 12, 8): ["F-n2048-8bit-I"],
    ("kgt_col", 12, 22): ["F-n2048-ja98-I"],
    ("kgt_col", 13, 2): ["F-n4096-P0", "F-n4096-P1", "F-n4096-I", "F-n4096-I2", "F-n4096-PPQQ", "F-n4096-coherence",
        "F-n4096-IQUV"],
    ("kgt_col", 13, 8): ["F-n4096-8bit-I"],
    ("kgt_col", 13, 22): ["F-n4096-ja98-I"],
    ("kgt_row", 10, "I"): ["F-n512-I", "F-n512-ja98-I", "F-n512-8bit-I"],
    ("kgt_row", 10, "I2"): ["F-n512-I2"],
    ("kgt_row", 10, "P0"): ["F-n512-P0"],
    ("kgt_row", 10, "P1"): ["F-n512-P1"],
    ("kgt_row", 10, "IQUV"): ["F-n512-IQUV"],
    ("kgt_row", 10, "PPQQ"): ["F-n512-PPQQ"],
    ("kgt_row", 10, "coherence"): ["F-n512-coherence"],
    ("kgt_row", 11, "I"): ["F-n1024-I", "F-n1024-ja98-I", "F-n1024-8bit-I"],
    ("kgt_row", 11, "I2"): ["F-n1024-I2"],
    ("kgt_row", 11, "P0"): ["F-n1024-P0"],
    ("kgt_row", 11, "P1"): ["F-n1024-P1"],
    ("kgt_row", 11, "IQUV"): ["F-n1024-IQUV"],
    ("kgt_row", 11, "PPQQ"): ["F-n1024-PPQQ"],
    ("kgt_row", 11, "coherence"): ["F-n1024-coherence"],
    ("kgt_row", 12, "I"): ["F-n2048-I", "F-n2048-ja98-I", "F-n2048-8bit-I"],
    ("kgt_row", 12, "I2"): ["F-n2048-I2"],
    ("kgt_row", 12, "P0"): ["F-n2048-P0"],
    ("kgt_row", 12, "P1"): ["F-n2048-P1"],
    ("kgt_row", 12, "IQUV"): ["F-n2048-IQUV"],
    ("kgt_row", 12, "PPQQ"): ["F-n2048-PPQQ"],
    ("kgt_row", 12, "coherence"): ["F-n2048-coherence"],
    ("kgt_row", 13, "I"): ["F-n4096-I", "F-n4096-ja98-I", "F-n4096-8bit-I"],
    ("kgt_row", 13, "I2"): ["F-n4096-I2"],
    ("kgt_row", 13, "P0"): ["F-n4096-P0"],
    ("kgt_row", 13, "P1"): ["F-n4096-P1"],
    ("kgt_row", 13, "IQUV"): ["F-n4096-IQUV"],
    ("kgt_row", 13, "PPQQ"): ["F-n4096-PPQQ"],
    ("kgt_row", 13, "coherence"): ["F-n4096-coherence"],
    ("kl_detect", "I"): ["G-n64-I", "H-long-n8"],
    ("kl_detect", "I2"): ["G-n64-I2"],
    ("kl_detect", "P0"): ["G-n64-P0"],
    ("kl_detect", "P1"): ["G-n64-P1"],
    ("kl_detect", "IQUV"): ["G-n64-IQUV", "G-n16-fr8192-IQUV"],
    ("kl_detect", "PPQQ"): ["G-n64-PPQQ"],
    ("kl_detect", "coherence"): ["G-n64-coherence", "G-n64-batch1-coherence", "G-n64-batch5-coherence", "G-n64-trials",
        "G-n8-fr8192-coherence", "G-n8-trials", "H-long-n64"],
    ("kl_pass", "f"): ["G-n64-P0", "G-n64-P1", "G-n64-I", "G-n64-I2", "G-n64-PPQQ", "G-n64-coherence", "G-n64-IQUV",
        "G-n64-batch1-coherence", "G-n64-batch5-coherence", "G-n64-trials", "G-n8-fr8192-coherence", "G-n8-trials",
        "G-n16-fr8192-IQUV", "H-long-n8", "H-long-n64"],
    ("kl_pass", "unmix"): ["G-n64-P0", "G-n64-P1", "G-n64-I", "G-n64-I2", "G-n64-PPQQ", "G-n64-coherence", "G-n64-IQUV",
        "G-n64-batch1-coherence", "G-n64-batch5-coherence", "G-n64-trials", "G-n8-fr8192-coherence", "G-n8-trials",
        "G-n16-fr8192-IQUV", "H-long-n8", "H-long-n64"],
    ("kl_pass", "stream"): ["G-n64-P0", "G-n64-P1", "G-n64-I", "G-n64-I2", "G-n64-PPQQ", "G-n64-coherence", "G-n64-IQUV",
        "G-n64-batch1-coherence", "G-n64-batch5-coherence", "G-n64-trials", "G-n8-fr8192-coherence", "G-n8-trials",
        "G-n16-fr8192-IQUV", "H-long-n8", "H-long-n64"],
    ("kr", 16, "I"): ["C-n8-I-split"],
    ("kr", 16, "IQUV"): ["C-n8-IQUV-split"],
    ("kr", 16, "coherence"): ["C-n8-coherence-split"],
    ("kr", 32, "I"): ["C-n16-I-split"],
    ("kr", 32, "IQUV"): ["C-n16-IQUV-split"],
    ("kr", 32, "coherence"): ["C-n16-coherence-split"],
    ("kr", 64, "I"): ["C-n32-I-split"],
    ("kr", 64, "IQUV"): ["C-n32-IQUV-split"],
    ("kr", 64, "coherence"): ["C-n32-coherence-split"],
    ("kr", 128, "I"): ["C-n64-I-split"],
    ("kr", 128, "IQUV"): ["C-n64-IQUV-split"],
    ("kr", 128, "coherence"): ["C-n64-coherence-split"],
    ("kr", 512, "I"): ["C-n256-I-split"],
    ("kr", 512, "IQUV"): ["C-n256-IQUV-split"],
    ("kr", 512, "coherence"): ["C-n256-coherence-split"],
    ("kx",): ["E-n2048-dedisp-I", "E-n2048-dedisp-IQUV", "E-n2048-dedisp-trials", "H-generic-n128"],
}


# ---------------------------------------------------------------- oracle, with the channelisations shared between cases
_streams, _chan = {}, {}


def _lru(cache, key, make, keep):
    if key in cache:
        cache[key] = cache.pop(key)
        return cache[key]
    while len(cache) >= keep:
        cache.pop(next(iter(cache)))
    cache[key] = make()
    return cache[key]


def inputs(c):
    """(VDIF per IF, signed bw, centre freq).  Several IFs: alternating sidebands, first IF LSB, fault mix per IF (clean,
    invalid frames, fill words); one IF: LSB at 1254 MHz or USB at 1286 MHz with both kinds of fault."""
    nif = c["nif"]
    if nif == 1:
        bws, freqs, faults = [BW if c["usb"] else -BW], [1286.0 if c["usb"] else 1254.0], [{"invalid_frac": 0.01, "fill_frac": 0.01}]
    else:
        bws, freqs, faults = [BW if i % 2 else -BW for i in range(nif)], [1254.0 + BW * i for i in range(nif)], None
    key = (nif, c["usb"], c["nframes"], c["nbit"], c["seed"])
    vd = _lru(_streams, key, lambda: streams(nif, c["nframes"], c["seed"], nbit=c["nbit"], faults=faults), 2)
    return vd, bws, freqs


def channelise(vd, bws, freqs, c, L, dm, nfilt, dtype=np.float64):
    """Per IF (yP, yQ): the oracle's complex channel samples [t, chan] in natural channel order, cut to the shortest IF."""
    out = []
    for v, b, f in zip(vd, bws, freqs):
        x = o.decode_vdif(v, nbit=c["nbit"], header_bytes=32, frame_bytes=8032, mode=c["decode"])
        if dm > 0:
            H = o.chirp(c["nchan"], L, f, b, dm)
            out.append([o.filterbank_dedisp(x[p], c["nchan"], L, H, nfilt[0], nfilt[1], dtype) for p in (0, 1)])
        else:
            out.append([o.filterbank(x[p], c["nchan"], L, dtype) for p in (0, 1)])
        del x
    n = min(y[0].shape[0] for y in out)
    return [(a[:n], q[:n]) for a, q in out]


def channelised(c, L, dm, nfilt):
    vd, bws, freqs = inputs(c)
    key = (c["nif"], c["usb"], c["nframes"], c["nbit"], c["seed"], c["decode"], c["nchan"], L, dm, tuple(nfilt))
    return _lru(_chan, key, lambda: channelise(vd, bws, freqs, c, L, dm, nfilt), 1)


def products(ch, pol, D):
    """Detected, integrated products per IF [t, nprod, chan], in pieces of about 4M samples to bound the memory."""
    out = []
    for a, q in ch:
        n = a.shape[0] // D * D
        step = max(D, (1 << 22) // a.shape[1] // D * D)
        out.append(np.concatenate([o.tscrunch(o.detect(a[t:min(t + step, n)], q[t:min(t + step, n)], MODE[pol]), D)
                                   for t in range(0, n, step)]))
    return out


# ---------------------------------------------------------------- running a case
def plan_kw(c, bws, freqs, chunk, dm=None):
    kw = dict(nchan=c["nchan"], bw=bws, freq=freqs, tscrunch=c["D"], pol_mode=c["pol"], in_nbit=c["nbit"], chunk_units=chunk)
    if c["freq_res"]:
        kw["freq_res"] = c["freq_res"]
    if c["decode"] == "ja98":
        kw["decode_mode"] = _lib.DECODE_JA98
    if c["trials"]:
        kw.update(coherent=True, dm_trials=list(c["trials"]))
    elif dm:
        kw.update(coherent=True, dm=dm)
    return kw


def probe(kw):
    """Plan geometry and path, no data."""
    cfg = dict(kw)
    cfg["bw_mhz"], cfg["freq_mhz"] = cfg.pop("bw"), cfg.pop("freq")
    with Plan(PlanConfig(**cfg)) as pl:
        return pl.geometry, pl.path


def _keep(g):
    return int(g.freq_res) - int(g.nfilt_pos) - int(g.nfilt_neg)


def dm_edge(c, bws, freqs):
    """Largest DM (to 1e-7) whose plan is accepted with freq_res L and keeps at least keep_min samples of each block."""
    def ok(dm):
        try:
            g, _ = probe(plan_kw(c, bws, freqs, c["push"] or 1, dm))
        except _lib.B2FError as e:
            if e.code != _lib.EUNSUPPORTED:
                raise
            return False
        return int(g.freq_res) == c["L"] and _keep(g) >= max(1, c["keep_min"])
    lo, hi = 1.0, 2.0
    assert ok(lo)
    while ok(hi):
        lo, hi = hi, 2 * hi
    while hi - lo > 1e-7 * hi:
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if ok(mid) else (lo, mid)
    return lo


def chunk_units(c, bws, freqs, dm):
    """Push size: the case's frames on the carry paths; on the tuned 512-point shapes whole push units, about a third of
    the input with dedispersion (units of a few frames), one unit otherwise."""
    if c["push"] or c["L"] != 512:
        return c["push"]
    if not (c["dm"] or c["trials"]):
        return 1
    g, _ = probe(plan_kw(c, bws, freqs, 1, dm))
    return max(1, c["nframes"] // 3 // int(g.unit_frames))


def run(c, vd, bws, freqs, chunk, dm, monkeypatch):
    with monkeypatch.context() as m:
        for k in ENV:
            m.delenv(k, raising=False)
        for k, v in c["env"].items():
            m.setenv(k, v)
        return run_plan(vd, out_nbit=-32, keep_bandpass=True, profile=True, **plan_kw(c, bws, freqs, chunk, dm))


def check(rows, fl, bws, info, c, what, redo32):
    """The plan's tiles against the float64 oracle; a failure also reports how far the oracle itself moves when its
    channelisation runs in float32 -- the rounding to expect of a correct float32 kernel."""
    try:
        check_splice(rows, expected_tiles(fl, bws, out_nbit=-32), info["if_order"], pol=c["pol"], nchan=c["nchan"], out_nbit=-32,
                     pol_major=False, what=what)
    except AssertionError as ex:
        f32 = redo32()
        e32 = max(assert_rel(a, b, np.inf, power=(b[:, 0] + b[:, 1] if c["pol"] == COH else b[:, 0]) if c["pol"] in (COH, IQUV) else None)
                  for a, b in zip(f32, fl))
        raise AssertionError(f"{ex}\nthe float32 oracle differs from the float64 one by {e32:.2e} (max rel err)") from None


@pytest.mark.parametrize("cid", list(CASES))
def test_dispatch_case(gpu, monkeypatch, cid):
    c = CASES[cid]
    vd, bws, freqs = inputs(c)
    dm = dm_edge(c, bws, freqs) if c["dm"] == "edge" else c["dm"]
    top = max(c["trials"]) if c["trials"] else dm
    chunk = chunk_units(c, bws, freqs, dm)
    rows, info = run(c, vd, bws, freqs, chunk, dm, monkeypatch)
    g, L, D = info["geometry"], c["L"], c["D"]

    # the arm that ran: path, geometry, launch counts
    exp = expected_arms(c, L)
    assert exp["arms"] == {k for k, ids in MATRIX.items() if cid in ids}
    assert info["path"] == exp["path"] and int(g.freq_res) == L
    assert int(g.ndm) == (len(c["trials"]) if c["trials"] else 1)
    counts = {k: info["times"][k][1] for k in TIMED}
    assert {k for k, n in counts.items() if n > 0} == exp["launched"], counts
    nf = (int(g.nfilt_pos), int(g.nfilt_neg))
    if top:
        assert nf[0] == nf[1] > 0 and nf[0] % kernel_D(D, L, True) == 0
        if c["fam"] == "D":                                          # 2 nfilt ~ 0.6 x 512
            assert 0.55 * 512 < 2 * nf[0] < 0.7 * 512, nf
        if c["dm"] == "edge":
            keep, Dk = _keep(g), kernel_D(D, L, True)
            assert keep // Dk >= 1
            if c["keep_min"]:                                        # the next DM step would leave less than keep_min
                assert c["keep_min"] <= keep < c["keep_min"] + 2 * Dk, (keep, Dk)
            else:                                                    # the next DM step would leave nothing
                assert keep == 2 * Dk, (keep, Dk)
    else:
        assert nf == (0, 0)
    if c["fam"] in ("E", "F", "G") and c["push"]:
        assert info["chunk_frames"] == c["push"] < c["nframes"]      # blocks straddle pushes

    # the rows against the oracle, every trial with the plan's nfilt and freq_res
    dms = c["trials"] or [dm]
    parts = np.split(rows.reshape(rows.shape[0], -1), len(dms), axis=1)
    for k, (dmk, part) in enumerate(zip(dms, parts)):
        if len(dms) > 1:
            ch = channelise(vd, bws, freqs, c, L, dmk, nf)             # trials: not kept
        else:
            ch = channelised(c, L, dmk, nf)
        fl = products(ch, c["pol"], D)
        del ch
        what = f"{cid}" + (f" trial DM {dmk:.2f}" if len(dms) > 1 else "")
        check(part, fl, bws, info, c, what, lambda: products(channelise(vd, bws, freqs, c, L, dmk, nf, np.float32), c["pol"], D))

    # batches, and the largest trial, change no bit of what the reference case computes
    if c["same_as"]:
        ref = CASES[c["same_as"]]
        one, _ = run(ref, vd, bws, freqs, chunk_units(ref, bws, freqs, top), top, monkeypatch)
        got = np.ascontiguousarray(parts[-1] if c["trials"] else rows)
        assert np.array_equal(got.view(np.uint8), one.view(np.uint8).reshape(one.shape[0], -1)), \
            f"{cid} differs from {c['same_as']} in {(got != one.reshape(got.shape)).mean():.2e} of its samples"


def test_ja98_tuned_dedispersion_refuses_unaligned_blocks(gpu):
    """nchan 8 at 2 nfilt ~ 0.6 x 512 with tscrunch 4: keep = 200, so blocks start every 3200 samples and the JA98 windows
    of a later push would not be the scan's.  The plan refuses it; the static levels and tscrunch 16 (D-n8-ja98-coherence)
    are accepted."""
    c = dict(CASES["D-n8-ja98-coherence"], D=4)
    bws, freqs = [-BW, BW], [1254.0, 1254.0 + BW]
    with pytest.raises(_lib.B2FError) as e:
        probe(plan_kw(c, bws, freqs, 1, c["dm"]))
    assert e.value.code == _lib.EUNSUPPORTED and "512" in e.value.message
    g, _ = probe(plan_kw(dict(c, decode="static"), bws, freqs, 1, c["dm"]))
    assert _keep(g) * 16 % 512
    g, _ = probe(plan_kw(CASES["D-n8-ja98-coherence"], bws, freqs, 1, c["dm"]))
    assert _keep(g) * 16 % 512 == 0
