#!/usr/bin/env python3
"""B200 drop-in for the per-subband wrapper of frb-baseband.

Contract kept (all citations into /root/reference/process_vdif.py):
  * command line: every flag, default and choice list of `options()` (:9-99), so the call
    base2fil.sh:61-64 makes works unchanged;
  * `make_hdr(...)` writes the same 12-line DSPSR header to <dir>/<vdif>_pol<p>.hdr (:115-139);
  * `run_digifil(...)` keeps its signature and output naming, refuses to clobber an existing
    file without overwrite, and never unlinks a FIFO (:142-155);
  * `InputError` / `RunError` carry `.message` (:231-255); neither/both of -l/-u is an
    InputError (:260-265).
What differs: the arithmetic runs in libb2f.so on the GPU instead of in a `digifil` child
process.  No library or no GPU -> RunError; nothing is computed on the CPU.
"""
import argparse
import os
import stat
import subprocess
import sys


# (flags, argparse keywords, option group) -- one row per option of the reference CLI
_G, _D, _P = "General info about the data.", "Input to digifil.", "Input to prepdata/prepsubband"
_CLI = [
    (("psrname",), dict(type=str, help="B/J name of the target; unknown sources also need --ra/--dec"), _G),
    (("filename",), dict(type=str, help="split VDIF file of one subband (two channels = two polarisations)"), _G),
    (("-f", "--freq"), dict(type=float, default=1608.0, help="centre frequency [MHz] (%(default)s)"), _G),
    (("--ra",), dict(type=str, default=None, help="hh:mm:ss.ss"), _G),
    (("--dec",), dict(type=str, default=None, help="dd:mm:ss.ss"), _G),
    (("-b", "--bw"), dict(type=float, default=16.0, help="subband bandwidth [MHz] (%(default)s)"), _G),
    (("-u", "--usb"), dict(action="store_true", help="upper sideband; exactly one of -u/-l is required"), _G),
    (("-l", "--lsb"), dict(action="store_true", help="lower sideband; exactly one of -u/-l is required"), _G),
    (("-t", "--telescope"), dict(type=str, default="ONSALA85", help="tempo2 telescope name (%(default)s)"), _G),
    (("--use_tmp",), dict(action="store_true", help="write the .hdr to /tmp"), _G),
    (("--hdr_only",), dict(action="store_true", help="stop after writing the .hdr"), _G),
    (("--fil_out_dir",), dict(type=str, default=None, help="directory (or FIFO directory) for the .fil"), _D),
    (("--nchan",), dict(type=int, default=512, help="channels per subband (%(default)s)"), _D),
    (("--nsec",), dict(type=float, default=120, help="seconds to process (%(default)s)"), _D),
    (("--start",), dict(type=float, default=1, help="seconds to skip at the start of the file (%(default)s)"), _D),
    (("--force",), dict(action="store_true", help="replace an existing regular output file"), _D),
    (("--pol",), dict(type=int, default=2, choices=[0, 1, 2, 3, 4],
                      help="0/1 one polarisation, 2 Stokes I, 3 (PP+QQ)^2, 4 PP,QQ,PQ,QP (%(default)s)"), _D),
    (("--nbit",), dict(type=int, default=8, choices=[2, 8, 16, -32], help="output bits, -32 = float (%(default)s)"), _D),
    (("--keepBP",), dict(action="store_true", help="no rescaling: keep the bandpass (digifil -I0)"), _D),
    (("--tscrunch",), dict(type=int, default=1, help="time integration factor, digifil -t (%(default)s)"), _D),
    (("--nthreads",), dict(type=int, default=1, help="accepted for compatibility, unused on the GPU"), _D),
    (("--device",), dict(type=int, default=int(os.environ.get("B2F_DEVICE", "0")), help="CUDA ordinal (extension)"), _D),
    (("--coherent_dm",), dict(type=float, default=0.0,
                              help="extension: coherently dedisperse inside each channel at this DM "
                                   "(run_digifil's dm/coherent arguments, which the reference CLI never sets)"), _D),
    (("--coherent_numdms",), dict(type=int, default=1,
                                  help="extension: with N >= 2, coherent dedispersion at the N trial DMs coherent_dm + k "
                                       "coherent_dmstep in one pass, one <stem>_DM<dm>.fil per trial (%(default)s)"), _D),
    (("--coherent_dmstep",), dict(type=float, default=0.0, help="extension: DM step of the coherent trials"), _D),
    (("--remove_delays",), dict(action="store_true",
                                help="extension: also remove the inter-channel dispersion delays at the coherent DM (or each "
                                     "trial DM), aligned to the top channel (digifil -K)"), _D),
    (("--do_prepdata",), dict(action="store_true", help="run PRESTO prepdata/prepsubband afterwards"), _P),
    (("--ncpus",), dict(type=int, default=1, help="1: prepdata, >1: prepsubband"), _P),
    (("--dm",), dict(type=float, default=None, help="DM for prepdata (default: psrcat)"), _P),
    (("--nozerodm",), dict(action="store_false", help="drop -zerodm"), _P),
    (("--clip",), dict(type=int, default=5, help="prepdata -clip, 0 disables (%(default)s)"), _P),
    (("--dm2",), dict(type=float, default=0.0, help="upper DM of a prepsubband range"), _P),
    (("--dmstep",), dict(type=float, default=1.0, help="DM step of that range"), _P),
]


class Error(Exception):
    """Base class of this module's exceptions."""


class InputError(Error):
    """Bad input from the caller."""

    def __init__(self, message):
        super().__init__(message)
        self.message = message


class RunError(Error):
    """The processing itself failed."""

    def __init__(self, message):
        super().__init__(message)
        self.message = message


def options(argv=None):
    parser = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    groups = {}
    for flags, kw, grp in _CLI:
        g = groups.setdefault(grp, parser.add_argument_group(grp))
        g.add_argument(*flags, **kw)
    return parser.parse_args(argv)


def psr_info(psr):
    """(raj, decj, dm) from psrcat, as the reference does for known pulsars (:102-108)."""
    try:
        fields = subprocess.check_output(["psrcat", "-c", "raj decj dm", "-o", "short", "-nohead", "-nonumber", psr]).split()
        ra, dec, dm = fields
    except Exception:
        raise RunError("psrcat died on given source {0}".format(psr))
    return ra.decode(), dec.decode(), float(dm)


def make_hdr(psr, freq, filename, pol=2, usb=True, ra=None, dec=None, bw=16.0, telescope="ONSALA85", npol=2, tmp=False):
    """Write the DSPSR ASCII header and return its path.  BW carries the sideband as its sign."""
    if ra is None or dec is None:
        ra, dec, _ = psr_info(psr)
    signed_bw = bw if usb else -bw
    rows = [("HDR_VERSION", "0.1", 1), ("TELESCOPE", telescope, 2), ("SOURCE", psr, 5), ("RA", ra, 9), ("DEC", dec, 8),
            ("FREQ", freq, 7), ("BW", signed_bw, 9), ("DATAFILE", filename, 3), ("INSTRUMENT", "VDIF", 1),
            ("MODE", "PSR", 7), ("BASIS", "Circular", 6), ("NPOL", npol, 7)]
    text = "\n".join("{0}{1}{2}".format(k, " " * pad, v) for k, v, pad in rows)
    where = "/tmp/" if tmp else os.path.dirname(filename)
    hdrfile = "{0}/{1}_pol{2}.hdr".format(where, os.path.basename(filename), pol)
    with open(hdrfile, "w") as f:
        f.write(text)
    return hdrfile


def read_hdr(hdrfile):
    """keyword -> value of a DSPSR ASCII header"""
    kv = {}
    with open(hdrfile) as f:
        for line in f:
            parts = line.split(None, 1)
            if len(parts) == 2:
                kv[parts[0]] = parts[1].strip()
    return kv


def _output_path(hdr, fil_out_dir, overwrite):
    fil = hdr[:-4] + ".fil" if hdr.endswith(".hdr") else hdr.replace(".hdr", ".fil")
    if fil_out_dir is not None:
        fil = "{0}/{1}".format(fil_out_dir, os.path.basename(fil))
    if os.path.exists(fil):
        if not overwrite:
            raise InputError("Filterbankfile {0} exists already. Delete first or set --force to overwrite".format(fil))
        if not stat.S_ISFIFO(os.stat(fil).st_mode):      # a FIFO made by base2fil.sh:348-349 is kept
            os.remove(fil)
    return fil


def coherent_trials(dm, numdms, dmstep):
    """Trial DMs of --coherent_dm/--coherent_numdms/--coherent_dmstep (prepsubband's -lodm/-numdms/-dmstep), or None
    for a single DM (numdms 1)."""
    if numdms < 1:
        raise InputError(f"--coherent_numdms {numdms}: must be >= 1")
    if numdms == 1:
        return None
    if not dmstep > 0:
        raise InputError("--coherent_numdms >= 2 needs --coherent_dmstep > 0")
    if dm < 0:
        raise InputError("--coherent_dm must be >= 0")
    return [dm + k * dmstep for k in range(numdms)]


def trial_output_paths(hdr, fil_out_dir, dm_trials):
    """<stem>_DM<dm:.2f>.fil per trial DM, in fil_out_dir (or beside the .hdr)."""
    fil = hdr[:-4] + ".fil" if hdr.endswith(".hdr") else hdr.replace(".hdr", ".fil")
    if fil_out_dir is not None:
        fil = "{0}/{1}".format(fil_out_dir, os.path.basename(fil))
    stem = fil[:-4]
    return ["{0}_DM{1:.2f}.fil".format(stem, d) for d in dm_trials]


def run_digifil(hdr, fil_out_dir=None, start=1, nsecs=120, nchan=128, overwrite=False, pol=2, nbit=8,
                tscrunch=1, nthreads=1, dm=0.0, coherent=False, keepBP=False, device=0, dm_trials=None, remove_delays=False):
    """Baseband -> filterbank for the subband described by `hdr`; returns the .fil path.  With `dm_trials` (a list of
    DMs) one pass writes a coherently dedispersed filterbank per trial and the list of their paths is returned.
    `remove_delays` (digifil -K): the inter-channel delays at `dm` (or each trial DM) are removed as well; with
    coherent=False that is incoherent dedispersion alone."""
    if dm_trials is not None:
        fils = trial_output_paths(hdr, fil_out_dir, dm_trials)
        for f in fils:
            if os.path.exists(f):
                if not overwrite:
                    raise InputError("Filterbankfile {0} exists already. Delete first or set --force to overwrite".format(f))
                if stat.S_ISFIFO(os.stat(f).st_mode):
                    raise InputError("{0}: trial DM outputs must be regular files, not FIFOs".format(f))
                os.remove(f)
        fil = fils
        dm, coherent = 0.0, True
    else:
        fil = _output_path(hdr, fil_out_dir, overwrite)
    if nbit not in (2, 8, 16, -32):
        raise InputError(f"nbit={nbit} not in supported values of [2, 8, 16, -32]. ")
    if pol not in (0, 1, 2, 3, 4):
        raise InputError(f"pol = {pol} not implemented. Choices are 0, 1, 2, 3, 4")
    from . import _lib, sigproc, vdif
    from .admission import GpuSlot
    from .plan import Plan, PlanConfig, pol_mode_from_reference, reference_freq_res

    kv = read_hdr(hdr)
    datafile, freq, bw = kv["DATAFILE"], float(kv["FREQ"]), float(kv["BW"])
    dedisp = "D -D {0}".format(dm) if (coherent and dm > 0) else reference_freq_res(nchan)
    if dm_trials is not None:
        dedisp = "D -D {0}".format(",".join("{0:.2f}".format(d) for d in dm_trials))
    if remove_delays and not (coherent and dm > 0) and dm_trials is None:
        dedisp = "{0} -D {1}".format(dedisp, dm)
    print("running b2f -b{0} -S{1} -T{2} -t {3} -o {4} {5} pol={6} -F{7}:{8}{9}{10} (libb2f.so, cuda:{11})".format(
        nbit, start, nsecs, tscrunch, " ".join(fil) if dm_trials is not None else fil, hdr, pol, nchan, dedisp,
        " -K" if remove_delays else "", " -I0" if keepBP else "", device))
    try:
        with open(datafile, "rb") as src:
            info = vdif.parse_header(src.read(32))
        fps = vdif.frames_per_second(bw, info)
        if abs(fps - round(fps)) > 1e-6:
            raise InputError(f"{datafile}: {fps} frames per second is not an integer for bw={bw}")
        cfg = PlanConfig(nchan=nchan, bw_mhz=[bw], freq_mhz=[freq], tscrunch=max(1, tscrunch),
                         pol_mode=pol_mode_from_reference(pol), out_nbit=nbit, in_nbit=info.nbit,
                         frame_bytes=info.frame_bytes, header_bytes=info.header_bytes, keep_bandpass=keepBP,
                         device=device, dm=float(dm), coherent=bool(coherent and (dm > 0.0 or dm_trials is not None)),
                         dm_trials=None if dm_trials is None else [float(d) for d in dm_trials],
                         remove_delays=bool(remove_delays),
                         # the reference passes -2 (:157,160): DSPSR's dynamic 2-bit levels; this build defaults to the
                         # static optimal levels, B2F_DECODE_MODE=ja98 selects the reference-faithful unpacker
                         decode_mode=_lib.DECODE_JA98 if os.environ.get("B2F_DECODE_MODE", "").lower() == "ja98" else _lib.DECODE_STATIC)
        # pwait (base2fil.sh:21-28,404-405) counts processes named digifil; B2F_MAX_CONCURRENT is the same throttle here
        with GpuSlot(device), Plan(cfg) as pl:
            # the digifil child process (reference :191): file in, .fil (or FIFO) out, inside libb2f
            c = pl.run_scan([datafile], fil, start_s=start, nsec=nsecs, source_name=kv.get("SOURCE", "unknown"),
                            telescope_id=sigproc.TELESCOPE_IDS.get(kv.get("TELESCOPE", "").lower(), 0),
                            src_raj=sigproc.sexagesimal_to_sigproc(kv.get("RA")),
                            src_dej=sigproc.sexagesimal_to_sigproc(kv.get("DEC")),
                            refdm=None if dm_trials is not None else dm)["counters"]
        if c["frames_invalid"] or c["frames_with_fill"] or c["frames_badhdr"]:
            print("b2f: masked {frames_invalid} invalid, {frames_with_fill} fill-pattern and {frames_badhdr} "
                  "malformed frames".format(**c), file=sys.stderr)
    except _lib.B2FError as e:
        if e.code == _lib.EINVAL:
            raise InputError(e.message)
        raise RunError("b2f died: {0}".format(e.message))
    except OSError as e:
        raise RunError("b2f died: {0}".format(e))
    return fil


def prepdata(filterbankfile, dm1, zerodm=True, clip=5, dm2=0, dmstep=1.0, ncpus=1):
    """Optional PRESTO step after the filterbank exists (reference :202-229); not part of the hot path."""
    if dm2 > 0.0 and dm2 < dm1:
        raise InputError("DM2 must be larger than DM1.")
    stem = filterbankfile.replace(".fil", "")
    if dm2 > 0.0:
        argv = ["prepsubband", "-lodm", str(dm1), "-numdms", str(int((dm2 - dm1) // dmstep + 1)), "-dmstep", str(dmstep)]
        outfile = stem
    else:
        argv = ["prepdata", "-dm", str(dm1)]
        outfile = "{0}_dm{1}".format(stem, dm1)
    argv += ["-filterbank", "-noweights", "-noscales", "-nobary", "-ncpus", str(ncpus)]
    argv += ["-zerodm"] if zerodm else []
    argv += ["-clip", str(clip)] if clip > 0 else []
    argv += ["-o", outfile, filterbankfile]
    print("running " + " ".join(argv))
    try:
        subprocess.check_call(argv)
    except (subprocess.CalledProcessError, OSError):
        raise RunError("Prepdata died.")


def main(argv=None):
    a = options(argv)
    if a.usb == a.lsb:
        raise InputError("You MUST supply either -l OR -u " +
                         ("not both." if a.usb else "to specify if data are LSB or USB"))
    hdr = make_hdr(a.psrname, a.freq, a.filename, usb=a.usb, bw=a.bw, telescope=a.telescope, tmp=a.use_tmp,
                   ra=a.ra, dec=a.dec, pol=a.pol)
    if a.hdr_only:
        print("Not creating filterbanks. Hdr files done.")
        return 0
    trials = coherent_trials(a.coherent_dm, a.coherent_numdms, a.coherent_dmstep)
    if a.do_prepdata and trials is not None:
        raise InputError("--do_prepdata takes one filterbank: not with --coherent_numdms >= 2")
    fil = run_digifil(hdr, a.fil_out_dir, a.start, a.nsec, a.nchan, overwrite=a.force, pol=a.pol, nbit=a.nbit,
                      tscrunch=a.tscrunch, nthreads=a.nthreads, keepBP=a.keepBP, device=a.device,
                      dm=a.coherent_dm, coherent=a.coherent_dm > 0.0, dm_trials=trials, remove_delays=a.remove_delays)
    if a.do_prepdata:
        prepdata(fil, a.dm if a.dm is not None else psr_info(a.psrname)[2], zerodm=a.nozerodm, clip=a.clip,
                 dm2=a.dm2, dmstep=a.dmstep, ncpus=a.ncpus)
    return 0


if __name__ == "__main__":
    sys.exit(main())
