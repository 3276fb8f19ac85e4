"""Python face of a libb2f plan: one object = one `digifil` invocation per IF plus the
`splice` that joins them (/root/reference/process_vdif.py:142-199,
/root/reference/base2fil.sh:404-448), running on one GPU.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from ._lib import B2FError  # noqa: F401  (re-export)


def reference_freq_res(nchan: int) -> int:
    """leakage factor digifil is given: /root/reference/process_vdif.py:162"""
    return 512 if nchan <= 128 else 2 * nchan


def pol_mode_from_reference(pol: int) -> int:
    """--pol of process_vdif (/root/reference/process_vdif.py:58-64,163-176) -> b2f_pol_mode"""
    try:
        return {0: _lib.POL_P0, 1: _lib.POL_P1, 2: _lib.POL_I, 3: _lib.POL_I2, 4: _lib.POL_COHERENCE}[pol]
    except KeyError:
        raise ValueError(f"pol = {pol} not implemented. Choices are 0, 1, 2, 3, 4")


@dataclass
class PlanConfig:
    nchan: int
    bw_mhz: list[float]                     # signed per IF: negative = LSB
    freq_mhz: list[float] | None = None
    if_order: list[int] | None = None       # output tile s <- IF index; default: descending frequency
    tscrunch: int = 1
    pol_mode: int = _lib.POL_I
    out_nbit: int = 8
    in_nbit: int = 2
    frame_bytes: int = 8032
    header_bytes: int = 32
    freq_res: int = 0
    frame_time_mode: int = 0
    mask_faults: bool = True
    keep_bandpass: bool = False
    splice_pol_major: bool = False
    chunk_units: int = 0                     # 0 = library default (about 2048 frames per IF and push)
    rescale_interval_s: float = 10.0
    device: int = 0
    profile: bool = False
    stream: int | None = None
    dm: float = 0.0                          # digifil -D
    coherent: bool = False                   # digifil -F nchan:D
    dm_trials: list[float] | None = None     # coherent dedispersion at each of these DMs in one pass (dm stays 0)
    raw_word_bits: int = 0                   # 16/32/64: one raw multi-BBC VDIF stream, corner turn on the GPU
    raw_bits: list | None = None             # per IF: 4 source bit positions (spif2file recipe)
    raw_format: int = 0                      # 0 VDIF frames, 1 Mark5B disk frames (16 B header, 10000 B payload)
    decode_mode: int = 0                     # 0 static optimal levels, 1 Jenet-Anderson dynamic levels per 512 samples (SURVEY D2)
    in8_offset_mode: int = 0                 # 8-bit input: 0 code - 127.5, 1 code - 128 (D3)
    fft_normalised: bool = False             # D4
    rescale_mode: int = 0                    # 0 digifil -c (first interval, frozen), 1 running (D8)
    digi_sigma: float = 0.0                  # D9: 0 = 6 sigma
    remove_delays: bool = False              # digifil -K: inter-channel dispersion delays at dm (or each trial) removed
    delay_ref_mhz: float = 0.0               # -K reference frequency; 0 = the plan's highest channel centre
    extra: dict = field(default_factory=dict)


class Plan:
    def __init__(self, cfg: PlanConfig):
        self.cfg = cfg
        nif = len(cfg.bw_mhz)
        p = _lib.Params()
        p.struct_size = C.sizeof(_lib.Params)
        p.device = cfg.device
        p.nif = nif
        p.nchan = cfg.nchan
        p.freq_res = cfg.freq_res
        p.tscrunch = cfg.tscrunch
        p.pol_mode = cfg.pol_mode
        p.out_nbit = cfg.out_nbit
        p.in_nbit = cfg.in_nbit
        p.frame_bytes = cfg.frame_bytes
        p.header_bytes = cfg.header_bytes
        p.frame_time_mode = cfg.frame_time_mode
        p.mask_faults = int(cfg.mask_faults)
        p.keep_bandpass = int(cfg.keep_bandpass)
        p.splice_pol_major = int(cfg.splice_pol_major)
        p.chunk_units = cfg.chunk_units
        p.rescale_interval_s = cfg.rescale_interval_s
        freq = cfg.freq_mhz if cfg.freq_mhz is not None else [1400.0 + abs(cfg.bw_mhz[0]) * i for i in range(nif)]
        order = cfg.if_order
        if order is None:  # highest sky frequency first, like base2fil's splice_list (base2fil.sh:350,367)
            order = sorted(range(nif), key=lambda i: -freq[i])
        if nif > _lib.B2F_MAX_IF:
            raise B2FError(_lib.EINVAL, "nif out of range")
        for i in range(nif):
            p.bw_mhz[i] = cfg.bw_mhz[i]
            p.freq_mhz[i] = freq[i]
            p.if_order[i] = order[i]
        p.dm = cfg.dm
        p.coherent = int(cfg.coherent)
        trials = list(cfg.dm_trials or [])
        if len(trials) > _lib.B2F_MAX_DM:
            raise B2FError(_lib.EINVAL, f"at most {_lib.B2F_MAX_DM} trial DMs")
        p.ndm = len(trials)
        for k, d in enumerate(trials):
            p.dm_trials[k] = float(d)
        p.profile = int(cfg.profile)
        p.raw_word_bits = cfg.raw_word_bits
        p.raw_format = cfg.raw_format
        if cfg.raw_word_bits:
            for i in range(nif):
                b = list(cfg.raw_bits[i])
                if len(b) == 2:                                   # 1-bit samples: (pol 0, pol 1) -> entries 0 and 2
                    b = [b[0], b[0], b[1], b[1]]
                for k in range(4):
                    p.raw_bits[i][k] = int(b[k])
        p.stream = cfg.stream
        p.decode_mode = cfg.decode_mode
        p.in8_offset_mode = cfg.in8_offset_mode
        p.fft_normalised = int(cfg.fft_normalised)
        p.rescale_mode = cfg.rescale_mode
        p.digi_sigma = cfg.digi_sigma
        p.remove_delays = int(cfg.remove_delays)
        p.delay_ref_mhz = float(cfg.delay_ref_mhz)
        self.if_order = list(order)
        self.freq_mhz = list(freq)
        self._h = C.c_void_p()
        self.nif = nif
        _lib.check(_lib.lib().b2f_plan_create(C.byref(p), C.byref(self._h)))
        g = _lib.Geometry()
        _lib.check(_lib.lib().b2f_get_geometry(self._h, C.byref(g)))
        self.geometry = g
        self.nprod = g.nprod
        self.row_bytes = g.row_bytes
        #: trial DMs of the plan (1 without trials); a row holds ndm slices of trial_row_bytes, trial-major
        self.ndm = g.ndm
        self.trial_row_bytes = g.trial_row_bytes
        self.chunk_frames = g.chunk_frames
        self.chunk_rows = g.chunk_rows
        self.tsamp_s = g.tsamp_s
        #: 2 = fused column + row kernel (L2 ring), 1 = the same as two launches, 0 = round-1 kernels
        self.path = _lib.lib().b2f_channeliser_path(self._h)

    # ------------------------------------------------------------------ lifecycle
    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().b2f_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ------------------------------------------------------------------ streaming
    def push(self, frames, nframes: int | None = None, on_device: bool = False):
        """frames: list (one per IF) of numpy uint8 arrays (host) or integer device pointers."""
        ptrs = (C.c_void_p * self.nif)()
        if on_device:
            assert nframes is not None
            for i, f in enumerate(frames):
                ptrs[i] = int(f)
        else:
            keep = []
            if self.cfg.raw_word_bits:
                frames = list(frames)[:1]
            for i, f in enumerate(frames):
                a = np.ascontiguousarray(f, dtype=np.uint8)
                keep.append(a)
                ptrs[i] = a.ctypes.data
                n = a.size // self.cfg.frame_bytes
                nframes = n if nframes is None else min(nframes, n)
            self._keep = keep   # host buffers must outlive the asynchronous copy
        _lib.check(_lib.lib().b2f_push(self._h, ptrs, int(nframes), int(on_device)))

    def flush(self):
        _lib.check(_lib.lib().b2f_flush(self._h))

    def pull(self, max_rows: int | None = None) -> np.ndarray:
        """Finished rows as a host array [rows, row_bytes] uint8 (view as needed)."""
        if max_rows is None:
            max_rows = int(self.geometry.interval_rows + 2 * self.chunk_rows)
        out = np.empty((max_rows, self.row_bytes), dtype=np.uint8)
        n = C.c_int64(0)
        _lib.check(_lib.lib().b2f_pull(self._h, out.ctypes.data, max_rows, 0, C.byref(n)))
        return out[: n.value]

    def pull_async(self, host_ptr: int, max_rows: int) -> int:
        """Queue finished rows into pinned host memory; call sync() before reading them."""
        n = C.c_int64(0)
        _lib.check(_lib.lib().b2f_pull(self._h, C.c_void_p(host_ptr), max_rows, 2, C.byref(n)))
        return n.value

    def pull_device(self, dev_ptr: int, max_rows: int) -> int:
        n = C.c_int64(0)
        _lib.check(_lib.lib().b2f_pull(self._h, C.c_void_p(dev_ptr), max_rows, 1, C.byref(n)))
        return n.value

    def pull_strided(self, dev_ptr: int, max_rows: int, row_pitch_bytes: int) -> int:
        """Rows into device (or NVLink-mapped peer) memory with a row pitch: in-GPU splice across ranks."""
        n = C.c_int64(0)
        _lib.check(_lib.lib().b2f_pull_strided(self._h, C.c_void_p(dev_ptr), max_rows, row_pitch_bytes, C.byref(n)))
        return n.value

    def sync(self):
        _lib.check(_lib.lib().b2f_sync(self._h))

    def mark(self) -> int:
        t = C.c_int64(0)
        _lib.check(_lib.lib().b2f_mark(self._h, C.byref(t)))
        return t.value

    def wait(self, ticket: int):
        _lib.check(_lib.lib().b2f_wait(self._h, int(ticket)))

    def run_scan(self, paths, out_path, *, start_s: float = 0.0, nsec: float | None = None,
                 source_name: str = "unknown", rawdatafile: str | None = None, telescope_id: int = 0,
                 machine_id: int = 0, src_raj: float = 0.0, src_dej: float = 0.0, refdm: float | None = None,
                 ring: int = 0, readers_per_file: int = 0, part: tuple[int, int] | None = None,
                 stats_only: bool = False) -> dict:
        """Files in, filterbank file out, entirely inside libb2f (b2f_run_scan): threaded readers, pinned ring,
        pipelined pushes/pulls.  `paths`: one split VDIF file per IF in plan order (or the one raw recording).
        `part=(k, n)`: only time segment k of n, written at its final offset of `out_path` (needs set_rescale
        unless keep_bandpass); `stats_only`: measure the first rescale interval, write nothing.  A plan with trial DMs
        takes a list of `ndm` output paths, one filterbank per trial with refdm = its DM."""
        io = _lib.ScanIO()
        io.struct_size = C.sizeof(_lib.ScanIO)
        io.start_s = float(start_s)
        io.nsec = -1.0 if nsec is None else float(nsec)
        io.source_name = source_name.encode()
        io.rawdatafile = None if rawdatafile is None else rawdatafile.encode()
        io.telescope_id, io.machine_id = int(telescope_id), int(machine_id)
        io.src_raj, io.src_dej = float(src_raj), float(src_dej)
        io.refdm = 0.0 if refdm is None else float(refdm)
        io.write_refdm = int(refdm is not None)
        io.ring = ring
        io.readers_per_file = readers_per_file
        io.part_index, io.part_count = part if part else (0, 0)
        io.stats_only = int(stats_only)
        if isinstance(out_path, (list, tuple)):
            if len(out_path) != self.ndm or not self.cfg.dm_trials:
                raise B2FError(_lib.EINVAL, f"a list of output paths needs a plan with {len(out_path)} trial DMs")
            tarr = (C.c_char_p * len(out_path))(*[os.fsencode(p) for p in out_path])
            io.trial_out_paths = C.cast(tarr, C.POINTER(C.c_char_p))
            out_path = None
        arr = (C.c_char_p * len(paths))(*[os.fsencode(p) for p in paths])
        res = _lib.ScanResult()
        _lib.check(_lib.lib().b2f_run_scan(self._h, len(paths), arr, None if out_path is None else os.fsencode(out_path),
                                           C.byref(io), C.byref(res)))
        return {"rows": int(res.rows), "frames_per_if": int(res.frames_per_if), "bytes_in": int(res.bytes_in),
                "bytes_out": int(res.bytes_out), "tstart_mjd": res.tstart_mjd, "seconds_of_data": res.seconds_of_data,
                "wall_s": res.wall_s, "setup_s": res.setup_s, "wait_read_s": res.wait_read_s,
                "wait_gpu_s": res.wait_gpu_s, "write_s": res.write_s, "counters": res.counters.as_dict()}

    def reset(self):
        _lib.check(_lib.lib().b2f_reset(self._h))

    # ------------------------------------------------------------------ introspection
    def counters(self) -> dict:
        c = _lib.Counters()
        _lib.check(_lib.lib().b2f_get_counters(self._h, C.byref(c)))
        return c.as_dict()

    def rescale(self):
        """mean, scale as [nif, nprod, nchan]; [ndm, nif, nprod, nchan] for a plan with trial DMs."""
        n = self.ndm * self.nif * self.nprod * self.cfg.nchan
        mean = np.empty(n, np.float32)
        scale = np.empty(n, np.float32)
        _lib.check(_lib.lib().b2f_get_rescale(self._h, mean.ctypes.data, scale.ctypes.data))
        shp = (self.nif, self.nprod, self.cfg.nchan)
        if self.cfg.dm_trials:
            shp = (self.ndm,) + shp
        return mean.reshape(shp), scale.reshape(shp)

    def set_rescale(self, mean: np.ndarray | None, scale: np.ndarray | None = None):
        """Freeze the digitiser's mean/scale (arrays as `rescale()` returns them); None returns to measuring."""
        if mean is None:
            _lib.check(_lib.lib().b2f_set_rescale(self._h, None, None))
            return
        m = np.ascontiguousarray(mean, np.float32).reshape(-1)
        s = np.ascontiguousarray(scale, np.float32).reshape(-1)
        assert m.size == s.size == self.ndm * self.nif * self.nprod * self.cfg.nchan
        _lib.check(_lib.lib().b2f_set_rescale(self._h, m.ctypes.data, s.ctypes.data))

    def delays(self) -> np.ndarray:
        """Inter-channel delays the plan removes (remove_delays), in channel samples: int64 [ndm, nif, nchan] in plan IF
        order and natural channel order (ndm = 1 without trials); zeros without remove_delays."""
        out = np.empty((self.ndm, self.nif, self.cfg.nchan), np.int64)
        _lib.check(_lib.lib().b2f_get_delays(self._h, out.ctypes.data))
        return out

    def kernel_times(self) -> dict:
        out = {}
        for k, name in enumerate(_lib.KERNEL_NAMES):
            ms = C.c_double(0)
            n = C.c_int64(0)
            _lib.check(_lib.lib().b2f_kernel_time(self._h, k, C.byref(ms), C.byref(n)))
            out[name] = (ms.value, n.value)
        return out

    def reset_timers(self):
        _lib.check(_lib.lib().b2f_reset_timers(self._h))

    def debug(self, which: int, dtype, count: int | None = None) -> np.ndarray:
        need = C.c_size_t(0)
        _lib.check(_lib.lib().b2f_debug_copy(self._h, which, None, 0, C.byref(need)))
        nbytes = need.value if count is None else min(need.value, count * np.dtype(dtype).itemsize)
        buf = np.empty(nbytes, np.uint8)
        _lib.check(_lib.lib().b2f_debug_copy(self._h, which, buf.ctypes.data, nbytes, None))
        return buf.view(dtype)

    def trial_rows(self, raw: np.ndarray) -> np.ndarray:
        """[rows, row_bytes] uint8 -> [ndm, rows, trial_row_bytes] view: trial k's rows as a single-DM plan writes them."""
        raw = np.ascontiguousarray(raw, np.uint8).reshape(-1, self.row_bytes)
        v = raw.reshape(raw.shape[0], self.ndm, self.trial_row_bytes)
        return v.transpose(1, 0, 2)

    def view_rows(self, raw: np.ndarray) -> np.ndarray:
        """[rows, row_bytes] uint8 -> [rows, elems] in the output sample type."""
        nb = self.cfg.out_nbit
        if nb == 8 or nb == 2:
            return raw
        if nb == 16:
            return raw.view(np.uint16)
        return raw.view(np.float32)


def fp32_peak_tflops(device: int = 0) -> float:
    v = C.c_double(0)
    _lib.check(_lib.lib().b2f_fp32_peak(device, C.byref(v)))
    return v.value


def decode(frames: np.ndarray, *, frame_bytes: int = 8032, header_bytes: int = 32, in_nbit: int = 2,
           mask_faults: bool = True, device: int = 0):
    """Stand-alone GPU decode: VDIF bytes -> x[2, nsamp] float32 and the fault counters."""
    a = np.ascontiguousarray(frames, dtype=np.uint8)
    nframes = a.size // frame_bytes
    spf = (frame_bytes - header_bytes) * 8 // (in_nbit * 2)
    out = np.empty((2, nframes * spf), np.float32)
    c = _lib.Counters()
    _lib.check(_lib.lib().b2f_decode(a.ctypes.data, nframes, frame_bytes, header_bytes, in_nbit, int(mask_faults), 0,
                                     out.ctypes.data, 0, device, C.byref(c)))
    return out, c.as_dict()
