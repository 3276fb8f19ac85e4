/* b2f.h -- C ABI of libb2f.so: B200-native baseband(VDIF) -> SIGPROC filterbank.
 *
 * This is the drop-in boundary for the one stage of pharaofranz/frb-baseband that
 * process_vdif.py hands to DSPSR `digifil` (per subband) and base2fil.sh hands to SIGPROC
 * `splice`.  The reference has no FFI for this path -- it shells out to two executables --
 * so every entry point below cites the reference call site whose work it replaces:
 *
 *   digifil argv built at      process_vdif.py:156-182   -> b2f_params fields
 *   digifil process run at     process_vdif.py:191        -> b2f_run_file, or b2f_push / b2f_pull per chunk
 *   fan-out + FIFOs + splice   base2fil.sh:404-448        -> b2f_run_scan
 *   .hdr semantics             process_vdif.py:115-139   -> freq_mhz / bw_mhz (sign = sideband)
 *   one digifil per IF         base2fil.sh:60-66          -> nif > 1 batches the IFs in one plan
 *   splice ${splice_list}      base2fil.sh:422-446        -> spliced row layout written by b2f_pull
 *   splice order               base2fil.sh:350,367        -> IF slot s of the output row holds
 *                                                            plan IF index if_order[s]
 *
 * Plain pointers and sizes only; no torch / C++ types.  All functions return 0 on success
 * or a negative B2F_E* code; b2f_last_error() gives a thread-local message.  A plan owns
 * its device memory and streams and may be used from one host thread at a time.  There is
 * no CPU fallback: without a CUDA device every compute entry point fails with B2F_ECUDA.
 */
#ifndef B2F_H
#define B2F_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2F_VERSION 100            /* 0.1.0 */
#define B2F_MAX_IF 32
#define B2F_MAX_DM 64              /* trial DMs of one coherent search plan */

struct b2f_plan;                   /* opaque: created by b2f_plan_create, owned by the library */

enum b2f_error {
    B2F_OK = 0,
    B2F_EINVAL = -1,               /* bad parameter (InputError in process_vdif.py:236) */
    B2F_ECUDA = -2,                /* CUDA runtime failure or no device (RunError, :247) */
    B2F_ENOMEM = -3,
    B2F_ESTATE = -4,               /* call sequence error */
    B2F_EUNSUPPORTED = -5          /* valid request outside what the kernels implement */
};

/* detection products: process_vdif.py:163-176 maps --pol {0,1,2,3,4} to -P0,-P1,-d1,-d3,-d4 */
enum b2f_pol_mode {
    B2F_POL_P0 = 0,                /* -P0 : |pol0|^2                       */
    B2F_POL_P1 = 1,                /* -P1 : |pol1|^2                       */
    B2F_POL_I = 2,                 /* -d1 : PP+QQ                          */
    B2F_POL_I2 = 3,                /* -d3 : (PP+QQ)^2                      */
    B2F_POL_COHERENCE = 4,         /* -d4 : PP, QQ, Re PQ*, Im PQ*         */
    B2F_POL_IQUV = 5,              /* Stokes, circular basis: I, Q=2Re RL*, U=2Im RL*, V=RR-LL */
    B2F_POL_PPQQ = 6               /* -d2 : PP, QQ                         */
};

enum b2f_frame_time_mode {
    B2F_FRAMES_POSITIONAL = 0,     /* frame k of a push is time slot k (digifil's reader) */
    B2F_FRAMES_BY_HEADER = 1       /* slot from header seconds/frame#; gaps zero-filled; frames whose time lies outside the
                                      push are dropped, so this mode is for single pushes (b2f_run_scan / b2f_run_file,
                                      which read files positionally, refuse it) */
};

/* 2-bit reconstruction levels (SURVEY.md Appendix A2 / D2).  The reference calls `digifil -2` (process_vdif.py:157,160); DSPSR's
 * 2-bit unpacker then sets the two output magnitudes per polarisation and window of 512 samples from the fraction of samples
 * between the thresholds (Jenet & Anderson 1998, excision disabled), while the north star of this build names the static VLBI
 * optimal levels.  Both are selectable; static is the default. */
enum b2f_decode_mode {
    B2F_DECODE_STATIC = 0,         /* -hi, -lo, +lo, +hi with lo = 1, hi = 3.3359 */
    B2F_DECODE_JA98 = 1            /* per window of 512 samples: lo, hi = conditional means of |x| for the observed fraction;
                                      2-bit input, FFT blocks starting on multiples of 512 samples */
};

/* what `-c` freezes (SURVEY.md D8) */
enum b2f_rescale_mode {
    B2F_RESCALE_CONSTANT = 0,      /* digifil -c: mean / sigma of the first interval, applied from sample 0, frozen */
    B2F_RESCALE_RUNNING = 1        /* without -c: every interval is scaled with its own statistics */
};

/* framing of the raw multi-BBC stream (raw_word_bits != 0) */
enum b2f_raw_format {
    B2F_RAW_VDIF = 0,              /* VDIF frames (spif2file.sh:31-77)                                                    */
    B2F_RAW_MARK5B = 1             /* Mark5B disk frames: 16-byte header (sync 0xABADDEED, frame# in second, BCD JJJSSSSS time
                                      code), 10000-byte payload (spif2file.sh:79-93,105-108).  The recipes of these modes start
                                      with swap_sign_mag: fold that into raw_bits (source bit b -> b ^ 1, spif.parse_recipe) */
};

typedef struct b2f_params {
    uint32_t struct_size;          /* = sizeof(b2f_params) */
    int32_t device;                /* CUDA device ordinal */
    int32_t nif;                   /* dual-pol IFs (subbands) processed together, 1..B2F_MAX_IF */
    int32_t nchan;                 /* channels per IF        (--nchan, digifil -F<nchan>:..)  */
    int32_t freq_res;              /* digifil -F ..:<freq_res>; 0 = reference rule
                                      512 if nchan<=128 else 2*nchan (process_vdif.py:162); with `coherent` the
                                      dedispersion kernel may lengthen it (next power of two >= 4 nfilt, up to 4096,
                                      and for nchan 8..64 on up to 2^20 / (2 nchan): 65536 at nchan 8, 8192 at
                                      nchan 64) when the smearing does not fit: b2f_geometry.freq_res is what was
                                      chosen.  An explicit freq_res above 4096 (other than nchan 4096's 8192) needs
                                      coherent dedispersion and 2 nchan freq_res <= 2^20 */
    int32_t tscrunch;              /* digifil -t             (--tscrunch)                     */
    int32_t pol_mode;              /* enum b2f_pol_mode                                       */
    int32_t out_nbit;              /* digifil -b: 2, 8, 16, -32 (process_vdif.py:153)         */
    int32_t in_nbit;               /* VDIF bits/sample: 1, 2 or 8 (frb.conf nbits; digifil reads it from the header) */
    int32_t frame_bytes;           /* VDIF frame size incl. header (base2fil.sh:130-136)      */
    int32_t header_bytes;          /* 32, or 16 for legacy (base2fil.sh:137-147)              */
    int32_t frame_time_mode;       /* enum b2f_frame_time_mode                                */
    int32_t mask_faults;           /* 1: invalid-bit frames and 0x11223344 words -> 0.0       */
    int32_t keep_bandpass;         /* digifil -I0            (--keepBP)                       */
    int32_t splice_pol_major;      /* 0: row = per-IF [pol][chan] tiles back to back (splice);
                                      1: row = [pol][all channels]                            */
    int32_t chunk_units;           /* frames per push = chunk_units * unit (see b2f_geometry)  */
    double rescale_interval_s;     /* digifil -I (default 10 s), stats frozen after (-c)      */
    double bw_mhz[B2F_MAX_IF];     /* signed: <0 = LSB (process_vdif.py:117-118)              */
    double freq_mhz[B2F_MAX_IF];   /* centre frequency of each IF (-f)                        */
    int32_t if_order[B2F_MAX_IF];  /* output tile s <- IF index if_order[s]; descending sky
                                      frequency for base2fil's plan                           */
    double dm;                     /* digifil -D dm (process_vdif.py:177-178)                 */
    int32_t coherent;              /* digifil -F nchan:D: in-channel coherent dedispersion by overlap-save (:179-180);
                                      nchan <= 2048, smearing up to what 4096 points hold, or for nchan 8..64 up to
                                      what 2^20 / (2 nchan) points hold */
    int32_t profile;               /* 1: time every kernel launch with CUDA events            */
    void* stream;                  /* cudaStream_t to launch on; NULL = plan-owned stream     */
    int32_t raw_word_bits;         /* 0: frames[i] is the split 2-channel VDIF stream of IF i (what jive5ab's
                                      spif2file writes, spif2file.sh:178-186).  16/32/64: frames[0] is ONE raw
                                      multi-BBC VDIF stream whose raw_word_bits-bit words each hold one time
                                      sample of every BBC channel; the corner turn is done on the GPU          */
    uint8_t raw_bits[B2F_MAX_IF][4]; /* spif2file recipe (spif2file.sh:31-98): source bit of output bits 0..3
                                      (pol0 lsb, pol0 msb, pol1 lsb, pol1 msb) of IF i                        */
    /* ---- knobs for what cannot be pinned without a running digifil (SURVEY.md Appendix D); 0 = this build's default */
    int32_t decode_mode;           /* enum b2f_decode_mode; SURVEY D2                                           */
    int32_t in8_offset_mode;       /* 8-bit VDIF samples, SURVEY D3: 0 = code - 127.5, 1 = code - 128           */
    int32_t fft_normalised;        /* D4: 1 = detected power divided by M * freq_res (squared for -d3), i.e. the
                                      transforms normalised; only visible with keep_bandpass (cancels under -c)  */
    int32_t rescale_mode;          /* enum b2f_rescale_mode; SURVEY D8                                          */
    double digi_sigma;             /* D9: half the output range spans this many sigma (digifil: 6); 0 = 6       */
    int32_t raw_format;            /* enum b2f_raw_format; only read when raw_word_bits != 0                    */
    int32_t reserved0;             /* must be 0                                                                 */
    /* ---- coherent dedispersion at several trial DMs in one pass: the spectrum of every overlap-save block is computed once
       and each trial applies its own chirp to it, so one plan writes ndm filterbanks.  Needs coherent = 1 and dm = 0;
       trials finite, >= 0, strictly increasing, the largest > 0.  freq_res, nfilt and the push size follow the largest
       trial by the single-DM rule, and its refusals apply (smearing beyond 4096 points, or beyond 2^20 / (2 nchan) points
       for nchan 8..64; nchan 4096). */
    int32_t ndm;                   /* 0: one DM, taken from dm; 1..B2F_MAX_DM: trial DMs dm_trials[0..ndm-1]          */
    double dm_trials[B2F_MAX_DM];
    /* ---- digifil -K: remove the inter-channel dispersion delays after detection (DSPSR's SampleDelay; recalled, not pinned).
       Channel c of IF i, sky centre f_c = freq_mhz[i] - bw/2 + (c + 1/2) bw/nchan (bw signed), is delayed by
       d_c = llround(DM (1/2.41e-4 s MHz^2) (f_c^-2 - f_ref^-2) / tsamp0) channel samples, tsamp0 = nchan/|bw| us, at the DM of
       dm (with or without coherent dedispersion) or of each trial.  Output row r sums channel samples r D + k + d_c, k < D
       (D = tscrunch): rows are aligned to the arrival time at f_ref, the rescale statistics come from the delayed rows, and a
       scan of K0 channel samples yields floor((K0 - d_max) / D) rows (the tail is dropped; d_max over every IF and trial).
       All delays 0 (DM 0) runs exactly as remove_delays = 0.  Otherwise the plan holds about d_max + two pushes of channel
       samples per (trial, IF): d_max |bw| 4 B nprod nif ndm and more (B2F_ENOMEM names the bytes when that does not fit). */
    int32_t remove_delays;         /* 0 or 1                                                                         */
    double delay_ref_mhz;          /* f_ref; 0 = centre of the plan's highest channel (the fch1 b2f_run_scan writes); else
                                      finite and >= that centre.  A plan holding some IFs of a wider band (one rank of an
                                      IF-sharded scan) passes the band's fch1 so that all ranks align to one frequency   */
} b2f_params;

typedef struct b2f_geometry {
    int64_t unit_frames;           /* frames per IF that hold a whole number of FFT blocks    */
    int64_t unit_blocks;           /* FFT blocks per unit                                     */
    int64_t chunk_frames;          /* frames per IF expected by b2f_push                      */
    int64_t chunk_rows;            /* output time samples produced per full push              */
    int64_t block_samples;         /* M = 2*nchan*freq_res time samples                       */
    int64_t samples_per_frame;
    int64_t row_bytes;             /* bytes of one output time sample (all trials, IFs, products) = ndm * trial_row_bytes */
    int32_t nprod;                 /* detected streams (SIGPROC nifs)                         */
    int32_t freq_res;
    double tsamp_s;
    int64_t interval_rows;         /* rows held before the first rescale is frozen            */
    int32_t nfilt_pos, nfilt_neg;  /* overlap-save samples discarded per block and channel (dedispersion) */
    int32_t ndm;                   /* trial DMs; 1 when trials are off                        */
    int64_t trial_row_bytes;       /* bytes of one trial's slice of a row: trial k starts at k * trial_row_bytes and holds
                                      exactly the row a single-DM plan at dm_trials[k] writes (either splice layout)      */
} b2f_geometry;

typedef struct b2f_counters {
    uint64_t frames_ok, frames_invalid, frames_with_fill, fill_words;
    uint64_t frames_dropped, frames_misplaced, frames_badhdr, slots_missing;
    uint64_t rows_produced, rows_emitted, blocks_dirty;
    uint64_t kernel_launches;     /* kernels this plan has launched since it was created */
    uint64_t rescale_frozen;      /* 1 once mean/scale are fixed for this scan (measured, preset, or keep_bandpass) */
    uint64_t rescale_preset;      /* 1 while b2f_set_rescale values are in force */
} b2f_counters;

/* kernel ids for b2f_kernel_time */
enum b2f_kernel_id {
    B2F_K_VALIDATE = 0,            /* frame header validation + fill masking + de-framing     */
    B2F_K_COLUMN = 1,              /* decode + column pass of the channeliser                 */
    B2F_K_EPS = 2,                 /* block-constant correction                               */
    B2F_K_ROW = 3,                 /* row pass + detection + time integration                 */
    B2F_K_STATS = 4,               /* per-channel mean / sigma                                */
    B2F_K_QUANT = 5,               /* rescale + requantise + sideband flip + splice           */
    B2F_K_DECODE = 6,              /* stand-alone decode (tests / roofline)                   */
    B2F_K_DEDISP = 7,              /* un-mix + chirp + backward FFT + overlap discard + detect */
    B2F_K_FUSED = 8,               /* decode + column pass + row pass + detection in one persistent kernel */
    B2F_K_TSUM = 9,                /* sum of partial rows when tscrunch spans the rows of several warps; with remove_delays
                                      the delay + integration kernel kd_delay_sum                                     */
    B2F_K_COUNT = 10
};

int b2f_version(void);
const char* b2f_last_error(void);
int b2f_device_count(void);

int b2f_plan_create(const b2f_params* params, struct b2f_plan** plan);
int b2f_plan_destroy(struct b2f_plan* plan);
int b2f_get_geometry(const struct b2f_plan* plan, b2f_geometry* out);

/* Feed one chunk: frames[i] -> nframes VDIF frames of IF i, on the host (pinned memory makes
 * the copy asynchronous) or already on the device.  Asynchronous: returns once the work is
 * queued.  nframes must be chunk_frames except for the final push of a scan. */
int b2f_push(struct b2f_plan* plan, const void* const* frames, int64_t nframes, int on_device);

/* End of scan: freeze the rescale even if fewer than interval_rows rows were seen. */
int b2f_flush(struct b2f_plan* plan);

/* Write finished, requantised, band-ordered rows to out.  out_on_device: 0 = host memory,
 * returns when the rows are there; 1 = device memory, queued on the plan's stream; 2 = pinned
 * host memory, queued on the plan's copy-out stream -- call b2f_sync before reading.  Returns
 * through *nrows how many rows were (or will be) written: 0 while the first rescale interval
 * is still filling. */
int b2f_pull(struct b2f_plan* plan, void* out, int64_t max_rows, int out_on_device, int64_t* nrows);

/* Like b2f_pull with out_on_device = 1, but consecutive rows are row_pitch_bytes apart: a rank that
 * owns part of the band drops its tile into the wider spliced rows of the rank that owns the file --
 * `out` may be that rank's memory mapped over NVLink (the in-GPU form of base2fil.sh:422's splice). */
int b2f_pull_strided(struct b2f_plan* plan, void* out, int64_t max_rows, int64_t row_pitch_bytes, int64_t* nrows);
/* (B2F_EUNSUPPORTED for a plan with trial DMs) */

int b2f_sync(struct b2f_plan* plan);
int b2f_reset(struct b2f_plan* plan);        /* new scan, same parameters */
int b2f_get_counters(struct b2f_plan* plan, b2f_counters* out);
/* mean/scale the digitiser applies: arrays of ndm*nif*nprod*nchan floats (ndm = 1 without trials), trial-major,
 * natural channel order */
int b2f_get_rescale(struct b2f_plan* plan, float* mean, float* scale);
/* Freeze the digitiser's mean/scale from outside instead of measuring them on the first rescale interval: a scan
 * cut into time segments (several GPUs, or several calls) must requantise every segment with the statistics of the
 * scan's first interval, which is what digifil -c does (process_vdif.py:181-182).  Arrays as b2f_get_rescale
 * returns them.  Stays in force across b2f_reset; NULL, NULL returns to measuring. */
int b2f_set_rescale(struct b2f_plan* plan, const float* mean, const float* scale);
/* accumulated device time (ms) and launch count of one kernel kind since the last reset of
 * the timers; requires params.profile = 1 */
int b2f_kernel_time(struct b2f_plan* plan, int kernel_id, double* ms, int64_t* launches);
int b2f_reset_timers(struct b2f_plan* plan);

/* Ordering points for callers that pipeline pushes and pulls without b2f_sync: b2f_mark returns a ticket for
 * "everything queued on this plan so far" (host->device copies, kernels, device->host copies); b2f_wait blocks
 * until that point has been reached.  After waiting on a ticket taken after push k / pull k, the host buffers
 * given to push k may be overwritten and the rows of pull k (mode 2) may be read.  At most 8 tickets may be
 * outstanding. */
int b2f_mark(struct b2f_plan* plan, int64_t* ticket);
int b2f_wait(struct b2f_plan* plan, int64_t ticket);

/* Which channeliser kernels the plan runs: 2 = fused column + row kernel with the block intermediate kept in an
 * L2-resident ring (2-bit split streams, frames in order, freq_res 512, no dedispersion); 1 = the same kernels as
 * two launches over a full intermediate; 0 = the round-1 kernels (everything else).  B2F_PATH=legacy|split|fused in
 * the environment overrides the choice where the fused kernel applies. */
int b2f_channeliser_path(const struct b2f_plan* plan);

/* The parameters the plan was created with (freq_res resolved to its effective value). */
int b2f_get_params(const struct b2f_plan* plan, b2f_params* out);

/* The inter-channel delays the plan removes (remove_delays), in channel samples: ndm * nif * nchan values (ndm = 1 without
 * trials), trial-major, plan IF order, natural channel order; all 0 without remove_delays. */
int b2f_get_delays(const struct b2f_plan* plan, int64_t* out);

/* ---- file level: what one `digifil` process per IF plus `splice` do with files ------------------------------- */

/* SIGPROC filterbank header as digifil writes it at the top of every .fil (process_vdif.py:143-145) and splice
 * re-emits with nchans summed (base2fil.sh:422); the fields dm_utils.py:108-125 reads back are source_name and
 * nchans. */
typedef struct b2f_fil_header {
    uint32_t struct_size;
    const char* source_name;       /* SOURCE of the .hdr (process_vdif.py:125); NULL = "unknown" */
    const char* rawdatafile;
    int32_t telescope_id, machine_id;
    double src_raj, src_dej;       /* hhmmss.s / ddmmss.s */
    double tstart_mjd, tsamp_s;
    int32_t nbits;                 /* 2, 8, 16 or 32 (float) */
    double fch1_mhz, foff_mhz;     /* centre of the first channel; foff < 0: descending frequency */
    int32_t nchans, nifs;
    double refdm;
    int32_t write_refdm;
} b2f_fil_header;

/* Serialise the header; buf may be NULL to query the size. Pure host code. */
int b2f_sigproc_header(const b2f_fil_header* h, void* buf, size_t cap, size_t* nbytes);

typedef struct b2f_scan_io {
    uint32_t struct_size;          /* = sizeof(b2f_scan_io) */
    double start_s;                /* digifil -S: seconds skipped at the head of every input (process_vdif.py:157-161) */
    double nsec;                   /* digifil -T: seconds processed; <= 0: to the end of the shortest input */
    const char* source_name;       /* SIGPROC header fields, see b2f_fil_header */
    const char* rawdatafile;       /* NULL = basename of the last input path */
    int32_t telescope_id, machine_id;
    double src_raj, src_dej;
    double refdm;
    int32_t write_refdm;
    int32_t ring;                  /* pinned input chunks in flight, 2..6; 0 = 3 */
    int32_t readers_per_file;      /* reader threads per input, 1..8; 0 = as many as the host cores allow, up to 4 */
    int32_t part_index, part_count; /* time segment part_index of part_count (0, 0 or 0, 1 = the whole window): the
                                      window is cut on boundaries where frames, FFT blocks and output samples
                                      coincide; every part writes its rows at their final offset of the same
                                      out_path (regular file, not truncated; part 0 also writes the header), so
                                      parts may run concurrently on different GPUs.  Unless keep_bandpass is set
                                      the plan needs b2f_set_rescale first (statistics of the scan's first interval) */
    int32_t stats_only;            /* 1: stop as soon as the first rescale interval is measured, write nothing
                                      (out_path may be NULL); read the result with b2f_get_rescale */
    const char* const* trial_out_paths; /* plan with trial DMs: one regular file per trial (out_path must be NULL), each
                                      with its own header (refdm = dm_trials[k]) and that trial's slice of every row.
                                      FIFOs are refused (B2F_EINVAL: a reader of one of ndm pipes written in lockstep
                                      can deadlock), and so are parts (B2F_EUNSUPPORTED) */
} b2f_scan_io;

typedef struct b2f_scan_result {
    int64_t frames_per_if, rows, bytes_in, bytes_out;
    double tstart_mjd, seconds_of_data, wall_s;
    double setup_s, wait_read_s, wait_gpu_s, write_s;   /* where the calling thread spent wall_s */
    b2f_counters counters;
} b2f_scan_result;

/* All subbands of a scan -> one band-ordered filterbank file: vdif_paths[i] is the split file of plan IF i
 * (base2fil.sh:336,353), or the single raw recording when the plan does the corner turn (raw_word_bits != 0).
 * Replaces base2fil.sh:404-448 (run_process_vdif per IF, FIFOs, splice).  out_path may be an existing FIFO: it
 * is then opened for writing as it is (process_vdif.py:146-149, INSTALL.md:32-35).  One reader thread per input
 * fills a ring of pinned chunks while the calling thread feeds the GPU and writes finished rows.  io and result
 * may be NULL.  The plan is reset first, so one plan serves consecutive scans. */
int b2f_run_scan(struct b2f_plan* plan, int nfiles, const char* const* vdif_paths, const char* out_path,
                 const b2f_scan_io* io, b2f_scan_result* result);
/* b2f_run_scan keeps its pinned host buffers in a process-wide cache for the next scan; this frees the idle ones. */
int b2f_release_host_cache(void);
/* One subband -> its own filterbank: the `digifil` child process of process_vdif.py:191 (plan with nif = 1). */
int b2f_run_file(struct b2f_plan* plan, const char* vdif_path, const char* fil_path, const b2f_scan_io* io,
                 b2f_scan_result* result);

/* Stand-alone decode of VDIF frames (host or device) -> planar float samples
 * out[2][nframes*samples_per_frame] on the device or host (kernel 1 of the path without the
 * channeliser; bit-exact contract).  counters may be NULL. */
int b2f_decode(const void* frames, int64_t nframes, int frame_bytes, int header_bytes, int in_nbit,
               int mask_faults, int in_on_device, float* out, int out_on_device, int device,
               b2f_counters* counters);

/* Measured FP32 FMA throughput of the device in TFLOP/s (roofline denominator for the
 * channeliser; the reference path is FP32 FFTW inside digifil, process_vdif.py:157-161). */
int b2f_fp32_peak(int device, double* tflops);

/* Test hooks: copy an internal device buffer of the most recent push to the host.
 * which: 0 compact payload, 1 word mask, 2 frame status, 3 block dirty flags,
 *        4 column-pass output [blk][L][R] float2 (paths 1, 2: slots of [32][R/2][16][2] float2; path 2: only the ring),
 *        5 column sums [blk][R] float2,
 *        6 eps [blk][nchan] float2, 7 detected floats of held rows [trial][if][row][prod][chan]. */
int b2f_debug_copy(struct b2f_plan* plan, int which, void* dst, size_t nbytes, size_t* needed);

#ifdef __cplusplus
}
#endif
#endif /* B2F_H */
