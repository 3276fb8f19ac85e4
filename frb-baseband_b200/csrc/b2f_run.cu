// b2f_run.cu -- file-level runner above the streaming ABI: split VDIF files in, one SIGPROC filterbank out.
//
// This is the work of one `digifil ... -o <fifo> <hdr>` child per IF (/root/reference/process_vdif.py:157-191)
// plus `splice ${splice_list} > IFall.fil` (/root/reference/base2fil.sh:420-448) as a single native call:
// reader threads fill a ring of pinned chunks (one thread per input file), the caller's thread feeds the GPU
// plan and writes finished rows; nothing waits for the GPU except to recycle a ring slot.  Only the public ABI
// of include/b2f.h is used for the device side.
#include <cuda_runtime.h>
#include <fcntl.h>
#include <pthread.h>
#include <signal.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "../../include/b2f.h"

int b2f_internal_fail(int code, const char* msg);

namespace {

int failf(int code, const std::string& s) { return b2f_internal_fail(code, s.c_str()); }

// ---- VDIF header facts needed on the host (VDIF 1.1 words 0..3)
struct FrameHead {
    uint32_t seconds, frame_nr, epoch, frame_bytes, nbit, nchan, legacy;
};

FrameHead parse_head(const uint8_t* b) {
    uint32_t w[4];
    memcpy(w, b, 16);
    FrameHead h;
    h.seconds = w[0] & 0x3FFFFFFFu;
    h.legacy = (w[0] >> 30) & 1u;
    h.frame_nr = w[1] & 0xFFFFFFu;
    h.epoch = (w[1] >> 24) & 0x3Fu;
    h.frame_bytes = (w[2] & 0xFFFFFFu) * 8u;
    h.nchan = 1u << ((w[2] >> 24) & 0x1Fu);
    h.nbit = ((w[3] >> 26) & 0x1Fu) + 1u;
    return h;
}

// Mark5B disk frame header: sync word, frame number within the second (bits 0..14 of word 1), BCD time code
// JJJSSSSS (MJD mod 1000, second of day).  The thousands of the MJD are not recorded: the latest day that is not in the
// future is taken, as jive5ab does with the system clock.
bool mark5b_head(const uint8_t* b, double fps, double* tstart) {
    uint32_t w[4];
    memcpy(w, b, 16);
    if (w[0] != 0xABADDEEDu) return false;
    uint32_t sss = 0, jjj = 0;
    for (int d = 4; d >= 0; --d) sss = sss * 10 + ((w[2] >> (4 * d)) & 15u);
    for (int d = 7; d >= 5; --d) jjj = jjj * 10 + ((w[2] >> (4 * d)) & 15u);
    const int64_t mjd_now = 40587 + (int64_t)(time(nullptr) / 86400);
    int64_t mjd = (int64_t)jjj + (mjd_now - (int64_t)jjj) / 1000 * 1000;
    if (tstart) *tstart = (double)mjd + ((double)sss + (double)(w[1] & 0x7FFFu) / fps) / 86400.0;
    return true;
}

// MJD of 00:00 UTC on the first day of a VDIF reference epoch (six-month steps from 2000-01-01)
int64_t epoch_mjd(uint32_t epoch) {
    const int64_t year = 2000 + epoch / 2, month = (epoch & 1) ? 7 : 1;
    const int64_t a = (14 - month) / 12, y = year + 4800 - a, m = month + 12 * a - 3;
    const int64_t jdn = 1 + (153 * m + 2) / 5 + 365 * y + y / 4 - y / 100 + y / 400 - 32045;
    return jdn - 2400001;
}

// ---- SIGPROC header (keyword strings with a 32-bit length in front; SURVEY.md Appendix B2)
struct HeaderWriter {
    std::vector<uint8_t> b;
    void str(const char* s) {
        const int32_t n = (int32_t)strlen(s);
        raw(&n, 4);
        raw(s, (size_t)n);
    }
    void raw(const void* p, size_t n) {
        const uint8_t* q = static_cast<const uint8_t*>(p);
        b.insert(b.end(), q, q + n);
    }
    void i32(const char* k, int32_t v) { str(k); raw(&v, 4); }
    void f64(const char* k, double v) { str(k); raw(&v, 8); }
    void text(const char* k, const char* v) { str(k); str(v); }
};

struct Ring {
    std::mutex mu;
    std::condition_variable cv;
    std::vector<int64_t> filled;      // per input file: chunks read so far
    std::vector<int64_t> got_frames;  // [chunk % ring][file] frames actually read
    int64_t released = 0;             // chunks whose slot may be overwritten
    bool abort = false;
    std::string err;
};

bool read_fully(int fd, uint8_t* dst, size_t n, off_t off, size_t* got) {
    size_t done = 0;
    while (done < n) {
        const ssize_t r = pread(fd, dst + done, n - done, off + (off_t)done);
        if (r < 0) return false;
        if (r == 0) break;
        done += (size_t)r;
    }
    *got = done;
    return true;
}

bool write_fully(int fd, const uint8_t* src, size_t n, off_t pos = -1) {      // pos >= 0: at that file offset
    size_t done = 0;
    while (done < n) {
        const ssize_t r = pos >= 0 ? pwrite(fd, src + done, n - done, pos + (off_t)done) : write(fd, src + done, n - done);
        if (r < 0) return false;
        done += (size_t)r;
    }
    return true;
}

// Pinned blocks are expensive to make (about 1 GB/s) and a process that runs many scans wants the same sizes
// again: finished scans hand their blocks back to this cache; b2f_release_host_cache() frees the idle ones.
struct PinnedPool {
    struct Block { void* p; size_t n; bool busy; };
    std::mutex mu;
    std::vector<Block> blocks;
    void* acquire(size_t n) {
        {
            std::lock_guard<std::mutex> lk(mu);
            for (auto& b : blocks)
                if (!b.busy && b.n >= n && b.n <= n + n / 2) { b.busy = true; return b.p; }
        }
        void* p = nullptr;
        if (cudaHostAlloc(&p, n, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        std::lock_guard<std::mutex> lk(mu);
        blocks.push_back({p, n, true});
        return p;
    }
    void release(void* p) {
        std::lock_guard<std::mutex> lk(mu);
        for (auto& b : blocks) if (b.p == p) b.busy = false;
    }
    void trim() {
        std::lock_guard<std::mutex> lk(mu);
        std::vector<Block> keep;
        for (auto& b : blocks) {
            if (b.busy) keep.push_back(b);
            else cudaFreeHost(b.p);
        }
        blocks.swap(keep);
    }
};
PinnedPool g_pool;

// A reader that closes base2fil's FIFO early must surface as an error (EPIPE), not kill the caller: SIGPIPE is
// blocked for the duration of a run (threads started meanwhile inherit the mask) and a pending one is consumed
// before the caller's mask is restored.
struct SigpipeGuard {
    sigset_t old{};
    bool active = false;
    SigpipeGuard() {
        sigset_t s;
        sigemptyset(&s);
        sigaddset(&s, SIGPIPE);
        active = pthread_sigmask(SIG_BLOCK, &s, &old) == 0;
    }
    ~SigpipeGuard() {
        if (!active) return;
        sigset_t s;
        sigemptyset(&s);
        sigaddset(&s, SIGPIPE);
        const timespec zero{0, 0};
        while (sigtimedwait(&s, nullptr, &zero) > 0) {}
        pthread_sigmask(SIG_SETMASK, &old, nullptr);
    }
};

struct Closer {
    std::vector<int> fds;
    std::vector<void*> pinned;
    ~Closer() {
        for (int f : fds) if (f >= 0) close(f);
        for (void* p : pinned) if (p) g_pool.release(p);
    }
};

// Finished rows go to the file on their own thread, in the order they were queued.
struct Writer {
    std::mutex mu;
    std::condition_variable cv;
    std::vector<std::pair<int, size_t>> q;      // (buffer index, bytes), FIFO
    std::vector<int> free_bufs;
    bool done = false, failed = false;
    std::string err;
};

}  // namespace

extern "C" int b2f_release_host_cache(void) {
    g_pool.trim();
    return 0;
}

extern "C" int b2f_sigproc_header(const b2f_fil_header* h, void* buf, size_t cap, size_t* nbytes) {
    if (!h || !nbytes) return failf(B2F_EINVAL, "null argument");
    if (h->struct_size != sizeof(b2f_fil_header)) return failf(B2F_EINVAL, "b2f_fil_header.struct_size mismatch");
    HeaderWriter w;
    w.str("HEADER_START");
    w.i32("telescope_id", h->telescope_id);
    w.i32("machine_id", h->machine_id);
    w.i32("data_type", 1);
    w.text("rawdatafile", h->rawdatafile ? h->rawdatafile : "");
    w.text("source_name", h->source_name ? h->source_name : "unknown");
    w.i32("barycentric", 0);
    w.i32("pulsarcentric", 0);
    w.f64("az_start", 0.0);
    w.f64("za_start", 0.0);
    w.f64("src_raj", h->src_raj);
    w.f64("src_dej", h->src_dej);
    w.f64("tstart", h->tstart_mjd);
    w.f64("tsamp", h->tsamp_s);
    w.i32("nbits", h->nbits);
    w.f64("fch1", h->fch1_mhz);
    w.f64("foff", h->foff_mhz);
    w.i32("nchans", h->nchans);
    w.i32("nifs", h->nifs);
    if (h->write_refdm) w.f64("refdm", h->refdm);
    w.str("HEADER_END");
    *nbytes = w.b.size();
    if (buf) {
        if (cap < w.b.size()) return failf(B2F_EINVAL, "header buffer too small");
        memcpy(buf, w.b.data(), w.b.size());
    }
    return 0;
}

extern "C" int b2f_run_scan(b2f_plan* pl, int nfiles, const char* const* vdif_paths, const char* out_path,
                            const b2f_scan_io* io_in, b2f_scan_result* res) {
    if (!pl || !vdif_paths) return failf(B2F_EINVAL, "null argument");
    b2f_scan_io io{};
    if (io_in) {
        if (io_in->struct_size != sizeof(b2f_scan_io)) return failf(B2F_EINVAL, "b2f_scan_io.struct_size mismatch");
        io = *io_in;
    }
    const bool stats_only = io.stats_only != 0;
    const bool in_parts = io.part_count > 1;
    if (in_parts && (io.part_index < 0 || io.part_index >= io.part_count)) return failf(B2F_EINVAL, "part_index out of range");
    if (in_parts && stats_only) return failf(B2F_EINVAL, "stats_only measures the head of the whole window: do not combine it with parts");
    b2f_params prm;
    b2f_geometry g;
    int rc = b2f_get_params(pl, &prm);
    if (rc) return rc;
    rc = b2f_get_geometry(pl, &g);
    if (rc) return rc;
    // trial DMs: one file per trial, each with that trial's slice of every row
    const bool trials = prm.ndm > 0;
    if (trials) {
        if (out_path) return failf(B2F_EINVAL, "a plan with trial DMs writes trial_out_paths: out_path must be NULL");
        if (in_parts) return failf(B2F_EUNSUPPORTED, "a scan with trial DMs cannot be processed in parts");
        if (!stats_only) {
            if (!io.trial_out_paths) return failf(B2F_EINVAL, "a plan with trial DMs needs trial_out_paths (one file per trial)");
            for (int k = 0; k < prm.ndm; ++k)
                if (!io.trial_out_paths[k]) return failf(B2F_EINVAL, "null trial output path");
        }
    } else {
        if (io.trial_out_paths) return failf(B2F_EINVAL, "trial_out_paths needs a plan with trial DMs");
        if (!out_path && !stats_only) return failf(B2F_EINVAL, "null output path");
    }
    const int nout = trials ? prm.ndm : 1;
    auto path_of = [&](int k) { return trials ? io.trial_out_paths[k] : out_path; };
    // Placement by header time works inside one push: a frame whose header time lies beyond the push is dropped and
    // never presented again, while this runner reads files positionally chunk by chunk -- after a gap every later
    // chunk would lose its last frames.  Whole files are digifil's positional reader (process_vdif.py:157-161).
    if (prm.frame_time_mode == B2F_FRAMES_BY_HEADER)
        return failf(B2F_EUNSUPPORTED, "b2f_run_scan reads frames positionally: frame_time_mode = B2F_FRAMES_BY_HEADER is single-push only (b2f_push)");
    const int nstreams = prm.raw_word_bits ? 1 : prm.nif;
    if (nfiles != nstreams)
        return failf(B2F_EINVAL, "the plan expects " + std::to_string(nstreams) + " input file(s), got " + std::to_string(nfiles));
    const auto t_begin = std::chrono::steady_clock::now();
    const size_t fb = (size_t)prm.frame_bytes;
    const double fps_d = 2.0 * std::fabs(prm.bw_mhz[0]) * 1e6 / (double)g.samples_per_frame;
    const int64_t fps = llround(fps_d);
    if (std::fabs(fps_d - (double)fps) > 1e-6)
        return failf(B2F_EINVAL, "frames per second is not an integer for this bandwidth and frame size");

    SigpipeGuard no_sigpipe;
    Closer own;
    // ---- inputs: size, window (-S / -T), geometry check against the plan
    int64_t f0 = llround(io.start_s * (double)fps);
    int64_t nfr = INT64_MAX;
    for (int i = 0; i < nfiles; ++i) {
        const int fd = open(vdif_paths[i], O_RDONLY);
        if (fd < 0) return failf(B2F_EINVAL, std::string("cannot open ") + vdif_paths[i] + ": " + strerror(errno));
        own.fds.push_back(fd);
        struct stat st;
        if (fstat(fd, &st)) return failf(B2F_EINVAL, std::string("cannot stat ") + vdif_paths[i]);
        nfr = std::min<int64_t>(nfr, (int64_t)(st.st_size / (off_t)fb) - f0);
        uint8_t head[32];
        size_t got = 0;
        const bool mk5 = prm.raw_word_bits && prm.raw_format == B2F_RAW_MARK5B;
        if (mk5) {
            if (read_fully(fd, head, 16, 0, &got) && got == 16 && !mark5b_head(head, (double)fps, nullptr))
                return failf(B2F_EINVAL, std::string(vdif_paths[i]) + ": no Mark5B sync word at the start of the file");
        } else if (read_fully(fd, head, 32, 0, &got) && got == 32) {
            const FrameHead h = parse_head(head);
            if (h.frame_bytes != fb || (int)(h.legacy ? 16 : 32) != prm.header_bytes ||
                (!prm.raw_word_bits && (int)h.nbit != prm.in_nbit))
                return failf(B2F_EINVAL, std::string(vdif_paths[i]) + ": frame geometry differs from the plan (" +
                                             std::to_string(h.frame_bytes) + " B frames, " + std::to_string(h.nbit) + " bit)");
        }
    }
    if (io.nsec > 0) nfr = std::min<int64_t>(nfr, llround(io.nsec * (double)fps));
    nfr = std::max<int64_t>(nfr, 0);

    double tstart = 0.0;
    {
        uint8_t head[32];
        size_t got = 0;
        if (prm.raw_word_bits && prm.raw_format == B2F_RAW_MARK5B) {
            if (read_fully(own.fds[0], head, 16, (off_t)(f0 * (int64_t)fb), &got) && got == 16) mark5b_head(head, (double)fps, &tstart);
        } else if (read_fully(own.fds[0], head, 32, (off_t)(f0 * (int64_t)fb), &got) && got == 32) {
            const FrameHead h = parse_head(head);
            tstart = (double)epoch_mjd(h.epoch) + ((double)h.seconds + (double)h.frame_nr / (double)fps) / 86400.0;
        }
    }

    // ---- time segment of this call: cut where frames, FFT blocks (overlap-save steps) and output samples coincide
    int64_t row0 = 0, rows_limit = INT64_MAX;
    if (in_parts) {
        b2f_counters c0;
        rc = b2f_get_counters(pl, &c0);
        if (rc) return rc;
        if (!prm.keep_bandpass && !c0.rescale_preset)
            return failf(B2F_ESTATE, "a scan processed in parts needs the statistics of its first interval: call b2f_set_rescale first");
        const int64_t D = std::max(1, prm.tscrunch), spf = g.samples_per_frame, M = g.block_samples;
        if ((D & (D - 1)) || D > g.freq_res)
            return failf(B2F_EUNSUPPORTED, "a scan in time parts needs a power-of-two tscrunch <= freq_res (parts are cut where FFT blocks and "
                                           "output samples coincide)");
        const int64_t keep = g.freq_res - g.nfilt_pos - g.nfilt_neg, step = keep * 2 * prm.nchan;
        const int64_t T = nfr * spf, NB = T >= M ? (T - M) / step + 1 : 0;
        const int64_t gg = std::gcd(spf, step), ub = spf / gg;           // blocks between aligned boundaries
        const int64_t A = NB / ub, k = io.part_index, n = io.part_count;
        const int64_t b_lo = A * k / n * ub, b_hi = k == n - 1 ? NB : A * (k + 1) / n * ub;
        const int64_t skip = b_lo * step / spf;                           // exact: b_lo is a multiple of ub
        // remove_delays: the last own row also reads d_max channel samples further on, i.e. whole blocks beyond b_hi
        int64_t dl_max = 0;
        if (prm.remove_delays) {
            std::vector<int64_t> dl((size_t)g.ndm * prm.nif * prm.nchan);
            rc = b2f_get_delays(pl, dl.data());
            if (rc) return rc;
            for (int64_t d : dl) dl_max = std::max(dl_max, d);
        }
        const int64_t b_end = std::min(NB, b_hi + (dl_max + keep - 1) / keep);
        int64_t take = nfr - skip;
        if (k < n - 1) take = std::min(take, ((b_end - b_lo - 1) * step + M + spf - 1) / spf);   // includes the overlap halo
        if (b_hi <= b_lo) take = 0;
        f0 += skip;
        nfr = std::max<int64_t>(take, 0);
        row0 = b_lo * keep / D;
        rows_limit = (b_hi - b_lo) * keep / D;
    }

    // ---- output: an existing FIFO (base2fil.sh:348-349) is opened as it is, never unlinked (process_vdif.py:146-149)
    std::vector<int> ofds;                    // one file, or one per trial DM
    bool out_is_fifo = false;
    bool positioned = false;                  // parts write at their final offset (pwrite) into a file nobody truncates
    for (int k = 0; k < nout && !stats_only; ++k) {
        const char* op = path_of(k);
        struct stat st;
        const bool fifo = stat(op, &st) == 0 && S_ISFIFO(st.st_mode);
        if (fifo && in_parts) return failf(B2F_EINVAL, "parts of a scan cannot be written to a FIFO");
        // the trial files are written in lockstep: a reader that drains one pipe after another would deadlock the scan
        if (fifo && trials) return failf(B2F_EINVAL, std::string(op) + ": trial DM outputs must be regular files, not FIFOs");
        out_is_fifo = fifo;
        int ofd = -1;
        if (fifo) {
            ofd = open(op, O_WRONLY);
#ifdef F_SETPIPE_SZ
            // what setfifo.perl does for every FIFO of the splice list (setfifo.perl:10, base2fil.sh:417-419): 1 MiB pipe
            if (ofd >= 0) (void)fcntl(ofd, F_SETPIPE_SZ, 1048576);
#endif
        } else {
            ofd = open(op, in_parts ? (O_WRONLY | O_CREAT) : (O_WRONLY | O_CREAT | O_TRUNC), 0644);
        }
        if (ofd < 0) return failf(B2F_EINVAL, std::string("cannot open ") + op + " for writing: " + strerror(errno));
        own.fds.push_back(ofd);
        ofds.push_back(ofd);
        positioned = in_parts;
    }
    const int ofd = ofds.empty() ? -1 : ofds[0];
    int64_t bytes_out = 0;
    off_t out_pos = 0, hdr_bytes = 0;
    if (!stats_only) {
        double top = prm.freq_mhz[0];
        for (int i = 1; i < prm.nif; ++i) top = std::max(top, prm.freq_mhz[i]);
        const double abw = std::fabs(prm.bw_mhz[0]);
        std::string base = vdif_paths[nfiles - 1];
        base = base.substr(base.find_last_of('/') == std::string::npos ? 0 : base.find_last_of('/') + 1);
        b2f_fil_header fh{};
        fh.struct_size = sizeof fh;
        fh.source_name = io.source_name;
        fh.rawdatafile = io.rawdatafile ? io.rawdatafile : base.c_str();
        fh.telescope_id = io.telescope_id;
        fh.machine_id = io.machine_id;
        fh.src_raj = io.src_raj;
        fh.src_dej = io.src_dej;
        fh.tstart_mjd = tstart;
        fh.tsamp_s = g.tsamp_s;
        fh.nbits = prm.out_nbit == -32 ? 32 : prm.out_nbit;
        fh.fch1_mhz = top + abw / 2 - abw / (2.0 * prm.nchan);
        fh.foff_mhz = -abw / prm.nchan;
        fh.nchans = prm.nif * prm.nchan;
        fh.nifs = g.nprod;
        fh.refdm = io.refdm;
        fh.write_refdm = io.write_refdm;
        for (int k = 0; k < nout; ++k) {
            if (trials) {
                fh.refdm = prm.dm_trials[k];
                fh.write_refdm = 1;
            }
            uint8_t hb[1024];
            size_t hn = 0;
            rc = b2f_sigproc_header(&fh, hb, sizeof hb, &hn);
            if (rc) return rc;
            if (!positioned || io.part_index == 0) {
                if (!write_fully(ofds[k], hb, hn, positioned ? 0 : -1)) return failf(B2F_EINVAL, std::string("write failed: ") + strerror(errno));
                bytes_out += (int64_t)hn;
            }
            hdr_bytes = (off_t)hn;                                   // the same length for every trial: refdm is always written
            out_pos = (off_t)hn + (off_t)(row0 * g.row_bytes);
        }
    }

    // ---- pinned ring + output buffers
    const int ring = io.ring > 0 ? std::min(std::max(io.ring, 2), 6) : 3;   // < 2 cannot overlap reading with the GPU
    const int64_t cf = g.chunk_frames;
    const size_t file_stride = ((size_t)cf * fb + 255) / 256 * 256;
    const size_t slot_bytes = file_stride * (size_t)nfiles;
    const int64_t max_rows = std::max<int64_t>(4 * g.chunk_rows, 4096);      // rows per pull; a backlog takes several
    if (cudaSetDevice(prm.device) != cudaSuccess) return failf(B2F_ECUDA, "cudaSetDevice failed");
    std::vector<uint8_t*> slot(ring, nullptr);
    for (int s = 0; s < ring; ++s) {
        void* p = g_pool.acquire(slot_bytes);
        if (!p) return failf(B2F_ENOMEM, "cannot allocate pinned input ring");
        own.pinned.push_back(p);
        slot[s] = static_cast<uint8_t*>(p);
    }
    constexpr int kOut = 4;
    uint8_t* outb[kOut];
    for (int s = 0; s < kOut; ++s) {
        void* p = g_pool.acquire((size_t)max_rows * (size_t)g.row_bytes);
        if (!p) return failf(B2F_ENOMEM, "cannot allocate pinned output buffers");
        own.pinned.push_back(p);
        outb[s] = static_cast<uint8_t*>(p);
    }

    // ---- readers: file i, chunk k -> slot[k % ring] + i * file_stride
    const int64_t nchunks = (nfr + cf - 1) / cf;
    // Several threads per file: a page-cache read is a single-core memcpy (about 5 GB/s), far below what PCIe takes.
    const int hw = (int)std::max(1u, std::thread::hardware_concurrency());
    const int parts = io.readers_per_file > 0 ? std::min(io.readers_per_file, 8)
                                              : std::max(1, std::min(4, hw / std::max(1, nfiles)));
    const int nreaders = nfiles * parts;
    Ring R;
    R.filled.assign(nreaders, 0);
    R.got_frames.assign((size_t)ring * nreaders, 0);
    std::vector<std::thread> readers;
    for (int t = 0; t < nreaders; ++t) {
        readers.emplace_back([&, t] {
            const int i = t / parts, j = t % parts;
            for (int64_t k = 0; k < nchunks; ++k) {
                {
                    std::unique_lock<std::mutex> lk(R.mu);
                    R.cv.wait(lk, [&] { return R.abort || k < R.released + ring; });
                    if (R.abort) return;
                }
                const int64_t want = std::min<int64_t>(cf, nfr - k * cf);
                const int64_t a = want * j / parts, b = want * (j + 1) / parts;      // this thread's frames of the chunk
                size_t got = 0;
                const bool ok = read_fully(own.fds[i], slot[k % ring] + (size_t)i * file_stride + (size_t)a * fb,
                                           (size_t)(b - a) * fb, (off_t)((f0 + k * cf + a) * (int64_t)fb), &got);
                std::lock_guard<std::mutex> lk(R.mu);
                if (!ok) {
                    R.abort = true;
                    R.err = std::string("read failed on ") + vdif_paths[i] + ": " + strerror(errno);
                }
                // frames of this chunk that are contiguous from its start as far as this part knows
                R.got_frames[(size_t)(k % ring) * nreaders + t] = (int64_t)(got / fb) == b - a ? want : a + (int64_t)(got / fb);
                R.filled[t] = k + 1;
                R.cv.notify_all();
                if (!ok) return;
            }
        });
    }
    auto stop_readers = [&] {
        {
            std::lock_guard<std::mutex> lk(R.mu);
            R.abort = true;
        }
        R.cv.notify_all();
        for (auto& t : readers) if (t.joinable()) t.join();
    };

    std::vector<uint8_t> gather(trials && !stats_only ? (size_t)max_rows * (size_t)g.trial_row_bytes : 0);   // the writer's, per trial

    // ---- feed the plan; rows of chunk k are written while chunk k+1 is on the GPU
    int64_t rows_total = 0, frames_done = 0;
    double t_wait_read = 0, t_wait_gpu = 0, t_write = 0;
    auto since = [](std::chrono::steady_clock::time_point t0) {
        return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    };
    const double t_setup = since(t_begin);
    Writer W;
    for (int s = 0; s < kOut; ++s) W.free_bufs.push_back(s);
    std::thread writer([&] {
        for (;;) {
            std::pair<int, size_t> job;
            {
                std::unique_lock<std::mutex> lk(W.mu);
                W.cv.wait(lk, [&] { return W.done || !W.q.empty(); });
                if (W.q.empty()) return;
                job = W.q.front();
                W.q.erase(W.q.begin());
            }
            const auto t0 = std::chrono::steady_clock::now();
            // A regular file takes the rows of one pull as four concurrent pwrites: a single writer into the page cache
            // (or tmpfs) allocates and fills pages at about 3 GB/s, which at 100x real time is what the whole runner waits
            // for (320 MB of rows per 20 s of C2).  A FIFO is a byte stream: one writer, in order.
            bool ok = true;
            if (!W.failed && trials) {
                // each trial's slice of every row, gathered into one contiguous piece per file
                const int64_t trb = g.trial_row_bytes, nr = (int64_t)(job.second / (size_t)g.row_bytes);
                const off_t tpos = hdr_bytes + (off_t)((out_pos - hdr_bytes) / g.row_bytes * trb);   // rows written so far
                for (int k = 0; k < nout && ok; ++k) {
                    const uint8_t* src = outb[job.first] + k * trb;
                    for (int64_t r = 0; r < nr; ++r) memcpy(gather.data() + r * trb, src + r * g.row_bytes, (size_t)trb);
                    ok = write_fully(ofds[k], gather.data(), (size_t)(nr * trb), tpos);
                }
            } else if (!W.failed) {
                const uint8_t* src = outb[job.first];
                const size_t n = job.second;
                constexpr int kPar = 4;
                if (out_is_fifo || n < ((size_t)8 << 20)) {
                    ok = write_fully(ofd, src, n, out_is_fifo ? (off_t)-1 : out_pos);
                } else {
                    const size_t piece = ((n / kPar) + 4095) & ~(size_t)4095;
                    bool okp[kPar];
                    std::thread th[kPar];
                    for (int q = 0; q < kPar; ++q) {
                        const size_t a = std::min(n, (size_t)q * piece), b = std::min(n, (size_t)(q + 1) * piece);
                        okp[q] = true;
                        th[q] = std::thread([&, q, a, b] { if (b > a) okp[q] = write_fully(ofd, src + a, b - a, out_pos + (off_t)a); });
                    }
                    for (int q = 0; q < kPar; ++q) { th[q].join(); ok = ok && okp[q]; }
                }
            }
            out_pos += (off_t)job.second;
            std::lock_guard<std::mutex> lk(W.mu);
            t_write += since(t0);
            if (!ok && !W.failed) {
                W.failed = true;
                W.err = std::string("write failed: ") + strerror(errno);
            }
            W.free_bufs.push_back(job.first);
            W.cv.notify_all();
        }
    });
    auto take_buffer = [&]() -> int {
        std::unique_lock<std::mutex> lk(W.mu);
        W.cv.wait(lk, [&] { return !W.free_bufs.empty(); });
        const int b = W.free_bufs.back();
        W.free_bufs.pop_back();
        return b;
    };
    auto queue_write = [&](int buf, int64_t rows) {
        rows = std::max<int64_t>(0, std::min(rows, rows_limit - rows_total));       // a part ends at its last own row
        {
            std::lock_guard<std::mutex> lk(W.mu);
            if (rows > 0) W.q.emplace_back(buf, (size_t)rows * (size_t)g.row_bytes);
            else W.free_bufs.push_back(buf);
        }
        W.cv.notify_all();
        bytes_out += rows * g.row_bytes;
        rows_total += rows;
    };
    int64_t pend_rows[2] = {0, 0}, pend_ticket[2] = {-1, -1};
    int pend_buf[2] = {-1, -1};
    auto drain = [&](int b) -> int {        // rows queued into pend_buf[b] by the GPU -> writer
        if (pend_ticket[b] < 0) return 0;
        const auto t0 = std::chrono::steady_clock::now();
        const int r = b2f_wait(pl, pend_ticket[b]);
        t_wait_gpu += since(t0);
        pend_ticket[b] = -1;
        queue_write(pend_buf[b], r ? 0 : pend_rows[b]);
        pend_buf[b] = -1;
        pend_rows[b] = 0;
        return r;
    };
    rc = b2f_reset(pl);
    for (int64_t k = 0; rc == 0 && k < nchunks; ++k) {
        int64_t got = INT64_MAX;
        const auto tw = std::chrono::steady_clock::now();
        {
            std::unique_lock<std::mutex> lk(R.mu);
            R.cv.wait(lk, [&] {
                if (R.abort) return true;
                for (int t = 0; t < nreaders; ++t) if (R.filled[t] <= k) return false;
                return true;
            });
            if (R.abort) { rc = failf(B2F_EINVAL, R.err); break; }
            for (int t = 0; t < nreaders; ++t) got = std::min(got, R.got_frames[(size_t)(k % ring) * nreaders + t]);
        }
        t_wait_read += since(tw);
        if (got <= 0) break;
        const void* ptrs[B2F_MAX_IF];
        for (int i = 0; i < nfiles; ++i) ptrs[i] = slot[k % ring] + (size_t)i * file_stride;
        const int b = (int)(k & 1);
        rc = b2f_push(pl, ptrs, got, 0);
        if (rc) break;
        if (stats_only) {                    // measure, emit nothing; stop once the interval is complete
            int64_t n = 0;
            rc = b2f_pull(pl, nullptr, 0, 0, &n);
            if (rc) break;
            rc = b2f_sync(pl);               // the ring slot is reused right away
            if (rc) break;
            b2f_counters c;
            rc = b2f_get_counters(pl, &c);
            if (rc) break;
            frames_done += got;
            {
                std::lock_guard<std::mutex> lk(R.mu);
                R.released = k + 1;
            }
            R.cv.notify_all();
            if (c.rescale_frozen || got < std::min<int64_t>(cf, nfr - k * cf)) break;
            continue;
        }
        // while the GPU has chunk k queued: finish chunk k-1 (its copies and kernels are then behind us, so its
        // ring slot can be recycled) and write its rows, which keeps the file in time order
        rc = drain(b ^ 1);
        if (rc) break;
        for (;;) {                           // normally one pull; the first rescale interval comes out as a backlog
            int64_t n = 0;
            pend_buf[b] = take_buffer();
            rc = b2f_pull(pl, outb[pend_buf[b]], max_rows, 2, &n);
            if (rc) { queue_write(pend_buf[b], 0); pend_buf[b] = -1; break; }
            pend_rows[b] = n;
            rc = b2f_mark(pl, &pend_ticket[b]);
            if (rc || n < max_rows) break;
            rc = drain(b);
            if (rc) break;
        }
        if (rc) break;
        frames_done += got;
        {
            std::lock_guard<std::mutex> lk(R.mu);
            R.released = k;                  // chunks < k are consumed; chunk k's slot stays until the next turn
        }
        R.cv.notify_all();
        if (got < std::min<int64_t>(cf, nfr - k * cf)) break;      // short read: a file ended early
    }
    stop_readers();
    if (rc == 0) rc = drain((int)(nchunks & 1));          // older of the two pending buffers first
    if (rc == 0) rc = drain((int)(nchunks & 1) ^ 1);
    if (rc == 0) rc = b2f_flush(pl);
    if (rc == 0 && stats_only) {             // a window shorter than the interval: statistics of what there is
        int64_t n = 0;
        rc = b2f_pull(pl, nullptr, 0, 0, &n);
    }
    while (rc == 0 && !stats_only) {         // rows still held (first rescale interval, tail)
        int64_t n = 0;
        const int buf = take_buffer();
        rc = b2f_pull(pl, outb[buf], max_rows, 0, &n);
        queue_write(buf, rc ? 0 : n);
        if (rc || n == 0) break;
    }
    {
        std::lock_guard<std::mutex> lk(W.mu);
        W.done = true;
    }
    W.cv.notify_all();
    writer.join();
    if (rc == 0 && W.failed) rc = failf(B2F_EINVAL, W.err);
    if (rc) {
        b2f_sync(pl);                        // nothing may still be reading the pinned buffers when they are freed
        return rc;
    }
    rc = b2f_sync(pl);
    if (rc) return rc;
    if (res) {
        memset(res, 0, sizeof *res);
        res->frames_per_if = frames_done;
        res->rows = rows_total;
        res->bytes_in = frames_done * (int64_t)fb * nfiles;
        res->bytes_out = bytes_out;
        res->tstart_mjd = tstart;
        res->seconds_of_data = (double)frames_done / (double)fps;
        res->wall_s = since(t_begin);
        res->setup_s = t_setup;
        res->wait_read_s = t_wait_read;
        res->wait_gpu_s = t_wait_gpu;
        res->write_s = t_write;
        rc = b2f_get_counters(pl, &res->counters);
    }
    return rc;
}

extern "C" int b2f_run_file(b2f_plan* pl, const char* vdif_path, const char* fil_path, const b2f_scan_io* io,
                            b2f_scan_result* res) {
    const char* paths[1] = {vdif_path};
    if (!vdif_path) return failf(B2F_EINVAL, "null argument");
    return b2f_run_scan(pl, 1, paths, fil_path, io, res);
}
