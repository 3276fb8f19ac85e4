// libb2f.so: plan object, streaming state machine and the C ABI declared in include/b2f.h.
// Host side of the path /root/reference/process_vdif.py:142-199 (run_digifil) and
// /root/reference/base2fil.sh:404-448 (fan-out + splice) drive today with two executables.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

#define B2F_API_TU
#include "b2f_fused.cuh"
#include "b2f_generic.cuh"
#include "b2f_launch.h"
#include "b2f_long.h"

using namespace b2f;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CU(x)                                                                                   \
    do {                                                                                        \
        cudaError_t e__ = (x);                                                                  \
        if (e__ != cudaSuccess) {                                                               \
            return fail(B2F_ECUDA, std::string(#x) + ": " + cudaGetErrorString(e__));          \
        }                                                                                       \
    } while (0)

}  // namespace

int b2f_internal_fail(int code, const char* msg) { return fail(code, msg); }

namespace {

bool is_pow2(int64_t v) { return v > 0 && (v & (v - 1)) == 0; }

struct TimedLaunch {
    int kid;
    cudaEvent_t a, b;
};

}  // namespace

struct b2f_plan {
    b2f_params prm{};
    int R = 0, N = 0, L = 0, D = 0, nprod = 0, nstrips = 0, num_sms = 0;
    int64_t M = 0, spf = 0, fps = 0, payload = 0, groups_per_slot = 0;
    int64_t unit_frames = 0, unit_blocks = 0, chunk_frames = 0, chunk_blocks = 0, chunk_rows = 0;
    int64_t interval_rows = 0, F_cap_rows = 0;
    int out_elem_bits = 8;
    int64_t row_elems = 0, row_bytes = 0;
    // trial DMs (b2f_params.ndm): F, d_Fk, statistics and chirp tables hold ndm * nif slots, trial-major; 1 without trials
    int ndm = 1;
    int64_t trial_row_elems = 0;

    cudaStream_t stream = nullptr, copy_stream = nullptr, d2h_stream = nullptr;
    bool own_stream = false;
    cudaEvent_t ev_stage_free[2]{}, ev_h2d_done[2]{}, ev_out_free[2]{}, ev_kq_done[2]{};
    static constexpr int kMarks = 8;                  // b2f_mark / b2f_wait tickets in flight
    cudaEvent_t ev_mark[kMarks][3]{};
    int64_t marks_issued = 0;
    int stage_idx = 0, out_idx = 0;
    int64_t launches = 0;

    uint8_t* d_stage[2]{};
    size_t stage_if_stride = 0;
    uint8_t *d_compact = nullptr, *d_wmask = nullptr, *d_fstat = nullptr, *d_blkdirty = nullptr;
    size_t compact_stride = 0, wmask_stride = 0, fstat_stride = 0;
    int slot_bytes = 0;
    float2 *d_inter = nullptr, *d_colsum = nullptr, *d_eps = nullptr;
    float* d_F = nullptr;
    int64_t F_if_stride = 0;
    float *d_mean = nullptr, *d_scale = nullptr;
    double2* d_partial = nullptr;
    float2 *d_tab_g = nullptr, *d_tab_h = nullptr, *d_tab_w = nullptr, *d_tab_r = nullptr, *d_tab_beta = nullptr;
    unsigned long long* d_counters = nullptr;
    int64_t batch_blocks = 0;      // FFT blocks per column/row launch pair (0 = whole chunk)
    // coherent dedispersion (digifil -D dm -F nchan:D): overlap-save geometry and halo carry
    bool dedisp = false;
    bool generic = false;          // freq_res / nchan outside the tuned 512-point kernels
    bool longfft = false;          // dedispersion with freq_res 8192..65536 (b2f_kl.cu)
    // tscrunch that is not a power of two, or longer than freq_res (process_vdif.py:156-158 passes any -t): the kernels
    // integrate D = the largest power of two dividing it (<= freq_res), d_Fk holds their rows and kd_sum_rows adds tsq of them
    int tsq = 1;
    float* d_Fk = nullptr;
    int64_t Fk_if_stride = 0, fk_pending = 0;
    // digifil -K (remove_delays, some delay > 0): the row kernels integrate nothing (D = 1) and write channel samples into
    // d_Fk, a ring of dl_cap rows per (trial, IF) slot; kd_delay_sum adds Du = tscrunch of them at each channel's delay into F.
    // Logical sample j of the ring (j = 0: the first sample of the next output row) sits at row dl_off + j, minus dl_wrap
    // where that reaches dl_wrap.  A push that does not fit behind the held samples starts again at row 0 (dl_wrapped);
    // dl_cap = d_max + Du - 1 + two pushes guarantees it fits there, so nothing is ever moved.
    bool delays = false, dl_wrapped = false;
    int Du = 1;
    int64_t dl_max = 0, dl_cap = 0, dl_off = 0, dl_held = 0, dl_wrap = 0, dl_w = 0;
    std::vector<int64_t> dl_host;  // delays [trial][if][chan] (remove_delays = 1), for b2f_get_delays
    int64_t* d_delays = nullptr;
    int kgt_lg = 0;                // generic kernels with compile-time geometry (L = R = 2^kgt_lg), 0 = run-time kernels
    int kgt_cols = 0, kgt_rb = 0, kgt_col_ctas = 0, kgt_row_ctas = 0;
    bool carry_mode = false;       // pushes need not hold whole blocks: unconsumed samples are carried over
    float2 *d_tw_col = nullptr, *d_tw_row = nullptr;
    int nfilt_pos = 0, nfilt_neg = 0, keep = 0;
    int64_t step = 0;              // samples between block starts = keep * R
    int64_t carry_len = 0;         // samples of the previous push still needed (per IF)
    uint8_t* d_carry = nullptr;
    // 8-bit input in carry mode: the stream holds bps = 2 bytes per time sample and no code decodes to 0.0, so the word
    // masks travel with the samples: d_wmask is indexed by stream position (one byte per 32 stream bytes, carried part
    // in front) instead of by frame slot, and the masks of the carried samples wait in d_carry_mask.
    int bps = 1;
    bool smask = false;
    uint8_t* d_carry_mask = nullptr;
    // JA98 decode on the generic path: levels per window of 512 samples of the index-byte stream (kj_levels_stream)
    float4* d_levels_stream = nullptr;
    int64_t levels_stride = 0;
    float2* d_spec = nullptr;
    float2* d_chirp = nullptr;
    uint8_t* d_out_stage[2]{};
    size_t out_stage_bytes[2]{};
    // round-2 channeliser (b2f_fused.cuh): 0 = round-1 kernels, 1 = new kernels as two launches, 2 = fused
    int path = 0;
    uint8_t* d_tstream = nullptr;  size_t tstream_stride = 0;   // block-transposed index bytes
    int* d_fillflag = nullptr;     size_t fillflag_stride = 0;
    float* d_part = nullptr;       int64_t part_if_stride = 0;  // partial rows when tscrunch > 1024 / R
    int Dp = 0;                    // rows a warp integrates itself
    unsigned* d_fsync = nullptr;   // per-lane arrival counters + abort flag (last word)
    int f_grid = 0, f_lanes = 0, f_nslot = 3, f_lag = 2;        // fused ring: rows run 2 blocks behind the columns, 3 slots per lane
    bool f_aborted = false;
    float4* d_levels = nullptr;                                 // JA98 decode: output magnitudes per window of 512 samples
    unsigned long long* d_fprof = nullptr;                      // B2F_FUSED_PROF=1: per-warp cycle breakdown of the fused kernel

    // state
    int64_t rows_base = 0;         // rows already emitted and dropped from the front of F
    int64_t rows_off = 0;          // offset inside F of the first held row
    int64_t rows_held = 0;
    int64_t rows_produced = 0, rows_emitted = 0;
    bool stats_ready = false, flushed = false, have_base = false;
    int64_t rows_this_interval = 0;   // B2F_RESCALE_RUNNING: rows still to be emitted with the statistics in force
    bool preset_stats = false;        // rescale given by the caller (b2f_set_rescale): survives b2f_reset
    int64_t frames_pushed = 0;
    uint32_t base_sec0[B2F_MAX_IF]{}, base_fnum0[B2F_MAX_IF]{};
    int64_t last_nblk = 0, last_nframes = 0;
    unsigned long long blocks_dirty = 0;

    std::vector<TimedLaunch> pending;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool;
    double k_ms[B2F_K_COUNT]{};
    int64_t k_n[B2F_K_COUNT]{};
};

namespace {

static const int kStatSplit = 64;

// where the row kernels put their rows: straight into F, or behind the rows still waiting in the staging buffer
// (with remove_delays: channel samples into the delay ring)
inline float* row_dst(const b2f_plan* pl) { return pl->tsq > 1 || pl->delays ? pl->d_Fk : pl->d_F; }
inline int64_t row_dst_stride(const b2f_plan* pl) { return pl->tsq > 1 || pl->delays ? pl->Fk_if_stride : pl->F_if_stride; }
inline int64_t row_dst_row0(const b2f_plan* pl) {
    return pl->delays ? pl->dl_w : pl->tsq > 1 ? pl->fk_pending : pl->rows_off + pl->rows_held;
}

template <class Fn>
int timed(b2f_plan* pl, int kid, Fn&& fn) {
    pl->launches++;
    if (!pl->prm.profile) {
        fn();
        pl->k_n[kid]++;
        CU(cudaGetLastError());
        return 0;
    }
    std::pair<cudaEvent_t, cudaEvent_t> ev;
    if (!pl->ev_pool.empty()) {
        ev = pl->ev_pool.back();
        pl->ev_pool.pop_back();
    } else {
        CU(cudaEventCreate(&ev.first));
        CU(cudaEventCreate(&ev.second));
    }
    CU(cudaEventRecord(ev.first, pl->stream));
    fn();
    CU(cudaGetLastError());
    CU(cudaEventRecord(ev.second, pl->stream));
    pl->pending.push_back({kid, ev.first, ev.second});
    return 0;
}

int collect_times(b2f_plan* pl) {
    if (pl->pending.empty()) return 0;
    CU(cudaStreamSynchronize(pl->stream));
    for (auto& t : pl->pending) {
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, t.a, t.b));
        pl->k_ms[t.kid] += ms;
        pl->k_n[t.kid]++;
        pl->ev_pool.emplace_back(t.a, t.b);
    }
    pl->pending.clear();
    return 0;
}

int nprod_of(int mode) {
    switch (mode) {
        case B2F_POL_P0: case B2F_POL_P1: case B2F_POL_I: case B2F_POL_I2: return 1;
        case B2F_POL_PPQQ: return 2;
        case B2F_POL_COHERENCE: case B2F_POL_IQUV: return 4;
        default: return 0;
    }
}

int launch_kb(b2f_plan* pl, const KBParams& kp, int grid) {
    cudaError_t e = cudaSuccess;
    int rc = timed(pl, B2F_K_ROW, [&] { e = b2f_launch_kb(pl->R, pl->prm.pol_mode, kp, grid, pl->stream); });
    if (rc) return rc;
    if (e != cudaSuccess) return fail(B2F_ECUDA, std::string("row pass launch: ") + cudaGetErrorString(e));
    return 0;
}

int launch_ka(b2f_plan* pl, bool fwd_only, const KAParams& ka, unsigned grid) {
    cudaError_t e = cudaSuccess;
    int rc = timed(pl, B2F_K_COLUMN, [&] { e = b2f_launch_ka(pl->d_levels_stream ? 22 : pl->prm.in_nbit, pl->R, fwd_only, ka, grid, pl->stream); });
    if (rc) return rc;
    if (e != cudaSuccess) return fail(B2F_ECUDA, std::string("column pass launch: ") + cudaGetErrorString(e));
    return 0;
}

void kb_shape(int R, int* TR, int* PT) {
    switch (R) {
        case 16: *TR = 4; *PT = 4; break;
        case 32: *TR = 4; *PT = 8; break;
        case 64: *TR = 8; *PT = 8; break;
        case 128: *TR = 8; *PT = 16; break;
        case 256: *TR = 16; *PT = 16; break;
        default: *TR = 16; *PT = 32; break;
    }
}

int upload_tables(b2f_plan* pl) {
    const int R = pl->R;
    const double M = (double)pl->M;
    std::vector<float2> g(16 * R), h(32 * R), w(32 * 16);
    for (int q = 0; q < 16; ++q)
        for (int n1 = 0; n1 < R; ++n1) {
            const double ph = -2.0 * M_PI * (double)((int64_t)q * n1) / M;
            g[q * R + n1] = make_float2((float)cos(ph), (float)sin(ph));
        }
    for (int p = 0; p < 32; ++p)
        for (int n1 = 0; n1 < R; ++n1) {
            const double ph = -2.0 * M_PI * (double)((int64_t)16 * p * n1) / M;
            h[p * R + n1] = make_float2((float)cos(ph), (float)sin(ph));
        }
    for (int l = 0; l < 32; ++l)
        for (int q = 0; q < 16; ++q) {
            const double ph = -2.0 * M_PI * (double)(l * q) / 512.0;
            w[l * 16 + q] = make_float2((float)cos(ph), (float)sin(ph));
        }
    int TR, PT;
    kb_shape(R, &TR, &PT);
    std::vector<float2> r(PT * TR);
    for (int q = 0; q < PT; ++q)
        for (int s = 0; s < TR; ++s) {
            const double ph = -2.0 * M_PI * (double)(s * q) / (double)R;
            r[q * TR + s] = make_float2((float)cos(ph), (float)sin(ph));
        }
    std::vector<float2> beta((size_t)16 * 4 * R);
    for (int item = 0; item < 16; ++item)
        for (int k = 0; k < 4; ++k)
            for (int n1 = 0; n1 < R; ++n1) {
                const double ph = (double)(1 << k) * 2.0 * M_PI * ((double)item / 512.0 - (double)n1 / M);
                beta[((size_t)item * 4 + k) * R + n1] = make_float2((float)cos(ph), (float)sin(ph));
            }
    CU(cudaMalloc(&pl->d_tab_beta, beta.size() * sizeof(float2)));
    CU(cudaMemcpy(pl->d_tab_beta, beta.data(), beta.size() * sizeof(float2), cudaMemcpyHostToDevice));
    CU(cudaMalloc(&pl->d_tab_g, g.size() * sizeof(float2)));
    CU(cudaMalloc(&pl->d_tab_h, h.size() * sizeof(float2)));
    CU(cudaMalloc(&pl->d_tab_w, w.size() * sizeof(float2)));
    CU(cudaMalloc(&pl->d_tab_r, r.size() * sizeof(float2)));
    CU(cudaMemcpy(pl->d_tab_g, g.data(), g.size() * sizeof(float2), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(pl->d_tab_h, h.data(), h.size() * sizeof(float2), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(pl->d_tab_w, w.data(), w.size() * sizeof(float2), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(pl->d_tab_r, r.data(), r.size() * sizeof(float2), cudaMemcpyHostToDevice));
    return 0;
}

int launch_k0(b2f_plan* pl, const K0Params& kp, cudaStream_t st, bool profile_ok) {
    const bool vec = (kp.payload_bytes % 32 == 0) && (kp.frame_bytes % 16 == 0) && (kp.header_bytes % 16 == 0);
    bool aligned = true;
    const int nif = pl ? pl->prm.nif : 1;
    for (int i = 0; i < nif; ++i) aligned = aligned && ((reinterpret_cast<uintptr_t>(kp.frames[i]) & 15) == 0);
    const int stage_bytes = (kp.frame_bytes + 127) & ~127;
    int sms = pl ? pl->num_sms : 148;
    int gx = (int)std::max<int64_t>(1, std::min<int64_t>(kp.nframes, (kK0CtasPerSM * sms + nif - 1) / nif));
    dim3 grid(gx, nif);
    auto body = [&] {
        if (vec && aligned) {
            size_t smem = 128 + (size_t)kK0Stages * stage_bytes;
            cudaFuncSetAttribute(k0_validate_compact<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k0_validate_compact<true><<<grid, kK0Threads, smem, st>>>(kp);
        } else {
            size_t smem = 128 + (size_t)stage_bytes;
            cudaFuncSetAttribute(k0_validate_compact<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k0_validate_compact<false><<<grid, kK0Threads, smem, st>>>(kp);
        }
    };
    if (pl && profile_ok) return timed(pl, B2F_K_VALIDATE, body);
    body();
    CU(cudaGetLastError());
    return 0;
}

void free_plan(b2f_plan* pl) {
    if (!pl) return;
    cudaSetDevice(pl->prm.device);
    cudaDeviceSynchronize();
    for (int i = 0; i < 2; ++i) {
        if (pl->d_stage[i]) cudaFree(pl->d_stage[i]);
        if (pl->ev_stage_free[i]) cudaEventDestroy(pl->ev_stage_free[i]);
        if (pl->ev_h2d_done[i]) cudaEventDestroy(pl->ev_h2d_done[i]);
        if (pl->ev_out_free[i]) cudaEventDestroy(pl->ev_out_free[i]);
        if (pl->ev_kq_done[i]) cudaEventDestroy(pl->ev_kq_done[i]);
        if (pl->d_out_stage[i]) cudaFree(pl->d_out_stage[i]);
    }
    for (int i = 0; i < b2f_plan::kMarks; ++i)
        for (int k = 0; k < 3; ++k)
            if (pl->ev_mark[i][k]) cudaEventDestroy(pl->ev_mark[i][k]);
    void* bufs[] = {pl->d_compact, pl->d_wmask, pl->d_fstat, pl->d_blkdirty, pl->d_inter, pl->d_colsum,
                    pl->d_eps, pl->d_F, pl->d_mean, pl->d_scale, pl->d_partial, pl->d_tab_g, pl->d_tab_h,
                    pl->d_tab_w, pl->d_tab_r, pl->d_tab_beta, pl->d_counters, pl->d_carry, pl->d_spec, pl->d_chirp, pl->d_tw_col, pl->d_tw_row,
                    pl->d_tstream, pl->d_fillflag, pl->d_part, pl->d_fsync, pl->d_fprof, pl->d_levels, pl->d_carry_mask, pl->d_levels_stream,
                    pl->d_delays};
    for (void* b : bufs)
        if (b) cudaFree(b);
    if (pl->d_Fk) cudaFree(pl->d_Fk);
    for (auto& t : pl->pending) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
    for (auto& e : pl->ev_pool) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    if (pl->copy_stream) cudaStreamDestroy(pl->copy_stream);
    if (pl->d2h_stream) cudaStreamDestroy(pl->d2h_stream);
    if (pl->own_stream && pl->stream) cudaStreamDestroy(pl->stream);
    delete pl;
}

int init_state(b2f_plan* pl) {
    pl->rows_base = pl->rows_off = pl->rows_held = pl->rows_produced = pl->rows_emitted = 0;
    pl->stats_ready = pl->prm.keep_bandpass != 0 || pl->preset_stats;
    pl->flushed = false;
    pl->have_base = false;
    pl->frames_pushed = 0;
    pl->carry_len = 0;
    pl->fk_pending = 0;
    pl->dl_off = pl->dl_held = pl->dl_w = 0;
    pl->dl_wrap = pl->dl_cap;
    pl->dl_wrapped = false;
    pl->blocks_dirty = 0;
    pl->last_nblk = pl->last_nframes = 0;
    pl->rows_this_interval = 0;
    pl->f_aborted = false;
    if (pl->d_fsync) CU(cudaMemsetAsync(pl->d_fsync, 0, ((size_t)pl->f_lanes + 1) * FS_STRIDE * sizeof(unsigned), pl->stream));
    const int ncol = pl->nprod * pl->N;
    CU(cudaMemsetAsync(pl->d_counters, 0, C_COUNT * sizeof(unsigned long long), pl->stream));
    if (!pl->preset_stats) {
        CU(cudaMemsetAsync(pl->d_mean, 0, (size_t)pl->ndm * pl->prm.nif * ncol * sizeof(float), pl->stream));
        // keep_bandpass with normalised transforms (D4): the "scale" the digitiser applies is 1 / (M * freq_res), squared for -d3
        float unit = 1.0f;
        if (pl->prm.keep_bandpass && pl->prm.fft_normalised) {
            const double nrm = 1.0 / ((double)pl->M * pl->L);
            unit = (float)(pl->prm.pol_mode == B2F_POL_I2 ? nrm * nrm : nrm);
        }
        std::vector<float> ones((size_t)pl->ndm * pl->prm.nif * ncol, unit);
        CU(cudaMemcpyAsync(pl->d_scale, ones.data(), ones.size() * sizeof(float), cudaMemcpyHostToDevice, pl->stream));
    }
    CU(cudaStreamSynchronize(pl->stream));
    return 0;
}

}  // namespace

// JA98 decode outside the round-2 column kernel: levels per window of 512 samples of the de-framed stream of this push
// (T samples per IF, carried samples included); no-op for the static levels.
int stream_levels(b2f_plan* pl, int64_t T) {
    if (!pl->d_levels_stream) return 0;
    const int nif = pl->prm.nif;
    const int64_t nthreads = ((T + 511) / 512) * nif * 32;
    kj_levels_stream<<<(unsigned)((nthreads + 255) / 256), 256, 0, pl->stream>>>(pl->d_compact, pl->compact_stride, T, pl->d_levels_stream,
                                                                                pl->levels_stride, nif);
    pl->launches++;
    CU(cudaGetLastError());
    return 0;
}

// Carry-mode path of one push (dedispersion and / or the generic channeliser).  Tuned dedispersion: forward column pass ->
// row FFT (spectrum) -> un-mix, chirp, backward column FFT, overlap discard, detect, integrate; generic shapes: generic
// column and row kernels, with dedispersion the row pass leaves channel samples and kx_dedisp_generic finishes.  Leaves the
// unconsumed tail of the sample stream (and, for 8-bit input, of its word masks) in d_carry for the next push
// ("time-chunked coherent dedispersion carries its overlap halo").
int push_dedisp(b2f_plan* pl, int64_t nblk, int64_t T) {
    const int nif = pl->prm.nif;
    const int64_t nbt = (int64_t)nif * nblk;
    int rc = 0;
    if (nblk > 0 && pl->smask) {                              // which blocks hold a masked word (stream-coordinate masks)
        k8_blkdirty<<<dim3((unsigned)nblk, (unsigned)nif), 256, 0, pl->stream>>>(pl->d_wmask, pl->wmask_stride, pl->d_blkdirty, (int)nblk,
                                                                                pl->step * pl->bps / 32, pl->M * pl->bps / 32);
        pl->launches++;
        CU(cudaGetLastError());
    }
    if (nblk > 0 && pl->longfft) {
        // freq_res 8192..65536 (b2f_kl.cu): forward column transform and row FFT once, the backward part once per trial
        const int64_t NB = pl->batch_blocks > 0 ? std::min<int64_t>(pl->batch_blocks, nbt) : nbt;
        if ((rc = stream_levels(pl, T))) return rc;
        KLParams kl{};
        kl.compact = pl->d_compact; kl.compact_stride = pl->compact_stride;
        kl.wmask = pl->d_wmask; kl.wmask_stride = pl->wmask_stride; kl.blkdirty = pl->d_blkdirty;
        kl.levels = pl->d_levels_stream; kl.levels_stride = pl->levels_stride;
        kl.in8_offset = pl->prm.in8_offset_mode ? 128.0f : 127.5f;
        kl.in_nbit = pl->d_levels_stream ? 22 : (pl->bps == 2 ? 8 : 2);
        kl.step = pl->step;
        kl.inter = pl->d_inter; kl.spec = pl->d_spec;
        kl.F = row_dst(pl); kl.F_if_stride = row_dst_stride(pl); kl.row0 = row_dst_row0(pl);
        kl.R = pl->R; kl.lgR = 31 - __builtin_clz(pl->R); kl.L = pl->L; kl.lgL = 31 - __builtin_clz(pl->L);
        kl.lgLa = 8; kl.lgLb = kl.lgL - 8; kl.M = pl->M;
        kl.nblk = (int)nblk; kl.nif = nif; kl.D = pl->D; kl.mode = pl->prm.pol_mode;
        kl.nfilt_pos = pl->nfilt_pos; kl.keep = pl->keep;
        for (int64_t b0 = 0; b0 < nbt; b0 += NB) {
            kl.gb_begin = b0; kl.gb_end = b0 + std::min(NB, nbt - b0);
            cudaError_t le = cudaSuccess;
            if ((rc = timed(pl, B2F_K_COLUMN, [&] { le = b2f_launch_kl_column(kl, pl->stream); }))) return rc;
            if (le != cudaSuccess) return fail(B2F_ECUDA, std::string("long column transform: ") + cudaGetErrorString(le));
            if ((rc = timed(pl, B2F_K_ROW, [&] { le = b2f_launch_kl_row(kl, pl->stream); }))) return rc;
            if (le != cudaSuccess) return fail(B2F_ECUDA, std::string("long row FFT: ") + cudaGetErrorString(le));
            for (int t = 0; t < pl->ndm; ++t) {
                KLParams kt = kl;
                kt.chirp = pl->d_chirp + (int64_t)t * nif * pl->L * pl->N;
                kt.F = kl.F + (int64_t)t * nif * kl.F_if_stride;
                if ((rc = timed(pl, B2F_K_DEDISP, [&] { le = b2f_launch_kl_back(kt, pl->stream); }))) return rc;
                if (le != cudaSuccess) return fail(B2F_ECUDA, std::string("long dedispersion back end: ") + cudaGetErrorString(le));
            }
        }
    } else if (nblk > 0 && pl->generic) {
        const int64_t NB = pl->batch_blocks > 0 ? std::min<int64_t>(pl->batch_blocks, nbt) : nbt;
        KGParams kg{};
        kg.compact = pl->d_compact; kg.compact_stride = pl->compact_stride;
        kg.wmask = pl->d_wmask; kg.wmask_stride = pl->wmask_stride; kg.blkdirty = pl->d_blkdirty;
        kg.in8_offset = pl->prm.in8_offset_mode ? 128.0f : 127.5f;
        kg.step = pl->step;
        kg.levels = pl->d_levels_stream; kg.levels_stride = pl->levels_stride;
        const int nbit = pl->d_levels_stream ? 22 : pl->prm.in_nbit;          // 22: 2-bit input decoded with JA98 levels
        if ((rc = stream_levels(pl, T))) return rc;
        kg.inter = pl->d_inter; kg.colsum = pl->d_colsum; kg.eps = pl->d_eps;
        kg.tw_col = pl->d_tw_col; kg.tw_row = pl->d_tw_row;
        kg.F = row_dst(pl); kg.F_if_stride = row_dst_stride(pl); kg.row0 = row_dst_row0(pl);
        kg.L = pl->L; kg.lgL = 31 - __builtin_clz(pl->L); kg.R = pl->R; kg.lgR = 31 - __builtin_clz(pl->R);
        kg.C = std::min(16, 8192 / pl->L);                    // 64 KiB of column data per CTA, two CTAs per SM
        kg.lgC = 31 - __builtin_clz(kg.C);
        kg.nblk = (int)nblk; kg.nif = nif; kg.D = pl->D; kg.mode = pl->prm.pol_mode; kg.M = pl->M;
        const int RB = std::max(1, std::min(16, 4096 / pl->R));
        const size_t smem_col = ((size_t)pl->L + 32 + kg_padded((size_t)pl->L * kg.C)) * sizeof(float2);
        const size_t smem_row = ((size_t)pl->R + kg_padded((size_t)RB * pl->R) + 2 * (size_t)RB * pl->R) * sizeof(float2);
        if (!pl->kgt_lg) {
            CU(cudaFuncSetAttribute(kg_column_pass<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_col));
            CU(cudaFuncSetAttribute(kg_column_pass<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_col));
            CU(cudaFuncSetAttribute(kg_column_pass<22>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_col));
        }
        if (!pl->kgt_lg || pl->dedisp) {
            CU(cudaFuncSetAttribute(kg_row_pass<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_row));
            CU(cudaFuncSetAttribute(kg_row_pass<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_row));
        }
        // dedispersion behind the generic kernels (kx_dedisp_generic): the row pass leaves un-detected channel samples
        KXParams kx{};
        size_t smem_kx = 0;
        if (pl->dedisp) {
            kx.volt = pl->d_spec; kx.chirp = pl->d_chirp;
            kx.F = kg.F; kx.F_if_stride = kg.F_if_stride; kx.row0 = kg.row0;
            kx.L = pl->L; kx.lgL = kg.lgL; kx.N = pl->N; kx.CH = std::max(1, std::min(4, 8192 / pl->L));
            kx.nblk = (int)nblk; kx.nif = nif; kx.D = pl->D; kx.mode = pl->prm.pol_mode;
            kx.nfilt_pos = pl->nfilt_pos; kx.keep = pl->keep;
            smem_kx = ((size_t)pl->L / 2 + (size_t)kx.CH * 2 * (pl->L + pl->L / 16)) * sizeof(float2);     // one pad element per 16 (kx_ph)
            CU(cudaFuncSetAttribute(kx_dedisp_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_kx));
        }
        if (pl->R * sizeof(float2) > 48 * 1024)
            CU(cudaFuncSetAttribute(ke_eps, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(pl->R * sizeof(float2))));
        for (int64_t b0 = 0; b0 < nbt; b0 += NB) {
            const int64_t nb = std::min(NB, nbt - b0);
            kg.gb_begin = b0; kg.gb_end = b0 + nb;
            cudaError_t le = cudaSuccess;
            rc = timed(pl, B2F_K_COLUMN, [&] {
                if (pl->kgt_lg) {                           // compile-time geometry (b2f_generic.cuh): L = R = 2^kgt_lg
                    const int64_t work = nb * (pl->R / pl->kgt_cols);
                    le = b2f_launch_kgt_col(pl->kgt_lg, nbit, kg, (int)std::min<int64_t>(work, (int64_t)pl->kgt_col_ctas * pl->num_sms), pl->stream, nullptr);
                } else {
                    const int64_t work = nb * (pl->R / kg.C);
                    const unsigned grid = (unsigned)std::min<int64_t>(work, 2 * (int64_t)pl->num_sms);
                    if (nbit == 8) kg_column_pass<8><<<grid, 256, smem_col, pl->stream>>>(kg);
                    else if (nbit == 22) kg_column_pass<22><<<grid, 256, smem_col, pl->stream>>>(kg);
                    else kg_column_pass<2><<<grid, 256, smem_col, pl->stream>>>(kg);
                }
            });
            if (rc) return rc;
            if (le != cudaSuccess) return fail(B2F_ECUDA, std::string("generic column pass: ") + cudaGetErrorString(le));
            rc = timed(pl, B2F_K_EPS, [&] {
                ke_eps<<<(unsigned)nb, std::min(pl->R / 2, 512), pl->R * sizeof(float2), pl->stream>>>(pl->d_colsum + b0 * pl->R,
                                                                                       pl->d_eps + b0 * pl->N, pl->R);
            });
            if (rc) return rc;
            rc = timed(pl, B2F_K_ROW, [&] {
                if (pl->dedisp) {
                    KGParams kv = kg;
                    kv.mode = kModeVolt; kv.D = 1; kv.volt = pl->d_spec;
                    const int64_t nunits = nb * (pl->L / RB);
                    const unsigned grid = (unsigned)std::min<int64_t>(nunits, (int64_t)pl->num_sms * 2);
                    if (pl->N > 1024) kg_row_pass<8><<<grid, 256, smem_row, pl->stream>>>(kv);
                    else kg_row_pass<4><<<grid, 256, smem_row, pl->stream>>>(kv);
                } else if (pl->kgt_lg) {
                    const int64_t nunits = nb * (pl->L / std::max(pl->D, pl->kgt_rb));
                    le = b2f_launch_kgt_row(pl->kgt_lg, pl->prm.pol_mode, kg, (int)std::min<int64_t>(nunits, (int64_t)pl->kgt_row_ctas * pl->num_sms),
                                            pl->stream, nullptr);
                } else {
                    const int64_t nunits = nb * (pl->L / std::max(pl->D, RB));
                    if (pl->N > 1024) kg_row_pass<8><<<(unsigned)std::min<int64_t>(nunits, (int64_t)pl->num_sms * 2), 256, smem_row, pl->stream>>>(kg);
                    else kg_row_pass<4><<<(unsigned)std::min<int64_t>(nunits, (int64_t)pl->num_sms * 2), 256, smem_row, pl->stream>>>(kg);
                }
            });
            if (rc) return rc;
            if (le != cudaSuccess) return fail(B2F_ECUDA, std::string("generic row pass: ") + cudaGetErrorString(le));
            if (pl->dedisp) {
                kx.gb_begin = b0; kx.gb_end = b0 + nb;
                const int64_t work = nb * (pl->N / kx.CH);
                for (int t = 0; t < pl->ndm; ++t) {             // trial DMs: the same channel samples, each trial's chirp and F slots
                    KXParams kt = kx;
                    kt.chirp = kx.chirp + (int64_t)t * nif * pl->L * pl->N;
                    kt.F = kx.F + (int64_t)t * nif * kx.F_if_stride;
                    rc = timed(pl, B2F_K_DEDISP, [&] {
                        kx_dedisp_generic<<<(unsigned)std::min<int64_t>(work, (int64_t)pl->num_sms), kKXThreads, smem_kx, pl->stream>>>(kt);
                    });
                    if (rc) return rc;
                }
            }
        }
    } else if (nblk > 0) {
        const int64_t cap = pl->batch_blocks > 0 ? pl->batch_blocks : (int64_t)nif * pl->chunk_blocks;
        const int64_t NB = std::min<int64_t>(cap, nbt);
        KAParams ka{};
        ka.compact = pl->d_compact; ka.compact_stride = pl->compact_stride;
        ka.wmask = pl->d_wmask; ka.wmask_stride = pl->wmask_stride; ka.blkdirty = pl->d_blkdirty;
        ka.inter = pl->d_inter; ka.colsum = pl->d_colsum;
        ka.tab_g = pl->d_tab_g; ka.tab_h = pl->d_tab_h; ka.tab_w = pl->d_tab_w; ka.tab_beta = pl->d_tab_beta;
        ka.R = pl->R; ka.nstrips = pl->nstrips; ka.nblk = (int)nblk; ka.nif = nif;
        ka.payload_bytes = (int)pl->payload; ka.groups_per_slot = (int)pl->groups_per_slot;
        ka.blk_step_bytes = pl->step * pl->bps;                   // 2-bit: 1 index byte per sample; 8-bit: 2 bytes, masks by stream position
        ka.in8_offset = pl->prm.in8_offset_mode ? 128.0f : 127.5f;
        ka.levels = pl->d_levels_stream; ka.levels_stride = pl->levels_stride;
        if (int rcl = stream_levels(pl, T)) return rcl;
        KBParams kb{};
        kb.inter = pl->d_inter; kb.eps = nullptr; kb.tab_r = pl->d_tab_r; kb.spec = pl->d_spec;
        kb.F = nullptr; kb.nblk = (int)nblk; kb.nif = nif; kb.D = 1;
        KCParams kc{};
        kc.spec = pl->d_spec; kc.chirp = pl->d_chirp; kc.tab_w = pl->d_tab_w;
        kc.F = row_dst(pl); kc.F_if_stride = row_dst_stride(pl); kc.row0 = row_dst_row0(pl);
        kc.nblk = (int)nblk; kc.nif = nif; kc.D = pl->D; kc.mode = pl->prm.pol_mode;
        kc.nfilt_pos = pl->nfilt_pos; kc.keep = pl->keep; kc.ndm = pl->ndm;
        const bool trials = pl->prm.ndm > 0;            // kc_dedisp_trials: one CTA per SM (registers hold the un-mixed spectrum)
        int TR, PT;
        kb_shape(pl->R, &TR, &PT);
        const int RW = 32 / TR;
        for (int64_t b0 = 0; b0 < nbt; b0 += NB) {
            const int64_t nb = std::min(NB, nbt - b0);
            ka.gb_begin = b0; ka.gb_end = b0 + nb;
            int64_t grid = std::max<int64_t>(1, (kKACtasPerSM * pl->num_sms) / pl->nstrips) * pl->nstrips;
            grid = std::min<int64_t>(grid, nb * pl->nstrips);
            rc = launch_ka(pl, true, ka, (unsigned)grid);         // forward only: the chirp goes between row FFT and backward FFT
            if (rc) return rc;
            kb.gb_begin = b0; kb.gb_end = b0 + nb;
            const int64_t ngroups = nb * (kL / RW);
            const int64_t ctas = (ngroups + kKBThreads / 32 - 1) / (kKBThreads / 32);
            cudaError_t e = cudaSuccess;
            rc = timed(pl, B2F_K_ROW, [&] { e = b2f_launch_kb(pl->R, kModeSpectrum, kb, (int)std::min<int64_t>(ctas, (int64_t)pl->num_sms * 2), pl->stream); });
            if (rc) return rc;
            if (e != cudaSuccess) return fail(B2F_ECUDA, std::string("row pass launch: ") + cudaGetErrorString(e));
            kc.gb_begin = b0; kc.gb_end = b0 + nb;
            const int64_t work = nb * (pl->N / 8);
            rc = timed(pl, B2F_K_DEDISP, [&] {
                e = b2f_launch_kc(pl->R, kc, trials, (int)std::min<int64_t>(work, (int64_t)pl->num_sms * (trials ? 1 : 2)), pl->stream);
            });
            if (rc) return rc;
            if (e != cudaSuccess) return fail(B2F_ECUDA, std::string("dedispersion back end launch: ") + cudaGetErrorString(e));
        }
    }
    // keep what the next push still needs
    const int64_t used = nblk * pl->step;
    const int64_t tail = T - used;
    if (tail > pl->M) return fail(B2F_ESTATE, "internal: dedispersion carry larger than one block");
    for (int i = 0; i < nif; ++i)
        CU(cudaMemcpyAsync(pl->d_carry + (size_t)i * pl->M * pl->bps, pl->d_compact + i * pl->compact_stride + used * pl->bps,
                           (size_t)tail * pl->bps, cudaMemcpyDeviceToDevice, pl->stream));
    if (pl->smask)
        for (int i = 0; i < nif; ++i)
            CU(cudaMemcpyAsync(pl->d_carry_mask + (size_t)i * (pl->M * pl->bps / 32), pl->d_wmask + i * pl->wmask_stride + used * pl->bps / 32,
                               (size_t)(tail * pl->bps / 32), cudaMemcpyDeviceToDevice, pl->stream));
    pl->carry_len = tail;
    return 0;
}

cudaError_t b2f_launch_ka(int in_nbit, int R, bool fwd_only, const KAParams& p, unsigned grid, cudaStream_t st) {
    if (in_nbit == 22) return b2f_launch_ka_22(R, fwd_only, p, grid, st);                                         // 2-bit input, JA98 levels
    return in_nbit == 8 ? b2f_launch_ka_8(R, fwd_only, p, grid, st) : b2f_launch_ka_2(R, fwd_only, p, grid, st);   // 1- and 2-bit: index-byte stream
}
cudaError_t b2f_launch_kr(int R, int mode, const KBParams& p, int grid, cudaStream_t st) {     // R != 256: that row length uses the tile row pass
    if (R <= 64) return b2f_launch_kr_part0(R, mode, p, grid, st);
    return b2f_launch_kr_part1(R, mode, p, grid, st);
}
cudaError_t b2f_launch_kb(int R, int mode, const KBParams& p, int grid, cudaStream_t st) {
    if (R <= 64) return b2f_launch_kb_part0(R, mode, p, grid, st);
    if (R == 256) return b2f_launch_kb_part2(R, mode, p, grid, st);
    return b2f_launch_kb_part1(R, mode, p, grid, st);
}

cudaError_t b2f_launch_kf(int R, int mode, const FParams& p, int grid, int cooperative, cudaStream_t st, int* occ) {
    switch (R) {
        case 16: return b2f_launch_kf_16(mode, p, grid, cooperative, st, occ);
        case 32: return b2f_launch_kf_32(mode, p, grid, cooperative, st, occ);
        case 64: return b2f_launch_kf_64(mode, p, grid, cooperative, st, occ);
        case 128: return b2f_launch_kf_128(mode, p, grid, cooperative, st, occ);
        case 256: return b2f_launch_kf_256(mode, p, grid, cooperative, st, occ);
        case 512: return b2f_launch_kf_512(mode, p, grid, cooperative, st, occ);
    }
    return cudaErrorInvalidValue;
}

cudaError_t b2f_launch_kgt_col(int lg, int in_nbit, const KGParams& p, int grid, cudaStream_t st, int* ctas) {
    switch (lg) {
        case 10: return b2f_launch_kgt_col_10(in_nbit, p, grid, st, ctas);
        case 11: return b2f_launch_kgt_col_11(in_nbit, p, grid, st, ctas);
        case 12: return b2f_launch_kgt_col_12(in_nbit, p, grid, st, ctas);
        case 13: return b2f_launch_kgt_col_13(in_nbit, p, grid, st, ctas);
    }
    return cudaErrorInvalidValue;
}

cudaError_t b2f_launch_kgt_row(int lg, int mode, const KGParams& p, int grid, cudaStream_t st, int* ctas) {
    switch (lg) {
        case 10: return b2f_launch_kgt_row_10(mode, p, grid, st, ctas);
        case 11: return b2f_launch_kgt_row_11(mode, p, grid, st, ctas);
        case 12: return b2f_launch_kgt_row_12(mode, p, grid, st, ctas);
        case 13: return b2f_launch_kgt_row_13(mode, p, grid, st, ctas);
    }
    return cudaErrorInvalidValue;
}

void b2f_kgt_geometry(int lg, int* cols, int* rb) {
    switch (lg) {
        case 10: *cols = KGT<10>::C; *rb = KGT<10>::RB; break;
        case 11: *cols = KGT<11>::C; *rb = KGT<11>::RB; break;
        case 12: *cols = KGT<12>::C; *rb = KGT<12>::RB; break;
        default: *cols = KGT<13>::C; *rb = KGT<13>::RB; break;
    }
}

namespace {

// the fused kernel gives up (instead of hanging the GPU) if a warp waits ~1 s for another one: surface that
int check_fused_abort(b2f_plan* pl) {
    if (pl->path != 2 || !pl->d_fsync) return 0;
    if (!pl->f_aborted) {
        unsigned flag = 0;
        CU(cudaMemcpyAsync(&flag, pl->d_fsync + (size_t)pl->f_lanes * FS_STRIDE, sizeof(flag), cudaMemcpyDeviceToHost, pl->stream));
        CU(cudaStreamSynchronize(pl->stream));
        if (flag) pl->f_aborted = true;
    }
    if (pl->f_aborted) return fail(B2F_ECUDA, "fused channeliser: inter-warp wait timed out (results of this scan are invalid)");
    return 0;
}

// Round-2 channeliser of one push: header check, transposing de-framer, then either the fused kernel or its two
// halves as separate launches, then the sum of partial rows where tscrunch spans several warps' rows.
int push_fused(b2f_plan* pl, const K0Params& k0, int64_t nframes, int64_t nblk) {
    const int nif = pl->prm.nif;
    const int64_t nbt = (int64_t)nif * nblk;
    int rc = 0;
    for (int i = 0; i < nif; ++i)
        if (reinterpret_cast<uintptr_t>(k0.frames[i]) & 15) return fail(B2F_EINVAL, "frames must be 16-byte aligned");
    K0HParams kh{};
    K0TParams kt{};
    for (int i = 0; i < nif; ++i) {
        kh.frames[i] = k0.frames[i]; kt.frames[i] = k0.frames[i];
        kh.base_sec[i] = k0.base_sec[i]; kh.base_fnum[i] = k0.base_fnum[i];
    }
    kh.fstat = pl->d_fstat; kh.fstat_stride = pl->fstat_stride; kh.counters = pl->d_counters;
    kh.nframes = nframes; kh.frame_bytes = pl->prm.frame_bytes; kh.header_bytes = pl->prm.header_bytes;
    kh.in_nbit = pl->prm.in_nbit; kh.fps = (int)pl->fps; kh.nif = nif;
    kt.fstat = pl->d_fstat; kt.fstat_stride = pl->fstat_stride;
    kt.fillflag = pl->d_fillflag; kt.fillflag_stride = pl->fillflag_stride;
    kt.tstream = pl->d_tstream; kt.tstream_if_stride = pl->tstream_stride; kt.counters = pl->d_counters;
    kt.nblk = (int)nblk; kt.nif = nif; kt.R = pl->R; kt.frame_bytes = pl->prm.frame_bytes;
    kt.header_bytes = pl->prm.header_bytes; kt.payload_bytes = (int)pl->payload; kt.mask_faults = pl->prm.mask_faults;
    CU(cudaMemsetAsync(pl->d_fillflag, 0, pl->fillflag_stride * nif * sizeof(int), pl->stream));
    rc = timed(pl, B2F_K_VALIDATE, [&] {
        const int64_t n = nframes * nif;
        k0h_headers<<<(unsigned)((n + 255) / 256), 256, 0, pl->stream>>>(kh);
        if (nblk > 0) {
            const int sc = std::min(64, pl->R);
            const int64_t units = nbt * (pl->R / sc);
            const unsigned grid = (unsigned)std::min<int64_t>(units, (int64_t)pl->num_sms * (sc == 64 ? 6 : 8));
            if (sc == 64) k0t_transpose<64><<<grid, 256, 0, pl->stream>>>(kt);
            else if (sc == 32) k0t_transpose<32><<<grid, 256, 0, pl->stream>>>(kt);
            else k0t_transpose<16><<<grid, 256, 0, pl->stream>>>(kt);
        }
    });
    if (rc) return rc;
    pl->launches++;                                   // two kernels in one timed region
    if (nblk == 0) return 0;
    if (pl->d_levels) {
        KJParams kj{};
        for (int i = 0; i < nif; ++i) kj.frames[i] = k0.frames[i];
        kj.fstat = pl->d_fstat; kj.fstat_stride = pl->fstat_stride; kj.levels = pl->d_levels;
        kj.nblk = (int)nblk; kj.nif = nif; kj.R = pl->R; kj.frame_bytes = pl->prm.frame_bytes;
        kj.header_bytes = pl->prm.header_bytes; kj.payload_bytes = (int)pl->payload; kj.mask_faults = pl->prm.mask_faults;
        const int64_t nthreads = nbt * pl->R * 32;
        rc = timed(pl, B2F_K_VALIDATE, [&] { kj_ja98_levels<<<(unsigned)((nthreads + 255) / 256), 256, 0, pl->stream>>>(kj); });
        if (rc) return rc;
    }

    FParams fp{};
    fp.tstream = pl->d_tstream; fp.tstream_if_stride = pl->tstream_stride;
    fp.ring = pl->d_inter; fp.colsum = pl->d_colsum; fp.eps = pl->d_eps;
    fp.tab_h = pl->d_tab_h; fp.tab_w = pl->d_tab_w; fp.tab_beta = pl->d_tab_beta; fp.tab_r = pl->d_tab_r;
    const bool direct = pl->Dp == pl->D || pl->path == 1;
    fp.out = direct ? row_dst(pl) : pl->d_part;
    fp.out_if_stride = direct ? row_dst_stride(pl) : pl->part_if_stride;
    fp.out_row0 = direct ? row_dst_row0(pl) : 0;
    fp.Dp = pl->Dp; fp.nblk = (int)nblk; fp.nif = nif;
    fp.gb_begin = 0; fp.gb_end = nbt;
    fp.sync = pl->d_fsync; fp.abort_flag = pl->d_fsync + (size_t)pl->f_lanes * FS_STRIDE;
    fp.nslot = pl->f_nslot; fp.lag = pl->f_lag; fp.prof = pl->d_fprof; fp.levels = pl->d_levels;
    cudaError_t e = cudaSuccess;
    if (pl->path == 2) {
        CU(cudaMemsetAsync(pl->d_fsync, 0, (size_t)pl->f_lanes * FS_STRIDE * sizeof(unsigned), pl->stream));
        fp.phase = 0;
        rc = timed(pl, B2F_K_FUSED, [&] { e = b2f_launch_kf(pl->R, pl->prm.pol_mode, fp, pl->f_grid, 1, pl->stream, nullptr); });
        if (rc) return rc;
        if (e != cudaSuccess) return fail(B2F_ECUDA, std::string("fused channeliser launch: ") + cudaGetErrorString(e));
    } else {
        fp.phase = 1;
        // the column half does not depend on the detection product: always the Stokes I instantiation, which is free of the
        // spills the four-product row code brings into the kernel (C3: 90.8 -> 77 ms per 60 s)
        rc = timed(pl, B2F_K_COLUMN, [&] { e = b2f_launch_kf(pl->R, B2F_POL_I, fp, pl->f_grid, 0, pl->stream, nullptr); });
        if (rc) return rc;
        if (e != cudaSuccess) return fail(B2F_ECUDA, std::string("column half launch: ") + cudaGetErrorString(e));
        rc = timed(pl, B2F_K_EPS, [&] {
            ke_eps<<<(unsigned)nbt, std::min(pl->R / 2, 512), pl->R * sizeof(float2), pl->stream>>>(pl->d_colsum, pl->d_eps, pl->R);
        });
        if (rc) return rc;
        if (pl->R == 256) {
            // 16-row tiles are 32 KiB contiguous in the block layout: one bulk copy per tile, block-wide second FFT stage
            KTParams kt{};
            kt.inter = pl->d_inter; kt.eps = pl->d_eps; kt.tab_r = pl->d_tab_r;
            kt.F = row_dst(pl); kt.F_if_stride = row_dst_stride(pl); kt.row0 = row_dst_row0(pl);
            kt.nblk = (int)nblk; kt.nif = nif; kt.D = pl->D; kt.nb = nbt;
            const int64_t units = nbt * (32 / std::max(1, pl->D / 16));
            rc = timed(pl, B2F_K_ROW, [&] { e = b2f_launch_kt(pl->prm.pol_mode, kt, (int)std::min<int64_t>(units, (int64_t)pl->num_sms * 2), pl->stream); });
            if (rc) return rc;
            if (e != cudaSuccess) return fail(B2F_ECUDA, std::string("tile row pass launch: ") + cudaGetErrorString(e));
            return 0;
        }
        // other row lengths: per-warp cp.async ring over the same blocks, whole integration groups per warp -> F directly
        int TR, PT;
        kb_shape(pl->R, &TR, &PT);
        const int RW = 32 / TR, GW = std::max(pl->D, RW);
        KBParams kb{};
        kb.inter = pl->d_inter; kb.eps = pl->d_eps; kb.tab_r = pl->d_tab_r;
        kb.F = row_dst(pl); kb.F_if_stride = row_dst_stride(pl); kb.row0 = row_dst_row0(pl);
        kb.nblk = (int)nblk; kb.nif = nif; kb.D = pl->D; kb.gb_begin = 0; kb.gb_end = nbt;
        const int64_t ngroups = nbt * (kL / GW);
        const int64_t ctas = (ngroups + kKBThreads / 32 - 1) / (kKBThreads / 32);
        rc = timed(pl, B2F_K_ROW, [&] { e = b2f_launch_kr(pl->R, pl->prm.pol_mode, kb, (int)std::min<int64_t>(ctas, (int64_t)pl->num_sms * 2), pl->stream); });
        if (rc) return rc;
        if (e != cudaSuccess) return fail(B2F_ECUDA, std::string("row pass launch: ") + cudaGetErrorString(e));
        return 0;
    }
    if (!direct) {
        const int ncol = pl->nprod * pl->N;
        const int64_t rows = nblk * kL / pl->D;
        const int64_t n4 = rows * (ncol / 4);
        rc = timed(pl, B2F_K_TSUM, [&] {
            kt_sum_partials<<<dim3((unsigned)((n4 + 255) / 256), nif), 256, 0, pl->stream>>>(
                pl->d_part, pl->part_if_stride, row_dst(pl), row_dst_stride(pl), row_dst_row0(pl), rows, ncol, pl->D / pl->Dp);
        });
        if (rc) return rc;
    }
    return 0;
}

}  // namespace

// tscrunch beyond what the row kernels integrate: output row r = sum of tsq consecutive kernel rows, in a fixed order
static __global__ void kd_sum_rows(const float* __restrict__ Fk, int64_t Fk_if_stride, float* __restrict__ F, int64_t F_if_stride,
                                   int64_t row0, int64_t nrows, int ncol, int q) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= nrows * ncol) return;
    const int64_t r = i / ncol;
    const int c = (int)(i - r * ncol);
    const float* src = Fk + blockIdx.y * Fk_if_stride + r * q * (int64_t)ncol + c;
    float acc = 0.f;
    for (int k = 0; k < q; ++k) acc += src[(int64_t)k * ncol];
    F[blockIdx.y * F_if_stride + (row0 + r) * ncol + c] = acc;
}

namespace {
int sum_rows(b2f_plan* pl, int64_t krows, int64_t rows) {
    if (pl->tsq <= 1) return 0;
    const int ncol = pl->nprod * pl->N, nif = pl->ndm * pl->prm.nif;     // every (trial, IF) slot
    const int64_t total = pl->fk_pending + krows, left = total - rows * pl->tsq;
    if (rows > 0) {
        const int64_t n = rows * ncol;
        int rc = timed(pl, B2F_K_TSUM, [&] {
            kd_sum_rows<<<dim3((unsigned)((n + 255) / 256), nif), 256, 0, pl->stream>>>(pl->d_Fk, pl->Fk_if_stride, pl->d_F, pl->F_if_stride,
                                                                                      pl->rows_off + pl->rows_held, rows, ncol, pl->tsq);
        });
        if (rc) return rc;
        // the kernel rows of the unfinished sample (fewer than tsq, so they cannot overlap their destination) move to the front
        for (int i = 0; i < nif && left > 0; ++i)
            CU(cudaMemcpyAsync(pl->d_Fk + i * pl->Fk_if_stride, pl->d_Fk + i * pl->Fk_if_stride + rows * pl->tsq * (int64_t)ncol,
                               (size_t)left * ncol * sizeof(float), cudaMemcpyDeviceToDevice, pl->stream));
    }
    pl->fk_pending = left;
    return 0;
}
}  // namespace

// digifil -K: output row r of slot (trial, IF) = sum of the Du channel samples r Du + k + d_c (k < Du) of the delay ring, added
// in order k = 0, 1, ...  Threads run over (row, column) with the column fastest and the slot in blockIdx.y, so the CTAs in
// flight cover a narrow band of rows of one slot: a lane's load touches its own 32-byte sector (neighbouring channels sit at
// rows d_c apart), and the other channels of that sector are read by later rows while it is still in L2.  Each byte of the
// ring is read from DRAM about once.
struct KDParams {
    const float* Fk;
    int64_t Fk_stride, off, wrap;  // ring rows per slot, row of logical sample 0, wrap point
    float* F;
    int64_t F_stride, row0, nrows;
    const int64_t* delays;         // [slot][chan]
    int ncol, N, Du;
};

static __global__ void __launch_bounds__(256) kd_delay_sum(KDParams p) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= p.nrows * p.ncol) return;
    const int64_t r = i / p.ncol;
    const int col = (int)(i - r * p.ncol);
    const int c = col % p.N;
    const float* src = p.Fk + blockIdx.y * p.Fk_stride + col;
    int64_t q = p.off + r * p.Du + p.delays[(int64_t)blockIdx.y * p.N + c];
    if (q >= p.wrap) q -= p.wrap;
    float acc = src[q * p.ncol];
    for (int k = 1; k < p.Du; ++k) {
        if (++q == p.wrap) q = 0;
        acc += src[q * p.ncol];
    }
    p.F[blockIdx.y * p.F_stride + (p.row0 + r) * p.ncol + col] = acc;
}

namespace {
// where this push's channel samples go in the ring (before the row kernels run)
int delay_place(b2f_plan* pl, int64_t krows) {
    if (!pl->delays || krows == 0) return 0;
    int64_t w = pl->dl_off + pl->dl_held;
    if (!pl->dl_wrapped) {
        if (w + krows > pl->dl_cap) {
            pl->dl_wrap = w;
            pl->dl_wrapped = true;
            w = 0;
        }
    } else {
        w -= pl->dl_wrap;
    }
    if (pl->dl_wrapped && w + krows > pl->dl_off) return fail(B2F_ESTATE, "internal: delay ring overrun");
    pl->dl_w = w;
    return 0;
}

// rows of this push from the ring into F; the consumed samples leave the ring
int delay_sum(b2f_plan* pl, int64_t krows, int64_t rows) {
    const int ncol = pl->nprod * pl->N, nslot = pl->ndm * pl->prm.nif;
    if (rows > 0) {
        KDParams kd{};
        kd.Fk = pl->d_Fk; kd.Fk_stride = pl->Fk_if_stride; kd.off = pl->dl_off; kd.wrap = pl->dl_wrap;
        kd.F = pl->d_F; kd.F_stride = pl->F_if_stride; kd.row0 = pl->rows_off + pl->rows_held; kd.nrows = rows;
        kd.delays = pl->d_delays; kd.ncol = ncol; kd.N = pl->N; kd.Du = pl->Du;
        const int64_t n = rows * ncol;
        int rc = timed(pl, B2F_K_TSUM, [&] { kd_delay_sum<<<dim3((unsigned)((n + 255) / 256), nslot), 256, 0, pl->stream>>>(kd); });
        if (rc) return rc;
    }
    const int64_t used = rows * pl->Du;
    pl->dl_held += krows - used;
    pl->dl_off += used;
    if (pl->dl_wrapped && pl->dl_off >= pl->dl_wrap) {
        pl->dl_off -= pl->dl_wrap;
        pl->dl_wrap = pl->dl_cap;
        pl->dl_wrapped = false;
    }
    return 0;
}
}  // namespace

extern "C" {

int b2f_version(void) { return B2F_VERSION; }
const char* b2f_last_error(void) { return g_err.c_str(); }

int b2f_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int b2f_plan_create(const b2f_params* prm, b2f_plan** out) {
    if (!prm || !out) return fail(B2F_EINVAL, "null argument");
    if (prm->struct_size != sizeof(b2f_params)) return fail(B2F_EINVAL, "b2f_params.struct_size mismatch");
    *out = nullptr;
    if (prm->nif < 1 || prm->nif > B2F_MAX_IF) return fail(B2F_EINVAL, "nif out of range");
    const int nprod = nprod_of(prm->pol_mode);
    if (!nprod) return fail(B2F_EINVAL, "pol_mode not in 0..6 (process_vdif --pol choices map to 0,1,2,3,4)");
    if (!(prm->out_nbit == 2 || prm->out_nbit == 8 || prm->out_nbit == 16 || prm->out_nbit == -32))
        return fail(B2F_EINVAL, "nbit not in supported values of [2, 8, 16, -32]");
    if (!(prm->in_nbit == 1 || prm->in_nbit == 2 || prm->in_nbit == 8)) return fail(B2F_EUNSUPPORTED, "VDIF bits/sample must be 1, 2 or 8");
    if (prm->nchan < 1) return fail(B2F_EINVAL, "nchan");
    // trial DMs: one coherent plan writes ndm filterbanks; its geometry is that of a single-DM plan at the largest trial
    if (prm->ndm < 0 || prm->ndm > B2F_MAX_DM) return fail(B2F_EINVAL, "ndm must be 0..64 (B2F_MAX_DM)");
    double dm = prm->dm;
    if (prm->ndm > 0) {
        if (prm->coherent != 1) return fail(B2F_EINVAL, "trial DMs need coherent = 1");
        if (prm->dm != 0.0) return fail(B2F_EINVAL, "trial DMs are given in dm_trials: dm must be 0");
        for (int k = 0; k < prm->ndm; ++k) {
            const double t = prm->dm_trials[k];
            if (!std::isfinite(t) || t < 0) return fail(B2F_EINVAL, "trial DMs must be finite and >= 0");
            if (k > 0 && !(t > prm->dm_trials[k - 1])) return fail(B2F_EINVAL, "trial DMs must be strictly increasing");
        }
        dm = prm->dm_trials[prm->ndm - 1];
        if (!(dm > 0)) return fail(B2F_EINVAL, "the largest trial DM must be > 0");
    }
    int L = prm->freq_res > 0 ? prm->freq_res : (prm->nchan <= 128 ? 512 : 2 * prm->nchan);
    const int R = 2 * prm->nchan;
    if (!is_pow2(R) || R < 16 || R > 8192) return fail(B2F_EUNSUPPORTED, "nchan must be a power of two in 8..4096");
    const bool dedisp = prm->coherent && dm > 0.0;
    // the longest transform: 4096 points, or with dedispersion as many as keep a block at 2^20 points (nchan 8..64)
    const int long_cap = std::max(4096, (1 << 20) / R);
    // overlap-save samples discarded at each end of a block and channel: half the smearing across the lowest channel of
    // the lowest subband (8.3 us DM dnu/nu_GHz^3, the rule of submit_job.py:62) plus 10 %, rounded up to a multiple of the
    // integration factor so that every block yields whole output samples
    auto nfilt_half = [&](int Dint) {
        const double bw0 = std::fabs(prm->bw_mhz[0]);
        double fmin = 1e30;
        for (int i = 0; i < prm->nif; ++i) fmin = std::min(fmin, prm->freq_mhz[i] - bw0 / 2 + bw0 / prm->nchan / 2);
        const double ns = 8.3 * dm * (bw0 / prm->nchan) / std::pow(fmin / 1000.0, 3) / ((double)prm->nchan / bw0);
        int nf = (int)std::ceil(0.55 * ns);
        nf = (nf + Dint - 1) / Dint * Dint;
        return nf < Dint ? Dint : nf;
    };
    if (dedisp && prm->freq_res <= 0 && std::fabs(prm->bw_mhz[0]) > 0 && prm->nif >= 1 && prm->nif <= B2F_MAX_IF) {
        // digifil -F nchan:D lets the dedispersion kernel choose the transform length (SURVEY D5: the next power of two
        // >= 4 nfilt, at least the reference rule's length).  The rule's length is kept whenever the smearing fits it.
        int D0 = (prm->tscrunch < 1 ? 1 : prm->tscrunch) & -(prm->tscrunch < 1 ? 1 : prm->tscrunch);
        while (D0 > 128) D0 >>= 1;
        const int nf = nfilt_half(D0);
        if (2 * nf >= L) {
            while (L < 8 * nf && L < 4096) L *= 2;
            // where 4096 points do not hold the smearing: the long-transform path, up to 2^20 points per block
            if (2 * nf >= L) while (L < 8 * nf && L < long_cap) L *= 2;
            if (2 * nf >= L)
                return fail(B2F_EUNSUPPORTED, "dispersion smearing exceeds freq_res " + std::to_string(long_cap) + " channel samples at nchan " +
                                                  std::to_string(prm->nchan) + ": use more channels");
        }
    }
    if (!is_pow2(L) || L < 16 || L > 65536) return fail(B2F_EUNSUPPORTED, "freq_res must be a power of two in 16..8192");
    // freq_res above 4096 (other than nchan 4096's square blocks): coherent dedispersion on the long-transform path only
    const bool longfft = L > 4096 && L != R;
    if (longfft && (!dedisp || L > long_cap))
        return fail(B2F_EUNSUPPORTED, "freq_res " + std::to_string(L) + " needs coherent dedispersion and at most 2^20 points per block: freq_res <= " +
                                          std::to_string(long_cap) + " at nchan " + std::to_string(prm->nchan));
    if ((R > 4096 || L > 4096) && L != R && !longfft)
        return fail(B2F_EUNSUPPORTED, "nchan 4096 needs freq_res = 2 nchan (digifil -F nchan:2*nchan, process_vdif.py:162)");
    const bool generic = !(L == kL && R <= 512);        // tuned kernels: 512-point columns, rows up to 512
    const int D_user = prm->tscrunch < 1 ? 1 : prm->tscrunch;
    if (D_user > (1 << 20)) return fail(B2F_EUNSUPPORTED, "tscrunch above 2^20");
    int D = D_user & -D_user;                       // what the kernels integrate; kd_sum_rows adds tsq = D_user / D of their rows
    while (D > L) D >>= 1;
    if (dedisp) while (D > 128) D >>= 1;
    const int tsq = D_user / D;
    if (prm->header_bytes != 32 && prm->header_bytes != 16) return fail(B2F_EINVAL, "header_bytes must be 32 or 16");
    const int payload = prm->frame_bytes - prm->header_bytes;
    if (payload <= 0 || payload % 8) return fail(B2F_EINVAL, "frame_bytes");
    if ((dedisp || generic) && prm->in_nbit == 8 && payload % 32)
        return fail(B2F_EUNSUPPORTED, "8-bit input with coherent dedispersion, freq_res != 512 or nchan > 256 needs a payload that is a multiple of 32 bytes");
    if (dedisp && generic && !longfft && (R > 4096 || L > 4096))
        return fail(B2F_EUNSUPPORTED, "coherent dedispersion needs nchan <= 2048 and freq_res <= 4096 in this build");
    const double abw = std::fabs(prm->bw_mhz[0]);
    if (abw <= 0) return fail(B2F_EINVAL, "bw_mhz");
    for (int i = 0; i < prm->nif; ++i) {
        if (std::fabs(std::fabs(prm->bw_mhz[i]) - abw) > 1e-9) return fail(B2F_EINVAL, "all IFs must share |bw|");
        if (prm->if_order[i] < 0 || prm->if_order[i] >= prm->nif) return fail(B2F_EINVAL, "if_order");
    }
    if (prm->decode_mode != B2F_DECODE_STATIC && prm->decode_mode != B2F_DECODE_JA98) return fail(B2F_EINVAL, "decode_mode");
    if (prm->decode_mode == B2F_DECODE_JA98 && prm->in_nbit != 2) return fail(B2F_EINVAL, "decode_mode JA98 is a 2-bit unpacker");
    if (prm->rescale_mode != B2F_RESCALE_CONSTANT && prm->rescale_mode != B2F_RESCALE_RUNNING) return fail(B2F_EINVAL, "rescale_mode");
    if (prm->digi_sigma < 0) return fail(B2F_EINVAL, "digi_sigma");
    const int W = prm->raw_word_bits;
    if (W != 0 && W != 16 && W != 32 && W != 64) return fail(B2F_EINVAL, "raw_word_bits must be 0, 16, 32 or 64");
    if (W && prm->in_nbit != 2 && prm->in_nbit != 1) return fail(B2F_EUNSUPPORTED, "raw multi-BBC input must be 1- or 2-bit");
    if (prm->reserved0) return fail(B2F_EINVAL, "reserved0 must be 0");
    if (prm->raw_format != B2F_RAW_VDIF && prm->raw_format != B2F_RAW_MARK5B) return fail(B2F_EINVAL, "raw_format");
    if (W && prm->raw_format == B2F_RAW_MARK5B && prm->header_bytes != 16) return fail(B2F_EINVAL, "Mark5B frames have a 16-byte header");
    // whole groups of 4 words per payload; 64-bit words may end on a group of 2 (Mark5B: 1250 words in 10000 bytes)
    if (W && (prm->frame_bytes % 16 || payload % (W == 64 ? 16 : W / 2))) return fail(B2F_EUNSUPPORTED, "raw frame size");
    if (W) for (int i = 0; i < prm->nif; ++i) for (int k = 0; k < 4; ++k)
        if (prm->raw_bits[i][k] >= W) return fail(B2F_EINVAL, "raw_bits entry outside the word");
    const int64_t spf = W ? (int64_t)payload * 8 / W : (int64_t)payload * 8 / (prm->in_nbit * 2);
    const double fps_d = 2.0 * abw * 1e6 / (double)spf;
    const int64_t fps = (int64_t)llround(fps_d);
    if (std::fabs(fps_d - (double)fps) > 1e-6) return fail(B2F_EINVAL, "frames per second is not an integer");
    if (nprod * prm->nchan % 4 || (prm->out_nbit == 2 && (int64_t)prm->nif * nprod * prm->nchan % 4))
        return fail(B2F_EINVAL, "row size");
    // digifil -K: inter-channel delays [trial][if][chan] in channel samples (b2f.h), refused here before any device call
    if (prm->remove_delays != 0 && prm->remove_delays != 1) return fail(B2F_EINVAL, "remove_delays must be 0 or 1");
    if (!prm->remove_delays && prm->delay_ref_mhz != 0.0) return fail(B2F_EINVAL, "delay_ref_mhz needs remove_delays = 1");
    std::vector<int64_t> dl_table;
    int64_t dl_max = 0;
    if (prm->remove_delays) {
        if (!std::isfinite(prm->dm) || prm->dm < 0) return fail(B2F_EINVAL, "remove_delays needs a finite dm >= 0");
        double top = -1e300, bottom = 1e300;
        for (int i = 0; i < prm->nif; ++i) {
            top = std::max(top, prm->freq_mhz[i] + abw / 2 - abw / (2.0 * prm->nchan));
            bottom = std::min(bottom, prm->freq_mhz[i] - abw / 2 + abw / (2.0 * prm->nchan));
        }
        if (!(bottom > 0)) return fail(B2F_EINVAL, "remove_delays needs every channel centre above 0 MHz");
        if (!std::isfinite(prm->delay_ref_mhz) || (prm->delay_ref_mhz != 0.0 && prm->delay_ref_mhz < top - 1e-9))
            return fail(B2F_EINVAL, "delay_ref_mhz must be 0 (the plan's highest channel centre, " + std::to_string(top) +
                                        " MHz) or a finite frequency at least that high");
        const double ref = prm->delay_ref_mhz != 0.0 ? prm->delay_ref_mhz : top;
        const double tsamp0 = prm->nchan / (abw * 1e6);
        const int nd = std::max(1, prm->ndm);
        dl_table.resize((size_t)nd * prm->nif * prm->nchan);
        for (int t = 0; t < nd; ++t) {
            const double dmt = prm->ndm > 0 ? prm->dm_trials[t] : prm->dm;
            for (int i = 0; i < prm->nif; ++i) {
                const double bw = prm->bw_mhz[i];
                for (int c = 0; c < prm->nchan; ++c) {
                    const double fc = prm->freq_mhz[i] - bw / 2 + (c + 0.5) * bw / prm->nchan;
                    const double v = (1.0 / 2.41e-4) * dmt * (1.0 / (fc * fc) - 1.0 / (ref * ref)) / tsamp0;
                    if (!(v < 1e15)) return fail(B2F_EINVAL, "inter-channel delay beyond 1e15 channel samples");
                    const int64_t d = std::max<int64_t>(0, llround(v));
                    dl_table[((size_t)t * prm->nif + i) * prm->nchan + c] = d;
                    dl_max = std::max(dl_max, d);
                }
            }
        }
    }
    const bool delays = dl_max > 0;          // all delays 0 (DM 0): exactly the plan without remove_delays

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(B2F_ECUDA, "no CUDA device: libb2f has no CPU fallback");
    }
    if (prm->device < 0 || prm->device >= ndev) return fail(B2F_EINVAL, "device ordinal");
    CU(cudaSetDevice(prm->device));

    b2f_plan* pl = new b2f_plan();
    pl->prm = *prm;
    pl->prm.freq_res = L;
    pl->prm.tscrunch = D_user;
    pl->tsq = tsq;
    pl->R = R; pl->N = prm->nchan; pl->L = L; pl->D = D; pl->nprod = nprod;
    pl->nstrips = R / kStripCols;
    pl->M = (int64_t)R * L;
    pl->spf = spf; pl->fps = fps; pl->payload = payload;
    pl->groups_per_slot = (payload + 31) / 32;
    pl->dedisp = dedisp;
    pl->generic = generic;
    pl->longfft = longfft;
    pl->carry_mode = dedisp || generic;
    pl->bps = (!W && prm->in_nbit == 8) ? 2 : 1;
    pl->smask = pl->carry_mode && pl->bps == 2;
    pl->step = pl->M;
    pl->keep = L;
    if (dedisp) {
        // smearing across the lowest channel of the lowest subband (8.3 us DM dnu/nu_GHz^3, the rule of
        // submit_job.py:62), half of it on each side plus 10 %, rounded up to a multiple of tscrunch so
        // that every block yields whole output samples
        const int nf = nfilt_half(D);
        if (2 * nf >= L) {
            delete pl;
            return fail(B2F_EUNSUPPORTED, "dispersion smearing exceeds freq_res channel samples (freq_res up to " + std::to_string(long_cap) + " at nchan " +
                                              std::to_string(prm->nchan) + ")");
        }
        pl->nfilt_pos = pl->nfilt_neg = nf;
        pl->keep = L - 2 * nf;
        pl->step = (int64_t)pl->keep * R;
    }
    const int64_t g = std::gcd(pl->spf, pl->step);
    pl->unit_frames = pl->step / g;
    pl->unit_blocks = pl->spf / g;
    // default push: about 2048 frames per IF (0.5 s at 32 MHz) -- fewer, longer launches (C2: 352x real time at
    // 1024 frames, 369x at 2048, 377x at 4096) -- as long as the [blocks][L][R] intermediate stays under 4 GiB
    int cu = prm->chunk_units > 0 ? prm->chunk_units : (int)std::max<int64_t>(1, 2048 / pl->unit_frames);
    if (prm->chunk_units <= 0 && !dedisp) {
        const int64_t unit_bytes = (int64_t)prm->nif * pl->unit_blocks * L * R * (int64_t)sizeof(float2);
        cu = (int)std::max<int64_t>(1, std::min<int64_t>(cu, (4ll << 30) / std::max<int64_t>(unit_bytes, 1)));
    }
    if (dedisp && prm->chunk_units <= 0) {
        // the three-kernel dedispersion path holds two [blocks][512][R] buffers: pushes of about 4096 frames per IF (C4, 20 s:
        // 139.8 ms at 1024 frames, 134.9 at 2048, 134.0 at 4096; profiles/r02_c4_push_size_sweep.jsonl) as long as each buffer
        // stays under 8 GiB.
        const int64_t unit_bytes = (int64_t)prm->nif * (pl->unit_blocks + 1) * L * R * (int64_t)sizeof(float2);
        cu = (int)std::max<int64_t>(1, std::min<int64_t>(4096 / pl->unit_frames, (8ll << 30) / std::max<int64_t>(unit_bytes, 1)));
    }
    if (generic) {                 // blocks span seconds: pushes are plain 1024-frame pieces, the carry does the rest
        pl->unit_frames = 1;
        pl->unit_blocks = 0;
        cu = prm->chunk_units > 0 ? prm->chunk_units : 1024;
    }
    pl->chunk_frames = pl->unit_frames * cu;
    pl->chunk_blocks = pl->unit_blocks * cu;
    if (generic) pl->chunk_blocks = pl->chunk_frames * pl->spf / pl->step;
    if (pl->carry_mode) pl->chunk_blocks += 1;                 // carried samples can complete one more block
    pl->chunk_rows = pl->chunk_blocks * pl->keep / D;
    if (tsq > 1) pl->chunk_rows = pl->chunk_rows / tsq + 1;       // a push can complete one more output sample than its share
    pl->dl_host = dl_table;
    if (delays) {
        // the geometry above is the plain plan's; only the kernels' integration factor changes
        const int64_t P = pl->chunk_blocks * pl->keep;            // channel samples of one push at most
        pl->delays = true;
        pl->Du = D_user;
        pl->D = 1;
        pl->tsq = 1;
        pl->dl_max = dl_max;
        pl->dl_cap = dl_max + D_user - 1 + 2 * P;
        pl->chunk_rows = (P + D_user - 1) / D_user;               // held samples short of a row + one push
    }
    const double tsamp = (double)D_user * prm->nchan / (abw * 1e6);
    const double interval = prm->rescale_interval_s > 0 ? prm->rescale_interval_s : 10.0;
    pl->interval_rows = prm->keep_bandpass ? 0 : (int64_t)llround(interval / tsamp);
    pl->F_cap_rows = pl->interval_rows + 2 * pl->chunk_rows;
    pl->out_elem_bits = prm->out_nbit == -32 ? 32 : prm->out_nbit;
    pl->ndm = std::max(1, prm->ndm);
    pl->trial_row_elems = (int64_t)prm->nif * nprod * prm->nchan;
    pl->row_elems = pl->ndm * pl->trial_row_elems;
    pl->row_bytes = pl->row_elems * pl->out_elem_bits / 8;
    {
        // FFT blocks per column/row launch pair.  0 = the whole push.  L2-sized sub-batches (e.g. 72
        // blocks = 72 MiB) were measured SLOWER on B200: the per-block kernel cost is the same whether
        // or not the intermediate stays in L2, and every extra launch costs ~7 us (DESIGN.md section 5).
        const char* b = getenv("B2F_BATCH_BLOCKS");
        pl->batch_blocks = b ? atoll(b) : 0;
        if (!b && generic) pl->batch_blocks = std::max<int64_t>(1, (1ll << 30) / ((int64_t)L * R * (int64_t)sizeof(float2)));
    }

    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, prm->device) != cudaSuccess) { free_plan(pl); return fail(B2F_ECUDA, "device properties"); }
    pl->num_sms = prop.multiProcessorCount;
    {
        // Which channeliser.  Measured on B200 for C2 (20 s of 8 IF x 32 MHz, profiles/r02_bench_C2_20s_*.json): round-1
        // kernels 46.1 ms (column 31.1 + row 15.0); round-2 column kernel + tile row pass 42.8 (23.5 + 19.0 -> see DESIGN 5b);
        // fused kernel 60 with 6-12x less DRAM traffic (the intermediate stays in the L2 ring) -- its inter-warp ordering costs
        // more than the HBM round trip it saves.  So: nchan 128 (R = 256: C2, C3, C5) runs the round-2 column kernel and the
        // tile row pass (path 1); every other shape the round-1 kernels (path 0).  B2F_PATH=legacy|split|fused overrides where
        // the round-2 kernels apply (2-bit split streams, frames in order, 512-point columns, no dedispersion, products I /
        // coherence / IQUV); the JA98 decode exists only in the round-2 column kernel and selects it by itself.
        const bool eligible = !generic && !dedisp && prm->in_nbit == 2 && W == 0 && prm->frame_time_mode == B2F_FRAMES_POSITIONAL &&
                              payload % 16 == 0 && prm->frame_bytes % 16 == 0 && prop.cooperativeLaunch;
        const char* e = getenv("B2F_PATH");
        int want = R == 256 ? 1 : (prm->decode_mode == B2F_DECODE_JA98 ? 2 : 0);
        if (e && !strcmp(e, "legacy")) want = 0;
        else if (e && !strcmp(e, "split")) want = 1;
        else if (e && !strcmp(e, "fused")) want = 2;
        pl->path = eligible ? want : 0;
        // JA98 decode: the round-2 column kernel has its own implementation (levels per block from the frames); every other
        // kernel family (generic, round-1 tuned, dedispersion, raw input) reads levels per window of 512 samples of the
        // de-framed stream (kj_levels_stream).  Its windows count from the first carried sample of each push, so they are
        // the scan's windows only if blocks start on multiples of 512 samples.  That holds for every shape without
        // dedispersion (step = M = 512 R on the tuned path); with dedispersion the overlap-save step is keep R, which
        // at nchan 8..64 need not be a multiple of 512.
        if (prm->decode_mode == B2F_DECODE_JA98 && pl->step % 512) {
            delete pl;
            return fail(B2F_EUNSUPPORTED, "decode_mode JA98 needs FFT blocks that start on multiples of 512 samples");
        }
        if (pl->path) {
            int occ = 0;
            FParams dummy{};
            if (prm->decode_mode == B2F_DECODE_JA98) dummy.levels = reinterpret_cast<const float4*>(&dummy);   // selects the instantiation
            if (b2f_launch_kf(R, prm->pol_mode, dummy, 0, 0, nullptr, &occ) != cudaSuccess || occ < 1) {
                cudaGetLastError();
                pl->path = 0;            // JA98 with the other detection products: the round-1 column kernel with stream levels
            } else {
                const int npair = R / 2;                                   // warps per lane (one block per lane and round)
                pl->f_grid = pl->num_sms;                                  // one 16-warp CTA per SM
                pl->f_lanes = pl->f_grid * kFWarps / npair;
                if (pl->f_lanes < 1) pl->path = 0;
                pl->Dp = std::min(pl->D, 1024 / R);
            }
        }
    }

    auto bail = [&](int rc) { free_plan(pl); return rc; };
#define CUB(x)                                                                                      \
    do {                                                                                            \
        cudaError_t e__ = (x);                                                                      \
        if (e__ != cudaSuccess) {                                                                   \
            g_err = std::string(#x) + ": " + cudaGetErrorString(e__);                              \
            return bail(e__ == cudaErrorMemoryAllocation ? B2F_ENOMEM : B2F_ECUDA);                \
        }                                                                                           \
    } while (0)

    if (prm->stream) {
        pl->stream = (cudaStream_t)prm->stream;
    } else {
        CUB(cudaStreamCreateWithFlags(&pl->stream, cudaStreamNonBlocking));
        pl->own_stream = true;
    }
    CUB(cudaStreamCreateWithFlags(&pl->copy_stream, cudaStreamNonBlocking));
    CUB(cudaStreamCreateWithFlags(&pl->d2h_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        CUB(cudaEventCreateWithFlags(&pl->ev_stage_free[i], cudaEventDisableTiming));
        CUB(cudaEventCreateWithFlags(&pl->ev_h2d_done[i], cudaEventDisableTiming));
        CUB(cudaEventCreateWithFlags(&pl->ev_out_free[i], cudaEventDisableTiming));
        CUB(cudaEventCreateWithFlags(&pl->ev_kq_done[i], cudaEventDisableTiming));
    }
    const int nif = prm->nif;
    const int64_t nbt = (int64_t)nif * pl->chunk_blocks;
    const int nslot = pl->ndm * nif;                        // F / statistics slots: (trial, IF), trial-major
    pl->F_if_stride = pl->F_cap_rows * nprod * pl->N;
    if (pl->tsq > 1) pl->Fk_if_stride = (pl->chunk_blocks * pl->keep / D + tsq) * nprod * pl->N;
    if (pl->delays) pl->Fk_if_stride = pl->dl_cap * nprod * pl->N;
    if (prm->ndm > 0) {
        // what grows with the trials, and the two spectrum-sized buffers, against what the device has free
        const int64_t blocks = pl->batch_blocks > 0 ? std::min<int64_t>(pl->batch_blocks, nbt) : nbt;
        const double need = (double)nslot * ((pl->F_if_stride + pl->Fk_if_stride) * sizeof(float) +
                                             (double)nprod * pl->N * (kStatSplit * sizeof(double2) + 2 * sizeof(float)) +
                                             (double)L * pl->N * sizeof(float2)) +
                            2.0 * blocks * L * R * sizeof(float2);
        size_t fr = 0, tot = 0;
        CUB(cudaMemGetInfo(&fr, &tot));
        if (need > (double)fr) {
            g_err = "ndm = " + std::to_string(prm->ndm) + " trial DMs need " + std::to_string((int64_t)(need / (1 << 20))) + " MiB of device memory, " +
                    std::to_string((int64_t)(fr >> 20)) + " MiB are free: use fewer trials or a smaller chunk_units";
            return bail(B2F_ENOMEM);
        }
    }
    if (pl->delays) {
        const double hold = (double)nslot * pl->Fk_if_stride * sizeof(float);
        size_t fr = 0, tot = 0;
        CUB(cudaMemGetInfo(&fr, &tot));
        if (hold > (double)fr) {
            g_err = "remove_delays holds " + std::to_string((int64_t)hold) + " bytes of channel samples (d_max = " + std::to_string(dl_max) +
                    " samples plus two pushes, per trial and IF), " + std::to_string((int64_t)fr) +
                    " bytes are free: use fewer IFs or trials per plan, or a smaller chunk_units";
            return bail(B2F_ENOMEM);
        }
    }
    pl->slot_bytes = W ? (int)spf : (prm->in_nbit == 8 ? payload : (int)spf);         // 1- and 2-bit: one index byte per time sample
    pl->compact_stride = (size_t)((pl->chunk_frames * (int64_t)pl->slot_bytes + (pl->carry_mode ? pl->M * pl->bps : 0) + 255) / 256 * 256);
    pl->wmask_stride = (size_t)((pl->chunk_frames * pl->groups_per_slot + (pl->smask ? pl->M * pl->bps / 32 : 0) + 255) / 256 * 256);
    pl->fstat_stride = (size_t)((pl->chunk_frames + 255) / 256 * 256);
    if (!pl->path) {
        CUB(cudaMalloc(&pl->d_compact, pl->compact_stride * nif));
        CUB(cudaMalloc(&pl->d_wmask, pl->wmask_stride * nif));
        CUB(cudaMalloc(&pl->d_blkdirty, (size_t)nbt));
    } else {
        pl->tstream_stride = (size_t)((pl->chunk_blocks * pl->M + 255) / 256 * 256);
        pl->fillflag_stride = (size_t)((pl->chunk_frames + 63) / 64 * 64);
        CUB(cudaMalloc(&pl->d_tstream, pl->tstream_stride * nif));
        CUB(cudaMalloc(&pl->d_fillflag, pl->fillflag_stride * nif * sizeof(int)));
        CUB(cudaMalloc(&pl->d_fsync, ((size_t)pl->f_lanes + 1) * FS_STRIDE * sizeof(unsigned)));
        CUB(cudaMemset(pl->d_fsync, 0, ((size_t)pl->f_lanes + 1) * FS_STRIDE * sizeof(unsigned)));
        if (prm->decode_mode == B2F_DECODE_JA98) CUB(cudaMalloc(&pl->d_levels, (size_t)nbt * R * sizeof(float4)));
        if (getenv("B2F_FUSED_PROF")) {
            CUB(cudaMalloc(&pl->d_fprof, (size_t)pl->f_grid * kFWarps * 8 * sizeof(unsigned long long)));
            CUB(cudaMemset(pl->d_fprof, 0, (size_t)pl->f_grid * kFWarps * 8 * sizeof(unsigned long long)));
        }
        if (pl->Dp < pl->D && pl->path == 2) {
            pl->part_if_stride = pl->chunk_blocks * (L / pl->Dp) * nprod * pl->N;
            CUB(cudaMalloc(&pl->d_part, (size_t)pl->part_if_stride * nif * sizeof(float)));
        }
    }
    CUB(cudaMalloc(&pl->d_fstat, pl->fstat_stride * nif));
    int64_t inter_blocks = pl->batch_blocks > 0 ? std::min<int64_t>(pl->batch_blocks, nbt) : nbt;
    if (pl->path == 2) inter_blocks = (int64_t)pl->f_lanes * pl->f_nslot;         // the ring: it lives in L2
    CUB(cudaMalloc(&pl->d_inter, (size_t)inter_blocks * L * R * sizeof(float2)));
    CUB(cudaMalloc(&pl->d_colsum, (size_t)nbt * R * sizeof(float2)));
    CUB(cudaMalloc(&pl->d_eps, (size_t)nbt * pl->N * sizeof(float2)));
    CUB(cudaMalloc(&pl->d_F, (size_t)pl->F_if_stride * nslot * sizeof(float)));
    if (pl->tsq > 1 || pl->delays) CUB(cudaMalloc(&pl->d_Fk, (size_t)pl->Fk_if_stride * nslot * sizeof(float)));
    if (pl->delays) {
        CUB(cudaMalloc(&pl->d_delays, dl_table.size() * sizeof(int64_t)));
        CUB(cudaMemcpy(pl->d_delays, dl_table.data(), dl_table.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
    }
    CUB(cudaMalloc(&pl->d_mean, (size_t)nslot * nprod * pl->N * sizeof(float)));
    CUB(cudaMalloc(&pl->d_scale, (size_t)nslot * nprod * pl->N * sizeof(float)));
    CUB(cudaMalloc(&pl->d_partial, (size_t)nslot * kStatSplit * nprod * pl->N * sizeof(double2)));
    CUB(cudaMalloc(&pl->d_counters, C_COUNT * sizeof(unsigned long long)));
    if (pl->carry_mode) CUB(cudaMalloc(&pl->d_carry, (size_t)pl->M * pl->bps * nif));
    if (pl->smask) CUB(cudaMalloc(&pl->d_carry_mask, (size_t)pl->M * pl->bps / 32 * nif));
    if (prm->decode_mode == B2F_DECODE_JA98 && (generic || pl->path == 0)) {
        pl->levels_stride = (pl->chunk_frames * pl->spf + pl->M) / 512 + 2;
        CUB(cudaMalloc(&pl->d_levels_stream, (size_t)pl->levels_stride * nif * sizeof(float4)));
    }
    if (generic && L == R && L >= 1024) {
        // the shapes process_vdif.py:162 produces (-F nchan:2*nchan): kernels with compile-time geometry
        const char* e = getenv("B2F_GENERIC");
        const int lg = 31 - __builtin_clz(L);
        if (!(e && !strcmp(e, "runtime") && L <= 4096)) {
            int cc = 0, rc2 = 0;
            if (b2f_launch_kgt_col(lg, prm->decode_mode == B2F_DECODE_JA98 ? 22 : prm->in_nbit, KGParams{}, 0, nullptr, &cc) != cudaSuccess || cc < 1 ||
                b2f_launch_kgt_row(lg, prm->pol_mode, KGParams{}, 0, nullptr, &rc2) != cudaSuccess || rc2 < 1) {
                cudaGetLastError();
                if (L > 4096) { g_err = "generic kernels for nchan 4096 do not fit this device"; return bail(B2F_EUNSUPPORTED); }
            } else {
                pl->kgt_lg = lg;
                pl->kgt_col_ctas = cc; pl->kgt_row_ctas = rc2;
                b2f_kgt_geometry(lg, &pl->kgt_cols, &pl->kgt_rb);
            }
        }
    }
    if (generic && !longfft) {
        auto pass_tables = [](int len) {                 // layout of kg_tw_offset: per outer pass, [q - 1][lo]
            std::vector<float2> t((size_t)len, make_float2(1.f, 0.f));
            const int lg = 31 - __builtin_clz(len);
            for (int f = 0; f < kg_outer_passes(lg); ++f) {
                const int n = len >> (4 * f), m = n / 16, off = kg_tw_offset(lg, f);
                for (int q = 1; q < 16; ++q)
                    for (int lo = 0; lo < m; ++lo) {
                        const double ph = -2.0 * M_PI * (double)lo * q / n;
                        t[(size_t)off + (size_t)(q - 1) * m + lo] = make_float2((float)cos(ph), (float)sin(ph));
                    }
            }
            return t;
        };
        std::vector<float2> tc = pass_tables(L), tr = pass_tables(R);
        CUB(cudaMalloc(&pl->d_tw_col, tc.size() * sizeof(float2)));
        CUB(cudaMalloc(&pl->d_tw_row, tr.size() * sizeof(float2)));
        CUB(cudaMemcpy(pl->d_tw_col, tc.data(), tc.size() * sizeof(float2), cudaMemcpyHostToDevice));
        CUB(cudaMemcpy(pl->d_tw_row, tr.data(), tr.size() * sizeof(float2), cudaMemcpyHostToDevice));
    }
    if (dedisp) {
        CUB(cudaMalloc(&pl->d_spec, (size_t)inter_blocks * L * R * sizeof(float2)));
        // chirp H[trial][if][k2][c] = exp(-i 2 pi D DM 1e6 f^2 / (fc^2 (fc + f))), conjugated for LSB, in double
        std::vector<float2> h((size_t)nslot * L * prm->nchan);
        for (int t = 0; t < pl->ndm; ++t) {
            const double dmt = prm->ndm > 0 ? prm->dm_trials[t] : prm->dm;
            for (int i = 0; i < nif; ++i) {
                const double bw = prm->bw_mhz[i], chbw = bw / prm->nchan;
                for (int c = 0; c < prm->nchan; ++c) {
                    const double fc = prm->freq_mhz[i] - bw / 2 + (c + 0.5) * chbw;
                    for (int k2 = 0; k2 < L; ++k2) {
                        const double f = ((double)k2 / L - 0.5) * chbw;
                        double ph = 2.0 * M_PI * (1.0 / 2.41e-4) * 1e6 * dmt * f * f / (fc * fc * (fc + f));
                        if (bw < 0) ph = -ph;
                        h[(((size_t)t * nif + i) * L + k2) * prm->nchan + c] = make_float2((float)cos(ph), (float)-sin(ph));
                    }
                }
            }
        }
        CUB(cudaMalloc(&pl->d_chirp, h.size() * sizeof(float2)));
        CUB(cudaMemcpy(pl->d_chirp, h.data(), h.size() * sizeof(float2), cudaMemcpyHostToDevice));
    }
#undef CUB
    int rc = upload_tables(pl);
    if (rc) return bail(rc);
    rc = init_state(pl);
    if (rc) return bail(rc);
    *out = pl;
    return 0;
}

int b2f_plan_destroy(b2f_plan* pl) {
    free_plan(pl);
    return 0;
}

int b2f_get_geometry(const b2f_plan* pl, b2f_geometry* g) {
    if (!pl || !g) return fail(B2F_EINVAL, "null argument");
    g->unit_frames = pl->unit_frames;
    g->unit_blocks = pl->unit_blocks;
    g->chunk_frames = pl->chunk_frames;
    g->chunk_rows = pl->chunk_rows;
    g->block_samples = pl->M;
    g->samples_per_frame = pl->spf;
    g->row_bytes = pl->row_bytes;
    g->nprod = pl->nprod;
    g->freq_res = pl->L;
    g->tsamp_s = (double)pl->prm.tscrunch * pl->N / (std::fabs(pl->prm.bw_mhz[0]) * 1e6);
    g->unit_blocks = pl->unit_blocks;
    g->interval_rows = pl->interval_rows;
    g->nfilt_pos = pl->nfilt_pos;
    g->nfilt_neg = pl->nfilt_neg;
    g->ndm = pl->ndm;
    g->trial_row_bytes = pl->trial_row_elems * pl->out_elem_bits / 8;
    return 0;
}

int b2f_reset(b2f_plan* pl) {
    if (!pl) return fail(B2F_EINVAL, "null plan");
    CU(cudaSetDevice(pl->prm.device));
    CU(cudaStreamSynchronize(pl->stream));
    CU(cudaStreamSynchronize(pl->copy_stream));
    CU(cudaStreamSynchronize(pl->d2h_stream));
    return init_state(pl);
}

int b2f_push(b2f_plan* pl, const void* const* frames, int64_t nframes, int on_device) {
    if (!pl || !frames) return fail(B2F_EINVAL, "null argument");
    if (nframes < 0 || nframes > pl->chunk_frames) return fail(B2F_EINVAL, "nframes exceeds chunk_frames");
    if (pl->flushed) return fail(B2F_ESTATE, "push after flush; call b2f_reset for a new scan");
    CU(cudaSetDevice(pl->prm.device));
    const int nif = pl->prm.nif;
    const int64_t T = pl->carry_len + nframes * pl->spf;          // samples available per IF (carry + new)
    const int64_t nblk = pl->carry_mode ? (T >= pl->M ? (T - pl->M) / pl->step + 1 : 0) : nframes * pl->spf / pl->M;
    const int64_t krows = nblk * pl->keep / pl->D;                     // rows the kernels write
    int64_t rows = pl->tsq > 1 ? (pl->fk_pending + krows) / pl->tsq : krows;
    if (pl->delays) rows = pl->dl_held + krows >= pl->dl_max ? (pl->dl_held + krows - pl->dl_max) / pl->Du : 0;   // tail dropped
    if (nblk == 0 && !pl->carry_mode) return 0;
    if (pl->rows_off + pl->rows_held + rows > pl->F_cap_rows && pl->rows_off > 0 && pl->rows_held + rows <= pl->F_cap_rows) {
        // running rescale keeps the rows of an unfinished interval: move them to the front of the buffer, in pieces no
        // longer than the gap so that source and destination of one copy never overlap
        const int64_t ncolF = (int64_t)pl->nprod * pl->N;
        for (int i = 0; i < pl->ndm * pl->prm.nif; ++i)
            for (int64_t r0 = 0; r0 < pl->rows_held; r0 += pl->rows_off) {
                const int64_t n = std::min(pl->rows_off, pl->rows_held - r0);
                float* base = pl->d_F + i * pl->F_if_stride;
                CU(cudaMemcpyAsync(base + r0 * ncolF, base + (pl->rows_off + r0) * ncolF, (size_t)n * ncolF * sizeof(float),
                                   cudaMemcpyDeviceToDevice, pl->stream));
            }
        pl->rows_off = 0;
    }
    if (pl->rows_off + pl->rows_held + rows > pl->F_cap_rows)
        return fail(B2F_ESTATE, "row buffer full: call b2f_pull before pushing more");
    if (int rcd = delay_place(pl, krows)) return rcd;
    const size_t fbytes = (size_t)nframes * pl->prm.frame_bytes;

    if (!pl->have_base) {
        for (int i = 0; i < (pl->prm.raw_word_bits ? 1 : nif); ++i) {
            uint32_t w[4];
            if (on_device) CU(cudaMemcpy(w, frames[i], 16, cudaMemcpyDeviceToHost));
            else memcpy(w, frames[i], 16);
            if (pl->prm.raw_word_bits && pl->prm.raw_format == B2F_RAW_MARK5B) {
                pl->base_sec0[i] = mark5b_seconds(w[2]);
                pl->base_fnum0[i] = w[1] & 0x7FFFu;
            } else {
                pl->base_sec0[i] = w[0] & 0x3FFFFFFFu;
                pl->base_fnum0[i] = w[1] & 0xFFFFFFu;
            }
        }
        pl->have_base = true;
    }

    K0Params k0{};
    if (on_device) {
        for (int i = 0; i < (pl->prm.raw_word_bits ? 1 : nif); ++i) k0.frames[i] = static_cast<const uint8_t*>(frames[i]);
    } else {
        const int idx = pl->stage_idx;
        if (!pl->d_stage[idx]) {
            pl->stage_if_stride = (size_t)((pl->chunk_frames * pl->prm.frame_bytes + 255) / 256 * 256);
            CU(cudaMalloc(&pl->d_stage[idx], pl->stage_if_stride * nif));
        }
        CU(cudaStreamWaitEvent(pl->copy_stream, pl->ev_stage_free[idx], 0));
        const int nstreams = pl->prm.raw_word_bits ? 1 : nif;
        for (int i = 0; i < nstreams; ++i) {
            CU(cudaMemcpyAsync(pl->d_stage[idx] + i * pl->stage_if_stride, frames[i], fbytes, cudaMemcpyHostToDevice,
                               pl->copy_stream));
            k0.frames[i] = pl->d_stage[idx] + i * pl->stage_if_stride;
        }
        CU(cudaEventRecord(pl->ev_h2d_done[idx], pl->copy_stream));
        CU(cudaStreamWaitEvent(pl->stream, pl->ev_h2d_done[idx], 0));
    }

    // ---- kernel 1: validate + de-frame
    k0.compact = pl->d_compact + pl->carry_len * pl->bps; k0.compact_stride = pl->compact_stride;   // carried halo sits in front
    k0.wmask = pl->d_wmask + (pl->smask ? pl->carry_len * pl->bps / 32 : 0); k0.wmask_stride = pl->wmask_stride;
    k0.fstat = pl->d_fstat; k0.fstat_stride = pl->fstat_stride;
    k0.counters = pl->d_counters;
    k0.nframes = nframes; k0.nslots = nframes;
    k0.frame_bytes = pl->prm.frame_bytes; k0.header_bytes = pl->prm.header_bytes;
    k0.payload_bytes = (int)pl->payload; k0.groups_per_slot = (int)pl->groups_per_slot;
    k0.slot_bytes = pl->slot_bytes;
    k0.in_nbit = pl->prm.in_nbit; k0.time_mode = pl->prm.frame_time_mode; k0.mask_faults = pl->prm.mask_faults;
    k0.fps = (int)pl->fps;
    for (int i = 0; i < nif; ++i) {
        const int64_t tot = (int64_t)pl->base_fnum0[i] + pl->frames_pushed;
        k0.base_sec[i] = pl->base_sec0[i] + (uint32_t)(tot / pl->fps);
        k0.base_fnum[i] = (uint32_t)(tot % pl->fps);
    }
    if (pl->carry_mode && pl->carry_len) {
        for (int i = 0; i < nif; ++i)
            CU(cudaMemcpyAsync(pl->d_compact + i * pl->compact_stride, pl->d_carry + (size_t)i * pl->M * pl->bps, (size_t)pl->carry_len * pl->bps,
                               cudaMemcpyDeviceToDevice, pl->stream));
        if (pl->smask)
            for (int i = 0; i < nif; ++i)
                CU(cudaMemcpyAsync(pl->d_wmask + i * pl->wmask_stride, pl->d_carry_mask + (size_t)i * (pl->M * pl->bps / 32),
                                   (size_t)(pl->carry_len * pl->bps / 32), cudaMemcpyDeviceToDevice, pl->stream));
    }
    int rc = 0;
    if (pl->path) {
        rc = push_fused(pl, k0, nframes, nblk);
        if (rc) return rc;
        if (!on_device) {
            CU(cudaEventRecord(pl->ev_stage_free[pl->stage_idx], pl->stream));
            pl->stage_idx ^= 1;
        }
        rc = pl->delays ? delay_sum(pl, krows, rows) : sum_rows(pl, krows, rows);
        if (rc) return rc;
        pl->rows_held += rows;
        pl->rows_produced += rows;
        pl->frames_pushed += nframes;
        pl->last_nblk = nblk;
        pl->last_nframes = nframes;
        return 0;
    }
    CU(cudaMemsetAsync(pl->d_fstat, 0, pl->fstat_stride * nif, pl->stream));
    if (nblk > 0) CU(cudaMemsetAsync(pl->d_blkdirty, 0, (size_t)nif * nblk, pl->stream));
    if (pl->prm.raw_word_bits) {                      // corner turn + validation in one pass over the raw stream
        K0RParams kr{};
        kr.frames = k0.frames[0];
        kr.compact = k0.compact; kr.compact_stride = pl->compact_stride;
        kr.fstat = pl->d_fstat; kr.fstat_stride = pl->fstat_stride; kr.counters = pl->d_counters;
        kr.nframes = nframes; kr.nslots = nframes;
        kr.frame_bytes = pl->prm.frame_bytes; kr.header_bytes = pl->prm.header_bytes; kr.payload_bytes = (int)pl->payload;
        kr.word_bits = pl->prm.raw_word_bits; kr.nif = nif; kr.time_mode = pl->prm.frame_time_mode;
        kr.mask_faults = pl->prm.mask_faults; kr.fps = (int)pl->fps; kr.slot_bytes = pl->slot_bytes;
        kr.base_sec = k0.base_sec[0]; kr.base_fnum = k0.base_fnum[0]; kr.format = pl->prm.raw_format; kr.sample_bits = pl->prm.in_nbit;
        for (int i = 0; i < nif; ++i) for (int k = 0; k < 4; ++k) kr.bit[i][k] = pl->prm.raw_bits[i][k];
        if (reinterpret_cast<uintptr_t>(kr.frames) & 15) return fail(B2F_EINVAL, "raw frames must be 16-byte aligned");
        const int stage_bytes = (kr.frame_bytes + 127) & ~127;
        const size_t smem = 128 + (size_t)kK0Stages * stage_bytes;
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(nframes, 4 * pl->num_sms));
        rc = timed(pl, B2F_K_VALIDATE, [&] {
            if (kr.word_bits == 16) {
                cudaFuncSetAttribute(k0r_corner_turn<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                k0r_corner_turn<16><<<grid, kK0Threads, smem, pl->stream>>>(kr);
            } else if (kr.word_bits == 32) {
                cudaFuncSetAttribute(k0r_corner_turn<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                k0r_corner_turn<32><<<grid, kK0Threads, smem, pl->stream>>>(kr);
            } else {
                cudaFuncSetAttribute(k0r_corner_turn<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                k0r_corner_turn<64><<<grid, kK0Threads, smem, pl->stream>>>(kr);
            }
        });
    } else {
        rc = launch_k0(pl, k0, pl->stream, true);
    }
    if (rc) return rc;
    if (!on_device) {
        CU(cudaEventRecord(pl->ev_stage_free[pl->stage_idx], pl->stream));
        pl->stage_idx ^= 1;
    }
    {
        K0bParams kb{};
        kb.wmask = k0.wmask; kb.wmask_stride = pl->wmask_stride;
        kb.fstat = pl->d_fstat; kb.fstat_stride = pl->fstat_stride;
        kb.blkdirty = pl->d_blkdirty; kb.counters = pl->d_counters;
        kb.nslots = nframes; kb.nif = nif; kb.nblk = pl->carry_mode ? 0 : (int)nblk;
        kb.groups_per_slot = (int)pl->groups_per_slot; kb.samples_per_frame = (int)pl->spf;
        kb.block_samples = pl->M;
        kb.compact = k0.compact; kb.compact_stride = pl->compact_stride;
        kb.slot_bytes = pl->slot_bytes; kb.in_nbit = pl->prm.in_nbit;
        const int64_t n = nframes * nif;
        k0b_finish_slots<<<(unsigned)((n + 255) / 256), 256, 0, pl->stream>>>(kb);
        pl->launches++;
        CU(cudaGetLastError());
    }
    if (pl->carry_mode) {
        rc = push_dedisp(pl, nblk, T);
        if (rc) return rc;
    } else
    // ---- round-1 channeliser: the column pass writes the whole [nb][512][R] float2 intermediate to HBM and the row pass
    // streams it back (97 % of the step's DRAM traffic; L2-sized sub-batches were measured slower, see plan_create)
    {
        const int64_t nbt = (int64_t)nif * nblk;
        const int64_t NB = pl->batch_blocks > 0 ? std::min<int64_t>(pl->batch_blocks, nbt) : nbt;
        int TR, PT;
        kb_shape(pl->R, &TR, &PT);
        const int RW = 32 / TR;                                   // rows per warp pass
        const int GW = std::max(pl->D, RW);
        KAParams ka{};
        ka.compact = pl->d_compact; ka.compact_stride = pl->compact_stride;
        ka.wmask = pl->d_wmask; ka.wmask_stride = pl->wmask_stride;
        ka.blkdirty = pl->d_blkdirty;
        ka.inter = pl->d_inter; ka.colsum = pl->d_colsum;
        ka.tab_g = pl->d_tab_g; ka.tab_h = pl->d_tab_h; ka.tab_w = pl->d_tab_w; ka.tab_beta = pl->d_tab_beta;
        ka.R = pl->R; ka.nstrips = pl->nstrips; ka.nblk = (int)nblk; ka.nif = nif;
        ka.payload_bytes = (int)pl->payload; ka.groups_per_slot = (int)pl->groups_per_slot;
        ka.blk_step_bytes = pl->M * pl->bps;
        ka.in8_offset = pl->prm.in8_offset_mode ? 128.0f : 127.5f;
        ka.levels = pl->d_levels_stream; ka.levels_stride = pl->levels_stride;
        if (int rcl = stream_levels(pl, T)) return rcl;
        KBParams kb{};
        kb.inter = pl->d_inter; kb.eps = pl->d_eps; kb.tab_r = pl->d_tab_r;
        kb.F = row_dst(pl); kb.F_if_stride = row_dst_stride(pl);
        kb.row0 = row_dst_row0(pl);
        kb.nblk = (int)nblk; kb.nif = nif; kb.D = pl->D;
        for (int64_t b0 = 0; b0 < nbt; b0 += NB) {
            const int64_t nb = std::min(NB, nbt - b0);
            ka.gb_begin = b0; ka.gb_end = b0 + nb;
            const int64_t work = nb * pl->nstrips;
            int64_t grid = std::max<int64_t>(1, (kKACtasPerSM * pl->num_sms) / pl->nstrips) * pl->nstrips;
            grid = std::min<int64_t>(grid, work);
            rc = launch_ka(pl, false, ka, (unsigned)grid);
            if (rc) return rc;
            rc = timed(pl, B2F_K_EPS, [&] {
                ke_eps<<<(unsigned)nb, std::min(pl->R / 2, 512), pl->R * sizeof(float2), pl->stream>>>(pl->d_colsum + b0 * pl->R,
                                                                                       pl->d_eps + b0 * pl->N, pl->R);
            });
            if (rc) return rc;
            kb.gb_begin = b0; kb.gb_end = b0 + nb;
            const int64_t ngroups = nb * (kL / GW);
            const int64_t ctas = (ngroups + kKBThreads / 32 - 1) / (kKBThreads / 32);
            rc = launch_kb(pl, kb, (int)std::min<int64_t>(ctas, (int64_t)pl->num_sms * 2));
            if (rc) return rc;
        }
    }
    rc = pl->delays ? delay_sum(pl, krows, rows) : sum_rows(pl, krows, rows);
    if (rc) return rc;
    pl->rows_held += rows;
    pl->rows_produced += rows;
    pl->frames_pushed += nframes;
    pl->last_nblk = nblk;
    pl->last_nframes = nframes;
    return 0;
}

int b2f_flush(b2f_plan* pl) {
    if (!pl) return fail(B2F_EINVAL, "null plan");
    pl->flushed = true;
    return 0;
}

static int pull_impl(b2f_plan* pl, void* out, int64_t max_rows, int out_on_device, int64_t pitch_bytes, int64_t* nrows);

int b2f_pull(b2f_plan* pl, void* out, int64_t max_rows, int out_on_device, int64_t* nrows) {
    return pull_impl(pl, out, max_rows, out_on_device, 0, nrows);
}

int b2f_pull_strided(b2f_plan* pl, void* out, int64_t max_rows, int64_t row_pitch_bytes, int64_t* nrows) {
    if (pl && pl->prm.ndm > 0) return fail(B2F_EUNSUPPORTED, "b2f_pull_strided splices the tiles of one DM: not with trial DMs");
    if (pl && row_pitch_bytes < pl->row_bytes) return fail(B2F_EINVAL, "row pitch smaller than one output row");
    {
        // kq_quantise stores 4 output elements at a time: 4 bytes for 8-bit (1 byte for 2-bit), 8 for 16-bit, 16 for float
        const int align = !pl ? 4 : (pl->prm.out_nbit == 16 ? 8 : (pl->prm.out_nbit == -32 ? 16 : 4));
        if (row_pitch_bytes % align || (reinterpret_cast<uintptr_t>(out) % align))
            return fail(B2F_EINVAL, "row pitch and output pointer must be multiples of " + std::to_string(align) + " bytes for this nbit");
    }
    return pull_impl(pl, out, max_rows, 1, row_pitch_bytes, nrows);
}

static int pull_impl(b2f_plan* pl, void* out, int64_t max_rows, int out_on_device, int64_t pitch_bytes, int64_t* nrows) {
    if (!pl || !nrows) return fail(B2F_EINVAL, "null argument");
    *nrows = 0;
    CU(cudaSetDevice(pl->prm.device));
    const int nif = pl->prm.nif;
    const int ncol = pl->nprod * pl->N;
    if (!pl->stats_ready) {
        if (pl->rows_held >= pl->interval_rows || (pl->flushed && pl->rows_held > 0)) {
            const int64_t nstat = std::min(pl->rows_held, pl->interval_rows);
            int rc = timed(pl, B2F_K_STATS, [&] {
                dim3 g1((ncol + 127) / 128, pl->ndm * nif, kStatSplit);
                ks_partial<<<g1, 128, 0, pl->stream>>>(pl->d_F + pl->rows_off * ncol, pl->F_if_stride, nstat, ncol, pl->d_partial);
                dim3 g2((ncol + 127) / 128, pl->ndm * nif);
                ks_final<<<g2, 128, 0, pl->stream>>>(pl->d_partial, kStatSplit, nstat, ncol, pl->d_mean, pl->d_scale);
            });
            if (rc) return rc;
            pl->stats_ready = true;
            pl->rows_this_interval = nstat;
        } else {
            return 0;
        }
    }
    const bool running = pl->prm.rescale_mode == B2F_RESCALE_RUNNING && !pl->prm.keep_bandpass && !pl->preset_stats;
    int64_t n = std::min(pl->rows_held, max_rows);
    if (running) n = std::min(n, pl->rows_this_interval);       // the statistics in force cover only their own interval
    if (n <= 0) return 0;
    if (!out) return fail(B2F_EINVAL, "null output buffer");
    void* dst = out;
    const size_t bytes = (size_t)n * pl->row_bytes;
    const int oi = pl->out_idx;
    if (out_on_device != 1) {
        if (pl->out_stage_bytes[oi] < bytes) {
            CU(cudaStreamSynchronize(pl->d2h_stream));
            if (pl->d_out_stage[oi]) CU(cudaFree(pl->d_out_stage[oi]));
            pl->d_out_stage[oi] = nullptr;
            pl->out_stage_bytes[oi] = 0;
            CU(cudaMalloc(&pl->d_out_stage[oi], bytes));
            pl->out_stage_bytes[oi] = bytes;
        }
        dst = pl->d_out_stage[oi];
        CU(cudaStreamWaitEvent(pl->stream, pl->ev_out_free[oi], 0));
    }
    KQParams kq{};
    kq.F = pl->d_F + pl->rows_off * ncol; kq.F_if_stride = pl->F_if_stride;
    kq.mean = pl->d_mean; kq.scale = pl->d_scale; kq.out = dst;
    kq.rows = n; kq.out_row_elems = pl->row_elems;
    kq.out_pitch_bytes = pitch_bytes > 0 ? pitch_bytes : pl->row_bytes;
    kq.nif = nif; kq.nprod = pl->nprod; kq.nchan = pl->N; kq.out_nbit = pl->prm.out_nbit;
    kq.pol_major = pl->prm.splice_pol_major;
    kq.inv_digi_sigma = (float)(1.0 / (pl->prm.digi_sigma > 0 ? pl->prm.digi_sigma : 6.0));
    kq.trial_row_elems = (int)pl->trial_row_elems;
    for (int i = 0; i < nif; ++i) {
        kq.if_order[i] = pl->prm.if_order[i];
        kq.flip[i] = pl->prm.bw_mhz[i] > 0 ? 1 : 0;
    }
    const int64_t quads = n * (pl->row_elems / 4);
    int rc = timed(pl, B2F_K_QUANT, [&] { kq_quantise<<<(unsigned)((quads + 255) / 256), 256, 0, pl->stream>>>(kq); });
    if (rc) return rc;
    if (out_on_device != 1) {
        // device -> host on its own stream so the next chunk's kernels are not held up
        CU(cudaEventRecord(pl->ev_kq_done[oi], pl->stream));
        CU(cudaStreamWaitEvent(pl->d2h_stream, pl->ev_kq_done[oi], 0));
        CU(cudaMemcpyAsync(out, dst, bytes, cudaMemcpyDeviceToHost, pl->d2h_stream));
        CU(cudaEventRecord(pl->ev_out_free[oi], pl->d2h_stream));
        pl->out_idx ^= 1;
        if (out_on_device == 0) {
            CU(cudaStreamSynchronize(pl->d2h_stream));
            int rc2 = check_fused_abort(pl);
            if (rc2) return rc2;
        }
    }
    pl->rows_held -= n;
    pl->rows_emitted += n;
    pl->rows_off = pl->rows_held ? pl->rows_off + n : 0;
    if (running) {
        pl->rows_this_interval -= n;
        if (pl->rows_this_interval == 0) pl->stats_ready = false;     // the next interval measures itself
    }
    *nrows = n;
    return 0;
}

int b2f_sync(b2f_plan* pl) {
    if (!pl) return fail(B2F_EINVAL, "null plan");
    CU(cudaSetDevice(pl->prm.device));
    CU(cudaStreamSynchronize(pl->copy_stream));
    CU(cudaStreamSynchronize(pl->stream));
    CU(cudaStreamSynchronize(pl->d2h_stream));
    return check_fused_abort(pl);
}

int b2f_mark(b2f_plan* pl, int64_t* ticket) {
    if (!pl || !ticket) return fail(B2F_EINVAL, "null argument");
    CU(cudaSetDevice(pl->prm.device));
    const int slot = (int)(pl->marks_issued % b2f_plan::kMarks);
    cudaStream_t st[3] = {pl->copy_stream, pl->stream, pl->d2h_stream};
    for (int k = 0; k < 3; ++k) {
        if (!pl->ev_mark[slot][k]) CU(cudaEventCreateWithFlags(&pl->ev_mark[slot][k], cudaEventDisableTiming));
        CU(cudaEventRecord(pl->ev_mark[slot][k], st[k]));
    }
    *ticket = pl->marks_issued++;
    return 0;
}

int b2f_wait(b2f_plan* pl, int64_t ticket) {
    if (!pl) return fail(B2F_EINVAL, "null plan");
    if (ticket < 0 || ticket >= pl->marks_issued) return fail(B2F_EINVAL, "unknown ticket");
    if (pl->marks_issued - ticket > b2f_plan::kMarks)          // its events were re-recorded by a newer mark
        return fail(B2F_ESTATE, "ticket too old: at most 8 marks may be outstanding");
    CU(cudaSetDevice(pl->prm.device));
    const int slot = (int)(ticket % b2f_plan::kMarks);
    for (int k = 0; k < 3; ++k) CU(cudaEventSynchronize(pl->ev_mark[slot][k]));
    return 0;
}

int b2f_channeliser_path(const b2f_plan* pl) { return pl ? pl->path : B2F_EINVAL; }

int b2f_get_delays(const b2f_plan* pl, int64_t* out) {
    if (!pl || !out) return fail(B2F_EINVAL, "null argument");
    const size_t n = (size_t)pl->ndm * pl->prm.nif * pl->N;
    if (pl->dl_host.size() == n) std::copy(pl->dl_host.begin(), pl->dl_host.end(), out);
    else std::fill(out, out + n, (int64_t)0);
    return 0;
}

int b2f_get_params(const b2f_plan* pl, b2f_params* out) {
    if (!pl || !out) return fail(B2F_EINVAL, "null argument");
    *out = pl->prm;
    out->freq_res = pl->L;
    return 0;
}

int b2f_get_counters(b2f_plan* pl, b2f_counters* c) {
    if (!pl || !c) return fail(B2F_EINVAL, "null argument");
    CU(cudaSetDevice(pl->prm.device));
    unsigned long long h[C_COUNT];
    CU(cudaStreamSynchronize(pl->stream));
    { int rc = check_fused_abort(pl); if (rc) return rc; }
    CU(cudaMemcpy(h, pl->d_counters, sizeof(h), cudaMemcpyDeviceToHost));
    c->frames_ok = h[C_OK]; c->frames_invalid = h[C_INVALID]; c->frames_with_fill = h[C_FILLFRAMES];
    c->fill_words = h[C_FILLWORDS]; c->frames_dropped = h[C_DROPPED]; c->frames_misplaced = h[C_MISPLACED];
    c->frames_badhdr = h[C_BADHDR]; c->slots_missing = h[C_MISSING];
    c->rows_produced = pl->rows_produced; c->rows_emitted = pl->rows_emitted; c->blocks_dirty = h[C_DIRTY];
    c->kernel_launches = (uint64_t)pl->launches;
    c->rescale_frozen = pl->stats_ready ? 1 : 0;
    c->rescale_preset = pl->preset_stats ? 1 : 0;
    return 0;
}

int b2f_get_rescale(b2f_plan* pl, float* mean, float* scale) {
    if (!pl || !mean || !scale) return fail(B2F_EINVAL, "null argument");
    CU(cudaSetDevice(pl->prm.device));
    CU(cudaStreamSynchronize(pl->stream));
    const size_t n = (size_t)pl->ndm * pl->prm.nif * pl->nprod * pl->N * sizeof(float);
    CU(cudaMemcpy(mean, pl->d_mean, n, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(scale, pl->d_scale, n, cudaMemcpyDeviceToHost));
    return 0;
}

int b2f_set_rescale(b2f_plan* pl, const float* mean, const float* scale) {
    if (!pl) return fail(B2F_EINVAL, "null plan");
    if ((mean == nullptr) != (scale == nullptr)) return fail(B2F_EINVAL, "mean and scale must both be given or both be NULL");
    CU(cudaSetDevice(pl->prm.device));
    if (!mean) {
        pl->preset_stats = false;
        pl->stats_ready = pl->prm.keep_bandpass != 0;
        return 0;
    }
    const size_t n = (size_t)pl->ndm * pl->prm.nif * pl->nprod * pl->N * sizeof(float);
    CU(cudaStreamSynchronize(pl->stream));
    CU(cudaMemcpy(pl->d_mean, mean, n, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(pl->d_scale, scale, n, cudaMemcpyHostToDevice));
    pl->preset_stats = true;
    pl->stats_ready = true;
    return 0;
}

int b2f_kernel_time(b2f_plan* pl, int kid, double* ms, int64_t* launches) {
    if (!pl || kid < 0 || kid >= B2F_K_COUNT) return fail(B2F_EINVAL, "kernel id");
    CU(cudaSetDevice(pl->prm.device));
    int rc = collect_times(pl);
    if (rc) return rc;
    if (ms) *ms = pl->k_ms[kid];
    if (launches) *launches = pl->k_n[kid];
    return 0;
}

int b2f_reset_timers(b2f_plan* pl) {
    if (!pl) return fail(B2F_EINVAL, "null plan");
    CU(cudaSetDevice(pl->prm.device));
    int rc = collect_times(pl);
    if (rc) return rc;
    for (int i = 0; i < B2F_K_COUNT; ++i) { pl->k_ms[i] = 0; pl->k_n[i] = 0; }
    return 0;
}

int b2f_decode(const void* frames, int64_t nframes, int frame_bytes, int header_bytes, int in_nbit, int mask_faults,
               int in_on_device, float* out, int out_on_device, int device, b2f_counters* counters) {
    if (!frames || !out || nframes <= 0) return fail(B2F_EINVAL, "null argument");
    if (!(in_nbit == 1 || in_nbit == 2 || in_nbit == 8)) return fail(B2F_EUNSUPPORTED, "VDIF bits/sample must be 1, 2 or 8");
    const int payload = frame_bytes - header_bytes;
    if (payload <= 0 || payload % 8 || (header_bytes != 32 && header_bytes != 16)) return fail(B2F_EINVAL, "frame geometry");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(B2F_ECUDA, "no CUDA device: libb2f has no CPU fallback");
    }
    CU(cudaSetDevice(device));
    const int64_t spf = (int64_t)payload * 8 / (in_nbit * 2);
    const int64_t nsamp = nframes * spf;
    const int gps = (payload + 31) / 32;
    uint8_t *d_in = nullptr, *d_compact = nullptr, *d_wmask = nullptr, *d_fstat = nullptr, *d_dirty = nullptr;
    unsigned long long* d_cnt = nullptr;
    float* d_out = nullptr;
    int rc = 0;
    auto cleanup = [&] {
        if (d_in) cudaFree(d_in);
        if (d_compact) cudaFree(d_compact);
        if (d_wmask) cudaFree(d_wmask);
        if (d_fstat) cudaFree(d_fstat);
        if (d_dirty) cudaFree(d_dirty);
        if (d_cnt) cudaFree(d_cnt);
        if (d_out && !out_on_device) cudaFree(d_out);
    };
#define CUD(x)                                                                     \
    do {                                                                           \
        cudaError_t e__ = (x);                                                     \
        if (e__ != cudaSuccess) {                                                  \
            cleanup();                                                             \
            return fail(B2F_ECUDA, std::string(#x) + ": " + cudaGetErrorString(e__)); \
        }                                                                          \
    } while (0)
    const uint8_t* src = static_cast<const uint8_t*>(frames);
    if (!in_on_device) {
        CUD(cudaMalloc(&d_in, (size_t)nframes * frame_bytes));
        CUD(cudaMemcpy(d_in, frames, (size_t)nframes * frame_bytes, cudaMemcpyHostToDevice));
        src = d_in;
    }
    const int slot_bytes = in_nbit == 8 ? payload : (int)spf;             // 1- and 2-bit: one index byte per time sample
    CUD(cudaMalloc(&d_compact, (size_t)nframes * slot_bytes));
    CUD(cudaMalloc(&d_wmask, (size_t)nframes * gps));
    CUD(cudaMalloc(&d_fstat, (size_t)nframes));
    CUD(cudaMalloc(&d_dirty, 1));
    CUD(cudaMalloc(&d_cnt, C_COUNT * sizeof(unsigned long long)));
    CUD(cudaMemset(d_cnt, 0, C_COUNT * sizeof(unsigned long long)));
    CUD(cudaMemset(d_fstat, 0, (size_t)nframes));
    if (out_on_device) d_out = out;
    else CUD(cudaMalloc(&d_out, (size_t)2 * nsamp * sizeof(float)));
    K0Params k0{};
    k0.frames[0] = src;
    k0.compact = d_compact; k0.wmask = d_wmask; k0.fstat = d_fstat; k0.counters = d_cnt;
    k0.nframes = nframes; k0.nslots = nframes;
    k0.frame_bytes = frame_bytes; k0.header_bytes = header_bytes; k0.payload_bytes = payload; k0.groups_per_slot = gps;
    k0.slot_bytes = slot_bytes;
    k0.in_nbit = in_nbit; k0.time_mode = 0; k0.mask_faults = mask_faults; k0.fps = 1;
    rc = launch_k0(nullptr, k0, 0, false);
    if (rc) { cleanup(); return rc; }
    const int64_t nwords = nframes * (int64_t)(slot_bytes / 4);      // 2-bit: index words of 4 time samples
    if (in_nbit != 8)
        k_decode<2><<<(unsigned)((nwords + 255) / 256), 256>>>(d_compact, d_wmask, payload, gps, nwords, d_out, nsamp);
    else
        k_decode<8><<<(unsigned)((nwords + 255) / 256), 256>>>(d_compact, d_wmask, payload, gps, nwords, d_out, nsamp);
    CUD(cudaGetLastError());
    CUD(cudaDeviceSynchronize());
    if (!out_on_device) CUD(cudaMemcpy(out, d_out, (size_t)2 * nsamp * sizeof(float), cudaMemcpyDeviceToHost));
    if (counters) {
        unsigned long long h[C_COUNT];
        CUD(cudaMemcpy(h, d_cnt, sizeof(h), cudaMemcpyDeviceToHost));
        memset(counters, 0, sizeof(*counters));
        counters->frames_ok = h[C_OK]; counters->frames_invalid = h[C_INVALID];
        counters->frames_with_fill = h[C_FILLFRAMES]; counters->fill_words = h[C_FILLWORDS];
        counters->frames_badhdr = h[C_BADHDR]; counters->frames_misplaced = h[C_MISPLACED];
    }
#undef CUD
    cleanup();
    return 0;
}

// FP32 FMA-loop peak of this device (the denominator of the FFT roofline: MEASURED_PEAKS.json
// only holds the HBM copy and bf16 GEMM figures).  8 independent FMA chains per thread.
__global__ void k_fma_peak(float* out, int iters) {
    float a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const float b = 1.0000001f, c = 1e-7f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            a0 = fmaf(a0, b, c); a1 = fmaf(a1, b, c); a2 = fmaf(a2, b, c); a3 = fmaf(a3, b, c);
            a4 = fmaf(a4, b, c); a5 = fmaf(a5, b, c); a6 = fmaf(a6, b, c); a7 = fmaf(a7, b, c);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

int b2f_fp32_peak(int device, double* tflops) {
    if (!tflops) return fail(B2F_EINVAL, "null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(B2F_ECUDA, "no CUDA device");
    }
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    float* d = nullptr;
    CU(cudaMalloc(&d, (size_t)blocks * threads * sizeof(float)));
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    double best = 0;
    for (int rep = 0; rep < 6; ++rep) {
        CU(cudaEventRecord(a));
        k_fma_peak<<<blocks, threads>>>(d, iters);
        CU(cudaEventRecord(b));
        CU(cudaEventSynchronize(b));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, a, b));
        const double fl = 2.0 * 64.0 * iters * (double)blocks * threads;
        if (rep >= 2) best = std::max(best, fl / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(d);
    *tflops = best;
    return 0;
}

int b2f_debug_copy(b2f_plan* pl, int which, void* dst, size_t nbytes, size_t* needed) {
    if (!pl) return fail(B2F_EINVAL, "null plan");
    CU(cudaSetDevice(pl->prm.device));
    CU(cudaStreamSynchronize(pl->stream));
    const int nif = pl->prm.nif;
    const int64_t nbt = (int64_t)nif * pl->last_nblk;
    const void* src = nullptr;
    size_t n = 0;
    switch (which) {
        case 0:
            if (pl->path) { src = pl->d_tstream; n = pl->tstream_stride * nif; }
            else { src = pl->d_compact; n = pl->compact_stride * nif; }
            break;
        case 1: src = pl->d_wmask; n = pl->wmask_stride * nif; break;
        case 2: src = pl->d_fstat; n = pl->fstat_stride * nif; break;
        case 3: src = pl->d_blkdirty; n = (size_t)nbt; break;
        case 4: {       // intermediate of the last sub-batch only (whole push when batching is off)
            int64_t nbk = pl->batch_blocks > 0 ? std::min<int64_t>(pl->batch_blocks, nbt) : nbt;
            if (pl->path == 2) nbk = (int64_t)pl->f_lanes * pl->f_nslot;     // the ring ([pair][512][2] slots), not the whole push
            src = pl->d_inter; n = (size_t)nbk * pl->L * pl->R * sizeof(float2); break;
        }
        case 5: src = pl->d_colsum; n = (size_t)nbt * pl->R * sizeof(float2); break;
        case 6: src = pl->d_eps; n = (size_t)nbt * pl->N * sizeof(float2); break;
        case 7: src = pl->d_F; n = (size_t)pl->F_if_stride * pl->ndm * nif * sizeof(float); break;
        case 8: src = pl->d_fprof; n = (size_t)pl->f_grid * kFWarps * 8 * sizeof(unsigned long long); break;
        default: return fail(B2F_EINVAL, "which");
    }
    if (!src) return fail(B2F_EINVAL, "this buffer is not used by the plan's channeliser path");
    if (needed) *needed = n;
    if (!dst) return 0;
    CU(cudaMemcpy(dst, src, std::min(n, nbytes), cudaMemcpyDeviceToHost));
    return 0;
}

}  // extern "C"
