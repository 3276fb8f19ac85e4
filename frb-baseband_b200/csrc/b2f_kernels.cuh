// Hand-written sm_100a kernels of the baseband -> filterbank path.  See DESIGN.md section 3
// for the algebra (column pass / row pass / block-constant correction) and section 4 for
// the HBM layout.  Replaces the arithmetic `digifil` performs for
// /root/reference/process_vdif.py:156-182 and `splice` for /root/reference/base2fil.sh:422.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/b2f.h"
#include "fft_inreg.cuh"

namespace b2f {

constexpr int kL = 512;                 // column FFT length (= digifil freq_res) of the fused path
#ifndef B2F_STRIP_COLS
#define B2F_STRIP_COLS 16
#endif
constexpr int kStripCols = B2F_STRIP_COLS;   // columns per column-pass CTA (8 or 16)
constexpr int kKAThreads = 16 * kStripCols;  // 16 work items x columns
constexpr int kKACtasPerSM = 32 / kStripCols;  // 4 x 128 threads or 2 x 256 threads: 16 warps per SM either way
#ifndef B2F_P3_SPLIT
#define B2F_P3_SPLIT 1
#endif
#ifndef B2F_KB_THREADS
#define B2F_KB_THREADS 256
#endif
#ifndef B2F_KB_STAGES
#define B2F_KB_STAGES 2
#endif
constexpr int kKBThreads = B2F_KB_THREADS;
constexpr int kKBStages = B2F_KB_STAGES;        // TMA ring depth per warp: kKBStages - 1 row tiles in flight
constexpr uint32_t kFillWord = 0x11223344u;
constexpr float kLevLo = 1.0f;          // standard VLBI optimal 2-bit reconstruction levels
constexpr float kLevHi = 3.3359f;

enum Counter {
    C_OK = 0, C_INVALID, C_FILLFRAMES, C_FILLWORDS, C_DROPPED, C_MISPLACED, C_BADHDR, C_MISSING,
    C_DIRTY, C_COUNT
};

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// TMA bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ float2 lds_v2_volatile(const void* p) {
    float2 v;
    asm volatile("ld.volatile.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(smem_u32(p)));
    return v;
}
__device__ __forceinline__ void stg_v2_volatile(void* p, float2 v) {
    asm volatile("st.volatile.global.v2.f32 [%0], {%1, %2};" : : "l"(p), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void cp_async8(void* dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ================================================================== kernel 1: validate + de-frame
// One launch covers every IF (blockIdx.y).  Frames are staged whole into shared memory by
// TMA bulk copies (4-deep ring), the header is validated, every 32-bit payload word is
// compared with the recorder fill pattern, and the payload is written with 128-bit stores to
// the de-framed sample stream the channeliser reads.  One mask bit per payload word and one
// status byte per frame record what must decode to 0.0.
struct K0Params {
    const uint8_t* frames[B2F_MAX_IF];
    uint8_t* compact;  size_t compact_stride;
    uint8_t* wmask;    size_t wmask_stride;
    uint8_t* fstat;    size_t fstat_stride;
    unsigned long long* counters;
    int64_t nframes, nslots;
    int frame_bytes, header_bytes, payload_bytes, groups_per_slot;
    int in_nbit, time_mode, mask_faults, fps;
    int slot_bytes;            // bytes one frame occupies in the de-framed stream
    uint32_t base_sec[B2F_MAX_IF], base_fnum[B2F_MAX_IF];
};

// 2-bit payload word (8 time samples x 2 pols) -> 8 index bytes, one per time sample:
// (ch1 code << 2 | ch0 code) << 3, i.e. the byte offset of that sample's (pol0, pol1) float2 in
// the 17-entry decode table; index 16 selects the (0, 0) entry for masked samples.
__device__ __forceinline__ uint2 expand_word_2bit(uint32_t w, bool masked) {
    if (masked) return make_uint2(0x80808080u, 0x80808080u);
    const uint32_t x = w & 0x0F0F0F0Fu, y = (w >> 4) & 0x0F0F0F0Fu;      // even / odd nibbles
    const uint32_t lo = __byte_perm(x, y, 0x5140), hi = __byte_perm(x, y, 0x7362);
    return make_uint2(lo << 3, hi << 3);
}

// 1-bit payload word (16 time samples x 2 channels, bit 2t = ch0, bit 2t+1 = ch1) -> 16 index bytes.  A 1-bit sample decodes
// to -1.0 / +1.0 = the inner levels of the 2-bit table (codes 1 and 2): index = ((s0 ? 2 : 1) | (s1 ? 8 : 4)) << 3
// = 0x28 + 8 s0 + 32 s1, so everything behind this kernel sees the same index-byte stream as for 2-bit input.
__device__ __forceinline__ uint4 expand_word_1bit(uint32_t w, bool masked) {
    if (masked) return make_uint4(0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u);
    auto four = [](uint32_t x) {                             // 4 (s0, s1) pairs in the low byte -> 4 index bytes
        const uint32_t t = (x | (x << 6) | (x << 12) | (x << 18)) & 0x03030303u;
        return 0x28282828u + ((t & 0x01010101u) << 3) + ((t & 0x02020202u) << 4);
    };
    return make_uint4(four(w & 255u), four((w >> 8) & 255u), four((w >> 16) & 255u), four(w >> 24));
}

constexpr int kK0Threads = 256;
constexpr int kK0Stages = 4;
constexpr int kK0CtasPerSM = 4;

template <bool VEC>
__global__ void __launch_bounds__(kK0Threads) k0_validate_compact(const K0Params p) {
    extern __shared__ __align__(128) uint8_t k0_smem[];
    uint64_t* mbar = reinterpret_cast<uint64_t*>(k0_smem);
    const int stage_bytes = (p.frame_bytes + 127) & ~127;
    uint8_t* bufs = k0_smem + 128;
    const int ifi = blockIdx.y;
    const int tid = threadIdx.x;
    const uint8_t* src = p.frames[ifi];
    uint8_t* compact = p.compact + ifi * p.compact_stride;
    uint8_t* wmask = p.wmask + ifi * p.wmask_stride;
    uint8_t* fstat = p.fstat + ifi * p.fstat_stride;

    if (VEC) {
        if (tid == 0) {
            for (int s = 0; s < kK0Stages; ++s) mbar_init(&mbar[s], 1);
            mbar_fence_init();
        }
        __syncthreads();
        if (tid == 0) {
            for (int s = 0; s < kK0Stages; ++s) {
                int64_t f = blockIdx.x + (int64_t)s * gridDim.x;
                if (f < p.nframes) {
                    mbar_expect_tx(&mbar[s], p.frame_bytes);
                    bulk_g2s(bufs + s * stage_bytes, src + f * p.frame_bytes, p.frame_bytes, &mbar[s]);
                }
            }
        }
    }

    unsigned long long c_ok = 0, c_inv = 0, c_fillf = 0, c_fillw = 0, c_drop = 0, c_mis = 0, c_bad = 0;
    int it = 0;
    for (int64_t f = blockIdx.x; f < p.nframes; f += gridDim.x, ++it) {
        const int stage = VEC ? (it % kK0Stages) : 0;
        uint8_t* buf = bufs + stage * stage_bytes;
        if (VEC) {
            mbar_wait(&mbar[stage], (it / kK0Stages) & 1);
        } else {
            const uint2* s8 = reinterpret_cast<const uint2*>(src + f * p.frame_bytes);
            for (int i = tid; i < p.frame_bytes / 8; i += kK0Threads) reinterpret_cast<uint2*>(buf)[i] = s8[i];
            __syncthreads();
        }
        const uint32_t* hw = reinterpret_cast<const uint32_t*>(buf);
        const uint32_t w0 = hw[0], w1 = hw[1], w2 = hw[2], w3 = hw[3];
        const bool invalid = (w0 >> 31) != 0;
        const bool bad = ((w2 & 0xFFFFFFu) * 8u != (uint32_t)p.frame_bytes) ||
                         ((int)((w3 >> 26) & 31u) + 1 != p.in_nbit) ||
                         ((int)((w0 >> 30) & 1u) != (p.header_bytes == 16 ? 1 : 0));
        const int64_t tslot = ((int64_t)(w0 & 0x3FFFFFFFu) - (int64_t)p.base_sec[ifi]) * p.fps +
                              ((int64_t)(w1 & 0xFFFFFFu) - (int64_t)p.base_fnum[ifi]);
        const int64_t slot = p.time_mode ? tslot : f;
        int any_fill = 0;
        unsigned nfill = 0;
        const bool in_range = (slot >= 0 && slot < p.nslots);
        if (in_range) {
            const bool dead = invalid || bad;
            const int ngroups = p.groups_per_slot;
            uint8_t* dst = compact + slot * (int64_t)p.slot_bytes;
            const uint8_t* pay = buf + p.header_bytes;
            const bool two = p.in_nbit == 2, one = p.in_nbit == 1;
            for (int g = tid; g < ngroups; g += kK0Threads) {
                uint32_t m = 0;
                uint32_t w[8];
                const int nw = VEC ? 8 : min(8, (p.payload_bytes - 32 * g) / 4);
                if (VEC) {
                    const uint4 a = *reinterpret_cast<const uint4*>(pay + 32 * g);
                    const uint4 b = *reinterpret_cast<const uint4*>(pay + 32 * g + 16);
                    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
                } else {
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        w[k] = k < nw ? *reinterpret_cast<const uint32_t*>(pay + 32 * g + 4 * k) : 0u;
                }
#pragma unroll
                for (int k = 0; k < 8; ++k) m |= (uint32_t)(k < nw && w[k] == kFillWord) << k;
                if (!dead) nfill += __popc(m);
                if (!p.mask_faults) m = 0;
                else if (dead) m = 0xFF;
                wmask[slot * (int64_t)ngroups + g] = (uint8_t)m;
                any_fill |= (m != 0);
                if (one) {               // 8 words -> 128 index bytes
                    for (int k = 0; k < nw; ++k) {
                        const uint4 e = expand_word_1bit(w[k], (m >> k) & 1);
                        if (VEC) {
                            reinterpret_cast<uint4*>(dst + 128 * g)[k] = e;
                        } else {
                            reinterpret_cast<uint2*>(dst + 128 * g)[2 * k] = make_uint2(e.x, e.y);
                            reinterpret_cast<uint2*>(dst + 128 * g)[2 * k + 1] = make_uint2(e.z, e.w);
                        }
                    }
                } else if (two) {        // 8 words -> 64 index bytes
                    uint2 e[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) e[k] = expand_word_2bit(w[k], (m >> k) & 1);
                    if (VEC) {
                        uint4* d4 = reinterpret_cast<uint4*>(dst + 64 * g);
#pragma unroll
                        for (int k = 0; k < 4; ++k) d4[k] = make_uint4(e[2 * k].x, e[2 * k].y, e[2 * k + 1].x, e[2 * k + 1].y);
                    } else {
                        for (int k = 0; k < nw; ++k) reinterpret_cast<uint2*>(dst + 64 * g)[k] = e[k];
                    }
                } else if (VEC) {
                    *reinterpret_cast<uint4*>(dst + 32 * g) = make_uint4(w[0], w[1], w[2], w[3]);
                    *reinterpret_cast<uint4*>(dst + 32 * g + 16) = make_uint4(w[4], w[5], w[6], w[7]);
                } else {
                    for (int k = 0; k < nw; ++k) *reinterpret_cast<uint32_t*>(dst + 32 * g + 4 * k) = w[k];
                }
            }
        }
        // barrier: everybody is done with buf; also reduces the fill flag
        any_fill = __syncthreads_or(any_fill);
        if (nfill) atomicAdd(&p.counters[C_FILLWORDS], (unsigned long long)nfill);
        if (tid == 0) {
            if (!in_range) {
                ++c_drop;
            } else {
                const bool dead = invalid || bad;
                fstat[slot] = dead ? 2 : (any_fill ? 3 : 1);
                if (bad) ++c_bad;
                else if (invalid) ++c_inv;
                else if (any_fill) { ++c_fillf; }
                else ++c_ok;
                if (tslot != f) ++c_mis;
            }
            if (VEC) {
                const int64_t fn = f + (int64_t)kK0Stages * gridDim.x;
                if (fn < p.nframes) {
                    fence_proxy_async();
                    mbar_expect_tx(&mbar[stage], p.frame_bytes);
                    bulk_g2s(buf, src + fn * p.frame_bytes, p.frame_bytes, &mbar[stage]);
                }
            }
        }
        (void)c_fillw;
    }
    if (tid == 0) {
        if (c_ok) atomicAdd(&p.counters[C_OK], c_ok);
        if (c_inv) atomicAdd(&p.counters[C_INVALID], c_inv);
        if (c_fillf) atomicAdd(&p.counters[C_FILLFRAMES], c_fillf);
        if (c_drop) atomicAdd(&p.counters[C_DROPPED], c_drop);
        if (c_mis) atomicAdd(&p.counters[C_MISPLACED], c_mis);
        if (c_bad) atomicAdd(&p.counters[C_BADHDR], c_bad);
    }
}

// ================================================================== kernel 1r: corner turn front end
// Raw multi-BBC VDIF (what the recorder holds before jive5ab's spif2file splits it,
// /root/reference/spif2file.sh:31-98,178-186): every W-bit word is one time sample of all BBC
// channels.  For IF i the recipe names the 4 source bits (sign, magnitude of pol A; sign,
// magnitude of pol B) that form its 2-channel 2-bit sample.  This kernel validates the raw
// frames like k0 and writes every IF's index-byte stream directly, so the split files, the FIFOs and
// the scratch-disk round trip disappear.
struct K0RParams {
    const uint8_t* frames;
    uint8_t* compact; size_t compact_stride;
    uint8_t* fstat;   size_t fstat_stride;
    unsigned long long* counters;
    int64_t nframes, nslots;
    int frame_bytes, header_bytes, payload_bytes, word_bits, nif, time_mode, mask_faults, fps, slot_bytes;
    uint32_t base_sec, base_fnum;
    uint8_t bit[B2F_MAX_IF][4];
    int format;                 // enum b2f_raw_format
    int sample_bits;            // 2, or 1: bit[i][0] / bit[i][2] are the source bits of pol 0 / pol 1 (spif2file.sh:58-61)
};

// Mark5B time code word (BCD JJJSSSSS: MJD mod 1000, second of day) -> JJJ * 86400 + SSSSS
__host__ __device__ inline uint32_t mark5b_seconds(uint32_t w2) {
    uint32_t sss = 0, jjj = 0;
    for (int d = 4; d >= 0; --d) sss = sss * 10 + ((w2 >> (4 * d)) & 15u);
    for (int d = 7; d >= 5; --d) jjj = jjj * 10 + ((w2 >> (4 * d)) & 15u);
    return jjj * 86400u + sss;
}
constexpr uint32_t kMark5BSync = 0xABADDEEDu;

template <typename WORD>
__device__ __forceinline__ uint32_t gather_nibble_index(WORD w, const uint8_t (&b)[4]) {
    return (uint32_t)(((w >> b[0]) & 1) << 3 | ((w >> b[1]) & 1) << 4 | ((w >> b[2]) & 1) << 5 | ((w >> b[3]) & 1) << 6);
}
// 1-bit samples: 0 -> -1.0, 1 -> +1.0 = the inner levels of the 2-bit table (codes 1 and 2), so the same decode LUT serves
template <typename WORD>
__device__ __forceinline__ uint32_t gather_1bit_index(WORD w, const uint8_t (&b)[4]) {
    const uint32_t s0 = (uint32_t)((w >> b[0]) & 1), s1 = (uint32_t)((w >> b[2]) & 1);
    return ((s0 ? 2u : 1u) | (s1 ? 8u : 4u)) << 3;
}

template <int WBITS>
__global__ void __launch_bounds__(kK0Threads) k0r_corner_turn(const K0RParams p) {
    using WORD = typename std::conditional<WBITS == 64, unsigned long long, uint32_t>::type;
    extern __shared__ __align__(128) uint8_t k0_smem[];
    uint64_t* mbar = reinterpret_cast<uint64_t*>(k0_smem);
    const int stage_bytes = (p.frame_bytes + 127) & ~127;
    uint8_t* bufs = k0_smem + 128;
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < kK0Stages; ++s) mbar_init(&mbar[s], 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0) {
        for (int s = 0; s < kK0Stages; ++s) {
            const int64_t f = blockIdx.x + (int64_t)s * gridDim.x;
            if (f < p.nframes) {
                mbar_expect_tx(&mbar[s], p.frame_bytes);
                bulk_g2s(bufs + s * stage_bytes, p.frames + f * p.frame_bytes, p.frame_bytes, &mbar[s]);
            }
        }
    }
    constexpr int SPW = WBITS == 16 ? 2 : 1;                  // time samples per 32-bit payload unit (16-bit words: 2)
    const bool one_bit = p.sample_bits == 1;
    const int nquads = p.slot_bytes / 4;                      // groups of 4 consecutive time samples per frame
    // Mark5B payloads of 64-bit words hold 1250 samples: a last group of 2, and slots that start on odd 16-bit boundaries
    const bool half = WBITS == 64 && (p.slot_bytes & 2) != 0;
    const int ngroups = nquads + (half ? 1 : 0);
    unsigned long long c_ok = 0, c_inv = 0, c_fillf = 0, c_drop = 0, c_mis = 0, c_bad = 0;
    int it = 0;
    for (int64_t f = blockIdx.x; f < p.nframes; f += gridDim.x, ++it) {
        const int stage = it % kK0Stages;
        uint8_t* buf = bufs + stage * stage_bytes;
        mbar_wait(&mbar[stage], (it / kK0Stages) & 1);
        const uint32_t* hw = reinterpret_cast<const uint32_t*>(buf);
        const uint32_t w0 = hw[0], w1 = hw[1], w2 = hw[2], w3 = hw[3];
        const bool mk5 = p.format == B2F_RAW_MARK5B;
        // Mark5B: no invalid bit and no length field; the sync word pins the framing, test-vector frames carry no sky data
        const bool invalid = mk5 ? ((w1 >> 15) & 1u) != 0 : (w0 >> 31) != 0;
        const bool bad = mk5 ? w0 != kMark5BSync
                             : ((w2 & 0xFFFFFFu) * 8u != (uint32_t)p.frame_bytes) || ((int)((w3 >> 26) & 31u) + 1 != p.sample_bits) ||
                                   ((int)((w0 >> 30) & 1u) != (p.header_bytes == 16 ? 1 : 0));
        const int64_t tslot = mk5 ? ((int64_t)mark5b_seconds(w2) - (int64_t)p.base_sec) * p.fps + ((int64_t)(w1 & 0x7FFFu) - (int64_t)p.base_fnum)
                                  : ((int64_t)(w0 & 0x3FFFFFFFu) - (int64_t)p.base_sec) * p.fps +
                                        ((int64_t)(w1 & 0xFFFFFFu) - (int64_t)p.base_fnum);
        const int64_t slot = p.time_mode ? tslot : f;
        const bool in_range = (slot >= 0 && slot < p.nslots);
        const bool dead = invalid || bad;
        int any_fill = 0;
        unsigned nfill = 0;
        if (in_range) {
            const uint8_t* pay = buf + p.header_bytes;
            for (int g = tid; g < ngroups; g += kK0Threads) {
                const int ns = (half && g == nquads) ? 2 : 4;           // samples in this group
                WORD w[4];
                bool masked[4];
                if (WBITS == 16) {
                    const uint2 v = *reinterpret_cast<const uint2*>(pay + 8 * g);
                    w[0] = v.x & 0xFFFFu; w[1] = v.x >> 16; w[2] = v.y & 0xFFFFu; w[3] = v.y >> 16;
                    masked[0] = masked[1] = v.x == kFillWord;
                    masked[2] = masked[3] = v.y == kFillWord;
                    nfill += (v.x == kFillWord) + (v.y == kFillWord);
                } else if (WBITS == 32) {
                    const uint4 v = *reinterpret_cast<const uint4*>(pay + 16 * g);
                    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
#pragma unroll
                    for (int k = 0; k < 4; ++k) { masked[k] = (uint32_t)w[k] == kFillWord; nfill += masked[k]; }
                } else {
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        if (2 * k >= ns) {                               // beyond the payload
                            w[2 * k] = w[2 * k + 1] = 0;
                            masked[2 * k] = masked[2 * k + 1] = false;
                            continue;
                        }
                        const uint4 v = *reinterpret_cast<const uint4*>(pay + 32 * g + 16 * k);
                        w[2 * k] = (WORD)v.x | ((WORD)v.y << 32);
                        w[2 * k + 1] = (WORD)v.z | ((WORD)v.w << 32);
                        masked[2 * k] = v.x == kFillWord || v.y == kFillWord;
                        masked[2 * k + 1] = v.z == kFillWord || v.w == kFillWord;
                        nfill += (v.x == kFillWord) + (v.y == kFillWord) + (v.z == kFillWord) + (v.w == kFillWord);
                    }
                }
                (void)SPW;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    masked[k] = p.mask_faults && (masked[k] || dead);
                    any_fill |= masked[k] && !dead;
                }
                for (int i = 0; i < p.nif; ++i) {
                    uint32_t o = 0;
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        o |= (masked[k] ? 0x80u : one_bit ? gather_1bit_index<WORD>(w[k], p.bit[i]) : gather_nibble_index<WORD>(w[k], p.bit[i])) << (8 * k);
                    uint8_t* d = p.compact + i * p.compact_stride + slot * (int64_t)p.slot_bytes + 4 * g;
                    if (half) {
                        reinterpret_cast<uint16_t*>(d)[0] = (uint16_t)(o & 0xFFFFu);
                        if (ns == 4) reinterpret_cast<uint16_t*>(d)[1] = (uint16_t)(o >> 16);
                    } else {
                        *reinterpret_cast<uint32_t*>(d) = o;
                    }
                }
            }
        }
        any_fill = __syncthreads_or(any_fill);
        if (nfill && !dead) atomicAdd(&p.counters[C_FILLWORDS], (unsigned long long)nfill);
        if (tid == 0) {
            if (!in_range) {
                ++c_drop;
            } else {
                for (int i = 0; i < p.nif; ++i) p.fstat[i * p.fstat_stride + slot] = dead ? 2 : (any_fill ? 3 : 1);
                if (bad) ++c_bad;
                else if (invalid) ++c_inv;
                else if (any_fill) ++c_fillf;
                else ++c_ok;
                if (tslot != f) ++c_mis;
            }
            const int64_t fn = f + (int64_t)kK0Stages * gridDim.x;
            if (fn < p.nframes) {
                fence_proxy_async();
                mbar_expect_tx(&mbar[stage], p.frame_bytes);
                bulk_g2s(buf, p.frames + fn * p.frame_bytes, p.frame_bytes, &mbar[stage]);
            }
        }
    }
    if (tid == 0) {
        if (c_ok) atomicAdd(&p.counters[C_OK], c_ok);
        if (c_inv) atomicAdd(&p.counters[C_INVALID], c_inv);
        if (c_fillf) atomicAdd(&p.counters[C_FILLFRAMES], c_fillf);
        if (c_drop) atomicAdd(&p.counters[C_DROPPED], c_drop);
        if (c_mis) atomicAdd(&p.counters[C_MISPLACED], c_mis);
        if (c_bad) atomicAdd(&p.counters[C_BADHDR], c_bad);
    }
}

// slots no frame landed in are masked; blocks touched by any non-clean slot are flagged
struct K0bParams {
    uint8_t* wmask;    size_t wmask_stride;
    const uint8_t* fstat; size_t fstat_stride;
    uint8_t* blkdirty;                         // [nif][nblk]
    unsigned long long* counters;
    int64_t nslots; int nif, nblk, groups_per_slot, samples_per_frame; int64_t block_samples;
    uint8_t* compact; size_t compact_stride; int slot_bytes, in_nbit;   // 2-bit: missing slots get the zero-entry index
};
#ifdef B2F_API_TU        // non-template kernels are launched from b2f_api.cu only: compile them once
static __global__ void k0b_finish_slots(const K0bParams p) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= p.nslots * p.nif) return;
    const int ifi = (int)(i / p.nslots);
    const int64_t slot = i % p.nslots;
    const uint8_t st = p.fstat[ifi * p.fstat_stride + slot];
    if (st == 1) return;
    if (st == 0) {
        uint8_t* m = p.wmask + ifi * p.wmask_stride + slot * (int64_t)p.groups_per_slot;
        for (int g = 0; g < p.groups_per_slot; ++g) m[g] = 0xFF;
        if (p.in_nbit != 8) {                                   // masking lives in the index stream for 1- and 2-bit input
            // 32-bit stores: a slot is a whole number of words, but with raw 64-bit input (slot_bytes = 1000) neither a
            // multiple of 16 bytes nor 16-byte aligned
            uint8_t* d8 = p.compact + ifi * p.compact_stride + slot * (int64_t)p.slot_bytes;
            if (p.slot_bytes & 2) {                              // Mark5B, 64-bit words: 1250 samples per frame
                uint16_t* d = reinterpret_cast<uint16_t*>(d8);
                for (int k = 0; k < p.slot_bytes / 2; ++k) d[k] = 0x8080u;
            } else {
                uint32_t* d = reinterpret_cast<uint32_t*>(d8);
                for (int k = 0; k < p.slot_bytes / 4; ++k) d[k] = 0x80808080u;
            }
        }
        atomicAdd(&p.counters[C_MISSING], 1ull);
    }
    const int64_t s0 = slot * p.samples_per_frame;
    const int64_t b0 = s0 / p.block_samples, b1 = (s0 + p.samples_per_frame - 1) / p.block_samples;
    for (int64_t b = b0; b <= b1 && b < p.nblk; ++b) p.blkdirty[ifi * (int64_t)p.nblk + b] = 1;
}
#endif

#ifdef B2F_API_TU
// JA98 decode on the generic path (NBIT = 22 in the column kernels): one warp per window of 512 samples of the index-byte
// stream (carried samples in front, so windows count from the start of the scan as long as blocks start on multiples of
// 512) counts, per polarisation, the samples between the thresholds among those that are not masked, and turns the
// fraction into the two output magnitudes -- the arithmetic of kj_ja98_levels (b2f_fused.cuh) and of the oracle's ja98_levels.
static __global__ void kj_levels_stream(const uint8_t* compact, size_t compact_stride, int64_t T, float4* levels, int64_t levels_stride, int nif) {
    const int lane = threadIdx.x & 31;
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwin = (T + 511) >> 9;
    if (w >= nwin * nif) return;
    const int ifi = (int)(w / nwin);
    const int64_t wi = w % nwin, pos = wi * 512 + lane * 16;
    const uint8_t* src = compact + ifi * compact_stride + pos;
    unsigned lowP = 0, lowQ = 0, nval = 0;
    uint32_t x[4] = {0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u};
    if (pos + 16 <= T) {
        const uint4 v = *reinterpret_cast<const uint4*>(src);
        x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
    } else {
        for (int k = 0; k < 16 && pos + k < T; ++k) x[k >> 2] = (x[k >> 2] & ~(0xFFu << (8 * (k & 3)))) | ((uint32_t)src[k] << (8 * (k & 3)));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {                                  // index byte = (c1 << 2 | c0) << 3, 0x80 = masked
        const uint32_t ok = (~x[k] >> 7) & 0x01010101u;
        lowP += __popc(((x[k] >> 3) ^ (x[k] >> 4)) & ok);           // code 1 or 2: the two bits differ
        lowQ += __popc(((x[k] >> 5) ^ (x[k] >> 6)) & ok);
        nval += __popc(ok);
    }
    for (int m = 16; m; m >>= 1) {
        lowP += __shfl_xor_sync(0xffffffffu, lowP, m);
        lowQ += __shfl_xor_sync(0xffffffffu, lowQ, m);
        nval += __shfl_xor_sync(0xffffffffu, nval, m);
    }
    if (lane == 0) {
        float lv[4];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            double phi = nval ? (double)(q ? lowQ : lowP) / (double)nval : 0.5;
            phi = fmin(fmax(phi, 1.0 / 512.0), 1.0 - 1.0 / 512.0);
            const double t = 1.4142135623730951 * erfinv(phi);
            const double e = exp(-0.5 * t * t);
            lv[2 * q] = (float)(0.7978845608028654 * (1.0 - e) / phi);
            lv[2 * q + 1] = (float)(0.7978845608028654 * e / (1.0 - phi));
        }
        levels[ifi * levels_stride + wi] = make_float4(lv[0], lv[1], lv[2], lv[3]);
    }
}

// 8-bit input in carry mode keeps its word masks by stream position (b2f_plan::smask): a block is dirty when any mask
// byte of its M samples is set.  step32 / blk32: block stride and block length in mask bytes.
static __global__ void k8_blkdirty(const uint8_t* wmask, size_t wmask_stride, uint8_t* blkdirty, int nblk, int64_t step32, int64_t blk32) {
    const int b = blockIdx.x, ifi = blockIdx.y;
    const uint8_t* m = wmask + ifi * wmask_stride + b * step32;
    int any = 0;
    for (int64_t i = threadIdx.x; i < blk32; i += blockDim.x) any |= m[i];
    any = __syncthreads_or(any);
    if (threadIdx.x == 0) blkdirty[ifi * (int64_t)nblk + b] = any ? 1 : 0;
}
#endif

// ================================================================== stand-alone decode
// compact payload (+ word mask) -> planar float samples out[2][nsamp].  HBM-bound expansion
// (2 bit -> 32 bit); the production path never runs it, the column pass decodes on the fly.
template <int NBIT>
__global__ void k_decode(const uint8_t* __restrict__ compact, const uint8_t* __restrict__ wmask,
                         int payload_bytes, int groups_per_slot, int64_t nwords, float* __restrict__ out,
                         int64_t nsamp) {
    const int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (w >= nwords) return;
    const uint32_t v = reinterpret_cast<const uint32_t*>(compact)[w];
    if (NBIT == 2) {
        // w counts index words: 4 time samples each, masking already folded into the index
        float a[4], b[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t idx = ((v >> (8 * k)) & 255u) >> 3;
            const uint32_t c0 = idx & 3u, c1 = (idx >> 2) & 3u;
            const float m0 = (c0 == 0 || c0 == 3) ? kLevHi : kLevLo;
            const float m1 = (c1 == 0 || c1 == 3) ? kLevHi : kLevLo;
            a[k] = idx >= 16 ? 0.f : ((c0 & 2) ? m0 : -m0);
            b[k] = idx >= 16 ? 0.f : ((c1 & 2) ? m1 : -m1);
        }
        reinterpret_cast<float4*>(out)[w] = make_float4(a[0], a[1], a[2], a[3]);
        reinterpret_cast<float4*>(out + nsamp)[w] = make_float4(b[0], b[1], b[2], b[3]);
    } else {
        const int words_per_slot = payload_bytes / 4;
        const int64_t slot = w / words_per_slot;
        const int ws = (int)(w % words_per_slot);
        const bool bad = (wmask[slot * groups_per_slot + (ws >> 3)] >> (ws & 7)) & 1;
        float2* o0 = reinterpret_cast<float2*>(out + w * 2);
        float2* o1 = reinterpret_cast<float2*>(out + nsamp + w * 2);
        const float x0 = bad ? 0.f : (float)(v & 255u) - 127.5f, y0 = bad ? 0.f : (float)((v >> 8) & 255u) - 127.5f;
        const float x1 = bad ? 0.f : (float)((v >> 16) & 255u) - 127.5f, y1 = bad ? 0.f : (float)(v >> 24) - 127.5f;
        o0[0] = make_float2(x0, x1);
        o1[0] = make_float2(y0, y1);
    }
}

// JA98 decode of a 2-bit sample pair: sign and size class from the static lookup, magnitude from the window's levels
__device__ __forceinline__ float2 kg_ja98(float2 v, float4 lv) {
    const float ax = fabsf(v.x), ay = fabsf(v.y);
    return make_float2(ax == 0.f ? 0.f : copysignf(ax > 2.f ? lv.y : lv.x, v.x), ay == 0.f ? 0.f : copysignf(ay > 2.f ? lv.w : lv.z, v.y));
}

// ================================================================== kernel 3a: column pass
// A block of M = R*512 dual-pol samples z[n] = xP[n] + i xQ[n] is viewed as a 512 x R matrix
// (n = n1 + R n2).  One CTA owns a strip of 16 columns: lane = column, so every shared-memory
// access is [index][lane] (conflict-free, no padding) and every twiddle except the two
// column-dependent tables is uniform across the 16 lanes.  Per column:
//   decode -> FFT_512 (16 x 32) -> * W_M^(k2 n1) -> IFFT_512 (32 x 16)  ->  B[m][n1]
// with only two shared-memory exchanges: the 32-point forward and inverse FFTs around the
// diagonal multiply act on the same 32 values, so they run back to back in registers.
// pw[q] = b^q, q = 1..15, from the exactly rounded seeds b, b^2, b^4, b^8 (host table, computed in
// double): every power is a product of at most four seeds (3 roundings), so no phase error of a base
// is amplified by the exponent.  Computing these twiddles in registers replaces shared-memory table
// reads, which -- not FP32 issue -- are what the column pass is short of (DESIGN.md section 5:
// dropping every butterfly gains 18 %, dropping the table reads 20 %).
__device__ __forceinline__ void cpowers15(const float2 (&sd)[4], float2 (&pw)[16]) {
    pw[0] = make_float2(1.f, 0.f);
    pw[1] = sd[0]; pw[2] = sd[1]; pw[4] = sd[2]; pw[8] = sd[3];
    pw[3] = cmul(sd[0], sd[1]);
    pw[5] = cmul(sd[0], sd[2]);
    pw[6] = cmul(sd[1], sd[2]);
    pw[7] = cmul(pw[3], sd[2]);
    pw[9] = cmul(sd[0], sd[3]);
    pw[10] = cmul(sd[1], sd[3]);
    pw[11] = cmul(pw[3], sd[3]);
    pw[12] = cmul(sd[2], sd[3]);
    pw[13] = cmul(pw[5], sd[3]);
    pw[14] = cmul(pw[6], sd[3]);
    pw[15] = cmul(pw[7], sd[3]);
}

struct KAParams {
    const uint8_t* compact;  size_t compact_stride;
    const uint8_t* wmask;    size_t wmask_stride;
    const uint8_t* blkdirty;
    float2* inter;           // [nif*nblk][512][R]
    float2* colsum;          // [nif*nblk][R]
    const float2* tab_g;     // [16][R]  W_M^(q n1)
    const float2* tab_h;     // [32][R]  W_M^(16 p n1)
    const float2* tab_w;     // [32][16] W_512^(l q)
    const float2* tab_beta;  // [16 items][4 seeds k = 1,2,4,8][R]  (W_M^(n1) conj W_512^(item))^k
    int R, nstrips, nblk, nif, payload_bytes, groups_per_slot;
    int64_t gb_begin, gb_end;   // this launch covers FFT blocks [gb_begin, gb_end); inter is indexed gb - gb_begin
    int64_t blk_step_bytes;     // stream bytes between the starts of consecutive blocks (= block size unless overlap-save)
    float in8_offset;        // 8-bit samples: value = code - in8_offset (127.5, or 128: SURVEY D3)
    const float4* levels; int64_t levels_stride;   // NBIT 22 (JA98): levels per window of 512 stream samples and IF (kj_levels_stream)
};

template <int NBIT>
struct KASmem {
    static constexpr int kPiece = (NBIT != 8 ? 1 : 2) * kStripCols;   // staged bytes per (row, strip); NBIT 22 = 2-bit with JA98 levels
    static constexpr int kRawBytes = kL * kPiece;
    static constexpr int kLutEntries = NBIT != 8 ? 32 : 0;      // index byte >> 3 -> (pol0, pol1); 16 = zero
    static constexpr size_t kBytes =
        (size_t)(kL * kStripCols + 512 + 512 + 32 * kStripCols + 16 * kStripCols + kLutEntries) * sizeof(float2) + 2 * kRawBytes;
};

// R (row length = 2*nchan) is a template parameter so that every global and shared address
// in the loop body is base + immediate.
// FWD_ONLY: forward transform only.  The kernel stops after A'[k2][n1] = FFT_512(column) * W_M^(k2 n1)
// and stores it; used by the dedispersion path, where the chirp has to be applied between the row FFT
// and the backward FFT.
template <int NBIT, int R, bool FWD_ONLY>
__global__ void __launch_bounds__(kKAThreads, kKACtasPerSM) ka_column_pass(const KAParams p) {
    using S = KASmem<NBIT>;
    extern __shared__ __align__(16) uint8_t ka_smem[];
    float2* data = reinterpret_cast<float2*>(ka_smem);      // 512 points x 16 lanes, as [256 pairs][16] float4
    float4* data4 = reinterpret_cast<float4*>(ka_smem);
    constexpr int C = kStripCols;
    float2* s_w = data + kL * C;                             // [32][16]  W_512^(l q)
    float2* s_wT = s_w + 512;                                // [16][32]
    float2* s_h = s_wT + 512;                                // [16][16 lanes] float4 = (h^p, h^(p+16))
    float2* s_g = s_h + 32 * C;                              // [8][C lanes]  float4 = (g^q, g^(q+8))
    float4* s_h4 = reinterpret_cast<float4*>(s_h);
    float4* s_g4 = reinterpret_cast<float4*>(s_g);
    float2* s_lut = s_g + 16 * C;                               // 17 used: sample index -> (pol0, pol1)
    uint8_t* s_raw = reinterpret_cast<uint8_t*>(s_lut + S::kLutEntries);   // [2][512][kPiece]

    const int tid = threadIdx.x;
    const int lane16 = tid % C;          // column within the strip
    const int item = tid / C;            // 0..15
    const int strip = blockIdx.x % p.nstrips;
    const int n1 = strip * kStripCols + lane16;

    for (int i = tid; i < 512; i += kKAThreads) {
        const float2 w = p.tab_w[i];
        s_w[i] = w;
        s_wT[(i & 15) * 32 + (i >> 4)] = w;
    }
    for (int i = tid; i < 32 * C; i += kKAThreads) {       // entry (p, lane) -> pair slot ((p & 15) * C + lane) * 2 + (p >> 4)
        const int pp = i / C, ln = i % C;
        s_h[((pp & 15) * C + ln) * 2 + (pp >> 4)] = p.tab_h[pp * R + strip * C + ln];
    }
    for (int i = tid; i < 16 * C; i += kKAThreads) {
        const int q = i / C, ln = i % C;
        s_g[((q & 7) * C + ln) * 2 + (q >> 3)] = p.tab_g[q * R + strip * C + ln];
    }
    if (NBIT != 8 && tid < 32) {
        // 16 entries span exactly the 32 banks once (conflict-free for any index pattern);
        // entry 16 = (0, 0) is what masked samples point at
        const int c0 = tid & 3, c1 = (tid >> 2) & 3;
        const float m0 = (c0 == 0 || c0 == 3) ? kLevHi : kLevLo;
        const float m1 = (c1 == 0 || c1 == 3) ? kLevHi : kLevLo;
        s_lut[tid] = tid < 16 ? make_float2((c0 & 2) ? m0 : -m0, (c1 & 2) ? m1 : -m1) : make_float2(0.f, 0.f);
    }

    // P3's merged twiddle base for m1 = item: beta = W_M^(n1) * conj(W_512^(item))
    float2 betaS[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) betaS[k] = p.tab_beta[(size_t)(item * 4 + k) * R + n1];
    __syncthreads();

    const int64_t nbt = p.gb_end;
    const int64_t first = p.gb_begin + blockIdx.x / p.nstrips;
    const int64_t step = gridDim.x / p.nstrips;
    const int64_t row_bytes = (int64_t)R * (NBIT != 8 ? 1 : 2);   // stream bytes per time sample: 1 index / 2 raw
    const int64_t blk_bytes = row_bytes * kL;

    auto issue_raw = [&](int64_t gb, int buf) {
        const int ifi = (int)(gb / p.nblk);
        const int64_t blk = gb % p.nblk;
        const uint8_t* src = p.compact + ifi * p.compact_stride + blk * p.blk_step_bytes + (int64_t)strip * S::kPiece;
        uint8_t* dst = s_raw + buf * S::kRawBytes;
        if (S::kPiece == 8) {
#pragma unroll
            for (int k = 0; k < kL / kKAThreads; ++k) {
                const int row = tid + k * kKAThreads;
                cp_async8(dst + row * 8, src + row * row_bytes);
            }
        } else {
            constexpr int PPR = S::kPiece / 16;                 // 16-byte pieces per row
#pragma unroll
            for (int k = 0; k < kL * PPR / kKAThreads; ++k) {
                const int j = tid + k * kKAThreads;
                const int row = j / PPR, h = j % PPR;
                cp_async16(dst + row * S::kPiece + h * 16, src + row * row_bytes + h * 16);
            }
        }
    };

    if (first < nbt) issue_raw(first, 0);
    cp_async_commit();
    uint8_t dirty_next = first < nbt ? p.blkdirty[first] : 0;

    int it = 0;
    for (int64_t gb = first; gb < nbt; gb += step, ++it) {
        const int buf = it & 1;
        const bool dirty = dirty_next != 0;
        if (gb + step < nbt) {
            issue_raw(gb + step, buf ^ 1);
            dirty_next = p.blkdirty[gb + step];           // consumed one work item later
        }
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();

        const uint8_t* raw = s_raw + buf * S::kRawBytes;
        const int ifi = (int)(gb / p.nblk);
        const int64_t blk = gb % p.nblk;

        // Shared-memory exchanges move float4 = the same element of rounds `item` and `item+16`,
        // so every exchange is one 128-bit access per two points (the LSU instruction queue, not
        // bandwidth, was the limiter with 64-bit accesses).
        // ---- P1: decode + 16-point FFT over r (n2 = 32 r + l) for l = item and item+16, twiddle W_512^(l q)
        {
            float2 vA[16], vB[16];
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int rowA = 32 * r + item, rowB = rowA + 16;
                if (NBIT != 8) {
                    vA[r] = *reinterpret_cast<const float2*>(reinterpret_cast<const uint8_t*>(s_lut) + raw[rowA * C + lane16]);
                    vB[r] = *reinterpret_cast<const float2*>(reinterpret_cast<const uint8_t*>(s_lut) + raw[rowB * C + lane16]);
                } else {
                    const uint32_t a = *reinterpret_cast<const uint16_t*>(raw + rowA * 2 * C + lane16 * 2);
                    const uint32_t b = *reinterpret_cast<const uint16_t*>(raw + rowB * 2 * C + lane16 * 2);
                    vA[r] = make_float2((float)(a & 255u) - p.in8_offset, (float)(a >> 8) - p.in8_offset);
                    vB[r] = make_float2((float)(b & 255u) - p.in8_offset, (float)(b >> 8) - p.in8_offset);
                }
            }
            if (NBIT == 22) {       // JA98: a row of R <= 512 samples lies in one window of 512 stream samples
                const float4* lvb = p.levels + ifi * p.levels_stride;
                const int64_t s0 = blk * p.blk_step_bytes;           // index bytes = samples
#pragma unroll
                for (int r = 0; r < 16; ++r) {
                    const int rowA = 32 * r + item;
                    vA[r] = kg_ja98(vA[r], __ldg(lvb + ((s0 + (int64_t)rowA * R) >> 9)));
                    vB[r] = kg_ja98(vB[r], __ldg(lvb + ((s0 + (int64_t)(rowA + 16) * R) >> 9)));
                }
            }
            if (NBIT == 8 && dirty) {
                const uint8_t* wm = p.wmask + ifi * p.wmask_stride;
#pragma unroll 1
                for (int rr = 0; rr < 32; ++rr) {
                    const int r = rr & 15;
                    const int row = 32 * r + item + (rr >> 4) * 16;
                    const int64_t off = blk * p.blk_step_bytes + row * row_bytes + (int64_t)strip * S::kPiece + lane16 * 2;
                    const int64_t slot = off / p.payload_bytes;
                    const int w = (int)(off % p.payload_bytes) >> 2;
                    if ((wm[slot * p.groups_per_slot + (w >> 3)] >> (w & 7)) & 1) {
#pragma unroll
                        for (int k = 0; k < 16; ++k) {       // static indexing keeps v[] in registers
                            if (k == r && rr < 16) vA[k] = make_float2(0.f, 0.f);
                            if (k == r && rr >= 16) vB[k] = make_float2(0.f, 0.f);
                        }
                    }
                }
            }
            fft_inreg<16, false>(vA); fft_inreg<16, false>(vB);
            // (measured: computing these and the h^p powers in registers as well costs more FP than the
            //  32 table reads it saves -- 99.6 vs 96.8 ms/step -- so they stay in shared memory)
            const float4* twA = reinterpret_cast<const float4*>(s_w + item * 16);
            const float4* twB = reinterpret_cast<const float4*>(s_w + (item + 16) * 16);
#pragma unroll
            for (int q = 0; q < 16; q += 2) {
                const float4 ta = twA[q >> 1], tb = twB[q >> 1];
                if (q) vA[q] = cmul(vA[q], make_float2(ta.x, ta.y));
                vA[q + 1] = cmul(vA[q + 1], make_float2(ta.z, ta.w));
                if (q) vB[q] = cmul(vB[q], make_float2(tb.x, tb.y));
                vB[q + 1] = cmul(vB[q + 1], make_float2(tb.z, tb.w));
            }
#pragma unroll
            for (int q = 0; q < 16; ++q)
                data4[(q * 16 + item) * C + lane16] = make_float4(vA[q].x, vA[q].y, vB[q].x, vB[q].y);
        }
        __syncthreads();

        // ---- Mid: FFT_32 over l -> p ; * W_M^(16 p n1) ; IFFT_32 over p -> m1 ; * conj W_512^(q m1)
        {
            const int q = item;
            float2 u[32];
#pragma unroll
            for (int l = 0; l < 16; ++l) {
                const float4 t = data4[(q * 16 + l) * C + lane16];
                u[l] = make_float2(t.x, t.y);
                u[l + 16] = make_float2(t.z, t.w);
            }
            fft_inreg<32, false>(u);
            if (FWD_ONLY) {
                // u[pp] = A[k2 = q + 16 pp]; full twiddle W_M^(k2 n1) = h^pp g^q, then straight to global
                const float4 g4 = s_g4[(q & 7) * C + lane16];
                const float2 gq = (q & 8) ? make_float2(g4.z, g4.w) : make_float2(g4.x, g4.y);
                float2* dst = p.inter + ((gb - p.gb_begin) * (int64_t)kL + q) * R + n1;
#pragma unroll
                for (int pp = 0; pp < 16; ++pp) {
                    const float4 h = s_h4[pp * C + lane16];
                    dst[(int64_t)(16 * pp) * R] = cmul(cmul(u[pp], make_float2(h.x, h.y)), gq);
                    dst[(int64_t)(16 * (pp + 16)) * R] = cmul(cmul(u[pp + 16], make_float2(h.z, h.w)), gq);
                }
            } else {
            if (q == 0) p.colsum[gb * R + n1] = u[0];          // A[k2 = 0]: column sum
#pragma unroll
            for (int pp = 0; pp < 16; ++pp) {
                const float4 h = s_h4[pp * C + lane16];
                if (pp) u[pp] = cmul(u[pp], make_float2(h.x, h.y));
                u[pp + 16] = cmul(u[pp + 16], make_float2(h.z, h.w));
            }
            fft_inreg<32, true>(u);
            // (the conj W_512^(q m1) twiddle of this stage is applied in P3, merged with W_M^(q n1))
#pragma unroll
            for (int m = 0; m < 16; ++m)
                data4[(q * 16 + m) * C + lane16] = make_float4(u[m].x, u[m].y, u[m + 16].x, u[m + 16].y);
            }   // !FWD_ONLY
        }
        __syncthreads();
        if (FWD_ONLY) continue;

        // ---- P3: * W_M^(q n1) ; IFFT_16 over q -> m2 ; m = m1 + 32 m2 for m1 = item and item+16
        // twiddle of element q: W_M^(q n1) conj W_512^(q m1) = beta^q, beta = g conj(W_512^m1).
        // Round B has m1 + 16: beta_B^q = beta_A^q conj(W_32^q), a compile-time constant factor.
        {
            float2 pw[16];
            cpowers15(betaS, pw);
            float2* dA = p.inter + ((gb - p.gb_begin) * (int64_t)kL + item) * R + n1;
            float2* dB = dA + 16 * R;
#if B2F_P3_SPLIT
            // Round A is finished and stored before round B is even loaded (volatile accesses keep the assembler
            // from regrouping them), so A's stores drain under B's arithmetic instead of all 32 stores arriving
            // in one burst at the end of the work item (ncu: 38 % of this section's stall samples sat on the
            // clustered STGs, lg_throttle).  Costs 16 more 64-bit shared loads; measured 31.8 -> 31.2 ms / 20 s.
            float2 yA[16], yB[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) yA[q] = lds_v2_volatile(&data4[(q * 16 + item) * C + lane16]);
#pragma unroll
            for (int q = 1; q < 16; ++q) yA[q] = cmul(yA[q], pw[q]);
            fft_inreg<16, true>(yA);
#pragma unroll
            for (int m2 = 0; m2 < 16; ++m2) stg_v2_volatile(&dA[32 * m2 * R], yA[m2]);
#pragma unroll
            for (int q = 0; q < 16; ++q)
                yB[q] = lds_v2_volatile(reinterpret_cast<const float2*>(&data4[(q * 16 + item) * C + lane16]) + 1);
#pragma unroll
            for (int q = 1; q < 16; ++q) {
                const float2 cb = make_float2(cos64(2 * q), sin64(2 * q));
                yB[q] = cmul(cmul(yB[q], cb), pw[q]);
            }
            fft_inreg<16, true>(yB);
#pragma unroll
            for (int m2 = 0; m2 < 16; ++m2) dB[32 * m2 * R] = yB[m2];
#else
            float2 yA[16], yB[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const float4 t = data4[(q * 16 + item) * C + lane16];
                yA[q] = make_float2(t.x, t.y);
                yB[q] = make_float2(t.z, t.w);
            }
#pragma unroll
            for (int q = 1; q < 16; ++q) {
                yA[q] = cmul(yA[q], pw[q]);
                const float2 cb = make_float2(cos64(2 * q), sin64(2 * q));      // conj(W_32^q) = exp(+2 pi i q/32)
                yB[q] = cmul(cmul(yB[q], cb), pw[q]);
            }
            fft_inreg<16, true>(yA); fft_inreg<16, true>(yB);
#pragma unroll
            for (int m2 = 0; m2 < 16; ++m2) {
                dA[32 * m2 * R] = yA[m2];
                dB[32 * m2 * R] = yB[m2];
            }
#endif
        }
        __syncthreads();
    }
    cp_async_wait<0>();
}

// ================================================================== kernel 3b: eps
// eps_c = conj(G[R-1-c] - G[(R-c) mod R]),  G = FFT_R(column sums): the one block-constant
// term that separating the two real polarisations after the row pass needs (DESIGN.md 3.3).
#ifdef B2F_API_TU        // non-template kernels are launched from b2f_api.cu only: compile them once
static __global__ void ke_eps(const float2* __restrict__ colsum, float2* __restrict__ eps, int R) {
    extern __shared__ float2 ke_s[];
    const int lg = 31 - __clz(R);
    const float2* src = colsum + (int64_t)blockIdx.x * R;
    for (int i = threadIdx.x; i < R; i += blockDim.x) ke_s[__brev(i) >> (32 - lg)] = src[i];
    __syncthreads();
    for (int s = 1; s <= lg; ++s) {
        const int half = 1 << (s - 1);
        for (int t = threadIdx.x; t < R / 2; t += blockDim.x) {      // one butterfly per thread and pass
            const int j = t & (half - 1);
            const int i0 = ((t >> (s - 1)) << s) + j, i1 = i0 + half;
            float sn, cs;
            sincospif(-(float)j / (float)half, &sn, &cs);
            const float2 a = ke_s[i0], b = ke_s[i1];
            const float2 wb = make_float2(b.x * cs - b.y * sn, b.x * sn + b.y * cs);
            ke_s[i0] = make_float2(a.x + wb.x, a.y + wb.y);
            ke_s[i1] = make_float2(a.x - wb.x, a.y - wb.y);
        }
        __syncthreads();
    }
    for (int t = threadIdx.x; t < R / 2; t += blockDim.x) {
        const float2 g0 = ke_s[R - 1 - t], g1 = ke_s[(R - t) & (R - 1)];
        eps[(int64_t)blockIdx.x * (R / 2) + t] = make_float2(g0.x - g1.x, -(g0.y - g1.y));
    }
}
#endif

// ================================================================== kernel 3c+4: row pass
// FFT_R across the R columns of every row m of the column-pass output, separation of the two
// polarisations (channel c with its mirror R-1-c, minus eps_c), detection and time
// integration over D rows.  TR lanes cooperate on one row (PT points each, R = TR*PT):
// radix-PT in registers, one transpose through padded shared memory, radix-TR in registers,
// mirror exchange by shuffle.
struct KBParams {
    const float2* inter;
    const float2* eps;          // [nif*nblk][R/2]
    const float2* tab_r;        // [PT][TR]  W_R^(s q)
    float* F;                   // [nif][cap_rows][nprod][R/2]
    int64_t F_if_stride;        // floats between IFs
    int64_t row0;               // first output row of this push inside F
    int nblk, nif, D;
    int64_t gb_begin, gb_end;   // FFT blocks of this launch; inter is indexed gb - gb_begin
    float2* spec;               // kModeSpectrum: [gb - gb_begin][512][R] output
};

// row-pass mode of the dedispersion path: no un-mixing or detection, store Z[k2][c] for all R channels
constexpr int kModeSpectrum = 100;

__host__ __device__ constexpr int nprod_of_mode(int mode) {
    return (mode == B2F_POL_COHERENCE || mode == B2F_POL_IQUV) ? 4 : (mode == B2F_POL_PPQQ ? 2 : 1);
}

// P = 2 yP, Q = 2i yQ (the un-mixed polarisations up to constant factors); MODE is compile-time
template <int MODE>
__device__ __forceinline__ void detect_acc(float (&acc)[nprod_of_mode(MODE)], float2 P, float2 Q) {
    const float pp = 0.25f * (P.x * P.x + P.y * P.y);
    const float qq = 0.25f * (Q.x * Q.x + Q.y * Q.y);
    if (MODE == B2F_POL_I) {
        acc[0] += pp + qq;
    } else if (MODE == B2F_POL_P0) {
        acc[0] += pp;
    } else if (MODE == B2F_POL_P1) {
        acc[0] += qq;
    } else if (MODE == B2F_POL_I2) {
        const float s = pp + qq;
        acc[0] = fmaf(s, s, acc[0]);
    } else if (MODE == B2F_POL_PPQQ) {
        acc[0] += pp;
        acc[nprod_of_mode(MODE) > 1 ? 1 : 0] += qq;
    } else {
        // yP yQ* = (i/4) P conj(Q):  Re = -Im(P conj Q)/4,  Im = Re(P conj Q)/4
        constexpr int n = nprod_of_mode(MODE);
        const float xr = P.x * Q.x + P.y * Q.y, xi = P.y * Q.x - P.x * Q.y;
        const float re = -0.25f * xi, im = 0.25f * xr;
        if (MODE == B2F_POL_COHERENCE) {
            acc[0] += pp; acc[1 % n] += qq; acc[2 % n] += re; acc[3 % n] += im;
        } else {
            acc[0] += pp + qq; acc[1 % n] += 2.f * re; acc[2 % n] += 2.f * im; acc[3 % n] += pp - qq;
        }
    }
}

template <int TR, int PT>
struct KBSmem {
    static constexpr int R = TR * PT;
    static constexpr int N = R / 2;
    static constexpr int RW = 32 / TR;                          // rows one warp transforms per pass
    static constexpr int kWarps = kKBThreads / 32;
    // rows of different row slots that share a half-warp must not share banks: short rows are padded
    static constexpr int kPitch = R * (int)sizeof(float2) + (TR < 16 ? TR * (int)sizeof(float2) : 0);
    static constexpr int kRows = RW * kPitch;
    static constexpr int kXch = RW * TR * (PT + 1) * (int)sizeof(float2);   // aliases the rows just consumed
    static constexpr int kBody = kRows > kXch ? kRows : kXch;
    static constexpr int kEps = N * (int)sizeof(float2);
    static constexpr int kStage = (kBody + kEps + 127) / 128 * 128;
    static constexpr int kWarpBytes = kKBStages * kStage;
    static constexpr int kTw = PT * TR * (int)sizeof(float2);
    static constexpr int kBarBytes = (kWarps * kKBStages * 8 + 127) / 128 * 128;
    static constexpr size_t kBytes = kBarBytes + (size_t)kWarps * kWarpBytes + kTw;
};

// Every warp is its own pipeline: it owns whole time-integration groups (D consecutive rows
// of one FFT block), walks them RW rows per pass, and keeps a private two-stage TMA ring
// (cp.async.bulk + mbarrier) so the next pass's rows land in shared memory while this pass is
// transformed.  Nothing in the loop synchronises the block.
template <int TR, int PT, int MODE>
__global__ void __launch_bounds__(kKBThreads, 2) kb_row_pass(const KBParams p) {
    using S = KBSmem<TR, PT>;
    constexpr int NPROD = nprod_of_mode(MODE);
    constexpr int R = TR * PT, N = R / 2, RW = S::RW, QPT = PT / TR, HP = TR / 2;
    extern __shared__ __align__(128) uint8_t kb_smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = lane % TR, rsw = lane / TR;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(kb_smem) + kKBStages * warp;
    uint8_t* stage0 = kb_smem + S::kBarBytes + (size_t)warp * S::kWarpBytes;
    float2* s_tw = reinterpret_cast<float2*>(kb_smem + S::kBarBytes + (size_t)S::kWarps * S::kWarpBytes);

    for (int i = tid; i < PT * TR; i += kKBThreads) s_tw[i] = p.tab_r[i];
    if (lane == 0) {
        for (int k = 0; k < kKBStages; ++k) mbar_init(&mbar[k], 1);
        mbar_fence_init();
    }
    __syncthreads();

    const int D = MODE == kModeSpectrum ? 1 : p.D;
    const int GW = D > RW ? D : RW;                 // rows per group
    const int passes = GW / RW;
    const int nout = GW / D;                        // output samples per group (1 unless D < RW)
    const int slots_per_out = RW / nout;
    const int groups_per_blk = kL / GW;
    const int64_t ngroups = (p.gb_end - p.gb_begin) * groups_per_blk;      // groups of this launch
    const int64_t wstride = (int64_t)gridDim.x * S::kWarps;

    auto issue = [&](int64_t grp, int pass, int buf) {
        const int64_t lb = grp / groups_per_blk;                // block index inside this launch
        const int64_t gb = p.gb_begin + lb;
        const int row0 = (int)(grp % groups_per_blk) * GW + pass * RW;
        uint8_t* dst = stage0 + buf * S::kStage;
        const float2* src = p.inter + (lb * (int64_t)kL + row0) * R;
        fence_proxy_async();
        if (lane == 0)
            mbar_expect_tx(&mbar[buf], (uint32_t)(RW * R * sizeof(float2) + ((pass == 0 && MODE != kModeSpectrum) ? S::kEps : 0)));
        __syncwarp();
        if (S::kPitch == R * (int)sizeof(float2)) {
            if (lane == 0) bulk_g2s(dst, src, (uint32_t)(RW * R * sizeof(float2)), &mbar[buf]);
        } else if (lane < RW) {
            bulk_g2s(dst + lane * S::kPitch, src + (int64_t)lane * R, (uint32_t)(R * sizeof(float2)), &mbar[buf]);
        }
        if (lane == 0 && pass == 0 && MODE != kModeSpectrum) bulk_g2s(dst + S::kBody, p.eps + gb * N, (uint32_t)S::kEps, &mbar[buf]);
    };

    int64_t grp_cur = (int64_t)blockIdx.x * S::kWarps + warp;
    int pass_cur = 0;
    auto advance = [&](int64_t& g, int& ps) {
        if (++ps == passes) { ps = 0; g += wstride; }
    };
    // the issue pointer runs kKBStages - 1 tiles ahead of the tile being transformed
    int64_t grp_iss = grp_cur;
    int pass_iss = 0, iss = 0;
    for (int k = 0; k < kKBStages - 1 && grp_iss < ngroups; ++k) {
        issue(grp_iss, pass_iss, iss % kKBStages);
        ++iss;
        advance(grp_iss, pass_iss);
    }

    float acc[QPT][HP][NPROD];
    float2 e[QPT][HP];
    int it = 0;
    while (grp_cur < ngroups) {
        const int buf = it % kKBStages;
        // the stage consumed one iteration ago (program order) is free: refill it
        if (grp_iss < ngroups) {
            issue(grp_iss, pass_iss, iss % kKBStages);
            ++iss;
            advance(grp_iss, pass_iss);
        }

        mbar_wait(&mbar[buf], (it / kKBStages) & 1);
        uint8_t* st = stage0 + buf * S::kStage;
        const float2* tile = reinterpret_cast<const float2*>(st + rsw * S::kPitch);
        if (pass_cur == 0 && MODE != kModeSpectrum) {
            const float2* s_eps = reinterpret_cast<const float2*>(st + S::kBody);
#pragma unroll
            for (int j = 0; j < QPT; ++j)
#pragma unroll
                for (int pp = 0; pp < HP; ++pp) {
                    e[j][pp] = s_eps[(s + TR * j) + PT * pp];
#pragma unroll
                    for (int k = 0; k < NPROD; ++k) acc[j][pp][k] = 0.f;
                }
        }
        float2 v[PT];
#pragma unroll
        for (int a = 0; a < PT; ++a) v[a] = tile[s + TR * a];
        fft_inreg<PT, false>(v);
#pragma unroll
        for (int q = 1; q < PT; ++q) v[q] = cmul(v[q], s_tw[q * TR + s]);
        // transpose PT x TR through the (now consumed) row area of this stage
        float2* myx = reinterpret_cast<float2*>(st) + (size_t)rsw * TR * (PT + 1);
        __syncwarp();
#pragma unroll
        for (int q = 0; q < PT; ++q) myx[s * (PT + 1) + q] = v[q];
        __syncwarp();
        float2 z[QPT][TR];
#pragma unroll
        for (int j = 0; j < QPT; ++j)
#pragma unroll
            for (int t = 0; t < TR; ++t) z[j][t] = myx[t * (PT + 1) + s + TR * j];
#pragma unroll
        for (int j = 0; j < QPT; ++j) fft_inreg<TR, false>(z[j]);
        if (MODE == kModeSpectrum) {
            // z[j][pp] = Z[k2 = this row][c = (s + TR j) + PT pp]: store the whole row
            const int64_t lb = grp_cur / groups_per_blk;
            const int row = (int)(grp_cur % groups_per_blk) * GW + pass_cur * RW + rsw;
            float2* dst = p.spec + (lb * (int64_t)kL + row) * R;
#pragma unroll
            for (int j = 0; j < QPT; ++j)
#pragma unroll
                for (int pp = 0; pp < TR; ++pp) dst[(s + TR * j) + PT * pp] = z[j][pp];
            advance(grp_cur, pass_cur);
            ++it;
            continue;
        }
        // z[j][pp] = Z_c at c = (s + TR j) + PT pp.  Mirror R-1-c lives in lane s^(TR-1),
        // register [QPT-1-j][TR-1-pp].
#pragma unroll
        for (int j = 0; j < QPT; ++j)
#pragma unroll
            for (int pp = 0; pp < HP; ++pp) {
                const float2 a = z[j][pp];
                const float2 bs = z[QPT - 1 - j][TR - 1 - pp];
                const float bx = __shfl_xor_sync(0xffffffffu, bs.x, TR - 1);
                const float by = __shfl_xor_sync(0xffffffffu, bs.y, TR - 1);
                const float2 bp = make_float2(bx - e[j][pp].x, -by - e[j][pp].y);
                if (MODE == B2F_POL_I) {
                    // |yP|^2 + |yQ|^2 = (|a + b'|^2 + |a - b'|^2) / 4 = (|a|^2 + |b'|^2) / 2: no need to form P and Q
                    float t = a.x * a.x;
                    t = fmaf(a.y, a.y, t);
                    t = fmaf(bp.x, bp.x, t);
                    t = fmaf(bp.y, bp.y, t);
                    acc[j][pp][0] = fmaf(0.5f, t, acc[j][pp][0]);
                } else {
                    detect_acc<MODE == kModeSpectrum ? B2F_POL_P0 : MODE>(acc[j][pp], make_float2(a.x + bp.x, a.y + bp.y), make_float2(a.x - bp.x, a.y - bp.y));
                }
            }
        if (pass_cur == passes - 1) {
            // add up the row slots that integrate into the same output sample
            for (int m = TR; m < TR * slots_per_out; m <<= 1) {
#pragma unroll
                for (int j = 0; j < QPT; ++j)
#pragma unroll
                    for (int pp = 0; pp < HP; ++pp)
#pragma unroll
                        for (int k = 0; k < NPROD; ++k)
                            acc[j][pp][k] += __shfl_xor_sync(0xffffffffu, acc[j][pp][k], m);
            }
            if (rsw % slots_per_out == 0) {
                const int64_t gb = p.gb_begin + grp_cur / groups_per_blk;
                const int ifi = (int)(gb / p.nblk);
                const int64_t blk = gb % p.nblk;
                const int g0 = (int)(grp_cur % groups_per_blk) * GW;
                const int64_t t = p.row0 + (blk * kL + g0) / D + rsw / slots_per_out;
                float* dst = p.F + ifi * p.F_if_stride + t * (int64_t)(NPROD * N);
#pragma unroll
                for (int k = 0; k < NPROD; ++k)
#pragma unroll
                    for (int j = 0; j < QPT; ++j)
#pragma unroll
                        for (int pp = 0; pp < HP; ++pp) dst[k * N + (s + TR * j) + PT * pp] = acc[j][pp][k];
            }
        }
        advance(grp_cur, pass_cur);
        ++it;
    }
}

// Row pass over the block layout the round-2 column kernel writes, [R/2 column pairs][512 rows][2 columns] float2 per block
// (b2f_fused.cuh): a row is R/2 pieces of 16 bytes, 8 KiB apart, so the per-warp ring is filled with cp.async (LDGSTS)
// pieces -- two neighbouring rows of a pair are one 32-byte sector -- instead of one bulk copy.  From HBM that access
// pattern costs twice the time of kb_row_pass's contiguous rows (28.8 vs 15.0 ms per 20 s of C2): this kernel exists for the
// two-launch form of the round-2 path (B2F_PATH=split), a debugging and profiling aid.  Everything after the load is kb_row_pass: each warp owns whole integration groups, the next pass's
// rows land while this pass is transformed, nothing synchronises the block.
template <int TR, int PT, int MODE>
__global__ void __launch_bounds__(kKBThreads, 2) kr_row_pass(const KBParams p) {
    using S = KBSmem<TR, PT>;
    constexpr int NPROD = nprod_of_mode(MODE);
    constexpr int R = TR * PT, N = R / 2, RW = S::RW, QPT = PT / TR, HP = TR / 2;
    extern __shared__ __align__(128) uint8_t kb_smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = lane % TR, rsw = lane / TR;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(kb_smem) + kKBStages * warp;
    uint8_t* stage0 = kb_smem + S::kBarBytes + (size_t)warp * S::kWarpBytes;
    float2* s_tw = reinterpret_cast<float2*>(kb_smem + S::kBarBytes + (size_t)S::kWarps * S::kWarpBytes);

    for (int i = tid; i < PT * TR; i += kKBThreads) s_tw[i] = p.tab_r[i];
    (void)mbar;
    __syncthreads();

    const int D = MODE == kModeSpectrum ? 1 : p.D;
    const int GW = D > RW ? D : RW;                 // rows per group
    const int passes = GW / RW;
    const int nout = GW / D;                        // output samples per group (1 unless D < RW)
    const int slots_per_out = RW / nout;
    const int groups_per_blk = kL / GW;
    const int64_t ngroups = (p.gb_end - p.gb_begin) * groups_per_blk;      // groups of this launch
    const int64_t wstride = (int64_t)gridDim.x * S::kWarps;

    auto issue = [&](int64_t grp, int pass, int buf) {
        const int64_t lb = grp / groups_per_blk;                // block index inside this launch
        const int64_t gb = p.gb_begin + lb;
        const int row0 = (int)(grp % groups_per_blk) * GW + pass * RW;
        uint8_t* dst = stage0 + buf * S::kStage;
        const float2* src = p.inter + lb * (int64_t)kL * R;     // block slot [32 row tiles][column pair][16 rows][2 columns]
        __syncwarp();                                           // everybody is done with the tile this refills
        constexpr int NPC = RW * (R / 2);                       // 16-byte pieces: lane -> (pair, row), row fastest
#pragma unroll
        for (int k = 0; k < (NPC + 31) / 32; ++k) {
            const int idx = lane + 32 * k;
            if (NPC % 32 == 0 || idx < NPC) {
                const int r = idx % RW, pp = idx / RW;
                const int m = row0 + r;
                cp_async16(dst + r * S::kPitch + pp * 16, src + ((((m >> 4) * (R / 2) + pp) * 16 + (m & 15)) * 2));
            }
        }
        if (pass == 0 && MODE != kModeSpectrum)
            for (int idx = lane; idx < N / 2; idx += 32) cp_async16(dst + S::kBody + idx * 16, p.eps + gb * N + idx * 2);
    };

    int64_t grp_cur = (int64_t)blockIdx.x * S::kWarps + warp;
    int pass_cur = 0;
    auto advance = [&](int64_t& g, int& ps) {
        if (++ps == passes) { ps = 0; g += wstride; }
    };
    // the issue pointer runs kKBStages - 1 tiles ahead of the tile being transformed
    int64_t grp_iss = grp_cur;
    int pass_iss = 0, iss = 0;
    for (int k = 0; k < kKBStages - 1; ++k) {
        if (grp_iss < ngroups) {
            issue(grp_iss, pass_iss, iss % kKBStages);
            ++iss;
            advance(grp_iss, pass_iss);
        }
        cp_async_commit();
    }

    float acc[QPT][HP][NPROD];
    float2 e[QPT][HP];
    int it = 0;
    while (grp_cur < ngroups) {
        const int buf = it % kKBStages;
        // the stage consumed one iteration ago (program order) is free: refill it
        if (grp_iss < ngroups) {
            issue(grp_iss, pass_iss, iss % kKBStages);
            ++iss;
            advance(grp_iss, pass_iss);
        }
        cp_async_commit();                              // one group per iteration (possibly empty): uniform accounting
        cp_async_wait<kKBStages - 1>();                 // everything but the newest kKBStages - 1 groups has landed
        __syncwarp();
        uint8_t* st = stage0 + buf * S::kStage;
        const float2* tile = reinterpret_cast<const float2*>(st + rsw * S::kPitch);
        if (pass_cur == 0 && MODE != kModeSpectrum) {
            const float2* s_eps = reinterpret_cast<const float2*>(st + S::kBody);
#pragma unroll
            for (int j = 0; j < QPT; ++j)
#pragma unroll
                for (int pp = 0; pp < HP; ++pp) {
                    e[j][pp] = s_eps[(s + TR * j) + PT * pp];
#pragma unroll
                    for (int k = 0; k < NPROD; ++k) acc[j][pp][k] = 0.f;
                }
        }
        float2 v[PT];
#pragma unroll
        for (int a = 0; a < PT; ++a) v[a] = tile[s + TR * a];
        fft_inreg<PT, false>(v);
#pragma unroll
        for (int q = 1; q < PT; ++q) v[q] = cmul(v[q], s_tw[q * TR + s]);
        // transpose PT x TR through the (now consumed) row area of this stage
        float2* myx = reinterpret_cast<float2*>(st) + (size_t)rsw * TR * (PT + 1);
        __syncwarp();
#pragma unroll
        for (int q = 0; q < PT; ++q) myx[s * (PT + 1) + q] = v[q];
        __syncwarp();
        float2 z[QPT][TR];
#pragma unroll
        for (int j = 0; j < QPT; ++j)
#pragma unroll
            for (int t = 0; t < TR; ++t) z[j][t] = myx[t * (PT + 1) + s + TR * j];
#pragma unroll
        for (int j = 0; j < QPT; ++j) fft_inreg<TR, false>(z[j]);
        if (MODE == kModeSpectrum) {
            // z[j][pp] = Z[k2 = this row][c = (s + TR j) + PT pp]: store the whole row
            const int64_t lb = grp_cur / groups_per_blk;
            const int row = (int)(grp_cur % groups_per_blk) * GW + pass_cur * RW + rsw;
            float2* dst = p.spec + (lb * (int64_t)kL + row) * R;
#pragma unroll
            for (int j = 0; j < QPT; ++j)
#pragma unroll
                for (int pp = 0; pp < TR; ++pp) dst[(s + TR * j) + PT * pp] = z[j][pp];
            advance(grp_cur, pass_cur);
            ++it;
            continue;
        }
        // z[j][pp] = Z_c at c = (s + TR j) + PT pp.  Mirror R-1-c lives in lane s^(TR-1),
        // register [QPT-1-j][TR-1-pp].
#pragma unroll
        for (int j = 0; j < QPT; ++j)
#pragma unroll
            for (int pp = 0; pp < HP; ++pp) {
                const float2 a = z[j][pp];
                const float2 bs = z[QPT - 1 - j][TR - 1 - pp];
                const float bx = __shfl_xor_sync(0xffffffffu, bs.x, TR - 1);
                const float by = __shfl_xor_sync(0xffffffffu, bs.y, TR - 1);
                const float2 bp = make_float2(bx - e[j][pp].x, -by - e[j][pp].y);
                if (MODE == B2F_POL_I) {
                    // |yP|^2 + |yQ|^2 = (|a + b'|^2 + |a - b'|^2) / 4 = (|a|^2 + |b'|^2) / 2: no need to form P and Q
                    float t = a.x * a.x;
                    t = fmaf(a.y, a.y, t);
                    t = fmaf(bp.x, bp.x, t);
                    t = fmaf(bp.y, bp.y, t);
                    acc[j][pp][0] = fmaf(0.5f, t, acc[j][pp][0]);
                } else {
                    detect_acc<MODE == kModeSpectrum ? B2F_POL_P0 : MODE>(acc[j][pp], make_float2(a.x + bp.x, a.y + bp.y), make_float2(a.x - bp.x, a.y - bp.y));
                }
            }
        if (pass_cur == passes - 1) {
            // add up the row slots that integrate into the same output sample
            for (int m = TR; m < TR * slots_per_out; m <<= 1) {
#pragma unroll
                for (int j = 0; j < QPT; ++j)
#pragma unroll
                    for (int pp = 0; pp < HP; ++pp)
#pragma unroll
                        for (int k = 0; k < NPROD; ++k)
                            acc[j][pp][k] += __shfl_xor_sync(0xffffffffu, acc[j][pp][k], m);
            }
            if (rsw % slots_per_out == 0) {
                const int64_t gb = p.gb_begin + grp_cur / groups_per_blk;
                const int ifi = (int)(gb / p.nblk);
                const int64_t blk = gb % p.nblk;
                const int g0 = (int)(grp_cur % groups_per_blk) * GW;
                const int64_t t = p.row0 + (blk * kL + g0) / D + rsw / slots_per_out;
                float* dst = p.F + ifi * p.F_if_stride + t * (int64_t)(NPROD * N);
#pragma unroll
                for (int k = 0; k < NPROD; ++k)
#pragma unroll
                    for (int j = 0; j < QPT; ++j)
#pragma unroll
                        for (int pp = 0; pp < HP; ++pp) dst[k * N + (s + TR * j) + PT * pp] = acc[j][pp][k];
            }
        }
        advance(grp_cur, pass_cur);
        ++it;
    }
    cp_async_wait<0>();
}


// ================================================================== kernel 2: dedispersion back end
// Dedispersion path only (digifil -D dm -F nchan:D).  Input: the full spectrum Z[k2][k1] of one
// overlap-save block (forward column pass + row FFT).  One CTA owns 8 channels x 2 polarisations =
// 16 lanes and, per lane, un-mixes the polarisation (Z[k] with conj Z[M-k]), multiplies by the
// chirp H[c][k2], runs the 512-point backward FFT (16 x 32, one exchange), keeps samples
// [nfilt_pos, 512 - nfilt_neg), detects (partner polarisation by shuffle) and integrates D samples.
struct KCParams {
    const float2* spec;         // [gb - gb_begin][512][R]
    const float2* chirp;        // [ndm][nif][512][N]  H[c][k2] stored k2-major
    const float2* tab_w;        // [32][16] W_512^(l q)
    float* F; int64_t F_if_stride; int64_t row0;  // F slot of (trial t, IF i): t * nif + i
    int nblk, nif, D, mode, nfilt_pos, keep;      // keep = 512 - nfilt_pos - nfilt_neg (multiple of D)
    int64_t gb_begin, gb_end;
    int ndm;                                      // trial DMs (kc_dedisp_trials); kc_dedisp_back runs trial 0
};

constexpr size_t kKCSmemBytes = (size_t)(kL * 16 + 512) * sizeof(float2);

// (z1 + conj z2)/2 for pol 0, (z1 - conj z2)/(2i) for pol 1: the spectrum of one polarisation from the mixed block spectrum
__device__ __forceinline__ float2 kc_unmix(float2 z1, float2 z2, int pol) {
    float2 x;
    if (pol == 0) x = make_float2(0.5f * (z1.x + z2.x), 0.5f * (z1.y - z2.y));
    else          x = make_float2(0.5f * (z1.y + z2.y), -0.5f * (z1.x - z2.x));
    return x;
}

// Spectrum bin k2 = 32 a + item + 16 h of channel c, and its mirror M - (c L + k2): row L - k2, channel R-1-c (k2 > 0) or
// row 0, channel (R-c) mod R.
template <int R>
__device__ __forceinline__ float2 kc_load_unmixed(const float2* Z, int k2, int c, int pol) {
    const float2 z1 = Z[(int64_t)k2 * R + c];
    const float2 z2 = k2 ? Z[(int64_t)(kL - k2) * R + (R - 1 - c)] : Z[(R - c) & (R - 1)];
    return kc_unmix(z1, z2, pol);
}

// Everything after the chirp for one (block, 8-channel strip): vA / vB hold the chirped bins k2 = 32 a + item (+ 16).
// IFFT_16 over a, twiddle, exchange, IFFT_32 over l, detect into shared memory, integrate D kept samples per output row
// into F slot `slot` (trial * nif + IF).  Ends with a barrier: the shared buffers are free again.
template <int R>
__device__ __forceinline__ void kc_backward_detect(float2 (&vA)[16], float2 (&vB)[16], const KCParams& p, float4* data4, float* pw,
                                                   const float2* s_w, int nprod, bool own_only, int slot, int64_t blk, int strip) {
    constexpr int N = R / 2;
    const int tid = threadIdx.x, lane16 = tid & 15, item = tid >> 4;
    const int ch8 = lane16 >> 1, pol = lane16 & 1;
    {
        fft_inreg<16, true>(vA);
        fft_inreg<16, true>(vB);
        const float4* twA = reinterpret_cast<const float4*>(s_w + item * 16);
        const float4* twB = reinterpret_cast<const float4*>(s_w + (item + 16) * 16);
#pragma unroll
        for (int q = 0; q < 16; q += 2) {            // * conj W_512^(l m_lo)
            const float4 ta = twA[q >> 1], tb = twB[q >> 1];
            if (q) vA[q] = cmul_conj(vA[q], make_float2(ta.x, ta.y));
            vA[q + 1] = cmul_conj(vA[q + 1], make_float2(ta.z, ta.w));
            if (q) vB[q] = cmul_conj(vB[q], make_float2(tb.x, tb.y));
            vB[q + 1] = cmul_conj(vB[q + 1], make_float2(tb.z, tb.w));
        }
#pragma unroll
        for (int q = 0; q < 16; ++q)
            data4[(q * 16 + item) * 16 + lane16] = make_float4(vA[q].x, vA[q].y, vB[q].x, vB[q].y);
    }
    __syncthreads();
    // ---- P2: IFFT_32 over l for m_lo = item -> y[m = m_lo + 16 m_hi]; detect into smem
    {
        float2 u[32];
#pragma unroll
        for (int l = 0; l < 16; ++l) {
            const float4 t = data4[(item * 16 + l) * 16 + lane16];
            u[l] = make_float2(t.x, t.y);
            u[l + 16] = make_float2(t.z, t.w);
        }
        fft_inreg<32, true>(u);
        __syncthreads();                   // everyone has its u[]: the exchange buffer becomes the power buffer
        if (own_only) {
            // products without a cross term: every lane squares its own polarisation, [m][ch][pol]
#pragma unroll
            for (int mh = 0; mh < 32; ++mh)
                pw[(size_t)(item + 16 * mh) * 16 + lane16] = u[mh].x * u[mh].x + u[mh].y * u[mh].y;
        } else {
#pragma unroll
        for (int mh = 0; mh < 32; ++mh) {
            const float ox = __shfl_xor_sync(0xffffffffu, u[mh].x, 1), oy = __shfl_xor_sync(0xffffffffu, u[mh].y, 1);
            if (pol == 0) {                 // this lane holds yP, its neighbour yQ
                const float2 yP = u[mh], yQ = make_float2(ox, oy);
                const float pp = yP.x * yP.x + yP.y * yP.y, qq = yQ.x * yQ.x + yQ.y * yQ.y;
                const float re = yP.x * yQ.x + yP.y * yQ.y, im = yP.y * yQ.x - yP.x * yQ.y;   // yP conj(yQ)
                float* dst = pw + (size_t)(item + 16 * mh) * 8 + ch8;
                constexpr size_t PS = (size_t)kL * 8;        // product stride
                switch (p.mode) {
                    case B2F_POL_I2: dst[0] = (pp + qq) * (pp + qq); break;
                    case B2F_POL_COHERENCE: dst[0] = pp; dst[PS] = qq; dst[2 * PS] = re; dst[3 * PS] = im; break;
                    default: dst[0] = pp + qq; dst[PS] = 2.f * re; dst[2 * PS] = 2.f * im; dst[3 * PS] = pp - qq; break;
                }
            }
        }
        }
    }
    __syncthreads();
    // ---- integrate D kept samples per output row
    const int nrow = p.keep / p.D;
    const int64_t t0 = p.row0 + blk * nrow;
    for (int o = tid; o < nprod * nrow * 8; o += 256) {
        const int ch = o & 7, r = (o >> 3) % nrow, k = (o >> 3) / nrow;
        float sum = 0.f;
        if (own_only) {
            const float2* src = reinterpret_cast<const float2*>(pw) + (size_t)(p.nfilt_pos + r * p.D) * 8 + ch;
            float s0 = 0.f, s1 = 0.f;
            for (int i = 0; i < p.D; ++i) {
                const float2 v = src[i * 8];
                s0 += v.x;
                s1 += v.y;
            }
            sum = p.mode == B2F_POL_I ? s0 + s1 : p.mode == B2F_POL_P0 ? s0 : p.mode == B2F_POL_P1 ? s1 : (k == 0 ? s0 : s1);
        } else {
            const float* src = pw + ((size_t)k * kL + p.nfilt_pos + r * p.D) * 8 + ch;
            for (int i = 0; i < p.D; ++i) sum += src[i * 8];
        }
        p.F[slot * p.F_if_stride + (t0 + r) * (int64_t)(nprod * N) + k * N + strip * 8 + ch] = sum;
    }
    __syncthreads();
}

template <int R>
__global__ void __launch_bounds__(256, 2) kc_dedisp_back(const KCParams p) {
    constexpr int N = R / 2;
    extern __shared__ __align__(16) uint8_t kc_smem[];
    float4* data4 = reinterpret_cast<float4*>(kc_smem);             // [256 pairs][16 lanes]
    float* pw = reinterpret_cast<float*>(kc_smem);                  // aliases data: [prod][512][8 ch]
    float2* s_w = reinterpret_cast<float2*>(kc_smem) + kL * 16;     // [32][16] W_512^(l q)
    const int tid = threadIdx.x, lane16 = tid & 15, item = tid >> 4;
    const int ch8 = lane16 >> 1, pol = lane16 & 1;
    for (int i = tid; i < 512; i += 256) s_w[i] = p.tab_w[i];
    __syncthreads();

    const int nstrips = N / 8;
    const int nprod = nprod_of_mode(p.mode);
    const bool own_only = p.mode == B2F_POL_P0 || p.mode == B2F_POL_P1 || p.mode == B2F_POL_I || p.mode == B2F_POL_PPQQ;
    const int64_t nwork = (p.gb_end - p.gb_begin) * nstrips;
    for (int64_t w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int64_t lb = w / nstrips;
        const int64_t gb = p.gb_begin + lb;
        const int ifi = (int)(gb / p.nblk);
        const int64_t blk = gb % p.nblk;
        const int c = (int)(w % nstrips) * 8 + ch8;
        const float2* Z = p.spec + lb * (int64_t)kL * R;
        const float2* H = p.chirp + (int64_t)ifi * kL * N;

        // ---- P1: un-mix + chirp on load, IFFT_16 over a (k2 = 32 a + l) for l = item, item + 16
        {
            float2 vA[16], vB[16];
#pragma unroll
            for (int a = 0; a < 16; ++a) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int k2 = 32 * a + item + 16 * h;
                    const float2 z1 = Z[(int64_t)k2 * R + c];
                    // mirror bin M - (c L + k2): row L - k2, channel R-1-c (k2 > 0) or row 0, channel (R-c) mod R
                    const float2 z2 = k2 ? Z[(int64_t)(kL - k2) * R + (R - 1 - c)] : Z[(R - c) & (R - 1)];
                    float2 x;
                    if (pol == 0) x = make_float2(0.5f * (z1.x + z2.x), 0.5f * (z1.y - z2.y));          // (z1 + conj z2)/2
                    else          x = make_float2(0.5f * (z1.y + z2.y), -0.5f * (z1.x - z2.x));         // (z1 - conj z2)/(2i)
                    x = cmul(x, H[(int64_t)k2 * N + c]);
                    if (h == 0) vA[a] = x; else vB[a] = x;
                }
            }
            fft_inreg<16, true>(vA);
            fft_inreg<16, true>(vB);
            const float4* twA = reinterpret_cast<const float4*>(s_w + item * 16);
            const float4* twB = reinterpret_cast<const float4*>(s_w + (item + 16) * 16);
#pragma unroll
            for (int q = 0; q < 16; q += 2) {            // * conj W_512^(l m_lo)
                const float4 ta = twA[q >> 1], tb = twB[q >> 1];
                if (q) vA[q] = cmul_conj(vA[q], make_float2(ta.x, ta.y));
                vA[q + 1] = cmul_conj(vA[q + 1], make_float2(ta.z, ta.w));
                if (q) vB[q] = cmul_conj(vB[q], make_float2(tb.x, tb.y));
                vB[q + 1] = cmul_conj(vB[q + 1], make_float2(tb.z, tb.w));
            }
#pragma unroll
            for (int q = 0; q < 16; ++q)
                data4[(q * 16 + item) * 16 + lane16] = make_float4(vA[q].x, vA[q].y, vB[q].x, vB[q].y);
        }
        __syncthreads();
        // ---- P2: IFFT_32 over l for m_lo = item -> y[m = m_lo + 16 m_hi]; detect into smem
        {
            float2 u[32];
#pragma unroll
            for (int l = 0; l < 16; ++l) {
                const float4 t = data4[(item * 16 + l) * 16 + lane16];
                u[l] = make_float2(t.x, t.y);
                u[l + 16] = make_float2(t.z, t.w);
            }
            fft_inreg<32, true>(u);
            __syncthreads();                   // everyone has its u[]: the exchange buffer becomes the power buffer
            if (own_only) {
                // products without a cross term: every lane squares its own polarisation, [m][ch][pol]
#pragma unroll
                for (int mh = 0; mh < 32; ++mh)
                    pw[(size_t)(item + 16 * mh) * 16 + lane16] = u[mh].x * u[mh].x + u[mh].y * u[mh].y;
            } else {
#pragma unroll
            for (int mh = 0; mh < 32; ++mh) {
                const float ox = __shfl_xor_sync(0xffffffffu, u[mh].x, 1), oy = __shfl_xor_sync(0xffffffffu, u[mh].y, 1);
                if (pol == 0) {                 // this lane holds yP, its neighbour yQ
                    const float2 yP = u[mh], yQ = make_float2(ox, oy);
                    const float pp = yP.x * yP.x + yP.y * yP.y, qq = yQ.x * yQ.x + yQ.y * yQ.y;
                    const float re = yP.x * yQ.x + yP.y * yQ.y, im = yP.y * yQ.x - yP.x * yQ.y;   // yP conj(yQ)
                    float* dst = pw + (size_t)(item + 16 * mh) * 8 + ch8;
                    constexpr size_t PS = (size_t)kL * 8;        // product stride
                    switch (p.mode) {
                        case B2F_POL_I2: dst[0] = (pp + qq) * (pp + qq); break;
                        case B2F_POL_COHERENCE: dst[0] = pp; dst[PS] = qq; dst[2 * PS] = re; dst[3 * PS] = im; break;
                        default: dst[0] = pp + qq; dst[PS] = 2.f * re; dst[2 * PS] = 2.f * im; dst[3 * PS] = pp - qq; break;
                    }
                }
            }
            }
        }
        __syncthreads();
        // ---- integrate D kept samples per output row
        const int nrow = p.keep / p.D;
        const int64_t t0 = p.row0 + blk * nrow;
        for (int o = tid; o < nprod * nrow * 8; o += 256) {
            const int ch = o & 7, r = (o >> 3) % nrow, k = (o >> 3) / nrow;
            float sum = 0.f;
            if (own_only) {
                const float2* src = reinterpret_cast<const float2*>(pw) + (size_t)(p.nfilt_pos + r * p.D) * 8 + ch;
                float s0 = 0.f, s1 = 0.f;
                for (int i = 0; i < p.D; ++i) {
                    const float2 v = src[i * 8];
                    s0 += v.x;
                    s1 += v.y;
                }
                sum = p.mode == B2F_POL_I ? s0 + s1 : p.mode == B2F_POL_P0 ? s0 : p.mode == B2F_POL_P1 ? s1 : (k == 0 ? s0 : s1);
            } else {
                const float* src = pw + ((size_t)k * kL + p.nfilt_pos + r * p.D) * 8 + ch;
                for (int i = 0; i < p.D; ++i) sum += src[i * 8];
            }
            p.F[ifi * p.F_if_stride + (t0 + r) * (int64_t)(nprod * N) + k * N + (int)(w % nstrips) * 8 + ch] = sum;
        }
        __syncthreads();
    }
}

// Several trial DMs in one pass (b2f_params.ndm): per (block, 8-channel strip) the spectrum is loaded and un-mixed once and
// kept in registers (64 per thread, hence one CTA of 256 threads per SM); then, for each trial, the same chirp multiply,
// backward FFT, overlap discard, detection and integration as kc_dedisp_back, into that trial's F slots.  The arithmetic
// per trial is kc_dedisp_back's, so every trial is bit-identical to a single-DM plan with the same nfilt.
template <int R>
__global__ void __launch_bounds__(256, 1) kc_dedisp_trials(const KCParams p) {
    constexpr int N = R / 2;
    extern __shared__ __align__(16) uint8_t kc_smem[];
    float4* data4 = reinterpret_cast<float4*>(kc_smem);
    float* pw = reinterpret_cast<float*>(kc_smem);
    float2* s_w = reinterpret_cast<float2*>(kc_smem) + kL * 16;
    const int tid = threadIdx.x, lane16 = tid & 15, item = tid >> 4;
    const int ch8 = lane16 >> 1, pol = lane16 & 1;
    for (int i = tid; i < 512; i += 256) s_w[i] = p.tab_w[i];
    __syncthreads();

    const int nstrips = N / 8;
    const int nprod = nprod_of_mode(p.mode);
    const bool own_only = p.mode == B2F_POL_P0 || p.mode == B2F_POL_P1 || p.mode == B2F_POL_I || p.mode == B2F_POL_PPQQ;
    const int64_t nwork = (p.gb_end - p.gb_begin) * nstrips;
    for (int64_t w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int64_t lb = w / nstrips;
        const int64_t gb = p.gb_begin + lb;
        const int ifi = (int)(gb / p.nblk);
        const int64_t blk = gb % p.nblk;
        const int strip = (int)(w % nstrips);
        const int c = strip * 8 + ch8;
        const float2* Z = p.spec + lb * (int64_t)kL * R;
        float2 xA[16], xB[16];                       // un-mixed bins k2 = 32 a + item (+ 16)
#pragma unroll
        for (int a = 0; a < 16; ++a) {
            xA[a] = kc_load_unmixed<R>(Z, 32 * a + item, c, pol);
            xB[a] = kc_load_unmixed<R>(Z, 32 * a + item + 16, c, pol);
        }
        for (int t = 0; t < p.ndm; ++t) {
            const int slot = t * p.nif + ifi;
            const float2* H = p.chirp + (int64_t)slot * kL * N;
            float2 vA[16], vB[16];
#pragma unroll
            for (int a = 0; a < 16; ++a) {
                vA[a] = cmul(xA[a], H[(int64_t)(32 * a + item) * N + c]);
                vB[a] = cmul(xB[a], H[(int64_t)(32 * a + item + 16) * N + c]);
            }
            kc_backward_detect<R>(vA, vB, p, data4, pw, s_w, nprod, own_only, slot, blk, strip);
        }
    }
}

// ================================================================== generic channeliser
// Any power-of-two freq_res (L) and row length (R = 2 nchan) outside the tuned 512-point kernels,
// e.g. process_vdif's default --nchan 512 -> -F512:1024 (/root/reference/process_vdif.py:46,162) and the
// 1024 channels per IF that submit_job.py:58-76 asks for at DM 560.  Same algebra as the tuned path
// (DESIGN.md section 3).  FFTs are in-place Sande-Tukey passes of radix 16 held in registers: a pass
// over segments of length n = 16 m computes y_q[lo] = W_n^(lo q) * sum_j x[j m + lo] W_16^(j q) and
// stores it at q m + lo, so after all passes frequency k sits at its digit-reversed position.  The
// inverse undoes the passes in reverse order, so the diagonal W_M^(k2 n1) is applied in that order
// and no reordering pass exists.  The innermost pass (radix 2..16, m = 1) of the forward transform,
// the diagonal and the innermost inverse pass act on the same values and run back to back in registers.
// 2-bit input (index stream) only.
struct KGParams {
    const uint8_t* compact; size_t compact_stride;
    float2* inter;               // [gb - gb_begin][L][R]
    float2* colsum;              // [nif*nblk][R]
    const float2* eps;           // [nif*nblk][R/2]
    const float2* tw_col;        // [L]  per-pass twiddle rows for L-point FFTs, see kg_tw_offset
    const float2* tw_row;        // [R]  the same for R-point FFTs
    float* F; int64_t F_if_stride; int64_t row0;
    int L, lgL, R, lgR, C, lgC, nblk, nif, D, mode;
    int64_t M, gb_begin, gb_end;
    // 8-bit input: word masks in stream coordinates (one byte per 32 bytes of the de-framed stream, carried over with the
    // samples), blocks that hold a masked word, the offset of the code -> value map (127.5 or 128, SURVEY D3)
    const uint8_t* wmask; size_t wmask_stride;
    const uint8_t* blkdirty;
    float in8_offset;
    int64_t step;                // samples between the starts of consecutive blocks (M, or less with overlap-save)
    const float4* levels; int64_t levels_stride;   // JA98 decode: (lo0, hi0, lo1, hi1) per window of 512 stream samples and IF
    float2* volt;                // mode kModeVolt: [gb - gb_begin][L][2][R/2] un-detected channel samples (P, Q)
};
// kg_row_pass mode: no detection, the two polarisations of every channel sample go to KGParams::volt (dedispersion)
constexpr int kModeVolt = 101;

// One 32-bit word of an 8-bit stream = two time samples x (pol 0, pol 1).  `o` = byte offset of the word from s.byte0,
// which in turn counts from the start of the IF's de-framed stream of this push (carried samples included).
struct KG8 { const uint8_t* wm; int64_t byte0; float off; bool dirty; const float4* levels; };

__device__ __forceinline__ void kg_decode8(uint32_t four, const KG8& s, int64_t o, float2& a, float2& b) {
    a = make_float2((float)(four & 255u) - s.off, (float)((four >> 8) & 255u) - s.off);
    b = make_float2((float)((four >> 16) & 255u) - s.off, (float)(four >> 24) - s.off);
    if (s.dirty) {
        const int64_t w = (s.byte0 + o) >> 2;
        if ((s.wm[w >> 3] >> (w & 7)) & 1) a = b = make_float2(0.f, 0.f);
    }
}

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }

// Shared-memory index swizzles (XOR within aligned 16-element groups, so buffers need no padding).  Every pass
// reads 64-bit elements either contiguously or at the stride of the innermost passes; the swizzle keeps the 16
// lanes of a half-warp on 16 different 8-byte banks in both cases:
//   columns, layout [index][C] with C < 16: the innermost passes step 32 elements between neighbouring segments
//     -> bits 5..6 of the element number are folded into bits 2..3;
//   rows, layout [row][R]: the innermost pass steps RM = 2..16 elements, the one before it R/256, and detection
//     reads digit-reversed positions (neighbouring channels are R/16 elements apart)
//     -> bits 4..6 and 8..10 are folded into bits 0..2 and bit 7 into bit 3.
// (ncu before: 45 % of the column kernel's and 65 % of the row kernel's shared wavefronts were bank conflicts
// with one pad element per 16.)
template <bool ROWS>
__device__ __forceinline__ int kg_phys(int e) {
    return ROWS ? (e ^ (((e >> 4) ^ (e >> 8)) & 7) ^ (((e >> 7) & 1) << 3)) : (e ^ (((e >> 5) & 3) << 2));
}
__host__ __device__ constexpr size_t kg_padded(size_t n) { return (n + 15) / 16 * 16; }

// number of radix-16 passes outside the innermost one, and the innermost radix, for a 2^lg point FFT
__host__ __device__ __forceinline__ int kg_outer_passes(int lg) { return (lg - 1) / 4; }
__host__ __device__ __forceinline__ int kg_inner_lg(int lg) { return lg - 4 * ((lg - 1) / 4); }

// Twiddles of outer pass f (segments of n = len >> 4f points, m = n / 16): 15 rows of m entries,
// table[offset(f) + (q - 1) m + lo] = exp(-2 pi i lo q / n), so the lanes of a warp (consecutive lo) read
// consecutive entries.  All passes together need fewer than `len` entries.
__host__ __device__ __forceinline__ int kg_tw_offset(int lg, int f) {
    int off = 0;
    for (int g = 0; g < f; ++g) off += 15 << (lg - 4 * g - 4);
    return off;
}

// frequency index <-> position after the forward passes (base-16 digits of the segment number reversed)
__device__ __forceinline__ int kg_freq_of_pos(int pos, int lg) {
    const int nf = kg_outer_passes(lg), lgi = kg_inner_lg(lg);
    const int seg = pos >> lgi, q = pos & ((1 << lgi) - 1);
    int k = 0;
    for (int f = 0; f < nf; ++f) k |= ((seg >> (4 * (nf - 1 - f))) & 15) << (4 * f);
    return k | (q << (4 * nf));
}
__device__ __forceinline__ int kg_pos_of_freq(int k, int lg) {
    const int nf = kg_outer_passes(lg), lgi = kg_inner_lg(lg);
    int seg = 0;
    for (int f = 0; f < nf; ++f) seg |= ((k >> (4 * f)) & 15) << (4 * (nf - 1 - f));
    return (seg << lgi) | (k >> (4 * nf));
}

// One radix-16 pass over `cnt` transforms.  Sequences are interleaved [index][1 << lgC] (columns) or stored one
// after the other with lgC = 0 and `seq_len` elements each (rows).  SRC: 0 shared, 1 index bytes (decode),
// 2 global float2.  DST: 0 shared, 1 global float2.
template <bool INV, int SRC, int DST, bool ROWS>
__device__ __forceinline__ void kg_pass16(float2* sm, const float2* tw, int lgLen, int lgn, int lgC, int cnt,
                                          const uint8_t* gsrc_b, const float2* gsrc_f, float2* gdst, int64_t gstride,
                                          const float2* lut) {
    const int lgm = lgn - 4, m = 1 << lgm, lgT = lgLen - 4;         // transforms per sequence = 2^lgT
    for (int t = threadIdx.x; t < cnt; t += blockDim.x) {
        const int cl = t & ((1 << lgC) - 1), u = t >> lgC;
        const int seq = u >> lgT, w = u & ((1 << lgT) - 1);          // seq > 0 only for rows (lgC = 0)
        const int lo = w & (m - 1), seg = w >> lgm;
        const int base = (seq << lgLen) + (seg << lgn) + lo;
        const float2* twl = tw + lo;                                 // this pass's table, [q - 1][lo]: lanes read neighbours
        float2 v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int idx = base + j * m;
            if (SRC == 1) v[j] = *reinterpret_cast<const float2*>(reinterpret_cast<const uint8_t*>(lut) + gsrc_b[(int64_t)idx * gstride + cl]);
            else if (SRC == 2) v[j] = gsrc_f[(int64_t)seq * gstride + (idx & ((1 << lgLen) - 1))];
            else v[j] = sm[kg_phys<ROWS>((idx << lgC) + cl)];
        }
        if (INV) {
#pragma unroll
            for (int q = 1; q < 16; ++q) v[q] = cmul_conj(v[q], twl[(q - 1) << lgm]);
            fft_inreg<16, true>(v);
        } else {
            fft_inreg<16, false>(v);
#pragma unroll
            for (int q = 1; q < 16; ++q) v[q] = cmul(v[q], twl[(q - 1) << lgm]);
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int idx = base + j * m;
            if (DST == 1) gdst[(int64_t)idx * gstride + cl] = v[j];
            else sm[kg_phys<ROWS>((idx << lgC) + cl)] = v[j];
        }
    }
}

// Column passes with two neighbouring columns per thread: one 128-bit shared access and one twiddle read serve
// both (the shared-memory instruction queue is what the column kernel runs out of first), and the two
// independent 16-point transforms interleave.  SRC: 0 shared, 1 index bytes.  DST: 0 shared, 1 global.
template <bool INV, int SRC, int DST>
__device__ __forceinline__ void kg_pass16_pair(float2* sm, const float2* tw, int lgLen, int lgn, int lgC, int cnt,
                                               const uint8_t* gsrc_b, float2* gdst, int64_t gstride, const float2* lut,
                                               const KG8* s8 = nullptr) {
    const int lgm = lgn - 4, m = 1 << lgm, lgP = lgC - 1;           // 2^lgP column pairs per strip
    for (int t = threadIdx.x; t < cnt; t += blockDim.x) {
        const int c2 = (t & ((1 << lgP) - 1)) * 2, w = t >> lgP;
        const int lo = w & (m - 1), seg = w >> lgm;
        const int base = (seg << lgn) + lo;
        const float2* twl = tw + lo;
        float2 a[16], b[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int idx = base + j * m;
            if (SRC == 1) {
                const uint32_t two = *reinterpret_cast<const uint16_t*>(gsrc_b + (int64_t)idx * gstride + c2);
                a[j] = *reinterpret_cast<const float2*>(reinterpret_cast<const uint8_t*>(lut) + (two & 255u));
                b[j] = *reinterpret_cast<const float2*>(reinterpret_cast<const uint8_t*>(lut) + (two >> 8));
            } else if (SRC == 2) {                                   // 8-bit sample pairs
                const int64_t o = ((int64_t)idx * gstride + c2) * 2;
                kg_decode8(*reinterpret_cast<const uint32_t*>(gsrc_b + o), *s8, o, a[j], b[j]);
            } else if (SRC == 3) {                                   // index bytes, JA98 levels of the sample's window
                const int64_t o = (int64_t)idx * gstride + c2;
                const uint32_t two = *reinterpret_cast<const uint16_t*>(gsrc_b + o);
                const float4 lv = __ldg(s8->levels + ((s8->byte0 + o) >> 9));
                a[j] = kg_ja98(*reinterpret_cast<const float2*>(reinterpret_cast<const uint8_t*>(lut) + (two & 255u)), lv);
                b[j] = kg_ja98(*reinterpret_cast<const float2*>(reinterpret_cast<const uint8_t*>(lut) + (two >> 8)), lv);
            } else {
                const float4 v4 = *reinterpret_cast<const float4*>(&sm[kg_phys<false>((idx << lgC) + c2)]);
                a[j] = make_float2(v4.x, v4.y);
                b[j] = make_float2(v4.z, v4.w);
            }
        }
        if (INV) {
#pragma unroll
            for (int q = 1; q < 16; ++q) {
                const float2 wq = twl[(q - 1) << lgm];
                a[q] = cmul_conj(a[q], wq);
                b[q] = cmul_conj(b[q], wq);
            }
            fft_inreg<16, true>(a);
            fft_inreg<16, true>(b);
        } else {
            fft_inreg<16, false>(a);
            fft_inreg<16, false>(b);
#pragma unroll
            for (int q = 1; q < 16; ++q) {
                const float2 wq = twl[(q - 1) << lgm];
                a[q] = cmul(a[q], wq);
                b[q] = cmul(b[q], wq);
            }
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int idx = base + j * m;
            const float4 v4 = make_float4(a[j].x, a[j].y, b[j].x, b[j].y);
            if (DST == 1) *reinterpret_cast<float4*>(gdst + (int64_t)idx * gstride + c2) = v4;
            else *reinterpret_cast<float4*>(&sm[kg_phys<false>((idx << lgC) + c2)]) = v4;
        }
    }
}

template <int RM>
__device__ __forceinline__ void kg_column_inner_pair(float2* sm, const KGParams& p, int n1_0, float2* colsum) {
    constexpr int LGI = ilog2(RM);
    const int lgC = p.lgC, lgP = lgC - 1, cnt = (p.L >> LGI) << lgP;
    const int nf = kg_outer_passes(p.lgL);
    const float inv_half_m = 2.0f / (float)p.M;
    for (int t = threadIdx.x; t < cnt; t += blockDim.x) {
        const int c2 = (t & ((1 << lgP) - 1)) * 2, seg = t >> lgP;
        float2 a[RM], b[RM];
#pragma unroll
        for (int q = 0; q < RM; ++q) {
            const float4 v4 = *reinterpret_cast<const float4*>(&sm[kg_phys<false>(((seg * RM + q) << lgC) + c2)]);
            a[q] = make_float2(v4.x, v4.y);
            b[q] = make_float2(v4.z, v4.w);
        }
        fft_inreg<RM, false>(a);
        fft_inreg<RM, false>(b);
        if (seg == 0) {                                             // A[k2 = 0]
            colsum[c2] = a[0];
            colsum[c2 + 1] = b[0];
        }
        int kseg = 0;
        for (int f = 0; f < nf; ++f) kseg |= ((seg >> (4 * (nf - 1 - f))) & 15) << (4 * f);
        const int n1 = n1_0 + c2;
#pragma unroll
        for (int q = 0; q < RM; ++q) {                              // * W_M^(k2 n1), phase reduced exactly in integers
            const int k2 = kseg | (q << (4 * nf));
            const int pa = (int)(((int64_t)k2 * n1) & (p.M - 1)), pb = (int)(((int64_t)pa + k2) & (p.M - 1));
            float sn, cs;
            sincospif(-(float)pa * inv_half_m, &sn, &cs);
            a[q] = cmul(a[q], make_float2(cs, sn));
            sincospif(-(float)pb * inv_half_m, &sn, &cs);
            b[q] = cmul(b[q], make_float2(cs, sn));
        }
        fft_inreg<RM, true>(a);
        fft_inreg<RM, true>(b);
#pragma unroll
        for (int q = 0; q < RM; ++q)
            *reinterpret_cast<float4*>(&sm[kg_phys<false>(((seg * RM + q) << lgC) + c2)]) = make_float4(a[q].x, a[q].y, b[q].x, b[q].y);
    }
}

// innermost step of the column pass: FFT_RM, diagonal, IFFT_RM on the RM values of one segment
template <int RM, bool GLOBAL>
__device__ __forceinline__ void kg_column_inner(float2* sm, const KGParams& p, int n1_0, float2* colsum, const uint8_t* gsrc_b,
                                                float2* gdst, const float2* lut, const KG8* s8 = nullptr) {
    constexpr int LGI = ilog2(RM);
    const int lgC = p.lgC, cnt = (p.L >> LGI) << lgC;
    const int nf = kg_outer_passes(p.lgL);
    const float inv_half_m = 2.0f / (float)p.M;
    for (int t = threadIdx.x; t < cnt; t += blockDim.x) {
        const int cl = t & ((1 << lgC) - 1), seg = t >> lgC;
        float2 v[RM];
#pragma unroll
        for (int q = 0; q < RM; ++q) {
            const int idx = seg * RM + q;
            if (GLOBAL && s8 && s8->levels) {                       // 2-bit, JA98 levels
                const int64_t o = (int64_t)idx * p.R + cl;
                v[q] = kg_ja98(*reinterpret_cast<const float2*>(reinterpret_cast<const uint8_t*>(lut) + gsrc_b[o]), __ldg(s8->levels + ((s8->byte0 + o) >> 9)));
            } else if (GLOBAL && s8) {                              // 8-bit: one (pol 0, pol 1) pair = half a stream word
                const int64_t o = ((int64_t)idx * p.R + cl) * 2;
                float2 lo, hi;
                kg_decode8(*reinterpret_cast<const uint32_t*>(gsrc_b + (o & ~(int64_t)3)), *s8, o & ~(int64_t)3, lo, hi);
                v[q] = (o & 2) ? hi : lo;
            } else if (GLOBAL) v[q] = *reinterpret_cast<const float2*>(reinterpret_cast<const uint8_t*>(lut) + gsrc_b[(int64_t)idx * p.R + cl]);
            else v[q] = sm[kg_phys<false>((idx << lgC) + cl)];
        }
        fft_inreg<RM, false>(v);
        if (seg == 0) colsum[cl] = v[0];                            // A[k2 = 0]
        int kseg = 0;
        for (int f = 0; f < nf; ++f) kseg |= ((seg >> (4 * (nf - 1 - f))) & 15) << (4 * f);
        const int n1 = n1_0 + cl;
#pragma unroll
        for (int q = 0; q < RM; ++q) {                              // * W_M^(k2 n1), phase reduced exactly in integers
            const int k2 = kseg | (q << (4 * nf));
            const int ph = (int)(((int64_t)k2 * n1) & (p.M - 1));
            float sn, cs;
            sincospif(-(float)ph * inv_half_m, &sn, &cs);
            v[q] = cmul(v[q], make_float2(cs, sn));
        }
        fft_inreg<RM, true>(v);
#pragma unroll
        for (int q = 0; q < RM; ++q) {
            const int idx = seg * RM + q;
            if (GLOBAL) gdst[(int64_t)idx * p.R + cl] = v[q];
            else sm[kg_phys<false>((idx << lgC) + cl)] = v[q];
        }
    }
}

#ifdef B2F_API_TU        // non-template kernels are launched from b2f_api.cu only: compile them once
template <int NBIT>
static __global__ void __launch_bounds__(256, 2) kg_column_pass(const KGParams p) {
    extern __shared__ __align__(16) uint8_t kg_smem[];
    float2* tw = reinterpret_cast<float2*>(kg_smem);                     // [L]
    float2* lut = tw + p.L;                                               // [32]
    float2* data = lut + 32;                                              // [L][C], padded
    const int tid = threadIdx.x, L = p.L, C = p.C, R = p.R, lgL = p.lgL, lgC = p.lgC;
    for (int i = tid; i < L; i += 256) tw[i] = p.tw_col[i];
    if (tid < 32) {
        const int c0 = tid & 3, c1 = (tid >> 2) & 3;
        const float m0 = (c0 == 0 || c0 == 3) ? kLevHi : kLevLo, m1 = (c1 == 0 || c1 == 3) ? kLevHi : kLevLo;
        lut[tid] = tid < 16 ? make_float2((c0 & 2) ? m0 : -m0, (c1 & 2) ? m1 : -m1) : make_float2(0.f, 0.f);
    }
    __syncthreads();
    const int nstrips = R / C;
    const int nf = kg_outer_passes(lgL), lgi = kg_inner_lg(lgL);
    const int64_t nwork = (p.gb_end - p.gb_begin) * nstrips;
    const int cnt16 = (L >> 4) << lgC;
    for (int64_t w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int64_t lb = w / nstrips, gb = p.gb_begin + lb;
        const int strip = (int)(w % nstrips);
        const int ifi = (int)(gb / p.nblk);
        const int64_t blk = gb % p.nblk;
        const int64_t off = (blk * p.step + (int64_t)strip * C) * (NBIT == 8 ? 2 : 1);
        const uint8_t* src = p.compact + ifi * p.compact_stride + off;
        const KG8 s8{p.wmask + ifi * p.wmask_stride, off, p.in8_offset, NBIT == 8 && p.blkdirty[gb] != 0,
                     NBIT == 22 ? p.levels + ifi * p.levels_stride : nullptr};
        float2* dst = p.inter + lb * (int64_t)L * R + strip * C;
        float2* colsum = p.colsum + gb * R + strip * C;
        if (nf == 0) {                                       // L = 16: one register-resident step, no shared memory
            kg_column_inner<16, true>(data, p, strip * C, colsum, src, dst, lut, NBIT != 2 ? &s8 : nullptr);
            continue;
        }
        const int cnt2 = cnt16 >> 1;                         // two neighbouring columns per thread
        for (int f = 0; f < nf; ++f) {                       // forward, outermost first
            if (f == 0) kg_pass16_pair<false, NBIT == 8 ? 2 : (NBIT == 22 ? 3 : 1), 0>(data, tw, lgL, lgL, lgC, cnt2, src, nullptr, R, lut, &s8);
            else kg_pass16_pair<false, 0, 0>(data, tw + kg_tw_offset(lgL, f), lgL, lgL - 4 * f, lgC, cnt2, nullptr, nullptr, 0, lut);
            __syncthreads();
        }
        switch (lgi) {
            case 1: kg_column_inner_pair<2>(data, p, strip * C, colsum); break;
            case 2: kg_column_inner_pair<4>(data, p, strip * C, colsum); break;
            case 3: kg_column_inner_pair<8>(data, p, strip * C, colsum); break;
            default: kg_column_inner_pair<16>(data, p, strip * C, colsum); break;
        }
        __syncthreads();
        for (int f = nf - 1; f >= 0; --f) {                  // inverse, innermost first
            if (f == 0) kg_pass16_pair<true, 0, 1>(data, tw, lgL, lgL, lgC, cnt2, nullptr, dst, R, lut);
            else kg_pass16_pair<true, 0, 0>(data, tw + kg_tw_offset(lgL, f), lgL, lgL - 4 * f, lgC, cnt2, nullptr, nullptr, 0, lut);
            __syncthreads();
        }
    }
}
#endif

template <int RM>
__device__ __forceinline__ void kg_row_inner(float2* sm, int lgR, int cnt) {
    constexpr int LGI = ilog2(RM);
    (void)lgR;
    for (int t = threadIdx.x; t < cnt; t += blockDim.x) {           // t = global segment number over all rows of the batch
        float2 v[RM];
#pragma unroll
        for (int q = 0; q < RM; ++q) v[q] = sm[kg_phys<true>((t << LGI) + q)];
        fft_inreg<RM, false>(v);
#pragma unroll
        for (int q = 0; q < RM; ++q) sm[kg_phys<true>((t << LGI) + q)] = v[q];
    }
}

// generic row pass: a CTA holds RB rows of a block in shared memory, transforms them together, detects and
// integrates D rows per output sample
template <int CPT>                                                       // channels per thread: nchan <= 256 * CPT
__global__ void __launch_bounds__(256, 2) kg_row_pass(const KGParams p) {
    extern __shared__ __align__(16) uint8_t kg_smem[];
    float2* tw = reinterpret_cast<float2*>(kg_smem);                     // [R]
    float2* rows = tw + p.R;                                              // [RB][R], swizzled
    const int tid = threadIdx.x, R = p.R, N = R / 2, lgR = p.lgR, L = p.L, D = p.D;
    for (int i = tid; i < R; i += 256) tw[i] = p.tw_row[i];
    __syncthreads();
    const int nprod = nprod_of_mode(p.mode);
    const int RB = min(16, 4096 / R) < 1 ? 1 : min(16, 4096 / R);        // rows per batch
    const int U = max(D, RB);                                            // rows per work unit (whole output samples)
    const int units_per_blk = L / U;
    const int64_t nunits = (p.gb_end - p.gb_begin) * units_per_blk;
    const int nf = kg_outer_passes(lgR), lgi = kg_inner_lg(lgR);
    const int cnt16 = RB * (R >> 4);
    int posA[CPT], posB[CPT];
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        const int c = tid + 256 * k;
        posA[k] = c < N ? kg_pos_of_freq(c, lgR) : 0;
        posB[k] = c < N ? kg_pos_of_freq(R - 1 - c, lgR) : 0;
    }
    // the next batch of rows is copied into shared memory (cp.async, two buffers) while this one is transformed
    const int batch = RB * R;
    float2* stage = rows + kg_padded((size_t)batch);                     // [2][RB][R], natural order
    auto prefetch = [&](int64_t g, int b0, int buf) {
        const int64_t lb = g / units_per_blk;
        const float2* src = p.inter + (lb * (int64_t)L + (int)(g % units_per_blk) * U + b0) * R;
        float2* dst = stage + (size_t)buf * batch;
        for (int i = tid * 2; i < batch; i += 512) cp_async16(dst + i, src + i);
    };
    int it = 0;
    if (blockIdx.x < nunits) prefetch(blockIdx.x, 0, 0);
    cp_async_commit();
    for (int64_t g = blockIdx.x; g < nunits; g += gridDim.x) {
        const int64_t lb = g / units_per_blk, gb = p.gb_begin + lb;
        const int r0 = (int)(g % units_per_blk) * U;
        const int ifi = (int)(gb / p.nblk);
        const int64_t blk = gb % p.nblk;
        float acc[CPT][4];
        float2 epsr[CPT];
#pragma unroll
        for (int k = 0; k < CPT; ++k) {
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[k][q] = 0.f;
            epsr[k] = tid + 256 * k < N ? p.eps[gb * N + tid + 256 * k] : make_float2(0.f, 0.f);
        }
        for (int b0 = 0; b0 < U; b0 += RB, ++it) {
            {
                int64_t gn = g;
                int bn = b0 + RB;
                if (bn >= U) { bn = 0; gn += gridDim.x; }
                if (gn < nunits) prefetch(gn, bn, (it + 1) & 1);
                cp_async_commit();
                cp_async_wait<1>();
                __syncthreads();
            }
            const float2* src = stage + (size_t)(it & 1) * batch;
            if (nf == 0) {                                   // R = 16: rows go straight to the innermost step
                for (int i = tid; i < RB * R; i += 256) rows[kg_phys<true>(i)] = src[i];
            } else {
                for (int f = 0; f < nf; ++f) {
                    if (f == 0) kg_pass16<false, 2, 0, true>(rows, tw, lgR, lgR, 0, cnt16, nullptr, src, nullptr, R, nullptr);
                    else kg_pass16<false, 0, 0, true>(rows, tw + kg_tw_offset(lgR, f), lgR, lgR - 4 * f, 0, cnt16, nullptr, nullptr, nullptr, 0, nullptr);
                    __syncthreads();
                }
            }
            if (nf == 0) __syncthreads();
            switch (lgi) {
                case 1: kg_row_inner<2>(rows, lgR, RB * (R >> 1)); break;
                case 2: kg_row_inner<4>(rows, lgR, RB * (R >> 2)); break;
                case 3: kg_row_inner<8>(rows, lgR, RB * (R >> 3)); break;
                default: kg_row_inner<16>(rows, lgR, RB * (R >> 4)); break;
            }
            __syncthreads();
            for (int r = 0; r < RB; ++r) {
                const float2* row = rows;
                const int rbase = r << lgR;
#pragma unroll
                for (int k = 0; k < CPT; ++k) {
                    const int c = tid + 256 * k;
                    if (c < N) {
                        const float2 a = row[kg_phys<true>(rbase + posA[k])];
                        const float2 b = row[kg_phys<true>(rbase + posB[k])];
                        const float2 e = epsr[k];
                        const float2 bp = make_float2(b.x - e.x, -b.y - e.y);
                        const float2 P = cadd(a, bp), Q = csub(a, bp);
                        if (p.mode == kModeVolt) {
                            float2* v = p.volt + ((lb * (int64_t)L + (r0 + b0 + r)) * 2) * N;
                            v[c] = P;
                            v[N + c] = Q;
                            continue;
                        }
                        const float pp = 0.25f * (P.x * P.x + P.y * P.y), qq = 0.25f * (Q.x * Q.x + Q.y * Q.y);
                        const float xr = P.x * Q.x + P.y * Q.y, xi = P.y * Q.x - P.x * Q.y;
                        const float re = -0.25f * xi, im = 0.25f * xr;
                        switch (p.mode) {
                            case B2F_POL_P0: acc[k][0] += pp; break;
                            case B2F_POL_P1: acc[k][0] += qq; break;
                            case B2F_POL_I: acc[k][0] += pp + qq; break;
                            case B2F_POL_I2: acc[k][0] += (pp + qq) * (pp + qq); break;
                            case B2F_POL_PPQQ: acc[k][0] += pp; acc[k][1] += qq; break;
                            case B2F_POL_COHERENCE: acc[k][0] += pp; acc[k][1] += qq; acc[k][2] += re; acc[k][3] += im; break;
                            default: acc[k][0] += pp + qq; acc[k][1] += 2.f * re; acc[k][2] += 2.f * im; acc[k][3] += pp - qq; break;
                        }
                    }
                }
                const int rr = r0 + b0 + r;                  // row of the block
                if (p.mode != kModeVolt && ((rr + 1) & (D - 1)) == 0) {             // an output sample is complete
                    const int64_t t = p.row0 + (blk * L + rr) / D;
                    float* dst = p.F + ifi * p.F_if_stride + t * (int64_t)(nprod * N);
#pragma unroll
                    for (int k = 0; k < CPT; ++k) {
                        const int c = tid + 256 * k;
                        if (c < N)
                            for (int q = 0; q < nprod; ++q) dst[q * N + c] = acc[k][q];
#pragma unroll
                        for (int q = 0; q < 4; ++q) acc[k][q] = 0.f;
                    }
                }
            }
            __syncthreads();
        }
    }
    cp_async_wait<0>();
}

// ================================================================== dedispersion behind the generic channeliser
// digifil -D dm -F nchan:D for the shapes the tuned 512-point path does not take (nchan > 256, or smearing that needs
// freq_res > 512: SURVEY D5).  The generic column and row kernels run unchanged up to the detector and leave the channel
// samples y_c[m], m = 0..L-1 of every overlap-save block in `volt` (kg_row_pass, mode kModeVolt).  Multiplying the L bins
// of channel c by the chirp before the backward transform is the circular convolution of y_c with the chirp's impulse
// response, so this kernel does FFT_L, * H[c][k] / L, IFFT_L per channel and polarisation, keeps the samples
// [nfilt_pos, nfilt_pos + keep), detects and integrates D of them.  In-place radix-2 in shared memory: decimation in
// frequency forward (output bit-reversed), the chirp is read at the bit-reversed index, decimation in time backward
// (input bit-reversed, output in order) -- no reordering pass; two stages per pass over the data (points base +
// {0, q, 2q, 3q} in registers).  A fallback for rare shapes: two extra transforms per
// channel and one more HBM round trip than the tuned path, not tuned further.
struct KXParams {
    const float2* volt;         // [gb - gb_begin][L][2][N]: (P, Q) = (2 yP, 2i yQ) as the detector takes them
    const float2* chirp;        // [nif][L][N]  H[c][k] stored k-major
    float* F; int64_t F_if_stride; int64_t row0;
    int L, lgL, N, CH, nblk, nif, D, mode, nfilt_pos, keep;
    int64_t gb_begin, gb_end;
};
#ifdef B2F_API_TU
// shared-memory position of element e of a sequence: one pad element per 16, so that the passes with small spans (a thread's
// four points 1, 2, 4 ... elements apart, neighbouring threads 4, 8, 16 ... apart) spread over the banks
__device__ __forceinline__ int kx_ph(int e) { return e + (e >> 4); }
constexpr int kKXThreads = 1024;              // one CTA per SM (up to 147 KiB of shared memory): 32 warps hide the shared-memory latency
static __global__ void __launch_bounds__(kKXThreads) kx_dedisp_generic(const KXParams p) {
    extern __shared__ __align__(16) uint8_t kx_smem[];
    const int tid = threadIdx.x, NT = kKXThreads, L = p.L, lgL = p.lgL, N = p.N, CH = p.CH, nseq = 2 * CH, H2 = L >> 1, Q4 = L >> 2;
    float2* tw = reinterpret_cast<float2*>(kx_smem);                // [L / 2]  W_L^t
    float2* data = tw + H2;                                         // [CH][2][LP], one pad element per 16 (kx_ph)
    const int LP = L + (L >> 4);
    for (int t = tid; t < H2; t += NT) {
        float sn, cs;
        sincospif(-(float)(2 * t) / (float)L, &sn, &cs);
        tw[t] = make_float2(cs, sn);
    }
    __syncthreads();
    const int ngroups = N / CH, nprod = nprod_of_mode(p.mode), nout = p.keep / p.D;
    const float inv_l = 1.0f / (float)L;
    const int64_t nwork = (p.gb_end - p.gb_begin) * ngroups;
    // two radix-2 stages (spans 2q and q) per pass over the data: points base + {0, q, 2q, 3q} of one sequence
    auto quad = [&](int b, int lgq, float2*& x, int& j, int& base) {
        const int seq = b >> (lgL - 2), i = b & (Q4 - 1);
        j = i & ((1 << lgq) - 1);
        x = data + seq * LP;
        base = ((i >> lgq) << (lgq + 2)) + j;
    };
    auto span1 = [&]() {                                            // the stage of span 1 (odd log2 L): no twiddle
        for (int b = tid; b < nseq * H2; b += NT) {
            float2* x = data + (b >> (lgL - 1)) * LP;
            const int e = 2 * (b & (H2 - 1));
            const float2 u = x[kx_ph(e)], v = x[kx_ph(e + 1)];
            x[kx_ph(e)] = cadd(u, v);
            x[kx_ph(e + 1)] = csub(u, v);
        }
        __syncthreads();
    };
    for (int64_t w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int64_t lb = w / ngroups, gb = p.gb_begin + lb;
        const int c0 = (int)(w % ngroups) * CH;
        const int ifi = (int)(gb / p.nblk);
        const int64_t blk = gb % p.nblk;
        const float2* V = p.volt + lb * (int64_t)L * 2 * N;
        for (int e = tid; e < L * nseq; e += NT) {                  // channel fastest: CH neighbouring float2 per access
            const int ch = e % CH, pol = (e / CH) & 1, m = e / nseq;
            data[(ch * 2 + pol) * LP + kx_ph(m)] = V[((int64_t)m * 2 + pol) * N + c0 + ch];
        }
        __syncthreads();
        int lgh = lgL - 1;
        for (; lgh >= 1; lgh -= 2) {                                // forward, decimation in frequency
            const int lgq = lgh - 1, q = 1 << lgq, sh = lgL - 1 - lgh;       // W_4q^t = tw[t << sh], W_2q^t = tw[t << (sh + 1)]
            for (int b = tid; b < nseq * Q4; b += NT) {
                float2* x;
                int j, e;
                quad(b, lgq, x, j, e);
                const int p0 = kx_ph(e), p1 = kx_ph(e + q), p2 = kx_ph(e + 2 * q), p3 = kx_ph(e + 3 * q);
                const float2 x0 = x[p0], x1 = x[p1], x2 = x[p2], x3 = x[p3];
                const float2 u0 = cadd(x0, x2), u2 = cmul(csub(x0, x2), tw[j << sh]);
                const float2 u1 = cadd(x1, x3), u3 = cmul(csub(x1, x3), tw[(j + q) << sh]);
                const float2 wq = tw[j << (sh + 1)];
                x[p0] = cadd(u0, u1);
                x[p1] = cmul(csub(u0, u1), wq);
                x[p2] = cadd(u2, u3);
                x[p3] = cmul(csub(u2, u3), wq);
            }
            __syncthreads();
        }
        if (lgh == 0) span1();
        const float2* H = p.chirp + (int64_t)ifi * L * N;
        for (int e = tid; e < nseq * L; e += NT) {                  // bin k sits at the bit-reversed position
            const int seq = e >> lgL, pos = e & (L - 1);
            const int k = (int)(__brev((unsigned)pos) >> (32 - lgL));
            const float2 h = H[(int64_t)k * N + c0 + (seq >> 1)];
            float2* x = data + seq * LP + kx_ph(pos);
            const float2 y = cmul(*x, h);
            *x = make_float2(y.x * inv_l, y.y * inv_l);
        }
        __syncthreads();
        int lgq = 0;
        if (lgL & 1) { span1(); lgq = 1; }
        for (; lgq <= lgL - 2; lgq += 2) {                          // backward, decimation in time
            const int q = 1 << lgq, sh = lgL - 2 - lgq;
            for (int b = tid; b < nseq * Q4; b += NT) {
                float2* x;
                int j, e;
                quad(b, lgq, x, j, e);
                const int p0 = kx_ph(e), p1 = kx_ph(e + q), p2 = kx_ph(e + 2 * q), p3 = kx_ph(e + 3 * q);
                const float2 x0 = x[p0], x1 = x[p1], x2 = x[p2], x3 = x[p3];
                const float2 wq = tw[j << (sh + 1)];
                const float2 v1 = cmul_conj(x1, wq), v3 = cmul_conj(x3, wq);
                const float2 y0 = cadd(x0, v1), y1 = csub(x0, v1), y2 = cadd(x2, v3), y3 = csub(x2, v3);
                const float2 w2 = cmul_conj(y2, tw[j << sh]), w3 = cmul_conj(y3, tw[(j + q) << sh]);
                x[p0] = cadd(y0, w2);
                x[p2] = csub(y0, w2);
                x[p1] = cadd(y1, w3);
                x[p3] = csub(y1, w3);
            }
            __syncthreads();
        }
        for (int o = tid; o < CH * nout; o += NT) {                 // detect + integrate D samples
            const int ch = o % CH, sidx = o / CH;
            const float2* xp = data + (ch * 2) * LP;
            const float2* xq = xp + LP;
            const int m0 = p.nfilt_pos + sidx * p.D;
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            for (int d = 0; d < p.D; ++d) {
                const float2 P = xp[kx_ph(m0 + d)], Q = xq[kx_ph(m0 + d)];
                const float pp = 0.25f * (P.x * P.x + P.y * P.y), qq = 0.25f * (Q.x * Q.x + Q.y * Q.y);
                const float xr = P.x * Q.x + P.y * Q.y, xi = P.y * Q.x - P.x * Q.y;
                const float re = -0.25f * xi, im = 0.25f * xr;
                switch (p.mode) {
                    case B2F_POL_P0: acc[0] += pp; break;
                    case B2F_POL_P1: acc[0] += qq; break;
                    case B2F_POL_I: acc[0] += pp + qq; break;
                    case B2F_POL_I2: acc[0] += (pp + qq) * (pp + qq); break;
                    case B2F_POL_PPQQ: acc[0] += pp; acc[1] += qq; break;
                    case B2F_POL_COHERENCE: acc[0] += pp; acc[1] += qq; acc[2] += re; acc[3] += im; break;
                    default: acc[0] += pp + qq; acc[1] += 2.f * re; acc[2] += 2.f * im; acc[3] += pp - qq; break;
                }
            }
            const int64_t t = p.row0 + blk * nout + sidx;
            float* dst = p.F + ifi * p.F_if_stride + t * (int64_t)(nprod * N) + c0 + ch;
            for (int q = 0; q < nprod; ++q) dst[q * N] = acc[q];
        }
        __syncthreads();
    }
}
#endif

// ================================================================== kernel 5a: statistics
// mean / sigma per (IF, product, channel) over the first rescale interval, fp64 accumulators,
// deterministic two-level reduction.
#ifdef B2F_API_TU        // non-template kernels are launched from b2f_api.cu only: compile them once
static __global__ void ks_partial(const float* __restrict__ F, int64_t F_if_stride, int64_t rows, int ncol,
                           double2* __restrict__ partial) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= ncol) return;
    const int ifi = blockIdx.y, split = blockIdx.z, nsplit = gridDim.z;
    const int64_t r0 = rows * split / nsplit, r1 = rows * (split + 1) / nsplit;
    const float* f = F + ifi * F_if_stride + col;
    double s = 0.0, ss = 0.0;
    for (int64_t r = r0; r < r1; ++r) {
        const double x = f[r * ncol];
        s += x;
        ss += x * x;
    }
    partial[((int64_t)ifi * nsplit + split) * ncol + col] = make_double2(s, ss);
}
#endif
#ifdef B2F_API_TU        // non-template kernels are launched from b2f_api.cu only: compile them once
static __global__ void ks_final(const double2* __restrict__ partial, int nsplit, int64_t rows, int ncol,
                         float* __restrict__ mean, float* __restrict__ scale) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= ncol) return;
    const int ifi = blockIdx.y;
    double s = 0.0, ss = 0.0;
    for (int k = 0; k < nsplit; ++k) {
        const double2 v = partial[((int64_t)ifi * nsplit + k) * ncol + col];
        s += v.x;
        ss += v.y;
    }
    const double m = rows > 0 ? s / (double)rows : 0.0;
    const double var = rows > 0 ? ss / (double)rows - m * m : 0.0;
    mean[ifi * ncol + col] = (float)m;
    scale[ifi * ncol + col] = var > 0.0 ? (float)(1.0 / sqrt(var)) : 1.0f;
}
#endif

// ================================================================== kernel 5b: requantise + flip + splice
// One thread = 4 consecutive output channels of one output row.  The band flip of USB
// subbands, the splice order and the trial-major layout of a row with trial DMs are index arithmetic on the load side.
struct KQParams {
    const float* F; int64_t F_if_stride;
    const float* mean; const float* scale;        // [nif][nprod*nchan]
    void* out;
    int64_t rows; int64_t out_row_elems;
    int64_t out_pitch_bytes;                       // bytes between output rows (>= one row); rows may live on a peer GPU
    int nif, nprod, nchan, out_nbit, pol_major;
    int if_order[B2F_MAX_IF];
    int flip[B2F_MAX_IF];                          // 1: channel reversal (USB)
    float inv_digi_sigma;                          // 1 / (sigmas spanned by half the output range): 1/6 for digifil
    int trial_row_elems;                           // elements of one trial's slice of a row (= out_row_elems without trials);
                                                   // trial k reads F / mean / scale slots k * nif + IF
};

__device__ __forceinline__ float quant(float y, float dscale, float dmean, float dmax) {
    return fminf(fmaxf(floorf(fmaf(y, dscale, dmean + 0.5f)), 0.f), dmax);
}

#ifdef B2F_API_TU        // non-template kernels are launched from b2f_api.cu only: compile them once
static __global__ void kq_quantise(const KQParams p) {
    const int64_t quads_per_row = p.out_row_elems / 4;
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= p.rows * quads_per_row) return;
    const int64_t row = i / quads_per_row;
    const int jr = (int)(i % quads_per_row) * 4;   // element of the whole row
    const int trial = jr / p.trial_row_elems;
    const int j = jr - trial * p.trial_row_elems;  // element of this trial's slice
    int tile, prod, k;
    if (p.pol_major) {
        prod = j / (p.nif * p.nchan);
        tile = (j / p.nchan) % p.nif;
        k = j % p.nchan;
    } else {
        tile = j / (p.nprod * p.nchan);
        prod = (j / p.nchan) % p.nprod;
        k = j % p.nchan;
    }
    const int ifi = p.if_order[tile];
    const int slot = trial * p.nif + ifi;
    const int ncol = p.nprod * p.nchan;
    const float* f = p.F + slot * p.F_if_stride + row * (int64_t)ncol + prod * p.nchan;
    const float* mu = p.mean + slot * ncol + prod * p.nchan;
    const float* sc = p.scale + slot * ncol + prod * p.nchan;
    float y[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int c = p.flip[ifi] ? (p.nchan - 1 - (k + a)) : (k + a);
        y[a] = (f[c] - mu[c]) * sc[c];
    }
    // byte address of element j of this row: the row pitch lets a rank drop its tile into the
    // owner's wider spliced rows (possibly peer memory over NVLink)
    uint8_t* orow = reinterpret_cast<uint8_t*>(p.out) + row * p.out_pitch_bytes;
    if (p.out_nbit == 8) {
        uint32_t w = 0;
#pragma unroll
        for (int a = 0; a < 4; ++a) w |= (uint32_t)quant(y[a], 127.5f * p.inv_digi_sigma, 127.5f, 255.f) << (8 * a);
        *reinterpret_cast<uint32_t*>(orow + jr) = w;
    } else if (p.out_nbit == 16) {
        ushort4 w;
        w.x = (unsigned short)quant(y[0], 32768.0f * p.inv_digi_sigma, 32768.0f, 65535.f);
        w.y = (unsigned short)quant(y[1], 32768.0f * p.inv_digi_sigma, 32768.0f, 65535.f);
        w.z = (unsigned short)quant(y[2], 32768.0f * p.inv_digi_sigma, 32768.0f, 65535.f);
        w.w = (unsigned short)quant(y[3], 32768.0f * p.inv_digi_sigma, 32768.0f, 65535.f);
        *reinterpret_cast<ushort4*>(orow + 2 * (int64_t)jr) = w;
    } else if (p.out_nbit == 2) {
        uint32_t w = 0;
#pragma unroll
        for (int a = 0; a < 4; ++a) w |= (uint32_t)quant(y[a], 1.0f, 1.5f, 3.f) << (2 * a);
        orow[jr / 4] = (uint8_t)w;
    } else {
        *reinterpret_cast<float4*>(orow + 4 * (int64_t)jr) = make_float4(y[0], y[1], y[2], y[3]);
    }
}
#endif

}  // namespace b2f
