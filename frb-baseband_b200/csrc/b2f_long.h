// Coherent dedispersion with overlap-save transforms of 8192..65536 points (nchan 8..64, at most 2^20 points per block).
// Kernels in b2f_kl.cu, launched from b2f_api.cu; DESIGN.md section 5f.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

namespace b2f {
struct KLParams {
    // de-framed stream of this push (carried samples in front), as the generic column kernel reads it
    const uint8_t* compact; size_t compact_stride;
    const uint8_t* wmask; size_t wmask_stride;      // 8-bit input: word masks by stream position
    const uint8_t* blkdirty;                        // 8-bit input: blocks that hold a masked word
    const float4* levels; int64_t levels_stride;    // JA98: levels per window of 512 stream samples
    float in8_offset;
    int in_nbit;                 // 2: index bytes (1- and 2-bit input), 8, 22: index bytes with JA98 levels
    int64_t step;                // samples between block starts
    float2* inter;               // [gb - gb_begin][M]: forward column transform, then the block spectrum Z
    float2* spec;                // [gb - gb_begin][M]: one trial's chirped channel spectra, then its channel samples
    const float2* chirp;         // [nif][L][N] of one trial
    float* F; int64_t F_if_stride; int64_t row0;
    int R, lgR, L, lgL, lgLa, lgLb, nblk, nif, D, mode, nfilt_pos, keep;
    int64_t M, gb_begin, gb_end;
};
}  // namespace b2f

// forward column transform (decode, L-point FFT, * W_M^(n1 k2)), row FFT to the block spectrum, and per trial the backward
// part (un-mix, chirp, inverse L-point FFT, overlap discard, detection, integration)
cudaError_t b2f_launch_kl_column(const b2f::KLParams& p, cudaStream_t st);
cudaError_t b2f_launch_kl_row(const b2f::KLParams& p, cudaStream_t st);
cudaError_t b2f_launch_kl_back(const b2f::KLParams& p, cudaStream_t st);
