// Row-pass instantiations for a subset of row lengths (-DB2F_PART=0|1|2).
#include "b2f_launch.h"

using namespace b2f;

#define B2F_CAT2(a, b) a##b
#define B2F_CAT(a, b) B2F_CAT2(a, b)

template <int TR, int PT, int MODE>
static cudaError_t go(const KBParams& p, int grid, cudaStream_t st) {
    auto kern = kb_row_pass<TR, PT, MODE>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)KBSmem<TR, PT>::kBytes);
    if (e != cudaSuccess) return e;
    kern<<<grid, kKBThreads, KBSmem<TR, PT>::kBytes, st>>>(p);
    return cudaGetLastError();
}

template <int TR, int PT, int MODE>
static cudaError_t go_r(const KBParams& p, int grid, cudaStream_t st) {
    auto kern = kr_row_pass<TR, PT, MODE>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)KBSmem<TR, PT>::kBytes);
    if (e != cudaSuccess) return e;
    kern<<<grid, kKBThreads, KBSmem<TR, PT>::kBytes, st>>>(p);
    return cudaGetLastError();
}

template <int TR, int PT>
static cudaError_t by_mode_r(int mode, const KBParams& p, int grid, cudaStream_t st) {
    switch (mode) {
#ifndef B2F_KF_MAIN_MODES
        case B2F_POL_P0: return go_r<TR, PT, B2F_POL_P0>(p, grid, st);
        case B2F_POL_P1: return go_r<TR, PT, B2F_POL_P1>(p, grid, st);
        case B2F_POL_I2: return go_r<TR, PT, B2F_POL_I2>(p, grid, st);
        case B2F_POL_PPQQ: return go_r<TR, PT, B2F_POL_PPQQ>(p, grid, st);
#endif
        case B2F_POL_I: return go_r<TR, PT, B2F_POL_I>(p, grid, st);
        case B2F_POL_COHERENCE: return go_r<TR, PT, B2F_POL_COHERENCE>(p, grid, st);
        case B2F_POL_IQUV: return go_r<TR, PT, B2F_POL_IQUV>(p, grid, st);
    }
    return cudaErrorInvalidValue;
}

template <int TR, int PT>
static cudaError_t by_mode(int mode, const KBParams& p, int grid, cudaStream_t st) {
    switch (mode) {
        case B2F_POL_P0: return go<TR, PT, B2F_POL_P0>(p, grid, st);
        case B2F_POL_P1: return go<TR, PT, B2F_POL_P1>(p, grid, st);
        case B2F_POL_I: return go<TR, PT, B2F_POL_I>(p, grid, st);
        case B2F_POL_I2: return go<TR, PT, B2F_POL_I2>(p, grid, st);
        case B2F_POL_COHERENCE: return go<TR, PT, B2F_POL_COHERENCE>(p, grid, st);
        case B2F_POL_IQUV: return go<TR, PT, B2F_POL_IQUV>(p, grid, st);
        case B2F_POL_PPQQ: return go<TR, PT, B2F_POL_PPQQ>(p, grid, st);
        case kModeSpectrum: return go<TR, PT, kModeSpectrum>(p, grid, st);
    }
    return cudaErrorInvalidValue;
}

cudaError_t B2F_CAT(b2f_launch_kb_part, B2F_PART)(int R, int mode, const KBParams& p, int grid, cudaStream_t st) {
    switch (R) {
#if B2F_PART == 0
        case 16: return by_mode<4, 4>(mode, p, grid, st);
        case 32: return by_mode<4, 8>(mode, p, grid, st);
        case 64: return by_mode<8, 8>(mode, p, grid, st);
#elif B2F_PART == 1
        case 128: return by_mode<8, 16>(mode, p, grid, st);
        case 512: return by_mode<16, 32>(mode, p, grid, st);
#else
        case 256: return by_mode<16, 16>(mode, p, grid, st);
#endif
    }
    return cudaErrorInvalidValue;
}

// the same row lengths for the [pair][row][2] block layout of the round-2 column kernel; R = 256 uses the tile row pass
// (b2f_kt.cu) instead
#if B2F_PART != 2
cudaError_t B2F_CAT(b2f_launch_kr_part, B2F_PART)(int R, int mode, const KBParams& p, int grid, cudaStream_t st) {
    switch (R) {
#if B2F_PART == 0
        case 16: return by_mode_r<4, 4>(mode, p, grid, st);
        case 32: return by_mode_r<4, 8>(mode, p, grid, st);
        case 64: return by_mode_r<8, 8>(mode, p, grid, st);
#else
        case 128: return by_mode_r<8, 16>(mode, p, grid, st);
        case 512: return by_mode_r<16, 32>(mode, p, grid, st);
#endif
    }
    return cudaErrorInvalidValue;
}
#endif
