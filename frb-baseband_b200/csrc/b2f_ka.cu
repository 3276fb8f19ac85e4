// Column-pass instantiations for one input bit depth (-DB2F_NBIT=2|8|22; 22 = 2-bit input decoded with JA98 levels).
#include "b2f_launch.h"

using namespace b2f;

#define B2F_CAT2(a, b) a##b
#define B2F_CAT(a, b) B2F_CAT2(a, b)

template <int R, bool FWD_ONLY>
static cudaError_t go(const KAParams& p, unsigned grid, cudaStream_t st) {
    auto kern = ka_column_pass<B2F_NBIT, R, FWD_ONLY>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)KASmem<B2F_NBIT>::kBytes);
    if (e != cudaSuccess) return e;
    kern<<<grid, kKAThreads, KASmem<B2F_NBIT>::kBytes, st>>>(p);
    return cudaGetLastError();
}

cudaError_t B2F_CAT(b2f_launch_ka_, B2F_NBIT)(int R, bool fwd_only, const KAParams& p, unsigned grid, cudaStream_t st) {
    if (fwd_only) {                            // forward-only product mode of the dedispersion path
        switch (R) {
            case 16: return go<16, true>(p, grid, st);
            case 32: return go<32, true>(p, grid, st);
            case 64: return go<64, true>(p, grid, st);
            case 128: return go<128, true>(p, grid, st);
            case 256: return go<256, true>(p, grid, st);
            case 512: return go<512, true>(p, grid, st);
        }
        return cudaErrorInvalidValue;
    }
    switch (R) {
        case 16: return go<16, false>(p, grid, st);
        case 32: return go<32, false>(p, grid, st);
        case 64: return go<64, false>(p, grid, st);
        case 128: return go<128, false>(p, grid, st);
        case 256: return go<256, false>(p, grid, st);
        case 512: return go<512, false>(p, grid, st);
    }
    return cudaErrorInvalidValue;
}
