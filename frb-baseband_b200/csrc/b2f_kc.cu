// Dedispersion back-end instantiations (one per row length): one trial DM, and several in one pass.
#include "b2f_launch.h"

using namespace b2f;

template <int R>
static cudaError_t go(const KCParams& p, bool trials, int grid, cudaStream_t st) {
    auto kern = trials ? kc_dedisp_trials<R> : kc_dedisp_back<R>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kKCSmemBytes);
    if (e != cudaSuccess) return e;
    kern<<<grid, 256, kKCSmemBytes, st>>>(p);
    return cudaGetLastError();
}

cudaError_t b2f_launch_kc(int R, const KCParams& p, bool trials, int grid, cudaStream_t st) {
    switch (R) {
        case 16: return go<16>(p, trials, grid, st);
        case 32: return go<32>(p, trials, grid, st);
        case 64: return go<64>(p, trials, grid, st);
        case 128: return go<128>(p, trials, grid, st);
        case 256: return go<256>(p, trials, grid, st);
        case 512: return go<512>(p, trials, grid, st);
    }
    return cudaErrorInvalidValue;
}
