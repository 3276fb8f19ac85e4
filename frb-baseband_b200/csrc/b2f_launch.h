// Launchers of the two heavily templated kernels, compiled in separate translation units
// (b2f_ka.cu, b2f_kb.cu with -DB2F_PART=n) so that `make -j` builds them in parallel.
#pragma once
#include "b2f_kernels.cuh"

// fwd_only: the column pass stops after the forward transform (dedispersion path)
cudaError_t b2f_launch_ka(int in_nbit, int R, bool fwd_only, const b2f::KAParams& p, unsigned grid, cudaStream_t st);
cudaError_t b2f_launch_ka_22(int R, bool fwd_only, const b2f::KAParams& p, unsigned grid, cudaStream_t st);
cudaError_t b2f_launch_kb(int R, int mode, const b2f::KBParams& p, int grid, cudaStream_t st);
cudaError_t b2f_launch_kr(int R, int mode, const b2f::KBParams& p, int grid, cudaStream_t st);     // [pair][row][2] blocks, R != 256
cudaError_t b2f_launch_kr_part0(int R, int mode, const b2f::KBParams& p, int grid, cudaStream_t st);
cudaError_t b2f_launch_kr_part1(int R, int mode, const b2f::KBParams& p, int grid, cudaStream_t st);
cudaError_t b2f_launch_kc(int R, const b2f::KCParams& p, bool trials, int grid, cudaStream_t st);   // trials: kc_dedisp_trials
cudaError_t b2f_launch_ka_2(int R, bool fwd_only, const b2f::KAParams& p, unsigned grid, cudaStream_t st);
cudaError_t b2f_launch_ka_8(int R, bool fwd_only, const b2f::KAParams& p, unsigned grid, cudaStream_t st);
cudaError_t b2f_launch_kb_part0(int R, int mode, const b2f::KBParams& p, int grid, cudaStream_t st);   // R = 16, 32, 64
cudaError_t b2f_launch_kb_part1(int R, int mode, const b2f::KBParams& p, int grid, cudaStream_t st);   // R = 128, 512
cudaError_t b2f_launch_kb_part2(int R, int mode, const b2f::KBParams& p, int grid, cudaStream_t st);   // R = 256

// fused column + row kernel (b2f_fused.cuh), one translation unit per row length.  With max_ctas_per_sm != NULL the
// call only reports how many CTAs of the kernel fit on one SM.
namespace b2f { struct FParams; }
cudaError_t b2f_launch_kf(int R, int mode, const b2f::FParams& p, int grid, int cooperative, cudaStream_t st, int* max_ctas_per_sm);
cudaError_t b2f_launch_kf_16(int mode, const b2f::FParams& p, int grid, int cooperative, cudaStream_t st, int* max_ctas_per_sm);
cudaError_t b2f_launch_kf_32(int mode, const b2f::FParams& p, int grid, int cooperative, cudaStream_t st, int* max_ctas_per_sm);
cudaError_t b2f_launch_kf_64(int mode, const b2f::FParams& p, int grid, int cooperative, cudaStream_t st, int* max_ctas_per_sm);
cudaError_t b2f_launch_kf_128(int mode, const b2f::FParams& p, int grid, int cooperative, cudaStream_t st, int* max_ctas_per_sm);
cudaError_t b2f_launch_kf_256(int mode, const b2f::FParams& p, int grid, int cooperative, cudaStream_t st, int* max_ctas_per_sm);
cudaError_t b2f_launch_kf_512(int mode, const b2f::FParams& p, int grid, int cooperative, cudaStream_t st, int* max_ctas_per_sm);
namespace b2f { struct KTParams; }
cudaError_t b2f_launch_kt(int mode, const b2f::KTParams& p, int grid, cudaStream_t st);      // tile row pass, R = 256

// generic channeliser with compile-time geometry (b2f_generic.cuh), one translation unit per size L = R = 2^lg, lg = 10..13.
// With ctas != NULL the call only reports how many CTAs of the kernel fit on one SM.
namespace b2f { struct KGParams; }
cudaError_t b2f_launch_kgt_col(int lg, int in_nbit, const b2f::KGParams& p, int grid, cudaStream_t st, int* ctas);
cudaError_t b2f_launch_kgt_row(int lg, int mode, const b2f::KGParams& p, int grid, cudaStream_t st, int* ctas);
void b2f_kgt_geometry(int lg, int* cols_per_cta, int* rows_per_batch);
#define B2F_KGT_DECL(LG)                                                                                         \
    cudaError_t b2f_launch_kgt_col_##LG(int in_nbit, const b2f::KGParams& p, int grid, cudaStream_t st, int* ctas);           \
    cudaError_t b2f_launch_kgt_row_##LG(int mode, const b2f::KGParams& p, int grid, cudaStream_t st, int* ctas);
B2F_KGT_DECL(10) B2F_KGT_DECL(11) B2F_KGT_DECL(12) B2F_KGT_DECL(13)
#undef B2F_KGT_DECL
