// Long-transform coherent dedispersion (b2f_long.h, DESIGN.md section 5f).
//
// A block of M = R L dual-pol samples z[n] = xP[n] + i xQ[n] (R = 2 nchan, L = 8192..65536) is transformed in the
// two-transposition order of the tuned dedispersion path (n = n1 + R n2, k = k2 + L k1):
//   forward column transform  A'[k2][n1] = W_M^(n1 k2) FFT_L over n2 of z[n1 + R n2]
//   row FFT                   Z[k2 + L k1] = FFT_R over n1 of A'[k2][n1]
//   backward, per trial       channel c, bin j: (Z[k] +- conj Z[M - k]) * H[c][j], k = c L + j; inverse FFT_L;
//                             drop nfilt_pos / nfilt_neg samples, detect, integrate.
// An L-point transform does not fit one SM (512 KiB at L = 65536), so it is split once more, L = La Lb with La = 256:
// every transform runs as passes of N <= 256 points over HBM-resident blocks (8 MiB at most).  One kernel, kl_pass, does
// every pass: a CTA loads 4096 points (P = 4096 / N transforms of N points, strided in HBM as the pass needs), runs a
// radix-2 FFT in shared memory, multiplies by the four-step twiddle and stores in place.  What differs between passes is
// the addressing, the twiddle exponent and where the first pass reads from (the de-framed stream, or the spectrum with
// the un-mixing and the chirp).
#include "b2f_kernels.cuh"
#include "b2f_long.h"

using namespace b2f;

namespace {

constexpr int kKLThreads = 256;
constexpr int kKLTile = 4096;                  // points per CTA

enum { kLoadF = 0, kLoadStream = 1, kLoadUnmix = 2 };

// one pass: element (block b, o, j, q) at b Bs + o Os + j Js + q Qs; an N-point transform over j for every (b, o, q).
// After the transform, output k is multiplied by W_T^e (W_T^-e for the inverse), e = (q >> qsh)(o co + k ck) + o k cok.
struct KLPass {
    float2* data;
    int64_t Bs, Os, Js, Qs;
    int lgN, lgP, On, Qn;
    bool inv;
    int qsh, lgT;                               // lgT = 0: no twiddle
    unsigned co, ck, cok;
};

template <int LOAD>
__global__ void __launch_bounds__(kKLThreads) kl_pass(const KLPass s, const KLParams p) {
    __shared__ float2 x[kKLTile + 256];         // [N][P + 1]: the pad keeps column and row accesses on distinct banks
    __shared__ float2 tw[128];                  // W_N^t (conjugated for the inverse), t < N / 2
    __shared__ float2 lut[32];                  // index byte >> 3 -> (pol 0, pol 1), 2-bit static levels; 16 = masked
    const int tid = threadIdx.x, lgN = s.lgN, lgP = s.lgP, N = 1 << lgN, P = 1 << lgP, PS = P + 1;
    const int64_t tiles = s.Qn >> lgP;
    int64_t w = blockIdx.x;
    const int q0 = (int)(w % tiles) << lgP;
    w /= tiles;
    const int o = (int)(w % s.On);
    const int64_t lb = w / s.On, gb = p.gb_begin + lb;
    const int ifi = (int)(gb / p.nblk);
    const int64_t blk = gb % p.nblk;
    for (int t = tid; t < N / 2; t += kKLThreads) {
        float sn, cs;
        sincospif(-(float)(2 * t) / (float)N, &sn, &cs);
        tw[t] = make_float2(cs, s.inv ? -sn : sn);
    }
    if (LOAD == kLoadStream && tid < 32) {
        const int c0 = tid & 3, c1 = (tid >> 2) & 3;
        const float m0 = (c0 == 0 || c0 == 3) ? kLevHi : kLevLo, m1 = (c1 == 0 || c1 == 3) ? kLevHi : kLevLo;
        lut[tid] = tid < 16 ? make_float2((c0 & 2) ? m0 : -m0, (c1 & 2) ? m1 : -m1) : make_float2(0.f, 0.f);
    }
    __syncthreads();
    const int64_t base = lb * s.Bs + o * s.Os;
    const bool jfast = s.Js == 1;               // the row FFT: a transform is contiguous in HBM
    const int cnt = N << lgP;
    for (int i = tid; i < cnt; i += kKLThreads) {
        const int j = jfast ? (i & (N - 1)) : (i >> lgP), q = jfast ? (i >> lgN) : (i & (P - 1));
        float2 v;
        if (LOAD == kLoadF) {
            v = s.data[base + j * s.Js + (int64_t)(q0 + q) * s.Qs];
        } else if (LOAD == kLoadStream) {       // sample n of the block, stream position blk step + n of the IF
            const int64_t pos = blk * p.step + j * s.Js + (int64_t)(q0 + q) * s.Qs;
            const uint8_t* src = p.compact + ifi * p.compact_stride;
            if (p.in_nbit == 8) {                // one 32-bit word = two time samples x (pol 0, pol 1)
                const int64_t ob = pos * 2;
                const KG8 k8{p.wmask + ifi * p.wmask_stride, 0, p.in8_offset, p.blkdirty[gb] != 0, nullptr};
                float2 lo, hi;
                kg_decode8(*reinterpret_cast<const uint32_t*>(src + (ob & ~(int64_t)3)), k8, ob & ~(int64_t)3, lo, hi);
                v = (ob & 2) ? hi : lo;
            } else {
                v = lut[src[pos] >> 3];
                if (p.in_nbit == 22) v = kg_ja98(v, __ldg(p.levels + ifi * p.levels_stride + (pos >> 9)));
            }
        } else {                                // o = jb, j = ja, q0 + q = 2 c + pol: bin jb + Lb ja of channel c
            const int bin = o + (j << p.lgLb), c = (q0 + q) >> 1;
            const int64_t k = ((int64_t)c << p.lgL) + bin, km = (p.M - k) & (p.M - 1);
            const float2* Z = p.inter + lb * p.M;    // Z[k2 + L k1] at ((k2 % Lb) La + k2 / Lb) R + k1
            auto at = [&](int64_t kk) {
                const int k1 = (int)(kk >> p.lgL), k2 = (int)(kk & (p.L - 1));
                return ((int64_t)((k2 & ((1 << p.lgLb) - 1)) << p.lgLa) + (k2 >> p.lgLb)) * p.R + k1;
            };
            const float2 a = Z[at(k)], b = Z[at(km)];
            const float2 u = (q & 1) ? make_float2(a.x - b.x, a.y + b.y) : make_float2(a.x + b.x, a.y - b.y);   // a -+ conj b
            v = cmul(u, __ldg(p.chirp + ((int64_t)ifi * p.L + bin) * (p.R >> 1) + c));
        }
        x[(int)(__brev((unsigned)j) >> (32 - lgN)) * PS + q] = v;
    }
    __syncthreads();
    for (int lgs = 0; lgs < lgN; ++lgs) {       // decimation in time: bit-reversed in, natural order out
        const int sp = 1 << lgs;
        for (int i = tid; i < (cnt >> 1); i += kKLThreads) {
            const int q = i & (P - 1), b = i >> lgP;
            const int pos = b & (sp - 1), i0 = ((b >> lgs) << (lgs + 1)) + pos;
            float2* x0 = x + i0 * PS + q;
            float2* x1 = x0 + sp * PS;
            const float2 u = *x0, t = cmul(*x1, tw[pos << (lgN - 1 - lgs)]);
            *x0 = make_float2(u.x + t.x, u.y + t.y);
            *x1 = make_float2(u.x - t.x, u.y - t.y);
        }
        __syncthreads();
    }
    const unsigned tmask = (1u << s.lgT) - 1;
    const float tscale = (s.inv ? 2.f : -2.f) / (float)(1u << s.lgT);
    for (int i = tid; i < cnt; i += kKLThreads) {
        const int k = jfast ? (i & (N - 1)) : (i >> lgP), q = jfast ? (i >> lgN) : (i & (P - 1));
        float2 v = x[k * PS + q];
        if (s.lgT) {                             // exponent reduced exactly: T divides 2^32
            const unsigned e = (((unsigned)(q0 + q) >> s.qsh) * ((unsigned)o * s.co + (unsigned)k * s.ck) + (unsigned)o * (unsigned)k * s.cok) & tmask;
            float sn, cs;
            sincospif(tscale * (float)e, &sn, &cs);
            v = cmul(v, make_float2(cs, sn));
        }
        s.data[base + k * s.Js + (int64_t)(q0 + q) * s.Qs] = v;
    }
}

// channel samples y[m][2c + pol] of every block -> keep samples from nfilt_pos, detected and integrated D at a time (the
// products and scaling of kx_dedisp_generic: (P, Q) = (2 yP, 2i yQ))
__global__ void __launch_bounds__(256) kl_detect(const KLParams p) {
    const int N = p.R >> 1, nout = p.keep / p.D, nprod = nprod_of_mode(p.mode);
    const int64_t per_blk = (int64_t)nout * N, i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (p.gb_end - p.gb_begin) * per_blk) return;
    const int64_t lb = i / per_blk, gb = p.gb_begin + lb;
    const int r = (int)(i - lb * per_blk), sidx = r / N, c = r - sidx * N;
    const int ifi = (int)(gb / p.nblk);
    const int64_t blk = gb % p.nblk;
    const float4* y = reinterpret_cast<const float4*>(p.spec + lb * p.M);      // (P, Q) of channel c at m N + c
    const int m0 = p.nfilt_pos + sidx * p.D;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int d = 0; d < p.D; ++d) {
        const float4 v = y[(int64_t)(m0 + d) * N + c];
        const float2 P = make_float2(v.x, v.y), Q = make_float2(v.z, v.w);
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
    float* dst = p.F + ifi * p.F_if_stride + (p.row0 + blk * nout + sidx) * (int64_t)(nprod * N) + c;
    for (int q = 0; q < nprod; ++q) dst[q * N] = acc[q];
}

template <int LOAD>
cudaError_t run_pass(const KLPass& s, const KLParams& p, cudaStream_t st) {
    const int64_t ctas = (p.gb_end - p.gb_begin) * (p.M / kKLTile);
    kl_pass<LOAD><<<(unsigned)ctas, kKLThreads, 0, st>>>(s, p);
    return cudaGetLastError();
}

}  // namespace

// La = 256 points over n2 mod La (stride R), Lb = L / 256 over n2 / La (stride R La); four-step twiddles in between
cudaError_t b2f_launch_kl_column(const KLParams& p, cudaStream_t st) {
    const int Lb = 1 << p.lgLb, La = 1 << p.lgLa;
    KLPass a{};                                  // q = n1 + R na, j = nb -> U[kb][na][n1] * W_L^(na kb)
    a.data = p.inter; a.Bs = p.M; a.Os = 0; a.On = 1; a.Js = (int64_t)p.R * La; a.Qs = 1; a.Qn = p.R * La;
    a.lgN = p.lgLb; a.lgP = 12 - p.lgLb; a.qsh = p.lgR; a.co = 0; a.ck = 1; a.cok = 0; a.lgT = p.lgL;
    cudaError_t e = run_pass<kLoadStream>(a, p, st);
    if (e != cudaSuccess) return e;
    KLPass b{};                                  // o = kb, j = na, q = n1 -> A[k2 = kb + Lb ka][n1] * W_M^(n1 k2)
    b.data = p.inter; b.Bs = p.M; b.Os = (int64_t)p.R * La; b.On = Lb; b.Js = p.R; b.Qs = 1; b.Qn = p.R;
    b.lgN = p.lgLa; b.lgP = 12 - p.lgLa; b.qsh = 0; b.co = 1; b.ck = (unsigned)Lb; b.cok = 0; b.lgT = p.lgR + p.lgL;
    return run_pass<kLoadF>(b, p, st);
}

cudaError_t b2f_launch_kl_row(const KLParams& p, cudaStream_t st) {
    KLPass r{};                                  // rows kb La + ka of R points -> Z[k2 + L k1] at row R + k1
    r.data = p.inter; r.Bs = p.M; r.Os = 0; r.On = 1; r.Js = 1; r.Qs = p.R; r.Qn = p.L;
    r.lgN = p.lgR; r.lgP = 12 - p.lgR;
    return run_pass<kLoadF>(r, p, st);
}

cudaError_t b2f_launch_kl_back(const KLParams& p, cudaStream_t st) {
    const int Lb = 1 << p.lgLb, La = 1 << p.lgLa;
    KLPass a{};                                  // o = jb, j = ja, q = 2c + pol -> T[jb][ma][q] * W_L^-(jb ma)
    a.data = p.spec; a.Bs = p.M; a.Os = (int64_t)La * p.R; a.On = Lb; a.Js = p.R; a.Qs = 1; a.Qn = p.R;
    a.lgN = p.lgLa; a.lgP = 12 - p.lgLa; a.inv = true; a.qsh = 0; a.co = 0; a.ck = 0; a.cok = 1; a.lgT = p.lgL;
    cudaError_t e = run_pass<kLoadUnmix>(a, p, st);
    if (e != cudaSuccess) return e;
    KLPass b{};                                  // j = jb, q = ma R + q -> y[m = ma + La mb] at m R + q
    b.data = p.spec; b.Bs = p.M; b.Os = 0; b.On = 1; b.Js = (int64_t)La * p.R; b.Qs = 1; b.Qn = La * p.R;
    b.lgN = p.lgLb; b.lgP = 12 - p.lgLb; b.inv = true;
    e = run_pass<kLoadF>(b, p, st);
    if (e != cudaSuccess) return e;
    const int64_t n = (p.gb_end - p.gb_begin) * (int64_t)(p.keep / p.D) * (p.R >> 1);
    kl_detect<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p);
    return cudaGetLastError();
}
