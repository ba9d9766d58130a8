/*
 * vvb_fir_kernels.cuh -- batched FIR filtering by FFT convolution (overlap-save) on the M-point register FFT.
 * Template only, so several translation units may include it.
 *
 * One partition of Lp taps, M-point complex transform, output blocks of L = M - Lp + 1 samples.  A team (the same T = M/E
 * threads and register layout as fft_c2c_kernel) owns a work item = one signal and a PAIR of consecutive output blocks:
 * convolution with a real h is C-linear, so with z = x_a + i x_b (the frames of blocks a and b) conv(z, h) carries block a
 * in its real part and block b in its imaginary part -- two real blocks per complex transform, no split step.
 *   1. load both frames x[start - (Lp - 1) + i], i < M (zeros outside [0, n)), in pass-1 order;
 *   2. forward team_fft in registers;
 *   3. times H (the partition's spectrum, 1/M folded in, natural order: one coalesced float2 load per element), parked
 *      in the team's exchange buffer and re-read in pass-1 order with re / im swapped;
 *   4. the second team_fft on the swapped data is the inverse;
 *   5. the last L samples of the frame are the block: re -> block a, im -> block b, clipped to n_out.
 * With ACCUM the block is added to what `y` holds (the passes p > 0 of a filter cut into partitions).
 */
#pragma once
#include "vvb_stft_kernels.cuh"

namespace vvb {

struct FirArgs {
    const float* x;          /* [batch][x_pitch], n valid samples */
    long long x_pitch, n;
    float* y;                /* [batch][y_pitch], n_out samples */
    long long y_pitch, n_out;
    long long n_full;        /* n + num_taps - 1: the full convolution; positions >= n_full are 0 */
    const float2* H;         /* spectrum of this pass's partition of signal b's filter: H + b * h_stride, M values */
    long long h_stride;      /* 0: one filter for every signal */
    long long delay;         /* p * Lp: this partition's delay */
    int lp, L;               /* taps per partition, samples per output block */
    long long pairs;         /* block pairs per signal = ceil(ceil(n_out / L) / 2) */
    long long blocks;        /* blocks per signal = ceil(n_out / L) */
    long long count;         /* batch * pairs */
    const float* tables;     /* Tables<C> blob of the M-point C2C plan */
};

/* v clamped to [0, M] as an int */
template <int M> VVB_DEV int clamp_m(long long v) { return v < 0 ? 0 : (v > M ? M : (int)v); }

template <class C, int G, bool ACCUM>
__global__ void __launch_bounds__(C::T* G) fir_ols_kernel(const FirArgs a)
{
    using TB = Tables<C>;
    using L = LastPass<C>;
    constexpr int M = C::M, E = C::E, T = C::T;
#ifdef VVB_EMU
    float* smem = reinterpret_cast<float*>(vvb_emu::g_dyn_smem);
#else
    extern __shared__ __align__(16) float smem[];
#endif
    float2* s_tw2 = reinterpret_cast<float2*>(smem);
    float2* s_tw3 = s_tw2 + C::TW2;
    float2* s_xb = s_tw3 + C::TW3;
    copy_table(reinterpret_cast<float*>(s_tw2), a.tables + TB::TW2, 2 * (C::TW2 + C::TW3));
    __syncthreads();
    const int team = threadIdx.x / T, t = threadIdx.x % T;
    float2* xb = s_xb + team * C::XBUF;
    const long long groups = (a.count + G - 1) / G;
    for (long long group = blockIdx.x; group < groups; group += gridDim.x) {
        const long long id = group * G + team;
        const bool active = id < a.count;
        const long long b = active ? id / a.pairs : 0;
        const long long blk = 2 * (active ? id - b * a.pairs : 0);         /* block a; block b = blk + 1 */
        const bool has_b = blk + 1 < a.blocks;
        const long long out_a = blk * a.L;                                  /* first output sample of block a */
        const long long src_a = out_a - a.delay - (a.lp - 1);               /* frame origin of block a */
        /* frame element i of block a is x[src_a + i], of block b x[src_a + L + i]: valid for i in [lo_a, hi_a) / [lo_b, hi_b)
         * (32-bit bounds, so the per-element tests are plain integer compares) */
        const float* xa = a.x + b * a.x_pitch + src_a;
        const int lo_a = clamp_m<M>(-src_a), hi_a = active ? clamp_m<M>(a.n - src_a) : 0;
        const int lo_b = clamp_m<M>(-src_a - a.L), hi_b = (active && has_b) ? clamp_m<M>(a.n - src_a - a.L) : 0;
        float2 v[E];
        {
            constexpr int R = C::R1, NQ = E / R, STRIDE = M / R;
#pragma unroll
            for (int q = 0; q < NQ; ++q)
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int i = t + T * q + r * STRIDE;
                    float2 s = make_float2(0.f, 0.f);
                    if (i >= lo_a && i < hi_a) s.x = __ldg(xa + i);
                    if (i >= lo_b && i < hi_b) s.y = __ldg(xa + a.L + i);
                    v[q * R + r] = s;
                }
        }
        team_fft<C>(v, xb, s_tw2, s_tw3, t, team);
        /* times H (1/M folded in), parked in natural order, re-read in pass-1 order with re / im swapped */
        const float2* H = a.H + b * a.h_stride;
#pragma unroll
        for (int q = 0; q < L::NQ; ++q)
#pragma unroll
            for (int r = 0; r < L::R; ++r) {
                const int k = t + T * q + r * L::NS;
                xb[C::pad(k)] = cmul(v[q * L::R + ct_bitrev(r, L::R)], __ldg(H + k));
            }
        team_sync<T>(team);
        {
            constexpr int R = C::R1, NQ = E / R, STRIDE = M / R;
#pragma unroll
            for (int q = 0; q < NQ; ++q)
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const float2 z = xb[C::pad(t + T * q + r * STRIDE)];
                    v[q * R + r] = make_float2(z.y, z.x);
                }
        }
        team_sync<T>(team);
        team_fft<C>(v, xb, s_tw2, s_tw3, t, team);
        if (active) {
            /* frame element k >= Lp - 1 is output sample out_a + k - (Lp - 1) of block a (and that + L of block b): written
             * for k < end (n_out), with the convolution's value below full (n_full) and 0 from there on */
            float* ya = a.y + b * a.y_pitch + out_a - (a.lp - 1);
            const long long base = out_a - (a.lp - 1);
            const int end_a = clamp_m<M>(a.n_out - base), full_a = clamp_m<M>(a.n_full - base);
            const int end_b = has_b ? clamp_m<M>(a.n_out - base - a.L) : 0, full_b = clamp_m<M>(a.n_full - base - a.L);
#pragma unroll
            for (int q = 0; q < L::NQ; ++q)
#pragma unroll
                for (int r = 0; r < L::R; ++r) {
                    const int k = t + T * q + r * L::NS;
                    if (k < a.lp - 1) continue;                                 /* the wrapped (circular) part of the frame */
                    const float2 zs = v[q * L::R + ct_bitrev(r, L::R)];          /* swapped: block a in .y, block b in .x */
                    if (k < end_a) {
                        if constexpr (ACCUM) { if (k < full_a) ya[k] += zs.y; }
                        else ya[k] = k < full_a ? zs.y : 0.0f;
                    }
                    if (k < end_b) {
                        if constexpr (ACCUM) { if (k < full_b) ya[a.L + k] += zs.x; }
                        else ya[a.L + k] = k < full_b ? zs.x : 0.0f;
                    }
                }
        }
        team_sync<T>(team);
    }
}

/* zero-padded, 1/M-scaled partitions of the filters: out[f][p][i] = (h_f[p lp + i] / M, 0) for i < lp and p lp + i < taps,
 * else 0 -- the input of the in-place M-point forward transforms that make the filter spectra */
struct FirPadArgs {
    const float* h;          /* [filters][h_pitch] */
    long long h_pitch, taps;
    float2* out;             /* [filters][parts][M] */
    long long total;         /* filters * parts * M */
    int m, lp, parts;
};

}  // namespace vvb
