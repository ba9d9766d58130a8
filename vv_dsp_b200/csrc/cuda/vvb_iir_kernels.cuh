/*
 * vvb_iir_kernels.cuh -- batched IIR filtering by a cascade of second-order sections (scipy.signal.sosfilt /
 * sosfiltfilt semantics, transposed direct form II).  Template only, so several translation units may include it.
 *
 * Blocked scan.  Section s is the linear system z' = A z + B u, y = z0 + b0 u with A = [[-a1, 1], [-a2, 0]].  A CTA walks
 * one segment of one row in tiles of IIR_THREADS runs of L samples, the tile held in registers (L per thread) across all
 * S sections.  For each section in order:
 *   1. every thread runs the recurrence over its L inputs from the zero state (thread 0 from the tile's carry) and keeps
 *      its end state b_t: the run is the affine map z -> M z + b_t with M = A^L;
 *   2. the CTA scans these maps (Hillis-Steele, inclusive): at level d, S_t += A^(L 2^d) S_(t - 2^d), through three
 *      rotating shared-memory buffers (one barrier per level), in float64.  Every level crosses warps (a warp-shuffle level would
 *      leave lane l of warp w with the window [32 w, 32 w + l] only, and joining warps then needs A^(L k) for every
 *      k < 32).  The matrices come from the handle's table, computed on the host in double: the device forms no
 *      matrix products.  The scan runs in float64 because A^k of a pole pair near z = 1 has entries far larger than
 *      A^k z (a 20 Hz high-pass at 48 kHz: ~100x), so a float32 product loses that factor in cancellation, many times
 *      what the sequential float32 recurrence loses; the entering state is rounded to float32 once;
 *   3. every thread reruns the recurrence over its L inputs from its true entering state S_(t-1) (thread 0: the carry),
 *      writing the outputs over the inputs; the last thread's end state is the carry of the next tile.
 * The input is read once and the output written once, through a padded shared-memory transpose so that both are
 * coalesced: 8 bytes per sample.
 *
 * Segments.  Rows of more than `segment` samples are cut into segments (a multiple of the tile, independent of the batch,
 * so results are too).  Launch A (STATES) runs the cascade from the zero state over every segment but the last of each
 * row and writes only its 2S end-state floats; iir_chain_kernel (launch B) chains z_(g+1) = Phi z_g + e_g per row from
 * the row's initial state, Phi the cascade's transition over one segment (host, double); launch C runs every segment from
 * its true entering state.  A row of at most one segment takes launch C alone.  No CTA ever waits on another.
 *
 * The state after the last sample of a segment (zf, or e_g in launch A) is the rerun state of the thread that owns that
 * sample, so a ragged tail does not propagate the state over the padding zeros past it.
 */
#pragma once
#include "vvb_fft_core.cuh"
#include "../../../include/vvb200_cuda.h"

namespace vvb {

constexpr int IIR_THREADS = VVB_IIR_THREADS;
constexpr int IIR_LEVELS = VVB_IIR_LEVELS;
constexpr int IIR_TABLE = VVB_IIR_TABLE;
constexpr int IIR_CHAIN_THREADS = 128;       /* launch B: one thread per state of the cascade (2 S <= 128) */
static_assert((1 << IIR_LEVELS) == IIR_THREADS, "one scan level per doubling of the threads");

struct IirArgs {
    const float* x;          /* [batch][x_pitch] */
    long long x_pitch, n;
    int in_mode, padtype;    /* VVB_IIR_IN_*, VVB_IIR_PAD_* */
    long long pad, nv;       /* virtual row: nv samples */
    float* y;                /* [batch][y_pitch] */
    long long y_pitch;
    int out_mode;            /* VVB_IIR_OUT_* */
    const double* table;     /* [S][IIR_TABLE] */
    int sections;
    const float* phi;        /* [2S][2S] */
    const float* zi;         /* NULL: zero state */
    long long zi_sstride, zi_rstride;
    int zi_scale_first;
    float* zf;               /* NULL: not written */
    long long zf_sstride;
    float* seg;              /* [batch][segs][2S]: A writes e_g in slot g + 1, B replaces slot g by z_g, C reads it */
    long long segment, segs;
    long long count;         /* work items of the launch */
};

/* virtual sample j of a row: the row itself, scipy's odd / even / constant extension of it, or the row reversed */
VVB_DEV float iir_in(const IirArgs& a, const float* xb, long long j)
{
    if (j < 0 || j >= a.nv) return 0.0f;
    if (a.in_mode == VVB_IIR_IN_PLAIN) return __ldg(xb + j);
    if (a.in_mode == VVB_IIR_IN_REV) return __ldg(xb + (a.nv - 1 - j));
    const long long i = j - a.pad;
    if (i >= 0 && i < a.n) return __ldg(xb + i);
    const bool left = i < 0;
    const float edge = __ldg(xb + (left ? 0 : a.n - 1));
    if (a.padtype == VVB_IIR_PAD_CONSTANT) return edge;
    const float m = __ldg(xb + (left ? -i : 2 * (a.n - 1) - i));     /* the sample mirrored about the edge */
    return a.padtype == VVB_IIR_PAD_ODD ? 2.0f * edge - m : m;
}

/* the state row b enters its first segment with in section s */
VVB_DEV float2 iir_entry(const IirArgs& a, const float* xb, long long b, int s)
{
    if (!a.zi) return make_float2(0.0f, 0.0f);
    const float* z = a.zi + s * a.zi_sstride + b * a.zi_rstride;
    float z0 = __ldg(z), z1 = __ldg(z + 1);
    if (a.zi_scale_first) {
        const float v0 = iir_in(a, xb, 0);
        z0 *= v0;
        z1 *= v0;
    }
    return make_float2(z0, z1);
}

VVB_DEV void iir_store(const IirArgs& a, float* yb, long long j, float v)
{
    if (a.out_mode == VVB_IIR_OUT_DIRECT) {
        yb[j] = v;
    } else {
        const long long i = a.nv - 1 - j - a.pad;
        if (i >= 0 && i < a.n) yb[i] = v;
    }
}

/* The scan writes IIR_LEVELS + 1 buffers per section (the levels, then the exclusive states), write w into buffer w mod 3:
 * the last reads of a buffer are then always two barriers old when it is written again, also across sections. */
static_assert((IIR_LEVELS + 1) % 3 == 0, "the scan buffers rotate the same way in every section");

/* dynamic shared memory of iir_tile_kernel: table, carries, three scan buffers, the padded tile */
template <int L> inline size_t iir_smem_bytes(int sections)
{
    return sizeof(double) * ((size_t)sections * IIR_TABLE + 6 * IIR_THREADS) + sizeof(float) * (2 * (size_t)sections + IIR_THREADS * (L + 1));
}

template <int L, bool STATES>
__global__ void __launch_bounds__(IIR_THREADS, 3) iir_tile_kernel(const IirArgs a)
{
#ifdef VVB_EMU
    double* smem_d = reinterpret_cast<double*>(vvb_emu::g_dyn_smem);
#else
    extern __shared__ __align__(16) float smem[];
    double* smem_d = reinterpret_cast<double*>(smem);
#endif
    constexpr int TILE = IIR_THREADS * L;
    const int S = a.sections, t = threadIdx.x;
    double* tab = smem_d;                              /* [S][IIR_TABLE] */
    double* scan = tab + S * IIR_TABLE;                /* [3][IIR_THREADS][2] */
    float* carry = reinterpret_cast<float*>(scan + 6 * IIR_THREADS);   /* [S][2]: the state entering the tile */
    float* xs = carry + 2 * S;                                        /* the tile: sample k of run t at t (L + 1) + k */
    for (int i = t; i < S * IIR_TABLE; i += IIR_THREADS) tab[i] = a.table[i];
    const long long per_row = STATES ? a.segs - 1 : a.segs;
    for (long long item = blockIdx.x; item < a.count; item += gridDim.x) {
        const long long b = item / per_row, g = item - b * per_row;
        const float* xb = a.x + b * a.x_pitch;
        float* yb = a.y + b * a.y_pitch;
        const long long start = g * a.segment;
        const long long len = a.nv - start < a.segment ? a.nv - start : a.segment;
        /* where the state after the segment's last sample goes: slot g + 1 (A), zf of the last segment (C), nowhere */
        float* endp = nullptr;
        long long end_stride = 2;
        if (STATES) endp = a.seg + (b * a.segs + g + 1) * 2 * S;
        else if (g == a.segs - 1 && a.zf) { endp = a.zf + 2 * b; end_stride = a.zf_sstride; }
        __syncthreads();                               /* the previous item's last carries are written */
        if (t < S) {
            float2 z = make_float2(0.0f, 0.0f);
            if (!STATES) {
                if (a.segs > 1) {
                    const float* p = a.seg + (b * a.segs + g) * 2 * S + 2 * t;
                    z = make_float2(p[0], p[1]);
                } else {
                    z = iir_entry(a, xb, b, t);
                }
            }
            carry[2 * t] = z.x;
            carry[2 * t + 1] = z.y;
        }
        for (long long t0 = 0; t0 < len; t0 += TILE) {
            const long long j0 = start + t0;
            const int valid = len - t0 < TILE ? (int)(len - t0) : TILE;
            __syncthreads();                           /* carries set, the previous tile's stores done */
#pragma unroll
            for (int k = 0; k < L; ++k) {
                const int j = k * IIR_THREADS + t;
                xs[j + j / L] = j < valid ? iir_in(a, xb, j0 + j) : 0.0f;
            }
            __syncthreads();
            float v[L];
#pragma unroll
            for (int k = 0; k < L; ++k) v[k] = xs[t * (L + 1) + k];
            const int last = (t0 + TILE >= len) ? valid - 1 - t * L : -1;   /* in [0, L): this run holds the last sample */
            for (int s = 0; s < S; ++s) {
                const double* c = tab + s * IIR_TABLE;
                const float b0 = (float)c[0], b1 = (float)c[1], b2 = (float)c[2], na1 = -(float)c[3], na2 = -(float)c[4];
                float c0 = 0.0f, c1 = 0.0f;
                if (t == 0) { c0 = carry[2 * s]; c1 = carry[2 * s + 1]; }
                /* 1. the run's end state from the zero state (thread 0: from the carry) */
                float z0 = c0, z1 = c1;
#pragma unroll
                for (int k = 0; k < L; ++k) {
                    const float y = __fmaf_rn(b0, v[k], z0);
                    z0 = __fmaf_rn(b1, v[k], __fmaf_rn(na1, y, z1));
                    z1 = __fmaf_rn(b2, v[k], na2 * y);
                }
                /* 2. inclusive scan of z -> A^L z + b_t over the runs, in float64, one barrier per level */
                double s0 = z0, s1 = z1;
#pragma unroll
                for (int d = 0; d < IIR_LEVELS; ++d) {
                    double* buf = scan + (d % 3) * 2 * IIR_THREADS;
                    buf[2 * t] = s0;
                    buf[2 * t + 1] = s1;
                    __syncthreads();
                    const int off = 1 << d;
                    if (t >= off) {
                        const double* m = c + 8 + 4 * d;
                        const double p0 = buf[2 * (t - off)], p1 = buf[2 * (t - off) + 1];
                        s0 = fma(m[0], p0, fma(m[1], p1, s0));
                        s1 = fma(m[2], p0, fma(m[3], p1, s1));
                    }
                }
                {   /* exclusive: the state entering run t, rounded to float32 once */
                    double* buf = scan + (IIR_LEVELS % 3) * 2 * IIR_THREADS;
                    buf[2 * t] = s0;
                    buf[2 * t + 1] = s1;
                    __syncthreads();
                    if (t > 0) { z0 = (float)buf[2 * (t - 1)]; z1 = (float)buf[2 * (t - 1) + 1]; }
                    else { z0 = c0; z1 = c1; }
                }
                /* 3. rerun from the true entering state, outputs over inputs */
                float e0 = 0.0f, e1 = 0.0f;
#pragma unroll
                for (int k = 0; k < L; ++k) {
                    const float u = v[k];
                    const float y = __fmaf_rn(b0, u, z0);
                    z0 = __fmaf_rn(b1, u, __fmaf_rn(na1, y, z1));
                    z1 = __fmaf_rn(b2, u, na2 * y);
                    v[k] = y;
                    if (k == last) { e0 = z0; e1 = z1; }
                }
                if (t == IIR_THREADS - 1) { carry[2 * s] = z0; carry[2 * s + 1] = z1; }
                if (endp && last >= 0 && last < L) { endp[s * end_stride] = e0; endp[s * end_stride + 1] = e1; }
            }
            if (!STATES) {
#pragma unroll
                for (int k = 0; k < L; ++k) xs[t * (L + 1) + k] = v[k];
                __syncthreads();
#pragma unroll
                for (int k = 0; k < L; ++k) {
                    const int j = k * IIR_THREADS + t;
                    if (j < valid) iir_store(a, yb, j0 + j, xs[j + j / L]);
                }
            }
        }
    }
}

/* launch B: per row, z_0 = the row's initial state, then z_g = Phi z_(g-1) + e_(g-1) over the segments, in place */
template <int THREADS>
__global__ void __launch_bounds__(THREADS) iir_chain_kernel(const IirArgs a)
{
#ifdef VVB_EMU
    float* z = reinterpret_cast<float*>(vvb_emu::g_dyn_smem);
#else
    extern __shared__ __align__(16) float z[];       /* THREADS floats */
#endif
    const int n2 = 2 * a.sections, i = threadIdx.x;
    for (long long b = blockIdx.x; b < a.count; b += gridDim.x) {
        const float* xb = a.x + b * a.x_pitch;
        float* slots = a.seg + b * a.segs * n2;
        __syncthreads();                               /* the previous row's readers of z are done */
        if (i < n2) {
            const float2 e = iir_entry(a, xb, b, i >> 1);
            z[i] = (i & 1) ? e.y : e.x;
            slots[i] = z[i];
        }
        for (long long g = 1; g < a.segs; ++g) {
            __syncthreads();
            float acc = 0.0f;
            if (i < n2) {
                const float* row = a.phi + (long long)i * n2;
                acc = slots[g * n2 + i];
                for (int j = 0; j < n2; ++j) acc = __fmaf_rn(__ldg(row + j), z[j], acc);
            }
            __syncthreads();
            if (i < n2) { z[i] = acc; slots[g * n2 + i] = acc; }
        }
    }
}

}  // namespace vvb
