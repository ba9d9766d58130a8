/*
 * vvb_resample_kernels.cuh -- batched rational-ratio resampling by a polyphase FIR (scipy.signal.resample_poly semantics,
 * zero padding).  Template only, so several translation units may include it.
 *
 * With the filter h (K taps, already scaled by up), half = (K - 1) / 2 and the polyphase bank bank[j][phi] = h[phi + j up]
 * (T = ceil(K / up) taps per phase, zero past K):
 *   y[m] = sum_{j < T} bank[j][phi] x[i0 - j],   q0 = m down + half,  phi = q0 mod up,  i0 = q0 div up,
 * with x = 0 outside [0, n).
 *
 * Work split.  A thread owns a RUN of R outputs s, s + up, ..., s + (R - 1) up: they share the phase phi, so each tap is
 * loaded once for R outputs, and their newest inputs are exactly `down` apart.  Runs are numbered q = u up + w: band u
 * holds the R up outputs [u R up, (u + 1) R up), and w is the run's phase, so the lanes of a warp walk consecutive phases
 * and their tap loads from the phase-minor bank are coalesced (warp-uniform when up == 1).  The run of phase w starts at
 * s = u R up + v with v = (w - half) down^-1 mod up.
 *
 * Register window.  The taps are walked in residue classes c = j mod down (c < min(down, T)), then k = j div down
 * ascending.  Output r at tap j = c + k down reads x[i0 + (r - k) down - c] = X_c[r - k], so one class needs the R + nk - 1
 * values X_c[1 - nk ... R - 1]: each step k >= 1 loads ONE new input (X_c[-k]) into the slot of the value that just left
 * the window and does R FMAs from registers.  Slots rotate at compile time (steps come in groups of R).  When down >= T
 * every class has one tap and the loop degenerates to R loads per tap, the best a single signal allows there.
 *
 * Every output sums its T products in one fixed order (c ascending, then k), in float32 with one FMA per product,
 * whatever its run, tile, chunk or batch: a signal resampled alone is bit-identical to itself inside any batch.
 *
 * SMEM: a CTA owns a tile of RS_THREADS consecutive runs of one signal and first stages the contiguous input span its
 * bands read (zeros outside [0, n)) into shared memory, one padding word per 32 (so lanes whose windows are a multiple of
 * 32 samples apart do not hit one bank).  Without SMEM (the span of a tile would not fit: large down / up with long
 * filters) the inputs are read through L1 with bounds checks.
 */
#pragma once
#include "vvb_fft_core.cuh"

namespace vvb {

constexpr int RS_THREADS = 256;        /* runs per tile = threads per CTA */
constexpr int RS_RUN = 8;              /* R: outputs per run */

struct ResampleArgs {
    const float* x;          /* [batch][x_pitch], n valid samples */
    long long x_pitch, n;
    float* y;                /* [batch][y_pitch], n_out samples */
    long long y_pitch, n_out;
    const float* bank;       /* [taps][up], phase-minor */
    long long up, down, half;
    long long dinv;          /* down^-1 mod up (0 when up == 1) */
    long long half_mod;      /* half mod up */
    int taps;                /* T: taps per phase */
    long long tiles;         /* tiles per signal */
    long long count;         /* batch * tiles */
    int span;                /* SMEM: staged samples a tile may need (the buffer holds span + span / 32 + 1 floats) */
};

/* padded shared-memory index of staged sample k */
VVB_DEV int rs_pad(int k) { return k + (k >> 5); }

template <bool SMEM>
VVB_DEV float rs_x(const float* xs, const float* xb, long long lo, long long n, long long i)
{
    if constexpr (SMEM) return xs[rs_pad((int)(i - lo))];
    else return (i >= 0 && i < n) ? __ldg(xb + i) : 0.0f;
}

template <int R, bool SMEM>
__global__ void __launch_bounds__(RS_THREADS) resample_poly_kernel(const ResampleArgs a)
{
    float* xs = nullptr;
    if constexpr (SMEM) {
#ifdef VVB_EMU
        xs = reinterpret_cast<float*>(vvb_emu::g_dyn_smem);
#else
        extern __shared__ __align__(16) float smem[];
        xs = smem;
#endif
    }
    const long long band = (long long)R * a.up;        /* outputs per band */
    for (long long item = blockIdx.x; item < a.count; item += gridDim.x) {
        const long long b = item / a.tiles, tile = item - b * a.tiles;
        const float* xb = a.x + b * a.x_pitch;
        long long lo = 0;
        if constexpr (SMEM) {
            /* the bands of this tile's runs, [u0, u1], read inputs lo ... hi */
            const long long u0 = tile * RS_THREADS / a.up, u1 = (tile * RS_THREADS + RS_THREADS - 1) / a.up;
            lo = (u0 * band * a.down + a.half) / a.up - (a.taps - 1);
            const long long hi = (((u1 + 1) * band - 1) * a.down + a.half) / a.up;
            const int span = (int)(hi - lo + 1);
            for (int k = threadIdx.x; k < span; k += RS_THREADS) {
                const long long i = lo + k;
                xs[rs_pad(k)] = (i >= 0 && i < a.n) ? __ldg(xb + i) : 0.0f;
            }
            __syncthreads();
        }
        const long long q = tile * RS_THREADS + threadIdx.x;
        const long long u = q / a.up, w = q - u * a.up;                     /* band, phase */
        const long long s = u * band + ((w - a.half_mod + a.up) % a.up) * a.dinv % a.up;
        if (s < a.n_out) {
            const long long i0 = (s * a.down + a.half) / a.up;              /* newest input of output s */
            const float* tap = a.bank + w;                                  /* tap j of this phase: tap[j up] */
            float acc[R];
#pragma unroll
            for (int r = 0; r < R; ++r) acc[r] = 0.0f;
            const int classes = a.down < a.taps ? (int)a.down : a.taps;
            for (int c = 0; c < classes; ++c) {
                const int nk = (int)((a.taps - c + a.down - 1) / a.down);   /* taps c, c + down, ... below T */
                const long long base = i0 - c;                              /* X_c[t] = x[base + t down], in slot t mod R */
                float win[R];
#pragma unroll
                for (int r = 0; r < R; ++r) win[r] = rs_x<SMEM>(xs, xb, lo, a.n, base + r * a.down);
                float h = __ldg(tap + (long long)c * a.up);
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] = __fmaf_rn(h, win[r], acc[r]);
                for (int k0 = 1; k0 < nk; k0 += R) {                        /* k0 = 1 mod R: the slots below are constants */
#pragma unroll
                    for (int kk = 0; kk < R; ++kk) {
                        const int k = k0 + kk;
                        if (k < nk) {
                            win[(2 * R - 1 - kk) % R] = rs_x<SMEM>(xs, xb, lo, a.n, base - (long long)k * a.down);   /* X_c[-k] */
                            h = __ldg(tap + (long long)(c + (long long)k * a.down) * a.up);
#pragma unroll
                            for (int r = 0; r < R; ++r) acc[r] = __fmaf_rn(h, win[(r + 2 * R - 1 - kk) % R], acc[r]);
                        }
                    }
                }
            }
            float* yb = a.y + b * a.y_pitch;
#pragma unroll
            for (int r = 0; r < R; ++r)
                if (s + r * a.up < a.n_out) yb[s + r * a.up] = acc[r];
        }
        if constexpr (SMEM) __syncthreads();
    }
}

/* dynamic shared memory of a SMEM launch staging `span` samples */
inline size_t resample_smem_bytes(long long span) { return sizeof(float) * (size_t)(span + span / 32 + 1); }

}  // namespace vvb
