/*
 * vvb_stft_kernels.cuh -- the STFT / ISTFT hot-path kernels (sm_100a).
 *
 * stft_forward_kernel  replaces, for a whole batch, the per-frame chain
 *     frame gather + zero/reflect pad   src/spectral/stft.c:127-130, src/core/framing.c:95-118
 *     window multiply                   src/core/vv_dsp_vectorized_math_fallback.c:24-26
 *     real->complex pack + C2C forward  src/spectral/stft.c:85-90, src/spectral/fft_kiss.c:27-67
 *     magnitude / power                 src/spectral/stft.c:133-140
 *   in ONE kernel: the window is applied while the samples are loaded into the registers
 *   of the first FFT pass, the N-point real transform is an N/2-point complex Stockham FFT
 *   plus a split step, and |X|^2 / |X| / X is formed in the split step and stored once.
 *
 * stft_inverse_kernel  replaces
 *     C2C backward + 1/n                src/spectral/fft_kiss.c:27-74
 *     synthesis window + OLA + norm     src/spectral/stft.c:103-108
 *     caller-side normalise             tools/dump_stft_roundtrip.c:50-54
 *   in ONE kernel: Hermitian half spectrum -> merged N/2-point complex spectrum -> inverse
 *   Stockham FFT (forward machinery on re/im-swapped data) -> times w/M -> each team parks
 *   its windowed frame in its own shared-memory slot -> after a CTA barrier every output
 *   sample is summed ONCE, by one thread, from the slots that cover it, in ascending frame
 *   order (the reference's accumulation order) -> times 1/sum(w^2) -> one coalesced store.
 *   No atomics anywhere; partial sums that belong to later frames are carried in shared
 *   memory from one round of G frames to the next.
 */
#pragma once
#include "vvb_fft_core.cuh"
#include <stdint.h>

#ifndef VVB_FWD_HALF_SPLIT
#define VVB_FWD_HALF_SPLIT 1          /* forward kernels: publish only the half column the partner thread needs */
#endif
#ifndef VVB_FWD_BASETW
#define VVB_FWD_BASETW 0              /* marching STFT, 32 x 32: 1 = re-read the twiddle bases per frame instead of keeping them in registers */
#endif
#ifndef VVB_INV_BASETW
#define VVB_INV_BASETW 1              /* marching ISTFT, 32 x 32: 5 twiddle bases from shared memory + computed powers */
#endif
#ifndef VVB_INV_PAIRMERGE
#define VVB_INV_PAIRMERGE 0           /* marching ISTFT, 32 x 32: merge bins k and M-k together (0 = every thread merges all its bins alone,
                                         1 = partner values through warp shuffles, 2 = through the exchange buffer) */
#endif
#ifndef VVB_PAIR_TW3
#define VVB_PAIR_TW3 true             /* pair ISTFT (fft_size 256 / 512): inter-pass twiddles computed from bases instead of 13-23 table loads */
#endif
#ifndef VVB_FWD_TABLE_TWIDDLES
#define VVB_FWD_TABLE_TWIDDLES 0      /* 1: the generic forward kernel loads twiddles / window from shared memory (A/B builds) */
#endif

namespace vvb {

enum { OUT_COMPLEX = 0, OUT_POWER = 1, OUT_MAGNITUDE = 2, OUT_LOGMEL = 3 };   /* OUT_LOGMEL: marching kernel and generic kernel with sub-warp teams, see mel_phase */
#ifndef VVB_MEL_NF_MAX
#define VVB_MEL_NF_MAX 4             /* generic forward kernel, fused log-mel: frames of a warp that share the weight loads (A/B builds: 8) */
#endif
constexpr int MEL_U = 4;              /* fused log-mel: four-tap groups ("quads") per schedule segment */
enum { PAD_ZERO = 0, PAD_REFLECT = 1 };

/* float offsets of the per-plan table blob in global memory (host builds it, vvb_runtime.cu) */
template <class C> struct Tables {
    static constexpr int N = 2 * C::M;
    static constexpr int WIN = 0;                      /* analysis window w[N] */
    static constexpr int WSYN = WIN + N;               /* synthesis window w[N]/M */
    static constexpr int TW2 = WSYN + N;               /* float2[C::TW2] */
    static constexpr int TW3 = TW2 + 2 * C::TW2;       /* float2[C::TW3] */
    static constexpr int POST = TW3 + 2 * C::TW3;      /* float2[C::POST] = (cos,sin)(2 pi k/N)/2 */
    static constexpr int WSYN_NORM = POST + 2 * C::POST + 1;   /* w[p]/M * 1/sum_w2[p % hop]: normalisation folded in */
    static constexpr int MIDNORM = WSYN_NORM + N;      /* sum_w2[c], c < hop (steady state, all frames present) */
    static constexpr int TOTAL = MIDNORM + N;
};

struct FwdArgs {
    const float* x;          /* [batch][x_pitch] */
    long long x_pitch, n;
    int frames, hop, pad_mode;
    void* out;               /* [batch][frames][out_pitch] float2 or float */
    long long out_pitch;
    const float* tables;
    int num_groups, groups_per_signal;
    /* OUT_LOGMEL only (tables: csrc/host/mel.c, build_fused_tables): out = [batch][frames][n_mels] log-mel rows */
    const float4* mel_w;     /* [mel_S * MEL_U][32]: the four weights of lane l's quad at schedule step i */
    const int2* mel_seg;     /* [mel_S][32]: { float offset of the segment's first quad in the power row, reset | (band + 1) << 1 } */
    int mel_S, mel_prow, n_mels;
    int mel_unit;            /* quads per schedule segment: MEL_U in the marching kernel, 2 or 4 in the generic kernel */
    int mel_pair;            /* 1: the band sums of two consecutive frames of a warp run together and share every weight load */
    float mel_eps;
};

/* bytes of shared memory the fused log-mel phase adds to a marching forward kernel with G one-warp teams */
VVB_CX size_t mel_smem_bytes(int G, int mel_S, int n_mels, int mel_prow, int pair)
{
    return (size_t)(8 * (G & 1)) + (size_t)mel_S * 32 * (16 * MEL_U + 8) + sizeof(float) * (size_t)G * (size_t)((n_mels + 31) & ~31) * (pair ? 2 : 1) +
           (pair ? sizeof(float) * (size_t)G * (size_t)mel_prow : 0);
}

/* OUT_LOGMEL in the generic forward kernel: the NF = min(4, 32 / T) teams of a group make consecutive frames and leave their
 * power rows in [row 0 | band sums of the NF frames | pad | row 1 | pad | ... ].  The pads put the rows of a warp's teams T banks
 * apart (row j of a group at j T, group stride NF T mod 32), so the split step's row stores -- lane t of every team writes bin
 * k0 + t -- never meet in a bank (ncu before: 23 % of the kernel's shared-memory store wavefronts were such conflicts). */
VVB_CX int mel_up_mod32(int x, int r) { return x + ((r - x) & 31); }                       /* smallest y >= x with y = r mod 32 */
VVB_CX int mel_row_offset(int j, int mel_prow, int nmp, int T, int NF, bool spread)
{
    int off = 0;
    for (int i = 1; i <= j; ++i) {
        const int end = (i == 1) ? mel_prow + NF * nmp : off + mel_prow;
        off = spread ? mel_up_mod32(end, (i * T) & 31) : end;
    }
    return off;
}
VVB_CX int mel_group_stride(int mel_prow, int nmp, int T, int NF, bool spread)
{
    const int end = (NF == 1 ? mel_prow + nmp : mel_row_offset(NF - 1, mel_prow, nmp, T, NF, spread) + mel_prow);
    return spread ? mel_up_mod32(end, (NF * T) & 31) : end;
}

struct InvArgs {
    const float2* spec;      /* [batch][frames][spec_pitch] */
    long long spec_pitch;
    int frames, hop;
    float* y;                /* OLA: [batch][y_pitch];  FRAMES: [count][N] */
    long long y_pitch, n_out;
    const float* inv_norm;   /* [head L | mid hop | tail L], L = N - hop; or nullptr = raw sum */
    const float* tables;
    int num_items, chunks_per_signal, chunk_frames;
    /* frame-range shard of a longer stream (marching kernels only; whole signals: 0, 1, 1).  The first halo_frames
     * rows of every signal's spectra belong to the PREVIOUS shard: they are synthesised only for their overlap into
     * this shard's samples (the same halo re-synthesis a warp does when its range starts mid-signal), nothing is
     * emitted for them and output position 0 is the first sample of frame halo_frames.  head_edge / tail_edge say
     * whether the shard starts / ends at the true start / end of the stream: only there fewer than N/hop frames
     * overlap (edge normalisation tables) and only at the true end the N - hop samples after the last frame's
     * hop-block are emitted.  Every output sample is the same ascending-frame FMA chain as in the unsharded call,
     * so shards concatenate to a bit-identical result. */
    int halo_frames, head_edge, tail_edge;
};

/* edge-inclusive reflection of any index into [0, n): ... 1 0 | 0 1 .. n-1 | n-1 n-2 ...
 * (same map as the reference's reflect_index, src/core/framing.c:21-56) */
VVB_DEV long long reflect_index(long long idx, long long n)
{
    const long long period = 2 * n;
    long long m = idx % period;
    if (m < 0) m += period;
    return m < n ? m : period - 1 - m;
}

VVB_DEV float fetch_sample(const float* xs, long long n, long long idx, int pad_mode)
{
    if (pad_mode == PAD_REFLECT) return n > 0 ? xs[reflect_index(idx, n)] : 0.0f;
    return (idx < 0 || idx >= n) ? 0.0f : xs[idx];
}

/* cooperative global -> shared copy of `count` floats */
VVB_DEV void copy_table(float* dst, const float* src, int count)
{
    for (int i = threadIdx.x; i < count; i += blockDim.x) dst[i] = __ldg(src + i);
}

/* ============================================================== forward (analysis) */
template <int OUT> VVB_DEV void emit_bin(void* out, long long idx, float2 x)
{
    if constexpr (OUT == OUT_COMPLEX) reinterpret_cast<float2*>(out)[idx] = x;
    else if constexpr (OUT == OUT_POWER) reinterpret_cast<float*>(out)[idx] = x.x * x.x + x.y * x.y;
    else if constexpr (OUT == OUT_LOGMEL) reinterpret_cast<float*>(out)[(int)idx] = x.x * x.x + x.y * x.y;   /* the team's power row in shared memory */
    else reinterpret_cast<float*>(out)[idx] = sqrtf(x.x * x.x + x.y * x.y);
}

/* Fused log-mel (reference: src/features/mel.c:204-245, log(sum_k P[k] W[m][k] + eps) with an ascending float32 sum, separate
 * multiply and add).  The warp that has just split a frame keeps the frame's power row in shared memory instead of storing
 * it, and its 32 lanes sum the bands: the host has packed the bands into 32 lane schedules of mel_S segments of MEL_U quads
 * (a quad = four consecutive bins, 16-byte aligned in the row; a band occupies whole segments of ONE lane, padded with zero
 * weights, which add exactly 0 like the zero weights of the reference's full-row sum).  All lanes walk the same number of
 * steps, band changes happen only at segment boundaries, so there is no divergence; per quad one LDS.128 of weights
 * ([step][lane]: conflict-free), one LDS.128 of power values, 4 FMUL + 4 FADD.  No power spectrogram reaches HBM.
 * NF = 2: a warp parks the row of every other frame in a second buffer and sums two frames at once -- two independent
 * chains that share every weight load (the phase is bound by shared-memory wavefronts: 4 + 4 per quad and frame -> 2 + 4). */
template <int NF>
VVB_DEV void mel_phase(const FwdArgs& a, const float4* s_w, const int2* s_seg, const float* row0, const float* row1, float* mout, int t,
                       long long out_row0, long long out_row1)
{
    __syncwarp();                                                      /* the power rows are complete */
    const int nmp = (a.n_mels + 31) & ~31;
    /* NF == 2: the band sums sit right behind the parked row, so their address comes off the register that already holds
     * the row pointer (the compiler otherwise re-derives the buffer address at every emit: ~20 instructions per segment) */
    if constexpr (NF == 2) mout = const_cast<float*>(row0) + a.mel_prow;
    float acc0 = 0.f, acc1 = 0.f;
    const float4* wq = s_w + t;
#pragma unroll 1
    for (int s = 0; s < a.mel_S; ++s) {
        const int2 d = s_seg[s * 32 + t];
        if (d.y & 1) { acc0 = 0.f; acc1 = 0.f; }
        const float4* p0 = reinterpret_cast<const float4*>(row0 + d.x);
        const float4* p1 = reinterpret_cast<const float4*>(row1 + d.x);
#pragma unroll
        for (int u = 0; u < MEL_U; ++u) {
            const float4 w = wq[(s * MEL_U + u) * 32];
            const float4 x0 = p0[u];
            acc0 = __fadd_rn(acc0, __fmul_rn(x0.x, w.x));
            acc0 = __fadd_rn(acc0, __fmul_rn(x0.y, w.y));
            acc0 = __fadd_rn(acc0, __fmul_rn(x0.z, w.z));
            acc0 = __fadd_rn(acc0, __fmul_rn(x0.w, w.w));
            if constexpr (NF == 2) {
                const float4 x1 = p1[u];
                acc1 = __fadd_rn(acc1, __fmul_rn(x1.x, w.x));
                acc1 = __fadd_rn(acc1, __fmul_rn(x1.y, w.y));
                acc1 = __fadd_rn(acc1, __fmul_rn(x1.z, w.z));
                acc1 = __fadd_rn(acc1, __fmul_rn(x1.w, w.w));
            }
        }
        if (d.y >> 1) {
            mout[(d.y >> 1) - 1] = acc0;
            if constexpr (NF == 2) mout[nmp + (d.y >> 1) - 1] = acc1;
        }
    }
    __syncwarp();
    float* o0 = reinterpret_cast<float*>(a.out) + out_row0 * a.out_pitch;
    float* o1 = reinterpret_cast<float*>(a.out) + out_row1 * a.out_pitch;
    /* NF * n_mels logarithms dealt evenly over the lanes (80 bands, two frames: 5 rounds instead of 6) */
    for (int i = t; i < NF * a.n_mels; i += 32) {
        const bool second = NF == 2 && i >= a.n_mels;
        const int m = second ? i - a.n_mels : i;
        (second ? o1 : o0)[m] = logf(mout[(second ? nmp : 0) + m] + a.mel_eps);
    }
    __syncwarp();                                                      /* the rows and the band sums are free again */
}
/* mel_phase for the generic forward kernel: NF consecutive frames of one signal (rows at base + roff[j], band sums behind row 0)
 * share every weight load -- per quad 4 shared-memory wavefronts of weights and 4 per frame -- with U quads per segment; the first
 * `nact` frames exist and leave as ONE contiguous run of nact * n_mels logarithms. */
template <int NF, int U>
VVB_DEV void mel_phase_multi(const FwdArgs& a, const float4* s_w, const int2* s_seg, const float* base, int T, int nmp,
                             int t, long long out_row0, int nact)
{
    __syncwarp();                                                      /* the power rows are complete */
    int roff[NF];                                                      /* (recomputed here: NF registers less across the transform) */
    roff[0] = 0;
#pragma unroll
    for (int j = 1; j < NF; ++j) {
        const int end = (j == 1) ? a.mel_prow + NF * nmp : roff[j - 1] + a.mel_prow;
        roff[j] = (a.mel_pair & 1) ? mel_up_mod32(end, (j * T) & 31) : end;
    }
    float* mout = const_cast<float*>(base) + a.mel_prow;
    float acc[NF];
#pragma unroll
    for (int j = 0; j < NF; ++j) acc[j] = 0.f;
    const float4* wq = s_w + t;
#pragma unroll 1
    for (int s = 0; s < a.mel_S; ++s) {
        const int2 d = s_seg[s * 32 + t];
        if (d.y & 1) {
#pragma unroll
            for (int j = 0; j < NF; ++j) acc[j] = 0.f;
        }
        const float* p = base + d.x;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const float4 w = wq[(s * U + u) * 32];
#pragma unroll
            for (int j = 0; j < NF; ++j) {
                const float4 x = *reinterpret_cast<const float4*>(p + roff[j] + 4 * u);
                acc[j] = __fadd_rn(acc[j], __fmul_rn(x.x, w.x));
                acc[j] = __fadd_rn(acc[j], __fmul_rn(x.y, w.y));
                acc[j] = __fadd_rn(acc[j], __fmul_rn(x.z, w.z));
                acc[j] = __fadd_rn(acc[j], __fmul_rn(x.w, w.w));
            }
        }
        if (d.y >> 1) {
#pragma unroll
            for (int j = 0; j < NF; ++j) mout[j * nmp + (d.y >> 1) - 1] = acc[j];
        }
    }
    __syncwarp();
    float* o = reinterpret_cast<float*>(a.out) + out_row0 * a.out_pitch;      /* out_pitch = n_mels: the frames' rows are contiguous */
    const int count = nact * a.n_mels;
    for (int i = t; i < count; i += 32) {
        int j = 0, m = i;
#pragma unroll
        for (int q = 1; q < NF; ++q) if (i >= q * a.n_mels) { j = q; m = i - q * a.n_mels; }
        o[i] = logf(mout[j * nmp + m] + a.mel_eps);
    }
    __syncwarp();                                                      /* the rows and the band sums are free again */
}

/* X[k] = sm/2 - g, X[M-k] = conj(sm/2 + g) with sm = A + conj(Bc), g = ((sin + j cos)/2) (A - conj(Bc)) */
VVB_DEV void split_math(float2 A, float2 Bc, float2 hw, float2& x0, float2& x1)
{
    const float2 sm = __fadd2_rn(A, make_float2(Bc.x, -Bc.y));
    const float2 df = __fadd2_rn(A, make_float2(-Bc.x, Bc.y));
    const float2 g = cmul(df, make_float2(hw.y, hw.x));
    x0 = __ffma2_rn(splat(0.5f), sm, make_float2(-g.x, -g.y));
    x1 = __ffma2_rn(make_float2(0.5f, -0.5f), sm, make_float2(g.x, -g.y));
}
/* ---- split step that exchanges only what the partner needs.
 * After the last pass thread t of a team holds its whole column, Z[t + T i] for every i < E, in
 * v[(i % NQ) * R + i / NQ] (NQ, R: sub-transforms and radix of the last pass).  Bin k = t + T i (i < E/2) pairs with
 * M - k = (T - t) + T (E - 1 - i): thread T - t, column index E - 1 - i >= E/2.  So a thread only has to publish the
 * upper half of its column and to read E/2 partner values; the A operand is already in its own registers.
 * E/2 STS.64 + E/2 LDS.64 per frame instead of E + E: at fft_size 2048 that is 64 shared-memory wavefronts fewer,
 * in a kernel that sits at 86 % of that peak.  ROT: twiddle = per-thread value x compile-time rotation; otherwise
 * it is read from the shared-memory table (fft_size 8192, where computing it was measured slower). */
template <class C, int I> VVB_DEV constexpr int column_slot()
{
    using L = LastPass<C>;
    return (I % L::NQ) * L::R + ct_bitrev(I / L::NQ, L::R);
}
template <class C, int OUT, bool ROT, int I>
VVB_DEV void split_pair_half(const float2 (&v)[C::E], const float2* xb, float2 hw_t, const float2* s_post, int t, void* out, long long row)
{
    constexpr int M = C::M, T = C::T;
    const int k = t + T * I;
    const float2 A = v[column_slot<C, I>()];
    float2 Bc = xb[C::pad(neg_mod<M>(k))];
    if constexpr (I == 0) { if (t == 0) Bc = A; }                      /* k = 0 pairs with itself (slot 0 is not published) */
    float2 hw;
    if constexpr (ROT) {
        constexpr float cr = TwC<2 * C::E, I>::c, sr = TwC<2 * C::E, I>::s;
        hw = cmul(hw_t, make_float2(cr, sr));
    } else {
        hw = s_post[k];
    }
    float2 x0, x1;
    split_math(A, Bc, hw, x0, x1);
    emit_bin<OUT>(out, row + k, x0);
    emit_bin<OUT>(out, row + M - k, x1);
}
template <class C, int OUT, bool ROT, int... Is>
VVB_DEV void split_pairs_half(const float2 (&v)[C::E], const float2* xb, float2 hw_t, const float2* s_post, int t, void* out, long long row, iseq<Is...>)
{
    (split_pair_half<C, OUT, ROT, Is>(v, xb, hw_t, s_post, t, out, row), ...);
}
template <class C, int... Is> VVB_DEV void publish_upper_half(const float2 (&v)[C::E], float2* xb, int t, iseq<Is...>)
{
    ((xb[C::pad(t + C::T * (C::E / 2 + Is))] = v[column_slot<C, C::E / 2 + Is>()]), ...);
}
/* publish the upper half of the column, then split; the caller syncs the team before xb is reused */
template <class C, int OUT, bool ROT>
VVB_DEV void split_and_store_half(const float2 (&v)[C::E], float2* xb, float2 hw_t, const float2* s_post, int t, int team, void* out, long long row)
{
    constexpr int M = C::M, E = C::E;
    publish_upper_half<C>(v, xb, t, typename make_iseq<E / 2>::type{});
    team_sync<C::T>(team);
    split_pairs_half<C, OUT, ROT>(v, xb, hw_t, s_post, t, out, row, typename make_iseq<E / 2>::type{});
    if (t == 0) {                                                      /* k = M/2 = T E/2: X = conj(Z[M/2]) */
        const float2 A = v[column_slot<C, E / 2>()];
        emit_bin<OUT>(out, row + M / 2, make_float2(A.x, -A.y));
    }
}

template <class C, int OUT> VVB_DEV void split_and_store(const float2* xb, const float2* s_post, int t, void* out, long long row);
template <class C, int OUT> VVB_DEV void split_and_store_rot(const float2* xb, float2 hw_t, int t, void* out, long long row);

template <class C, int G, int OUT>
__global__ void __launch_bounds__(C::T* G, (C::E <= 16 ? 2 : 1)) stft_forward_kernel(const FwdArgs a)
{
    using TB = Tables<C>;
    constexpr int M = C::M, N = 2 * M, E = C::E, T = C::T;
#ifdef VVB_EMU
    float* smem = reinterpret_cast<float*>(vvb_emu::g_dyn_smem);
#else
    extern __shared__ __align__(16) float smem[];
#endif
    float* s_win = smem;                                              /* N floats */
    float2* s_tw2 = reinterpret_cast<float2*>(s_win + N);
    float2* s_tw3 = s_tw2 + C::TW2;
    float2* s_post = s_tw3 + C::TW3;
    float2* s_xb = s_post + C::POST + 1;                              /* +1 keeps 16 B alignment */
    copy_table(s_win, a.tables + TB::WIN, N);
    copy_table(reinterpret_cast<float*>(s_tw2), a.tables + TB::TW2, 2 * (C::TW2 + C::TW3 + C::POST));
    /* OUT_LOGMEL in this kernel (sub-warp teams: fft_size 256 ... 1024 and the speech framings): a warp's 32 / T teams make
     * consecutive frames; each team leaves its power row in shared memory and the warp then runs mel_phase_multi on every group
     * of NF rows with the lane schedules of csrc/host/mel.c -- no CTA barrier, so the band sums of one warp overlap the
     * transforms of the others.  Layout per group: mel_row_offset / mel_group_stride; row tails stay zero. */
    constexpr int TPW = T <= 32 ? 32 / T : 1;                         /* teams (= consecutive frames) per warp */
    constexpr int NF = TPW < VVB_MEL_NF_MAX ? (TPW < 2 ? 1 : TPW) : VVB_MEL_NF_MAX;   /* frames that share the weight loads */
    float4* s_melw = nullptr;
    int2* s_melseg = nullptr;
    float* s_rows = nullptr;
    int nmp = 0, gstride = 0, my_row = 0;
    int rowb = 0;                                                     /* NF == 2: the odd frame's row */
    if constexpr (OUT == OUT_LOGMEL) {
        static_assert(T <= 16 && G % NF == 0, "two or more teams per warp");
        s_melw = reinterpret_cast<float4*>(smem + ((N + 2 * (C::TW2 + C::TW3 + C::POST + 1) + 2 * G * C::XBUF + 3) & ~3));
        s_melseg = reinterpret_cast<int2*>(s_melw + a.mel_S * a.mel_unit * 32);
        s_rows = reinterpret_cast<float*>(s_melseg + a.mel_S * 32);
        nmp = (a.n_mels + 31) & ~31;
        const bool spread = (a.mel_pair & 1) != 0;                    /* (A/B switch: rows T banks apart, or back to back) */
        rowb = mel_row_offset(1, a.mel_prow, nmp, T, NF, spread);
        gstride = mel_group_stride(a.mel_prow, nmp, T, NF, spread);
        my_row = (int)(threadIdx.x / T / NF) * gstride + mel_row_offset((int)(threadIdx.x / T) % NF, a.mel_prow, nmp, T, NF, spread);
        copy_table(reinterpret_cast<float*>(s_melw), reinterpret_cast<const float*>(a.mel_w), a.mel_S * a.mel_unit * 32 * 4);
        copy_table(reinterpret_cast<float*>(s_melseg), reinterpret_cast<const float*>(a.mel_seg), a.mel_S * 32 * 2);
        for (int i = threadIdx.x; i < (G / NF) * gstride; i += blockDim.x) s_rows[i] = 0.f;
    }
    __syncthreads();

    const int team = threadIdx.x / T, t = threadIdx.x % T;
    float2* xb = s_xb + team * C::XBUF;
    const float2* win2 = reinterpret_cast<const float2*>(s_win);
    /* These kernels are bound by shared-memory wavefronts (ncu: LSU 85 % at fft_size 512), so what can be
     * computed or kept in registers is: inter-pass twiddles as powers of a per-thread base (two-pass
     * configurations), split twiddles as per-thread value x compile-time rotation, and the window in
     * registers where E is small enough to keep two CTAs per SM. */
    constexpr bool REGTW = (C::NP == 2) && (E <= 32) && !VVB_FWD_TABLE_TWIDDLES;    /* (E = 60: the bases and powers on top of 120 data registers spill) */
    constexpr bool WINREG = (E <= 16) && !VVB_FWD_TABLE_TWIDDLES;
    TwBase twb;
    if constexpr (REGTW) twb = load_tw_base2<C>(reinterpret_cast<const float2*>(a.tables + TB::TW2), t);
    const float2 hw_t = __ldg(reinterpret_cast<const float2*>(a.tables + TB::POST) + t);   /* t < T <= M/2 */
    float2 wreg[WINREG ? E : 1];
    if constexpr (WINREG) {
        constexpr int R = C::R1, NQ = E / R, STRIDE = M / R;
#pragma unroll
        for (int q = 0; q < NQ; ++q)
#pragma unroll
            for (int r = 0; r < R; ++r) wreg[q * R + r] = win2[t + T * q + r * STRIDE];
    }
    auto win_at = [&](int slot, int i) -> float2 {
        if constexpr (WINREG) { (void)i; return wreg[slot]; } else { (void)slot; return win2[i]; }
    };

    for (int group = blockIdx.x; group < a.num_groups; group += gridDim.x) {
        const int b = group / a.groups_per_signal;
        const int f = (group % a.groups_per_signal) * G + team;
        const bool active = f < a.frames;
        const float* xs = a.x + (long long)b * a.x_pitch;
        long long start = (long long)f * a.hop;
        if (a.pad_mode == PAD_REFLECT) start -= M;                   /* nfft/2 */

        /* ---- framing + window, straight into the registers of pass 1 */
        float2 v[E];
        {
            constexpr int R = C::R1, NQ = E / R, STRIDE = M / R;
            const bool inside = active && start >= 0 && start + N <= a.n;
            if (inside) {
                const float* p = xs + start;
                if ((reinterpret_cast<uintptr_t>(p) & 7) == 0) {
                    const float2* p2 = reinterpret_cast<const float2*>(p);
#pragma unroll
                    for (int q = 0; q < NQ; ++q)
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const int i = t + T * q + r * STRIDE;
                            const float2 s = __ldg(p2 + i), w = win_at(q * R + r, i);
                            v[q * R + r] = make_float2(s.x * w.x, s.y * w.y);
                        }
                } else {
#pragma unroll
                    for (int q = 0; q < NQ; ++q)
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const int i = t + T * q + r * STRIDE;
                            const float2 w = win_at(q * R + r, i);
                            v[q * R + r] = make_float2(__ldg(p + 2 * i) * w.x, __ldg(p + 2 * i + 1) * w.y);
                        }
                }
            } else if (active) {
#pragma unroll
                for (int q = 0; q < NQ; ++q)
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const int i = t + T * q + r * STRIDE;
                        const float2 w = win_at(q * R + r, i);
                        v[q * R + r] = make_float2(fetch_sample(xs, a.n, start + 2 * i, a.pad_mode) * w.x,
                                                   fetch_sample(xs, a.n, start + 2 * i + 1, a.pad_mode) * w.y);
                    }
            } else {
#pragma unroll
                for (int i = 0; i < E; ++i) v[i] = make_float2(0.f, 0.f);
            }
        }

        /* ---- M-point complex FFT of z[i] = x[2i] + j x[2i+1] */
        if constexpr (REGTW) team_fft_regtw2<C>(v, xb, twb, t, team);
        else team_fft<C>(v, xb, s_tw2, s_tw3, t, team);

        /* ---- split step: X[k] = (Z[k] + conj Z[M-k])/2 - (j/2) W_N^k (Z[k] - conj Z[M-k]) */
        const long long row = ((long long)b * a.frames + f) * a.out_pitch;
        if constexpr (OUT == OUT_LOGMEL) {
            static_assert(VVB_FWD_HALF_SPLIT && !VVB_FWD_TABLE_TWIDDLES, "the fused log-mel phase takes the half-column split");
            publish_upper_half<C>(v, xb, t, typename make_iseq<E / 2>::type{});
            team_sync<T>(team);
            if (active) {                                             /* the power row goes to shared memory */
                float* pw = s_rows + my_row;
                split_pairs_half<C, OUT, (C::M <= 2048)>(v, xb, hw_t, s_post, t, pw, 0, typename make_iseq<E / 2>::type{});
                if (t == 0) {
                    const float2 A = v[column_slot<C, E / 2>()];
                    emit_bin<OUT>(pw, M / 2, make_float2(A.x, -A.y));
                }
            }
            const int lane = threadIdx.x & 31, wteam = (threadIdx.x >> 5) * TPW, fw = f - (team - wteam);
#pragma unroll 1
            for (int q = 0; q < TPW / NF; ++q) {
                const int fe = fw + NF * q;                           /* the same for all lanes of the warp */
                if (fe >= a.frames) break;
                const float* pb = s_rows + (wteam / NF + q) * gstride;
                const long long orow = (long long)b * a.frames + fe;
                const int nact = min(NF, a.frames - fe);
                if constexpr (NF == 2) {
                    /* two frames per warp (T = 16): the marching kernel's phase, four quads per segment (same-box A/B against
                     * mel_phase_multi<2, U>: fft_size 1024 2.92 vs 3.04 (U = 4) / 3.09 ms (U = 2), 640: 1.45 vs 1.54 / 1.53 ms) */
                    float* mo = const_cast<float*>(pb) + a.mel_prow;
                    if (nact == 2) mel_phase<2>(a, s_melw, s_melseg, pb, pb + rowb, mo, lane, orow, orow + 1);
                    else mel_phase<1>(a, s_melw, s_melseg, pb, pb, mo, lane, orow, orow);
                } else {
                    /* four frames share the weight loads (T <= 8); short bands take two quads per segment (fft_size 400:
                     * 1.19 -> 1.11 ms with four frames, -> 1.09 ms with two-quad segments; 256: 1.15 -> 1.02 -> 0.98 ms) */
                    if (a.mel_unit == 2) mel_phase_multi<NF, 2>(a, s_melw, s_melseg, pb, T, nmp, lane, orow, nact);
                    else mel_phase_multi<NF, 4>(a, s_melw, s_melseg, pb, T, nmp, lane, orow, nact);
                }
            }
        } else if constexpr (VVB_FWD_HALF_SPLIT && !VVB_FWD_TABLE_TWIDDLES) {
            publish_upper_half<C>(v, xb, t, typename make_iseq<E / 2>::type{});
            team_sync<T>(team);
            if (active) {
                split_pairs_half<C, OUT, (C::M <= 2048)>(v, xb, hw_t, s_post, t, a.out, row, typename make_iseq<E / 2>::type{});
                if (t == 0) {
                    const float2 A = v[column_slot<C, E / 2>()];
                    emit_bin<OUT>(a.out, row + M / 2, make_float2(A.x, -A.y));
                }
            }
        } else {
            team_store_natural<C>(v, xb, t);
            team_sync<T>(team);
            if constexpr (!VVB_FWD_TABLE_TWIDDLES && C::M <= 2048) {
                if (active) split_and_store_rot<C, OUT>(xb, hw_t, t, a.out, row);
            } else {
                if (active) split_and_store<C, OUT>(xb, s_post, t, a.out, row);
            }
        }
        team_sync<T>(team);                                           /* xb is reused next group */
    }
}

/* ================================================= forward, warp-marching specialisation */
/* One-warp teams (fft_size 2048), hop = 64*S, zero padding.  A warp walks consecutive frames of one
 * signal.  Consecutive frames share N - hop samples, so the warp keeps a ring of N/hop + 1 hop-blocks
 * in shared memory and, per frame, fetches only the ONE new hop-block -- with a TMA 1-D bulk copy
 * (cp.async.bulk, completion on an mbarrier) issued one frame ahead by a single lane.  Every input
 * sample therefore leaves L2 once per warp-range instead of N/hop times, and its latency is
 * covered by a whole frame of FFT work.  The window lives in registers (it depends only on the lane
 * and the register slot), the split step and |X|^2 are fused as in stft_forward_kernel.  There are no
 * CTA-wide barriers after the tables are loaded. */
template <class C, int OUT>
VVB_DEV void split_and_store(const float2* xb, const float2* s_post, int t, void* out, long long row)
{
    constexpr int M = C::M, E = C::E, T = C::T;
    auto emit = [&](int k, float xr, float xi) {
        if constexpr (OUT == OUT_COMPLEX) reinterpret_cast<float2*>(out)[row + k] = make_float2(xr, xi);
        else if constexpr (OUT == OUT_POWER) reinterpret_cast<float*>(out)[row + k] = xr * xr + xi * xi;
        else reinterpret_cast<float*>(out)[row + k] = sqrtf(xr * xr + xi * xi);
    };
#pragma unroll
    for (int i = 0; i < E / 2; ++i) {
        const int k = t + T * i;                                      /* 0 .. M/2-1 */
        const float2 A = xb[C::pad(k)];
        const float2 Bc = xb[C::pad(neg_mod<M>(k))];
        const float2 hw = s_post[k];                                  /* (cos, sin)/2 */
        const float2 sm = __fadd2_rn(A, make_float2(Bc.x, -Bc.y));    /* A + conj(Bc) */
        const float2 df = __fadd2_rn(A, make_float2(-Bc.x, Bc.y));    /* A - conj(Bc) */
        const float2 g = cmul(df, make_float2(hw.y, hw.x));           /* (sin + j cos)/2 * df */
        const float2 x0 = __ffma2_rn(splat(0.5f), sm, make_float2(-g.x, -g.y));              /* X[k] = sm/2 - g */
        const float2 x1 = __ffma2_rn(make_float2(0.5f, -0.5f), sm, make_float2(g.x, -g.y));  /* X[M-k] = conj(sm/2 + g) */
        emit(k, x0.x, x0.y);
        emit(M - k, x1.x, x1.y);
    }
    if (t == 0) {                                                     /* k = M/2: X = conj(Z[M/2]) */
        const float2 A = xb[C::pad(M / 2)];
        emit(M / 2, A.x, -A.y);
    }
}

/* split step with the twiddle of bin k = t + T*i formed as (per-thread value) x (compile-time rotation
 * by 2 pi i T / N) instead of loaded from the table: 16 LDS.64 fewer per frame */
template <class C, int OUT, int I> VVB_DEV void split_pair_rot(const float2* xb, float2 hw_t, int t, void* out, long long row)
{
    constexpr int M = C::M, T = C::T;
    const int k = t + T * I;
    const float2 A = xb[C::pad(k)];
    const float2 Bc = xb[C::pad(neg_mod<M>(k))];
    constexpr float cr = TwC<2 * C::E, I>::c, sr = TwC<2 * C::E, I>::s;
    const float2 hw = cmul(hw_t, make_float2(cr, sr));
    const float2 sm = __fadd2_rn(A, make_float2(Bc.x, -Bc.y));
    const float2 df = __fadd2_rn(A, make_float2(-Bc.x, Bc.y));
    const float2 g = cmul(df, make_float2(hw.y, hw.x));
    const float2 x0 = __ffma2_rn(splat(0.5f), sm, make_float2(-g.x, -g.y));
    const float2 x1 = __ffma2_rn(make_float2(0.5f, -0.5f), sm, make_float2(g.x, -g.y));
    if constexpr (OUT == OUT_COMPLEX) {
        reinterpret_cast<float2*>(out)[row + k] = x0;
        reinterpret_cast<float2*>(out)[row + M - k] = x1;
    } else if constexpr (OUT == OUT_POWER) {
        reinterpret_cast<float*>(out)[row + k] = x0.x * x0.x + x0.y * x0.y;
        reinterpret_cast<float*>(out)[row + M - k] = x1.x * x1.x + x1.y * x1.y;
    } else {
        reinterpret_cast<float*>(out)[row + k] = sqrtf(x0.x * x0.x + x0.y * x0.y);
        reinterpret_cast<float*>(out)[row + M - k] = sqrtf(x1.x * x1.x + x1.y * x1.y);
    }
}
template <class C, int OUT, int... Is> VVB_DEV void split_pairs_rot(const float2* xb, float2 hw_t, int t, void* out, long long row, iseq<Is...>)
{
    (split_pair_rot<C, OUT, Is>(xb, hw_t, t, out, row), ...);
}
template <class C, int OUT>
VVB_DEV void split_and_store_rot(const float2* xb, float2 hw_t, int t, void* out, long long row)
{
    constexpr int M = C::M;
    split_pairs_rot<C, OUT>(xb, hw_t, t, out, row, typename make_iseq<C::E / 2>::type{});
    if (t == 0) {                                                     /* k = M/2: X = conj(Z[M/2]) */
        const float2 A = xb[C::pad(M / 2)];
        if constexpr (OUT == OUT_COMPLEX) reinterpret_cast<float2*>(out)[row + M / 2] = make_float2(A.x, -A.y);
        else if constexpr (OUT == OUT_POWER) reinterpret_cast<float*>(out)[row + M / 2] = A.x * A.x + A.y * A.y;
        else reinterpret_cast<float*>(out)[row + M / 2] = sqrtf(A.x * A.x + A.y * A.y);
    }
}

/* ---- split step without shared memory (one-warp 32 x 32 transforms).
 * After the last pass lane t holds column t: Z[t + 32 r] in v[r].  The partner bin of k = t + 32 r is
 * M - k = (32 - t) + 32 (31 - r): lane 32-t, slot 31-r.  Each lane handles its EVEN slots: it fetches the
 * partner's odd slot 31-r with two shuffles (the register index is the same for every lane), forms X[k]
 * and X[M-k] and stores both (lanes are consecutive in k, so both stores are coalesced).  Together the
 * lanes 1..31 cover every bin that is not a multiple of 32 exactly once.  Column 0 (lane 0, bins 32 r) is
 * paired with itself (r <-> 32 - r): all lanes run the same register-only code on their own column and
 * only lane 0 stores.  This replaces a natural-order store (32 STS.64), 32 paired LDS.64 and two team
 * barriers per frame by 32 SHFL -- the kernel is bound by shared-memory/LSU wavefronts. */
template <class C, int OUT, int R2> VVB_DEV void split_shfl_pair(const float2 (&v)[C::E], float2 hw_t, int t, int src, void* out, long long row)
{
    constexpr int R = 2 * R2, M = C::M;                                /* even slot */
    float2 Bc;
    Bc.x = __shfl_sync(0xffffffffu, v[31 - R].x, src);
    Bc.y = __shfl_sync(0xffffffffu, v[31 - R].y, src);
    constexpr float cr = TwC<64, R>::c, sr = TwC<64, R>::s;
    float2 x0, x1;
    split_math(v[R], Bc, cmul(hw_t, make_float2(cr, sr)), x0, x1);
    if (t != 0) {
        const int k = t + 32 * R;
        emit_bin<OUT>(out, row + k, x0);
        emit_bin<OUT>(out, row + M - k, x1);
    }
}
template <class C, int OUT, int R> VVB_DEV void split_col0_pair(const float2 (&v)[C::E], int t, void* out, long long row)
{
    constexpr int M = C::M;                                            /* bins 32 R and M - 32 R of column 0 */
    constexpr float hc = 0.5f * TwC<64, R>::c, hs = 0.5f * TwC<64, R>::s;
    float2 x0, x1;
    split_math(v[R], v[(32 - R) % 32], make_float2(hc, hs), x0, x1);
    if (t == 0) {
        emit_bin<OUT>(out, row + 32 * R, x0);
        if constexpr (R != 16) emit_bin<OUT>(out, row + M - 32 * R, x1);
    }
}
template <class C, int OUT, int... Is> VVB_DEV void split_shfl_all(const float2 (&v)[C::E], float2 hw_t, int t, int src, void* out, long long row, iseq<Is...>)
{
    (split_shfl_pair<C, OUT, Is>(v, hw_t, t, src, out, row), ...);
}
template <class C, int OUT, int... Is> VVB_DEV void split_col0_all(const float2 (&v)[C::E], int t, void* out, long long row, iseq<Is...>)
{
    (split_col0_pair<C, OUT, Is>(v, t, out, row), ...);
}
template <class C, int OUT> VVB_DEV void split_shuffle_store(const float2 (&v)[C::E], float2 hw_t, int t, void* out, long long row)
{
    static_assert(C::T == 32 && C::E == 32, "one-warp 32 x 32 transforms");
    split_shfl_all<C, OUT>(v, hw_t, t, (32 - t) & 31, out, row, typename make_iseq<16>::type{});
    split_col0_all<C, OUT>(v, t, out, row, typename make_iseq<17>::type{});
}

template <class C, int S, int G, int MINB, int OUT>
__global__ void __launch_bounds__(C::T* G, MINB) stft_march_kernel(const FwdArgs a)
{
    static_assert(C::T >= 32 && C::R1 == C::E && C::E % S == 0, "whole-warp teams, pass-1 radix == points per thread");
    using TB = Tables<C>;
    constexpr int M = C::M, E = C::E, T = C::T;
    constexpr int NB = E / S, HB = T * S, HOP = 2 * HB, RING = NB + 1;    /* HB float2 per hop-block */
#ifdef VVB_EMU
    float* smem = reinterpret_cast<float*>(vvb_emu::g_dyn_smem);
#else
    extern __shared__ __align__(16) float smem[];
#endif
    float2* s_tw2 = reinterpret_cast<float2*>(smem);
    float2* s_tw3 = s_tw2 + C::TW2;
    float2* s_post = s_tw3 + C::TW3;
    float2* s_xb = s_post + C::POST + 1;
    float2* s_ring = s_xb + G * C::XBUF;                              /* G x RING x HB float2, 16-byte aligned */
    unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(s_ring + G * RING * HB);
    copy_table(reinterpret_cast<float*>(s_tw2), a.tables + TB::TW2, 2 * (C::TW2 + C::TW3 + C::POST));
    const int team = threadIdx.x / T, t = threadIdx.x % T;
    /* OUT_LOGMEL: schedule tables | one power row per team (tail kept at zero) | one row of band sums per team */
    float4* s_melw = reinterpret_cast<float4*>(s_bar + ((G + 1) & ~1));
    int2* s_melseg = nullptr;
    float *prow = nullptr, *mout = nullptr, *row_a = nullptr;
    if constexpr (OUT == OUT_LOGMEL) {
        static_assert(T == 32, "the fused log-mel phase is written for one-warp teams");
        s_melseg = reinterpret_cast<int2*>(s_melw + a.mel_S * MEL_U * 32);
        float* s_mout = reinterpret_cast<float*>(s_melseg + a.mel_S * 32);
        const int nmp = (a.n_mels + 31) & ~31;
        copy_table(reinterpret_cast<float*>(s_melw), reinterpret_cast<const float*>(a.mel_w), a.mel_S * MEL_U * 32 * 4);
        copy_table(reinterpret_cast<float*>(s_melseg), reinterpret_cast<const float*>(a.mel_seg), a.mel_S * 32 * 2);
        /* the power row lives in the lower half of the team's exchange buffer: the split step publishes and reads only the
         * upper half (floats >= 2 pad(M/2)), and the next frame's first pass overwrites it after the closing team barrier */
        prow = reinterpret_cast<float*>(s_xb + team * C::XBUF);
        mout = s_mout + team * nmp;
        if (a.mel_pair) {                /* per team: [parked row (written only by the split step, tail stays zero) | band sums of two frames] */
            const int stride = a.mel_prow + 2 * nmp;
            for (int i = threadIdx.x; i < G * stride; i += blockDim.x) s_mout[i] = 0.f;
            row_a = s_mout + team * stride;
            mout = row_a + a.mel_prow;
        }
    }
    bool have_a = false;                                                  /* OUT_LOGMEL, pairs: row_a holds a frame that waits for its partner */
    long long out_a = 0;
    if (t == 0) mbar_init(&s_bar[team], 1);
    __syncthreads();

    float2* xb = s_xb + team * C::XBUF;
    float2* ring = s_ring + team * RING * HB;
    unsigned long long* bar = &s_bar[team];
    unsigned parity = 0;

    float2 win[E];                                                    /* window of this thread's sample pairs */
#pragma unroll
    for (int r = 0; r < E; ++r) win[r] = __ldg(reinterpret_cast<const float2*>(a.tables + TB::WIN) + t + T * r);
    constexpr bool REGTW = (C::T == 32 && C::NP == 2 && C::R1 == 32 && C::R2 == 32);
    TwBase twb;
    if constexpr (REGTW && !VVB_FWD_BASETW) twb = load_tw_base<C>(reinterpret_cast<const float2*>(a.tables + TB::TW2), t);
    const float2 hw_t = __ldg(reinterpret_cast<const float2*>(a.tables + TB::POST) + t);   /* (cos, sin)(2 pi t/N)/2, t < T <= M/2 */

    const int F = a.frames;
    const long long total = (long long)a.num_groups * F;              /* num_groups carries the batch */
    const long long nteams = (long long)gridDim.x * G;
    const long long quota = (total + nteams - 1) / nteams;
    long long g0 = ((long long)blockIdx.x * G + team) * quota;
    const long long g1 = min(total, g0 + quota);

    while (g0 < g1) {
        const int b = (int)(g0 / F);
        const int f_begin = (int)(g0 - (long long)b * F);
        const int f_end = (int)min((long long)F, (long long)f_begin + (g1 - g0));
        const float* xs = a.x + (long long)b * a.x_pitch;
        const bool bulk_ok = (reinterpret_cast<uintptr_t>(xs) & 15) == 0;
        g0 += f_end - f_begin;

        /* bring hop-block j into its ring slot: samples [origin + j*HOP, origin + (j+1)*HOP), where origin is
         * 0 (frames start at f*hop, zeros outside the signal) or -N/2 (centred frames, edge-inclusive
         * reflection outside the signal: src/core/framing.c:21-56,86-102).  Returns true if a TMA copy was
         * issued (completion must then be awaited on the mbarrier); blocks that touch a signal edge are
         * filled by the threads with the padding rule. */
        const long long origin = (a.pad_mode == PAD_REFLECT) ? -(long long)M : 0;      /* M = N/2 */
        auto load_block = [&](int j) -> bool {
            float2* dst = ring + (j % RING) * HB;
            const long long s0 = origin + (long long)j * HOP;
            if (bulk_ok && s0 >= 0 && s0 + HOP <= a.n) {
                if (t == 0) {
                    fence_proxy_async();
                    mbar_expect_tx(bar, HOP * 4);
                    bulk_load(dst, xs + s0, HOP * 4, bar);
                }
                return true;
            }
#pragma unroll
            for (int r = 0; r < S; ++r) {
                const long long i0 = s0 + 2 * (t + T * r);
                dst[t + T * r] = make_float2(fetch_sample(xs, a.n, i0, a.pad_mode), fetch_sample(xs, a.n, i0 + 1, a.pad_mode));
            }
            return false;
        };

        /* prologue: the N/hop blocks of the first frame.  All TMA copies are issued at once against ONE transaction
         * count (a range then starts after one memory latency instead of N/hop of them: with ~36 frames per team, as on
         * 8 GPUs of a sharded stream, that was ~5 % of the kernel); blocks that touch a signal edge are filled by hand */
        team_sync<T>(team);
        {
            int nbulk = 0;
#pragma unroll 1
            for (int q = 0; q < NB; ++q) {
                const long long s0 = origin + (long long)(f_begin + q) * HOP;
                nbulk += (bulk_ok && s0 >= 0 && s0 + HOP <= a.n) ? 1 : 0;
            }
            if (nbulk && t == 0) { fence_proxy_async(); mbar_expect_tx(bar, (unsigned)nbulk * HOP * 4); }
#pragma unroll 1
            for (int q = 0; q < NB; ++q) {
                const int j = f_begin + q;
                float2* dst = ring + (j % RING) * HB;
                const long long s0 = origin + (long long)j * HOP;
                if (bulk_ok && s0 >= 0 && s0 + HOP <= a.n) {
                    if (t == 0) bulk_load(dst, xs + s0, HOP * 4, bar);
                } else {
#pragma unroll
                    for (int r = 0; r < S; ++r) {
                        const long long i0 = s0 + 2 * (t + T * r);
                        dst[t + T * r] = make_float2(fetch_sample(xs, a.n, i0, a.pad_mode), fetch_sample(xs, a.n, i0 + 1, a.pad_mode));
                    }
                }
            }
            if (nbulk) { mbar_wait(bar, parity); parity ^= 1; }
        }
        bool pending = false;

#pragma unroll 1
        for (int frame = f_begin; frame < f_end; ++frame) {
            if (pending) { mbar_wait(bar, parity); parity ^= 1; }      /* block frame+NB-1 has landed */
            team_sync<T>(team);                                        /* ... and manual fills are visible */
            /* fetch the next frame's new block now: it goes to the slot of block frame-1, which nobody
             * reads any more, and has this whole frame's FFT to arrive */
            pending = (frame + 1 < f_end) ? load_block(frame + NB) : false;
            float2 v[E];
#pragma unroll
            for (int r = 0; r < E; ++r) {
                v[r] = __fmul2_rn(ring[((frame + r / S) % RING) * HB + t + T * (r % S)], win[r]);
            }
#ifdef VVB_SPLIT_SHFL
            constexpr bool SPLIT_SHFL = REGTW;
#else
            constexpr bool SPLIT_SHFL = false;     /* measured on B200: 3.05 ms vs 1.72 ms -- SHFL is the slower path */
#endif
            if constexpr (SPLIT_SHFL) {
                team_fft_regtw<C>(v, xb, twb, t, team);
                split_shuffle_store<C, OUT>(v, hw_t, t, a.out, ((long long)b * F + frame) * a.out_pitch);
            } else if constexpr (REGTW) {
                if constexpr (VVB_FWD_BASETW) team_fft_basetw<C>(v, xb, s_tw2, t, team);
                else team_fft_regtw<C>(v, xb, twb, t, team);
                if constexpr (OUT == OUT_LOGMEL) {
                    const long long orow = (long long)b * F + frame;
                    const bool park = a.mel_pair && !have_a;
                    split_and_store_half<C, OUT, true>(v, xb, hw_t, s_post, t, team, park ? row_a : prow, 0);
                    if (park) {
                        have_a = true; out_a = orow;
                    } else {
                        if (M + 1 + t < a.mel_prow) prow[M + 1 + t] = 0.f;  /* quads past the last bin read zeros, not stale exchange data */
                        if (a.mel_pair) mel_phase<2>(a, s_melw, s_melseg, row_a, prow, mout, t, out_a, orow);
                        else mel_phase<1>(a, s_melw, s_melseg, prow, prow, mout, t, orow, orow);
                        have_a = false;
                    }
                } else if constexpr (VVB_FWD_HALF_SPLIT) {
                    split_and_store_half<C, OUT, true>(v, xb, hw_t, s_post, t, team, a.out, ((long long)b * F + frame) * a.out_pitch);
                } else {
                    team_store_natural<C>(v, xb, t);
                    team_sync<T>(team);
                    split_and_store_rot<C, OUT>(xb, hw_t, t, a.out, ((long long)b * F + frame) * a.out_pitch);
                }
                team_sync<T>(team);                                    /* xb is reused by the next frame */
            } else {
                /* computed inter-pass twiddles, same-box A/B (1024 x 480000 samples): fft_size 4096 complex 2.528 -> 2.472 ms,
                 * power 2.218 -> 2.263 ms; fft_size 8192 complex unchanged, power 2.476 -> 2.619 ms: kept where they pay */
                /* (fft_size 4096, 32.8.8: the computed version also exchanges only half of the data between passes 2 and 3,
                 * complex 2.455 -> 2.274 ms on one box, so every output kind takes it there) */
                team_fft_march<C, (C::M == 2048)>(v, xb, s_tw2, s_tw3, t, team);
                /* computed split twiddles help at fft_size 4096 (2.94 -> 2.86 ms) and hurt at 8192 (3.24 -> 3.75 ms) */
                /* (fft_size 8192 with power / magnitude output is the one case measured slower with the half exchange:
                 * 2.46 -> 2.58 ms, while its complex output gains 8 %) */
                if constexpr (VVB_FWD_HALF_SPLIT && !(C::M == 4096 && OUT != OUT_COMPLEX)) {
                    split_and_store_half<C, OUT, (C::M <= 2048)>(v, xb, hw_t, s_post, t, team, a.out, ((long long)b * F + frame) * a.out_pitch);
                } else {
                    team_store_natural<C>(v, xb, t);
                    team_sync<T>(team);
                    if constexpr (C::M <= 2048) split_and_store_rot<C, OUT>(xb, hw_t, t, a.out, ((long long)b * F + frame) * a.out_pitch);
                    else split_and_store<C, OUT>(xb, s_post, t, a.out, ((long long)b * F + frame) * a.out_pitch);
                }
                team_sync<T>(team);                                    /* xb is reused by the next frame */
            }
        }
    }
    if constexpr (OUT == OUT_LOGMEL) {
        if (have_a) mel_phase<1>(a, s_melw, s_melseg, row_a, row_a, mout, t, out_a, out_a);    /* odd number of frames in this team's range */
    }
}

/* =============================================================== inverse (synthesis) */
/* Load the half spectrum of one frame, merge to Z (stored re/im swapped so the forward FFT
 * machinery computes the inverse), run the FFT, multiply by the synthesis window.
 * On exit: out2[i] = (x[2i], x[2i+1]) * wsyn for this thread's items i = j + r*NS. */
template <class C>
VVB_DEV void team_inverse_frame(float2 (&v)[C::E], const float2* X, bool active, float2* xb, const float2* s_tw2,
                                const float2* s_tw3, const float2* s_post, int t, int team)
{
    constexpr int M = C::M, E = C::E, T = C::T;
    /* ---- merge: Z[k] = (X[k]+conj X[M-k])/2 + (j/2) conj(W_N^k) (X[k]-conj X[M-k]) */
#pragma unroll
    for (int i = 0; i < E / 2; ++i) {
        const int k = t + T * i;                                      /* 0 .. M/2-1 */
        float2 a = make_float2(0.f, 0.f), b = make_float2(0.f, 0.f);
        if (active) { a = __ldg(X + k); b = __ldg(X + (M - k)); }
        if (k == 0) { a.y = 0.f; b.y = 0.f; }                         /* Re(IDFT): DC / Nyquist imag drop out */
        const float2 hw = s_post[k];
        const float sr = a.x + b.x, si = a.y - b.y;                   /* a + conj(b) */
        const float dr = a.x - b.x, di = a.y + b.y;                   /* a - conj(b) */
        const float ur = -hw.y * dr - hw.x * di, ui = -hw.y * di + hw.x * dr;
        const float zr = 0.5f * sr + ur, zi = 0.5f * si + ui;         /* Z[k]   */
        const float yr = 0.5f * sr - ur, yi = -(0.5f * si - ui);      /* Z[M-k] */
        xb[C::pad(k)] = make_float2(zi, zr);                          /* swapped */
        if (k != 0) xb[C::pad(M - k)] = make_float2(yi, yr);
    }
    if (t == 0) {                                                     /* k = M/2: Z = conj(X[M/2]) */
        float2 a = make_float2(0.f, 0.f);
        if (active) a = __ldg(X + M / 2);
        xb[C::pad(M / 2)] = make_float2(-a.y, a.x);
    }
    team_sync<T>(team);
    {   /* pass-1 operands from the natural-order buffer */
        constexpr int R = C::R1, NQ = E / R, STRIDE = M / R;
#pragma unroll
        for (int q = 0; q < NQ; ++q)
#pragma unroll
            for (int r = 0; r < R; ++r) v[q * R + r] = xb[C::pad(t + T * q + r * STRIDE)];
    }
    team_sync<T>(team);
    team_fft<C>(v, xb, s_tw2, s_tw3, t, team);
}

/* one round of the slot-based overlap-add of stft_inverse_kernel (V samples per thread and step) */
template <class C, int G, int V>
VVB_DEV void ola_combine(const InvArgs& a, const float2* s_xb, const float* carry_in, float* carry_out, float* yb,
                         long long fb, int hop, int edge, int K, int nblk, long long out_lo, long long out_hi, bool normalise)
{
    using TB = Tables<C>;
    constexpr int N = 2 * C::M;
    const long long tail0 = (long long)a.frames * hop;
    /* one flat index space over (hop-block, sample group): with a loop over the hop-blocks and the threads dealt over ONE
     * block, a hop of 160 kept 40 of 256 threads busy (fft_size 400 / hop 160: ISTFT 3.39 ms, 4.5 x the forward kernel) */
    const int per_blk = (hop + V - 1) / V;
    for (int w = threadIdx.x; w < nblk * per_blk; w += blockDim.x) {
        const int hb = w / per_blk;
        const int g_lo = max(0, hb - K + 1), g_hi = min(G - 1, hb);
        {
            const int cidx = (w - hb * per_blk) * V;
            const int s = hb * hop + cidx;
            if (s >= G * hop + edge) continue;
            float acc[V];
#pragma unroll
            for (int j = 0; j < V; ++j) acc[j] = (s < edge) ? carry_in[s + j] : 0.f;
            for (int g = g_lo; g <= g_hi; ++g) {
                const int p = s - g * hop;
                if (p < N) {
                    const float* slot = reinterpret_cast<const float*>(s_xb + g * C::XBUF) + p;
                    if constexpr (V == 4) {
                        const float4 q = *reinterpret_cast<const float4*>(slot);
                        acc[0] += q.x; acc[1] += q.y; acc[2] += q.z; acc[3] += q.w;
                    } else {
                        acc[0] += slot[0];
                    }
                }
            }
            if (s < G * hop) {
                const long long tt = fb * hop + s;
                if (normalise && (tt < edge || tt + V > tail0)) {
                    /* edge region: undo the steady-state factor folded into the window, apply the true one */
#pragma unroll
                    for (int j = 0; j < V; ++j) {
                        const long long u = tt + j;
                        float sc;
                        if (u >= tail0) sc = (u - tail0 < edge) ? __ldg(a.inv_norm + edge + hop + (u - tail0)) : 0.f;
                        else if (u < edge) sc = __ldg(a.inv_norm + u);
                        else sc = __ldg(a.inv_norm + edge + cidx + j);
                        acc[j] *= sc * __ldg(a.tables + TB::MIDNORM + cidx + j);
                    }
                }
                if constexpr (V == 4) {
                    if (tt >= out_lo && tt + 3 < out_hi) {
                        *reinterpret_cast<float4*>(yb + tt) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                        continue;
                    }
                }
#pragma unroll
                for (int j = 0; j < V; ++j)
                    if (tt + j >= out_lo && tt + j < out_hi) yb[tt + j] = acc[j];
            } else {
#pragma unroll
                for (int j = 0; j < V; ++j) carry_out[s - G * hop + j] = acc[j];
            }
        }
    }
}

template <class C, int G, bool OLA>
__global__ void __launch_bounds__(C::T* G) stft_inverse_kernel(const InvArgs a)
{
    using TB = Tables<C>;
    using L = LastPass<C>;
    constexpr int M = C::M, N = 2 * M, E = C::E, T = C::T;
#ifdef VVB_EMU
    float* smem = reinterpret_cast<float*>(vvb_emu::g_dyn_smem);
#else
    extern __shared__ __align__(16) float smem[];
#endif
    float* s_wsyn = smem;                                             /* N floats */
    float2* s_tw2 = reinterpret_cast<float2*>(s_wsyn + N);
    float2* s_tw3 = s_tw2 + C::TW2;
    float2* s_post = s_tw3 + C::TW3;
    float2* s_xb = s_post + C::POST + 1;
    float* s_carry = reinterpret_cast<float*>(s_xb + G * C::XBUF);    /* 2 x (N - hop) floats (OLA) */
    /* normalised overlap-add: steady-state 1/sum(w^2) folded into the synthesis window (see istft_march_kernel) */
    const bool normalise = OLA && a.inv_norm != nullptr;
    copy_table(s_wsyn, a.tables + (normalise ? TB::WSYN_NORM : TB::WSYN), N);
    copy_table(reinterpret_cast<float*>(s_tw2), a.tables + TB::TW2, 2 * (C::TW2 + C::TW3 + C::POST));
    __syncthreads();

    const int team = threadIdx.x / T, t = threadIdx.x % T;
    float2* xb = s_xb + team * C::XBUF;
    const float2* wsyn2 = reinterpret_cast<const float2*>(s_wsyn);
    const int hop = a.hop;

    if constexpr (!OLA) {
        /* windowed frames out, no overlap-add: item = group of G frames of the flat frame list */
        for (int item = blockIdx.x; item < a.num_items; item += gridDim.x) {
            const int f = item * G + team;
            const bool active = f < a.frames;
            float2 v[E];
            team_inverse_frame<C>(v, a.spec + (long long)f * a.spec_pitch, active, xb, s_tw2, s_tw3, s_post, t, team);
            if (active) {
                float2* dst = reinterpret_cast<float2*>(a.y + (long long)f * N);
#pragma unroll
                for (int q = 0; q < L::NQ; ++q)
#pragma unroll
                    for (int r = 0; r < L::R; ++r) {
                        const int i = t + T * q + r * L::NS;
                        const float2 z = v[q * L::R + ct_bitrev(r, L::R)], w = wsyn2[i];
                        dst[i] = make_float2(z.y * w.x, z.x * w.y);   /* (Re z, Im z) after un-swap */
                    }
            }
            team_sync<T>(team);
        }
        return;
    } else {
        const int edge = N - hop;                                     /* samples a frame shares with later ones */
        const int K = (N + hop - 1) / hop;                            /* frames covering one sample */
        const int nblk = (G * hop + edge + hop - 1) / hop;            /* hop-blocks in the accumulation span */
        for (int item = blockIdx.x; item < a.num_items; item += gridDim.x) {
            const int b = item / a.chunks_per_signal;
            const int c = item % a.chunks_per_signal;
            const int f_begin = c * a.chunk_frames;
            const int f_end = min(a.frames, f_begin + a.chunk_frames);
            const bool last = (f_end >= a.frames);
            const long long out_lo = (long long)f_begin * hop;
            const long long out_hi = last ? a.n_out : min(a.n_out, (long long)f_end * hop);
            const int fr0 = f_begin - min(K - 1, f_begin);            /* halo frames re-synthesised */
            const float2* specb = a.spec + (long long)b * a.frames * a.spec_pitch;
            float* yb = a.y + (long long)b * a.y_pitch;

            for (int i = threadIdx.x; i < 2 * edge; i += blockDim.x) s_carry[i] = 0.f;
            int cur = 0;
            __syncthreads();

            for (long long fb = fr0; fb * hop < out_hi; fb += G) {
                const long long f = fb + team;
                const bool active = f < f_end;
                float2 v[E];
                team_inverse_frame<C>(v, specb + f * a.spec_pitch, active, xb, s_tw2, s_tw3, s_post, t, team);
                /* park the windowed frame in this team's slot, natural sample order */
#pragma unroll
                for (int q = 0; q < L::NQ; ++q)
#pragma unroll
                    for (int r = 0; r < L::R; ++r) {
                        const int i = t + T * q + r * L::NS;
                        const float2 z = v[q * L::R + ct_bitrev(r, L::R)], w = wsyn2[i];
                        xb[i] = make_float2(z.y * w.x, z.x * w.y);
                    }
                __syncthreads();

                /* conflict-free overlap-add: every output sample is summed once, by one thread, from the slots
                 * that cover it, in ascending frame order; four samples per thread (128-bit shared-memory and
                 * global accesses) when hop and the output row are 4-sample aligned */
                const float* carry_in = s_carry + cur * edge;
                float* carry_out = s_carry + (cur ^ 1) * edge;
                const bool vec4 = ((hop & 3) == 0) && ((reinterpret_cast<uintptr_t>(yb) & 15) == 0);
                if (vec4) ola_combine<C, G, 4>(a, s_xb, carry_in, carry_out, yb, fb, hop, edge, K, nblk, out_lo, out_hi, normalise);
                else ola_combine<C, G, 1>(a, s_xb, carry_in, carry_out, yb, fb, hop, edge, K, nblk, out_lo, out_hi, normalise);
                cur ^= 1;
                __syncthreads();
            }
        }
    }
}

/* ================================================= inverse, warp-marching specialisation */
/* For one-warp teams (T == 32, i.e. fft_size 2048) and hop = 64*S: a warp walks consecutive
 * frames of one signal and keeps the overlap-add accumulator IN REGISTERS.  Thread t owns the
 * sample pairs (2i, 2i+1), i = t + 32 r, of every frame; advancing one frame shifts positions by
 * hop = 2*32*S samples = S register slots of the SAME thread, so the accumulator is a register
 * ring rotated by S slots per frame (compile-time indices: the frame loop is unrolled 32/S
 * times).  After frame f is added, the first S slots hold finished samples [f*hop, (f+1)*hop):
 * they are scaled by 1/sum(w^2) and stored with coalesced 64-bit stores, then cleared.
 * No shared-memory slots, no carry buffers, no CTA barriers, no atomics; frames are added in
 * ascending order exactly like the reference accumulates out_add (src/spectral/stft.c:103-108).
 * Work is split into equal ranges of the flattened (signal, frame) sequence, one range per
 * warp; a range that starts mid-signal first re-synthesises the 32/S - 1 frames before it. */
/* merge step of the marching ISTFT for one bin k = t + T*R of this thread (R compile time):
 *     Z[k] = (X[k] + conj X[M-k])/2 + (j/2) conj(W_N^k) (X[k] - conj X[M-k]),  W_N^k = W_N^t * W_{2E}^R
 * read from the staged half spectrum, result stored re/im swapped for the forward-FFT trick */
template <class C, int R> VVB_DEV void march_merge_one(float2 (&v)[C::E], const float2* st, int t, float2 hw_t)
{
    constexpr int M = C::M, T = C::T;
    float2 x = st[t + T * R];                                         /* st: staged X[0..M], natural order */
    float2 y = st[M - t - T * R];
    if constexpr (R == 0) {
        if (t == 0) { x.y = 0.f; y.y = 0.f; }                          /* Re(IDFT): DC / Nyquist imag drop out */
    }
    constexpr float cr = TwC<2 * C::E, R>::c, sr = TwC<2 * C::E, R>::s;
    const float2 h = cmul(hw_t, make_float2(cr, sr));                 /* (cos, sin)(2 pi k/N)/2 = hw_t rotated */
    const float2 sm = __fadd2_rn(x, make_float2(y.x, -y.y));          /* x + conj(y) */
    const float2 df = __fadd2_rn(x, make_float2(-y.x, y.y));          /* x - conj(y) */
    const float2 u = cmul(df, make_float2(-h.y, h.x));                /* (j/2) conj(W_N^k) * df */
    v[R] = __ffma2_rn(splat(0.5f), make_float2(sm.y, sm.x), make_float2(u.y, u.x));   /* (Im Z, Re Z) */
}
template <class C, int... Rs> VVB_DEV void march_merge(float2 (&v)[C::E], const float2* st, int t, float2 hw_t, iseq<Rs...>)
{
    (march_merge_one<C, Rs>(v, st, t, hw_t), ...);
}

/* ---- the same merge with every pair (k, M-k) formed ONCE (one-warp 32 x 32 transforms).
 * Lane t owns column t of the first pass: bins k = t + 32 R in slot R.  The partner bin M - k = (32 - t) + 32 (31 - R)
 * lives in lane 32 - t, slot 31 - R, so lane t forms Z[k] AND Z[M-k] for its lower slots R < 16 from one load of
 * (X[k], X[M-k]) and one shared sum / difference / twiddle product (8 packed instructions per pair instead of 2 x 7,
 * 32 staged loads per frame instead of 64), keeps Z[k] and hands Z[M-k] to lane 32 - t, which files it in slot 31 - R.
 * Lane 16 is its own partner (the shuffle returns its own value); lane 0 owns the self-paired column 0, whose partner
 * of slot R is slot 32 - R: it takes its own values one slot further up, and slot 16 (k = M/2) is conj X[M/2].
 * MODE 1 moves the partner values with SHFL, MODE 2 through the team's exchange buffer at their natural position. */
/* streaming 8-byte load of a spectrum bin straight from global memory (read once, not worth a place in L1) */
VVB_DEV float2 load_bin_global(const float2* p)
{
#ifdef VVB_EMU
    return *p;
#else
    return __ldcs(p);
#endif
}
/* phase 1 of a pair: the two loads (GLOBAL: from the spectrum row in HBM / L2; otherwise from the staged copy) */
template <class C, int R, bool GLOBAL> VVB_DEV void march_pair_load(float2 (&x)[C::E / 2], float2 (&y)[C::E / 2], const float2* st, int t)
{
    constexpr int M = C::M, T = C::T;
    if constexpr (GLOBAL) { x[R] = load_bin_global(st + t + T * R); y[R] = load_bin_global(st + M - t - T * R); }
    else { x[R] = st[t + T * R]; y[R] = st[M - t - T * R]; }
}
template <class C, int R> VVB_DEV void march_merge_pair_math(float2 (&v)[C::E], float2 (&zp)[C::E / 2], float2 x, float2 y, int t, float2 hw_t)
{
    if constexpr (R == 0) {
        if (t == 0) { x.y = 0.f; y.y = 0.f; }                          /* Re(IDFT): DC / Nyquist imag drop out */
    }
    constexpr float cr = TwC<2 * C::E, R>::c, sr = TwC<2 * C::E, R>::s;
    const float2 h = cmul(hw_t, make_float2(cr, sr));                 /* (cos, sin)(2 pi k/N)/2 */
    const float2 sm = __fadd2_rn(x, make_float2(y.x, -y.y));          /* x + conj(y) */
    const float2 df = __fadd2_rn(x, make_float2(-y.x, y.y));          /* x - conj(y) */
    const float2 u = cmul(df, make_float2(-h.y, h.x));                /* (j/2) conj(W_N^k) * df */
    v[R] = __ffma2_rn(splat(0.5f), make_float2(sm.y, sm.x), make_float2(u.y, u.x));                  /* Z[k]   as (Im, Re) */
    zp[R] = __ffma2_rn(make_float2(-0.5f, 0.5f), make_float2(sm.y, sm.x), make_float2(u.y, -u.x));   /* Z[M-k] = conj(sm/2 - u) as (Im, Re) */
}
template <class C, bool GLOBAL, int... Rs> VVB_DEV void march_merge_pairs_compute(float2 (&v)[C::E], float2 (&zp)[C::E / 2], const float2* st, int t, float2 hw_t, iseq<Rs...>)
{
    float2 x[C::E / 2], y[C::E / 2];
    (march_pair_load<C, Rs, GLOBAL>(x, y, st, t), ...);               /* all loads in flight before the first use */
    (march_merge_pair_math<C, Rs>(v, zp, x[Rs], y[Rs], t, hw_t), ...);
}
template <class C, int MODE, bool GLOBAL = false> VVB_DEV void march_merge_pairs(float2 (&v)[C::E], const float2* st, float2* xb, int t, float2 hw_t)
{
    static_assert(C::T == 32 && C::E == 32, "one-warp 32 x 32 transforms");
    constexpr int M = C::M, H = C::E / 2;
    float2 zp[H];
    const float2 nyq = GLOBAL ? load_bin_global(st + M / 2) : st[M / 2];   /* k = M/2 (lane 0, slot 16): Z = conj X[M/2] */
    march_merge_pairs_compute<C, GLOBAL>(v, zp, st, t, hw_t, typename make_iseq<H>::type{});
    if constexpr (MODE == 1) {
        const int src = (32 - t) & 31;
        float2 rc[H];
#pragma unroll
        for (int r = 0; r < H; ++r) {
            rc[r].x = __shfl_sync(0xffffffffu, zp[r].x, src);
            rc[r].y = __shfl_sync(0xffffffffu, zp[r].y, src);
        }
        const bool col0 = (t == 0);
#pragma unroll
        for (int r = 0; r < H - 1; ++r) {                              /* slot 31 - r <- partner's pair r (lane 0: its own pair r + 1) */
            v[31 - r].x = col0 ? rc[r + 1].x : rc[r].x;
            v[31 - r].y = col0 ? rc[r + 1].y : rc[r].y;
        }
        v[H].x = col0 ? -nyq.y : rc[H - 1].x;
        v[H].y = col0 ? nyq.x : rc[H - 1].y;
    } else {
#pragma unroll
        for (int r = 0; r < H; ++r) {
            const int p = (M - t - 32 * r) & (M - 1);                  /* natural position of Z[M-k]; k = 0 has no partner slot */
            if (r > 0 || t > 0) xb[C::pad(p)] = zp[r];
        }
        if (t == 0) xb[C::pad(M / 2)] = make_float2(-nyq.y, nyq.x);
        __syncwarp();
#pragma unroll
        for (int r = H; r < 2 * H; ++r) v[r] = xb[C::pad(t + 32 * r)];
        __syncwarp();                                                  /* all partner values read before pass 1 overwrites xb */
    }
}

template <class C, int S, int G, int MINB>
__global__ void __launch_bounds__(C::T* G, MINB) istft_march_kernel(const InvArgs a)
{
    static_assert(C::T >= 32 && C::R1 == C::E && C::E % S == 0, "whole-warp teams, pass-1 radix == points per thread");
    using TB = Tables<C>;
    using L = LastPass<C>;
    constexpr int M = C::M, N = 2 * M, E = C::E, T = C::T;
    constexpr int PERIOD = E / S, HOP = 2 * T * S, EDGE = N - HOP;    /* PERIOD frames overlap one sample */
    constexpr int STG = M + 2;                                        /* staged half spectrum X[-1|0 .. M] */
#ifdef VVB_EMU
    float* smem = reinterpret_cast<float*>(vvb_emu::g_dyn_smem);
#else
    extern __shared__ __align__(16) float smem[];
#endif
    float* s_wsyn = smem;
    float2* s_tw2 = reinterpret_cast<float2*>(s_wsyn + N);
    float2* s_tw3 = s_tw2 + C::TW2;
    float2* s_xb = s_tw3 + C::TW3;
    float2* s_stage = s_xb + G * C::XBUF;
    unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(s_stage + G * STG);
    /* normalised synthesis: the steady-state 1/sum(w^2) is already folded into the window table, so the
     * main path has no per-sample table load or multiply; only the first/last PERIOD-1 hop-blocks of a
     * signal (fewer frames overlap there) are rescaled, below */
    const bool normalise = a.inv_norm != nullptr;
    copy_table(s_wsyn, a.tables + (normalise ? TB::WSYN_NORM : TB::WSYN), N);
    copy_table(reinterpret_cast<float*>(s_tw2), a.tables + TB::TW2, 2 * (C::TW2 + C::TW3));
    const int team = threadIdx.x / T, t = threadIdx.x % T;
    if (t == 0) mbar_init(&s_bar[team], 1);
    __syncthreads();

    float2* xb = s_xb + team * C::XBUF;                               /* FFT exchange buffer of this team */
    float2* stage = s_stage + team * STG;                             /* next frame's spectrum lands here */
    unsigned long long* bar = &s_bar[team];
    unsigned parity = 0;
    const float2* wsyn2 = reinterpret_cast<const float2*>(s_wsyn);
    /* split-step twiddle of this thread: (cos, sin)(2 pi t / N) / 2; its bins k = t + T r differ from it
     * by the compile-time rotation 2 pi r / (2E) */
    const float2 hw_t = __ldg(reinterpret_cast<const float2*>(a.tables + TB::POST) + t);   /* t < T <= M/2 */
    /* Twiddle bases held in registers across frames, as in the forward kernel, push this kernel from 242 to 255
     * registers and into spills (2.25 vs 2.12 ms measured) because of the 64-register accumulator.  The 32 x 32
     * configuration instead re-reads the five bases from shared memory every frame (team_fft_basetw below):
     * they are live only during the twiddle phase, 26 of the 31 LDS.64 disappear, 2.02 -> 1.91 ms. */
    constexpr bool REGTW = false;
    [[maybe_unused]] TwBase twb;
    if constexpr (REGTW) twb = load_tw_base<C>(reinterpret_cast<const float2*>(a.tables + TB::TW2), t);
    const int F = a.frames;
    const long long total = (long long)a.num_items * F;               /* num_items carries the batch */
    const long long nteams = (long long)gridDim.x * G;
    const long long quota = (total + nteams - 1) / nteams;
    long long g0 = ((long long)blockIdx.x * G + team) * quota;
    const long long g1 = min(total, g0 + quota);

    while (g0 < g1) {
        const int b = (int)(g0 / F);
        const int f_begin = (int)(g0 - (long long)b * F);
        const int f_end = (int)min((long long)F, (long long)f_begin + (g1 - g0));
        const int emit_end = (f_end == F && a.tail_edge) ? f_end + PERIOD - 1 : f_end;   /* hop-blocks [f_begin, emit_end) are ours */
        const int emit_begin = max(f_begin, a.halo_frames);            /* halo frames: overlap only, nothing emitted */
        const int fr0 = f_begin - min(PERIOD - 1, f_begin);            /* halo frames re-synthesised */
        [[maybe_unused]] const float2* specb = a.spec + (long long)b * F * a.spec_pitch;
        float* yb = a.y + (long long)b * a.y_pitch;
        const bool y8 = (reinterpret_cast<uintptr_t>(yb) & 7) == 0;    /* 64-bit stores possible for this signal's row */
        g0 += f_end - f_begin;

        /* asynchronous copy of one frame's half spectrum X[0..M] into the team's staging buffer, issued right
         * after the previous frame's merge has consumed the buffer, so it is in flight for a whole frame.
         * Preferred: ONE TMA bulk copy (cp.async.bulk) by one thread.  Rows are (M+1)*8 bytes, i.e. only
         * 8-byte aligned on odd rows; the copy then starts 8 bytes early (the previous row's last bin) and
         * the merge reads at an offset of one element.  Both cases move (M+2)*8 bytes.  Fallback (base not
         * 16-byte aligned, odd pitch overflow, or the very last row of the buffer, where reading 8 bytes
         * past the end would leave the allocation): per-thread 8-byte cp.async (LDGSTS). */
        const bool spec16 = (reinterpret_cast<uintptr_t>(a.spec) & 15) == 0;
        auto prefetch = [&](int frame, int& off, bool& bulk) {
            off = 0; bulk = false;
            if (frame < f_end) {
                const long long rowi = (long long)b * F + frame;
                const float2* X = a.spec + rowi * a.spec_pitch;
                const int mis = (int)((rowi * a.spec_pitch) & 1);     /* 1: row starts 8 bytes past a 16-byte boundary */
                const bool last_row = (b == a.num_items - 1) && (frame == F - 1);
                if (spec16 && !last_row && (rowi > 0 || mis == 0)) {
                    off = mis; bulk = true;
                    if (t == 0) {
                        fence_proxy_async();
                        mbar_expect_tx(bar, STG * 8);
                        bulk_load(stage, X - mis, STG * 8, bar);
                    }
                } else {
#pragma unroll
                    for (int r = 0; r < E; ++r) cp_async8(&stage[t + T * r], X + t + T * r);
                    if (t == 0) cp_async8(&stage[M], X + M);
                }
            }
            cp_async_commit();
        };
        int off_next = 0, off_cur = 0;
        bool bulk_next = false, bulk_cur = false;

        float2 acc[E];
#pragma unroll
        for (int i = 0; i < E; ++i) acc[i] = make_float2(0.f, 0.f);
        prefetch(fr0, off_next, bulk_next);

#pragma unroll 1
        for (int frame = fr0; frame < emit_end; ++frame) {
            if (frame < f_end) {                                       /* team-uniform */
                float2 v[E];
                off_cur = off_next; bulk_cur = bulk_next;
                if (bulk_cur) { mbar_wait(bar, parity); parity ^= 1; } else cp_async_wait_all();
                team_sync<T>(team);
                /* merge straight into the pass-1 registers (see march_merge_one) */
                if constexpr (VVB_INV_PAIRMERGE != 0 && C::T == 32 && C::E == 32)
                    march_merge_pairs<C, VVB_INV_PAIRMERGE>(v, stage + off_cur, xb, t, hw_t);
                else
                    march_merge<C>(v, stage + off_cur, t, hw_t, typename make_iseq<E>::type{});
                team_sync<T>(team);                                    /* all reads of the staged X are done */
                prefetch(frame + 1, off_next, bulk_next);
                if constexpr (REGTW) team_fft_regtw<C>(v, xb, twb, t, team);
                else if constexpr (VVB_INV_BASETW && C::T == 32 && C::R1 == 32 && C::R2 == 32 && C::NP == 2) team_fft_basetw<C>(v, xb, s_tw2, t, team);
                else team_fft_march<C>(v, xb, s_tw2, s_tw3, t, team);   /* three passes: computed twiddles (fft_size 4096: 2.576 -> 2.522 ms, 8192: 2.830 -> 2.581 ms) */
                /* v[q*RL + r] is sample pair i = t + T*(q + NQ*r): accumulate into that slot */
#pragma unroll
                for (int q = 0; q < L::NQ; ++q)
#pragma unroll
                    for (int r = 0; r < L::R; ++r) {
                        const int sl = q + L::NQ * r;
                        const float2 z = v[q * L::R + r];
                        acc[sl] = __ffma2_rn(make_float2(z.y, z.x), wsyn2[t + T * sl], acc[sl]);   /* z is stored swapped */
                    }
            }
            if (frame >= emit_begin) {
                const long long base = (long long)(frame - a.halo_frames) * HOP;
                if (normalise && ((a.head_edge && frame < PERIOD - 1) || frame >= F)) {
                    /* edge block: fewer than PERIOD frames overlap; undo the folded steady-state factor and
                     * apply this block's own 1/sum(w^2) (head or tail table of InvArgs::inv_norm) */
                    const float* edge = (frame >= F) ? a.inv_norm + EDGE + HOP + (long long)(frame - F) * HOP
                                                     : a.inv_norm + (long long)frame * HOP;
                    const float* mid = a.tables + TB::MIDNORM;
#pragma unroll
                    for (int r = 0; r < S; ++r) {
                        const int c = 2 * (t + T * r);
                        acc[r].x *= __ldg(edge + c) * __ldg(mid + c);
                        acc[r].y *= __ldg(edge + c + 1) * __ldg(mid + c + 1);
                    }
                }
#pragma unroll
                for (int r = 0; r < S; ++r) {
                    const long long tt = base + 2 * (t + T * r);
                    if (y8 && tt + 1 < a.n_out) *reinterpret_cast<float2*>(yb + tt) = acc[r];
                    else {                                             /* row not 8-byte aligned (odd pitch), or the last sample */
                        if (tt < a.n_out) yb[tt] = acc[r].x;
                        if (tt + 1 < a.n_out) yb[tt + 1] = acc[r].y;
                    }
                }
            }
            /* advance one hop: slot r now means what slot r+S meant (register moves; an unrolled ring
             * of PERIOD frame bodies would not fit the instruction cache) */
#pragma unroll
            for (int r = 0; r < E - S; ++r) acc[r] = acc[r + S];
#pragma unroll
            for (int r = E - S; r < E; ++r) acc[r] = make_float2(0.f, 0.f);
        }
        cp_async_wait_all();                                           /* nothing in flight across pieces */
        team_sync<T>(team);
        if (f_end == F && a.tail_edge) {                               /* nothing covers [cov, n_out): zeros */
            const long long cov = (long long)(F - 1 - a.halo_frames) * HOP + N;
            for (long long tt = cov + t; tt < a.n_out; tt += T) yb[tt] = 0.f;
        }
    }
}

/* ================================================= inverse, two frames per complex transform */
/* fft_size N <= 1024: a warp turns TWO consecutive frames into one N-point COMPLEX transform,
 *     Z = X_f + j X_{f+1}  (Hermitian extensions)   =>   IDFT_N(Z) = x_f + j x_{f+1},
 * so there is no merge step and no merge twiddle, and the one-warp configurations with M = N apply
 * (N = 256: 8.8.4, N = 512: 16.16.2, N = 1024: 32.32).  Thread t owns the samples i = t + 32 s of both
 * frames (every output index of these configurations is congruent to t mod 32), the hop is HS slots of 32
 * samples, and the overlap-add accumulator is E + HS registers rotated by 2 HS slots per pair, exactly as
 * in istft_march_kernel: finished hop-blocks leave with coalesced 128-byte stores, no shared-memory slots,
 * no CTA barriers.  Frames are added in ascending order.  The window table is the real-transform one
 * (w / (N/2) [x 1/sum w^2]); the factor 1/2 that turns it into w / N is applied when it is loaded. */
struct PairArgs {
    const float2* spec; long long spec_pitch;
    int frames, num_items;
    float* y; long long y_pitch, n_out;
    const float* inv_norm;           /* edge tables as in InvArgs, nullptr = raw sum */
    const float* tables;             /* Tables<C> of the N-point complex plan (twiddles only) */
    const float* wsyn;               /* N floats: synthesis window of the real plan (normalisation folded in when inv_norm) */
    const float* midnorm;            /* hop floats: steady-state sum w^2 */
};

template <class C, int HS, int G, int MINB>
__global__ void __launch_bounds__(32 * G, MINB) istft_pair_kernel(const PairArgs a)
{
    static_assert(C::T == 32, "one-warp complex transform of size fft_size");
    using TB = Tables<C>;
    using L = LastPass<C>;
    constexpr int N = C::M, E = C::E, T = 32;
    constexpr int HOP = 32 * HS, PERIOD = E / HS, EDGE = N - HOP, HALO_PAIRS = PERIOD / 2;
    static_assert(E % HS == 0 && PERIOD >= 2 && L::NS % 32 == 0, "hop must divide fft_size");
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
    const bool normalise = a.inv_norm != nullptr;
    float w[E];                                                        /* w[s] for sample t + 32 s, already / N */
#pragma unroll
    for (int s2 = 0; s2 < E; ++s2) w[s2] = 0.5f * __ldg(a.wsyn + t + 32 * s2);

    const int F = a.frames;
    const int FP = (F + 1) / 2;                                        /* frame pairs per signal */
    const long long total = (long long)a.num_items * FP;
    const long long nteams = (long long)gridDim.x * G;
    const long long quota = (total + nteams - 1) / nteams;
    long long g0 = ((long long)blockIdx.x * G + team) * quota;
    const long long g1 = min(total, g0 + quota);

    while (g0 < g1) {
        const int b = (int)(g0 / FP);
        const int p_begin = (int)(g0 - (long long)b * FP);
        const int p_end = (int)min((long long)FP, (long long)p_begin + (g1 - g0));
        const int blk_begin = 2 * p_begin;                             /* hop-blocks [blk_begin, blk_end) are ours */
        const int blk_end = (p_end == FP) ? F + PERIOD - 1 : 2 * p_end;
        const int p0 = p_begin - min(HALO_PAIRS, p_begin);            /* halo pairs re-synthesised */
        const float2* specb = a.spec + (long long)b * F * a.spec_pitch;
        float* yb = a.y + (long long)b * a.y_pitch;
        g0 += p_end - p_begin;

        float acc[E + HS];
#pragma unroll
        for (int i = 0; i < E + HS; ++i) acc[i] = 0.f;

#pragma unroll 1
        for (int pair = p0; 2 * pair < blk_end; ++pair) {
            const int f0 = 2 * pair;
            if (pair < p_end) {                                        /* warp-uniform */
                const bool have1 = f0 + 1 < F;
                const float2* X1 = specb + (long long)f0 * a.spec_pitch;
                const float2* X2 = X1 + (have1 ? a.spec_pitch : 0);
                float2 v[E];
                {
                    constexpr int R = C::R1, NQ = E / R, STRIDE = N / R;
#pragma unroll
                    for (int q = 0; q < NQ; ++q)
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const int i = t + T * q + r * STRIDE;
                            const int k = (2 * i <= N) ? i : N - i;
                            float2 x1 = __ldg(X1 + k), x2 = __ldg(X2 + k);
                            if (!have1) x2 = make_float2(0.f, 0.f);
                            if (2 * i > N) { x1.y = -x1.y; x2.y = -x2.y; }           /* Hermitian extension */
                            if (k == 0 || 2 * k == N) { x1.y = 0.f; x2.y = 0.f; }    /* Re(IDFT): DC / Nyquist imag drop out */
                            /* Z = x1 + j x2, stored re/im swapped so the forward machinery computes the inverse */
                            v[q * R + r] = make_float2(x1.y + x2.x, x1.x - x2.y);
                        }
                }
                if constexpr (VVB_INV_BASETW && C::R1 == 32 && C::R2 == 32 && C::NP == 2) team_fft_basetw<C>(v, xb, s_tw2, t, team);
                else team_fft_march<C, VVB_PAIR_TW3>(v, xb, s_tw2, s_tw3, t, team);      /* three passes: computed inter-pass twiddles */
                /* v = (N x_{f+1}[i], N x_f[i]) for i = t + 32 (q + r NS/32) */
#pragma unroll
                for (int q = 0; q < L::NQ; ++q)
#pragma unroll
                    for (int r = 0; r < L::R; ++r) {
                        const int sl = q + r * (L::NS / 32);
                        const float2 z = v[q * L::R + ct_bitrev(r, L::R)];
                        acc[sl] = fmaf(z.y, w[sl], acc[sl]);
                    }
                /* an odd frame count leaves the last pair without its second frame: the imaginary part is then only the
                 * transform's rounding noise, which must not reach the tail samples (after the divide by a window-sum
                 * that falls towards 0 there it would be amplified without bound) */
                if (have1) {
#pragma unroll
                    for (int q = 0; q < L::NQ; ++q)
#pragma unroll
                        for (int r = 0; r < L::R; ++r) {
                            const int sl = q + r * (L::NS / 32);
                            const float2 z = v[q * L::R + ct_bitrev(r, L::R)];
                            acc[sl + HS] = fmaf(z.x, w[sl], acc[sl + HS]);
                        }
                }
            }
            /* the two oldest hop-blocks are complete: blocks f0 (slots 0..HS-1) and f0+1 (slots HS..2HS-1) */
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int blk = f0 + h;
                if (blk >= blk_begin && blk < blk_end) {
                    const long long base = (long long)blk * HOP;
                    const bool edge_blk = normalise && (blk < PERIOD - 1 || blk >= F);
                    const float* edge = nullptr;
                    if (edge_blk) edge = (blk >= F) ? a.inv_norm + EDGE + HOP + (long long)(blk - F) * HOP
                                                    : a.inv_norm + (long long)blk * HOP;
#pragma unroll
                    for (int s2 = 0; s2 < HS; ++s2) {
                        const int c = t + 32 * s2;
                        float val = acc[h * HS + s2];
                        if (edge_blk) val *= __ldg(edge + c) * __ldg(a.midnorm + c);
                        if (base + c < a.n_out) yb[base + c] = val;
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < E - HS; ++i) acc[i] = acc[i + 2 * HS];
#pragma unroll
            for (int i = E - HS; i < E + HS; ++i) acc[i] = 0.f;
        }
        if (p_end == FP) {                                             /* nothing covers [cov, n_out): zeros */
            const long long cov = (long long)(F - 1) * HOP + N;
            for (long long tt = cov + t; tt < a.n_out; tt += T) yb[tt] = 0.f;
        }
    }
}

/* ===================================================== batched complex FFT (plan API) */
struct C2CArgs {
    const float2* in;
    float2* out;
    int batch;
    int inverse;             /* 1: backward, scaled 1/M */
    const float* tables;
};

template <class C, int G>
__global__ void __launch_bounds__(C::T* G) fft_c2c_kernel(const C2CArgs a)
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
    const int groups = (a.batch + G - 1) / G;
    const float scale = a.inverse ? 1.0f / (float)M : 1.0f;
    for (int group = blockIdx.x; group < groups; group += gridDim.x) {
        const int id = group * G + team;
        const bool active = id < a.batch;
        float2 v[E];
        {
            constexpr int R = C::R1, NQ = E / R, STRIDE = M / R;
#pragma unroll
            for (int q = 0; q < NQ; ++q)
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    float2 s = make_float2(0.f, 0.f);
                    if (active) s = __ldg(a.in + (long long)id * M + t + T * q + r * STRIDE);
                    v[q * R + r] = a.inverse ? make_float2(s.y, s.x) : s;
                }
        }
        /* in == out is allowed (reference fft_kiss.c:112): every load of this transform is done
         * before its first store because team_fft contains team barriers */
        team_fft<C>(v, xb, s_tw2, s_tw3, t, team);
        if (active) {
#pragma unroll
            for (int q = 0; q < L::NQ; ++q)
#pragma unroll
                for (int r = 0; r < L::R; ++r) {
                    const float2 z = v[q * L::R + ct_bitrev(r, L::R)];
                    a.out[(long long)id * M + t + T * q + r * L::NS] =
                        a.inverse ? make_float2(z.y * scale, z.x * scale) : z;
                }
        }
        team_sync<T>(team);
    }
}

}  // namespace vvb
