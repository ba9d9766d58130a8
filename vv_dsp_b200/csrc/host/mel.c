/*
 * mel.c -- mel filterbank (host) and log-mel spectrogram (GPU) behind the reference's API
 * (include/vv_dsp/features/mel.h:12-66, src/features/mel.c:14-245), plus the batched
 * STFT -> log-mel entry point of include/vv_dsp/b200.h.  SURVEY.md section 8f, rank 2.
 *
 * The filterbank is built on the host with the reference's float32 formulas, so it is
 * bit-identical: HTK scale 2595 log10f(1 + hz/700), n_mels + 2 points equally spaced in mel
 * (start + step*i), lower-bound search of each edge in the bin frequencies k*sr/n_fft, rising
 * slope on [left, center), falling on [center, right), every filter divided by its sum.
 * The log-mel reduction runs on the GPU (csrc/cuda/vvb_direct_kernels.cuh: logmel_kernel).
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "vv_dsp/b200.h"
#include "vv_dsp/features/mel.h"
#include "vvb200_cuda.h"
#include "internal.h"

vv_dsp_real vv_dsp_hz_to_mel(vv_dsp_real hz) { return hz < 0.0f ? 0.0f : 2595.0f * log10f(1.0f + hz / 700.0f); }

vv_dsp_real vv_dsp_mel_to_hz(vv_dsp_real mel) { return mel < 0.0f ? 0.0f : 700.0f * (powf(10.0f, mel / 2595.0f) - 1.0f); }

static size_t first_not_below(const float* v, size_t n, float x)
{
    size_t a = 0, b = n;
    while (a < b) {
        const size_t mid = a + (b - a) / 2;
        if (v[mid] < x) a = mid + 1; else b = mid;
    }
    return a;
}

vv_dsp_status vv_dsp_mel_filterbank_create(size_t n_fft, size_t n_mels, vv_dsp_real sample_rate, vv_dsp_real fmin,
                                           vv_dsp_real fmax, vv_dsp_mel_variant variant, vv_dsp_real** out_filterbank_weights,
                                           size_t* out_num_filters, size_t* out_filter_len)
{
    size_t bins, npts, i, m, k;
    float *fb, *edges, *freqs, mel_lo, mel_hi, step;
    if (!out_filterbank_weights || !out_num_filters || !out_filter_len) return VV_DSP_ERROR_NULL_POINTER;
    if (n_fft == 0 || n_mels == 0 || sample_rate <= 0.0f || fmin < 0.0f || fmax <= fmin) return VV_DSP_ERROR_INVALID_SIZE;
    if (fmax > sample_rate / 2.0f) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (variant != VV_DSP_MEL_VARIANT_HTK) return VV_DSP_ERROR_OUT_OF_RANGE;
    bins = n_fft / 2 + 1;
    if (n_mels >= bins) return VV_DSP_ERROR_INVALID_SIZE;
    npts = n_mels + 2;
    fb = (float*)calloc(n_mels * bins, sizeof(float));
    edges = (float*)malloc(npts * sizeof(float));
    freqs = (float*)malloc(bins * sizeof(float));
    if (!fb || !edges || !freqs) { free(fb); free(edges); free(freqs); return VV_DSP_ERROR_INTERNAL; }
    mel_lo = vv_dsp_hz_to_mel(fmin);
    mel_hi = vv_dsp_hz_to_mel(fmax);
    step = (mel_hi - mel_lo) / (float)(npts - 1);
    for (i = 0; i < npts; ++i) edges[i] = vv_dsp_mel_to_hz(mel_lo + step * (float)i);
    for (k = 0; k < bins; ++k) freqs[k] = (float)k * sample_rate / (float)n_fft;
    for (m = 0; m < n_mels; ++m) {
        const float left = edges[m], center = edges[m + 1], right = edges[m + 2];
        const size_t il = first_not_below(freqs, bins, left), ic = first_not_below(freqs, bins, center),
                     ir = first_not_below(freqs, bins, right);
        float* w = fb + m * bins;
        float total = 0.0f;
        for (k = il; k < ic && k < bins; ++k) w[k] = (freqs[k] - left) / (center - left);
        for (k = ic; k < ir && k < bins; ++k) w[k] = (right - freqs[k]) / (right - center);
        for (k = 0; k < bins; ++k) total += w[k];
        if (total > 0.0f) for (k = 0; k < bins; ++k) w[k] /= total;
    }
    free(edges); free(freqs);
    *out_filterbank_weights = fb; *out_num_filters = n_mels; *out_filter_len = bins;
    return VV_DSP_OK;
}

void vv_dsp_mel_filterbank_free(vv_dsp_real* filterbank_weights, size_t n_mels)
{
    (void)n_mels;
    free(filterbank_weights);
}

/* dense [n_mels][bins] -> device-resident sparse form.
 *   meta : lo[n_mels] | len[n_mels] | off[n_mels]            one contiguous non-zero run per filter
 *          header[12]: slot_ptr start (x4), group start (x4), quad-weight offset, spare
 *          then, for each of the four tile shapes of the log-mel kernel (16, 32, 64, 128 band slots):
 *          slot_ptr[slots + 1] and the slot-ordered group list {first bin, quad index, taps | 8*last, band}
 *   w    : the packed runs | the same runs padded with zeros to groups of four taps (16-byte loads)
 * A group is four consecutive taps of one filter.  Filters are dealt to slots longest first, each to the
 * least loaded slot, so that every slot of the kernel walks about the same number of groups. */
void vvdsp_internal_mel_device_free(mel_device* md)
{
    vvb_free(md->d_meta); vvb_free(md->d_w); vvb_free(md->d_fw); vvb_free(md->d_fseg);
    md->d_meta = NULL; md->d_w = NULL; md->d_fw = NULL; md->d_fseg = NULL; md->f_segments = 0; md->f_prow = 0; md->f_unit = 0;
}

/* Lane schedules of the fused STFT -> log-mel kernel (csrc/cuda/vvb_stft_kernels.cuh, mel_phase).  The warp that has just
 * computed a frame's power row sums the bands with its 32 lanes.  A band's ordered float32 sum is one dependent chain, so a
 * band goes to ONE lane; to keep the 32 lanes in step without any divergence every lane walks the same S segments of
 * FUSED_U quads (a quad = four consecutive bins starting at a multiple of four) and a band occupies whole consecutive
 * segments of its lane, from the quad that contains its first non-zero weight on.  Weights are taken from the dense row, so
 * everything outside the band's support inside those segments is an exact zero that adds nothing -- like the zero weights
 * of the reference's full-row sum (src/features/mel.c:229-236).  Bands are dealt longest first, each to the fullest lane
 * that still has room (best fit decreasing), for the smallest S that works.
 *   d_fw   float4 [S * FUSED_U][32]   weights of lane l's quad at step i
 *   d_fseg int2   [S][32]             { float offset of the segment's first quad in the power row, (band + 1) << 1 | reset }
 *                                      reset: the accumulator starts from zero here; band + 1: emit the sum after this segment
 * Bank conflicts: a lane reads its quad with one LDS.128, which the hardware serves a quarter warp (8 lanes x 16 bytes) at
 * a time, conflict-free iff the eight quad indices differ mod 8.  Lanes advance in step, so what matters is the residue
 * of every segment's first quad.  A first placement gave 2.7 wavefronts where one suffices (ncu: +162 conflicts per frame,
 * the whole fused kernel bound by shared-memory wavefronts), so the schedules are then improved by a deterministic local
 * search over (a) which physical lane runs which schedule, (b) the order of the bands inside a schedule and (c) starting a
 * band up to `slack` quads early (zero weights) where its last segment has room: 260 -> 108 wavefronts per frame for the
 * 80-band / 1025-bin filterbank, against 96 without any conflict.  Idle segments read the least loaded residue.
 * Not built (the chained kernels serve the call) when the schedule would exceed FUSED_MAX_STEPS quad steps. */
#define FUSED_LANES 32
#define FUSED_MAX_STEPS 48
typedef struct fused_sched {
    size_t S, n_mels;
    int U;                      /* quads per segment: 4, or 2 where the bands are short (small bin counts) */
    const int *nseg, *q0;
    int* delta;                 /* quads a band starts early */
    int* list;                  /* [32][n_mels]: bands of schedule v in execution order */
    int count[FUSED_LANES];     /* bands per schedule */
    int perm[FUSED_LANES];      /* physical lane -> schedule */
} fused_sched;

/* residue (mod 8) of the first quad of every segment of schedule v, -1 = idle */
static void fused_residues(const fused_sched* fs, int v, int* res)
{
    size_t s = 0;
    int i, j;
    for (i = 0; i < fs->count[v]; ++i) {
        const int b = fs->list[(size_t)v * fs->n_mels + (size_t)i];
        for (j = 0; j < fs->nseg[b]; ++j) res[s++] = (fs->q0[b] - fs->delta[b] + j * fs->U) & 7;
    }
    while (s < fs->S) res[s++] = -1;
}

/* shared-memory wavefronts of the power-row loads per frame: per quarter warp and segment, U loads of max-multiplicity */
static long fused_cost(const fused_sched* fs, int* scratch)
{
    long total = 0;
    int quarter, i;
    size_t s;
    for (quarter = 0; quarter < FUSED_LANES / 8; ++quarter) {
        for (i = 0; i < 8; ++i) fused_residues(fs, fs->perm[quarter * 8 + i], scratch + (size_t)i * fs->S);
        for (s = 0; s < fs->S; ++s) {
            int cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0}, idle = 0, worst = 0, k;
            for (i = 0; i < 8; ++i) { const int r = scratch[(size_t)i * fs->S + s]; if (r < 0) ++idle; else ++cnt[r]; }
            while (idle-- > 0) { int least = 0; for (k = 1; k < 8; ++k) if (cnt[k] < cnt[least]) least = k; ++cnt[least]; }
            for (k = 0; k < 8; ++k) if (cnt[k] > worst) worst = cnt[k];
            total += (long)worst * fs->U;
        }
    }
    return total;
}

/* segments per lane the best-fit-decreasing placement needs with `unit` quads per segment (0: none within FUSED_MAX_STEPS) */
static size_t fused_min_segments(const int* lo, const int* len, size_t n_mels, int unit)
{
    int load[FUSED_LANES];
    size_t m, l, total = 0, S;
    int maxseg = 1;
    int* nseg = (int*)malloc(n_mels * sizeof(int));
    int* order = (int*)malloc(n_mels * sizeof(int));
    if (!nseg || !order) { free(nseg); free(order); return 0; }
    for (m = 0; m < n_mels; ++m) {
        const int first = len[m] > 0 ? lo[m] : 0, end = len[m] > 0 ? lo[m] + len[m] : 1;
        size_t q = m;
        nseg[m] = ((end + 3) / 4 - first / 4 + unit - 1) / unit;
        if (nseg[m] > maxseg) maxseg = nseg[m];
        total += (size_t)nseg[m];
        while (q > 0 && nseg[order[q - 1]] < nseg[m]) { order[q] = order[q - 1]; --q; }
        order[q] = (int)m;
    }
    S = (total + FUSED_LANES - 1) / FUSED_LANES;
    if (S < (size_t)maxseg) S = (size_t)maxseg;
    for (; S * (size_t)unit <= FUSED_MAX_STEPS; ++S) {
        int ok = 1;
        for (l = 0; l < FUSED_LANES; ++l) load[l] = 0;
        for (m = 0; m < n_mels && ok; ++m) {
            int best = -1;
            for (l = 0; l < FUSED_LANES; ++l)
                if (load[l] + nseg[order[m]] <= (int)S && (best < 0 || load[l] > load[best])) best = (int)l;
            if (best < 0) ok = 0; else load[best] += nseg[order[m]];
        }
        if (ok) break;
    }
    free(nseg); free(order);
    return S * (size_t)unit <= FUSED_MAX_STEPS ? S : 0;
}

/* Quads per segment.  The marching kernel (fft_size 2048) and the generic forward kernel with two frames per warp (fft_size 512,
 * 640, 1024) are written for four.  With four frames per warp (fft_size <= 480: at most 241 bins) the generic kernel takes two or
 * four: with short bands (five taps at fft_size 400 / 80 bands) a four-quad segment is mostly zero padding, so the choice goes by
 * the shared-memory wavefronts of a segment: ~6 of bookkeeping + 20 per quad (weights once, four power rows). */
static int fused_choose_unit(const int* lo, const int* len, size_t n_mels, size_t bins)
{
    size_t s2, s4;
    if (bins > 241 || getenv("VVB_MEL_UNIT4")) return 4;
    s2 = fused_min_segments(lo, len, n_mels, 2);
    s4 = fused_min_segments(lo, len, n_mels, 4);
    if (!s2) return 4;
    if (!s4) return 2;
    return s2 * (6 + 20 * 2) < s4 * (6 + 20 * 4) ? 2 : 4;
}

static int build_fused_tables(const float* weights, size_t n_mels, size_t bins, const int* lo, const int* len, int unit, void* stream, mel_device* md)
{
    int *nseg = NULL, *q0 = NULL, *nq = NULL, *order = NULL, *seg = NULL, *scratch = NULL;
    int load[FUSED_LANES];
    fused_sched fs;
    float* wq = NULL;
    size_t m, total = 0, S, l, prow_quads = (bins + 3) / 4;
    int st = 0, maxseg = 1, ok = 0, p;
    unsigned long long rng = 0x9E3779B97F4A7C15ull;
    long cost;
    const int FUSED_U = unit;
    md->d_fw = NULL; md->d_fseg = NULL; md->f_segments = 0; md->f_prow = 0; md->f_unit = 0;
    memset(&fs, 0, sizeof(fs));
    if (n_mels == 0 || n_mels > 1024 || bins == 0 || bins > (1u << 20)) return 0;
    nseg = (int*)malloc(n_mels * sizeof(int)); q0 = (int*)malloc(n_mels * sizeof(int)); nq = (int*)malloc(n_mels * sizeof(int));
    order = (int*)malloc(n_mels * sizeof(int));
    fs.delta = (int*)calloc(n_mels, sizeof(int)); fs.list = (int*)malloc(FUSED_LANES * n_mels * sizeof(int));
    if (!nseg || !q0 || !nq || !order || !fs.delta || !fs.list) { st = 4; goto done; }
    for (m = 0; m < n_mels; ++m) {
        const int first = len[m] > 0 ? lo[m] : 0, end = len[m] > 0 ? lo[m] + len[m] : 1;
        const int qa = first / 4, qb = (end + 3) / 4;
        q0[m] = qa; nq[m] = qb - qa;
        nseg[m] = (nq[m] + FUSED_U - 1) / FUSED_U;
        if (nseg[m] > maxseg) maxseg = nseg[m];
        total += (size_t)nseg[m];
        if ((size_t)(qa + nseg[m] * FUSED_U) > prow_quads) prow_quads = (size_t)(qa + nseg[m] * FUSED_U);
    }
    for (m = 0; m < n_mels; ++m) {                                     /* bands by descending segment count */
        size_t q = m;
        while (q > 0 && nseg[order[q - 1]] < nseg[m]) { order[q] = order[q - 1]; --q; }
        order[q] = (int)m;
    }
    S = (total + FUSED_LANES - 1) / FUSED_LANES;
    if (S < (size_t)maxseg) S = (size_t)maxseg;
    for (; S * FUSED_U <= FUSED_MAX_STEPS; ++S) {                      /* best fit decreasing for the smallest S that works */
        ok = 1;
        for (l = 0; l < FUSED_LANES; ++l) { load[l] = 0; fs.count[l] = 0; }
        for (m = 0; m < n_mels && ok; ++m) {
            const int b = order[m];
            int best = -1;
            for (l = 0; l < FUSED_LANES; ++l)
                if (load[l] + nseg[b] <= (int)S && (best < 0 || load[l] > load[best])) best = (int)l;
            if (best < 0) { ok = 0; break; }
            fs.list[(size_t)best * n_mels + (size_t)fs.count[best]++] = b;
            load[best] += nseg[b];
        }
        if (ok) break;
    }
    if (!ok) goto done;                                                /* no schedule short enough: not an error */
    fs.S = S; fs.n_mels = n_mels; fs.nseg = nseg; fs.q0 = q0; fs.U = unit;
    for (p = 0; p < FUSED_LANES; ++p) fs.perm[p] = p;
    scratch = (int*)malloc(8 * S * sizeof(int));
    if (!scratch) { st = 4; goto done; }
    cost = fused_cost(&fs, scratch);
    {   /* local search (deterministic): keep every move that does not make the loads slower */
        const long floor_cost = (long)(S * FUSED_U * (FUSED_LANES / 8));
        int it;
        for (it = 0; it < 30000 && cost > floor_cost; ++it) {
            unsigned r0, r1, r2;
            rng = rng * 6364136223846793005ull + 1442695040888963407ull; r0 = (unsigned)(rng >> 33);
            rng = rng * 6364136223846793005ull + 1442695040888963407ull; r1 = (unsigned)(rng >> 33);
            rng = rng * 6364136223846793005ull + 1442695040888963407ull; r2 = (unsigned)(rng >> 33);
            if (r0 % 10 < 5) {                                         /* swap the schedules of two lanes */
                const int a = (int)(r1 % FUSED_LANES), b = (int)(r2 % FUSED_LANES), t = fs.perm[a];
                long c2;
                if (a == b) continue;
                fs.perm[a] = fs.perm[b]; fs.perm[b] = t;
                c2 = fused_cost(&fs, scratch);
                if (c2 <= cost) cost = c2; else { fs.perm[b] = fs.perm[a]; fs.perm[a] = t; }
            } else if (r0 % 10 < 8) {                                  /* start a band early, inside the room of its last segment */
                const int b = (int)(r1 % n_mels), room = nseg[b] * FUSED_U - nq[b], slack = room < q0[b] ? room : q0[b];
                const int old = fs.delta[b];
                long c2;
                if (slack <= 0) continue;
                fs.delta[b] = (int)(r2 % (unsigned)(slack + 1));
                c2 = fused_cost(&fs, scratch);
                if (c2 <= cost) cost = c2; else fs.delta[b] = old;
            } else {                                                   /* exchange two bands inside one schedule */
                const int v = (int)(r1 % FUSED_LANES);
                if (fs.count[v] > 1) {
                    int* li = fs.list + (size_t)v * n_mels;
                    const int i = (int)(r2 % (unsigned)fs.count[v]), j = (int)((r2 >> 8) % (unsigned)fs.count[v]), t = li[i];
                    long c2;
                    if (i == j) continue;
                    li[i] = li[j]; li[j] = t;
                    c2 = fused_cost(&fs, scratch);
                    if (c2 <= cost) cost = c2; else { li[j] = li[i]; li[i] = t; }
                }
            }
        }
    }
    if (getenv("VVB_MEL_DEBUG"))
        fprintf(stderr, "vvb: fused log-mel schedule: %zu bands, %zu segments of %d quads per lane, %ld shared-memory wavefronts per frame for the power row (%zu without conflicts)\n",
                n_mels, S, FUSED_U, cost, S * FUSED_U * (FUSED_LANES / 8));
    wq = (float*)calloc(S * FUSED_U * FUSED_LANES * 4, sizeof(float));
    seg = (int*)calloc(S * FUSED_LANES * 2, sizeof(int));
    if (!wq || !seg) { st = 4; goto done; }
    for (p = 0; p < FUSED_LANES; p += 8) {                             /* a quarter warp at a time: idle segments take the least loaded residue */
        size_t s;
        int i;
        for (i = 0; i < 8; ++i) fused_residues(&fs, fs.perm[p + i], scratch + (size_t)i * S);
        for (s = 0; s < S; ++s) {
            int cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0}, k;
            for (i = 0; i < 8; ++i) if (scratch[(size_t)i * S + s] >= 0) ++cnt[scratch[(size_t)i * S + s]];
            for (i = 0; i < 8; ++i)
                if (scratch[(size_t)i * S + s] < 0) {
                    int least = 0;
                    for (k = 1; k < 8; ++k) if (cnt[k] < cnt[least]) least = k;
                    ++cnt[least];
                    seg[2 * (s * FUSED_LANES + (size_t)(p + i))] = 4 * least;          /* weights stay zero, nothing is emitted */
                }
        }
    }
    for (p = 0; p < FUSED_LANES; ++p) {
        const int v = fs.perm[p];
        int i, j, u, e, s = 0;
        for (i = 0; i < fs.count[v]; ++i) {
            const int b = fs.list[(size_t)v * n_mels + (size_t)i], first_quad = q0[b] - fs.delta[b];
            for (j = 0; j < nseg[b]; ++j, ++s) {
                int* d = seg + 2 * ((size_t)s * FUSED_LANES + (size_t)p);
                d[0] = 4 * (first_quad + j * FUSED_U);
                d[1] = (j == 0 ? 1 : 0) | (j + 1 == nseg[b] ? (b + 1) << 1 : 0);
                for (u = 0; u < FUSED_U; ++u)
                    for (e = 0; e < 4; ++e) {
                        const size_t k = (size_t)d[0] + 4 * (size_t)u + (size_t)e;
                        wq[4 * (((size_t)s * FUSED_U + (size_t)u) * FUSED_LANES + (size_t)p) + (size_t)e] = k < bins ? weights[(size_t)b * bins + k] : 0.0f;
                    }
            }
        }
    }
    st = vvb_malloc((void**)&md->d_fw, S * FUSED_U * FUSED_LANES * 4 * sizeof(float));
    if (!st) st = vvb_malloc((void**)&md->d_fseg, S * FUSED_LANES * 2 * sizeof(int));
    if (!st) st = vvb_memcpy_h2d(md->d_fw, wq, S * FUSED_U * FUSED_LANES * 4 * sizeof(float), stream);
    if (!st) st = vvb_memcpy_h2d(md->d_fseg, seg, S * FUSED_LANES * 2 * sizeof(int), stream);
    if (!st) st = vvb_stream_sync(stream);
    if (!st) { md->f_segments = S; md->f_prow = 4 * prow_quads; md->f_unit = (size_t)unit; }
    else { vvb_free(md->d_fw); vvb_free(md->d_fseg); md->d_fw = NULL; md->d_fseg = NULL; }
done:
    free(nseg); free(q0); free(nq); free(order); free(fs.delta); free(fs.list); free(scratch); free(wq); free(seg);
    return st;
}

int vvdsp_internal_mel_device_build(const float* weights, size_t n_mels, size_t bins, void* stream, mel_device* md)
{
    const size_t hdr = 3 * n_mels;
    size_t m, k, total = 0, groups = 0, meta_len, w_len, quad0, v, pos;
    int *meta = NULL, *order = NULL, *gcount = NULL, *gfirst = NULL, *load = NULL, *owner = NULL;
    float* packed = NULL;
    int st = 4;
    md->d_meta = NULL; md->d_w = NULL; md->n_groups = 0;
    md->d_fw = NULL; md->d_fseg = NULL; md->f_segments = 0; md->f_prow = 0; md->f_unit = 0;
    gcount = (int*)malloc(n_mels * sizeof(int)); gfirst = (int*)malloc(n_mels * sizeof(int));
    order = (int*)malloc(n_mels * sizeof(int)); owner = (int*)malloc(n_mels * sizeof(int));
    load = (int*)malloc(128 * sizeof(int));
    packed = (float*)malloc((2 * n_mels * bins + 8 * n_mels + 8) * sizeof(float));
    if (!gcount || !gfirst || !order || !owner || !load || !packed) goto done;
    /* first pass: runs and group counts, to size the tables */
    for (m = 0; m < n_mels; ++m) {
        const float* w = weights + m * bins;
        size_t lo = bins, hi = 0;
        for (k = 0; k < bins; ++k) if (w[k] != 0.0f) { if (lo == bins) lo = k; hi = k + 1; }
        if (lo == bins) { lo = 0; hi = 0; }
        gcount[m] = (int)((hi - lo + 3) / 4);
        if (gcount[m] == 0) gcount[m] = 1;              /* an all-zero filter still has to emit log(eps) */
        gfirst[m] = (int)groups;
        groups += (size_t)gcount[m];
        total += hi - lo;
    }
    meta_len = hdr + 12;
    for (v = 0; v < 4; ++v) meta_len += ((size_t)(16u << v) + 1 + 3) / 4 * 4 + 4 * groups;
    meta_len = (meta_len + 3) / 4 * 4 + 4;
    meta = (int*)calloc(meta_len, sizeof(int));
    if (!meta) goto done;
    quad0 = (total + 3) / 4 * 4;
    w_len = quad0 + 4 * groups;
    memset(packed, 0, (w_len ? w_len : 1) * sizeof(float));
    total = 0;
    for (m = 0; m < n_mels; ++m) {
        const float* w = weights + m * bins;
        size_t lo = bins, hi = 0;
        for (k = 0; k < bins; ++k) if (w[k] != 0.0f) { if (lo == bins) lo = k; hi = k + 1; }
        if (lo == bins) { lo = 0; hi = 0; }
        meta[m] = (int)lo; meta[n_mels + m] = (int)(hi - lo); meta[2 * n_mels + m] = (int)total;
        memcpy(packed + total, w + lo, (hi - lo) * sizeof(float));
        memcpy(packed + quad0 + 4 * (size_t)gfirst[m], w + lo, (hi - lo) * sizeof(float));
        total += hi - lo;
    }
    /* filters by descending group count (insertion sort: n_mels is small) */
    for (m = 0; m < n_mels; ++m) {
        size_t q = m;
        while (q > 0 && gcount[order[q - 1]] < gcount[m]) { order[q] = order[q - 1]; --q; }
        order[q] = (int)m;
    }
    meta[hdr + 8] = (int)quad0;
    pos = (hdr + 12 + 3) / 4 * 4;
    for (v = 0; v < 4; ++v) {
        const size_t slots = (size_t)16u << v;
        size_t s, q, g, at;
        int* slot_ptr = meta + pos;
        int* desc;
        meta[hdr + v] = (int)pos;
        pos += (slots + 1 + 3) / 4 * 4;
        meta[hdr + 4 + v] = (int)pos;
        desc = meta + pos;
        pos += 4 * groups;
        for (s = 0; s < slots; ++s) load[s] = 0;
        for (q = 0; q < n_mels; ++q) {
            size_t best = 0;
            for (s = 1; s < slots; ++s) if (load[s] < load[best]) best = s;
            owner[order[q]] = (int)best;
            load[best] += gcount[order[q]];
        }
        at = 0;
        for (s = 0; s < slots; ++s) {
            slot_ptr[s] = (int)at;
            for (m = 0; m < n_mels; ++m) {
                if (owner[m] != (int)s) continue;
                for (g = 0; g < (size_t)gcount[m]; ++g) {
                    const int len = meta[n_mels + m], left = len - (int)(4 * g);
                    const int taps = left > 4 ? 4 : (left > 0 ? left : 0);
                    int* d = desc + 4 * at++;
                    d[0] = meta[m] + (int)(4 * g);
                    d[1] = gfirst[m] + (int)g;
                    d[2] = taps | ((g + 1 == (size_t)gcount[m]) ? 8 : 0);
                    d[3] = (int)m;
                }
            }
        }
        slot_ptr[slots] = (int)at;
    }
    st = vvb_malloc((void**)&md->d_meta, meta_len * sizeof(int));
    if (!st) st = vvb_malloc((void**)&md->d_w, (w_len ? w_len : 1) * sizeof(float));
    if (!st) st = vvb_memcpy_h2d(md->d_meta, meta, meta_len * sizeof(int), stream);
    if (!st && w_len) st = vvb_memcpy_h2d(md->d_w, packed, w_len * sizeof(float), stream);
    if (!st) st = vvb_stream_sync(stream);          /* the host staging arrays die below */
    if (!st) md->n_groups = groups;
    if (!st) st = build_fused_tables(weights, n_mels, bins, meta, meta + n_mels, fused_choose_unit(meta, meta + n_mels, n_mels, bins), stream, md);
done:
    free(meta); free(packed); free(order); free(gcount); free(gfirst); free(load); free(owner);
    if (st) vvdsp_internal_mel_device_free(md);
    return st;
}

int vvdsp_internal_logmel(const mel_device* md, const float* d_power, size_t frames, size_t bins, size_t n_mels, float eps,
                          float* d_out, void* stream)
{
    return vvb_logmel(d_power, frames, bins, bins, md->d_meta, md->d_w, n_mels, md->n_groups, eps, d_out, stream);
}

vv_dsp_status vv_dsp_compute_log_mel_spectrogram(const vv_dsp_real* power_spectrogram, size_t num_frames, size_t n_fft_bins,
                                                 const vv_dsp_real* filterbank_weights, size_t n_mels, vv_dsp_real log_epsilon,
                                                 vv_dsp_real* out_log_mel_spectrogram)
{
    mel_device md;
    float *d_p = NULL, *d_o = NULL;
    void* stream = NULL;
    int st;
    if (!power_spectrogram || !filterbank_weights || !out_log_mel_spectrogram) return VV_DSP_ERROR_NULL_POINTER;
    if (num_frames == 0 || n_fft_bins == 0 || n_mels == 0) return VV_DSP_ERROR_INVALID_SIZE;
    if (log_epsilon < 0.0f) return VV_DSP_ERROR_OUT_OF_RANGE;
    memset(&md, 0, sizeof(md));
    st = vvb_device_ready();                         /* no CUDA device -> UNSUPPORTED, never a CPU computation */
    if (st) return vvdsp_internal_status(st);
    st = vvb_stream_create(&stream);
    if (!st) st = vvdsp_internal_mel_device_build(filterbank_weights, n_mels, n_fft_bins, stream, &md);
    if (!st) st = vvb_malloc((void**)&d_p, num_frames * n_fft_bins * sizeof(float));
    if (!st) st = vvb_malloc((void**)&d_o, num_frames * n_mels * sizeof(float));
    if (!st) st = vvb_memcpy_h2d(d_p, power_spectrogram, num_frames * n_fft_bins * sizeof(float), stream);
    if (!st) st = vvdsp_internal_logmel(&md, d_p, num_frames, n_fft_bins, n_mels, log_epsilon, d_o, stream);
    if (!st) st = vvb_memcpy_d2h(out_log_mel_spectrogram, d_o, num_frames * n_mels * sizeof(float), stream);
    if (stream) { int s2 = vvb_stream_sync(stream); if (!st) st = s2; }
    vvb_free(d_p); vvb_free(d_o); vvdsp_internal_mel_device_free(&md);
    if (stream) vvb_stream_destroy(stream);
    return vvdsp_internal_status(st);
}

/* ------------------------------------------------------------------ MFCC (src/features/mel.c:249-461) */
void vvdsp_internal_mfcc_device_free(mfcc_device* md) { vvb_free(md->d_table); vvb_free(md->d_lifter); md->d_table = NULL; md->d_lifter = NULL; }

/* cos(pi (n + 1/2) k / N) and the lifter factors, evaluated in float32 exactly as the reference evaluates
 * them per term (src/spectral/dct.c:25, mel.c:292) */
int vvdsp_internal_mfcc_device_build(size_t n_mels, size_t n_coeffs, float lifter, void* stream, mfcc_device* md)
{
    const float pi = (float)3.141592653589793238462643383279502884;
    float* tab = (float*)malloc(n_coeffs * n_mels * sizeof(float));
    float* lif = (float*)malloc(n_coeffs * sizeof(float));
    size_t k, n;
    int st = 4;
    md->d_table = NULL; md->d_lifter = NULL; md->n_mels = n_mels; md->n_coeffs = n_coeffs; md->lifter = lifter;
    if (tab && lif) {
        for (k = 0; k < n_coeffs; ++k) {
            for (n = 0; n < n_mels; ++n) {
                const float ang = pi * ((float)n + 0.5f) * (float)k / (float)n_mels;
                tab[k * n_mels + n] = cosf(ang);
            }
            lif[k] = 1.0f;
            if (lifter > 0.0f && k >= 1) lif[k] = 1.0f + (lifter / 2.0f) * sinf((float)3.14159265358979323846 * (float)k / lifter);
        }
        st = vvb_malloc((void**)&md->d_table, n_coeffs * n_mels * sizeof(float));
        if (!st) st = vvb_malloc((void**)&md->d_lifter, n_coeffs * sizeof(float));
        if (!st) st = vvb_memcpy_h2d(md->d_table, tab, n_coeffs * n_mels * sizeof(float), stream);
        if (!st) st = vvb_memcpy_h2d(md->d_lifter, lif, n_coeffs * sizeof(float), stream);
        if (!st) st = vvb_stream_sync(stream);
    }
    free(tab); free(lif);
    if (st) vvdsp_internal_mfcc_device_free(md);
    return st;
}

static vv_dsp_status mfcc_validate(size_t num_frames, size_t n_mels, size_t n_coeffs, vv_dsp_dct_type dct_type, vv_dsp_real lifter)
{
    if (num_frames == 0 || n_mels == 0 || n_coeffs == 0) return VV_DSP_ERROR_INVALID_SIZE;
    if (n_coeffs > n_mels) return VV_DSP_ERROR_INVALID_SIZE;
    if (dct_type != VV_DSP_DCT_II) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (lifter < 0.0f) return VV_DSP_ERROR_OUT_OF_RANGE;
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_mfcc(const vv_dsp_real* log_mel_spectrogram, size_t num_frames, size_t n_mels, size_t num_mfcc_coeffs,
                          vv_dsp_dct_type dct_type, vv_dsp_real lifter_coeff, vv_dsp_real* out_mfcc_coeffs)
{
    mfcc_device md;
    float *d_in = NULL, *d_out = NULL;
    void* stream = NULL;
    vv_dsp_status v;
    int st;
    if (!log_mel_spectrogram || !out_mfcc_coeffs) return VV_DSP_ERROR_NULL_POINTER;
    v = mfcc_validate(num_frames, n_mels, num_mfcc_coeffs, dct_type, lifter_coeff);
    if (v != VV_DSP_OK) return v;
    md.d_table = NULL; md.d_lifter = NULL;
    st = vvb_device_ready();
    if (st) return vvdsp_internal_status(st);
    st = vvb_stream_create(&stream);
    if (!st) st = vvdsp_internal_mfcc_device_build(n_mels, num_mfcc_coeffs, lifter_coeff, stream, &md);
    if (!st) st = vvb_malloc((void**)&d_in, num_frames * n_mels * sizeof(float));
    if (!st) st = vvb_malloc((void**)&d_out, num_frames * num_mfcc_coeffs * sizeof(float));
    if (!st) st = vvb_memcpy_h2d(d_in, log_mel_spectrogram, num_frames * n_mels * sizeof(float), stream);
    if (!st) st = vvb_mfcc(d_in, num_frames, n_mels, num_mfcc_coeffs, md.d_table, md.d_lifter, d_out, stream);
    if (!st) st = vvb_memcpy_d2h(out_mfcc_coeffs, d_out, num_frames * num_mfcc_coeffs * sizeof(float), stream);
    if (stream) { int s2 = vvb_stream_sync(stream); if (!st) st = s2; }
    vvb_free(d_in); vvb_free(d_out); vvdsp_internal_mfcc_device_free(&md);
    if (stream) vvb_stream_destroy(stream);
    return vvdsp_internal_status(st);
}

struct vv_dsp_mfcc_plan {
    size_t n_fft, n_mels, n_coeffs, bins;
    vv_dsp_dct_type dct_type;
    vv_dsp_real lifter, log_epsilon;
    vv_dsp_real* weights;            /* host filterbank, as the reference keeps it */
    mel_device mel; mfcc_device mfcc; int on_device;
    void* stream;
};

vv_dsp_status vv_dsp_mfcc_init(size_t n_fft, size_t n_mels, size_t num_mfcc_coeffs, vv_dsp_real sample_rate, vv_dsp_real fmin,
                               vv_dsp_real fmax, vv_dsp_mel_variant variant, vv_dsp_dct_type dct_type, vv_dsp_real lifter_coeff,
                               vv_dsp_real log_epsilon, vv_dsp_mfcc_plan** out_plan)
{
    vv_dsp_mfcc_plan* p;
    size_t nf = 0, fl = 0;
    vv_dsp_status v;
    if (!out_plan) return VV_DSP_ERROR_NULL_POINTER;
    if (n_fft == 0 || n_mels == 0 || num_mfcc_coeffs == 0 || sample_rate <= 0.0f) return VV_DSP_ERROR_INVALID_SIZE;
    if (num_mfcc_coeffs > n_mels || fmin < 0.0f || fmax <= fmin || fmax > sample_rate / 2.0f) return VV_DSP_ERROR_OUT_OF_RANGE;
    p = (vv_dsp_mfcc_plan*)calloc(1, sizeof(*p));
    if (!p) return VV_DSP_ERROR_INTERNAL;
    p->n_fft = n_fft; p->n_mels = n_mels; p->n_coeffs = num_mfcc_coeffs; p->bins = n_fft / 2 + 1;
    p->dct_type = dct_type; p->lifter = lifter_coeff; p->log_epsilon = log_epsilon;
    v = vv_dsp_mel_filterbank_create(n_fft, n_mels, sample_rate, fmin, fmax, variant, &p->weights, &nf, &fl);
    if (v != VV_DSP_OK) { free(p); return v; }
    *out_plan = p;                   /* device tables are built on first use, so init works like the reference's */
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_mfcc_process(const vv_dsp_mfcc_plan* plan, const vv_dsp_real* power_spectrogram, size_t num_frames,
                                  vv_dsp_real* out_mfcc_coeffs)
{
    vv_dsp_mfcc_plan* p = (vv_dsp_mfcc_plan*)plan;    /* the device tables are a cache, not logical state */
    float *d_p = NULL, *d_lm = NULL, *d_o = NULL;
    vv_dsp_status v;
    int st;
    if (!plan || !power_spectrogram || !out_mfcc_coeffs) return VV_DSP_ERROR_NULL_POINTER;
    if (num_frames == 0) return VV_DSP_ERROR_INVALID_SIZE;
    if (p->log_epsilon < 0.0f) return VV_DSP_ERROR_OUT_OF_RANGE;         /* compute_log_mel's check comes first */
    v = mfcc_validate(num_frames, p->n_mels, p->n_coeffs, p->dct_type, p->lifter);
    if (v != VV_DSP_OK) return v;
    st = vvb_device_ready();
    if (st) return vvdsp_internal_status(st);
    if (!p->on_device) {
        st = vvb_stream_create(&p->stream);
        if (!st) st = vvdsp_internal_mel_device_build(p->weights, p->n_mels, p->bins, p->stream, &p->mel);
        if (!st) st = vvdsp_internal_mfcc_device_build(p->n_mels, p->n_coeffs, p->lifter, p->stream, &p->mfcc);
        if (st) {
            vvdsp_internal_mel_device_free(&p->mel); vvdsp_internal_mfcc_device_free(&p->mfcc);
            if (p->stream) { vvb_stream_destroy(p->stream); p->stream = NULL; }
            return vvdsp_internal_status(st);
        }
        p->on_device = 1;
    }
    st = vvb_malloc((void**)&d_p, num_frames * p->bins * sizeof(float));
    if (!st) st = vvb_malloc((void**)&d_lm, num_frames * p->n_mels * sizeof(float));
    if (!st) st = vvb_malloc((void**)&d_o, num_frames * p->n_coeffs * sizeof(float));
    if (!st) st = vvb_memcpy_h2d(d_p, power_spectrogram, num_frames * p->bins * sizeof(float), p->stream);
    if (!st) st = vvdsp_internal_logmel(&p->mel, d_p, num_frames, p->bins, p->n_mels,
                             p->log_epsilon, d_lm, p->stream);
    if (!st) st = vvb_mfcc(d_lm, num_frames, p->n_mels, p->n_coeffs, p->mfcc.d_table, p->mfcc.d_lifter, d_o, p->stream);
    if (!st) st = vvb_memcpy_d2h(out_mfcc_coeffs, d_o, num_frames * p->n_coeffs * sizeof(float), p->stream);
    { int s2 = vvb_stream_sync(p->stream); if (!st) st = s2; }
    vvb_free(d_p); vvb_free(d_lm); vvb_free(d_o);
    return vvdsp_internal_status(st);
}

vv_dsp_status vv_dsp_mfcc_destroy(vv_dsp_mfcc_plan* plan)
{
    if (!plan) return VV_DSP_ERROR_NULL_POINTER;
    if (plan->on_device) { vvdsp_internal_mel_device_free(&plan->mel); vvdsp_internal_mfcc_device_free(&plan->mfcc); }
    if (plan->stream) vvb_stream_destroy(plan->stream);
    vv_dsp_mel_filterbank_free(plan->weights, plan->n_mels);
    free(plan);
    return VV_DSP_OK;
}
