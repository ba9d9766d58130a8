/*
 * fir.c -- batched FIR filtering by FFT convolution (overlap-save) on the device: vv_dsp_fir_* of include/vv_dsp/b200.h
 * (host, C99).  This file picks the transform size and the filter partitions, builds the filter spectra per call and
 * stages HOST buffers in chunks; the arithmetic is fir_ols_kernel (csrc/cuda/vvb_fir_kernels.cuh).
 */
#include <stdlib.h>
#include "vv_dsp/b200.h"
#include "vvb200_cuda.h"
#include "internal.h"

/* bound of the handle's filter-spectra scratch: per-signal filters beyond it are processed in chunks of signals */
#define FIR_SPEC_TARGET_BYTES ((size_t)128 << 20)
#define FIR_MIN_FFT 128
#define FIR_MAX_FFT 8192
#define FIR_MAX_TAPS ((size_t)0x7fffffff)    /* keeps the plan search short and every product of the cost model in range */

struct vv_dsp_fir {
    size_t taps, fft_size, parts, lp;
    handle_core core;
    vvb_fir_engine* eng;
    float* d_h;     size_t h_bytes;   /* filters staged from HOST */
    vvb_cpx* d_spec; size_t spec_bytes;
    float* d_x;     size_t x_bytes;   /* signals staged from HOST */
    float* d_y;     size_t y_bytes;   /* output staged for HOST */
};

/* The plan rule (documented in b200.h): over transform sizes N = 128 ... 8192 and partition counts P with
 * Lp = ceil(M / P) <= N, the smallest P N log2(N) / (N - Lp + 1); ties to the smaller N, then the fewer passes.
 * P beyond 4 ceil(M / N) never wins (at P = 2 ceil(M / N) a block already holds N / 2 samples), so the search stops there.
 * Costs are compared exactly, as cross products of integers. */
static void fir_plan(size_t m, size_t* fft_size, size_t* parts)
{
    unsigned long long best_num = 0, best_den = 0;
    size_t n, p;
    int lg;
    *fft_size = 0; *parts = 0;
    for (n = FIR_MIN_FFT, lg = 7; n <= FIR_MAX_FFT; n *= 2, ++lg) {
        const size_t p0 = (m + n - 1) / n;
        for (p = p0; p <= 4 * p0 && p <= m; ++p) {
            const size_t lp = (m + p - 1) / p;
            const unsigned long long num = (unsigned long long)p * n * (unsigned long long)lg, den = n - lp + 1;
            if (lp > n) continue;
            if (*parts == 0 || num * best_den < best_num * den) {
                best_num = num; best_den = den; *fft_size = n; *parts = p;
            }
        }
    }
}

static void fir_free(vv_dsp_fir* f)
{
    if (!f) return;
    vvb_free(f->d_h); vvb_free(f->d_spec); vvb_free(f->d_x); vvb_free(f->d_y);
    vvb_fir_engine_destroy(f->eng);
    vvdsp_internal_core_free(&f->core);
    free(f);
}

vv_dsp_status vv_dsp_fir_create(size_t num_taps, vv_dsp_fir** out)
{
    vv_dsp_fir* f;
    int st;
    if (!out) return VV_DSP_ERROR_NULL_POINTER;
    *out = NULL;
    if (num_taps == 0 || num_taps > FIR_MAX_TAPS) return VV_DSP_ERROR_INVALID_SIZE;
    f = (vv_dsp_fir*)calloc(1, sizeof(*f));
    if (!f) return VV_DSP_ERROR_INTERNAL;
    f->taps = num_taps;
    fir_plan(num_taps, &f->fft_size, &f->parts);
    f->lp = (num_taps + f->parts - 1) / f->parts;
    st = vvdsp_internal_core_init(&f->core);
    if (!st) st = vvb_fir_engine_create(f->fft_size, &f->eng);
    if (st) { fir_free(f); return st == 6 ? VV_DSP_ERROR_UNSUPPORTED : VV_DSP_ERROR_INTERNAL; }
    *out = f;
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_fir_destroy(vv_dsp_fir* f)
{
    int prev;
    if (!f) return VV_DSP_ERROR_NULL_POINTER;
    prev = vvdsp_internal_enter(&f->core);
    fir_free(f);
    vvdsp_internal_leave(prev);
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_fir_set_stream(vv_dsp_fir* f, void* cuda_stream)
{
    return vvdsp_internal_set_stream(f ? &f->core : NULL, cuda_stream);
}

vv_dsp_status vv_dsp_fir_synchronize(vv_dsp_fir* f)
{
    return vvdsp_internal_synchronize(f ? &f->core : NULL);
}

vv_dsp_status vv_dsp_fir_get_config(const vv_dsp_fir* f, size_t* fft_size, size_t* partitions)
{
    if (!f || !fft_size || !partitions) return VV_DSP_ERROR_NULL_POINTER;
    *fft_size = f->fft_size;
    *partitions = f->parts;
    return VV_DSP_OK;
}

/* filter spectra of `count` filters (rows of `filters` at `pitch`) into d_spec */
static int make_spectra(vv_dsp_fir* f, const vv_dsp_real* filters, vv_dsp_mem_space space, size_t count, size_t pitch)
{
    int st = 0;
    if (space == VV_DSP_MEM_HOST) {
        st = vvb_memcpy2d_h2d(f->d_h, f->taps * sizeof(float), filters, pitch * sizeof(float), f->taps * sizeof(float), count,
                              f->core.stream);
        filters = f->d_h; pitch = f->taps;
    }
    if (!st) st = vvb_fir_spectra(f->eng, filters, count, pitch, f->taps, f->lp, f->parts, f->d_spec, f->core.stream);
    return st;
}

static int filter_impl(vv_dsp_fir* f, const vv_dsp_real* filters, vv_dsp_mem_space filters_space, size_t num_filters,
                       size_t filter_pitch, const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch, size_t n,
                       size_t signal_pitch, vv_dsp_real* out, vv_dsp_mem_space out_space, size_t n_out, size_t out_pitch)
{
    const int shared = num_filters == 1;
    const size_t spec_per = f->parts * f->fft_size * sizeof(vvb_cpx);      /* one filter's spectra */
    const size_t x_per = signals_space == VV_DSP_MEM_HOST ? n * sizeof(float) : 0;
    const size_t y_per = out_space == VV_DSP_MEM_HOST ? n_out * sizeof(float) : 0;
    const size_t h_per = (!shared && filters_space == VV_DSP_MEM_HOST) ? f->taps * sizeof(float) : 0;
    const size_t stage_per = (x_per > y_per ? x_per : y_per) + h_per;
    const int any_host = signals_space == VV_DSP_MEM_HOST || out_space == VV_DSP_MEM_HOST || filters_space == VV_DSP_MEM_HOST;
    size_t cs = vvdsp_internal_chunk_rows(&f->core, batch, stage_per), done;
    int st = 0;
    if (!shared && FIR_SPEC_TARGET_BYTES / spec_per < cs) cs = FIR_SPEC_TARGET_BYTES / spec_per;
    if (cs < 1) cs = 1;
    st = vvdsp_internal_reserve(&f->core, (void**)&f->d_spec, &f->spec_bytes, (shared ? 1 : cs) * spec_per);
    if (!st && filters_space == VV_DSP_MEM_HOST)
        st = vvdsp_internal_reserve(&f->core, (void**)&f->d_h, &f->h_bytes, (shared ? 1 : cs) * f->taps * sizeof(float));
    if (!st && x_per) st = vvdsp_internal_reserve(&f->core, (void**)&f->d_x, &f->x_bytes, cs * x_per);
    if (!st && signals_space == VV_DSP_MEM_HOST && !f->d_x)                                               /* n == 0 */
        st = vvdsp_internal_reserve(&f->core, (void**)&f->d_x, &f->x_bytes, sizeof(float));
    if (!st && y_per) st = vvdsp_internal_reserve(&f->core, (void**)&f->d_y, &f->y_bytes, cs * y_per);
    if (!st && shared) st = make_spectra(f, filters, filters_space, 1, filter_pitch);
    /* every chunk runs on the handle's stream, so stream order keeps the scratch buffers of consecutive chunks apart */
    for (done = 0; done < batch && !st; done += cs) {
        const size_t nb = batch - done < cs ? batch - done : cs;
        const float* d_x = signals + done * signal_pitch;
        float* d_y = out + done * out_pitch;
        size_t xp = signal_pitch, yp = out_pitch;
        if (!shared) st = make_spectra(f, filters + done * filter_pitch, filters_space, nb, filter_pitch);
        if (!st && signals_space == VV_DSP_MEM_HOST) {
            if (n)
                st = vvb_memcpy2d_h2d(f->d_x, n * sizeof(float), d_x, signal_pitch * sizeof(float), n * sizeof(float), nb,
                                      f->core.stream);
            d_x = f->d_x; xp = n;
        }
        if (out_space == VV_DSP_MEM_HOST) { d_y = f->d_y; yp = n_out; }
        if (!st) st = vvb_fir_filter(f->eng, f->d_spec, shared ? 0 : f->parts * f->fft_size, f->taps, f->lp, f->parts, d_x, nb, n, xp,
                                     d_y, n_out, yp, f->core.stream);
        if (!st && out_space == VV_DSP_MEM_HOST)
            st = vvb_memcpy2d_d2h(out + done * out_pitch, out_pitch * sizeof(float), f->d_y, n_out * sizeof(float), n_out * sizeof(float),
                                  nb, f->core.stream);
    }
    return vvdsp_internal_finish(&f->core, st, any_host);
}

vv_dsp_status vv_dsp_fir_filter_batch(vv_dsp_fir* f, const vv_dsp_real* filters, vv_dsp_mem_space filters_space, size_t num_filters,
                                      size_t filter_pitch, const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch,
                                      size_t n, size_t signal_pitch, vv_dsp_real* out, vv_dsp_mem_space out_space, size_t n_out,
                                      size_t out_pitch)
{
    int prev, st;
    if (!f || !filters || !signals || !out) return VV_DSP_ERROR_NULL_POINTER;
    if ((unsigned)filters_space > 1u || (unsigned)signals_space > 1u || (unsigned)out_space > 1u) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (filter_pitch == 0) filter_pitch = f->taps;
    if (signal_pitch == 0) signal_pitch = n;
    if (out_pitch == 0) out_pitch = n_out;
    if ((num_filters != 1 && num_filters != batch) || filter_pitch < f->taps || signal_pitch < n || out_pitch < n_out)
        return VV_DSP_ERROR_INVALID_SIZE;
    if ((const void*)out == (const void*)signals) return VV_DSP_ERROR_UNSUPPORTED;      /* no in-place filtering */
    if (batch == 0 || n_out == 0) return VV_DSP_OK;
    prev = vvdsp_internal_enter(&f->core);
    st = filter_impl(f, filters, filters_space, num_filters, filter_pitch, signals, signals_space, batch, n, signal_pitch, out, out_space,
                     n_out, out_pitch);
    vvdsp_internal_leave(prev);
    return vvdsp_internal_status(st);
}
