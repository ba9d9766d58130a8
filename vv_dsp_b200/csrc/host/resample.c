/*
 * resample.c -- batched rational-ratio resampling by a polyphase FIR on the device: vv_dsp_resample_poly_* of
 * include/vv_dsp/b200.h (host, C99).  This file reduces the ratio, designs the default filter in double, builds the
 * polyphase bank once per handle and stages HOST buffers in chunks of rows; the arithmetic is resample_poly_kernel
 * (csrc/cuda/vvb_resample_kernels.cuh).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "vv_dsp/b200.h"
#include "vvb200_cuda.h"
#include "internal.h"

#define RS_MAX_BANK ((size_t)65536)             /* up T: the default design of every pair of standard rates fits */
#define RS_MAX_RATIO ((size_t)0x7fffffff)       /* up and down after reduction: keeps the kernel's index products in range */
#define RS_MAX_UPSAMPLED ((size_t)1 << 62)      /* n up */

struct vv_dsp_resample_poly {
    size_t up, down, taps, per_phase, half;
    handle_core core;
    float* d_bank;                    /* [per_phase][up], NULL for the identity ratio */
    float* d_x;     size_t x_bytes;   /* signals staged from HOST */
    float* d_y;     size_t y_bytes;   /* output staged for HOST */
};

static size_t gcd(size_t a, size_t b)
{
    while (b) { const size_t t = a % b; a = b; b = t; }
    return a;
}

/* modified Bessel function of the first kind, order 0, by its power series */
static double bessel_i0(double x)
{
    double sum = 1.0, term = 1.0;
    int k;
    for (k = 1; k < 500; ++k) {
        const double f = x / (2.0 * k);
        term *= f * f;
        sum += term;
        if (term < sum * 1e-17) break;
    }
    return sum;
}

/* scipy.signal.firwin(2 half + 1, 1 / max_rate, window=('kaiser', 5.0)): the windowed sinc normalised to unit DC gain */
static void design_default(size_t half, size_t max_rate, double* h)
{
    const size_t k_taps = 2 * half + 1;
    const double fc = 1.0 / (double)max_rate, beta = 5.0, i0b = bessel_i0(beta);
    const double pi = 3.14159265358979323846;
    double sum = 0.0;
    size_t k;
    for (k = 0; k < k_taps; ++k) {
        const double m = (double)k - (double)half;
        const double xm = fc * m;
        const double sinc = m == 0.0 ? 1.0 : sin(pi * xm) / (pi * xm);
        const double ratio = half ? m / (double)half : 0.0;
        const double win = bessel_i0(beta * sqrt(fmax(0.0, 1.0 - ratio * ratio))) / i0b;
        h[k] = fc * sinc * win;
        sum += h[k];
    }
    for (k = 0; k < k_taps; ++k) h[k] /= sum;
}

static void rs_free(vv_dsp_resample_poly* r)
{
    if (!r) return;
    vvb_free(r->d_bank); vvb_free(r->d_x); vvb_free(r->d_y);
    vvdsp_internal_core_free(&r->core);
    free(r);
}

vv_dsp_status vv_dsp_resample_poly_create(size_t up, size_t down, const vv_dsp_real* taps, size_t num_taps,
                                          vv_dsp_resample_poly** out)
{
    vv_dsp_resample_poly* r;
    int st;
    size_t g;
    if (!out) return VV_DSP_ERROR_NULL_POINTER;
    *out = NULL;
    if (!taps && num_taps > 0) return VV_DSP_ERROR_NULL_POINTER;
    if (up == 0 || down == 0 || (taps && num_taps == 0)) return VV_DSP_ERROR_INVALID_SIZE;
    g = gcd(up, down);
    up /= g; down /= g;
    if (up > RS_MAX_RATIO || down > RS_MAX_RATIO) return VV_DSP_ERROR_INVALID_SIZE;
    r = (vv_dsp_resample_poly*)calloc(1, sizeof(*r));
    if (!r) return VV_DSP_ERROR_INTERNAL;
    r->up = up; r->down = down;
    r->taps = taps ? num_taps : 20 * (up > down ? up : down) + 1;
    r->half = (r->taps - 1) / 2;
    r->per_phase = (r->taps + up - 1) / up;
    if (!(up == 1 && down == 1) && (r->per_phase > RS_MAX_BANK / up)) { free(r); return VV_DSP_ERROR_INVALID_SIZE; }
    st = vvdsp_internal_core_init(&r->core);
    if (!st && !(up == 1 && down == 1)) {        /* the identity ratio copies: no filter, no bank */
        const size_t bank_n = up * r->per_phase;
        double* h = (double*)malloc(r->taps * sizeof(double));
        float* bank = (float*)malloc(bank_n * sizeof(float));
        size_t j, phi;
        if (!h || !bank) st = 4;
        if (!st) {
            if (taps) for (j = 0; j < r->taps; ++j) h[j] = (double)taps[j];
            else design_default(r->half, up > down ? up : down, h);
            /* bank[j][phi] = up h[phi + j up], rounded to float32 once */
            for (j = 0; j < r->per_phase; ++j)
                for (phi = 0; phi < up; ++phi) {
                    const size_t k = phi + j * up;
                    bank[j * up + phi] = k < r->taps ? (float)((double)up * h[k]) : 0.0f;
                }
            st = vvb_malloc((void**)&r->d_bank, bank_n * sizeof(float));
            if (!st) st = vvb_memcpy_h2d(r->d_bank, bank, bank_n * sizeof(float), r->core.stream);
            if (!st) st = vvb_stream_sync(r->core.stream);
        }
        free(h); free(bank);
    }
    if (st) { rs_free(r); return st == 6 ? VV_DSP_ERROR_UNSUPPORTED : VV_DSP_ERROR_INTERNAL; }
    *out = r;
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_resample_poly_destroy(vv_dsp_resample_poly* r)
{
    int prev;
    if (!r) return VV_DSP_ERROR_NULL_POINTER;
    prev = vvdsp_internal_enter(&r->core);
    rs_free(r);
    vvdsp_internal_leave(prev);
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_resample_poly_set_stream(vv_dsp_resample_poly* r, void* cuda_stream)
{
    return vvdsp_internal_set_stream(r ? &r->core : NULL, cuda_stream);
}

vv_dsp_status vv_dsp_resample_poly_synchronize(vv_dsp_resample_poly* r)
{
    return vvdsp_internal_synchronize(r ? &r->core : NULL);
}

vv_dsp_status vv_dsp_resample_poly_get_config(const vv_dsp_resample_poly* r, size_t* up, size_t* down, size_t* num_taps,
                                              size_t* taps_per_phase)
{
    if (!r || !up || !down || !num_taps || !taps_per_phase) return VV_DSP_ERROR_NULL_POINTER;
    *up = r->up; *down = r->down; *num_taps = r->taps; *taps_per_phase = r->per_phase;
    return VV_DSP_OK;
}

size_t vv_dsp_resample_poly_output_length(const vv_dsp_resample_poly* r, size_t n)
{
    if (!r) return 0;
    /* ceil(n up / down) without forming n up */
    return (n / r->down) * r->up + ((n % r->down) * r->up + r->down - 1) / r->down;
}

static int copy_rows(vv_dsp_resample_poly* r, const vv_dsp_real* src, vv_dsp_mem_space ss, size_t sp, vv_dsp_real* dst,
                     vv_dsp_mem_space ds, size_t dp, size_t rows, size_t n)
{
    const size_t w = n * sizeof(float);
    size_t b;
    if (ss == VV_DSP_MEM_HOST && ds == VV_DSP_MEM_HOST) {
        for (b = 0; b < rows; ++b) memcpy(dst + b * dp, src + b * sp, w);
        return 0;
    }
    if (ss == VV_DSP_MEM_HOST) return vvb_memcpy2d_h2d(dst, dp * sizeof(float), src, sp * sizeof(float), w, rows, r->core.stream);
    if (ds == VV_DSP_MEM_HOST) return vvb_memcpy2d_d2h(dst, dp * sizeof(float), src, sp * sizeof(float), w, rows, r->core.stream);
    return vvb_memcpy2d_d2d(dst, dp * sizeof(float), src, sp * sizeof(float), w, rows, r->core.stream);
}

static int resample_impl(vv_dsp_resample_poly* r, const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch,
                         size_t n, size_t signal_pitch, vv_dsp_real* out, vv_dsp_mem_space out_space, size_t n_out,
                         size_t out_pitch)
{
    const size_t x_per = signals_space == VV_DSP_MEM_HOST ? n * sizeof(float) : 0;
    const size_t y_per = out_space == VV_DSP_MEM_HOST ? n_out * sizeof(float) : 0;
    const size_t cs = vvdsp_internal_chunk_rows(&r->core, batch, x_per > y_per ? x_per : y_per);
    const int any_host = signals_space == VV_DSP_MEM_HOST || out_space == VV_DSP_MEM_HOST;
    size_t done;
    int st = 0;
    if (!r->d_bank) {                             /* identity ratio: a copy, bit for bit */
        st = copy_rows(r, signals, signals_space, signal_pitch, out, out_space, out_pitch, batch, n);
        return vvdsp_internal_finish(&r->core, st, any_host);
    }
    if (x_per) st = vvdsp_internal_reserve(&r->core, (void**)&r->d_x, &r->x_bytes, cs * x_per);
    if (!st && y_per) st = vvdsp_internal_reserve(&r->core, (void**)&r->d_y, &r->y_bytes, cs * y_per);
    /* every chunk runs on the handle's stream, so stream order keeps the scratch buffers of consecutive chunks apart */
    for (done = 0; done < batch && !st; done += cs) {
        const size_t nb = batch - done < cs ? batch - done : cs;
        const float* d_x = signals + done * signal_pitch;
        float* d_y = out + done * out_pitch;
        size_t xp = signal_pitch, yp = out_pitch;
        if (signals_space == VV_DSP_MEM_HOST) {
            st = vvb_memcpy2d_h2d(r->d_x, n * sizeof(float), d_x, signal_pitch * sizeof(float), n * sizeof(float), nb, r->core.stream);
            d_x = r->d_x; xp = n;
        }
        if (out_space == VV_DSP_MEM_HOST) { d_y = r->d_y; yp = n_out; }
        if (!st)
            st = vvb_resample_poly(r->d_bank, r->up, r->down, r->per_phase, r->half, d_x, nb, n, xp, d_y, n_out, yp, r->core.stream);
        if (!st && out_space == VV_DSP_MEM_HOST)
            st = vvb_memcpy2d_d2h(out + done * out_pitch, out_pitch * sizeof(float), r->d_y, n_out * sizeof(float), n_out * sizeof(float),
                                  nb, r->core.stream);
    }
    return vvdsp_internal_finish(&r->core, st, any_host);
}

vv_dsp_status vv_dsp_resample_poly_batch(vv_dsp_resample_poly* r, const vv_dsp_real* signals, vv_dsp_mem_space signals_space,
                                         size_t batch, size_t n, size_t signal_pitch, vv_dsp_real* out,
                                         vv_dsp_mem_space out_space, size_t out_pitch, size_t* out_len)
{
    int prev, st;
    size_t n_out;
    if (!r || !signals || !out || !out_len) return VV_DSP_ERROR_NULL_POINTER;
    if ((unsigned)signals_space > 1u || (unsigned)out_space > 1u) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (n > (RS_MAX_UPSAMPLED - 1) / r->up) return VV_DSP_ERROR_INVALID_SIZE;              /* n up >= 2^62 */
    n_out = vv_dsp_resample_poly_output_length(r, n);
    if (signal_pitch == 0) signal_pitch = n;
    if (out_pitch == 0) out_pitch = n_out;
    if (signal_pitch < n || out_pitch < n_out) return VV_DSP_ERROR_INVALID_SIZE;
    if ((const void*)out == (const void*)signals) return VV_DSP_ERROR_UNSUPPORTED;      /* no in-place resampling */
    *out_len = n_out;
    if (batch == 0 || n == 0) return VV_DSP_OK;
    prev = vvdsp_internal_enter(&r->core);
    st = resample_impl(r, signals, signals_space, batch, n, signal_pitch, out, out_space, n_out, out_pitch);
    vvdsp_internal_leave(prev);
    return vvdsp_internal_status(st);
}
