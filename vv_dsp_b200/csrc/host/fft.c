/*
 * fft.c -- vv_dsp_fft_* plan API on top of the CUDA engine (host, C99).
 *
 * Boundary behaviour follows the reference's src/spectral/fft.c:15-107:
 *   set_backend      >= 3 -> OUT_OF_RANGE; backend not available -> UNSUPPORTED (:15-26)
 *   make_plan        NULL out -> NULL_POINTER, *out = NULL first, n == 0 -> INVALID_SIZE,
 *                    bad type / dir -> OUT_OF_RANGE (:63-72); plan captures the backend (:82)
 *   execute          NULL anything -> NULL_POINTER (:95-100)
 *   destroy(NULL)    -> OK (:102-107)
 *   set_fftw_flag / flush_fftw_cache -> UNSUPPORTED when FFTW is not compiled in (:54-61)
 * Backend id 0 ("KISS" in the reference) is the B200 engine here; FFTW and FFTS are never
 * available.  Data pointers are host memory; each execute is synchronous: pinned staging ->
 * H2D -> kernel -> D2H -> stream sync.  Unlike the reference the selector is not the place
 * where arithmetic changes: there is exactly one implementation, on the GPU.
 */
#include <stdlib.h>
#include <string.h>
#include "vv_dsp/spectral/fft.h"
#include "vv_dsp/b200.h"
#include "vvb200_cuda.h"
#include "internal.h"

struct vv_dsp_fft_plan {
    size_t n;
    vv_dsp_fft_type type;
    vv_dsp_fft_dir dir;
    vv_dsp_fft_backend backend;
    vvb_fft_engine* eng;
    void* stream;
    void *h_in, *h_out;      /* pinned staging */
    int zero_copy;           /* vv_dsp_fft_execute runs the kernel on h_in / h_out directly */
    void *d_in, *d_out;
    size_t in_bytes, out_bytes;
};

static vv_dsp_fft_backend g_backend = VV_DSP_FFT_BACKEND_KISS;

vv_dsp_status vv_dsp_fft_set_backend(vv_dsp_fft_backend backend)
{
    if ((unsigned)backend >= 3u) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (!vv_dsp_fft_is_backend_available(backend)) return VV_DSP_ERROR_UNSUPPORTED;
    g_backend = backend;
    return VV_DSP_OK;
}

vv_dsp_fft_backend vv_dsp_fft_get_backend(void) { return g_backend; }

int vv_dsp_fft_is_backend_available(vv_dsp_fft_backend backend) { return backend == VV_DSP_FFT_BACKEND_KISS; }

vv_dsp_status vv_dsp_fft_set_fftw_flag(vv_dsp_fftw_flag flag)
{
    (void)flag;
    return VV_DSP_ERROR_UNSUPPORTED;
}

vv_dsp_status vv_dsp_fft_flush_fftw_cache(void) { return VV_DSP_ERROR_UNSUPPORTED; }

static void plan_free(vv_dsp_fft_plan* p)
{
    if (!p) return;
    vvb_fft_engine_destroy(p->eng);
    vvb_host_free(p->h_in); vvb_host_free(p->h_out);
    vvb_free(p->d_in); vvb_free(p->d_out);
    if (p->stream) vvb_stream_destroy(p->stream);
    free(p);
}

vv_dsp_status vv_dsp_fft_make_plan(size_t n, vv_dsp_fft_type type, vv_dsp_fft_dir dir, vv_dsp_fft_plan** out_plan)
{
    vv_dsp_fft_plan* p;
    int st;
    const size_t cpx = 2 * sizeof(float);
    if (!out_plan) return VV_DSP_ERROR_NULL_POINTER;
    *out_plan = NULL;
    if (n == 0) return VV_DSP_ERROR_INVALID_SIZE;
    if (type != VV_DSP_FFT_C2C && type != VV_DSP_FFT_R2C && type != VV_DSP_FFT_C2R) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (dir != VV_DSP_FFT_FORWARD && dir != VV_DSP_FFT_BACKWARD) return VV_DSP_ERROR_OUT_OF_RANGE;
    p = (vv_dsp_fft_plan*)calloc(1, sizeof(*p));
    if (!p) return VV_DSP_ERROR_INTERNAL;
    p->n = n; p->type = type; p->dir = dir; p->backend = g_backend;
    p->in_bytes = (type == VV_DSP_FFT_C2C) ? n * cpx : (type == VV_DSP_FFT_R2C ? n * sizeof(float) : (n / 2 + 1) * cpx);
    p->out_bytes = (type == VV_DSP_FFT_C2C) ? n * cpx : (type == VV_DSP_FFT_R2C ? (n / 2 + 1) * cpx : n * sizeof(float));
    st = vvb_fft_engine_create(n, (int)type, (int)dir, &p->eng);
    if (!st) st = vvb_stream_create(&p->stream);
    if (!st) st = vvb_host_alloc(&p->h_in, p->in_bytes);
    if (!st) st = vvb_host_alloc(&p->h_out, p->out_bytes);
    p->zero_copy = !st && vvb_fft_engine_is_single_kernel(p->eng) && vvb_host_memory_is_device_visible() && getenv("VVB_PERFRAME_STAGED") == NULL;
    if (!st) st = vvb_malloc(&p->d_in, p->in_bytes);
    if (!st) st = vvb_malloc(&p->d_out, p->out_bytes);
    if (st) {
        plan_free(p);
        return st == 6 ? VV_DSP_ERROR_UNSUPPORTED : VV_DSP_ERROR_INTERNAL;
    }
    *out_plan = p;
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_fft_execute(const vv_dsp_fft_plan* plan, const void* in, void* out)
{
    int st;
    if (!plan || !in || !out) return VV_DSP_ERROR_NULL_POINTER;
    memcpy(plan->h_in, in, plan->in_bytes);
    if (plan->zero_copy) {
        /* single-kernel plans run straight on the pinned, device-visible staging buffers: one launch instead of three operations */
        st = vvb_fft_exec(plan->eng, plan->h_in, plan->h_out, 1, plan->stream);
    } else {
        st = vvb_memcpy_h2d(plan->d_in, plan->h_in, plan->in_bytes, plan->stream);
        if (!st) st = vvb_fft_exec(plan->eng, plan->d_in, plan->d_out, 1, plan->stream);
        if (!st) st = vvb_memcpy_d2h(plan->h_out, plan->d_out, plan->out_bytes, plan->stream);
    }
    if (!st) st = vvb_stream_sync(plan->stream);
    if (st) return VV_DSP_ERROR_INTERNAL;
    memcpy(out, plan->h_out, plan->out_bytes);
    /* even-n R2C: the Nyquist bin is exactly real (reference fft_kiss.c:140-143 forces +0) */
    if (plan->type == VV_DSP_FFT_R2C && plan->n % 2 == 0 && plan->n > 1) ((vv_dsp_cpx*)out)[plan->n / 2].im = 0.0f;
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_fft_destroy(vv_dsp_fft_plan* plan)
{
    plan_free(plan);   /* NULL is fine, like the reference */
    return VV_DSP_OK;
}

/* batched execute (include/vv_dsp/b200.h): the same engine, `batch` transforms per launch */
vv_dsp_status vv_dsp_fft_execute_batch(const vv_dsp_fft_plan* plan, const void* in, vv_dsp_mem_space in_space, void* out,
                                       vv_dsp_mem_space out_space, size_t batch, void* cuda_stream)
{
    void *d_in = NULL, *d_out = NULL, *stream;
    int st = 0;
    if (!plan || !in || !out) return VV_DSP_ERROR_NULL_POINTER;
    if ((unsigned)in_space > 1u || (unsigned)out_space > 1u) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (batch == 0) return VV_DSP_OK;
    stream = cuda_stream ? cuda_stream : plan->stream;
    if (in_space == VV_DSP_MEM_DEVICE && out_space == VV_DSP_MEM_DEVICE) {
        return vvdsp_internal_status(vvb_fft_exec(plan->eng, in, out, batch, stream));
    }
    if (in_space == VV_DSP_MEM_HOST) {
        st = vvb_malloc(&d_in, plan->in_bytes * batch);
        if (!st) st = vvb_memcpy_h2d(d_in, in, plan->in_bytes * batch, stream);
    }
    if (!st && out_space == VV_DSP_MEM_HOST) st = vvb_malloc(&d_out, plan->out_bytes * batch);
    if (!st) st = vvb_fft_exec(plan->eng, d_in ? d_in : in, d_out ? d_out : out, batch, stream);
    if (!st && out_space == VV_DSP_MEM_HOST) st = vvb_memcpy_d2h(out, d_out, plan->out_bytes * batch, stream);
    { int s2 = vvb_stream_sync(stream); if (!st) st = s2; }
    vvb_free(d_in); vvb_free(d_out);
    if (st) return vvdsp_internal_status(st);
    if (out_space == VV_DSP_MEM_HOST && plan->type == VV_DSP_FFT_R2C && plan->n % 2 == 0 && plan->n > 1) {
        size_t b, bins = plan->n / 2 + 1;
        for (b = 0; b < batch; ++b) ((vv_dsp_cpx*)out)[b * bins + plan->n / 2].im = 0.0f;
    }
    return VV_DSP_OK;
}
