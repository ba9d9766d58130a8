/*
 * stream.c -- ONE long stream sharded by frame range over several GPUs of this process
 * (include/vv_dsp/b200.h, SURVEY.md section 8e, BASELINE config 4; host, C99).
 *
 * What the reference does with such a stream is the per-frame loop of tools/dump_stft_roundtrip.c:44-54 over
 * the whole signal: process(frame f) ... reconstruct(frame f) into recon + f*hop, divide by the window sum.
 * Frames interact only through the overlap-add of src/spectral/stft.c:103-108, i.e. within nfft - hop samples.
 *
 * Here every device runs the two fused kernels of the batched path on its own frame range; the coupling at a
 * shard boundary is carried by sample halos (see b200.h): each shard recomputes the K-1 frames in front of its
 * range from its left halo, so synthesis needs no exchange and is bit-identical to the unsharded call.  Per
 * step and device: one small kernel that loads the two halos of nfft - hop floats from the neighbours' memory
 * (peer-to-peer over NVLink), the analysis
 * kernel, the synthesis kernel -- enqueued on the device's own stream, replayed as one CUDA graph per device
 * after the first step.  The devices never wait for one another inside a step: the halos are read from the
 * neighbours' owned INPUT samples, which no step writes.
 */
#include <stdlib.h>
#include <string.h>
#include "vv_dsp/b200.h"
#include "vvb200_cuda.h"
#include "internal.h"

typedef struct shard {
    int device;
    vv_dsp_stft* h;
    void* stream;
    size_t f0, f1, s0, s1, halo_frames, lh, rh, x_len, spec_frames;
    float* d_x;
    vvb_cpx* d_spec;
    float* d_y;
    void* graph;                 /* roundtrip step of this device, captured after the first run */
    void *ev0, *ev1;             /* timing */
} shard;

struct vv_dsp_stft_stream {
    size_t n, nfft, hop, bins, frames, ndev, halo;
    shard* sh;
    int graphs_tried;
};

static void stream_free(vv_dsp_stft_stream* s)
{
    size_t d;
    int cur = 0;
    if (!s) return;
    vvb_get_device(&cur);
    for (d = 0; s->sh && d < s->ndev; ++d) {
        shard* k = &s->sh[d];
        vvb_set_device(k->device);
        if (k->stream) vvb_stream_sync(k->stream);
        vvb_graph_destroy(k->graph);
        if (k->ev0) vvb_event_destroy(k->ev0);
        if (k->ev1) vvb_event_destroy(k->ev1);
        vvb_free(k->d_x); vvb_free(k->d_spec); vvb_free(k->d_y);
        if (k->h) (void)vv_dsp_stft_destroy(k->h);
    }
    vvb_set_device(cur);
    free(s->sh);
    free(s);
}

vv_dsp_status vv_dsp_stft_stream_create(const vv_dsp_stft_params* params, size_t n, size_t num_devices, const int* device_ids,
                                        vv_dsp_stft_stream** out)
{
    vv_dsp_stft_stream* s;
    size_t d, K;
    int st = 0, cur = 0, count = 0;
    if (!out || !params) return VV_DSP_ERROR_NULL_POINTER;
    *out = NULL;
    if (params->fft_size == 0 || params->hop_size == 0 || params->hop_size > params->fft_size || num_devices == 0)
        return VV_DSP_ERROR_INVALID_SIZE;
    if (params->fft_size % params->hop_size) return VV_DSP_ERROR_UNSUPPORTED;       /* halo frames need hop | fft_size */
    if (n < params->fft_size) return VV_DSP_ERROR_INVALID_SIZE;
    st = vvb_device_count(&count);
    if (st) return vvdsp_internal_status(st);
    for (d = 0; d < num_devices; ++d) {
        const int id = device_ids ? device_ids[d] : (int)d;
        if (id < 0 || id >= count) return VV_DSP_ERROR_OUT_OF_RANGE;
    }
    s = (vv_dsp_stft_stream*)calloc(1, sizeof(*s));
    if (!s) return VV_DSP_ERROR_INTERNAL;
    s->n = n; s->nfft = params->fft_size; s->hop = params->hop_size; s->bins = s->nfft / 2 + 1;
    s->frames = 1 + (n - s->nfft) / s->hop;
    s->ndev = num_devices; s->halo = s->nfft - s->hop;
    K = s->nfft / s->hop;
    /* every shard must hold the halo of its neighbours: at least K own frames */
    if (s->frames / num_devices < K) { free(s); return VV_DSP_ERROR_INVALID_SIZE; }
    s->sh = (shard*)calloc(num_devices, sizeof(shard));
    if (!s->sh) { free(s); return VV_DSP_ERROR_INTERNAL; }
    vvb_get_device(&cur);
    for (d = 0; d < num_devices && !st; ++d) {
        shard* k = &s->sh[d];
        vv_dsp_status vs;
        k->device = device_ids ? device_ids[d] : (int)d;
        k->f0 = s->frames * d / num_devices; k->f1 = s->frames * (d + 1) / num_devices;
        k->s0 = k->f0 * s->hop; k->s1 = (d == num_devices - 1) ? n : k->f1 * s->hop;
        k->halo_frames = d ? K - 1 : 0;
        k->lh = d ? s->halo : 0;
        k->rh = (d == num_devices - 1) ? 0 : s->halo;
        k->x_len = k->lh + (k->s1 - k->s0) + k->rh;
        k->spec_frames = k->halo_frames + (k->f1 - k->f0);
        st = vvb_set_device(k->device);
        if (st) break;
        vs = vv_dsp_stft_create(params, &k->h);
        if (vs != VV_DSP_OK) { st = (int)vs; break; }
        k->stream = vv_dsp_stft_get_stream(k->h);
        st = vvb_malloc((void**)&k->d_x, k->x_len * sizeof(float));
        if (!st) st = vvb_memset(k->d_x, 0, k->x_len * sizeof(float), k->stream);
        if (!st) st = vvb_malloc((void**)&k->d_spec, k->spec_frames * s->bins * sizeof(vvb_cpx));
        if (!st) st = vvb_malloc((void**)&k->d_y, ((k->s1 - k->s0 + 1) & ~(size_t)1) * sizeof(float));
        if (!st) st = vvb_event_create_timing(&k->ev0);
        if (!st) st = vvb_event_create_timing(&k->ev1);
        if (!st) st = vvb_stream_sync(k->stream);
    }
    /* the halo copies read the neighbours' memory */
    for (d = 0; d + 1 < num_devices && !st; ++d) {
        st = vvb_enable_peer_access(s->sh[d].device, s->sh[d + 1].device);
        if (!st) st = vvb_enable_peer_access(s->sh[d + 1].device, s->sh[d].device);
    }
    vvb_set_device(cur);
    if (st) { stream_free(s); return vvdsp_internal_status(st); }
    *out = s;
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_stft_stream_destroy(vv_dsp_stft_stream* s)
{
    if (!s) return VV_DSP_ERROR_NULL_POINTER;
    stream_free(s);
    return VV_DSP_OK;
}

size_t vv_dsp_stft_stream_num_frames(const vv_dsp_stft_stream* s) { return s ? s->frames : 0; }

vv_dsp_status vv_dsp_stft_stream_get_shard(const vv_dsp_stft_stream* s, size_t d, vv_dsp_stft_stream_shard* out)
{
    const shard* k;
    if (!s || !out) return VV_DSP_ERROR_NULL_POINTER;
    if (d >= s->ndev) return VV_DSP_ERROR_OUT_OF_RANGE;
    k = &s->sh[d];
    out->device = k->device;
    out->frame0 = k->f0; out->frame1 = k->f1; out->sample0 = k->s0; out->sample1 = k->s1;
    out->halo_frames = k->halo_frames; out->left_halo = k->lh; out->right_halo = k->rh;
    out->signal = k->d_x; out->spectra = (vv_dsp_cpx*)k->d_spec; out->output = k->d_y;
    out->cuda_stream = k->stream;
    return VV_DSP_OK;
}

vv_dsp_status vv_dsp_stft_stream_synchronize(vv_dsp_stft_stream* s)
{
    size_t d;
    int st = 0, cur = 0;
    if (!s) return VV_DSP_ERROR_NULL_POINTER;
    vvb_get_device(&cur);
    for (d = 0; d < s->ndev; ++d) {
        int s2 = vvb_set_device(s->sh[d].device);
        if (!s2) s2 = vvb_stream_sync(s->sh[d].stream);
        if (!st) st = s2;
    }
    vvb_set_device(cur);
    return vvdsp_internal_status(st);
}

vv_dsp_status vv_dsp_stft_stream_upload(vv_dsp_stft_stream* s, const vv_dsp_real* signal)
{
    size_t d;
    int st = 0, cur = 0;
    if (!s || !signal) return VV_DSP_ERROR_NULL_POINTER;
    vvb_get_device(&cur);
    for (d = 0; d < s->ndev && !st; ++d) {
        shard* k = &s->sh[d];
        st = vvb_set_device(k->device);
        if (!st) st = vvb_memcpy_h2d(k->d_x + k->lh, signal + k->s0, (k->s1 - k->s0) * sizeof(float), k->stream);
    }
    vvb_set_device(cur);
    if (st) return vvdsp_internal_status(st);
    return vv_dsp_stft_stream_synchronize(s);
}

/* the two halos of shard d: the last nfft-hop owned samples of d-1 and the first nfft-hop owned samples of d+1, read
 * straight from the neighbours' memory by a small kernel on d's own device (peer-to-peer loads over NVLink) */
static int enqueue_halos(vv_dsp_stft_stream* s, size_t d)
{
    shard* k = &s->sh[d];
    float *dl = NULL, *dr = NULL;
    const float *sl = NULL, *sr = NULL;
    if (k->lh) {
        const shard* l = &s->sh[d - 1];
        dl = k->d_x; sl = l->d_x + l->lh + (l->s1 - l->s0) - s->halo;
    }
    if (k->rh) {
        const shard* r = &s->sh[d + 1];
        dr = k->d_x + k->lh + (k->s1 - k->s0); sr = r->d_x + r->lh;
    }
    return vvb_halo_gather(dl, sl, dr, sr, s->halo, k->stream);
}

static int enqueue_forward(vv_dsp_stft_stream* s, size_t d)
{
    shard* k = &s->sh[d];
    size_t fr = 0;
    int st = enqueue_halos(s, d);
    if (!st) st = (int)vv_dsp_stft_batch_forward(k->h, k->d_x, VV_DSP_MEM_DEVICE, 1, k->x_len, k->x_len, VV_DSP_FRAMES_VALID,
                                                 VV_DSP_SPEC_COMPLEX, k->d_spec, VV_DSP_MEM_DEVICE, 0, &fr);
    if (!st && fr != k->spec_frames) st = 4;
    return st;
}

static int enqueue_inverse(vv_dsp_stft_stream* s, size_t d)
{
    shard* k = &s->sh[d];
    return (int)vv_dsp_stft_shard_inverse(k->h, (const vv_dsp_cpx*)k->d_spec, k->spec_frames, k->halo_frames, d == 0, d == s->ndev - 1,
                                          k->d_y, k->s1 - k->s0);
}

typedef int (*enqueue_fn)(vv_dsp_stft_stream*, size_t);

static vv_dsp_status for_each_device(vv_dsp_stft_stream* s, enqueue_fn a, enqueue_fn b)
{
    size_t d;
    int st = 0, cur = 0;
    if (!s) return VV_DSP_ERROR_NULL_POINTER;
    vvb_get_device(&cur);
    for (d = 0; d < s->ndev && !st; ++d) {
        st = vvb_set_device(s->sh[d].device);
        if (!st) st = a(s, d);
        if (!st && b) st = b(s, d);
    }
    vvb_set_device(cur);
    return vvdsp_internal_status(st);
}

vv_dsp_status vv_dsp_stft_stream_forward(vv_dsp_stft_stream* s) { return for_each_device(s, enqueue_forward, NULL); }
vv_dsp_status vv_dsp_stft_stream_inverse(vv_dsp_stft_stream* s) { return for_each_device(s, enqueue_inverse, NULL); }

/* Capture the step of every device into a graph.  Runs after one plain step, so every lazily built table
 * (normalisation edges, occupancy queries) exists and nothing in the captured region allocates or synchronises. */
static void try_capture(vv_dsp_stft_stream* s)
{
    size_t d;
    int cur = 0;
    s->graphs_tried = 1;
    if (getenv("VVB_STREAM_NO_GRAPH")) return;
    vvb_get_device(&cur);
    for (d = 0; d < s->ndev; ++d) {
        shard* k = &s->sh[d];
        int st = vvb_set_device(k->device);
        if (!st) st = vvb_stream_sync(k->stream);
        if (!st) st = vvb_graph_capture_begin(k->stream);
        if (st) break;                                       /* graphs unavailable: plain enqueue stays in use */
        st = enqueue_forward(s, d);
        if (!st) st = enqueue_inverse(s, d);
        {
            void* g = NULL;
            const int s2 = vvb_graph_capture_end(k->stream, &g);
            if (!st && !s2) k->graph = g; else vvb_graph_destroy(g);
        }
    }
    /* all or nothing */
    for (d = 0; d < s->ndev; ++d) if (!s->sh[d].graph) break;
    if (d < s->ndev)
        for (d = 0; d < s->ndev; ++d) { vvb_set_device(s->sh[d].device); vvb_graph_destroy(s->sh[d].graph); s->sh[d].graph = NULL; }
    vvb_set_device(cur);
}

static int enqueue_roundtrip(vv_dsp_stft_stream* s, size_t d)
{
    shard* k = &s->sh[d];
    int st;
    if (k->graph) return vvb_graph_launch(k->graph, k->stream);
    st = enqueue_forward(s, d);
    if (!st) st = enqueue_inverse(s, d);
    return st;
}

vv_dsp_status vv_dsp_stft_stream_roundtrip(vv_dsp_stft_stream* s)
{
    vv_dsp_status st;
    if (!s) return VV_DSP_ERROR_NULL_POINTER;
    st = for_each_device(s, enqueue_roundtrip, NULL);
    if (st == VV_DSP_OK && !s->graphs_tried) {
        st = vv_dsp_stft_stream_synchronize(s);
        if (st == VV_DSP_OK) try_capture(s);
    }
    return st;
}

vv_dsp_status vv_dsp_stft_stream_download(vv_dsp_stft_stream* s, vv_dsp_real* out)
{
    size_t d;
    int st = 0, cur = 0;
    if (!s || !out) return VV_DSP_ERROR_NULL_POINTER;
    vvb_get_device(&cur);
    for (d = 0; d < s->ndev && !st; ++d) {
        shard* k = &s->sh[d];
        st = vvb_set_device(k->device);
        if (!st) st = vvb_memcpy_d2h(out + k->s0, k->d_y, (k->s1 - k->s0) * sizeof(float), k->stream);
    }
    vvb_set_device(cur);
    if (st) return vvdsp_internal_status(st);
    return vv_dsp_stft_stream_synchronize(s);
}

vv_dsp_status vv_dsp_stft_stream_download_spectra(vv_dsp_stft_stream* s, vv_dsp_cpx* spectra)
{
    size_t d;
    int st = 0, cur = 0;
    if (!s || !spectra) return VV_DSP_ERROR_NULL_POINTER;
    vvb_get_device(&cur);
    for (d = 0; d < s->ndev && !st; ++d) {
        shard* k = &s->sh[d];
        st = vvb_set_device(k->device);
        if (!st) st = vvb_memcpy_d2h(spectra + k->f0 * s->bins, k->d_spec + k->halo_frames * s->bins,
                                     (k->f1 - k->f0) * s->bins * sizeof(vvb_cpx), k->stream);
    }
    vvb_set_device(cur);
    if (st) return vvdsp_internal_status(st);
    return vv_dsp_stft_stream_synchronize(s);
}

vv_dsp_status vv_dsp_stft_stream_time_roundtrip(vv_dsp_stft_stream* s, size_t warmup, size_t steps, double* ms_per_step)
{
    size_t d, i;
    int st = 0, cur = 0;
    vv_dsp_status vs;
    double worst = 0.0;
    if (!s || !ms_per_step) return VV_DSP_ERROR_NULL_POINTER;
    if (steps == 0) return VV_DSP_ERROR_INVALID_SIZE;
    for (i = 0; i < warmup + 1; ++i) {                       /* at least one: the step after it runs from the graphs */
        vs = vv_dsp_stft_stream_roundtrip(s);
        if (vs != VV_DSP_OK) return vs;
    }
    vs = vv_dsp_stft_stream_synchronize(s);
    if (vs != VV_DSP_OK) return vs;
    vvb_get_device(&cur);
    for (d = 0; d < s->ndev && !st; ++d) {
        st = vvb_set_device(s->sh[d].device);
        if (!st) st = vvb_event_record(s->sh[d].ev0, s->sh[d].stream);
    }
    for (i = 0; i < steps && !st; ++i)
        for (d = 0; d < s->ndev && !st; ++d) {
            st = vvb_set_device(s->sh[d].device);
            if (!st) st = enqueue_roundtrip(s, d);
        }
    for (d = 0; d < s->ndev && !st; ++d) {
        st = vvb_set_device(s->sh[d].device);
        if (!st) st = vvb_event_record(s->sh[d].ev1, s->sh[d].stream);
    }
    for (d = 0; d < s->ndev && !st; ++d) {
        float ms = 0.0f;
        st = vvb_set_device(s->sh[d].device);
        if (!st) st = vvb_stream_sync(s->sh[d].stream);
        if (!st) st = vvb_event_elapsed_ms(s->sh[d].ev0, s->sh[d].ev1, &ms);
        if ((double)ms > worst) worst = (double)ms;
    }
    vvb_set_device(cur);
    if (st) return vvdsp_internal_status(st);
    *ms_per_step = worst / (double)steps;
    return VV_DSP_OK;
}
