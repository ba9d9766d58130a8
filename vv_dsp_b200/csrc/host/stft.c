/*
 * stft.c -- vv_dsp_stft_* handle API and the batched extension (host, C99).
 *
 * Per-frame entry points keep the reference's contract (src/spectral/stft.c:30-144,
 * include/vv_dsp/spectral/stft.h:30-56): host pointers in and out, synchronous, same
 * validation order and status codes.  All arithmetic happens on the GPU through
 * include/vvb200_cuda.h; this file only validates, stages and mirrors.
 *
 * The batched entry points (include/vv_dsp/b200.h) are the throughput path: one fused
 * kernel per direction for a whole batch, device-resident or staged through pinned
 * double buffers so host<->device copies overlap the kernels.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "vv_dsp/b200.h"
#include "vv_dsp/core.h"
#include "vv_dsp/window.h"
#include "vvb200_cuda.h"
#include "internal.h"

#define NORM_CACHE 4
#define NSLOT 4            /* slots 0,1: analysis (host -> device staging); slots 2,3: synthesis (device -> host) */
#define NDEP 64            /* per-chunk completion events of the last stream-ordered analysis call */
/* per slot and direction (default; see stage_target below).  e2e step of the headline shape against the chunk size, same box:
 * 192 MB 45.8 ms, 96 MB 44.9, 48 MB 45.2, 24 MB 47.3 (the first chunk's upload and the last chunk's download are not overlapped) */
#define STAGE_TARGET_BYTES ((size_t)96 << 20)

typedef struct stage_slot {
    void* stream;
    void* d_in;  size_t in_bytes;
    void* d_out; size_t out_bytes;
    void* d_raw; size_t raw_bytes;     /* PCM ingest: the undecoded samples of a chunk */
} stage_slot;

struct vv_dsp_stft {
    size_t nfft, hop, bins;
    vv_dsp_stft_window win_type;
    vv_dsp_real* win;                 /* host copy of the window (bit-identical to the reference's) */
    vvb_engine* eng;
    int device;                       /* the CUDA device the handle was created on: every entry point runs there */
    void* own_stream;
    void* stream;                     /* own_stream or the caller's */
    /* per-frame staging */
    float* h_in;   vvb_cpx* h_spec;   float* h_frame;   /* pinned */
    float* d_in;   vvb_cpx* d_spec;   float* d_frame;
    /* batched staging (host-space arguments) */
    stage_slot slot[NSLOT];
    /* stream-ordered mode (vv_dsp_stft_set_async): host-space calls only enqueue work; a later call that
     * reads a device buffer produced chunk by chunk by an earlier one waits per chunk, on these events */
    int async;
    int zero_copy;                    /* per-frame calls: the kernels read / write the pinned staging buffers directly */
    struct { const char* lo; const char* hi; void* ev; int valid; } dep[NDEP];
    int dep_next;
    size_t stage_target;              /* staging bytes per slot and direction */
    /* log-mel chain: power scratch (grown on demand) and the last filterbank in device-sparse form */
    float* d_mel_scratch; size_t mel_scratch_bytes;
    mel_device mel; const float* mel_key_ptr; size_t mel_key_n; unsigned long long mel_key_hash;
    /* MFCC tail of that chain: log-mel scratch and the cosine / lifter tables of the last (n_mels, n_coeffs, lifter) */
    float* d_logmel_scratch; size_t logmel_scratch_bytes;
    mfcc_device mfcc;
    /* 1/sum(w^2) tables per frame count: [head nfft-hop | mid hop | tail nfft-hop] */
    struct { size_t frames; float* d_tab; int used; } norm[NORM_CACHE];
    int norm_next;
};

static vv_dsp_status map_status(int st)
{
    if (st == 0) return VV_DSP_OK;
    if (st >= 1 && st <= 6 && st != 5) return (vv_dsp_status)st;
    return VV_DSP_ERROR_INTERNAL;
}

/* A handle lives on the device that was current when it was created.  Entry points switch to it when the caller's
 * current device is another one and switch back before returning (multi-device callers: csrc/host/stream.c). */
static int dev_enter(const vv_dsp_stft* h)
{
    int cur = -1;
    if (!h || vvb_get_device(&cur) != 0 || cur == h->device) return -1;
    return vvb_set_device(h->device) == 0 ? cur : -1;
}
static void dev_leave(int prev) { if (prev >= 0) vvb_set_device(prev); }

const char* vv_dsp_b200_version(void) { return "vv-dsp_b200 0.1.0 (sm_100a)"; }
const char* vv_dsp_b200_last_error(void) { return vvb_last_error(); }
unsigned long long vv_dsp_b200_kernel_launches(void) { return vvb_kernel_launches(); }
vv_dsp_status vv_dsp_b200_fp32_peak(int packed, double* tflops) { return map_status(vvb_fp32_peak(packed, tflops)); }
vv_dsp_status vv_dsp_b200_sm_clock_mhz(void* cuda_stream, double* mhz) { return map_status(vvb_sm_clock_mhz(cuda_stream, mhz)); }

/* ---------------------------------------------------------------- create / destroy */
static void handle_free(vv_dsp_stft* h)
{
    int i;
    if (!h) return;
    for (i = 0; i < NSLOT; ++i) {
        vvb_free(h->slot[i].d_in); vvb_free(h->slot[i].d_out); vvb_free(h->slot[i].d_raw);
        if (h->slot[i].stream) vvb_stream_destroy(h->slot[i].stream);
    }
    for (i = 0; i < NORM_CACHE; ++i) vvb_free(h->norm[i].d_tab);
    vvb_free(h->d_mel_scratch); vvdsp_internal_mel_device_free(&h->mel);
    vvb_free(h->d_logmel_scratch); vvdsp_internal_mfcc_device_free(&h->mfcc);
    for (i = 0; i < NDEP; ++i) if (h->dep[i].ev) vvb_event_destroy(h->dep[i].ev);
    vvb_host_free(h->h_in); vvb_host_free(h->h_spec); vvb_host_free(h->h_frame);
    vvb_free(h->d_in); vvb_free(h->d_spec); vvb_free(h->d_frame);
    vvb_engine_destroy(h->eng);
    if (h->own_stream) vvb_stream_destroy(h->own_stream);
    free(h->win);
    free(h);
}

vv_dsp_status vv_dsp_stft_create(const vv_dsp_stft_params* params, vv_dsp_stft** out)
{
    vv_dsp_stft* h;
    vv_dsp_status ws;
    int st;
    if (!out || !params) return VV_DSP_ERROR_NULL_POINTER;
    *out = NULL;
    if (params->fft_size == 0 || params->hop_size == 0 || params->hop_size > params->fft_size)
        return VV_DSP_ERROR_INVALID_SIZE;
    h = (vv_dsp_stft*)calloc(1, sizeof(*h));
    if (!h) return VV_DSP_ERROR_INTERNAL;
    h->nfft = params->fft_size; h->hop = params->hop_size; h->bins = h->nfft / 2 + 1;
    h->win_type = params->window;
    h->stage_target = STAGE_TARGET_BYTES;
    {   /* test hook: a small staging size makes a modest batch span many chunks (tests/test_gpu_parity.py) */
        const char* env = getenv("VVB_STAGE_TARGET_BYTES");
        if (env && atol(env) > 0) h->stage_target = (size_t)atol(env);
    }
    h->win = (vv_dsp_real*)malloc(h->nfft * sizeof(vv_dsp_real));
    if (!h->win) { handle_free(h); return VV_DSP_ERROR_INTERNAL; }
    switch (params->window) {
    case VV_DSP_STFT_WIN_BOXCAR: ws = vv_dsp_window_boxcar(h->nfft, h->win); break;
    case VV_DSP_STFT_WIN_HANN: ws = vv_dsp_window_hann(h->nfft, h->win); break;
    case VV_DSP_STFT_WIN_HAMMING: ws = vv_dsp_window_hamming(h->nfft, h->win); break;
    default: ws = VV_DSP_ERROR_OUT_OF_RANGE; break;
    }
    if (ws != VV_DSP_OK) { handle_free(h); return ws; }
    st = vvb_device_ready();                      /* 6 = no usable device: reported as UNSUPPORTED, never a CPU fallback */
    if (!st) st = vvb_get_device(&h->device);
    if (!st) st = vvb_engine_create(h->nfft, h->hop, h->win, &h->eng);
    if (!st) st = vvb_stream_create(&h->own_stream);
    h->stream = h->own_stream;
    if (!st) st = vvb_host_alloc((void**)&h->h_in, h->nfft * sizeof(float));
    if (!st) st = vvb_host_alloc((void**)&h->h_spec, h->bins * sizeof(vvb_cpx));
    if (!st) st = vvb_host_alloc((void**)&h->h_frame, h->nfft * sizeof(float));
    /* (emulator builds and VVB_PERFRAME_STAGED=1 keep the explicit copies) */
    h->zero_copy = vvb_host_memory_is_device_visible() && getenv("VVB_PERFRAME_STAGED") == NULL;
    if (!st) st = vvb_malloc((void**)&h->d_in, h->nfft * sizeof(float));
    if (!st) st = vvb_malloc((void**)&h->d_spec, h->bins * sizeof(vvb_cpx));
    if (!st) st = vvb_malloc((void**)&h->d_frame, h->nfft * sizeof(float));
    if (st) { handle_free(h); return st == 6 ? VV_DSP_ERROR_UNSUPPORTED : VV_DSP_ERROR_INTERNAL; }
    *out = h;
    return VV_DSP_OK;
}

static vv_dsp_status destroy_impl(vv_dsp_stft* h)
{
    if (!h) return VV_DSP_ERROR_NULL_POINTER;     /* reference stft.c:63 */
    handle_free(h);
    return VV_DSP_OK;
}

/* ------------------------------------------------------------------ per-frame API */
static vv_dsp_status process_impl(vv_dsp_stft* h, const vv_dsp_real* in, vv_dsp_cpx* out)
{
    int st;
    size_t k;
    if (!h || !in || !out) return VV_DSP_ERROR_NULL_POINTER;
    memcpy(h->h_in, in, h->nfft * sizeof(float));
    if (h->zero_copy) {
        /* one launch instead of copy + launch + copy: the pinned staging buffers are mapped into the device's address
         * space (unified addressing), so the kernel reads the frame and writes the spectrum over the host link itself */
        st = vvb_stft_forward(h->eng, h->h_in, 1, h->nfft, h->nfft, 1, VVB_PAD_ZERO, VVB_OUT_COMPLEX, h->h_spec, h->bins, h->stream);
    } else {
        st = vvb_memcpy_h2d(h->d_in, h->h_in, h->nfft * sizeof(float), h->stream);
        if (!st) st = vvb_stft_forward(h->eng, h->d_in, 1, h->nfft, h->nfft, 1, VVB_PAD_ZERO, VVB_OUT_COMPLEX,
                                       h->d_spec, h->bins, h->stream);
        if (!st) st = vvb_memcpy_d2h(h->h_spec, h->d_spec, h->bins * sizeof(vvb_cpx), h->stream);
    }
    if (!st) st = vvb_stream_sync(h->stream);
    if (st) return map_status(st);
    /* bins 0..nfft/2 from the device; the rest is the conjugate mirror of a real input's spectrum */
    for (k = 0; k < h->bins; ++k) { out[k].re = h->h_spec[k].re; out[k].im = h->h_spec[k].im; }
    for (k = 1; k < h->bins; ++k)
        if (h->nfft - k > k) { out[h->nfft - k].re = h->h_spec[k].re; out[h->nfft - k].im = -h->h_spec[k].im; }
    return VV_DSP_OK;
}

static vv_dsp_status reconstruct_impl(vv_dsp_stft* h, const vv_dsp_cpx* in, vv_dsp_real* out_add, vv_dsp_real* norm_add)
{
    int st;
    size_t k, i;
    const size_t n = h ? h->nfft : 0;
    if (!h || !in || !out_add) return VV_DSP_ERROR_NULL_POINTER;
    /* Re(IDFT(X)) == IDFT of the Hermitian part of X: Xh[k] = (X[k] + conj X[n-k]) / 2 */
    for (k = 0; k < h->bins; ++k) {
        const vv_dsp_cpx a = in[k], b = in[(n - k) % n];
        h->h_spec[k].re = 0.5f * (a.re + b.re);
        h->h_spec[k].im = 0.5f * (a.im - b.im);
    }
    if (h->zero_copy) {
        st = vvb_stft_inverse_frames(h->eng, h->h_spec, 1, h->bins, h->h_frame, h->stream);
    } else {
        st = vvb_memcpy_h2d(h->d_spec, h->h_spec, h->bins * sizeof(vvb_cpx), h->stream);
        if (!st) st = vvb_stft_inverse_frames(h->eng, h->d_spec, 1, h->bins, h->d_frame, h->stream);
        if (!st) st = vvb_memcpy_d2h(h->h_frame, h->d_frame, n * sizeof(float), h->stream);
    }
    if (!st) st = vvb_stream_sync(h->stream);
    if (st) return map_status(st);
    for (i = 0; i < n; ++i) {
        out_add[i] += h->h_frame[i];
        if (norm_add) norm_add[i] += h->win[i] * h->win[i];
    }
    return VV_DSP_OK;
}

/* ------------------------------------------------------------------ frame counting */
size_t vv_dsp_stft_num_bins(const vv_dsp_stft* h) { return h ? h->bins : 0; }

size_t vv_dsp_stft_num_frames(const vv_dsp_stft* h, size_t n, vv_dsp_frame_convention convention)
{
    if (!h) return 0;
    switch (convention) {
    case VV_DSP_FRAMES_VALID: return n < h->nfft ? 0 : 1 + (n - h->nfft) / h->hop;
    case VV_DSP_FRAMES_SPECTROGRAM: return n < h->nfft ? 1 : 1 + (n - h->nfft + h->hop) / h->hop;
    case VV_DSP_FRAMES_PADDED_TAIL: return n / h->hop;   /* starts with start + nfft <= n + nfft - hop */
    case VV_DSP_FRAMES_CENTER: return (n + h->hop - 1) / h->hop;
    default: return 0;
    }
}

vv_dsp_status vv_dsp_stft_set_stream(vv_dsp_stft* h, void* cuda_stream)
{
    if (!h) return VV_DSP_ERROR_NULL_POINTER;
    h->stream = cuda_stream ? cuda_stream : h->own_stream;
    return VV_DSP_OK;
}

static vv_dsp_status synchronize_impl(vv_dsp_stft* h)
{
    int i, st;
    if (!h) return VV_DSP_ERROR_NULL_POINTER;
    st = vvb_stream_sync(h->stream);
    for (i = 0; i < NSLOT; ++i)
        if (h->slot[i].stream) { int s2 = vvb_stream_sync(h->slot[i].stream); if (!st) st = s2; }
    for (i = 0; i < NDEP; ++i) h->dep[i].valid = 0;
    return map_status(st);
}

vv_dsp_status vv_dsp_stft_set_async(vv_dsp_stft* h, int enable)
{
    if (!h) return VV_DSP_ERROR_NULL_POINTER;
    if (h->async && !enable) { vv_dsp_status st = synchronize_impl(h); if (st != VV_DSP_OK) return st; }
    h->async = enable ? 1 : 0;
    return VV_DSP_OK;
}

/* remember that the device range [lo, hi) is complete once everything enqueued so far on `stream` is */
static int dep_record(vv_dsp_stft* h, const void* lo, size_t bytes, void* stream)
{
    int k = h->dep_next, st = 0;
    h->dep_next = (h->dep_next + 1) % NDEP;
    if (!h->dep[k].ev) st = vvb_event_create(&h->dep[k].ev);
    /* the ring wrapped onto a chunk nobody has been told to wait for yet: a dependency is never dropped -- the
     * host waits for that (NDEP chunks old, almost certainly finished) chunk, after which no consumer needs an
     * event to read its range */
    if (!st && h->dep[k].valid) { st = vvb_event_sync(h->dep[k].ev); h->dep[k].valid = 0; }
    if (!st) st = vvb_event_record(h->dep[k].ev, stream);
    h->dep[k].lo = (const char*)lo; h->dep[k].hi = (const char*)lo + bytes; h->dep[k].valid = !st;
    return st;
}

/* make `stream` wait for every recorded producer chunk that overlaps [lo, hi) */
static int dep_wait(vv_dsp_stft* h, const void* lo, size_t bytes, void* stream)
{
    const char* a = (const char*)lo; const char* b = a + bytes;
    int k, st = 0;
    for (k = 0; k < NDEP && !st; ++k)
        if (h->dep[k].valid && h->dep[k].lo < b && a < h->dep[k].hi) st = vvb_stream_wait_event(stream, h->dep[k].ev);
    return st;
}

/* ---------------------------------------------------------------- staging helpers */
static int slot_reserve(stage_slot* s, size_t in_bytes, size_t out_bytes)
{
    int st = 0;
    if (!s->stream) st = vvb_stream_create(&s->stream);
    if (!st && in_bytes > s->in_bytes) {
        vvb_free(s->d_in); s->d_in = NULL; s->in_bytes = 0;
        st = vvb_malloc(&s->d_in, in_bytes);
        if (!st) s->in_bytes = in_bytes;
    }
    if (!st && out_bytes > s->out_bytes) {
        vvb_free(s->d_out); s->d_out = NULL; s->out_bytes = 0;
        st = vvb_malloc(&s->d_out, out_bytes);
        if (!st) s->out_bytes = out_bytes;
    }
    return st;
}

static size_t chunk_signals(const vv_dsp_stft* h, size_t batch, size_t bytes_per_signal)
{
    size_t c = bytes_per_signal ? h->stage_target / bytes_per_signal : batch;
    if (c < 1) c = 1;
    if (c > batch) c = batch;
    return c;
}

/* ------------------------------------------------------------------ batched forward */
/* pcm_format 0: `signals_v` are float32 samples; 16 / 24 / 32 / -32: HOST rows of little-endian PCM (or float32) samples as
 * they sit in a WAV data chunk (mono, one signal per row, pitch in samples), decoded on the device chunk by chunk with the
 * scaling of the reference's reader (src/audio/wav.c:458-521) -- the upload then carries 2 or 3 bytes per sample */
static vv_dsp_status batch_forward_impl(vv_dsp_stft* h, const void* signals_v, int pcm_format, vv_dsp_mem_space signals_space,
                                        size_t batch, size_t n, size_t signal_pitch,
                                        vv_dsp_frame_convention convention, vv_dsp_spec_kind kind, void* out,
                                        vv_dsp_mem_space out_space, size_t spec_pitch, size_t* out_frames)
{
    const vv_dsp_real* signals = (const vv_dsp_real*)signals_v;
    const size_t bps = pcm_format ? (size_t)(pcm_format < 0 ? -pcm_format : pcm_format) / 8 : sizeof(float);
    size_t frames, esize, done;
    int pad, st = 0, c = 0, fast;
    if (!h || !signals || !out) return VV_DSP_ERROR_NULL_POINTER;
    if (pcm_format && signals_space != VV_DSP_MEM_HOST) return VV_DSP_ERROR_UNSUPPORTED;   /* device PCM: vv_dsp_b200_pcm_to_planar first */
    fast = vvb_engine_is_fast(h->eng);
    if ((unsigned)convention > 3u || (unsigned)kind > 2u || (unsigned)signals_space > 1u || (unsigned)out_space > 1u)
        return VV_DSP_ERROR_OUT_OF_RANGE;
    if (signal_pitch == 0) signal_pitch = n;
    if (spec_pitch == 0) spec_pitch = h->bins;
    if (signal_pitch < n || spec_pitch < h->bins) return VV_DSP_ERROR_INVALID_SIZE;
    frames = vv_dsp_stft_num_frames(h, n, convention);
    if (out_frames) *out_frames = frames;
    if (batch == 0 || frames == 0) return VV_DSP_OK;
    pad = (convention == VV_DSP_FRAMES_CENTER) ? VVB_PAD_REFLECT_CENTER : VVB_PAD_ZERO;
    esize = (kind == VV_DSP_SPEC_COMPLEX) ? sizeof(vvb_cpx) : sizeof(float);

    if (signals_space == VV_DSP_MEM_DEVICE && out_space == VV_DSP_MEM_DEVICE)
        return map_status(vvb_stft_forward(h->eng, signals, batch, n, signal_pitch, frames, pad, (int)kind, out,
                                           spec_pitch, h->stream));

    /* at least one side lives in host memory: stream chunks of signals through two slots */
    {
        const size_t in_per = (signals_space == VV_DSP_MEM_HOST) ? (n ? n : 1) * sizeof(float) : 0;
        const size_t out_per = (out_space == VV_DSP_MEM_HOST) ? frames * h->bins * esize : 0;
        const size_t cs = chunk_signals(h, batch, in_per > out_per ? in_per : out_per);
        if (!h->async) st = vvb_stream_sync(h->stream);   /* device-side operands may still be in flight */
        for (done = 0; done < batch && !st; done += cs, ++c) {
            /* sizes without a Stockham kernel keep per-engine scratch buffers (chirp-z work buffer, synthesis frames):
             * their chunks all run on ONE stream, in order, in both directions */
            stage_slot* s = &h->slot[fast ? c % 2 : 0];
            const size_t nb = (batch - done < cs) ? batch - done : cs;
            const float* d_x;
            char* d_o;
            size_t xp, op;
            if (s->in_bytes < in_per * cs || s->out_bytes < out_per * cs || !s->stream || (pcm_format && s->raw_bytes < n * bps * cs)) {
                if (s->stream) st = vvb_stream_sync(s->stream);        /* about to reallocate its buffers */
                if (!st) st = slot_reserve(s, in_per * cs, out_per * cs);
                if (!st && pcm_format && s->raw_bytes < n * bps * cs) {
                    vvb_free(s->d_raw); s->d_raw = NULL; s->raw_bytes = 0;
                    st = vvb_malloc(&s->d_raw, n * bps * cs);
                    if (!st) s->raw_bytes = n * bps * cs;
                }
            }
            if (!st && !h->async) st = vvb_stream_sync(s->stream);     /* slot free again (stream order suffices when async) */
            if (st) break;
            if (pcm_format) {
                if (n) {
                    st = vvb_memcpy2d_h2d(s->d_raw, n * bps, (const char*)signals_v + done * signal_pitch * bps, signal_pitch * bps,
                                          n * bps, nb, s->stream);
                    /* the dense chunk is one channel of nb * n samples for the decoder */
                    if (!st) st = vvb_pcm_to_planar(s->d_raw, pcm_format, nb * n, 1, (float*)s->d_in, nb * n, s->stream);
                }
                d_x = (const float*)s->d_in; xp = n;
            } else if (signals_space == VV_DSP_MEM_HOST) {
                if (n)
                    st = vvb_memcpy2d_h2d(s->d_in, n * sizeof(float), signals + done * signal_pitch,
                                          signal_pitch * sizeof(float), n * sizeof(float), nb, s->stream);
                d_x = (const float*)s->d_in; xp = n;
            } else { d_x = signals + done * signal_pitch; xp = signal_pitch; }
            if (out_space == VV_DSP_MEM_HOST) { d_o = (char*)s->d_out; op = h->bins; }
            else { d_o = (char*)out + done * frames * spec_pitch * esize; op = spec_pitch; }
            if (!st && h->async && signals_space == VV_DSP_MEM_DEVICE)
                st = dep_wait(h, d_x, nb * xp * sizeof(float), s->stream);
            if (!st) st = vvb_stft_forward(h->eng, d_x, nb, n, xp, frames, pad, (int)kind, d_o, op, s->stream);
            if (!st && out_space == VV_DSP_MEM_HOST)
                st = vvb_memcpy2d_d2h((char*)out + done * frames * spec_pitch * esize, spec_pitch * esize, s->d_out,
                                      h->bins * esize, h->bins * esize, nb * frames, s->stream);
            if (!st && h->async && out_space == VV_DSP_MEM_DEVICE)
                st = dep_record(h, d_o, nb * frames * op * esize, s->stream);
        }
        if (!h->async)
            for (c = 0; c < NSLOT; ++c)
                if (h->slot[c].stream) { int s2 = vvb_stream_sync(h->slot[c].stream); if (!st) st = s2; }
    }
    return map_status(st);
}

/* --------------------------------------------------- 1/sum(w^2) tables for the ISTFT */
/* norm(t) = sum over frames f covering t, ASCENDING f, of w[t - f*hop]^2 in float32 -- the
 * order the reference accumulates norm_add in (src/spectral/stft.c:107 driven by
 * tools/dump_stft_roundtrip.c:44-47); entry = norm > 1e-12 ? 1/norm : 0 (dump tool :50-52). */
static float inv_norm_at(const vv_dsp_stft* h, size_t frames, size_t t)
{
    const size_t nfft = h->nfft, hop = h->hop;
    size_t f_lo = (t < nfft) ? 0 : (t - nfft) / hop + 1;
    size_t f_hi = t / hop, f;
    float acc = 0.0f;
    if (frames == 0) return 0.0f;
    if (f_hi > frames - 1) f_hi = frames - 1;
    for (f = f_lo; f <= f_hi && f_hi != (size_t)-1; ++f) {
        const float w = h->win[t - f * hop];
        acc += w * w;
    }
    return acc > 1e-12f ? 1.0f / acc : 0.0f;
}

static int norm_tables(vv_dsp_stft* h, size_t frames, const float** d_tab)
{
    const size_t edge = h->nfft - h->hop, total = 2 * edge + h->hop;
    size_t i;
    int k, st;
    float* host;
    for (k = 0; k < NORM_CACHE; ++k)
        if (h->norm[k].used && h->norm[k].frames == frames) { *d_tab = h->norm[k].d_tab; return 0; }
    host = (float*)malloc(total * sizeof(float));
    if (!host) return 4;
    for (i = 0; i < edge; ++i) host[i] = inv_norm_at(h, frames, i);                       /* head: t = i */
    for (i = 0; i < h->hop; ++i) {                                                       /* mid: all K frames present */
        /* any t >= edge with t % hop == i and t < frames*hop; computed as if frames were unlimited */
        const size_t t = ((edge + h->hop - 1) / h->hop) * h->hop + i;
        host[edge + i] = inv_norm_at(h, (size_t)-2, t);
    }
    for (i = 0; i < edge; ++i) host[edge + h->hop + i] = inv_norm_at(h, frames, frames * h->hop + i);  /* tail */
    k = h->norm_next; h->norm_next = (h->norm_next + 1) % NORM_CACHE;
    st = vvb_stream_sync(h->stream);                 /* the evicted table may still be in use */
    for (i = 0; i < NSLOT && !st; ++i) if (h->slot[i].stream) st = vvb_stream_sync(h->slot[i].stream);
    vvb_free(h->norm[k].d_tab); h->norm[k].d_tab = NULL; h->norm[k].used = 0;
    if (!st) st = vvb_malloc((void**)&h->norm[k].d_tab, total * sizeof(float));
    if (!st) st = vvb_memcpy_h2d(h->norm[k].d_tab, host, total * sizeof(float), h->stream);
    if (!st) st = vvb_stream_sync(h->stream);
    free(host);
    if (st) return st;
    h->norm[k].frames = frames; h->norm[k].used = 1;
    *d_tab = h->norm[k].d_tab;
    return 0;
}

/* ------------------------------------------------------------------ batched inverse */
static vv_dsp_status batch_inverse_impl(vv_dsp_stft* h, const vv_dsp_cpx* spectra, vv_dsp_mem_space spectra_space,
                                        size_t batch, size_t frames, size_t spec_pitch, vv_dsp_real* out,
                                        vv_dsp_mem_space out_space, size_t n_out, size_t out_pitch, int normalise)
{
    const float* d_tab = NULL;
    size_t done;
    int st = 0, c = 0, fast;
    if (!h || !out || (!spectra && frames)) return VV_DSP_ERROR_NULL_POINTER;
    fast = vvb_engine_is_fast(h->eng);
    if ((unsigned)spectra_space > 1u || (unsigned)out_space > 1u) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (spec_pitch == 0) spec_pitch = h->bins;
    if (out_pitch == 0) out_pitch = n_out;
    if (spec_pitch < h->bins || out_pitch < n_out) return VV_DSP_ERROR_INVALID_SIZE;
    if (batch == 0 || n_out == 0) return VV_DSP_OK;
    if (normalise) { st = norm_tables(h, frames, &d_tab); if (st) return map_status(st); }

    if (spectra_space == VV_DSP_MEM_DEVICE && out_space == VV_DSP_MEM_DEVICE)
        return map_status(vvb_stft_inverse(h->eng, (const vvb_cpx*)spectra, batch, frames, spec_pitch, out, n_out,
                                           out_pitch, d_tab, h->stream));
    {
        const size_t in_per = (spectra_space == VV_DSP_MEM_HOST) ? frames * h->bins * sizeof(vvb_cpx) : 0;
        const size_t out_per = (out_space == VV_DSP_MEM_HOST) ? n_out * sizeof(float) : 0;
        const size_t cs = chunk_signals(h, batch, in_per > out_per ? in_per : out_per);
        if (!h->async) st = vvb_stream_sync(h->stream);
        for (done = 0; done < batch && !st; done += cs, ++c) {
            stage_slot* s = &h->slot[fast ? 2 + c % 2 : 0];            /* own streams: D2H overlaps the analysis H2D */
            const size_t nb = (batch - done < cs) ? batch - done : cs;
            const vvb_cpx* d_s;
            float* d_y;
            size_t sp, yp;
            if (s->in_bytes < in_per * cs || s->out_bytes < out_per * cs || !s->stream) {
                if (s->stream) st = vvb_stream_sync(s->stream);
                if (!st) st = slot_reserve(s, in_per * cs, out_per * cs);
            }
            if (!st && !h->async) st = vvb_stream_sync(s->stream);
            if (st) break;
            if (spectra_space == VV_DSP_MEM_HOST) {
                if (frames)
                    st = vvb_memcpy2d_h2d(s->d_in, h->bins * sizeof(vvb_cpx), spectra + done * frames * spec_pitch,
                                          spec_pitch * sizeof(vvb_cpx), h->bins * sizeof(vvb_cpx), nb * frames, s->stream);
                d_s = (const vvb_cpx*)s->d_in; sp = h->bins;
            } else { d_s = (const vvb_cpx*)spectra + done * frames * spec_pitch; sp = spec_pitch; }
            if (out_space == VV_DSP_MEM_HOST) { d_y = (float*)s->d_out; yp = n_out; }
            else { d_y = out + done * out_pitch; yp = out_pitch; }
            if (!st && h->async && spectra_space == VV_DSP_MEM_DEVICE && frames)
                st = dep_wait(h, d_s, nb * frames * sp * sizeof(vvb_cpx), s->stream);
            if (!st) st = vvb_stft_inverse(h->eng, d_s, nb, frames, sp, d_y, n_out, yp, d_tab, s->stream);
            if (!st && out_space == VV_DSP_MEM_HOST)
                st = vvb_memcpy2d_d2h(out + done * out_pitch, out_pitch * sizeof(float), s->d_out, n_out * sizeof(float),
                                      n_out * sizeof(float), nb, s->stream);
            if (!st && h->async && out_space == VV_DSP_MEM_DEVICE)
                st = dep_record(h, d_y, nb * yp * sizeof(float), s->stream);
        }
        if (!h->async)
            for (c = 0; c < NSLOT; ++c)
                if (h->slot[c].stream) { int s2 = vvb_stream_sync(h->slot[c].stream); if (!st) st = s2; }
    }
    return map_status(st);
}

vv_dsp_status vv_dsp_stft_istft(vv_dsp_stft* h, const vv_dsp_cpx* half_spectra, size_t frames, vv_dsp_real* out, size_t n_out)
{
    return vv_dsp_stft_batch_inverse(h, half_spectra, VV_DSP_MEM_HOST, 1, frames, 0, out, VV_DSP_MEM_HOST, n_out, 0, 1);
}

/* ---------------------------------------------------- whole-signal magnitude (reference API) */
vv_dsp_status vv_dsp_stft_spectrogram(vv_dsp_stft* h, const vv_dsp_real* signal, size_t n, vv_dsp_real* out_mag,
                                      size_t* out_frames)
{
    size_t frames, f, k;
    float* half;
    vv_dsp_status st;
    static const float zero = 0.0f;
    if (!h || !signal || !out_mag || !out_frames) return VV_DSP_ERROR_NULL_POINTER;
    frames = vv_dsp_stft_num_frames(h, n, VV_DSP_FRAMES_SPECTROGRAM);
    *out_frames = frames;
    half = (float*)malloc(frames * h->bins * sizeof(float));
    if (!half) return VV_DSP_ERROR_INTERNAL;
    st = vv_dsp_stft_batch_forward(h, n ? signal : &zero, VV_DSP_MEM_HOST, 1, n, n ? n : 1, VV_DSP_FRAMES_SPECTROGRAM,
                                   VV_DSP_SPEC_MAGNITUDE, half, VV_DSP_MEM_HOST, 0, NULL);
    if (st == VV_DSP_OK) {
        /* the reference writes all fft_size bins per frame (stft.c:133-140); |X[n-k]| = |X[k]| */
        for (f = 0; f < frames; ++f) {
            const float* src = half + f * h->bins;
            float* dst = out_mag + f * h->nfft;
            for (k = 0; k < h->bins; ++k) dst[k] = src[k];
            for (k = 1; k < h->bins; ++k) if (h->nfft - k > k) dst[h->nfft - k] = src[k];
        }
    }
    free(half);
    return st;
}

/* -------------------------------------------------- STFT -> power -> log-mel (include/vv_dsp/b200.h) */
/* Chunks of signals whose power spectrogram fits a bounded device scratch; per chunk the fused power
 * kernel and the HBM-bound log-mel kernel run back to back on one stream. */
/* STFT -> power -> log-mel [-> MFCC when n_coeffs > 0]; `width` = floats per output frame */
/* pcm_format 0: float32 signals; 16 / 24 / 32 / -32: HOST rows of WAV samples, decoded on the device chunk by chunk (see
 * batch_forward_impl) */
static vv_dsp_status batch_mel_chain(vv_dsp_stft* h, const void* signals_v, int pcm_format, vv_dsp_mem_space signals_space, size_t batch,
                                     size_t n, size_t signal_pitch, vv_dsp_frame_convention convention,
                                     const vv_dsp_real* filterbank_weights, size_t n_mels, vv_dsp_real log_epsilon,
                                     size_t n_coeffs, vv_dsp_real lifter,
                                     vv_dsp_real* out, vv_dsp_mem_space out_space, size_t* out_frames)
{
    const size_t scratch_target = (size_t)768 << 20;
    const size_t width = n_coeffs ? n_coeffs : n_mels;
    size_t frames, per_signal, cs, done, i;
    const vv_dsp_real* signals = (const vv_dsp_real*)signals_v;
    const size_t bps = pcm_format ? (size_t)(pcm_format < 0 ? -pcm_format : pcm_format) / 8 : sizeof(float);
    float *d_power, *d_x = NULL, *d_o = NULL;
    void* d_raw = NULL;
    unsigned long long hash = 1469598103934665603ull;
    void* stream;
    int st = 0, pad, fused;
    if (!h || !signals || !filterbank_weights || !out) return VV_DSP_ERROR_NULL_POINTER;
    if (pcm_format && signals_space != VV_DSP_MEM_HOST) return VV_DSP_ERROR_UNSUPPORTED;
    if ((unsigned)convention > 3u || (unsigned)signals_space > 1u || (unsigned)out_space > 1u) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (n_mels == 0) return VV_DSP_ERROR_INVALID_SIZE;
    if (log_epsilon < 0.0f) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (n_coeffs > n_mels) return VV_DSP_ERROR_INVALID_SIZE;
    if (lifter < 0.0f) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (signal_pitch == 0) signal_pitch = n;
    if (signal_pitch < n) return VV_DSP_ERROR_INVALID_SIZE;
    frames = vv_dsp_stft_num_frames(h, n, convention);
    if (out_frames) *out_frames = frames;
    if (batch == 0 || frames == 0) return VV_DSP_OK;
    pad = (convention == VV_DSP_FRAMES_CENTER) ? VVB_PAD_REFLECT_CENTER : VVB_PAD_ZERO;
    per_signal = frames * h->bins * sizeof(float);
    cs = scratch_target / per_signal; if (cs < 1) cs = 1; if (cs > batch) cs = batch;
    stream = h->stream;
    /* the device-sparse filterbank is cached per handle; fingerprint = pointer, size and an FNV-1a hash of EVERY weight
     * (about 80 k words: negligible next to the kernels, and an in-place edit of any weight is seen) */
    for (i = 0; i < n_mels * h->bins; ++i) {
        unsigned int bits; memcpy(&bits, filterbank_weights + i, sizeof(bits));
        hash = (hash ^ bits) * 1099511628211ull;
    }
    if (!h->mel.d_meta || h->mel_key_ptr != filterbank_weights || h->mel_key_n != n_mels || h->mel_key_hash != hash) {
        st = vvb_stream_sync(stream);
        vvdsp_internal_mel_device_free(&h->mel);
        if (!st) st = vvdsp_internal_mel_device_build(filterbank_weights, n_mels, h->bins, stream, &h->mel);
        if (!st) { h->mel_key_ptr = filterbank_weights; h->mel_key_n = n_mels; h->mel_key_hash = hash; }
        else { h->mel_key_ptr = NULL; h->mel_key_n = 0; }
    }
    /* one kernel from samples to log-mel rows where the plan has it (fft_size 2048 marching kernel): the power spectrogram
     * then never exists in HBM and there is no scratch; chunks only bound the host staging buffers */
    fused = !st && h->mel.d_fw && vvb_stft_forward_logmel_ok(h->eng, h->mel.f_segments, h->mel.f_prow, h->mel.f_unit, n_mels);
    if (getenv("VVB_MEL_DEBUG")) {
        /* 2 / 1: marching kernel with two frames / one frame per band-sum phase; 3: generic kernel, band sums per warp */
        const int mode = fused ? vvb_stft_forward_logmel_ok(h->eng, h->mel.f_segments, h->mel.f_prow, h->mel.f_unit, n_mels) : 0;
        fprintf(stderr, "vvb: STFT -> log-mel: %s\n", mode == 2 ? "one fused kernel, two frames per band-sum phase"
                                                    : mode == 1 ? "one fused kernel, one frame per band-sum phase"
                                                    : mode ? "one fused kernel, band sums per warp" : "power kernel + log-mel kernel");
    }
    if (fused) {
        const size_t stage_target = h->stage_target;                   /* VVB_STAGE_TARGET_BYTES applies here too */
        cs = batch;
        if (signals_space == VV_DSP_MEM_HOST || out_space == VV_DSP_MEM_HOST) {
            const size_t per = (n ? n : 1) * sizeof(float) + frames * n_mels * sizeof(float);
            cs = stage_target / per;
        } else if (n_coeffs) {
            cs = scratch_target / (frames * n_mels * sizeof(float));    /* the log-mel rows between the two kernels */
        }
        if (cs < 1) cs = 1;
        if (cs > batch) cs = batch;
    }
    if (!st && !fused && h->mel_scratch_bytes < cs * per_signal) {
        st = vvb_stream_sync(stream);
        vvb_free(h->d_mel_scratch); h->d_mel_scratch = NULL; h->mel_scratch_bytes = 0;
        if (!st) st = vvb_malloc((void**)&h->d_mel_scratch, cs * per_signal);
        if (!st) h->mel_scratch_bytes = cs * per_signal;
    }
    d_power = h->d_mel_scratch;
    if (!st && n_coeffs) {
        if (!h->mfcc.d_table || h->mfcc.n_mels != n_mels || h->mfcc.n_coeffs != n_coeffs || h->mfcc.lifter != lifter) {
            st = vvb_stream_sync(stream);
            vvdsp_internal_mfcc_device_free(&h->mfcc);
            if (!st) st = vvdsp_internal_mfcc_device_build(n_mels, n_coeffs, lifter, stream, &h->mfcc);
        }
        if (!st && h->logmel_scratch_bytes < cs * frames * n_mels * sizeof(float)) {
            st = vvb_stream_sync(stream);
            vvb_free(h->d_logmel_scratch); h->d_logmel_scratch = NULL; h->logmel_scratch_bytes = 0;
            if (!st) st = vvb_malloc((void**)&h->d_logmel_scratch, cs * frames * n_mels * sizeof(float));
            if (!st) h->logmel_scratch_bytes = cs * frames * n_mels * sizeof(float);
        }
    }
    if (!st && fused && signals_space == VV_DSP_MEM_HOST && batch > cs) {
        /* host signals through the fused kernel, more than one chunk: two staging sets on the handle's two slot streams, so
         * the upload of chunk c + 1 overlaps the kernel and the download of chunk c (a single stream serialises them) */
        float *px[2] = {NULL, NULL}, *po[2] = {NULL, NULL}, *pl[2] = {NULL, NULL};
        void *ps[2] = {NULL, NULL}, *pr[2] = {NULL, NULL};
        size_t c = 0;
        int k;
        for (k = 0; k < 2 && !st; ++k) {
            st = slot_reserve(&h->slot[k], 0, 0);                          /* makes sure the slot's stream exists */
            ps[k] = h->slot[k].stream;
            if (!st) st = vvb_stream_sync(ps[k]);
            if (!st) st = vvb_malloc((void**)&px[k], cs * (n ? n : 1) * sizeof(float));
            if (!st && pcm_format) st = vvb_malloc(&pr[k], cs * (n ? n : 1) * bps);
            if (!st && out_space == VV_DSP_MEM_HOST) st = vvb_malloc((void**)&po[k], cs * frames * width * sizeof(float));
            if (!st && n_coeffs) st = vvb_malloc((void**)&pl[k], cs * frames * n_mels * sizeof(float));
        }
        if (!st) st = vvb_stream_sync(stream);                              /* device-side operands may still be in flight */
        for (done = 0; done < batch && !st; done += cs, ++c) {
            const size_t nb = (batch - done < cs) ? batch - done : cs;
            float* o_dev = (out_space == VV_DSP_MEM_HOST) ? po[c & 1] : out + done * frames * width;
            float* lm_dev = n_coeffs ? pl[c & 1] : o_dev;
            void* sq = ps[c & 1];
            if (c >= 2) st = vvb_stream_sync(sq);                           /* this set's previous chunk has left */
            if (!st && n && pcm_format) {
                st = vvb_memcpy2d_h2d(pr[c & 1], n * bps, (const char*)signals_v + done * signal_pitch * bps, signal_pitch * bps, n * bps, nb, sq);
                if (!st) st = vvb_pcm_to_planar(pr[c & 1], pcm_format, nb * n, 1, px[c & 1], nb * n, sq);
            } else if (!st && n) {
                st = vvb_memcpy2d_h2d(px[c & 1], n * sizeof(float), signals + done * signal_pitch, signal_pitch * sizeof(float),
                                      n * sizeof(float), nb, sq);
            }
            if (!st) st = vvb_stft_forward_logmel(h->eng, px[c & 1], nb, n, n ? n : 1, frames, pad, h->mel.d_fw, h->mel.d_fseg,
                                                  h->mel.f_segments, h->mel.f_prow, h->mel.f_unit, n_mels, log_epsilon, lm_dev, sq);
            if (!st && n_coeffs) st = vvb_mfcc(lm_dev, nb * frames, n_mels, n_coeffs, h->mfcc.d_table, h->mfcc.d_lifter, o_dev, sq);
            if (!st && out_space == VV_DSP_MEM_HOST)
                st = vvb_memcpy_d2h(out + done * frames * width, po[c & 1], nb * frames * width * sizeof(float), sq);
        }
        for (k = 0; k < 2; ++k) {
            if (ps[k]) { int s2 = vvb_stream_sync(ps[k]); if (!st) st = s2; }
            vvb_free(px[k]); vvb_free(po[k]); vvb_free(pl[k]); vvb_free(pr[k]);
        }
        return map_status(st);
    }
    if (!st && signals_space == VV_DSP_MEM_HOST) st = vvb_malloc((void**)&d_x, cs * (n ? n : 1) * sizeof(float));
    if (!st && pcm_format) st = vvb_malloc(&d_raw, cs * (n ? n : 1) * bps);
    if (!st && out_space == VV_DSP_MEM_HOST) st = vvb_malloc((void**)&d_o, cs * frames * width * sizeof(float));
    for (done = 0; done < batch && !st; done += cs) {
        const size_t nb = (batch - done < cs) ? batch - done : cs;
        const float* x_dev = signals + done * signal_pitch;
        size_t xp = signal_pitch;
        float* o_dev = out + done * frames * width;
        float* lm_dev;
        if (pcm_format) {
            if (n) {
                st = vvb_memcpy2d_h2d(d_raw, n * bps, (const char*)signals_v + done * signal_pitch * bps, signal_pitch * bps, n * bps, nb, stream);
                if (!st) st = vvb_pcm_to_planar(d_raw, pcm_format, nb * n, 1, d_x, nb * n, stream);
            }
            x_dev = d_x; xp = n ? n : 1;
        } else if (signals_space == VV_DSP_MEM_HOST) {
            if (n) st = vvb_memcpy2d_h2d(d_x, n * sizeof(float), signals + done * signal_pitch, signal_pitch * sizeof(float),
                                         n * sizeof(float), nb, stream);
            x_dev = d_x; xp = n ? n : 1;
        }
        if (out_space == VV_DSP_MEM_HOST) o_dev = d_o;
        lm_dev = n_coeffs ? h->d_logmel_scratch : o_dev;
        if (fused) {
            if (!st) st = vvb_stft_forward_logmel(h->eng, x_dev, nb, n, xp, frames, pad, h->mel.d_fw, h->mel.d_fseg, h->mel.f_segments,
                                                  h->mel.f_prow, h->mel.f_unit, n_mels, log_epsilon, lm_dev, stream);
        } else {
            if (!st) st = vvb_stft_forward(h->eng, x_dev, nb, n, xp, frames, pad, VVB_OUT_POWER, d_power, h->bins, stream);
            if (!st) st = vvdsp_internal_logmel(&h->mel, d_power, nb * frames, h->bins, n_mels, log_epsilon, lm_dev, stream);
        }
        if (!st && n_coeffs) st = vvb_mfcc(lm_dev, nb * frames, n_mels, n_coeffs, h->mfcc.d_table, h->mfcc.d_lifter, o_dev, stream);
        if (!st && out_space == VV_DSP_MEM_HOST)
            st = vvb_memcpy_d2h(out + done * frames * width, d_o, nb * frames * width * sizeof(float), stream);
        if (!st && signals_space == VV_DSP_MEM_HOST) st = vvb_stream_sync(stream);   /* staging buffer reuse */
    }
    /* device-resident calls only enqueue (scratch and filterbank live in the handle); host buffers: synchronous */
    if (signals_space == VV_DSP_MEM_HOST || out_space == VV_DSP_MEM_HOST) {
        int s2 = vvb_stream_sync(stream); if (!st) st = s2;
        vvb_free(d_x); vvb_free(d_o); vvb_free(d_raw);
    }
    return map_status(st);
}

vv_dsp_status vv_dsp_stft_batch_logmel_pcm(vv_dsp_stft* h, const void* pcm, int format, size_t batch, size_t n, size_t signal_pitch,
                                           vv_dsp_frame_convention convention, const vv_dsp_real* filterbank_weights, size_t n_mels,
                                           vv_dsp_real log_epsilon, vv_dsp_real* out, vv_dsp_mem_space out_space, size_t* out_frames)
{
    int prev;
    vv_dsp_status st;
    if (format != 16 && format != 24 && format != 32 && format != -32) return VV_DSP_ERROR_OUT_OF_RANGE;
    prev = dev_enter(h);
    st = batch_mel_chain(h, pcm, format, VV_DSP_MEM_HOST, batch, n, signal_pitch, convention, filterbank_weights, n_mels, log_epsilon, 0, 0.0f,
                         out, out_space, out_frames);
    dev_leave(prev);
    return st;
}

vv_dsp_status vv_dsp_stft_batch_logmel(vv_dsp_stft* h, const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch,
                                       size_t n, size_t signal_pitch, vv_dsp_frame_convention convention,
                                       const vv_dsp_real* filterbank_weights, size_t n_mels, vv_dsp_real log_epsilon,
                                       vv_dsp_real* out, vv_dsp_mem_space out_space, size_t* out_frames)
{
    const int prev = dev_enter(h);
    const vv_dsp_status st = batch_mel_chain(h, signals, 0, signals_space, batch, n, signal_pitch, convention, filterbank_weights, n_mels,
                                             log_epsilon, 0, 0.0f, out, out_space, out_frames);
    dev_leave(prev);
    return st;
}

vv_dsp_status vv_dsp_stft_batch_mfcc(vv_dsp_stft* h, const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch,
                                     size_t n, size_t signal_pitch, vv_dsp_frame_convention convention,
                                     const vv_dsp_real* filterbank_weights, size_t n_mels, vv_dsp_real log_epsilon,
                                     size_t num_mfcc_coeffs, vv_dsp_real lifter_coeff,
                                     vv_dsp_real* out, vv_dsp_mem_space out_space, size_t* out_frames)
{
    int prev;
    vv_dsp_status st;
    if (num_mfcc_coeffs == 0) return VV_DSP_ERROR_INVALID_SIZE;
    prev = dev_enter(h);
    st = batch_mel_chain(h, signals, 0, signals_space, batch, n, signal_pitch, convention, filterbank_weights, n_mels, log_epsilon,
                         num_mfcc_coeffs, lifter_coeff, out, out_space, out_frames);
    dev_leave(prev);
    return st;
}

/* ------------------------------------------------- one frame-range shard of a longer stream (include/vv_dsp/b200.h) */
static vv_dsp_status shard_inverse_impl(vv_dsp_stft* h, const vv_dsp_cpx* spectra, size_t local_frames, size_t halo_frames,
                                        int is_first, int is_last, vv_dsp_real* out, size_t n_out)
{
    const float* d_tab = NULL;
    int st;
    if (!h || !spectra || !out) return VV_DSP_ERROR_NULL_POINTER;
    if (local_frames == 0 || halo_frames >= local_frames || n_out == 0) return VV_DSP_ERROR_INVALID_SIZE;
    if (h->nfft % h->hop) return VV_DSP_ERROR_UNSUPPORTED;
    if (halo_frames != (is_first ? 0 : h->nfft / h->hop - 1)) return VV_DSP_ERROR_INVALID_SIZE;
    /* the edge tables depend on the frame count only when fewer than nfft/hop frames exist: a shard that carries its
     * halo sees the same head / tail factors as the whole stream */
    if (!is_first && local_frames - halo_frames < h->nfft / h->hop - 1) return VV_DSP_ERROR_INVALID_SIZE;
    st = norm_tables(h, local_frames, &d_tab);
    if (!st) st = vvb_stft_inverse_shard(h->eng, (const vvb_cpx*)spectra, local_frames, halo_frames, is_first, is_last, h->bins,
                                         out, n_out, d_tab, h->stream);
    return map_status(st);
}

/* ------------------------------------------------- public entry points: run on the handle's device */
vv_dsp_status vv_dsp_stft_destroy(vv_dsp_stft* h)
{
    const int prev = dev_enter(h);
    const vv_dsp_status st = destroy_impl(h);
    dev_leave(prev);
    return st;
}
vv_dsp_status vv_dsp_stft_process(vv_dsp_stft* h, const vv_dsp_real* in, vv_dsp_cpx* out)
{
    const int prev = dev_enter(h);
    const vv_dsp_status st = process_impl(h, in, out);
    dev_leave(prev);
    return st;
}
vv_dsp_status vv_dsp_stft_reconstruct(vv_dsp_stft* h, const vv_dsp_cpx* in, vv_dsp_real* out_add, vv_dsp_real* norm_add)
{
    const int prev = dev_enter(h);
    const vv_dsp_status st = reconstruct_impl(h, in, out_add, norm_add);
    dev_leave(prev);
    return st;
}
vv_dsp_status vv_dsp_stft_synchronize(vv_dsp_stft* h)
{
    const int prev = dev_enter(h);
    const vv_dsp_status st = synchronize_impl(h);
    dev_leave(prev);
    return st;
}
vv_dsp_status vv_dsp_stft_batch_forward(vv_dsp_stft* h, const vv_dsp_real* signals, vv_dsp_mem_space signals_space,
                                        size_t batch, size_t n, size_t signal_pitch,
                                        vv_dsp_frame_convention convention, vv_dsp_spec_kind kind, void* out,
                                        vv_dsp_mem_space out_space, size_t spec_pitch, size_t* out_frames)
{
    const int prev = dev_enter(h);
    const vv_dsp_status st = batch_forward_impl(h, signals, 0, signals_space, batch, n, signal_pitch, convention, kind, out, out_space,
                                                spec_pitch, out_frames);
    dev_leave(prev);
    return st;
}
vv_dsp_status vv_dsp_stft_batch_forward_pcm(vv_dsp_stft* h, const void* pcm, int format, size_t batch, size_t n, size_t signal_pitch,
                                            vv_dsp_frame_convention convention, vv_dsp_spec_kind kind, void* out,
                                            vv_dsp_mem_space out_space, size_t spec_pitch, size_t* out_frames)
{
    int prev;
    vv_dsp_status st;
    if (format != 16 && format != 24 && format != 32 && format != -32) return VV_DSP_ERROR_OUT_OF_RANGE;
    prev = dev_enter(h);
    st = batch_forward_impl(h, pcm, format, VV_DSP_MEM_HOST, batch, n, signal_pitch, convention, kind, out, out_space, spec_pitch, out_frames);
    dev_leave(prev);
    return st;
}
vv_dsp_status vv_dsp_stft_batch_inverse(vv_dsp_stft* h, const vv_dsp_cpx* spectra, vv_dsp_mem_space spectra_space,
                                        size_t batch, size_t frames, size_t spec_pitch, vv_dsp_real* out,
                                        vv_dsp_mem_space out_space, size_t n_out, size_t out_pitch, int normalise)
{
    const int prev = dev_enter(h);
    const vv_dsp_status st = batch_inverse_impl(h, spectra, spectra_space, batch, frames, spec_pitch, out, out_space, n_out, out_pitch,
                                                normalise);
    dev_leave(prev);
    return st;
}
vv_dsp_status vv_dsp_stft_shard_inverse(vv_dsp_stft* h, const vv_dsp_cpx* spectra, size_t local_frames, size_t halo_frames,
                                        int is_first, int is_last, vv_dsp_real* out, size_t n_out)
{
    const int prev = dev_enter(h);
    const vv_dsp_status st = shard_inverse_impl(h, spectra, local_frames, halo_frames, is_first, is_last, out, n_out);
    dev_leave(prev);
    return st;
}
int vv_dsp_stft_device(const vv_dsp_stft* h) { return h ? h->device : -1; }
void* vv_dsp_stft_get_stream(const vv_dsp_stft* h) { return h ? h->stream : NULL; }
const vv_dsp_real* vv_dsp_stft_window_ptr(const vv_dsp_stft* h) { return h ? h->win : NULL; }
