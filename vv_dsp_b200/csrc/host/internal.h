/* internal.h -- helpers shared between the C99 host translation units (not part of the ABI) */
#ifndef VVDSP_B200_HOST_INTERNAL_H
#define VVDSP_B200_HOST_INTERNAL_H
#include <stddef.h>
#include <stdlib.h>
#include "vv_dsp/vv_dsp_types.h"
#include "vvb200_cuda.h"

/* What every stream-bound handle (STFT, FIR, resampler, SOS) holds: the device it lives on, its stream and the size of a
 * staging chunk of HOST rows.  Handles embed it as their member `core`.  The functions below are static inline so that every
 * host unit compiles and links on its own, whichever set of units a library is built from. */
typedef struct handle_core {
    int device;                       /* the CUDA device the handle was created on: every entry point runs there */
    void* own_stream;
    void* stream;                     /* own_stream or the caller's */
    size_t stage_target;              /* staging bytes per chunk of HOST rows (per slot and direction for the STFT) */
} handle_core;

/* default bytes per staging chunk (and, for the STFT, per slot and direction).  e2e step of the headline STFT shape against
 * the chunk size, same box: 192 MB 45.8 ms, 96 MB 44.9, 48 MB 45.2, 24 MB 47.3 (the first chunk's upload and the last
 * chunk's download are not overlapped) */
#define STAGE_TARGET_BYTES ((size_t)96 << 20)

/* internal status (0 = success, 1..6 as vv_dsp_status, anything else a runtime failure) -> vv_dsp_status */
static inline vv_dsp_status vvdsp_internal_status(int st)
{
    if (st == 0) return VV_DSP_OK;
    if (st >= 1 && st <= 6 && st != 5) return (vv_dsp_status)st;
    return VV_DSP_ERROR_INTERNAL;
}

/* device ready -> current device -> own stream; returns the internal status (6 = no usable device) */
static inline int vvdsp_internal_core_init(handle_core* c)
{
    const char* env = getenv("VVB_STAGE_TARGET_BYTES");   /* a small staging size makes a modest batch span many chunks (tests) */
    int st = vvb_device_ready();                          /* 6 = no usable device: reported as UNSUPPORTED, never a CPU fallback */
    if (!st) st = vvb_get_device(&c->device);
    if (!st) st = vvb_stream_create(&c->own_stream);
    c->stream = c->own_stream;
    c->stage_target = (env && atol(env) > 0) ? (size_t)atol(env) : STAGE_TARGET_BYTES;
    return st;
}

static inline void vvdsp_internal_core_free(handle_core* c)
{
    if (c->own_stream) vvb_stream_destroy(c->own_stream);
}

/* A handle lives on the device that was current when it was created.  Entry points switch to it when the caller's
 * current device is another one and switch back before returning (multi-device callers: csrc/host/stream.c).  c may be
 * NULL; the return value goes to vvdsp_internal_leave. */
static inline int vvdsp_internal_enter(const handle_core* c)
{
    int cur = -1;
    if (!c || vvb_get_device(&cur) != 0 || cur == c->device) return -1;
    return vvb_set_device(c->device) == 0 ? cur : -1;
}

static inline void vvdsp_internal_leave(int prev) { if (prev >= 0) vvb_set_device(prev); }

/* NULL cuda_stream: the handle's own stream; c == NULL: VV_DSP_ERROR_NULL_POINTER */
static inline vv_dsp_status vvdsp_internal_set_stream(handle_core* c, void* cuda_stream)
{
    if (!c) return VV_DSP_ERROR_NULL_POINTER;
    c->stream = cuda_stream ? cuda_stream : c->own_stream;
    return VV_DSP_OK;
}

/* waits for the handle's stream, on the handle's device; c == NULL: VV_DSP_ERROR_NULL_POINTER */
static inline vv_dsp_status vvdsp_internal_synchronize(const handle_core* c)
{
    int prev, st;
    if (!c) return VV_DSP_ERROR_NULL_POINTER;
    prev = vvdsp_internal_enter(c);
    st = vvb_stream_sync(c->stream);
    vvdsp_internal_leave(prev);
    return vvdsp_internal_status(st);
}

/* grow a device scratch to `bytes`; work already enqueued may still use the old one */
static inline int vvdsp_internal_reserve(const handle_core* c, void** buf, size_t* have, size_t bytes)
{
    int st;
    if (bytes <= *have) return 0;
    st = vvb_stream_sync(c->stream);
    vvb_free(*buf); *buf = NULL; *have = 0;
    if (!st) st = vvb_malloc(buf, bytes);
    if (!st) *have = bytes;
    return st;
}

/* rows of `batch` (>= 1) per chunk, so that every chunk's HOST staging fits the target: at least 1 */
static inline size_t vvdsp_internal_chunk_rows(const handle_core* c, size_t batch, size_t bytes_per_row)
{
    size_t cs = batch;
    if (bytes_per_row && c->stage_target / bytes_per_row < cs) cs = c->stage_target / bytes_per_row;
    return cs < 1 ? 1 : cs;
}

/* a call that read or wrote a HOST buffer returns once the stream is done with it; the first error wins */
static inline int vvdsp_internal_finish(const handle_core* c, int st, int any_host)
{
    if (any_host) { int s2 = vvb_stream_sync(c->stream); if (!st) st = s2; }
    return st;
}

/* device-resident sparse mel filterbank: meta = lo | len | off per band, packed non-zero weights */
/* d_fw / d_fseg (may be NULL): lane schedules of the fused STFT -> log-mel kernel (f_segments segments per lane, power row of
 * f_prow floats, f_unit quads per segment), see mel.c build_fused_tables */
typedef struct mel_device { int* d_meta; float* d_w; size_t n_groups; float* d_fw; int* d_fseg; size_t f_segments, f_prow, f_unit; } mel_device;
int vvdsp_internal_mel_device_build(const float* dense_weights, size_t n_mels, size_t bins, void* stream, mel_device* md);
void vvdsp_internal_mel_device_free(mel_device* md);
/* log-mel of densely packed power rows on the device (the four-tap group kernels) */
int vvdsp_internal_logmel(const mel_device* md, const float* d_power, size_t frames, size_t bins, size_t n_mels, float eps,
                          float* d_out, void* stream);

/* MFCC tables on the device: cosine table [n_coeffs][n_mels] and lifter factors [n_coeffs] */
typedef struct mfcc_device { float* d_table; float* d_lifter; size_t n_mels, n_coeffs; float lifter; } mfcc_device;
int vvdsp_internal_mfcc_device_build(size_t n_mels, size_t n_coeffs, float lifter, void* stream, mfcc_device* md);
void vvdsp_internal_mfcc_device_free(mfcc_device* md);

#endif
