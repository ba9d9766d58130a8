/*
 * vvb200_cuda.h -- the thin C-ABI between the C99 host library (csrc/host/ *.c) and
 * the CUDA translation units (csrc/cuda/ *.cu).  Plain pointers and sizes only; no
 * CUDA or torch types cross it (streams travel as void*).  INTERNAL: consumers bind
 * vv_dsp/ *.h; this header exists so the host side stays pure C99.
 *
 * Every function returns 0 on success or a vv_dsp_status-compatible code
 * (4 = CUDA failure, text via vvb_last_error(); 6 = no device / unsupported size).
 */
#ifndef VVB200_CUDA_H
#define VVB200_CUDA_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vvb_engine vvb_engine;     /* device-resident STFT plan: tables + stream */
typedef struct vvb_fft_engine vvb_fft_engine; /* device-resident FFT plan */
typedef struct { float re, im; } vvb_cpx;

enum { VVB_OUT_COMPLEX = 0, VVB_OUT_POWER = 1, VVB_OUT_MAGNITUDE = 2 };
enum { VVB_PAD_ZERO = 0, VVB_PAD_REFLECT_CENTER = 1 };

const char* vvb_last_error(void);
unsigned long long vvb_kernel_launches(void);
int vvb_device_ready(void);   /* 0 when a usable sm_100-class device is current */
int vvb_fp32_peak(int packed, double* tflops);   /* diagnostics: measured FFMA (0) / FFMA2 (1) throughput */
int vvb_sm_clock_mhz(void* stream, double* mhz); /* diagnostics: SM clock right now (cycles per global-timer ns), after the work queued on stream */

/* ---- memory / stream plumbing (device = the engine's device) */
int vvb_malloc(void** dptr, size_t bytes);
int vvb_free(void* dptr);
int vvb_host_alloc(void** hptr, size_t bytes);   /* pinned */
int vvb_host_memory_is_device_visible(void);     /* 1: kernels may dereference vvb_host_alloc memory (unified addressing) */
int vvb_host_free(void* hptr);
int vvb_memcpy_h2d(void* dst, const void* src, size_t bytes, void* stream);
int vvb_memcpy_d2h(void* dst, const void* src, size_t bytes, void* stream);
int vvb_memcpy2d_h2d(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t height, void* stream);
int vvb_memcpy2d_d2h(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t height, void* stream);
int vvb_memcpy2d_d2d(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t height, void* stream);
int vvb_memset(void* dst, int value, size_t bytes, void* stream);
int vvb_stream_create(void** stream);
int vvb_stream_destroy(void* stream);
int vvb_stream_sync(void* stream);
int vvb_event_create(void** ev);
int vvb_event_destroy(void* ev);
int vvb_event_record(void* ev, void* stream);
int vvb_event_sync(void* ev);                    /* host waits for the recorded work */
int vvb_stream_wait_event(void* stream, void* ev);

/* ---- several devices in one process (frame-range sharding of one stream, csrc/host/stream.c) */
int vvb_device_count(int* count);
int vvb_get_device(int* device);
int vvb_set_device(int device);
int vvb_enable_peer_access(int device, int peer);   /* device may then read / write peer's memory; 0 also when already on or device == peer */
/* dst_left[i] = src_left[i], dst_right[i] = src_right[i], i < count, by a kernel on the current device; the sources may be
 * memory of a peer device (vvb_enable_peer_access) -- the halo exchange of stream.c.  Either pair may be NULL. */
int vvb_halo_gather(float* dst_left, const float* src_left, float* dst_right, const float* src_right, size_t count, void* stream);
int vvb_event_create_timing(void** ev);
int vvb_event_elapsed_ms(void* ev_start, void* ev_end, float* ms);
/* capture what is enqueued on `stream` between begin and end into an executable graph; 6 = not supported here */
int vvb_graph_capture_begin(void* stream);
int vvb_graph_capture_end(void* stream, void** graph_exec);
int vvb_graph_launch(void* graph_exec, void* stream);
int vvb_graph_destroy(void* graph_exec);

/* ---- STFT engine.  window: nfft host floats (the analysis == synthesis window). */
int vvb_engine_create(size_t nfft, size_t hop, const float* window, vvb_engine** out);
void vvb_engine_destroy(vvb_engine* e);
int vvb_engine_is_fast(const vvb_engine* e);   /* 1 if nfft has a Stockham kernel (pow2 256..8192) */

/* frames of every signal b < batch: frame f covers x[start .. start+nfft), start = f*hop
 * (VVB_PAD_ZERO, zeros outside [0,n)) or f*hop - nfft/2 with edge-inclusive reflection
 * (VVB_PAD_REFLECT_CENTER).  d_out: [batch][frames][out_pitch] of vvb_cpx (COMPLEX) or
 * float (POWER / MAGNITUDE), bins 0..nfft/2. */
int vvb_stft_forward(vvb_engine* e, const float* d_x, size_t batch, size_t n, size_t x_pitch, size_t frames,
                     int pad_mode, int out_kind, void* d_out, size_t out_pitch, void* stream);
/* STFT -> log-mel in one kernel (no power spectrogram in HBM): d_out = [batch][frames][n_mels].  d_mel_w / d_mel_seg: the lane
 * schedules built by the host (csrc/host/mel.c, build_fused_tables): mel_segments segments of mel_unit quads per lane (4; the
 * generic kernel also takes 2), power
 * row of mel_prow floats.  Plans: fft_size 2048 with hop N/8, N/4, N/2 (marching kernel) and every Stockham size <= 1024 with
 * any hop (generic kernel).  Returns 6 when the plan or the schedule has no fused kernel. */
int vvb_stft_forward_logmel_ok(const vvb_engine* e, size_t mel_segments, size_t mel_prow, size_t mel_unit, size_t n_mels);
int vvb_stft_forward_logmel(vvb_engine* e, const float* d_x, size_t batch, size_t n, size_t x_pitch, size_t frames, int pad_mode,
                            const float* d_mel_w, const int* d_mel_seg, size_t mel_segments, size_t mel_prow, size_t mel_unit,
                            size_t n_mels, float eps, float* d_out, void* stream);

/* overlap-add synthesis of d_spec [batch][frames][spec_pitch] into d_y [batch][y_pitch]
 * (n_out valid samples each).  d_inv_norm: table set built by vvb_norm_tables_build, or
 * NULL for the raw (un-normalised) sum. */
int vvb_stft_inverse(vvb_engine* e, const vvb_cpx* d_spec, size_t batch, size_t frames, size_t spec_pitch,
                     float* d_y, size_t n_out, size_t y_pitch, const float* d_inv_norm, void* stream);

/* One frame-range shard of a longer stream: d_spec [frames][spec_pitch] = halo_frames rows that belong to the previous
 * shard (synthesised only for their overlap into this shard's samples) followed by the shard's own frames; d_y receives
 * the n_out samples starting at the first own frame's position.  head_edge / tail_edge: the shard starts / ends at the
 * true start / end of the stream (edge normalisation; the trailing nfft-hop samples are emitted only at the true end).
 * Shards concatenate to the bit-identical result of vvb_stft_inverse on the whole stream.  6 if (nfft, hop) has no
 * marching kernel. */
int vvb_stft_inverse_shard(vvb_engine* e, const vvb_cpx* d_spec, size_t frames, size_t halo_frames, int head_edge,
                           int tail_edge, size_t spec_pitch, float* d_y, size_t n_out, const float* d_inv_norm, void* stream);

/* windowed synthesis frames without overlap-add: d_frames [count][nfft] =
 * Re(IDFT(spec)/nfft) * w  (what vv_dsp_stft_reconstruct adds into out_add). */
int vvb_stft_inverse_frames(vvb_engine* e, const vvb_cpx* d_spec, size_t count, size_t spec_pitch,
                            float* d_frames, void* stream);

/* ---- log-mel: d_out[f][m] = logf(sum_{k in [lo[m], lo[m]+len[m])} d_power[f][k] * w[off[m] + k - lo[m]] + eps).
 * d_meta: int[3*n_mels] = lo | len | off, followed by the slot-ordered group tables csrc/host/mel.c builds;
 * d_w: packed non-zero weights, ascending k per band, followed by the same runs in zero-padded groups of four.
 * n_groups: number of four-tap groups in those tables (0 = tables absent: only the plain kernel is used). */
int vvb_logmel(const float* d_power, size_t frames, size_t bins, size_t power_pitch, const int* d_meta, const float* d_w,
               size_t n_mels, size_t n_groups, float eps, float* d_out, void* stream);

/* ---- MFCC: d_out[f][k] = d_lifter[k] * sum_n d_logmel[f][n] * d_table[k*n_mels + n], n ascending */
int vvb_mfcc(const float* d_logmel, size_t frames, size_t n_mels, size_t n_coeffs, const float* d_table,
             const float* d_lifter, float* d_out, void* stream);

/* ---- PCM decode: interleaved little-endian samples (format 16/24/32 = signed PCM, -32 = float32) -> planar float32 */
int vvb_pcm_to_planar(const void* d_interleaved, int format, size_t num_samples, size_t channels, float* d_planar,
                      size_t pitch, void* stream);

/* ---- FFT engine (plan API): type 0 C2C, 1 R2C, 2 C2R; dir +1 / -1 */
int vvb_fft_engine_create(size_t n, int type, int dir, vvb_fft_engine** out);
void vvb_fft_engine_destroy(vvb_fft_engine* e);
int vvb_fft_engine_is_single_kernel(const vvb_fft_engine* e);   /* one kernel that reads its input once */
int vvb_fft_exec(vvb_fft_engine* e, const void* d_in, void* d_out, size_t batch, void* stream);

/* ---- FIR by overlap-save (csrc/host/fir.c): m = transform size, a power of two in [128, 8192] */
typedef struct vvb_fir_engine vvb_fir_engine;
int vvb_fir_engine_create(size_t m, vvb_fir_engine** out);
void vvb_fir_engine_destroy(vvb_fir_engine* e);
/* filter spectra: d_spec [filters][parts][m] = FFT_m of the zero-padded partition h_f[p lp .. (p+1) lp) (taps beyond
 * num_taps read as 0), times 1/m.  d_h: [filters][h_pitch] floats. */
int vvb_fir_spectra(vvb_fir_engine* e, const float* d_h, size_t filters, size_t h_pitch, size_t num_taps, size_t lp,
                    size_t parts, vvb_cpx* d_spec, void* stream);
/* d_y[b][i] = sum_j h_b[j] x_b[i - j], i < n_out (0 from n + num_taps - 1 on), by `parts` passes of the overlap-save
 * kernel in ascending partition order (pass p delayed by p lp, passes after the first add into d_y).  d_spec as built by
 * vvb_fir_spectra; spec_stride: complex values from one signal's spectra to the next's (0: one filter for all). */
int vvb_fir_filter(vvb_fir_engine* e, const vvb_cpx* d_spec, size_t spec_stride, size_t num_taps, size_t lp, size_t parts,
                   const float* d_x, size_t batch, size_t n, size_t x_pitch, float* d_y, size_t n_out, size_t y_pitch,
                   void* stream);

/* ---- polyphase resampling (csrc/host/resample.c): up, down coprime; d_bank [taps_per_phase][up] (phase-minor) holds
 * h[phi + j up], the filter already scaled by up, 0 past its end; half = (num_taps - 1) / 2.
 *   d_y[b][m] = sum_{j < T} d_bank[j][phi] x_b[i0 - j],  q0 = m down + half, phi = q0 mod up, i0 = q0 div up,  m < n_out,
 * x_b = 0 outside [0, n); every output sums its products in one fixed order, whatever the batch. */
int vvb_resample_poly(const float* d_bank, size_t up, size_t down, size_t taps_per_phase, size_t half,
                      const float* d_x, size_t batch, size_t n, size_t x_pitch, float* d_y, size_t n_out, size_t y_pitch,
                      void* stream);

/* ---- IIR second-order sections (csrc/host/sos.c).  A tile is VVB_IIR_THREADS runs of VVB_IIR_RUN samples.
 * d_table [S][VVB_IIR_TABLE] (double): b0 b1 b2 a1 a2 0 0 0 (float32 values), then A^(RUN 2^d) row-major for d < VVB_IIR_LEVELS, A = [[-a1, 1],
 * [-a2, 0]].  d_phi [2S][2S]: the cascade's state transition over one segment (state index 2 s + c).  The kernels run
 * the cascade over the virtual rows v_b[j], 0 <= j < nv:
 *   VVB_IIR_IN_PLAIN: x_b[j] (nv = n);  VVB_IIR_IN_EXT: x_b padded by `pad` samples at both ends by `padtype` (scipy's
 *   odd_ext / even_ext / const_ext; nv = n + 2 pad);  VVB_IIR_IN_REV: x_b[nv - 1 - j] (x rows of nv samples).
 * and store output j at y_b[j] (VVB_IIR_OUT_DIRECT) or at y_b[nv - 1 - j - pad] when that lies in [0, n)
 * (VVB_IIR_OUT_REVTRIM).  The entering state of section s is zi[s zi_sstride + b zi_rstride + c] (0 when zi is NULL),
 * times v_b[0] when zi_scale_first; the state after the last sample goes to zf[s zf_sstride + 2 b + c] unless zf is NULL.
 * Rows longer than `segment` samples take three launches and need d_seg [batch][ceil(nv / segment)][2S] of scratch. */
#define VVB_IIR_THREADS 256
#define VVB_IIR_RUN 16
#define VVB_IIR_LEVELS 8             /* log2(VVB_IIR_THREADS) */
#define VVB_IIR_TABLE (8 + 4 * VVB_IIR_LEVELS)
enum { VVB_IIR_IN_PLAIN = 0, VVB_IIR_IN_EXT = 1, VVB_IIR_IN_REV = 2 };
enum { VVB_IIR_OUT_DIRECT = 0, VVB_IIR_OUT_REVTRIM = 1 };
enum { VVB_IIR_PAD_ODD = 1, VVB_IIR_PAD_EVEN = 2, VVB_IIR_PAD_CONSTANT = 3 };   /* the values of VV_DSP_PAD_* */
typedef struct {
    const double* d_table; const float* d_phi; size_t sections, segment;
    const float* x; size_t x_pitch, n; int in_mode, padtype; size_t pad, nv;
    float* y; size_t y_pitch; int out_mode;
    const float* zi; size_t zi_sstride, zi_rstride; int zi_scale_first;
    float* zf; size_t zf_sstride;
    float* d_seg;
    size_t batch;
} vvb_iir_call;
int vvb_iir_sos(const vvb_iir_call* c, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* VVB200_CUDA_H */
