/*
 * vv_dsp/b200.h -- batched, device-resident extension of the STFT handle API.
 *
 * NOT in the reference: its API is one host frame per call (include/vv_dsp/spectral/
 * stft.h:30-56), which cannot express BASELINE's batched workloads.  These entry
 * points are defined so that, frame for frame, they equal looping the per-frame API
 * the way the reference's own callers do:
 *   analysis   tools/dump_stft_roundtrip.c:44-45   process(h, x + f*hop, spec)
 *   synthesis  tools/dump_stft_roundtrip.c:46-54   reconstruct(h, spec, recon + f*hop,
 *              norm + f*hop); y[i] = norm[i] > 1e-12 ? recon[i]/norm[i] : 0
 *
 * Layouts (row-major, contiguous unless a pitch is given):
 *   signals   [batch][signal_pitch]         float32, n valid samples per row
 *   spectra   [batch][frames][spec_pitch]   bins k = 0..fft_size/2 (fft_size/2+1 per
 *             frame, the Hermitian half; X[fft_size-k] = conj X[k] is implied).
 *             vv_dsp_cpx for COMPLEX, float32 for POWER (re^2+im^2, what
 *             include/vv_dsp/features/mel.h:74-77 consumes) and MAGNITUDE (sqrtf).
 *   A pitch of 0 means dense (n, resp. fft_size/2+1).  No padding is ever added
 *   behind the caller's back.
 *
 * Memory spaces: every buffer argument carries its own space.  HOST buffers are
 * caller-owned host memory (pinned memory makes the copies asynchronous and
 * overlapped); DEVICE buffers are CUDA device pointers on the handle's device.
 * If every buffer of a call is DEVICE the call only enqueues work on the handle's
 * stream (vv_dsp_stft_set_stream) and returns; otherwise it returns after the
 * results are in host memory.
 *
 * Every fft_size >= 1 is served on the GPU: powers of two in [256, 8192] by the fused
 * Stockham kernels (the throughput path), 320 / 400 / 480 / 640 by mixed-radix Stockham
 * kernels, other sizes in [32, 4096] by the fused
 * chirp-z kernel, larger ones up to 2^22 by the chirp-z pipeline on four-step plans, the
 * rest by direct-DFT kernels (correct, O(n^2) like the reference's path for those
 * sizes).  There is no CPU fallback anywhere.
 */
#ifndef VV_DSP_B200_H
#define VV_DSP_B200_H

#include <stddef.h>
#include "vv_dsp/vv_dsp_types.h"
#include "vv_dsp/spectral/stft.h"
#include "vv_dsp/spectral/fft.h"
#include "vv_dsp/features/mel.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef enum vv_dsp_mem_space {
    VV_DSP_MEM_HOST = 0,
    VV_DSP_MEM_DEVICE = 1
} vv_dsp_mem_space;

/* The reference's four coexisting frame-count rules (SURVEY.md section 8a):
 *   VALID        n < fft ? 0 : 1 + (n-fft)/hop          src/core/framing.c:66-67, dump tool loop
 *   SPECTROGRAM  n < fft ? 1 : 1 + (n-fft+hop)/hop      src/spectral/stft.c:119 (zero-padded tail)
 *   PADDED_TAIL  frames while start+fft <= n+(fft-hop)  tests/spectral_tests.c:101 (zero-padded tail)
 *   CENTER       ceil(n/hop), frame centred at f*hop, edge-inclusive reflect padding
 *                src/core/framing.c:61-63,21-56,86-102 */
typedef enum vv_dsp_frame_convention {
    VV_DSP_FRAMES_VALID = 0,
    VV_DSP_FRAMES_SPECTROGRAM = 1,
    VV_DSP_FRAMES_PADDED_TAIL = 2,
    VV_DSP_FRAMES_CENTER = 3
} vv_dsp_frame_convention;

typedef enum vv_dsp_spec_kind {
    VV_DSP_SPEC_COMPLEX = 0,
    VV_DSP_SPEC_POWER = 1,
    VV_DSP_SPEC_MAGNITUDE = 2
} vv_dsp_spec_kind;

/* frame count for a signal of n samples under a convention; fft_size/2+1 */
size_t vv_dsp_stft_num_frames(const vv_dsp_stft* h, size_t n, vv_dsp_frame_convention convention);
size_t vv_dsp_stft_num_bins(const vv_dsp_stft* h);

/* Bind the handle to a caller-owned cudaStream_t.  NULL = the handle's own (non-blocking) stream;
 * to address CUDA's default streams pass cudaStreamLegacy ((void*)1) or cudaStreamPerThread ((void*)2). */
vv_dsp_status vv_dsp_stft_set_stream(vv_dsp_stft* h, void* cuda_stream);
/* Block until everything the handle has enqueued (its stream and its staging streams) has finished. */
vv_dsp_status vv_dsp_stft_synchronize(vv_dsp_stft* h);
/* Stream-ordered mode for calls with HOST buffers (off by default).  When enabled such calls only
 * enqueue their copies and kernels and return, like cudaMemcpyAsync: host buffers (pin them) must stay
 * valid and untouched until vv_dsp_stft_synchronize().  The library orders a call that reads a DEVICE
 * buffer after the earlier stream-ordered call of the same handle that produced it, chunk by chunk,
 * so the host->device copies of an analysis call overlap the device->host copies of the synthesis call
 * that follows it (PCIe is full duplex).  Calls whose buffers are all DEVICE are not ordered against
 * stream-ordered calls; synchronize in between. */
vv_dsp_status vv_dsp_stft_set_async(vv_dsp_stft* h, int enable);

/* Analysis of `batch` signals: framing + window + real FFT (+ |X|^2 or |X|) fused in
 * one kernel.  *out_frames receives the per-signal frame count (may be NULL). */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_batch_forward(
    vv_dsp_stft* h,
    const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch, size_t n, size_t signal_pitch,
    vv_dsp_frame_convention convention, vv_dsp_spec_kind kind,
    void* out, vv_dsp_mem_space out_space, size_t spec_pitch, size_t* out_frames);

/* The same analysis fed with the samples as they sit in a WAV data chunk: HOST rows of mono little-endian PCM
 * (format 16 / 24 / 32) or IEEE float32 (format -32), signal_pitch in SAMPLES (0 = n).  Chunks are uploaded undecoded (2 or 3
 * bytes per sample instead of 4) and converted on the device with the scaling of the reference's WAV reader
 * (src/audio/wav.c:458-521: sample * 2^-15 / 2^-23 / 2^-31), so the spectra equal those of vv_dsp_stft_batch_forward on the
 * decoded floats bit for bit.  Follows vv_dsp_stft_set_async like the float call. */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_batch_forward_pcm(
    vv_dsp_stft* h,
    const void* pcm, int format, size_t batch, size_t n, size_t signal_pitch,
    vv_dsp_frame_convention convention, vv_dsp_spec_kind kind,
    void* out, vv_dsp_mem_space out_space, size_t spec_pitch, size_t* out_frames);

/* Synthesis: inverse real FFT + synthesis window + overlap-add of `frames` frames per
 * signal at positions f*hop, into n_out samples per signal (positions >= n_out are
 * dropped like vv_dsp_overlap_add does, src/core/framing.c:139-145; positions no
 * frame covers are 0).  normalise != 0 divides by the accumulated sum of w^2 with the
 * callers' guard (norm > 1e-12 ? y/norm : 0); normalise == 0 returns the raw sum. */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_batch_inverse(
    vv_dsp_stft* h,
    const vv_dsp_cpx* spectra, vv_dsp_mem_space spectra_space, size_t batch, size_t frames, size_t spec_pitch,
    vv_dsp_real* out, vv_dsp_mem_space out_space, size_t n_out, size_t out_pitch, int normalise);

/* One-signal host convenience: ISTFT with window-sum normalisation
 * (= reconstruct-all-frames + the caller-side divide of tools/dump_stft_roundtrip.c:50-54). */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_istft(vv_dsp_stft* h, const vv_dsp_cpx* half_spectra, size_t frames,
                                                 vv_dsp_real* out, size_t n_out);

/* ---------------------------------------------------------------------------------------------------------------
 * ONE long stream sharded by frame range over several GPUs (SURVEY.md section 8e, BASELINE config 4).
 *
 * Shard d owns the valid frames [F d / G, F (d+1) / G) of the n-sample stream and the samples [f0 hop, f1 hop)
 * (the last shard: up to n).  Frames of different shards interact only through the overlap of nfft - hop samples at
 * a boundary, and both directions resolve it with a HALO that is (nfft - hop) samples long:
 *   analysis   a shard's local signal is [left halo | owned samples | right halo]; the right halo lets its last
 *              frames reach into the next shard's samples, the left halo makes it ALSO compute the K - 1 = nfft/hop - 1
 *              frames before its own first frame.  Local spectra: [K - 1 halo frames | own frames][bins].
 *   synthesis  the halo frames are synthesised only for their overlap into the shard's first nfft - hop samples
 *              (exactly what a warp of the batched kernel does when its range starts mid-signal); nothing is
 *              exchanged, every output sample is the same ascending-frame sum as in the unsharded call, and the
 *              shards' outputs CONCATENATE to the bit-identical result of vv_dsp_stft_batch_inverse on the whole
 *              stream.  A frame-wise modification of the spectra must be applied to the halo rows as well.
 * The only communication is the two sample halos per boundary (nfft - hop floats each way, 12 KB at 4096 / 1024),
 * copied device to device over NVLink.  Needs hop | fft_size, fft_size in {512 ... 8192} and hop in {N/8, N/4, N/2}.
 * (Bit-identical to the unsharded call for fft_size >= 2048, where both run the same kernel; at 512 / 1024 the
 * unsharded call pairs frames two per transform, so the two agree to rounding -- and any two shard counts bit for bit.)
 * ------------------------------------------------------------------------------------------------------------- */

/* Synthesis of one shard, building block of the multi-process flavour (one process per GPU, vv_dsp_b200/sharding.py):
 * spectra = DEVICE [local_frames][fft_size/2+1] holding halo_frames (0 for the first shard, else fft_size/hop - 1) rows
 * of the previous shard followed by the shard's own frames; out = DEVICE, n_out owned samples, normalised.
 * Enqueued on the handle's stream.  The analysis of a shard is vv_dsp_stft_batch_forward (VALID) of its local signal. */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_shard_inverse(vv_dsp_stft* h, const vv_dsp_cpx* spectra, size_t local_frames,
                                                         size_t halo_frames, int is_first, int is_last,
                                                         vv_dsp_real* out, size_t n_out);
/* the CUDA device a handle lives on (every entry point switches to it and back), and the stream it enqueues on */
int vv_dsp_stft_device(const vv_dsp_stft* h);
void* vv_dsp_stft_get_stream(const vv_dsp_stft* h);

/* The single-process flavour: one handle drives `num_devices` GPUs (device_ids NULL = 0 .. num_devices-1; the same id
 * may appear more than once, which shards the stream on one GPU).  All buffers are owned by the handle and resident
 * on the devices; per step the library enqueues, on each device's own stream, the two halo copies from the
 * neighbouring devices (peer to peer), the fused analysis kernel and the fused synthesis kernel -- replayed as one
 * CUDA graph per device once the first step has run.  No call blocks except upload / download / synchronize. */
typedef struct vv_dsp_stft_stream vv_dsp_stft_stream;
typedef struct vv_dsp_stft_stream_shard {
    int device;
    size_t frame0, frame1;          /* own frames of the stream */
    size_t sample0, sample1;        /* own samples of the stream */
    size_t halo_frames;             /* leading rows of `spectra` that belong to the previous shard */
    size_t left_halo, right_halo;   /* samples in front of / behind the owned samples in `signal` */
    vv_dsp_real* signal;            /* DEVICE [left_halo + (sample1 - sample0) + right_halo] */
    vv_dsp_cpx* spectra;            /* DEVICE [halo_frames + frame1 - frame0][fft_size/2+1] */
    vv_dsp_real* output;            /* DEVICE [sample1 - sample0] */
    void* cuda_stream;              /* the stream the shard's work is enqueued on */
} vv_dsp_stft_stream_shard;

VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_stream_create(const vv_dsp_stft_params* params, size_t n, size_t num_devices,
                                                         const int* device_ids, vv_dsp_stft_stream** out);
vv_dsp_status vv_dsp_stft_stream_destroy(vv_dsp_stft_stream* s);
size_t vv_dsp_stft_stream_num_frames(const vv_dsp_stft_stream* s);
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_stream_get_shard(const vv_dsp_stft_stream* s, size_t d, vv_dsp_stft_stream_shard* out);
/* host signal [n] -> the shards' owned samples (synchronous); the halos are filled by every analysis step */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_stream_upload(vv_dsp_stft_stream* s, const vv_dsp_real* signal);
/* halo exchange + analysis of every shard (COMPLEX spectra into the shards' buffers); enqueue only */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_stream_forward(vv_dsp_stft_stream* s);
/* normalised synthesis of every shard from its spectra buffer into its output buffer; enqueue only */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_stream_inverse(vv_dsp_stft_stream* s);
/* forward + inverse as ONE enqueue per device (a captured CUDA graph after the first call) */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_stream_roundtrip(vv_dsp_stft_stream* s);
vv_dsp_status vv_dsp_stft_stream_synchronize(vv_dsp_stft_stream* s);
/* gather to host (synchronous): out [n] samples; spectra [num_frames][fft_size/2+1] without the halo rows */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_stream_download(vv_dsp_stft_stream* s, vv_dsp_real* out);
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_stream_download_spectra(vv_dsp_stft_stream* s, vv_dsp_cpx* spectra);
/* device-timed benchmark of `steps` roundtrip steps after `warmup` untimed ones: every device's stream is timed with
 * its own pair of CUDA events between two full synchronisations; *ms_per_step = the slowest device's time / steps */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_stream_time_roundtrip(vv_dsp_stft_stream* s, size_t warmup, size_t steps, double* ms_per_step);

/* STFT -> power -> mel filterbank -> log for a whole batch (SURVEY.md section 8f, rank 2):
 * out[b][f][m] = logf(sum_k |X_bf[k]|^2 W[m][k] + log_epsilon), i.e. vv_dsp_compute_log_mel_spectrogram
 * applied to the power output of vv_dsp_stft_batch_forward.  filterbank_weights: HOST, dense
 * [n_mels][fft_size/2+1] as produced by vv_dsp_mel_filterbank_create.  out: [batch][frames][n_mels]
 * float32.  ONE kernel from samples to log-mel rows (no power spectrogram in device memory) at fft_size 2048 with hop N/8, N/4,
 * N/2 and at every Stockham size <= 1024 (256 / 512 / 1024, 320 / 400 / 480 / 640) with any hop; elsewhere two kernels (power,
 * then an HBM-bound log-mel kernel) chained per chunk of signals through a bounded device scratch.  Same rows either way. */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_batch_logmel(
    vv_dsp_stft* h,
    const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch, size_t n, size_t signal_pitch,
    vv_dsp_frame_convention convention,
    const vv_dsp_real* filterbank_weights, size_t n_mels, vv_dsp_real log_epsilon,
    vv_dsp_real* out, vv_dsp_mem_space out_space, size_t* out_frames);

/* vv_dsp_stft_batch_logmel fed with HOST rows of WAV samples (format 16 / 24 / 32 PCM or -32 float32, mono, signal_pitch in
 * samples): uploaded undecoded, converted on the device like vv_dsp_stft_batch_forward_pcm; the same log-mel rows bit for bit. */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_batch_logmel_pcm(
    vv_dsp_stft* h, const void* pcm, int format, size_t batch, size_t n, size_t signal_pitch,
    vv_dsp_frame_convention convention, const vv_dsp_real* filterbank_weights, size_t n_mels, vv_dsp_real log_epsilon,
    vv_dsp_real* out, vv_dsp_mem_space out_space, size_t* out_frames);

/* The same chain followed by the MFCC stage of vv_dsp_mfcc (unnormalised DCT-II of every log-mel frame, first
 * num_mfcc_coeffs kept, liftering when lifter_coeff > 0): out is [batch][frames][num_mfcc_coeffs].  Frame for
 * frame equal to vv_dsp_mfcc(vv_dsp_compute_log_mel_spectrogram(|process|^2)). */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_stft_batch_mfcc(
    vv_dsp_stft* h,
    const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch, size_t n, size_t signal_pitch,
    vv_dsp_frame_convention convention,
    const vv_dsp_real* filterbank_weights, size_t n_mels, vv_dsp_real log_epsilon,
    size_t num_mfcc_coeffs, vv_dsp_real lifter_coeff,
    vv_dsp_real* out, vv_dsp_mem_space out_space, size_t* out_frames);

/* Many transforms through one plan (SURVEY.md section 8f, rank 1): `batch` contiguous transforms,
 * C2C: cpx[batch][n] -> cpx[batch][n];  R2C: real[batch][n] -> cpx[batch][n/2+1];  C2R: the reverse.
 * Same conventions as vv_dsp_fft_execute (forward unscaled, backward 1/n, R2C Nyquist real, C2R =
 * Re of the inverse of the Hermitian extension).  DEVICE buffers: enqueued on `cuda_stream` (NULL = the
 * plan's stream) and not awaited; any HOST buffer: staged and synchronous.  in == out is allowed for C2C
 * with n in [32, 4096] or a power of two up to 8192 (not for the direct-DFT sizes). */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_fft_execute_batch(const vv_dsp_fft_plan* plan, const void* in,
                                                        vv_dsp_mem_space in_space, void* out,
                                                        vv_dsp_mem_space out_space, size_t batch, void* cuda_stream);

/* WAV sample decode on the device (SURVEY.md section 8f, rank 4): interleaved little-endian samples, as they
 * sit in the data chunk of a WAV file, to planar float32 [channels][planar_pitch] with the scaling of the
 * reference's reader (src/audio/wav.c:458-521): format 16 / 24 / 32 = signed PCM times 2^-15 / 2^-23 / 2^-31,
 * format -32 = IEEE float32.  planar_pitch 0 = num_samples.  A HOST input is staged (the upload carries 2 or
 * 3 bytes per sample instead of 4); DEVICE in and out: enqueued on cuda_stream and not awaited. */
VV_DSP_NODISCARD vv_dsp_status vv_dsp_b200_pcm_to_planar(const void* interleaved, vv_dsp_mem_space in_space, int format,
                                                         size_t num_samples, size_t channels, vv_dsp_real* planar,
                                                         vv_dsp_mem_space out_space, size_t planar_pitch, void* cuda_stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Batched FIR filtering by FFT convolution (overlap-save), one fused kernel per filter partition.
 *
 *   out[b][i] = sum_{j < num_taps} h_b[j] x_b[i - j],   0 <= i < n_out,
 * where x_b[k] = 0 outside [0, n) and h_b = filters[num_filters == 1 ? 0 : b] (rows of num_taps taps).
 * n_out = n is causal FIR filtering (scipy.signal.lfilter(h, 1, x)); n_out = n + num_taps - 1 is the full linear
 * convolution; samples beyond that are 0.  Pitches (in elements) of 0 mean dense.  Memory spaces as above: if every
 * buffer is DEVICE the call only enqueues on the handle's stream, otherwise it returns once the results are in host
 * memory.  `out` must not overlap `signals`; an identical base pointer is rejected with VV_DSP_ERROR_UNSUPPORTED.
 *
 * Plan: a handle is created for a tap count M and picks, as a pure function of M, a complex transform size
 * N in {128, 256, ..., 8192} and P partitions of Lp = ceil(M / P) <= N taps: the smallest P N log2(N) / (N - Lp + 1)
 * (transform work per output sample), ties to the smaller N and then the fewer partitions.  That gives N = 128 for
 * M <= 29, 256 to M = 52, 512 to 94, 1024 to 171, 2048 to 316, 4096 to 586 and 8192 from M = 587; one partition up to
 * M = 5462, two from 5463, 12 at 48 000.  Every M >= 1 runs on the GPU: partition p (taps p Lp ... (p+1) Lp) is one
 * pass of the kernel delayed by p Lp samples that adds into `out`, in ascending p, so results are deterministic.
 * The filter spectra are built on the device in every call (filters change per batch in augmentation); per-signal
 * filters are processed in chunks of signals whose spectra fit a bounded scratch of the handle.
 *
 * Status: NULL pointer -> VV_DSP_ERROR_NULL_POINTER; num_taps == 0 (or above 2^31 - 1), num_filters not in {1, batch}
 * or a pitch smaller than its row -> VV_DSP_ERROR_INVALID_SIZE; a bad memory space -> VV_DSP_ERROR_OUT_OF_RANGE;
 * out == signals -> VV_DSP_ERROR_UNSUPPORTED; batch == 0 or n_out == 0 -> VV_DSP_OK with no work; CUDA failures
 * -> VV_DSP_ERROR_INTERNAL (no usable device at creation: VV_DSP_ERROR_UNSUPPORTED).
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct vv_dsp_fir vv_dsp_fir;
VV_DSP_NODISCARD vv_dsp_status vv_dsp_fir_create(size_t num_taps, vv_dsp_fir** out);
vv_dsp_status vv_dsp_fir_destroy(vv_dsp_fir* f);
/* same rules as vv_dsp_stft_set_stream (NULL = the handle's own stream) */
vv_dsp_status vv_dsp_fir_set_stream(vv_dsp_fir* f, void* cuda_stream);
vv_dsp_status vv_dsp_fir_synchronize(vv_dsp_fir* f);
/* the transform size N and the number of filter partitions P (passes) the handle uses */
vv_dsp_status vv_dsp_fir_get_config(const vv_dsp_fir* f, size_t* fft_size, size_t* partitions);
VV_DSP_NODISCARD vv_dsp_status vv_dsp_fir_filter_batch(
    vv_dsp_fir* f,
    const vv_dsp_real* filters, vv_dsp_mem_space filters_space, size_t num_filters, size_t filter_pitch,
    const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch, size_t n, size_t signal_pitch,
    vv_dsp_real* out, vv_dsp_mem_space out_space, size_t n_out, size_t out_pitch);

/* ---------------------------------------------------------------------------------------------------------------
 * Batched rational-ratio resampling by a polyphase FIR: scipy.signal.resample_poly(x, up, down, window=..., padtype=
 * 'constant') row by row.  up / down are first divided by their gcd.  With K taps w, h = up w and half = (K - 1) / 2:
 *
 *   y[m] = sum_k h[k] xu[m down + half - k],   0 <= m < n_out = ceil(n up / down),
 *   xu[q] = x[q / up] if up divides q and 0 <= q / up < n, else 0.
 *
 * taps == NULL (num_taps 0) designs scipy's default filter, firwin(2 half + 1, 1 / max(up, down), window=('kaiser', 5.0))
 * with half = 10 max(up, down), in double; otherwise the num_taps host floats are the window argument of resample_poly.
 * The bank of T = ceil(K / up) taps per phase is rounded to float32 once and lives on the device.  up == down == 1 after
 * reduction copies the input bit for bit and ignores the filter.  Every output sums its T products in one fixed order,
 * so a signal gives the same bits alone or inside any batch, from HOST or DEVICE buffers.
 *
 * Pitches (in elements) of 0 mean dense.  Memory spaces as above: if both buffers are DEVICE the call only enqueues on
 * the handle's stream, otherwise it returns once the results are in host memory.  `out` must not overlap `signals`; an
 * identical base pointer is rejected with VV_DSP_ERROR_UNSUPPORTED.  *out_len receives n_out.
 *
 * Status: NULL handle / signals / out / out_len, or taps == NULL with num_taps > 0 -> VV_DSP_ERROR_NULL_POINTER; up or
 * down == 0, taps with num_taps == 0, a bank up T above 65 536 taps, up or down above 2^31 - 1 after reduction, a pitch
 * smaller than its row or n up >= 2^62 -> VV_DSP_ERROR_INVALID_SIZE; a bad memory space -> VV_DSP_ERROR_OUT_OF_RANGE;
 * out == signals -> VV_DSP_ERROR_UNSUPPORTED; batch == 0 or n == 0 -> VV_DSP_OK with no work; CUDA failures ->
 * VV_DSP_ERROR_INTERNAL (no usable device at creation: VV_DSP_ERROR_UNSUPPORTED).
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct vv_dsp_resample_poly vv_dsp_resample_poly;
VV_DSP_NODISCARD vv_dsp_status vv_dsp_resample_poly_create(size_t up, size_t down, const vv_dsp_real* taps /* HOST or NULL */,
                                                           size_t num_taps, vv_dsp_resample_poly** out);
vv_dsp_status vv_dsp_resample_poly_destroy(vv_dsp_resample_poly* r);
/* same rules as vv_dsp_stft_set_stream (NULL = the handle's own stream) */
vv_dsp_status vv_dsp_resample_poly_set_stream(vv_dsp_resample_poly* r, void* cuda_stream);
vv_dsp_status vv_dsp_resample_poly_synchronize(vv_dsp_resample_poly* r);
/* the reduced up / down, the filter length K and the taps per phase T */
vv_dsp_status vv_dsp_resample_poly_get_config(const vv_dsp_resample_poly* r, size_t* up, size_t* down, size_t* num_taps,
                                              size_t* taps_per_phase);
/* ceil(n up / down); 0 for a NULL handle */
size_t vv_dsp_resample_poly_output_length(const vv_dsp_resample_poly* r, size_t n);
VV_DSP_NODISCARD vv_dsp_status vv_dsp_resample_poly_batch(
    vv_dsp_resample_poly* r,
    const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch, size_t n, size_t signal_pitch,
    vv_dsp_real* out, vv_dsp_mem_space out_space, size_t out_pitch, size_t* out_len);

/* ---------------------------------------------------------------------------------------------------------------
 * Batched IIR filtering by a cascade of S second-order sections: scipy.signal.sosfilt / sosfiltfilt row by row.  Row s
 * of sos[S][6] is (b0, b1, b2, 1, a1, a2); every section runs transposed direct form II in scipy's order,
 *
 *   y = b0 u + z0,   z0 <- b1 u - a1 y + z1,   z1 <- b2 u - a2 y,   (the input u of section s + 1 is y of section s)
 *
 * filter:   sosfilt(sos, x, zi=zi) row by row.  zi and zf have scipy's layout [S][batch][2] (row pitch 2, section
 *           pitch 2 batch); zi == NULL is the zero state, zf == NULL does not write zf.  zf may be zi.
 * filtfilt: sosfiltfilt(sos, x, padtype, padlen) row by row.  padtype is VV_DSP_PAD_NONE (padlen is then 0), _ODD,
 *           _EVEN or _CONSTANT; padlen == (size_t)-1 is scipy's default 3 (2S + 1 - min(#{b2 == 0}, #{a2 == 0})).  The
 *           forward pass runs over the padded signal from sosfilt_zi(sos) x_ext[0], the backward pass from
 *           sosfilt_zi(sos) y_fwd[last], and the result is trimmed by padlen at both ends.  The padding is an index rule
 *           of the kernel's loads; the forward pass writes n + 2 padlen floats per row to a device scratch of the handle.
 *
 * Arithmetic is float32 on the float32-rounded coefficients (sos is rounded once, at creation): exactly the filter
 * scipy applies to float32 sos and x, but not the float64 arithmetic scipy uses when sos is float64.  The device runs the
 * recurrence as a blocked scan: tiles of VV_DSP_SOS_TILE samples whose per-thread runs are joined by the constant maps
 * A^k of each section (tables computed on the host in double; the join itself runs in float64).  Rows longer than the segment length (VV_DSP_SOS_SEGMENT
 * samples unless the handle reports another, a multiple of the tile) are cut into segments that are joined through the
 * cascade's state transition over one segment, so a few long rows still fill the device.  Output bits depend only on
 * (sos, n, zi, x) of a row: not on the batch, the memory spaces or the staging chunks.
 *
 * Rejected filters: a section whose poles are not strictly inside the unit circle (|a2| < 1 and |a1| < 1 + a2 fails)
 * is rejected with VV_DSP_ERROR_OUT_OF_RANGE.  scipy runs such a filter and diverges; the scan has no error bound for it.
 *
 * Pitches (in elements) of 0 mean dense.  Memory spaces as above: if every buffer is DEVICE the call only enqueues on
 * the handle's stream, otherwise it returns once the results are in host memory.  `out` must not overlap `signals`; an
 * identical base pointer is rejected with VV_DSP_ERROR_UNSUPPORTED.
 *
 * Status: NULL handle / signals / out / sos -> VV_DSP_ERROR_NULL_POINTER; S outside [1, 64], a pitch smaller than its
 * row, or 0 < n <= padlen in filtfilt -> VV_DSP_ERROR_INVALID_SIZE; a coefficient that is not finite ->
 * VV_DSP_ERROR_NAN_INF; a0 != 1, a pole on or outside the unit circle, a bad memory space or a bad padtype ->
 * VV_DSP_ERROR_OUT_OF_RANGE; out == signals -> VV_DSP_ERROR_UNSUPPORTED; batch == 0 or n == 0 -> VV_DSP_OK with no
 * filtering (filter then writes zf = zi, or zeros); CUDA failures -> VV_DSP_ERROR_INTERNAL (no usable device at
 * creation: VV_DSP_ERROR_UNSUPPORTED).
 * ------------------------------------------------------------------------------------------------------------- */
#define VV_DSP_SOS_MAX_SECTIONS 64
#define VV_DSP_SOS_TILE 4096                      /* samples per tile: 256 threads x 16 */
#define VV_DSP_SOS_SEGMENT ((size_t)1 << 20)      /* samples per segment of a long row */
enum { VV_DSP_PAD_NONE = 0, VV_DSP_PAD_ODD = 1, VV_DSP_PAD_EVEN = 2, VV_DSP_PAD_CONSTANT = 3 };
typedef struct vv_dsp_sos vv_dsp_sos;
VV_DSP_NODISCARD vv_dsp_status vv_dsp_sos_create(const vv_dsp_real* sos /* HOST [S][6] */, size_t n_sections,
                                                 vv_dsp_sos** out);
vv_dsp_status vv_dsp_sos_destroy(vv_dsp_sos* h);
/* same rules as vv_dsp_stft_set_stream (NULL = the handle's own stream) */
vv_dsp_status vv_dsp_sos_set_stream(vv_dsp_sos* h, void* cuda_stream);
vv_dsp_status vv_dsp_sos_synchronize(vv_dsp_sos* h);
/* S and the segment length in samples */
vv_dsp_status vv_dsp_sos_get_config(const vv_dsp_sos* h, size_t* n_sections, size_t* segment_length);
VV_DSP_NODISCARD vv_dsp_status vv_dsp_sos_filter_batch(
    vv_dsp_sos* h,
    const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch, size_t n, size_t signal_pitch,
    const vv_dsp_real* zi, vv_dsp_mem_space zi_space,     /* [S][batch][2] or NULL */
    vv_dsp_real* zf, vv_dsp_mem_space zf_space,           /* [S][batch][2] or NULL */
    vv_dsp_real* out, vv_dsp_mem_space out_space, size_t out_pitch);
VV_DSP_NODISCARD vv_dsp_status vv_dsp_sos_filtfilt_batch(
    vv_dsp_sos* h,
    const vv_dsp_real* signals, vv_dsp_mem_space signals_space, size_t batch, size_t n, size_t signal_pitch,
    int padtype, size_t padlen,
    vv_dsp_real* out, vv_dsp_mem_space out_space, size_t out_pitch);

/* Library / device introspection */
const char* vv_dsp_b200_version(void);
/* last CUDA error text seen by the calling thread ("" if none) */
const char* vv_dsp_b200_last_error(void);
/* diagnostics: measured FP32 FMA throughput of the current device in TFLOP/s (scalar FFMA when packed == 0,
 * packed FFMA2 otherwise); the denominator of the FP32 side of the roofline */
vv_dsp_status vv_dsp_b200_fp32_peak(int packed, double* tflops);
/* diagnostics: the SM clock in MHz at this moment, measured on the device (SM cycles per nanosecond of the global
 * timer over ~50 us) after everything queued on cuda_stream; synchronises that stream */
vv_dsp_status vv_dsp_b200_sm_clock_mhz(void* cuda_stream, double* mhz);
/* number of kernels this process has launched through the library (bench.py's gpu_launches) */
unsigned long long vv_dsp_b200_kernel_launches(void);

#ifdef __cplusplus
}
#endif

#endif /* VV_DSP_B200_H */
