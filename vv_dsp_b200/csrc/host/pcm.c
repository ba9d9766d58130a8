/*
 * pcm.c -- vv_dsp_b200_pcm_to_planar (include/vv_dsp/b200.h): the sample conversion of the reference's WAV
 * reader (src/audio/wav.c:458-521) as a device kernel, so that config 1 style inputs can be uploaded as
 * PCM and converted next to the STFT.  SURVEY.md section 8f, rank 4.  File parsing stays with the caller.
 */
#include <stdlib.h>
#include "vv_dsp/b200.h"
#include "vvb200_cuda.h"
#include "internal.h"

vv_dsp_status vv_dsp_b200_pcm_to_planar(const void* interleaved, vv_dsp_mem_space in_space, int format, size_t num_samples,
                                        size_t channels, vv_dsp_real* planar, vv_dsp_mem_space out_space, size_t planar_pitch,
                                        void* cuda_stream)
{
    const size_t bytes_per = (size_t)(format < 0 ? -format : format) / 8;
    const void* d_in = interleaved;
    float *d_out = planar, *d_tmp_out = NULL;
    void *d_tmp_in = NULL, *stream = cuda_stream, *own = NULL;
    int st;
    if (!interleaved || !planar) return VV_DSP_ERROR_NULL_POINTER;
    if ((unsigned)in_space > 1u || (unsigned)out_space > 1u) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (format != 16 && format != 24 && format != 32 && format != -32) return VV_DSP_ERROR_OUT_OF_RANGE;
    if (num_samples == 0 || channels == 0) return VV_DSP_ERROR_INVALID_SIZE;
    if (planar_pitch == 0) planar_pitch = num_samples;
    if (planar_pitch < num_samples) return VV_DSP_ERROR_INVALID_SIZE;
    st = vvb_device_ready();                 /* no CUDA device -> UNSUPPORTED, never a CPU conversion */
    if (st) return vvdsp_internal_status(st);
    if (!stream && (in_space == VV_DSP_MEM_HOST || out_space == VV_DSP_MEM_HOST)) { st = vvb_stream_create(&own); stream = own; }
    if (!st && in_space == VV_DSP_MEM_HOST) {
        st = vvb_malloc(&d_tmp_in, num_samples * channels * bytes_per);
        if (!st) st = vvb_memcpy_h2d(d_tmp_in, interleaved, num_samples * channels * bytes_per, stream);
        d_in = d_tmp_in;
    }
    if (!st && out_space == VV_DSP_MEM_HOST) {
        st = vvb_malloc((void**)&d_tmp_out, channels * num_samples * sizeof(float));
        d_out = d_tmp_out;
    }
    if (!st) st = vvb_pcm_to_planar(d_in, format, num_samples, channels, d_out,
                                    out_space == VV_DSP_MEM_HOST ? num_samples : planar_pitch, stream);
    if (!st && out_space == VV_DSP_MEM_HOST)
        st = vvb_memcpy2d_d2h(planar, planar_pitch * sizeof(float), d_tmp_out, num_samples * sizeof(float),
                              num_samples * sizeof(float), channels, stream);
    if (in_space == VV_DSP_MEM_HOST || out_space == VV_DSP_MEM_HOST) {
        int s2 = vvb_stream_sync(stream); if (!st) st = s2;
        vvb_free(d_tmp_in); vvb_free(d_tmp_out);
    }
    if (own) vvb_stream_destroy(own);
    return vvdsp_internal_status(st);
}
