"""vv-dsp_b200: B200-native (sm_100a) STFT / ISTFT / FFT hot path behind vv-dsp's C API.

The product is ``lib/libvvdsp_b200.so`` (C99 host library + hand-written CUDA kernels,
built by ``python -m vv_dsp_b200.build``).  This package is the thin ctypes mirror of
that C API used by the tests and bench.py; names, argument meaning and status codes
follow the reference's ``vv_dsp_stft_*`` / ``vv_dsp_fft_*`` interface
(reference include/vv_dsp/spectral/stft.h, fft.h).  There is no CPU fallback: loading
fails loudly when the CUDA library has not been built.
"""
from .api import (  # noqa: F401
    CONVENTIONS, KINDS, WINDOWS, FftPlan, FirFilter, Library, Resampler, SosFilter, Stft, StftStream, VvDspError, default_library,
    fetch_frame, get_num_frames, overlap_add, window, mel_filterbank, log_mel_spectrogram, mfcc, MfccPlan, pcm_to_planar,
)

__all__ = ["Stft", "StftStream", "FftPlan", "FirFilter", "Resampler", "SosFilter", "Library", "VvDspError", "default_library", "window", "get_num_frames",
           "fetch_frame", "overlap_add", "WINDOWS", "CONVENTIONS", "KINDS"]
