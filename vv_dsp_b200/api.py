"""ctypes mirror of the C API in include/vv_dsp/*.h (see package docstring)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

PKG = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.path.join(PKG, "lib", "libvvdsp_b200.so")

WINDOWS = {"boxcar": 0, "hann": 1, "hamming": 2}
CONVENTIONS = {"valid": 0, "spectrogram": 1, "padded_tail": 2, "center": 3}
KINDS = {"complex": 0, "power": 1, "magnitude": 2}
HOST, DEVICE = 0, 1
STATUS = {0: "VV_DSP_OK", 1: "VV_DSP_ERROR_NULL_POINTER", 2: "VV_DSP_ERROR_INVALID_SIZE",
          3: "VV_DSP_ERROR_OUT_OF_RANGE", 4: "VV_DSP_ERROR_INTERNAL", 5: "VV_DSP_ERROR_NAN_INF",
          6: "VV_DSP_ERROR_UNSUPPORTED"}
FFT_C2C, FFT_R2C, FFT_C2R = 0, 1, 2
FFT_FORWARD, FFT_BACKWARD = 1, -1

_sz = C.c_size_t
_vp = C.c_void_p


class VvDspError(RuntimeError):
    def __init__(self, status, where, detail=""):
        self.status = int(status)
        super().__init__(f"{where}: {STATUS.get(int(status), status)}" + (f" ({detail})" if detail else ""))


class StftParams(C.Structure):
    """vv_dsp_stft_params (reference include/vv_dsp/spectral/stft.h:23-27)"""
    _fields_ = [("fft_size", _sz), ("hop_size", _sz), ("window", C.c_int)]


class Library:
    """A loaded libvvdsp_b200.so with prototypes declared for every exported entry point."""

    # name -> (restype, argtypes); the exported C-ABI of include/vv_dsp/*.h
    PROTOS = {
        "vv_dsp_stft_create": (C.c_int, [C.POINTER(StftParams), C.POINTER(_vp)]),
        "vv_dsp_stft_destroy": (C.c_int, [_vp]),
        "vv_dsp_stft_process": (C.c_int, [_vp, _vp, _vp]),
        "vv_dsp_stft_reconstruct": (C.c_int, [_vp, _vp, _vp, _vp]),
        "vv_dsp_stft_spectrogram": (C.c_int, [_vp, _vp, _sz, _vp, C.POINTER(_sz)]),
        "vv_dsp_fft_set_backend": (C.c_int, [C.c_int]),
        "vv_dsp_fft_get_backend": (C.c_int, []),
        "vv_dsp_fft_is_backend_available": (C.c_int, [C.c_int]),
        "vv_dsp_fft_set_fftw_flag": (C.c_int, [C.c_int]),
        "vv_dsp_fft_flush_fftw_cache": (C.c_int, []),
        "vv_dsp_fft_make_plan": (C.c_int, [_sz, C.c_int, C.c_int, C.POINTER(_vp)]),
        "vv_dsp_fft_execute": (C.c_int, [_vp, _vp, _vp]),
        "vv_dsp_fft_destroy": (C.c_int, [_vp]),
        "vv_dsp_fft_execute_batch": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int, _sz, _vp]),
        "vv_dsp_window_boxcar": (C.c_int, [_sz, _vp]),
        "vv_dsp_window_hann": (C.c_int, [_sz, _vp]),
        "vv_dsp_window_hamming": (C.c_int, [_sz, _vp]),
        "vv_dsp_get_num_frames": (_sz, [_sz, _sz, _sz, C.c_int]),
        "vv_dsp_fetch_frame": (C.c_int, [_vp, _sz, _vp, _sz, _sz, _sz, C.c_int, _vp]),
        "vv_dsp_overlap_add": (C.c_int, [_vp, _vp, _sz, _sz, _sz, _sz]),
        "vv_dsp_vectorized_window_apply": (C.c_int, [_vp, _vp, _vp, _sz]),
        "vv_dsp_stft_num_frames": (_sz, [_vp, _sz, C.c_int]),
        "vv_dsp_stft_num_bins": (_sz, [_vp]),
        "vv_dsp_stft_set_stream": (C.c_int, [_vp, _vp]),
        "vv_dsp_stft_synchronize": (C.c_int, [_vp]),
        "vv_dsp_stft_set_async": (C.c_int, [_vp, C.c_int]),
        "vv_dsp_stft_batch_forward": (C.c_int, [_vp, _vp, C.c_int, _sz, _sz, _sz, C.c_int, C.c_int, _vp, C.c_int, _sz,
                                                C.POINTER(_sz)]),
        "vv_dsp_stft_batch_forward_pcm": (C.c_int, [_vp, _vp, C.c_int, _sz, _sz, _sz, C.c_int, C.c_int, _vp, C.c_int, _sz,
                                                    C.POINTER(_sz)]),
        "vv_dsp_stft_batch_inverse": (C.c_int, [_vp, _vp, C.c_int, _sz, _sz, _sz, _vp, C.c_int, _sz, _sz, C.c_int]),
        "vv_dsp_stft_istft": (C.c_int, [_vp, _vp, _sz, _vp, _sz]),
        "vv_dsp_hz_to_mel": (C.c_float, [C.c_float]),
        "vv_dsp_mel_to_hz": (C.c_float, [C.c_float]),
        "vv_dsp_mel_filterbank_create": (C.c_int, [_sz, _sz, C.c_float, C.c_float, C.c_float, C.c_int, C.POINTER(C.POINTER(C.c_float)),
                                                   C.POINTER(_sz), C.POINTER(_sz)]),
        "vv_dsp_mel_filterbank_free": (None, [C.POINTER(C.c_float), _sz]),
        "vv_dsp_compute_log_mel_spectrogram": (C.c_int, [_vp, _sz, _sz, _vp, _sz, C.c_float, _vp]),
        "vv_dsp_stft_batch_logmel": (C.c_int, [_vp, _vp, C.c_int, _sz, _sz, _sz, C.c_int, _vp, _sz, C.c_float, _vp, C.c_int,
                                               C.POINTER(_sz)]),
        "vv_dsp_stft_batch_logmel_pcm": (C.c_int, [_vp, _vp, C.c_int, _sz, _sz, _sz, C.c_int, _vp, _sz, C.c_float, _vp, C.c_int,
                                                   C.POINTER(_sz)]),
        "vv_dsp_stft_batch_mfcc": (C.c_int, [_vp, _vp, C.c_int, _sz, _sz, _sz, C.c_int, _vp, _sz, C.c_float, _sz, C.c_float, _vp, C.c_int,
                                             C.POINTER(_sz)]),
        "vv_dsp_mfcc": (C.c_int, [_vp, _sz, _sz, _sz, C.c_int, C.c_float, _vp]),
        "vv_dsp_mfcc_init": (C.c_int, [_sz, _sz, _sz, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int, C.c_float, C.c_float,
                                       C.POINTER(_vp)]),
        "vv_dsp_mfcc_process": (C.c_int, [_vp, _vp, _sz, _vp]),
        "vv_dsp_mfcc_destroy": (C.c_int, [_vp]),
        "vv_dsp_b200_pcm_to_planar": (C.c_int, [_vp, C.c_int, C.c_int, _sz, _sz, _vp, C.c_int, _sz, _vp]),
        "vv_dsp_b200_version": (C.c_char_p, []),
        "vv_dsp_b200_last_error": (C.c_char_p, []),
        "vv_dsp_b200_kernel_launches": (C.c_ulonglong, []),
        "vv_dsp_b200_fp32_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
        "vv_dsp_b200_sm_clock_mhz": (C.c_int, [_vp, C.POINTER(C.c_double)]),
        "vv_dsp_stft_shard_inverse": (C.c_int, [_vp, _vp, _sz, _sz, C.c_int, C.c_int, _vp, _sz]),
        "vv_dsp_stft_device": (C.c_int, [_vp]),
        "vv_dsp_stft_get_stream": (_vp, [_vp]),
        "vv_dsp_stft_stream_create": (C.c_int, [C.POINTER(StftParams), _sz, _sz, C.POINTER(C.c_int), C.POINTER(_vp)]),
        "vv_dsp_stft_stream_destroy": (C.c_int, [_vp]),
        "vv_dsp_stft_stream_num_frames": (_sz, [_vp]),
        "vv_dsp_stft_stream_get_shard": (C.c_int, [_vp, _sz, _vp]),
        "vv_dsp_stft_stream_upload": (C.c_int, [_vp, _vp]),
        "vv_dsp_stft_stream_forward": (C.c_int, [_vp]),
        "vv_dsp_stft_stream_inverse": (C.c_int, [_vp]),
        "vv_dsp_stft_stream_roundtrip": (C.c_int, [_vp]),
        "vv_dsp_stft_stream_synchronize": (C.c_int, [_vp]),
        "vv_dsp_stft_stream_download": (C.c_int, [_vp, _vp]),
        "vv_dsp_stft_stream_download_spectra": (C.c_int, [_vp, _vp]),
        "vv_dsp_stft_stream_time_roundtrip": (C.c_int, [_vp, _sz, _sz, C.POINTER(C.c_double)]),
        "vv_dsp_fir_create": (C.c_int, [_sz, C.POINTER(_vp)]),
        "vv_dsp_fir_destroy": (C.c_int, [_vp]),
        "vv_dsp_fir_set_stream": (C.c_int, [_vp, _vp]),
        "vv_dsp_fir_synchronize": (C.c_int, [_vp]),
        "vv_dsp_fir_get_config": (C.c_int, [_vp, C.POINTER(_sz), C.POINTER(_sz)]),
        "vv_dsp_fir_filter_batch": (C.c_int, [_vp, _vp, C.c_int, _sz, _sz, _vp, C.c_int, _sz, _sz, _sz, _vp, C.c_int, _sz, _sz]),
        "vv_dsp_resample_poly_create": (C.c_int, [_sz, _sz, _vp, _sz, C.POINTER(_vp)]),
        "vv_dsp_resample_poly_destroy": (C.c_int, [_vp]),
        "vv_dsp_resample_poly_set_stream": (C.c_int, [_vp, _vp]),
        "vv_dsp_resample_poly_synchronize": (C.c_int, [_vp]),
        "vv_dsp_resample_poly_get_config": (C.c_int, [_vp, C.POINTER(_sz), C.POINTER(_sz), C.POINTER(_sz), C.POINTER(_sz)]),
        "vv_dsp_resample_poly_output_length": (_sz, [_vp, _sz]),
        "vv_dsp_resample_poly_batch": (C.c_int, [_vp, _vp, C.c_int, _sz, _sz, _sz, _vp, C.c_int, _sz, C.POINTER(_sz)]),
        "vv_dsp_sos_create": (C.c_int, [_vp, _sz, C.POINTER(_vp)]),
        "vv_dsp_sos_destroy": (C.c_int, [_vp]),
        "vv_dsp_sos_set_stream": (C.c_int, [_vp, _vp]),
        "vv_dsp_sos_synchronize": (C.c_int, [_vp]),
        "vv_dsp_sos_get_config": (C.c_int, [_vp, C.POINTER(_sz), C.POINTER(_sz)]),
        "vv_dsp_sos_filter_batch": (C.c_int, [_vp, _vp, C.c_int, _sz, _sz, _sz, _vp, C.c_int, _vp, C.c_int, _vp, C.c_int, _sz]),
        "vv_dsp_sos_filtfilt_batch": (C.c_int, [_vp, _vp, C.c_int, _sz, _sz, _sz, C.c_int, _sz, _vp, C.c_int, _sz]),
    }
    # entry points newer than round 1: absent from an old library variant loaded for an A/B measurement
    OPTIONAL = {"vv_dsp_b200_sm_clock_mhz", "vv_dsp_stft_shard_inverse", "vv_dsp_stft_device", "vv_dsp_stft_get_stream",
                "vv_dsp_stft_stream_create", "vv_dsp_stft_stream_destroy", "vv_dsp_stft_stream_num_frames",
                "vv_dsp_stft_stream_get_shard", "vv_dsp_stft_stream_upload", "vv_dsp_stft_stream_forward",
                "vv_dsp_stft_stream_inverse", "vv_dsp_stft_stream_roundtrip", "vv_dsp_stft_stream_synchronize",
                "vv_dsp_stft_stream_download", "vv_dsp_stft_stream_download_spectra", "vv_dsp_stft_stream_time_roundtrip",
                "vv_dsp_fir_create", "vv_dsp_fir_destroy", "vv_dsp_fir_set_stream", "vv_dsp_fir_synchronize", "vv_dsp_fir_get_config",
                "vv_dsp_fir_filter_batch", "vv_dsp_resample_poly_create", "vv_dsp_resample_poly_destroy",
                "vv_dsp_resample_poly_set_stream", "vv_dsp_resample_poly_synchronize", "vv_dsp_resample_poly_get_config",
                "vv_dsp_resample_poly_output_length", "vv_dsp_resample_poly_batch", "vv_dsp_sos_create", "vv_dsp_sos_destroy",
                "vv_dsp_sos_set_stream", "vv_dsp_sos_synchronize", "vv_dsp_sos_get_config", "vv_dsp_sos_filter_batch",
                "vv_dsp_sos_filtfilt_batch"}

    def __init__(self, path: str | None = None):
        path = path or DEFAULT_LIB
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} not found: the CUDA library has not been built (python -m vv_dsp_b200.build). "
                "vv-dsp_b200 has no CPU fallback.")
        self.path = path
        self.dll = C.CDLL(path)
        for name, (res, args) in self.PROTOS.items():
            if name in self.OPTIONAL and not hasattr(self.dll, name):
                continue
            fn = getattr(self.dll, name)
            fn.restype = res
            fn.argtypes = args

    def __getattr__(self, name):
        return getattr(self.dll, name)

    def last_error(self) -> str:
        return (self.dll.vv_dsp_b200_last_error() or b"").decode()

    def kernel_launches(self) -> int:
        return int(self.dll.vv_dsp_b200_kernel_launches())

    def fp32_peak(self, packed: bool = False) -> float:
        """measured FP32 FMA throughput of the current device, TFLOP/s"""
        v = C.c_double(0.0)
        st = self.dll.vv_dsp_b200_fp32_peak(int(packed), C.byref(v))
        if st != 0:
            raise VvDspError(st, "vv_dsp_b200_fp32_peak", self.last_error())
        return float(v.value)

    def sm_clock_mhz(self, cuda_stream=None) -> float:
        """SM clock measured on the device right after the work queued on cuda_stream (synchronises it)"""
        v = C.c_double(0.0)
        st = self.dll.vv_dsp_b200_sm_clock_mhz(_vp(cuda_stream or 0), C.byref(v))
        if st != 0:
            raise VvDspError(st, "vv_dsp_b200_sm_clock_mhz", self.last_error())
        return float(v.value)

    def version(self) -> str:
        return self.dll.vv_dsp_b200_version().decode()


_default = None


def default_library() -> Library:
    global _default
    if _default is None:
        # VVDSP_B200_LIB: path of another nvcc-built libvvdsp_b200 variant (A/B measurements only)
        _default = Library(os.environ.get("VVDSP_B200_LIB") or None)
    return _default


def _check(lib, st, where):
    if st != 0:
        raise VvDspError(st, where, lib.last_error())


def _is_device(a) -> bool:
    return hasattr(a, "data_ptr") and getattr(a, "is_cuda", False)


def _ptr(a):
    if a is None:
        return None
    if hasattr(a, "data_ptr"):          # torch tensor, CUDA (device space) or CPU (host space)
        return _vp(a.data_ptr())
    return a.ctypes.data_as(_vp)


def _space(t):
    return DEVICE if _is_device(t) else HOST


def _check_device_tensor(t, dtype_name, what):
    """device tensors are handed to the C API as raw pointers: the layout has to be what it expects"""
    import torch
    want = {"float32": torch.float32, "complex64": torch.complex64}[dtype_name]
    if t.dtype != want:
        raise TypeError(f"{what}: expected a {dtype_name} CUDA tensor, got {t.dtype}")
    if t.stride(-1) != 1:
        raise ValueError(f"{what}: the innermost dimension must be contiguous (stride {t.stride(-1)})")


def _rows(a, what):
    """(container, rows, row length, row pitch in elements); device tensors keep their layout (odd pitches of views
    included), host arrays are made dense float32"""
    if _is_device(a):
        _check_device_tensor(a, "float32", what)
        if a.ndim != 2:
            raise ValueError(f"{what}: expected a 2-D tensor")
        return a, int(a.shape[0]), int(a.shape[1]), (int(a.stride(0)) if a.shape[0] > 1 else 0)
    a = np.ascontiguousarray(a, np.float32)
    if a.ndim != 2:
        raise ValueError(f"{what}: expected a 2-D array")
    return a, int(a.shape[0]), int(a.shape[1]), 0


def _out_rows(out, like, batch, n):
    """the output container ([batch, n] float32 in the container of `like` unless given) and its row pitch"""
    if out is None:
        if _is_device(like):
            import torch
            out = torch.empty((batch, n), device=like.device, dtype=torch.float32)
        else:
            out = np.empty((batch, n), np.float32)
    elif not _is_device(out):
        if not (isinstance(out, np.ndarray) and out.dtype == np.float32 and out.flags.c_contiguous):
            raise ValueError("out: expected a C-contiguous float32 numpy array")
    opitch = 0
    if _is_device(out):
        _check_device_tensor(out, "float32", "out")
        opitch = int(out.stride(0)) if batch > 1 else 0
    if tuple(out.shape) != (batch, n):
        raise ValueError(f"out: expected shape {(batch, n)}, got {tuple(out.shape)}")
    return out, opitch


def _win_id(w):
    return WINDOWS[w] if isinstance(w, str) else int(w)


# ----------------------------------------------------------------------------- free functions
def window(kind, n, lib: Library | None = None):
    """vv_dsp_window_{boxcar,hann,hamming}(N, out) -> (status, float32[n])"""
    lib = lib or default_library()
    out = np.empty(max(n, 1), np.float32)
    st = getattr(lib, f"vv_dsp_window_{kind}")(n, _ptr(out))
    return st, out[:n]


def get_num_frames(signal_len, frame_len, hop_len, center=0, lib: Library | None = None) -> int:
    lib = lib or default_library()
    return int(lib.vv_dsp_get_num_frames(signal_len, frame_len, hop_len, int(center)))


def fetch_frame(signal, frame_len, hop_len, frame_index, center=0, win=None, lib: Library | None = None):
    lib = lib or default_library()
    signal = np.ascontiguousarray(signal, np.float32)
    out = np.zeros(max(frame_len, 1), np.float32)
    w = np.ascontiguousarray(win, np.float32) if win is not None else None
    st = lib.vv_dsp_fetch_frame(_ptr(signal), signal.size, _ptr(out), frame_len, hop_len, frame_index, int(center), _ptr(w))
    return st, out[:frame_len]


def overlap_add(frame, output, hop_len, frame_index, lib: Library | None = None) -> int:
    lib = lib or default_library()
    frame = np.ascontiguousarray(frame, np.float32)
    assert output.dtype == np.float32 and output.flags.c_contiguous
    return lib.vv_dsp_overlap_add(_ptr(frame), _ptr(output), output.size, frame.size, hop_len, frame_index)


def mel_filterbank(n_fft, n_mels, sample_rate, fmin, fmax, variant=0, lib: Library | None = None):
    """vv_dsp_mel_filterbank_create -> (status, float32[n_mels, n_fft/2+1] or None)"""
    lib = lib or default_library()
    w = C.POINTER(C.c_float)()
    nf, fl = _sz(0), _sz(0)
    st = lib.vv_dsp_mel_filterbank_create(n_fft, n_mels, sample_rate, fmin, fmax, variant, C.byref(w), C.byref(nf), C.byref(fl))
    if st != 0:
        return st, None
    out = np.ctypeslib.as_array(w, shape=(nf.value, fl.value)).copy()
    lib.vv_dsp_mel_filterbank_free(w, nf)
    return st, out


def log_mel_spectrogram(power, weights, log_epsilon, lib: Library | None = None):
    """vv_dsp_compute_log_mel_spectrogram: power [frames, bins], weights [n_mels, bins] (host) -> [frames, n_mels]"""
    lib = lib or default_library()
    power = np.ascontiguousarray(power, np.float32)
    weights = np.ascontiguousarray(weights, np.float32)
    out = np.empty((power.shape[0], weights.shape[0]), np.float32)
    st = lib.vv_dsp_compute_log_mel_spectrogram(_ptr(power), power.shape[0], power.shape[1], _ptr(weights), weights.shape[0],
                                                log_epsilon, _ptr(out))
    _check(lib, st, "vv_dsp_compute_log_mel_spectrogram")
    return out


def pcm_to_planar(raw, fmt, channels, out=None, stream=0, lib: Library | None = None):
    """vv_dsp_b200_pcm_to_planar: interleaved little-endian samples (bytes / numpy uint8 / torch CUDA uint8) of
    format 16 / 24 / 32 (PCM) or -32 (float32) -> float32 [channels, samples] (numpy, or torch when out is)."""
    lib = lib or default_library()
    dev_in = _is_device(raw)
    if not dev_in:
        raw = np.frombuffer(bytes(raw), np.uint8) if not isinstance(raw, np.ndarray) else np.ascontiguousarray(raw).view(np.uint8)
    nbytes = int(raw.numel()) if dev_in else int(raw.size)
    n = nbytes // (abs(fmt) // 8) // max(channels, 1)
    if out is None:
        if dev_in:
            import torch
            out = torch.empty((channels, n), device=raw.device, dtype=torch.float32)
        else:
            out = np.empty((channels, n), np.float32)
    pitch = int(out.stride(0)) if _is_device(out) else n
    st = lib.vv_dsp_b200_pcm_to_planar(_ptr(raw), DEVICE if dev_in else HOST, fmt, n, channels, _ptr(out),
                                       _space(out), pitch, stream)
    _check(lib, st, "vv_dsp_b200_pcm_to_planar")
    return out


DCT_II = 2


def mfcc(log_mel, num_coeffs, lifter=0.0, dct_type=DCT_II, lib: Library | None = None):
    """vv_dsp_mfcc: log_mel [frames, n_mels] (host) -> (status, [frames, num_coeffs])"""
    lib = lib or default_library()
    log_mel = np.ascontiguousarray(log_mel, np.float32)
    out = np.empty((log_mel.shape[0], max(int(num_coeffs), 1)), np.float32)
    st = lib.vv_dsp_mfcc(_ptr(log_mel), log_mel.shape[0], log_mel.shape[1], num_coeffs, dct_type, lifter, _ptr(out))
    return st, out[:, :num_coeffs]


class MfccPlan:
    """vv_dsp_mfcc_init / process / destroy (power spectrogram -> log-mel -> MFCC, host buffers)"""

    def __init__(self, n_fft, n_mels, num_coeffs, sample_rate, fmin, fmax, variant=0, dct_type=DCT_II, lifter=0.0,
                 log_epsilon=1e-10, lib: Library | None = None):
        self.lib = lib or default_library()
        self._p = _vp()
        self.num_coeffs = num_coeffs
        self.status = self.lib.vv_dsp_mfcc_init(n_fft, n_mels, num_coeffs, sample_rate, fmin, fmax, variant, dct_type, lifter,
                                                log_epsilon, C.byref(self._p))

    def process(self, power):
        power = np.ascontiguousarray(power, np.float32)
        out = np.empty((power.shape[0], self.num_coeffs), np.float32)
        st = self.lib.vv_dsp_mfcc_process(self._p, _ptr(power), power.shape[0], _ptr(out))
        return st, out

    def close(self):
        if self._p:
            self.lib.vv_dsp_mfcc_destroy(self._p)
            self._p = _vp()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


# ----------------------------------------------------------------------------- stream-bound handles
class _StreamHandle:
    """A handle of include/vv_dsp/b200.h that enqueues its device work on one CUDA stream: vv_dsp_<_prefix>_destroy,
    _set_stream and _synchronize, and the binding to torch's current stream."""

    _prefix = ""

    def __init__(self, lib: Library | None):
        self.lib = lib or default_library()
        self._h = _vp()
        self._stream_pinned = False      # set_stream() called by the user: never rebind behind their back
        self._bound_stream = None        # what the handle is bound to right now (None = its own stream)

    def _call(self, what, *args):
        name = f"vv_dsp_{self._prefix}_{what}"
        _check(self.lib, getattr(self.lib, name)(self._h, *args), name)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            getattr(self.lib, f"vv_dsp_{self._prefix}_destroy")(self._h)
            self._h = _vp()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_stream(self, cuda_stream):
        """Pin the handle to a stream.  cuda_stream: a cudaStream_t as an integer.  None = the handle's own stream
        (and back to automatic binding, see _bind_torch_stream); 0 (the legacy default stream, what torch reports
        for its default stream) is passed as cudaStreamLegacy (0x1), because the C API reserves NULL for "the
        handle's own stream"."""
        self._stream_pinned = cuda_stream is not None
        self._set_stream_raw(cuda_stream)

    def _set_stream_raw(self, cuda_stream):
        self._call("set_stream", None if cuda_stream is None else _vp(int(cuda_stream) or 1))
        self._bound_stream = None if cuda_stream is None else (int(cuda_stream) or 1)

    def _bind_torch_stream(self, tensor):
        """Stream contract of the device path: calls whose buffers are torch CUDA tensors are enqueued on torch's
        CURRENT stream of that device (like any torch op), so they are ordered after the ops that produced the
        inputs and before the ops that consume the outputs -- unless the user pinned a stream with set_stream(),
        in which case ordering against torch's streams is theirs to establish."""
        if self._stream_pinned:
            return
        import torch
        cur = int(torch.cuda.current_stream(tensor.device).cuda_stream) or 1
        if cur != self._bound_stream:
            self._set_stream_raw(cur)

    def _bind(self, *tensors):
        """_bind_torch_stream to the first device tensor among `tensors` (None entries allowed), if there is one"""
        dev = next((t for t in tensors if _is_device(t)), None)
        if dev is not None:
            self._bind_torch_stream(dev)

    def synchronize(self):
        self._call("synchronize")


# ----------------------------------------------------------------------------- STFT handle
class Stft(_StreamHandle):
    """vv_dsp_stft handle: create / process / reconstruct / spectrogram + the batched extension."""

    _prefix = "stft"

    def __init__(self, fft_size, hop_size, window="hann", lib: Library | None = None):
        super().__init__(lib)
        self.nfft, self.hop = int(fft_size), int(hop_size)
        self.bins = self.nfft // 2 + 1
        p = StftParams(self.nfft, self.hop, _win_id(window))
        st = self.lib.vv_dsp_stft_create(C.byref(p), C.byref(self._h))
        _check(self.lib, st, "vv_dsp_stft_create")

    # --- reference per-frame API
    def process(self, frame):
        frame = np.ascontiguousarray(frame, np.float32)
        assert frame.size == self.nfft
        out = np.empty(self.nfft, np.complex64)
        _check(self.lib, self.lib.vv_dsp_stft_process(self._h, _ptr(frame), _ptr(out)), "vv_dsp_stft_process")
        return out

    def reconstruct(self, spec, out_add, norm_add=None):
        spec = np.ascontiguousarray(spec, np.complex64)
        assert spec.size == self.nfft and out_add.dtype == np.float32 and out_add.size >= self.nfft
        _check(self.lib, self.lib.vv_dsp_stft_reconstruct(self._h, _ptr(spec), _ptr(out_add), _ptr(norm_add)),
               "vv_dsp_stft_reconstruct")

    def spectrogram(self, signal):
        signal = np.ascontiguousarray(signal, np.float32)
        frames = self.num_frames(signal.size, "spectrogram")
        out = np.empty((frames, self.nfft), np.float32)
        nf = _sz(0)
        keep = signal if signal.size else np.zeros(1, np.float32)
        _check(self.lib, self.lib.vv_dsp_stft_spectrogram(self._h, _ptr(keep), signal.size, _ptr(out), C.byref(nf)),
               "vv_dsp_stft_spectrogram")
        assert nf.value == frames
        return out

    # --- batched extension (include/vv_dsp/b200.h)
    def num_frames(self, n, convention="valid") -> int:
        return int(self.lib.vv_dsp_stft_num_frames(self._h, n, CONVENTIONS[convention]))

    def set_async(self, enable=True):
        """stream-ordered mode for HOST-buffer calls (see include/vv_dsp/b200.h); finish with synchronize()"""
        _check(self.lib, self.lib.vv_dsp_stft_set_async(self._h, int(bool(enable))), "vv_dsp_stft_set_async")

    def batch_forward(self, signals, kind="complex", convention="valid", out=None):
        """signals: [batch, n] float32, numpy (host) or torch CUDA tensor (device).  Returns
        [batch, frames, bins] complex64 / float32 in the same kind of container unless `out` is given."""
        dev_in = _is_device(signals)
        if not dev_in:
            signals = np.ascontiguousarray(signals, np.float32)
        assert signals.ndim == 2
        batch, n = int(signals.shape[0]), int(signals.shape[1])
        pitch = (int(signals.stride(0)) if batch > 1 else n) if dev_in else n
        frames = self.num_frames(n, convention)
        if out is None:
            if dev_in:
                import torch
                out = torch.empty((batch, frames, self.bins), device=signals.device,
                                  dtype=torch.complex64 if kind == "complex" else torch.float32)
            else:
                out = np.empty((batch, frames, self.bins), np.complex64 if kind == "complex" else np.float32)
        spec_pitch = 0
        if dev_in:
            _check_device_tensor(signals, "float32", "signals")
        if _is_device(out):
            _check_device_tensor(out, "complex64" if kind == "complex" else "float32", "out")
            assert tuple(out.shape) == (batch, frames, self.bins), (tuple(out.shape), (batch, frames, self.bins))
            spec_pitch = self._spec_pitch(out)
        self._bind(out, signals)
        nf = _sz(0)
        st = self.lib.vv_dsp_stft_batch_forward(self._h, _ptr(signals), DEVICE if dev_in else HOST, batch, n, pitch,
                                                CONVENTIONS[convention], KINDS[kind], _ptr(out),
                                                _space(out), spec_pitch, C.byref(nf))
        _check(self.lib, st, "vv_dsp_stft_batch_forward")
        assert nf.value == frames
        return out

    def batch_forward_pcm(self, pcm, fmt=16, kind="complex", convention="valid", out=None):
        """vv_dsp_stft_batch_forward_pcm: pcm = HOST [batch, n] numpy array of WAV samples -- int16 (fmt 16), int32 (fmt 32),
        float32 (fmt -32) or uint8 [batch, 3 n] (fmt 24, packed little-endian).  The upload carries the undecoded bytes."""
        dt = {16: np.int16, 32: np.int32, -32: np.float32, 24: np.uint8}[fmt]
        pcm = np.ascontiguousarray(pcm, dt)
        assert pcm.ndim == 2
        batch, n = int(pcm.shape[0]), int(pcm.shape[1]) // (3 if fmt == 24 else 1)
        frames = self.num_frames(n, convention)
        if out is None:
            out = np.empty((batch, frames, self.bins), np.complex64 if kind == "complex" else np.float32)
        spec_pitch = 0
        if _is_device(out):
            _check_device_tensor(out, "complex64" if kind == "complex" else "float32", "out")
            assert tuple(out.shape) == (batch, frames, self.bins)
            spec_pitch = self._spec_pitch(out)
            self._bind_torch_stream(out)
        nf = _sz(0)
        st = self.lib.vv_dsp_stft_batch_forward_pcm(self._h, _ptr(pcm), fmt, batch, n, n, CONVENTIONS[convention], KINDS[kind],
                                                    _ptr(out), _space(out), spec_pitch, C.byref(nf))
        _check(self.lib, st, "vv_dsp_stft_batch_forward_pcm")
        assert nf.value == frames
        return out

    def _prepare_device_args(self, signals, out):
        """dtype / layout checks and stream binding of the feature chains (dense float32 output)"""
        if _is_device(signals):
            _check_device_tensor(signals, "float32", "signals")
        if _is_device(out):
            _check_device_tensor(out, "float32", "out")
            if not out.is_contiguous():
                raise ValueError("out: must be contiguous")
        self._bind(out, signals)

    def _spec_pitch(self, t):
        """row pitch (elements) of a [batch, frames, bins] device tensor whose rows follow each other at one pitch;
        0 = dense"""
        if t.shape[1] > 1 and t.shape[0] > 1 and t.stride(0) != t.shape[1] * t.stride(1):
            raise ValueError("spectra: frames of consecutive signals must follow each other at the row pitch")
        p = int(t.stride(1)) if t.shape[1] > 1 else (int(t.stride(0)) if t.shape[0] > 1 else self.bins)
        if p < self.bins:
            raise ValueError("spectra: row pitch smaller than fft_size/2+1")
        return 0 if p == self.bins else p

    def batch_logmel(self, signals, weights, log_epsilon=1e-10, convention="valid", out=None):
        """STFT -> power -> mel -> log: signals [batch, n] (numpy or torch CUDA), weights [n_mels, bins] numpy"""
        dev_in = _is_device(signals)
        if not dev_in:
            signals = np.ascontiguousarray(signals, np.float32)
        weights = np.ascontiguousarray(weights, np.float32)
        assert weights.shape[1] == self.bins
        batch, n = int(signals.shape[0]), int(signals.shape[1])
        pitch = (int(signals.stride(0)) if batch > 1 else n) if dev_in else n
        frames = self.num_frames(n, convention)
        if out is None:
            if dev_in:
                import torch
                out = torch.empty((batch, frames, weights.shape[0]), device=signals.device, dtype=torch.float32)
            else:
                out = np.empty((batch, frames, weights.shape[0]), np.float32)
        self._prepare_device_args(signals, out)
        nf = _sz(0)
        st = self.lib.vv_dsp_stft_batch_logmel(self._h, _ptr(signals), DEVICE if dev_in else HOST, batch, n, pitch,
                                               CONVENTIONS[convention], _ptr(weights), weights.shape[0], log_epsilon,
                                               _ptr(out), _space(out), C.byref(nf))
        _check(self.lib, st, "vv_dsp_stft_batch_logmel")
        return out

    def batch_logmel_pcm(self, pcm, weights, fmt=16, log_epsilon=1e-10, convention="valid", out=None):
        """vv_dsp_stft_batch_logmel_pcm: pcm = HOST [batch, n] WAV samples (int16 / int32 / float32, or uint8 [batch, 3 n] for
        24-bit), uploaded undecoded; returns [batch, frames, n_mels] log-mel rows (numpy, or the torch CUDA tensor `out`)"""
        dt = {16: np.int16, 32: np.int32, -32: np.float32, 24: np.uint8}[fmt]
        pcm = np.ascontiguousarray(pcm, dt)
        weights = np.ascontiguousarray(weights, np.float32)
        assert pcm.ndim == 2 and weights.shape[1] == self.bins
        batch, n = int(pcm.shape[0]), int(pcm.shape[1]) // (3 if fmt == 24 else 1)
        frames = self.num_frames(n, convention)
        if out is None:
            out = np.empty((batch, frames, weights.shape[0]), np.float32)
        if _is_device(out):
            _check_device_tensor(out, "float32", "out")
            self._bind_torch_stream(out)
        nf = _sz(0)
        st = self.lib.vv_dsp_stft_batch_logmel_pcm(self._h, _ptr(pcm), fmt, batch, n, n, CONVENTIONS[convention], _ptr(weights),
                                                   weights.shape[0], log_epsilon, _ptr(out), _space(out), C.byref(nf))
        _check(self.lib, st, "vv_dsp_stft_batch_logmel_pcm")
        return out

    def batch_mfcc(self, signals, weights, num_coeffs, lifter=0.0, log_epsilon=1e-10, convention="valid", out=None):
        """STFT -> power -> mel -> log -> DCT-II (+ liftering): [batch, frames, num_coeffs]"""
        dev_in = _is_device(signals)
        if not dev_in:
            signals = np.ascontiguousarray(signals, np.float32)
        weights = np.ascontiguousarray(weights, np.float32)
        assert weights.shape[1] == self.bins
        batch, n = int(signals.shape[0]), int(signals.shape[1])
        pitch = (int(signals.stride(0)) if batch > 1 else n) if dev_in else n
        frames = self.num_frames(n, convention)
        if out is None:
            if dev_in:
                import torch
                out = torch.empty((batch, frames, num_coeffs), device=signals.device, dtype=torch.float32)
            else:
                out = np.empty((batch, frames, num_coeffs), np.float32)
        self._prepare_device_args(signals, out)
        nf = _sz(0)
        st = self.lib.vv_dsp_stft_batch_mfcc(self._h, _ptr(signals), DEVICE if dev_in else HOST, batch, n, pitch,
                                             CONVENTIONS[convention], _ptr(weights), weights.shape[0], log_epsilon,
                                             num_coeffs, lifter, _ptr(out), _space(out), C.byref(nf))
        _check(self.lib, st, "vv_dsp_stft_batch_mfcc")
        return out

    def batch_inverse(self, spectra, n_out, normalise=True, out=None):
        """spectra: [batch, frames, bins] complex64 (numpy or torch CUDA).  Returns [batch, n_out] float32."""
        dev_in = _is_device(spectra)
        if not dev_in:
            spectra = np.ascontiguousarray(spectra, np.complex64)
        assert spectra.ndim == 3 and spectra.shape[2] == self.bins
        batch, frames = int(spectra.shape[0]), int(spectra.shape[1])
        if out is None:
            if dev_in:
                import torch
                out = torch.empty((batch, n_out), device=spectra.device, dtype=torch.float32)
            else:
                out = np.empty((batch, n_out), np.float32)
        keep = spectra if frames else None
        spec_pitch = out_pitch = 0
        if dev_in:
            _check_device_tensor(spectra, "complex64", "spectra")
            spec_pitch = self._spec_pitch(spectra)
        if _is_device(out):
            _check_device_tensor(out, "float32", "out")
            assert out.ndim == 2 and int(out.shape[0]) == batch and int(out.shape[1]) == n_out
            out_pitch = int(out.stride(0)) if batch > 1 else 0
        self._bind(out, spectra)
        st = self.lib.vv_dsp_stft_batch_inverse(self._h, _ptr(keep), DEVICE if dev_in else HOST, batch, frames, spec_pitch,
                                                _ptr(out), _space(out), n_out, out_pitch, int(normalise))
        _check(self.lib, st, "vv_dsp_stft_batch_inverse")
        return out

    def shard_inverse(self, spectra, halo_frames, is_first, is_last, n_out, out=None):
        """Synthesis of one frame-range shard of a longer stream (include/vv_dsp/b200.h): spectra = CUDA tensor
        [halo_frames + own frames, bins], out = CUDA tensor [n_out] (the shard's owned samples)."""
        import torch
        _check_device_tensor(spectra, "complex64", "spectra")
        assert spectra.ndim == 2 and spectra.shape[1] == self.bins and spectra.is_contiguous()
        if out is None:
            out = torch.empty(n_out, device=spectra.device, dtype=torch.float32)
        _check_device_tensor(out, "float32", "out")
        self._bind_torch_stream(out)
        st = self.lib.vv_dsp_stft_shard_inverse(self._h, _ptr(spectra), int(spectra.shape[0]), int(halo_frames), int(bool(is_first)),
                                                int(bool(is_last)), _ptr(out), int(n_out))
        _check(self.lib, st, "vv_dsp_stft_shard_inverse")
        return out

    def shard_inverse_raw(self, spectra, halo_frames, is_first, is_last, out):
        """the same through raw pointers (numpy arrays standing in for device memory: emulator library only)"""
        st = self.lib.vv_dsp_stft_shard_inverse(self._h, _ptr(spectra), int(spectra.shape[0]), int(halo_frames), int(bool(is_first)),
                                                int(bool(is_last)), _ptr(out), int(out.size))
        _check(self.lib, st, "vv_dsp_stft_shard_inverse")
        return out

    def istft(self, half_spectra, n_out):
        half_spectra = np.ascontiguousarray(half_spectra, np.complex64)
        out = np.empty(n_out, np.float32)
        st = self.lib.vv_dsp_stft_istft(self._h, _ptr(half_spectra) if half_spectra.size else None,
                                        half_spectra.shape[0], _ptr(out), n_out)
        _check(self.lib, st, "vv_dsp_stft_istft")
        return out


# ----------------------------------------------------------------------------- one stream over several GPUs
class StreamShard(C.Structure):
    """vv_dsp_stft_stream_shard (include/vv_dsp/b200.h)"""
    _fields_ = [("device", C.c_int), ("frame0", _sz), ("frame1", _sz), ("sample0", _sz), ("sample1", _sz),
                ("halo_frames", _sz), ("left_halo", _sz), ("right_halo", _sz),
                ("signal", _vp), ("spectra", _vp), ("output", _vp), ("cuda_stream", _vp)]


class StftStream:
    """vv_dsp_stft_stream: ONE long stream sharded by frame range over several GPUs of this process."""

    def __init__(self, fft_size, hop_size, n, devices, window="hann", lib: Library | None = None):
        self.lib = lib or default_library()
        self.nfft, self.hop, self.n = int(fft_size), int(hop_size), int(n)
        self.bins = self.nfft // 2 + 1
        self.devices = list(devices)
        self._s = _vp()
        p = StftParams(self.nfft, self.hop, _win_id(window))
        ids = (C.c_int * len(self.devices))(*self.devices)
        st = self.lib.vv_dsp_stft_stream_create(C.byref(p), self.n, len(self.devices), ids, C.byref(self._s))
        _check(self.lib, st, "vv_dsp_stft_stream_create")
        self.frames = int(self.lib.vv_dsp_stft_stream_num_frames(self._s))

    def close(self):
        if getattr(self, "_s", None) is not None and self._s.value:
            self.lib.vv_dsp_stft_stream_destroy(self._s)
            self._s = _vp()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def shard(self, d) -> StreamShard:
        sh = StreamShard()
        _check(self.lib, self.lib.vv_dsp_stft_stream_get_shard(self._s, d, C.byref(sh)), "vv_dsp_stft_stream_get_shard")
        return sh

    def upload(self, signal):
        signal = np.ascontiguousarray(signal, np.float32)
        assert signal.size == self.n
        _check(self.lib, self.lib.vv_dsp_stft_stream_upload(self._s, _ptr(signal)), "vv_dsp_stft_stream_upload")

    def forward(self):
        _check(self.lib, self.lib.vv_dsp_stft_stream_forward(self._s), "vv_dsp_stft_stream_forward")

    def inverse(self):
        _check(self.lib, self.lib.vv_dsp_stft_stream_inverse(self._s), "vv_dsp_stft_stream_inverse")

    def roundtrip(self):
        _check(self.lib, self.lib.vv_dsp_stft_stream_roundtrip(self._s), "vv_dsp_stft_stream_roundtrip")

    def synchronize(self):
        _check(self.lib, self.lib.vv_dsp_stft_stream_synchronize(self._s), "vv_dsp_stft_stream_synchronize")

    def download(self):
        out = np.empty(self.n, np.float32)
        _check(self.lib, self.lib.vv_dsp_stft_stream_download(self._s, _ptr(out)), "vv_dsp_stft_stream_download")
        return out

    def download_spectra(self):
        out = np.empty((self.frames, self.bins), np.complex64)
        _check(self.lib, self.lib.vv_dsp_stft_stream_download_spectra(self._s, _ptr(out)), "vv_dsp_stft_stream_download_spectra")
        return out

    def time_roundtrip(self, warmup=3, steps=10) -> float:
        """ms per forward + inverse step, CUDA events on every device's stream, slowest device"""
        ms = C.c_double(0.0)
        _check(self.lib, self.lib.vv_dsp_stft_stream_time_roundtrip(self._s, warmup, steps, C.byref(ms)),
               "vv_dsp_stft_stream_time_roundtrip")
        return float(ms.value)


# ----------------------------------------------------------------------------- FIR filtering
class FirFilter(_StreamHandle):
    """vv_dsp_fir handle (include/vv_dsp/b200.h): batched FIR filtering by FFT convolution on the device.
    out[b][i] = sum_j h_b[j] x_b[i - j] for i < n_out; n_out = n is lfilter(h, 1, x), n + num_taps - 1 the full convolution."""

    _prefix = "fir"
    _f = property(lambda self: self._h)        # the handle's name before the handles shared a base class

    def __init__(self, num_taps, lib: Library | None = None):
        super().__init__(lib)
        self.num_taps = int(num_taps)
        _check(self.lib, self.lib.vv_dsp_fir_create(self.num_taps, C.byref(self._h)), "vv_dsp_fir_create")
        n, p = _sz(0), _sz(0)
        _check(self.lib, self.lib.vv_dsp_fir_get_config(self._h, C.byref(n), C.byref(p)), "vv_dsp_fir_get_config")
        self.fft_size, self.partitions = int(n.value), int(p.value)

    def filter(self, filters, signals, n_out=None, out=None):
        """filters: [1 or batch, num_taps], signals: [batch, n] float32 (numpy, or torch CUDA tensors).  Returns
        [batch, n_out] float32 (default n_out = n) in the container of `signals` unless `out` is given."""
        filters, nf, taps, fpitch = _rows(filters, "filters")
        signals, batch, n, spitch = _rows(signals, "signals")
        if taps != self.num_taps:
            raise ValueError(f"filters: rows of {taps} taps, the handle was created for {self.num_taps}")
        n_out = n if n_out is None else int(n_out)
        out, opitch = _out_rows(out, signals, batch, n_out)
        self._bind(out, signals, filters)
        st = self.lib.vv_dsp_fir_filter_batch(self._h, _ptr(filters), _space(filters), nf, fpitch, _ptr(signals), _space(signals),
                                              batch, n, spitch, _ptr(out), _space(out), n_out, opitch)
        _check(self.lib, st, "vv_dsp_fir_filter_batch")
        return out


# ----------------------------------------------------------------------------- resampling
class Resampler(_StreamHandle):
    """vv_dsp_resample_poly handle (include/vv_dsp/b200.h): batched rational-ratio resampling by a polyphase FIR on the
    device, scipy.signal.resample_poly(x, up, down, window=taps, padtype='constant') row by row.  taps=None designs scipy's
    default Kaiser (beta 5) filter; up / down are reduced by their gcd."""

    _prefix = "resample_poly"
    _r = property(lambda self: self._h)        # the handle's name before the handles shared a base class

    def __init__(self, up, down, taps=None, lib: Library | None = None):
        super().__init__(lib)
        t = None if taps is None else np.ascontiguousarray(np.asarray(taps, np.float32).ravel())
        st = self.lib.vv_dsp_resample_poly_create(int(up), int(down), None if t is None else t.ctypes.data_as(_vp),
                                                  0 if t is None else t.size, C.byref(self._h))
        _check(self.lib, st, "vv_dsp_resample_poly_create")
        u, d, k, tp = _sz(0), _sz(0), _sz(0), _sz(0)
        _check(self.lib, self.lib.vv_dsp_resample_poly_get_config(self._h, C.byref(u), C.byref(d), C.byref(k), C.byref(tp)),
               "vv_dsp_resample_poly_get_config")
        self.up, self.down, self.num_taps, self.taps_per_phase = int(u.value), int(d.value), int(k.value), int(tp.value)

    def output_length(self, n) -> int:
        """ceil(n up / down)"""
        return int(self.lib.vv_dsp_resample_poly_output_length(self._h, int(n)))

    def resample(self, signals, out=None):
        """signals: [batch, n] float32 (numpy, or a torch CUDA tensor, views with a row pitch included).  Returns
        [batch, output_length(n)] float32 in the container of `signals` unless `out` is given."""
        signals, batch, n, spitch = _rows(signals, "signals")
        out, opitch = _out_rows(out, signals, batch, self.output_length(n))
        self._bind(out, signals)
        got = _sz(0)
        st = self.lib.vv_dsp_resample_poly_batch(self._h, _ptr(signals), _space(signals), batch, n, spitch, _ptr(out), _space(out),
                                                 opitch, C.byref(got))
        _check(self.lib, st, "vv_dsp_resample_poly_batch")
        return out


# ----------------------------------------------------------------------------- IIR second-order sections
PADTYPES = {None: 0, "none": 0, "odd": 1, "even": 2, "constant": 3}


class SosFilter(_StreamHandle):
    """vv_dsp_sos handle (include/vv_dsp/b200.h): batched IIR filtering by a cascade of second-order sections on the
    device, scipy.signal.sosfilt / sosfiltfilt row by row.  sos: [S][6] rows (b0, b1, b2, 1, a1, a2), rounded to float32
    once; every section must have its poles strictly inside the unit circle."""

    _prefix = "sos"

    def __init__(self, sos, lib: Library | None = None):
        super().__init__(lib)
        s = np.ascontiguousarray(np.asarray(sos, np.float32))
        if s.ndim != 2 or s.shape[1] != 6:
            raise ValueError("sos: expected an array of shape (n_sections, 6)")
        _check(self.lib, self.lib.vv_dsp_sos_create(s.ctypes.data_as(_vp), s.shape[0], C.byref(self._h)), "vv_dsp_sos_create")
        ns, seg = _sz(0), _sz(0)
        _check(self.lib, self.lib.vv_dsp_sos_get_config(self._h, C.byref(ns), C.byref(seg)), "vv_dsp_sos_get_config")
        self.n_sections, self.segment_length = int(ns.value), int(seg.value)

    def _state(self, z, batch, what):
        """a [S, batch, 2] float32 state in either space, dense"""
        if _is_device(z):
            _check_device_tensor(z, "float32", what)
            if not z.is_contiguous():
                raise ValueError(f"{what}: expected a contiguous tensor")
        else:
            z = np.ascontiguousarray(z, np.float32)
        if tuple(z.shape) != (self.n_sections, batch, 2):
            raise ValueError(f"{what}: expected shape {(self.n_sections, batch, 2)}, got {tuple(z.shape)}")
        return z

    def filter(self, signals, zi=None, return_zf=False, out=None):
        """scipy.signal.sosfilt(sos, signals, zi=zi) row by row.  signals: [batch, n] float32 (numpy, or a torch CUDA
        tensor, views with a row pitch included); zi: [S, batch, 2] or None (zero state).  Returns the output in the
        container of `signals` unless `out` is given, and (output, zf) when return_zf."""
        signals, batch, n, spitch = _rows(signals, "signals")
        out, opitch = _out_rows(out, signals, batch, n)
        if zi is not None:
            zi = self._state(zi, batch, "zi")
        zf = None
        if return_zf:
            if _is_device(signals):
                import torch
                zf = torch.empty((self.n_sections, batch, 2), device=signals.device, dtype=torch.float32)
            else:
                zf = np.empty((self.n_sections, batch, 2), np.float32)
        self._bind(out, signals, zi, zf)
        st = self.lib.vv_dsp_sos_filter_batch(self._h, _ptr(signals), _space(signals), batch, n, spitch, _ptr(zi), _space(zi),
                                              _ptr(zf), _space(zf), _ptr(out), _space(out), opitch)
        _check(self.lib, st, "vv_dsp_sos_filter_batch")
        return (out, zf) if return_zf else out

    def filtfilt(self, signals, padtype="odd", padlen=None, out=None):
        """scipy.signal.sosfiltfilt(sos, signals, padtype=padtype, padlen=padlen) row by row; padlen=None is scipy's
        default.  Returns the output in the container of `signals` unless `out` is given."""
        if padtype not in PADTYPES:
            raise ValueError(f"padtype: expected one of {sorted(k for k in PADTYPES if k)} or None")
        signals, batch, n, spitch = _rows(signals, "signals")
        out, opitch = _out_rows(out, signals, batch, n)
        self._bind(out, signals)
        st = self.lib.vv_dsp_sos_filtfilt_batch(self._h, _ptr(signals), _space(signals), batch, n, spitch, PADTYPES[padtype],
                                                (1 << 64) - 1 if padlen is None else int(padlen), _ptr(out), _space(out), opitch)
        _check(self.lib, st, "vv_dsp_sos_filtfilt_batch")
        return out


# ----------------------------------------------------------------------------- FFT plan
class FftPlan:
    """vv_dsp_fft_plan: make_plan / execute / destroy (reference include/vv_dsp/spectral/fft.h:190-252)."""

    def __init__(self, n, ftype=FFT_C2C, direction=FFT_FORWARD, lib: Library | None = None):
        self.lib = lib or default_library()
        self.n, self.type, self.dir = int(n), int(ftype), int(direction)
        self._p = _vp()
        st = self.lib.vv_dsp_fft_make_plan(self.n, self.type, self.dir, C.byref(self._p))
        _check(self.lib, st, "vv_dsp_fft_make_plan")

    def execute(self, x):
        n = self.n
        if self.type == FFT_C2C:
            x = np.ascontiguousarray(x, np.complex64); out = np.empty(n, np.complex64)
        elif self.type == FFT_R2C:
            x = np.ascontiguousarray(x, np.float32); out = np.empty(n // 2 + 1, np.complex64)
        else:
            x = np.ascontiguousarray(x, np.complex64); out = np.empty(n, np.float32)
        _check(self.lib, self.lib.vv_dsp_fft_execute(self._p, _ptr(x), _ptr(out)), "vv_dsp_fft_execute")
        return out

    def execute_batch(self, x, out=None, stream=None):
        """x: [batch, n] (C2C complex64 / R2C float32) or [batch, n/2+1] complex64 (C2R); numpy or torch CUDA"""
        dev = _is_device(x)
        n, bins = self.n, self.n // 2 + 1
        if not dev:
            x = np.ascontiguousarray(x, np.float32 if self.type == FFT_R2C else np.complex64)
        batch = int(x.shape[0])
        oshape = (batch, n if self.type != FFT_R2C else bins)
        if out is None:
            if dev:
                import torch
                out = torch.empty(oshape, device=x.device, dtype=torch.float32 if self.type == FFT_C2R else torch.complex64)
            else:
                out = np.empty(oshape, np.float32 if self.type == FFT_C2R else np.complex64)
        st = self.lib.vv_dsp_fft_execute_batch(self._p, _ptr(x), DEVICE if dev else HOST, _ptr(out),
                                               _space(out), batch,
                                               _vp(int(stream) or 1) if stream is not None else None)
        _check(self.lib, st, "vv_dsp_fft_execute_batch")
        return out

    def close(self):
        if getattr(self, "_p", None) is not None and self._p.value:
            self.lib.vv_dsp_fft_destroy(self._p)
            self._p = _vp()

    __del__ = close
