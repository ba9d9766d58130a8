"""CPU tests (-m "not gpu"): the kernel SOURCES and the host library, executed under the
test-only fibre emulator (tests/emu), against the oracle.  This is not a product path --
it exists because the build container has no GPU; the same checks run on the B200 in
test_gpu_parity.py through the nvcc-built library."""
import os
import sys

import pytest

import parity_cases as pc

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def emu():
    sys.path.insert(0, os.path.join(HERE, "emu"))
    import build_emu
    from vv_dsp_b200 import Library
    return Library(build_emu.build())


def test_status_codes(emu):
    pc.check_status_codes(emu)
    pc.check_live_handle_null_args(emu)


def test_reference_known_answers(emu):
    pc.check_reference_known_answers(emu)


@pytest.mark.parametrize("nfft,hop,win", [(2048, 512, "hann"), (256, 64, "hamming"), (64, 32, "hann"), (12, 5, "boxcar")])
def test_per_frame_api(emu, oracle, nfft, hop, win):
    pc.check_per_frame_api(emu, oracle, nfft, hop, win)


@pytest.mark.parametrize("nfft,hop,n", [(256, 64, 2000), (512, 128, 3000), (1024, 256, 5000), (2048, 512, 9000),
                                        (4096, 1024, 14000), (8192, 2048, 30000), (2048, 300, 7000), (100, 30, 900)])
def test_batch_forward_and_inverse(emu, oracle, nfft, hop, n):
    pc.check_batch_forward(emu, oracle, nfft, hop, "hann", n)
    pc.check_batch_inverse(emu, oracle, nfft, hop, "hann", n)


def test_short_and_ragged_inputs(emu, oracle):
    # signal shorter than a frame, shorter than half a frame (multiple reflections), exactly one frame
    for n in (1, 100, 700, 2048, 2049):
        pc.check_batch_forward(emu, oracle, 2048, 512, "hann", n, batch=1)
    pc.check_batch_forward(emu, oracle, 256, 64, "hamming", 3001, batch=3)
    pc.check_batch_inverse(emu, oracle, 256, 256, "boxcar", 2000)


def test_marching_istft_partitions(emu, oracle):
    """fft_size 2048 warp-marching ISTFT: warp ranges that start mid-signal (halo re-synthesis) and span
    signal boundaries; all three instantiated hops; truncated and extended output lengths"""
    for hop in (256, 512, 1024):
        pc.check_batch_inverse(emu, oracle, 2048, hop, "hann", 2048 + hop * 10 + 100, batch=3)
        pc.check_batch_inverse(emu, oracle, 2048, hop, "hamming", 2048 + hop * 37 + 1, batch=5)
    for nfft, hop in ((512, 128), (512, 64), (1024, 256), (1024, 512), (4096, 1024), (4096, 2048), (8192, 2048), (8192, 1024)):
        pc.check_batch_forward(emu, oracle, nfft, hop, "hann", nfft + hop * 9 + 77, batch=3, conventions=("valid", "spectrogram"))
        pc.check_batch_inverse(emu, oracle, nfft, hop, "hann", nfft + hop * 9 + 77, batch=3)
    pc.check_batch_inverse(emu, oracle, 2048, 512, "hann", 2048, batch=2)          # one frame per signal
    pc.check_batch_inverse(emu, oracle, 2048, 512, "hann", 2048 + 511, batch=1)


def test_spectrogram(emu, oracle):
    pc.check_spectrogram(emu, oracle, 512, 128, "hann", 3000)
    pc.check_spectrogram(emu, oracle, 64, 16, "hamming", 40)     # n < nfft: one zero-padded frame


def test_fft_plans(emu, oracle):
    pc.check_fft_plans(emu, oracle, [1, 2, 3, 8, 16, 100, 128, 256, 1024, 2048, 8192])    # 8192: three-pass C2C, 256-thread team


def test_fft_four_step(emu, oracle):
    """powers of two above 8192: two batched Stockham plans + transposes (the reference runs its radix-2 loop at any
    power of two, src/spectral/fft_kiss.c:108-116); C2C both directions, R2C, C2R"""
    pc.check_fft_plans(emu, oracle, [16384])
    pc.check_fft_large(emu, oracle, [16384, 32768])


def test_fft_execute_batch(emu, oracle):
    pc.check_fft_batch(emu, oracle, [1, 8, 100, 128, 256, 1024])


def test_mel(emu, oracle):
    pc.check_mel(emu, oracle, 2048, 512, 80, 48000.0, 12000)
    pc.check_mel(emu, oracle, 512, 128, 26, 16000.0, 6000)


def test_mel_fused(emu, oracle):
    pc.check_mel_fused(emu, oracle, cases=((512, 80, 48000.0), (1024, 40, 16000.0)), n=6000, batch=3)


def test_mel_fused_cta(emu, oracle, capfd):
    pc.check_mel_fused_cta(emu, oracle, cases=((400, 160, 80, 16000.0), (512, 128, 26, 16000.0), (1024, 256, 40, 44100.0), (256, 64, 23, 8000.0),
                                               (320, 160, 40, 16000.0)), n=4000, batch=3, capfd=capfd)


def test_mel_fused_fallback(emu, capfd):
    pc.check_mel_fused_fallback(emu, capfd)


def test_mel_fused_random_filterbanks(emu):
    pc.check_mel_fused_random_filterbanks(emu)


def test_mel_host_pipeline(emu, monkeypatch):
    monkeypatch.setenv("VVB_STAGE_TARGET_BYTES", "100000")            # two signals per chunk: four chunks
    pc.check_mel_host_pipeline(emu)


def test_mfcc(emu, oracle):
    pc.check_mfcc(emu, oracle)


def test_golden_slices(emu, golden):
    pc.check_golden_slices(emu, golden)


def test_config1_voicebank(emu, golden):
    pc.check_config1_voicebank(emu, golden)


def test_accuracy_vs_truth(emu, oracle):
    for nfft in (256, 2048, 8192):
        mine, theirs = pc.check_accuracy_vs_truth(emu, oracle, nfft)
        assert mine < theirs


def test_batch_forward_pcm(emu, monkeypatch):
    monkeypatch.setenv("VVB_STAGE_TARGET_BYTES", "40000")              # three chunks
    pc.check_batch_forward_pcm(emu)


def test_pcm_decode(emu, oracle):
    import os
    pc.check_pcm_decode(emu, oracle, os.path.join(os.path.dirname(__file__), "golden"))


def test_mixed_radix_speech_sizes(emu, oracle):
    print(pc.check_bluestein(emu, oracle, [(400, 160), (320, 80), (480, 160), (640, 160)]))


def test_bluestein_sizes(emu, oracle):
    report = pc.check_bluestein(emu, oracle, [(440, 160), (33, 11), (96, 24), (1000, 250)])
    print("error vs float64 truth (mine, reference):", report)


def test_bluestein_unfused_and_direct_paths(emu, oracle, monkeypatch):
    """the multi-kernel chirp-z pipeline and the O(n^2) kernels stay selectable (read when a plan is created)"""
    monkeypatch.setenv("VVB_BLUESTEIN_UNFUSED", "1")
    pc.check_bluestein(emu, oracle, [(440, 110), (100, 25)])
    monkeypatch.delenv("VVB_BLUESTEIN_UNFUSED")
    monkeypatch.setenv("VVB_NO_BLUESTEIN", "1")
    pc.check_bluestein(emu, oracle, [(100, 25)])


def test_inverse_few_frames(emu, oracle):
    pc.check_inverse_few_frames(emu, oracle, [(256, 64), (512, 256), (1024, 128), (2048, 512)], (1, 2, 3, 5))


def test_reconstruct_non_hermitian(emu, oracle):
    pc.check_reconstruct_non_hermitian(emu, oracle)


def test_staged_chunks_do_not_overlap(emu, monkeypatch):
    one = pc.check_staged_chunks_equal_single(emu, 100, 30, n=900, batch=5)
    monkeypatch.setenv("VVB_STAGE_TARGET_BYTES", str(8 * 1024))
    many = pc.check_staged_chunks_equal_single(emu, 100, 30, n=900, batch=5)
    import numpy as np
    assert np.array_equal(one[0], many[0]) and np.array_equal(one[1], many[1])


@pytest.mark.parametrize("nfft,hop", [(2048, 512), (4096, 1024), (512, 256), (1024, 128)])
def test_stream_sharding_bit_identical(emu, nfft, hop):
    pc.check_stream_sharding(emu, nfft, hop, nfft + hop * 45 + 17, shard_counts=(1, 2, 3))


# reduced route matrix: every kernel family, Hann plus one other window (the full matrix runs in test_gpu_parity.py)
EMU_ROUTES = [(2048, 512, "hamming"), (4096, 1024, "boxcar"), (8192, 2048, "hann"), (1024, 512, "hann"), (256, 32, "hamming"),
              (2048, 441, "hamming"), (512, 75, "boxcar"), (4096, 1000, "hann"), (8192, 441, "hann"), (1024, 100, "hamming"),
              (480, 160, "hamming"), (100, 25, "hann"), (1000, 1000, "hamming"), (31, 9, "hamming")]


@pytest.mark.parametrize("nfft,hop,win", EMU_ROUTES)
def test_route_vs_float64_truth(emu, oracle, capfd, nfft, hop, win):
    """one (fft_size, hop) per kernel family against float64 truth (parity_cases.check_route); the route is asserted from
    the library's VVB_ROUTE_DEBUG lines, and the slot overlap-add cuts one signal into at least 4 chunks"""
    fwd, inv = next((r[2], r[3]) for r in pc.ROUTES if r[:2] == (nfft, hop))
    n = pc.route_length(nfft, hop, inv)
    worst = pc.check_route(emu, oracle, nfft, hop, win, n, batch=2, big_batch=5, capfd=capfd, fwd=fwd, inv=inv,
                           min_chunks=4 if inv == "stft_inverse_kernel" else None)
    print("route", nfft, hop, win, fwd, inv, worst)


@pytest.mark.parametrize("env,nfft,hop,fwd,inv", pc.SWITCH_ROUTES)
def test_switch_route_vs_float64_truth(emu, oracle, capfd, monkeypatch, env, nfft, hop, fwd, inv):
    """the separate-kernel chirp-z pipeline and the O(n^2) kernels, selected by their switches, against float64 truth"""
    monkeypatch.setenv(env, "1")
    pc.check_route(emu, oracle, nfft, hop, "hann", pc.route_length(nfft, hop, inv), big_batch=5, capfd=capfd, fwd=fwd, inv=inv)


@pytest.mark.parametrize("env,nfft,hop,fwd,inv", [(None, 512, 128, "stft_forward_kernel", "stft_inverse_kernel"),
                                                  (None, 400, 160, "stft_forward_kernel", "stft_inverse_kernel"),
                                                  (None, 1000, 250, "chirp_fused_fwd", "chirp_fused_inv"),
                                                  (None, 12, 5, "stft_forward_direct_kernel", "stft_inverse_direct_kernel")]
                         + pc.SWITCH_ROUTES)
def test_per_frame_route_vs_float64_truth(emu, oracle, capfd, monkeypatch, env, nfft, hop, fwd, inv):
    """vv_dsp_stft_process / reconstruct against float64 truth, one row per family (the staged chirp-z one by its switch)"""
    if env:
        monkeypatch.setenv(env, "1")
    pc.check_per_frame_route(emu, oracle, nfft, hop, "hamming", frames=3, capfd=capfd, fwd=fwd, inv=inv)


# one row per log-mel path: fused marching kernel (pair, single), fused generic kernel, chained logmel_tma_kernel (a chirp-z
# size), chained logmel_kernel (> 512 bands)
EMU_LOGMEL_ROUTES = [r for r in pc.LOGMEL_ROUTES if r[:3] in ((2048, 512, 80), (2048, 1024, 40), (400, 160, 80), (1000, 250, 40), (4096, 1024, 600))
                     and r[6] is None]


@pytest.mark.parametrize("nfft,hop,n_mels,sr,route,mode,env", EMU_LOGMEL_ROUTES)
def test_logmel_route_vs_float64_truth(emu, oracle, capfd, nfft, hop, n_mels, sr, route, mode, env):
    win = "hamming" if nfft in (400, 4096) else "hann"
    print(pc.check_logmel_route(emu, oracle, nfft, hop, n_mels, sr, win, route, mode, capfd=capfd, n=nfft + 12 * hop + hop // 3))


@pytest.mark.parametrize("env,nfft,hop,inv", [("VVB_NO_WS", 2048, 256, "istft_march_kernel"),
                                              ("VVB_NO_PAIR", 512, 64, "istft_march_kernel"), ("VVB_NO_PAIR", 1024, 512, "istft_march_kernel"),
                                              ("VVB_NO_PAIR", 256, 128, "stft_inverse_kernel"),
                                              ("VVB_NO_MARCH", 8192, 1024, "stft_inverse_kernel"), ("VVB_NO_MARCH", 1024, 256, "stft_inverse_kernel")])
def test_cross_check_switch_routes(emu, oracle, capfd, monkeypatch, env, nfft, hop, inv):
    """the cross-check kernels behind VVB_NO_WS / VVB_NO_PAIR / VVB_NO_MARCH against float64 truth"""
    monkeypatch.setenv(env, "1")
    fwd = "stft_forward_kernel" if env == "VVB_NO_MARCH" or nfft <= 1024 else "stft_march_kernel"
    pc.check_route(emu, oracle, nfft, hop, "hann", pc.route_length(nfft, hop, None), big_batch=3, capfd=capfd, fwd=fwd, inv=inv)


def test_mel_switches_bit_identical(emu):
    pc.check_mel_switches(emu, cases=((2048, 512, 80, 48000.0), (512, 128, 40, 16000.0), (400, 160, 80, 16000.0)), n=9000)


def test_stream_sharding_without_graphs(emu, monkeypatch):
    monkeypatch.setenv("VVB_STREAM_NO_GRAPH", "1")
    pc.check_stream_sharding(emu, 2048, 512, 2048 + 512 * 45 + 17, shard_counts=(1, 3))
