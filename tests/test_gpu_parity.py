"""GPU tests (-m gpu): the product library (nvcc, sm_100a) through its C-ABI against the
oracle on identical seeded inputs, the committed golden slices of the real reference, and --
at BASELINE's full sizes -- size-independent properties (round trip, linearity, Parseval).
Nothing here reads /root/reference."""
import numpy as np
import pytest

import parity_cases as pc
from _util import ROUNDTRIP_REL_L2, noise, rel_l2, spectra_close
from vv_dsp_b200 import FftPlan, Stft

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vv_dsp_b200 import default_library
    lib = default_library()           # raises if the CUDA library is missing: no fallback
    return lib


def test_library_loaded_and_launches(lib, oracle):
    before = lib.kernel_launches()
    pc.check_per_frame_api(lib, oracle, 2048, 512, "hann")
    assert lib.kernel_launches() > before            # the CUDA kernels really ran
    assert "sm_100a" in lib.version()


def test_status_codes(lib):
    pc.check_status_codes(lib)
    pc.check_live_handle_null_args(lib)


def test_reference_known_answers(lib):
    pc.check_reference_known_answers(lib)


@pytest.mark.parametrize("nfft,hop,win", [(2048, 512, "hann"), (1024, 256, "hamming"), (256, 64, "boxcar"),
                                          (4096, 1024, "hann"), (64, 32, "hann"), (12, 5, "boxcar"), (200, 50, "hann"), (400, 160, "hann")])
def test_per_frame_api(lib, oracle, nfft, hop, win):
    pc.check_per_frame_api(lib, oracle, nfft, hop, win)


@pytest.mark.parametrize("nfft,hop,n", [(256, 64, 20000), (512, 128, 20000), (1024, 256, 30000), (2048, 512, 60000),
                                        (4096, 1024, 60000), (8192, 2048, 90000), (2048, 300, 30000),
                                        (2048, 2048, 20000), (100, 30, 3000), (64, 16, 3000)])
def test_batch_forward_and_inverse(lib, oracle, nfft, hop, n):
    pc.check_batch_forward(lib, oracle, nfft, hop, "hann", n, batch=3)
    pc.check_batch_inverse(lib, oracle, nfft, hop, "hann", n, batch=3)


@pytest.mark.parametrize("win", ["boxcar", "hamming"])
def test_other_windows(lib, oracle, win):
    pc.check_batch_forward(lib, oracle, 1024, 256, win, 20000)
    pc.check_batch_inverse(lib, oracle, 1024, 256, win, 20000)


def test_short_and_ragged_inputs(lib, oracle):
    for n in (1, 100, 700, 2048, 2049, 2559, 2560):
        pc.check_batch_forward(lib, oracle, 2048, 512, "hann", n, batch=1)
    pc.check_batch_forward(lib, oracle, 256, 64, "hamming", 3001, batch=5)
    pc.check_batch_inverse(lib, oracle, 256, 256, "boxcar", 2000)
    pc.check_batch_inverse(lib, oracle, 2048, 512, "hann", 2048 + 512 * 3 + 5, batch=1)


def test_marching_istft_partitions(lib, oracle):
    for hop in (256, 512, 1024):
        pc.check_batch_inverse(lib, oracle, 2048, hop, "hann", 2048 + hop * 10 + 100, batch=3)
        pc.check_batch_inverse(lib, oracle, 2048, hop, "hamming", 2048 + hop * 37 + 1, batch=5)
        pc.check_batch_inverse(lib, oracle, 2048, hop, "hann", 300000, batch=9)
    for nfft, hop in ((512, 128), (512, 64), (512, 256), (1024, 256), (1024, 128), (1024, 512), (4096, 1024), (4096, 2048), (4096, 512), (8192, 2048), (8192, 1024), (8192, 4096)):
        pc.check_batch_forward(lib, oracle, nfft, hop, "hann", nfft + hop * 9 + 77, batch=3, conventions=("valid", "spectrogram", "padded_tail"))
        pc.check_batch_inverse(lib, oracle, nfft, hop, "hann", nfft + hop * 9 + 77, batch=3)
        pc.check_batch_inverse(lib, oracle, nfft, hop, "hamming", 400000, batch=5)
    pc.check_batch_inverse(lib, oracle, 2048, 512, "hann", 2048, batch=2)
    pc.check_batch_inverse(lib, oracle, 2048, 512, "hann", 2048 + 511, batch=1)


def test_many_signals_chunking(lib, oracle, capfd):
    """more work items than resident CTAs, several chunks per signal in the ISTFT (hop 100: the slot overlap-add of
    stft_inverse_kernel, which cuts every signal into chunks that re-synthesise their halo frames)"""
    nfft, hop, n, B = 1024, 100, 200000, 7
    x = np.stack([noise(300 + i, n) for i in range(B)])
    from vv_dsp_b200 import Stft
    with Stft(nfft, hop, "hann", lib=lib) as h:
        s = h.batch_forward(x, "complex", "valid")
        ref = oracle.batch_forward(x, nfft, hop, threads=4)
        ok, frac = spectra_close(s, ref)
        assert ok, frac
        y, lines = pc.routed(capfd, lambda: h.batch_inverse(ref, n, True))
        assert pc.launched(lines, "stft_inverse_kernel", nfft) and pc.ola_chunks(lines) >= 2, lines
        refy = np.stack([oracle.istft(ref[i], nfft, hop, n) for i in range(B)])
        assert rel_l2(y[:, nfft:-nfft], refy[:, nfft:-nfft]) < 5e-5
        assert rel_l2(h.batch_inverse(s, n, True)[:, nfft:-nfft], x[:, nfft:-nfft]) < ROUNDTRIP_REL_L2


def test_device_resident_torch_tensors(lib, oracle):
    import torch
    from vv_dsp_b200 import Stft
    nfft, hop, n, B = 2048, 512, 48000, 4
    x = np.stack([noise(400 + i, n) for i in range(B)])
    xd = torch.from_numpy(x).cuda()
    with Stft(nfft, hop, "hann", lib=lib) as h:
        h.set_stream(torch.cuda.current_stream().cuda_stream)
        sd = h.batch_forward(xd, "complex", "valid")
        pd = h.batch_forward(xd, "power", "valid")
        yd = h.batch_inverse(sd, n, True)
        torch.cuda.synchronize()
        ref = oracle.batch_forward(x, nfft, hop, threads=4)
        ok, frac = spectra_close(sd.cpu().numpy(), ref)
        assert ok, frac
        ok, frac = spectra_close(pd.cpu().numpy(), oracle.batch_power(x, nfft, hop, threads=4), rtol=1e-4, atol=1e-4)
        assert ok, frac
        assert rel_l2(yd.cpu().numpy()[:, nfft:-nfft], x[:, nfft:-nfft]) < ROUNDTRIP_REL_L2
        # host-staged and device-resident paths give identical bits
        assert np.array_equal(h.batch_forward(x, "complex", "valid"), sd.cpu().numpy())


def test_stream_ordered_host_mode(lib, oracle):
    """vv_dsp_stft_set_async: same bits as the synchronous host path, many chunks, pinned buffers"""
    import torch
    from vv_dsp_b200 import Stft
    nfft, hop, n, B = 2048, 512, 480000, 260          # > 2 staging chunks of ~100 signals
    xh = torch.empty((B, n), dtype=torch.float32).pin_memory()
    xh.copy_(torch.from_numpy(np.stack([noise(700 + i % 7, n) for i in range(B)])))
    yh = torch.empty((B, n), dtype=torch.float32).pin_memory()
    spec = torch.empty((B, 934, 1025), dtype=torch.complex64, device="cuda")
    with Stft(nfft, hop, "hann", lib=lib) as h:
        ref = h.batch_inverse(h.batch_forward(xh.numpy(), "complex", "valid"), n, True)      # synchronous
        h.set_async(True)
        for _ in range(2):                                                                    # twice: slot reuse
            yh.zero_()
            h.batch_forward(xh.numpy(), "complex", "valid", out=spec)
            h.batch_inverse(spec, n, True, out=yh.numpy())
            h.synchronize()
            assert np.array_equal(yh.numpy(), ref)
        h.set_async(False)
    assert rel_l2(ref[:, nfft:-nfft], xh.numpy()[:, nfft:-nfft]) < ROUNDTRIP_REL_L2


def test_spectrogram(lib, oracle):
    pc.check_spectrogram(lib, oracle, 2048, 512, "hann", 30000)
    pc.check_spectrogram(lib, oracle, 64, 16, "hamming", 40)


def test_fft_plans(lib, oracle):
    pc.check_fft_plans(lib, oracle, [1, 2, 3, 4, 8, 16, 32, 64, 100, 128, 200, 256, 512, 1024, 2048, 4096, 8192])


def test_fft_execute_batch(lib, oracle):
    pc.check_fft_batch(lib, oracle, [1, 2, 8, 16, 100, 128, 200, 256, 512, 1024, 2048, 4096, 8192], batch=7)
    # device-resident, in place for a Stockham size
    import torch
    from vv_dsp_b200 import FftPlan
    x = (torch.randn(64, 1024, device="cuda") + 1j * torch.randn(64, 1024, device="cuda")).to(torch.complex64)
    ref = torch.fft.fft(x.to(torch.complex128), dim=-1)
    p = FftPlan(1024, 0, +1, lib=lib)
    y = x.clone()
    p.execute_batch(y, out=y, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert float((y - ref).abs().max() / ref.abs().max()) < 2e-6


def test_mel(lib, oracle):
    pc.check_mel(lib, oracle, 2048, 512, 80, 48000.0, 60000, batch=5)
    pc.check_mel(lib, oracle, 1024, 256, 40, 44100.0, 30000)
    pc.check_mel(lib, oracle, 4096, 1024, 128, 48000.0, 60000)
    pc.check_mel(lib, oracle, 400, 160, 40, 16000.0, 16000)          # non power of two fft_size (direct path)


@pytest.mark.gpu
def test_mel_fused_kernel_equals_chained_kernels(lib, oracle):
    pc.check_mel_fused(lib, oracle)


@pytest.mark.gpu
def test_mel_fused_in_generic_kernel_equals_chained_kernels(lib, oracle, capfd):
    pc.check_mel_fused_cta(lib, oracle, capfd=capfd)
    pc.check_mel_fused_cta(lib, oracle, cases=((400, 160, 80, 16000.0), (1024, 256, 128, 48000.0)), n=160000, batch=37)


def test_mel_fused_fallback_to_chained_kernels(lib, capfd):
    pc.check_mel_fused_fallback(lib, capfd)


def test_mel_fused_random_filterbanks(lib):
    pc.check_mel_fused_random_filterbanks(lib, seeds=range(25))


def test_mel_host_pipeline(lib, monkeypatch):
    monkeypatch.setenv("VVB_STAGE_TARGET_BYTES", "100000")
    pc.check_mel_host_pipeline(lib)
    monkeypatch.setenv("VVB_STAGE_TARGET_BYTES", "3000000")
    pc.check_mel_host_pipeline(lib, n=200000, batch=11)


def test_mfcc(lib, oracle):
    pc.check_mfcc(lib, oracle)


def test_golden_slices_of_the_real_reference(lib, golden):
    pc.check_golden_slices(lib, golden)


def test_config1_voicebank(lib, golden):
    err = pc.check_config1_voicebank(lib, golden)
    print(f"config1 interior round-trip rel-L2 = {err:.3e}")


@pytest.mark.parametrize("nfft", [256, 1024, 2048, 4096, 8192])
def test_accuracy_vs_float64_truth(lib, oracle, nfft):
    mine, theirs = pc.check_accuracy_vs_truth(lib, oracle, nfft)
    print(f"nfft={nfft}: max err/max|X| vs float64: library {mine:.2e}, oracle {theirs:.2e}")
    assert mine < theirs


def test_full_size_properties_config2_3():
    """BASELINE configs 2/3 at FULL size (1024 x 480000, nfft=2048 hop=512), device-resident:
    frame count, Parseval per frame, linearity, and the STFT->ISTFT round trip."""
    import torch
    from vv_dsp_b200 import Stft
    B, n, nfft, hop = 1024, 480000, 2048, 512
    g = torch.Generator(device="cuda").manual_seed(1234)
    x = torch.rand((B, n), device="cuda", generator=g) * 2 - 1
    with Stft(nfft, hop, "hann") as h:
        h.set_stream(torch.cuda.current_stream().cuda_stream)
        assert h.num_frames(n) == 934
        spec = h.batch_forward(x, "complex", "valid")
        assert tuple(spec.shape) == (B, 934, 1025)
        power = h.batch_forward(x, "power", "valid")
        y = h.batch_inverse(spec, n, True)
        torch.cuda.synchronize()
        # round trip on the interior, every signal
        num = torch.linalg.vector_norm((y - x)[:, nfft:-nfft].double(), dim=1)
        den = torch.linalg.vector_norm(x[:, nfft:-nfft].double(), dim=1)
        assert float((num / den).max()) <= ROUNDTRIP_REL_L2
        # uncovered tail is exactly zero, first sample (w[0] = 0 -> norm 0) is zero
        cov = 933 * hop + nfft
        assert float(y[:, cov:].abs().max()) == 0.0 and float(y[:, 0].abs().max()) == 0.0
        # power == |spec|^2
        p2 = spec.real ** 2 + spec.imag ** 2
        assert float(((power - p2).abs() / (p2.abs().amax(dim=-1, keepdim=True) + 1e-30)).max()) < 1e-6
        # Parseval per frame against the windowed frame energy (checked on a subset of signals)
        w = torch.hann_window(nfft, periodic=False, device="cuda")
        fr = x[:8].unfold(1, nfft, hop) * w
        e_time = (fr.double() ** 2).sum(-1)
        pw = power[:8].double()
        e_freq = (pw[..., 0] + pw[..., -1] + 2 * pw[..., 1:-1].sum(-1)) / nfft
        assert float(((e_time - e_freq).abs() / e_time).max()) < 1e-5
        # linearity: STFT(a x1 + b x2) == a STFT(x1) + b STFT(x2)
        x1, x2 = x[:4], x[4:8]
        lhs = h.batch_forward(0.5 * x1 - 1.5 * x2, "complex", "valid")
        rhs = 0.5 * spec[:4] - 1.5 * spec[4:8]
        torch.cuda.synchronize()
        assert float((lhs - rhs).abs().max() / rhs.abs().max()) < 2e-6
        del spec, power, y, p2


def test_full_size_spot_check_against_oracle(oracle):
    """same full-size batch: 3 signals spot-checked bin by bin against the oracle"""
    import torch
    from vv_dsp_b200 import Stft
    B, n, nfft, hop = 64, 480000, 2048, 512
    x = np.stack([noise(5000 + i, n) for i in range(B)])
    with Stft(nfft, hop, "hann") as h:
        s = h.batch_forward(x, "complex", "valid")
        y = h.batch_inverse(s, n, True)
    for i in (0, 31, 63):
        ref = oracle.stft(x[i], nfft, hop)
        ok, frac = spectra_close(s[i], ref)
        assert ok, (i, frac)
        refy = oracle.istft(ref, nfft, hop, n)
        assert rel_l2(y[i][nfft:-nfft], refy[nfft:-nfft]) < 2e-5


def test_full_size_batch_1024_spot_check_against_oracle(oracle):
    """BASELINE configs 2/3 at their full size (1024 x 480000 samples, device-resident): the first, a middle and the LAST
    signal -- the last CTA's range, where a partition error would sit -- bin by bin against the oracle, and the fused
    log-mel kernel's rows of those signals against the same signals processed alone (range partition independence)."""
    import torch
    from vv_dsp_b200 import Stft, mel_filterbank
    B, n, nfft, hop = 1024, 480000, 2048, 512
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(77)
    x = torch.rand((B, n), device=dev, generator=g) * 2 - 1
    st, w = mel_filterbank(nfft, 80, 48000.0, 0.0, 24000.0)
    assert st == 0
    with Stft(nfft, hop, "hann") as h:
        s = h.batch_forward(x, "complex", "valid")
        y = h.batch_inverse(s, n, True)
        lm = h.batch_logmel(x, w, 1e-10)
        torch.cuda.synchronize()
        for i in (0, 517, B - 1):
            xi = x[i].cpu().numpy()
            ref = oracle.stft(xi, nfft, hop)
            ok, frac = spectra_close(s[i].cpu().numpy(), ref)
            assert ok, (i, frac)
            refy = oracle.istft(ref, nfft, hop, n)
            assert rel_l2(y[i].cpu().numpy()[nfft:-nfft], refy[nfft:-nfft]) < 2e-5
            alone = h.batch_logmel(x[i:i + 1].contiguous(), w, 1e-10)
            torch.cuda.synchronize()
            assert torch.equal(lm[i], alone[0]), i
    del x, s, y, lm
    torch.cuda.empty_cache()


def test_per_frame_api_with_explicit_copies(lib, oracle, monkeypatch):
    """per-frame calls normally run their kernel on the pinned staging buffers (zero-copy); VVB_PERFRAME_STAGED=1 keeps
    the copy + launch + copy sequence: both must give the same bits"""
    x = noise(31, 2048)
    z = (noise(32, 512) + 1j * noise(33, 512)).astype(np.complex64)
    with Stft(2048, 512, "hann", lib=lib) as h:
        a = h.process(x)
    fa = FftPlan(512, 0, +1, lib=lib).execute(z)
    monkeypatch.setenv("VVB_PERFRAME_STAGED", "1")
    pc.check_per_frame_api(lib, oracle, 2048, 512, "hann")
    pc.check_per_frame_api(lib, oracle, 400, 160, "hamming")
    with Stft(2048, 512, "hann", lib=lib) as h:
        b = h.process(x)
    fb = FftPlan(512, 0, +1, lib=lib).execute(z)
    assert np.array_equal(a, b) and np.array_equal(fa, fb)


def test_one_handle_per_thread_concurrently(lib, oracle):
    """INTEGRATION.md section 4: one handle (and one plan) per thread, like the reference (src/spectral/stft.c:13-18).  Four threads
    run different sizes at once -- batched calls, the fused log-mel kernel, the per-frame API and a plan -- and every result
    equals the one computed alone (ctypes releases the GIL, so the calls really overlap)."""
    import threading
    from vv_dsp_b200 import mel_filterbank
    jobs = [(2048, 512), (512, 128), (400, 160), (4096, 1024)]
    xs = [np.stack([noise(2100 + 10 * j + i, 30000) for i in range(4)]) for j in range(len(jobs))]
    st, w = mel_filterbank(2048, 40, 16000.0, 0.0, 8000.0, lib=lib)
    assert st == 0

    def work(j, out):
        nfft, hop = jobs[j]
        res = []
        with Stft(nfft, hop, "hann", lib=lib) as h:
            for _ in range(3):
                s = h.batch_forward(xs[j], "complex", "center")
                y = h.batch_inverse(s, xs[j].shape[1], True)
                res += [s, y]
            if nfft == 2048:
                res.append(h.batch_logmel(xs[j], w, 1e-6))
            res.append(h.process(xs[j][0, :nfft]))
        z = (xs[j][0, :256] + 1j * xs[j][1, :256]).astype(np.complex64)
        res.append(FftPlan(256, 0, +1, lib=lib).execute(z))
        out[j] = res

    alone, together = {}, {}
    for j in range(len(jobs)):
        work(j, alone)
    threads = [threading.Thread(target=work, args=(j, together)) for j in range(len(jobs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for j in range(len(jobs)):
        assert len(alone[j]) == len(together[j])
        for a, b in zip(alone[j], together[j]):
            assert np.array_equal(a, b), jobs[j]


def test_stream_sharding_nccl():
    """config-4 style frame-range sharding over NCCL; needs >= 2 GPUs (skipped on a 1-GPU box)"""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    n = min(torch.cuda.device_count(), 4)
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.join(here, "nccl_stream_check.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "nccl stream sharding ok" in r.stdout


def test_batch_forward_pcm(lib, monkeypatch):
    monkeypatch.setenv("VVB_STAGE_TARGET_BYTES", "40000")
    pc.check_batch_forward_pcm(lib)
    monkeypatch.delenv("VVB_STAGE_TARGET_BYTES")
    pc.check_batch_forward_pcm(lib, 2048, 512, 30000, 5)


def test_pcm_decode(lib, oracle):
    import os
    pc.check_pcm_decode(lib, oracle, os.path.join(os.path.dirname(__file__), "golden"))


def test_bluestein_sizes(lib, oracle):
    report = pc.check_bluestein(lib, oracle, [(400, 160), (33, 11), (96, 24), (480, 120), (1000, 250), (1536, 384), (2000, 500), (2047, 512), (64, 16),
                                              (3000, 750), (4095, 1365)])
    print("error vs float64 truth (mine, reference):", report)


def test_bluestein_above_4096(lib, oracle):
    """non-power-of-two sizes whose chirp-z length exceeds the largest one-kernel transform (M = 16384 ... 131072: four-step
    plans underneath).  The reference serves these with its O(n^2) float DFT (src/spectral/fft_kiss.c:76-92,115)."""
    report = pc.check_bluestein(lib, oracle, [(5000, 1250), (12000, 3000)])
    print("error vs float64 truth (mine, reference):", report)
    rng = np.random.default_rng(5)
    for n in (48000, 100003):                       # plan API only: float64 truth (the O(n^2) oracle would take minutes here)
        z = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)
        xr = rng.uniform(-1, 1, n).astype(np.float32)
        f = FftPlan(n, 0, +1, lib=lib).execute(z)
        t = np.fft.fft(z.astype(np.complex128))
        assert np.abs(f - t).max() <= 3e-6 * np.abs(t).max(), (n, np.abs(f - t).max() / np.abs(t).max())
        back = FftPlan(n, 0, -1, lib=lib).execute(f)
        assert np.abs(back - z).max() < 1e-5
        r = FftPlan(n, 1, +1, lib=lib).execute(xr)
        tr = np.fft.rfft(xr.astype(np.float64))
        assert r.shape == (n // 2 + 1,) and np.abs(r - tr).max() <= 3e-6 * np.abs(tr).max()
        assert np.abs(FftPlan(n, 2, -1, lib=lib).execute(r) - xr).max() < 1e-5


def test_mixed_radix_speech_sizes(lib, oracle, monkeypatch):
    """fft_size 400 / 320 / 480 / 640 (25 / 20 / 30 / 40 ms at 16 kHz) run register Stockham kernels with 5- and 3-point leaves instead
    of the chirp-z transform: same checks against float64 truth and the oracle, several hops, and against the chirp-z path"""
    report = pc.check_bluestein(lib, oracle, [(400, 160), (400, 100), (320, 80), (320, 160), (400, 200), (480, 160), (480, 120), (640, 160)])
    print("error vs float64 truth (mine, reference):", report)
    x = np.stack([noise(900 + i, 16000) for i in range(3)])
    for nfft, hop in ((400, 160), (320, 80), (480, 160), (640, 320)):
        with Stft(nfft, hop, "hann", lib=lib) as h:
            a = h.batch_forward(x, "complex", "center")
        monkeypatch.setenv("VVB_NO_MIXED_RADIX", "1")
        with Stft(nfft, hop, "hann", lib=lib) as h:
            b = h.batch_forward(x, "complex", "center")
        monkeypatch.delenv("VVB_NO_MIXED_RADIX")
        assert np.abs(a - b).max() <= 1e-6 * np.abs(b).max()


def test_bluestein_unfused_and_direct_paths(lib, oracle, monkeypatch):
    """the multi-kernel chirp-z pipeline and the O(n^2) kernels stay selectable (read when a plan is created)"""
    monkeypatch.setenv("VVB_BLUESTEIN_UNFUSED", "1")
    pc.check_bluestein(lib, oracle, [(440, 110), (100, 25)])
    monkeypatch.delenv("VVB_BLUESTEIN_UNFUSED")
    monkeypatch.setenv("VVB_NO_BLUESTEIN", "1")
    pc.check_bluestein(lib, oracle, [(100, 25)])


def test_inverse_few_frames(lib, oracle):
    pc.check_inverse_few_frames(lib, oracle, [(256, 64), (256, 32), (256, 128), (512, 128), (512, 256), (1024, 256), (1024, 128), (1024, 512), (2048, 512), (4096, 1024), (8192, 2048)], (1, 2, 3, 4, 5, 9))


def test_mel_chain_device_buffers(lib, oracle):
    """device-resident signals / outputs of the log-mel and MFCC chains give the same bits as the host-buffer path,
    on a caller-provided stream, with strided (pitched) signal rows"""
    import torch
    from vv_dsp_b200 import Stft, mel_filterbank
    nfft, hop, n_mels = 2048, 512, 80
    _, w = mel_filterbank(nfft, n_mels, 48000.0, 0.0, 24000.0, lib=lib)
    x = np.stack([noise(200 + i, 40000) for i in range(6)])
    s = torch.cuda.Stream()
    big = torch.zeros((6, 40960), device="cuda")
    big[:, :40000] = torch.from_numpy(x).cuda()
    xd = big[:, :40000]                                        # row pitch 40960 != n
    torch.cuda.synchronize()
    with Stft(nfft, hop, "hann", lib=lib) as h:
        lm_host = h.batch_logmel(x, w)
        mf_host = h.batch_mfcc(x, w, 13, lifter=22.0)
        h.set_stream(s.cuda_stream)
        lm_dev = h.batch_logmel(xd, w)
        mf_dev = h.batch_mfcc(xd, w, 13, lifter=22.0)
        s.synchronize()
        assert lm_dev.is_cuda and mf_dev.is_cuda
        assert lm_dev.cpu().numpy().tobytes() == lm_host.tobytes()
        assert mf_dev.cpu().numpy().tobytes() == mf_host.tobytes()


def test_fft_four_step_sizes(lib, oracle):
    """plan API above 8192: four-step C2C / R2C / C2R against the oracle (whose power-of-two path is the radix-2 loop)"""
    pc.check_fft_plans(lib, oracle, [16384])
    print("error vs float64 truth (mine, reference):", pc.check_fft_large(lib, oracle, [16384, 32768, 65536, 1 << 20, 1 << 22]))
    pc.check_fft_batch(lib, oracle, [16384], batch=3)


def test_reconstruct_non_hermitian(lib, oracle):
    pc.check_reconstruct_non_hermitian(lib, oracle)


def test_async_more_chunks_than_the_dependency_ring(lib, oracle, monkeypatch):
    """150 one-signal chunks through the 64-entry dependency ring of the stream-ordered host mode"""
    monkeypatch.setenv("VVB_STAGE_TARGET_BYTES", str(64 * 1024))
    pc.check_async_many_chunks(lib, oracle)


@pytest.mark.parametrize("nfft,hop", [(400, 160), (100, 30), (2048, 512), (3000, 750)])
def test_staged_chunks_do_not_overlap(lib, nfft, hop, monkeypatch):
    """multi-chunk host-staged calls (chirp-z / direct sizes share per-engine scratch) == single-chunk calls"""
    one_spec, one_y = pc.check_staged_chunks_equal_single(lib, nfft, hop)
    monkeypatch.setenv("VVB_STAGE_TARGET_BYTES", str(32 * 1024))
    many_spec, many_y = pc.check_staged_chunks_equal_single(lib, nfft, hop)
    assert np.array_equal(one_spec, many_spec) and np.array_equal(one_y, many_y)


def test_device_calls_follow_torchs_current_stream(lib):
    """No set_stream(): device-tensor calls are enqueued on torch's current stream, so they are ordered against the
    torch ops that produce their inputs and consume their outputs (also on a side stream)."""
    import torch
    nfft, hop, n, B = 2048, 512, 48000, 64
    g = torch.Generator(device="cuda").manual_seed(7)
    base = torch.rand((B, n), device="cuda", generator=g) * 2 - 1
    with Stft(nfft, hop, "hann", lib=lib) as h:
        torch.cuda.synchronize()
        want = h.batch_forward(base * 0.5, "complex", "valid")
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        for s in (torch.cuda.current_stream(), side):
            with torch.cuda.stream(s):
                big = torch.rand((4096, 4096), device="cuda")
                for _ in range(20):
                    big = big @ big * 1e-3                           # keeps the stream busy: the input below is late
                x = base * 0.5                                        # produced on this stream
                spec = h.batch_forward(x, "complex", "valid")
                back = h.batch_inverse(spec, n, True)
                err = (back - x)[:, nfft:-nfft].abs().max()          # consumed on this stream
            torch.cuda.synchronize()
            assert torch.equal(spec, want)
            assert float(err) < 1e-5
        # layout / dtype are checked instead of silently misread
        with pytest.raises(TypeError):
            h.batch_forward(base.double(), "complex", "valid")
        with pytest.raises(ValueError):
            h.batch_forward(base[:, ::2], "complex", "valid")
        # a row pitch larger than the row is honoured: signals and spectra as views into wider buffers
        wide = torch.zeros((B, n + 96), device="cuda"); wide[:, :n] = base * 0.5
        wspec = torch.zeros((B, want.shape[1], h.bins + 3), device="cuda", dtype=torch.complex64)
        h.batch_forward(wide[:, :n], "complex", "valid", out=wspec[:, :, :h.bins])
        torch.cuda.synchronize()
        assert torch.equal(wspec[:, :, :h.bins], want) and float(wspec[:, :, h.bins:].abs().max()) == 0.0
        wy = torch.zeros((B, n + 10), device="cuda")
        h.batch_inverse(wspec[:, :, :h.bins], n, True, out=wy[:, :n])
        torch.cuda.synchronize()
        assert float((wy[:, :n] - base * 0.5)[:, nfft:-nfft].abs().max()) < 1e-5 and float(wy[:, n:].abs().max()) == 0.0


@pytest.mark.parametrize("nfft,hop", [(4096, 1024), (2048, 512), (2048, 256), (8192, 4096), (1024, 256), (512, 64)])
def test_stream_sharding_bit_identical(lib, nfft, hop):
    """BASELINE config 4 in miniature: 1 / 2 / 3 / 5 / 8 shards == the unsharded result, bit for bit"""
    y, x = pc.check_stream_sharding(lib, nfft, hop, nfft + hop * 997 + 123, shard_counts=(1, 2, 3, 5, 8))
    assert rel_l2(y[nfft:-nfft], x[nfft:-nfft]) <= ROUNDTRIP_REL_L2


def test_stream_sharding_over_all_visible_gpus(lib):
    """the same on every GPU the box has (the driver's test box has one: then this is the 1-device case)"""
    import torch
    g = torch.cuda.device_count()
    nfft, hop, n = 4096, 1024, 48000 * 60
    x = noise(77, n)
    with Stft(nfft, hop, "hann", lib=lib) as h:
        spec = h.batch_forward(x[None], "complex", "valid")[0]
        y = h.batch_inverse(spec[None], n, True)[0]
    from vv_dsp_b200 import StftStream
    with StftStream(nfft, hop, n, list(range(g)), lib=lib) as s:
        s.upload(x)
        for _ in range(3):
            s.roundtrip()
        s.synchronize()
        assert np.array_equal(s.download_spectra(), spec)
        assert np.array_equal(s.download(), y)
        assert {s.shard(d).device for d in range(g)} == set(range(g))


@pytest.mark.parametrize("win", ["hann", "hamming", "boxcar"])
@pytest.mark.parametrize("nfft,hop,fwd,inv", pc.ROUTES)
def test_route_vs_float64_truth(lib, oracle, capfd, nfft, hop, fwd, inv, win):
    """Every kernel family at the (fft_size, hop) rows that reach it (parity_cases.ROUTES) against float64 truth, with
    the route read from VVB_ROUTE_DEBUG; stft_inverse_kernel rows cut one signal into >= 4 overlap-add chunks.
    Worst error against truth over the three windows, relative to the per-signal maximum, measured on one NVIDIA B200
    (power limit 1000 W); bounds in parity_cases.TRUTH_*:
      stft_march_kernel    complex 2.3e-7, magnitude 2.4e-7, power 4.3e-7
      stft_forward_kernel  complex 2.4e-7, magnitude 2.9e-7, power 4.9e-7
      istft_ws_kernel      raw 3.4e-7, normalised 1.4e-6, weighted 4.0e-7
      istft_march_kernel   raw 3.9e-7, normalised 1.7e-6, weighted 4.4e-7
      istft_pair_kernel    raw 3.4e-7, normalised 1.2e-6, weighted 3.7e-7
      stft_inverse_kernel  raw 4.1e-7, normalised 1.9e-6, weighted 4.3e-7
    (istft_pair_kernel was at 6.5e-6 normalised and up to 5e-4 weighted before its unpaired last frame stopped adding
    the transform's rounding noise to the tail samples.)
    The rows of the other branches of the dispatcher are held to the same bounds; their worst B200 errors are not measured:
      mixed radix, fft_size 320 / 480 / 400 at hop 400 (stft_forward_kernel, stft_inverse_kernel)
      chirp_fused_kernel MODE 0 / MODE 1 + overlap_add_kernel
      staged chirp-z (chirp_pre_* / chirp_mul / chirp_post_* on four-step plans) + overlap_add_kernel
      stft_forward_direct_kernel, stft_inverse_direct_kernel + overlap_add_kernel
    In the CPU emulator (tests/emu, not a B200 number) these stay below complex 2.8e-7, power 3.9e-7, raw 3.7e-7,
    normalised 1.4e-6, weighted 4.6e-7.  Every row also requires exact zeros in the imaginary parts of the DC and Nyquist bins."""
    worst = pc.check_route(lib, oracle, nfft, hop, win, pc.route_length(nfft, hop, inv), batch=2, big_batch=64, capfd=capfd,
                           fwd=fwd, inv=inv, min_chunks=4 if inv == "stft_inverse_kernel" else None, device_views=True)
    with capfd.disabled():
        print("route", nfft, hop, win, fwd, inv, " ".join(f"{k} {v:.2e}" for k, v in worst.items()))


@pytest.mark.parametrize("hop", [256, 512, 1024])
def test_no_ws_switch(lib, oracle, capfd, monkeypatch, hop):
    """VVB_NO_WS: the ISTFT of fft_size 2048 through istft_march_kernel<Cfg1024> instead of istft_ws_kernel, within the
    truth bounds.  Not bit-identical to the default path: measured on a B200, the raw overlap-add differs in the last bits
    (up to 2.4e-7 of max|y|) and the normalised output by up to 1.3e-6 where the window-sum is above 1e-2."""
    monkeypatch.setenv("VVB_NO_WS", "1")
    for win in ("hann", "hamming", "boxcar"):
        pc.check_route(lib, oracle, 2048, hop, win, pc.route_length(2048, hop, None), capfd=capfd,
                       fwd="stft_march_kernel", inv="istft_march_kernel", device_views=True)


@pytest.mark.parametrize("nfft,hop", [(N, N // d) for N in (256, 512, 1024) for d in (8, 4, 2)])
def test_no_pair_switch(lib, oracle, capfd, monkeypatch, nfft, hop):
    """VVB_NO_PAIR: unsharded ISTFT of fft_size 512 / 1024 through the whole-warp marching kernel, of 256 through the slot
    overlap-add -- within the truth bounds (not claimed bit-identical to istft_pair_kernel)"""
    monkeypatch.setenv("VVB_NO_PAIR", "1")
    inv = "stft_inverse_kernel" if nfft == 256 else "istft_march_kernel"
    for win in ("hann", "hamming", "boxcar"):
        pc.check_route(lib, oracle, nfft, hop, win, pc.route_length(nfft, hop, None), capfd=capfd,
                       fwd="stft_forward_kernel", inv=inv, device_views=True)


@pytest.mark.parametrize("win", ["hann", "hamming", "boxcar"])
@pytest.mark.parametrize("env,nfft,hop,fwd,inv", pc.SWITCH_ROUTES)
def test_switch_route_vs_float64_truth(lib, oracle, capfd, monkeypatch, env, nfft, hop, fwd, inv, win):
    """The chirp-z pipeline of separate kernels (VVB_BLUESTEIN_UNFUSED) and the O(n^2) kernels (VVB_NO_BLUESTEIN) at a size
    that otherwise takes the fused chirp-z kernel: the same checks as test_route_vs_float64_truth."""
    monkeypatch.setenv(env, "1")
    worst = pc.check_route(lib, oracle, nfft, hop, win, pc.route_length(nfft, hop, inv), capfd=capfd, fwd=fwd, inv=inv, device_views=True)
    with capfd.disabled():
        print("route", env, nfft, hop, win, fwd, inv, " ".join(f"{k} {v:.2e}" for k, v in worst.items()))


@pytest.mark.parametrize("nfft,hop,batch,frames", [(5000, 1250, 3, 1000), (16384, 4096, 2, 600)])
def test_staged_chirp_multipass(lib, oracle, capfd, nfft, hop, batch, frames):
    """The staged chirp-z pipeline's work buffer holds 2048 transforms at M = 16384 (fft_size 5000) and 1024 at M = 32768
    (fft_size 16384): 3000 and 1200 transforms in one device-resident call take two passes, the second starting inside a
    signal.  Against float64 truth and bit-identical to each signal alone.  Worst B200 error: not measured."""
    worst = pc.check_multipass(lib, oracle, nfft, hop, batch, frames, capfd=capfd)
    with capfd.disabled():
        print("multipass", nfft, hop, " ".join(f"{k} {v:.2e}" for k, v in worst.items()))


@pytest.mark.parametrize("env,nfft,hop,fwd,inv", [(None, 2048, 512, "stft_march_kernel", "stft_inverse_kernel"),
                                                  (None, 512, 128, "stft_forward_kernel", "stft_inverse_kernel"),
                                                  (None, 400, 160, "stft_forward_kernel", "stft_inverse_kernel"),
                                                  (None, 1000, 250, "chirp_fused_fwd", "chirp_fused_inv"),
                                                  (None, 5000, 1250, "chirp_staged_fwd", "chirp_staged_inv"),
                                                  (None, 12, 5, "stft_forward_direct_kernel", "stft_inverse_direct_kernel")]
                         + pc.SWITCH_ROUTES)
def test_per_frame_route_vs_float64_truth(lib, oracle, capfd, monkeypatch, env, nfft, hop, fwd, inv):
    """vv_dsp_stft_process / reconstruct, one row per kernel family, against float64 truth at the TRUTH_* bounds; the
    synthesis is the per-frame flavour of each family (stft_inverse_kernel without overlap-add, chirp_fused_kernel MODE 1,
    the chirp-z pipeline's frames, the O(n^2) inverse).  Worst B200 error: not measured (complex 2.2e-7, raw 2.8e-7 in the
    CPU emulator)."""
    if env:
        monkeypatch.setenv(env, "1")
    for win in ("hann", "hamming", "boxcar"):
        worst = pc.check_per_frame_route(lib, oracle, nfft, hop, win, capfd=capfd, fwd=fwd, inv=inv)
        with capfd.disabled():
            print("per-frame", env, nfft, hop, win, " ".join(f"{k} {v:.2e}" for k, v in worst.items()))


@pytest.mark.parametrize("win", ["hann", "hamming"])
@pytest.mark.parametrize("nfft,hop,n_mels,sr,route,mode,env", pc.LOGMEL_ROUTES)
def test_logmel_route_vs_float64_truth(lib, oracle, capfd, monkeypatch, nfft, hop, n_mels, sr, route, mode, env, win):
    """Every STFT -> log-mel path (parity_cases.LOGMEL_ROUTES) and the batched MFCC on top, in all four frame conventions,
    against float64 truth: |exp(lm) - (mel + eps)| within TRUTH_LOGMEL times sum_k |w_mk| |X_k| max|X| per band and frame,
    the MFCC within the bound propagated from it.  The route is read from VVB_ROUTE_DEBUG and VVB_MEL_DEBUG.
    Worst error over TRUTH_LOGMEL's term on a B200: not measured (3.4e-7 in the CPU emulator, uniform across the paths)."""
    if env:
        monkeypatch.setenv(env, "1")
    worst = pc.check_logmel_route(lib, oracle, nfft, hop, n_mels, sr, win, route, mode, capfd=capfd)
    with capfd.disabled():
        print("logmel", nfft, hop, n_mels, win, route, mode, env, f"logmel {worst['logmel']:.2e} mfcc/bound {worst['mfcc']:.2e}")


def test_logmel_pcm_vs_float64_truth(lib, oracle):
    pc.check_logmel_pcm_truth(lib, oracle)


@pytest.mark.parametrize("nfft,hop", [(r[0], r[1]) for r in pc.ROUTES if r[3] in ("istft_ws_kernel", "istft_march_kernel", "istft_pair_kernel")])
def test_no_march_switch(lib, oracle, capfd, monkeypatch, nfft, hop):
    """VVB_NO_MARCH: the generic forward kernel and the slot overlap-add for every (fft_size, hop) that normally takes a
    marching, warp-specialised or pair kernel -- within the truth bounds"""
    monkeypatch.setenv("VVB_NO_MARCH", "1")
    for win in ("hann", "hamming", "boxcar"):
        pc.check_route(lib, oracle, nfft, hop, win, pc.route_length(nfft, hop, None), capfd=capfd,
                       fwd="stft_forward_kernel", inv="stft_inverse_kernel", device_views=True)


def test_mel_switches_bit_identical(lib):
    pc.check_mel_switches(lib)


@pytest.mark.parametrize("nfft,hop", [(2048, 512), (4096, 1024), (1024, 256)])
def test_stream_sharding_without_graphs(lib, monkeypatch, nfft, hop):
    """VVB_STREAM_NO_GRAPH: the stream handle's launches enqueued one by one instead of replaying a CUDA graph -- still
    bit-identical to the unsharded calls"""
    monkeypatch.setenv("VVB_STREAM_NO_GRAPH", "1")
    pc.check_stream_sharding(lib, nfft, hop, nfft + hop * 997 + 123, shard_counts=(1, 2, 5))
