"""CPU tests (-m "not gpu"): pin the oracle restatement.

 (a) against sha256 digests and slices generated from the real reference (tests/golden/),
 (b) bit for bit against the reference's outputs: digests recorded from it (tests/golden/reference_digests.json),
     and live against oracle/_ref/libvvdsp_ref.so where it was built,
 (c) against the known answers in the reference's own tests (cited per test),
 (d) its accuracy envelope vs float64 (SURVEY.md section 8c).
"""
import json
import os

import numpy as np
import pytest

from _util import noise, sha, rel_l2, stft_truth_f64


# ------------------------------------------------------------------ (a) golden digests
def test_golden_windows(oracle, golden):
    n = 0
    for c in golden["cases"]:
        if c["kind"] != "window":
            continue
        st, w = oracle.window(c["window"], c["n"])
        assert st == c["status"]
        assert sha(w) == c["sha256"], c
        n += 1
    assert n == 24


def test_golden_fft(oracle, golden):
    for c in golden["cases"]:
        if c["kind"] != "fft":
            continue
        n = c["n"]
        rng = np.random.default_rng(c["seed"])
        x = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)
        xr = rng.uniform(-1, 1, n).astype(np.float32)
        assert sha(oracle.fft_c2c(x, +1)) == c["c2c_fwd"], n
        assert sha(oracle.fft_c2c(x, -1)) == c["c2c_bwd"], n
        r2c = oracle.fft_r2c(xr)
        assert sha(r2c) == c["r2c"], n
        if "c2r" in c:
            assert sha(oracle.fft_c2r(r2c, n)) == c["c2r"], n


def test_golden_stft(oracle, golden):
    seen = 0
    for c in golden["cases"]:
        if c["kind"] != "stft":
            continue
        nfft, hop, win, n = c["nfft"], c["hop"], c["window"], c["n"]
        x = noise(c["seed"], n)
        for conv, frames in c["frames"].items():
            assert oracle.num_frames(n, nfft, hop, conv) == frames, (c, conv)
            s = oracle.stft(x, nfft, hop, win, convention=conv)
            assert s.shape[0] == frames
            assert sha(s) == c["sha256"]["stft_" + conv], (nfft, hop, conv)
        assert sha(oracle.roundtrip(x, nfft, hop, win)) == c["sha256"]["roundtrip"]
        assert sha(oracle.batch_roundtrip(x[None], nfft, hop, win)[0]) == c["sha256"]["roundtrip"]
        assert sha(oracle.power(x, nfft, hop, win)) == c["sha256"]["power"]
        assert sha(oracle.spectrogram(x, nfft, hop, win)) == c["sha256"]["spectrogram_mag"]
        sv = oracle.stft(x, nfft, hop, win)
        assert sha(oracle.istft(sv, nfft, hop, n, win)) == c["sha256"]["istft_half_valid"]
        key = f"n{nfft}_h{hop}_{win}_s{c['seed']}"
        if sv.shape[0]:
            assert np.array_equal(sv[0], golden["slices"][key + "_stft_row0"])
            assert np.array_equal(sv[-1], golden["slices"][key + "_stft_rowlast"])
        seen += 1
    assert seen == 12


def test_golden_config1_voicebank(oracle, golden):
    """BASELINE config 1: voicebank/_a'ka'sa.wav, nfft=1024 hop=256 Hann (621 valid frames)."""
    c = [c for c in golden["cases"] if c["kind"] == "config1"][0]
    wav = golden["pcm"].astype(np.float32) / np.float32(32768.0)   # src/audio/wav.c:471-483
    assert wav.size == 159856 and c["frames"] == 621
    assert sha(wav) == c["sha256"]["input"]
    s = oracle.batch_forward(wav[None], 1024, 256)[0]
    assert s.shape == (621, 513)
    assert sha(s) == c["sha256"]["stft_valid"]
    y = oracle.batch_roundtrip(wav[None], 1024, 256)[0]
    assert sha(y) == c["sha256"]["roundtrip"]
    assert sha(oracle.batch_power(wav[None], 1024, 256)[0]) == c["sha256"]["power"]
    assert np.array_equal(y[80000:81024], golden["slices"]["config1_roundtrip_80000"])
    # interior round-trip error of the reference path itself (SURVEY.md 8c: 2.3e-6)
    assert rel_l2(y[1024:-1024], wav[1024:-1024]) < 5e-6


# ------------------------------------------------------------------ (b) bit for bit vs reference
# Each case is (key, what the oracle computes, what the reference library computes from the same input).  Where
# oracle/_ref was built the reference side runs live; the oracle's result must also equal the sha256 digest (or status
# code) recorded from the reference under that key in tests/golden/reference_digests.json, so that the comparison
# holds in every checkout.
def bits(v):
    return int(v) if isinstance(v, (int, np.integer)) else sha(v)


def check_against_reference(oracle, reference, recorded, cases):
    for key, mine, theirs in cases:
        got = bits(mine(oracle))
        assert got == recorded[key], key
        if reference is not None:
            assert got == bits(theirs(reference)), key


LIVE_STFT = [(2048, 512, "hann"), (1024, 256, "hamming"), (96, 40, "hann"), (8, 3, "boxcar")]


def stft_cases(oracle, nfft, hop, win):
    k = f"stft_n{nfft}_h{hop}_{win}/"
    x = np.stack([noise(100 + i, 6000) for i in range(3)])
    yield k + "batch_forward", lambda o: o.batch_forward(x, nfft, hop, win), lambda r: r.batch_forward(x, nfft, hop, win, threads=2)
    yield k + "batch_roundtrip", lambda o: o.batch_roundtrip(x, nfft, hop, win, threads=3), lambda r: r.batch_roundtrip(x, nfft, hop, win)
    yield k + "batch_power", lambda o: o.batch_power(x, nfft, hop, win), lambda r: r.batch_power(x, nfft, hop, win)
    for conv in ("valid", "spectrogram", "padded_tail", "center"):
        yield (k + "stft_" + conv, lambda o, c=conv: o.stft(x[0, :1500], nfft, hop, win, convention=c),
               lambda r, c=conv: r.stft(x[0, :1500], nfft, hop, win, convention=c))
    s = oracle.stft(x[1], nfft, hop, win)
    for norm in (True, False):
        yield (k + f"istft_normalise{int(norm)}", lambda o, m=norm: o.istft(s, nfft, hop, 6000, win, normalise=m),
               lambda r, m=norm: r.istft(s, nfft, hop, 6000, win, normalise=m))
    f = noise(7, nfft)
    yield k + "process", lambda o: o.process(f, nfft, hop, win), lambda r: r.process(f, nfft, hop, win)


def status_cases(oracle):
    for args in [(0, 1, 1), (8, 0, 1), (8, 9, 1), (8, 4, 7), (2, 1, 0), (8, 8, 2)]:
        yield "create_status_{}_{}_{}".format(*args), lambda o, a=args: o.create_status(*a), lambda r, a=args: r.create_status(*a)


MEL_ARGS = [(2048, 80, 48000.0, 0.0, 24000.0), (2048, 128, 48000.0, 20.0, 20000.0), (1024, 40, 44100.0, 0.0, 22050.0),
            (512, 26, 16000.0, 300.0, 8000.0)]
MEL_BAD_ARGS = [(0, 10, 48000.0, 0.0, 100.0), (512, 0, 48000.0, 0.0, 100.0), (512, 300, 48000.0, 0.0, 100.0),
                (512, 10, 48000.0, 0.0, 30000.0), (512, 10, 48000.0, 100.0, 50.0), (512, 10, 48000.0, 0.0, 8000.0, 1)]


def mel_cases(oracle):
    for args in MEL_ARGS:
        k = "mel_n{}_m{}_sr{:g}_{:g}_{:g}/".format(*args)
        yield k + "status", lambda o, a=args: o.mel_filterbank(*a)[0], lambda r, a=args: r.mel_filterbank(*a)[0]
        yield k + "weights", lambda o, a=args: o.mel_filterbank(*a)[1], lambda r, a=args: r.mel_filterbank(*a)[1]
        p = np.random.default_rng(1).uniform(0, 10, (5, args[0] // 2 + 1)).astype(np.float32)
        yield (k + "log_mel", lambda o, a=args, p=p: o.log_mel(p, o.mel_filterbank(*a)[1], 1e-10),
               lambda r, a=args, p=p: r.log_mel(p, r.mel_filterbank(*a)[1], 1e-10))
    for bad in MEL_BAD_ARGS:
        yield ("mel_bad_" + "_".join(f"{v:g}" for v in bad), lambda o, a=bad: o.mel_filterbank(*a)[0],
               lambda r, a=bad: r.mel_filterbank(*a)[0])


def mfcc_cases(oracle):
    rng = np.random.default_rng(5)
    for n_mels, n_coeffs, lifter in ((80, 13, 0.0), (40, 40, 22.0), (26, 12, 22.0), (7, 1, 3.5)):
        lm = rng.normal(-3, 4, (17, n_mels)).astype(np.float32)
        k = f"mfcc_m{n_mels}_c{n_coeffs}_l{lifter:g}/"
        yield k + "status", lambda o, a=(lm, n_coeffs, lifter): o.mfcc(*a)[0], lambda r, a=(lm, n_coeffs, lifter): r.mfcc(*a)[0]
        yield k + "coeffs", lambda o, a=(lm, n_coeffs, lifter): o.mfcc(*a)[1], lambda r, a=(lm, n_coeffs, lifter): r.mfcc(*a)[1]
    lm = np.zeros((2, 8), np.float32)
    for bad in ((0, 0.0, 2), (9, 0.0, 2), (4, -1.0, 2), (4, 0.0, 3), (4, 0.0, 4)):
        yield "mfcc_bad_{}_{:g}_{}".format(*bad), lambda o, a=bad: o.mfcc(lm, *a)[0], lambda r, a=bad: r.mfcc(lm, *a)[0]
    p = rng.uniform(0, 5, (9, 257)).astype(np.float32)
    w = oracle.mel_filterbank(512, 40, 16000.0, 0.0, 8000.0)[1]
    plan = (p, 512, 40, 13, 16000.0, 0.0, 8000.0, 22.0, 1e-10)
    yield "mfcc_plan/status", lambda o: o.mfcc(o.log_mel(p, w, 1e-10), 13, 22.0)[0], lambda r: r.mfcc_plan_process(*plan)[0]
    yield "mfcc_plan/coeffs", lambda o: o.mfcc(o.log_mel(p, w, 1e-10), 13, 22.0)[1], lambda r: r.mfcc_plan_process(*plan)[1]


def write_wav(path, raw, fmt, channels, rate=48000):
    import struct
    bits = abs(fmt)
    tag = 3 if fmt < 0 else 1
    block = channels * bits // 8
    hdr = b"RIFF" + struct.pack("<I", 36 + len(raw)) + b"WAVEfmt " + struct.pack("<IHHIIHH", 16, tag, channels, rate, rate * block,
                                                                                 block, bits) + b"data" + struct.pack("<I", len(raw))
    with open(path, "wb") as f:
        f.write(hdr + raw)


def pcm_cases(oracle, tmp_dir):
    rng = np.random.default_rng(3)
    for fmt in (16, 24, 32, -32):
        for channels in (1, 2):
            n = 1001
            if fmt == -32:
                raw = rng.uniform(-1, 1, n * channels).astype("<f4").tobytes()
            elif fmt == 24:
                v = rng.integers(-2**23, 2**23, n * channels, dtype=np.int64)
                v[:4] = [-2**23, 2**23 - 1, -1, 0]
                raw = b"".join(int(q & 0xFFFFFF).to_bytes(3, "little") for q in v)
            else:
                lim = 2 ** (fmt - 1)
                v = rng.integers(-lim, lim, n * channels, dtype=np.int64)
                v[:4] = [-lim, lim - 1, -1, 0]
                raw = v.astype("<i2" if fmt == 16 else "<i4").tobytes()
            path = os.path.join(tmp_dir, f"t_{fmt}_{channels}.wav")
            write_wav(path, raw, fmt, channels)
            yield (f"pcm_{fmt}_{channels}ch", lambda o, a=(raw, fmt, channels): o.pcm_to_planar(*a),
                   lambda r, p=path: r.wav_read(p))


@pytest.fixture(scope="module")
def recorded():
    return json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")))["digests"]


@pytest.mark.parametrize("nfft,hop,win", LIVE_STFT)
def test_live_against_reference(oracle, reference, recorded, nfft, hop, win):
    check_against_reference(oracle, reference, recorded, stft_cases(oracle, nfft, hop, win))


def test_live_status_codes(oracle, reference, recorded):
    """src/spectral/stft.c:31-34,21-28: NULL->1 (not reachable here), sizes->2, bad enum->3."""
    check_against_reference(oracle, reference, recorded, status_cases(oracle))
    assert oracle.create_status(0, 1, 1) == 2 and oracle.create_status(8, 9, 1) == 2
    assert oracle.create_status(8, 4, 7) == 3 and oracle.create_status(2, 1, 0) == 0


# ------------------------------------------------------------------ (c) the reference's own known answers
def test_framing_goldens(oracle):
    """tests/framing_tests.c:17-45 (frame counts), :56-73 (zero-padded tail), :85-102 (reflect),
    :116-121 (window), :130-150 / :159-192 (overlap-add)."""
    assert oracle.num_frames(1024, 256, 128, "valid") == 7
    assert oracle.num_frames(1024, 256, 128, "center") == 8
    assert oracle.num_frames(100, 256, 128, "valid") == 0
    assert oracle.num_frames(100, 256, 128, "center") == 1
    assert oracle.num_frames(1024, 256, 0, "valid") == 0
    sig = np.arange(10, dtype=np.float32)
    assert oracle.fetch_frame(sig, 4, 2, 0)[1].tolist() == [0, 1, 2, 3]
    assert oracle.fetch_frame(sig, 4, 2, 1)[1].tolist() == [2, 3, 4, 5]
    assert oracle.fetch_frame(sig, 4, 2, 4)[1].tolist() == [8, 9, 0, 0]
    sig1 = np.arange(1, 11, dtype=np.float32)
    assert oracle.fetch_frame(sig1, 4, 2, 0, center=True)[1].tolist() == [2, 1, 1, 2]
    assert oracle.fetch_frame(sig1, 4, 2, 1, center=True)[1].tolist() == [1, 2, 3, 4]
    w = np.array([0.5, 1.0, 1.0, 0.5], np.float32)
    assert oracle.fetch_frame(sig1, 4, 2, 0, window=w)[1].tolist() == [0.5, 2.0, 3.0, 2.0]
    out = np.zeros(8, np.float32)
    oracle.overlap_add(np.array([1, 2, 3, 4], np.float32), out, 2, 0)
    oracle.overlap_add(np.array([0.5, 1, 1.5, 2], np.float32), out, 2, 1)
    assert out.tolist() == [1, 2, 3.5, 5, 1.5, 2, 0, 0]
    out = np.zeros(8, np.float32)
    for i, fr in enumerate([[1, 2, 3, 4], [3, 4, 5, 6], [5, 6, 7, 8]]):
        oracle.overlap_add(np.array(fr, np.float32), out, 2, i)
    assert out.tolist() == [1, 2, 6, 8, 10, 12, 7, 8]
    assert oracle.fetch_frame(sig, 0, 2, 0)[0] == 2   # INVALID_SIZE, framing_tests.c:197-219


def test_frame_count_conventions_at_baseline_shapes(oracle):
    """SURVEY.md 8(a): S / V / C / T at C2, C1, C4."""
    for (n, nfft, hop), exp in {(480000, 2048, 512): (935, 934, 938, 937), (159856, 1024, 256): (622, 621, 625, 624),
                                (172800000, 4096, 1024): (168748, 168747, 168750, 168750)}.items():
        got = tuple(oracle.num_frames(n, nfft, hop, c) for c in ("spectrogram", "valid", "center", "padded_tail"))
        assert got == exp


def test_window_known_answers(oracle):
    """tests/gtest/test_window.cpp:50-68,154-176,212-214; tests/window_tests.c:109-131."""
    for n in (8, 17):
        st, w = oracle.window("hann", n)
        ref = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(n) / (n - 1))
        assert st == 0 and np.abs(w - ref).max() < 1e-6
        assert abs(w[0]) < 1e-6 and abs(w[-1]) < 1e-6
        assert np.abs(w - w[::-1]).max() < 1e-6
    assert oracle.window("hann", 1)[1].tolist() == [1.0]
    assert oracle.window("hann", 0)[0] == 2
    st, w = oracle.window("hamming", 16)
    assert np.abs(w - np.hamming(16)).max() < 1e-6
    assert np.abs(oracle.window("hann", 2048)[1] - np.hanning(2048)).max() < 2e-6   # python/test_stft.py:52


def test_fft_known_answers(oracle):
    """impulse -> ones: tests/spectral_tests.c:14-35 (N=8, 1e-4), tests/fft_backend_tests.c:70-99 (N=16, 1e-5);
    N=1 identity, tone peaks: tests/gtest/test_fft.cpp:190-227,370-408; round trips :155-188,261-304."""
    for n, tol in ((8, 1e-4), (16, 1e-5)):
        x = np.zeros(n, np.complex64)
        x[0] = 1
        X = oracle.fft_c2c(x)
        assert np.abs(X - 1).max() <= tol
    assert oracle.fft_c2c(np.array([3 - 2j], np.complex64))[0] == np.complex64(3 - 2j)
    n = 1024
    X = oracle.fft_c2c(np.exp(2j * np.pi * 10 * np.arange(n) / n).astype(np.complex64))
    assert np.argmax(np.abs(X)) == 10
    rng = np.random.default_rng(5)
    for n in (1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 3, 5, 7, 12, 100, 200):
        x = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)
        tol = 1e-5 if n <= 64 else (5e-5 if n <= 256 else 1e-4)
        assert np.abs(oracle.fft_c2c(oracle.fft_c2c(x, +1), -1) - x).max() < tol
        xr = rng.uniform(-1, 1, n).astype(np.float32)
        X = oracle.fft_r2c(xr)
        assert abs(X[0].imag) < 1e-5
        if n % 2 == 0 and n > 1:
            assert X[-1].imag == 0.0          # src/spectral/fft_kiss.c:140-143
        if n <= 256:
            assert np.abs(oracle.fft_c2r(X, n) - xr).max() < 1e-3
    # python/test_fft.py: n=16 vs numpy at 5e-5
    x = np.random.default_rng(0).standard_normal(16).astype(np.float32)
    assert np.allclose(oracle.fft_r2c(x), np.fft.rfft(x), rtol=5e-5, atol=5e-5)


def test_stft_known_answers(oracle):
    """zero frame -> zero spectrum (tests/gtest/test_stft.cpp:400-407); sine peak (:154-197);
    3-tone round trip nfft=512 hop=128: max<1e-3, RMS<1e-5 on [512,1536) (:452-522);
    tests/spectral_tests.c:83-121 padded-tail round trip MSE<1e-2; python/test_stft.py (5e-2)."""
    assert np.abs(oracle.process(np.zeros(64, np.float32), 64, 16)).max() < 1e-10
    for nfft in (16, 32, 64, 128):
        for win in ("hann", "hamming"):
            t = np.arange(nfft)
            X = oracle.process(np.sin(2 * np.pi * (nfft // 8) * t / nfft).astype(np.float32), nfft, 8, win)
            mag = np.abs(X[: nfft // 2])
            assert mag[0] < 0.1 and abs(int(np.argmax(mag)) - nfft // 8) <= 1 and mag.max() > 1
    n, nfft, hop = 2048, 512, 128
    t = np.arange(n) / 16000.0
    x = (0.5 * np.sin(2 * np.pi * 440 * t) + 0.3 * np.sin(2 * np.pi * 880 * t) + 0.2 * np.sin(2 * np.pi * 1320 * t)).astype(np.float32)
    y = oracle.roundtrip(x, nfft, hop)
    e = (y - x)[512:1536]
    assert np.abs(e).max() < 1e-3 and np.sqrt(np.mean(e.astype(np.float64) ** 2)) < 1e-5
    x = np.sin(2 * np.pi * np.arange(256) / 32.0).astype(np.float32)
    s = oracle.stft(x, 64, 32, convention="padded_tail", half=False)
    assert s.shape[0] == 8
    y = oracle.istft(s, 64, 32, 256, half=False)
    assert np.mean((y - x) ** 2) < 1e-2
    x = np.random.default_rng(2).standard_normal(4096).astype(np.float32)
    y = oracle.roundtrip(x, 512, 128)
    assert np.abs(y - x)[512:-512].max() < 5e-2


# ------------------------------------------------------------------ (d) accuracy envelope
@pytest.mark.parametrize("nfft,bound", [(256, 3e-6), (1024, 8e-6), (2048, 1e-5), (4096, 6e-5), (8192, 1.2e-4)])
def test_oracle_accuracy_envelope(oracle, nfft, bound):
    """SURVEY.md section 0.7 / 8c: the reference's own float32 drift vs float64 grows with N."""
    hop = nfft // 4
    x = noise(40 + nfft, nfft * 6)
    s = oracle.stft(x, nfft, hop)
    w = oracle.window("hann", nfft)[1]
    truth = stft_truth_f64(x, w, nfft, hop, s.shape[0])
    err = np.abs(s - truth).max() / np.abs(truth).max()
    assert err < bound, err


# ------------------------------------------------------------------ groundwork for SURVEY.md 8(f) rank 2
def test_mel_oracle_against_reference(oracle, reference, recorded):
    """The mel filterbank / log-mel restatement (src/features/mel.c:14-245) is bit-exact against the
    compiled reference."""
    check_against_reference(oracle, reference, recorded, mel_cases(oracle))
    for args in MEL_ARGS:
        so, wo = oracle.mel_filterbank(*args)
        assert so == 0 and np.allclose(wo.sum(axis=1), 1.0, atol=1e-5), args


def test_mfcc_oracle_against_reference(oracle, reference, recorded):
    """orc_mfcc (DCT-II of src/spectral/dct.c:21-30 + liftering, src/features/mel.c:249-310) is bit-exact against the
    reference, and so is the plan pipeline power -> log-mel -> MFCC (mel.c:333-450) rebuilt from the oracle's pieces."""
    check_against_reference(oracle, reference, recorded, mfcc_cases(oracle))
    assert all(mine(oracle) == 0 for key, mine, _ in mfcc_cases(oracle) if key.endswith("/status"))


def test_pcm_decode_oracle_against_reference(oracle, reference, recorded, tmp_path):
    """orc_pcm_to_planar (src/audio/wav.c:458-521) is bit-exact against vv_dsp_wav_read of the same bytes, for every
    sample format the reference reads, mono and interleaved stereo, including the extreme codes."""
    check_against_reference(oracle, reference, recorded, pcm_cases(oracle, str(tmp_path)))
