"""Parity checks of the library against the oracle, parameterised by the loaded library.

The same functions run (a) on the CPU through tests/emu (kernel sources under the
fibre emulator: test_emu_kernels.py, -m "not gpu") and (b) on the B200 through the
product C-ABI (test_gpu_parity.py, -m gpu).  Tolerances are the north-star's:
spectra |X-Xref| <= 5e-5*max|Xref| + 5e-5*|Xref| (per frame), ISTFT(STFT(x)) interior
relative L2 <= 1e-5; frame counts, padding and indexing bit-exact.
"""
import numpy as np

from _util import ATOL, ROUNDTRIP_REL_L2, RTOL, istft_truth_f64, noise, rel_l2, spectra_close, stft_truth_f64
from vv_dsp_b200 import StftStream, FftPlan, Stft
from vv_dsp_b200.api import VvDspError


def check_per_frame_api(lib, oracle, nfft, hop, win):
    """vv_dsp_stft_process / reconstruct against the oracle's (reference tools/dump_stft_roundtrip.c:44-54)."""
    n = nfft * 3 + 17
    x = noise(900 + nfft, n)
    with Stft(nfft, hop, win, lib=lib) as h:
        recon = np.zeros(n, np.float32); norm = np.zeros(n, np.float32)
        orecon = np.zeros(n, np.float32); onorm = np.zeros(n, np.float32)
        f = 0
        while f * hop + nfft <= n:
            fr = x[f * hop: f * hop + nfft]
            s = h.process(fr)
            so = oracle.process(fr, nfft, hop, win)
            ok, frac = spectra_close(s, so)
            assert ok, (nfft, hop, win, f, frac)
            h.reconstruct(so, recon[f * hop:], norm[f * hop:])      # same input to both sides
            a, b = oracle.reconstruct(so, nfft, hop, win)
            orecon[f * hop: f * hop + nfft] += a
            onorm[f * hop: f * hop + nfft] += b
            f += 1
        assert np.array_equal(norm, onorm)                           # host float32 accumulation: bit-exact
        scale = max(np.abs(orecon).max(), 1e-30)
        assert np.abs(recon - orecon).max() <= 5e-5 * scale, np.abs(recon - orecon).max() / scale


def check_batch_forward(lib, oracle, nfft, hop, win, n, batch=2, conventions=("valid", "spectrogram", "padded_tail", "center")):
    x = np.stack([noise(10 + nfft + i, n) for i in range(batch)])
    worst = 0.0
    with Stft(nfft, hop, win, lib=lib) as h:
        for conv in conventions:
            s = h.batch_forward(x, "complex", conv)
            assert s.shape[1] == oracle.num_frames(n, nfft, hop, conv), conv      # frame counts bit-exact
            ref = np.stack([oracle.stft(x[i], nfft, hop, win, convention=conv) for i in range(batch)])
            ok, frac = spectra_close(s, ref)
            assert ok, (nfft, hop, win, conv, frac)
            worst = max(worst, frac)
        p = h.batch_forward(x, "power", "valid")
        refp = np.stack([oracle.power(x[i], nfft, hop, win) for i in range(batch)])
        ok, frac = spectra_close(p, refp, rtol=2 * RTOL, atol=2 * ATOL)            # |X|^2: twice the relative budget
        assert ok, ("power", nfft, hop, frac)
        m = h.batch_forward(x, "magnitude", "valid")
        ok, frac = spectra_close(m, np.sqrt(refp), rtol=RTOL, atol=ATOL)
        assert ok, ("magnitude", nfft, hop, frac)
    return worst


def check_batch_inverse(lib, oracle, nfft, hop, win, n, batch=2):
    x = np.stack([noise(50 + nfft + i, n) for i in range(batch)])
    with Stft(nfft, hop, win, lib=lib) as h:
        frames = h.num_frames(n)
        spec = np.stack([oracle.stft(x[i], nfft, hop, win) for i in range(batch)])   # same spectra to both sides
        y = h.batch_inverse(spec, n, True)
        raw = h.batch_inverse(spec, n, False)
        refy = np.stack([oracle.istft(spec[i], nfft, hop, n, win) for i in range(batch)])
        refraw = np.stack([oracle.istft(spec[i], nfft, hop, n, win, normalise=False) for i in range(batch)])
        scale = max(np.abs(refraw).max(), 1e-30)
        assert np.abs(raw - refraw).max() <= 5e-5 * scale, np.abs(raw - refraw).max() / scale
        cov = (frames - 1) * hop + nfft if frames else 0
        assert np.all(y[:, cov:] == 0) and np.all(raw[:, cov:] == 0)               # no frame covers: exactly 0
        lo, hi = nfft, n - nfft
        # normalised comparisons only where the divide is well conditioned (Hann/Hamming at hop > nfft/2
        # leave window-sums near zero; the raw overlap-add above is still compared everywhere)
        if hi > lo and (2 * hop <= nfft or win == "boxcar"):
            assert rel_l2(y[:, lo:hi], refy[:, lo:hi]) <= 5e-5
            # the library's own STFT -> ISTFT round trip must meet the north-star bound
            own = h.batch_inverse(h.batch_forward(x, "complex", "valid"), n, True)
            err = rel_l2(own[:, lo:hi], x[:, lo:hi])
            assert err <= ROUNDTRIP_REL_L2, err
            # single-signal host convenience == batch entry
            one = h.istft(spec[0], n)
            assert np.array_equal(one, y[0])
        # truncated / extended output lengths (vv_dsp_overlap_add's drop rule, framing.c:139-145)
        if frames and (2 * hop <= nfft or win == "boxcar"):
            short = h.batch_inverse(spec, n // 2, True)
            refshort = oracle.istft(spec[0], nfft, hop, n // 2, win)
            m = slice(nfft, max(nfft, n // 2 - nfft))
            assert np.allclose(short[0][m], refshort[m], rtol=0, atol=5e-5 * max(np.abs(refshort).max(), 1e-30))


def check_inverse_few_frames(lib, oracle, sizes, frame_counts=(1, 2, 3, 4, 5, 9)):
    """ISTFT of very short signals (1..9 frames: every range is head + tail, odd and even pair counts) and of outputs longer
    than the frames cover, raw and normalised, against the oracle.  Normalised values are compared where the window-sum
    is above 1e-2 (below that the reference's own divide amplifies float32 rounding without bound)."""
    worst = 0.0
    for nfft, hop in sizes:
        w = oracle.window("hann", nfft)[1].astype(np.float64)
        with Stft(nfft, hop, "hann", lib=lib) as h:
            for F in frame_counts:
                n = (F - 1) * hop + nfft
                x = np.stack([noise(3 + F + i, n) for i in range(3)])
                spec = np.stack([oracle.stft(x[i], nfft, hop) for i in range(3)])
                assert spec.shape[1] == F
                for extra in (0, 7, nfft):
                    # float64 truth: overlap-add of irfft(spec) * w in double, and the double window-sum
                    acc, nn = istft_truth_f64(spec, w, nfft, hop, n + extra)
                    good = np.broadcast_to(nn > 1e-2, (3, n + extra))
                    for norm in (False, True):
                        if norm and 2 * hop > nfft:
                            continue
                        y = h.batch_inverse(spec, n + extra, norm)
                        ref = np.stack([oracle.istft(spec[i], nfft, hop, n + extra, "hann", normalise=norm) for i in range(3)])
                        assert np.all(y[:, n:] == 0)                                  # nothing covers: exactly zero
                        if norm:
                            err = np.abs((y - ref)[good]).max() / max(np.abs(ref[good]).max(), 1e-30)
                        else:
                            err = np.abs(y - ref).max() / max(np.abs(ref).max(), 1e-30)
                        worst = max(worst, float(err))
                        # the reference's twiddle recurrence is 2.3e-5 / 4.3e-5 of max|X| off at fft_size 4096 / 8192
                        # (SURVEY.md section 8c) and the divide by a window-sum of 1e-2 amplifies that up to 100 times
                        tol = 1e-4 if (nfft <= 2048 or not norm) else 5e-3
                        assert err < tol, (nfft, hop, F, extra, norm, err)
                        # ... so the binding check for this library is float64 truth at the north-star bound:
                        # overlap-add of irfft(spec) * w in double, divided by the double window-sum
                        if norm:
                            truth = np.where(good, acc / np.where(nn > 1e-2, nn, 1.0), 0.0)
                            terr = np.abs((y - truth)[good]).max() / max(np.abs(truth[good]).max(), 1e-30)
                            # a sample is divided by a window-sum >= 1e-2, which amplifies the float32 rounding of
                            # the synthesis (~2e-7 of max|x|) by up to 100
                            assert terr < 5e-5, ("truth", nfft, hop, F, extra, terr)
                        else:
                            terr = np.abs(y - acc).max() / max(np.abs(acc).max(), 1e-30)
                            assert terr < 1e-5, ("truth", nfft, hop, F, extra, terr)
    return worst


def check_spectrogram(lib, oracle, nfft, hop, win, n):
    x = noise(77 + nfft, n)
    with Stft(nfft, hop, win, lib=lib) as h:
        mag = h.spectrogram(x)
        ref = oracle.spectrogram(x, nfft, hop, win)
        assert mag.shape == ref.shape
        ok, frac = spectra_close(mag, ref)
        assert ok, frac


def check_fft_plans(lib, oracle, sizes):
    rng = np.random.default_rng(3)
    for n in sizes:
        x = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)
        xr = rng.uniform(-1, 1, n).astype(np.float32)
        f = FftPlan(n, 0, +1, lib=lib).execute(x)
        b = FftPlan(n, 0, -1, lib=lib).execute(x)
        r = FftPlan(n, 1, +1, lib=lib).execute(xr)
        c = FftPlan(n, 2, -1, lib=lib).execute(r)
        for got, ref, what in ((f, oracle.fft_c2c(x, +1), "c2c fwd"), (b, oracle.fft_c2c(x, -1), "c2c bwd"),
                               (r, oracle.fft_r2c(xr), "r2c")):
            ok, frac = spectra_close(got, ref)
            assert ok, (n, what, frac)
        if n % 2 == 0 and n > 1:
            assert r[-1].imag == 0.0
        assert np.abs(c - xr).max() < 1e-5, (n, np.abs(c - xr).max())            # reference tolerance is 1e-3
        # forward -> backward round trip (tests/gtest/test_fft.cpp:155-188)
        back = FftPlan(n, 0, -1, lib=lib).execute(f)
        assert np.abs(back - x).max() < 1e-5


def check_fft_large(lib, oracle, sizes):
    """Plan API at powers of two above 8192 (four-step kernels).  The reference's radix-2 loop carries a float32 twiddle
    recurrence whose error grows with n (4.3e-5 of max|X| at 8192, SURVEY.md section 8c), so the yardstick is float64
    truth: this library within 2e-6 of it, and within the triangle bound (own error + the oracle's) of the oracle."""
    rng = np.random.default_rng(31)
    report = {}
    for n in sizes:
        x = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)
        xr = rng.uniform(-1, 1, n).astype(np.float32)
        for direction, truth in ((+1, np.fft.fft(x.astype(np.complex128))), (-1, np.fft.ifft(x.astype(np.complex128)))):
            got = FftPlan(n, 0, direction, lib=lib).execute(x)
            ref = oracle.fft_c2c(x, direction)
            mx = np.abs(truth).max()
            mine, theirs = np.abs(got - truth).max() / mx, np.abs(ref - truth).max() / mx
            assert mine < 2e-6, (n, direction, mine)
            assert np.abs(got - ref).max() / mx <= mine + theirs + 1e-7
            report[(n, direction)] = (float(mine), float(theirs))
        r = FftPlan(n, 1, +1, lib=lib).execute(xr)
        tr = np.fft.rfft(xr.astype(np.float64))
        assert np.abs(r - tr).max() / np.abs(tr).max() < 2e-6 and r[-1].imag == 0.0 and r.shape == (n // 2 + 1,)
        c = FftPlan(n, 2, -1, lib=lib).execute(r)
        assert np.abs(c - xr).max() < 1e-5, (n, np.abs(c - xr).max())
        back = FftPlan(n, 0, -1, lib=lib).execute(FftPlan(n, 0, +1, lib=lib).execute(x))
        assert np.abs(back - x).max() < 1e-5
    return report


def check_fft_batch(lib, oracle, sizes, batch=5):
    """vv_dsp_fft_execute_batch == looping vv_dsp_fft_execute == the oracle, transform by transform"""
    rng = np.random.default_rng(11)
    for n in sizes:
        x = (rng.uniform(-1, 1, (batch, n)) + 1j * rng.uniform(-1, 1, (batch, n))).astype(np.complex64)
        xr = rng.uniform(-1, 1, (batch, n)).astype(np.float32)
        pf, pb, pr, pc = (FftPlan(n, 0, +1, lib=lib), FftPlan(n, 0, -1, lib=lib), FftPlan(n, 1, +1, lib=lib), FftPlan(n, 2, -1, lib=lib))
        F, B, R = pf.execute_batch(x), pb.execute_batch(x), pr.execute_batch(xr)
        Cr = pc.execute_batch(R)
        for i in range(batch):
            for got, ref, what in ((F[i], oracle.fft_c2c(x[i], +1), "c2c fwd"), (B[i], oracle.fft_c2c(x[i], -1), "c2c bwd"),
                                   (R[i], oracle.fft_r2c(xr[i]), "r2c")):
                ok, frac = spectra_close(got, ref)
                assert ok, (n, i, what, frac)
            assert np.array_equal(F[i], pf.execute(x[i])) and np.array_equal(R[i], pr.execute(xr[i]))
            assert np.abs(Cr[i] - xr[i]).max() < 1e-5
        assert np.all(R[:, -1].imag == 0) if n % 2 == 0 and n > 1 else True


def check_mel(lib, oracle, nfft=2048, hop=512, n_mels=80, sr=48000.0, n=30000, batch=3):
    """mel filterbank (host, bit-exact), log-mel on given power (sum order = reference's; logf within 2 ulp),
    and the batched STFT -> log-mel chain against the oracle's process -> power -> log-mel."""
    from vv_dsp_b200 import log_mel_spectrogram, mel_filterbank
    st, w = mel_filterbank(nfft, n_mels, sr, 0.0, sr / 2, lib=lib)
    so, wo = oracle.mel_filterbank(nfft, n_mels, sr, 0.0, sr / 2)
    assert st == so == 0 and w.tobytes() == wo.tobytes()
    for bad in [(0, 10, sr, 0.0, 100.0), (512, 0, sr, 0.0, 100.0), (512, 300, sr, 0.0, 100.0), (512, 10, sr, 0.0, sr),
                (512, 10, sr, 100.0, 50.0), (512, 10, sr, 0.0, 8000.0, 1)]:
        assert mel_filterbank(*bad, lib=lib)[0] == oracle.mel_filterbank(*bad)[0], bad
    p = np.random.default_rng(1).uniform(0, 10, (70, nfft // 2 + 1)).astype(np.float32)
    a, b = log_mel_spectrogram(p, w, 1e-10, lib=lib), oracle.log_mel(p, wo, 1e-10)
    assert np.abs(a - b).max() <= 1e-6                                # same float32 sums; only logf may differ in the last ulp
    # every tile shape of the log-mel kernel: 32/16/8/4 frames per tile, more than 128 bands (two passes),
    # ragged last tile, a single frame
    for nf2, nm2, frames2 in ((256, 40, 100), (512, 200, 67), (4096, 128, 21), (8192, 64, 9), (2048, 150, 1), (16384, 30, 5)):
        st2, w2 = mel_filterbank(nf2, nm2, sr, 20.0, sr / 2, lib=lib)
        assert st2 == 0
        p2 = np.random.default_rng(nf2).uniform(0, 3, (frames2, nf2 // 2 + 1)).astype(np.float32)
        a2, b2 = log_mel_spectrogram(p2, w2, 1e-10, lib=lib), oracle.log_mel(p2, w2, 1e-10)
        assert a2.shape == b2.shape and np.abs(a2 - b2).max() <= 1e-6, (nf2, nm2, frames2)
    x = np.stack([noise(60 + i, n) for i in range(batch)])
    with Stft(nfft, hop, "hann", lib=lib) as h:
        for conv in ("valid", "center"):
            lm = h.batch_logmel(x, w, 1e-10, conv)
            ref = np.stack([oracle.log_mel(np.abs(oracle.stft(x[i], nfft, hop, convention=conv)) ** 2, wo, 1e-10) for i in range(batch)])
            assert lm.shape == ref.shape
            e, er = np.exp(lm.astype(np.float64)), np.exp(ref.astype(np.float64))
            assert np.abs(e - er).max() <= 1e-4 * er.max(), np.abs(e - er).max() / er.max()


def check_mel_fused(lib, oracle, cases=((512, 80, 48000.0), (256, 128, 48000.0), (1024, 40, 16000.0), (512, 23, 8000.0)), n=9000, batch=5):
    """STFT -> log-mel in ONE kernel (fft_size 2048 marching kernel, band sums by the warp that made the frame) against the
    chained power and log-mel kernels (VVB_MEL_UNFUSED=1): bit for bit, every hop with a marching kernel, zero-padded and
    centred frames, filterbanks with short and long schedules; plus a filterbank with an all-zero band, a band whose
    support has holes and negative weights (nothing in the kernel assumes a triangular shape)."""
    import os
    from vv_dsp_b200 import mel_filterbank
    nfft = 2048
    x = np.stack([noise(160 + i, n + 37 * i)[:n] for i in range(batch)])
    rng = np.random.default_rng(9)
    for hop, n_mels, sr in cases:
        st, w = mel_filterbank(nfft, n_mels, sr, 0.0, sr / 2, lib=lib)
        assert st == 0
        banks = [w]
        odd = w.copy()
        odd[1] = 0.0                                                   # an empty band: log(eps)
        odd[n_mels // 2, ::3] = 0.0                                    # holes inside a support
        odd[n_mels - 2] *= -1.0                                        # negative weights (sum + eps stays whatever it is)
        odd[0, :150] = rng.uniform(0, 1e-3, 150).astype(np.float32)      # a wide band out of order
        banks.append(odd)
        with Stft(nfft, hop, "hann", lib=lib) as h:
            for wb in banks:
                for conv in ("valid", "center"):
                    fused = h.batch_logmel(x, wb, 1e-6, conv)
                    os.environ["VVB_MEL_SINGLE"] = "1"                   # one frame per band-sum phase instead of two
                    try:
                        single = h.batch_logmel(x, wb, 1e-6, conv)
                    finally:
                        del os.environ["VVB_MEL_SINGLE"]
                    os.environ["VVB_MEL_UNFUSED"] = "1"
                    try:
                        chained = h.batch_logmel(x, wb, 1e-6, conv)
                    finally:
                        del os.environ["VVB_MEL_UNFUSED"]
                    assert fused.shape == chained.shape
                    assert np.array_equal(fused, chained, equal_nan=True), (hop, n_mels, conv, np.nanmax(np.abs(fused - chained)))
                    assert np.array_equal(single, chained, equal_nan=True), (hop, n_mels, conv)
            ref = np.stack([oracle.log_mel(np.abs(oracle.stft(x[i], nfft, hop)) ** 2, w, 1e-6) for i in range(2)])
            lm = h.batch_logmel(x[:2], w, 1e-6, "valid")
            e, er = np.exp(lm.astype(np.float64)), np.exp(ref.astype(np.float64))
            assert np.abs(e - er).max() <= 1e-4 * er.max()


def check_mel_fused_cta(lib, oracle, cases=((400, 160, 80, 16000.0), (512, 128, 26, 16000.0), (1024, 256, 40, 44100.0), (256, 64, 23, 8000.0),
                                           (320, 160, 40, 16000.0), (480, 160, 64, 16000.0), (640, 160, 80, 16000.0), (512, 100, 128, 48000.0)),
                        n=7000, batch=4, capfd=None):
    """STFT -> log-mel in ONE kernel for the sizes of the generic forward kernel (sub-warp teams: every warp keeps the power rows
    of its frames in shared memory and sums the bands there) against the chained power and log-mel kernels (VVB_MEL_UNFUSED=1): bit for
    bit, zero-padded and centred frames, frame counts that are no multiple of the CTA's frame group, filterbanks with an empty
    band, holes, negative weights and a wide out-of-order band; MFCC on top; and against the oracle's chain.  With capfd the
    library's VVB_MEL_DEBUG line proves which path ran."""
    import os
    from vv_dsp_b200 import mel_filterbank
    rng = np.random.default_rng(19)
    for nfft, hop, n_mels, sr in cases:
        x = np.stack([noise(260 + i, n + 31 * i)[:n] for i in range(batch)])
        st, w = mel_filterbank(nfft, n_mels, sr, 0.0, sr / 2, lib=lib)
        assert st == 0
        odd = w.copy()
        odd[1] = 0.0
        odd[n_mels // 2, ::3] = 0.0
        odd[n_mels - 2] *= -1.0
        odd[0, :nfft // 8] = rng.uniform(0, 1e-3, nfft // 8).astype(np.float32)
        with Stft(nfft, hop, "hann", lib=lib) as h:
            for wb in (w, odd):
                for conv in ("valid", "center"):
                    if capfd is not None:
                        capfd.readouterr()
                        os.environ["VVB_MEL_DEBUG"] = "1"
                    try:
                        fused = h.batch_logmel(x, wb, 1e-6, conv)
                    finally:
                        os.environ.pop("VVB_MEL_DEBUG", None)
                    if capfd is not None:
                        assert "one fused kernel" in capfd.readouterr().err, (nfft, hop)
                    fused_mf = h.batch_mfcc(x, wb, min(13, n_mels), lifter=22.0, log_epsilon=1e-6, convention=conv)
                    os.environ["VVB_MEL_UNFUSED"] = "1"
                    try:
                        chained = h.batch_logmel(x, wb, 1e-6, conv)
                        chained_mf = h.batch_mfcc(x, wb, min(13, n_mels), lifter=22.0, log_epsilon=1e-6, convention=conv)
                    finally:
                        del os.environ["VVB_MEL_UNFUSED"]
                    assert fused.shape == chained.shape
                    assert np.array_equal(fused, chained, equal_nan=True), (nfft, hop, conv, np.nanmax(np.abs(fused - chained)))
                    assert np.array_equal(fused_mf, chained_mf, equal_nan=True), (nfft, hop, conv)
            one = h.batch_logmel(x[1:2, :nfft + 3], w, 1e-6, "valid")    # a single frame, and a signal shorter than a frame
            assert one.shape == (1, 1, n_mels) and np.array_equal(one[0], h.batch_logmel(x[1:2, :nfft + hop], w, 1e-6, "valid")[0, :1])
            assert h.batch_logmel(x[:1, :nfft - 1], w, 1e-6, "valid").shape == (1, 0, n_mels)
            ref = np.stack([oracle.log_mel(np.abs(oracle.stft(x[i], nfft, hop)) ** 2, w, 1e-6) for i in range(2)])
            lm = h.batch_logmel(x[:2], w, 1e-6, "valid")
            e, er = np.exp(lm.astype(np.float64)), np.exp(ref.astype(np.float64))
            assert np.abs(e - er).max() <= 1e-4 * er.max(), (nfft, hop)


def check_mel_fused_fallback(lib, capfd=None):
    """Filterbanks whose band sums do not fit the fused kernel's shared memory (200 bands at fft_size 400) or whose lane schedule
    is too long to build (400 bands at 1024) take the chained kernels -- silently and with the same rows; 128 bands still fuse."""
    import os
    from vv_dsp_b200 import mel_filterbank
    rng = np.random.default_rng(23)
    for nfft, hop, n_mels, sr, expect in ((400, 160, 200, 16000.0, "power kernel + log-mel kernel"), (400, 160, 128, 16000.0, "one fused kernel"),
                                          (1024, 256, 400, 48000.0, "power kernel + log-mel kernel"), (256, 64, 128, 8000.0, "one fused kernel")):
        st, w = mel_filterbank(nfft, n_mels, sr, 0.0, sr / 2, lib=lib)
        assert st == 0
        x = rng.uniform(-1, 1, (3, nfft * 9 + 17)).astype(np.float32)
        with Stft(nfft, hop, "hann", lib=lib) as h:
            if capfd is not None:
                capfd.readouterr()
                os.environ["VVB_MEL_DEBUG"] = "1"
            try:
                a = h.batch_logmel(x, w, 1e-6, "center")
            finally:
                os.environ.pop("VVB_MEL_DEBUG", None)
            if capfd is not None:
                assert expect in capfd.readouterr().err, (nfft, n_mels)
            os.environ["VVB_MEL_UNFUSED"] = "1"
            try:
                b = h.batch_logmel(x, w, 1e-6, "center")
            finally:
                del os.environ["VVB_MEL_UNFUSED"]
            assert a.shape == (3, h.num_frames(x.shape[1], "center"), n_mels) and np.array_equal(a, b), (nfft, n_mels)


def check_mel_fused_random_filterbanks(lib, seeds=range(6), nfft=2048, hop=512):
    """The fused kernel takes ANY weight matrix whose lane schedule fits: random band counts, supports, orders, holes and
    signs, odd and even frame counts per signal (pair flush), against the chained kernels bit for bit."""
    import os
    bins = nfft // 2 + 1
    for seed in seeds:
        rng = np.random.default_rng(1000 + seed)
        n_mels = int(rng.integers(1, 97))
        w = np.zeros((n_mels, bins), np.float32)
        for m in range(n_mels):
            length = int(rng.integers(0, 120))                        # 0: an empty band
            lo = int(rng.integers(0, bins - length + 1))
            vals = rng.uniform(-0.2, 1.0, length).astype(np.float32)
            vals[rng.uniform(size=length) < 0.15] = 0.0
            w[m, lo:lo + length] = vals
        frames = int(rng.integers(1, 6))
        n = nfft + hop * (frames - 1) + int(rng.integers(0, hop))
        x = np.stack([noise(300 + seed * 7 + i, n) for i in range(3)])
        with Stft(nfft, hop, "hann", lib=lib) as h:
            fused = h.batch_logmel(x, w, 1e-3)
            os.environ["VVB_MEL_UNFUSED"] = "1"
            try:
                chained = h.batch_logmel(x, w, 1e-3)
            finally:
                del os.environ["VVB_MEL_UNFUSED"]
        assert fused.shape == chained.shape == (3, frames, n_mels)
        assert np.array_equal(fused, chained, equal_nan=True), (seed, n_mels, frames)


def check_mel_host_pipeline(lib, nfft=2048, hop=512, n=9000, batch=7):
    """host signals through the fused log-mel kernel in several chunks (two staging sets, two streams): the same bytes as
    one device-resident call; log-mel to host and to device memory, MFCC on top"""
    from vv_dsp_b200 import mel_filterbank
    st, w = mel_filterbank(nfft, 40, 16000.0, 0.0, 8000.0, lib=lib)
    assert st == 0
    x = np.stack([noise(2500 + i, n) for i in range(batch)])
    with Stft(nfft, hop, "hann", lib=lib) as h:
        lm = h.batch_logmel(x, w, 1e-6, "center")                     # chunked by VVB_STAGE_TARGET_BYTES (set by the caller)
        mf = h.batch_mfcc(x, w, 13, lifter=22.0, log_epsilon=1e-6, convention="center")
        one = np.stack([h.batch_logmel(x[i:i + 1], w, 1e-6, "center")[0] for i in range(batch)])
        one_mf = np.stack([h.batch_mfcc(x[i:i + 1], w, 13, lifter=22.0, log_epsilon=1e-6, convention="center")[0] for i in range(batch)])
    assert np.array_equal(lm, one) and np.array_equal(mf, one_mf)
    # ... and fed with 16-bit PCM (uploaded undecoded): the same rows as the float call on the decoded samples
    from vv_dsp_b200 import pcm_to_planar
    raw = np.random.default_rng(3).integers(-32768, 32768, (batch, n), dtype=np.int16)
    xf = np.stack([pcm_to_planar(raw[i].tobytes(), 16, 1, lib=lib)[0] for i in range(batch)])
    with Stft(nfft, hop, "hann", lib=lib) as h:
        assert np.array_equal(h.batch_logmel_pcm(raw, w, 16, 1e-6, "center"), h.batch_logmel(xf, w, 1e-6, "center"))
    with Stft(512, 128, "hann", lib=lib) as h:                         # the generic forward kernel's fused flavour
        st2, w2 = mel_filterbank(512, 26, 16000.0, 0.0, 8000.0, lib=lib)
        assert np.array_equal(h.batch_logmel_pcm(raw, w2, 16, 1e-6, "valid"), h.batch_logmel(xf, w2, 1e-6, "valid"))
        # the other WAV sample formats: 24-bit packed, 32-bit PCM, float32
        rng = np.random.default_rng(4)
        r24 = rng.integers(0, 256, (batch, 3 * n), dtype=np.uint8)
        r32 = rng.integers(-2**31, 2**31, (batch, n), dtype=np.int64).astype(np.int32)
        rf = rng.uniform(-1, 1, (batch, n)).astype(np.float32)
        for fmt, rawf in ((24, r24), (32, r32), (-32, rf)):
            dec = np.stack([pcm_to_planar(rawf[i].tobytes(), fmt, 1, lib=lib)[0] for i in range(batch)])
            assert np.array_equal(h.batch_logmel_pcm(rawf, w2, fmt, 1e-6, "center"), h.batch_logmel(dec, w2, 1e-6, "center")), fmt
    with Stft(4096, 1024, "hann", lib=lib) as h:                       # a size without a fused kernel: the chained path
        st3, w3 = mel_filterbank(4096, 40, 48000.0, 0.0, 24000.0, lib=lib)
        assert np.array_equal(h.batch_logmel_pcm(raw, w3, 16, 1e-6, "center"), h.batch_logmel(xf, w3, 1e-6, "center"))


def check_mfcc(lib, oracle):
    """vv_dsp_mfcc, the MFCC plan and the batched STFT -> MFCC chain against the oracle (same float32 sums as the
    reference: only the logf feeding the DCT may differ in the last ulp)."""
    from vv_dsp_b200 import MfccPlan, mel_filterbank, mfcc
    rng = np.random.default_rng(9)
    for n_mels, n_coeffs, lifter, frames in ((80, 13, 22.0, 70), (40, 40, 0.0, 33), (26, 12, 22.0, 1), (128, 20, 5.5, 65)):
        lm = rng.normal(-3, 4, (frames, n_mels)).astype(np.float32)
        st, a = mfcc(lm, n_coeffs, lifter, lib=lib)
        so, b = oracle.mfcc(lm, n_coeffs, lifter)
        assert st == so == 0 and a.tobytes() == b.tobytes(), (n_mels, n_coeffs, lifter)
    lm = np.zeros((2, 8), np.float32)
    for bad in ((0, 0.0, 2), (9, 0.0, 2), (4, -1.0, 2), (4, 0.0, 3), (4, 0.0, 4)):
        assert mfcc(lm, bad[0], bad[1], bad[2], lib=lib)[0] == oracle.mfcc(lm, bad[0], bad[1], bad[2])[0], bad
    # plan: power -> log-mel -> MFCC
    nfft, n_mels, n_coeffs, sr = 512, 40, 13, 16000.0
    p = rng.uniform(0, 5, (37, nfft // 2 + 1)).astype(np.float32)
    _, w = oracle.mel_filterbank(nfft, n_mels, sr, 0.0, sr / 2)
    want = oracle.mfcc(oracle.log_mel(p, w, 1e-10), n_coeffs, 22.0)[1]
    with MfccPlan(nfft, n_mels, n_coeffs, sr, 0.0, sr / 2, lifter=22.0, lib=lib) as plan:
        assert plan.status == 0
        st, got = plan.process(p)
        assert st == 0 and np.abs(got - want).max() <= 2e-5 * max(1.0, np.abs(want).max())
        assert plan.process(np.zeros((0, nfft // 2 + 1), np.float32))[0] == 2
    for bad in ((0, 40, 13, sr, 0.0, 8000.0, 2), (512, 40, 41, sr, 0.0, 8000.0, 3), (512, 40, 13, sr, 0.0, 9000.0, 3),
                (512, 40, 13, 0.0, 0.0, 8000.0, 2)):
        plan = MfccPlan(*bad[:6], lib=lib)
        assert plan.status == bad[6], bad
        plan.close()
    with MfccPlan(nfft, n_mels, n_coeffs, sr, 0.0, sr / 2, dct_type=3, lib=lib) as plan:     # rejected at process time, as in mel.c:249-270
        assert plan.status == 0 and plan.process(p)[0] == 3
    # batched chain
    nfft, hop, n_mels = 1024, 256, 64
    _, w = mel_filterbank(nfft, n_mels, 48000.0, 0.0, 24000.0, lib=lib)
    x = np.stack([noise(80 + i, 12000) for i in range(2)])
    with Stft(nfft, hop, "hann", lib=lib) as h:
        got = h.batch_mfcc(x, w, 20, lifter=22.0)
        lm = h.batch_logmel(x, w)
        want = np.stack([oracle.mfcc(lm[i], 20, 22.0)[1] for i in range(2)])
        assert got.shape == want.shape and got.tobytes() == want.tobytes()       # same log-mel in, same sums


def check_pcm_decode(lib, oracle, golden_dir=None):
    """vv_dsp_b200_pcm_to_planar against the oracle's restatement of the reference's WAV sample conversion: bit-exact
    for every format, mono and stereo, extreme codes, and the config-1 voicebank samples."""
    import ctypes as C
    from vv_dsp_b200 import pcm_to_planar
    rng = np.random.default_rng(3)
    for fmt in (16, 24, 32, -32):
        for channels in (1, 2, 3):
            n = 4099
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
            got = pcm_to_planar(raw, fmt, channels, lib=lib)
            assert got.tobytes() == oracle.pcm_to_planar(raw, fmt, channels).tobytes(), (fmt, channels)
    if golden_dir is not None:
        pcm = np.load(f"{golden_dir}/voicebank_aka_sa_pcm16.npz")["pcm"]
        got = pcm_to_planar(pcm.astype("<i2").tobytes(), 16, 1, lib=lib)[0]
        assert got.tobytes() == (pcm.astype(np.float32) / np.float32(32768.0)).tobytes()
    buf = np.zeros(8, np.uint8)
    out = np.zeros(8, np.float32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)                                      # noqa: E731
    f = lib.vv_dsp_b200_pcm_to_planar
    assert f(None, 0, 16, 4, 1, vp(out), 0, 0, None) == 1 and f(vp(buf), 0, 16, 4, 1, None, 0, 0, None) == 1
    assert f(vp(buf), 0, 8, 4, 1, vp(out), 0, 0, None) == 3 and f(vp(buf), 2, 16, 4, 1, vp(out), 0, 0, None) == 3
    assert f(vp(buf), 0, 16, 0, 1, vp(out), 0, 0, None) == 2 and f(vp(buf), 0, 16, 4, 0, vp(out), 0, 0, None) == 2
    assert f(vp(buf), 0, 16, 4, 1, vp(out), 0, 3, None) == 2


def check_batch_forward_pcm(lib, nfft=512, hop=128, n=5000, batch=7):
    """vv_dsp_stft_batch_forward_pcm: WAV samples uploaded undecoded and converted next to the STFT equal the float call on
    the samples decoded like the reference's reader does (src/audio/wav.c:458-521), bit for bit; several chunks."""
    from vv_dsp_b200 import pcm_to_planar
    rng = np.random.default_rng(12)
    with Stft(nfft, hop, "hann", lib=lib) as h:
        for fmt in (16, 24, 32, -32):
            if fmt == 16:
                raw = rng.integers(-32768, 32768, (batch, n), dtype=np.int16)
            elif fmt == 32:
                raw = rng.integers(-2**31, 2**31, (batch, n), dtype=np.int64).astype(np.int32)
            elif fmt == -32:
                raw = rng.uniform(-1, 1, (batch, n)).astype(np.float32)
            else:
                raw = rng.integers(0, 256, (batch, 3 * n), dtype=np.uint8)
            x = np.stack([pcm_to_planar(raw[i].tobytes(), fmt, 1, lib=lib)[0] for i in range(batch)])
            want = h.batch_forward(x, "complex", "center")
            got = h.batch_forward_pcm(raw, fmt, "complex", "center")
            assert np.array_equal(want, got), fmt
            assert np.array_equal(h.batch_forward(x, "power", "valid"), h.batch_forward_pcm(raw, fmt, "power", "valid")), fmt
        assert lib.vv_dsp_stft_batch_forward_pcm(h._h, 1, 8, 1, n, n, 0, 0, 1, 0, 0, None) == 3      # a format the reader has not
        assert lib.vv_dsp_stft_batch_forward_pcm(h._h, None, 16, 1, n, n, 0, 0, 1, 0, 0, None) == 1


def check_status_codes(lib):
    """Return codes of the reference boundary (SURVEY.md section 4 'lifecycle/validation')."""
    import ctypes as C
    from vv_dsp_b200.api import StftParams
    h = C.c_void_p()
    for (nfft, hop, win), want in (((0, 1, 1), 2), ((8, 0, 1), 2), ((8, 9, 1), 2), ((8, 4, 7), 3)):
        p = StftParams(nfft, hop, win)
        assert lib.vv_dsp_stft_create(C.byref(p), C.byref(h)) == want
        assert not h.value
    assert lib.vv_dsp_stft_create(None, C.byref(h)) == 1
    p = StftParams(8, 4, 1)
    assert lib.vv_dsp_stft_create(C.byref(p), None) == 1
    assert lib.vv_dsp_stft_destroy(None) == 1
    assert lib.vv_dsp_fft_destroy(None) == 0
    plan = C.c_void_p()
    assert lib.vv_dsp_fft_make_plan(0, 0, 1, C.byref(plan)) == 2
    assert lib.vv_dsp_fft_make_plan(8, 5, 1, C.byref(plan)) == 3
    assert lib.vv_dsp_fft_make_plan(8, 0, 0, C.byref(plan)) == 3
    assert lib.vv_dsp_fft_make_plan(8, 0, 1, None) == 1
    assert lib.vv_dsp_fft_execute(None, None, None) == 1
    assert lib.vv_dsp_fft_set_backend(1) == 6 and lib.vv_dsp_fft_set_backend(2) == 6
    assert lib.vv_dsp_fft_set_backend(3) == 3 and lib.vv_dsp_fft_set_backend(0) == 0
    assert lib.vv_dsp_fft_get_backend() == 0
    assert lib.vv_dsp_fft_is_backend_available(0) == 1 and lib.vv_dsp_fft_is_backend_available(1) == 0
    assert lib.vv_dsp_fft_set_fftw_flag(0) == 6 and lib.vv_dsp_fft_flush_fftw_cache() == 6


def check_live_handle_null_args(lib):
    import ctypes as C
    with Stft(16, 8, "hann", lib=lib) as h:
        buf = np.zeros(16, np.complex64)
        assert lib.vv_dsp_stft_process(h._h, None, buf.ctypes.data_as(C.c_void_p)) == 1
        assert lib.vv_dsp_stft_process(h._h, buf.ctypes.data_as(C.c_void_p), None) == 1
        assert lib.vv_dsp_stft_reconstruct(h._h, None, buf.ctypes.data_as(C.c_void_p), None) == 1
        assert np.abs(h.process(np.zeros(16, np.float32))).max() < 1e-10        # zero frame -> zero spectrum
    with Stft(2, 1, "boxcar", lib=lib) as h:                                     # test_stft.cpp:423-449
        s = h.process(np.array([1.0, 2.0], np.float32))
        assert np.allclose(s, [3, -1])


def check_reference_known_answers(lib):
    """The reference's own tolerance tests, run against this library (SURVEY.md section 4)."""
    for n, tol in ((8, 1e-4), (16, 1e-5)):
        x = np.zeros(n, np.complex64); x[0] = 1
        assert np.abs(FftPlan(n, 0, 1, lib=lib).execute(x) - 1).max() <= tol
    assert FftPlan(1, 0, 1, lib=lib).execute(np.array([3 - 2j], np.complex64))[0] == np.complex64(3 - 2j)
    n = 1024
    X = FftPlan(n, 0, 1, lib=lib).execute(np.exp(2j * np.pi * 10 * np.arange(n) / n).astype(np.complex64))
    assert int(np.argmax(np.abs(X))) == 10
    # 3-tone round trip, nfft=512 hop=128 (tests/gtest/test_stft.cpp:452-522): max<1e-3, RMS<1e-5 on [512,1536)
    n, nfft, hop = 2048, 512, 128
    t = np.arange(n) / 16000.0
    x = (0.5 * np.sin(2 * np.pi * 440 * t) + 0.3 * np.sin(2 * np.pi * 880 * t) + 0.2 * np.sin(2 * np.pi * 1320 * t)).astype(np.float32)
    with Stft(nfft, hop, "hann", lib=lib) as h:
        recon = np.zeros(n, np.float32); norm = np.zeros(n, np.float32)
        f = 0
        while f * hop + nfft <= n:
            h.reconstruct(h.process(x[f * hop: f * hop + nfft]), recon[f * hop:], norm[f * hop:])
            f += 1
        y = np.where(norm > 1e-10, recon / np.maximum(norm, 1e-30), recon)
        e = (y - x)[512:1536]
        assert np.abs(e).max() < 1e-3 and np.sqrt(np.mean(e.astype(np.float64) ** 2)) < 1e-5
    # sine peak tests (tests/gtest/test_stft.cpp:154-197)
    for nfft in (16, 32, 64, 128):
        for win in ("hann", "hamming"):
            with Stft(nfft, 8, win, lib=lib) as h:
                X = h.process(np.sin(2 * np.pi * (nfft // 8) * np.arange(nfft) / nfft).astype(np.float32))
                mag = np.abs(X[: nfft // 2])
                assert mag[0] < 0.1 and abs(int(np.argmax(mag)) - nfft // 8) <= 1 and mag.max() > 1


def check_accuracy_vs_truth(lib, oracle, nfft):
    """error vs float64 truth, reported next to the oracle's own (SURVEY.md section 0.7)."""
    hop = nfft // 4
    x = noise(40 + nfft, nfft * 6)
    with Stft(nfft, hop, "hann", lib=lib) as h:
        s = h.batch_forward(x[None], "complex", "valid")[0]
    so = oracle.stft(x, nfft, hop)
    w = oracle.window("hann", nfft)[1]
    truth = stft_truth_f64(x, w, nfft, hop, s.shape[0])
    mine = np.abs(s - truth).max() / np.abs(truth).max()
    theirs = np.abs(so - truth).max() / np.abs(truth).max()
    assert mine < 2e-6, mine            # table twiddles: no growth with N
    return mine, theirs


# Bounds against float64 truth, relative to the per-signal maximum of the truth: about 4 times the worst error of any
# route (test_gpu_parity.py::test_route_vs_float64_truth lists them per kernel family).  The north-star parity bound
# (5e-5) would let a wrong twiddle, a dropped halo frame or a small race through.
TRUTH_COMPLEX = 1e-6          # complex and magnitude spectra
TRUTH_POWER = 2e-6
TRUTH_RAW = 1e-6              # overlap-add without normalisation
TRUTH_NORM = 1e-5             # normalised ISTFT, samples whose window-sum is above 1e-2
TRUTH_WEIGHTED = 2e-6         # normalised ISTFT, every sample with a window-sum above 1e-10, error times sqrt(window-sum)

# kernel family -> the launcher that VVB_ROUTE_DEBUG names, and fft_size / (the M of its Cfg); None: no Cfg parameter
ROUTE_LAUNCHERS = {
    "stft_march_kernel": ("launch_fwd_march_t", 2),
    "stft_forward_kernel": ("launch_forward_t", 2),
    "istft_pair_kernel": ("launch_inv_pair_s", 1),
    "istft_ws_kernel": ("launch_inv_ws_s", None),
    "istft_march_kernel": ("launch_inv_march_s", 2),
    "stft_inverse_kernel": ("launch_inverse_t", 2),          # the slot overlap-add (OLA = true) instantiation
}


def routed(capfd, fn):
    """fn() with VVB_ROUTE_DEBUG=1 and VVB_MEL_DEBUG=1: (its result, the library's stderr lines)"""
    import os
    capfd.readouterr()
    os.environ["VVB_ROUTE_DEBUG"] = "1"
    os.environ["VVB_MEL_DEBUG"] = "1"
    try:
        r = fn()
    finally:
        del os.environ["VVB_ROUTE_DEBUG"], os.environ["VVB_MEL_DEBUG"]
    return r, capfd.readouterr().err.splitlines()


def chirp_m(nfft):
    """length of the chirp-z convolution of a size without a Stockham kernel: the power of two >= 2 fft_size - 1, at least 128"""
    m = 128
    while m < 2 * nfft - 1:
        m *= 2
    return m


def route_needles(family, nfft, frames=False):
    """What VVB_ROUTE_DEBUG prints when `family` runs at this fft_size: a list of groups of substrings, every group on one
    line.  Besides the Stockham families of ROUTE_LAUNCHERS:
      chirp_fused_fwd / chirp_fused_inv: chirp_fused_kernel on the M-point plan (M = chirp_m), MODE 0 analysis / MODE 1
        synthesis;
      chirp_staged_fwd / chirp_staged_inv: the multi-kernel chirp-z pipeline (pre-multiply, M-point transforms, chirp_mul,
        post-multiply) with a four-step plan underneath when M > 8192;
      stft_forward_direct_kernel / stft_inverse_direct_kernel: the O(n^2) kernels;
      logmel_march / logmel_generic: the fused STFT -> log-mel instantiations of stft_march_kernel (fft_size 2048) and of
        the generic forward kernel; logmel_tma_kernel / logmel_kernel: the log-mel kernel of the chained path.
    Inverses of the non-Stockham families end in overlap_add_kernel.  frames: the per-frame synthesis
    (vvb_stft_inverse_frames), which has no overlap-add."""
    if family in ROUTE_LAUNCHERS:
        fn, div = ROUTE_LAUNCHERS[family]
        group = ["vvb: launch ", f"vvb::{fn}("] + ([f"C = Cfg<{nfft // div},"] if div is not None else [])
        if family == "stft_inverse_kernel":
            group.append("bool OLA = false" if frames else "bool OLA = true")
        return [group]
    M = chirp_m(nfft)
    ola = [] if frames else [["vvb: launch overlap_add_kernel in", "vvb_stft_inverse("]]
    fused = lambda mode: [["vvb: launch kern in", "vvb::launch_chirp_fused_m(", f"C = Cfg<{M},", f"int MODE = {mode}]"]]  # noqa: E731
    m_point = [["vvb: launch fourstep_transpose_kernel in"]] if M > 8192 else [["vvb::launch_c2c(", f"C = Cfg<{M},"]]
    staged = lambda pre, post: [[f"vvb: launch {pre} in"], ["vvb: launch chirp_mul_kernel in"], [f"vvb: launch {post} in"]] + m_point  # noqa: E731
    return {
        "chirp_fused_fwd": fused(0),
        "chirp_fused_inv": fused(1) + ola,
        "chirp_staged_fwd": staged("chirp_pre_stft_kernel", "chirp_post_stft_kernel"),
        "chirp_staged_inv": staged("chirp_pre_spec_kernel", "chirp_post_frames_kernel") + ola,
        "stft_forward_direct_kernel": [["vvb: launch stft_forward_direct_kernel in", "vvb_stft_forward("]],
        "stft_inverse_direct_kernel": [["vvb: launch stft_inverse_direct_kernel in",
                                        "vvb_stft_inverse_frames(" if frames else "vvb_stft_inverse("]] + ola,
        "logmel_march": [["vvb: launch kern in", "vvb::launch_fwd_march_t(", "C = Cfg<1024,", "int OUT = 3]"]],
        "logmel_generic": [["vvb: launch kern in", "vvb::launch_forward_logmel(", f"C = Cfg<{nfft // 2},"]],
        "logmel_tma_kernel": [["vvb: launch (logmel_tma_kernel<"]],
        "logmel_kernel": [["vvb: launch logmel_kernel in"]],
    }[family]


def launched(lines, family, nfft, frames=False):
    """did the VVB_ROUTE_DEBUG lines launch `family` in the configuration of this fft_size?  (route_needles)"""
    return all(any(all(s in ln for s in group) for ln in lines) for group in route_needles(family, nfft, frames))


def ola_chunks(lines):
    """chunks per signal of the last stft_inverse_kernel overlap-add launch (VVB_ROUTE_DEBUG)"""
    found = [int(ln.split("chunks_per_signal ")[1].split(",")[0]) for ln in lines if "chunks_per_signal" in ln]
    assert found, lines
    return found[-1]


def _rel(got, truth, axis):
    """worst over signals of max|got - truth| / max|truth|, both maxima per signal"""
    got = np.asarray(got)
    err = np.abs(got.astype(truth.dtype) - truth).max(axis=axis)
    return float((err / np.maximum(np.abs(truth).max(axis=axis), 1e-30)).max())


def check_route(lib, oracle, nfft, hop, win, n, batch=2, big_batch=64, capfd=None, fwd=None, inv=None, min_chunks=None,
                device_views=False):
    """One (fft_size, hop, window) against float64 truth, through whatever kernels the dispatcher picks for it:
      - forward complex in all four frame conventions, power and magnitude of valid frames (stft_truth_f64);
      - inverse raw and normalised (istft_truth_f64), fed with the library's own spectra and with the oracle's;
        normalised samples are compared where the window-sum is above 1e-2, and wherever the library divides with the
        error weighted by sqrt(window-sum); uncovered samples must be exactly zero;
      - the interior round trip at ROUNDTRIP_REL_L2 where the window-sum has no near-zeros;
      - batch invariance: signal 0 alone == signal 0 in a batch of big_batch, forward and inverse, bit for bit (the two
        calls split the signal into different work ranges / overlap-add chunks);
      - with device_views (GPU): input, spectra and output as torch views with odd row pitches (unaligned rows: the
        scalar overlap-add combine and the 32-bit stores of the marching kernels) == the host-buffer results, bit for bit.
    With capfd, the VVB_ROUTE_DEBUG lines of the single-signal calls must name the kernel families fwd / inv, and an
    inverse through stft_inverse_kernel must cut the signal into at least min_chunks chunks.
    Returns the worst error per check relative to the per-signal maximum of the truth."""
    bins = nfft // 2 + 1
    x = np.stack([noise(7000 + nfft + hop + i, n) for i in range(batch)])
    w = oracle.window(win, nfft)[1]
    worst = dict.fromkeys(("complex", "power", "magnitude", "raw", "norm", "weighted"), 0.0)

    def bound(what, e, lim, *ctx):
        worst[what] = max(worst[what], e)
        assert e <= lim, (what, nfft, hop, win, *ctx, e)

    with Stft(nfft, hop, win, lib=lib) as h:
        for conv in ("valid", "spectrogram", "padded_tail", "center"):
            s = h.batch_forward(x, "complex", conv)
            truth = stft_truth_f64(x, w, nfft, hop, convention=conv)
            assert s.shape == truth.shape == (batch, oracle.num_frames(n, nfft, hop, conv), bins), conv
            bound("complex", _rel(s, truth, (1, 2)), TRUTH_COMPLEX, conv)
            # the spectrum of a real frame is real at DC and, for an even fft_size, at Nyquist: exactly, not to rounding
            assert np.all(s[..., 0].imag == 0) and (nfft % 2 == 1 or np.all(s[..., -1].imag == 0)), (nfft, hop, win, conv)
            if conv == "valid":
                spec, tv = s, truth
        F = spec.shape[1]
        bound("power", _rel(h.batch_forward(x, "power", "valid"), np.abs(tv) ** 2, (1, 2)), TRUTH_POWER)
        bound("magnitude", _rel(h.batch_forward(x, "magnitude", "valid"), np.abs(tv), (1, 2)), TRUTH_COMPLEX)

        cov = (F - 1) * hop + nfft
        ospec = np.stack([oracle.stft(x[i], nfft, hop, win) for i in range(batch)])
        for which, sp in (("own", spec), ("oracle", ospec)):
            acc, wsum = istft_truth_f64(sp, w, nfft, hop, n)
            raw = h.batch_inverse(sp, n, False)
            y = h.batch_inverse(sp, n, True)
            bound("raw", _rel(raw, acc, 1), TRUTH_RAW, which)
            good = wsum > 1e-2
            if good.any():
                bound("norm", _rel(y[:, good], acc[:, good] / wsum[good], 1), TRUTH_NORM, which)
            # every sample the library divides, the error weighted by sqrt(window-sum): the synthesis error at a sample
            # scales with the windows that cover it, so this stays at the raw-sum level even where the divide
            # amplifies it (the window tails at both ends of the signal)
            div = wsum > 1e-10
            sc = np.sqrt(wsum[div])
            bound("weighted", _rel(y[:, div] * sc, acc[:, div] / sc, 1), TRUTH_WEIGHTED, which)
            assert np.all(y[:, cov:] == 0) and np.all(raw[:, cov:] == 0), which
            if which == "own":
                own_y, own_raw = y, raw
        lo, hi = nfft, n - nfft
        if hi > lo and (2 * hop <= nfft or win == "boxcar"):
            err = rel_l2(own_y[:, lo:hi], x[:, lo:hi])
            assert err <= ROUNDTRIP_REL_L2, (nfft, hop, win, err)

        # batch invariance (and, with capfd, the route of the single-signal calls)
        call = (lambda f: routed(capfd, f)) if capfd is not None else (lambda f: (f(), []))
        s1, lines_f = call(lambda: h.batch_forward(x[:1], "complex", "valid"))
        y1, lines_i = call(lambda: h.batch_inverse(s1, n, True))
        r1 = h.batch_inverse(s1, n, False)
        assert np.array_equal(s1[0], spec[0]) and np.array_equal(y1[0], own_y[0]) and np.array_equal(r1[0], own_raw[0])
        if big_batch:
            xb = np.concatenate([x[:1], np.stack([noise(9000 + i, n) for i in range(big_batch - 1)])])
            sb = h.batch_forward(xb, "complex", "valid")
            assert np.array_equal(sb[0], s1[0]), (nfft, hop, win, "forward: alone != in a batch")
            assert np.array_equal(h.batch_inverse(sb, n, True)[0], y1[0]), (nfft, hop, win, "inverse: alone != in a batch")
            assert np.array_equal(h.batch_inverse(sb, n, False)[0], r1[0]), (nfft, hop, win, "raw: alone != in a batch")
            del xb, sb
        if capfd is not None:
            assert fwd is None or launched(lines_f, fwd, nfft), (nfft, hop, fwd, lines_f)
            assert inv is None or launched(lines_i, inv, nfft), (nfft, hop, inv, lines_i)
            if min_chunks is not None:
                assert ola_chunks(lines_i) >= min_chunks, (nfft, hop, lines_i)

        if device_views:
            import torch
            assert batch > 1                                       # (a single row has no pitch)
            px = n + (1 if n % 2 == 0 else 2)                      # odd row pitches: rows start at every alignment
            xd = torch.zeros((batch, px), device="cuda")
            xd[:, :n] = torch.from_numpy(x)
            sd = torch.zeros((batch, F, bins + 2), dtype=torch.complex64, device="cuda")
            yd = torch.zeros((batch, px), device="cuda")
            rd = torch.zeros((batch, px), device="cuda")
            h.batch_forward(xd[:, :n], "complex", "valid", out=sd[:, :, :bins])
            h.batch_inverse(sd[:, :, :bins], n, True, out=yd[:, :n])
            h.batch_inverse(sd[:, :, :bins], n, False, out=rd[:, :n])
            torch.cuda.synchronize()
            assert np.array_equal(sd[:, :, :bins].cpu().numpy(), spec) and float(sd[:, :, bins:].abs().max()) == 0.0
            assert np.array_equal(yd[:, :n].cpu().numpy(), own_y) and float(yd[:, n:].abs().max()) == 0.0
            assert np.array_equal(rd[:, :n].cpu().numpy(), own_raw) and float(rd[:, n:].abs().max()) == 0.0
    return worst


# Every STFT / ISTFT kernel family with the (fft_size, hop) rows that reach it: (fft_size, hop, forward family, inverse family).
# Hops 441 and 75 are no multiple of 4 (scalar overlap-add combine); 441 is 10 ms at 44.1 kHz.
ROUTES = ([(2048, h, "stft_march_kernel", "istft_ws_kernel") for h in (256, 512, 1024)]
          + [(N, N // d, "stft_march_kernel", "istft_march_kernel") for N in (4096, 8192) for d in (8, 4, 2)]
          + [(N, N // d, "stft_forward_kernel", "istft_pair_kernel") for N in (256, 512, 1024) for d in (8, 4, 2)]
          + [(N, h, "stft_forward_kernel", "stft_inverse_kernel") for N, h in
             ((256, 100), (512, 75), (1024, 100), (2048, 480), (2048, 441), (4096, 1000), (4096, 441), (4096, 4096),
              (8192, 441), (8192, 3000), (400, 160), (640, 160))]
          # mixed radix (3- and 5-point leaves): 320 and 480 besides 400 / 640 above; hop = fft_size leaves window-sum zeros
          + [(N, h, "stft_forward_kernel", "stft_inverse_kernel") for N, h in ((320, 80), (320, 160), (480, 120), (480, 160), (400, 400))]
          # chirp-z in one kernel per transform (M <= 8192), the powers of two below 256 included
          + [(N, h, "chirp_fused_fwd", "chirp_fused_inv") for N, h in
             ((64, 16), (128, 32), (100, 25), (440, 110), (1000, 250), (2047, 512), (4095, 1365), (1000, 1000))]
          # chirp-z through the multi-kernel pipeline on four-step plans (M = 16384, 32768)
          + [(N, h, "chirp_staged_fwd", "chirp_staged_inv") for N, h in ((5000, 1250), (16384, 4096))]
          # O(n^2) kernels (n < 32)
          + [(N, h, "stft_forward_direct_kernel", "stft_inverse_direct_kernel") for N, h in ((12, 5), (24, 6), (31, 9), (30, 30))])

# rows that reach a family only under a selection switch (read when a handle is created): (switch, fft_size, hop, fwd, inv)
SWITCH_ROUTES = [("VVB_BLUESTEIN_UNFUSED", 440, 110, "chirp_staged_fwd", "chirp_staged_inv"),
                 ("VVB_NO_BLUESTEIN", 100, 25, "stft_forward_direct_kernel", "stft_inverse_direct_kernel")]

# frames per round (teams G per CTA) of stft_inverse_kernel at each fft_size: 256 threads / (fft_size/2 / points per thread)
OLA_TEAMS = {256: 32, 512: 16, 1024: 16, 2048: 8, 4096: 4, 8192: 2, 320: 32, 400: 64, 480: 64, 640: 16}


def route_length(nfft, hop, inv, chunks=4):
    """Signal length for a route row.  Where the inverse is stft_inverse_kernel: enough frames for the slot overlap-add
    to cut ONE signal into `chunks` chunks (it keeps >= 16 rounds of G frames per chunk), with a ragged last chunk;
    elsewhere 41 frames.  A ragged tail after the last frame either way."""
    frames = 16 * OLA_TEAMS[nfft] * chunks + OLA_TEAMS[nfft] // 2 + 3 if inv == "stft_inverse_kernel" else 41
    return (frames - 1) * hop + nfft + hop // 3


def check_per_frame_route(lib, oracle, nfft, hop, win, frames=5, capfd=None, fwd=None, inv=None):
    """vv_dsp_stft_process / reconstruct against float64 truth at the TRUTH_* bounds: the spectrum of each frame (all fft_size
    bins) against the float64 DFT of the windowed frame, and the frame that reconstruct adds (vvb_stft_inverse_frames: the
    synthesis without overlap-add) against the float64 inverse DFT of the same spectrum times the window; the window-sum it
    adds is the float32 w*w.  With capfd the VVB_ROUTE_DEBUG lines must name fwd and inv (its per-frame flavour)."""
    w = oracle.window(win, nfft)[1]
    x = noise(1300 + nfft + hop, (frames - 1) * hop + nfft)
    worst = {"complex": 0.0, "raw": 0.0}
    call = (lambda f: routed(capfd, f)) if capfd is not None else (lambda f: (f(), []))
    with Stft(nfft, hop, win, lib=lib) as h:
        for f in range(frames):
            fr = x[f * hop: f * hop + nfft]
            s, lines_f = call(lambda: h.process(fr))
            truth = np.fft.fft(fr.astype(np.float64) * w)
            e = _rel(s, truth, None)
            worst["complex"] = max(worst["complex"], e)
            assert e <= TRUTH_COMPLEX, ("process", nfft, hop, win, f, e)
            assert s[0].imag == 0 and (nfft % 2 == 1 or s[nfft // 2].imag == 0), ("process", nfft, hop, win, f)
            out = np.zeros(nfft, np.float32)
            norm = np.zeros(nfft, np.float32)
            _, lines_i = call(lambda: h.reconstruct(s, out, norm))
            frame_truth = np.fft.ifft(s.astype(np.complex128)).real * w
            e = _rel(out, frame_truth, None)
            worst["raw"] = max(worst["raw"], e)
            assert e <= TRUTH_RAW, ("reconstruct", nfft, hop, win, f, e)
            assert np.array_equal(norm, w * w)
            if capfd is not None:
                assert fwd is None or launched(lines_f, fwd, nfft), (nfft, hop, fwd, lines_f)
                assert inv is None or launched(lines_i, inv, nfft, frames=True), (nfft, hop, inv, lines_i)
    return worst


def check_multipass(lib, oracle, nfft, hop, batch, frames, win="hann", capfd=None, min_passes=2):
    """The staged chirp-z pipeline over more transforms than its work buffer holds (chirp_reserve caps it at 256 MB, the
    four-step plans underneath alike): device-resident signals, so one call carries batch * frames transforms and the pass
    boundaries fall inside a signal.  Spectra, raw and normalised ISTFT against float64 truth at the TRUTH_* bounds, and bit
    for bit equal to each signal run alone.  With capfd: the pipeline ran min_passes passes or more, forward and inverse."""
    import torch
    n = (frames - 1) * hop + nfft + hop // 3
    x = np.stack([noise(1700 + nfft + i, n) for i in range(batch)])
    w = oracle.window(win, nfft)[1]
    xd = torch.from_numpy(x).cuda()
    call = (lambda f: routed(capfd, f)) if capfd is not None else (lambda f: (f(), []))
    worst = {}
    with Stft(nfft, hop, win, lib=lib) as h:
        def fwd():
            r = h.batch_forward(xd, "complex", "valid")
            torch.cuda.synchronize()
            return r
        sd, lines_f = call(fwd)
        assert tuple(sd.shape) == (batch, frames, nfft // 2 + 1)

        def inv(norm):
            r = h.batch_inverse(sd, n, norm)
            torch.cuda.synchronize()
            return r.cpu().numpy()
        y, lines_i = call(lambda: inv(True))
        raw = inv(False)
        s = sd.cpu().numpy()
        if capfd is not None:
            assert launched(lines_f, "chirp_staged_fwd", nfft) and launched(lines_i, "chirp_staged_inv", nfft), (lines_f, lines_i)
            for lines, kern in ((lines_f, "chirp_pre_stft_kernel"), (lines_i, "chirp_pre_spec_kernel")):
                passes = sum(f"vvb: launch {kern} in" in ln for ln in lines)
                assert passes >= min_passes, (nfft, kern, passes)
        worst["complex"] = _rel(s, stft_truth_f64(x, w, nfft, hop), (1, 2))
        assert worst["complex"] <= TRUTH_COMPLEX, worst
        acc, wsum = istft_truth_f64(s, w, nfft, hop, n)
        worst["raw"] = _rel(raw, acc, 1)
        assert worst["raw"] <= TRUTH_RAW, worst
        good = wsum > 1e-2
        worst["norm"] = _rel(y[:, good], acc[:, good] / wsum[good], 1)
        assert worst["norm"] <= TRUTH_NORM, worst
        assert np.all(y[:, (frames - 1) * hop + nfft:] == 0)
        for i in range(batch):
            one = h.batch_forward(xd[i:i + 1].contiguous(), "complex", "valid")
            y1 = h.batch_inverse(one, n, True)
            torch.cuda.synchronize()
            assert np.array_equal(one.cpu().numpy()[0], s[i]), (nfft, i, "forward: alone != in the batch")
            assert np.array_equal(y1.cpu().numpy()[0], y[i]), (nfft, i, "inverse: alone != in the batch")
    return worst


# Bound of the log-mel routes against float64 truth, per band and frame:
#   |exp(lm) - (mel + eps)| <= TRUTH_LOGMEL * sum_k |w_mk| |X_k| * max|X|  +  2^-22 * max(|log(mel + eps)|, 1) * (mel + eps)
# The first term is the float32 error of |X_k|^2 (about max|X| |X_k| times the spectrum's relative error) carried through
# the band's weights; the second is two units in the last place of the float32 logarithm itself, which is all a band with
# no power (log(eps)) may differ by.  A flat bound on the log would hold quiet bands (a few 1e-6 of the frame's power)
# to the error of the loud bins around them.  About 6 times the worst error in the CPU emulator (3.4e-7); the worst on a B200
# is not measured yet (test_logmel_route_vs_float64_truth).
TRUTH_LOGMEL = 2e-6


def logmel_truth(x, w, nfft, hop, convention, weights, eps):
    """float64 mel + eps of |X_truth|^2 under the library's float32 filterbank, and the propagated bound above"""
    X = stft_truth_f64(x, w, nfft, hop, convention=convention)
    A = np.abs(X)
    W = np.asarray(weights, np.float64)
    mel = (A * A) @ W.T + eps
    bound = TRUTH_LOGMEL * (A @ np.abs(W).T) * A.max(axis=(-2, -1), keepdims=True)
    return mel, bound + 2.0 ** -22 * np.maximum(np.abs(np.log(mel)), 1.0) * mel


def mfcc_truth(mel, bound, n_coeffs, lifter):
    """float64 DCT-II (cos(pi (n + 1/2) k / n_mels), unnormalised) of log(mel + eps) with the lifter 1 + L/2 sin(pi k / L), and
    a bound propagated from the log-mel bound: a log-mel error below bound/(mel+eps) <= 1/2 is at most twice that in the log;
    plus the float32 cosine table (angle rounded to float32), the float32 sum over n_mels terms and the float32 lifter."""
    n_mels = mel.shape[-1]
    k = np.arange(n_coeffs)[:, None]
    ang = np.pi * (np.arange(n_mels)[None, :] + 0.5) * k / n_mels
    D = np.cos(ang)
    lif = np.ones(n_coeffs)
    if lifter > 0:
        lif[1:] = 1.0 + lifter / 2.0 * np.sin(np.pi * np.arange(1, n_coeffs) / lifter)
    lm = np.log(mel)
    r = bound / mel
    assert r.max() <= 0.5, r.max()
    c = (lm @ D.T) * lif
    absl = np.abs(lm)
    err = (2 * r) @ np.abs(D).T + absl @ (2.0 ** -22 * (1 + np.abs(ang))).T + n_mels * 2.0 ** -23 * absl.sum(-1, keepdims=True)
    return c, np.abs(lif) * err + 2.0 ** -21 * np.abs(c)


LOGMEL_MODES = {"pair": "one fused kernel, two frames per band-sum phase", "single": "one fused kernel, one frame per band-sum phase",
                "warp": "one fused kernel, band sums per warp", "chained": "power kernel + log-mel kernel"}


def check_logmel_route(lib, oracle, nfft, hop, n_mels, sr, win, route=None, mode=None, capfd=None, batch=2, n=None, eps=1e-10,
                       n_coeffs=13, lifter=22.0):
    """batch_logmel and batch_mfcc in all four frame conventions against float64 truth (logmel_truth, mfcc_truth), through
    whatever path the handle picks for this filterbank.  With capfd the call must launch `route` (route_needles) and the
    VVB_MEL_DEBUG line must name `mode` (LOGMEL_MODES).  Returns the worst error over TRUTH_LOGMEL's term (relative to
    sum |w||X| max|X|) and the worst MFCC error as a fraction of its bound."""
    from vv_dsp_b200 import mel_filterbank
    st, weights = mel_filterbank(nfft, n_mels, sr, 0.0, sr / 2, lib=lib)
    assert st == 0
    n = n or nfft + 40 * hop + hop // 3
    x = np.stack([noise(2900 + nfft + hop + i, n) for i in range(batch)])
    w = oracle.window(win, nfft)[1]
    worst = {"logmel": 0.0, "mfcc": 0.0}
    call = (lambda f: routed(capfd, f)) if capfd is not None else (lambda f: (f(), []))
    with Stft(nfft, hop, win, lib=lib) as h:
        for conv in ("valid", "spectrogram", "padded_tail", "center"):
            lm, lines = call(lambda: h.batch_logmel(x, weights, eps, conv))
            if capfd is not None:
                assert route is None or launched(lines, route, nfft), (nfft, hop, n_mels, route, lines)
                assert mode is None or f"vvb: STFT -> log-mel: {LOGMEL_MODES[mode]}" in lines, (nfft, hop, n_mels, mode, lines)
            mel, bound = logmel_truth(x, w, nfft, hop, conv, weights, eps)
            assert lm.shape == mel.shape == (batch, h.num_frames(n, conv), n_mels), conv
            err = np.abs(np.exp(lm.astype(np.float64)) - mel)
            assert np.all(err <= bound), (nfft, hop, n_mels, win, conv, float((err / bound).max()))
            prop = (bound - 2.0 ** -22 * np.maximum(np.abs(np.log(mel)), 1.0) * mel) / TRUTH_LOGMEL
            worst["logmel"] = max(worst["logmel"], float((err / np.maximum(prop, 1e-300)).max()))
            mf = h.batch_mfcc(x, weights, n_coeffs, lifter=lifter, log_epsilon=eps, convention=conv)
            c, cb = mfcc_truth(mel, bound, n_coeffs, lifter)
            e = np.abs(mf - c)
            assert np.all(e <= cb), (nfft, hop, n_mels, win, conv, "mfcc", float((e / cb).max()))
            worst["mfcc"] = max(worst["mfcc"], float((e / cb).max()))
    return worst


def check_logmel_pcm_truth(lib, oracle, nfft=2048, hop=512, n_mels=80, sr=48000.0, n=30000, batch=3, eps=1e-10):
    """batch_logmel_pcm (16-bit samples decoded on the device) against the float64 truth of the decoded samples"""
    from vv_dsp_b200 import mel_filterbank
    st, weights = mel_filterbank(nfft, n_mels, sr, 0.0, sr / 2, lib=lib)
    raw = np.random.default_rng(41).integers(-32768, 32768, (batch, n), dtype=np.int16)
    x = raw.astype(np.float64) / 32768.0
    w = oracle.window("hann", nfft)[1]
    with Stft(nfft, hop, "hann", lib=lib) as h:
        for conv in ("valid", "center"):
            lm = h.batch_logmel_pcm(raw, weights, 16, eps, conv)
            mel, bound = logmel_truth(x, w, nfft, hop, conv, weights, eps)
            err = np.abs(np.exp(lm.astype(np.float64)) - mel)
            assert lm.shape == mel.shape and np.all(err <= bound), (conv, float((err / bound).max()))


# Every log-mel path: (fft_size, hop, n_mels, sample rate, route, mode, switch).  The fused marching kernel at fft_size 2048
# sums two frames per band-sum phase where shared memory allows; the generic forward kernel fuses the sizes <= 1024 and the
# mixed-radix ones; every other size, and filterbanks the fused kernels cannot hold, chain the power kernel and a log-mel kernel
# (logmel_tma_kernel up to 512 bands, logmel_kernel above).
LOGMEL_ROUTES = ([(2048, h, 80, 48000.0, "logmel_march", "pair", None) for h in (256, 512, 1024)]
                 + [(2048, 1024, 40, 48000.0, "logmel_march", "single", None)]          # (its short schedule leaves no room for a pair)
                 + [(2048, 512, 80, 48000.0, "logmel_march", "single", "VVB_MEL_SINGLE"), (2048, 256, 40, 16000.0, "logmel_march", "single", "VVB_MEL_SINGLE")]
                 + [(N, h, m, sr, "logmel_generic", "warp", None) for N, h, m, sr in
                    ((256, 64, 40, 8000.0), (512, 128, 40, 16000.0), (1024, 256, 64, 44100.0), (320, 80, 40, 16000.0), (400, 160, 80, 16000.0),
                     (480, 160, 64, 16000.0), (640, 160, 80, 16000.0))]
                 + [(N, h, m, sr, "logmel_tma_kernel", "chained", None) for N, h, m, sr in
                    ((4096, 1024, 128, 48000.0), (8192, 2048, 256, 48000.0), (1000, 250, 40, 16000.0))]
                 + [(4096, 1024, 600, 48000.0, "logmel_kernel", "chained", None)]
                 # the filterbanks of check_mel_fused_fallback
                 + [(400, 160, 200, 16000.0, "logmel_tma_kernel", "chained", None), (400, 160, 128, 16000.0, "logmel_generic", "warp", None),
                    (1024, 256, 400, 48000.0, "logmel_tma_kernel", "chained", None), (256, 64, 128, 8000.0, "logmel_generic", "warp", None)])


MEL_SWITCHES = ("VVB_MEL_NO_TMA", "VVB_MEL_UNIT4", "VVB_MEL_NO_GENERIC", "VVB_MEL_ROW_SPREAD_OFF")


def check_mel_switches(lib, cases=((2048, 512, 80, 48000.0), (2048, 256, 40, 16000.0), (512, 128, 40, 16000.0), (400, 160, 80, 16000.0),
                                   (1024, 256, 64, 44100.0)), n=20000, batch=3):
    """The log-mel diagnostic switches are documented as bit-identical to the default path: log-mel and MFCC rows of the
    batched chain (each switch alone and on top of VVB_MEL_UNFUSED, where the log-mel kernel of the chain runs), and
    log_mel_spectrogram on a dense power matrix (logmel_tma_kernel against the register-transposing kernel)."""
    import os
    from vv_dsp_b200 import log_mel_spectrogram, mel_filterbank
    for nfft, hop, n_mels, sr in cases:
        st, w = mel_filterbank(nfft, n_mels, sr, 0.0, sr / 2, lib=lib)
        assert st == 0
        x = np.stack([noise(4000 + nfft + i, n) for i in range(batch)])

        def rows(*envs):
            for e in envs:
                os.environ[e] = "1"
            try:
                with Stft(nfft, hop, "hann", lib=lib) as h:       # (VVB_MEL_UNIT4 is read when a handle builds its schedules)
                    return (h.batch_logmel(x, w, 1e-6, "center"), h.batch_logmel(x, w, 1e-6, "valid"),
                            h.batch_mfcc(x, w, 13, lifter=22.0, log_epsilon=1e-6, convention="center"))
            finally:
                for e in envs:
                    del os.environ[e]
        fused, chained = rows(), rows("VVB_MEL_UNFUSED")
        for env in MEL_SWITCHES:
            for base, got in ((fused, rows(env)), (chained, rows("VVB_MEL_UNFUSED", env))):
                for a, b in zip(base, got):
                    assert a.shape == b.shape and np.array_equal(a, b, equal_nan=True), (nfft, hop, env)
        p = np.random.default_rng(nfft).uniform(0, 3, (77, nfft // 2 + 1)).astype(np.float32)
        a = log_mel_spectrogram(p, w, 1e-10, lib=lib)
        os.environ["VVB_MEL_NO_TMA"] = "1"
        try:
            b = log_mel_spectrogram(p, w, 1e-10, lib=lib)
        finally:
            del os.environ["VVB_MEL_NO_TMA"]
        assert np.array_equal(a, b), (nfft, "log_mel_spectrogram")


def check_bluestein(lib, oracle, sizes):
    """Sizes served by the chirp-z path (no Stockham kernel, 32 <= n <= 4096).  The reference serves them with an O(n^2)
    float32 DFT whose own error grows with n (measured here: 2.5e-5 at n=400, 6e-5 at 1000, 1.5e-4 at 2000 of max|X|),
    so the yardstick is float64 truth: the CUDA result must be within 3e-6 of it, and within the triangle bound
    (own error + the oracle's error) of the oracle.  Frame counts and zero regions stay bit-exact."""
    report = {}
    rng = np.random.default_rng(21)
    for nfft, hop in sizes:
        n = nfft + hop * 7 + 13
        x = np.stack([noise(70 + nfft + i, n) for i in range(2)])
        for win in ("hann", "hamming"):
            w = oracle.window(win, nfft)[1]
            with Stft(nfft, hop, win, lib=lib) as h:
                for conv in ("valid", "center", "spectrogram"):
                    s = h.batch_forward(x, "complex", conv)
                    assert s.shape[1] == oracle.num_frames(n, nfft, hop, conv), conv
                s = h.batch_forward(x, "complex", "valid")
                p = h.batch_forward(x, "power", "valid")
                F = s.shape[1]
                truth = np.stack([stft_truth_f64(x[i], w, nfft, hop, F) for i in range(2)])
                ref = np.stack([oracle.stft(x[i], nfft, hop, win) for i in range(2)])
                mx = np.abs(truth).max()
                mine, theirs = np.abs(s - truth).max() / mx, np.abs(ref - truth).max() / mx
                assert mine < 3e-6, (nfft, win, mine)
                assert np.abs(s - ref).max() / mx <= mine + theirs + 1e-7
                assert np.abs(p - np.abs(truth) ** 2).max() <= 6e-6 * mx * mx
                # synthesis: float64 overlap-add of irfft(spec) * w, divided by sum(w^2) where > 1e-12
                y = h.batch_inverse(ref, n, True)
                raw = h.batch_inverse(ref, n, False)
                acc, norm = istft_truth_f64(ref, w, nfft, hop, n)
                assert np.abs(raw - acc).max() <= 3e-6 * np.abs(acc).max()
                cov = (F - 1) * hop + nfft
                assert np.all(y[:, cov:] == 0) and np.all(raw[:, cov:] == 0)
                if 2 * hop <= nfft:
                    good = norm > 1e-3
                    yt = np.where(good, acc / np.where(good, norm, 1), 0)
                    assert np.abs(y - yt)[:, good].max() <= 2e-5 * np.abs(yt).max()
                    own = h.batch_inverse(s, n, True)
                    assert rel_l2(own[:, nfft:n - nfft], x[:, nfft:n - nfft]) <= ROUNDTRIP_REL_L2
                    oref = np.stack([oracle.istft(ref[i], nfft, hop, n, win) for i in range(2)])
                    # the oracle's O(n^2) float32 inverse DFT error dominates here and grows with the size
                    assert rel_l2(y[:, nfft:n - nfft], oref[:, nfft:n - nfft]) <= 2e-4 * max(1.0, nfft / 2048)
                    # binding check beside the widened tolerance: float64 truth of the same spectra, relative L2
                    assert rel_l2(y[:, nfft:n - nfft], yt[:, nfft:n - nfft]) <= ROUNDTRIP_REL_L2
        report[nfft] = (float(mine), float(theirs))
        # plan API
        z = (rng.uniform(-1, 1, (3, nfft)) + 1j * rng.uniform(-1, 1, (3, nfft))).astype(np.complex64)
        xr = rng.uniform(-1, 1, (3, nfft)).astype(np.float32)
        f = FftPlan(nfft, 0, +1, lib=lib).execute_batch(z)
        b = FftPlan(nfft, 0, -1, lib=lib).execute_batch(z)
        r = FftPlan(nfft, 1, +1, lib=lib).execute_batch(xr)
        c = FftPlan(nfft, 2, -1, lib=lib).execute_batch(r)
        z64 = z.astype(np.complex128)
        assert np.abs(f - np.fft.fft(z64, axis=-1)).max() <= 3e-6 * np.abs(np.fft.fft(z64, axis=-1)).max()
        assert np.abs(b - np.fft.ifft(z64, axis=-1)).max() <= 3e-6 * np.abs(np.fft.ifft(z64, axis=-1)).max()
        rt = np.fft.rfft(xr.astype(np.float64), axis=-1)
        assert np.abs(r - rt).max() <= 3e-6 * np.abs(rt).max()
        assert np.abs(c - xr).max() < 5e-6
        assert np.array_equal(f[1], FftPlan(nfft, 0, +1, lib=lib).execute(z[1]))
        fo = oracle.fft_c2c(z[0], +1)
        assert np.abs(f[0] - fo).max() <= np.abs(f[0] - np.fft.fft(z64[0])).max() + np.abs(fo - np.fft.fft(z64[0])).max() + 1e-6
    return report


def check_golden_slices(lib, golden):
    """GPU/emulator output against slices of the REAL reference's output (tests/golden/)."""
    for c in golden["cases"]:
        if c["kind"] != "stft" or c["nfft"] < 16:
            continue
        nfft, hop, win, n = c["nfft"], c["hop"], c["window"], c["n"]
        x = noise(c["seed"], n)
        key = f"n{nfft}_h{hop}_{win}_s{c['seed']}"
        with Stft(nfft, hop, win, lib=lib) as h:
            s = h.batch_forward(x[None], "complex", "valid")[0]
            assert s.shape[0] == c["frames"]["valid"]
            for conv in ("spectrogram", "padded_tail", "center"):
                assert h.num_frames(n, conv) == c["frames"][conv]
            ok, frac = spectra_close(s[0], golden["slices"][key + "_stft_row0"])
            assert ok, (key, frac)
            ok, frac = spectra_close(s[-1], golden["slices"][key + "_stft_rowlast"])
            assert ok, (key, frac)
            y = h.batch_inverse(s[None], n, True)[0]
            ref = golden["slices"][key + "_istft_mid"]
            # (hop > nfft/2 with Hann: the window-sum has near-zeros, the divide is ill-conditioned; skip)
            if n // 2 >= nfft and n // 2 + 256 <= n - nfft and 2 * hop <= nfft:
                # the golden slice is the REFERENCE's round trip, which carries its own float32 drift
                # (interior rel-L2 2.2e-5 at 4096, 3.9e-5 at 8192: SURVEY.md section 8c); allow for it,
                # and hold this library to the true signal at the north-star bound
                tol = 5e-5 if nfft <= 2048 else 4e-4
                assert np.abs(y[n // 2: n // 2 + 256] - ref).max() <= tol * max(np.abs(ref).max(), 1e-30), key
                # binding check beside the widened tolerance: the true signal, max-norm, at the north-star scale
                assert np.abs(y[n // 2: n // 2 + 256] - x[n // 2: n // 2 + 256]).max() <= 1e-5 * np.abs(x).max(), key
                if 2 * hop <= nfft:   # with less overlap the Hann window-sum has near-zeros: ill-conditioned divide
                    assert rel_l2(y[n // 2: n // 2 + 256], x[n // 2: n // 2 + 256]) <= ROUNDTRIP_REL_L2, key


def check_config1_voicebank(lib, golden):
    """BASELINE config 1: voicebank WAV, nfft=1024 hop=256 Hann, forward + ISTFT round trip."""
    wav = golden["pcm"].astype(np.float32) / np.float32(32768.0)
    with Stft(1024, 256, "hann", lib=lib) as h:
        s = h.batch_forward(wav[None], "complex", "valid")[0]
        assert s.shape == (621, 513)
        for f in (0, 310, 620):
            ok, frac = spectra_close(s[f], golden["slices"][f"config1_stft_row{f}"])
            assert ok, (f, frac)
        y = h.batch_inverse(s[None], wav.size, True)[0]
    ref = golden["slices"]["config1_roundtrip_80000"]
    assert np.abs(y[80000:81024] - ref).max() <= 5e-5 * np.abs(ref).max()
    err = rel_l2(y[1024:-1024], wav[1024:-1024])
    assert err <= ROUNDTRIP_REL_L2, err
    return err


def check_reconstruct_non_hermitian(lib, oracle, sizes=((256, 64), (2048, 512), (100, 30), (8, 4))):
    """vv_dsp_stft_reconstruct with a spectrum that is NOT Hermitian (a caller edited only bins 0..n/2, or anything
    else): the reference adds Re(IDFT(X)) * w (src/spectral/stft.c:95-110); here the host forms the Hermitian part
    (X[k] + conj X[n-k]) / 2 first.  Same arbitrary input to both sides."""
    rng = np.random.default_rng(99)
    for nfft, hop in sizes:
        for case in ("random", "lower_half_only", "imag_dc_nyquist"):
            X = (rng.uniform(-1, 1, nfft) + 1j * rng.uniform(-1, 1, nfft)).astype(np.complex64)
            if case == "lower_half_only":
                x = rng.uniform(-1, 1, nfft).astype(np.float32)
                X = np.fft.fft(x).astype(np.complex64)
                X[nfft // 2 + 1:] = 0                                   # upper half wiped: a common caller shortcut
            elif case == "imag_dc_nyquist":
                X = np.fft.fft(rng.uniform(-1, 1, nfft)).astype(np.complex64)
                X[0] += 3j
                X[nfft // 2] -= 2j
            with Stft(nfft, hop, "hann", lib=lib) as h:
                out = np.full(nfft, 0.25, np.float32); nrm = np.full(nfft, 0.5, np.float32)
                h.reconstruct(X, out, nrm)
            a, b = oracle.reconstruct(X, nfft, hop, "hann")
            w = oracle.window("hann", nfft)[1].astype(np.float64)
            truth = np.fft.ifft(X.astype(np.complex128)).real * w
            scale = max(np.abs(truth).max(), 1e-30)
            assert np.abs((out - 0.25) - truth).max() <= 1e-5 * scale, (nfft, case)              # float64 truth
            assert np.abs((out - 0.25) - a).max() <= 5e-5 * scale + 1e-7, (nfft, case)           # the reference's result
            assert np.array_equal(nrm, np.float32(0.5) + b), (nfft, case)                        # norm_add += w*w, float32


def check_async_many_chunks(lib, oracle, nfft=256, hop=64, n=4000, batch=150):
    """Stream-ordered host mode with MORE chunks than the dependency ring holds (64): the analysis call leaves its
    spectra in HBM chunk by chunk, the synthesis call that follows must wait for every one of them.  Caller sets
    VVB_STAGE_TARGET_BYTES small enough that a chunk is one signal (test hook read at handle creation)."""
    import torch
    x = np.stack([noise(500 + i, n) for i in range(batch)])
    with Stft(nfft, hop, "hann", lib=lib) as h:
        F = h.num_frames(n, "valid")
        ref_spec = h.batch_forward(x, "complex", "valid")             # synchronous reference run
        ref_y = h.batch_inverse(ref_spec, n, True)
        xh = torch.from_numpy(x).pin_memory()
        yh = torch.empty((batch, n), dtype=torch.float32).pin_memory()
        for rep in range(3):
            spec = torch.zeros((batch, F, h.bins), device="cuda", dtype=torch.complex64)
            yh.zero_()
            torch.cuda.synchronize()
            h.set_async(True)
            h.batch_forward(xh.numpy(), "complex", "valid", out=spec)
            h.batch_inverse(spec, n, True, out=yh.numpy())
            h.synchronize()
            h.set_async(False)
            assert np.array_equal(spec.cpu().numpy(), ref_spec), rep
            assert np.array_equal(yh.numpy(), ref_y), rep


def check_staged_chunks_equal_single(lib, nfft, hop, n=3000, batch=9):
    """host-staged calls split into many chunks == the same call in one chunk (sizes with per-engine scratch buffers
    included: their chunks must not overlap in time).  Caller sets VVB_STAGE_TARGET_BYTES for the chunked handle."""
    x = np.stack([noise(900 + nfft + i, n) for i in range(batch)])
    with Stft(nfft, hop, "hann", lib=lib) as h:
        spec = h.batch_forward(x, "complex", "valid")
        y = h.batch_inverse(spec, n, True)
        for rep in range(3):
            assert np.array_equal(h.batch_forward(x, "complex", "valid"), spec)
            assert np.array_equal(h.batch_inverse(spec, n, True), y)
    return spec, y


def check_stream_sharding(lib, nfft, hop, n, shard_counts=(1, 2, 3, 5), win="hann", device=0):
    """vv_dsp_stft_stream (one stream, frame-range shards with sample halos) against the UNSHARDED batched calls:
    spectra and the normalised ISTFT must be bit-identical for every shard count -- the shards re-synthesise the
    nfft/hop - 1 frames in front of their range instead of exchanging partial sums.  All shards on one device here
    (peer copies degenerate to device copies), so the whole path runs on a 1-GPU box and in the emulator."""
    x = noise(4242 + nfft, n)
    with Stft(nfft, hop, win, lib=lib) as h:
        spec = h.batch_forward(x[None], "complex", "valid")[0]
        y = h.batch_inverse(spec[None], n, True)[0]
    first = None
    for g in shard_counts:
        with StftStream(nfft, hop, n, [device] * g, win, lib=lib) as s:
            assert s.frames == spec.shape[0]
            cover = 0
            for d in range(g):
                sh = s.shard(d)
                assert sh.frame0 == s.frames * d // g and sh.frame1 == s.frames * (d + 1) // g        # SURVEY.md 8e
                assert sh.sample0 == sh.frame0 * hop and sh.sample1 == (n if d == g - 1 else sh.frame1 * hop)
                assert sh.halo_frames == (0 if d == 0 else nfft // hop - 1)
                assert sh.left_halo == (0 if d == 0 else nfft - hop) and sh.right_halo == (0 if d == g - 1 else nfft - hop)
                cover += sh.sample1 - sh.sample0
            assert cover == n
            s.upload(x)
            s.forward(); s.inverse(); s.synchronize()
            assert np.array_equal(s.download_spectra(), spec), (nfft, hop, g, "spectra")
            # fft_size >= 2048: shards and the unsharded call run the same marching kernel -> bit-identical.  Below, the
            # unsharded call pairs frames (two per complex transform), a shard does not: equal to rounding, and the
            # shard counts must still agree bit for bit among themselves.
            same = (lambda a, b: np.array_equal(a, b)) if nfft >= 2048 else \
                   (lambda a, b: np.abs(a - b)[nfft:-nfft].max() <= 2e-6 * np.abs(b).max())
            got = s.download()
            assert same(got, y), (nfft, hop, g, "istft")
            if first is None:
                first = got
            assert np.array_equal(got, first), (nfft, hop, g, "shard counts disagree")
            for _ in range(3):                                    # first call plain, later ones replay the captured graphs
                s.roundtrip()
            s.synchronize()
            assert np.array_equal(s.download(), first), (nfft, hop, g, "roundtrip")
            assert s.time_roundtrip(1, 2) >= 0.0
    return y, x
