"""Batched polyphase resampling (vv_dsp_resample_poly_*, include/vv_dsp/b200.h) against scipy.signal.resample_poly in float64.

One set of check_* functions runs in the CPU emulator (tests/emu: the kernel sources compiled for the CPU, small sizes) and
on the B200 (the nvcc-built library, -m gpu, full sizes).  Every ratio row asserts the handle's configuration and the
launches VVB_ROUTE_DEBUG reports: resample_poly_kernel with the input span staged in shared memory, or read through L1
when it would not fit, and no kernel at all for the identity ratio."""
import ctypes
import os
import sys
from math import gcd

import numpy as np
import pytest
from scipy.signal import firwin, resample_poly

import parity_cases as pc
from vv_dsp_b200 import Resampler, VvDspError

HERE = os.path.dirname(os.path.abspath(__file__))
HOST, DEVICE = 0, 1
EPS32 = 2.0 ** -24

# (up, down) as given -> (reduced up, reduced down, K, T, input span in shared memory) of the default Kaiser design.
# The standard-rate rows, both directions, small ratios, a ratio that reduces, the largest bank of any pair of the standard
# rates (11 025 -> 192 000: 53 760 taps), and 192 -> 8 kHz, whose tile span does not fit in shared memory.
ROWS = {(1, 3): (1, 3, 61, 61, True), (3, 1): (3, 1, 61, 21, True), (160, 441): (160, 441, 8821, 56, True),
        (441, 160): (441, 160, 8821, 21, True), (147, 160): (147, 160, 3201, 22, True), (160, 147): (160, 147, 3201, 21, True),
        (2, 1): (2, 1, 41, 21, True), (1, 2): (1, 2, 41, 41, True), (5, 4): (5, 4, 101, 21, True), (6, 4): (3, 2, 61, 21, True),
        (2560, 147): (2560, 147, 51201, 21, True), (1, 24): (1, 24, 481, 481, False)}


@pytest.fixture(scope="module")
def emu():
    sys.path.insert(0, os.path.join(HERE, "emu"))
    import build_emu
    from vv_dsp_b200 import Library
    return Library(build_emu.build())


@pytest.fixture(scope="module")
def lib():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from vv_dsp_b200 import default_library
    return default_library()


def is_gpu(lib):
    return "emu" not in lib.path


# ----------------------------------------------------------------------------- helpers
def default_window(up, down):
    """scipy's default design of resample_poly, passed to it explicitly so that truth and bound use the same taps"""
    g = gcd(up, down)
    m = max(up // g, down // g)
    return firwin(2 * 10 * m + 1, 1.0 / m, window=("kaiser", 5.0))


def truth(x, up, down, w):
    """float64 resample_poly of every row"""
    return np.stack([resample_poly(row.astype(np.float64), up, down, window=w, padtype="constant") for row in x])


def worst_ratio(y, x, up, down, w, taps_per_phase):
    """max over outputs of |y - y64| over (T + 2) 2^-24 sum_j |h_j x_(i0-j)| (a T-term float32 dot product plus the one
    rounding of the taps); the right-hand side is resample_poly(|x|, window=|w|) in float64"""
    err = np.abs(np.asarray(y, np.float64) - truth(x, up, down, w))
    rhs = (taps_per_phase + 2) * EPS32 * truth(np.abs(x.astype(np.float64)), up, down, np.abs(w))
    return float(np.where(err > 0, err / np.maximum(rhs, 1e-300), 0.0).max()) if err.size else 0.0


def data(seed, rows, cols):
    return np.random.default_rng(seed).standard_normal((rows, cols)).astype(np.float32)


def to_space(lib, a, space):
    """an array in the requested memory space: numpy for HOST (and for DEVICE in the emulator, where device memory is
    host memory), a torch CUDA tensor for DEVICE on the GPU"""
    if space == DEVICE and is_gpu(lib):
        import torch
        return torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return np.ascontiguousarray(a)


def ptr(a):
    return ctypes.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)


def to_host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def raw_resample(lib, r, x, xs, os_, n, xp=0, op=0, batch=None):
    """vv_dsp_resample_poly_batch with both buffers in the space asked for; x is a 2-D numpy array whose row length is its
    pitch when xp is given; the output buffer is prefilled with 7.5.  Returns (status, out_len, output as numpy)"""
    batch = x.shape[0] if batch is None else batch
    n_out = r.output_length(n)
    out = np.full((max(batch, 1), max(op or n_out, 1)), np.float32(7.5))
    xd, od = to_space(lib, x, xs), to_space(lib, out, os_)
    got = ctypes.c_size_t(12345)
    st = lib.vv_dsp_resample_poly_batch(r._r, ptr(xd), xs, batch, n, xp, ptr(od), os_, op, ctypes.byref(got))
    r.synchronize()
    return st, got.value, to_host(od)


def routed_lines(capfd, fn):
    """fn() with VVB_ROUTE_DEBUG=1: (its result, the library's stderr lines)"""
    return pc.routed(capfd, fn) if capfd is not None else (fn(), None)


def check_launches(lines, smem, launches=1):
    kern = [ln for ln in lines if "resample_poly_kernel" in ln]
    assert len(kern) == launches, lines
    assert all("vvb::launch_resample(" in ln and "int R = 8" in ln and f"bool SMEM = {'true' if smem else 'false'}" in ln
               for ln in kern), kern


def check_config(r, up, down, k, t):
    assert (r.up, r.down, r.num_taps, r.taps_per_phase) == (up, down, k, t)


def lengths(up, down, t, long_n):
    """n = 1, shorter than down, shorter than T, n up not a multiple of down (there is none when down == 1), a long signal"""
    ns = {1, max(down - 1, 1), max(t - 1, 1), long_n}
    if down > 1:
        odd = down + 1
        while (odd * up) % down == 0:
            odd += 1
        ns.add(odd)
    return sorted(ns)


# ----------------------------------------------------------------------------- checks
def check_row(lib, up, down, capfd=None, long_n=3000, batch=2):
    """One ratio with the default design against float64 truth over every signal-length class, with the configuration,
    the launches and the output length asserted.  Returns the worst error over the bound."""
    ru, rd, k, t, smem = ROWS[(up, down)]
    w = default_window(up, down)
    worst = 0.0
    with Resampler(up, down, lib=lib) as r:
        check_config(r, ru, rd, k, t)
        for i, n in enumerate(lengths(ru, rd, t, long_n)):
            x = data(100 + i, batch, n)
            y, lines = routed_lines(capfd, lambda: r.resample(x))
            if lines is not None:
                check_launches(lines, smem)
            y = to_host(y)
            assert y.shape == (batch, len(resample_poly(x[0].astype(np.float64), up, down, window=w)))
            worst = max(worst, worst_ratio(y, x, up, down, w, t))
    assert worst <= 1.0, (up, down, worst)
    return worst


def check_exact(lib, up, down, n=None, k=None, seed=1):
    """integer signals in [-8, 8] and taps that are multiples of 1/4: every product and partial sum is exact in float32, so
    the output equals float64 truth bit for bit -- a phase, offset or edge error shows whatever the tolerance"""
    rng = np.random.default_rng(seed)
    g = gcd(up, down)
    k = k or 2 * 10 * max(up // g, down // g) + 1
    w = (rng.integers(-8, 9, k) / 4.0).astype(np.float32)
    for nn in ([n] if n else lengths(up // g, down // g, -(-k // (up // g)), 700)):
        x = rng.integers(-8, 9, (2, nn)).astype(np.float32)
        with Resampler(up, down, taps=w, lib=lib) as r:
            y = to_host(r.resample(x))
        want = truth(x, up, down, w.astype(np.float64))
        assert np.array_equal(y, want.astype(np.float32)) and np.array_equal(y.astype(np.float64), want), (up, down, nn)


def check_custom_filters(lib, capfd=None):
    """a filter of one tap, of even length, shorter than up (empty phases), and a ratio that reduces to 1 / 1 with a filter
    (a copy that ignores it)"""
    x = data(7, 3, 1001)
    for up, down, k in ((3, 2, 1), (2, 3, 30), (1, 3, 8), (7, 3, 4), (5, 4, 3)):
        w = np.random.default_rng(k).standard_normal(k).astype(np.float32)
        with Resampler(up, down, taps=w, lib=lib) as r:
            check_config(r, up, down, k, -(-k // up))
            y, lines = routed_lines(capfd, lambda: r.resample(x))
            if lines is not None:
                check_launches(lines, True)
            assert worst_ratio(to_host(y), x, up, down, w.astype(np.float64), r.taps_per_phase) <= 1.0, (up, down, k)
        check_exact(lib, up, down, n=1001, k=k, seed=k)
    w = np.ones(5, np.float32)
    for up, down, taps in ((7, 7, None), (4, 4, w)):
        with Resampler(up, down, taps=taps, lib=lib) as r:
            assert (r.up, r.down) == (1, 1)
            y, lines = routed_lines(capfd, lambda: r.resample(x))
            if lines is not None:
                assert not any("resample_poly_kernel" in ln for ln in lines), lines
            assert np.array_equal(to_host(y), x)


def check_lengths(lib):
    """output_length and *out_len equal scipy's output length for every n tried, 0 included"""
    for up, down in ((1, 3), (3, 1), (160, 441), (147, 160), (5, 4), (6, 4)):
        with Resampler(up, down, lib=lib) as r:
            for n in (0, 1, 2, 3, 146, 147, 160, 441, 442, 1000, 4409):
                want = -(-n * r.up // r.down)
                if n:
                    assert want == len(resample_poly(np.ones(n), up, down))
                assert r.output_length(n) == want
                st, got, _ = raw_resample(lib, r, np.ones((2, max(n, 1)), np.float32), HOST, HOST, n, xp=max(n, 1))
                assert st == 0 and got == want, (up, down, n)


def check_batch_identity(lib, up, down, n, monkeypatch=None, capfd=None):
    """one signal alone is bit-identical to itself inside a batch of 64; several staging chunks equal one"""
    x = data(11, 64, n)
    with Resampler(up, down, lib=lib) as r:
        n_out = r.output_length(n)
        many = to_host(r.resample(x))
        for b in (0, 37, 63):
            assert np.array_equal(to_host(r.resample(x[b:b + 1])), many[b:b + 1])
    if monkeypatch is not None:
        with monkeypatch.context() as mp:
            mp.setenv("VVB_STAGE_TARGET_BYTES", str(4 * 5 * max(n, n_out)))         # five signals per chunk
            with Resampler(up, down, lib=lib) as r2:
                y, lines = routed_lines(capfd, lambda: r2.resample(x))
                assert np.array_equal(y, many)
                if lines is not None:
                    check_launches(lines, ROWS[(up, down)][4], launches=13)


def check_spaces(lib, up, down, n, batch=5):
    """HOST / DEVICE for signals and out, dense and with odd row pitches: bit-identical to the dense HOST result, with
    nothing written into the pitch padding"""
    xw = data(12, batch, n + 5)
    with Resampler(up, down, lib=lib) as r:
        n_out = r.output_length(n)
        st, got, ref = raw_resample(lib, r, np.ascontiguousarray(xw[:, :n]), HOST, HOST, n)
        assert st == 0 and got == n_out
        for xs in (HOST, DEVICE):
            for os_ in (HOST, DEVICE):
                st, got, y = raw_resample(lib, r, np.ascontiguousarray(xw[:, :n]), xs, os_, n)
                assert st == 0 and got == n_out and np.array_equal(y, ref), (xs, os_)
                st, got, y = raw_resample(lib, r, xw, xs, os_, n, xp=n + 5, op=n_out + 7)
                assert st == 0 and got == n_out, (xs, os_)
                assert np.array_equal(y[:, :n_out], ref), (xs, os_)
                assert np.all(y[:, n_out:] == np.float32(7.5)), (xs, os_)


def check_status_codes(lib):
    h = ctypes.c_void_p()
    w = np.ones(4, np.float32)
    create = lib.vv_dsp_resample_poly_create
    assert create(1, 3, None, 0, None) == 1                                    # NULL out pointer
    assert create(1, 3, None, 4, ctypes.byref(h)) == 1                         # taps == NULL with num_taps > 0
    assert create(0, 3, None, 0, ctypes.byref(h)) == 2                         # up == 0
    assert create(1, 0, None, 0, ctypes.byref(h)) == 2                         # down == 0
    assert create(1, 3, ptr(w), 0, ctypes.byref(h)) == 2                       # taps given with num_taps == 0
    assert create(1, 3277, None, 0, ctypes.byref(h)) == 2                      # default bank 65 541 taps > 65 536
    big = np.zeros(65537, np.float32)
    assert create(2, 1, ptr(big), big.size, ctypes.byref(h)) == 2              # bank 2 x 32 769
    assert lib.vv_dsp_resample_poly_destroy(None) == 1
    assert lib.vv_dsp_resample_poly_set_stream(None, None) == 1
    assert lib.vv_dsp_resample_poly_synchronize(None) == 1
    assert lib.vv_dsp_resample_poly_output_length(None, 10) == 0
    with pytest.raises(VvDspError):
        Resampler(0, 1, lib=lib)
    with Resampler(2560, 147, lib=lib):                                        # the largest standard-rate bank: 53 760 taps
        pass
    with Resampler(1, 3, lib=lib) as r:
        s = ctypes.c_size_t()
        assert lib.vv_dsp_resample_poly_get_config(None, ctypes.byref(s), ctypes.byref(s), ctypes.byref(s), ctypes.byref(s)) == 1
        assert lib.vv_dsp_resample_poly_get_config(r._r, None, ctypes.byref(s), ctypes.byref(s), ctypes.byref(s)) == 1
        x, y = np.ones((3, 300), np.float32), np.zeros((3, 100), np.float32)
        call = lambda *a: lib.vv_dsp_resample_poly_batch(r._r, *a)              # noqa: E731
        ok = (ptr(x), HOST, 3, 300, 0, ptr(y), HOST, 0, ctypes.byref(s))
        assert call(*ok) == 0 and s.value == 100
        assert lib.vv_dsp_resample_poly_batch(None, *ok) == 1                  # NULL handle
        for i in (0, 5, 8):                                                    # signals, out, out_len
            assert call(*ok[:i], None, *ok[i + 1:]) == 1
        for i in (1, 6):                                                       # memory spaces
            assert call(*ok[:i], 2, *ok[i + 1:]) == 3
        assert call(*ok[:4], 299, *ok[5:]) == 2                                # signal pitch below its row
        assert call(*ok[:7], 99, ok[8]) == 2                                   # out pitch below its row
        assert call(*ok[:3], 1 << 62, *ok[4:]) == 2                           # n up >= 2^62
        assert call(*ok[:5], ptr(x), *ok[6:]) == 6                             # out == signals
        y[:] = 3.0
        s.value = 99
        assert call(*ok[:2], 0, *ok[3:]) == 0 and np.all(y == 3.0) and s.value == 100     # batch == 0
        assert call(*ok[:3], 0, *ok[4:]) == 0 and np.all(y == 3.0) and s.value == 0       # n == 0
    with Resampler(3, 1, lib=lib) as r:
        s = ctypes.c_size_t()
        x, y = np.ones((1, 8), np.float32), np.zeros((1, 24), np.float32)
        n_big = ((1 << 62) + 2) // 3                                           # n up just reaches 2^62
        assert lib.vv_dsp_resample_poly_batch(r._r, ptr(x), HOST, 1, n_big, 0, ptr(y), HOST, 0, ctypes.byref(s)) == 2
        assert lib.vv_dsp_resample_poly_batch(r._r, ptr(x), HOST, 1, 8, 0, ptr(y), HOST, 0, ctypes.byref(s)) == 0


# ----------------------------------------------------------------------------- CPU emulator
@pytest.mark.parametrize("up,down", sorted(ROWS))
def test_emu_row_vs_float64_truth(emu, capfd, up, down):
    worst = check_row(emu, up, down, capfd=capfd, long_n=3000 if up < 1000 else 600)
    with capfd.disabled():
        print(f"\nresample ({up}, {down}): worst error / bound = {worst:.2e}")


@pytest.mark.parametrize("up,down", sorted(ROWS))
def test_emu_exact_indexing(emu, up, down):
    check_exact(emu, up, down, n=None if up < 1000 else 300)


def test_emu_custom_filters_and_identity(emu, capfd):
    check_custom_filters(emu, capfd=capfd)


def test_emu_lengths(emu):
    check_lengths(emu)


def test_emu_batch_identity_and_chunks(emu, monkeypatch, capfd):
    check_batch_identity(emu, 1, 3, 900, monkeypatch=monkeypatch, capfd=capfd)
    check_batch_identity(emu, 160, 147, 300)


@pytest.mark.parametrize("up,down", [(1, 3), (160, 441)])
def test_emu_spaces(emu, up, down):
    check_spaces(emu, up, down, 1201, batch=3)


def test_emu_status_codes(emu):
    check_status_codes(emu)


# ----------------------------------------------------------------------------- B200
@pytest.mark.gpu
@pytest.mark.parametrize("up,down", sorted(ROWS))
def test_gpu_row_vs_float64_truth(lib, capfd, up, down):
    worst = check_row(lib, up, down, capfd=capfd, long_n=480000, batch=3)
    with capfd.disabled():
        print(f"\nresample ({up}, {down}): worst error / bound = {worst:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("up,down", sorted(ROWS))
def test_gpu_exact_indexing(lib, up, down):
    check_exact(lib, up, down)
    check_exact(lib, up, down, n=480001)


@pytest.mark.gpu
def test_gpu_custom_filters_lengths_and_status(lib, capfd):
    check_custom_filters(lib, capfd=capfd)
    check_lengths(lib)
    check_status_codes(lib)


@pytest.mark.gpu
def test_gpu_batch_identity_and_chunks(lib, monkeypatch, capfd):
    check_batch_identity(lib, 1, 3, 160000, monkeypatch=monkeypatch, capfd=capfd)
    check_batch_identity(lib, 160, 147, 48000)
    check_batch_identity(lib, 1, 24, 48000)


@pytest.mark.gpu
@pytest.mark.parametrize("up,down", [(1, 3), (3, 1), (160, 441), (1, 24)])
def test_gpu_spaces(lib, up, down):
    check_spaces(lib, up, down, 48001, batch=5)


@pytest.mark.gpu
def test_gpu_torch_views_equal_host_path(lib):
    """torch views with odd row pitches (signals, out) give the host path's result bit for bit"""
    import torch
    n, batch = 30001, 5
    x = data(13, batch, n)
    with Resampler(160, 441, lib=lib) as r:
        want = r.resample(x)
        n_out = r.output_length(n)
        xw = torch.zeros((batch, n + 5), device="cuda"); xw[:, :n] = torch.from_numpy(x).cuda()
        ow = torch.full((batch, n_out + 7), 7.5, device="cuda")
        got = r.resample(xw[:, :n], out=ow[:, :n_out])
        torch.cuda.synchronize()
        assert got.data_ptr() == ow.data_ptr()
        assert np.array_equal(got.cpu().numpy(), want)
        assert bool((ow[:, n_out:] == 7.5).all())
        assert np.array_equal(r.resample(xw[:, :n]).cpu().numpy(), want)
        with pytest.raises(TypeError):
            r.resample(xw[:, :n].double())
        with pytest.raises(ValueError):
            r.resample(xw[:, :2 * (n // 2):2])


@pytest.mark.gpu
def test_gpu_device_calls_follow_torchs_current_stream(lib):
    """No set_stream(): device-tensor calls are enqueued on torch's current stream, so they are ordered against the torch
    ops that produce their inputs and consume their outputs (also on a side stream)."""
    import torch
    n, batch = 480000, 16
    g = torch.Generator(device="cuda").manual_seed(7)
    base = torch.rand((batch, n), device="cuda", generator=g) * 2 - 1
    with Resampler(1, 3, lib=lib) as r:
        torch.cuda.synchronize()
        want = r.resample(base * 0.5)
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        for s in (torch.cuda.current_stream(), side):
            with torch.cuda.stream(s):
                big = torch.rand((4096, 4096), device="cuda")
                for _ in range(20):
                    big = big @ big * 1e-3                       # keeps the stream busy: the input below is late
                x = base * 0.5                                    # produced on this stream
                y = r.resample(x)
                z = y * 2.0                                       # consumed on this stream
            torch.cuda.synchronize()
            assert torch.equal(y, want)
            assert torch.equal(z, want * 2.0)


@pytest.mark.gpu
def test_gpu_11025_to_192000(lib, capfd):
    """the largest bank of the standard rates (2560 / 147, 53 760 taps) with the default design, on 2 x 110 250 samples"""
    up, down = 2560, 147
    x = data(14, 2, 110250)
    w = default_window(up, down)
    with Resampler(192000, 11025, lib=lib) as r:
        check_config(r, up, down, 51201, 21)
        y, lines = pc.routed(capfd, lambda: r.resample(x))
        check_launches(lines, True)
        assert y.shape == (2, 1920000)
        assert worst_ratio(y, x, up, down, w, 21) <= 1.0
