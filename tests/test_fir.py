"""Batched FIR filtering by FFT convolution (vv_dsp_fir_*, include/vv_dsp/b200.h) against float64 truth.

One set of check_* functions runs in the CPU emulator (tests/emu: the kernel sources compiled for the CPU, small sizes) and
on the B200 (the nvcc-built library, -m gpu, full sizes).  Every row asserts the (transform size, partitions) the handle
picked and the launches VVB_ROUTE_DEBUG reports: fir_ols_kernel in that configuration, one plain pass and P - 1 ACCUM
passes per chunk of signals."""
import os
import sys

import numpy as np
import pytest
from scipy.signal import oaconvolve

import parity_cases as pc
from vv_dsp_b200 import FirFilter, VvDspError

HERE = os.path.dirname(os.path.abspath(__file__))
HOST, DEVICE = 0, 1

# num_taps -> (transform size, partitions) of the plan rule in b200.h; the rows reach every transform size, the last
# one-pass and first two-pass M, 3 and 12 passes
PLAN = {1: (128, 1), 2: (128, 1), 31: (256, 1), 64: (512, 1), 128: (1024, 1), 255: (2048, 1), 512: (4096, 1), 1000: (8192, 1),
        2049: (8192, 1), 5462: (8192, 1), 5463: (8192, 2), 10000: (8192, 3), 48000: (8192, 12)}
# the edges of the rule's table: the last M of each size and the first of the next
PLAN_EDGES = {29: (128, 1), 30: (256, 1), 52: (256, 1), 53: (512, 1), 94: (512, 1), 95: (1024, 1), 171: (1024, 1), 172: (2048, 1),
              316: (2048, 1), 317: (4096, 1), 586: (4096, 1), 587: (8192, 1), 16000: (8192, 4)}

# bound of max_i |y - y64| per signal: FIR_C * log2(N) * sqrt(P) * ||h||_2 * max over N-sample frames of ||x_frame||_2
# (Cauchy-Schwarz bounds |y| by ||h|| ||x_frame||).  Worst ratio to the bound without FIR_C: 8.9e-9 in the emulator, 9.1e-9
# on one NVIDIA B200 (power limit 1000 W).
FIR_C = 4e-8


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
def truth(h, x, n_out):
    """float64 full linear convolution of every row with its filter, cut or zero-extended to n_out"""
    out = np.zeros((x.shape[0], n_out))
    for b in range(x.shape[0]):
        hb = h[0 if h.shape[0] == 1 else b].astype(np.float64)
        full = oaconvolve(x[b].astype(np.float64), hb) if x.shape[1] else np.zeros(0)
        k = min(n_out, full.size)
        out[b, :k] = full[:k]
    return out


def bound(h, x, fft_size, parts):
    """per-signal error bound (see FIR_C) without FIR_C"""
    c2 = np.concatenate([np.zeros((x.shape[0], 1)), np.cumsum(x.astype(np.float64) ** 2, axis=1)], axis=1)
    w = min(fft_size, x.shape[1])
    frame = np.sqrt(np.maximum((c2[:, w:] - c2[:, :-w]).max(axis=1), 0.0)) if x.shape[1] else np.zeros(x.shape[0])
    hn = np.linalg.norm(h.astype(np.float64), axis=1)
    hn = np.broadcast_to(hn if h.shape[0] > 1 else hn[:1], (x.shape[0],))
    return np.log2(fft_size) * np.sqrt(parts) * hn * frame


def worst_ratio(y, h, x, n_out, f):
    """max over signals of the error against float64 truth over the bound without FIR_C"""
    err = np.abs(np.asarray(y, np.float64) - truth(h, x, n_out)).max(axis=1) if n_out else np.zeros(x.shape[0])
    return float((err / np.maximum(bound(h, x, f.fft_size, f.partitions), 1e-30)).max())


def data(seed, rows, cols, scale=1.0):
    return (np.random.default_rng(seed).standard_normal((rows, cols)) * scale).astype(np.float32)


def to_space(lib, a, space):
    """an array in the requested memory space: numpy for HOST (and for DEVICE in the emulator, where device memory is
    host memory), a torch CUDA tensor for DEVICE on the GPU"""
    if space == DEVICE and is_gpu(lib):
        import torch
        return torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return np.ascontiguousarray(a)


def ptr(a):
    import ctypes
    return ctypes.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)


def to_host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def raw_filter(lib, f, h, hs, x, xs, n_out, os_, hp=0, xp=0, op=0, n=None, out_rows=None):
    """vv_dsp_fir_filter_batch with every buffer in the space asked for; h / x are 2-D numpy arrays whose row length
    is their pitch when hp / xp are given (n = valid samples per row); returns (status, output as numpy [batch, pitch])"""
    n = x.shape[1] if n is None else n
    batch = x.shape[0]
    width = op or n_out
    out = np.full((batch if out_rows is None else out_rows, max(width, 1)), np.float32(7.5))
    hd, xd, od = to_space(lib, h, hs), to_space(lib, x, xs), to_space(lib, out, os_)
    st = lib.vv_dsp_fir_filter_batch(f._f, ptr(hd), hs, h.shape[0], hp, ptr(xd), xs, batch, n, xp, ptr(od), os_, n_out, op)
    f.synchronize()
    return st, to_host(od)


def routed_lines(lib, capfd, fn):
    """fn() with VVB_ROUTE_DEBUG=1: (its result, the library's stderr lines)"""
    return pc.routed(capfd, fn) if capfd is not None else (fn(), None)


def check_launches(lines, fft_size, parts, chunks=1):
    """one plain and parts - 1 ACCUM passes of fir_ols_kernel at this size per chunk, nothing else of the FIR family"""
    fir = [ln for ln in lines if "fir_ols_kernel" in ln]
    assert all("vvb::launch_fir(" in ln and f"C = Cfg<{fft_size}," in ln for ln in fir), fir
    assert sum("bool ACCUM = false" in ln for ln in fir) == chunks, fir
    assert sum("bool ACCUM = true" in ln for ln in fir) == chunks * (parts - 1), fir
    assert any("fir_pad_kernel" in ln for ln in lines) and any(f"vvb::launch_c2c(" in ln and f"C = Cfg<{fft_size}," in ln
                                                                for ln in lines), lines


# ----------------------------------------------------------------------------- checks
def lengths(m, block, long_n):
    """n shorter than M, shorter than one block, exactly L and L +- 1, an odd and an even block count, a long signal"""
    ns = {max(m // 2, 1), max(block // 2, 1), block, block - 1, block + 1, 3 * block - 5, 4 * block, long_n}
    return sorted(k for k in ns if k >= 1)


def check_row(lib, m, capfd=None, long_n=30000, batch=3):
    """One tap count against float64 truth: plan, launches, every signal length class, every n_out class, shared and
    per-signal filters.  Returns the worst error over the bound without FIR_C."""
    worst = 0.0
    with FirFilter(m, lib=lib) as f:
        assert (f.fft_size, f.partitions) == PLAN[m]
        block = f.fft_size - -(-m // f.partitions) + 1
        for i, n in enumerate(lengths(m, block, long_n)):
            nf = 1 if i % 2 == 0 else batch
            h, x = data(10 + i, nf, m, 1.0 / np.sqrt(m)), data(20 + i, batch, n)
            n_outs = [n, n + m - 1] if i != 3 else [0, max(n - 7, 1), n, n + m - 1, n + m + 100]
            for n_out in n_outs:
                y, lines = routed_lines(lib, capfd, lambda: f.filter(h, x, n_out))
                if lines is not None and n_out:
                    check_launches(lines, f.fft_size, f.partitions)
                y = to_host(y)
                assert y.shape == (batch, n_out)
                if n_out > n + m - 1:
                    assert not y[:, n + m - 1:].any()           # beyond the full convolution: exactly 0
                worst = max(worst, worst_ratio(y, h, x, n_out, f))
    assert worst < FIR_C, (m, worst)
    return worst


def check_known_answers(lib):
    """h = [1] returns x, h = delta[j - d] returns x delayed by d, to rounding"""
    x = data(3, 2, 5000)
    with FirFilter(1, lib=lib) as f:
        y = to_host(f.filter(np.ones((1, 1), np.float32), x))
        assert np.abs(y - x).max() <= 1e-6 * np.abs(x).max()
    for m, d in ((64, 17), (5463, 5000), (10000, 9999)):
        h = np.zeros((1, m), np.float32)
        h[0, d] = 1.0
        with FirFilter(m, lib=lib) as f:
            y = to_host(f.filter(h, x, x.shape[1] + m - 1))
        want = np.zeros_like(y)
        want[:, d:d + x.shape[1]] = x
        assert np.abs(y - want).max() <= 1e-6 * np.abs(x).max(), (m, d)


def check_filters_and_batch(lib, m, n):
    """a shared filter is bit-identical to the same filter repeated in every row; one signal alone is bit-identical to the
    same signal inside a batch of 64"""
    h, x = data(5, 1, m, 0.1), data(6, 64, n)
    with FirFilter(m, lib=lib) as f:
        shared = to_host(f.filter(h, x))
        per_signal = to_host(f.filter(np.repeat(h, 64, axis=0), x))
        assert np.array_equal(shared, per_signal)
        for b in (0, 37, 63):
            assert np.array_equal(to_host(f.filter(h, x[b:b + 1])), shared[b:b + 1])
        hs = data(7, 64, m, 0.1)
        many = to_host(f.filter(hs, x))
        assert np.array_equal(to_host(f.filter(hs[37:38], x[37:38])), many[37:38])


def check_spaces(lib, m, n, batch=5, monkeypatch=None, capfd=None):
    """HOST / DEVICE in every combination, with row pitches wider than the rows (odd), equal to the dense HOST result bit for
    bit, and nothing written into the pitch padding; several staging chunks (VVB_STAGE_TARGET_BYTES) equal one chunk.
    The rows pick n so that n_out = n + M - 1 is an odd multiple of the block length: the last pair of blocks has an
    empty half, whose samples would start right in the padding."""
    n_out = n + m - 1
    with FirFilter(m, lib=lib) as f:
        block = f.fft_size - -(-m // f.partitions) + 1
    assert n_out % block == 0 and (n_out // block) % 2 == 1, (m, n)
    hp, xp, op = m + 3, n + 5, n_out + 7
    hw, xw = data(8, batch, hp, 0.1), data(9, batch, xp)
    for nf in (1, batch):
        h = np.ascontiguousarray(hw[:nf, :m])
        with FirFilter(m, lib=lib) as f:
            st, ref = raw_filter(lib, f, h, HOST, np.ascontiguousarray(xw[:, :n]), HOST, n_out, HOST)
            assert st == 0
            assert worst_ratio(ref[:, :n_out], h, xw[:, :n], n_out, f) < FIR_C
            for spaces in [(a, b, c) for a in (HOST, DEVICE) for b in (HOST, DEVICE) for c in (HOST, DEVICE)]:
                st, y = raw_filter(lib, f, hw[:nf], spaces[0], xw, spaces[1], n_out, spaces[2], hp=hp, xp=xp, op=op, n=n)
                assert st == 0, spaces
                assert np.array_equal(y[:, :n_out], ref), (nf, spaces)
                assert np.all(y[:, n_out:] == np.float32(7.5)), (nf, spaces)
        if monkeypatch is not None:
            with monkeypatch.context() as mp:
                mp.setenv("VVB_STAGE_TARGET_BYTES", str(4 * (n + m)))        # one signal per chunk
                with FirFilter(m, lib=lib) as f:
                    y, lines = routed_lines(lib, capfd, lambda: raw_filter(lib, f, h, HOST, np.ascontiguousarray(xw[:, :n]), HOST,
                                                                           n_out, HOST))
                    assert y[0] == 0 and np.array_equal(y[1], ref), nf
                    if lines is not None:
                        check_launches(lines, f.fft_size, f.partitions, chunks=batch)


def check_status_codes(lib):
    import ctypes
    from vv_dsp_b200.api import _vp
    h = _vp()
    assert lib.vv_dsp_fir_create(0, ctypes.byref(h)) == 2
    assert lib.vv_dsp_fir_create(16, None) == 1
    assert lib.vv_dsp_fir_destroy(None) == 1
    assert lib.vv_dsp_fir_set_stream(None, None) == 1
    assert lib.vv_dsp_fir_synchronize(None) == 1
    with pytest.raises(VvDspError):
        FirFilter(0, lib=lib)
    with FirFilter(16, lib=lib) as f:
        n1, n2 = ctypes.c_size_t(), ctypes.c_size_t()
        assert lib.vv_dsp_fir_get_config(None, ctypes.byref(n1), ctypes.byref(n2)) == 1
        assert lib.vv_dsp_fir_get_config(f._f, None, ctypes.byref(n2)) == 1
        h, x, y = np.ones((3, 16), np.float32), np.ones((3, 100), np.float32), np.zeros((3, 100), np.float32)
        call = lambda *a: lib.vv_dsp_fir_filter_batch(f._f, *a)       # noqa: E731
        ok = (ptr(h), HOST, 3, 0, ptr(x), HOST, 3, 100, 0, ptr(y), HOST, 100, 0)
        assert call(*ok) == 0
        assert lib.vv_dsp_fir_filter_batch(None, *ok) == 1
        for i in (0, 4, 9):                                            # filters, signals, out
            assert call(*ok[:i], None, *ok[i + 1:]) == 1
        for i in (1, 5, 10):                                           # memory spaces
            assert call(*ok[:i], 2, *ok[i + 1:]) == 3
        assert call(*ok[:2], 2, *ok[3:]) == 2                          # num_filters not in {1, batch}
        assert call(*ok[:2], 0, *ok[3:]) == 2
        assert call(*ok[:3], 15, *ok[4:]) == 2                         # pitches below their rows
        assert call(*ok[:8], 99, *ok[9:]) == 2
        assert call(*ok[:12], 99) == 2
        assert call(*ok[:9], ptr(x), *ok[10:]) == 6                    # out == signals
        y[:] = 3.0
        assert call(*ok[:2], 1, *ok[3:6], 0, *ok[7:]) == 0 and np.all(y == 3.0)     # batch == 0
        assert call(*ok[:11], 0, 0) == 0 and np.all(y == 3.0)          # n_out == 0
        with pytest.raises(ValueError):                                # a HOST out of another shape
            f.filter(h, x, out=np.zeros((3, 101), np.float32))


def check_plan_edges(lib):
    for m, cfg in PLAN_EDGES.items():
        with FirFilter(m, lib=lib) as f:
            assert (f.fft_size, f.partitions) == cfg, m


# ----------------------------------------------------------------------------- CPU emulator
EMU_ROWS = [1, 2, 31, 64, 128, 255, 512, 1000, 2049, 5462, 5463, 10000]


@pytest.mark.parametrize("m", EMU_ROWS)
def test_emu_row_vs_float64_truth(emu, capfd, m):
    worst = check_row(emu, m, capfd=capfd, long_n=12000 if m < 5000 else 25000, batch=2)
    with capfd.disabled():
        print(f"\nFIR M={m}: worst error / bound without C = {worst:.2e} (C = {FIR_C:.0e})")


def test_emu_plan_edges(emu):
    check_plan_edges(emu)


def test_emu_known_answers(emu):
    check_known_answers(emu)


def test_emu_filters_and_batch(emu):
    check_filters_and_batch(emu, 31, 700)
    check_filters_and_batch(emu, 5463, 9000)


@pytest.mark.parametrize("m,n", [(64, 3 * 449 - 63), (5463, 3 * 5461 - 5462)])
def test_emu_spaces_and_chunks(emu, monkeypatch, capfd, m, n):
    check_spaces(emu, m, n, batch=3, monkeypatch=monkeypatch, capfd=capfd)


def test_emu_status_codes(emu):
    check_status_codes(emu)


# ----------------------------------------------------------------------------- B200
@pytest.mark.gpu
@pytest.mark.parametrize("m", sorted(PLAN))
def test_gpu_row_vs_float64_truth(lib, capfd, m):
    worst = check_row(lib, m, capfd=capfd, long_n=480000 if m < 20000 else 200000, batch=4)
    with capfd.disabled():
        print(f"\nFIR M={m}: worst error / bound without C = {worst:.2e} (C = {FIR_C:.0e})")


@pytest.mark.gpu
def test_gpu_plan_edges_and_known_answers(lib):
    check_plan_edges(lib)
    check_known_answers(lib)


@pytest.mark.gpu
def test_gpu_filters_and_batch(lib):
    check_filters_and_batch(lib, 31, 48000)
    check_filters_and_batch(lib, 5463, 48000)
    check_filters_and_batch(lib, 10000, 30000)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(64, 107 * 449 - 63), (1000, 3 * 7193 - 999), (10000, 7 * 4859 - 9999)])
def test_gpu_spaces_and_chunks(lib, monkeypatch, capfd, m, n):
    check_spaces(lib, m, n, batch=6, monkeypatch=monkeypatch, capfd=capfd)


@pytest.mark.gpu
def test_gpu_status_codes(lib):
    check_status_codes(lib)


@pytest.mark.gpu
def test_gpu_torch_views_equal_host_path(lib):
    """torch views with odd row pitches (filters, signals, out) give the host path's result bit for bit"""
    import torch
    m, n, batch = 2049, 30001, 5
    h, x = data(11, batch, m, 0.03), data(12, batch, n)
    with FirFilter(m, lib=lib) as f:
        want = f.filter(h, x, n + m - 1)
        hw = torch.zeros((batch, m + 3), device="cuda"); hw[:, :m] = torch.from_numpy(h).cuda()
        xw = torch.zeros((batch, n + 5), device="cuda"); xw[:, :n] = torch.from_numpy(x).cuda()
        ow = torch.full((batch, n + m - 1 + 7), 7.5, device="cuda")
        got = f.filter(hw[:, :m], xw[:, :n], n + m - 1, out=ow[:, :n + m - 1])
        torch.cuda.synchronize()
        assert got.data_ptr() == ow.data_ptr()
        assert np.array_equal(got.cpu().numpy(), want)
        assert bool((ow[:, n + m - 1:] == 7.5).all())
        with pytest.raises(TypeError):
            f.filter(hw[:, :m].double(), xw[:, :n])
        with pytest.raises(ValueError):
            f.filter(hw[:, :m], xw[:, :2 * (n // 2):2])


@pytest.mark.gpu
def test_gpu_filter_scratch_chunks(lib, capfd):
    """per-signal filters of 48 000 taps for 200 signals: the spectra (12 x 8192 complex values per filter) exceed the
    handle's 128 MB filter scratch, so the call runs in two chunks of signals -- against float64 truth, and each signal
    bit-identical to itself filtered alone"""
    m, n, batch = 48000, 20000, 200
    h, x = data(13, batch, m, 1.0 / np.sqrt(m)), data(14, batch, n)
    with FirFilter(m, lib=lib) as f:
        y, lines = pc.routed(capfd, lambda: f.filter(h, x))
        check_launches(lines, 8192, 12, chunks=2)
        assert worst_ratio(y, h, x, n, f) < FIR_C
        for b in (0, 170, 199):
            assert np.array_equal(f.filter(h[b:b + 1], x[b:b + 1]), y[b:b + 1])


@pytest.mark.gpu
def test_gpu_device_calls_follow_torchs_current_stream(lib):
    """No set_stream(): device-tensor calls are enqueued on torch's current stream, so they are ordered against the torch
    ops that produce their inputs and consume their outputs (also on a side stream)."""
    import torch
    m, n, batch = 5463, 480000, 16
    g = torch.Generator(device="cuda").manual_seed(7)
    base = torch.rand((batch, n), device="cuda", generator=g) * 2 - 1
    h = torch.rand((batch, m), device="cuda", generator=g) * 1e-2
    with FirFilter(m, lib=lib) as f:
        torch.cuda.synchronize()
        want = f.filter(h, base * 0.5)
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        for s in (torch.cuda.current_stream(), side):
            with torch.cuda.stream(s):
                big = torch.rand((4096, 4096), device="cuda")
                for _ in range(20):
                    big = big @ big * 1e-3                       # keeps the stream busy: the input below is late
                x = base * 0.5                                    # produced on this stream
                y = f.filter(h, x)
                z = y * 2.0                                       # consumed on this stream
            torch.cuda.synchronize()
            assert torch.equal(y, want)
            assert torch.equal(z, want * 2.0)
