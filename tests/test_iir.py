"""Batched IIR filtering by second-order sections (vv_dsp_sos_*, include/vv_dsp/b200.h) against scipy.signal.sosfilt /
sosfiltfilt in float64.

One set of check_* functions runs in the CPU emulator (tests/emu: the kernel sources compiled for the CPU, small sizes) and
on the B200 (the nvcc-built library, -m gpu, full sizes).  Truth is scipy in float64 on the float32-rounded sos and the
float32 input; a row passes when max|y - y64| <= 4 e32 + 16 2^-24 max|y64|, e32 being the error of scipy's own
sequential float32 recurrence against the same truth.  Every call asserts the launches VVB_ROUTE_DEBUG reports: launch C
alone for rows of at most one segment, A, B and C for longer ones (the emulator reaches those through VVB_IIR_SEGMENT)."""
import ctypes
import os
import sys

import numpy as np
import pytest
from scipy.signal import butter, ellip, sosfilt, sosfilt_zi, sosfiltfilt
from scipy.signal._arraytools import const_ext, even_ext, odd_ext

import parity_cases as pc
from vv_dsp_b200 import SosFilter, VvDspError

HERE = os.path.dirname(os.path.abspath(__file__))
HOST, DEVICE = 0, 1
EPS32 = 2.0 ** -24
RUN, TILE, SEGMENT = 16, 4096, 1 << 20
EMU_SEGMENT = 2 * TILE                      # VVB_IIR_SEGMENT of the emulator's segmented rows


def random_sections(seed, count, radius=0.99):
    """seeded stable sections: complex pole pairs (or two real poles) of radius <= `radius`, random zeros"""
    rng = np.random.default_rng(seed)
    rows = []
    for _ in range(count):
        r, th = radius * np.sqrt(rng.uniform(0.05, 1.0)), rng.uniform(0.0, np.pi)
        if rng.uniform() < 0.25:
            p1, p2 = radius * rng.uniform(-1, 1), radius * rng.uniform(-1, 1)
            a1, a2 = -(p1 + p2), p1 * p2
        else:
            a1, a2 = -2.0 * r * np.cos(th), r * r
        rows.append([*rng.standard_normal(3) * 0.5, 1.0, a1, a2])
    return np.array(rows)


FILTERS = {
    "identity": np.array([[1.0, 0, 0, 1, 0, 0]]),
    "lowpass_1k": butter(2, 1000, fs=48000, output="sos"),
    "highpass_20": butter(2, 20, "highpass", fs=48000, output="sos"),
    "bandpass_50_8k": butter(4, [50, 8000], "bandpass", fs=48000, output="sos"),
    "ellip8": ellip(8, 0.5, 80, 0.05, output="sos"),
    "dc_blocker": np.array([[1.0, -1.0, 0, 1, -0.995, 0]]),
    "preemphasis": np.array([[1.0, -0.97, 0, 1, 0, 0]]),
    "butter32": butter(32, 0.1, output="sos"),
    "random64": random_sections(5, 64),
}
SECTIONS = {"identity": 1, "lowpass_1k": 1, "highpass_20": 1, "bandpass_50_8k": 4, "ellip8": 4, "dc_blocker": 1,
            "preemphasis": 1, "butter32": 16, "random64": 64}


def sos32(name):
    return np.asarray(FILTERS[name], np.float32)


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
    return None if a is None else ctypes.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)


def to_host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def zi_unit32(sos):
    """sosfilt_zi in float64 on the float32 sos, rounded to float32 once (as the handle does)"""
    return sosfilt_zi(sos.astype(np.float64)).astype(np.float32)


def default_padlen(sos):
    return 3 * (2 * len(sos) + 1 - min(int((sos[:, 2] == 0).sum()), int((sos[:, 5] == 0).sum())))


def filtfilt32(sos, x, padtype, padlen):
    """sosfiltfilt composed from float32 pieces: the textbook float32 forward-backward the device is held to"""
    edge = 0 if padtype is None else (default_padlen(sos) if padlen is None else padlen)
    ext = {"odd": odd_ext, "even": even_ext, "constant": const_ext}[padtype](x, edge, axis=-1) if edge else x
    zi = zi_unit32(sos)[:, None, :]
    y, _ = sosfilt(sos, ext, axis=-1, zi=zi * ext[None, :, :1])
    y, _ = sosfilt(sos, y[:, ::-1], axis=-1, zi=zi * y[None, :, -1:])
    y = y[:, ::-1]
    return y[:, edge:y.shape[1] - edge] if edge else y


# zf is held to a wider bound than the outputs: a finding, explained in DESIGN.md section 4 (IIR accuracy).  With a pole
# pair near z = 1 (the 20 Hz high-pass) the end state's error reaches ~47 e32 in the emulator, while every output stays
# within 4 e32 + 16 2^-24 max|y64|.
ZF_E32, ZF_REL = 64, 256


def check_bound(y, y64, y32, what, c32=4, rel=16):
    """per row: max|y - y64| <= c32 e32 + rel 2^-24 max|y64|.  Returns the worst ratio of the error to the bound."""
    y, y64, y32 = (np.asarray(a, np.float64).reshape(len(y64), -1) for a in (y, y64, y32))
    worst = 0.0
    for r in range(len(y64)):
        err = float(np.abs(y[r] - y64[r]).max(initial=0.0))
        bound = c32 * float(np.abs(y32[r] - y64[r]).max(initial=0.0)) + rel * EPS32 * float(np.abs(y64[r]).max(initial=0.0))
        assert err <= bound or err == 0.0, (what, r, err, bound)
        worst = max(worst, err / bound if bound > 0 else 0.0)
    return worst


def routed_lines(capfd, fn):
    return pc.routed(capfd, fn) if capfd is not None else (fn(), None)


def check_launches(lines, nv, segment, passes=1):
    """per pass: launch C alone for nv <= segment, else A, B and C in that order"""
    kern = [ln for ln in lines if "iir_tile_kernel" in ln or "iir_chain_kernel" in ln]
    one = ["C"] if nv <= segment else ["A", "B", "C"]
    got = []
    for ln in kern:
        if "iir_chain_kernel" in ln:
            assert "vvb::launch_iir_chain(" in ln, ln
            got.append("B")
        else:
            assert "vvb::launch_iir_tile(" in ln and "int L = 16" in ln, ln
            got.append("A" if "bool STATES = true" in ln else "C")
    assert got == one * passes, (got, lines)


# ----------------------------------------------------------------------------- checks
def check_filter_row(lib, name, ns, batch=2, capfd=None, segment=SEGMENT):
    """sosfilt without and with zi, zf against scipy's, over every length in ns.  Returns the worst error / bound."""
    s32 = sos32(name)
    s64 = s32.astype(np.float64)
    S = len(s32)
    worst = 0.0
    with SosFilter(s32, lib=lib) as f:
        assert (f.n_sections, f.segment_length) == (S, segment)
        for i, n in enumerate(ns):
            x = data(100 + i, batch, n)
            y, lines = routed_lines(capfd, lambda: f.filter(x))
            if lines is not None:
                check_launches(lines, n, segment)
            y64 = sosfilt(s64, x.astype(np.float64), axis=-1)
            if name == "identity":
                assert np.array_equal(y, x)
            worst = max(worst, check_bound(y, y64, sosfilt(s32, x, axis=-1), (name, n)))
            zi = (np.random.default_rng(200 + i).standard_normal((S, batch, 2)) * 0.5).astype(np.float32)
            (y, zf), lines = routed_lines(capfd, lambda: f.filter(x, zi=zi, return_zf=True))
            if lines is not None:
                check_launches(lines, n, segment)
            y64, zf64 = sosfilt(s64, x.astype(np.float64), axis=-1, zi=zi.astype(np.float64))
            y32, zf32 = sosfilt(s32, x, axis=-1, zi=zi)
            worst = max(worst, check_bound(y, y64, y32, (name, n, "zi")))
            worst = max(worst, check_bound(zf.transpose(1, 0, 2), zf64.transpose(1, 0, 2), zf32.transpose(1, 0, 2),
                                           (name, n, "zf"), c32=ZF_E32, rel=ZF_REL))
    return worst


def check_chained(lib, name, n, batch=2):
    """three calls passing zf -> zi equal one scipy call over the whole rows, within the bound"""
    s32 = sos32(name)
    x = data(21, batch, n)
    cuts = [0, n // 3, n // 3 + 1, n]
    parts = []
    with SosFilter(s32, lib=lib) as f:
        z = np.zeros((len(s32), batch, 2), np.float32)
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b > a:
                y, z = f.filter(np.ascontiguousarray(x[:, a:b]), zi=z, return_zf=True)
                parts.append(y)
    y = np.concatenate(parts, axis=1)
    y64, zf64 = sosfilt(s32.astype(np.float64), x.astype(np.float64), axis=-1, zi=np.zeros((len(s32), batch, 2)))
    y32, zf32 = sosfilt(s32, x, axis=-1, zi=np.zeros((len(s32), batch, 2), np.float32))
    return max(check_bound(y, y64, y32, (name, "chained")),
               check_bound(z.transpose(1, 0, 2), zf64.transpose(1, 0, 2), zf32.transpose(1, 0, 2), (name, "chained zf"),
                           c32=ZF_E32, rel=ZF_REL))


def check_filtfilt_row(lib, name, ns, batch=2, capfd=None, segment=SEGMENT, padlens=(None,)):
    """sosfiltfilt with every padtype and the given padlens (None: scipy's default) over every length in ns"""
    s32 = sos32(name)
    s64 = s32.astype(np.float64)
    worst = 0.0
    with SosFilter(s32, lib=lib) as f:
        for i, n in enumerate(ns):
            x = data(300 + i, batch, n)
            for padtype in ("odd", "even", "constant", None):
                for padlen in padlens:
                    edge = 0 if padtype is None else (default_padlen(s32) if padlen is None else padlen)
                    if n <= edge:
                        with pytest.raises(VvDspError):
                            f.filtfilt(x, padtype=padtype, padlen=padlen)
                        continue
                    y, lines = routed_lines(capfd, lambda: f.filtfilt(x, padtype=padtype, padlen=padlen))
                    if lines is not None:
                        check_launches(lines, n + 2 * edge, segment, passes=2)
                    y64 = sosfiltfilt(s64, x.astype(np.float64), axis=-1, padtype=padtype, padlen=padlen)
                    worst = max(worst, check_bound(y, y64, filtfilt32(s32, x, padtype, padlen), (name, n, padtype, padlen)))
    return worst


def check_batch_identity(lib, name, n, monkeypatch=None, capfd=None):
    """one row alone is bit-identical to itself inside a batch of 40; several staging chunks equal one (filter, zf and
    filtfilt)"""
    s32 = sos32(name)
    x = data(31, 40, n)
    zi = (np.random.default_rng(32).standard_normal((len(s32), 40, 2))).astype(np.float32)
    with SosFilter(s32, lib=lib) as f:
        many, zf = f.filter(x, zi=zi, return_zf=True)
        ff = f.filtfilt(x)
        for b in (0, 17, 39):
            y1, z1 = f.filter(x[b:b + 1], zi=np.ascontiguousarray(zi[:, b:b + 1]), return_zf=True)
            assert np.array_equal(y1, many[b:b + 1]) and np.array_equal(z1, zf[:, b:b + 1])
            assert np.array_equal(f.filtfilt(x[b:b + 1]), ff[b:b + 1])
    if monkeypatch is not None:
        with monkeypatch.context() as mp:
            mp.setenv("VVB_STAGE_TARGET_BYTES", str(4 * 3 * n))                 # three rows per chunk
            with SosFilter(s32, lib=lib) as f2:
                (y, z), lines = routed_lines(capfd, lambda: f2.filter(x, zi=zi, return_zf=True))
                assert np.array_equal(y, many) and np.array_equal(z, zf)
                if lines is not None:
                    check_launches(lines, n, f2.segment_length, passes=14)
                assert np.array_equal(f2.filtfilt(x), ff)


def raw_filter(lib, f, x, xs, zs, fs, os_, zi, with_zf, xp=0, op=0):
    """vv_dsp_sos_filter_batch with every buffer in the space asked for; x is 2-D numpy whose row length is its pitch when
    xp is given; out is prefilled with 7.5.  Returns (status, out, zf) as numpy"""
    batch, n = x.shape[0], (x.shape[1] if not xp else xp - 5)
    out = np.full((batch, op or n), np.float32(7.5))
    xd, od = to_space(lib, x, xs), to_space(lib, out, os_)
    zid = None if zi is None else to_space(lib, zi, zs)
    zfd = to_space(lib, np.full((f.n_sections, batch, 2), np.float32(9.0)), fs) if with_zf else None
    st = lib.vv_dsp_sos_filter_batch(f._h, ptr(xd), xs, batch, n, xp, ptr(zid), zs, ptr(zfd), fs, ptr(od), os_, op)
    f.synchronize()
    return st, to_host(od), None if zfd is None else to_host(zfd)


def check_spaces(lib, name, n, batch=3):
    """HOST / DEVICE for signals, zi, zf and out, dense and with odd row pitches: bit-identical to the all-HOST result,
    nothing written into the pitch padding; filtfilt likewise for signals and out"""
    s32 = sos32(name)
    xw = data(41, batch, n + 5)
    x = np.ascontiguousarray(xw[:, :n])
    zi = np.random.default_rng(42).standard_normal((len(s32), batch, 2)).astype(np.float32)
    with SosFilter(s32, lib=lib) as f:
        st, ref, zref = raw_filter(lib, f, x, HOST, HOST, HOST, HOST, zi, True)
        assert st == 0
        for xs in (HOST, DEVICE):
            for zs in (HOST, DEVICE):
                for fs in (HOST, DEVICE):
                    for os_ in (HOST, DEVICE):
                        st, y, z = raw_filter(lib, f, x, xs, zs, fs, os_, zi, True)
                        assert st == 0 and np.array_equal(y, ref) and np.array_equal(z, zref), (xs, zs, fs, os_)
                st, y, z = raw_filter(lib, f, xw, xs, zs, zs, 1 - xs, zi, True, xp=n + 5, op=n + 7)
                assert st == 0 and np.array_equal(y[:, :n], ref) and np.all(y[:, n:] == np.float32(7.5)), (xs, zs)
                assert np.array_equal(z, zref)
        ffref = f.filtfilt(x)
        for xs in (HOST, DEVICE):
            for os_ in (HOST, DEVICE):
                out = np.full((batch, n + 7), np.float32(7.5))
                xd, od = to_space(lib, xw, xs), to_space(lib, out, os_)
                assert lib.vv_dsp_sos_filtfilt_batch(f._h, ptr(xd), xs, batch, n, n + 5, 1, 2 ** 64 - 1, ptr(od), os_,
                                                     n + 7) == 0
                f.synchronize()
                y = to_host(od)
                assert np.array_equal(y[:, :n], ffref) and np.all(y[:, n:] == np.float32(7.5)), (xs, os_)


def check_status_codes(lib):
    h = ctypes.c_void_p()
    create = lib.vv_dsp_sos_create
    good = sos32("bandpass_50_8k")

    def made(sos, count=None):
        s = np.ascontiguousarray(sos, np.float32)
        st = create(ptr(s), len(s) if count is None else count, ctypes.byref(h))
        if st == 0:
            lib.vv_dsp_sos_destroy(h)
        return st

    assert create(ptr(good), 4, None) == 1                                     # NULL out
    assert create(None, 4, ctypes.byref(h)) == 1                               # NULL sos
    assert made(good, 0) == 2                                                  # S == 0
    assert made(np.tile(good, (17, 1)), 65) == 2                               # S == 65
    assert made(np.tile(good, (16, 1))) == 0                                   # S == 64
    for i in range(6):
        for bad in (np.nan, np.inf):
            s = good.copy()
            s[2, i] = bad
            assert made(s) == 5, (i, bad)                                      # not finite
    s = good.copy(); s[1, 3] = 2.0
    assert made(s) == 3                                                        # a0 != 1
    for a1, a2 in ((0.0, 1.0), (-2.0, 1.0), (0.0, -1.0), (-1.0, 0.0), (1.0, 0.0), (-1.5, 0.4), (0.0, 1.2)):
        assert made([[1, 0, 0, 1, a1, a2]]) == 3, (a1, a2)                    # a pole on or outside the unit circle
    assert made([[1, 0, 0, 1, -1.998, 0.998001]]) == 0                         # radius 0.999
    assert lib.vv_dsp_sos_destroy(None) == 1
    assert lib.vv_dsp_sos_set_stream(None, None) == 1
    assert lib.vv_dsp_sos_synchronize(None) == 1
    with pytest.raises(VvDspError):
        SosFilter([[1, 0, 0, 1, 0, 1.5]], lib=lib)
    with pytest.raises(ValueError):
        SosFilter([1, 0, 0, 1, 0, 0], lib=lib)
    with SosFilter(good, lib=lib) as f:
        s = ctypes.c_size_t()
        assert lib.vv_dsp_sos_get_config(None, ctypes.byref(s), ctypes.byref(s)) == 1
        assert lib.vv_dsp_sos_get_config(f._h, None, ctypes.byref(s)) == 1
        assert lib.vv_dsp_sos_get_config(f._h, ctypes.byref(s), None) == 1
        x, y = np.ones((3, 300), np.float32), np.zeros((3, 300), np.float32)
        zi = np.full((4, 3, 2), 2.5, np.float32)
        zf = np.zeros((4, 3, 2), np.float32)
        call = lambda *a: lib.vv_dsp_sos_filter_batch(f._h, *a)                 # noqa: E731
        ok = (ptr(x), HOST, 3, 300, 0, ptr(zi), HOST, ptr(zf), HOST, ptr(y), HOST, 0)
        assert call(*ok) == 0
        assert lib.vv_dsp_sos_filter_batch(None, *ok) == 1                     # NULL handle
        for i in (0, 9):                                                       # signals, out
            assert call(*ok[:i], None, *ok[i + 1:]) == 1
        for i in (1, 6, 8, 10):                                                # memory spaces
            assert call(*ok[:i], 2, *ok[i + 1:]) == 3
        assert call(*ok[:4], 299, *ok[5:]) == 2                                # signal pitch below its row
        assert call(*ok[:11], 299) == 2                                        # out pitch below its row
        assert call(*ok[:9], ptr(x), *ok[10:]) == 6                            # out == signals
        y[:] = 3.0
        zf[:] = 7.0
        assert call(*ok[:2], 0, *ok[3:]) == 0 and np.all(y == 3.0) and np.all(zf == 7.0)     # batch == 0
        assert call(*ok[:3], 0, *ok[4:]) == 0 and np.all(y == 3.0) and np.all(zf == 2.5)     # n == 0: zf = zi
        assert call(*ok[:5], None, HOST, *ok[7:]) == 0                          # zi == NULL: the zero state
        zf[:] = 7.0
        assert call(*ok[:3], 0, 0, None, HOST, *ok[7:]) == 0 and np.all(zf == 0.0)          # n == 0, no zi: zeros
        ff = lambda *a: lib.vv_dsp_sos_filtfilt_batch(f._h, *a)                # noqa: E731
        okf = (ptr(x), HOST, 3, 300, 0, 1, 2 ** 64 - 1, ptr(y), HOST, 0)
        assert ff(*okf) == 0
        assert lib.vv_dsp_sos_filtfilt_batch(None, *okf) == 1
        for i in (0, 7):
            assert ff(*okf[:i], None, *okf[i + 1:]) == 1
        for i in (1, 8):
            assert ff(*okf[:i], 2, *okf[i + 1:]) == 3
        for bad in (-1, 4):                                                    # padtype
            assert ff(*okf[:5], bad, *okf[6:]) == 3
        assert ff(*okf[:4], 299, *okf[5:]) == 2
        assert ff(*okf[:9], 299) == 2
        assert ff(*okf[:7], ptr(x), *okf[8:]) == 6
        assert ff(*okf[:6], 300, *okf[7:]) == 2                                # n <= padlen
        assert ff(*okf[:6], 299, *okf[7:]) == 0
        xs = np.ones((3, 27), np.float32)                                      # default padlen 27 for 4 sections
        assert ff(ptr(xs), HOST, 3, 27, 0, 1, 2 ** 64 - 1, ptr(y), HOST, 0) == 2
        assert ff(ptr(xs), HOST, 3, 27, 0, 0, 2 ** 64 - 1, ptr(y), HOST, 0) == 0            # padtype none: no padding
        assert ff(*okf[:2], 0, *okf[3:]) == 0 and ff(*okf[:3], 0, *okf[4:]) == 0            # batch == 0, n == 0
        with pytest.raises(ValueError):
            f.filtfilt(x, padtype="reflect")
        with pytest.raises(ValueError):
            f.filter(x, zi=np.zeros((4, 2, 2), np.float32))
    with SosFilter(sos32("dc_blocker"), lib=lib) as f:                          # first-order section: default padlen 6
        assert default_padlen(sos32("dc_blocker")) == 6
        x7 = data(1, 1, 7)
        assert np.array_equal(f.filtfilt(x7).shape, (1, 7))
        with pytest.raises(VvDspError):
            f.filtfilt(x7[:, :6])


# ----------------------------------------------------------------------------- CPU emulator
EMU_LENGTHS = [1, 2, RUN - 1, RUN, RUN + 1, TILE - 1, TILE, TILE + 1, 2 * TILE + 1234]


@pytest.mark.parametrize("name", sorted(FILTERS))
def test_emu_filter_vs_float64_truth(emu, capfd, name):
    ns = EMU_LENGTHS if SECTIONS[name] <= 4 else [1, RUN + 1, TILE + 1]
    worst = check_filter_row(emu, name, ns, capfd=capfd)
    with capfd.disabled():
        print(f"\nsosfilt {name}: worst error / bound = {worst:.2e}")


@pytest.mark.parametrize("name", sorted(FILTERS))
def test_emu_filtfilt_vs_float64_truth(emu, capfd, name):
    ns = [200, TILE + 1] if SECTIONS[name] <= 4 else [200]
    worst = check_filtfilt_row(emu, name, ns, capfd=capfd, padlens=(None, 0, 17))
    with capfd.disabled():
        print(f"\nsosfiltfilt {name}: worst error / bound = {worst:.2e}")


@pytest.mark.parametrize("name", ["highpass_20", "bandpass_50_8k", "ellip8", "dc_blocker"])
def test_emu_segments(emu, capfd, monkeypatch, name):
    """rows of several segments plus a ragged one (VVB_IIR_SEGMENT = two tiles): launches A, B and C"""
    monkeypatch.setenv("VVB_IIR_SEGMENT", str(EMU_SEGMENT - 100))              # rounded up to a whole number of tiles
    n = 3 * EMU_SEGMENT + 1000
    check_filter_row(emu, name, [EMU_SEGMENT, EMU_SEGMENT + 1, n], capfd=capfd, segment=EMU_SEGMENT)
    check_filtfilt_row(emu, name, [n], capfd=capfd, segment=EMU_SEGMENT)
    assert check_chained(emu, name, n) <= 1.0


def test_emu_chained_calls(emu):
    for name in ("highpass_20", "ellip8"):
        check_chained(emu, name, 3 * TILE + 7)


def test_emu_batch_identity_and_chunks(emu, monkeypatch, capfd):
    check_batch_identity(emu, "bandpass_50_8k", 700, monkeypatch=monkeypatch, capfd=capfd)


def test_emu_spaces(emu):
    check_spaces(emu, "ellip8", 1201)


def test_emu_status_codes(emu):
    check_status_codes(emu)


# ----------------------------------------------------------------------------- B200
GPU_LENGTHS = [1, 2, RUN - 1, RUN, RUN + 1, TILE - 1, TILE, TILE + 1, 480000, SEGMENT, 3 * SEGMENT + 12345]


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FILTERS))
def test_gpu_filter_vs_float64_truth(lib, capfd, name):
    worst = check_filter_row(lib, name, GPU_LENGTHS, batch=3, capfd=capfd)
    with capfd.disabled():
        print(f"\nsosfilt {name}: worst error / bound = {worst:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FILTERS))
def test_gpu_filtfilt_vs_float64_truth(lib, capfd, name):
    worst = check_filtfilt_row(lib, name, [200, 48000, 2 * SEGMENT + 777], batch=2, capfd=capfd, padlens=(None, 0, 1000))
    with capfd.disabled():
        print(f"\nsosfiltfilt {name}: worst error / bound = {worst:.2e}")


@pytest.mark.gpu
def test_gpu_chained_calls(lib):
    for name in ("highpass_20", "ellip8", "butter32"):
        assert check_chained(lib, name, 2 * SEGMENT + 4097) <= 1.0


@pytest.mark.gpu
def test_gpu_batch_identity_and_chunks(lib, monkeypatch, capfd):
    check_batch_identity(lib, "bandpass_50_8k", 48000, monkeypatch=monkeypatch, capfd=capfd)
    check_batch_identity(lib, "highpass_20", SEGMENT + 5)


@pytest.mark.gpu
def test_gpu_spaces(lib):
    check_spaces(lib, "ellip8", 48001)
    check_spaces(lib, "highpass_20", SEGMENT + 3)


@pytest.mark.gpu
def test_gpu_status_codes(lib):
    check_status_codes(lib)


@pytest.mark.gpu
def test_gpu_torch_views_equal_host_path(lib):
    """torch views with odd row pitches (signals, out) give the host path's result bit for bit, zi / zf included"""
    import torch
    n, batch = 30001, 5
    x = data(51, batch, n)
    zi = np.random.default_rng(52).standard_normal((4, batch, 2)).astype(np.float32)
    with SosFilter(sos32("ellip8"), lib=lib) as f:
        want, zwant = f.filter(x, zi=zi, return_zf=True)
        ffwant = f.filtfilt(x, padtype="even")
        xw = torch.zeros((batch, n + 5), device="cuda"); xw[:, :n] = torch.from_numpy(x).cuda()
        ow = torch.full((batch, n + 7), 7.5, device="cuda")
        got, zf = f.filter(xw[:, :n], zi=torch.from_numpy(zi).cuda(), return_zf=True, out=ow[:, :n])
        torch.cuda.synchronize()
        assert got.data_ptr() == ow.data_ptr() and zf.is_cuda
        assert np.array_equal(got.cpu().numpy(), want) and np.array_equal(zf.cpu().numpy(), zwant)
        assert bool((ow[:, n:] == 7.5).all())
        got = f.filtfilt(xw[:, :n], padtype="even", out=ow[:, :n])
        torch.cuda.synchronize()
        assert np.array_equal(got.cpu().numpy(), ffwant) and bool((ow[:, n:] == 7.5).all())
        with pytest.raises(TypeError):
            f.filter(xw[:, :n].double())
        with pytest.raises(ValueError):
            f.filter(xw[:, :2 * (n // 2):2])


@pytest.mark.gpu
def test_gpu_device_calls_follow_torchs_current_stream(lib):
    """No set_stream(): device-tensor calls are enqueued on torch's current stream, so they are ordered against the torch
    ops that produce their inputs and consume their outputs (also on a side stream)."""
    import torch
    n, batch = 480000, 16
    g = torch.Generator(device="cuda").manual_seed(7)
    base = torch.rand((batch, n), device="cuda", generator=g) * 2 - 1
    with SosFilter(sos32("bandpass_50_8k"), lib=lib) as f:
        torch.cuda.synchronize()
        want = f.filter(base * 0.5)
        wantff = f.filtfilt(base * 0.5)
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        for s in (torch.cuda.current_stream(), side):
            with torch.cuda.stream(s):
                big = torch.rand((4096, 4096), device="cuda")
                for _ in range(20):
                    big = big @ big * 1e-3                       # keeps the stream busy: the input below is late
                x = base * 0.5                                    # produced on this stream
                y = f.filter(x)
                yy = f.filtfilt(x)
                z = y * 2.0                                       # consumed on this stream
            torch.cuda.synchronize()
            assert torch.equal(y, want) and torch.equal(yy, wantff)
            assert torch.equal(z, want * 2.0)
