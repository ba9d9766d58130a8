"""Batched polyphase resampling (vv_dsp_resample_poly_batch) on device-resident signals, against torch and scipy baselines.

    python benchmarks/resample_bench.py [--batch 1024] [--seconds 10] [--iters 5] [--rows 3] [--scipy-signals 4]
                                        [--out FILE.jsonl]

Workload: `batch` signals of `seconds` at the input rate, the default Kaiser design, for 48 -> 16 kHz (1, 3), 16 -> 48 kHz
(3, 1), 44.1 -> 16 kHz (160, 441), 48 -> 44.1 kHz (147, 160), 44.1 -> 48 kHz (160, 147) and 11.025 -> 192 kHz (2560, 147).
Timed with CUDA events after a warm-up call; every input is at least 0.65 GB, above the L2.  One JSON line per row:
  - ms per call and Gsamples/s of output;
  - the model's bytes (4 n + 4 n_out per signal plus the bank) and flops (2 per tap summed: T per output), and the share
    of the larger of the HBM bound (MEASURED_PEAKS.json if present, else the data sheet, labelled) and the FP32 bound
    (vv_dsp_b200_fp32_peak, scalar FFMA);
  - the worst error of sampled rows against float64 scipy.signal.resample_poly, over the bound of tests/test_resample.py;
  - baselines held to the same truth: torch conv1d(stride=down) for (1, 3) and conv_transpose1d(stride=up) for (3, 1) on
    the same GPU (TF32 off), and scipy.signal.resample_poly on one host core over a few signals, scaled to the batch.
The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

# (input rate, up, down): the five rows of a speech / audio front end and the largest bank of the standard rates
ROWS = [(48000, 1, 3), (16000, 3, 1), (44100, 160, 441), (48000, 147, 160), (44100, 160, 147), (11025, 2560, 147)]


def timed(fn, iters):
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--rows", type=int, default=3, help="sampled rows checked against float64 truth")
    ap.add_argument("--scipy-signals", type=int, default=4, help="signals resampled by scipy on one host core")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("resample_bench.py needs a CUDA device: nothing is measured without one")
    import torch.nn.functional as F
    from scipy.signal import resample_poly
    from fir_bench import card, hbm_peak
    from test_resample import default_window, worst_ratio
    from vv_dsp_b200 import Resampler, default_library

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    lib = default_library()
    name, power = card()
    hbm_gbs, hbm_src = hbm_peak()
    fp32 = lib.fp32_peak(False)
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        print(json.dumps(rec), flush=True)
        if out:
            out.write(json.dumps(rec) + "\n")

    emit(dict(card=name, power_limit_and_max_sm_clock=power, hbm_gbs=hbm_gbs, hbm_source=hbm_src, fp32_tflops=fp32,
              fp32_source="vv_dsp_b200_fp32_peak (scalar FFMA)"))
    B = args.batch
    g = torch.Generator(device="cuda").manual_seed(1)
    for rate, up, down in ROWS:
        n = int(round(rate * args.seconds))
        x = torch.rand((B, n), device="cuda", generator=g) * 2 - 1
        rows = np.linspace(0, B - 1, args.rows).astype(int)
        w = default_window(up, down)
        with Resampler(up, down, lib=lib) as r:
            n_out, T = r.output_length(n), r.taps_per_phase
            y = torch.empty((B, n_out), device="cuda")
            ms = timed(lambda: r.resample(x, out=y), args.iters)
            torch.cuda.synchronize()
            xs = x[rows].cpu().numpy()
            err_lib = worst_ratio(y[rows].cpu().numpy(), xs, up, down, w, T)
        bytes_ = B * (4 * n + 4 * n_out) + 4 * up * T
        flops = 2 * B * n_out * T
        t_hbm = bytes_ / (hbm_gbs * 1e9) * 1e3
        t_fp32 = flops / (fp32 * 1e12) * 1e3
        rec = dict(rate_in=rate, rate_out=rate * up // down, up=up, down=down, batch=B, n=n, n_out=n_out, num_taps=r.num_taps,
                   taps_per_phase=T, input_gb=round(4 * B * n / 1e9, 3), ms=round(ms, 3),
                   gsamples_per_s=round(B * n_out / ms / 1e6, 2), model_bytes=bytes_, model_flops=flops,
                   hbm_bound_ms=round(t_hbm, 3), fp32_bound_ms=round(t_fp32, 3), bound="HBM" if t_hbm >= t_fp32 else "FP32",
                   share_of_bound=round(max(t_hbm, t_fp32) / ms, 3), worst_err_over_bound_lib=err_lib,
                   lib_within_bound=bool(err_lib <= 1.0))
        # torch baselines on the same GPU, aligned to the same outputs: y[m] = sum_k h[k] xu[m down + half - k]
        h = torch.from_numpy((up * w).astype(np.float32)).cuda()
        half = (len(w) - 1) // 2
        base = None
        if up == 1:
            base = lambda: F.conv1d(x[:, None, :], h.flip(0)[None, None, :], stride=down, padding=half)[:, 0, :]   # noqa: E731
            label = "torch conv1d(stride=down)"
        elif down == 1:
            opad = up * n - ((n - 1) * up - 2 * half + len(w))
            base = lambda: F.conv_transpose1d(x[:, None, :], h[None, None, :], stride=up, padding=half,          # noqa: E731
                                              output_padding=opad)[:, 0, :]
            label = "torch conv_transpose1d(stride=up)"
        if base is not None:
            ms_t = timed(base, args.iters)
            yt = base()
            torch.cuda.synchronize()
            assert tuple(yt.shape) == (B, n_out), yt.shape
            rec.update(torch_baseline=label, torch_ms=round(ms_t, 3), speedup_vs_torch=round(ms_t / ms, 2),
                       worst_err_over_bound_torch=worst_ratio(yt[rows].cpu().numpy(), xs, up, down, w, T))
            del yt
        # scipy on one host core, a few signals, scaled to the batch
        k = max(1, min(args.scipy_signals, B))
        xh = x[:k].cpu().numpy()
        t0 = time.perf_counter()
        ys = [resample_poly(row, up, down, window=w, padtype="constant") for row in xh]
        ms_s = (time.perf_counter() - t0) * 1e3 * B / k
        rec.update(scipy_one_core_ms_scaled=round(ms_s, 1), scipy_signals_timed=k, speedup_vs_scipy_one_core=round(ms_s / ms, 1),
                   worst_err_over_bound_scipy_float32_input=worst_ratio(np.stack(ys), xh, up, down, w, T))
        emit(rec)
        del x, y
        torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
