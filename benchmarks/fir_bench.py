"""Batched FIR filtering (vv_dsp_fir_filter_batch) on device-resident signals, against a torch rfft / irfft convolution.

    python benchmarks/fir_bench.py [--batch 1024] [--n 480000] [--taps 64,512,2048,5462,16000,48000] [--iters 5]
                                   [--out FILE.jsonl]

Workload: `batch` signals of n samples (default: the headline shape, 1024 x 480 000), causal filtering (n_out = n), each
tap count with one shared filter and with a filter per signal.  Timed with CUDA events after a warm-up call; the inputs
(2 GB) are far larger than the L2.  One JSON line per workload:
  - ms per call, Gsamples/s (output samples), the plan's (N, P);
  - the model's bytes (P (4 n + 4 n_out) per signal plus the filter spectra) and flops (per pass and transform of two blocks:
    2 x 5 N log2 N for the forward and inverse transforms plus 6 N for the multiply; plus 5 N log2 N per filter partition for
    the spectra), and the share of the larger of the HBM and FP32 bounds (HBM bandwidth from MEASURED_PEAKS.json, FP32 from
    vv_dsp_b200_fp32_peak);
  - the baseline: torch.fft rfft / irfft convolution of the whole signal on the same GPU (a baseline only: the library does
    not use cuFFT), and the worst error of both against float64 truth on sampled rows, over the bound of tests/test_fir.py.
The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except (ValueError, KeyError):
            pass
    return 7700.0, "data sheet (MEASURED_PEAKS.json absent)"


def card():
    import torch
    name = torch.cuda.get_device_name()
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or "not read"
    except (OSError, subprocess.SubprocessError):
        power = "not read"
    return name, power


def model(batch, n, n_out, taps, fft_size, parts, num_filters):
    lp = -(-taps // parts)
    block = fft_size - lp + 1
    pairs = -(-(-(-n_out // block)) // 2)
    spectra = num_filters * parts * fft_size * 8
    bytes_ = batch * parts * (4 * n + 4 * n_out) + spectra
    lg = math.log2(fft_size)
    flops = parts * batch * pairs * (2 * 5 * fft_size * lg + 6 * fft_size) + num_filters * parts * 5 * fft_size * lg
    return bytes_, flops


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
    ap.add_argument("--n", type=int, default=480000)
    ap.add_argument("--taps", default="64,512,2048,5462,16000,48000")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--rows", type=int, default=3, help="sampled rows checked against float64 truth")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("fir_bench.py needs a CUDA device: nothing is measured without one")
    from test_fir import FIR_C, worst_ratio
    from vv_dsp_b200 import FirFilter, default_library

    lib = default_library()
    name, power = card()
    hbm_gbs, hbm_src = hbm_peak()
    fp32 = lib.fp32_peak(False)
    B, n = args.batch, args.n
    n_out = n
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.rand((B, n), device="cuda", generator=g) * 2 - 1
    y = torch.empty((B, n_out), device="cuda")
    rows = np.linspace(0, B - 1, args.rows).astype(int)
    out = open(args.out, "a") if args.out else None
    head = dict(card=name, power_limit_and_max_sm_clock=power, hbm_gbs=hbm_gbs, hbm_source=hbm_src, fp32_tflops=fp32,
                fp32_source="vv_dsp_b200_fp32_peak (scalar FFMA)")
    print(json.dumps(head), flush=True)
    if out:
        out.write(json.dumps(head) + "\n")
    for taps in [int(t) for t in args.taps.split(",")]:
        for mode in ("shared", "per_signal"):
            nf = 1 if mode == "shared" else B
            h = (torch.rand((nf, taps), device="cuda", generator=g) * 2 - 1) / math.sqrt(taps)
            with FirFilter(taps, lib=lib) as f:
                ms = timed(lambda: f.filter(h, x, n_out, out=y), args.iters)
                fft_size, parts = f.fft_size, f.partitions
                torch.cuda.synchronize()
                hs = h.cpu().numpy()
                xs = x[rows].cpu().numpy()
                hrows = hs if nf == 1 else hs[rows]
                err_lib = worst_ratio(y[rows].cpu().numpy(), hrows, xs, n_out, f)
            # baseline: one rfft / irfft convolution of every whole signal, cut to n_out
            nfft = 1 << (n + taps - 2).bit_length()

            def torch_conv():
                H = torch.fft.rfft(h, nfft)
                return torch.fft.irfft(torch.fft.rfft(x, nfft) * H, nfft)[:, :n_out]

            ms_torch = timed(torch_conv, max(1, args.iters // 2))
            yt = torch_conv()
            torch.cuda.synchronize()
            plan = SimpleNamespace(fft_size=fft_size, partitions=parts)     # the baseline is held to the library's bound
            err_torch = worst_ratio(yt[rows].cpu().numpy(), hrows, xs, n_out, plan)
            del yt
            torch.cuda.empty_cache()
            bytes_, flops = model(B, n, n_out, taps, fft_size, parts, nf)
            t_hbm = bytes_ / (hbm_gbs * 1e9) * 1e3
            t_fp32 = flops / (fp32 * 1e12) * 1e3
            rec = dict(taps=taps, filters=mode, batch=B, n=n, n_out=n_out, fft_size=fft_size, partitions=parts,
                       ms=round(ms, 3), gsamples_per_s=round(B * n_out / ms / 1e6, 2),
                       model_bytes=bytes_, model_flops=flops, bound="HBM" if t_hbm >= t_fp32 else "FP32",
                       share_of_bound=round(max(t_hbm, t_fp32) / ms, 3),
                       torch_fft_ms=round(ms_torch, 3), speedup_vs_torch_fft=round(ms_torch / ms, 2),
                       worst_err_over_bound_lib=err_lib, worst_err_over_bound_torch=err_torch, bound_C=FIR_C,
                       torch_within_bound=bool(err_torch < FIR_C), lib_within_bound=bool(err_lib < FIR_C))
            print(json.dumps(rec), flush=True)
            if out:
                out.write(json.dumps(rec) + "\n")
            del h
    if out:
        out.close()


if __name__ == "__main__":
    main()
