"""Batched IIR filtering by second-order sections (vv_dsp_sos_*) on device-resident signals, against torchaudio and scipy.

    python benchmarks/iir_bench.py [--batch 1024] [--seconds 10] [--iters 5] [--rows 2] [--scipy-signals 2]
                                   [--torch-rows 16] [--segments 18,20,22] [--out FILE.jsonl]

Workload: `batch` signals of `seconds` at 48 kHz through the 20 Hz high-pass (1 section), the 50 Hz - 8 kHz band-pass
(4 sections) and a 16-section butter(32) low-pass; sosfiltfilt of the band-pass; and 8 signals of one hour through the
band-pass, which takes the segmented path (launches A, B and C), once per segment length in --segments (log2 samples,
set through VVB_IIR_SEGMENT at creation; 20 is the library's default).  Timed with CUDA events after a warm-up call;
every input is at least 1.9 GB, above the L2.  One JSON line per row:
  - ms per call and Gsamples/s;
  - the model's bytes (8 per sample for one pass over a row, 12 on the segmented path where launch A reads the input once
    more, 16 for filtfilt: the forward pass writes and the backward pass reads a scratch row) and flops (22 per sample and
    section per pass: 9 for each of the two runs of the recurrence and 4 for the scan, 8 levels of 4 FMA shared by 16
    samples), and the share of the larger of the HBM bound (MEASURED_PEAKS.json if present, else the data sheet,
    labelled) and the FP32 bound (vv_dsp_b200_fp32_peak, scalar FFMA);
  - the worst error of sampled rows against float64 scipy, over the bound of tests/test_iir.py;
  - baselines: torchaudio.functional.lfilter section by section (clamp=False) on the same GPU, timed on --torch-rows rows
    and scaled to the batch (labelled), and scipy.signal.sosfilt / sosfiltfilt on one host core over a few signals,
    scaled.
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

FS = 48000
FLOPS_PER_SAMPLE_SECTION = 22


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


def err_over_bound(y, y64, y32):
    """max over rows of max|y - y64| / (4 e32 + 16 2^-24 max|y64|), the bound of tests/test_iir.py"""
    worst = 0.0
    for r in range(len(y64)):
        err = float(np.abs(y[r].astype(np.float64) - y64[r]).max())
        bound = 4.0 * float(np.abs(y32[r].astype(np.float64) - y64[r]).max()) + 16.0 * 2.0 ** -24 * float(np.abs(y64[r]).max())
        worst = max(worst, err / bound if bound > 0 else (0.0 if err == 0 else float("inf")))
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--rows", type=int, default=2, help="sampled rows checked against float64 truth")
    ap.add_argument("--scipy-signals", type=int, default=2, help="signals filtered by scipy on one host core")
    ap.add_argument("--torch-rows", type=int, default=16, help="rows torchaudio's lfilter is timed on, scaled to the batch")
    ap.add_argument("--segments", default="18,20,22", help="log2 segment lengths of the one-hour row")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("iir_bench.py needs a CUDA device: nothing is measured without one")
    from scipy.signal import sosfilt, sosfiltfilt
    from fir_bench import card, hbm_peak
    from test_iir import filtfilt32, sos32
    from vv_dsp_b200 import SosFilter, default_library
    try:
        import torchaudio.functional as taf
    except Exception:                                  # noqa: BLE001 -- the baseline is optional
        taf = None

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
              fp32_source="vv_dsp_b200_fp32_peak (scalar FFMA)", torchaudio=taf is not None))
    g = torch.Generator(device="cuda").manual_seed(1)
    n10 = int(round(FS * args.seconds))
    hour = FS * 3600
    rows = [("highpass_20", "filter", args.batch, n10, None), ("bandpass_50_8k", "filter", args.batch, n10, None),
            ("butter32", "filter", args.batch, n10, None), ("bandpass_50_8k", "filtfilt", args.batch, n10, None)]
    rows += [("bandpass_50_8k", "filter", 8, hour, int(s)) for s in args.segments.split(",")]
    for fname, op, B, n, log2_seg in rows:
        s32 = sos32(fname)
        S = len(s32)
        x = torch.rand((B, n), device="cuda", generator=g) * 2 - 1
        y = torch.empty_like(x)
        if log2_seg is not None:
            os.environ["VVB_IIR_SEGMENT"] = str(1 << log2_seg)
        try:
            f = SosFilter(s32, lib=lib)
        finally:
            os.environ.pop("VVB_IIR_SEGMENT", None)
        with f:
            call = (lambda: f.filter(x, out=y)) if op == "filter" else (lambda: f.filtfilt(x, out=y))
            ms = timed(call, args.iters if n <= 10 * n10 else 2)
            torch.cuda.synchronize()
            seg = f.segment_length
            pick = np.linspace(0, B - 1, min(args.rows, B)).astype(int)
            if n > 10 * n10:
                pick = pick[:1]
            xs, ys = x[pick].cpu().numpy(), y[pick].cpu().numpy()
        s64 = s32.astype(np.float64)
        if op == "filter":
            y64 = sosfilt(s64, xs.astype(np.float64), axis=-1)
            err = err_over_bound(ys, y64, sosfilt(s32, xs, axis=-1))
        else:
            y64 = sosfiltfilt(s64, xs.astype(np.float64), axis=-1)
            err = err_over_bound(ys, y64, filtfilt32(s32, xs, "odd", None))
        samples = B * n
        segs = -(-n // seg)
        passes = 1 if op == "filter" else 2
        per_sample = (8 if op == "filter" else 16) + (4 * passes * (segs - 1) / segs if segs > 1 else 0)
        bytes_ = int(samples * per_sample)
        flops = FLOPS_PER_SAMPLE_SECTION * S * samples * passes * (1 + ((segs - 1) / segs if segs > 1 else 0))
        t_hbm = bytes_ / (hbm_gbs * 1e9) * 1e3
        t_fp32 = flops / (fp32 * 1e12) * 1e3
        rec = dict(filter=fname, op=op, sections=S, batch=B, n=n, segment_length=seg, segments_per_row=segs,
                   input_gb=round(4 * samples / 1e9, 3), ms=round(ms, 3), gsamples_per_s=round(samples / ms / 1e6, 2),
                   model_bytes=bytes_, model_flops=int(flops), hbm_bound_ms=round(t_hbm, 3), fp32_bound_ms=round(t_fp32, 3),
                   bound="HBM" if t_hbm >= t_fp32 else "FP32", share_of_bound=round(max(t_hbm, t_fp32) / ms, 3),
                   worst_err_over_bound_lib=err, lib_within_bound=bool(err <= 1.0))
        if taf is not None and op == "filter" and log2_seg in (None, 20):
            k = max(1, min(args.torch_rows, B))
            xk = x[:k].contiguous()
            coeffs = [(torch.tensor(s[3:], device="cuda"), torch.tensor(s[:3], device="cuda")) for s in s32]

            def ta():
                v = xk
                for a, b in coeffs:
                    v = taf.lfilter(v, a, b, clamp=False)
                return v
            ms_t = timed(ta, 1) * B / k
            rec.update(torchaudio_baseline=f"torchaudio.functional.lfilter per section, clamp=False, timed on {k} rows, "
                                           f"scaled to {B}",
                       torchaudio_ms_scaled=round(ms_t, 1), speedup_vs_torchaudio=round(ms_t / ms, 1))
        k = max(1, min(args.scipy_signals, B if n <= 10 * n10 else 1))
        xh = x[:k].cpu().numpy()
        t0 = time.perf_counter()
        if op == "filter":
            sosfilt(s32, xh, axis=-1)
        else:
            sosfiltfilt(s32, xh, axis=-1)
        ms_s = (time.perf_counter() - t0) * 1e3 * B / k
        rec.update(scipy_one_core_float32_ms_scaled=round(ms_s, 1), scipy_signals_timed=k,
                   speedup_vs_scipy_one_core=round(ms_s / ms, 1))
        emit(rec)
        del x, y
        torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
