#!/usr/bin/env python
"""bench.py -- the headline benchmark of BASELINE.json, on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): "STFT+ISTFT Msamples/s at nfft=2048 hop=512".  One step = one pass
of the hot path over one batch of synthetic input = configs[1]+configs[2]:
    batched STFT (framing + Hann + real FFT -> complex half spectra [B][934][1025] in HBM)
  + batched ISTFT (half spectra -> inverse FFT -> synthesis window -> overlap-add ->
    window-sum normalisation -> [B][480000])
for B = 1024 signals x 10 s @ 48 kHz per GPU, valid frames only (934 per signal).

  value   whole-job Msamples/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e     the same metric through the C-ABI with HOST (pinned) buffers: signals H2D ->
          STFT -> ISTFT -> reconstructed signals D2H inside the timed region (spectra stay
          in HBM between the two calls, as a user of the batched API would keep them)
  roofline   the dominant kernel's algorithmic HBM bytes / its CUDA-event duration vs the
          measured copy bandwidth in MEASURED_PEAKS.json; roofline_fp32 gives the
          north-star's other bound (5 N log2 N flops vs a measured FFMA peak)
  cpu_baseline  the reference's own CPU path (oracle/_ref, else the oracle port) on this
          box's host cores, bounded sample
Multi-GPU: signals are sharded by signal across ranks, no collective on the data path
(weak scaling: every rank owns B signals).  --impl reference times the CPU reference.

--dump-outputs DIR writes what the last timed step returned on rank 0, for comparing two builds
output for output (the inputs are seeded, so the same arguments give the same inputs): a fixed,
seeded sample of DUMP_SIGNALS signals, as DIR/spectra.npy (float32 [signals][934][1025][2], real
and imaginary parts) and DIR/reconstruction.npy (float32 [signals][480000]), 57.5 MB in all.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NFFT, HOP, N_SAMPLES, BATCH = 2048, 512, 480_000, 1024
FRAMES = 1 + (N_SAMPLES - NFFT) // HOP          # 934 (valid-only convention)
BINS = NFFT // 2 + 1
METRIC = "STFT+ISTFT Msamples/s at nfft=2048 hop=512"
UNIT = "Msamples/s"
WORKLOAD = ("configs[1]+[2]: batched STFT -> complex half spectra -> batched ISTFT (OLA, window-sum normalised), "
            "1024 synthetic mono signals x 10 s @48 kHz per GPU, nfft=2048 hop=512 Hann, 934 valid frames/signal")
DUMP_SIGNALS, DUMP_SEED = 6, 0      # 6 x (7.66 MB spectra + 1.92 MB signal) stays under 64 MB


def dump_outputs(out_dir, spec, y):
    """The timed path's outputs for a fixed, seeded sample of signals, as float32 .npy files under out_dir."""
    import numpy as np
    import torch
    B = spec.shape[0]
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(B, min(B, DUMP_SIGNALS), replace=False))
    idx = torch.as_tensor(rows, device=spec.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "spectra.npy"), torch.view_as_real(spec.index_select(0, idx)).cpu().numpy())
    np.save(os.path.join(out_dir, "reconstruction.npy"), y.index_select(0, idx).cpu().numpy())


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel_substr):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the named kernel, read from the NEWEST ncu summary under
    profiles/ (r*_ncu_full_*.csv: metric rows, one column per kernel) that has a column for it.  Returns (bytes, file)."""
    import csv
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full_*.csv")), reverse=True):
        try:
            rows = [r for r in csv.reader(open(path)) if r and not r[0].startswith("#")]
            hdr = rows[0]
            cols = [i for i, h in enumerate(hdr) if kernel_substr in h]
            if not cols:
                continue
            vals = {r[0]: (r[1], r[cols[0]]) for r in rows[1:] if len(r) > cols[0]}
            scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
            rd, wr = vals["dram__bytes_read.sum"], vals["dram__bytes_write.sum"]
            return float(rd[1]) * scale[rd[0]] + float(wr[1]) * scale[wr[0]], os.path.relpath(path, ROOT)
        except Exception:
            continue
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [l.split(", ") for ts, l in self.lines if t0 - 0.05 <= ts <= t1 + 0.15] or [l.split(", ") for _, l in self.lines]
        sm, mx, reasons, power = [], [], set(), []
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference(threads, target_seconds, signals=None):
    """Time the reference's CPU implementation of the step (process -> reconstruct -> normalise,
    tools/dump_stft_roundtrip.c:44-54) on a bounded sample: `signals` signals of the headline shape if given, else as
    many as fit target_seconds.  Returns (run() -> seconds, signals per run, kind, pilot seconds per signal and thread)."""
    import numpy as np
    from oracle.oracle import Oracle, Reference
    if Reference.available():
        impl, kind = Reference(), "reference"
    else:
        impl, kind = Oracle(), "port"
    rng = np.random.default_rng(1234)
    pilot = rng.uniform(-1, 1, (threads, N_SAMPLES)).astype(np.float32)
    t = time.perf_counter()
    impl.batch_roundtrip(pilot, NFFT, HOP, "hann", threads=threads, want_output=False)
    dt = time.perf_counter() - t
    if signals is None:
        per_thread = max(1, min(64, int(target_seconds / max(dt, 1e-3))))
        B = threads * per_thread
    else:
        B = int(signals)
    reps = -(-B // threads)
    x = np.tile(pilot, (reps, 1))[:B] if B != threads else pilot

    def run():
        t0 = time.perf_counter()
        impl.batch_roundtrip(x, NFFT, HOP, "hann", threads=threads, want_output=False)
        return time.perf_counter() - t0
    run.pilot_seconds = dt
    return run, B, kind


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the step on this box's host cores (oracle/_ref =
    the unmodified reference compiled by oracle/Makefile; the oracle port if that is absent).  One step = the SAME
    workload as the GPU arm's step (1024 signals) whenever K + W such steps fit in about four minutes on this host;
    otherwise a bounded sample of it (the metric is per-sample throughput on identical signal shapes)."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    probe, _, _ = cpu_reference(cores, target_seconds=1.0)
    est_full = probe.pilot_seconds * BATCH / cores                        # seconds per step of 1024 signals
    nsteps = max(1, args.steps + args.warmup)
    if est_full * nsteps <= 240.0:
        run, B, kind = cpu_reference(cores, 0.0, signals=BATCH)
        note = "same workload as the GPU arm's step"
    else:
        run, B, kind = cpu_reference(cores, target_seconds=max(2.0, 240.0 / nsteps))
        note = (f"bounded sample: {BATCH} signals per step would take ~{est_full * nsteps:.0f} s for {nsteps} steps on {cores} cores; "
                "throughput is per sample on identical signal shapes")
    for _ in range(args.warmup):
        run()
    times = [run() for _ in range(args.steps)]
    total = sum(times)
    val = B * N_SAMPLES * args.steps / total / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "nfft": NFFT, "hop": HOP, "window": "hann", "signals_per_gpu": BATCH,
                   "signal_samples": N_SAMPLES, "frames_per_signal": FRAMES, "bins": BINS,
                   "sample_signals_per_step": B, "sample_note": note,
                   "note": "CPU reference path on the box's host cores, one vv_dsp_stft handle per thread"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{B} signals x {N_SAMPLES} samples per step, STFT->ISTFT->normalise loop of tools/dump_stft_roundtrip.c:44-54"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def stream_config4(lib, n_gpus, seconds=3600, steps=10, warmup=3):
    """BASELINE config 4: ONE 1-hour 48 kHz stream, nfft=4096 hop=1024 Hann, sharded by frame range over n_gpus GPUs
    by the C library's multi-device handle (vv_dsp_stft_stream_*: peer-to-peer sample halos, one CUDA graph per
    device and step).  Timed on the devices (CUDA events on every device's stream, slowest device); the sharded
    result is compared bit for bit with the one-device result of the same stream."""
    import numpy as np
    from vv_dsp_b200 import StftStream
    nfft, hop = 4096, 1024
    n = 48000 * seconds
    frames, bins = 1 + (n - nfft) // hop, nfft // 2 + 1
    rng = np.random.default_rng(4)
    x = np.tile(rng.uniform(-1, 1, 48000 * 30).astype(np.float32), seconds // 30 + 1)[:n]
    out = {"workload": f"configs[3]: single {seconds}-s 48 kHz stream ({n} samples, {frames} frames), nfft={nfft} hop={hop} Hann, "
                       f"STFT -> complex half spectra -> normalised ISTFT, frame-range sharded over {n_gpus} GPU(s), "
                       f"(nfft-hop)-sample halos peer to peer",
           "n_gpus": n_gpus, "steps": steps, "halo_bytes_per_boundary_and_direction": (nfft - hop) * 4}
    with StftStream(nfft, hop, n, [0], lib=lib) as s1:
        s1.upload(x)
        ms1 = s1.time_roundtrip(warmup, steps)
        y1 = s1.download()
    lo, hi = nfft, n - nfft
    out["roundtrip_rel_l2"] = float(np.linalg.norm((y1[lo:hi] - x[lo:hi]).astype(np.float64)) / np.linalg.norm(x[lo:hi].astype(np.float64)))
    hbm_peak, _ = measured_peaks()
    gbytes = 2 * (4 * n + 8 * frames * bins) / 1e9
    out["ms_per_step_1gpu"] = ms1
    out["hbm_frac_1gpu"] = gbytes / (ms1 * 1e-3) / hbm_peak
    ms = ms1
    if n_gpus > 1:
        with StftStream(nfft, hop, n, list(range(n_gpus)), lib=lib) as s:
            s.upload(x)
            ms = s.time_roundtrip(warmup, steps)
            out["bit_identical_to_unsharded"] = bool(np.array_equal(s.download(), y1))
            out["devices"] = sorted({s.shard(d).device for d in range(n_gpus)})
        out["strong_scaling_efficiency"] = ms1 / (n_gpus * ms)
    out["ms_per_step"] = ms
    out["value"] = n / (ms * 1e-3) / 1e6
    out["unit"] = UNIT
    out["algorithmic_GB_per_step"] = gbytes
    out["hbm_frac_aggregate"] = gbytes / (ms * 1e-3) / (hbm_peak * n_gpus)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="signals per GPU (default: the BASELINE shape)")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stream", action="store_true", help="skip the config-4 single-stream leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's spectra and reconstructed signals (seeded sample) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the launcher set it (the driver reads communicator ranks from it); NCCL's own log
        # lines go to stderr so that stdout carries the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    # CPU-side rendezvous for the phases in which ONE rank drives every GPU (the config-4 stream leg): the other
    # ranks must wait on the host, not inside an NCCL kernel on a GPU that rank 0 is using
    cpu_group = dist.new_group(backend="gloo") if world > 1 else None

    from vv_dsp_b200 import Stft, default_library
    lib = default_library()
    B = args.batch
    stream = torch.cuda.Stream(device=dev)      # explicit non-default stream: kernels AND events live on it
    torch.cuda.set_stream(stream)
    h = Stft(NFFT, HOP, "hann")
    h.set_stream(stream.cuda_stream)

    # synthetic inputs of the named shape, i.i.d. uniform(-1,1), resident in HBM
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.rand((B, N_SAMPLES), device=dev, generator=g) * 2 - 1
    spec = torch.empty((B, FRAMES, BINS), device=dev, dtype=torch.complex64)
    y = torch.empty((B, N_SAMPLES), device=dev, dtype=torch.float32)

    def step():
        h.batch_forward(x, "complex", "valid", out=spec)
        h.batch_inverse(spec, N_SAMPLES, True, out=y)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step()
    barrier()

    # ---- timed region: exactly K steps, CUDA events on the launching stream
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    launches0 = lib.kernel_launches()
    barrier()
    t0 = time.perf_counter()
    start = torch.cuda.Event(enable_timing=True); end = torch.cuda.Event(enable_timing=True)
    start.record(stream)
    for k in range(args.steps):
        ev[k][0].record(stream)
        h.batch_forward(x, "complex", "valid", out=spec)
        ev[k][1].record(stream)
        h.batch_inverse(spec, N_SAMPLES, True, out=y)
        ev[k][2].record(stream)
    end.record(stream)
    barrier()
    t1 = time.perf_counter()
    launches = lib.kernel_launches() - launches0
    clocks = sampler.stop(t0, t1)
    ms_total = start.elapsed_time(end)
    fwd_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / args.steps
    inv_ms = sum(e[1].elapsed_time(e[2]) for e in ev) / args.steps
    tmax = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total_max = float(tmax.item())
    ms_per_step = ms_total_max / args.steps
    value = world * B * N_SAMPLES / (ms_per_step * 1e-3) / 1e6

    # ---- sanity inside the bench: the timed outputs are the real thing (round trip on the interior)
    err = float(torch.linalg.vector_norm((y - x)[:, NFFT:-NFFT].double()) / torch.linalg.vector_norm(x[:, NFFT:-NFFT].double()))
    if args.dump_outputs and rank == 0:             # before the legs below reuse spec
        dump_outputs(args.dump_outputs, spec, y)

    # ---- power-spectrum variant (configs[1] as literally stated), device-resident, for the record
    pw = torch.empty((B, FRAMES, BINS), device=dev, dtype=torch.float32)
    for _ in range(2):
        h.batch_forward(x, "power", "valid", out=pw)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(5):
        h.batch_forward(x, "power", "valid", out=pw)
    e1.record(stream)
    torch.cuda.synchronize()
    pow_ms = e0.elapsed_time(e1) / 5
    del pw

    # ---- end to end through the C-ABI with HOST buffers (pinned), copies inside the timed region
    e2e_steps = args.e2e_steps or max(2, min(args.steps, 5))
    xh = torch.empty((B, N_SAMPLES), dtype=torch.float32).pin_memory()
    yh = torch.empty((B, N_SAMPLES), dtype=torch.float32).pin_memory()
    xh.copy_(x)
    xh_np, yh_np = xh.numpy(), yh.numpy()

    # stream-ordered mode (vv_dsp_stft_set_async): both calls only enqueue; the library chains the synthesis
    # of each chunk of signals to the analysis chunk that produced its spectra, so the H2D of later chunks
    # overlaps the D2H of earlier ones.  synchronize() returns when yh is complete.
    h.set_async(True)

    def e2e_step():
        h.batch_forward(xh_np, "complex", "valid", out=spec)      # H2D inside, spectra stay in HBM
        h.batch_inverse(spec, N_SAMPLES, True, out=yh_np)          # D2H inside
        h.synchronize()

    e2e_step()
    barrier()
    te = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - te) / e2e_steps
    te_t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te_t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * N_SAMPLES / float(te_t.item()) / 1e6
    sel = [0, 1, B // 2, B - 1]
    e2e_err = float(np.linalg.norm((yh_np[sel] - xh_np[sel])[:, NFFT:-NFFT]) / np.linalg.norm(xh_np[sel][:, NFFT:-NFFT]))

    # ---- the same step fed with 16-bit PCM as it sits in a WAV file (vv_dsp_stft_batch_forward_pcm): the upload is half
    # the bytes, the samples are decoded on the device next to the STFT; the output is still float32 in host memory
    x16 = torch.empty((B, N_SAMPLES), dtype=torch.int16).pin_memory()
    x16.copy_((x * 32767.0).round().to(torch.int16))
    x16_np = x16.numpy()

    def e2e_pcm_step():
        h.batch_forward_pcm(x16_np, 16, "complex", "valid", out=spec)
        h.batch_inverse(spec, N_SAMPLES, True, out=yh_np)
        h.synchronize()

    e2e_pcm_step()
    barrier()
    tp = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_pcm_step()
    torch.cuda.synchronize()
    pcm_s = (time.perf_counter() - tp) / e2e_steps
    tp_t = torch.tensor([pcm_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tp_t, op=dist.ReduceOp.MAX)
    e2e_pcm_value = world * B * N_SAMPLES / float(tp_t.item()) / 1e6
    ref16 = x16_np[sel].astype(np.float32) / 32768.0
    e2e_pcm_err = float(np.linalg.norm((yh_np[sel] - ref16)[:, NFFT:-NFFT]) / np.linalg.norm(ref16[:, NFFT:-NFFT]))
    h.set_async(False)
    del x16, x16_np

    fp32_scalar = fp32_packed = None
    if rank == 0:
        try:
            fp32_scalar, fp32_packed = lib.fp32_peak(False), lib.fp32_peak(True)
        except Exception:
            pass
    # ---- config 4: one long stream over all GPUs, driven by rank 0 through the C library's multi-device handle
    stream_line = None
    if not args.no_stream:
        del xh, yh, xh_np, yh_np
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=cpu_group)
        if rank == 0:
            try:
                stream_line = stream_config4(lib, world)
            except Exception as exc:                       # the headline line must still be printed
                stream_line = {"error": f"{type(exc).__name__}: {exc}"}
        if world > 1:
            dist.barrier(group=cpu_group)
    if rank == 0:
        hbm_peak, peak_src = measured_peaks()
        bytes_fwd = B * (4 * N_SAMPLES + 8 * FRAMES * BINS)       # SURVEY.md 8(d): read samples once + write half spectra once
        bytes_inv = B * (8 * FRAMES * BINS + 4 * N_SAMPLES)
        dom = ("istft_ws_kernel", inv_ms, bytes_inv) if inv_ms >= fwd_ms else ("stft_march_kernel", fwd_ms, bytes_fwd)
        # measured DRAM traffic of that kernel at this shape: the newest ncu --set full summary committed under profiles/
        traffic, traffic_file = ncu_traffic(dom[0]) if B == BATCH else (None, None)
        achieved = dom[2] / (dom[1] * 1e-3) / 1e9
        flops_dir = B * FRAMES * 5 * NFFT * 11                     # 5 N log2 N per frame per direction
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "nfft": NFFT, "hop": HOP, "window": "hann", "signals_per_gpu": B,
                       "signal_samples": N_SAMPLES, "frames_per_signal": FRAMES, "bins": BINS,
                       "l2": "inputs larger than L2 (1.97 GB signals, 7.84 GB spectra per GPU vs 126 MB L2)",
                       "parallelism": f"shard-by-signal x{world}, no collective"},
            "roofline": {"bound": "hbm", "kernel": dom[0], "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak,
                         "traffic": traffic, "traffic_source": traffic_file, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": dom[2], "ms_per_launch": dom[1]},
            "kernels": {"stft_forward_ms": fwd_ms, "stft_inverse_ms": inv_ms, "stft_forward_power_ms": pow_ms,
                        "stft_forward_GBps": bytes_fwd / (fwd_ms * 1e-3) / 1e9, "stft_inverse_GBps": bytes_inv / (inv_ms * 1e-3) / 1e9,
                        "stft_power_Gsamples_per_s": B * N_SAMPLES / (pow_ms * 1e-3) / 1e9,
                        "step_hbm_frac": (bytes_fwd + bytes_inv) / ((fwd_ms + inv_ms) * 1e-3) / 1e9 / hbm_peak},
            "roofline_fp32": {"flops_per_direction": flops_dir, "convention": "5*N*log2(N) per frame (north-star)",
                              "achieved_tflops_forward": flops_dir / (fwd_ms * 1e-3) / 1e12,
                              "achieved_tflops_inverse": flops_dir / (inv_ms * 1e-3) / 1e12,
                              "nominal_peak_tflops": 74.5, "measured_peak_tflops_ffma": fp32_scalar,
                              "measured_peak_tflops_ffma2": fp32_packed,
                              "roofline_ms_power_variant": max(flops_dir / ((fp32_scalar or 74.5) * 1e12), B * (4 * N_SAMPLES + 4 * FRAMES * BINS) / (hbm_peak * 1e9)) * 1e3,
                              "frac_power_variant": max(flops_dir / ((fp32_scalar or 74.5) * 1e12), B * (4 * N_SAMPLES + 4 * FRAMES * BINS) / (hbm_peak * 1e9)) * 1e3 / pow_ms},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * N_SAMPLES * 4, "d2h_bytes_per_step": B * N_SAMPLES * 4,
                    "ms_per_step": float(te_t.item()) * 1e3, "steps": e2e_steps, "roundtrip_rel_l2": e2e_err,
                    "api": "vv_dsp_stft_set_async(1); vv_dsp_stft_batch_forward(HOST signals -> DEVICE spectra); vv_dsp_stft_batch_inverse(DEVICE spectra -> HOST signals); vv_dsp_stft_synchronize()"},
            "e2e_pcm16": {"value": e2e_pcm_value, "unit": UNIT, "h2d_bytes_per_step": B * N_SAMPLES * 2, "d2h_bytes_per_step": B * N_SAMPLES * 4,
                          "ms_per_step": float(tp_t.item()) * 1e3, "steps": e2e_steps, "roundtrip_rel_l2_vs_decoded_samples": e2e_pcm_err,
                          "api": "the same with vv_dsp_stft_batch_forward_pcm(HOST 16-bit PCM as in a WAV data chunk): decoded on the device, output still float32 on the host"},
            "gpu_launches": int(launches), "clocks": clocks, "roundtrip_rel_l2": err,
        }
        if stream_line is not None:
            line["stream_config4"] = stream_line
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            run, Bc, kind = cpu_reference(cores, target_seconds=12.0)
            dt = run()
            line["cpu_baseline"] = {"value": Bc * N_SAMPLES / dt / 1e6, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": f"{Bc} signals x {N_SAMPLES} samples, STFT->ISTFT->normalise loop of "
                                              f"tools/dump_stft_roundtrip.c:44-54, one handle per thread, {dt:.1f} s"}
            run1, B1, _ = cpu_reference(1, target_seconds=4.0)        # BASELINE.md section 3: also on ONE thread
            dt1 = run1()
            line["cpu_baseline_1thread"] = {"value": B1 * N_SAMPLES / dt1 / 1e6, "unit": UNIT, "cores": 1, "kind": kind,
                                            "sample": f"{B1} signals x {N_SAMPLES} samples, same loop, {dt1:.1f} s"}
            # SURVEY.md section 8(d): also the forward + re^2 + im^2 loop (configs[1] as literally stated), all cores, a few seconds
            try:
                import numpy as np
                from oracle.oracle import Oracle, Reference
                impl = Reference() if Reference.available() else Oracle()
                xp = np.random.default_rng(4321).uniform(-1, 1, (cores * 32, N_SAMPLES)).astype(np.float32)
                tp0 = time.perf_counter()
                impl.batch_power(xp, NFFT, HOP, "hann", threads=cores, want_output=False)
                dtp = time.perf_counter() - tp0
                line["cpu_baseline_power"] = {"value": xp.shape[0] * N_SAMPLES / dtp / 1e6, "unit": UNIT, "cores": cores, "kind": kind,
                                              "sample": f"{xp.shape[0]} signals x {N_SAMPLES} samples, vv_dsp_stft_process + re^2 + im^2 per frame, {dtp:.1f} s",
                                              "gpu_value": B * N_SAMPLES / (pow_ms * 1e-3) / 1e6}
            except Exception as exc:                        # a reported extra, never fatal
                line["cpu_baseline_power"] = {"error": f"{type(exc).__name__}: {exc}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
