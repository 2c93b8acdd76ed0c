"""Cost of the float64 sections (FORM 2) on the synthetic corpus of bench.py (4620 utterances, U(32000, 64000)
samples at 16 kHz, seed 1) through a bank float32 cannot hold: 16 kHz, 128 channels, LOW_FREQ = 20, width 1
(its last group of 32 channels runs FORM 2).  Compares the resident window-store pass (whole utterances, as
bench.py runs it) with the same bank forced to float32 (F2CNN_B200_ALLOW_IMPRECISE=1), and reports:
  * pass time and fused-kernel time of each (device events, median of --reps passes);
  * the time of the FORM 2 launch alone and of the float32 launch next to it (torch.profiler, separate run);
  * the FORM 2 launch's DFMA rate as a share of the DFMA peak tools/fma_peak measured (--peak FILE: its
    output), counting the DFMAs of the cascade (the magnitude, low-pass and stores are float32).
Usage: python tools/float64_sections_bench.py [--peak fma_peak.log] [--reps 10]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from f2cnn_b200 import engine, synth
from f2cnn_b200.gammatone import filters

STEP, DOTS, CUTOFF = 160, 11, 50


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--peak", help="output of tools/fma_peak (JSON lines); its dfma_reg sustained rate is the peak")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--utts", type=int, default=4620)
    args = ap.parse_args()
    co = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 20), 1.0)
    C = co.shape[0]
    lengths = synth.corpus_lengths(args.utts, 32000, 64000, seed=1)
    flat, offsets = synth.corpus_waves_i16(lengths, seed=1)
    wave = torch.from_numpy(flat).cuda()
    f64 = engine.Plan(co, float64_sections=True)
    os.environ["F2CNN_B200_ALLOW_IMPRECISE"] = "1"
    f32 = engine.Plan(co, float64_sections=False)
    del os.environ["F2CNN_B200_ALLOW_IMPRECISE"]
    assert f64.float64_groups == (3,) and f32.float64_groups == ()
    res = {"device": device_info(), "bank": "16 kHz, 128 ch, LOW_FREQ 20, width 1", "utterances": int(args.utts),
           "samples": int(offsets[-1]), "float64_groups": list(f64.float64_groups),
           "predicted_float32_error_per_group": [round(float(v), 3) for v in engine.bank_check_groups(co)]}
    runs = {}
    for name, plan in (("float64_sections", f64), ("forced_float32", f32)):
        b = plan.batch(lengths, step=STEP, target_items=1)
        offs, rows = b.grid_windows(DOTS)
        win = torch.empty((rows, DOTS, C), dtype=torch.float32, device="cuda")
        runs[name] = (b, offs, win)

    def step(name, ev=None):
        b, offs, win = runs[name]
        b.run(wave, lpf=True, cutoff=CUTOFF, windows=(offs, DOTS, win), fused_events=ev)

    for name in runs:
        for _ in range(3):
            step(name)
    torch.cuda.synchronize()
    times = {n: {"pass_ms": [], "fused_ms": []} for n in runs}
    for _ in range(args.reps):          # alternating, so that both see the same clocks
        for name in runs:
            a, b_, f0, f1 = (engine.DeviceEvent() for _ in range(4))
            a.record()
            step(name, (f0, f1))
            b_.record()
            b_.synchronize()
            times[name]["pass_ms"].append(a.elapsed_ms(b_))
            times[name]["fused_ms"].append(f0.elapsed_ms(f1))
    for name, t in times.items():
        res[name] = {k: round(float(np.median(v)), 3) for k, v in t.items()}
        res[name]["pass_ms_min_max"] = [round(min(t["pass_ms"]), 3), round(max(t["pass_ms"]), 3)]
    w_imag, w_edge, _ = f64.get_warmup()
    # FORM 2 DFMAs per channel: per sample 2 x 12 (real and imaginary sections) + 4 (injection e*G) + 2 (g4);
    # warm-up of the imaginary path 16 per sample over w_imag; edge pass 12 per sample over the last w_edge (tiles)
    n = lengths.astype(np.float64)
    edge = np.minimum(n, np.ceil(w_edge / 256.0) * 256.0 + 256.0)
    dfma = 32.0 * float(np.sum(30.0 * n + 16.0 * w_imag + 12.0 * edge))
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            step("float64_sections")
            step("forced_float32")
        torch.cuda.synchronize()
    ktime = {}
    for e in prof.key_averages():
        for tag in ("fused_kernel<true", "fused_kernel<false", "ring_cluster", "edge"):   # <true: FORM 2 (float64)
            if tag in e.key:
                ktime.setdefault(tag, []).append((e.key[:90], e.count, e.device_time_total / max(e.count, 1) / 1e3))
    f64_ms = sum(t for k, c, t in ktime.get("fused_kernel<true", []))
    res["kernels_ms_per_call"] = {k: [(name, c, round(t, 3)) for name, c, t in v] for k, v in ktime.items()}
    res["form2_launch_ms"] = round(f64_ms, 3)
    res["form2_dfma_per_pass"] = dfma
    if f64_ms > 0:
        res["form2_dfma_tflops"] = round(2.0 * dfma / (f64_ms * 1e-3) / 1e12, 3)
    if args.peak:
        for line in open(args.peak):
            line = line.strip()
            if line.startswith("{") and '"dfma_reg"' in line:
                peak = json.loads(line)["sustained_tflops"]
                res["dfma_peak_tflops"] = peak
                if f64_ms > 0:
                    res["form2_share_of_dfma_peak"] = round(res["form2_dfma_tflops"] / peak, 3)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
