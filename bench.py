#!/usr/bin/env python
"""bench.py -- channel-samples/s of the F2CNN feature-extraction hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm (oracle port, all host threads)
    python bench.py ... --dump-outputs DIR                   # also write a seeded sample of the output

Workload (BASELINE.json configs[1], SURVEY.md section 8d config 2): a synthetic
TIMIT-TRAIN-sized corpus -- 4620 utterances, lengths U(32000, 64000) samples at 16 kHz,
int16 white noise -- through the 128-channel ERB gammatone filterbank, the ENV1 envelope
with the 50 Hz low-pass and the window gather on the full label grid, producing the
(N, 11, 128) float32 input tensor.  One step = one pass of that path over the whole corpus.
Multi-GPU (configs[2]): the SAME corpus, utterances dealt to the ranks by length-sorted
round-robin (engine.shard_utterances), no collective on the data path, rows of all ranks placed
into ONE shared host tensor (strong scaling); value = channel-samples of the corpus /
max-over-ranks time.

One JSON line on stdout (rank 0).  `value`: inputs resident in HBM, device-timed.  `e2e`: the
same metric through the public call api.features_to_windows with HOST buffers -- pinned int16
waves in, the float32 input tensor in host memory out, wall clock around the call.  `roofline`: the fused kernel against
the FP32 FMA peak (80 FLOP per channel-sample, SURVEY.md 8d), timed with CUDA events on its
own stream inside the timed region.  `cpu_baseline`: the float64 oracle port (the reference's
algorithm restated in C, reference Python cannot travel to the GPU box) on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS, C, LOW, CUTOFF, RADIUS, STEP = 16000, 128, 100, 50, 5, 160
N_UTTS, LEN_LO, LEN_HI = 4620, 32000, 64000
FLOP_PER_CS = 80.0  # 40 FP32 FMA per channel-sample: filterbank + envelope + LPF (SURVEY.md 8d)
TRAFFIC_1GPU = 11.520e9  # bytes per fused_kernel launch (window-store mode): 4.08 GB read + 7.44 GB written (ncu, DESIGN.md section 5)
KERNELS_PER_STEP = 2  # ring_cluster_kernel (whole pre-pass of the corpus sizes), fused_kernel (stores the windows)
DUMP_ROWS = 8192  # --dump-outputs: 8192 x 11 x 128 float32 = 46 MB of the 7.5 GB windows tensor


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--utts", type=int, default=N_UTTS, help="utterances of the corpus (default: the config's 4620)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the side configs (single utterance, 600 s stream, evalnoise)")
    ap.add_argument("--no-verify", action="store_true", help="N > 1: skip the bit-for-bit check against the 1-GPU result")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write DIR/windows.npy: %d seeded rows (sorted, rows in corpus order) of "
                         "the float32 (N, 11, %d) windows the last timed step stored" % (DUMP_ROWS, C))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; the CPU arm times a bounded sample of "
                 "the corpus and has no output of the whole step to write")
    return args


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ---- clocks --------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([f.strip() for f in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                power.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        load = [s for s, p in zip(sm, power) if p >= 0.5 * max(power)] if power else sm
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "reasons": sorted(reasons), "samples": len(sm)}


# ---- CPU arm -------------------------------------------------------------------------------
def cpu_arm(coefs, lengths, seed, seconds, steps=1, warmup=0):
    """Time the oracle port (erb_filterbank -> ExtractEnvelopeFromMatrix(True,50) -> window
    gather, float64, in memory) on a bounded sample of the corpus with all host threads."""
    from f2cnn_b200 import synth
    from oracle import oracle as orc
    orc.lib()
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every core it may run on
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    orc.set_num_threads(avail)
    cores = orc.num_threads()
    rng = np.random.default_rng(seed)
    order = rng.permutation(len(lengths))

    def run(idx):
        n = int(lengths[idx])
        w = synth.white_noise_i16(n, seed=10_000 + int(idx))
        t = time.perf_counter()
        orc.utterance(w, coefs, True, CUTOFF, synth.label_grid(n), RADIUS, STEP)
        return time.perf_counter() - t, n

    dt, n0 = run(order[0])  # calibration (also warms the twiddle / page cache)
    per_step = max(2, min(len(order), int(seconds / max(dt, 1e-3) / max(steps, 1))))
    for _ in range(warmup):
        run(order[0])
    total_t, total_n = 0.0, 0
    pos = 0
    step_rates = []
    for _ in range(steps):
        st, sn = 0.0, 0
        for _ in range(per_step):
            d, n = run(order[pos % len(order)])
            pos += 1
            st += d
            sn += n
        step_rates.append(C * sn / st)
        total_t += st
        total_n += sn
    # single-core figure beside it (SURVEY.md 8d): two utterances on one thread
    orc.set_num_threads(1)
    t1, n1 = 0.0, 0
    for k in range(2):
        d, n = run(order[(pos + k) % len(order)])
        t1 += d
        n1 += n
    orc.set_num_threads(avail)
    return {"value": C * total_n / total_t, "unit": "channel-samples/s", "cores": cores, "kind": "port",
            "value_single_core": C * n1 / t1,
            "sample": "%d utterances (%d samples) of the corpus per step x %d steps, float64 C port of the "
                      "reference algorithm, OpenMP over channels, in memory" % (per_step, total_n // max(steps, 1),
                                                                                steps),
            "seconds": total_t}, total_t / max(steps, 1)


def other_configs(coefs128):
    """The BASELINE.json configs that are not the headline, timed on the device (rank 0, N = 1):
    configs[0] one 3 s utterance (latency of the public call), configs[3] the 600 s x 256-channel stream
    at 20/50/100 Hz cut-off, configs[4] evalnoise -- noisy float64 utterances through filterbank,
    envelope and the tensor-core CNN on every stride-1 frame."""
    import torch
    from f2cnn_b200 import api, cnn, engine, synth
    from f2cnn_b200.gammatone import filters

    def timed(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = engine.DeviceEvent(), engine.DeviceEvent()
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_ms(b) / reps

    out = {}
    fma_peak = 148 * 128 * 2 * 1965e6
    # ---- configs[0]: single utterance, host wave in -> host windows out ----
    w = synth.white_noise_i16(48000, 0)
    centers = synth.label_grid(48000)
    api.features_to_windows([w], coefs128, [centers], True, CUTOFF)
    t = time.perf_counter()
    for _ in range(20):
        api.features_to_windows([w], coefs128, [centers], True, CUTOFF)
    ms = (time.perf_counter() - t) / 20 * 1e3
    out["config1_single_utterance"] = {"host_ms_per_call": ms, "channel_samples_per_s": C * 48000 / ms * 1e3,
                                       "path": "api.features_to_windows, 3 s x 128 ch, time-chunked"}
    # ---- configs[3]: 600 s stream, 256 channels ----
    n = 9_600_000
    co256 = filters.make_erb_filters(FS, filters.centre_freqs(FS, 256, LOW))
    plan4 = engine.plan_for(co256)
    w4 = torch.from_numpy(synth.white_noise_i16(n, seed=2)).cuda()
    b4 = plan4.batch([n])
    dec4 = torch.empty((b4.total_frames, 256), dtype=torch.float32, device="cuda")
    for cut in (20, 50, 100):
        ms = timed(lambda: b4.run(w4, lpf=True, cutoff=cut, out={"dec": dec4}), reps=3, warm=1)
        rate = 256.0 * n / ms * 1e3
        out["config4_stream_600s_256ch_cutoff%d" % cut] = {"device_ms": ms, "channel_samples_per_s": rate, "items": b4.num_items,
                                                           "fma_roofline_frac": FLOP_PER_CS * rate / fma_peak}
    del w4, dec4, b4
    # ---- configs[4]: evalnoise ----
    model = cnn.seeded_model(0)
    net = cnn.TensorCoreCNN(model)
    plan = engine.plan_for(coefs128)
    base = synth.speech_like_i16(48000, seed=31).astype(np.float64)
    rms = float(np.sqrt(np.mean(base ** 2)))
    for snr_db in (0, 10, 20):
        noisy = base + np.random.default_rng(3 + snr_db).normal(scale=rms / 10 ** (snr_db / 20.0), size=48000)
        wd = torch.from_numpy(noisy).cuda()
        b5 = plan.batch([48000])

        def run():
            env_t = b5.run(wd, lpf=True, cutoff=CUTOFF, env_t=True)["env_t"]
            return env_t, net.predict_envelope(env_t, STEP)

        ms_all = timed(run, reps=5)
        env_t, scores = run()
        ms_cnn = timed(lambda: net.predict_envelope(env_t, STEP), reps=5)
        frames = 48000 - 11 * STEP
        out["config5_evalnoise_snr%ddB" % snr_db] = {
            "frames": frames, "device_ms_filterbank_envelope_cnn": ms_all, "device_ms_cnn": ms_cnn,
            "frames_per_s": frames / ms_all * 1e3, "cnn_tflops": frames * 2 * 21.0e6 / ms_cnn / 1e9,
            "rising_fraction": float((scores[:, 1] > scores[:, 0]).float().mean()),
            "cnn": "tcgen05 kernels (csrc/f2_cnn.cu), bf16 x bf16 -> fp32, seeded weights (no trained model ships with the reference)"}
    return out


def dump_windows(path, windows, shards, nwin_all, rank):
    """--dump-outputs: a fixed, seeded sample of the corpus's windows, rows numbered as in the whole corpus.
    Rank r's `windows` holds the rows of its utterances shards[r]; every sampled row is copied from the rank
    that computed it, so the file is the same, bit for bit, for any number of GPUs."""
    import torch
    import torch.distributed as dist
    first = np.concatenate([[0], np.cumsum(nwin_all)])
    rows = np.sort(np.random.default_rng(0).choice(int(first[-1]), size=min(DUMP_ROWS, int(first[-1])), replace=False))
    owner = np.empty(len(nwin_all), dtype=np.int64)        # utterance -> rank
    local_first = np.empty(len(nwin_all), dtype=np.int64)  # utterance -> its first row in its rank's `windows`
    for r, utts in enumerate(shards):
        owner[utts] = r
        local_first[utts] = np.cumsum(nwin_all[utts]) - nwin_all[utts]
    utt = np.searchsorted(first, rows, side="right") - 1
    src = local_first[utt] + rows - first[utt]

    def of_rank(r):
        return torch.from_numpy(np.flatnonzero(owner[utt] == r)).to(windows.device)

    sample = torch.zeros((len(rows),) + tuple(windows.shape[1:]), dtype=windows.dtype, device=windows.device)
    mine = of_rank(rank)
    sample[mine] = windows[torch.from_numpy(src).to(windows.device)[mine]]
    if len(shards) > 1:
        parts = [torch.empty_like(sample) for _ in shards] if rank == 0 else None
        dist.gather(sample, parts, dst=0)
        if rank == 0:
            for r in range(1, len(shards)):
                sel = of_rank(r)
                sample[sel] = parts[r][sel]
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        np.save(os.path.join(path, "windows.npy"), sample.cpu().numpy())


def main():
    args = parse()
    rank, local_rank, world = dist_env()
    from f2cnn_b200 import synth
    from f2cnn_b200.gammatone import filters
    coefs = filters.make_erb_filters(FS, filters.centre_freqs(FS, C, LOW))
    dots = 2 * RADIUS + 1
    config = {"workload": "synthetic TIMIT-TRAIN-sized corpus: %d utterances x U(%d,%d) samples @16 kHz int16 (seed 1), "
                          "%d-ch ERB gammatone -> ENV1 (LPF %d Hz) -> (N,11,%d) float32 windows on the full label "
                          "grid%s" % (args.utts, LEN_LO, LEN_HI, C, CUTOFF, C,
                                      "" if world == 1 else "; the SAME corpus dealt to %d GPUs by length-sorted "
                                      "round-robin, rows placed into ONE shared host tensor" % world),
              "utterances": args.utts, "utterances_per_gpu": args.utts / world, "channels": C, "lpf_hz": CUTOFF,
              "l2": "inputs larger than L2 (rings %.1f GB per pass and GPU), no flush needed" %
                    (args.utts / world * 65536 * 16 / 1e9)}

    if args.impl == "reference":
        if rank != 0:
            return
        lengths = synth.corpus_lengths(args.utts, LEN_LO, LEN_HI, seed=1)
        cb, ms = cpu_arm(coefs, lengths, 1, args.cpu_seconds * 4, steps=args.steps, warmup=min(args.warmup, 1))
        print(json.dumps({"impl": "reference", "metric": "channel-samples/sec (filterbank+envelope)",
                          "value": cb["value"], "unit": "channel-samples/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms * 1e3,
                          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                          "data": "synthetic", "config": config, "cpu_baseline": cb,
                          "e2e": {"value": cb["value"], "unit": "channel-samples/s", "h2d_bytes_per_step": 0,
                                  "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from f2cnn_b200 import api, engine, hostmem

    # every rank holds the SAME corpus (config 3: "same corpus utterance-sharded"); its shard is what
    # engine.shard_utterances deals it
    lengths = synth.corpus_lengths(args.utts, LEN_LO, LEN_HI, seed=1)
    flat, offsets = synth.corpus_waves_i16(lengths, seed=1)
    total_samples = int(offsets[-1])
    cs_per_step = float(C) * total_samples          # the WHOLE job, whatever the number of GPUs
    shards = engine.shard_utterances(lengths, world)
    mine = shards[rank]
    my_lengths = lengths[mine]

    plan = engine.plan_for(coefs, local_rank)
    # whole utterances (target_items=1): bit for bit what the 1-GPU pass computes, and a shard of >= 578
    # utterances x 4 channel groups already fills the 2368 CTA slots of the device
    batch = plan.batch(my_lengths, step=STEP, phase=0, target_items=1)
    # label grid: centres 800 + 160k, k < int(n/160 - 12): first frame of window k is frame k
    nwin_all = np.maximum((lengths / STEP - dots - 1).astype(np.int64), 0)
    n_windows_all = int(nwin_all.sum())
    nwin = nwin_all[mine]
    n_windows = int(nwin.sum())
    base = np.concatenate([batch.frame_offsets[u] + np.arange(nwin[u], dtype=np.int64) for u in range(len(my_lengths))])

    wave_host = torch.from_numpy(flat).pin_memory()
    wave_dev = torch.cat([torch.from_numpy(flat[offsets[u]:offsets[u + 1]]) for u in mine]).to(dev)
    base_dev = torch.from_numpy(base).to(dev)
    dec = torch.empty((batch.total_frames, C), dtype=torch.float32, device=dev)
    windows = torch.empty((n_windows, dots, C), dtype=torch.float32, device=dev)

    grid_offsets, grid_rows = batch.grid_windows(dots)
    assert grid_rows == n_windows

    def step(events=None):
        # the label-grid windows are stored by the fused kernel itself (no decimated round trip)
        batch.run(wave_dev, lpf=True, cutoff=CUTOFF, windows=(grid_offsets, dots, windows), fused_events=events)

    # the fused window store must equal decimated frames + gather (the general path), bit for bit
    step()
    batch.run(wave_dev, lpf=True, cutoff=CUTOFF, out={"dec": dec})
    check = torch.empty((min(n_windows, 4096), dots, C), dtype=torch.float32, device=dev)
    for r0 in (0, max(n_windows // 2 - 2048, 0), max(n_windows - 4096, 0)):
        engine.gather_windows(dec, base_dev[r0:r0 + check.shape[0]], dots, 1, out=check[:min(4096, n_windows - r0)])
        assert torch.equal(check[:min(4096, n_windows - r0)], windows[r0:r0 + 4096]), "window store differs from gather"

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    # nvidia-smi samples every 100 ms and a sharded step lasts a few ms: keep the device under the same load
    # (untimed steps) until the sampler has seen it, then time
    t_load = time.perf_counter()
    while time.perf_counter() - t_load < 0.6:
        step()
        torch.cuda.synchronize()
    ev = [(engine.DeviceEvent(), engine.DeviceEvent()) for _ in range(args.steps)]
    t_start, t_stop = engine.DeviceEvent(), engine.DeviceEvent()
    barrier()
    t_start.record()
    for i in range(args.steps):
        step(ev[i])
    t_stop.record()
    barrier()
    clocks = sampler.stop()
    fused_ms = float(np.mean([a.elapsed_ms(b) for a, b in ev]))
    ms_step = max_over_ranks(t_start.elapsed_ms(t_stop)) / args.steps
    value = cs_per_step / (ms_step * 1e-3)
    windows_head = windows[:64].cpu() if rank == 0 else None
    if args.dump_outputs:
        dump_windows(args.dump_outputs, windows, shards, nwin_all, rank)
    del windows, dec, check

    # ---- e2e: THE PUBLIC CALL, host int16 waves in, host float32 input tensor out ---------------------
    e2e = None
    if not args.no_e2e:
        centers = np.concatenate([STEP * RADIUS + STEP * np.arange(k, dtype=np.int64) for k in nwin_all])
        shard = None if world == 1 else (rank, world)
        shared = None
        backing = "private array (engine.host_empty: anonymous memory advised to huge pages)"
        if world == 1:
            out_arr = engine.host_empty((n_windows_all, dots, C), np.float32)
        else:
            # ONE host tensor for all ranks: a shared mapping on the RAM-backed filesystem
            need = n_windows_all * dots * C * 4
            d = hostmem.shm_dir()
            if d is None or hostmem.shm_free_bytes(d) < need + (64 << 20):
                import tempfile
                d = tempfile.gettempdir()
            path = os.path.join(d, "f2cnn_b200_bench_%s.f32" % os.environ.get("MASTER_PORT", "0"))
            if rank == 0:
                shared = hostmem.SharedArray(path, (n_windows_all, dots, C), create=True)
            barrier()
            if rank != 0:
                shared = hostmem.SharedArray(path, (n_windows_all, dots, C))
            out_arr = shared.array
            backing = "one shared mapping under %s, mapped by all %d ranks" % (d, world)

        def call(out):
            return api.features_to_windows((wave_host, lengths), coefs, centers, True, CUTOFF, RADIUS, STEP,
                                           out=out, counts=nwin_all, shard=shard)

        barrier()
        t0 = time.perf_counter()
        call(out_arr)                     # first call: builds and caches the pipeline, touches `out`
        cold_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
        call(out_arr)
        k = args.steps
        barrier()
        t0 = time.perf_counter()
        for _ in range(k):
            call(out_arr)
        torch.cuda.synchronize()
        warm_local = (time.perf_counter() - t0) * 1e3 / k
        barrier()
        ms_e2e = max_over_ranks(warm_local)
        fresh_ms = None
        if world == 1:
            # the same call when the caller does not hand in an output array: a new 7.5 GB array per call
            # (the first one faults its pages in; once dropped, its block is pooled for the next call)
            fresh_ms = []
            for _ in range(3):
                t0 = time.perf_counter()
                tmp = api.features_to_windows((wave_host, lengths), coefs, centers, True, CUTOFF, RADIUS, STEP, counts=nwin_all)
                fresh_ms.append((time.perf_counter() - t0) * 1e3)
                del tmp
        barrier()
        # the same corpus for a consumer that reads windows as VIEWS of the decimated frames (api.features_to_frames):
        # nothing is expanded on the host, so this is the end-to-end time of the GPU side alone -- a side figure,
        # NOT the contract's input_data.npy tensor
        api.features_to_frames((wave_host, lengths), coefs, True, CUTOFF, RADIUS, STEP, counts=nwin_all, shard=shard)
        barrier()
        t0 = time.perf_counter()
        for _ in range(k):
            fw = api.features_to_frames((wave_host, lengths), coefs, True, CUTOFF, RADIUS, STEP, counts=nwin_all, shard=shard)
        frames_local = (time.perf_counter() - t0) * 1e3 / k
        barrier()
        ms_frames = max_over_ranks(frames_local)
        if rank == 0 and world == 1:
            assert np.array_equal(fw.windows(0), out_arr[:int(nwin_all[0])]), "frame views differ from the placed rows"
        del fw
        pipe_subs = None
        with api._pipelines_lock:
            for p_ in api._pipelines.values():
                pipe_subs = (len(p_.subs), p_.placer.threads)
        verified = None
        if rank == 0:
            # the host path must produce exactly what the resident path produced ...
            g0 = int(np.cumsum(nwin_all)[mine[0]] - nwin_all[mine[0]])   # first row of this rank's first utterance
            k0 = min(64, int(nwin[0]))
            assert np.array_equal(out_arr[g0:g0 + k0], windows_head.numpy()[:k0]), "e2e path differs from resident path"
            if world > 1 and not args.no_verify:
                # ... and the tensor the N ranks assembled must equal the 1-GPU result, bit for bit
                one = api.features_to_windows((wave_host, lengths), coefs, centers, True, CUTOFF, RADIUS, STEP, counts=nwin_all)
                verified = bool(np.array_equal(one, out_arr))
                assert verified, "sharded result differs from the single-GPU result"
                del one
        barrier()
        my_frames = int(np.sum((my_lengths + STEP - 1) // STEP))
        e2e = {"value": cs_per_step / (ms_e2e * 1e-3), "unit": "channel-samples/s",
               "h2d_bytes_per_step": total_samples * 2,
               "d2h_bytes_per_step": int(np.sum((lengths + STEP - 1) // STEP)) * C * 4,
               "host_tensor_bytes": n_windows_all * dots * C * 4,
               "ms_per_step": ms_e2e, "first_call_ms": cold_ms, "fresh_output_ms": fresh_ms,
               "frames_as_views": {"ms_per_step": ms_frames, "value": cs_per_step / (ms_frames * 1e-3),
                                   "what": "api.features_to_frames: host waves in, decimated frames on the host, windows "
                                           "read as overlapping views of them (0.71 GB instead of the 7.5 GB tensor); "
                                           "side figure, not the input_data.npy contract"}, "timer": "host wall clock "
               "around the call (it returns when the last row is placed), max over ranks",
               "path": "api.features_to_windows((pinned int16 waves, lengths), coefs, centres, LPF=True, 50, out=..., "
                       "counts=...%s): cached engine.WindowPipeline, %s sub-batches, uploads on one stream, kernels on two, the "
                       "fused kernel stores its decimated frames into pinned host memory, rows placed by %s host threads per rank" %
                       ("" if world == 1 else ", shard=(rank, world)", pipe_subs[0] if pipe_subs else "?",
                        pipe_subs[1] if pipe_subs else "?"),
               "output": backing, "equals_single_gpu_result": verified, "frames_per_rank": my_frames}
        if shared is not None:
            barrier()
            if rank == 0:
                shared.unlink()
        api.release_cached_pipelines()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except OSError:
        pass
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    fma_peak = 148 * 128 * 2 * sm_max * 1e6 / 1e12  # TFLOP/s, nominal FP32 FMA at max clock
    my_cs = float(C) * float(my_lengths.sum())
    achieved = FLOP_PER_CS * my_cs / (fused_ms * 1e-3) / 1e12
    roofline = {"bound": "fp32_fma", "kernel": "fused_kernel", "achieved": achieved, "peak": fma_peak,
                "unit": "TFLOP/s", "frac": achieved / fma_peak,
                # dram__bytes_read.sum + dram__bytes_write.sum of one fused_kernel launch on the 1-GPU workload,
                # ncu --set full capture summarised in profiles/ (see DESIGN.md section 5)
                "traffic": TRAFFIC_1GPU if (args.utts == N_UTTS and world == 1) else None,
                "peak_source": "148 SM x 128 lanes x 2 x sm_max_mhz (MEASURED_PEAKS.json has no FP32 entry); "
                               "tools/fma_peak.cu measured 73.8 TFLOP/s sustained (FFMA2) on this pool",
                "kernel_ms": fused_ms, "kernel_share_of_step": fused_ms / ms_step,
                "algorithmic_flop_per_channel_sample": FLOP_PER_CS,
                # ring tiles (x, xi, G: 12 B per sample, shared by the C channels) + every decimated frame
                # stored into the 2R+1 window rows that contain it
                "hbm": {"algorithmic_bytes_per_channel_sample": 12.0 / C + 4.0 * dots / STEP,
                        "achieved_GBps": (12.0 / C + 4.0 * dots / STEP) * my_cs / (fused_ms * 1e-3) / 1e9,
                        "peak_GBps": peaks.get("hbm_gbs")}}
    cpu = None
    if not args.no_cpu and world == 1:
        cpu, _ = cpu_arm(coefs, lengths, 1, args.cpu_seconds)
    others = None
    if world == 1 and not args.no_configs:
        del wave_dev, wave_host
        torch.cuda.empty_cache()
        try:
            others = other_configs(coefs)
        except Exception as e:  # the headline line must not depend on the side configs
            others = {"error": repr(e)}
    out = {"metric": "channel-samples/sec (filterbank+envelope)", "value": value, "unit": "channel-samples/s",
           "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": config, "clocks": clocks, "e2e": e2e, "gpu_launches": KERNELS_PER_STEP * args.steps,
           "roofline": roofline, "cpu_baseline": cpu, "windows_per_step": n_windows_all, "other_configs": others}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
