"""Cutoff sweep against separate runs, on the GPU, in one process.

1. The 600 s x 256-channel stream of BASELINE.json configs[3] with the settings (20, 50, 100, None): one
   Batch.run_cutoffs against the four single-setting Batch.run calls, alternated, CUDA events, warm.
2. The 4620-utterance bench corpus: api.features_to_windows_sweep with (20, 50, 100) against three
   api.features_to_windows calls, alternated, host clock around calls that end synchronised, both filling the
   same preallocated host outputs; the rows are asserted equal bit for bit in the same run.

Prints the card's name and power limit with the numbers.  Usage: python tools/cutoff_sweep.py [reps]"""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from f2cnn_b200 import api, engine, synth
from f2cnn_b200.gammatone import filters


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def device_ms(fn):
    a, b = engine.DeviceEvent(), engine.DeviceEvent()
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_ms(b)


def stats(v):
    v = np.asarray(v)
    return "median %.3f  min %.3f  max %.3f ms (n=%d)" % (np.median(v), v.min(), v.max(), v.size)


def main(reps=20):
    print("card:", card())
    settings = (20, 50, 100, None)

    # ---- 1. configs[3]: 600 s stream, 256 channels ----
    n = 9_600_000
    co256 = filters.make_erb_filters(16000, filters.centre_freqs(16000, 256, 100))
    plan = engine.plan_for(co256)
    wd = torch.from_numpy(synth.white_noise_i16(n, seed=2)).cuda()
    b = plan.batch([n])
    dec = torch.empty((b.total_frames, 256), device="cuda")
    planes = torch.empty((len(settings), b.total_frames, 256), device="cuda")
    print("stream: %d samples x 256 channels, %d work items, settings %s" % (n, b.num_items, settings))

    def separate():
        for c in settings:
            b.run(wd, lpf=c is not None, cutoff=100 if c is None else c, out={"dec": dec})

    def sweep():
        b.run_cutoffs(wd, settings, out=planes)

    for _ in range(3):
        separate()
        sweep()
    t_sep, t_sw = [], []
    for _ in range(reps):
        t_sep.append(device_ms(separate))
        t_sw.append(device_ms(sweep))
    print("stream, four separate runs: ", stats(t_sep))
    print("stream, one sweep:          ", stats(t_sw))
    print("stream, sweep / separate:    %.3f" % (np.median(t_sw) / np.median(t_sep)))
    for j, c in enumerate(settings):
        b.run(wd, lpf=c is not None, cutoff=100 if c is None else c, out={"dec": dec})
        d = (planes[j] - dec).abs().max().item()
        print("stream, plane %s: max |sweep - single run| = %.3g (rms %.3g)" % (c, d, dec.pow(2).mean().sqrt().item()))
    del wd, dec, planes, b

    # ---- 2. bench corpus, public calls ----
    co128 = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))
    lengths = synth.corpus_lengths(4620, 32000, 64000, seed=1)
    flat, _ = synth.corpus_waves_i16(lengths, seed=1)
    wave_host = torch.from_numpy(flat).pin_memory()
    counts = np.maximum((lengths / 160 - 11 - 1).astype(np.int64), 0)
    centers = np.concatenate([160 * 5 + 160 * np.arange(k, dtype=np.int64) for k in counts])
    cut3 = (20, 50, 100)
    print("corpus: %d utterances, %d windows x 11 x 128, settings %s" % (lengths.size, int(counts.sum()), cut3))
    outs = [engine.host_empty((int(counts.sum()), 11, 128), np.float32) for _ in cut3]
    one = engine.host_empty((int(counts.sum()), 11, 128), np.float32)

    def separate3():
        for c, o in zip(cut3, outs):
            api.features_to_windows((wave_host, lengths), co128, centers, True, c, counts=counts, out=o)

    def sweep3():
        api.features_to_windows_sweep((wave_host, lengths), co128, centers, cut3, counts=counts, out=outs)

    separate3()
    sweep3()
    for c, o in zip(cut3, outs):
        api.features_to_windows((wave_host, lengths), co128, centers, True, c, counts=counts, out=one)
        assert np.array_equal(o, one), "cutoff %s: sweep differs from features_to_windows" % c
    print("corpus: sweep rows == features_to_windows rows bit for bit for", cut3)
    del one
    corpus_reps = max(3, reps // 4)
    h_sep, h_sw = [], []
    for _ in range(corpus_reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        separate3()
        h_sep.append((time.perf_counter() - t) * 1e3)
        t = time.perf_counter()
        sweep3()
        h_sw.append((time.perf_counter() - t) * 1e3)
    print("corpus, three features_to_windows calls:  ", stats(h_sep))
    print("corpus, one features_to_windows_sweep call:", stats(h_sw))
    print("corpus, sweep / separate:                  %.3f" % (np.median(h_sw) / np.median(h_sep)))
    print("card:", card())


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 20)
