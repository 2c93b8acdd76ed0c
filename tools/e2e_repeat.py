"""The public call on the bench corpus, N times: per-call wall times (ms), median and min.
usage: tools/e2e_repeat.py [calls]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from f2cnn_b200 import api, engine, synth
from f2cnn_b200.gammatone import filters

calls = int(sys.argv[1]) if len(sys.argv) > 1 else 12
co = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))
lengths = synth.corpus_lengths(4620, 32000, 64000, seed=1)
flat, _ = synth.corpus_waves_i16(lengths, seed=1)
wave = torch.from_numpy(flat).pin_memory()
nwin = np.maximum((lengths / 160 - 12).astype(np.int64), 0)
centers = np.concatenate([800 + 160 * np.arange(k, dtype=np.int64) for k in nwin])
out = engine.host_empty((int(nwin.sum()), 11, 128), np.float32)
ms = []
for i in range(calls + 2):
    t = time.perf_counter()
    api.features_to_windows((wave, lengths), co, centers, True, 50, 5, 160, out=out, counts=nwin)
    ms.append((time.perf_counter() - t) * 1e3)
warm = np.array(ms[2:])
print("first %.1f ms; warm calls: %s -> median %.2f min %.2f ms; checksum %.6e" % (
    ms[0], " ".join("%.1f" % m for m in warm), np.median(warm), warm.min(),
    float(out[::997].astype(np.float64).sum())))
