"""Which stage is late when one public call in six takes 4 ms longer?  12 timed pipeline runs: end of the
GPU chain (CUDA events) and end of placement per run, plus gc activity."""
import gc, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from f2cnn_b200 import engine, synth
from f2cnn_b200.gammatone import filters

co = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))
plan = engine.plan_for(co)
lengths = synth.corpus_lengths(4620, 32000, 64000, seed=1)
flat, offs = synth.corpus_waves_i16(lengths, seed=1)
wave_host = torch.from_numpy(flat).pin_memory()
nwin = np.maximum((lengths / 160 - 12).astype(np.int64), 0)
centers = np.concatenate([800 + 160 * np.arange(k, dtype=np.int64) for k in nwin])
out = engine.host_empty((int(nwin.sum()), 11, 128), np.float32)
pipe = engine.WindowPipeline(plan, lengths, placer=engine.Placer(15))
runs, _, _ = engine.window_runs(centers, nwin, lengths, pipe.frame_offsets)
for _ in range(3):
    pipe.run(wave_host, runs, out)
pipe.timing = True
if len(sys.argv) > 1 and sys.argv[1] == "nogc":
    gc.disable()
for i in range(14):
    g0 = gc.get_count()
    t = time.perf_counter()
    pipe.run(wave_host, runs, out)
    total = (time.perf_counter() - t) * 1e3
    subs, jobs = pipe.timeline()
    print("run %2d total %.2f ms | kernels end %.2f | first runnable %.2f last placed %.2f | per-sub place ms %s | gc %s" % (
        i, total, max(s["kernels"] for s in subs), jobs[0]["runnable"], max(j["placed"] for j in jobs),
        " ".join("%.1f" % (j["placed"] - j["runnable"]) for j in jobs), g0), flush=True)
