"""Timeline of one corpus-sized pipeline run: when each sub-batch's waves, kernels (and with them its
frames, which the fused kernel stores into host memory) and rows were done (ms since the start of the call)."""
import os, sys, time
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
out[:] = 0
threads = int(sys.argv[1]) if len(sys.argv) > 1 else 0
pipe = engine.WindowPipeline(plan, lengths, placer=engine.Placer(threads))
runs, _, _ = engine.window_runs(centers, nwin, lengths, pipe.frame_offsets)
for _ in range(3):
    pipe.run(wave_host, runs, out)
pipe.timing = True
t = time.perf_counter()
pipe.run(wave_host, runs, out)
total = (time.perf_counter() - t) * 1e3
subs, jobs = pipe.timeline()
print("placement threads %d, total %.2f ms (includes the leading synchronize)" % (pipe.placer.threads, total))
print("sub  utts   waves-on-device  kernels-done | rows runnable   placed   (rows)")
for i, s in enumerate(subs):
    j = jobs[i] if i < len(jobs) else dict(runnable=float("nan"), placed=float("nan"), rows=0)
    print("%3d %5d %12.2f %14.2f | %12.2f %10.2f %9d" % (i, s["utterances"], s["h2d"], s["kernels"],
                                                       j["runnable"], j["placed"], j["rows"]))
