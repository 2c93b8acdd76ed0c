"""Full-rate output modes -- (C, n) in either dtype, alone, mixed or next to the time-major envelope: parity
against the oracle and the HBM roofline figure of SURVEY.md 8d (16.04 / 12.04 / 8.04 bytes per channel-sample)
on 256 corpus utterances."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from f2cnn_b200 import engine, synth
from f2cnn_b200.gammatone import filters
from oracle import oracle

co = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))
plan = engine.plan_for(co)
lengths = synth.corpus_lengths(256, seed=1)
flat, _ = synth.corpus_waves_i16(lengths, seed=1)
fd = torch.from_numpy(flat).cuda()
bq = plan.batch(lengths)
cs = 128.0 * float(lengths.sum())
for tag, kw, bpc in (("gfb+env f64 (reference layout)", dict(gfb=torch.float64, env=torch.float64), 16.04),
                     ("gfb+env f32", dict(gfb=torch.float32, env=torch.float32), 8.04),
                     ("env f64 only", dict(env=torch.float64), 8.02), ("gfb f64 only", dict(gfb=torch.float64), 8.02),
                     ("env f64 + env_t f32", dict(env=torch.float64, env_t=True), 12.04),
                     ("gfb f64 + env f32", dict(gfb=torch.float64, env=torch.float32), 12.04)):
    res = bq.run(fd, lpf=True, cutoff=50, **kw)
    torch.cuda.synchronize()
    a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        bq.run(fd, lpf=True, cutoff=50, out=res, **kw)
    z.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(z) / 3
    print("%-32s %.3f ms  %.3e ch-samples/s  %.0f GB/s algorithmic = %.2f of the 6533 GB/s HBM peak" % (tag, ms, cs / ms * 1e3, bpc * cs / ms / 1e6, bpc * cs / ms / 1e6 / 6533.5))
    # spot parity of the first and last utterance
    for u in (0, 255):
        n = int(lengths[u]); off = int(lengths[:u].sum())
        w = flat[off:off + n]
        go = oracle.erb_filterbank(w, co); eo = oracle.extract_envelope(go, True, 50)
        for key, want in (("gfb", go), ("env", eo)):
            if key in res:
                got = res[key][128 * off:128 * (off + n)].double().cpu().numpy().reshape(128, n)
                err = (np.max(np.abs(got - want), axis=1) / np.sqrt(np.mean(want ** 2, axis=1))).max()
                assert err <= 1e-4, (tag, u, key, err)
    del res
print("parity ok")
