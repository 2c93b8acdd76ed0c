"""The one-kernel ring transform (ring_cluster_kernel) against scipy.signal.hilbert on rows that pad to
N2 = 32768 and 65536, and the per-utterance frame checksums of a corpus slice with and without it
(F2CNN_B200_RING_CLUSTER=0 in a child process: the multi-pass kernels)."""
import os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch


def errors():
    from scipy.signal import hilbert
    from f2cnn_b200 import api
    rng = np.random.default_rng(7)
    for n in (20000, 32768, 32769, 47001, 65535, 65536, 65537, 100003, 131072):
        m = rng.normal(0, 3000, (6, n))
        N2 = 1 << int(np.ceil(np.log2(n)))
        want = np.imag(hilbert(np.concatenate([m, np.zeros((6, N2 - n))], axis=1), axis=1))[:, :n]
        got = api.hilbert_imag_rows(m)
        print("n=%6d N2=%6d  max |xi - scipy| / rms = %.2e" % (n, N2, np.max(np.abs(got - want)) / np.sqrt(np.mean(want ** 2))), flush=True)


def checksums():
    from f2cnn_b200 import engine, synth
    from f2cnn_b200.gammatone import filters
    coefs = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))
    lengths = synth.corpus_lengths(4620, seed=1)
    if os.environ.get("RING_CHECK_LONG"):   # a corpus of 4.1 ... 8.2 s utterances: rings of 131072 samples
        lengths = synth.corpus_lengths(2310, 65537, 131072, seed=1)
    flat = torch.from_numpy(synth.corpus_waves_i16(lengths, seed=1)[0]).cuda()
    plan = engine.plan_for(coefs)
    batch = plan.batch(lengths, step=160, phase=0)
    out = {"dec": torch.empty((batch.total_frames, 128), dtype=torch.float32, device="cuda")}
    batch.run(flat, lpf=True, cutoff=50, dec=True, out=out)
    torch.cuda.synchronize()
    sums = torch.stack([out["dec"][int(a):int(b)].double().sum() for a, b in zip(batch.frame_offsets[:-1], batch.frame_offsets[1:])]).cpu().numpy()
    np.save("gpurun_out/ring_sums_%s.npy" % os.environ.get("F2CNN_B200_RING_CLUSTER", "1"), sums)
    np.save("gpurun_out/ring_lengths.npy", lengths)
    print("cluster=%s  checksum %.9e" % (os.environ.get("F2CNN_B200_RING_CLUSTER", "1"), float(out["dec"].double().sum())),
          flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "checksums":
        checksums()
    else:
        errors()
        for v in ("1", "0"):
            subprocess.run([sys.executable, __file__, "checksums"], env=dict(os.environ, F2CNN_B200_RING_CLUSTER=v))
        a, b = np.load("gpurun_out/ring_sums_1.npy"), np.load("gpurun_out/ring_sums_0.npy")
        lengths = np.load("gpurun_out/ring_lengths.npy")
        rel = np.abs(a - b) / np.abs(b)
        bad = np.nonzero(rel > 1e-6)[0]
        print("per-utterance checksums: max rel diff %.2e, %d utterances above 1e-6" % (rel.max(), bad.size))
        for u in bad[:20]:
            print("   utt %d n=%d rel %.2e" % (u, lengths[u], rel[u]))
