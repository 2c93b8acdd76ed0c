"""Scoring a corpus with the tensor-core CNN: per-utterance calls against api.cnn_evaluate_corpus, on the GPU.

The bench's seed-1 corpus (4620 utterances of U(32000, 64000) int16 samples, or its first --utts), LPF at 50 Hz,
seeded weights.  Three timings, host clock around calls that end with the scores on the host:
  1. a loop of api.cnn_evaluate(..., with_envelopes=False), one call per utterance;
  2. api.cnn_evaluate_corpus on one GPU;
  3. api.cnn_evaluate_corpus with shard=(rank, world) over every visible GPU, one process per GPU writing into
     one hostmem.SharedArray: from the moment all ranks are ready (warmed up) to the last rank's return.  With one
     visible GPU: rank 0's share of a 2-, 4- and 8-GPU run, timed alone on that GPU.
The scores of 2 and 3 are asserted equal bit for bit; those of 1 are compared with 2.  Prints every card's name
and power limit with the numbers.  Usage: python tools/cnn_corpus.py [--utts N] [--reps R]"""
import argparse
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

LPF, CUTOFF, SEED_MODEL = True, 50, 0


def cards():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "nvidia-smi unavailable"


def corpus(n_utts):
    from f2cnn_b200 import synth
    lengths = synth.corpus_lengths(4620, 32000, 64000, seed=1)
    flat, _ = synth.corpus_waves_i16(lengths, seed=1)
    return flat[:int(lengths[:n_utts].sum())], lengths[:n_utts]


def coefs():
    from f2cnn_b200.gammatone import filters
    return filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))


def rank_main(rank, world, n_utts, path, total, reps, barrier, q):
    import torch
    torch.cuda.set_device(rank)
    from f2cnn_b200 import api, cnn, hostmem
    flat, lengths = corpus(n_utts)
    wave_host = torch.from_numpy(flat).pin_memory()
    model = cnn.seeded_model(SEED_MODEL)
    out = hostmem.SharedArray(path, (total, 2), np.float32)
    api.cnn_evaluate_corpus((wave_host, lengths), coefs(), model, LPF, CUTOFF, out=out.array, shard=(rank, world))
    for _ in range(reps):
        barrier.wait()
        t0 = time.time()
        api.cnn_evaluate_corpus((wave_host, lengths), coefs(), model, LPF, CUTOFF, out=out.array, shard=(rank, world))
        q.put((rank, t0, time.time()))
    barrier.wait()


def stats(v):
    v = np.asarray(v)
    return "median %.3f  min %.3f  max %.3f s (n=%d)" % (np.median(v), v.min(), v.max(), v.size)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=4620)
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    import torch
    from f2cnn_b200 import api, cnn, engine, hostmem
    print("cards:\n" + cards())
    flat, lengths = corpus(args.utts)
    wave_host = torch.from_numpy(flat).pin_memory()
    co = coefs()
    model = cnn.seeded_model(SEED_MODEL)
    nb = np.maximum(lengths - 11 * 160, 0)
    offsets = np.concatenate([[0], np.cumsum(nb)])
    total = int(offsets[-1])
    print("corpus: %d utterances, %d samples, %d stride-1 frames (%.3g FLOP at 2 x 21.0 MMAC per frame)"
          % (lengths.size, int(lengths.sum()), total, total * 2 * 21.0e6))

    # 1. per-utterance calls
    looped = np.empty((total, 2), np.float32)
    starts = np.concatenate([[0], np.cumsum(lengths)])

    def loop():
        for u in range(lengths.size):
            looped[offsets[u]:offsets[u + 1]] = api.cnn_evaluate(flat[starts[u]:starts[u + 1]], co, model, LPF, CUTOFF,
                                                                 with_envelopes=False)[0]

    for u in range(3):
        api.cnn_evaluate(flat[starts[u]:starts[u + 1]], co, model, LPF, CUTOFF, with_envelopes=False)
    t_loop = []
    for _ in range(args.reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        loop()
        t_loop.append(time.perf_counter() - t)
    print("1. loop of cnn_evaluate:              ", stats(t_loop))

    # 2. one call on one GPU
    one = np.empty((total, 2), np.float32)
    api.cnn_evaluate_corpus((wave_host[:int(lengths[:16].sum())], lengths[:16]), co, model, LPF, CUTOFF)
    t_one = []
    for _ in range(args.reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        api.cnn_evaluate_corpus((wave_host, lengths), co, model, LPF, CUTOFF, out=one)
        t_one.append(time.perf_counter() - t)
    print("2. cnn_evaluate_corpus, 1 GPU:        ", stats(t_one))
    same = sum(np.array_equal(one[offsets[u]:offsets[u + 1]], looped[offsets[u]:offsets[u + 1]]) for u in range(lengths.size))
    print("   against the loop: %d of %d utterances bit for bit, max |difference| %.3g"
          % (same, lengths.size, float(np.abs(one - looped).max()) if total else 0.0))
    print("   per GPU: %.1f frames/us, %.0f TFLOP/s of useful work" % (total / np.median(t_one) / 1e6,
                                                                      total * 2 * 21.0e6 / np.median(t_one) / 1e12))

    # 3. sharded over every visible GPU, one process each
    world = torch.cuda.device_count()
    if world < 2:
        # what one rank of a W-GPU run computes, alone on this GPU: the W-GPU run itself is not measured here
        print("3. sharded: 1 visible GPU; rank 0's share of a W-GPU run, timed alone on this GPU:")
        part = np.empty((total, 2), np.float32)
        for w in (2, 4, 8):
            t_w = []
            for _ in range(args.reps):
                torch.cuda.synchronize()
                t = time.perf_counter()
                api.cnn_evaluate_corpus((wave_host, lengths), co, model, LPF, CUTOFF, out=part, shard=(0, w))
                t_w.append(time.perf_counter() - t)
            mine = np.repeat(np.isin(np.arange(lengths.size), engine.shard_utterances(lengths, w)[0]), nb)
            assert np.array_equal(part[mine], one[mine]), "shard (0, %d) differs from the 1-GPU call" % w
            print("   W = %d: %s, 1-GPU time / W = %.3f s; rows equal the 1-GPU call bit for bit"
                  % (w, stats(t_w), np.median(t_one) / w))
    else:
        with tempfile.TemporaryDirectory(dir=hostmem.shm_dir()) as d:
            path = os.path.join(d, "scores.f32")
            shared = hostmem.SharedArray(path, (total, 2), np.float32, create=True)
            ctx = mp.get_context("spawn")
            barrier, q = ctx.Barrier(world + 1, timeout=900), ctx.Queue()
            procs = [ctx.Process(target=rank_main, args=(r, world, args.utts, path, total, args.reps, barrier, q))
                     for r in range(world)]
            for p in procs:
                p.start()
            t_sh = []
            try:
                for _ in range(args.reps):
                    barrier.wait()
                    marks = [q.get(timeout=600) for _ in range(world)]
                    t_sh.append(max(m[2] for m in marks) - min(m[1] for m in marks))
                barrier.wait()
                for p in procs:
                    p.join(timeout=120)
            finally:
                for p in procs:     # no rank stays behind on its GPU, whatever happened above
                    if p.is_alive():
                        p.kill()
                        p.join()
            assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
            print("3. cnn_evaluate_corpus, %d GPUs:       " % world, stats(t_sh))
            print("   speedup over 1 GPU: %.2f, over the loop: %.2f" % (np.median(t_one) / np.median(t_sh),
                                                                        np.median(t_loop) / np.median(t_sh)))
            assert np.array_equal(shared.array, one), "sharded scores differ from the 1-GPU call"
            print("   sharded scores == 1-GPU scores bit for bit")
    print("cards:\n" + cards())


if __name__ == "__main__":
    main()
