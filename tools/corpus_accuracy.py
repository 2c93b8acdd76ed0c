"""The reference's label accuracy of every utterance of a labelled corpus, on the GPU: api.cnn_label_accuracy_corpus.

The bench's seed-1 corpus (4620 utterances of U(32000, 64000) int16 samples, or its first --utts), LPF at 50 Hz,
seeded weights with the output bias centred (centred_model); labels per utterance: a seeded sorted subset (about
half) of synth.label_grid with random classes, as ExtractLabel would keep them.  Host clock around calls that end with their results on the host.
  1. cnn_label_accuracy_corpus against cnn_evaluate_corpus alone, alternated: what counting on the device adds,
     and what it saves against bringing the scores back (with_scores=True is timed as well);
  2. the corpus clean and at SNRdB = 0 / 10 / 20: Evaluating.MixNoise per utterance on the host (numpy.random
     seeded, on the float64 samples) into one float64 flat buffer, then one cnn_label_accuracy_corpus call; corpus
     accuracy sum(hits) / sum(counted).  MixNoise's sigma is RMS / 10^(SNRdB/10), the reference's power ratio
     applied to an amplitude: a true SNR of 0 / 20 / 40 dB;
  3. the host restatement Evaluating._label_accuracy on 20 utterances of the clean scores, timed, and asserted
     equal to hits / counted of the device counters (ZeroDivisionError where counted is 0).
Prints the card's name and power limit with the numbers and writes everything to --log as well.
Usage: python tools/corpus_accuracy.py [--utts N] [--reps R] [--log PATH]"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

LPF, CUTOFF, SEED_MODEL, SEED_LABELS, STEP = True, 50, 0, 3, 160
_lines = []


def say(*parts):
    line = " ".join(str(p) for p in parts)
    print(line, flush=True)
    _lines.append(line)


def cards():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "nvidia-smi unavailable"


def corpus(n_utts):
    from f2cnn_b200 import synth
    lengths = synth.corpus_lengths(4620, 32000, 64000, seed=1)
    flat, _ = synth.corpus_waves_i16(lengths, seed=1)
    return flat[:int(lengths[:n_utts].sum())], lengths[:n_utts]


def labels_for(lengths):
    from f2cnn_b200 import synth
    rng = np.random.default_rng(SEED_LABELS)
    times = [g[rng.random(g.size) < 0.5] for g in (synth.label_grid(int(n)) for n in lengths)]
    counts = np.asarray([t.size for t in times], dtype=np.int64)
    times = np.concatenate(times)
    return times, rng.integers(0, 2, times.size).astype(np.int32), counts


def centred_model(wave_host, lengths, co):
    """Seeded weights whose output bias is moved so that the median frame of the first 16 utterances sits on the
    decision boundary: the seeded network alone decides 0 (falling) on every frame, which no noise would change."""
    import torch
    from f2cnn_b200 import api, cnn
    model = cnn.seeded_model(SEED_MODEL)
    for _ in range(2):      # a second pass where float32 softmax scores saturated in the first
        sc, _ = api.cnn_evaluate_corpus((wave_host[:int(lengths[:16].sum())], lengths[:16]), co, model, LPF, CUTOFF)
        logit = np.log(np.maximum(sc.astype(np.float64), 1e-300))
        with torch.no_grad():
            model.d2.bias[1] -= float(np.median(logit[:, 1] - logit[:, 0]))
    return model


def stats(v):
    v = np.asarray(v)
    return "median %.3f  min %.3f  max %.3f s (n=%d)" % (np.median(v), v.min(), v.max(), v.size)


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    return time.perf_counter() - t, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=4620)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--log", default=os.path.join(ROOT, "profiles", "r03f_corpus_accuracy.log"))
    args = ap.parse_args()
    import torch
    from f2cnn_b200 import api
    from f2cnn_b200.gammatone import filters
    from f2cnn_b200.scripts.CNN import Evaluating
    say("cards:\n" + cards())
    flat, lengths = corpus(args.utts)
    wave_host = torch.from_numpy(flat).pin_memory()
    co = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))
    model = centred_model(wave_host, lengths, co)
    labels = labels_for(lengths)
    times, classes, counts = labels
    nb = np.maximum(lengths - 11 * STEP, 0)
    say("corpus: %d utterances, %d samples, %d stride-1 frames, %d labels (%.0f per utterance)"
        % (lengths.size, int(lengths.sum()), int(nb.sum()), times.size, times.size / max(lengths.size, 1)))

    # warm-up on a few utterances: plan, network, pinned staging
    head = int(lengths[:16].sum()), lengths[:16]
    api.cnn_label_accuracy_corpus((wave_host[:head[0]], head[1]), co, model,
                                  (times[:int(counts[:16].sum())], classes[:int(counts[:16].sum())], counts[:16]),
                                  LPF, CUTOFF)
    api.cnn_evaluate_corpus((wave_host[:head[0]], head[1]), co, model, LPF, CUTOFF)

    # 1. counting on the device against scoring alone, alternated
    t_acc, t_eval = [], []
    scores = np.empty((int(nb.sum()), 2), np.float32)
    for _ in range(args.reps):
        t, (hits, counted) = timed(lambda: api.cnn_label_accuracy_corpus((wave_host, lengths), co, model, labels,
                                                                         LPF, CUTOFF))
        t_acc.append(t)
        t, _ = timed(lambda: api.cnn_evaluate_corpus((wave_host, lengths), co, model, LPF, CUTOFF, out=scores))
        t_eval.append(t)
    say("1. cnn_label_accuracy_corpus (2 x %d int64 back):  %s" % (lengths.size, stats(t_acc)))
    say("   cnn_evaluate_corpus alone (%.2f GB of scores back): %s" % (scores.nbytes / 1e9, stats(t_eval)))
    t_ws, (h_ws, c_ws, sc_ws, off) = timed(lambda: api.cnn_label_accuracy_corpus((wave_host, lengths), co, model,
                                                                                labels, LPF, CUTOFF, with_scores=True))
    say("   cnn_label_accuracy_corpus, with_scores=True:      %.3f s" % t_ws)
    assert np.array_equal(sc_ws, scores), "with_scores differs from cnn_evaluate_corpus"
    assert np.array_equal(h_ws, hits) and np.array_equal(c_ws, counted)
    say("   with_scores: scores equal cnn_evaluate_corpus bit for bit, counters equal the call without scores")

    # 2. accuracy clean and at 0 / 10 / 20 dB
    def report(name, h, c, t, extra=""):
        say("2. %-8s corpus accuracy %.6f (%d / %d counted frames), %d utterances with nothing counted; "
            "call %.3f s%s" % (name, h.sum() / max(int(c.sum()), 1), int(h.sum()), int(c.sum()), int((c == 0).sum()), t,
                               extra))

    say("   seeded, untrained weights (output bias centred, centred_model) and random classes: the accuracy says nothing "
        "about a network; the clean scores decide 1 (rising) on %d of %d frames"
        % (int((sc_ws[:, 1] > sc_ws[:, 0]).sum()), sc_ws.shape[0]))
    report("clean", hits, counted, float(np.median(t_acc)))
    starts = np.concatenate([[0], np.cumsum(lengths)])
    noisy = np.empty(int(lengths.sum()), np.float64)
    for snr in (0, 10, 20):
        np.random.seed(1000 + snr)
        t0 = time.perf_counter()
        for u in range(lengths.size):
            # float64 samples: on int16 ones the reference's RMS squares wrap around (often a NaN sigma)
            noisy[starts[u]:starts[u + 1]] = Evaluating.MixNoise(flat[starts[u]:starts[u + 1]].astype(np.float64), snr)
        t_mix = time.perf_counter() - t0
        t, (h, c) = timed(lambda: api.cnn_label_accuracy_corpus((noisy, lengths), co, model, labels, LPF, CUTOFF))
        report("SNRdB=%d" % snr, h, c, t, " (MixNoise on the host %.1f s)" % t_mix)

    # 3. the host restatement on 20 utterances, and the counters against it
    pick = np.linspace(0, lengths.size - 1, min(20, lengths.size)).astype(int)
    loff = np.concatenate([[0], np.cumsum(counts)])
    t_host, frames_host = 0.0, 0
    for u in pick:
        lab = list(zip(times[loff[u]:loff[u + 1]].tolist(), classes[loff[u]:loff[u + 1]].tolist()))
        sc = sc_ws[off[u]:off[u + 1]]
        t0 = time.perf_counter()
        try:
            ref = Evaluating._label_accuracy(lab, Evaluating._decisions(sc), STEP)
        except ZeroDivisionError:
            ref = None
        t_host += time.perf_counter() - t0
        frames_host += sc.shape[0]
        assert ref == (hits[u] / counted[u] if counted[u] else None), "utterance %d: %r vs %d / %d" % (
            u, ref, hits[u], counted[u])
    say("3. Evaluating._label_accuracy on %d utterances (%d frames, %d labels): %.2f s, %.3f s per utterance; "
        "the device counters give the same accuracy on every one"
        % (pick.size, frames_host, int(counts[pick].sum()), t_host, t_host / pick.size))
    say("   at that rate the %d utterances would take %.0f s on this host" % (lengths.size,
                                                                            t_host / pick.size * lengths.size))
    say("cards:\n" + cards())
    os.makedirs(os.path.dirname(os.path.abspath(args.log)), exist_ok=True)
    with open(args.log, "w") as f:
        f.write("# python tools/corpus_accuracy.py --utts %d --reps %d\n" % (args.utts, args.reps))
        f.write("\n".join(_lines) + "\n")


if __name__ == "__main__":
    main()
