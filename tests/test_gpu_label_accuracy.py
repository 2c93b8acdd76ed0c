"""The label accuracy of `cnn eval*` on the GPU (f2_label_accuracy, engine.label_accuracy, api.label_accuracy,
api.cnn_label_accuracy_corpus, Evaluating.EvaluateOneWavArray).

The counts are integers, so the bar is equality with what the reference's rule implies.  The rule is the host
restatement Evaluating._label_accuracy, unchanged: it is handed decisions that record each comparison it makes,
so the number of comparisons is `counted` and the number that came out true is `hits` (it returns only their
ratio, and raises ZeroDivisionError when nothing is counted)."""
import os
import sys
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
STEP = 160
DOTS = 11


class _Decision:
    """A 0/1 decision that logs every comparison _label_accuracy makes with a target class."""

    def __init__(self, value, log):
        self.value, self.log = value, log

    def __eq__(self, target):
        hit = self.value == target
        self.log.append(bool(hit))
        return hit


def _reference_counts(labels, scores, step):
    from f2cnn_b200.scripts.CNN.Evaluating import _decisions, _label_accuracy
    log = []
    decisions = [_Decision(d, log) for d in _decisions(scores)]
    try:
        ratio = _label_accuracy(labels, decisions, step)
    except ZeroDivisionError:
        ratio = None
    hits, counted = sum(log), len(log)
    assert ratio == (hits / counted if counted else None)
    return hits, counted


def _scores(rng, nf):
    """Random float32 scores with some rows of equal scores and some NaN (both decide 0)."""
    s = rng.random((nf, 2)).astype(np.float32)
    if nf:
        eq = rng.random(nf) < 0.1
        s[eq, 1] = s[eq, 0]
        s[rng.random(nf) < 0.05, rng.integers(0, 2)] = np.nan
    return s


def _labels(rng, nf, step, kind):
    """(time, class) pairs, times non-decreasing, of one kind of the cases the kernel has to get right."""
    if kind == "none":
        t = np.zeros(0, np.int64)
    elif kind == "single":
        t = rng.integers(-5, nf + 5, 1)
    elif kind == "duplicates":
        # beyond both ends as well, and repeated times (an empty interval)
        t = np.sort(rng.integers(-3 * step, nf + 3 * step, int(rng.integers(2, 40))))
        t = np.sort(np.concatenate([t, t[rng.integers(0, t.size, 4)]]))
    elif kind == "gaps":
        # gaps of at least 2*step: frames far from both ends of an interval are not counted
        t = -step + np.cumsum(rng.integers(2 * step, 4 * step + 1, int(rng.integers(2, 12))))
    else:
        # equidistant frames: even gaps of up to 2*step put a frame at distance < step from both ends
        t = -3 + np.cumsum(2 * rng.integers(1, step + 1, int(rng.integers(2, 30))))
    return [(int(a), int(c)) for a, c in zip(t, rng.integers(0, 2, t.size))]


FRAMES = (0, 1, 2, 31, 32, 33, 63, 255, 256, 257, 2047, 2048, 2049, 5000)
KINDS = ("none", "single", "duplicates", "gaps", "ties")


@pytest.mark.parametrize("step", [1, 2, 160])
def test_ragged_utterances_in_one_launch_count_what_the_reference_counts(step):
    import torch
    from f2cnn_b200 import api, engine
    rng = np.random.default_rng(100 + step)
    utts = []
    for nf in FRAMES:
        for kind in KINDS:
            utts.append((_scores(rng, nf), _labels(rng, nf, step, kind)))
    order = rng.permutation(len(utts))
    utts = [utts[i] for i in order]
    want = np.asarray([_reference_counts(lab, sc, step) for sc, lab in utts], dtype=np.int64)
    assert want[:, 1].sum() > 0 or step == 1      # step 1: no frame lies strictly inside and closer than 1

    score_off = np.concatenate([[0], np.cumsum([sc.shape[0] for sc, _ in utts])]).astype(np.int64)
    label_off = np.concatenate([[0], np.cumsum([len(lab) for _, lab in utts])]).astype(np.int64)
    times = np.asarray([t for _, lab in utts for t, _ in lab], dtype=np.int64)
    classes = np.asarray([c for _, lab in utts for _, c in lab], dtype=np.int32)
    dev = torch.device("cuda")
    scores = torch.from_numpy(np.concatenate([sc for sc, _ in utts])).to(dev)
    got = engine.label_accuracy(scores, torch.from_numpy(score_off).to(dev), torch.from_numpy(times).to(dev),
                                torch.from_numpy(classes).to(dev), torch.from_numpy(label_off).to(dev), step)
    assert got.dtype == torch.int64 and got.shape == (2, len(utts))
    assert np.array_equal(got.cpu().numpy().T, want)

    # one utterance at a time through the public call: host float32, device tensor, host float64
    for (sc, lab), w in zip(utts, want):
        assert api.label_accuracy(sc, lab, step) == tuple(w)
        assert api.label_accuracy(torch.from_numpy(sc).to(dev), lab, step) == tuple(w)
        assert api.label_accuracy(sc.astype(np.float64), lab, step) == tuple(w)


def test_float64_scores_keep_their_own_decisions():
    """Two float64 scores that round to the same float32 still decide 1 when the second is larger, as the
    reference's comparison of the Keras output does."""
    from f2cnn_b200 import api
    s = np.full((600, 2), 0.5)
    s[:, 1] += 1e-12
    s[::3, 1] = 0.5 - 1e-12
    labels = [(100, 1), (300, 1), (400, 1)]
    want = _reference_counts(labels, s, STEP)
    assert api.label_accuracy(s, labels, STEP) == want
    assert want[0] not in (0, want[1])
    assert api.label_accuracy(s.astype(np.float32), labels, STEP) == (0, want[1])   # float32 ties decide 0


def test_more_frames_than_the_grid_holds():
    """A launch larger than one pass of the grid (148 SMs x 8 CTAs x 256 threads on a B200) counts every frame
    once: the utterances in one launch equal the utterances one at a time."""
    import torch
    from f2cnn_b200 import api, engine
    rng = np.random.default_rng(7)
    dev = torch.device("cuda")
    nfs = rng.integers(20000, 40000, 40)
    utts = [(_scores(rng, int(nf)), _labels(rng, int(nf), STEP, "ties" if u % 2 else "duplicates"))
            for u, nf in enumerate(nfs)]
    for u in (0, 1, 39):
        assert api.label_accuracy(*utts[u], STEP) == _reference_counts(utts[u][1], utts[u][0], STEP)
    one = np.asarray([api.label_accuracy(sc, lab, STEP) for sc, lab in utts])
    score_off = np.concatenate([[0], np.cumsum(nfs)]).astype(np.int64)
    label_off = np.concatenate([[0], np.cumsum([len(lab) for _, lab in utts])]).astype(np.int64)
    got = engine.label_accuracy(torch.from_numpy(np.concatenate([sc for sc, _ in utts])).to(dev),
                                torch.from_numpy(score_off).to(dev),
                                torch.tensor([t for _, lab in utts for t, _ in lab], dtype=torch.int64, device=dev),
                                torch.tensor([c for _, lab in utts for _, c in lab], dtype=torch.int32, device=dev),
                                torch.from_numpy(label_off).to(dev), STEP)
    assert int(score_off[-1]) > torch.cuda.get_device_properties(dev).multi_processor_count * 8 * 256
    assert np.array_equal(got.cpu().numpy().T, one) and one[:, 1].sum() > 0


def test_abi_rejects_bad_arguments():
    import ctypes
    import torch
    from f2cnn_b200 import _native
    L = _native.lib()
    buf = torch.zeros(64, dtype=torch.int64, device="cuda")
    p = ctypes.c_void_p(buf.data_ptr())
    odd = ctypes.c_void_p(buf.data_ptr() + 4)
    null = ctypes.c_void_p(0)
    assert L.f2_label_accuracy(p, p, p, p, p, 0, STEP, p, p, None) == _native.F2_OK        # nothing to count
    assert L.f2_label_accuracy(p, p, p, p, p, -1, STEP, p, p, None) == _native.F2_ERR_INVALID
    assert L.f2_label_accuracy(p, p, p, p, p, 1, 0, p, p, None) == _native.F2_ERR_INVALID
    assert L.f2_label_accuracy(odd, p, p, p, p, 1, STEP, p, p, None) == _native.F2_ERR_INVALID
    for k in range(7):
        args = [p, p, p, p, p, 1, STEP, p, p]
        args[k if k < 5 else k + 2] = null
        assert L.f2_label_accuracy(*args, None) == _native.F2_ERR_INVALID, k


# ---- the corpus call -------------------------------------------------------------------------------------------

def _coefs():
    from f2cnn_b200.gammatone import filters
    return filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))


def _wave(n, seed):
    """A speech-like int16 utterance with a little noise (no stretch of exact zeros)."""
    from f2cnn_b200 import synth
    rng = np.random.default_rng(seed + 7)
    w = (synth.speech_like_i16(n, seed=seed).astype(np.int32) + rng.integers(-40, 41, n)).clip(-32768, 32767)
    return np.where(w == 0, 1, w).astype(np.int16)


# frames per utterance: 0, 1 and 2 between longer ones
LENGTHS = [9000, DOTS * STEP, DOTS * STEP + 1, 20000, DOTS * STEP + 2, 30000, 5000, 14000]


def _corpus_labels(lengths, seed):
    """Per utterance a seeded sorted subset of the label grid (with repeats) and a few times outside the frames,
    random classes; flattened as (times, classes, counts)."""
    from f2cnn_b200 import synth
    rng = np.random.default_rng(seed)
    times, counts = [], []
    for n in lengths:
        grid = synth.label_grid(int(n))
        t = rng.choice(grid, size=min(grid.size, 25)) if grid.size else np.zeros(0, np.int64)
        t = np.sort(np.concatenate([t, rng.integers(-400, max(int(n) - DOTS * STEP, 0) + 400, 3)]))
        times.append(t)
        counts.append(t.size)
    times = np.concatenate(times)
    return times, rng.integers(0, 2, times.size).astype(np.int32), np.asarray(counts)


@pytest.fixture(scope="module")
def corpus():
    from f2cnn_b200 import api, cnn
    model = cnn.seeded_model(seed=3)
    waves = [_wave(n, 600 + i) for i, n in enumerate(LENGTHS)]
    labels = _corpus_labels(LENGTHS, 11)
    scores, offsets = api.cnn_evaluate_corpus(waves, _coefs(), model, LPF=True, CUTOFF=50)
    return model, waves, labels, scores, offsets


def test_corpus_counts_equal_the_reference_on_the_corpus_scores(corpus):
    from f2cnn_b200 import api
    model, waves, labels, scores, offsets = corpus
    times, classes, counts = labels
    loff = np.concatenate([[0], np.cumsum(counts)])
    want = np.asarray([_reference_counts(list(zip(times[loff[u]:loff[u + 1]].tolist(),
                                                  classes[loff[u]:loff[u + 1]].tolist())),
                                         scores[offsets[u]:offsets[u + 1]], STEP) for u in range(len(LENGTHS))])
    assert want[:, 1].sum() > 0 and want[1, 1] == 0            # utterance 1 has no frame
    hits, counted, got_scores, got_offsets = api.cnn_label_accuracy_corpus(waves, _coefs(), model, labels, LPF=True,
                                                                          CUTOFF=50, with_scores=True)
    assert hits.dtype == counted.dtype == np.int64
    assert np.array_equal(np.stack([hits, counted], 1), want)
    assert np.array_equal(got_scores, scores) and np.array_equal(got_offsets, offsets)
    # (flat, lengths) input, without scores
    flat = np.concatenate(waves)
    h2, c2 = api.cnn_label_accuracy_corpus((flat, np.asarray(LENGTHS)), _coefs(), model, labels, True, 50)
    assert np.array_equal(h2, hits) and np.array_equal(c2, counted)


def test_corpus_counts_do_not_depend_on_sub_batches_or_shards(corpus, monkeypatch):
    from f2cnn_b200 import api
    model, waves, labels, scores, offsets = corpus
    whole = api.cnn_label_accuracy_corpus(waves, _coefs(), model, labels, True, 50)
    monkeypatch.setattr(api, "_CNN_ENV_BYTES", 25000 * 128 * 4)    # one to three utterances per sub-batch
    split = api.cnn_label_accuracy_corpus(waves, _coefs(), model, labels, True, 50, with_scores=True)
    assert np.array_equal(split[0], whole[0]) and np.array_equal(split[1], whole[1])
    assert np.array_equal(split[2], scores)
    shared = (np.full(len(LENGTHS), -1, np.int64), np.full(len(LENGTHS), -1, np.int64))
    for rank in range(2):
        out = api.cnn_label_accuracy_corpus(waves, _coefs(), model, labels, True, 50, out=shared, shard=(rank, 2))
        assert out[0] is shared[0] and out[1] is shared[1]
    assert np.array_equal(shared[0], whole[0]) and np.array_equal(shared[1], whole[1])


# ---- the drop-in -----------------------------------------------------------------------------------------------

def _conf(channels):
    return ("[FILTERBANK]\nFRAMERATE=16000\nNCHANNELS=%d\nLOW_FREQ=100\n"
            "[CNN]\nFORMANT=2\nCENTERED=True\nRADIUS=5\nBATCH_SIZE=32\nEPOCHS=20\nRISK=0.05\nSAMPLING_PERIOD=10000\n"
            % channels)


@pytest.fixture()
def evaluating(tmp_path, monkeypatch):
    """A tree with one labelled utterance, the reference's figure replaced by a recorder; returns (module, wave,
    path, what the figure received)."""
    from scipy.io import wavfile
    from f2cnn_b200 import dropin, synth
    monkeypatch.chdir(tmp_path)
    d = tmp_path / "resources" / "f2cnn" / "TEST"
    d.mkdir(parents=True)
    n = 7000
    w = synth.speech_like_i16(n, seed=n)
    wav = str(d / "DR1.SPK2.SI3.WAV")
    wavfile.write(wav, 16000, w)
    synth.write_fb(str(d / "DR1.SPK2.SI3.FB"), synth.formant_tracks_khz(n // 160 + 3, seed=n))
    synth.write_phn(str(d / "DR1.SPK2.SI3.PHN"), synth.phoneme_segments(n, seed=n))
    seen = {}
    dropin.install()
    try:
        for name, attrs in {"scripts.plotting": {}, "scripts.plotting.PlottingCNN": dict(
                PlotEnvelopesAndCNNResultsWithPhonemes=lambda *a: seen.update(plot=a))}.items():
            m = types.ModuleType(name)
            m.__dict__.update(attrs)
            if not attrs:
                m.__path__ = []
            monkeypatch.setitem(sys.modules, name, m)
        from scripts.CNN import Evaluating
        yield Evaluating, w, wav, seen
    finally:
        dropin.uninstall()


def _expected_accuracy(Evaluating, wav, scores):
    from configparser import ConfigParser
    from f2cnn_b200.scripts.processing.LabelDataGenerator import ExtractLabel
    cfg = ConfigParser()
    cfg.read("configF2CNN.conf")
    rows = ExtractLabel(wav, cfg)
    assert rows, "the fixture should give labels"
    labels = [(r[-4], r[-1]) for r in rows]
    return Evaluating._label_accuracy(labels, Evaluating._decisions(scores), STEP), labels


def test_evaluate_one_wav_array_plots_the_reference_accuracy_tensor_cores(evaluating, tmp_path, monkeypatch):
    from f2cnn_b200 import cnn
    Evaluating, w, wav, seen = evaluating
    (tmp_path / "configF2CNN.conf").write_text(_conf(128))
    cnn.save_weights(str(tmp_path / "model.npz"), cnn.seeded_model(seed=2))
    Evaluating.EvaluateOneWavArray(w, 16000, wav, model=str(tmp_path / "model.npz"))
    scores, acc = seen["plot"][1], seen["plot"][2]
    assert scores.shape == (len(w) - DOTS * STEP, 2)
    want, labels = _expected_accuracy(Evaluating, wav, scores)
    assert isinstance(acc, float) and acc == want

    # no labels: None; labels no frame lies between: the reference's ZeroDivisionError
    from f2cnn_b200.scripts.processing import LabelDataGenerator
    monkeypatch.setattr(LabelDataGenerator, "ExtractLabel", lambda *a: None)
    Evaluating.EvaluateOneWavArray(w, 16000, wav, model=str(tmp_path / "model.npz"))
    assert seen["plot"][2] is None
    row = ["TEST", "DR1", "SPK2", "SI3", "aa"]
    monkeypatch.setattr(LabelDataGenerator, "ExtractLabel",
                        lambda *a: [row + [800, 0.1, 0.01, 1], row + [801, -0.1, 0.01, 0]])
    with pytest.raises(ZeroDivisionError):
        Evaluating.EvaluateOneWavArray(w, 16000, wav, model=str(tmp_path / "model.npz"))


def test_evaluate_one_wav_array_plots_the_reference_accuracy_keras(evaluating, tmp_path, monkeypatch):
    """The Keras branch (a geometry the tensor cores are not built for): float64 scores, some of them pairs that
    float32 could not tell apart, and some equal."""
    Evaluating, w, wav, seen = evaluating
    (tmp_path / "configF2CNN.conf").write_text(_conf(32))
    rng = np.random.default_rng(5)

    class _Net:
        def predict(self, x, verbose=0):
            s = rng.random((x.shape[0], 2))
            s[::4, 1] = s[::4, 0] + 1e-13
            s[1::4, 1] = s[1::4, 0]
            return s

    keras = types.ModuleType("keras")
    keras.models = types.SimpleNamespace(load_model=lambda name: _Net())
    keras.backend = types.SimpleNamespace(clear_session=lambda: None)
    monkeypatch.setitem(sys.modules, "keras", keras)
    Evaluating.EvaluateOneWavArray(w, 16000, wav)
    scores, acc = seen["plot"][1], seen["plot"][2]
    assert scores.dtype == np.float64
    want, _ = _expected_accuracy(Evaluating, wav, scores)
    assert acc == want
