"""api.label_accuracy and api.cnn_label_accuracy_corpus refuse malformed labels and arguments with ValueError
before anything reaches the device (no GPU needed: a launch would fail here)."""
import numpy as np
import pytest


class _Launched(Exception):
    pass


def _no_launch(*a, **k):
    raise _Launched()


@pytest.fixture()
def api(monkeypatch):
    import torch
    from f2cnn_b200 import api, engine
    monkeypatch.setattr(engine, "plan_for", _no_launch)
    monkeypatch.setattr(engine, "label_accuracy", _no_launch)
    monkeypatch.setattr(api, "_to_device", _no_launch)
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)   # naming a device is not a launch
    return api


WAVES = [np.ones(4000, np.int16), np.ones(5000, np.int16)]
COEFS = np.zeros((128, 10))
# times may fall from one utterance to the next, not within one
GOOD = (np.array([10, 20, 5, 9]), np.array([0, 1, 1, 0]), np.array([2, 2]))


@pytest.mark.parametrize("labels, match", [
    ((np.array([20, 10, 5, 9]), GOOD[1], GOOD[2]), "utterance 0 decrease"),
    ((np.array([10, 20, 9, 5]), GOOD[1], GOOD[2]), "utterance 1 decrease"),
    ((GOOD[0], GOOD[1], np.array([2, 1])), "counts"),
    ((GOOD[0], GOOD[1], np.array([4])), "counts"),
    ((GOOD[0], GOOD[1], np.array([5, -1])), "counts"),
    ((GOOD[0], GOOD[1][:3], GOOD[2]), "4 label times, 3 classes"),
    ((np.array([10.5, 20, 5, 9]), GOOD[1], GOOD[2]), "times must be integers"),
    ((GOOD[0], np.array([0, 1, 2 ** 31, 0]), GOOD[2]), "classes must be integers"),
    ((GOOD[0], np.array([0, np.nan, 1, 0]), GOOD[2]), "classes must be integers"),
])
def test_corpus_labels_are_checked_before_any_launch(api, labels, match):
    with pytest.raises(ValueError, match=match):
        api.cnn_label_accuracy_corpus(WAVES, COEFS, None, labels)
    with pytest.raises(_Launched):       # well-formed labels get as far as the device
        api.cnn_label_accuracy_corpus(WAVES, COEFS, None, GOOD)
    # integral floats are integers
    with pytest.raises(_Launched):
        api.cnn_label_accuracy_corpus(WAVES, COEFS, None, tuple(a.astype(np.float64) for a in GOOD))


def test_corpus_arguments_are_checked_before_any_launch(api):
    with pytest.raises(ValueError, match="RADIUS = 5 and 128"):
        api.cnn_label_accuracy_corpus(WAVES, COEFS, None, GOOD, radius=4)
    with pytest.raises(ValueError, match="RADIUS = 5 and 128"):
        api.cnn_label_accuracy_corpus(WAVES, COEFS[:64], None, GOOD)
    with pytest.raises(ValueError, match="shared `out`"):
        api.cnn_label_accuracy_corpus(WAVES, COEFS, None, GOOD, shard=(0, 2))
    with pytest.raises(ValueError, match="with_scores"):
        api.cnn_label_accuracy_corpus(WAVES, COEFS, None, GOOD, shard=(0, 2), with_scores=True,
                                      out=(np.zeros(2, np.int64), np.zeros(2, np.int64)))
    with pytest.raises(ValueError, match="int64"):
        api.cnn_label_accuracy_corpus(WAVES, COEFS, None, GOOD, out=(np.zeros(2, np.int32), np.zeros(2, np.int64)))
    with pytest.raises(ValueError, match="int64"):
        api.cnn_label_accuracy_corpus(WAVES, COEFS, None, GOOD, out=(np.zeros(3, np.int64), np.zeros(3, np.int64)))
    with pytest.raises(ValueError, match=r"\(times, classes, counts\)"):
        api.cnn_label_accuracy_corpus(WAVES, COEFS, None, GOOD[:2])
    with pytest.raises(_Launched):
        api.cnn_label_accuracy_corpus(WAVES, COEFS, None, GOOD, out=(np.zeros(2, np.int64), np.zeros(2, np.int64)),
                                      shard=(1, 2))


def test_one_utterance_is_checked_before_any_launch(api):
    scores = np.zeros((50, 2), np.float32)
    with pytest.raises(ValueError, match="decrease"):
        api.label_accuracy(scores, [(10, 1), (30, 0), (20, 1)])
    with pytest.raises(ValueError, match="integers"):
        api.label_accuracy(scores, [(10, 1), (30.5, 0)])
    with pytest.raises(ValueError, match=r"\(F, 2\)"):
        api.label_accuracy(np.zeros((50, 3), np.float32), [(10, 1), (30, 0)])
    with pytest.raises(ValueError, match=r"\(F, 2\)"):
        api.label_accuracy(np.zeros(50, np.float32), [(10, 1), (30, 0)])
    for labels in ([(10, 1), (30, 0)], [(10, 1), (10, 0)], [(5, 1)], []):
        with pytest.raises(_Launched):
            api.label_accuracy(scores, labels)
