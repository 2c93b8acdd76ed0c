"""Host-only checks of the per-group float32 prediction that chooses the float64 (FORM 2) channel groups:
f2_bank_check_groups flags exactly the banks f2_bank_check refuses, and the group holding the refused
channel.  No device is needed."""
import numpy as np
import pytest

from f2cnn_b200 import _native, engine
from f2cnn_b200.gammatone import filters

# tools/fuzz_parity.py 120 7: the banks f2_bank_check refuses (profiles/r02z_fuzz.log)
REFUSED_FUZZ_CASES = [10, 12, 13, 19, 20, 22, 26, 29, 32, 35, 39, 45, 48, 57, 60, 65, 72, 75, 77, 82, 84, 93, 97,
                      109, 113, 114, 118]


def fuzz_cases(cases=120, seed=7):
    """The parameters tools/fuzz_parity.py draws, with the same generator calls in the same order."""
    rng = np.random.default_rng(seed)
    out = []
    for case in range(cases):
        fs = int(rng.choice([8000, 16000, 16000, 22050, 44100]))
        C = int(rng.choice([1, 7, 32, 40, 64, 96, 128, 160, 256]))
        low = int(rng.choice([20, 50, 100, 100, 300]))
        width = float(rng.choice([1.0, 1.0, 0.5, 2.0]))
        n = int(rng.choice([300, 1000, 4096, 8191, 20000, 48000, 65536, 65537, 100000])) + int(rng.integers(0, 50))
        kind = str(rng.choice(["white", "speech", "tone", "chirp"]))
        freq = float(rng.choice([low, 2 * low, 440.0, 1000.0, fs / 4.0])) if kind == "tone" else None
        dtype = [np.int16, np.float32, np.float64][int(rng.integers(0, 3))]
        lpf = bool(rng.random() < 0.7)
        cutoff = float(rng.choice([20, 50, 100, 400]))
        step = int(rng.choice([160, 80, 441]))
        target = int(rng.choice([0, 0, 1, 64]))
        out.append(dict(case=case, fs=fs, C=C, low=low, width=width, n=n, kind=kind, freq=freq, dtype=dtype, lpf=lpf,
                        cutoff=cutoff, step=step, target=target))
    return out


def bank(p):
    return filters.make_erb_filters(p["fs"], filters.centre_freqs(p["fs"], p["C"], p["low"]), p["width"])


def test_groups_flagged_exactly_where_the_bank_check_refuses():
    refused, flagged = [], []
    for p in fuzz_cases():
        co = bank(p)
        pred, worst = engine.bank_check(co)
        groups = engine.bank_check_groups(co)
        assert groups.shape == ((p["C"] + 31) // 32,)
        assert np.all(np.isfinite(groups)) and np.all(groups >= 0.0)
        if pred > 1.0:
            refused.append(p["case"])
            assert groups[worst // 32] > 1.0, (p, groups, worst)
        if np.any(groups > 1.0):
            flagged.append(p["case"])
    assert refused == REFUSED_FUZZ_CASES
    assert flagged == REFUSED_FUZZ_CASES


def test_configured_banks_flag_no_group():
    for C in (128, 256):
        groups = engine.bank_check_groups(filters.make_erb_filters(16000, filters.centre_freqs(16000, C, 100)))
        assert groups.shape == (C // 32,) and np.all(groups < 1.0), groups


def test_the_refused_group_is_the_low_frequency_one():
    """16 kHz, 96 channels, LOW_FREQ = 20, width 2 (the bank the float32 check refuses at 4.7x): only the
    last group, the one nearest z = 1, is above the bar."""
    groups = engine.bank_check_groups(filters.make_erb_filters(16000, filters.centre_freqs(16000, 96, 20), 2.0))
    assert groups[2] > 1.0 and np.all(groups[:2] < 1.0), groups


def test_bad_arguments_are_rejected_like_the_bank_check():
    with pytest.raises(ValueError):
        engine.bank_check_groups(np.zeros((4, 9)))
    for bad in (np.zeros((4, 10)), np.ones((0, 10))):
        with pytest.raises((_native.F2Error, ValueError)) as e1:
            engine.bank_check(bad)
        with pytest.raises((_native.F2Error, ValueError)) as e2:
            engine.bank_check_groups(bad)
        assert type(e1.value) is type(e2.value)
        if isinstance(e1.value, _native.F2Error):
            assert e1.value.code == e2.value.code == _native.F2_ERR_INVALID
