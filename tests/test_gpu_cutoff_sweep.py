"""Cutoff sweep: the decimated frames of several envelope settings from one filterbank and Hilbert pass
(f2_batch_run_cutoffs, engine.Batch.run_cutoffs, api.features_to_windows_sweep, GenerateInputDataSweep),
against single-setting runs of the same batch and the float64 oracle."""
import csv
import ctypes
import math
import os

import numpy as np
import pytest

from test_float64_sections_cpu import REFUSED_FUZZ_CASES, bank, fuzz_cases

pytestmark = pytest.mark.gpu
TOL = 1e-4          # the project's bar against the float64 oracle, x channel RMS
WARM_TOL = 1e-6     # a longer warm-start of a chunk against the single run's, x channel RMS (short utterances)
# The same on a 200000-sample utterance in time chunks.  The truncated history of a warm start is below 1e-9,
# but two float32 runs that start a chunk from different states round differently from there on: the one-pole
# low-pass sums ~1/(1-k) rounded samples, and the no-low-pass plane's cascade starts w_lpf samples earlier than in
# its own run.  Measured on a B200 the planes other than the lowest cutoff differ from their single runs by up to
# 1.8e-6 x channel RMS (c128 bank, 50 Hz) and 6.8e-6 (no low-pass), more than the 1e-6 expected; each is as far
# from the float64 oracle as its single run (within 7e-7).  The bound is the float32 error level of the envelope
# (DESIGN.md section 3: <= 1e-5 of the channel RMS).
CHUNK_TOL = 1e-5
LENGTHS = [1, 255, 256, 257, 65536, 48000]
CONF = ("[FILTERBANK]\nFRAMERATE=16000\nNCHANNELS=32\nLOW_FREQ=100\n"
        "[CNN]\nFORMANT=2\nCENTERED=True\nRADIUS=5\nBATCH_SIZE=32\nEPOCHS=20\nRISK=0.05\nSAMPLING_PERIOD=10000\n")


@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from f2cnn_b200 import _native, api, engine, synth
    from f2cnn_b200.gammatone import filters
    return dict(torch=torch, native=_native, api=api, engine=engine, synth=synth, filters=filters)


@pytest.fixture(scope="module")
def banks(gpu):
    """name -> plan: the 128- and 256-channel banks, and banks float32 refuses, run with float64 sections"""
    engine, filters = gpu["engine"], gpu["filters"]
    plans = {"c128": engine.Plan(filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))),
             "c256": engine.Plan(filters.make_erb_filters(16000, filters.centre_freqs(16000, 256, 100)))}
    cases = {p["case"]: p for p in fuzz_cases()}
    for case in REFUSED_FUZZ_CASES[:2]:
        plans["fuzz%d" % case] = engine.Plan(bank(cases[case]), float64_sections=True)
    plans["low20"] = engine.Plan(filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 20)),
                                 float64_sections=True)
    for name in ("fuzz%d" % REFUSED_FUZZ_CASES[0], "low20"):
        assert plans[name].float64_groups, name
    return plans


def waves(gpu, lengths, dtype=np.int16, seed=3):
    synth, torch = gpu["synth"], gpu["torch"]
    w = np.concatenate([synth.speech_like_i16(n, seed=seed + i) if n else np.zeros(0, np.int16)
                        for i, n in enumerate(lengths)]).astype(dtype)
    return w, torch.from_numpy(w).cuda()


def single(batch, wd, c):
    return batch.run(wd, dec=True, lpf=c is not None, cutoff=100 if c is None else c)["dec"].cpu().numpy()


def rel_rms(got, want):
    """max |got - want| per channel (last axis) over the channel's RMS of `want`"""
    want = np.asarray(want, dtype=np.float64)
    axes = tuple(range(want.ndim - 1))
    rms = np.maximum(np.sqrt(np.mean(want ** 2, axis=axes)), 1e-300)
    return float((np.max(np.abs(np.asarray(got, dtype=np.float64) - want), axis=axes) / rms).max())


@pytest.mark.parametrize("target", [1, 64])
def test_one_setting_is_the_existing_run(gpu, banks, target):
    """run_cutoffs([c]) == run(dec=True, lpf=c is not None, cutoff=c) bit for bit: whole utterances and time
    chunks, every wave dtype, steps 1 / 7 / 160 and a nonzero phase, short and long utterances, 128 and 256
    channels and banks with float64 sections"""
    modes = [("c128", np.int16, 160, 0), ("c128", np.float32, 7, 3), ("c128", np.float64, 1, 0),
             ("c128", np.int16, 160, 37), ("c256", np.int16, 160, 0)]
    modes += [(name, np.int16, 160, 0) for name in banks if name.startswith(("fuzz", "low"))]
    for name, dtype, step, phase in modes:
        plan = banks[name]
        w, wd = waves(gpu, LENGTHS, dtype)
        b = plan.batch(LENGTHS, step=step, phase=phase, target_items=target)
        if target > 1:
            assert b.num_items > len(LENGTHS) * ((plan.n_channels + 31) // 32), "not time-chunked"
        for c in (None, 20, 50, 400):
            got = b.run_cutoffs(wd, [c])
            assert got.shape == (1, b.total_frames, plan.n_channels)
            assert np.array_equal(got[0].cpu().numpy(), single(b, wd, c)), (name, dtype, step, phase, c)


@pytest.mark.parametrize("step", [160, 7, 1])
def test_several_settings_on_whole_utterances(gpu, banks, step):
    """every plane of (20, 50, 100, None), of a permuted order and of two- and three-setting sweeps equals its
    single run bit for bit"""
    for name in ("c128", "low20"):
        plan = banks[name]
        w, wd = waves(gpu, LENGTHS)
        b = plan.batch(LENGTHS, step=step, phase=step // 2, target_items=1)
        ref = {c: single(b, wd, c) for c in (20, 50, 100, None)}
        for settings in ((20, 50, 100, None), (None, 100, 20, 50), (50, None), (100, 20, None)):
            got = b.run_cutoffs(wd, settings).cpu().numpy()
            for j, c in enumerate(settings):
                assert np.array_equal(got[j], ref[c]), (name, settings, c)


def test_several_settings_on_time_chunks(gpu, banks, oracle):
    """a long utterance in time chunks: every chunk warms up for the lowest cutoff, so that plane is bit for bit
    its single run; the others meet the oracle's bar and stay within WARM_TOL of their single runs"""
    orc = oracle
    n, step, phase = 200000, 160, 80
    settings = (50, 20, 100, None)
    for name in ("c128", "low20"):
        plan = banks[name]
        w, wd = waves(gpu, [n], seed=11)
        b = plan.batch([n], step=step, phase=phase, target_items=64)
        assert b.num_items > (plan.n_channels + 31) // 32, "not time-chunked"
        got = b.run_cutoffs(wd, settings).cpu().numpy()
        gfb = orc.erb_filterbank(w, plan.coefs)
        worst = {}
        for j, c in enumerate(settings):
            one = single(b, wd, c)
            if c == 20:
                assert np.array_equal(got[j], one), name
                continue
            env = orc.extract_envelope(gfb, c is not None, 100 if c is None else c)
            want = env[:, phase::step].T
            rms = np.sqrt(np.mean(env ** 2, axis=1))
            e = lambda a, b_: float((np.max(np.abs(np.asarray(a, np.float64) - b_), axis=0) / rms).max())
            worst[c] = dict(sweep_vs_oracle=e(got[j], want), single_vs_oracle=e(one, want), sweep_vs_single=e(got[j], one))
        print(name, "error x channel RMS:", worst)
        for c, w_ in worst.items():
            assert w_["sweep_vs_oracle"] <= TOL, (name, c, w_)
            assert w_["sweep_vs_single"] <= CHUNK_TOL, (name, c, w_)


def label_corpus(gpu, n_utts, lo, hi, seed, keep=0.85):
    """waves and label-grid timepoints with some rows dropped, as a CSV has them"""
    synth = gpu["synth"]
    rng = np.random.default_rng(seed)
    lengths = rng.integers(lo, hi, n_utts)
    ws = [synth.white_noise_i16(int(n), seed=seed + i) for i, n in enumerate(lengths)]
    tps = []
    for n in lengths:
        grid = synth.label_grid(int(n))
        tps.append(grid[rng.random(grid.shape[0]) < keep])
    return ws, tps


def test_public_sweep_on_the_pipeline_path(gpu):
    """a corpus above the pipeline threshold: every cutoff's rows equal features_to_windows' bit for bit"""
    api, filters = gpu["api"], gpu["filters"]
    co = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))
    ws, tps = label_corpus(gpu, 200, 44000, 52000, seed=5)
    total = sum(len(t) for t in tps)
    assert total * 11 * 128 * 4 >= api._PIPELINE_BYTES
    settings = (20, 100, None)
    got = api.features_to_windows_sweep(ws, co, tps, settings)
    assert any(k[-1] == len(settings) for k in api._pipelines), "the sweep did not take the pipeline path"
    for j, c in enumerate(settings):
        want = api.features_to_windows(ws, co, tps, LPF=c is not None, CUTOFF=100 if c is None else c)
        assert got[j].shape == want.shape == (total, 11, 128) and got[j].dtype == np.float32
        assert np.array_equal(got[j], want), c
    api.release_cached_pipelines()


def test_public_sweep_on_the_small_path(gpu, oracle):
    """one batch (time-chunked here): the lowest cutoff bit for bit, the others within WARM_TOL of
    features_to_windows and within the bar of the oracle; off-grid timepoints raise ValueError"""
    api, filters = gpu["api"], gpu["filters"]
    orc = oracle
    co = filters.make_erb_filters(16000, filters.centre_freqs(16000, 32, 100))
    ws, tps = label_corpus(gpu, 3, 9000, 30000, seed=9)
    settings = (None, 20, 50)
    got = api.features_to_windows_sweep(ws, co, tps, settings)
    for j, c in enumerate(settings):
        want = api.features_to_windows(ws, co, tps, LPF=c is not None, CUTOFF=100 if c is None else c)
        assert got[j].shape == want.shape
        if c == 20:
            assert np.array_equal(got[j], want)
        else:
            assert rel_rms(got[j], want) <= WARM_TOL, c
        ref = np.concatenate([orc.utterance(w, co, c is not None, 100 if c is None else c, t)[2]
                              for w, t in zip(ws, tps)])
        assert rel_rms(got[j], ref) <= TOL, c
    # a window index off the grid of the others
    with pytest.raises(ValueError, match="features_to_windows"):
        api.features_to_windows_sweep(ws, co, [tps[0], tps[1] + 1, tps[2]], settings)
    with pytest.raises(ValueError):
        api.features_to_windows_sweep(ws, co, tps, (20, 0))


def test_argument_checks(gpu, banks):
    """the documented status codes from the C entry point, ValueError from Python"""
    torch, _native = gpu["torch"], gpu["native"]
    plan = banks["c128"]
    w, wd = waves(gpu, [4000])
    b = plan.batch([4000])
    L = _native.lib()
    K_max = 4
    plane = b.total_frames * plan.n_channels
    dec = torch.empty(K_max * plane, dtype=torch.float32, device="cuda")
    ws = torch.empty(b.workspace_bytes(), dtype=torch.uint8, device="cuda")

    def call(hz, n=None, stride=plane, dec_ptr=dec.data_ptr(), ws_bytes=ws.numel()):
        arr = (ctypes.c_double * max(len(hz), 1))(*hz)
        return L.f2_batch_run_cutoffs(b._h, ctypes.c_void_p(wd.data_ptr()), _native.F2_I16, arr,
                                      len(hz) if n is None else n, ctypes.c_void_p(dec_ptr), stride,
                                      ctypes.c_void_p(ws.data_ptr()), ws_bytes, None)

    assert call([20.0, 0.0]) == _native.F2_OK
    torch.cuda.synchronize()
    for n in (0, 5, -1):
        assert call([20.0] * 5, n=n) == _native.F2_ERR_INVALID, n
    for bad in (-1.0, 8000.0, math.nan):
        assert call([20.0, bad]) == _native.F2_ERR_INVALID, bad
        assert "cutoff" in L.f2_last_error().decode()
    assert call([20.0, 50.0], stride=plane - 1) == _native.F2_ERR_INVALID
    assert call([20.0], dec_ptr=0) == _native.F2_ERR_INVALID
    assert call([20.0], ws_bytes=ws.numel() - 1) == _native.F2_ERR_WORKSPACE

    for bad in ([], [20, 50, 100, None, 400], [-1], [8000], [math.nan], [0], [None, 0.0]):
        with pytest.raises(ValueError):
            b.run_cutoffs(wd, bad)
    short = torch.empty(2 * plane, dtype=torch.float32, device="cuda").as_strided(
        (2, b.total_frames, plan.n_channels), (plane - plan.n_channels, plan.n_channels, 1))
    with pytest.raises(ValueError):
        b.run_cutoffs(wd, [20, 50], out=short)


@pytest.fixture()
def tree(tmp_path, monkeypatch):
    from scipy.io import wavfile
    from f2cnn_b200 import synth
    monkeypatch.chdir(tmp_path)
    (tmp_path / "configF2CNN.conf").write_text(CONF)
    rows = []
    for tt, name, n in (("TRAIN", "DR1.SPK0.SA1", 9000), ("TRAIN", "DR2.SPK1.SX7", 12000), ("TEST", "DR1.SPK2.SI3", 7000)):
        d = tmp_path / "resources" / "f2cnn" / tt
        d.mkdir(parents=True, exist_ok=True)
        wavfile.write(str(d / (name + ".WAV")), 16000, synth.speech_like_i16(n, seed=n))
        dr, spk, sent = name.split(".")
        for tp in synth.label_grid(n)[::3]:
            rows.append([tt, dr, spk, sent, "aa", int(tp), 0.1, 0.01, 1])
    os.makedirs("trainingData")
    with open(os.path.join("trainingData", "label_data.csv"), "w") as f:
        wr = csv.writer(f, lineterminator="\n")
        for r in rows[::-1]:
            wr.writerow(r)
    return tmp_path


def test_driver_writes_every_cutoff(gpu, tree):
    """GenerateInputDataSweep writes input_data_LPF<k>.npy / input_data_NOLPF.npy, each matching
    GenerateInputData for that cutoff (computed from the WAVs, no .ENV1.npy present)"""
    from f2cnn_b200 import dropin
    dropin.install()
    try:
        from scripts.processing import InputGenerator
        InputGenerator.GenerateInputDataSweep(CUTOFFS=(50, None, 20))
        names = {50: "input_data_LPF50.npy", None: "input_data_NOLPF.npy", 20: "input_data_LPF20.npy"}
        assert sorted(os.listdir("trainingData")) == sorted(list(names.values()) + ["label_data.csv"])
        for c, name in names.items():
            got = np.load(os.path.join("trainingData", name))
            InputGenerator.GenerateInputData(inputFile=os.path.join("single", name), LPF=c is not None,
                                             CUTOFF=100 if c is None else c)
            want = np.load(os.path.join("single", name))
            assert got.dtype == np.float32 and got.shape == want.shape
            if c == 20:
                assert np.array_equal(got, want)
            else:
                assert rel_rms(got, want) <= WARM_TOL, c
        os.remove(str(tree / "resources" / "f2cnn" / "TEST" / "DR1.SPK2.SI3.WAV"))
        with pytest.raises(FileNotFoundError):
            InputGenerator.GenerateInputDataSweep(CUTOFFS=(20,))
    finally:
        dropin.uninstall()
