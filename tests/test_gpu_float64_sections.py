"""Float64 sections (FORM 2): the channel groups float32 cannot hold to 1e-4 x RMS run their cascade in
float64 when the plan asks for it (Plan(float64_sections=True) / F2CNN_B200_FLOAT64_SECTIONS=1).

Bounds of the fuzz test were set from a run on a B200 (see test_refused_fuzz_banks_meet_the_bar)."""
import numpy as np
import pytest

from test_float64_sections_cpu import REFUSED_FUZZ_CASES, bank, fuzz_cases

pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from f2cnn_b200 import api, engine, synth
    from f2cnn_b200.gammatone import filters
    return api, engine, filters, synth, torch


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle as o
    o.lib()
    return o


def err(got, want, floor=0.01):
    """max |got - want| per channel over the channel's RMS floored at `floor` of the loudest, in units of TOL"""
    want = np.asarray(want, dtype=np.float64)
    rms = np.sqrt(np.mean(want ** 2, axis=-1))
    rms = np.maximum(np.maximum(rms, floor * rms.max()), 1e-300)
    return float((np.max(np.abs(np.asarray(got, dtype=np.float64) - want), axis=-1) / rms).max()) / TOL


def refused_128(filters):
    """16 kHz, 128 channels, LOW_FREQ = 20, width 1: refused in float32 (2.4x the bar predicted)"""
    return filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 20), 1.0)


def test_refused_bank_runs_with_float64_sections(gpu, orc, monkeypatch):
    """The bank of test_banks_outside_the_float32_tolerance_raise_instead_of_answering (float32 misses the
    fs/4 tone by 4.7x): accepted with float64 sections, its last group in float64, within the bar on the
    tone and on white noise; the float32 groups are bit for bit the forced-float32 run's."""
    api, engine, filters, synth, torch = gpu
    fs, C, n = 16000, 96, 4111
    co = filters.make_erb_filters(fs, filters.centre_freqs(fs, C, 20), 2.0)
    monkeypatch.delenv("F2CNN_B200_ALLOW_IMPRECISE", raising=False)
    plan = engine.Plan(co, float64_sections=True)
    assert plan.float64_sections and 2 in plan.float64_groups
    f32 = [g for g in range(3) if g not in plan.float64_groups]
    rows = np.concatenate([np.arange(32 * g, 32 * g + 32) for g in f32]).astype(np.int64)
    monkeypatch.setenv("F2CNN_B200_ALLOW_IMPRECISE", "1")
    forced = engine.Plan(co, float64_sections=False)
    assert forced.float64_groups == ()
    for kind, w in (("white", synth.white_noise_i16(n, seed=32)), ("tone", synth.tone_i16(n, freq=fs / 4.0, fs=fs))):
        go = orc.erb_filterbank(w, co)
        eo = orc.extract_envelope(go, False, 100)
        wd = torch.from_numpy(w).cuda()
        r = plan.batch([n]).run(wd, gfb=torch.float64, env=torch.float64)
        r32 = forced.batch([n]).run(wd, gfb=torch.float64, env=torch.float64)
        gfb, env = (r[k].cpu().numpy().reshape(C, n) for k in ("gfb", "env"))
        assert err(gfb, go) <= 1.0, kind
        assert err(env, eo) <= 1.0, kind
        for k in ("gfb", "env"):
            assert np.array_equal(r[k].cpu().numpy().reshape(C, n)[rows], r32[k].cpu().numpy().reshape(C, n)[rows])


def test_refused_fuzz_banks_meet_the_bar(gpu, orc):
    """The 27 banks tools/fuzz_parity.py 120 7 draws and the float32 check refuses, with their drawn lengths,
    input kinds, dtypes, low-pass settings, steps and chunk targets: filterbank, envelope and decimated frames
    against the float64 oracle, channel RMS floored at 1 % of the loudest.  Observed on a B200 (1000 W): worst
    gfb 0.155 / env 0.258 / dec 0.244 of the bar; float32 misses the same banks by up to 4.7x.  Bounds: about
    1.5x the observed worst."""
    api, engine, filters, synth, torch = gpu
    BOUND = {"gfb": 0.25, "env": 0.4, "dec": 0.4}
    worst = {"gfb": 0.0, "env": 0.0, "dec": 0.0}
    for p in fuzz_cases():
        if p["case"] not in REFUSED_FUZZ_CASES:
            continue
        co, n, fs, case = bank(p), p["n"], p["fs"], p["case"]
        if p["kind"] == "white":
            w = synth.white_noise_i16(n, seed=case)
        elif p["kind"] == "speech":
            w = synth.speech_like_i16(n, seed=case)
        elif p["kind"] == "tone":
            w = synth.tone_i16(n, freq=p["freq"], fs=fs)
        else:
            w = synth.chirp_i16(n, f0=float(p["low"]), f1=fs * 0.45, fs=fs)
        w = w.astype(p["dtype"])
        plan = engine.Plan(co, float64_sections=True)
        assert plan.float64_groups, case
        b = plan.batch([n], step=p["step"], target_items=p["target"])
        wd = torch.from_numpy(w).cuda()
        r = b.run(wd, lpf=p["lpf"], cutoff=p["cutoff"], gfb=torch.float64, env=torch.float64)
        dec = b.run(wd, lpf=p["lpf"], cutoff=p["cutoff"], dec=True)["dec"].cpu().numpy().T
        go = orc.erb_filterbank(w, co)
        eo = orc.extract_envelope(go, p["lpf"], p["cutoff"])
        C = p["C"]
        got = {"gfb": (r["gfb"].cpu().numpy().reshape(C, n), go), "env": (r["env"].cpu().numpy().reshape(C, n), eo)}
        for name, (g, want) in got.items():
            worst[name] = max(worst[name], err(g, want))
        sc = np.sqrt(np.mean(eo ** 2, axis=1))
        sc = np.maximum(sc, 0.01 * sc.max())
        worst["dec"] = max(worst["dec"], float((np.max(np.abs(dec - eo[:, ::p["step"]]), axis=1) / sc).max()) / TOL)
    print("refused fuzz banks with float64 sections, worst of the bar:", worst)
    for name, v in worst.items():
        assert v <= BOUND[name], (name, worst)


def test_output_modes_of_a_refused_bank(gpu, orc, monkeypatch):
    """One refused 128-channel bank through every output mode: window store == decimated frames + gather bit for
    bit; the (C, n) store == the transposed time-major output; gammatonegram; time chunks within the
    bound of test_time_chunking_is_transparent; batch == single runs bit for bit; two runs identical."""
    api, engine, filters, synth, torch = gpu
    co = refused_128(filters)
    plan = engine.Plan(co, float64_sections=True)
    assert plan.float64_groups == (3,)
    C, dots, step = 128, 11, 160
    lens = [9000, 1700, 48000, 2081]
    waves = [synth.speech_like_i16(n, seed=60 + i) for i, n in enumerate(lens)]
    flat = torch.from_numpy(np.concatenate(waves)).cuda()
    batch = plan.batch(lens, step=step)
    offs, rows = batch.grid_windows(dots)
    nb = [max(n // step - dots - 1, 0) for n in lens]
    win = torch.full((rows, dots, C), float("nan"), dtype=torch.float32, device="cuda")
    batch.run(flat, lpf=True, cutoff=50, windows=(offs, dots, win))
    dec = batch.run(flat, lpf=True, cutoff=50, dec=True)["dec"]
    base = np.concatenate([batch.frame_offsets[u] + np.arange(nb[u]) for u in range(len(lens))]).astype(np.int64)
    assert not torch.isnan(win).any()
    assert torch.equal(win, engine.gather_windows(dec, torch.from_numpy(base).cuda(), dots, 1))
    # (C, n) envelope alone, and next to the time-major envelope: the same bits, and env_t.T
    direct = batch.run(flat, lpf=True, cutoff=50, env=torch.float32)["env"]
    both = batch.run(flat, lpf=True, cutoff=50, env=torch.float32, env_t=True)
    assert torch.equal(direct, both["env"])
    o = 0
    for n in lens:
        assert torch.equal(direct[o * C:(o + n) * C].reshape(C, n), both["env_t"][o:o + n].T)
        o += n
    assert torch.equal(dec, batch.run(flat, lpf=True, cutoff=50, dec=True)["dec"])
    # whole utterances (target_items=1): batch == single runs bit for bit, and the oracle
    whole = plan.batch(lens, step=step, target_items=1)
    wdec = whole.run(flat, lpf=True, cutoff=50, dec=True)["dec"]
    for u, (n, w) in enumerate(zip(lens, waves)):
        one = plan.batch([n], step=step, target_items=1).run(torch.from_numpy(w).cuda(), lpf=True, cutoff=50,
                                                             dec=True)["dec"]
        f0 = int(whole.frame_offsets[u])
        assert torch.equal(one, wdec[f0:f0 + one.shape[0]])
    _, eo, _ = orc.utterance(waves[2], co, True, 50)
    for b_, d_ in ((whole, wdec), (batch, dec)):
        f0 = int(b_.frame_offsets[2])
        assert err(d_[f0:f0 + (48000 + step - 1) // step].cpu().numpy().T, eo[:, ::step]) <= 1.0
    # gammatonegram (through plan_for: the environment variable)
    monkeypatch.setenv("F2CNN_B200_FLOAT64_SECTIONS", "1")
    g = np.asarray(api.gammatonegram(waves[2], co, 160, True, 50))
    assert g.shape[0] == C and np.all(np.isfinite(g))
    assert err(g, eo[:, ::160][:, :g.shape[1]]) <= 1.0
    # a long stream in time chunks (edge residuals from the float64 edge pass)
    w = synth.speech_like_i16(60000, seed=9)
    go, eo, _ = orc.utterance(w, co, True, 20)
    wd = torch.from_numpy(w).cuda()
    ref = plan.batch([60000], target_items=1).run(wd, lpf=True, cutoff=20, env=torch.float64)["env"].cpu().numpy()
    b = plan.batch([60000], target_items=64)
    assert b.num_items > 4
    env = b.run(wd, lpf=True, cutoff=20, env=torch.float64)["env"].cpu().numpy().reshape(C, -1)
    assert err(env, eo, floor=0.0) <= 1.0
    assert err(env, ref.reshape(C, -1), floor=0.0) <= 0.2
    gfb = b.run(wd, gfb=torch.float64)["gfb"].cpu().numpy().reshape(C, -1)
    assert err(gfb, go, floor=0.0) <= 1.0


@pytest.mark.parametrize("C", [128, 256])
def test_accepted_banks_are_unchanged_by_the_flag(gpu, C):
    """A bank the float32 check accepts selects no group, and every output mode is bit for bit the same with
    the flag on and off."""
    api, engine, filters, synth, torch = gpu
    co = filters.make_erb_filters(16000, filters.centre_freqs(16000, C, 100))
    on, off = engine.Plan(co, float64_sections=True), engine.Plan(co, float64_sections=False)
    assert on.float64_groups == () and off.float64_groups == ()
    lens = [30000, 5000, 48000]
    flat = torch.from_numpy(np.concatenate([synth.speech_like_i16(n, seed=7 + i) for i, n in enumerate(lens)])).cuda()
    for target in (0, 64):
        outs = []
        for plan in (on, off):
            b = plan.batch(lens, target_items=target)
            offs, rows = b.grid_windows(11)
            win = torch.zeros((rows, 11, C), dtype=torch.float32, device="cuda")
            b.run(flat, lpf=True, cutoff=50, windows=(offs, 11, win))
            r = b.run(flat, lpf=True, cutoff=50, gfb=torch.float64, env=torch.float32, dec=True)
            r2 = b.run(flat, lpf=True, cutoff=50, env=torch.float64, env_t=True)
            outs.append([win] + [r[k] for k in ("gfb", "env", "dec")] + [r2[k] for k in ("env", "env_t")])
        for x, y in zip(*outs):
            assert torch.equal(x, y)


def test_public_calls_with_the_environment_variable(gpu, orc, monkeypatch):
    """F2CNN_B200_FLOAT64_SECTIONS=1 reaches the api.* functions and the drop-in scripts through plan_for:
    features_to_windows((flat, lengths), counts=...) == the device-side window store of the same batch, bit for
    bit; on the corpus path features_to_frames(...).materialize() == features_to_windows bit for bit (label
    grid, as test_frame_windows_are_views_of_the_decimated_frames); both against the oracle; the drop-in
    filterbank at 44.1 kHz, LOW_FREQ = 20."""
    api, engine, filters, synth, torch = gpu
    co = refused_128(filters)
    with pytest.raises(Exception):
        api.erb_filterbank(synth.white_noise_i16(2000, seed=1), co)
    monkeypatch.setenv("F2CNN_B200_FLOAT64_SECTIONS", "1")
    assert engine.plan_for(co).float64_groups == (3,)
    lens = np.array([20000, 33333], dtype=np.int64)
    waves = [synth.speech_like_i16(int(n), seed=80 + i) for i, n in enumerate(lens)]
    flat = np.concatenate(waves)
    counts = np.maximum((lens / 160 - 12).astype(np.int64), 0)
    centers = np.concatenate([800 + 160 * np.arange(k, dtype=np.int64) for k in counts])
    got = api.features_to_windows((flat, lens), co, centers, True, 50, counts=counts)
    plan = engine.plan_for(co)
    b = plan.batch(lens.tolist())
    offs, rows = b.grid_windows(11)
    win = torch.zeros((rows, 11, 128), dtype=torch.float32, device="cuda")
    b.run(torch.from_numpy(flat).cuda(), lpf=True, cutoff=50, windows=(offs, 11, win))
    assert np.array_equal(got, win.cpu().numpy())
    # the corpus path (sub-batches of whole utterances) for a ragged corpus, on the label grid
    monkeypatch.setattr(api, "_PIPELINE_BYTES", 0)
    rng = np.random.default_rng(17)
    clens = rng.integers(1500, 9000, size=13).astype(np.int64)
    cwaves = [synth.speech_like_i16(int(n), seed=300 + i) for i, n in enumerate(clens)]
    nwin = np.maximum((clens / 160 - 12).astype(np.int64), 0)
    ccenters = [800 + 160 * np.arange(k, dtype=np.int64) for k in nwin]
    corpus = api.features_to_windows(cwaves, co, ccenters, True, 50)
    cflat = torch.from_numpy(np.concatenate(cwaves))
    for source in (cwaves, (cflat, clens)):
        assert np.array_equal(api.features_to_frames(source, co, True, 50).materialize(), corpus)
    for x, ws, cs, ks in ((got, waves, [centers[:counts[0]], centers[counts[0]:]], counts), (corpus, cwaves, ccenters, nwin)):
        row = 0
        for w, c, k in zip(ws, cs, ks):
            if k == 0:
                continue
            _, eo, wo = orc.utterance(w, co, True, 50, c, 5, 160)
            scale = np.sqrt(np.mean(eo ** 2, axis=1))
            assert np.max(np.abs(x[row:row + k] - wo) / scale[None, None, :]) / TOL <= 1.0
            row += int(k)
    from f2cnn_b200.scripts.processing import GammatoneFiltering
    fs = 44100
    co44 = filters.make_erb_filters(fs, filters.centre_freqs(fs, 64, 20))
    assert engine.plan_for(co44).float64_groups == (1,)
    w = synth.speech_like_i16(30000, seed=5)
    out = GammatoneFiltering.GetFilteredOutputFromArray(w, co44)
    assert err(out, orc.erb_filterbank(w, co44)) <= 1.0


def test_cnn_evaluate_on_a_refused_bank(gpu, orc, monkeypatch):
    """api.cnn_evaluate (`cnn eval*`) on a refused 128-channel bank with F2CNN_B200_FLOAT64_SECTIONS=1: its
    envelopes are within the bar of the oracle, and its scores meet the bounds of test_gpu_cnn_reference.py
    (chained and stage-local) when oracle/cnn_bf16.py is fed those envelopes."""
    api, engine, filters, synth, torch = gpu
    from oracle import cnn_bf16
    from test_gpu_cnn_reference import CHUNK, _chained, _check, _stage_local
    monkeypatch.setenv("F2CNN_B200_FLOAT64_SECTIONS", "1")
    co = refused_128(filters)
    assert engine.plan_for(co).float64_groups == (3,)
    n = 48000
    w = synth.speech_like_i16(n, seed=21).astype(np.float64) + np.random.default_rng(6).normal(0, 30, n)
    model = cnn_bf16.spread_model().cuda()
    scores, envelopes = api.cnn_evaluate(w, co, model, True, 50, with_envelopes=True)
    nb = n - 1760
    assert scores.shape == (nb, 2) and envelopes.shape == (128, n)
    _, eo, _ = orc.utterance(w, co, True, 50)
    assert err(envelopes, eo) <= 1.0
    # the envelopes are the float32 time-major envelope the network read, widened
    env_t = torch.from_numpy(np.ascontiguousarray(envelopes.T)).float().cuda()
    assert np.array_equal(env_t.double().cpu().numpy().T, envelopes)
    ref = cnn_bf16.BF16Reference(model, device="cuda")
    got = torch.from_numpy(scores).cuda()
    for i0, i1 in ((0, 256), (CHUNK - 128, CHUNK + 128), (nb - 256, nb)):
        _chained(ref, env_t, 160, i0, i1, got[i0:i1], "refused bank [%d, %d)" % (i0, i1))
    tc = api._network_for(model)
    for i0, i1 in ((0, 300), (nb - 257, nb)):
        s = tc.predict_envelope(env_t, 160, frames=(i0, i1))
        _check(_stage_local(tc, ref, env_t, 160, i0, i1, s), "refused bank [%d, %d)" % (i0, i1))


def test_two_devices_shard_a_refused_bank(gpu, monkeypatch):
    """A refused bank sharded over two devices with shard=(rank, world): the rows equal the one-GPU result."""
    api, engine, filters, synth, torch = gpu
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    monkeypatch.setenv("F2CNN_B200_FLOAT64_SECTIONS", "1")
    co = refused_128(filters)
    lens = np.array([20000, 9000, 33333, 12000], dtype=np.int64)
    flat = np.concatenate([synth.speech_like_i16(int(n), seed=90 + i) for i, n in enumerate(lens)])
    whole = api.features_to_frames((flat, lens), co, True, 50)
    first_row = np.concatenate([[0], np.cumsum(whole.counts)])
    want = whole.materialize()
    for rank in range(2):
        with torch.cuda.device(rank):
            part = api.features_to_frames((flat, lens), co, True, 50, shard=(rank, 2))
        for j, u in enumerate(part.utterances):
            assert np.array_equal(part.windows(j), want[first_row[u]:first_row[u + 1]]), (rank, u)
