"""Parity of the CUDA path (through the C ABI) with the float64 oracle and with the golden
vectors recorded from the unmodified reference.

Tolerance (BASELINE.json north_star): max abs error <= 1e-4 x per-channel signal RMS for the
filterbank and the envelope; window indexing / row order exact.  The kernels compute in
float32, so the pure-tone KAT -- whose stop-band channels sit 60 dB below the input -- is held
to 1e-4 x max(channel RMS, 1 % of the loudest channel's RMS): that floor is float32's
resolution of the input itself, not an algorithmic error."""
import csv
import io

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu
TOL = 1e-4


@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from f2cnn_b200 import api, engine
    from f2cnn_b200.gammatone import filters
    return api, engine, filters, torch


def rel_err(got, want, rms=None, floor=0.0):
    want = np.asarray(want, dtype=np.float64)
    if rms is None:
        rms = np.sqrt(np.mean(want ** 2, axis=-1))
    rms = np.maximum(rms, floor * np.max(rms))
    rms = np.maximum(rms, 1e-300)
    return np.max(np.abs(np.asarray(got, dtype=np.float64) - want), axis=-1) / rms


def coefs128():
    return load_golden("coefs.npz")["coefs_fs16000_c128_l100"]


@pytest.mark.parametrize("name", ["white", "delta", "tone1k", "chirp", "speech"])
def test_golden_3s(gpu, name):
    """configs[0]: single 3 s utterance, 128 channels, against the reference's own outputs."""
    api, engine, filters, torch = gpu
    g = load_golden("utt3s_%s.npz" % name)
    co = coefs128()
    idx = g["idx"]
    floor = 1e-2 if name == "tone1k" else 0.0
    gfb = api.erb_filterbank(g["wave"], co)
    assert gfb.shape == (128, 48000) and gfb.dtype == np.float64
    assert rel_err(gfb[:, idx], g["gfb"], g["gfb_rms"], floor).max() <= TOL
    env50 = api.extract_envelope_from_matrix(gfb, True, 50)  # stand-alone rows path
    assert rel_err(env50[:, idx], g["env_lpf50"], g["env_lpf50_rms"], floor).max() <= TOL
    gfb2, env50f = api.filterbank_envelope(g["wave"], co, True, 50, with_gfb=True)  # fused path
    # same arithmetic, but the time chunks are warm-started from different points with and
    # without the low-pass warm-up: equal to float32 rounding noise (~1e-6), not bit for bit
    assert rel_err(gfb2, gfb, None, floor).max() <= 5e-5
    assert rel_err(env50f[:, idx], g["env_lpf50"], g["env_lpf50_rms"], floor).max() <= TOL
    envno = api.filterbank_envelope(g["wave"], co, False)
    assert rel_err(envno[:, idx], g["env_nolpf"], g["env_nolpf_rms"], floor).max() <= TOL
    # per-channel energy (checksum over all 48000 samples, not only the sampled columns)
    np.testing.assert_allclose(np.sqrt(np.mean(gfb ** 2, axis=1)), g["gfb_rms"], rtol=2e-5)
    np.testing.assert_allclose(np.sqrt(np.mean(env50f ** 2, axis=1)), g["env_lpf50_rms"], rtol=2e-5)
    if name == "white":
        for cut, key in ((20, "env_lpf20"), (100, "env_lpf100")):
            e = api.filterbank_envelope(g["wave"], co, True, cut)
            assert rel_err(e[:, idx], g[key], g[key + "_rms"]).max() <= TOL
        dec = g["dec_idx"]
        assert rel_err(env50f[:, dec], g["env_lpf50_dec"], g["env_lpf50_rms"]).max() <= TOL


def test_golden_small_lengths(gpu):
    """Ragged / tiny inputs: n = 1 .. 4097 (ring shorter than a tile, N2 = 1, 2, 4 ...)."""
    api, engine, filters, torch = gpu
    g = load_golden("small.npz")
    co = g["coefs"]
    for nn in (1, 2, 3, 4, 5, 16, 17, 255, 256, 257, 1000, 4096, 4097):
        w = g["wave_%d" % nn]
        gfb = api.erb_filterbank(w, co)
        assert gfb.shape == (8, nn)
        # a few samples of a just-starting filter have no meaningful RMS: scale by the peak
        scale = np.maximum(np.sqrt(np.mean(g["gfb_%d" % nn] ** 2, axis=1)), 1e-3 * np.abs(g["gfb_%d" % nn]).max())
        assert rel_err(gfb, g["gfb_%d" % nn], scale).max() <= TOL, nn
        for key, (lpf, cut) in {"env_lpf50": (True, 50), "env_nolpf": (False, 100)}.items():
            want = g["%s_%d" % (key, nn)]
            scale = np.maximum(np.sqrt(np.mean(want ** 2, axis=1)), 1e-3 * np.abs(want).max())
            got = api.filterbank_envelope(w, co, lpf, cut)
            # rings shorter than one tile (inputs under 16 ms): the periodic Hilbert path is driven
            # almost entirely by the edge injection and float32 holds it to ~1e-3 only (DESIGN.md)
            tol = 2e-3 if nn < 255 else TOL
            assert rel_err(got, want, scale).max() <= tol, (key, nn)
            got_rows = api.extract_envelope_from_matrix(g["gfb_%d" % nn], lpf, cut)
            assert rel_err(got_rows, want, scale).max() <= TOL, (key, nn, "rows")


def test_golden_pow2_lengths(gpu):
    """n = 65530 .. 65537: no padding at n = 2^16, N2 doubles at 2^16 + 1."""
    api, engine, filters, torch = gpu
    g = load_golden("pow2.npz")
    co = g["coefs"]
    for nn in (65530, 65535, 65536, 65537):
        idx = g["idx_%d" % nn]
        gfb, env = api.filterbank_envelope(g["wave_%d" % nn], co, True, 50, with_gfb=True)
        assert rel_err(gfb[:, idx], g["gfb_%d" % nn], g["gfb_rms_%d" % nn]).max() <= TOL
        assert rel_err(env[:, idx], g["env_lpf50_%d" % nn], g["env_lpf50_rms_%d" % nn]).max() <= TOL
        envno = api.filterbank_envelope(g["wave_%d" % nn], co, False)
        assert rel_err(envno[:, idx], g["env_nolpf_%d" % nn], g["env_nolpf_rms_%d" % nn]).max() <= TOL


def test_golden_c256_float64_and_dense_frames(gpu):
    """256 channels, float64 noise-mixed input (evalnoise path), dense framing + normalizeInput."""
    api, engine, filters, torch = gpu
    g = load_golden("c256_f64.npz")
    co = load_golden("coefs.npz")["coefs_fs16000_c256_l100"]
    idx = g["idx"]
    gfb, env = api.filterbank_envelope(g["wave"], co, True, 50, with_gfb=True)
    assert rel_err(gfb[:, idx], g["gfb"], g["gfb_rms"]).max() <= TOL
    assert rel_err(env[:, idx], g["env_lpf50"], g["env_lpf50_rms"]).max() <= TOL
    n = g["wave"].shape[0]
    raw = api.dense_frames(g["wave"], co, True, 50, normalize=False)
    assert raw.shape == (n - 11 * 160, 11, 256) and raw.dtype == np.float64
    norm = api.dense_frames(g["wave"], co, True, 50, normalize=True)
    for j, i in enumerate(g["frames_i"]):
        assert np.max(np.abs(raw[i] - g["frames"][j]) / g["env_lpf50_rms"][None, :]) <= TOL
        # log-min-max compresses: compare in the normalised domain with an absolute bound
        assert np.max(np.abs(norm[i] - g["frames_norm"][j])) <= 2e-4


def test_golden_input_generator_rows(gpu):
    """End to end windows: row order = sorted file key, then CSV order (InputGenerator.py:50,67-82)."""
    api, engine, filters, torch = gpu
    g = load_golden("inputgen.npz")
    files = {}
    for row in csv.reader(io.StringIO(str(g["csv"]))):
        key = (row[0], row[1], row[2], row[3])
        files.setdefault("%s/%s.%s.%s" % key, (key, []))[1].append(int(row[5]))
    keys = sorted(files)
    waves = [g["wave_%s_%s_%s_%s" % files[k][0]] for k in keys]
    tps = [np.asarray(files[k][1]) for k in keys]
    got = api.features_to_windows(waves, g["coefs"], tps, True, 50)
    want = g["input_data"]
    assert got.shape == want.shape and got.dtype == np.float32
    scale = np.sqrt(np.mean(want.astype(np.float64) ** 2, axis=(0, 1)))
    assert np.max(np.abs(got.astype(np.float64) - want) / scale[None, None, :]) <= TOL


def test_ragged_batch_matches_oracle_and_single_runs(gpu, oracle):
    """Several utterances of different lengths in one launch == each alone (bit-exact) == oracle."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    lens = [300, 16000, 1, 5000, 33000, 257]
    waves = [synth.white_noise_i16(n, seed=40 + i) for i, n in enumerate(lens)]
    plan = engine.plan_for(co)
    # target_items=1: whole utterances (no time chunks), the configuration of the corpus runs
    batch = plan.batch(lens, target_items=1)
    flat = torch.from_numpy(np.concatenate(waves)).cuda()
    res = batch.run(flat, lpf=True, cutoff=50, gfb=torch.float32, env=torch.float32, dec=True)
    chunked = plan.batch(lens).run(flat, lpf=True, cutoff=50, env=torch.float32)["env"].cpu().numpy()
    gfb_all, env_all, dec_all = res["gfb"].cpu().numpy(), res["env"].cpu().numpy(), res["dec"].cpu().numpy()
    off = 0
    for u, (n, w) in enumerate(zip(lens, waves)):
        gfb = gfb_all[128 * off:128 * (off + n)].reshape(128, n)
        env = env_all[128 * off:128 * (off + n)].reshape(128, n)
        single = plan.batch([n], target_items=1).run(torch.from_numpy(w).cuda(), lpf=True, cutoff=50,
                                                     gfb=torch.float32, env=torch.float32, dec=True)
        assert np.array_equal(single["gfb"].cpu().numpy().reshape(128, n), gfb)
        assert np.array_equal(single["env"].cpu().numpy().reshape(128, n), env)
        f0, f1 = batch.frame_offsets[u], batch.frame_offsets[u + 1]
        assert f1 - f0 == len(range(0, n, 160))
        assert np.array_equal(single["dec"].cpu().numpy(), dec_all[f0:f1])
        assert np.array_equal(dec_all[f0:f1], env[:, ::160].T)  # decimated grid == full-rate samples
        if n >= 256:
            go, eo, _ = oracle.utterance(w, co, True, 50)
            assert rel_err(gfb, go).max() <= TOL and rel_err(env, eo).max() <= TOL
            # the default decomposition (time chunks + per-utterance edge table) agrees as well
            assert rel_err(chunked[128 * off:128 * (off + n)].reshape(128, n), eo).max() <= TOL
        off += n


def test_time_chunking_is_transparent(gpu, oracle):
    """Splitting an utterance into warm-started time chunks changes nothing above 1e-5 x RMS."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    w = synth.speech_like_i16(60000, seed=9)
    go, eo, _ = oracle.utterance(w, co, True, 20)  # 20 Hz: the slowest low-pass pole
    plan = engine.plan_for(co)
    wd = torch.from_numpy(w).cuda()
    ref = plan.batch([60000], target_items=1).run(wd, lpf=True, cutoff=20, env=torch.float64)["env"].cpu().numpy()
    for target in (4, 16, 4096):
        b = plan.batch([60000], target_items=target)
        assert b.num_items > 1
        env = b.run(wd, lpf=True, cutoff=20, env=torch.float64)["env"].cpu().numpy()
        assert rel_err(env.reshape(128, -1), eo).max() <= TOL
        assert rel_err(env.reshape(128, -1), ref.reshape(128, -1)).max() <= 2e-5


def test_windows_off_grid_and_negative_index(gpu, oracle):
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    w = synth.white_noise_i16(9000, seed=77)
    _, eo, _ = oracle.utterance(w, co, True, 50)
    for centers in ([801, 1603, 5007], [100, 800], [900, 4000, 2000]):  # off-grid / wrapping / unsorted
        got = api.features_to_windows([w], co, [np.asarray(centers)], True, 50)
        want = oracle.gather_windows(eo, centers)
        scale = np.sqrt(np.mean(eo ** 2, axis=1))
        assert np.max(np.abs(got - want) / scale[None, None, :]) <= TOL
    with pytest.raises(IndexError):
        api.features_to_windows([w], co, [np.asarray([8500])], True, 50)


def test_linearity_and_determinism_full_size(gpu):
    """configs[1] scale (a slice of the 4620-utterance corpus at full utterance length): scaling the
    int16 input by 2 scales every output by exactly 2 (power-of-two scaling is exact in
    floating point), and two runs are bit-identical."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    lengths = synth.corpus_lengths(256, seed=1)
    flat, _ = synth.corpus_waves_i16(lengths, seed=1, sigma=1500.0)
    plan = engine.plan_for(co)
    batch = plan.batch(lengths)
    a = batch.run(torch.from_numpy(flat).cuda(), lpf=True, cutoff=50, dec=True)["dec"].clone()
    b = batch.run(torch.from_numpy(flat).cuda(), lpf=True, cutoff=50, dec=True)["dec"].clone()
    c = batch.run(torch.from_numpy((flat * 2).astype(np.int16)).cuda(), lpf=True, cutoff=50, dec=True)["dec"]
    assert torch.equal(a, b)
    assert torch.isfinite(a).all() and (a >= 0).all()
    assert torch.equal(a * 2, c)


def test_long_stream_config4_subset(gpu, oracle):
    """configs[3], reduced to what the float64 oracle finishes quickly: one 75 s stream
    (1.2 M samples, N2 = 2^21, two-pass FFT), 256 channels on the GPU, parity on a 24-channel
    subset at the three cut-offs."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = load_golden("coefs.npz")["coefs_fs16000_c256_l100"]
    n = 1_200_000
    w = synth.white_noise_i16(n, seed=2)
    sub = np.r_[0:8, 124:132, 248:256]
    go = oracle.erb_filterbank(w, co[sub])
    plan = engine.plan_for(co)
    batch = plan.batch([n])
    assert batch.num_items > 2  # the stream is chunked in time
    wd = torch.from_numpy(w).cuda()
    for cut in (20, 50, 100):
        eo = oracle.extract_envelope(go, True, cut)
        res = batch.run(wd, lpf=True, cutoff=cut, env_t=True, dec=True)
        env = res["env_t"][:, torch.from_numpy(sub).cuda()].T.cpu().numpy()
        assert rel_err(env, eo).max() <= TOL, cut
        dec = res["dec"].cpu().numpy()[:, sub]
        assert np.array_equal(dec, env[:, ::160].T)


def test_error_behaviour(gpu):
    api, engine, filters, torch = gpu
    co = coefs128()
    assert api.erb_filterbank(np.zeros(0, dtype=np.int16), co).shape == (128, 0)
    with pytest.raises(ValueError):
        api.erb_filterbank(np.zeros((2, 10)), co)
    with pytest.raises(ValueError):
        api.extract_envelope_from_matrix(np.zeros((4, 0)))
    bad = co.copy()
    bad[3, 8] = 1.5  # unstable pole
    with pytest.raises(Exception):
        engine.Plan(bad)
    with pytest.raises(ValueError):
        api.dense_frames(np.zeros(4000, dtype=np.int16), co, True, 50, normalize=True)  # all-zero frames: min <= 0


def test_evalnoise_config5_frames_and_cnn_forward(gpu, oracle):
    """configs[4]: noise-mixed float64 utterance at 0/10/20 dB SNR -> filterbank -> envelope ->
    dense framing -> normalizeInput -> CNN forward (seeded weights; there is no Keras oracle,
    so the forward pass is checked for consistency between GPU-made and oracle-made frames)."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import cnn, synth
    co = coefs128()
    base = synth.speech_like_i16(8000, seed=31)
    rng = np.random.default_rng(3)
    model = cnn.seeded_model(0)
    for snr_db in (0, 10, 20):
        rms = np.sqrt(np.mean(base.astype(np.float64) ** 2))
        wave = base + rng.normal(scale=rms / 10 ** (snr_db / 20.0), size=base.shape[0])
        frames = api.dense_frames(wave, co, True, 50, normalize=True)
        nb = base.shape[0] - 11 * 160
        assert frames.shape == (nb, 11, 128) and frames.dtype == np.float64
        _, eo, _ = oracle.utterance(wave, co, True, 50)
        pick = [0, 1, 777, nb - 1]
        want = np.stack([oracle.normalize_input(oracle.dense_frames(eo, 5, 160, i, i + 1)[0]) for i in pick])
        # log-min-max domain, values in [0, 1]: the log amplifies the relative error of the
        # near-silent samples at the start of the utterance
        assert np.max(np.abs(frames[pick] - want)) <= 2e-3
        s_gpu = cnn.predict(model, torch.from_numpy(frames[pick]).cuda().float()).cpu().numpy()
        s_ref = cnn.predict(model, torch.from_numpy(want).cuda().float()).cpu().numpy()
        assert s_gpu.shape == (4, 2) and np.allclose(s_gpu.sum(axis=1), 1.0, atol=1e-5)
        assert np.max(np.abs(s_gpu - s_ref)) <= 5e-3
    # the tensor-core options of the forward pass (bf16 autocast, NHWC layout) against fp32 NCHW
    many = torch.from_numpy(frames[:512]).cuda().float()
    s32 = cnn.predict(cnn.seeded_model(0), many).cpu().numpy()
    s16 = cnn.predict(cnn.seeded_model(0), many, autocast_dtype=torch.bfloat16, channels_last=True).cpu().numpy()
    s32n = cnn.predict(cnn.seeded_model(0), many, channels_last=True).cpu().numpy()
    assert np.max(np.abs(s32n - s32)) <= 1e-4 and np.max(np.abs(s16 - s32)) <= 3e-2


def test_chunked_batch_uses_per_utterance_edge_table(gpu, oracle):
    """A batch that is split in time AND has many (utterance, channel) pairs takes the sequential
    edge kernel (the single-utterance tests above take the chunked-scan edge kernel); both must
    agree with the oracle and with the unsplit run."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    lens = [9000 + 37 * i for i in range(640)]
    waves = [synth.white_noise_i16(n, seed=500 + i) for i, n in enumerate(lens)]
    flat = torch.from_numpy(np.concatenate(waves)).cuda()
    plan = engine.plan_for(co)
    split = plan.batch(lens, target_items=4096)  # forced time chunks on a many-utterance batch
    whole = plan.batch(lens, target_items=1)   # one item per utterance, in-kernel edge pass
    assert split.num_items > whole.num_items == 640 * 4  # one CTA per (utterance, 32 channels)
    a = split.run(flat, lpf=True, cutoff=50, dec=True)["dec"].cpu().numpy()
    b = whole.run(flat, lpf=True, cutoff=50, dec=True)["dec"].cpu().numpy()
    for u in (0, 319, 639):
        _, eo, _ = oracle.utterance(waves[u], co, True, 50)
        f0, f1 = split.frame_offsets[u], split.frame_offsets[u + 1]
        want = eo[:, ::160].T
        scale = np.sqrt(np.mean(eo ** 2, axis=1))[None, :]
        assert np.max(np.abs(a[f0:f1] - want) / scale) <= TOL
        assert np.max(np.abs(b[f0:f1] - want) / scale) <= TOL
        assert np.max(np.abs(a[f0:f1] - b[f0:f1]) / scale) <= 2e-5


@pytest.mark.parametrize("fs,C,low,n,dtype", [(44100, 100, 50, 30000, np.float32), (8000, 37, 50, 12345, np.int16),
                                               (16000, 300, 100, 5000, np.float64)])
def test_other_filterbanks_and_dtypes(gpu, oracle, fs, C, low, n, dtype):
    """Channel counts that are not multiples of 32 / 128, other sample rates (slower poles ->
    longer warm-ups derived at plan creation), float32 / float64 waves, whole and chunked."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = filters.make_erb_filters(fs, filters.centre_freqs(fs, C, low))
    w = synth.white_noise_i16(n, seed=n).astype(dtype)
    go = oracle.erb_filterbank(w, co)
    eo = oracle.extract_envelope(go, True, 50)
    plan = engine.plan_for(co)
    wd = torch.from_numpy(w).cuda()
    for target in (1, 0, 64):
        res = plan.batch([n], target_items=target).run(wd, lpf=True, cutoff=50, gfb=torch.float64, env=torch.float64,
                                                       dec=True)
        gfb = res["gfb"].cpu().numpy().reshape(C, n)
        env = res["env"].cpu().numpy().reshape(C, n)
        assert rel_err(gfb, go).max() <= TOL, (target, "gfb")
        assert rel_err(env, eo).max() <= TOL, (target, "env")
        assert np.array_equal(res["dec"].cpu().numpy(), env[:, ::160].astype(np.float32).T)


def test_corpus_sized_request_takes_the_pipelined_path(gpu, monkeypatch):
    """features_to_windows on many utterances: the sub-batched, three-stream pipeline returns
    exactly what the single-launch path returns."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    lengths = synth.corpus_lengths(96, lo=8000, hi=16000, seed=4)
    waves = [synth.white_noise_i16(int(n), seed=900 + i) for i, n in enumerate(lengths)]
    tps = [synth.label_grid(int(n)) for n in lengths]
    a = api.features_to_windows(waves, co, tps, True, 50)
    monkeypatch.setattr(api, "_PIPELINE_BYTES", 1)
    b = api.features_to_windows(waves, co, tps, True, 50)
    assert a.shape == b.shape == (sum(len(t) for t in tps), 11, 128)
    # sub-batches run whole utterances (no time chunks) while the single launch of a 96-utterance
    # batch splits them: same values to float32 noise, not bit for bit
    scale = np.sqrt(np.mean(a.astype(np.float64) ** 2, axis=(0, 1)))
    assert np.max(np.abs(a - b) / scale[None, None, :]) <= 5e-5


def test_long_stream_config4_full_length(gpu, oracle):
    """configs[3] at its full size on the GPU: 600 s (9.6 M samples, N2 = 2^24), 256 channels,
    cut-off 20 Hz (the slowest low-pass pole); the float64 oracle checks four channels."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = load_golden("coefs.npz")["coefs_fs16000_c256_l100"]
    n = 9_600_000
    w = synth.white_noise_i16(n, seed=2)
    sub = np.array([0, 85, 170, 255])
    eo = oracle.extract_envelope(oracle.erb_filterbank(w, co[sub]), True, 20)
    plan = engine.plan_for(co)
    batch = plan.batch([n])
    assert batch.num_items >= 148
    dec = batch.run(torch.from_numpy(w).cuda(), lpf=True, cutoff=20, dec=True)["dec"].cpu().numpy()
    assert dec.shape == (60000, 256)
    want = eo[:, ::160].T
    scale = np.sqrt(np.mean(eo ** 2, axis=1))[None, :]
    assert np.max(np.abs(dec[:, sub] - want) / scale) <= TOL


def test_fuzz_random_shapes(gpu, oracle):
    """Seeded fuzz over lengths (incl. rings shorter than a tile and powers of two), channel
    counts, sample dtypes, cut-offs, decimation grids and time-chunk targets, in ragged batches."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    rng = np.random.default_rng(2024)
    special = [255, 256, 257, 1023, 1024, 4096, 8191, 8192, 32768, 32769]
    for case in range(16):
        C = int(rng.choice([1, 5, 32, 33, 64, 100, 128, 129, 200]))
        fs = int(rng.choice([16000, 16000, 8000, 22050]))
        co = filters.make_erb_filters(fs, filters.centre_freqs(fs, C, int(rng.choice([50, 100, 200]))))
        U = int(rng.integers(1, 5))
        lens = [int(rng.choice(special)) if rng.random() < 0.4 else int(rng.integers(300, 40000)) for _ in range(U)]
        dtype = [np.int16, np.float32, np.float64][int(rng.integers(0, 3))]
        waves = [synth.white_noise_i16(n, seed=1000 * case + i).astype(dtype) for i, n in enumerate(lens)]
        lpf = bool(rng.random() < 0.7)
        cutoff = float(rng.choice([20, 50, 100, 400]))
        step = int(rng.choice([160, 80, 100, 7]))
        phase = int(rng.integers(0, step))
        target = int(rng.choice([0, 1, 16, 512]))
        plan = engine.plan_for(co)
        batch = plan.batch(lens, step=step, phase=phase, target_items=target)
        flat = torch.from_numpy(np.concatenate(waves)).cuda()
        res = batch.run(flat, lpf=lpf, cutoff=cutoff, gfb=torch.float64, env=torch.float64, dec=True)
        dec_only = batch.run(flat, lpf=lpf, cutoff=cutoff, dec=True)["dec"].cpu().numpy()
        gfb_all, env_all, dec_all = res["gfb"].cpu().numpy(), res["env"].cpu().numpy(), res["dec"].cpu().numpy()
        off = 0
        tag = (case, C, fs, lens, dtype.__name__, lpf, cutoff, step, phase, target)
        for u, (n, w) in enumerate(zip(lens, waves)):
            go = oracle.erb_filterbank(w, co)
            eo = oracle.extract_envelope(go, lpf, cutoff)
            gfb = gfb_all[C * off:C * (off + n)].reshape(C, n)
            env = env_all[C * off:C * (off + n)].reshape(C, n)
            sg = np.maximum(np.sqrt(np.mean(go ** 2, axis=1)), 1e-3 * np.abs(go).max())
            se = np.maximum(np.sqrt(np.mean(eo ** 2, axis=1)), 1e-3 * np.abs(eo).max())
            assert rel_err(gfb, go, sg).max() <= TOL, tag
            assert rel_err(env, eo, se).max() <= TOL, tag
            f0, f1 = batch.frame_offsets[u], batch.frame_offsets[u + 1]
            assert f1 - f0 == len(range(phase, n, step)), tag
            assert np.array_equal(dec_all[f0:f1], env[:, phase::step].astype(np.float32).T), tag
            assert np.max(np.abs(dec_only[f0:f1] - eo[:, phase::step].T) / se[None, :]) <= TOL, tag
            off += n


def test_warmup_lengths_are_what_keeps_truncation_below_float32(gpu, oracle):
    """f2_plan_set_warmup: the defaults derived from the slowest pole hold parity; cutting the
    history to 256 samples visibly breaks it (so the truncated-history design is load-bearing and
    its lengths are not arbitrary)."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    w = synth.white_noise_i16(30000, seed=12)
    _, eo, _ = oracle.utterance(w, co, True, 50)
    plan = engine.Plan(co)  # private plan: the cached one must keep its defaults
    wi, we, wc = plan.get_warmup()
    assert (wi, we, wc) == (1536, 2048, 2048)  # 21.5 / -ln r and 29 / -ln r for r = 0.98590, tile-rounded
    wd = torch.from_numpy(w).cuda()
    good = plan.batch([30000], target_items=8).run(wd, lpf=True, cutoff=50, env=torch.float64)["env"].cpu().numpy()
    assert rel_err(good.reshape(128, -1), eo).max() <= TOL
    plan.set_warmup(256, 256, 256)
    assert plan.get_warmup() == (256, 256, 256)
    bad = plan.batch([30000], target_items=8).run(wd, lpf=True, cutoff=50, env=torch.float64)["env"].cpu().numpy()
    assert rel_err(bad.reshape(128, -1), eo).max() > 10 * TOL


def test_fused_window_store_equals_decimated_frames_plus_gather(gpu, oracle):
    """`windows` output mode of f2_batch_run: for the label grid (window k = decimated frames
    k..k+dots-1, k < max(n//step - dots - 1, 0): LabelDataGenerator.py:38-50 + InputGenerator.py:73-80)
    the fused kernel stores every frame into the window rows that contain it.  Pure placement: bit
    for bit the decimated frames + gather, on ragged batches with too-short utterances, with time
    chunks, other radii / steps, a channel count that is not a multiple of 32, with and without
    low-pass; and equal to the oracle's windows."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    for C, lens, dots, step, lpf, target in (
            (128, [9000, 1700, 48000, 1919, 1920, 2081, 33000], 11, 160, True, 0),
            (128, [60000], 11, 160, True, 64),            # one utterance in time chunks
            (40, [5000, 12345, 800], 5, 80, False, 0),
            (7, [4000, 4001], 3, 100, True, 16)):
        co = filters.make_erb_filters(16000, filters.centre_freqs(16000, C, 100))
        waves = [synth.white_noise_i16(n, seed=40 + i) for i, n in enumerate(lens)]
        flat = torch.from_numpy(np.concatenate(waves)).cuda()
        plan = engine.plan_for(co)
        batch = plan.batch(lens, step=step, target_items=target)
        offs, rows = batch.grid_windows(dots)
        nb = [max(n // step - dots - 1, 0) for n in lens]
        assert rows == sum(nb) and offs.cpu().tolist() == np.concatenate([[0], np.cumsum(nb)]).tolist()
        win = torch.full((rows, dots, C), float("nan"), dtype=torch.float32, device="cuda")
        batch.run(flat, lpf=lpf, cutoff=50, windows=(offs, dots, win))
        dec = batch.run(flat, lpf=lpf, cutoff=50, dec=True)["dec"]
        base = np.concatenate([batch.frame_offsets[u] + np.arange(nb[u]) for u in range(len(lens))]).astype(np.int64)
        want = engine.gather_windows(dec, torch.from_numpy(base).cuda(), dots, 1)
        assert not torch.isnan(win).any()          # every entry of every row was written
        assert torch.equal(win, want)
        # and against the reference algorithm: rows of GenerateInputData for that label grid
        u = int(np.argmax(lens))
        _, eo, wo = oracle.utterance(waves[u], co, lpf, 50, step * (dots // 2) + step * np.arange(nb[u]), dots // 2, step)
        r0 = int(offs[u].item())
        scale = np.sqrt(np.mean(eo ** 2, axis=1))
        assert np.max(np.abs(win[r0:r0 + nb[u]].cpu().numpy() - wo) / scale[None, None, :]) <= TOL
    with pytest.raises(ValueError):
        batch.run(flat, lpf=True, cutoff=50, dec=True, windows=(offs, dots, win))


def test_banks_outside_the_float32_tolerance_raise_instead_of_answering(gpu, oracle, monkeypatch):
    """make_erb_filters(fs, cf, width) is public API (gammatone/filters.py:89): a bank whose poles sit so
    close to z = 1 that float32 cannot hold 1e-4 x RMS (LOW_FREQ = 20 Hz, width = 2: the family the
    round-1 fuzz found at 4.7x the bar, profiles/r01o_fuzz.log) must be an error, not a quiet answer.
    f2_plan_create predicts the error by running the worst channels on the host in float32 and float64;
    with the override the prediction is shown to be what the device then does."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import _native, synth
    fs, C, n = 16000, 96, 4111
    co = filters.make_erb_filters(fs, filters.centre_freqs(fs, C, 20), 2.0)
    predicted, channel = engine.bank_check(co)
    assert predicted > 1.0
    with pytest.raises(_native.F2Error) as exc:
        engine.Plan(co)
    assert exc.value.code == _native.F2_ERR_UNSUPPORTED and "float32" in str(exc.value)
    with pytest.raises(_native.F2Error):
        api.erb_filterbank(synth.tone_i16(n, freq=4000.0), co)
    # the same bank with the check overridden: white noise is fine, the loud stop-band tone is not, and
    # the prediction was the tone's error
    monkeypatch.setenv("F2CNN_B200_ALLOW_IMPRECISE", "1")
    plan = engine.Plan(co)
    worst = {}
    for kind, w in (("white", synth.white_noise_i16(n, seed=32)), ("tone", synth.tone_i16(n, freq=fs / 4.0, fs=fs))):
        go = oracle.erb_filterbank(w, co)
        gfb = plan.batch([n]).run(torch.from_numpy(w).cuda(), gfb=torch.float64)["gfb"].cpu().numpy().reshape(C, n)
        scale = np.sqrt(np.mean(go ** 2, axis=1))
        scale = np.maximum(scale, 0.01 * scale.max())
        worst[kind] = float((np.max(np.abs(gfb - go), axis=1) / scale).max()) / TOL
    assert worst["white"] <= 1.0
    assert worst["tone"] > 1.0 and abs(worst["tone"] - predicted) <= 0.25 * predicted
    # the configured bank and its neighbours stay far inside
    for low, width in ((100, 1.0), (100, 2.0), (50, 1.0)):
        assert engine.bank_check(filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, low), width))[0] < 0.5


def test_degenerate_requests_of_the_pipeline_and_the_framing(gpu):
    """No utterances / no windows through the corpus pipeline, and dense frames that would read past the
    envelope (the C ABI takes bare pointers: the bound travels with the call)."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import _native
    plan = engine.plan_for(coefs128())
    pipe = engine.WindowPipeline(plan, np.zeros(0, dtype=np.int64))
    assert pipe.subs == [] and pipe.total_frames == 0
    out = np.zeros((0, 11, 128), np.float32)
    pipe.run(torch.zeros(0, dtype=torch.int16), np.zeros((0, 3), np.int64), out)
    pipe = engine.WindowPipeline(plan, [3000, 1200])            # too short for any window
    runs, _, n_rows = engine.window_runs(np.zeros(0, np.int64), [0, 0], [3000, 1200], pipe.frame_offsets)
    assert n_rows == 0 and runs.shape == (0, 3)
    pipe.run(torch.zeros(4200, dtype=torch.int16).pin_memory(), runs, out)
    env_t = torch.rand((2000, 128), device="cuda") + 0.1
    frames, flag = engine.dense_frames(env_t, 11, 160, 0, 2000 - 1760 + 160)
    assert frames.shape[0] == 400 and int(flag.item()) == 0
    with pytest.raises(_native.F2Error):
        engine.dense_frames(env_t, 11, 160, 0, 401)


def test_corpus_pipeline_input_forms_out_argument_and_fallthrough(gpu, monkeypatch):
    """The pipelined path of features_to_windows: pinned flat buffer, pageable flat buffer and list of arrays
    give the same bits; out= is filled in place and validated; timepoints in flat (centres, counts) form;
    a request whose LATER utterances leave the grid (a wrapping window) falls through to the general path."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    lengths = synth.corpus_lengths(40, lo=6000, hi=15000, seed=6)
    waves = [synth.white_noise_i16(int(n), seed=300 + i) for i, n in enumerate(lengths)]
    tps = [synth.label_grid(int(n)) for n in lengths]
    flat = np.concatenate(waves)
    counts = np.asarray([len(t) for t in tps])
    monkeypatch.setattr(api, "_PIPELINE_BYTES", 1)
    a = api.features_to_windows((torch.from_numpy(flat).pin_memory(), lengths), co, tps, True, 50)
    b = api.features_to_windows((flat, lengths), co, np.concatenate(tps), True, 50, counts=counts)
    c = api.features_to_windows(waves, co, tps, True, 50)
    assert a.shape == (counts.sum(), 11, 128) and np.array_equal(a, b) and np.array_equal(a, c)
    out = np.full_like(a, np.nan)
    assert api.features_to_windows((flat, lengths), co, tps, True, 50, out=out) is out and np.array_equal(out, a)
    with pytest.raises(ValueError):
        api.features_to_windows((flat, lengths), co, tps, True, 50, out=np.zeros((3, 11, 128), np.float32))
    with pytest.raises(ValueError):
        api.features_to_windows((flat, lengths), co, tps, True, 50, shard=(0, 2))      # shard needs the shared out
    # shards of a 3-way split into one array == the whole
    parts = np.zeros_like(a)
    for r in range(3):
        api.features_to_windows((flat, lengths), co, tps, True, 50, out=parts, shard=(r, 3))
    assert np.array_equal(parts, a)
    # utterance 20 gets a window that wraps like a negative Python index: legal, but not a run of frames
    tps2 = [t.copy() for t in tps]
    tps2[20] = np.concatenate([[160], tps2[20]])
    d = api.features_to_windows(waves, co, tps2, True, 50)
    row20 = int(counts[:20].sum())
    scale = np.sqrt(np.mean(a.astype(np.float64) ** 2, axis=(0, 1)))[None, None, :]
    assert d.shape[0] == a.shape[0] + 1
    # same values as the pipelined result up to float32 noise (the single batch splits utterances in time)
    assert np.max(np.abs(np.delete(d, row20, axis=0) - a) / scale) <= 5e-5
    with pytest.raises(IndexError):
        bad = [t.copy() for t in tps]
        bad[30] = np.concatenate([bad[30], [int(lengths[30]) - 100]])
        api.features_to_windows(waves, co, bad, True, 50)


def test_one_kernel_ring_transform_sizes(gpu, oracle):
    """The cluster kernels that transform rings of 32768, 65536 (every corpus utterance) and 131072 samples in
    distributed shared memory: Im(paddedHilbert) of rows on both sides of its size range against the float64
    oracle (EnvelopeExtraction.py:20-36), including the sizes next to it that take the multi-pass kernels."""
    api, engine, filters, torch = gpu
    rng = np.random.default_rng(21)
    for n in (16384, 16385, 20001, 32768, 32769, 47001, 65535, 65536, 65537, 100003, 131072, 131073):
        m = rng.normal(0.0, 3000.0, (3, n))
        got = api.hilbert_imag_rows(m)
        for r in range(3):
            want = oracle.padded_hilbert(m[r]).imag
            assert np.max(np.abs(got[r] - want)) <= 1e-5 * np.sqrt(np.mean(want ** 2)), n


def test_ring_transform_is_independent_of_the_batch_and_of_wave_alignment(gpu):
    """An utterance gives the same bits alone, in a batch of hundreds (many clusters in flight, odd and even
    offsets into the int16 buffer: the cluster kernel's aligned and unaligned pair loads) and on a second run."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    plan = engine.plan_for(co)
    rng = np.random.default_rng(5)
    lens = rng.integers(16385, 65537, size=300).astype(np.int64)
    lens[::7] += 1 - (lens[::7] & 1)          # some odd lengths: the next utterance starts at an odd sample
    waves = [synth.white_noise_i16(int(n), seed=100 + i) for i, n in enumerate(lens)]
    flat = torch.from_numpy(np.concatenate(waves)).cuda()
    batch = plan.batch(lens, target_items=1)
    first = batch.run(flat, lpf=True, cutoff=50, dec=True)["dec"].cpu().numpy()
    again = batch.run(flat, lpf=True, cutoff=50, dec=True)["dec"].cpu().numpy()
    assert np.array_equal(first, again)
    for u in (0, 1, 6, 7, 8, 150, 299):
        single = plan.batch([int(lens[u])], target_items=1).run(torch.from_numpy(waves[u]).cuda(), lpf=True, cutoff=50,
                                                                 dec=True)["dec"].cpu().numpy()
        assert np.array_equal(single, first[batch.frame_offsets[u]:batch.frame_offsets[u + 1]]), u


def test_shared_injection_tables_equal_private_ones(gpu, oracle):
    """Ring sizes 2^8..2^20 read the injection kernel G from one table per size (four shifted copies);
    smaller and larger rings tabulate it per utterance.  Lengths on both sides of both limits, every
    residue of n mod 4 (which copy is read), against the oracle."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    for n in (120, 128, 129, 255, 256, 257, 1021, 1022, 1023, 1024, 4097):
        w = synth.white_noise_i16(n, seed=n)
        _, env = api.filterbank_envelope(w, co, False, 100, with_gfb=True)
        _, eo, _ = oracle.utterance(w, co, False, 100)
        tol = TOL if n >= 255 else 2e-3   # rings shorter than a tile: DESIGN.md section 2 (ii)
        assert rel_err(env, eo).max() <= tol, n


def test_pinned_block_is_addressable_from_kernels(gpu):
    """engine._pinned_empty: huge-page mapping registered with CUDA (f2_host_pin).  The fused kernel stores
    decimated frames straight into it; the result equals the device-buffer result."""
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    co = coefs128()
    plan = engine.plan_for(co)
    w = synth.white_noise_i16(40000, seed=3)
    batch = plan.batch([40000], target_items=1)
    host = engine._pinned_empty(batch.total_frames * 128, torch.float32).view(-1, 128)
    assert host.is_pinned()
    host.zero_()
    dev = batch.run(torch.from_numpy(w).cuda(), lpf=True, cutoff=50, dec=True)["dec"]
    batch.run(torch.from_numpy(w).cuda(), lpf=True, cutoff=50, out={"dec": host})
    torch.cuda.synchronize()
    assert np.array_equal(host.numpy(), dev.cpu().numpy())


def test_frame_windows_are_views_of_the_decimated_frames(gpu, monkeypatch):
    """api.features_to_frames: the windows of the label grid as overlapping views of the decimated frames --
    equal, bit for bit, to the rows api.features_to_windows builds on its corpus path (whole utterances);
    materialize() is that tensor; a shard holds its own utterances only."""
    api, engine, filters, torch = gpu
    monkeypatch.setattr(api, "_PIPELINE_BYTES", 0)   # a small corpus takes the corpus path too
    from f2cnn_b200 import synth
    co = coefs128()
    rng = np.random.default_rng(17)
    lens = rng.integers(1500, 9000, size=37).astype(np.int64)
    lens[5] = 1700                       # too short for a single window of the grid: 0 rows
    waves = [synth.white_noise_i16(int(n), seed=300 + i) for i, n in enumerate(lens)]
    nwin = np.maximum((lens / 160 - 12).astype(np.int64), 0)
    assert nwin[5] == 0
    centers = [800 + 160 * np.arange(k, dtype=np.int64) for k in nwin]
    want = api.features_to_windows(waves, co, centers, True, 50)
    flat = torch.from_numpy(np.concatenate(waves))
    for source in (waves, (flat, lens)):
        fw = api.features_to_frames(source, co, True, 50)
        assert len(fw) == want.shape[0] and np.array_equal(fw.counts, nwin)
        row = 0
        for u, k in enumerate(nwin):
            v = fw.windows(u)
            assert v.shape == (k, 11, 128) and (k == 0 or not v.flags["OWNDATA"])
            assert np.array_equal(v, want[row:row + k]), u
            row += int(k)
        for r in (0, 1, int(nwin[0]), want.shape[0] - 1, -1):
            assert np.array_equal(fw[r], want[r])
        with pytest.raises(IndexError):
            fw[want.shape[0]]
        assert np.array_equal(fw.materialize(), want)
    halves = [api.features_to_frames((flat, lens), co, True, 50, shard=(r, 2)) for r in range(2)]
    assert sorted(np.concatenate([h.utterances for h in halves]).tolist()) == list(range(37))
    first_row = np.concatenate([[0], np.cumsum(nwin)])
    for h in halves[::-1]:               # the second shard's buffer is still its own (another pipeline)
        for j, u in enumerate(h.utterances):
            assert np.array_equal(h.windows(j), want[first_row[u]:first_row[u + 1]]), u
    with pytest.raises(IndexError):
        api.features_to_frames(waves, co, True, 50, counts=nwin + 3)


def test_multi_pass_prepass_agrees_with_the_cluster_kernels(gpu):
    """F2CNN_B200_RING_CLUSTER=0 sends rings of 32768 / 65536 / 131072 samples through the generic
    multi-pass kernels (fft_cols / fft_rows / hilbert_mask, which serve every other ring size and are kept
    as the cluster kernels' cross-check): a child process computes the same decimated envelopes that way;
    the two agree far inside the tolerance (different FFT factorisations)."""
    import os
    import subprocess
    import sys
    import tempfile
    api, engine, filters, torch = gpu
    from f2cnn_b200 import synth
    lens = [20000, 40000, 65536, 70001]
    code = (
        "import sys, numpy as np, torch\n"
        "sys.path.insert(0, %r)\n"
        "from f2cnn_b200 import engine, synth\n"
        "from f2cnn_b200.gammatone import filters\n"
        "co = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))\n"
        "lens = %r\n"
        "flat = torch.from_numpy(np.concatenate([synth.white_noise_i16(n, seed=900 + i) for i, n in enumerate(lens)])).cuda()\n"
        "dec = engine.plan_for(co).batch(lens, target_items=1).run(flat, lpf=True, cutoff=50, dec=True)['dec']\n"
        "np.save(sys.argv[1], dec.cpu().numpy())\n" % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), lens))
    out = {}
    with tempfile.TemporaryDirectory() as d:
        for flag in ("1", "0"):
            path = os.path.join(d, "dec%s.npy" % flag)
            subprocess.run([sys.executable, "-c", code, path], check=True, env=dict(os.environ, F2CNN_B200_RING_CLUSTER=flag),
                           timeout=300)
            out[flag] = np.load(path).astype(np.float64)
    assert out["1"].shape == out["0"].shape and not np.array_equal(out["1"], out["0"])   # really two code paths
    rms = np.sqrt(np.mean(out["0"] ** 2, axis=0))
    assert (np.max(np.abs(out["1"] - out["0"]), axis=0) / rms).max() <= 2e-5
