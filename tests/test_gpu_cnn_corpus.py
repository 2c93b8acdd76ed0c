"""Scoring many utterances with the tensor-core CNN in one pass (f2_cnn_forward_segments,
TensorCoreCNN.predict_segments, api.cnn_evaluate_corpus).

Each frame's arithmetic in the three kernels depends on that frame alone, so the bar at the network stage is
exact equality with the one-utterance calls.  End to end, the corpus call runs whole utterances through the
front end (never time chunks); its scores are therefore compared bit for bit with the network on the envelope
of a whole-utterance batch, and with cnn_evaluate wherever cnn_evaluate does not split the lone utterance into
time chunks.  Where it does, both are held to the float32 forward on the float64 oracle's envelope with the 5e-3
score bound of test_gpu_cnn.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEP = 160
DOTS = 11


def _coefs():
    from f2cnn_b200.gammatone import filters
    return filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))


def _wave(n, seed, dtype):
    """A speech-like utterance with a little noise (no stretch of exact zeros)."""
    from f2cnn_b200 import synth
    rng = np.random.default_rng(seed + 7)
    w = synth.speech_like_i16(n, seed=seed) if n else np.zeros(0, np.int16)
    if dtype == np.int16:
        w = (w.astype(np.int32) + rng.integers(-40, 41, n)).clip(-32768, 32767)
        return np.where(w == 0, 1, w).astype(np.int16)
    return w.astype(np.float64) + rng.normal(0, 30, n)


def _nb(n):
    return max(int(n) - DOTS * STEP, 0)


def _oracle_scores(model, env_t, torch):
    """normalizeInput (float64) + the float32 network on every stride-1 frame of env_t ([n, 128] device)."""
    nb = env_t.shape[0] - DOTS * STEP
    out = []
    for i0 in range(0, nb, 4096):
        i1 = min(i0 + 4096, nb)
        idx = torch.arange(i0, i1, device=env_t.device)[:, None] + STEP * torch.arange(DOTS, device=env_t.device)[None, :]
        fr = env_t[idx].double()
        lo = fr.amin(dim=(1, 2), keepdim=True).log()
        hi = fr.amax(dim=(1, 2), keepdim=True).log()
        with torch.no_grad():
            out.append(model(((fr.log() - lo) / (hi - lo)).float()))
    return torch.cat(out)


@pytest.fixture(scope="module")
def setup():
    import torch
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    from f2cnn_b200 import cnn, engine
    model = cnn.seeded_model(seed=3)
    return torch, cnn, engine, model, cnn.TensorCoreCNN(model)


# frames per utterance: 1 and 0 around chunk-sized ones, so that the second chunk (frames 32 768 .. 65 535)
# holds the last frame of utterance 0, utterances 1 .. 3 and the start of utterance 4
NBS = (32769, 1, 0, 5, 32767, -860, 32768, 3)
LENGTHS = [nb + DOTS * STEP for nb in NBS]


@pytest.mark.parametrize("dtype", [np.int16, np.float64])
@pytest.mark.parametrize("lpf", [True, False])
def test_segments_equal_the_per_utterance_calls_bit_for_bit(setup, dtype, lpf):
    torch, cnn, engine, model, net = setup
    waves = [_wave(n, 100 + i, dtype) for i, n in enumerate(LENGTHS)]
    plan = engine.plan_for(_coefs())
    batch = plan.batch(LENGTHS, step=STEP, target_items=1)
    env_t = batch.run(torch.from_numpy(np.concatenate(waves)).cuda(), lpf=lpf, cutoff=50, env_t=True)["env_t"]
    rows = batch.sample_offsets[:-1]
    counts = np.asarray([_nb(n) for n in LENGTHS])
    got = net.predict_segments(env_t, STEP, rows, counts)
    assert got.shape == (int(counts.sum()), 2)
    at = 0
    for r, k in zip(rows, counts):
        want = net.predict_envelope(env_t, STEP, frames=(int(r), int(r + k)))
        assert torch.equal(got[at:at + k], want)
        at += int(k)
    # segments need not follow the utterances: any frame ranges of env_t, in any order, zero-frame ones included
    segs = [(40000, 300), (int(rows[-1]), 0), (0, 33000), (5, 7)]
    got = net.predict_segments(env_t, STEP, [s[0] for s in segs], [s[1] for s in segs])
    want = torch.cat([net.predict_envelope(env_t, STEP, frames=(r, r + k)) for r, k in segs])
    assert torch.equal(got, want)

    # end to end, in sub-batches of two or three utterances: the same scores as the one whole-utterance batch
    from f2cnn_b200 import api
    old = api._CNN_ENV_BYTES
    api._CNN_ENV_BYTES = 3 * 35000 * 128 * 4
    try:
        scores, offsets = api.cnn_evaluate_corpus(waves, _coefs(), model, LPF=lpf, CUTOFF=50)
    finally:
        api._CNN_ENV_BYTES = old
    assert np.array_equal(offsets, np.concatenate([[0], np.cumsum(counts)]))
    assert scores.dtype == np.float32 and np.array_equal(scores, net.predict_segments(env_t, STEP, rows, counts).cpu().numpy())


def test_corpus_against_cnn_evaluate_and_the_oracle(setup, oracle):
    torch, cnn, engine, model, net = setup
    from f2cnn_b200 import api
    co = _coefs()
    plan = engine.plan_for(co)
    lengths = (9000, 48000, 20000)
    waves = [_wave(n, 200 + i, np.float64) for i, n in enumerate(lengths)]
    scores, offsets = api.cnn_evaluate_corpus(waves, co, model, LPF=True, CUTOFF=50)
    # (flat, lengths) input gives the same
    flat = np.concatenate(waves)
    again, _ = api.cnn_evaluate_corpus((flat, np.asarray(lengths)), co, model, LPF=True, CUTOFF=50)
    assert np.array_equal(scores, again)
    chunked = 0
    for u, (w, n) in enumerate(zip(waves, lengths)):
        mine = scores[offsets[u]:offsets[u + 1]]
        single, none = api.cnn_evaluate(w, co, model, True, 50, with_envelopes=False)
        assert none is None and single.shape == mine.shape == (_nb(n), 2)
        whole = plan.batch([n], step=STEP, target_items=1)
        env_whole = whole.run(torch.from_numpy(w).cuda(), lpf=True, cutoff=50, env_t=True)["env_t"]
        assert np.array_equal(mine, net.predict_envelope(env_whole, STEP).cpu().numpy())
        if plan.batch([n], step=STEP).num_items == whole.num_items:
            # cnn_evaluate ran the utterance whole as well: the same envelope, the same scores
            assert np.array_equal(mine, single)
        else:
            chunked += 1
            _, eo, _ = oracle.utterance(w, co, True, 50)
            ref = _oracle_scores(model, torch.from_numpy(eo.T.copy()).cuda().float(), torch).cpu().numpy()
            assert float(np.abs(mine - ref).max()) <= 5e-3
            assert float(np.abs(single - ref).max()) <= 5e-3
    print("utterances cnn_evaluate splits into time chunks: %d of %d" % (chunked, len(lengths)))
    with pytest.raises(ValueError):
        api.cnn_evaluate_corpus(waves, co, model, radius=4)
    with pytest.raises(ValueError):
        api.cnn_evaluate_corpus(waves, co[:64], model)
    with pytest.raises(ValueError):
        api.cnn_evaluate_corpus(waves, co, model, out=np.zeros((3, 2), np.float32))


def test_non_positive_value_names_the_utterance(setup):
    torch, cnn, engine, model, net = setup
    from f2cnn_b200 import api
    co = _coefs()
    waves = [_wave(6000, 300 + i, np.int16) for i in range(5)]
    waves[3] = np.zeros(6000, np.int16)    # an all-zero envelope: normalizeInput raises ValueError
    old = api._CNN_ENV_BYTES
    api._CNN_ENV_BYTES = 2 * 6000 * 128 * 4   # the bad utterance is in the second sub-batch
    try:
        with pytest.raises(ValueError, match=r"positive \(utterance 3\)"):
            api.cnn_evaluate_corpus(waves, co, model)
    finally:
        api._CNN_ENV_BYTES = old
    with pytest.raises(ValueError, match="positive"):
        api.cnn_evaluate(waves[3], co, model, with_envelopes=False)
    # the network stage names the segment
    plan = engine.plan_for(co)
    batch = plan.batch([6000] * 5, step=STEP, target_items=1)
    env_t = batch.run(torch.from_numpy(np.concatenate(waves)).cuda(), env_t=True)["env_t"]
    with pytest.raises(cnn.NonPositiveInput) as exc:
        net.predict_segments(env_t, STEP, batch.sample_offsets[:-1], [_nb(6000)] * 5)
    assert exc.value.segment == 3
    ok = [0, 1, 2, 4]
    assert net.predict_segments(env_t, STEP, batch.sample_offsets[ok], [_nb(6000)] * 4).shape == (4 * _nb(6000), 2)


def _shard_corpus():
    from f2cnn_b200 import synth
    lengths = synth.corpus_lengths(12, lo=1000, hi=40000, seed=5)
    return lengths, np.concatenate([_wave(int(n), 400 + i, np.int16) for i, n in enumerate(lengths)])


def test_shards_fill_one_shared_array_like_the_single_call(setup, tmp_path):
    torch, cnn, engine, model, net = setup
    from f2cnn_b200 import api, hostmem
    co = _coefs()
    lengths, flat = _shard_corpus()
    whole, offsets = api.cnn_evaluate_corpus((flat, lengths), co, model, True, 50)
    shared = hostmem.SharedArray(str(tmp_path / "scores.f32"), whole.shape, np.float32, create=True)
    shared.array[...] = np.nan
    old = api._CNN_ENV_BYTES
    api._CNN_ENV_BYTES = 60000 * 128 * 4     # several sub-batches per shard
    try:
        for r in range(2):
            out, off = api.cnn_evaluate_corpus((flat, lengths), co, model, True, 50, out=shared.array, shard=(r, 2))
            assert out is shared.array and np.array_equal(off, offsets)
    finally:
        api._CNN_ENV_BYTES = old
    assert np.array_equal(shared.array, whole)
    with pytest.raises(ValueError):
        api.cnn_evaluate_corpus((flat, lengths), co, model, True, 50, shard=(0, 2))    # no shared `out`
    with pytest.raises(ValueError, match="host memory"):
        api.cnn_evaluate_corpus((torch.from_numpy(flat).cuda(), lengths), co, model, True, 50)
    if torch.cuda.device_count() < 2:
        return
    # one process per device, both writing into the one mapping
    shared.array[...] = np.nan
    np.savez(str(tmp_path / "corpus.npz"), flat=flat, lengths=lengths)
    code = (
        "import sys, numpy as np, torch\n"
        "sys.path.insert(0, %r)\n"
        "from f2cnn_b200 import api, cnn, hostmem\n"
        "from f2cnn_b200.gammatone import filters\n"
        "rank, d = int(sys.argv[1]), sys.argv[2]\n"
        "torch.cuda.set_device(rank)\n"
        "z = np.load(d + '/corpus.npz')\n"
        "co = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))\n"
        "out = hostmem.SharedArray(d + '/scores.f32', (%d, 2), np.float32)\n"
        "api.cnn_evaluate_corpus((z['flat'], z['lengths']), co, cnn.seeded_model(seed=3), True, 50, out=out.array,\n"
        "                        shard=(rank, 2))\n" % (ROOT, whole.shape[0]))
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r), str(tmp_path)]) for r in range(2)]
    try:
        assert [p.wait(timeout=600) for p in procs] == [0, 0]
    finally:
        for p in procs:     # a rank that did not finish must not stay behind on its GPU
            if p.poll() is None:
                p.kill()
                p.wait()
    assert np.array_equal(shared.array, whole)


def test_abi_rejects_segments_past_the_envelope_and_a_short_workspace(setup):
    torch, cnn, engine, model, net = setup
    import ctypes
    from f2cnn_b200 import _native
    L = _native.lib()
    n = 6000
    env_t = engine.plan_for(_coefs()).batch([n]).run(torch.from_numpy(_wave(n, 500, np.float64)).cuda(), env_t=True)["env_t"]
    last = n - (DOTS - 1) * STEP       # frames [0, last) read rows up to n - 1

    def call(rows, frames, ws_bytes=None):
        rows = np.asarray(rows, np.int64)
        frames = np.asarray(frames, np.int64)
        total = max(int(frames.sum()), 1)
        net._workspace(total)
        need = int(L.f2_cnn_workspace_bytes(net._h, total))
        scores = torch.zeros((total, 2), device="cuda")
        flags = torch.zeros(len(rows) + 1, dtype=torch.int32, device="cuda")
        rc = L.f2_cnn_forward_segments(net._h, ctypes.c_void_p(env_t.data_ptr()), n, STEP,
                                       rows.ctypes.data_as(ctypes.c_void_p), frames.ctypes.data_as(ctypes.c_void_p),
                                       len(rows), ctypes.c_void_p(scores.data_ptr()), ctypes.c_void_p(flags.data_ptr()),
                                       ctypes.c_void_p(net._ws.data_ptr()), need if ws_bytes is None else ws_bytes, None)
        torch.cuda.synchronize()
        return rc, scores, flags

    assert call([0, 100], [last, last])[0] == _native.F2_ERR_INVALID
    assert call([last], [1])[0] == _native.F2_ERR_INVALID
    assert call([0], [-1])[0] == _native.F2_ERR_INVALID
    assert call([-1], [3])[0] == _native.F2_ERR_INVALID
    assert call([2 ** 63 - 10], [5])[0] == _native.F2_ERR_INVALID     # a row whose end would overflow int64
    rc, _, _ = call([0, 10], [50, 60], ws_bytes=int(L.f2_cnn_workspace_bytes(net._h, 110)) - 1)
    assert rc == _native.F2_ERR_WORKSPACE
    # zero-frame segments, also beyond the envelope's rows, read nothing and are legal
    rc, scores, flags = call([n + 500, 10, 0, last - 1], [0, 50, 0, 1])
    assert rc == _native.F2_OK and not flags.any()
    want = torch.cat([net.predict_envelope(env_t, STEP, frames=(10, 60)),
                      # predict_envelope stops one step earlier (nb = n - 11*step): pad rows that frame last - 1 never reads
                      net.predict_envelope(torch.cat([env_t, env_t[:STEP]]), STEP, frames=(last - 1, last))])
    assert torch.equal(scores, want)
    assert call([0, 0], [0, 0])[0] == _native.F2_OK
    # more runs in one chunk than travel with the launch (f2::CnnRuns::kInline): the table goes through the workspace
    rows = 20 * np.arange(200)[::-1]
    got = net.predict_segments(env_t, STEP, rows, np.full(200, 3))
    full = net.predict_envelope(env_t, STEP)
    assert torch.equal(got, full[torch.from_numpy(rows[:, None] + np.arange(3)).reshape(-1).cuda()])
