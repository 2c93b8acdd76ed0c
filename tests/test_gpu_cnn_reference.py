"""The tensor-core CNN forward (csrc/f2_cnn.cu) against the bf16-faithful float64 reference
(oracle/cnn_bf16.py), which rounds to bf16 exactly where the kernels store bf16.

Stage-local comparisons feed each reference stage the kernel's own input to that stage (env_t -> p2,
the kernel's p2 -> features, the kernel's features -> scores), so one rounding flip upstream cannot hide
or blur anything downstream.  Bounds (set at about 4x the maxima observed on a B200, see OBSERVED):

  p2, features   |kernel - reference| <= ULPS * ulp_bf16(reference) + FLOOR * max|reference|,
                 and at least BIT_EQUAL of the elements bit-equal
  scores         stage-local: SCORE_TOL absolute; logits log(s1/s0) where min(s) > 1e-6: LOGIT_TOL
  chained        env_t -> scores through the whole reference: CHAINED_TOL absolute

Two networks: cnn.seeded_model(3) (what the other tests and tools use; its scores all sit near 0.5) and
cnn_bf16.spread_model() (He-scaled weights, biases of std 0.3, logit difference of std ~1), on which
every parameter moves the scores.  test_bounds_reject_every_mutation shows that each bound would fail
on a subtly wrong kernel: every mutated reference breaks one of them by at least 10x.

OBSERVED on one B200 (1000 W power limit), over the calls of this file, both networks: at least 99.988 %
of p2 and 99.935 % of the feature elements bit-equal; stage-local scores within 3.0e-6, logits within
1.3e-5; chained scores within 2.9e-3 on the spread network (1.9e-5 on seeded_model); every mutation
breaks a bound by at least 87x.  The rare elements
that differ are isolated rounding flips (the kernel normalises with float32 logf, the reference in float64;
a flipped bf16 input or conv1 value moves a p2 element by |w| x one bf16 ulp of the flipped value).  Where
that element is small next to its layer, the flip is many of ITS ulps (up to ~54 in p2, ~125 in the
features) and at most 6.9e-3 of the layer maximum: hence the absolute floor of 2^-6 of the layer
maximum, while the bit-equal fraction keeps the comparison tight everywhere else."""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ULPS = 2.0
FLOOR = 2.0 ** -6
BIT_EQUAL = 0.997
SCORE_TOL = 1.2e-5
LOGIT_TOL = 6e-5
CHAINED_TOL = 1e-2
CHUNK = 32768


def _coefs():
    from f2cnn_b200.gammatone import filters
    return filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))


def _env_t(n, seed, noise_seed):
    """Time-major float32 envelope ([n, 128], device) of a speech-like utterance, as test_gpu_cnn.py builds it."""
    import torch
    from f2cnn_b200 import engine, synth
    w = synth.speech_like_i16(n, seed=seed).astype(np.float64) + np.random.default_rng(noise_seed).normal(0, 30, n)
    return engine.plan_for(_coefs()).batch([n]).run(torch.from_numpy(w).cuda(), lpf=True, cutoff=50, env_t=True)["env_t"]


@pytest.fixture(scope="module")
def setup():
    import torch
    from f2cnn_b200 import cnn
    from oracle import cnn_bf16
    env_t = _env_t(20000, 11, 2)
    models = {"spread": cnn_bf16.spread_model().cuda(), "seeded": cnn.seeded_model(seed=3)}
    nets = {k: cnn.TensorCoreCNN(m) for k, m in models.items()}
    refs = {k: cnn_bf16.BF16Reference(m, device="cuda") for k, m in models.items()}
    return torch, cnn_bf16, env_t, models, nets, refs


@pytest.fixture(params=["spread", "seeded"])
def net(request, setup):
    torch, cnn_bf16, env_t, models, nets, refs = setup
    return request.param, nets[request.param], refs[request.param]


def _excess(got, ref, ulps=ULPS):
    """max |got - ref| / (ulps * ulp_bf16(ref) + FLOOR * max|ref|): <= 1 passes the bound."""
    from oracle import cnn_bf16
    tol = ulps * cnn_bf16.bf16_ulp(ref) + FLOOR * float(ref.abs().max())
    return float(((got.double() - ref).abs() / tol).max())


def _ulps(got, ref):
    """Largest error beyond the absolute floor, in bf16 ulps of the reference value."""
    from oracle import cnn_bf16
    d = (got.double() - ref).abs() - FLOOR * float(ref.abs().max())
    return float((d.clamp_min(0) / cnn_bf16.bf16_ulp(ref)).max())


def _rel_abs(got, ref):
    """max |got - ref| / max|ref|."""
    return float((got.double() - ref).abs().max()) / max(float(ref.abs().max()), 1e-300)


def _mismatch(got, ref):
    """Fraction of elements that are not bit-equal, in units of the allowed fraction 1 - BIT_EQUAL."""
    return float((got.double() != ref).double().mean()) / (1.0 - BIT_EQUAL)


def _logit_err(scores, logits):
    import torch
    s = scores.double()
    ok = s.min(dim=1).values > 1e-6
    if not bool(ok.any()):
        return 0.0
    got = torch.log(s[ok, 1] / s[ok, 0])
    return float((got - (logits[ok, 1] - logits[ok, 0])).abs().max())


def _stage_local(tc, ref, env_t, step, i0, i1, scores=None):
    """Run the kernels on frames [i0, i1) (unless `scores` of that call are given) and compare every stage
    with the reference applied to the kernel's own input to it."""
    import torch
    if scores is None:
        scores = tc.predict_envelope(env_t, step, frames=(i0, i1))
    torch.cuda.synchronize()
    gp2, gfeat = tc.intermediates(i1 - i0)
    rp2 = ref.front(ref.normalize(ref.frames(env_t, step, i0, i1)))
    rfeat = ref.mid(gp2.double())
    rlog = ref.logits(gfeat.double())
    rsc = torch.softmax(rlog, dim=1)
    return {
        "p2": _excess(gp2, rp2), "p2_ulps": _ulps(gp2, rp2), "p2_abs": _rel_abs(gp2, rp2), "p2_equal": float((gp2.double() == rp2).double().mean()),
        "feat": _excess(gfeat, rfeat), "feat_ulps": _ulps(gfeat, rfeat), "feat_abs": _rel_abs(gfeat, rfeat),
        "feat_equal": float((gfeat.double() == rfeat).double().mean()),
        "score": float((scores.double() - rsc).abs().max()), "logit": _logit_err(scores, rlog),
    }


def _check(m, what=""):
    print("observed %s: p2 %.2f ulps, %.2e of max (%.5f bit-equal), feat %.2f ulps, %.2e of max (%.5f bit-equal), "
          "scores %.2e, logits %.2e" % (what, m["p2_ulps"], m["p2_abs"], m["p2_equal"], m["feat_ulps"], m["feat_abs"],
                                        m["feat_equal"], m["score"], m["logit"]))
    assert m["p2"] <= 1.0 and m["feat"] <= 1.0, (what, m)
    assert m["p2_equal"] >= BIT_EQUAL and m["feat_equal"] >= BIT_EQUAL, (what, m)
    assert m["score"] <= SCORE_TOL and m["logit"] <= LOGIT_TOL, (what, m)


def _chained(ref, env_t, step, i0, i1, scores, what=""):
    err = float((scores.double() - ref.forward(env_t, step, i0, i1)["scores"]).abs().max())
    print("observed %s: chained scores %.2e" % (what, err))
    assert err <= CHAINED_TOL, (what, err)
    return err


# ---- (a) stage-local parity ------------------------------------------------------------------------------
def test_stage_local_parity(setup, net):
    torch, _, env_t, _, _, _ = setup
    name, tc, ref = net
    nb = env_t.shape[0] - 1760
    for i0, i1 in ((0, 300), (5000, 5700), (nb - 257, nb)):
        scores = tc.predict_envelope(env_t, 160, frames=(i0, i1))
        _check(_stage_local(tc, ref, env_t, 160, i0, i1, scores), "%s [%d, %d)" % (name, i0, i1))
        _chained(ref, env_t, 160, i0, i1, scores, "%s [%d, %d)" % (name, i0, i1))


# ---- (b) sensitivity: the bounds reject every mutation -----------------------------------------------------
def test_bounds_reject_every_mutation(setup, net):
    """Each mutated reference, compared with the kernels like the correct one, breaks a bound by >= 10x.
    Also prints which mutations the float32-oracle bounds of test_gpu_cnn.py (p2 and features within
    2e-2 of the layer max, scores within 5e-3) would have let through."""
    torch, cnn_bf16, env_t, models, _, _ = setup
    name, tc, _ = net
    i0, i1 = 5000, 5700
    scores = tc.predict_envelope(env_t, 160, frames=(i0, i1))
    torch.cuda.synchronize()
    gp2, gfeat = tc.intermediates(i1 - i0)
    gp2, gfeat = gp2.double(), gfeat.double()
    passed_old = []
    for mutation in cnn_bf16.MUTATIONS:
        ref = cnn_bf16.BF16Reference(models[name], device="cuda", mutation=mutation)
        rp2 = ref.front(ref.normalize(ref.frames(env_t, 160, i0, i1)))
        rfeat = ref.mid(gp2)
        rlog = ref.logits(gfeat)
        chain = ref.forward(env_t, 160, i0, i1)
        ratio = max(_excess(gp2, rp2), _excess(gfeat, rfeat), _mismatch(gp2, rp2), _mismatch(gfeat, rfeat),
                    float((scores.double() - torch.softmax(rlog, dim=1)).abs().max()) / SCORE_TOL,
                    _logit_err(scores, rlog) / LOGIT_TOL,
                    float((scores.double() - chain["scores"]).abs().max()) / CHAINED_TOL)
        old = (float((gp2 - chain["p2"]).abs().max()) <= 2e-2 * float(chain["p2"].abs().max())
               and float((gfeat - chain["feat"]).abs().max()) <= 2e-2 * float(chain["feat"].abs().max())
               and float((scores.double() - chain["scores"]).abs().max()) <= 5e-3)
        if old:
            passed_old.append(mutation)
        print("observed %s %s: breaks the bounds by %.3gx%s" % (name, mutation, ratio, " (old bounds: accepted)" if old else ""))
        assert ratio >= 10.0, (name, mutation, ratio)
    print("observed %s: the old bounds accept %s" % (name, passed_old))


# ---- (c) counts and offsets ---------------------------------------------------------------------------------
def test_frame_counts_at_the_persistent_grid_edges_are_bit_exact(setup, net):
    """grid = min(frames, SMs) (148 on a B200) and the front kernel prefetches frame f + 2 * grid: counts
    around 1, 128, 148, 2 * 148 and 3 * 148 from an odd first frame.  A frame goes through the same
    instructions whatever CTA, tile or chunk computes it, so every sub-range equals the whole bit for bit."""
    torch, _, env_t, _, _, _ = setup
    name, tc, ref = net
    i0, top = 12345, 445
    whole = tc.predict_envelope(env_t, 160, frames=(i0, i0 + top)).clone()
    for nf in (1, 2, 127, 128, 129, 147, 148, 149, 295, 296, 297, 445):
        got = tc.predict_envelope(env_t, 160, frames=(i0, i0 + nf))
        assert torch.equal(got, whole[:nf]), (name, nf)
        _check(_stage_local(tc, ref, env_t, 160, i0, i0 + nf, got), "%s nf=%d" % (name, nf))
        tail = tc.predict_envelope(env_t, 160, frames=(i0 + top - nf, i0 + top))
        assert torch.equal(tail, whole[top - nf:]), (name, nf)


# ---- (d) more than one chunk --------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def long_env(setup):
    nb = 2 * CHUNK + 5   # chunks of 32768, 32768 and 5 frames
    return _env_t(nb + 1760, 13, 4), nb


def test_chunk_splits_agree_bit_for_bit(setup, long_env, net):
    torch, _, _, _, _, _ = setup
    env, nb = long_env
    name, tc, ref = net
    full = tc.predict_envelope(env, 160)
    assert full.shape == (nb, 2)
    full = full.clone()
    for cuts in ((0, CHUNK, nb), (0, 1, CHUNK + 2, nb)):
        parts = [tc.predict_envelope(env, 160, frames=(a, b)) for a, b in zip(cuts[:-1], cuts[1:])]
        assert torch.equal(torch.cat(parts), full), (name, cuts)
    # the chained reference at both chunk edges of the whole call
    for i0, i1 in ((CHUNK - 128, CHUNK + 128), (nb - 256, nb)):
        _chained(ref, env, 160, i0, i1, full[i0:i1], "%s chunk edge [%d, %d)" % (name, i0, i1))


def test_non_positive_value_in_the_last_chunk_raises(setup, long_env):
    torch, _, _, _, nets, _ = setup
    env, nb = long_env
    tc = nets["spread"]
    bad = env.clone()
    row = nb - 1 + 10 * 160   # read only by the last frame (third chunk, as its 11th dot)
    bad[row, 7] = 0.0
    with pytest.raises(ValueError, match="positive"):
        tc.predict_envelope(bad, 160)
    with pytest.raises(ValueError, match="positive"):
        tc.predict_envelope(bad, 160, frames=(CHUNK - 3, nb))
    ok = tc.predict_envelope(bad, 160, frames=(0, nb - 1))
    assert torch.equal(ok, tc.predict_envelope(env, 160, frames=(0, nb - 1)))


# ---- (e) steps ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("step", [1, 37, 80, 160, 320])
def test_steps_and_the_last_legal_frame(setup, net, step):
    torch, _, env_t, _, _, _ = setup
    name, tc, ref = net
    nb = env_t.shape[0] - 11 * step
    for i0, i1 in ((0, 64), (nb - 64, nb)):
        scores = tc.predict_envelope(env_t, step, frames=(i0, i1))
        _check(_stage_local(tc, ref, env_t, step, i0, i1, scores), "%s step %d [%d, %d)" % (name, step, i0, i1))
        _chained(ref, env_t, step, i0, i1, scores, "%s step %d [%d, %d)" % (name, step, i0, i1))
    assert tc.predict_envelope(env_t, step).shape == (nb, 2)
    with pytest.raises(IndexError):
        tc.predict_envelope(env_t, step, frames=(nb - 1, nb + 1))


# ---- (f) inputs ---------------------------------------------------------------------------------------------
def test_flat_single_value_and_wide_range_frames(setup, net):
    torch, _, _, _, _, _ = setup
    name, tc, ref = net
    rows, nf = 2000, 240
    flat = torch.full((rows, 128), 3.0, device="cuda")
    single = flat.clone()
    single[800, 60] = 5.0                      # frames 0 and 160 see one value above the rest
    g = torch.Generator(device="cuda").manual_seed(9)
    wide = torch.pow(10.0, torch.rand((rows, 128), device="cuda", generator=g) * 40 - 20)
    wide[400, 0], wide[1000, 127] = 1e-20, 1e20
    # every value within 16 ulps of 3000: a float32 log(hi) - log(lo) would cancel to nothing or to one ulp of it
    near = 3000.0 + 2.0 ** -12 * torch.randint(0, 17, (rows, 128), device="cuda", generator=g).float()
    near[:, 0], near[:, 127] = 3000.0, 3000.0 + 16 * 2.0 ** -12
    for what, env in (("flat", flat), ("single", single), ("1e-20 .. 1e20", wide), ("near-flat", near)):
        scores = tc.predict_envelope(env, 160, frames=(0, nf))
        _check(_stage_local(tc, ref, env, 160, 0, nf, scores), "%s %s" % (name, what))
        _chained(ref, env, 160, 0, nf, scores, "%s %s" % (name, what))
        if what == "flat":
            assert bool((scores == scores[0]).all())
    x = ref.normalize(ref.frames(single, 160, 0, 1))
    assert int((x != 0).sum()) == 1 and float(x.max()) == 1.0


# ---- (g) api.cnn_evaluate ---------------------------------------------------------------------------------
def test_cnn_evaluate_on_a_3s_utterance(setup):
    """46 240 frames, two chunks; with and without envelopes; two networks alternating through the cache."""
    torch, cnn_bf16, _, models, nets, refs = setup
    from f2cnn_b200 import api, cnn, synth
    co = _coefs()
    n = 48000
    w = synth.speech_like_i16(n, seed=21).astype(np.float64) + np.random.default_rng(6).normal(0, 30, n)
    nb = n - 1760
    s_env, envelopes = api.cnn_evaluate(w, co, models["spread"], True, 50, with_envelopes=True)
    s_no, none = api.cnn_evaluate(w, co, models["spread"], True, 50, with_envelopes=False)
    assert none is None and envelopes.shape == (128, n)
    assert s_env.shape == (nb, 2) and np.array_equal(s_env.view(np.int32), s_no.view(np.int32))
    _, env_t = api.evaluate_front_end(w, co, True, 50, frames=False)
    got = torch.from_numpy(s_env).cuda()
    for i0, i1 in ((0, 256), (CHUNK - 128, CHUNK + 128), (nb - 256, nb)):
        _chained(refs["spread"], env_t, 160, i0, i1, got[i0:i1], "cnn_evaluate [%d, %d)" % (i0, i1))
    # A, B, A through the network cache (Keras-layout arrays for B)
    s_b, _ = api.cnn_evaluate(w, co, cnn.keras_arrays(models["seeded"]), True, 50, with_envelopes=False)
    s_a, _ = api.cnn_evaluate(w, co, models["spread"], True, 50, with_envelopes=False)
    assert np.array_equal(s_a, s_no)
    assert np.array_equal(s_b, nets["seeded"].predict_envelope(env_t, 160).cpu().numpy())
    assert not np.allclose(s_a, s_b, atol=1e-2)
    with pytest.raises(ValueError):
        api.cnn_evaluate(w, co, models["spread"], True, 50, radius=4)
    with pytest.raises(ValueError):
        api.cnn_evaluate(w, co[:64], models["spread"], True, 50)


# ---- (h) two devices --------------------------------------------------------------------------------------
def test_networks_on_two_devices_in_one_process(setup):
    """The kernels' shared-memory limit is a per-device function attribute: a network on a second device
    must run as well as one on the first, whichever device ran first, with bit-identical scores."""
    torch, _, env_t, models, nets, _ = setup
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 visible devices")
    from f2cnn_b200 import cnn
    env = env_t[:4000].contiguous()
    s0 = nets["spread"].predict_envelope(env, 160).cpu()
    tc1 = cnn.TensorCoreCNN(models["spread"], device=1)
    s1 = tc1.predict_envelope(env.to("cuda:1"), 160).cpu()
    assert torch.equal(s0, s1)
    from f2cnn_b200 import api
    with torch.cuda.device(1):
        via_api = api._network_for(models["spread"])
        assert via_api.device.index == 1
        assert torch.equal(via_api.predict_envelope(env.to("cuda:1"), 160).cpu(), s0)
    # device 1 first, in a fresh process
    code = (
        "import sys, numpy as np, torch\n"
        "sys.path.insert(0, %r)\n"
        "from f2cnn_b200 import cnn\n"
        "from oracle import cnn_bf16\n"
        "env = torch.from_numpy(np.load(sys.argv[1]))\n"
        "out = [cnn.TensorCoreCNN(cnn_bf16.spread_model(), device=d).predict_envelope(env.to('cuda:%%d' %% d), 160).cpu().numpy()\n"
        "       for d in (1, 0)]\n"
        "np.save(sys.argv[2], np.stack(out))\n" % ROOT)
    with tempfile.TemporaryDirectory() as d:
        src, dst = os.path.join(d, "env.npy"), os.path.join(d, "scores.npy")
        np.save(src, env.cpu().numpy())
        subprocess.run([sys.executable, "-c", code, src, dst], check=True, timeout=300)
        out = np.load(dst)
    assert np.array_equal(out[0], s0.numpy()) and np.array_equal(out[1], s0.numpy())
