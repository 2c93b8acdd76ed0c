"""The bf16-faithful CNN reference (oracle/cnn_bf16.py) on the CPU: with its rounding switched off it is
the float64 forward of cnn.F2CNN, its bf16 rounding is bf16_rne's, every mutation the GPU tests use to
prove their bounds changes its output, and the spread network is not saturated."""
import copy
import struct

import numpy as np
import pytest
import torch

from oracle import cnn_bf16
from oracle.cnn_bf16 import BF16Reference, MUTATIONS


@pytest.fixture(scope="module")
def env_t(oracle):
    """Time-major float32 envelope (4000 rows) of a speech-like utterance, from the CPU oracle."""
    from f2cnn_b200 import synth
    from f2cnn_b200.gammatone import filters
    co = filters.make_erb_filters(16000, filters.centre_freqs(16000, 128, 100))
    n = 4000
    w = synth.speech_like_i16(n, seed=11).astype(np.float64) + np.random.default_rng(2).normal(0, 30, n)
    _, env, _ = oracle.utterance(w, co, True, 50)
    return torch.from_numpy(env.T.copy()).float()


@pytest.fixture(scope="module")
def spread():
    """He-scaled weights, biases of std 0.3, last layer x4: see cnn_bf16.spread_model."""
    return cnn_bf16.spread_model()


@pytest.fixture(scope="module")
def seeded():
    from f2cnn_b200 import cnn
    return cnn.seeded_model(seed=3, device="cpu")


@pytest.fixture(params=["spread", "seeded"])
def model(request):
    return request.getfixturevalue(request.param)


def _bf16_rne(f):
    """f2_capi.cu's bf16_rne, line for line, on one float32."""
    u = struct.unpack("<I", struct.pack("<f", f))[0]
    if (u & 0x7FFFFFFF) > 0x7F800000:
        return ((u >> 16) | 0x40) & 0xFFFF
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFFFFFF
    return u >> 16


def _bits(x64):
    return (x64.to(torch.float32).view(torch.int32).to(torch.int64) >> 16) & 0xFFFF


def test_bf16_rounding_is_bf16_rne_and_torch():
    hi = [0x3F80, 0x3F81, 0xBF80, 0xBF81, 0x0001, 0x0080, 0x7F7F, 0xFF7F, 0x4B7F, 0x0000]
    lo = [0x0000, 0x0001, 0x7FFF, 0x8000, 0x8001, 0xFFFF]   # exact, next to a tie, a tie, past a tie
    words = [(h << 16) | l for h in hi for l in lo]
    words += [0x7F800001, 0x7FBFFFFF, 0xFFC00000, 0x7FC00001, 0xFF800000, 0x7F800000]   # NaNs and infinities
    rng = np.random.default_rng(0)
    words += [int(v) for v in rng.integers(0, 2 ** 32, 4000, dtype=np.uint64)]
    x = torch.tensor(np.array(words, dtype=np.uint32).view(np.float32))
    got = _bits(cnn_bf16.bf16(x))
    want = torch.tensor([_bf16_rne(float(v)) for v in x.tolist()])
    assert torch.equal(got, want)
    nan = torch.isnan(x)
    assert bool(torch.isnan(cnn_bf16.bf16(x))[nan].all()) and int(nan.sum()) >= 4
    # ties go to even, a hair past a tie goes up, a hair short of it goes down
    one = torch.tensor(np.array([0x3F808000, 0x3F818000, 0x3F808001, 0x3F807FFF], dtype=np.uint32).view(np.float32))
    assert _bits(cnn_bf16.bf16(one)).tolist() == [0x3F80, 0x3F82, 0x3F81, 0x3F80]
    fin = ~nan
    assert torch.equal(cnn_bf16.bf16(x[fin]), x[fin].to(torch.bfloat16).to(torch.float64))


def test_bf16_ulp_is_the_spacing_of_bf16_values():
    x = torch.tensor([1.0, 1.5, 2.0, 3.999, 0.75, -6.0, 1e-3], dtype=torch.float64)
    u = cnn_bf16.bf16_ulp(x)
    assert u.tolist()[:4] == [2.0 ** -7, 2.0 ** -7, 2.0 ** -6, 2.0 ** -6]
    b = cnn_bf16.bf16(x)
    assert torch.equal(cnn_bf16.bf16(b + cnn_bf16.bf16_ulp(b)), b + cnn_bf16.bf16_ulp(b))
    assert bool((cnn_bf16.bf16(b + 0.49 * cnn_bf16.bf16_ulp(b)) == b).all())


def _normalize_input(fr):
    """Training.normalizeInput on one (11, 128) frame, in numpy float64."""
    lo, hi = np.log(fr.min()), np.log(fr.max())
    return np.zeros_like(fr) if hi == lo else (np.log(fr) - lo) / (hi - lo)


@pytest.mark.parametrize("step, i0", [(160, 0), (37, 1234)])
def test_unrounded_reference_is_the_float64_forward(model, env_t, step, i0):
    i1 = min(i0 + 96, env_t.shape[0] - 11 * step)
    ref = BF16Reference(model, rounding=False)
    got = ref.forward(env_t, step, i0, i1)
    e = env_t.double().numpy()
    fr = np.stack([_normalize_input(e[i + step * np.arange(11)]) for i in range(i0, i1)])
    x = torch.from_numpy(fr)
    assert float((ref.normalize(ref.frames(env_t, step, i0, i1))[:, 0] - x).abs().max()) <= 1e-12
    m64 = copy.deepcopy(model).double()
    with torch.no_grad():
        want = m64(x)
        p2 = torch.nn.functional.max_pool2d(torch.relu(m64.c2(torch.relu(m64.c1(x.unsqueeze(1))))), 2)
    assert float((got["scores"] - want).abs().max()) <= 1e-12
    assert float((got["p2"] - p2).abs().max()) <= 1e-12
    assert float((want.sum(1) - 1).abs().max()) <= 1e-12


def test_rounding_happens_and_stays_within_bf16(model, env_t):
    """With rounding on, every stored activation is a bf16 value and the scores move, but only by the
    amount bf16 storage explains (the GPU tests hold the kernels far tighter, to this reference)."""
    a = BF16Reference(model).forward(env_t, 160, 0, 128)
    b = BF16Reference(model, rounding=False).forward(env_t, 160, 0, 128)
    for k in ("p2", "feat"):
        assert torch.equal(cnn_bf16.bf16(a[k]), a[k])
    assert not torch.equal(a["scores"], b["scores"])
    assert float((a["scores"] - b["scores"]).abs().max()) <= 5e-2


@pytest.mark.parametrize("mutation", MUTATIONS)
def test_every_mutation_changes_the_output(mutation, model, env_t):
    base = BF16Reference(model).forward(env_t, 160, 500, 628)
    mut = BF16Reference(model, mutation=mutation).forward(env_t, 160, 500, 628)
    assert not torch.equal(mut["scores"], base["scores"])
    # a mutation of the front end already shows in p2, one of conv3 .. flatten in the features
    stage = {"no_b3": "feat", "no_b4": "feat", "flatten_chw": "feat", "no_b5": "scores", "no_b6": "scores",
             "swap_b6": "scores", "swap_w6": "scores"}.get(mutation, "p2")
    assert not torch.equal(mut[stage], base[stage])


def test_reference_rejects_non_positive_values(env_t):
    bad = env_t.clone()
    bad[1000, 3] = 0.0
    ref = BF16Reference(cnn_bf16.spread_model())
    with pytest.raises(ValueError, match="positive"):
        ref.forward(bad, 160, 900, 1100)
    ref.forward(bad, 160, 1001, 1100)
    with pytest.raises(ValueError):
        BF16Reference(cnn_bf16.spread_model(), mutation="no_b7")


def test_spread_network_is_neither_dead_nor_saturated(spread, env_t):
    nb = env_t.shape[0] - 1760
    out = BF16Reference(spread).forward(env_t, 160, 0, nb)
    for k in ("p2", "feat"):
        nz = float((out[k] > 0).double().mean())
        assert 0.2 <= nz <= 0.8, (k, nz)
    d = out["logits"][:, 1] - out["logits"][:, 0]
    assert 0.5 <= float(d.std()) <= 3.0
    assert float(out["scores"].max(1).values.median()) < 0.95
