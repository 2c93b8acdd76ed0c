"""The kernels around the fused pass, each on inputs the test builds itself, against a plain float64 (numpy /
scipy) computation on the same float32 values -- not end to end, where the fused kernel's 1e-4 x RMS error
budget would hide a defect of theirs.

  (a) the (C, n) store, each output in its dtype  bit for bit against env_t.T / its float64 widening
  (b) gather_rows (vector and scalar), gather_index,
      gather_cn                                    bit for bit against numpy indexing / numpy.astype(float32)
  (c) dense_frames                                 raw: bit for bit; normalised: NORM_TOL absolute against
                                                   oracle.normalize_input in float64
  (d) rows_envelope / f2_rows_op                   LOWPASS: lp_tol(k) x RMS against scipy.signal.lfilter;
                                                   HILBERT, ENVELOPE: hb_tol(N2) (+ lp_tol) x RMS against
                                                   scipy.signal.hilbert of the float32 row (paddedHilbert)
  (e) label_fit                                    exact rational a, b, r; p against scipy.special.betainc

Bounds, from the float32 (float64) operations involved; RMS is that of the float32 row entering the kernel:
  NORM_TOL = 2e-6     the kernel and normalize_input both take log(v) - log(lo) over log(hi) - log(lo) in
                      float64.  Each log is within an ulp, 2^-52 x 88 at most; over the narrowest span of
                      distinct float32 values (hi / lo - 1 = 2^-24) that is 6.5e-7 of the result, per side.
  lp_tol(k)           2^-24 x (16 + 1 / (1 - |k|)): k = -a1 rounded to float32 moves the DC gain by
                      2^-25 / (1 - |k|), and each float32 rounding of the scan decays like |k|^t.
  hb_tol(N2)          2^-24 x 8 x log2(N2): a float32 FFT of N2 points and its inverse.
  label_fit           a, b, r within the rounding of float64 sums of 2R+1 products of the exact values
                      (computed as Fractions); p within 1e-11 relative, plus the (R - 1/2) x dr / (1 - |r|)
                      that an error dr of r makes of p ~ (1 - |r|)^(R - 1/2) near |r| = 1.

OBSERVED on one B200 (1000 W power limit), profiles/r03c_stage_kernels.log: normalised frames within 3.0e-8
(the float32 output's rounding); rows within 0.15 (LOWPASS), 0.13 (HILBERT, ENVELOPE), 0.19 (ENVELOPE + LPF)
of their bounds; label_fit p within 1.3e-3 of its bound; the (C, n) store bit-identical to env_t.T."""
import math
from fractions import Fraction

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -24
NORM_TOL = 2e-6
F2_ERR_INVALID, F2_ERR_UNSUPPORTED = 1, 4
OBSERVED = {}


def _observe(key, value):
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), float(value))


def _coefs(C):
    from f2cnn_b200.gammatone import filters
    return filters.make_erb_filters(16000, filters.centre_freqs(16000, C, 100))


@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available()
    from f2cnn_b200 import _native, api, engine, synth
    return torch, api, engine, synth, _native


def _bits(t):
    """int32 view of a float32 tensor or array, so that comparisons are bit for bit (NaN payloads too)."""
    a = t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t)
    return np.ascontiguousarray(a).view(np.int32 if a.dtype == np.float32 else np.int64)


# ---- (a) reference layouts ---------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [1, 31, 33, 128, 200])
def test_reference_layouts_transposed_and_direct(gpu, C):
    """The fused kernel stores (C, n) outputs itself, next to env_t or not: env must be env_t.T bit for bit in
    both dtypes, the float64 filterbank the widening of the float32 one, and the runs without env_t the same bits
    as those with it.  gfb and env in different dtypes each hold what the same-dtype runs hold."""
    torch, api, engine, synth, _ = gpu
    lens = [1, 31, 33, 131072, 131073, 4000, 2]
    waves = [synth.white_noise_i16(n, seed=70 + i) for i, n in enumerate(lens)]
    flat = torch.from_numpy(np.concatenate(waves)).cuda()
    batch = engine.plan_for(_coefs(C)).batch(lens)
    off = batch.sample_offsets
    t = {dt: batch.run(flat, lpf=True, cutoff=50, gfb=dt, env=dt, env_t=True) for dt in (torch.float32, torch.float64)}
    d = {dt: batch.run(flat, lpf=True, cutoff=50, gfb=dt, env=dt) for dt in (torch.float32, torch.float64)}
    mixed = [(gd, ed, batch.run(flat, lpf=True, cutoff=50, gfb=gd, env=ed, env_t=with_t))
             for gd, ed in ((torch.float64, torch.float32), (torch.float32, torch.float64)) for with_t in (False, True)]
    env_t = t[torch.float32]["env_t"]
    assert torch.equal(env_t, t[torch.float64]["env_t"])
    for u, n in enumerate(lens):
        blk = slice(C * int(off[u]), C * int(off[u + 1]))
        et = env_t[int(off[u]):int(off[u + 1])].T
        assert torch.equal(t[torch.float32]["env"][blk].view(C, n), et), (C, n)
        assert torch.equal(t[torch.float64]["env"][blk].view(C, n), et.double()), (C, n)
        assert torch.equal(t[torch.float64]["gfb"][blk], t[torch.float32]["gfb"][blk].double()), (C, n)
        for key in ("gfb", "env"):
            assert torch.equal(d[torch.float64][key][blk], d[torch.float32][key][blk].double()), (C, n, key)
            assert torch.equal(d[torch.float32][key][blk], t[torch.float32][key][blk]), (C, n, key)
        for gd, ed, m in mixed:
            assert torch.equal(m["gfb"][blk], d[gd]["gfb"][blk]), (C, n, gd, ed)
            assert torch.equal(m["env"][blk], d[ed]["env"][blk]), (C, n, gd, ed)
    for gd, ed, m in mixed:
        if "env_t" in m:
            assert torch.equal(m["env_t"], env_t), (C, gd, ed)


# ---- (b) gathers -------------------------------------------------------------------------------------------
def _random_bits(torch, numel, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(-2 ** 31, 2 ** 31 - 1, (numel,), device="cuda", generator=g, dtype=torch.int32).view(torch.float32)


@pytest.mark.parametrize("stride", [1, 160])
@pytest.mark.parametrize("C,shifted", [(128, None), (37, None), (126, None), (128, "frames"), (128, "out")])
def test_gather_windows_vector_and_scalar_paths(gpu, C, shifted, stride):
    """5000 windows (more than the 148 x 32 CTAs of the vector path, so its grid-stride loop runs); C % 4 != 0 or a
    frames / out view one float off 16-byte alignment takes the scalar kernel."""
    torch, api, engine, synth, _ = gpu
    dots, nw = 11, 5000
    R = 3000 + (dots - 1) * stride
    fs, os_ = int(shifted == "frames"), int(shifted == "out")
    frames = _random_bits(torch, R * C + fs, 1 + C + stride)[fs:].view(R, C)
    base = np.random.default_rng(C + stride).integers(0, R - (dots - 1) * stride, nw).astype(np.int64)
    base[:2] = (0, R - 1 - (dots - 1) * stride)
    out = torch.empty(nw * dots * C + os_, device="cuda")[os_:].view(nw, dots, C)
    engine.gather_windows(frames, torch.from_numpy(base).cuda(), dots, stride, out=out)
    want = _bits(frames)[base[:, None] + stride * np.arange(dots)[None, :]]
    assert np.array_equal(_bits(out), want)


@pytest.mark.parametrize("C", [128, 37])
def test_gather_index_wrapped_rows(gpu, C):
    torch, api, engine, synth, _ = gpu
    n = 4000
    src = _random_bits(torch, n * C, 3).view(n, C)
    centers = np.array([100, 800, 1599, 1600, 2500, n - 801, 0], dtype=np.int64)   # the first three wrap
    idx = api.window_indices(n, centers, 5, 160)
    raw = centers[:, None] + 160 * (np.arange(11) - 5)[None, :]
    assert (raw < 0).any()
    got = engine.gather_index(src, torch.from_numpy(np.ascontiguousarray(idx.reshape(-1))).cuda())
    want = _bits(src)[raw.reshape(-1)]                       # numpy's negative indices wrap like Python's
    assert np.array_equal(_bits(got), want)


FLT_MAX = float(np.finfo(np.float32).max)
SPECIALS = [1 + 2.0 ** -24, 1 + 3 * 2.0 ** -24, -(1 + 2.0 ** -24), 1 + 2.0 ** -24 + 2.0 ** -52, 2.0 ** -150,
            3 * 2.0 ** -150, 5 * 2.0 ** -150, 1e-40, -1e-40, 1e-310, -1e-310, 2.0 ** -126 * (1 - 2.0 ** -25),
            FLT_MAX, FLT_MAX + 2.0 ** 102, FLT_MAX + 2.0 ** 103, -(FLT_MAX + 2.0 ** 103), 1e39, -1e300,
            float("inf"), -float("inf"), 0.0, -0.0, 0.1, 1.0 / 3]


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_gather_cn_rounds_like_numpy(gpu, dtype):
    """(C, n) source -> float32 rows: ties to even, subnormals (float32 and float64), overflow past FLT_MAX."""
    torch, api, engine, synth, _ = gpu
    C, n = 37, 3001
    rng = np.random.default_rng(4)
    env = rng.normal(0, 1e3, (C, n))
    if dtype == "float64":
        sp = np.array(SPECIALS)
        env[np.arange(sp.size) % C, 7 * np.arange(sp.size)] = sp
        env[:, 1000:1000 + sp.size] = sp[None, :]
    env = env.astype(dtype)
    with np.errstate(over="ignore"):
        want_all = env.astype(np.float32)
    idx = rng.permutation(n).astype(np.int64)
    got = engine.gather_windows_cn(torch.from_numpy(env).cuda(), torch.from_numpy(idx).cuda())
    assert np.array_equal(_bits(got), _bits(np.ascontiguousarray(want_all[:, idx].T)))
    tps = np.array([100, 1500, n - 801], dtype=np.int64)         # the first wraps (InputGenerator.py:76)
    got_w = api.gather_windows_from_matrix(env, tps, 5, 160)
    raw = tps[:, None] + 160 * (np.arange(11) - 5)[None, :]
    assert np.array_equal(_bits(got_w), _bits(np.ascontiguousarray(np.moveaxis(want_all[:, raw], 0, -1))))


# ---- (c) dense_frames ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [1, 37, 128, 256])
def test_dense_frames_raw_slices_and_last_frame(gpu, C):
    torch, api, engine, synth, _native = gpu
    for dots in (1, 3, 11, 21):
        for step in (1, 7, 160):
            R = 400 + (dots - 1) * step
            env_t = torch.randn((R, C), device="cuda", generator=torch.Generator(device="cuda").manual_seed(dots + step))
            i1 = R - (dots - 1) * step                    # frame i1 - 1 reads the last row
            i0 = max(i1 - 300, 0)
            want = _bits(env_t)[np.arange(i0, i1)[:, None] + step * np.arange(dots)[None, :]]
            out32, _ = engine.dense_frames(env_t, dots, step, i0, i1, out_dtype=torch.float32)
            out64, _ = engine.dense_frames(env_t, dots, step, i0, i1, out_dtype=torch.float64)
            assert np.array_equal(_bits(out32), want), (C, dots, step)
            assert np.array_equal(out64.cpu().numpy(), want.view(np.float32).astype(np.float64)), (C, dots, step)
            with pytest.raises(_native.F2Error) as e:
                engine.dense_frames(env_t, dots, step, i0, i1 + 1)
            assert e.value.code == F2_ERR_INVALID


def _near_flat_rows(rng, R, C, lo, hi_or_k):
    """float32 rows whose every frame holds exactly lo and hi: column 0 is lo, column C-1 hi, the rest between."""
    lo = np.float32(lo)
    if isinstance(hi_or_k, int):
        grid = [lo]
        for _ in range(hi_or_k):
            grid.append(np.nextafter(grid[-1], np.float32(np.inf)))
        env = rng.choice(np.array(grid, dtype=np.float32), (R, C))
        hi = grid[-1]
    else:
        hi = np.float32(lo * (1 + hi_or_k))
        env = np.clip((lo + (hi - lo) * rng.random((R, C))).astype(np.float32), lo, hi)
    env[:, 0], env[:, -1] = lo, hi
    return env


def test_dense_frames_normalised_against_float64(gpu, oracle):
    """normalizeInput per frame against oracle.normalize_input of the same float32 values: envelope frames,
    1e-20 ... 1e20 frames, flat frames (exact zeros), values <= 0 (the flag), and near-flat frames -- hi a few
    ulps above lo, or lo x (1 + 1e-6 ... 1e-2) -- where a float32 log difference cancels."""
    torch, api, engine, synth, _ = gpu
    rng = np.random.default_rng(8)
    inputs = []
    n = 20000
    w = synth.speech_like_i16(n, seed=3).astype(np.float64) + rng.normal(0, 30, n)
    env = engine.plan_for(_coefs(128)).batch([n]).run(torch.from_numpy(w).cuda(), lpf=True, cutoff=50, env_t=True)["env_t"]
    inputs.append(("envelope", env.cpu().numpy(), 11, 160))
    inputs.append(("1e-20 .. 1e20", (10.0 ** rng.uniform(-20, 20, (2000, 37))).astype(np.float32), 11, 160))
    for lo in (1e-3, 3.0, 3000.0):
        for k in (1, 2, 16):
            inputs.append(("lo %g, hi = lo + %d ulps" % (lo, k), _near_flat_rows(rng, 60, 128, lo, k), 11, 1))
        for span in (1e-6, 1e-5, 1e-4, 1e-3, 1e-2):
            inputs.append(("lo %g, span %g" % (lo, span), _near_flat_rows(rng, 60, 128, lo, span), 11, 1))
    for what, rows, dots, step in inputs:
        env_t = torch.from_numpy(np.ascontiguousarray(rows)).cuda()
        i1 = min(rows.shape[0] - (dots - 1) * step, 200)
        frames = rows[np.arange(i1)[:, None] + step * np.arange(dots)[None, :]].astype(np.float64)
        want = np.stack([oracle.normalize_input(f) for f in frames])
        for dt in (torch.float64, torch.float32):
            got, flag = engine.dense_frames(env_t, dots, step, 0, i1, normalize=True, out_dtype=dt)
            err = np.abs(got.cpu().numpy().astype(np.float64) - want)
            _observe("normalised |kernel - float64|", np.nanmax(err))
            assert int(flag.item()) == 0, what
            assert np.all(err <= NORM_TOL), (what, dt, float(np.nanmax(err)))
    flat = torch.full((50, 128), 3.0, device="cuda")
    got, flag = engine.dense_frames(flat, 11, 1, 0, 40, normalize=True)
    assert int(flag.item()) == 0 and bool((got == 0).all())
    for bad in (0.0, -1.0):
        env_t = torch.rand((50, 128), device="cuda") + 1.0
        env_t[30, 5] = bad
        _, flag = engine.dense_frames(env_t, 11, 1, 0, 40, normalize=True)
        assert int(flag.item()) == 1


# ---- (d) stand-alone rows --------------------------------------------------------------------------------
def lp_tol(k):
    return EPS32 * (16.0 + 1.0 / (1.0 - abs(k)))


def hb_tol(n):
    return EPS32 * 8.0 * max(int(math.ceil(math.log2(n))), 1)


def _lowpass_scan_f32(x, k, b0, keep_carry_e=True, keep_carry_l=True):
    """rows_envelope_kernel's low-pass in numpy float32: one warp of 32 lanes x 8 samples per 256-sample
    iteration, each lane from zero state, a Kogge-Stone scan of (k^8, end state) across the lanes, the previous
    iteration's carry folded in.  keep_carry_e / keep_carry_l = False drop the carried envelope sample / state."""
    f32 = np.float32

    def fma(a, b, c):
        return (np.float64(a) * np.float64(b) + np.float64(c)).astype(f32)

    k, b0 = f32(k), f32(b0)
    kp = [f32(1)]
    for _ in range(8):
        kp.append(f32(kp[-1] * k))
    kp = np.array(kp, dtype=f32)
    out = np.empty(len(x), dtype=f32)
    carry_l = carry_e = f32(0)
    for base in range(0, len(x), 256):
        m = min(256, len(x) - base)
        e = np.zeros(256, dtype=f32)
        e[:m] = x[base:base + m]
        e = e.reshape(32, 8)
        ep = np.concatenate([[carry_e if keep_carry_e else f32(0)], e[:-1, 7]]).astype(f32)
        loc = np.empty((32, 8), dtype=f32)
        l = np.zeros(32, dtype=f32)
        for j in range(8):
            l = fma(k, l, (e[:, j] + ep).astype(f32))
            ep = e[:, j]
            loc[:, j] = l
        a, b = np.full(32, kp[8], dtype=f32), l.copy()
        off = 1
        while off < 32:
            a1 = np.concatenate([np.zeros(off, f32), a[:-off]])
            b1 = np.concatenate([np.zeros(off, f32), b[:-off]])
            lane = np.arange(32) >= off
            a, b = np.where(lane, (a * a1).astype(f32), a), np.where(lane, fma(a, b1, b), b)
            off *= 2
        c = carry_l if keep_carry_l else f32(0)
        end = fma(a, c, b)
        init = np.concatenate([[c], end[:-1]]).astype(f32)
        out[base:base + m] = (b0 * fma(kp[1:][None, :], init[:, None], loc)).astype(f32).reshape(-1)[:m]
        carry_l, carry_e = end[31], e[31, 7]
    return out


@pytest.mark.parametrize("cutoff", [0.5, 20, 50, 4000, 7999.5])
def test_lowpass_bound_rejects_a_scan_without_its_carries(gpu, oracle, cutoff):
    """The numpy restatement of the kernel's scan passes lp_tol; the same scan without carry_e (the envelope
    sample before each 256-sample iteration) or without carry_l (the state carried into it) fails it, and so
    does the kernel's own output if it loses either."""
    import scipy.signal
    torch, api, engine, synth, _ = gpu
    b, a = oracle.butter1_lowpass(cutoff / 8000.0)
    k = -a[1]
    x = (np.random.default_rng(2).normal(0, 1, 4096) + 5).astype(np.float32)
    want = scipy.signal.lfilter(b, a, x.astype(np.float64))
    rms = np.sqrt(np.mean(x.astype(np.float64) ** 2))
    err = lambda y: np.max(np.abs(y.astype(np.float64) - want)) / rms
    tol = lp_tol(k)
    assert err(_lowpass_scan_f32(x, k, b[0])) <= tol
    assert err(api.lowpass_rows(x[None, :], cutoff)[0]) <= tol
    assert err(_lowpass_scan_f32(x, k, b[0], keep_carry_e=False)) > 2 * tol
    if abs(k) > 1e-6:   # at 4000 Hz, k = 0: there is no state to carry
        assert err(_lowpass_scan_f32(x, k, b[0], keep_carry_l=False)) > 2 * tol


N_CASES = [1, 2, 3, 4, 5, 6, 7, 8, 9, 255, 256, 257, 8191, 8192, 8193, 12001, 32768, 40001, 131072, 131073,
           (1 << 20) + 3, (1 << 25)]
ROWS = [1, 2, 3, 5, 129]
IN_DTYPES = ["int16", "float32", "float64"]
OUT_DTYPES = ["float32", "float64"]
CUTOFFS = [0.5, 20, 50, 4000, 7999.5]
OPS = ["envelope+lpf", "envelope", "hilbert", "lowpass"]


def _fuzz_cases():
    """One case per row length; every other parameter cycles in a seeded order, so that each value appears."""
    rng = np.random.default_rng(2026)

    def cyc(vals):
        v = [vals[i % len(vals)] for i in range(len(N_CASES))]
        rng.shuffle(v)
        return v

    rows_small = cyc(ROWS)
    cases = []
    for i, (n, dt, ot, cut, op) in enumerate(zip(N_CASES, cyc(IN_DTYPES), cyc(OUT_DTYPES), cyc(CUTOFFS), cyc(OPS))):
        rows = rows_small[i] if n <= 8193 else (1 + i % 2 if n <= 1 << 17 else 1)   # the largest rows: one or two
        cases.append((n, rows, dt, ot, cut, op))
    for vals, j in ((ROWS, 1), (IN_DTYPES, 2), (OUT_DTYPES, 3), (CUTOFFS, 4), (OPS, 5)):
        assert set(vals) <= {c[j] for c in cases}
    return cases


def _rows_input(rng, dt, rows, n):
    if dt == "int16":
        return rng.integers(-20000, 20000, (rows, n)).astype(np.int16)
    return (rng.normal(0, 1000.0, (rows, n)) + 300.0).astype(dt)


@pytest.mark.parametrize("case", _fuzz_cases(), ids=lambda c: "n%d-r%d-%s-%s-%g-%s" % c)
def test_rows_ops_against_scipy(gpu, oracle, case):
    import scipy.signal
    torch, api, engine, synth, _ = gpu
    n, rows, dt, ot, cutoff, op = case
    rng = np.random.default_rng(n + rows)
    m = _rows_input(rng, dt, rows, n)
    plan = engine.any_plan()
    out_t = torch.float64 if ot == "float64" else torch.float32
    lpf = op in ("envelope+lpf", "lowpass")
    if op == "hilbert" and ot == "float64":
        got = api.hilbert_imag_rows(m)
    elif op == "lowpass" and ot == "float64":
        got = api.lowpass_rows(m, cutoff)
    elif op.startswith("envelope"):
        got = api.extract_envelope_from_matrix(m, lpf, cutoff, dtype=np.dtype(ot))
    else:
        code = {"hilbert": 1, "lowpass": 2}[op]
        got = plan.envelope_rows(torch.from_numpy(np.ascontiguousarray(m)).cuda(), lpf, cutoff, out_t, op=code).cpu().numpy()
    assert got.dtype == np.dtype(ot) and got.shape == (rows, n)
    b, a = oracle.butter1_lowpass(cutoff / 8000.0)
    N2 = 1 << max(int(math.ceil(math.log2(n))), 0)
    for r in range(rows):
        x = m[r].astype(np.float32).astype(np.float64)
        rms = np.sqrt(np.mean(x ** 2))
        if op == "lowpass":
            want, tol = scipy.signal.lfilter(b, a, x), lp_tol(-a[1])
        else:
            h = scipy.signal.hilbert(x, N2)[:n] if N2 > 1 else x.astype(np.complex128)
            want, tol = (h.imag, hb_tol(N2)) if op == "hilbert" else (np.abs(h), hb_tol(N2))
            if op == "envelope+lpf":
                want, tol = scipy.signal.lfilter(b, a, want), tol + lp_tol(-a[1])
        err = np.max(np.abs(got[r].astype(np.float64) - want)) / rms
        _observe("rows %s / bound" % op, err / tol)
        assert err <= tol, (case, r, err, tol)


def test_rows_op_refusals(gpu):
    """n = 2^25 + 1 is unsupported; cut-offs 0, 8000 and NaN are invalid with the low-pass; F2_ROWS_LOWPASS
    without lpf is invalid (the header's "lpf must be 1") instead of returning the rows unfiltered."""
    torch, api, engine, synth, _native = gpu
    plan = engine.any_plan()
    m = torch.ones((1, 1000), device="cuda")
    for cut in (0.0, 8000.0, float("nan")):
        for op in (0, 2):
            with pytest.raises(_native.F2Error) as e:
                plan.envelope_rows(m, True, cut, op=op)
            assert e.value.code == F2_ERR_INVALID, (cut, op)
    with pytest.raises(_native.F2Error) as e:
        plan.envelope_rows(m, False, 50, op=2)
    assert e.value.code == F2_ERR_INVALID
    with pytest.raises(_native.F2Error) as e:
        plan.envelope_rows(torch.ones((1, (1 << 25) + 1), device="cuda"), False, 50, op=1)
    assert e.value.code == F2_ERR_UNSUPPORTED


# ---- (e) label_fit -------------------------------------------------------------------------------------------
def _exact_fit(v, x):
    """(a, b, r, p) from exact rational sums; r from r^2, p from 1 - r = (1 - r^2) / (1 + r) without cancellation."""
    from scipy.special import betainc
    n = len(v)
    fv, fx = [Fraction(float(t)) for t in v], [Fraction(int(t)) for t in x]
    mv, mx = sum(fv) / n, sum(fx) / n
    sxx = sum((t - mx) ** 2 for t in fx)
    sxv = sum((s - mx) * (t - mv) for s, t in zip(fx, fv))
    svv = sum((t - mv) ** 2 for t in fv)
    if svv == 0 or sxv == 0:
        return float(sxv / sxx), float(mv - sxv / sxx * mx), math.nan, math.nan
    a = sxv / sxx
    r2 = sxv * sxv / (sxx * svv)
    r = math.sqrt(float(r2))
    one_minus_r = float(1 - r2) / (1 + r)
    ab = n / 2 - 1
    p = min(2 * betainc(ab, ab, one_minus_r / 2), 1.0)
    return float(a), float(mv - a * mx), r, p


def _tracks(rng, dots):
    k = np.arange(dots, dtype=np.float64)
    one_ulp = np.full(dots, 1234.5)
    one_ulp[dots // 3 if dots > 3 else 0] = np.nextafter(1234.5, np.inf)
    return {
        "random": 1500 + 300 * rng.normal(size=dots),
        "1e6 Hz + 0.01 Hz detail": 1e6 + 0.01 * rng.normal(size=dots),
        "almost linear": 1000 + 0.25 * k + 1e-11 * rng.normal(size=dots),
        "one value 1 ulp off": one_ulp,
        "constant": np.full(dots, 987.25),
        "symmetric V": np.abs(k - (dots - 1) / 2) + 7.0,
    }


@pytest.mark.parametrize("radius", [1, 2, 5, 10, 25, 50])
def test_label_fit_against_exact_and_lstsq(gpu, oracle, radius):
    from scipy.special import betainc
    torch, api, engine, synth, _ = gpu
    dots = 2 * radius + 1
    rng = np.random.default_rng(radius)
    i32max = np.iinfo(np.int32).max
    for step in (1, 160, 441):
        tracks = _tracks(rng, dots)
        names = list(tracks)
        centers = [radius * step, 123456, i32max - radius * step]
        flat = np.concatenate([tracks[nm] for nm in names])
        first = np.repeat(np.arange(len(names), dtype=np.int64) * dots, len(centers))
        center = np.tile(np.array(centers, dtype=np.int32), len(names))
        got = engine.label_fit(torch.from_numpy(flat).cuda(), torch.from_numpy(first).cuda(),
                               torch.from_numpy(center).cuda(), dots, step).cpu().numpy()
        for i in range(len(first)):
            name = names[i // len(centers)]
            v = flat[first[i]:first[i] + dots]
            x = int(center[i]) + step * (np.arange(dots, dtype=np.int64) - radius)
            want = _exact_fit(v, x)
            a, b, r, p = got[i]
            what = (name, radius, step, int(center[i]))
            if name in ("constant", "symmetric V"):
                assert math.isnan(r) and math.isnan(p), what
                continue
            # float64 sums of `dots` products: |error| <= dots x 2^-52 x sum |dx dv| (<= sqrt(sxx svv))
            dx = (x - int(center[i])).astype(np.float64)
            sxx, sdxdv = np.sum(dx * dx), np.sum(np.abs(dx * (v - np.mean(v))))
            atol = 2 * dots * 2.0 ** -52 * (sdxdv / sxx + abs(want[0]))
            rtol = 2 * dots * 2.0 ** -52
            assert abs(a - want[0]) <= atol, what + (a, want[0])
            assert abs(b - want[1]) <= 4 * 2.0 ** -52 * abs(want[1]) + atol * float(center[i]), what + (b, want[1])
            assert abs(r - want[2]) <= rtol, what + (r, want[2])
            # p ~ (1 - |r|)^(R - 1/2) near |r| = 1: an error dr in r moves it by (R - 1/2) dr / (1 - |r|)
            ptol = want[3] * (1e-11 + (radius - 0.5) * rtol / max(1.0 - want[2], 1e-300)) + 1e-300
            _observe("label |p - exact| / bound", abs(p - want[3]) / ptol)
            assert abs(p - want[3]) <= ptol, what + (p, want[3])
            assert abs(p - min(2 * betainc(dots / 2 - 1, dots / 2 - 1, (1 - abs(r)) / 2), 1.0)) <= 1e-11 * p + 1e-300, what
            if name == "random" and i % len(centers) < 2:   # lstsq + pearsonr, where lstsq is well conditioned
                la, lb, lr, lp = oracle.label_fit(v, x)
                assert abs(a - la) <= 1e-9 * abs(la) and abs(r - abs(lr)) <= 1e-9 and abs(p - lp) <= 1e-9 * lp, what


def test_zz_report_observed():
    """Prints the worst value of every quantity the bounds above are set from (run with -s)."""
    for key in sorted(OBSERVED):
        print("OBSERVED %-40s %.3e" % (key, OBSERVED[key]))
