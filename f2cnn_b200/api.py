"""numpy-in / numpy-out entry points behind the reference-named modules.

Each function stages its inputs through pinned host memory, launches the C-ABI sequence on
the current CUDA stream and returns freshly allocated numpy arrays of the reference's dtype
and layout.  All arithmetic happens in libf2cnn_b200.so."""
import hashlib
import threading
from collections import OrderedDict

import numpy as np
import torch

from . import engine

_WAVE_DTYPES = (np.int16, np.float32, np.float64)
_PIPELINE_BYTES = 256 << 20  # window tensors above this size go through engine.WindowPipeline


def _as_wave(wave):
    """The reference feeds scipy.signal.lfilter an int16 WAV array or a float64 noise-mixed
    array (Evaluating.py:200); anything else is promoted to float64 like lfilter would."""
    w = np.asarray(wave)
    if w.ndim != 1:
        raise ValueError("wave must be one-dimensional, got shape %s" % (w.shape,))
    if w.dtype not in [np.dtype(d) for d in _WAVE_DTYPES]:
        if w.dtype.kind in "iub" and w.dtype.itemsize <= 2:
            w = w.astype(np.int16) if w.dtype != np.uint16 else w.astype(np.float64)
        else:
            w = w.astype(np.float64)
    return np.ascontiguousarray(w)


def _as_matrix(matrix):
    """A (rows, n) matrix as the C ABI takes it: int16, float32 or float64, C-contiguous; anything else is
    promoted to float64."""
    m = np.asarray(matrix)
    if m.dtype not in (np.dtype(np.float32), np.dtype(np.float64), np.dtype(np.int16)):
        m = m.astype(np.float64)
    return np.ascontiguousarray(m)


def _torch_dtype(dtype):
    """The output dtype a call was asked for: float64, or float32 for anything else."""
    return torch.float64 if np.dtype(dtype) == np.float64 else torch.float32


def _to_device(a, device):
    """A host numpy array or tensor on `device`; 64 KiB and more go through pinned memory."""
    t = torch.from_numpy(a) if isinstance(a, np.ndarray) else a
    if t.numel() * t.element_size() >= (1 << 16) and not t.is_pinned():
        t = t.pin_memory()
    return t.to(device, non_blocking=True)


def _to_host(t):
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=t.numel() * t.element_size() >= (1 << 16))
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return host.numpy()


def _check_out(out, shape, dtype=np.float32, count=None, message=None):
    """An existing array for a call to fill: a C-contiguous numpy array of `dtype` and `shape` -- with `count`, a
    sequence of that many, returned as a list.  Anything else raises ValueError(message)."""
    outs = [out] if count is None else list(out)
    if (count is not None and len(outs) != count) or not all(
            isinstance(o, np.ndarray) and o.dtype == dtype and o.flags["C_CONTIGUOUS"] and o.shape == shape
            for o in outs):
        raise ValueError(message or "out must be a C-contiguous %s array of shape %s" % (np.dtype(dtype).name, shape))
    return out if count is None else outs


def _utterance(wave, coefs):
    """One waveform's (host wave, plan, n) for the single-utterance calls."""
    w = _as_wave(wave)
    plan = engine.plan_for(np.asarray(coefs, dtype=np.float64))
    return w, plan, int(w.shape[0])


def _run_utterance(plan, w, step=160, phase=0, **outputs):
    """The fused pass over one host waveform: Batch.run's result dict for the requested `outputs`."""
    return plan.batch([int(w.shape[0])], step=step, phase=phase).run(_to_device(w, plan.device), **outputs)


def _normalised_frames(env_t, dots, step, i0, i1, normalize, dtype):
    """Dense stride-1 frames i0..i1 of a time-major envelope on the host (Evaluating.py:70-78), normalised per frame
    (Training.normalizeInput) when `normalize`."""
    out, flag = engine.dense_frames(env_t, dots, step, i0, i1, normalize=normalize, out_dtype=_torch_dtype(dtype))
    host = _to_host(out)
    if normalize and int(flag.item()) != 0:
        raise ValueError("values must all be positive")  # Training.py:18-20
    return host


def erb_filterbank(wave, coefs, dtype=np.float64):
    """gammatone/filters.py:195-239 -> (C, n) float64 (the reference's dtype; float32 on request)."""
    w, plan, n = _utterance(wave, coefs)
    if n == 0:
        return np.zeros((plan.n_channels, 0), dtype=dtype)
    res = _run_utterance(plan, w, gfb=_torch_dtype(dtype))
    return _to_host(res["gfb"]).reshape(plan.n_channels, n)


def filterbank_envelope(wave, coefs, LPF=False, CUTOFF=100, with_gfb=False, dtype=np.float64):
    """Fused erb_filterbank + ExtractEnvelopeFromMatrix on one waveform: the (C,n) envelope
    (and optionally the filterbank output) without the intermediate host round trip."""
    w, plan, n = _utterance(wave, coefs)
    tdt = _torch_dtype(dtype)
    if n == 0:
        z = np.zeros((plan.n_channels, 0), dtype=dtype)
        return (z, z.copy()) if with_gfb else z
    res = _run_utterance(plan, w, lpf=LPF, cutoff=CUTOFF, env=tdt, gfb=tdt if with_gfb else None)
    env = _to_host(res["env"]).reshape(plan.n_channels, n)
    if with_gfb:
        return _to_host(res["gfb"]).reshape(plan.n_channels, n), env
    return env


def gammatonegram(wave, coefs, hop, LPF=False, CUTOFF=100, dtype=np.float64):
    """Every `hop`-th sample of the envelope of `filterbank_envelope` -- (C, ceil(n / hop)), the samples at
    t = 0, hop, 2*hop, ... -- stored by the fused kernel itself: what a plot of a whole file needs
    (scripts/plotting/PlottingProcessing.py:101-109 takes the full-rate matrix for it)."""
    w, plan, n = _utterance(wave, coefs)
    hop = int(hop)
    if hop < 1:
        raise ValueError("hop must be >= 1")
    if n == 0:
        return np.zeros((plan.n_channels, 0), dtype=dtype)
    dec = _run_utterance(plan, w, step=hop, lpf=LPF, cutoff=CUTOFF, dec=True)["dec"]
    return np.ascontiguousarray(_to_host(dec).T.astype(dtype, copy=False))


def extract_envelope_from_matrix(matrix, LPF=False, CUTOFF=100, dtype=np.float64):
    """scripts/processing/EnvelopeExtraction.py:51-67 on an arbitrary (rows, n) matrix:
    abs(paddedHilbert(row)) then lowPassFilter(row, CUTOFF) iff LPF -> float64 (float32 on request),
    same shape."""
    if np.ndim(matrix) != 2:
        raise ValueError("matrix must be two-dimensional (channels x samples)")
    m = _as_matrix(matrix)
    rows, n = m.shape
    if rows == 0:
        return np.zeros(m.shape, dtype=dtype)
    if n == 0:
        # paddedHilbert(empty) -> scipy.signal.hilbert raises "N must be positive."
        raise ValueError("N must be positive.")
    plan = engine.any_plan()
    return _to_host(plan.envelope_rows(_to_device(m, plan.device), LPF, CUTOFF, out_dtype=_torch_dtype(dtype)))


class MatrixStream:
    """Full-rate (C, n) matrices for MANY utterances -- what the file drivers `prepare filter` and `prepare
    envelope` write (GammatoneFiltering.py:69-83, EnvelopeExtraction.py:101-117) -- without paying the
    per-call set-up of the array functions: utterances are processed in batches that fill one of two
    pinned host slots; the matrices handed back are VIEWS into the slot, so writer threads save them
    without another copy while the next batch is computed into the other slot.  A slot is recycled when
    the futures registered with retire() for it have finished.

    mode "filterbank": waves -> erb_filterbank: process(list of waves).
    mode "envelope":   loaded .GFB matrices -> ExtractEnvelopeFromMatrix: process(list of (C, n) arrays)."""

    def __init__(self, coefs, mode="filterbank", LPF=False, CUTOFF=100, dtype=np.float64, slot_bytes=768 << 20):
        # the envelope of a loaded matrix does not depend on a filterbank: any plan of the device will do
        self.plan = engine.any_plan() if coefs is None else engine.plan_for(np.asarray(coefs, dtype=np.float64))
        self.mode, self.lpf, self.cutoff = mode, bool(LPF), CUTOFF
        self.dtype = np.dtype(dtype)
        self.tdt = _torch_dtype(self.dtype)
        self.slot_bytes = int(slot_bytes)
        self._slots = [torch.empty(self.slot_bytes, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        self._guards = [[], []]
        self._dev = torch.empty(self.slot_bytes, dtype=torch.uint8, device=self.plan.device)
        self._stage = None
        self._k = 0
        self.per_value = self.dtype.itemsize   # bytes of one matrix element in a slot

    def batches(self, sizes):
        """Split a list of matrix sizes (elements: C * n per utterance) into runs that fit a slot."""
        out, cur, used = [], [], 0
        for i, sz in enumerate(sizes):
            need = int(sz) * self.per_value
            if need > self.slot_bytes:
                raise ValueError("one matrix of %d bytes does not fit a slot of %d" % (need, self.slot_bytes))
            if used + need > self.slot_bytes and cur:
                out.append(cur)
                cur, used = [], 0
            cur.append(i)
            used += need
        if cur:
            out.append(cur)
        return out

    def retire(self, futures):
        """Futures (writer jobs) that still read the views returned by the last process() call."""
        self._guards[self._k ^ 1] = list(futures)

    def _pinned_stage(self, nbytes):
        if self._stage is None or self._stage.numel() < nbytes:
            self._stage = torch.empty(int(nbytes), dtype=torch.uint8, pin_memory=True)
        return self._stage

    def process(self, items):
        k = self._k
        for fut in self._guards[k]:
            fut.result()
        self._guards[k] = []
        C = self.plan.n_channels
        slot, dev = self._slots[k], self._dev
        stream = torch.cuda.current_stream(self.plan.device)
        views = []
        if self.mode == "filterbank":
            _, waves, lengths = _waves_lengths(list(items))
            total = int(lengths.sum())
            if total == 0:
                return [np.zeros((C, 0), dtype=self.dtype) for _ in waves]
            wdt = torch.from_numpy(waves[0][:0]).dtype
            stage = self._pinned_stage(total * waves[0].dtype.itemsize).view(wdt)[:total]
            np.concatenate(waves, out=stage.numpy())
            wave_dev = stage.to(self.plan.device, non_blocking=True)
            nbytes = C * total * self.per_value
            self.plan.batch(lengths).run(wave_dev, lpf=self.lpf, cutoff=self.cutoff,
                                         out={"gfb": dev[:nbytes].view(self.tdt)}, gfb=self.tdt)
            slot[:nbytes].copy_(dev[:nbytes], non_blocking=True)
            stream.synchronize()
            host = slot.numpy()
            off = 0
            for n in lengths:
                sz = C * int(n) * self.per_value
                views.append(host[off:off + sz].view(self.dtype).reshape(C, int(n)))
                off += sz
        else:
            off = 0
            placed = []
            for m in items:
                if np.ndim(m) != 2:
                    raise ValueError("matrix must be two-dimensional (channels x samples)")
                m = _as_matrix(m)
                rows, n = m.shape
                if n == 0:
                    raise ValueError("N must be positive.")
                src = self._pinned_stage(m.nbytes)[:m.nbytes]
                np.copyto(src.numpy().view(m.dtype).reshape(m.shape), m)
                m_dev = src.to(self.plan.device, non_blocking=True).view(torch.from_numpy(m[:0, :0]).dtype).view(rows, n)
                res = self.plan.envelope_rows(m_dev, self.lpf, self.cutoff, out_dtype=self.tdt)
                sz = rows * n * self.dtype.itemsize
                slot[off:off + sz].copy_(res.view(-1).view(torch.uint8), non_blocking=True)
                stream.synchronize()   # the staging buffer is reused by the next matrix
                placed.append((off, sz, rows, n))
                off += sz
            host = slot.numpy()
            views = [host[o:o + sz].view(self.dtype).reshape(r, n) for o, sz, r, n in placed]
        self._k ^= 1
        return views


def _rows_op(matrix, op, lpf, cutoff):
    m = _as_matrix(matrix)
    if m.shape[1] == 0:
        raise ValueError("N must be positive.")
    plan = engine.any_plan()
    out = plan.envelope_rows(_to_device(m, plan.device), lpf, cutoff, out_dtype=torch.float64, op=op)
    return _to_host(out)


def hilbert_imag_rows(matrix):
    """Imaginary part of paddedHilbert(row) for every row (EnvelopeExtraction.py:20-36)."""
    return _rows_op(matrix, 1, False, 100)


def lowpass_rows(matrix, freq):
    """lowPassFilter(row, freq) for every row (EnvelopeExtraction.py:39-48)."""
    return _rows_op(matrix, 2, True, freq)


def gather_windows_from_matrix(envelopes, timepoints, radius=5, step=160):
    """InputGenerator.py:73-80 on a loaded (C, n) envelope matrix -> (m, 2R+1, C) float32."""
    env = np.ascontiguousarray(envelopes)
    if env.dtype not in (np.dtype(np.float32), np.dtype(np.float64)):
        env = env.astype(np.float64)
    C, n = env.shape
    idx = window_indices(n, timepoints, radius, step)
    plan = engine.any_plan()
    out = engine.gather_windows_cn(_to_device(env, plan.device),
                                   _to_device(np.ascontiguousarray(idx.reshape(-1)), plan.device))
    return _to_host(out).reshape(idx.shape[0], 2 * radius + 1, C)


def window_indices(n, centers, radius, step):
    """Sample indices read by InputGenerator.py:76 for one file, with Python list
    semantics: a negative index wraps once, anything else out of range is an IndexError."""
    centers = np.asarray(centers, dtype=np.int64).reshape(-1)
    offs = step * (np.arange(2 * radius + 1, dtype=np.int64) - radius)
    idx = centers[:, None] + offs[None, :]
    idx = np.where(idx < 0, idx + n, idx)
    if idx.size and (idx.min() < 0 or idx.max() >= n):
        raise IndexError("index out of bounds")
    return idx


_pipelines = OrderedDict()   # corpus-sized requests: cached engine.WindowPipeline objects
_pipelines_lock = threading.Lock()
_MAX_PIPELINES = 2


def _pipeline_for(plan, lengths, dots, step, phase, LPF, CUTOFF, src_offsets=None, share=1, cutoffs=None):
    """The sub-batch layout, device buffers, pinned staging and worker pool of a corpus-sized request
    depend only on the utterance lengths and the grid: built once, reused by every later call with the
    same corpus (a second `prepare input --cutoff K` run, the next epoch's noise draw, a benchmark).
    cutoffs: the settings of a cutoff sweep (their number is part of the layout)."""
    key = (id(plan), hashlib.sha1(lengths.tobytes()).hexdigest(), int(dots), int(step), int(phase), int(share),
           None if src_offsets is None else hashlib.sha1(np.ascontiguousarray(src_offsets).tobytes()).hexdigest(),
           None if cutoffs is None else len(cutoffs))
    with _pipelines_lock:
        pipe = _pipelines.get(key)
        if pipe is None:
            # `share` processes of this box run a pipeline each: split the host cores between their pools
            # (one core stays free for the CUDA host-callback thread that hands frames to the pool)
            threads = max(1, engine.host_cores() // max(int(share), 1) - (1 if int(share) == 1 else 0))
            pipe = engine.WindowPipeline(plan, lengths, dots=dots, step=step, phase=phase, lpf=LPF, cutoff=CUTOFF,
                                         src_offsets=src_offsets, placer=engine.Placer(threads), cutoffs=cutoffs)
            _pipelines[key] = pipe
            while len(_pipelines) > _MAX_PIPELINES:
                _pipelines.popitem(last=False)
        else:
            _pipelines.move_to_end(key)
        pipe.lpf, pipe.cutoff = bool(LPF), CUTOFF
        if cutoffs is not None:
            pipe.cutoffs = tuple(cutoffs)
        return pipe


def release_cached_pipelines():
    """Drop the cached corpus pipelines (device buffers, pinned staging, worker threads) and the pooled
    output block."""
    with _pipelines_lock:
        _pipelines.clear()
    engine.release_host_pool()


def _waves_lengths(waves):
    """waves as a list of 1-D arrays or as (flat, lengths) -> (flat host tensor or None, list of waves or None,
    lengths).  Listed waves of different dtypes are promoted to float64."""
    flat_in = None
    if isinstance(waves, tuple) and len(waves) == 2:
        flat_in, lengths = waves
        lengths = np.ascontiguousarray(lengths, dtype=np.int64)
        if not torch.is_tensor(flat_in):
            flat_in = torch.from_numpy(_as_wave(flat_in))
        if flat_in.dim() != 1 or flat_in.numel() != int(lengths.sum()):
            raise ValueError("flat buffer holds %d samples, lengths add up to %d" % (flat_in.numel(), int(lengths.sum())))
    else:
        waves = [_as_wave(w) for w in waves]
        if len({w.dtype for w in waves}) > 1:
            waves = [w.astype(np.float64) for w in waves]
        lengths = np.asarray([w.shape[0] for w in waves], dtype=np.int64)
    return flat_in, waves, lengths


def _corpus(waves, timepoints, counts):
    """The (waves, timepoints, counts) arguments of features_to_windows -> (flat host tensor or None, list of
    waves or None, lengths, flat centres, counts)."""
    flat_in, waves, lengths = _waves_lengths(waves)
    n_utts = int(lengths.shape[0])
    if counts is not None:
        centers = np.ascontiguousarray(timepoints, dtype=np.int64).reshape(-1)
        counts = np.ascontiguousarray(counts, dtype=np.int64).reshape(-1)
        if counts.shape[0] != n_utts or int(counts.sum()) != centers.shape[0]:
            raise ValueError("counts: one entry per utterance, adding up to the number of timepoints")
    else:
        if len(timepoints) != n_utts:
            raise ValueError("%d utterances, %d timepoint lists" % (n_utts, len(timepoints)))
        counts = np.fromiter((len(t) for t in timepoints), dtype=np.int64, count=n_utts)
        centers = (np.concatenate([np.asarray(t, dtype=np.int64).reshape(-1) for t in timepoints])
                   if n_utts else np.zeros(0, dtype=np.int64))
    return flat_in, waves, lengths, centers, counts


def _shard(lengths, shard, shared_out=None):
    """shard=(rank, world) -> (the utterances engine.shard_utterances deals to `rank`, world); every utterance and
    1 without a shard.  shared_out: whether the call was given the `out` array all ranks fill (None: the call
    writes none)."""
    if shard is None:
        return np.arange(lengths.shape[0]), 1
    rank, world = int(shard[0]), int(shard[1])
    if (shared_out is not None and not shared_out) or not 0 <= rank < world:
        raise ValueError("shard=(rank, world) needs 0 <= rank < world" +
                         ("" if shared_out is None else " and the shared `out` array"))
    return engine.shard_utterances(lengths, world)[rank], world


def _gather_on_grid(dec, idx, phase, step, frame_offsets, dots):
    """Windows (total, dots, C) from the decimated frames `dec` ([frames, C] on the device) of a batch whose
    grid holds every index of `idx` (per utterance, from window_indices)."""
    bases, strided = [], True
    for u, i in enumerate(idx):
        if not i.size:
            continue
        rows = (i - phase) // step + frame_offsets[u]
        strided = strided and bool(np.all(np.diff(rows, axis=1) == 1))
        bases.append(rows)
    rows = np.concatenate(bases)
    if strided:
        base_dev = _to_device(np.ascontiguousarray(rows[:, 0]), dec.device)
        return engine.gather_windows(dec, base_dev, dots, 1)
    res_w = engine.gather_index(dec, _to_device(np.ascontiguousarray(rows.reshape(-1)), dec.device))
    return res_w.view(rows.shape[0], dots, dec.shape[1])


def _windows(waves, coefs, timepoints, counts, radius, step, out, settings=None, LPF=False, CUTOFF=100, shard=None,
             device_out=False):
    """The windows of features_to_windows (settings None: the one envelope setting LPF / CUTOFF, Batch.run) and of
    features_to_windows_sweep (settings: its list, Batch.run_cutoffs), as a list of one result per setting."""
    sweep = settings is not None
    K = len(settings) if sweep else 1
    plan = engine.plan_for(np.asarray(coefs, dtype=np.float64))
    C = plan.n_channels
    dots = 2 * radius + 1
    flat_in, waves, lengths, centers, counts = _corpus(waves, timepoints, counts)
    n_utts = int(lengths.shape[0])
    total = int(counts.sum())
    shape = (total, dots, C)
    outs = None
    if out is not None:
        if sweep:
            outs = _check_out(out, shape, count=K, message="out must be %d C-contiguous float32 arrays of shape %s"
                                                          % (K, shape))
        else:
            outs = [_check_out(out, shape)]
            if device_out:
                raise ValueError("out= is a host array; it cannot be combined with device_out")
    sel, world = _shard(lengths, shard, shared_out=out is not None)
    if total == 0:
        return [np.zeros((0, dots, C), dtype=np.float32) for _ in range(K)] if outs is None else outs

    on_one_grid = False
    if shard is not None or (not device_out and total * dots * C * 4 >= _PIPELINE_BYTES and n_utts >= 8):
        # corpus-sized request: decimated frames over PCIe, rows placed on the host (engine.WindowPipeline)
        first = int(centers[0]) - radius * step
        phase = first % step if first >= 0 else 0
        cen, lens, cnts, src_offsets, row_offsets = centers, lengths, counts, None, None
        if shard is not None:
            mine = np.zeros(n_utts, dtype=bool)
            mine[sel] = True
            cen, lens, cnts = centers[np.repeat(mine, counts)], lengths[sel], counts[sel]
            src_offsets = (np.cumsum(lengths) - lengths)[sel]
            row_offsets = (np.cumsum(counts) - counts)[sel]
        # cheap look at the first utterances before anything is built: a request that is not on one grid
        # goes straight to the one-batch path
        head = int(min(8, cnts.shape[0]))
        n_dec_h = np.where(lens[:head] > phase, (lens[:head] - phase + step - 1) // step, 0)
        probe, phase_h, _ = engine.window_runs(cen[:int(cnts[:head].sum())], cnts[:head], lens[:head],
                                               np.concatenate([[0], np.cumsum(n_dec_h)]), radius, step, phase)
        on_one_grid = probe is not None and phase_h == phase
    if on_one_grid:
        pipe = _pipeline_for(plan, lens, dots, step, phase, LPF, CUTOFF, src_offsets, world, cutoffs=settings)
        results = [engine.host_empty(shape, np.float32) for _ in range(K)] if outs is None else outs
        state = {}

        def detect():
            # runs on the host while the first sub-batch is already on the device
            runs, phase2, _ = engine.window_runs(cen, cnts, lens, pipe.frame_offsets, radius, step, phase,
                                                 row_offsets=row_offsets)
            state["ok"] = runs is not None and phase2 == phase
            return runs if state["ok"] else np.zeros((0, 3), dtype=np.int64)

        pipe.run(flat_in if flat_in is not None else waves if shard is None else [waves[u] for u in sel], detect,
                 results if sweep else results[0])
        if state["ok"]:
            return results
        # legal timepoints that are not windows of consecutive frames of one grid (a wrapping index, mixed
        # phases) further down the corpus: nothing was placed; the one-batch path below answers
        del results
    if shard is not None:
        raise ValueError("shard= needs timepoints that are windows of consecutive frames of one decimated grid")

    # one batch, windows gathered on the device
    cpos = np.concatenate([[0], np.cumsum(counts)])
    idx = [window_indices(int(n), centers[cpos[u]:cpos[u + 1]], radius, step) for u, n in enumerate(lengths)]
    # one decimated grid serves every window when all indices share a residue mod step
    allidx = np.concatenate([i.reshape(-1) for i in idx if i.size])
    phase = int(allidx[0] % step)
    on_grid = bool(np.all(allidx % step == phase))
    if sweep and not on_grid:
        raise ValueError("features_to_windows_sweep needs every window index on one decimated grid (all equal mod "
                         "step = %d); call features_to_windows once per cutoff for these timepoints" % step)
    wave_dev = _to_device(flat_in if flat_in is not None else np.concatenate(waves) if len(waves) > 1 else waves[0],
                          plan.device)
    if on_grid:
        batch = plan.batch(lengths, step=step, phase=phase)
        planes = (batch.run_cutoffs(wave_dev, settings) if sweep else
                  [batch.run(wave_dev, lpf=LPF, cutoff=CUTOFF, dec=True)["dec"]])
        res_w = [_gather_on_grid(p, idx, phase, step, batch.frame_offsets, dots) for p in planes]
    else:
        # an off-grid request (features_to_windows only): windows gathered from the full-rate envelope
        batch = plan.batch(lengths, step=step, phase=0)
        env_t = batch.run(wave_dev, lpf=LPF, cutoff=CUTOFF, env_t=True)["env_t"]
        rows = np.concatenate([i + batch.sample_offsets[u] for u, i in enumerate(idx) if i.size])
        res_w = [engine.gather_index(env_t, _to_device(np.ascontiguousarray(rows.reshape(-1)), plan.device))
                 .view(shape)]
    if device_out:
        return res_w
    host = [_to_host(r) for r in res_w]
    if outs is None:
        return host
    for o, h in zip(outs, host):
        o[...] = h
    return outs


def features_to_windows(waves, coefs, timepoints, LPF=False, CUTOFF=100, radius=5, step=160, device_out=False,
                        out=None, counts=None, shard=None):
    """Fused path from waveforms to the (N, 2R+1, C) float32 input tensor.

    waves: list of 1-D arrays (same dtype), or (flat, lengths) as returned by ingest.read_corpus
    (one buffer of all samples, pinned for full speed); timepoints: list of int arrays (window
    centres per utterance, in output order) -- or, with `counts`, ONE flat int array of all centres
    and counts[u] of them per utterance.  Equivalent to
    erb_filterbank -> ExtractEnvelopeFromMatrix(LPF, CUTOFF) -> the gather of
    InputGenerator.py:73-80 per utterance, rows concatenated in list order.  `out`: an existing
    C-contiguous (N, 2R+1, C) float32 numpy array to fill (a corpus-sized result is 7.5 GB: reusing
    it saves its page faults); by default a fresh array is returned.
    shard=(rank, world): one of `world` processes (one per GPU, e.g. under torchrun) that were all
    handed the SAME corpus and the SAME `out` -- a shared mapping, hostmem.SharedArray.  This call
    computes the utterances engine.shard_utterances deals to `rank` and writes their rows, and only
    theirs, at their final offsets; there is nothing to exchange afterwards."""
    return _windows(waves, coefs, timepoints, counts, radius, step, out, LPF=LPF, CUTOFF=CUTOFF, shard=shard,
                    device_out=device_out)[0]


def features_to_windows_sweep(waves, coefs, timepoints, cutoffs, radius=5, step=160, counts=None, out=None):
    """features_to_windows for several envelope settings at once: a list of K (N, 2R+1, C) float32 arrays, the
    k-th equal to features_to_windows(..., LPF=cutoffs[k] is not None, CUTOFF=cutoffs[k]).  cutoffs: 1..4
    entries, each a cutoff in (0, 8000) Hz or None for no low-pass.  The filterbank and the Hilbert transform
    run once for all settings (engine.Batch.run_cutoffs).  waves, timepoints, counts and `out` (here a list of
    K arrays) mean what they mean in features_to_windows.

    Every window index must lie on one decimated grid (all indices equal mod `step`), as those of
    LabelDataGenerator's CSV do; anything else raises ValueError (call features_to_windows per cutoff).
    Corpus-sized requests go through engine.WindowPipeline (bit for bit what features_to_windows gives per
    cutoff); smaller ones take one batch, whose time-chunked utterances all warm up for the slowest setting (the
    low-pass pole nearest the unit circle)."""
    settings = list(cutoffs)
    engine.cutoff_settings(settings)
    return _windows(waves, coefs, timepoints, counts, radius, step, out, settings=settings)


class FrameWindows:
    """The input tensor of a corpus WITHOUT its (2R+1)-fold redundancy: the decimated envelope frames of every
    utterance in one page-locked host array, and the windows as overlapping VIEWS of it.

    Row k of utterance u of `input_data.npy` is frames k .. k+dots-1 of that utterance
    (InputGenerator.py:73-80 on the label grid of LabelDataGenerator.py:38-50), i.e. dots*C consecutive floats
    starting at frame frame_offsets[u] + k: `windows(u)` is that (counts[u], dots, C) array as a strided view,
    `self[r]` is global row r, `materialize()` builds the reference's tensor (bit-identical to
    api.features_to_windows).  0.71 GB instead of 7.5 GB for the 4620-utterance corpus: a consumer that reads
    windows through the views (a training loop that gathers mini-batches) never pays for the expansion, which is
    what bounds the end-to-end time of the full tensor on any number of GPUs (DESIGN.md section 6).

    `frames` belongs to the cached pipeline of this corpus layout: it is valid until the next
    features_to_frames / features_to_windows call with the same lengths (copy it to keep it)."""

    def __init__(self, frames, frame_offsets, counts, dots, utterances, placer):
        self.frames, self.frame_offsets, self.counts, self.dots = frames, frame_offsets, counts, int(dots)
        self.utterances = utterances          # indices into the caller's utterance list (a shard holds a subset)
        self.row_offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        self._placer = placer

    def __len__(self):
        return int(self.row_offsets[-1])

    def windows(self, u):
        """(counts[u], dots, C) float32 view of the u-th utterance held here (no copy)."""
        C = self.frames.shape[1]
        k, f0 = int(self.counts[u]), int(self.frame_offsets[u])
        if k == 0:
            return np.zeros((0, self.dots, C), dtype=np.float32)
        base = self.frames[f0:f0 + k + self.dots - 1]
        return np.lib.stride_tricks.as_strided(base, shape=(k, self.dots, C), strides=(C * 4, C * 4, 4), writeable=False)

    def __getitem__(self, r):
        r = int(r)
        if r < 0:
            r += len(self)
        if not 0 <= r < len(self):
            raise IndexError("row %d of %d" % (r, len(self)))
        u = int(np.searchsorted(self.row_offsets, r, side="right") - 1)
        f = int(self.frame_offsets[u]) + r - int(self.row_offsets[u])
        return self.frames[f:f + self.dots]

    def materialize(self, out=None):
        """The (N, dots, C) float32 tensor of the reference, rows placed by the library's host pool."""
        C = self.frames.shape[1]
        out = engine.host_empty((len(self), self.dots, C), np.float32) if out is None else out
        runs = np.stack([self.frame_offsets[:-1], self.row_offsets[:-1], self.counts], axis=1).astype(np.int64)
        runs = np.ascontiguousarray(runs[runs[:, 2] > 0])
        if runs.shape[0]:
            self._placer.submit(torch.from_numpy(self.frames), runs, out, dots=self.dots, stream=None, after_stream=False)
            self._placer.wait()
        return out


def features_to_frames(waves, coefs, LPF=False, CUTOFF=100, radius=5, step=160, counts=None, shard=None):
    """Waveforms -> FrameWindows: the same filterbank -> envelope -> decimation as features_to_windows on the
    label grid (window k of an utterance is centred on step*radius + step*k, LabelDataGenerator.py:38-50), but the
    call ends when the decimated frames are on the host -- nothing is expanded.  waves: (flat, lengths) or a list
    of 1-D arrays; counts[u]: windows of utterance u (default: the label grid's int(n/step - dots - 1));
    shard=(rank, world): this process computes the utterances engine.shard_utterances deals to `rank`
    (FrameWindows.utterances)."""
    coefs = np.asarray(coefs, dtype=np.float64)
    plan = engine.plan_for(coefs)
    dots = 2 * radius + 1
    flat_in, waves, lengths = _waves_lengths(waves)
    n_frames = (lengths + step - 1) // step
    grid = np.maximum((lengths / step - dots - 1).astype(np.int64), 0)
    if counts is None:
        counts = grid
    else:
        counts = np.ascontiguousarray(counts, dtype=np.int64).reshape(-1)
        if counts.shape[0] != lengths.shape[0] or np.any(counts < 0) or np.any(counts + dots - 1 > np.maximum(n_frames, dots - 1)):
            raise IndexError("counts: one entry per utterance, windows must lie inside the utterance's frames")
    sel, world = _shard(lengths, shard)
    pipe = _pipeline_for(plan, lengths[sel], dots, step, 0, LPF, CUTOFF,
                         None if shard is None else (np.cumsum(lengths) - lengths)[sel], world)
    no_runs = np.zeros((0, 3), dtype=np.int64)
    pipe.run(flat_in if flat_in is not None else [waves[u] for u in sel], no_runs, None)
    return FrameWindows(pipe._dec_host.numpy(), pipe.frame_offsets, counts[sel], dots, sel, pipe.placer)


def dense_frames(wave, coefs, LPF=False, CUTOFF=100, radius=5, step=160, normalize=True, dtype=np.float64,
                 frames=None):
    """In-memory front end of Evaluating.EvaluateOneWavArray (Evaluating.py:52-80):
    filterbank -> envelope -> dense stride-1 framing (-> normalizeInput per frame).
    Returns (nb, 2R+1, C); `frames=(i0, i1)` restricts the frame range."""
    w, plan, n = _utterance(wave, coefs)
    dots = 2 * radius + 1
    nb = int(n - dots * step)
    i0, i1 = (0, nb) if frames is None else (int(frames[0]), int(frames[1]))
    if frames is not None and not (0 <= i0 <= i1 <= max(nb, 0)):
        raise IndexError("frames=(%d, %d) outside the %d frames of this utterance" % (i0, i1, max(nb, 0)))
    if nb <= 0 or i1 <= i0:
        return np.zeros((0, dots, plan.n_channels), dtype=dtype)
    env_t = _run_utterance(plan, w, step=step, lpf=LPF, cutoff=CUTOFF, env_t=True)["env_t"]
    return _normalised_frames(env_t, dots, step, i0, i1, normalize, dtype)


def evaluate_front_end(wave, coefs, LPF=False, CUTOFF=100, radius=5, step=160, frames=True, dtype=np.float64):
    """ONE filterbank pass for `cnn eval*` (Evaluating.py:52-80): the (C, n) envelopes the figure shows
    and the (nb, 2R+1, C) normalised frames model.predict takes, both from the same time-major envelope.
    frames=False returns (envelopes, device env_t) for a consumer on the device (api.cnn_evaluate)."""
    w, plan, n = _utterance(wave, coefs)
    dots = 2 * radius + 1
    if n == 0:
        raise ValueError("N must be positive.")
    res = _run_utterance(plan, w, step=step, lpf=LPF, cutoff=CUTOFF, env=torch.float64, env_t=True)
    envelopes = _to_host(res["env"]).reshape(plan.n_channels, n)
    if not frames:
        return envelopes, res["env_t"]
    nb = int(n - dots * step)
    if nb <= 0:
        return envelopes, np.zeros((0, dots, plan.n_channels), dtype=dtype)
    return envelopes, _normalised_frames(res["env_t"], dots, step, 0, nb, True, dtype)


_networks = OrderedDict()


def _check_cnn_geometry(radius, coefs):
    """coefs as float64, after checking that the tensor-core network takes this geometry."""
    coefs = np.asarray(coefs, dtype=np.float64)
    if radius != 5 or coefs.shape[0] != 128:
        raise ValueError("the tensor-core network is built for RADIUS = 5 and 128 channels")
    return coefs


def _network_for(weights):
    """Tensor-core network for a list of Keras-layout arrays (or an F2CNN module), cached by content."""
    from . import cnn
    arrays = cnn.keras_arrays(weights) if isinstance(weights, torch.nn.Module) else [np.asarray(a) for a in weights]
    h = hashlib.sha1()
    for a in arrays:
        h.update(np.ascontiguousarray(a, dtype=np.float32).tobytes())
    key = (h.hexdigest(), torch.cuda.current_device())
    net = _networks.get(key)
    if net is None:
        net = cnn.TensorCoreCNN(arrays)
        _networks[key] = net
        while len(_networks) > 4:
            _networks.popitem(last=False)
    return net


def cnn_evaluate(wave, coefs, weights, LPF=False, CUTOFF=100, radius=5, step=160, with_envelopes=True):
    """`cnn eval*` from waveform to scores on the device (Evaluating.py:52-87): filterbank -> envelope ->
    every stride-1 frame normalised and run through the reference network on the tensor cores
    (csrc/f2_cnn.cu), without materialising the (nb, 11, 128) frame tensor.  weights: the 12 arrays of
    Keras' model.get_weights() or an f2cnn_b200.cnn.F2CNN module.  Returns (scores (nb, 2) float32,
    envelopes (C, n) float64 or None).  Only the configured geometry (RADIUS = 5, 128 channels)."""
    coefs = _check_cnn_geometry(radius, coefs)
    net = _network_for(weights)
    if with_envelopes:
        envelopes, env_t = evaluate_front_end(wave, coefs, LPF, CUTOFF, radius, step, frames=False)
    else:
        w, plan, _ = _utterance(wave, coefs)
        envelopes, env_t = None, _run_utterance(plan, w, step=step, lpf=LPF, cutoff=CUTOFF, env_t=True)["env_t"]
    scores = net.predict_envelope(env_t, step)
    return _to_host(scores), envelopes


_CNN_ENV_BYTES = 2 << 30   # time-major envelope of one sub-batch of cnn_evaluate_corpus (512 bytes per sample)


def cnn_evaluate_corpus(waves, coefs, weights, LPF=False, CUTOFF=100, radius=5, step=160, out=None, shard=None):
    """cnn_evaluate for a whole corpus: the scores of every stride-1 frame of every utterance, e.g. a test set
    scored by a trained model.  waves: list of 1-D arrays, or (flat, lengths) as returned by ingest.read_corpus.
    Returns (scores, offsets): scores is the float32 (sum(nb_u), 2) host array with nb_u = max(n_u - (2R+1)*step,
    0) (Evaluating.py:70-78), and utterance u's scores are scores[offsets[u]:offsets[u+1]].

    Utterances go through the front end in sub-batches of whole utterances (never split into time chunks, so an
    utterance's envelope and scores do not depend on the sub-batch or shard it lands in), and each sub-batch
    through the network in one pass whose chunks run across utterance boundaries
    (TensorCoreCNN.predict_segments).  Scores equal cnn_evaluate's where cnn_evaluate computes the same envelope
    (it may split a lone long utterance into time chunks, whose envelope differs in the last float32 bits).
    Raises ValueError naming the first utterance with a frame value <= 0 (Training.normalizeInput).
    out: an existing C-contiguous float32 (sum(nb_u), 2) array to fill.  shard=(rank, world): one of `world`
    processes (one per GPU) handed the same corpus and the same `out` -- a shared mapping,
    hostmem.SharedArray -- scores the utterances engine.shard_utterances deals to `rank` and writes them, and
    only them, at their final offsets.  Only the configured geometry (RADIUS = 5, 128 channels)."""
    coefs, flat_in, waves, lengths, nb, offsets, sel = _scoring_corpus(waves, coefs, radius, step, shard, out is not None,
                                                                       "cnn_evaluate_corpus")
    total = int(offsets[-1])
    scores = np.empty((total, 2), dtype=np.float32) if out is None else _check_out(out, (total, 2))
    for _ in _scored_sub_batches(flat_in, waves, lengths, nb, sel, coefs, weights, LPF, CUTOFF, int(step),
                                 scores, offsets):
        pass
    return scores, offsets


def _scoring_corpus(waves, coefs, radius, step, shard, shared_out, caller):
    """The arguments common to the corpus scoring calls, checked -> (coefs, flat host tensor or None, list of waves
    or None, lengths, frames per utterance nb, score offsets, the utterances this call scores)."""
    coefs = _check_cnn_geometry(radius, coefs)
    flat_in, waves, lengths = _waves_lengths(waves)
    if flat_in is not None and flat_in.device.type != "cpu":
        raise ValueError("%s takes the flat wave buffer in host memory (it is on %s)" % (caller, flat_in.device))
    nb = np.maximum(lengths - (2 * radius + 1) * int(step), 0)
    offsets = np.concatenate([[0], np.cumsum(nb)]).astype(np.int64)
    sel, _ = _shard(lengths, shard, shared_out)
    return coefs, flat_in, waves, lengths, nb, offsets, sel


def _scored_sub_batches(flat_in, waves, lengths, nb, sel, coefs, weights, LPF, CUTOFF, step, scores=None,
                        offsets=None):
    """The utterances `sel` (ascending) through the front end and the network in sub-batches of whole utterances:
    yields (sub, device scores of sub's frames back to back) per sub-batch; the scores are valid until the next
    step.  With `scores`, utterance u's rows are also copied to scores[offsets[u]:offsets[u+1]] on the host."""
    from . import cnn
    sel = sel[nb[sel] > 0]          # an utterance without frames has nothing to score
    if sel.size == 0:
        return
    plan = engine.plan_for(coefs)
    net = _network_for(weights)
    # consecutive utterances (in `sel` order) whose envelopes fit _CNN_ENV_BYTES; a larger one goes alone
    env_bytes = lengths[sel] * plan.n_channels * 4
    subs, start, used = [], 0, 0
    for i, b in enumerate(env_bytes):
        if used + b > _CNN_ENV_BYTES and i > start:
            subs.append(sel[start:i])
            start, used = i, 0
        used += int(b)
    subs.append(sel[start:])
    src = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    host = flat_in.numpy() if flat_in is not None else None
    wdt = flat_in.dtype if flat_in is not None else torch.from_numpy(waves[0][:0]).dtype
    max_samples = max(int(lengths[sub].sum()) for sub in subs)
    max_frames = max(int(nb[sub].sum()) for sub in subs)
    stage = torch.empty(max_samples, dtype=wdt, pin_memory=True)
    wave_dev = torch.empty(max_samples, dtype=wdt, device=plan.device)
    env_buf = torch.empty((max_samples, plan.n_channels), dtype=torch.float32, device=plan.device)
    scores_host = torch.empty((max_frames, 2), dtype=torch.float32, pin_memory=True) if scores is not None else None
    for sub in subs:
        lens = lengths[sub]
        n = int(lens.sum())
        np.concatenate([host[src[u]:src[u + 1]] if host is not None else waves[u] for u in sub], out=stage.numpy()[:n])
        wave_dev[:n].copy_(stage[:n], non_blocking=True)
        batch = plan.batch(lens, step=step, target_items=1)
        env_t = batch.run(wave_dev[:n], lpf=LPF, cutoff=CUTOFF, out={"env_t": env_buf[:n]})["env_t"]
        try:
            # returns after a device synchronise: the staging buffer is free for the next sub-batch
            sc = net.predict_segments(env_t, step, batch.sample_offsets[:-1], nb[sub])
        except cnn.NonPositiveInput as e:
            raise ValueError("values must all be positive (utterance %d)" % int(sub[e.segment])) from None
        if scores is not None:
            k = int(sc.shape[0])
            scores_host[:k].copy_(sc)
            got = scores_host.numpy()
            at = 0
            for u in sub:
                scores[offsets[u]:offsets[u + 1]] = got[at:at + nb[u]]
                at += int(nb[u])
        yield sub, sc


def _label_ints(a, dtype, what):
    """A 1-D array of integers (integral floats included) that `dtype` holds, as `dtype`; else ValueError."""
    a = np.asarray(a).reshape(-1)
    lo, hi = np.iinfo(dtype).min, np.iinfo(dtype).max
    if a.size:
        if a.dtype.kind == "f":
            ok = bool(np.all(np.isfinite(a))) and np.array_equal(np.trunc(a), a) and a.min() >= lo and a.max() < -float(lo)
        else:
            ok = a.dtype.kind in "iub" and int(a.min()) >= lo and int(a.max()) <= hi
        if not ok:
            raise ValueError("label %s must be integers that %s holds" % (what, np.dtype(dtype).name))
    return np.ascontiguousarray(a, dtype=dtype)


def _label_arrays(times, classes, counts, n_utts):
    """Flattened labels, checked: (int64 times, int32 classes, int64 label offsets (n_utts + 1)).  ValueError for
    times and classes of different lengths, non-integer values, counts that do not add up to the number of labels
    and times that decrease within an utterance."""
    times, classes = _label_ints(times, np.int64, "times"), _label_ints(classes, np.int32, "classes")
    counts = _label_ints(counts, np.int64, "counts")
    if times.shape != classes.shape:
        raise ValueError("%d label times, %d classes" % (times.shape[0], classes.shape[0]))
    if counts.shape[0] != n_utts or np.any(counts < 0) or int(counts.sum()) != times.shape[0]:
        raise ValueError("label counts: one entry per utterance (%d), adding up to the %d labels"
                         % (n_utts, times.shape[0]))
    loff = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    falls = np.flatnonzero(np.diff(times) < 0) + 1      # label k is below label k - 1 ...
    falls = falls[~np.isin(falls, loff)]                 # ... of the same utterance
    if falls.size:
        u = int(np.searchsorted(loff, falls[0], side="right")) - 1
        raise ValueError("label times of utterance %d decrease (label %d)" % (u, int(falls[0] - loff[u])))
    return times, classes, loff


def label_accuracy(scores, labels, step=160):
    """The reference's label accuracy of one utterance (Evaluating.py:87-110) as two exact integers (hits,
    counted): accuracy = hits / counted.  scores: the (F, 2) scores of the utterance's stride-1 frames, a host
    array or a CUDA tensor (float32 on the device; a host array of another dtype is reduced to its decisions
    s[1] > s[0] first, which rounding it to float32 could change); labels: [(time in samples, class), ...],
    times non-decreasing, as ExtractLabel gives them.  Frame i counts when it lies strictly between two
    consecutive label times and closer than `step` to one of them, and hits when its decision equals the class of
    the nearer label (the earlier one on a tie).  Computed on the GPU (f2_label_accuracy)."""
    labels = [tuple(l) for l in labels]
    times, classes, loff = _label_arrays([l[0] for l in labels], [l[1] for l in labels], [len(labels)], 1)
    if torch.is_tensor(scores) and scores.is_cuda:
        if scores.dtype != torch.float32 or scores.dim() != 2 or scores.shape[1] != 2:
            raise ValueError("device scores must be a (F, 2) float32 tensor")
        sc = scores.contiguous()
    else:
        host = scores.numpy() if torch.is_tensor(scores) else np.asarray(scores)
        if host.ndim != 2 or host.shape[1] != 2:
            raise ValueError("scores must have shape (F, 2), got %s" % (host.shape,))
        if host.dtype != np.float32:
            rising = host[:, 1] > host[:, 0]
            host = np.zeros(host.shape, dtype=np.float32)
            host[:, 1] = rising
        sc = _to_device(np.ascontiguousarray(host), torch.device("cuda", torch.cuda.current_device()))
    dev = sc.device
    counts = engine.label_accuracy(sc, _to_device(np.asarray([0, sc.shape[0]], dtype=np.int64), dev),
                                   _to_device(times, dev), _to_device(classes, dev), _to_device(loff, dev), int(step))
    hits, counted = _to_host(counts)[:, 0]
    return int(hits), int(counted)


def cnn_label_accuracy_corpus(waves, coefs, weights, labels, LPF=False, CUTOFF=100, radius=5, step=160,
                              with_scores=False, out=None, shard=None):
    """The reference's label accuracy (Evaluating.py:87-110) of every utterance of a labelled corpus under one
    network: cnn_evaluate_corpus, with each sub-batch's scores counted on the device (f2_label_accuracy) before
    they leave it.  labels = (times, classes, counts): all label times (samples, non-decreasing within an
    utterance) and classes back to back, counts[u] of them for utterance u -- flattened like the (centres, counts)
    of features_to_windows.  Returns int64 arrays (hits, counted) of one entry per utterance, utterance u's
    accuracy being hits[u] / counted[u]; with_scores=True returns (hits, counted, scores, offsets) with the scores
    and offsets cnn_evaluate_corpus returns.  out=(hits, counted): existing C-contiguous int64 arrays to fill.
    shard=(rank, world): as in cnn_evaluate_corpus, with `out` the shared pair of arrays; it does not combine with
    with_scores (cnn_evaluate_corpus scores a shard into a shared array).  Raises ValueError before any launch on
    malformed labels or another geometry than RADIUS = 5, 128 channels."""
    if shard is not None and with_scores:
        raise ValueError("shard= does not combine with with_scores")
    coefs, flat_in, waves, lengths, nb, offsets, sel = _scoring_corpus(
        waves, coefs, radius, step, shard, out is not None, "cnn_label_accuracy_corpus")
    n_utts = int(lengths.shape[0])
    if len(labels) != 3:
        raise ValueError("labels = (times, classes, counts)")
    times, classes, loff = _label_arrays(*labels, n_utts)
    hits, counted = (np.zeros(n_utts, np.int64), np.zeros(n_utts, np.int64)) if out is None else _check_out(
        out, (n_utts,), np.int64, count=2, message="out must be two C-contiguous int64 arrays of shape (%d,)" % n_utts)
    hits[sel] = 0
    counted[sel] = 0
    scores = np.empty((int(offsets[-1]), 2), dtype=np.float32) if with_scores else None
    owner = np.repeat(np.arange(n_utts), np.diff(loff))
    mine = np.zeros(n_utts, dtype=bool)
    step = int(step)
    for sub, sc in _scored_sub_batches(flat_in, waves, lengths, nb, sel, coefs, weights, LPF, CUTOFF, step,
                                       scores, offsets):
        dev = sc.device
        mine[:] = False
        mine[sub] = True
        pick = mine[owner]        # sub's labels, in utterance order (sub is ascending)
        sub_loff = np.concatenate([[0], np.cumsum(np.diff(loff)[sub])]).astype(np.int64)
        sub_off = np.concatenate([[0], np.cumsum(nb[sub])]).astype(np.int64)
        got = _to_host(engine.label_accuracy(sc, _to_device(sub_off, dev), _to_device(times[pick], dev),
                                             _to_device(classes[pick], dev), _to_device(sub_loff, dev), step))
        hits[sub], counted[sub] = got[0], got[1]
    if with_scores:
        return hits, counted, scores, offsets
    return hits, counted


def label_fit(tracks, firsts, centers, radius=5, step=160):
    """Slope labels for a whole corpus in one launch (LabelDataGenerator.py:60-68).

    tracks[u]: float64 formant track of utterance u (Hz per 10 ms frame); firsts[u]: int array,
    index in tracks[u] of the first of the 2*radius+1 frames of each timepoint; centers[u]: the
    timepoints in samples.  Returns a float64 (N, 4) host array of (slope, intercept, r, p), rows in
    utterance order then timepoint order."""
    plan = engine.any_plan()
    dots = 2 * int(radius) + 1
    offs = np.concatenate([[0], np.cumsum([len(t) for t in tracks])]).astype(np.int64)
    first_parts, center_parts = [], []
    for u, (f, c) in enumerate(zip(firsts, centers)):
        f = np.asarray(f, dtype=np.int64)
        c = np.asarray(c, dtype=np.int64)
        if f.shape != c.shape:
            raise ValueError("firsts[%d] and centers[%d] differ in length" % (u, u))
        if f.size and (f.min() < 0 or f.max() + dots > len(tracks[u])):
            raise IndexError("utterance %d: a window leaves the formant track" % u)
        first_parts.append(f + offs[u])
        center_parts.append(c)
    first = np.concatenate(first_parts + [np.zeros(0, np.int64)])
    center = np.concatenate(center_parts + [np.zeros(0, np.int64)])
    if first.size == 0:
        return np.zeros((0, 4))
    if center.max() > np.iinfo(np.int32).max:
        raise OverflowError("timepoint beyond int32")
    flat = np.concatenate([np.asarray(t, dtype=np.float64) for t in tracks])
    out = engine.label_fit(_to_device(flat, plan.device), _to_device(first, plan.device),
                           _to_device(center.astype(np.int32), plan.device), dots, step)
    return _to_host(out)
