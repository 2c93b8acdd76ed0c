"""Host-side engine: plans, batches and launch helpers over the C ABI.

PyTorch is used only as plumbing (device memory, pinned host buffers, streams); every
computation of the hot path happens in libf2cnn_b200.so.  Nothing here falls back to
numpy/scipy/torch math: without the library or a CUDA device the calls raise."""
import ctypes
import hashlib
import os
import threading

import numpy as np
import torch

from . import _native
from ._native import F2_F32, F2_F64, F2_I16, RunArgs, check

_NP2F2 = {np.dtype(np.int16): F2_I16, np.dtype(np.float32): F2_F32, np.dtype(np.float64): F2_F64}
_T2F2 = {torch.int16: F2_I16, torch.float32: F2_F32, torch.float64: F2_F64}


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("f2cnn_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


def _stream_ptr(stream):
    s = stream if stream is not None else torch.cuda.current_stream()
    return ctypes.c_void_p(s.cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def lowpass_coefficients(cutoff_hz):
    """(b0, a1) of butter(1, cutoff/8000, 'low') -- reference EnvelopeExtraction.py:47."""
    b0 = ctypes.c_double()
    a1 = ctypes.c_double()
    check(_native.lib().f2_lowpass_coefficients(float(cutoff_hz), ctypes.byref(b0), ctypes.byref(a1)))
    return b0.value, a1.value


def bank_check(coefs):
    """(predicted worst float32 error in units of the 1e-4 x RMS tolerance, channel) of a
    make_erb_filters bank -- the host-only check Plan() applies (f2_bank_check)."""
    coefs = np.ascontiguousarray(coefs, dtype=np.float64)
    if coefs.ndim != 2 or coefs.shape[1] != 10:
        raise ValueError("coefs must be (n_channels, 10) as returned by make_erb_filters")
    pred, chan = ctypes.c_double(), ctypes.c_int()
    check(_native.lib().f2_bank_check(coefs.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), int(coefs.shape[0]),
                                      ctypes.byref(pred), ctypes.byref(chan)))
    return pred.value, chan.value


def bank_check_groups(coefs):
    """Predicted float32 error of every group of 32 channels, in units of the 1e-4 x RMS tolerance (numpy
    array, host only, f2_bank_check_groups).  Plan(..., float64_sections=True) runs the groups above 1.0
    in float64."""
    coefs = np.ascontiguousarray(coefs, dtype=np.float64)
    if coefs.ndim != 2 or coefs.shape[1] != 10:
        raise ValueError("coefs must be (n_channels, 10) as returned by make_erb_filters")
    out = np.zeros(max(1, (coefs.shape[0] + 31) // 32), dtype=np.float64)
    check(_native.lib().f2_bank_check_groups(coefs.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                             int(coefs.shape[0]), out.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
    return out


def float64_sections_default():
    """The float64_sections setting of Plan(..., float64_sections=None): F2CNN_B200_FLOAT64_SECTIONS=1."""
    return os.environ.get("F2CNN_B200_FLOAT64_SECTIONS", "0") == "1"


class Plan:
    """One gammatone filterbank on one device.  coefs = make_erb_filters output (C,10).

    float64_sections: the kernels compute in float32, and a bank float32 cannot hold to the 1e-4 x RMS
    tolerance (bank_check > 1: poles very near z = 1, e.g. LOW_FREQ = 20 Hz) is refused.  With True, the
    groups of 32 channels that bank_check_groups puts above 1 run their sections in float64 instead and
    the bank is accepted; the others are unchanged.  None: F2CNN_B200_FLOAT64_SECTIONS=1 (off by default)."""

    def __init__(self, coefs, device=None, float64_sections=None):
        _require_cuda()
        coefs = np.ascontiguousarray(coefs, dtype=np.float64)
        if coefs.ndim != 2 or coefs.shape[1] != 10:
            raise ValueError("coefs must be (n_channels, 10) as returned by make_erb_filters")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        self.n_channels = int(coefs.shape[0])
        self.coefs = coefs
        self.float64_sections = float64_sections_default() if float64_sections is None else bool(float64_sections)
        self._h = ctypes.c_void_p()
        flags = _native.F2_PLAN_FLOAT64_SECTIONS if self.float64_sections else 0
        check(_native.lib().f2_plan_create_ex(coefs.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), self.n_channels,
                                              self.device.index, flags, ctypes.byref(self._h)))
        n_groups = (self.n_channels + 31) // 32
        mask = (ctypes.c_ubyte * n_groups)()
        if _native.lib().f2_plan_float64_groups(self._h, mask, n_groups) < 0:
            raise _native.F2Error(_native.F2_ERR_INVALID, _native.lib().f2_last_error().decode())
        self.float64_groups = tuple(g for g in range(n_groups) if mask[g])
        self._ws = {}
        self._ws_lock = threading.Lock()
        self._frozen = False  # plan_for() hands the same object to every caller: no mutation there

    def __del__(self):
        try:
            h = getattr(self, "_h", None)
            if h is not None and h.value:
                _native.lib().f2_plan_destroy(h)
                self._h = None
        except Exception:  # interpreter shutdown: module globals may already be gone
            pass

    def set_warmup(self, w_imag=0, w_edge=0, w_casc=0):
        """Development knob (f2_plan_set_warmup).  Only on a plan you created yourself with Plan(...):
        the plans plan_for() caches are shared by every caller and stay as created."""
        if self._frozen:
            raise RuntimeError("set_warmup on a cached plan (engine.plan_for): create a private engine.Plan(coefs)")
        check(_native.lib().f2_plan_set_warmup(self._h, int(w_imag), int(w_edge), int(w_casc)))

    def get_warmup(self):
        a, b, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        check(_native.lib().f2_plan_get_warmup(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return a.value, b.value, c.value

    def batch(self, lengths, step=160, phase=0, target_items=0):
        return Batch(self, lengths, step, phase, target_items)

    def workspace(self, nbytes, stream=None):
        """Grow-only scratch of this plan's launches ON ONE STREAM (caller-owned per the C ABI).
        Launches on different streams get different blocks, so they may overlap; the block is
        allocated under the stream it serves, which is what makes handing a replaced block back to
        torch's caching allocator safe (it is only reused in that stream's order)."""
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        key = int(s.cuda_stream)
        with self._ws_lock:
            ws = self._ws.get(key)
            if ws is None or ws.numel() < nbytes:
                self._ws.pop(key, None)
                ws = None
                with torch.cuda.stream(s):
                    ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
                self._ws[key] = ws
            return ws

    # -- stand-alone envelope of matrix rows (ExtractEnvelopeFromMatrix on foreign data) ----
    def envelope_rows(self, matrix_dev, lpf, cutoff, out_dtype=torch.float64, stream=None, op=0):
        rows, n = matrix_dev.shape
        out = torch.empty((rows, n), dtype=out_dtype, device=self.device)
        if rows == 0 or n == 0:
            return out
        L = _native.lib()
        if not matrix_dev.is_contiguous() or matrix_dev.device != self.device:
            raise ValueError("envelope_rows wants a contiguous matrix on the plan's device")
        ws = self.workspace(L.f2_envelope_rows_workspace_bytes(rows, n), stream)
        check(L.f2_rows_op(self._h, _ptr(matrix_dev), _T2F2[matrix_dev.dtype], rows, n, int(op), int(bool(lpf)),
                           float(cutoff), _ptr(out), _T2F2[out_dtype], _ptr(ws), ws.numel(), _stream_ptr(stream)))
        return out


class Batch:
    """A set of utterances (by length) prepared for repeated runs on one plan."""

    def __init__(self, plan, lengths, step=160, phase=0, target_items=0):
        self.plan = plan
        self.lengths = np.ascontiguousarray(lengths, dtype=np.int64).reshape(-1)
        self.n_utts = int(self.lengths.shape[0])
        self.step, self.phase = int(step), int(phase)
        self._h = ctypes.c_void_p()
        L = _native.lib()
        check(L.f2_batch_create(plan._h, self.lengths.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), self.n_utts,
                                self.step, self.phase, int(target_items), ctypes.byref(self._h)))
        self.total_samples = int(L.f2_batch_total_samples(self._h))
        self.total_frames = int(L.f2_batch_total_frames(self._h))
        self.num_items = int(L.f2_batch_num_items(self._h))
        self.frame_offsets = np.zeros(self.n_utts + 1, dtype=np.int64)
        check(L.f2_batch_frame_offsets(self._h, self.frame_offsets.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
        self.sample_offsets = np.zeros(self.n_utts + 1, dtype=np.int64)
        np.cumsum(self.lengths, out=self.sample_offsets[1:])
        self._grid = {}
        self._grid_rows = {}

    def __del__(self):
        try:
            h = getattr(self, "_h", None)
            if h is not None and h.value:
                _native.lib().f2_batch_destroy(h)
                self._h = None
        except Exception:
            pass

    def workspace_bytes(self, want_full_gfb=False, want_full_env=False):
        return int(_native.lib().f2_batch_workspace_bytes(self._h, int(want_full_gfb), int(want_full_env)))

    def grid_windows(self, dots=11):
        """The label grid of LabelDataGenerator.py:38-50 on this batch's decimated frames: utterance
        u has nb = max(n // step - dots - 1, 0) windows, window k = frames k .. k+dots-1.  Returns the
        device int64 row offsets (n_utts+1) `run(windows=...)` wants, and the total row count."""
        key = int(dots)
        if key not in self._grid:
            nb = np.maximum(self.lengths // self.step - key - 1, 0)
            off = np.concatenate([[0], np.cumsum(nb)]).astype(np.int64)
            self._grid[key] = (torch.from_numpy(off).to(self.plan.device), int(off[-1]))
            self._grid_rows[int(self._grid[key][0].data_ptr())] = int(off[-1])
        return self._grid[key]

    def run(self, wave_dev, lpf=False, cutoff=100, gfb=None, env=None, env_t=False, dec=False, stream=None,
            out=None, fused_events=None, windows=None):
        """wave_dev: flat device tensor (int16/float32/float64) of total_samples.
        gfb/env: None or torch.float64/float32 -> (C*total_samples,) reference-layout blocks;
        env_t: time-major [total_samples, C] float32; dec: [total_frames, C] float32.
        `out` may carry preallocated tensors under the same keys.
        windows=(row_offsets_dev, dots[, out_tensor]): the fused kernel writes the (rows, dots, C)
        float32 windows itself (window k of utterance u = its decimated frames k..k+dots-1, rows
        row_offsets[u] + k); a stand-alone output mode, see grid_windows()."""
        plan = self.plan
        C = plan.n_channels
        if wave_dev.numel() != self.total_samples:
            raise ValueError("wave has %d samples, batch expects %d" % (wave_dev.numel(), self.total_samples))
        if wave_dev.device != plan.device:
            raise ValueError("wave is on %s, plan on %s" % (wave_dev.device, plan.device))
        if not wave_dev.is_contiguous() or wave_dev.dtype not in _T2F2:
            raise ValueError("wave must be a contiguous int16 / float32 / float64 tensor")
        res = {} if out is None else dict(out)
        # the C ABI takes bare pointers: whatever the caller preallocated is checked here
        want = {"gfb": (C * self.total_samples, (torch.float32, torch.float64)),
                "env": (C * self.total_samples, (torch.float32, torch.float64)),
                "env_t": (C * self.total_samples, (torch.float32,)), "dec": (C * self.total_frames, (torch.float32,))}
        for key, (numel, dts) in want.items():
            t = res.get(key)
            mapped = key == "dec" and t is not None and t.device.type == "cpu" and t.is_pinned()   # kernel stores over PCIe
            if t is not None and (t.numel() < numel or t.dtype not in dts or not t.is_contiguous() or
                                  (t.device != plan.device and not mapped)):
                raise ValueError("preallocated %r: need >= %d contiguous elements of %s on %s" % (key, numel, dts, plan.device))
        if gfb is not None and "gfb" not in res:
            res["gfb"] = torch.empty(C * self.total_samples, dtype=gfb, device=plan.device)
        if env is not None and "env" not in res:
            res["env"] = torch.empty(C * self.total_samples, dtype=env, device=plan.device)
        if env_t and "env_t" not in res:
            res["env_t"] = torch.empty((self.total_samples, C), dtype=torch.float32, device=plan.device)
        if dec and "dec" not in res:
            res["dec"] = torch.empty((self.total_frames, C), dtype=torch.float32, device=plan.device)
        a = RunArgs()
        a.wave = wave_dev.data_ptr()
        a.wave_dtype = _T2F2[wave_dev.dtype]
        a.lpf = int(bool(lpf))
        a.cutoff_hz = float(cutoff) if lpf else 0.0
        g, e = res.get("gfb"), res.get("env")
        a.gfb = g.data_ptr() if g is not None else None
        a.gfb_dtype = _T2F2[g.dtype] if g is not None else F2_F64
        a.env = e.data_ptr() if e is not None else None
        a.env_dtype = _T2F2[e.dtype] if e is not None else F2_F64
        a.env_t = res["env_t"].data_ptr() if "env_t" in res else None
        a.dec = res["dec"].data_ptr() if "dec" in res else None
        if windows is not None:
            if g is not None or e is not None or "env_t" in res or "dec" in res:
                raise ValueError("windows is a stand-alone output mode")
            offs, dots = windows[0], int(windows[1])
            if offs.dtype != torch.int64 or offs.device != plan.device or offs.numel() != len(self.lengths) + 1:
                raise ValueError("windows offsets: int64 device tensor of n_utts+1 entries")
            if len(windows) > 2 and windows[2] is not None:
                res["windows"] = windows[2]
            elif "windows" not in res:
                rows = self._grid_rows.get(int(offs.data_ptr()))
                rows = int(offs[-1].item()) if rows is None else rows
                res["windows"] = torch.empty((rows, dots, C), dtype=torch.float32, device=plan.device)
            w = res["windows"]
            if w.dtype != torch.float32 or not w.is_contiguous() or w.device != plan.device:
                raise ValueError("windows output: contiguous float32 tensor on the plan's device")
            rows = self._grid_rows.get(int(offs.data_ptr()))
            if rows is None:  # offsets that did not come from grid_windows(): one small D2H read
                rows = int(offs[-1].item())
            if w.numel() < rows * dots * C:
                raise ValueError("windows output holds %d floats, the offsets ask for %d rows x %d x %d" %
                                 (w.numel(), rows, dots, C))
            a.windows, a.win_offsets, a.win_dots = w.data_ptr(), offs.data_ptr(), dots
        if fused_events is not None:  # (DeviceEvent, DeviceEvent) around the fused kernel
            a.ev_fused_start, a.ev_fused_stop = fused_events[0].handle, fused_events[1].handle
        need = self.workspace_bytes(g is not None, e is not None and "env_t" not in res)
        ws = plan.workspace(need, stream)
        check(_native.lib().f2_batch_run(self._h, ctypes.byref(a), _ptr(ws), ws.numel(), _stream_ptr(stream)))
        return res


class DeviceEvent:
    """cudaEvent_t owned through the C ABI (recorded on the stream the kernels run on)."""

    def __init__(self):
        self.handle = ctypes.c_void_p()
        check(_native.lib().f2_event_create(ctypes.byref(self.handle)))

    def record(self, stream=None):
        check(_native.lib().f2_event_record(self.handle, _stream_ptr(stream)))

    def synchronize(self):
        check(_native.lib().f2_event_synchronize(self.handle))

    def elapsed_ms(self, stop):
        ms = ctypes.c_float()
        check(_native.lib().f2_event_elapsed_ms(self.handle, stop.handle, ctypes.byref(ms)))
        return float(ms.value)

    def __del__(self):
        try:
            if self.handle is not None and self.handle.value:
                _native.lib().f2_event_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


# ---- windowing helpers ---------------------------------------------------------------------
def gather_windows(frames_dev, base_rows_dev, dots, stride_rows=1, out=None, stream=None):
    """out[w, j, :] = frames[base_rows[w] + j*stride_rows, :]  (InputGenerator.py:73-80)."""
    n, C = int(base_rows_dev.numel()), int(frames_dev.shape[1])
    if out is None:
        out = torch.empty((n, dots, C), dtype=torch.float32, device=frames_dev.device)
    check(_native.lib().f2_gather_windows(_ptr(frames_dev), C, _ptr(base_rows_dev), n, int(dots), int(stride_rows),
                                          _ptr(out), _stream_ptr(stream)))
    return out


def gather_index(src_dev, idx_dev, out=None, stream=None):
    n, C = int(idx_dev.numel()), int(src_dev.shape[1])
    if out is None:
        out = torch.empty((n, C), dtype=torch.float32, device=src_dev.device)
    check(_native.lib().f2_gather_index(_ptr(src_dev), C, _ptr(idx_dev), n, _ptr(out), _stream_ptr(stream)))
    return out


def gather_windows_cn(env_dev, idx_dev, out=None, stream=None):
    """out[i, :] = float32(env[:, idx[i]]) for a (C, n) float64/float32 device matrix."""
    C, n = int(env_dev.shape[0]), int(env_dev.shape[1])
    m = int(idx_dev.numel())
    if out is None:
        out = torch.empty((m, C), dtype=torch.float32, device=env_dev.device)
    check(_native.lib().f2_gather_windows_cn(_ptr(env_dev), _T2F2[env_dev.dtype], C, n, _ptr(idx_dev), m, _ptr(out),
                                             _stream_ptr(stream)))
    return out


def dense_frames(env_t_dev, dots, step, i0, i1, normalize=False, out_dtype=torch.float64, stream=None):
    """Frames i0..i1 of Evaluating.py:70-78 (+ Training.normalizeInput when normalize)."""
    C = int(env_t_dev.shape[1])
    out = torch.empty((max(i1 - i0, 0), dots, C), dtype=out_dtype, device=env_t_dev.device)
    flag = torch.zeros(1, dtype=torch.int32, device=env_t_dev.device)
    if not env_t_dev.is_contiguous() or env_t_dev.dtype != torch.float32:
        raise ValueError("dense_frames wants a contiguous float32 [rows, C] envelope")
    check(_native.lib().f2_dense_frames(_ptr(env_t_dev), int(env_t_dev.shape[0]), C, int(dots), int(step), int(i0), int(i1),
                                        int(bool(normalize)), _ptr(out), _T2F2[out_dtype], _ptr(flag),
                                        _stream_ptr(stream)))
    return out, flag


def label_fit(formant_dev, first_dev, center_dev, dots, step, stream=None):
    """(slope, intercept, r, p) per timepoint: LabelDataGenerator.py:60-68 for every item at once.
    formant_dev float64, first_dev int64, center_dev int32 device tensors; returns (N, 4) float64."""
    if formant_dev.dtype != torch.float64 or first_dev.dtype != torch.int64 or center_dev.dtype != torch.int32:
        raise TypeError("label_fit wants float64 formants, int64 first indices, int32 centers")
    n = int(first_dev.shape[0])
    if int(center_dev.shape[0]) != n:
        raise ValueError("first and center differ in length")
    out = torch.empty((n, 4), dtype=torch.float64, device=formant_dev.device)
    check(_native.lib().f2_label_fit(_ptr(formant_dev), _ptr(first_dev), _ptr(center_dev), n, int(dots), int(step),
                                     _ptr(out), _stream_ptr(stream)))
    return out


def shard_utterances(lengths, world):
    """Length-sorted round-robin deal of utterances over `world` devices (SURVEY.md section 8e; the
    reference's unit of parallelism is the file, GammatoneFiltering.py:121-125): sort by length,
    longest first, and deal like cards, so that every shard sees the same length distribution and
    sum(n_u) differs by at most one utterance.  Returns `world` ascending index arrays."""
    lengths = np.asarray(lengths, dtype=np.int64).reshape(-1)
    world = max(1, int(world))
    order = np.argsort(-lengths, kind="stable")
    return [np.sort(order[r::world]) for r in range(world)]


def host_cores():
    """Cores this process may run on (cgroup / affinity aware)."""
    import os
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


class _PinnedBlock:
    """Page-locked, kernel-addressable host memory: a huge-page advised mapping registered with CUDA
    (f2_host_alloc + f2_host_pin) -- 0.17 s for the 0.71 GB frames buffer of the corpus where
    torch.empty(pin_memory=True) (cudaHostAlloc) takes 0.6 s of the first call."""

    def __init__(self, nbytes):
        self.nbytes = max(int(nbytes), 4096)
        self.ptr = ctypes.c_void_p()
        check(_native.lib().f2_host_alloc(self.nbytes, ctypes.byref(self.ptr)))
        rc = _native.lib().f2_host_pin(self.ptr, self.nbytes)
        if rc != 0:
            _native.lib().f2_host_free(self.ptr, self.nbytes)
            self.ptr = None
            check(rc)

    def __del__(self):
        try:
            if self.ptr is not None and self.ptr.value:
                L = _native.lib()
                L.f2_host_unpin(self.ptr)
                L.f2_host_free(self.ptr, self.nbytes)
                self.ptr = None
        except Exception:
            pass


def _pinned_empty(n, dtype):
    """Flat pinned host tensor of n elements; falls back to torch's pinned allocator where registering
    fails (memlock limits, exotic platforms)."""
    n = max(int(n), 1)
    esz = torch.empty(0, dtype=dtype).element_size()
    try:
        block = _PinnedBlock(n * esz)
    except Exception:
        return torch.empty(n, dtype=dtype, pin_memory=True)
    buf = (ctypes.c_char * (n * esz)).from_address(block.ptr.value)
    buf._f2_block = block   # the registration lives as long as the ctypes view numpy (and the tensor) hold on to
    np_dt = torch.empty(0, dtype=dtype).numpy().dtype
    return torch.from_numpy(np.frombuffer(buf, dtype=np_dt, count=n))


class WindowPipeline:
    """Host waves in, host (N, 2R+1, C) float32 windows out, for a whole corpus (or one shard of it).

    The input tensor of the reference is (2R+1)x redundant -- row k of an utterance is 2R+1
    consecutive decimated frames -- so the DECIMATED FRAMES travel over PCIe (0.68 GB for the
    4620-utterance corpus instead of 7.5 GB) and the rows are placed on the host by the worker pool
    of f2_host.cpp.  The utterances are cut into sub-batches: the waves of all of them are queued
    on an upload stream at the start, sub-batch i is filtered on a compute stream, and the fused
    kernel stores its decimated frames STRAIGHT INTO THE PINNED HOST BUFFER (posted PCIe writes
    spread over the kernel's run time: 16 GB/s on average; a device buffer plus one D2H copy per
    sub-batch arrives in bursts that fight the placement threads for the host's DRAM and was 3 ms
    slower per corpus -- `zero_copy = False` / F2CNN_B200_ZERO_COPY_FRAMES=0 brings it back).  The
    end of each sub-batch's kernels is followed, in stream order, by the host placement of its rows
    (cudaLaunchHostFunc -> thread pool), so the host never waits between sub-batches.  Consecutive sub-batches run on two alternating compute
    streams (each with its own ring workspace), so the tail of one launch overlaps the head of the
    next.

    lengths[u]: samples of utterance u; src_offsets[u]: where it starts in the host buffer passed
    to run() (default: back to back), so a shard can read its utterances out of the buffer that
    holds the whole corpus.  Frames are numbered over the pipeline's utterances in order
    (`frame_offsets`), which is what engine.window_runs wants."""

    def __init__(self, plan, lengths, dots=11, step=160, phase=0, lpf=True, cutoff=50, n_sub=None, src_offsets=None,
                 placer=None):
        self.plan, self.dots, self.lpf, self.cutoff = plan, int(dots), bool(lpf), cutoff
        self.step, self.phase = int(step), int(phase)
        lengths = np.ascontiguousarray(lengths, dtype=np.int64).reshape(-1)
        self.lengths = lengths
        U = int(lengths.shape[0])
        cum = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        self.src_offsets = cum[:-1].copy() if src_offsets is None else np.ascontiguousarray(src_offsets, dtype=np.int64)
        if self.src_offsets.shape[0] != U:
            raise ValueError("src_offsets: one entry per utterance")
        self.src_extent = int((self.src_offsets + lengths).max()) if U else 0
        n_dec = np.where(lengths > self.phase, (lengths - self.phase + self.step - 1) // self.step, 0)
        self.frame_offsets = np.concatenate([[0], np.cumsum(n_dec)]).astype(np.int64)
        self.total_frames = int(self.frame_offsets[-1])
        self.total_samples = int(cum[-1])
        # sub-batches of total/n_sub samples, except that the first few grow from an eighth of that (nothing
        # can be placed before the first sub-batch is uploaded, filtered and downloaded) and the last few
        # shrink to a quarter (the rows of the last sub-batch are placed after the GPU has gone idle)
        if n_sub is None and os.environ.get("F2CNN_B200_NSUB"):
            n_sub = int(os.environ["F2CNN_B200_NSUB"])   # development knob
        if n_sub is None:
            # a sub-batch should still fill the device: 592 utterances x 4 channel groups = one wave of CTAs
            n_sub = min(U // 576, 8)
        n_sub = max(1, min(int(n_sub), 32, max(U, 1)))
        per_sub = cum[-1] / n_sub
        head, size, at = [], per_sub / 8, 0.0
        ramp = os.environ.get("F2CNN_B200_RAMP")   # development knob: head sub-batches as fractions 1/d of the corpus
        if ramp:
            for d in ramp.split(","):
                at += cum[-1] / float(d)
                head.append(at)
            size = per_sub
        while size < per_sub and at + size < cum[-1] / 2:
            at += size
            head.append(at)
            size *= 2
        tail, size, back = [], per_sub / 4, float(cum[-1])
        while size < per_sub and back - size > cum[-1] / 2:
            back -= size
            tail.append(back)
            size *= 2
        body = []
        if back - at > per_sub:
            k = max(1, int(round((back - at) / per_sub)))
            body = [at + (back - at) * j / k for j in range(1, k)]
        marks = head + body + tail[::-1]
        cuts = sorted(set([0] + [int(np.searchsorted(cum, m)) for m in marks] + [U]))
        dev = plan.device
        C = plan.n_channels
        self.subs = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b <= a:
                continue
            # whole utterances only (target_items=1): same arithmetic as one big batch, bit for bit
            batch = plan.batch(lengths[a:b], step=self.step, phase=self.phase, target_items=1)
            assert batch.total_frames == int(self.frame_offsets[b] - self.frame_offsets[a])
            # contiguous source spans of this sub-batch (adjacent utterances merge into one copy)
            so, ln = self.src_offsets[a:b], lengths[a:b]
            brk = np.flatnonzero(so[1:] != so[:-1] + ln[:-1]) + 1
            first = np.concatenate([[0], brk])
            last = np.concatenate([brk, [b - a]])
            spans = (so[first].copy(), (cum[a:b][first]).copy(), (cum[a:b][last - 1] + ln[last - 1] - cum[a:b][first]).copy())
            self.subs.append(dict(batch=batch, u0=a, u1=b, s0=int(cum[a]), s1=int(cum[b]), spans=spans,
                                  f0=int(self.frame_offsets[a]), f1=int(self.frame_offsets[b])))
        self._wave_dev = None
        self._stage = None      # pinned staging for pageable input
        with torch.cuda.device(dev):
            self._dec_dev = None    # only the copy mode (zero_copy = False) needs a device-side frames buffer
            self._dec_host = _pinned_empty(max(self.total_frames, 1) * C, torch.float32).view(-1, C)
            self._s_in, self._s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
            # consecutive sub-batches alternate between two compute streams: a launch ends with a tail
            # of its longest utterances on half-empty SMs, and the next launch's CTAs fill them
            self._s_comp = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]
            self._ev_in = [torch.cuda.Event(enable_timing=True) for _ in self.subs]
            self._ev_done = [torch.cuda.Event(enable_timing=True) for _ in self.subs]
            self._ev_out = [torch.cuda.Event(enable_timing=True) for _ in self.subs]
            self._ev_start = torch.cuda.Event(enable_timing=True)
            self._ev_end = torch.cuda.Event(blocking=True)
        # True: the fused kernel stores the decimated frames straight into the pinned host buffer (posted PCIe
        # writes spread over the kernel's run time) instead of a device buffer + one D2H copy per sub-batch
        self.zero_copy = os.environ.get("F2CNN_B200_ZERO_COPY_FRAMES", "1") == "1"
        self.timing = False     # True: run() synchronises first and keeps a timeline (see timeline())
        self._t0 = None
        self.placer = placer if placer is not None else Placer()

    # -- uploads -------------------------------------------------------------------------------
    def _upload(self, sub, wave_host, esize):
        src, dst, cnt = sub["spans"]
        L = _native.lib()
        check(L.f2_upload_spans(_ptr(self._wave_dev), ctypes.c_void_p(wave_host.data_ptr()),
                                (src * esize).ctypes.data_as(ctypes.c_void_p), (dst * esize).ctypes.data_as(ctypes.c_void_p),
                                (cnt * esize).ctypes.data_as(ctypes.c_void_p), int(src.shape[0]),
                                ctypes.c_void_p(self._s_in.cuda_stream)))

    def _split_runs(self, runs):
        """runs (global frame numbering) -> one array per sub-batch."""
        runs = np.ascontiguousarray(runs, dtype=np.int64).reshape(-1, 3)
        bounds = np.asarray([s["f1"] for s in self.subs], dtype=np.int64)
        which = np.searchsorted(bounds, runs[:, 0], side="right")
        if runs.shape[0] and np.all(which[1:] >= which[:-1]):
            edges = np.searchsorted(which, np.arange(len(self.subs) + 1))
            return [runs[edges[i]:edges[i + 1]] for i in range(len(self.subs))]
        order = np.argsort(which, kind="stable")
        runs, which = runs[order], which[order]
        edges = np.searchsorted(which, np.arange(len(self.subs) + 1))
        return [np.ascontiguousarray(runs[edges[i]:edges[i + 1]]) for i in range(len(self.subs))]

    def run(self, wave_host, runs, out_host, keep_frames=False):
        """wave_host: flat host tensor (int16 / float32 / float64; pinned for full speed -- pageable
        input is staged through a pinned buffer sub-batch by sub-batch) or a list of per-utterance
        numpy arrays; runs: (n, 3) int64 from engine.window_runs on this pipeline's frame_offsets;
        out_host: the (N, dots, C) float32 host array or tensor the rows go to (any host memory).
        Returns when every row has been placed."""
        # no garbage-collector pause while the launch sequence is being queued: a generation-0/1 sweep of a
        # torch process takes ~5 ms, and when it hit between the kernel launches and the placement submits one
        # call in six finished 4 ms late (tools/e2e_hiccup.py); collection resumes while this thread waits
        import gc
        gc_was_on = gc.isenabled()
        gc.disable()
        try:
            return self._run(wave_host, runs, out_host, keep_frames, gc_was_on)
        finally:
            if gc_was_on:
                gc.enable()

    def _run(self, wave_host, runs, out_host, keep_frames, gc_was_on):
        caller = torch.cuda.current_stream(self.plan.device)
        dev = self.plan.device
        C = self.plan.n_channels
        listed = isinstance(wave_host, (list, tuple))
        if listed:
            dt = torch.from_numpy(wave_host[0][:0]).dtype if len(wave_host) else torch.int16
            pinned = False
        else:
            if not torch.is_tensor(wave_host):
                wave_host = torch.from_numpy(wave_host)
            if wave_host.dim() != 1 or wave_host.numel() < self.src_extent:
                raise ValueError("wave buffer holds %d samples, the pipeline reads up to %d" % (wave_host.numel(), self.src_extent))
            dt = wave_host.dtype
            pinned = wave_host.is_pinned()
        if dt not in _T2F2:
            raise TypeError("waves must be int16, float32 or float64")
        if self._wave_dev is None or self._wave_dev.dtype != dt:
            self._wave_dev = torch.empty(max(self.total_samples, 1), dtype=dt, device=dev)
        if not pinned and (self._stage is None or self._stage.dtype != dt):
            self._stage = _pinned_empty(self.total_samples, dt)
        out_flat = out_host
        esize = self._wave_dev.element_size()
        if self.timing:
            import time
            torch.cuda.synchronize(dev)
            self.placer.trace(clear=True)
            self._t0 = time.monotonic()
            self._ev_start.record(caller)
        for s_ in (self._s_in, self._s_out, self._s_comp[0], self._s_comp[1]):
            s_.wait_stream(caller)
        if pinned:
            # all uploads are queued at once (444 MB for the corpus): over after the first few ms
            for i, sub in enumerate(self.subs):
                self._upload(sub, wave_host, esize)
                self._ev_in[i].record(self._s_in)
        for i, sub in enumerate(self.subs):
            if not pinned:
                # pageable input: this sub-batch's samples -> pinned staging -> device, while the
                # previous sub-batches are being filtered
                stage = self._stage[sub["s0"]:sub["s1"]].numpy()
                if listed:
                    np.concatenate([np.asarray(w).reshape(-1) for w in wave_host[sub["u0"]:sub["u1"]]], out=stage)
                else:
                    src, dst, cnt = sub["spans"]
                    host_np = wave_host.numpy()
                    for so, do, n in zip(src, dst, cnt):
                        stage[do - sub["s0"]:do - sub["s0"] + n] = host_np[so:so + n]
                with torch.cuda.stream(self._s_in):
                    self._wave_dev[sub["s0"]:sub["s1"]].copy_(self._stage[sub["s0"]:sub["s1"]], non_blocking=True)
                    self._ev_in[i].record(self._s_in)
            comp = self._s_comp[i & 1]
            comp.wait_event(self._ev_in[i])
            if not self.zero_copy and self._dec_dev is None:
                self._dec_dev = torch.empty((max(self.total_frames, 1), C), dtype=torch.float32, device=dev)
            dec = (self._dec_host if self.zero_copy else self._dec_dev)[sub["f0"]:sub["f1"]]
            sub["batch"].run(self._wave_dev[sub["s0"]:sub["s1"]], lpf=self.lpf, cutoff=self.cutoff, out={"dec": dec},
                             stream=comp)
            self._ev_done[i].record(comp)
        # Uploads and kernels of every sub-batch are queued; only now is the placement plan needed.  `runs`
        # may be a callable: the run detection of a corpus (a few ms on the host) then happens while the
        # first sub-batch is already being filtered.
        if callable(runs):
            runs = runs()
        per_sub = self._split_runs(runs)
        with torch.cuda.stream(self._s_out):
            for i, sub in enumerate(self.subs):
                self._s_out.wait_event(self._ev_done[i])
                if sub["f1"] > sub["f0"] and not self.zero_copy:
                    self._dec_host[sub["f0"]:sub["f1"]].copy_(self._dec_dev[sub["f0"]:sub["f1"]], non_blocking=True)
                self._ev_out[i].record(self._s_out)
                if per_sub[i].shape[0]:
                    self.placer.submit(self._dec_host, per_sub[i], out_flat, dots=self.dots, stream=self._s_out)
            self._ev_end.record(self._s_out)
        for s_ in (self._s_out, self._s_comp[0], self._s_comp[1]):
            caller.wait_stream(s_)
        if gc_was_on:
            import gc
            gc.enable()                 # everything is queued: a sweep now costs nothing
        self._ev_end.synchronize()      # blocking event: the waiting thread sleeps, its core places rows
        self._s_out.synchronize()
        self.placer.wait()
        return out_host

    def timeline(self):
        """After a run() with timing = True: per sub-batch, milliseconds since the start of the run at
        which its waves were on the device, its kernels had finished, its frames were on the host (CUDA
        events), and at which its rows became runnable / were placed (host clock of the worker pool)."""
        torch.cuda.synchronize(self.plan.device)
        trace = self.placer.trace(clear=True)
        rows = []
        for i, sub in enumerate(self.subs):
            rows.append(dict(utterances=sub["u1"] - sub["u0"], h2d=self._ev_start.elapsed_time(self._ev_in[i]),
                             kernels=self._ev_start.elapsed_time(self._ev_done[i]),
                             d2h=self._ev_start.elapsed_time(self._ev_out[i])))
        jobs = [dict(runnable=(t[1] - self._t0) * 1e3, placed=(t[2] - self._t0) * 1e3, rows=int(t[3])) for t in trace]
        return rows, jobs

    @property
    def frames_host(self):
        """The decimated frames of the last run ([total_frames, C] float32, pinned host memory)."""
        return self._dec_host[:self.total_frames]


class MultiGpuWindowPipeline:
    """WindowPipeline over several GPUs of one box from ONE process: the utterances are dealt to
    the devices by shard_utterances (length-sorted round-robin), every device runs its own
    WindowPipeline over its shard, reading its utterances out of the one host wave buffer and
    placing its rows at their final offsets in the one host output.  Utterances are independent,
    so there is no collective -- the "gather" is each device's frames landing on the host and
    being placed (SURVEY.md section 8e).  One host thread drives all devices; the placement pool is
    shared."""

    def __init__(self, coefs, lengths, devices=None, **kw):
        lengths = np.ascontiguousarray(lengths, dtype=np.int64).reshape(-1)
        if devices is None:
            devices = list(range(torch.cuda.device_count()))
        devices = list(devices)[:max(1, min(len(devices), max(len(lengths), 1)))]
        self.lengths = lengths
        cum = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        self.placer = kw.pop("placer", None) or Placer()
        self.parts = []
        for d, idx in zip(devices, shard_utterances(lengths, len(devices))):
            with torch.cuda.device(d):
                pipe = WindowPipeline(plan_for(coefs, d), lengths[idx], src_offsets=cum[idx], placer=self.placer, **kw)
            self.parts.append(dict(device=d, utts=idx, pipe=pipe))

    def window_runs(self, centers, counts, radius=5):
        """Per-device runs for centres given in corpus order (rows in corpus order)."""
        counts = np.asarray(counts, dtype=np.int64)
        centers = np.asarray(centers, dtype=np.int64)
        cpos = np.concatenate([[0], np.cumsum(counts)])
        out = []
        for part in self.parts:
            idx, pipe = part["utts"], part["pipe"]
            cen = np.concatenate([centers[cpos[u]:cpos[u + 1]] for u in idx] + [np.zeros(0, np.int64)])
            runs, phase, _ = window_runs(cen, counts[idx], self.lengths[idx], pipe.frame_offsets, radius, pipe.step,
                                         pipe.phase, row_offsets=cpos[idx])
            if runs is None or phase != pipe.phase:
                raise ValueError("timepoints are not windows of consecutive frames of the pipeline's grid")
            out.append(runs)
        return out

    def run(self, wave_host, runs_per_part, out_host):
        import concurrent.futures as cf
        # every device needs its own driving thread only for the final wait; launches are asynchronous
        def drive(part, runs):
            with torch.cuda.device(part["device"]):
                part["pipe"].run(wave_host, runs, out_host)
        with cf.ThreadPoolExecutor(max_workers=len(self.parts)) as pool:
            list(pool.map(drive, self.parts, runs_per_part))
        return out_host


# ---- plan cache for the numpy-in / numpy-out drop-in functions -----------------------------
_plans = {}
_plans_lock = threading.Lock()


def plan_for(coefs, device=None):
    """One shared, immutable plan per (coefficient matrix, device, float64 sections setting): the setting is
    F2CNN_B200_FLOAT64_SECTIONS at the time of the call (Plan)."""
    _require_cuda()
    coefs = np.ascontiguousarray(coefs, dtype=np.float64)
    dev = torch.cuda.current_device() if device is None else int(device)
    f64 = float64_sections_default()
    key = (hashlib.sha1(coefs.tobytes()).hexdigest(), coefs.shape, dev, f64)
    with _plans_lock:
        p = _plans.get(key)
        if p is None:
            p = Plan(coefs, dev, float64_sections=f64)
            p._frozen = True
            _plans[key] = p
        return p


_generic_plan = {}


def any_plan(device=None):
    """A plan is only a device handle for the filterbank-independent entry points."""
    dev = torch.cuda.current_device() if device is None else int(device)
    with _plans_lock:
        for (k, shape, d, f64), p in _plans.items():
            if d == dev:
                return p
    from .gammatone import filters
    return plan_for(filters.make_erb_filters(16000, filters.centre_freqs(16000, 4, 100)), dev)


# ---- host side of the window stage (f2_host.cpp; HOST memory, no device needed) ----------------
def window_runs(centers, counts, lengths, frame_offsets, radius=5, step=160, phase=-1, row_offsets=None):
    """Label timepoints -> runs of consecutive windows on the decimated grid (f2_window_runs).

    centers: int64 window centres of all utterances back to back; counts[u] of them belong to
    utterance u (InputGenerator.py:73-80 output order).  Returns (runs, phase, n_rows): runs is an
    (n, 3) int64 array of (first_frame, row0, count), or None when the timepoints are legal but not
    windows of consecutive frames of one grid.  Raises IndexError where the reference would."""
    centers = np.ascontiguousarray(centers, dtype=np.int64).reshape(-1)
    counts = np.ascontiguousarray(counts, dtype=np.int64).reshape(-1)
    lengths = np.ascontiguousarray(lengths, dtype=np.int64).reshape(-1)
    frame_offsets = np.ascontiguousarray(frame_offsets, dtype=np.int64).reshape(-1)
    n_utts = int(counts.shape[0])
    if lengths.shape[0] != n_utts or frame_offsets.shape[0] < n_utts or int(counts.sum()) != centers.shape[0]:
        raise ValueError("window_runs: counts / lengths / frame_offsets / centers do not fit together")
    rows = None
    if row_offsets is not None:
        rows = np.ascontiguousarray(row_offsets, dtype=np.int64).reshape(-1)
        if rows.shape[0] < n_utts:
            raise ValueError("window_runs: row_offsets shorter than the utterance list")
    L = _native.lib()
    ph = ctypes.c_int(int(phase))
    n_runs, n_rows = ctypes.c_int64(), ctypes.c_int64()
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p) if a is not None and a.size else None

    def call(buf, room):
        ph.value = int(phase)
        rc = L.f2_window_runs(p(centers), p(counts), p(lengths), p(frame_offsets), p(rows), n_utts, int(radius),
                              int(step), ctypes.byref(ph), p(buf), room, ctypes.byref(n_runs), ctypes.byref(n_rows))
        if rc == _native.F2_ERR_INDEX:
            raise IndexError(L.f2_last_error().decode("utf-8", "replace"))
        check(rc)

    # one pass when the guess holds (a label grid is one run per utterance); the count comes back either way
    room = int(min(max(centers.shape[0], 1), max(4 * n_utts, 1024)))
    runs = np.empty((room, 3), dtype=np.int64)
    try:
        call(runs, room)
    except _native.F2Error as e:
        if e.code != _native.F2_ERR_WORKSPACE:
            raise
        runs = np.empty((max(n_runs.value, 1), 3), dtype=np.int64)
        call(runs, n_runs.value)
    if n_runs.value < 0:
        return None, ph.value, n_rows.value
    return runs[:n_runs.value], ph.value, n_rows.value


def _host_ptr(a):
    if torch.is_tensor(a):
        if a.device.type != "cpu" or not a.is_contiguous():
            raise ValueError("host placement wants contiguous CPU tensors")
        return ctypes.c_void_p(a.data_ptr())
    if not a.flags["C_CONTIGUOUS"]:
        raise ValueError("host placement wants C-contiguous arrays")
    return a.ctypes.data_as(ctypes.c_void_p)


def _check_placement(frames, runs, out, dots):
    C = int(frames.shape[-1])
    if str(frames.dtype).split(".")[-1] != "float32" or str(out.dtype).split(".")[-1] != "float32":
        raise TypeError("host placement copies float32 frames into float32 rows")
    runs = np.ascontiguousarray(runs, dtype=np.int64).reshape(-1, 3)
    if runs.shape[0]:
        n_frames = int(np.prod(frames.shape[:-1]))
        n_rows = int(np.prod(out.shape)) // (int(dots) * C)
        live = runs[runs[:, 2] > 0]
        if live.shape[0] and (live.min() < 0 or int((live[:, 0] + live[:, 2]).max()) + int(dots) - 1 > n_frames or
                              int((live[:, 1] + live[:, 2]).max()) > n_rows):
            raise IndexError("a window run leaves the frame matrix or the output tensor")
    return runs, C


def place_windows(frames, runs, out, dots=11, threads=0):
    """out[row0+i, j, :] = frames[first_frame+i+j, :] for every run (f2_place_windows): the rows of
    InputGenerator.py:73-80 from decimated frames, one contiguous copy per row.  Host arrays."""
    runs, C = _check_placement(frames, runs, out, dots)
    check(_native.lib().f2_place_windows(_host_ptr(frames), C, int(dots), runs.ctypes.data_as(ctypes.c_void_p),
                                         int(runs.shape[0]), _host_ptr(out), int(threads)))
    return out


class Placer:
    """Persistent host worker pool that places window rows in CUDA stream order (f2_placer_*)."""

    def __init__(self, threads=0):
        self._h = ctypes.c_void_p()
        check(_native.lib().f2_placer_create(int(threads), ctypes.byref(self._h)))
        self.threads = int(_native.lib().f2_placer_threads(self._h))
        self._keep = []

    def submit(self, frames, runs, out, dots=11, stream=None, after_stream=True):
        """Queue a placement; with after_stream it starts once everything queued on `stream` (default:
        the current stream) so far -- the D2H copy of `frames` -- has completed."""
        runs, C = _check_placement(frames, runs, out, dots)
        self._keep.append((frames, out))  # keep the buffers alive until wait()
        sp = _stream_ptr(stream) if after_stream else ctypes.c_void_p(0)
        check(_native.lib().f2_placer_submit(self._h, int(bool(after_stream)), sp, _host_ptr(frames), C, int(dots),
                                             runs.ctypes.data_as(ctypes.c_void_p), int(runs.shape[0]), _host_ptr(out)))

    def wait(self):
        check(_native.lib().f2_placer_wait(self._h))
        self._keep.clear()

    def trace(self, clear=True):
        """(jobs, 4) float64: submit, runnable, done (CLOCK_MONOTONIC seconds), rows -- per finished job."""
        L = _native.lib()
        n = int(L.f2_placer_trace(self._h, None, 0, 0))
        buf = np.zeros((max(n, 1), 4), dtype=np.float64)
        n = int(L.f2_placer_trace(self._h, buf.ctypes.data_as(ctypes.c_void_p), n, int(bool(clear))))
        return buf[:n]

    def __del__(self):
        try:
            h = getattr(self, "_h", None)
            if h is not None and h.value:
                _native.lib().f2_placer_destroy(h)
                self._h = None
        except Exception:
            pass


_host_pool = []            # [(address, nbytes)]: freed corpus-sized blocks waiting for the next request
_host_pool_lock = threading.Lock()
_HOST_POOL_MIN = 64 << 20  # smaller blocks are not worth keeping
_HOST_POOL_MAX_BLOCKS = 1


class _HostBlock:
    """Lease on a huge-page advised anonymous mapping (f2_host_alloc).  When the numpy array built on it
    is garbage collected, a corpus-sized block goes back to a one-entry pool instead of to the kernel:
    the next request of about that size -- the same call again -- gets memory whose pages are already
    there (a fresh 7.5 GB mapping costs ~0.1 s of page faults even with huge pages)."""

    def __init__(self, nbytes):
        want = max(int(nbytes), 1)
        self.ptr = None
        with _host_pool_lock:
            for i, (addr, size) in enumerate(_host_pool):
                if want <= size <= want + (want >> 2):
                    self.ptr, self.nbytes = ctypes.c_void_p(addr), size
                    del _host_pool[i]
                    break
        if self.ptr is None:
            self.nbytes = want
            self.ptr = ctypes.c_void_p()
            check(_native.lib().f2_host_alloc(self.nbytes, ctypes.byref(self.ptr)))

    def __del__(self):
        try:
            if self.ptr is None or not self.ptr.value:
                return
            addr, self.ptr = self.ptr.value, None
            with _host_pool_lock:
                if self.nbytes >= _HOST_POOL_MIN and len(_host_pool) < _HOST_POOL_MAX_BLOCKS:
                    _host_pool.append((addr, self.nbytes))
                    return
            _native.lib().f2_host_free(ctypes.c_void_p(addr), self.nbytes)
        except Exception:
            pass


def release_host_pool():
    """Give the pooled output blocks back to the operating system."""
    with _host_pool_lock:
        blocks, _host_pool[:] = list(_host_pool), []
    for addr, size in blocks:
        _native.lib().f2_host_free(ctypes.c_void_p(addr), size)


def host_empty(shape, dtype=np.float32):
    """Uninitialised numpy array on huge-page advised anonymous memory (f2_host_alloc): the fresh
    output tensor of a corpus-sized request without two million 4 KiB page faults."""
    shape = tuple(int(s) for s in shape)
    dt = np.dtype(dtype)
    nbytes = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
    block = _HostBlock(nbytes)
    buf = (ctypes.c_char * max(nbytes, 1)).from_address(block.ptr.value)
    buf._f2_block = block  # the mapping lives as long as the ctypes view numpy holds on to
    return np.frombuffer(buf, dtype=dt, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)
