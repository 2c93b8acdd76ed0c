"""Forward pass of the reference's F2-direction CNN (scripts/CNN/Training.py:93-114) in PyTorch,
for the `cnn eval*` path: Conv32 3x3 same -> Conv32 3x3 -> MaxPool2 -> Conv64 3x3 same ->
Conv64 3x3 -> MaxPool2 -> Flatten(1920) -> Dense516 -> Dense2 softmax, ReLU after every conv /
the first dense, dropout inactive at inference.

Two implementations of the same network:
  * TensorCoreCNN -- the product path of `cnn eval*`: hand-written tcgen05 kernels in
    libf2cnn_b200.so (csrc/f2_cnn.cu: implicit-GEMM convolutions with the accumulators in tensor
    memory, bf16 operands, float32 accumulation), fed straight from the time-major envelope.
  * F2CNN -- a plain PyTorch module (float32 through cuDNN).  It is the ORACLE the kernels are tested
    against (there is no Keras here and no trained model ships with the reference) and the carrier of
    the parameters: weights are seeded (benchmarks, tests) or loaded from arrays in Keras layout with
    `load_keras_arrays`."""
import ctypes

import numpy as np
import torch
import torch.nn.functional as F

from . import _native
from ._native import check


class F2CNN(torch.nn.Module):
    def __init__(self, dots=11, channels=128, num_classes=2):
        super().__init__()
        self.c1 = torch.nn.Conv2d(1, 32, 3, padding=1)
        self.c2 = torch.nn.Conv2d(32, 32, 3)
        self.c3 = torch.nn.Conv2d(32, 64, 3, padding=1)
        self.c4 = torch.nn.Conv2d(64, 64, 3)
        h = ((dots - 2) // 2 - 2) // 2
        w = ((channels - 2) // 2 - 2) // 2
        self.flat = 64 * h * w  # 1920 for 11 x 128
        self.d1 = torch.nn.Linear(self.flat, 516)
        self.d2 = torch.nn.Linear(516, num_classes)

    def forward(self, frames):
        """frames: (N, dots, channels) -> (N, num_classes) softmax scores [falling, rising]."""
        x = frames.unsqueeze(1)
        x = F.relu(self.c1(x))
        x = F.max_pool2d(F.relu(self.c2(x)), 2)
        x = F.relu(self.c3(x))
        x = F.max_pool2d(F.relu(self.c4(x)), 2)
        # Keras flattens channels-last (H, W, C); keep that order so Keras dense weights fit
        x = x.permute(0, 2, 3, 1).reshape(x.shape[0], -1)
        x = F.relu(self.d1(x))
        return F.softmax(self.d2(x), dim=1)

    @torch.no_grad()
    def load_keras_arrays(self, arrays):
        """arrays: [k1, b1, ..., k4, b4, W1, c1, W2, c2] in Keras layout (conv kernels HWIO,
        dense kernels (in, out))."""
        convs = [self.c1, self.c2, self.c3, self.c4]
        for i, conv in enumerate(convs):
            conv.weight.copy_(torch.as_tensor(arrays[2 * i]).permute(3, 2, 0, 1))
            conv.bias.copy_(torch.as_tensor(arrays[2 * i + 1]))
        for j, lin in enumerate([self.d1, self.d2]):
            lin.weight.copy_(torch.as_tensor(arrays[8 + 2 * j]).t())
            lin.bias.copy_(torch.as_tensor(arrays[9 + 2 * j]))


def seeded_model(seed=0, dots=11, channels=128, device="cuda", dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    m = F2CNN(dots, channels)
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * (0.05 if p.dim() > 1 else 0.01))
    return m.to(device=device, dtype=dtype).eval()


@torch.no_grad()
def predict(model, frames_dev, batch=8192, autocast_dtype=None, channels_last=False):
    """Scores for all frames, in batches (46 240 frames per 3 s utterance).  autocast_dtype =
    torch.bfloat16 runs the convolutions and dense layers on the tensor cores in bf16 (inputs are
    normalised to [0, 1], scores differ by ~1e-2); None keeps the parameters' precision.
    channels_last=True lays the convolution weights and activations out NHWC, the layout cuDNN's
    tensor-core kernels want (57 ms fp32 -> 49 ms bf16 -> 33 ms bf16 NHWC per 3 s utterance); it
    converts the module's parameters in place, the results do not depend on it."""
    out = []
    if channels_last:
        model.to(memory_format=torch.channels_last)
    dt = next(model.parameters()).dtype
    for i in range(0, frames_dev.shape[0], batch):
        x = frames_dev[i:i + batch].to(dt)
        if autocast_dtype is not None:
            with torch.autocast("cuda", dtype=autocast_dtype):
                y = model(x)
            out.append(y.float())
        else:
            out.append(model(x))
    return torch.cat(out) if out else torch.zeros((0, 2), device=frames_dev.device)


class TensorCoreCNN:
    """The network on the 5th-generation tensor cores (f2_cnn_* of the C ABI).  `source`: an F2CNN
    module or the 12 arrays of Keras' model.get_weights() (conv kernels HWIO, dense kernels (in, out))."""

    def __init__(self, source, device=None, dots=11, channels=128):
        if not torch.cuda.is_available():
            raise RuntimeError("TensorCoreCNN needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        arrays = keras_arrays(source) if isinstance(source, torch.nn.Module) else list(source)
        if len(arrays) != 12:
            raise ValueError("expected the 12 parameter arrays of the reference network, got %d" % len(arrays))
        shapes = [(3, 3, 1, 32), (32,), (3, 3, 32, 32), (32,), (3, 3, 32, 64), (64,), (3, 3, 64, 64), (64,),
                  (1920, 516), (516,), (516, 2), (2,)]
        host = []
        for a, shp in zip(arrays, shapes):
            a = np.ascontiguousarray(np.asarray(a, dtype=np.float32))
            if a.shape != shp:
                raise ValueError("parameter of shape %s where the reference network has %s" % (a.shape, shp))
            host.append(a)
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        ptrs = (ctypes.c_void_p * 12)(*[a.ctypes.data for a in host])
        self._h = ctypes.c_void_p()
        check(_native.lib().f2_cnn_create(self.device.index, ptrs, int(dots), int(channels), ctypes.byref(self._h)))
        self._ws = None
        self.step = None

    def __del__(self):
        try:
            h = getattr(self, "_h", None)
            if h is not None and h.value:
                _native.lib().f2_cnn_destroy(h)
                self._h = None
        except Exception:
            pass

    def predict_envelope(self, env_t, step=160, frames=None, stream=None):
        """Scores of the stride-1 frames of a time-major envelope ([n, 128] float32 on the device):
        frame i = rows i + k*step, k < 11, normalised per frame like Training.normalizeInput
        (Evaluating.py:70-87).  Returns an (n_frames, 2) float32 device tensor; raises ValueError where
        normalizeInput would (a value <= 0)."""
        self._check_env_t(env_t)
        n = int(env_t.shape[0])
        nb = max(n - 11 * int(step), 0)
        i0, i1 = (0, nb) if frames is None else (int(frames[0]), int(frames[1]))
        if not 0 <= i0 <= i1 <= nb:
            raise IndexError("frames=(%d, %d) outside the %d frames of this envelope" % (i0, i1, nb))
        scores = torch.empty((i1 - i0, 2), dtype=torch.float32, device=self.device)
        if i1 == i0:
            return scores
        L = _native.lib()
        self._workspace(i1 - i0)
        flags = torch.zeros(2, dtype=torch.int32, device=self.device)
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        check(L.f2_cnn_forward(self._h, ctypes.c_void_p(env_t.data_ptr()), n, int(step), i0, i1,
                               ctypes.c_void_p(scores.data_ptr()), ctypes.c_void_p(flags.data_ptr()),
                               ctypes.c_void_p(self._ws.data_ptr()), self._ws.numel(), ctypes.c_void_p(s.cuda_stream)))
        bad, status = (int(v) for v in flags.tolist())
        if status:
            raise RuntimeError("tensor-core pipeline did not complete (stage %d)" % status)
        if bad:
            raise ValueError("values must all be positive")  # Training.py:18-20
        return scores

    def predict_segments(self, env_t, step, rows, counts, stream=None):
        """Scores of several utterances whose envelopes lie in ONE time-major env_t ([n, 128] float32 on the
        device), in one pass: segment s is counts[s] stride-1 frames starting at row rows[s] (frame i of it =
        rows rows[s] + i + k*step, k < 11), e.g. every frame of utterance s (counts[s] = max(n_s - 11*step, 0)).
        Returns the (sum(counts), 2) float32 device tensor of the segments' scores back to back; each frame's
        scores are bit for bit those predict_envelope gives for it.  Raises NonPositiveInput (a ValueError)
        naming the first segment that has a frame holding a value <= 0 (Training.normalizeInput raises there)."""
        self._check_env_t(env_t)
        rows = np.ascontiguousarray(rows, dtype=np.int64).reshape(-1)
        counts = np.ascontiguousarray(counts, dtype=np.int64).reshape(-1)
        if rows.shape != counts.shape:
            raise ValueError("rows and counts: one entry per segment")
        n, step = int(env_t.shape[0]), int(step)
        live = counts > 0
        if np.any(rows < 0) or np.any(counts < 0) or np.any(rows[live] + counts[live] + 10 * step > n):
            raise IndexError("a segment's frames leave the %d rows of this envelope" % n)
        total = int(counts.sum())
        scores = torch.empty((total, 2), dtype=torch.float32, device=self.device)
        if total == 0:
            return scores
        L = _native.lib()
        self._workspace(total)
        n_segs = int(rows.shape[0])
        flags = torch.zeros(n_segs + 1, dtype=torch.int32, device=self.device)
        s = stream if stream is not None else torch.cuda.current_stream(self.device)
        check(L.f2_cnn_forward_segments(self._h, ctypes.c_void_p(env_t.data_ptr()), n, step,
                                        rows.ctypes.data_as(ctypes.c_void_p), counts.ctypes.data_as(ctypes.c_void_p),
                                        n_segs, ctypes.c_void_p(scores.data_ptr()), ctypes.c_void_p(flags.data_ptr()),
                                        ctypes.c_void_p(self._ws.data_ptr()), self._ws.numel(),
                                        ctypes.c_void_p(s.cuda_stream)))
        s.synchronize()
        flags = flags.cpu().numpy()
        if flags[-1]:
            raise RuntimeError("tensor-core pipeline did not complete (stage %d)" % flags[-1])
        bad = np.flatnonzero(flags[:-1])
        if bad.size:
            raise NonPositiveInput(int(bad[0]))
        return scores

    def _check_env_t(self, env_t):
        if env_t.dtype != torch.float32 or not env_t.is_contiguous() or env_t.dim() != 2 or env_t.shape[1] != 128 \
                or env_t.device != self.device:
            raise ValueError("env_t: contiguous float32 [n, 128] tensor on %s" % self.device)

    def _workspace(self, n_frames):
        need = int(_native.lib().f2_cnn_workspace_bytes(self._h, int(n_frames)))
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)

    def intermediates(self, n_frames):
        """(pooled conv2 output (n, 32, 4, 63), features (n, 1920)) of the last chunk, as float32 -- for
        the layer-by-layer tests (n_frames <= 32768 so that the chunk is the whole call)."""
        chunk, off = ctypes.c_int64(), ctypes.c_size_t()
        check(_native.lib().f2_cnn_workspace_layout(int(n_frames), ctypes.byref(chunk), ctypes.byref(off)))
        base = (self._ws.data_ptr() + 255) // 256 * 256 - self._ws.data_ptr()
        raw = self._ws[base:base + n_frames * 4 * 252 * 16].view(torch.bfloat16).view(n_frames, 4, 252, 8)
        pooled = raw.permute(0, 1, 3, 2).reshape(n_frames, 32, 4, 63).float()
        feat = self._ws[base + off.value:base + off.value + n_frames * 1920 * 2].view(torch.bfloat16).view(n_frames, 1920)
        return pooled, feat.float()


class NonPositiveInput(ValueError):
    """A frame of segment `segment` of TensorCoreCNN.predict_segments held a value <= 0: the ValueError
    Training.normalizeInput raises (Training.py:18-20)."""

    def __init__(self, segment):
        super().__init__("values must all be positive (segment %d)" % segment)
        self.segment = segment


def keras_arrays(model):
    """The parameters of an F2CNN module in Keras' get_weights() order and layout."""
    out = []
    for conv in (model.c1, model.c2, model.c3, model.c4):
        out.append(conv.weight.detach().float().permute(2, 3, 1, 0).contiguous().cpu().numpy())
        out.append(conv.bias.detach().float().cpu().numpy())
    for lin in (model.d1, model.d2):
        out.append(lin.weight.detach().float().t().contiguous().cpu().numpy())
        out.append(lin.bias.detach().float().cpu().numpy())
    return out


WEIGHT_NAMES = ("conv1_kernel", "conv1_bias", "conv2_kernel", "conv2_bias", "conv3_kernel", "conv3_bias",
                "conv4_kernel", "conv4_bias", "dense1_kernel", "dense1_bias", "dense2_kernel", "dense2_bias")


def save_weights(path, source):
    """Write the 12 parameter arrays (Keras get_weights() order and layout) as an .npz: what
    scripts.CNN.Evaluating takes as `model` where no Keras is installed."""
    arrays = keras_arrays(source) if isinstance(source, torch.nn.Module) else list(source)
    np.savez(path, **{n: np.asarray(a, dtype=np.float32) for n, a in zip(WEIGHT_NAMES, arrays)})


def load_weights(path):
    """The 12 arrays of an .npz written by save_weights (or by numpy.savez(path, *model.get_weights()))."""
    with np.load(path, allow_pickle=False) as z:
        if all(n in z.files for n in WEIGHT_NAMES):
            return [z[n] for n in WEIGHT_NAMES]
        if all("arr_%d" % i in z.files for i in range(12)):
            return [z["arr_%d" % i] for i in range(12)]
    raise ValueError("%s does not hold the 12 parameter arrays of the reference network" % path)
