"""A bf16-faithful float64 reference of the tensor-core CNN forward (f2cnn_b200/csrc/f2_cnn.cu).

The kernels keep weights and activations in bf16 and accumulate in float32.  A plain float32 forward
(cnn.F2CNN) does not round where they round, so it can only be compared with them at a bound far wider
than their error.  This reference computes in float64 and rounds to bf16 at exactly the points where the
kernels store bf16, and nowhere else:

  stage        kernel                                                  here
  input        float32 min/max/log normalisation, bf16 into the grid   float64 normalisation, bf16
  weights      conv kernels and W5 in bf16 (f2_capi.cu bf16_rne),       same
               biases and W6 float32
  conv1        fp32 accumulate, +b1, relu, bf16                         float64 accumulate, +b1, relu, bf16
  conv2 + pool max of accumulators over rows 0..7 and column pairs,     same (row 8 and the last column dropped)
               +b2, relu, bf16                  -> p2 (intermediates)
  conv3, conv4 +b, relu, bf16                                           same
  pool+flatten max of bf16 values, Keras HWC order -> feat              same
  dense        bf16 feat x bf16 W5 in fp32, +b5, relu; fp32 logits      float64
               with fp32 W6, +b6; softmax

Every stage can also be applied on its own (normalize, front, mid, dense), so that a test can feed it the
kernel's own input to that stage: one rounding flip upstream then cannot blur the bound downstream.

`mutation` names one deliberate bug (MUTATIONS); a test shows its bounds would reject a kernel with that
bug by showing they reject the mutated reference.  `rounding=False` switches every bf16 rounding off: the
reference then is the float64 forward of cnn.F2CNN."""
import torch
import torch.nn.functional as F

MUTATIONS = (
    "no_b1", "no_b2", "no_b3", "no_b4", "no_b5", "no_b6",   # one bias dropped
    "swap_b6",               # the two logit biases exchanged
    "swap_w6",               # the two columns of the last dense kernel exchanged
    "conv2_transposed",      # conv2 taps read (dx, dy) instead of (dy, dx)
    "conv1_pad_shift",       # conv1's `same` zero padding one column too far left
    "pool_rows_1_8",         # conv2's 2x2 pool over rows 1..8 instead of 0..7
    "flatten_chw",           # features flattened channels-first instead of Keras' HWC
    "normalize_per_row",     # normalizeInput's min/max per time row instead of per frame
    "frame_late",            # every frame read one envelope row late
)

DOTS, CHANNELS = 11, 128


def bf16(x):
    """Round to bf16 (round to nearest even) the way f2_capi.cu's bf16_rne and the kernels'
    __float2bfloat16 do: from float32, a NaN stays a (quiet) NaN.  Returns float64."""
    u = x.to(torch.float32).contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) & 0xFFFF
    r = torch.where((u & 0x7FFFFFFF) > 0x7F800000, (u >> 16) | 0x40, r)
    r = r << 16
    r = torch.where(r >= 1 << 31, r - (1 << 32), r)
    return r.to(torch.int32).view(torch.float32).to(torch.float64)


def bf16_ulp(x):
    """Spacing of bf16 values at |x| (that of the smallest normal below it)."""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.pow(2.0, e - 7)


def spread_model(seed=5, gain=4.0):
    """A float32 F2CNN (on the CPU) whose every parameter matters to the scores, unlike
    cnn.seeded_model's (std 0.05 weights, 0.01 biases: all scores within 0.48..0.52, and dropping a
    dense bias moves them by less than 5e-3).  He-scaled weights (std sqrt(2 / fan_in)), biases of
    std 0.3 (comparable to the activations), and the last layer scaled by `gain` so that on
    speech-like envelopes the logit difference spreads by about +-3 without saturating the softmax
    (seed 5, gain 4: standard deviation about 1, median top score about 0.85)."""
    from f2cnn_b200 import cnn
    g = torch.Generator().manual_seed(seed)
    m = cnn.F2CNN()
    with torch.no_grad():
        for lay in (m.c1, m.c2, m.c3, m.c4, m.d1, m.d2):
            fan_in = lay.weight[0].numel()
            lay.weight.copy_(torch.randn(lay.weight.shape, generator=g) * (2.0 / fan_in) ** 0.5)
            lay.bias.copy_(torch.randn(lay.bias.shape, generator=g) * 0.3)
        m.d2.weight.mul_(gain)
    return m.eval()


def _params(source):
    """float64 tensors (conv weights OIHW, dense weights (out, in)) of an F2CNN module or of the 12
    Keras-layout arrays, every value first made float32 as the kernels receive it."""
    if isinstance(source, torch.nn.Module):
        m = source
        w = [m.c1.weight, m.c1.bias, m.c2.weight, m.c2.bias, m.c3.weight, m.c3.bias, m.c4.weight, m.c4.bias,
             m.d1.weight, m.d1.bias, m.d2.weight, m.d2.bias]
        return [t.detach().float().double().cpu() for t in w]
    a = [torch.as_tensor(x).float().double() for x in source]
    for i in (0, 2, 4, 6):
        a[i] = a[i].permute(3, 2, 0, 1)
    a[8], a[10] = a[8].t(), a[10].t()
    return [t.contiguous() for t in a]


class BF16Reference:
    def __init__(self, source, device="cpu", rounding=True, mutation=None):
        if mutation is not None and mutation not in MUTATIONS:
            raise ValueError("unknown mutation %r" % (mutation,))
        self.mutation = mutation
        self.r = bf16 if rounding else (lambda t: t)
        p = [t.to(device) for t in _params(source)]
        k1, b1, k2, b2, k3, b3, k4, b4, w5, b5, w6, b6 = p
        # weights as the kernels hold them: conv kernels and W5 in bf16, biases and W6 in float32
        self.k1, self.k2, self.k3, self.k4, self.w5 = (self.r(k) for k in (k1, k2, k3, k4, w5))
        self.b1, self.b2, self.b3, self.b4, self.b5, self.w6, self.b6 = b1, b2, b3, b4, b5, w6, b6
        if mutation and mutation.startswith("no_b"):
            i = int(mutation[-1])
            setattr(self, "b%d" % i, torch.zeros_like(getattr(self, "b%d" % i)))
        if mutation == "swap_b6":
            self.b6 = self.b6.flip(0)
        if mutation == "swap_w6":
            self.w6 = self.w6.flip(0)
        if mutation == "conv2_transposed":
            self.k2 = self.k2.transpose(2, 3).contiguous()

    # ---- stages -------------------------------------------------------------------------------------
    def frames(self, env_t, step, i0, i1):
        """(i1 - i0, 11, 128) float64: frame i = envelope rows i + k*step, k < 11 (f2_cnn_forward)."""
        late = 1 if self.mutation == "frame_late" else 0
        dev = env_t.device
        idx = torch.arange(i0, i1, device=dev)[:, None] + late + step * torch.arange(DOTS, device=dev)[None, :]
        return env_t[idx].to(torch.float64)

    def normalize(self, fr):
        """normalizeInput (Training.py:13-28) per frame, in float64, then bf16: (n, 1, 11, 128).
        Raises ValueError on a value <= 0, as the reference does."""
        if not bool((fr > 0).all()):
            raise ValueError("values must all be positive")
        dims = (2,) if self.mutation == "normalize_per_row" else (1, 2)
        lo, hi = fr.amin(dim=dims, keepdim=True), fr.amax(dim=dims, keepdim=True)
        span = torch.log(hi) - torch.log(lo)
        x = torch.where(hi > lo, (torch.log(fr) - torch.log(lo)) / torch.where(hi > lo, span, 1.0), 0.0)
        return self.r(x).unsqueeze(1)

    def front(self, x):
        """conv1 + relu + conv2 + relu + max pool: the kernel's p2, (n, 32, 4, 63)."""
        if self.mutation == "conv1_pad_shift":
            y = F.conv2d(F.pad(x, (2, 0, 1, 1)), self.k1)
        else:
            y = F.conv2d(x, self.k1, padding=1)
        y = self.r(F.relu(y + self.b1[:, None, None]))
        acc = F.conv2d(y, self.k2)                           # (n, 32, 9, 126)
        rows = acc[:, :, 1:9] if self.mutation == "pool_rows_1_8" else acc[:, :, 0:8]
        return self.r(F.relu(F.max_pool2d(rows, 2) + self.b2[:, None, None]))

    def mid(self, p2):
        """conv3 + relu + conv4 + relu + max pool + flatten: the kernel's features, (n, 1920)."""
        y = self.r(F.relu(F.conv2d(p2, self.k3, padding=1) + self.b3[:, None, None]))
        y = self.r(F.relu(F.conv2d(y, self.k4) + self.b4[:, None, None]))
        y = F.max_pool2d(y, 2)                               # (n, 64, 1, 30)
        if self.mutation == "flatten_chw":
            return y.reshape(y.shape[0], -1)
        return y.permute(0, 2, 3, 1).reshape(y.shape[0], -1)

    def logits(self, feat):
        h = F.relu(feat.to(torch.float64) @ self.w5.t() + self.b5)
        return h @ self.w6.t() + self.b6

    def dense(self, feat):
        """dense 516 + relu + dense 2 + softmax: scores (n, 2)."""
        return torch.softmax(self.logits(feat), dim=1)

    # ---- chained ------------------------------------------------------------------------------------
    def forward(self, env_t, step, i0, i1):
        """env_t -> {"p2", "feat", "logits", "scores"} for frames i0 .. i1 - 1."""
        p2 = self.front(self.normalize(self.frames(env_t, step, i0, i1)))
        feat = self.mid(p2)
        lg = self.logits(feat)
        return {"p2": p2, "feat": feat, "logits": lg, "scores": torch.softmax(lg, dim=1)}
