"""Keras-protocol glue the reference's model files rely on: `Layer` (build-on-first-call),
`Dense`, `DNN`, `BatchNormalization`, `Dropout`, activations.

These are the dense MLP pieces either side of the hot path (SURVEY.md §8 f2): they stay on the
framework's GEMM (torch -> cuBLAS, fp32, TF32 off) and exist so that model code written
against the reference's layer API runs unchanged.  Initialisers follow Keras (App. A4):
glorot_uniform kernels, zero biases.
"""
from __future__ import annotations

import math
from typing import Callable, Optional, Sequence

import torch
import torch.nn.functional as F


class Layer(torch.nn.Module):
    """Keras-style layer: `build(input_shape)` runs once on the first call, then `call`."""

    def __init__(self, name: Optional[str] = None, **kwargs):
        super().__init__()
        self._built = False
        self._name = name

    def build(self, input_shape):  # noqa: D401
        pass

    def call(self, inputs, **kwargs):
        raise NotImplementedError

    def forward(self, inputs, *args, **kwargs):
        if not self._built:
            self.build(_shape_of(inputs))
            self._built = True
        return self.call(inputs, *args, **kwargs)

    def add_weight(self, name: str, shape, initializer="glorot_uniform", regularizer=None,
                   trainable: bool = True, dtype=torch.float32, device=None):
        w = torch.empty(tuple(shape), dtype=dtype, device=device or _default_device())
        _init_(w, initializer)
        p = torch.nn.Parameter(w, requires_grad=trainable)
        self.register_parameter(name, p)
        if regularizer is not None:
            self.__dict__.setdefault("_regularized", []).append((p, regularizer))
        return p

    def regularization_loss(self):
        """Sum of the l2(λ)·Σw² terms of this layer and its children (Keras adds them to the loss)."""
        total = 0.0
        for m in self.modules():
            for p, reg in m.__dict__.get("_regularized", []):
                total = total + reg(p)
        return total


def _default_device():
    return torch.device("cuda") if torch.cuda.is_available() else torch.device("cpu")


def _shape_of(x):
    if isinstance(x, (list, tuple)):
        return [_shape_of(t) for t in x]
    if isinstance(x, dict):
        return {k: _shape_of(v) for k, v in x.items()}
    return tuple(x.shape) if hasattr(x, "shape") else None


def _init_(w: torch.Tensor, initializer) -> None:
    if callable(initializer):
        initializer(w)
    elif initializer in ("glorot_uniform", None):
        if w.dim() >= 2:
            fan_in, fan_out = w.shape[0], w.shape[1]
        else:                         # Keras: scalar / 1-D -> fans (1,1) / (n,n)
            fan_in = fan_out = max(1, w.numel())
        lim = math.sqrt(6.0 / (fan_in + fan_out))
        with torch.no_grad():
            w.uniform_(-lim, lim)
    elif initializer == "random_normal":
        with torch.no_grad():
            w.normal_(0.0, 0.05)
    elif initializer == "random_uniform":
        with torch.no_grad():
            w.uniform_(-0.05, 0.05)
    elif initializer == "zeros":
        with torch.no_grad():
            w.zero_()
    elif initializer == "ones":
        with torch.no_grad():
            w.fill_(1.0)
    else:
        raise ValueError(f"unknown initializer {initializer!r}")


class l2:
    """tensorflow.keras.regularizers.l2: λ·Σ w² (no ½), App. A3."""

    def __init__(self, l2: float = 0.01):
        self.l2 = float(l2)

    def __call__(self, w):
        return self.l2 * (w * w).sum()


def get_activation(act) -> Optional[Callable]:
    if act is None or act == "linear":
        return None
    if callable(act):
        return act
    table = {"relu": F.relu, "sigmoid": torch.sigmoid, "tanh": torch.tanh, "softmax":
             lambda x: torch.softmax(x, -1)}
    if act not in table:
        # the reference's default att_activation='prelu' is not a Keras activation string either
        raise ValueError(f"Unknown activation function: {act}")
    return table[act]


class Dense(Layer):
    """tensorflow.keras.layers.Dense: y = act(x·W + b); contracts the last axis (A4)."""

    def __init__(self, units: int, activation=None, use_bias: bool = True,
                 kernel_regularizer=None, **kwargs):
        super().__init__(**kwargs)
        self.units, self.use_bias, self.kernel_regularizer = units, use_bias, kernel_regularizer
        self.activation = get_activation(activation)
        self._act_name = activation if isinstance(activation, str) else None
        if isinstance(activation, torch.nn.Module):
            self.activation_module = activation

    def build(self, input_shape):
        self.kernel = self.add_weight("kernel", (input_shape[-1], self.units), "glorot_uniform",
                                      self.kernel_regularizer)
        self.bias = self.add_weight("bias", (self.units,), "zeros") if self.use_bias else None

    def call(self, x, **kwargs):
        if self.bias is not None and x.dim() >= 2 and x.is_cuda:
            # rank-3 inputs contract the last axis (Keras tensordot, App. A4): the same GEMM on
            # the flattened (B*L, d) rows — tensor-core path, fused bias / ReLU / bias-gradient
            relu = self._act_name == "relu"
            lead = x.shape[:-1]
            x2 = x.reshape(-1, x.shape[-1]) if x.dim() > 2 else x
            y = _DenseFn.apply(x2, self.kernel, self.bias, relu)
            if x.dim() > 2:
                y = y.reshape(*lead, self.units)
            return y if (relu or self.activation is None) else self.activation(y)
        y = torch.matmul(x, self.kernel)
        if self.bias is not None:
            y = y + self.bias
        return self.activation(y) if self.activation is not None else y


# Dense GEMM backend: "bf16x6" = librtf_b200's tcgen05 GEMM (fp32 operands split into 3 bf16 terms,
# the 6 partial products above one fp32 ulp accumulated in fp32; csrc/dense_gemm.cuh), "library" =
# the framework's GEMM (cuBLAS).  Shapes the tensor-core path does not take (K or N not a multiple
# of 4, tiny problems, CPU tensors) always use the library.
DENSE_GEMM = "bf16x6"


def set_dense_gemm(kind: str) -> None:
    global DENSE_GEMM
    if kind not in ("bf16x6", "library"):
        raise ValueError(kind)
    DENSE_GEMM = kind


# bf16x6 layers large enough to repay splitting their operands into bf16 planes once (a pass at
# HBM rate per operand, 10 B per value) run the plane-fed GEMM (csrc/dense_gemm_planes.cuh), whose
# mainloop has no transform warps; the results are bit-identical to the fp32-fed GEMM.  Measured
# on a B200 at B = 65 536 (profiles/r4_dense_planes.jsonl), the saving beats the split passes when
# K N / (K + N) >= 256: the 480-1024-1024-512 layers of the DLRM top MLP, not its 512-256 or
# the bottom MLP's 512-256-128 layers.  set_dense_planes(False) forces the fp32-fed GEMM.
DENSE_PLANES = True


def set_dense_planes(on: bool) -> None:
    global DENSE_PLANES
    DENSE_PLANES = bool(on)


def _planes_pay(M: int, K: int, N: int) -> bool:
    return DENSE_PLANES and K % 8 == 0 and N % 8 == 0 and K * N >= 256 * (K + N)


def _x6_ok(*mats) -> bool:
    if DENSE_GEMM != "bf16x6":
        return False
    for m in mats:
        if not (m.is_cuda and m.dtype == torch.float32 and m.dim() == 2 and m.is_contiguous()
                and m.shape[0] % 4 == 0 and m.shape[1] % 4 == 0 and m.data_ptr() % 16 == 0):
            return False
    return True


def dense_gemm(kind: str, a: torch.Tensor, b: torch.Tensor, bias=None, relu: bool = False,
               splits: int = 1) -> torch.Tensor:
    """librtf_b200 fp32-accurate tensor-core GEMM on contiguous 2-D fp32 CUDA tensors.
    kind 'nn': a (M,K) @ b (K,N) [+ bias, ReLU];  'nt': a (M,K) @ b (N,K)^T;
    'tn': a (K,M)^T @ b (K,N), optionally as `splits` partial products over K summed in order."""
    import ctypes as C
    from . import _lib as L
    lib = L.lib()
    if kind == "nn":
        (M, K), N = a.shape, b.shape[1]
    elif kind == "nt":
        (M, K), N = a.shape, b.shape[0]
    elif kind == "tn":
        (K, M), N = a.shape, b.shape[1]
    else:
        raise ValueError(kind)
    fn = getattr(lib, f"rtf_dense_gemm_{kind}")
    wsq = getattr(lib, f"rtf_dense_gemm_{kind}_workspace")
    lda, ldb = a.stride(0), b.stride(0)
    sa = sb = sd = 0
    batch = 1
    if kind == "tn" and splits > 1:
        if K % splits or (K // splits) % 4:
            raise ValueError("splits must divide K into multiples of 4")
        batch, K = splits, K // splits
        sa, sb, sd = K * lda, K * ldb, M * N
    out = torch.empty((batch, M, N) if batch > 1 else (M, N), dtype=torch.float32, device=a.device)
    key = (kind, M, N, K, batch)
    if key not in _GEMM_WS_BYTES:
        nb = C.c_size_t(0)
        L.check(wsq(M, N, K, batch, C.byref(nb)), f"rtf_dense_gemm_{kind}_workspace")
        _GEMM_WS_BYTES[key] = max(nb.value, 16)
    ws = _scratch(_GEMM_WS_BYTES[key], a.device)
    rc = fn(a.data_ptr(), lda, sa, b.data_ptr(), ldb, sb, None if bias is None else bias.data_ptr(),
            int(relu), out.data_ptr(), N, sd, M, N, K, batch, ws.data_ptr(), ws.numel(),
            L.current_stream_ptr())
    L.check(rc, f"rtf_dense_gemm_{kind}")
    return out.sum(0) if batch > 1 else out


def split_planes(x: torch.Tensor) -> torch.Tensor:
    """Split a contiguous 2-D fp32 CUDA tensor (R, C) into its three bf16 planes, a (3, R, C)
    bf16 tensor with x ~= p0 + p1 * 2^-8 + p2 * 2^-16: the operand split the dense GEMM's
    mainloop makes (rtf_split_bf16x3)."""
    from . import _lib as L
    if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.is_contiguous()):
        raise ValueError("split_planes takes a contiguous 2-D fp32 CUDA tensor")
    R, Cc = x.shape
    p = torch.empty((3, R, Cc), dtype=torch.bfloat16, device=x.device)
    L.check(L.lib().rtf_split_bf16x3(x.data_ptr(), R, Cc, Cc, p.data_ptr(), Cc, R * Cc,
                                     L.current_stream_ptr()), "rtf_split_bf16x3")
    return p


def dense_gemm_planes(kind: str, a: torch.Tensor, b: torch.Tensor, bias=None, relu: bool = False,
                      splits: int = 1) -> torch.Tensor:
    """dense_gemm on operands given as bf16 planes (split_planes): a, b are (3, rows, cols)
    contiguous bf16 tensors holding the planes of the 2-D fp32 operands dense_gemm takes.  The
    result is bit-identical to dense_gemm on the fp32 operands the planes were split from."""
    import ctypes as C
    from . import _lib as L
    lib = L.lib()
    for m in (a, b):
        if not (m.is_cuda and m.dtype == torch.bfloat16 and m.dim() == 3 and m.shape[0] == 3
                and m.is_contiguous()):
            raise ValueError("plane operands are contiguous (3, rows, cols) bf16 CUDA tensors")
    if kind == "nn":
        (M, K), N = a.shape[1:], b.shape[2]
    elif kind == "nt":
        (M, K), N = a.shape[1:], b.shape[1]
    elif kind == "tn":
        (K, M), N = a.shape[1:], b.shape[2]
    else:
        raise ValueError(kind)
    fn = getattr(lib, f"rtf_dense_gemm_{kind}_planes")
    wsq = getattr(lib, f"rtf_dense_gemm_{kind}_planes_workspace")
    lda, ldb = a.stride(1), b.stride(1)
    sa = sb = sd = 0
    batch = 1
    if kind == "tn" and splits > 1:
        if K % splits or (K // splits) % 4:
            raise ValueError("splits must divide K into multiples of 4")
        batch, K = splits, K // splits
        sa, sb, sd = K * lda, K * ldb, M * N
    out = torch.empty((batch, M, N) if batch > 1 else (M, N), dtype=torch.float32, device=a.device)
    key = (kind + "_planes", M, N, K, batch)
    if key not in _GEMM_WS_BYTES:
        nb = C.c_size_t(0)
        L.check(wsq(M, N, K, batch, C.byref(nb)), f"rtf_dense_gemm_{kind}_planes_workspace")
        _GEMM_WS_BYTES[key] = max(nb.value, 16)
    ws = _scratch(_GEMM_WS_BYTES[key], a.device)
    rc = fn(a.data_ptr(), lda, sa, a.stride(0), b.data_ptr(), ldb, sb, b.stride(0),
            None if bias is None else bias.data_ptr(), int(relu), out.data_ptr(), N, sd, M, N, K,
            batch, ws.data_ptr(), ws.numel(), L.current_stream_ptr())
    L.check(rc, f"rtf_dense_gemm_{kind}_planes")
    return out.sum(0) if batch > 1 else out


_GEMM_WS_BYTES: dict = {}
_SCRATCH: dict = {}


def _scratch(nbytes: int, device) -> torch.Tensor:
    """A reusable kernel-scratch buffer per (device, stream): launches on one stream are ordered,
    so consecutive GEMMs / reductions may share it (saves an allocator round trip per launch —
    ~60 per training step, and the host has to stay ahead of the GPU)."""
    key = (device.index, torch._C._cuda_getCurrentRawStream(device.index if device.index is not None
                                                            else torch._C._cuda_getDevice()))
    buf = _SCRATCH.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = _SCRATCH[key] = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
    return buf


def _wgrad_splits(B: int, kin: int, n: int, clusters: int = 74) -> int:
    """Split count for dW = x^T g: the reduction runs over the batch while the output is only a
    few 256x128 tiles, so the K loop is cut into fixed chunks (>= 512 rows) until the tiles fill
    the 74 SM pairs with the least wave quantisation (e.g. 1024x1024: 32 tiles x 16 = 6.9 waves)."""
    tiles = ((kin + 255) // 256) * ((n + 127) // 128)
    best, best_eff = 1, 0.0
    s = 1
    while s <= 64 and B % s == 0 and (B // s) % 4 == 0 and B // s >= 512:
        waves = tiles * s / clusters
        eff = waves / -(-tiles * s // clusters)
        if eff > best_eff + 0.02:
            best, best_eff = s, eff
        s *= 2
    return best


def _wgrad(x: torch.Tensor, g: torch.Tensor) -> torch.Tensor:
    """dW = x^T g for a tall batch.  The reduction runs over the batch (K = 65 536 here) while the
    output is only a few 128x128 tiles, so a single GEMM leaves most SMs idle; a batched
    split-K (fixed chunking, partials summed in order => deterministic) measured 2-2.6x faster
    (tools/probe_wgrad.py)."""
    B = x.shape[0]
    if B >= 1024 and _x6_ok(x, g):
        return dense_gemm("tn", x, g, splits=_wgrad_splits(B, x.shape[1], g.shape[1]))
    S = 16
    if B >= 8192 and B % S == 0 and x.is_contiguous() and g.is_contiguous():
        return torch.bmm(x.view(S, B // S, -1).transpose(1, 2), g.view(S, B // S, -1)).sum(0)
    return x.t() @ g


def _relu_bwd_bias_grad(gy: torch.Tensor, y):
    """(g, db): g = gy * (y > 0) (g is gy itself when y is None) and db = g.sum(0), in one pass
    through librtf_b200 (rtf_relu_bwd_colsum) when the layout allows, else framework ops."""
    B, N = gy.shape
    if gy.is_cuda and N % 4 == 0 and B > 0:
        import ctypes as C
        from . import _lib as L
        gy = gy.contiguous()
        key = ("relu_bwd", B, N)
        if key not in _GEMM_WS_BYTES:
            nb = C.c_size_t(0)
            L.check(L.lib().rtf_relu_bwd_colsum_workspace(B, N, C.byref(nb)), "rtf_relu_bwd_colsum_workspace")
            _GEMM_WS_BYTES[key] = max(nb.value, 16)
        ws = _scratch(_GEMM_WS_BYTES[key], gy.device)
        g = torch.empty_like(gy) if y is not None else gy
        db = torch.empty(N, dtype=torch.float32, device=gy.device)
        L.check(L.lib().rtf_relu_bwd_colsum(gy.data_ptr(), None if y is None else y.data_ptr(), B, N,
                                            g.data_ptr(), db.data_ptr(), ws.data_ptr(),
                                            L.current_stream_ptr()), "rtf_relu_bwd_colsum")
        return g, db
    g = torch.ops.aten.threshold_backward(gy, y, 0.0) if y is not None else gy.contiguous()
    return g, g.sum(0)


class _DenseFn(torch.autograd.Function):
    """x W + b (optionally ReLU) with bias / ReLU in the library GEMM's epilogue — one pass over
    the output instead of three; backward masks the incoming gradient once, split-K weight grad."""

    @staticmethod
    def forward(ctx, x, w, b, relu):
        kpad = 0
        if (x.shape[1] % 4 and DENSE_GEMM == "bf16x6" and x.is_cuda and x.shape[0] >= 1024
                and w.shape[1] % 4 == 0 and x.shape[0] % 4 == 0):
            # e.g. the 13 dense Criteo features: zero-pad K to a multiple of 4 (16-byte rows for
            # TMA) so this layer runs on the tensor-core path too; the pad is sliced off again
            kpad = (-x.shape[1]) % 4
            x = F.pad(x, (0, kpad))
            w = F.pad(w, (0, 0, 0, kpad))
        ctx.kpad = kpad
        ctx.planes = False
        if x.shape[0] >= 1024 and _x6_ok(x, w) and b.data_ptr() % 16 == 0:
            if _planes_pay(*x.shape, w.shape[1]):
                # split x and W into bf16 planes once; the backward's dgrad and wgrad reuse them
                ctx.planes = True
                xp, wp = split_planes(x), split_planes(w)
                y = dense_gemm_planes("nn", xp, wp, b, relu)
                ctx.save_for_backward(xp, wp, y if relu else None)
                ctx.relu = relu
                return y
            y = dense_gemm("nn", x, w, b, relu)
        else:
            y = torch._addmm_activation(b, x, w, use_gelu=False) if relu else torch.addmm(b, x, w)
        ctx.save_for_backward(x, w, y if relu else None)
        ctx.relu = relu
        return y

    @staticmethod
    def backward(ctx, gy):
        x, w, y = ctx.saved_tensors
        g, gb = _relu_bwd_bias_grad(gy, y if ctx.relu else None)
        if ctx.planes:   # x, w are the planes of the forward's operands
            gp = split_planes(g)
            gx = dense_gemm_planes("nt", gp, w) if ctx.needs_input_grad[0] else None
            gw = None
            if ctx.needs_input_grad[1]:
                B = g.shape[0]
                gw = dense_gemm_planes("tn", x, gp, splits=_wgrad_splits(B, x.shape[2], g.shape[1]))
            if ctx.kpad:   # the K padding of the forward (e.g. a 479-wide interaction -> 480)
                gx = None if gx is None else gx[:, : gx.shape[1] - ctx.kpad].contiguous()
                gw = None if gw is None else gw[: gw.shape[0] - ctx.kpad]
            return gx, gw, gb, None
        gx = None
        if ctx.needs_input_grad[0]:
            gx = dense_gemm("nt", g, w) if (g.shape[0] >= 1024 and _x6_ok(g, w)) else g @ w.t()
        gw = _wgrad(x, g) if ctx.needs_input_grad[1] else None
        if ctx.kpad:
            # contiguous: a strided (B, 13) view sends BatchNorm's backward down a 2 ms generic path
            gx = None if gx is None else gx[:, : gx.shape[1] - ctx.kpad].contiguous()
            gw = None if gw is None else gw[: gw.shape[0] - ctx.kpad]
        return gx, gw, gb, None


class _BatchNormTrainFn(torch.autograd.Function):
    """Training-mode BatchNormalization through librtf_b200 (rtf_bn_fwd / rtf_bn_bwd): batch
    statistics + normalisation + the Keras moving-average update in the forward, (dx, dgamma,
    dbeta) in the backward; the column reductions are deterministic two-stage sums."""

    @staticmethod
    def forward(ctx, x2, gamma, beta, eps, momentum, moving_mean, moving_var):
        import ctypes as C
        from . import _lib as L
        L.require_cuda(x2, "BatchNormalization(x)")
        if x2.dtype != torch.float32:
            raise TypeError("BatchNormalization: fp32 activations only")
        if x2.stride(1) != 1:
            x2 = x2.contiguous()
        B, Cc = x2.shape
        key = ("bn", B, Cc)
        if key not in _GEMM_WS_BYTES:
            nb = C.c_size_t(0)
            L.check(L.lib().rtf_bn_workspace(B, Cc, C.byref(nb)), "rtf_bn_workspace")
            _GEMM_WS_BYTES[key] = nb.value
        ws = _scratch(_GEMM_WS_BYTES[key], x2.device)
        y = torch.empty((B, Cc), dtype=torch.float32, device=x2.device)
        stats = torch.empty((2, Cc), dtype=torch.float32, device=x2.device)
        L.check(L.lib().rtf_bn_fwd(x2.data_ptr(), x2.stride(0), B, Cc,
                                   None if gamma is None else gamma.data_ptr(),
                                   None if beta is None else beta.data_ptr(), eps, momentum,
                                   y.data_ptr(), y.stride(0), stats[0].data_ptr(), stats[1].data_ptr(),
                                   None if moving_mean is None else moving_mean.data_ptr(),
                                   None if moving_var is None else moving_var.data_ptr(),
                                   ws.data_ptr(), ws.numel(), L.current_stream_ptr()), "rtf_bn_fwd")
        ctx.save_for_backward(x2, stats, gamma)
        ctx.has_beta = beta is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        import ctypes as C
        from . import _lib as L
        x2, stats, gamma = ctx.saved_tensors
        B, Cc = x2.shape
        if dy.stride(1) != 1:
            dy = dy.contiguous()
        ws = _scratch(_GEMM_WS_BYTES[("bn", B, Cc)], x2.device)
        dx = torch.empty_like(dy) if ctx.needs_input_grad[0] else None
        dg = torch.empty(Cc, dtype=torch.float32, device=dy.device) if gamma is not None else None
        db = torch.empty(Cc, dtype=torch.float32, device=dy.device) if ctx.has_beta else None
        L.check(L.lib().rtf_bn_bwd(dy.data_ptr(), dy.stride(0), x2.data_ptr(), x2.stride(0), B, Cc,
                                   stats[0].data_ptr(), stats[1].data_ptr(),
                                   None if gamma is None else gamma.data_ptr(),
                                   None if dx is None else dx.data_ptr(),
                                   0 if dx is None else dx.stride(0),
                                   None if dg is None else dg.data_ptr(),
                                   None if db is None else db.data_ptr(),
                                   ws.data_ptr(), ws.numel(), L.current_stream_ptr()), "rtf_bn_bwd")
        return dx, dg, db, None, None, None, None


class BatchNormalization(Layer):
    """Keras defaults (A9): momentum 0.99, eps 1e-3, batch statistics in training."""

    def __init__(self, center: bool = True, scale: bool = True, momentum: float = 0.99,
                 epsilon: float = 1e-3, trainable: bool = True, **kwargs):
        super().__init__(**kwargs)
        self.center, self.scale, self.momentum, self.epsilon = center, scale, momentum, epsilon

    def build(self, input_shape):
        c = input_shape[-1]
        self.gamma = self.add_weight("gamma", (c,), "ones") if self.scale else None
        self.beta = self.add_weight("beta", (c,), "zeros") if self.center else None
        dev = _default_device()
        self.register_buffer("moving_mean", torch.zeros(c, device=dev))
        self.register_buffer("moving_variance", torch.ones(c, device=dev))

    def call(self, x, **kwargs):
        shp = x.shape
        x2 = x.reshape(-1, shp[-1])
        if self.training and x2.is_cuda and x2.shape[0] > 0:
            # batch statistics, normalisation and Keras' moving averages (BIASED batch variance;
            # torch's running_var would take the unbiased one) in rtf_bn_fwd
            y = _BatchNormTrainFn.apply(x2, self.gamma, self.beta, self.epsilon, self.momentum,
                                        self.moving_mean, self.moving_variance)
        elif self.training:       # CPU tensors: layer-building / checkpoint tests without a GPU
            y, mean, invstd = torch.native_batch_norm(x2, self.gamma, self.beta, None, None, True, 0.0,
                                                      self.epsilon)
            with torch.no_grad():
                var = 1.0 / (invstd * invstd) - self.epsilon
                self.moving_mean.mul_(self.momentum).add_(mean, alpha=1.0 - self.momentum)
                self.moving_variance.mul_(self.momentum).add_(var, alpha=1.0 - self.momentum)
        else:
            y = F.batch_norm(x2, self.moving_mean, self.moving_variance, self.gamma, self.beta,
                             False, 0.0, self.epsilon)
        return y.reshape(shp)


class Dropout(Layer):
    def __init__(self, rate: float = 0.0, **kwargs):
        super().__init__(**kwargs)
        self.rate = rate

    def call(self, x, **kwargs):
        return F.dropout(x, self.rate, self.training) if self.rate > 0 else x


class DNN(Layer):
    """ctr.layers.modules.DNN (src/ctr/layers/modules.py:114-135): a BatchNormalization created
    inside `call` (once, A5), the Dense stack, then dropout.  `input_bn=False` gives the
    match-side DNN (src/match/layers/modules.py:8-26), which has no BatchNormalization."""

    def __init__(self, hidden_units: Sequence[int], activation="relu", dnn_dropout: float = 0.0,
                 input_bn: bool = True, **kwargs):
        super().__init__(**kwargs)
        self.dnn_network = torch.nn.ModuleList([Dense(u, activation=activation) for u in hidden_units])
        self.dropout = Dropout(dnn_dropout)
        self.bn = BatchNormalization() if input_bn else None

    def call(self, inputs, **kwargs):
        x = inputs
        if self.bn is not None:
            x = self.bn(x)
        for dnn in self.dnn_network:
            x = dnn(x)
        return self.dropout(x)


class DenseAdam:
    """Keras-form Adam (App. A12; what every reference script compiles with,
    src/ctr/fm/train.py:49-50) for the dense variables, as ONE kernel (rtf_dense_adam) over flat
    buffers: the parameters are re-pointed at views of `flat`, their `.grad`s at views of
    `flat_grad` (autograd accumulates into them in place), so a data-parallel trainer all-reduces
    `flat_grad` directly and nothing is concatenated or copied back.  Same formulas and rounding
    as K2's sparse row update, so embeddings and MLPs follow one Adam form:
        m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  w -= lr sqrt(1-b2^t)/(1-b1^t) m/(sqrt(v)+eps)"""

    ALIGN = 64      # floats: every parameter starts on a 256-byte boundary (TMA / float4 loads)

    def __init__(self, params, lr: float = 1e-3, beta1: float = 0.9, beta2: float = 0.999,
                 eps: float = 1e-7):
        from . import _lib as L
        params = [p for p in params if p.requires_grad]
        if not params:
            raise ValueError("DenseAdam: no trainable parameters")
        for p in params:
            L.require_cuda(p, "DenseAdam(param)")
            if p.dtype != torch.float32:
                raise TypeError("DenseAdam: fp32 parameters only")
        self.params, self.lr, self.beta1, self.beta2, self.eps = params, lr, beta1, beta2, eps
        self.t = 0
        self.lr_dev = None
        offs, n = [], 0
        for p in params:
            offs.append(n)
            n += (p.numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        dev = params[0].device
        self.flat = torch.zeros(n, dtype=torch.float32, device=dev)
        self.flat_grad = torch.zeros_like(self.flat)
        self.m = torch.zeros_like(self.flat)
        self.v = torch.zeros_like(self.flat)
        with torch.no_grad():
            for p, o in zip(params, offs):
                view = self.flat[o:o + p.numel()].view(p.shape)
                view.copy_(p.data)
                p.data = view
                p.grad = self.flat_grad[o:o + p.numel()].view(p.shape)
        self.offsets = offs

    def zero_grad(self):
        self.flat_grad.zero_()
        for p, o in zip(self.params, self.offsets):     # someone may have set .grad to None
            if p.grad is None or p.grad.data_ptr() != self.flat_grad.data_ptr() + 4 * o:
                p.grad = self.flat_grad[o:o + p.numel()].view(p.shape)

    def lr_for_step(self, t: int) -> float:
        return self.lr * math.sqrt(1.0 - self.beta2 ** t) / (1.0 - self.beta1 ** t)

    def enable_device_lr(self):
        """Step size in a device scalar (rtf_opt.lr_dev), refreshed by advance() — see StepGraph."""
        if self.lr_dev is None:
            self.lr_dev = torch.zeros(1, dtype=torch.float32, device=self.flat.device)
            self.lr_dev.fill_(self.lr_for_step(max(self.t, 1)))

    def advance(self):
        self.t += 1
        if self.lr_dev is not None:
            self.lr_dev.fill_(self.lr_for_step(self.t))

    def apply(self):
        """The launch alone (step t was set by advance())."""
        import ctypes as C
        from . import _lib as L
        st = L.rtf_opt(L.OPT_ADAM, self.lr_for_step(max(self.t, 1)), self.beta1, self.beta2,
                       self.eps, 0.0, None if self.lr_dev is None else self.lr_dev.data_ptr())
        L.check(L.lib().rtf_dense_adam(self.flat.data_ptr(), self.flat_grad.data_ptr(),
                                       self.m.data_ptr(), self.v.data_ptr(), self.flat.numel(),
                                       C.byref(st), L.current_stream_ptr()), "rtf_dense_adam")

    def step(self):
        self.advance()
        self.apply()


def _tree_map(fn, x):
    if isinstance(x, torch.Tensor):
        return fn(x)
    if isinstance(x, (list, tuple)):
        return type(x)(_tree_map(fn, v) for v in x)
    if isinstance(x, dict):
        return {k: _tree_map(fn, v) for k, v in x.items()}
    return x


def _tree_leaves(x, out=None):
    out = [] if out is None else out
    if isinstance(x, torch.Tensor):
        out.append(x)
    elif isinstance(x, (list, tuple)):
        for v in x:
            _tree_leaves(v, out)
    elif isinstance(x, dict):
        for k in x:
            _tree_leaves(x[k], out)
    return out


class StepGraph:
    """One training step replayed from a CUDA graph.

    The small models of the reference (FM, DIN, YoutubeDNN at batch 4096) take 100-350 kernel
    launches of a few microseconds each per step: the step time is the host's launch rate, not
    the GPU.  The whole step — K1 lookups, interaction kernels, GEMMs, backward, K2's sort +
    row updates (side stream included), the dense Adam launch — is captured once and replayed
    with one cudaGraphLaunch.  What changes between steps stays outside the graph:
      * the batch: copied into static input buffers before the replay;
      * the Adam step size lr*sqrt(1-b2^t)/(1-b1^t): a device scalar the kernels read
        (rtf_opt.lr_dev), refreshed by `advance()` before the replay.
    `warmup` steps run eagerly first (lazy layer builds, allocator, library handles), then the
    capture; a batch whose shapes differ from the captured ones (a ragged last batch) runs
    eagerly.  The returned loss is a static buffer overwritten by the next step.

        sg = StepGraph(body, advance)       # body(inputs, labels) -> loss; advance() -> None
        loss = sg(inputs, labels)
    """

    def __init__(self, body, advance, warmup: int = 3):
        self.body, self.advance, self.warmup = body, advance, warmup
        self.graph = None
        self.n_eager = 0
        self.n_replays = 0

    @staticmethod
    def _sig(*trees):
        return tuple((tuple(t.shape), t.dtype, t.device) for t in _tree_leaves(list(trees)))

    def __call__(self, inputs, labels=None):
        if self.graph is None and self.n_eager < self.warmup:
            self.n_eager += 1
            self.advance()
            return self.body(inputs, labels)
        if self.graph is None:
            self._capture(inputs, labels)
        if self._sig(inputs, labels) != self.sig:
            self.advance()
            return self.body(inputs, labels)
        for dst, src in zip(self.static_leaves, _tree_leaves([inputs, labels])):
            if dst.data_ptr() != src.data_ptr():
                dst.copy_(src, non_blocking=True)
        self.advance()
        self.graph.replay()
        self.n_replays += 1
        return self.static_loss

    def _capture(self, inputs, labels):
        self.sig = self._sig(inputs, labels)
        self.static_in = _tree_map(lambda t: t.clone(), inputs)
        self.static_labels = _tree_map(lambda t: t.clone(), labels)
        self.static_leaves = _tree_leaves([self.static_in, self.static_labels])
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            loss = self.body(self.static_in, self.static_labels)
        self.graph, self.static_loss = g, loss


class _BCEFn(torch.autograd.Function):
    """Keras binary_crossentropy through librtf_b200 (rtf_bce_fwd): loss and d loss / d p in one
    pass + an ordered sum of the chunk partials — 2 launches instead of ~30 framework ones."""

    @staticmethod
    def forward(ctx, p, y):
        import ctypes as C
        from . import _lib as L
        n = p.numel()
        key = ("bce", n)
        if key not in _GEMM_WS_BYTES:
            nb = C.c_size_t(0)
            L.check(L.lib().rtf_bce_workspace(n, C.byref(nb)), "rtf_bce_workspace")
            _GEMM_WS_BYTES[key] = max(nb.value, 16)
        ws = _scratch(_GEMM_WS_BYTES[key], p.device)
        loss = torch.empty((), dtype=torch.float32, device=p.device)
        dp = torch.empty_like(p) if ctx.needs_input_grad[0] else None
        L.check(L.lib().rtf_bce_fwd(y.data_ptr(), p.data_ptr(), n, loss.data_ptr(),
                                    None if dp is None else dp.data_ptr(), ws.data_ptr(),
                                    L.current_stream_ptr()), "rtf_bce_fwd")
        if dp is not None:
            ctx.save_for_backward(dp)
        return loss

    @staticmethod
    def backward(ctx, g):
        (dp,) = ctx.saved_tensors
        return dp * g, None


def binary_crossentropy(y_true: torch.Tensor, y_pred: torch.Tensor) -> torch.Tensor:
    """Keras `binary_crossentropy` on probabilities (A11): clip to [1e-7, 1-1e-7], then
    -mean(y·log(p+1e-7) + (1-y)·log(1-p+1e-7)).  fp32 CUDA tensors take the one-pass kernel
    (`rtf_bce_fwd`); anything else the framework's elementwise ops."""
    if (y_pred.is_cuda and y_pred.dtype == torch.float32 and y_pred.numel() > 0
            and not y_true.requires_grad):
        y = y_true.to(torch.float32).reshape(y_pred.shape).contiguous()
        return _BCEFn.apply(y_pred.contiguous(), y)
    eps = 1e-7
    p = torch.clamp(y_pred, eps, 1.0 - eps)
    y = y_true.to(p.dtype).reshape(p.shape)
    return -(y * torch.log(p + eps) + (1.0 - y) * torch.log(1.0 - p + eps)).mean()
