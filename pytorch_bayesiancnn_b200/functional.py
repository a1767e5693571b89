"""Host side of the boundary: torch.autograd.Functions that call the C ABI.

PyTorch supplies device memory, the current stream and autograd; every number on
the Bayesian layer path is produced by libbbb_b200.so.  Nothing here computes a
layer with aten ops.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import itertools
import os
import threading
import weakref
from typing import Iterable, Optional

import torch

from . import _lib as L


# --------------------------------------------------------------------------- #
# noise bookkeeping (Python owns (seed, stream_id); kernels own the draws)
# --------------------------------------------------------------------------- #
_MASK64 = 0xFFFFFFFFFFFFFFFF
_MC_NAMESPACE = 1 << 63            # stream ids of Monte-Carlo evaluation samples (mc_sample): disjoint from training's
_instances = itertools.count()     # one _Noise per thread; the index keeps DataParallel replica threads apart


def _rank() -> int:
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank()
    except Exception:
        pass
    return int(os.environ.get("RANK", "0"))


class _Noise(threading.local):
    """(seed, stream counter) of the calling thread.

    Default seed: derived from ``torch.initial_seed()``, the process rank and the thread's index, so that
    ``torch.manual_seed(s)`` reseeds the engine like it reseeds the reference's CPU generator, and so that ranks /
    DataParallel replica threads do not draw identical noise.  ``manual_seed`` pins an explicit seed instead
    (same value on every rank = same noise on every rank, which is what MC sharding wants: see mc.py)."""

    def __init__(self):
        self.index = next(_instances)
        self.explicit = False
        self.seed = None
        self.torch_seed = None
        self.counter = 0
        self.queue = None          # external-eps queue (parity mode)
        self.base = None           # device int64[1] stream base (CUDA-graph capture mode)

    def current_seed(self) -> int:
        if not self.explicit:
            ts = torch.initial_seed()
            if self.seed is None or ts != self.torch_seed:      # first use, or torch.manual_seed() was called since
                self.torch_seed = ts
                mix = (ts * 0x9E3779B97F4A7C15 + _rank() * 0xD1B54A32D192ED03 + self.index * 0x94D049BB133111EB
                       + 0x5EEDB200) & _MASK64
                self.seed, self.counter = mix, 0
        return self.seed


_noise = _Noise()


def manual_seed(seed: int, counter: int = 0):
    """Seed the engine's Philox streams.  Every stochastic layer call consumes one
    stream id (counter += 1), so a fixed seed replays the same noise."""
    _noise.explicit = True
    _noise.seed = int(seed) & _MASK64
    _noise.counter = int(counter)


def current_seed() -> int:
    return _noise.current_seed()


def begin_sample(sample_id: int):
    """Position the stream counter for Monte-Carlo sample `sample_id` (global id):
    layer calls of that sample use stream ids (sample_id << 32) + 0, 1, 2, ...  so
    results do not depend on how samples are sharded over ranks (SURVEY.md 8e).
    Moves the calling thread's counter for good: prefer the ``mc_sample`` context manager,
    which restores the training counter afterwards."""
    _noise.counter = int(sample_id) << 32


@contextlib.contextmanager
def mc_sample(sample_id: int, seed: Optional[int] = None, offset: int = 0):
    """Layer calls inside draw Monte-Carlo evaluation sample `sample_id` (global id): stream ids
    2^63 + (sample_id << 40) + 0, 1, 2, ... (2^40 ids per sample: room for 2^20 CUDA-graph replays of 2^20 layer calls)
    -- a namespace training never reaches, independent of how the samples are sharded over ranks.  The thread's training counter (and seed) are restored on exit, so an evaluation pass
    between epochs does not make training replay its noise."""
    _noise.current_seed()
    saved = (_noise.seed, _noise.counter, _noise.explicit)
    if seed is not None:
        _noise.seed, _noise.explicit = int(seed) & _MASK64, True
    _noise.counter = (_MC_NAMESPACE | (int(sample_id) << 40)) + int(offset)     # offset: e.g. training step * 2^20
    try:
        yield
    finally:
        _noise.seed, _noise.counter, _noise.explicit = saved


@contextlib.contextmanager
def stream_base(base: Optional[torch.Tensor]):
    """Graph-capture mode: layer calls inside take stream ids 0, 1, 2, ... RELATIVE to
    the device scalar `base` (int64[1]), which kernels read at run time; advancing it
    (bbb_noise_advance, captured in the graph) gives every replay fresh noise."""
    prev, prev_ctr = _noise.base, _noise.counter
    _noise.base = base
    _noise.counter = 0
    try:
        yield
    finally:
        _noise.base, _noise.counter = prev, prev_ctr


def noise_advance(base: torch.Tensor, inc: int):
    rc = L.lib().bbb_noise_advance(_ptr(base), C.c_uint64(inc), _stream(base.device))
    L.check(rc, "bbb_noise_advance")


def next_stream() -> tuple[int, int]:
    seed = _noise.current_seed()
    s = _noise.counter
    _noise.counter += 1
    return seed, s


def noise_snapshot():
    """(counter, eps queue) -- lets a multi-layer caller roll the noise state back if it fails half-way."""
    return _noise.counter, (list(_noise.queue) if _noise.queue is not None else None)


def noise_restore(snap):
    _noise.counter = snap[0]
    if snap[1] is not None and _noise.queue is not None:
        _noise.queue[:] = snap[1]


@contextlib.contextmanager
def external_eps(tensors: Iterable[torch.Tensor]):
    """Parity mode: feed the layers the eps tensors the reference drew, in the
    reference's draw order (BBB: W_eps then bias_eps per layer -- BBB/BBBConv.py:63,68;
    LRT: one activation-shaped eps per layer -- BBB_LRT/BBBConv.py:78)."""
    prev = _noise.queue
    _noise.queue = list(tensors)
    try:
        yield
        if _noise.queue:
            raise RuntimeError(f"external_eps: {len(_noise.queue)} eps tensors were not consumed")
    finally:
        _noise.queue = prev


def _pop_eps(shape, device):
    q = _noise.queue
    if q is None:
        return None
    if not q:
        raise RuntimeError("external_eps: queue exhausted")
    e = q.pop(0)
    if tuple(e.shape) != tuple(shape):
        raise RuntimeError(f"external_eps: expected shape {tuple(shape)}, got {tuple(e.shape)}")
    return e.to(device=device, dtype=torch.float32).contiguous()


def external_eps_active() -> bool:
    return _noise.queue is not None


def draw_noise(variant, w_shape, b_shape, y_shape, device):
    """(eps_a, eps_b, seed, stream_id, base) of one stochastic layer call.  Under ``external_eps`` it pops the
    reference's draws (BBB: the weight eps, then the bias eps if ``b_shape`` is not None; LRT: one eps of the output
    shape ``y_shape``); otherwise it takes the next Philox stream id (relative to the ``stream_base`` scalar, if any)."""
    if not external_eps_active():
        seed, stream_id = next_stream()
        return None, None, seed, stream_id, _noise.base
    if variant == L.VARIANT_LRT:
        return _pop_eps(y_shape, device), None, 0, 0, None
    eps_a = _pop_eps(w_shape, device)
    eps_b = _pop_eps(b_shape, device) if b_shape is not None else None
    return eps_a, eps_b, 0, 0, None


# --------------------------------------------------------------------------- #
# helpers
# --------------------------------------------------------------------------- #
def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise L.EngineError(
            f"{what}: tensor is on {t.device}; the Bayesian layer engine runs on CUDA (sm_100a) only "
            "and has no CPU fallback")


_ws_cache: dict = {}                              # shared scratch: (device, stream) -> buffer
_ws_layer = weakref.WeakKeyDictionary()           # layer-private scratch: module -> {(device, slot): buffer}; dies with the layer
_ws_slot = 0


def current_workspace_slot() -> int:
    return _ws_slot


@contextlib.contextmanager
def workspace_slot(k: int):
    """Layer workspaces (prepared operand tiles, KL partials and counters) are private per (layer, slot).
    Forwards that may run CONCURRENTLY -- e.g. two captured graphs replayed on two streams -- must be built
    under different slots; everything on one stream can share slot 0 (the default)."""
    global _ws_slot
    prev, _ws_slot = _ws_slot, int(k)
    try:
        yield
    finally:
        _ws_slot = prev


def workspace(device, desc=None, owner=None) -> torch.Tensor:
    """Zero-initialised scratch.  Without `owner`: one per (device, stream) -- calls on
    one stream are ordered, so sharing is safe and the kernels leave the counters
    zeroed.  With `owner` (a layer module): a private buffer sized by bbb_workspace_bytes(desc),
    which on the tcgen05 path also holds that layer's prepared bf16 operand tiles; it is held
    through a weak reference to the layer, so it is freed with it and never re-bound to another one."""
    n = int(L.lib().bbb_workspace_bytes(C.byref(desc) if desc is not None else None))
    if owner is None:
        cache, key = _ws_cache, (device.index, torch.cuda.current_stream(device).cuda_stream)
    else:
        cache = _ws_layer.get(owner)
        if cache is None:
            cache = _ws_layer[owner] = {}
        key = (device.index, _ws_slot)
    ws = cache.get(key)
    if ws is None or ws.numel() < n:
        ws = torch.zeros(n, dtype=torch.uint8, device=device)
        cache[key] = ws
    return ws


def make_desc(x_shape, w_shape, conv, variant, sample, has_bias, prior_mu, prior_sigma,
              math=L.MATH_FP32, kl_convention=L.KL_REFERENCE, act=L.ACT_NONE,
              act_dtype=L.DTYPE_F32, pool=False, phase=0, fold=None) -> L.LayerDesc:
    """The bbb_layer_desc of one layer call.  ``pool``: fused 2x2 max-pool epilogue; ``phase``: 0, FUSED_PREP_ONLY or
    FUSED_SKIP_PREP; ``fold`` = (rows per MC sample, Philox stream stride) when MC samples are folded into the batch
    (include/bbb_b200.h)."""
    d = L.LayerDesc()
    if conv is None:
        d.batch, d.in_channels, d.in_h, d.in_w = x_shape[0], x_shape[1], 1, 1
        d.out_channels, d.kernel_h, d.kernel_w = w_shape[0], 1, 1
        d.stride_h = d.stride_w = d.dil_h = d.dil_w = 1
        d.pad_h = d.pad_w = 0
    else:
        (sh, sw), (ph, pw), (dh, dw) = conv
        d.batch, d.in_channels, d.in_h, d.in_w = x_shape
        d.out_channels, _, d.kernel_h, d.kernel_w = w_shape
        d.stride_h, d.stride_w, d.pad_h, d.pad_w, d.dil_h, d.dil_w = sh, sw, ph, pw, dh, dw
    d.variant, d.sample, d.has_bias = variant, int(bool(sample)), int(bool(has_bias))
    d.act_dtype, d.math, d.kl_convention, d.epilogue_act = act_dtype, math, kl_convention, act
    d.pool_k = d.pool_s = 2 if pool else 0
    d.reserved[0] = phase
    if fold is not None:
        rows, stride = fold
        d.reserved[1] = int(rows)
        d.reserved[2] = C.c_int32(stride & 0xFFFFFFFF).value
        d.reserved[3] = C.c_int32((stride >> 32) & 0xFFFFFFFF).value
    d.prior_mu, d.prior_sigma = float(prior_mu), float(prior_sigma)
    return d


def out_hw(h, w, kh, kw, conv):
    (sh, sw), (ph, pw), (dh, dw) = conv
    return ((h + 2 * ph - dh * (kh - 1) - 1) // sh + 1, (w + 2 * pw - dw * (kw - 1) - 1) // sw + 1)


# --------------------------------------------------------------------------- #
# tensor-core backward: wgrad / dgrad as role-swapped calls of the tcgen05 layer kernel
# --------------------------------------------------------------------------- #
_TC_K_MAX = 8192          # the gather kernel keeps an 8-byte table entry per reduction index in shared memory


def _tc_contract(x, w, conv, math):
    """Plain (mean-only, bias-free) conv2d / linear of fp32 `x` with the fp32 tensor `w` on the tcgen05 layer kernel
    (`math`: bf16 or tf32 operands like the layer's forward, fp32 TMEM accumulators): the engine's forward with
    sample=0, no KL."""
    lib = L.lib()
    x, w = x.contiguous(), w.contiguous()
    d = make_desc(tuple(x.shape), tuple(w.shape), conv, L.VARIANT_BBB, False, False, 0.0, 1.0, math)
    if conv is None:
        y = torch.empty(x.shape[0], w.shape[0], dtype=torch.float32, device=x.device)
        fn = lib.bbb_linear_forward
    else:
        oh, ow = out_hw(x.shape[2], x.shape[3], w.shape[2], w.shape[3], conv)
        y = torch.empty(x.shape[0], w.shape[0], oh, ow, dtype=torch.float32, device=x.device)
        fn = lib.bbb_conv2d_forward
    ws = workspace(x.device, d)
    rc = fn(C.byref(d), _ptr(x), _ptr(w), _ptr(w), None, None, _ptr(y), None, None, None, None,
            C.c_uint64(0), C.c_uint64(0), None, _ptr(ws), C.c_size_t(ws.numel()), _stream(x.device))
    L.check(rc, "tcgen05 contraction (backward)")
    return y


def _tc_dgrad(g, w, conv, x_shape, math):
    """d x of y = conv(x, w): the full correlation of (zero-inserted) g with the flipped, channel-transposed kernel --
    itself a stride-1 convolution, so it runs on the same tcgen05 layer kernel."""
    if conv is None:
        return _tc_contract(g, w.t(), None, math)                         # [B,N] x [K,N]^T -> [B,K]
    (sh, sw), (ph, pw), (dh, dw) = conv
    kh, kw = w.shape[2], w.shape[3]
    H, W = x_shape[2], x_shape[3]
    OH, OW = g.shape[2], g.shape[3]
    qh, qw = dh * (kh - 1) - ph, dw * (kw - 1) - pw
    if qh < 0 or qw < 0:
        return None
    hup = H - (dh * (kh - 1) - 2 * ph)                # rows of the zero-inserted gradient map: hup + 2*qh - dh*(kh-1) == H
    wup = W - (dw * (kw - 1) - 2 * pw)
    if (sh, sw) != (1, 1) or hup != OH or wup != OW:
        gu = g.new_zeros(g.shape[0], g.shape[1], hup, wup)
        gu[:, :, 0:(OH - 1) * sh + 1:sh, 0:(OW - 1) * sw + 1:sw] = g
        g = gu
    wt = w.flip(2, 3).transpose(0, 1)
    return _tc_contract(g, wt, ((1, 1), (qh, qw), (dh, dw)), math)


def _tc_wgrad(x, g, conv, w_shape, math):
    """d w of y = conv(x, w): a convolution with the batch as the reduction ("channel") axis -- input x^T [C,B,H,W],
    kernel g^T [N,B,OH,OW], stride <-> dilation swapped -- on the tcgen05 layer kernel.  Deterministic (no atomics);
    the batch is cut so that the reduction index fits the kernel's shared-memory table and the partial results summed."""
    if conv is None:
        out = _tc_contract(x.t(), g.t(), None, math)                       # [K,B] x [N,B]^T -> [K,N]
        return out.t()
    (sh, sw), (ph, pw), (dh, dw) = conv
    kh, kw = w_shape[2], w_shape[3]
    B = x.shape[0]
    per = max(1, _TC_K_MAX // (g.shape[2] * g.shape[3]))
    acc = None
    for b0 in range(0, B, per):
        xt = x[b0:b0 + per].transpose(0, 1)
        gt = g[b0:b0 + per].transpose(0, 1)
        part = _tc_contract(xt, gt, ((dh, dw), (ph, pw), (sh, sw)), math)[:, :, :kh, :kw]
        acc = part if acc is None else acc + part
    return acc.transpose(0, 1)


def _tc_backward_ok(cfg):
    return cfg["math"] in (L.MATH_BF16_TC, L.MATH_AUTO, L.MATH_TF32_TC)


# --------------------------------------------------------------------------- #
# the layer op
# --------------------------------------------------------------------------- #
class BayesLayerFn(torch.autograd.Function):
    """(y, kl) = layer(x; W_mu, W_rho, bias_mu, bias_rho).  One fused kernel forward;
    backward = bbb_*_backward + bbb_kl_backward accumulating into the same grads."""

    @staticmethod
    def forward(ctx, x, W_mu, W_rho, bias_mu, bias_rho, cfg):
        lib = L.lib()
        _require_cuda(x, "BayesLayerFn")
        _require_cuda(W_mu, "BayesLayerFn (parameters)")
        dev = x.device
        conv = cfg["conv"]
        variant, sample = cfg["variant"], cfg["sample"]
        x = x.contiguous()
        if x.dtype != torch.float32:
            x = x.float()
        W_mu_c, W_rho_c = W_mu.contiguous(), W_rho.contiguous()
        has_bias = bias_mu is not None
        d = make_desc(tuple(x.shape), tuple(W_mu.shape), conv, variant, sample, has_bias,
                      cfg["prior_mu"], cfg["prior_sigma"], cfg["math"], cfg["kl_convention"], cfg["act"])
        if conv is None:
            if x.dim() != 2 or x.shape[1] != W_mu.shape[1]:
                raise L.EngineError(f"linear: x {tuple(x.shape)} vs weight {tuple(W_mu.shape)}")
            yshape = (x.shape[0], W_mu.shape[0])
        else:
            if x.dim() != 4 or x.shape[1] != W_mu.shape[1]:
                raise L.EngineError(f"conv2d: x {tuple(x.shape)} vs weight {tuple(W_mu.shape)}")
            oh, ow = out_hw(x.shape[2], x.shape[3], W_mu.shape[2], W_mu.shape[3], conv)
            yshape = (x.shape[0], W_mu.shape[0], oh, ow)
        y = torch.empty(yshape, dtype=torch.float32, device=dev)
        kl = torch.empty((), dtype=torch.float32, device=dev)
        eps_a, eps_b, seed, stream_id, base = (
            draw_noise(variant, W_mu.shape, bias_mu.shape if has_bias else None, yshape, dev) if sample
            else (None, None, 0, 0, None))
        need_grad = any(ctx.needs_input_grad[:5])      # grad mode is off inside Function.forward
        act_std = None
        if variant == L.VARIANT_LRT and sample and need_grad:
            act_std = torch.empty(yshape, dtype=torch.float32, device=dev)
        ws = workspace(dev, d, cfg.get("owner"))
        fn = lib.bbb_linear_forward if conv is None else lib.bbb_conv2d_forward
        rc = fn(C.byref(d), _ptr(x), _ptr(W_mu_c), _ptr(W_rho_c), _ptr(bias_mu), _ptr(bias_rho),
                _ptr(y), _ptr(kl), _ptr(act_std), _ptr(eps_a), _ptr(eps_b),
                C.c_uint64(seed), C.c_uint64(stream_id), _ptr(base), _ptr(ws), C.c_size_t(ws.numel()), _stream(dev))
        L.check(rc, "bbb_linear_forward" if conv is None else "bbb_conv2d_forward")
        ctx.cfg = cfg
        ctx.desc = d
        ctx.noise = (seed, stream_id, base)
        ctx.has_bias = has_bias
        ctx.save_for_backward(x, W_mu_c, W_rho_c, bias_mu, bias_rho, act_std, eps_a, eps_b)
        return y, kl

    @staticmethod
    def backward(ctx, gy, gkl):
        lib = L.lib()
        x, W_mu, W_rho, bias_mu, bias_rho, act_std, eps_a, eps_b = ctx.saved_tensors
        cfg, d = ctx.cfg, ctx.desc
        dev = x.device
        if cfg["act"] != L.ACT_NONE:
            raise L.EngineError("backward through a fused activation epilogue is not available")
        g_W_mu = torch.zeros_like(W_mu)
        g_W_rho = torch.zeros_like(W_rho)
        g_b_mu = torch.zeros_like(bias_mu) if ctx.has_bias else None
        g_b_rho = torch.zeros_like(bias_rho) if ctx.has_bias else None
        gx = None
        done = False
        if gy is not None and _tc_backward_ok(cfg):
            try:
                out = BayesLayerFn._backward_tc(ctx, gy.contiguous().float())
            except L.EngineError as e:
                if e.code != L.E_UNSUPPORTED:              # a shape the tcgen05 kernel does not take
                    raise
                out = None
            if out is not None:
                gx, gw_mu, gw_rho, gb_mu, gb_rho = out
                g_W_mu += gw_mu.reshape(g_W_mu.shape)
                g_W_rho += gw_rho.reshape(g_W_rho.shape)
                if ctx.has_bias:
                    g_b_mu += gb_mu
                    g_b_rho += gb_rho
                done = True
        if gy is not None and not done:
            gy = gy.contiguous().float()
            if ctx.needs_input_grad[0]:
                gx = torch.zeros_like(x)
            ws = workspace(dev)
            fn = lib.bbb_linear_backward if cfg["conv"] is None else lib.bbb_conv2d_backward
            seed, stream_id, base = ctx.noise
            rc = fn(C.byref(d), _ptr(x), _ptr(gy), _ptr(W_mu), _ptr(W_rho), _ptr(bias_mu), _ptr(bias_rho),
                    _ptr(act_std), _ptr(eps_a), _ptr(eps_b), C.c_uint64(seed), C.c_uint64(stream_id), _ptr(base),
                    _ptr(gx), _ptr(g_W_mu), _ptr(g_W_rho), _ptr(g_b_mu), _ptr(g_b_rho),
                    _ptr(ws), C.c_size_t(ws.numel()), _stream(dev))
            L.check(rc, "bbb_*_backward")
        if gkl is not None:
            gkl = gkl.contiguous().float()
            rc = lib.bbb_kl_backward(_ptr(W_mu), _ptr(W_rho), C.c_uint64(W_mu.numel()),
                                     C.c_float(cfg["prior_mu"]), C.c_float(cfg["prior_sigma"]),
                                     C.c_int32(cfg["kl_convention"]), _ptr(gkl), _ptr(g_W_mu), _ptr(g_W_rho),
                                     _stream(dev))
            L.check(rc, "bbb_kl_backward")
            if ctx.has_bias:
                rc = lib.bbb_kl_backward(_ptr(bias_mu), _ptr(bias_rho), C.c_uint64(bias_mu.numel()),
                                         C.c_float(cfg["prior_mu"]), C.c_float(cfg["prior_sigma"]),
                                         C.c_int32(cfg["kl_convention"]), _ptr(gkl), _ptr(g_b_mu), _ptr(g_b_rho),
                                         _stream(dev))
                L.check(rc, "bbb_kl_backward")
        return gx, g_W_mu, g_W_rho, g_b_mu, g_b_rho, None


    @staticmethod
    def _backward_tc(ctx, gy):
        """SURVEY.md Appendix A on the tensor cores: every contraction of the backward (wgrad of the mean and of the
        variance path, dgrad of both) is a call of the tcgen05 layer kernel with the operands' roles swapped; eps is
        regenerated from the forward's Philox stream; the element-wise chain rule through sigma = softplus(rho) is
        parameter-sized glue.  Returns None when a shape does not fit (the caller then uses the CUDA-core kernels)."""
        x, W_mu, W_rho, bias_mu, bias_rho, act_std, eps_a, eps_b = ctx.saved_tensors
        cfg = ctx.cfg
        conv, variant, sample = cfg["conv"], cfg["variant"], cfg["sample"]
        dev = x.device
        math = L.MATH_TF32_TC if cfg["math"] == L.MATH_TF32_TC else L.MATH_BF16_TC      # same operand type as the forward
        seed, stream_id, base = ctx.noise
        if base is not None:
            stream_id = int(stream_id) + int(base.item())
        need_x = ctx.needs_input_grad[0]
        sig = torch.log1p(torch.exp(W_rho))
        dsig = torch.sigmoid(W_rho)
        gb_mu = gb_rho = None
        red = (0,) if conv is None else (0, 2, 3)
        if variant == L.VARIANT_LRT:
            gw_mu = _tc_wgrad(x, gy, conv, W_mu.shape, math)
            if sample:
                if eps_a is None:
                    z = philox_normal(gy.numel(), seed, stream_id, 0, device=dev)
                    eps = z.view(gy.shape) if conv is None else z.view(gy.shape[0], gy.shape[2], gy.shape[3], gy.shape[1]).permute(0, 3, 1, 2)
                else:
                    eps = eps_a
                gv = gy * eps / (2.0 * act_std)
                gw_rho = _tc_wgrad(x * x, gv, conv, W_mu.shape, math) * (2.0 * sig * dsig)
            else:
                gv, gw_rho = None, torch.zeros_like(W_rho)
            gx = None
            if need_x:
                gx = _tc_dgrad(gy, W_mu, conv, x.shape, math)
                if gx is None:
                    return None
                if sample:
                    gx2 = _tc_dgrad(gv, sig * sig, conv, x.shape, math)
                    gx = gx + 2.0 * x * gx2
            if ctx.has_bias:
                gb_mu = gy.sum(red)
                if sample:
                    sb = torch.log1p(torch.exp(bias_rho))
                    gb_rho = gv.sum(red) * (2.0 * sb * torch.sigmoid(bias_rho))
                else:
                    gb_rho = torch.zeros_like(bias_rho)
        else:
            nw = W_mu.numel()
            if sample:
                ew = eps_a if eps_a is not None else philox_normal(nw, seed, stream_id, 0, device=dev).view(W_mu.shape)
                W = W_mu + ew * sig
            else:
                ew, W = None, W_mu
            gw_mu = _tc_wgrad(x, gy, conv, W_mu.shape, math)
            gw_rho = gw_mu.reshape(W_mu.shape) * ew * dsig if sample else torch.zeros_like(W_rho)
            gx = None
            if need_x:
                gx = _tc_dgrad(gy, W, conv, x.shape, math)
                if gx is None:
                    return None
            if ctx.has_bias:
                gb_mu = gy.sum(red)
                if sample:
                    eb = eps_b if eps_b is not None else philox_normal(bias_mu.numel(), seed, stream_id, nw, device=dev)
                    gb_rho = gb_mu * eb * torch.sigmoid(bias_rho)
                else:
                    gb_rho = torch.zeros_like(bias_rho)
        return gx, gw_mu, gw_rho, gb_mu, gb_rho


class KLFn(torch.autograd.Function):
    """kl_loss() with no preceding forward: sigma recomputed from rho in the kernel."""

    @staticmethod
    def forward(ctx, W_mu, W_rho, bias_mu, bias_rho, prior_mu, prior_sigma, kl_convention):
        lib = L.lib()
        _require_cuda(W_mu, "kl_loss")
        dev = W_mu.device
        W_mu_c, W_rho_c = W_mu.contiguous(), W_rho.contiguous()
        kl = torch.empty((), dtype=torch.float32, device=dev)
        ws = workspace(dev)
        nb = 0 if bias_mu is None else bias_mu.numel()
        rc = lib.bbb_kl_forward(_ptr(W_mu_c), _ptr(W_rho_c), C.c_uint64(W_mu.numel()), _ptr(bias_mu), _ptr(bias_rho),
                                C.c_uint64(nb), C.c_float(prior_mu), C.c_float(prior_sigma), C.c_int32(kl_convention),
                                _ptr(kl), _ptr(ws), C.c_size_t(ws.numel()), _stream(dev))
        L.check(rc, "bbb_kl_forward")
        ctx.save_for_backward(W_mu_c, W_rho_c, bias_mu, bias_rho)
        ctx.cfg = (float(prior_mu), float(prior_sigma), int(kl_convention))
        return kl

    @staticmethod
    def backward(ctx, gkl):
        lib = L.lib()
        W_mu, W_rho, bias_mu, bias_rho = ctx.saved_tensors
        pm, ps, conv = ctx.cfg
        dev = W_mu.device
        gkl = gkl.contiguous().float()
        out = []
        for mu, rho in ((W_mu, W_rho), (bias_mu, bias_rho)):
            if mu is None:
                out += [None, None]
                continue
            g_mu, g_rho = torch.zeros_like(mu), torch.zeros_like(rho)
            rc = lib.bbb_kl_backward(_ptr(mu), _ptr(rho), C.c_uint64(mu.numel()), C.c_float(pm), C.c_float(ps),
                                     C.c_int32(conv), _ptr(gkl), _ptr(g_mu), _ptr(g_rho), _stream(dev))
            L.check(rc, "bbb_kl_backward")
            out += [g_mu, g_rho]
        return out[0], out[1], out[2], out[3], None, None, None


# --------------------------------------------------------------------------- #
# small direct wrappers
# --------------------------------------------------------------------------- #
def philox_normal(n: int, seed: int, stream_id: int, offset: int = 0, device="cuda") -> torch.Tensor:
    """The engine's own noise stream, drawn on the host side of the boundary."""
    out = torch.empty(n, dtype=torch.float32, device=device)
    rc = L.lib().bbb_philox_normal_fill(_ptr(out), C.c_uint64(n), C.c_uint64(seed), C.c_uint64(stream_id),
                                        C.c_uint64(offset), _stream(out.device))
    L.check(rc, "bbb_philox_normal_fill")
    return out


def mc_combine(logits: torch.Tensor, want_moments: bool = False):
    """logits [S,B,C] -> log_outputs [B,C] (main_bayesian.py:46-53) and optionally the
    [3,B,C] sums (softmax, softmax^2, logits) for uncertainty_estimation.py:70-96."""
    _require_cuda(logits, "mc_combine")
    logits = logits.contiguous().float()
    S, B, Cc = logits.shape
    out = torch.empty(B, Cc, dtype=torch.float32, device=logits.device)
    mom = torch.empty(3, B, Cc, dtype=torch.float32, device=logits.device) if want_moments else None
    rc = L.lib().bbb_mc_combine(_ptr(logits), S, B, Cc, _ptr(out), _ptr(mom), _stream(logits.device))
    L.check(rc, "bbb_mc_combine")
    return (out, mom) if want_moments else out
