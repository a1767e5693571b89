"""The reference's layer surface (SURVEY.md 8b) on top of the CUDA engine.

Same class names, constructor signatures, parameter names (``W_mu``, ``W_rho``,
``bias_mu``, ``bias_rho`` -- the state_dict keys), ``forward(x, sample=True)``,
``kl_loss()``, ``reset_parameters()``, ``ModuleWrapper.set_flag`` and
``FlattenLayer`` as layers/BBB/BBBConv.py, layers/BBB/BBBLinear.py,
layers/BBB_LRT/BBBConv.py, layers/BBB_LRT/BBBLinear.py and layers/misc.py, so that
models/BayesianModels/*.py import and train unchanged.  The bodies are new: one
fused CUDA kernel per forward (through the C ABI), KL computed in that kernel.

Engine knobs ride on ``set_flag`` (never on the constructor):
  math           'fp32' | 'bf16' | 'tf32' | 'auto'   arithmetic path (default from $BBB_B200_MATH or 'auto': the tcgen05 tensor-core
                                            path wherever the shape fits a UMMA tile, IEEE-fp32 CUDA cores otherwise;
                                            'fp32' forces the exact-arithmetic kernels everywhere)
  kl_convention  'reference' | 'textbook'   default 'reference' = the formula as executed (SURVEY D1)
"""
from __future__ import annotations

import os

import torch
from torch import nn
from torch.nn import Parameter

from . import _lib as L
from . import functional as Fn

_DEFAULT_PRIORS = {
    "prior_mu": 0,
    "prior_sigma": 0.1,
    "posterior_mu_initial": (0, 0.1),
    "posterior_rho_initial": (-3, 0.1),
}


def _default_math() -> str:
    return os.environ.get("BBB_B200_MATH", "auto")


def _default_fuse() -> bool:
    return os.environ.get("BBB_B200_FUSE", "1") != "0"


class ModuleWrapper(nn.Module):
    """layers/misc.py:4-25: universal forward returning (x, kl); recursive set_flag."""

    def __init__(self):
        super().__init__()

    def set_flag(self, flag_name, value):
        setattr(self, flag_name, value)
        self.__dict__.pop("_fused_plans", None)          # engine knobs (math, fuse, ...) change what can be fused
        for child in self.children():
            if hasattr(child, "set_flag"):
                child.set_flag(flag_name, value)

    def _try_fused(self, x):
        """Run the children as a fused tcgen05 chain if they match (see fused.py); None = not fusable."""
        if not (torch.is_tensor(x) and x.is_cuda and x.dim() == 4) or not getattr(self, "fuse", _default_fuse()):
            return None
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            return None                                    # the fused chain is forward-only
        from . import fused
        plans = self.__dict__.setdefault("_fused_plans", {})
        key = tuple(x.shape)
        if key not in plans:
            kids = list(self.children())
            plans[key] = fused.plan(kids, tuple(x.shape)) if kids else None
        steps = plans[key]
        if steps is None:
            return None
        try:
            return fused.run(steps, x, **fused._direct)     # (output, summed KL)
        except L.EngineError as e:
            if e.code != L.E_UNSUPPORTED:                  # anything else is a real error
                raise
            plans[key] = None
            return None

    def forward(self, x):
        out = self._try_fused(x)
        if out is not None:
            # the fused chain already reduced the per-layer KL scalars (each layer's kl_loss() still
            # returns its own term); same value as the loop below, one launch instead of one per layer
            return out
        for child in self.children():
            x = child(x)
        kl = 0.0
        for m in self.modules():
            if hasattr(m, "kl_loss"):
                kl = kl + m.kl_loss()
        return x, kl


class FlattenLayer(ModuleWrapper):
    """layers/misc.py:28-35: x.view(-1, num_features) (no shape check, like the reference)."""

    def __init__(self, num_features):
        super().__init__()
        self.num_features = num_features

    def forward(self, x):
        return x.reshape(-1, self.num_features) if not x.is_contiguous() else x.view(-1, self.num_features)


def _pair(v):
    return tuple(v) if isinstance(v, (tuple, list)) else (v, v)


class _BayesLayer(ModuleWrapper):
    """Shared machinery of the four reference layer classes."""
    _variant = L.VARIANT_BBB
    _params_on_device = True       # BBB creates params on cuda:0 if present (BBB/BBBConv.py:27,41);
                                   # LRT on CPU (BBB_LRT/BBBConv.py:43-44) -- kept (SURVEY D12)

    def _setup(self, w_shape, n_out, bias, priors):
        self.use_bias = bias
        self.device = torch.device("cuda:0" if torch.cuda.is_available() else "cpu")
        if priors is None:
            priors = dict(_DEFAULT_PRIORS)
        self.prior_mu = priors["prior_mu"]
        self.prior_sigma = priors["prior_sigma"]
        self.posterior_mu_initial = priors["posterior_mu_initial"]
        self.posterior_rho_initial = priors["posterior_rho_initial"]
        dev = self.device if self._params_on_device else torch.device("cpu")
        self.W_mu = Parameter(torch.empty(w_shape, device=dev))
        self.W_rho = Parameter(torch.empty(w_shape, device=dev))
        if self.use_bias:
            self.bias_mu = Parameter(torch.empty(n_out, device=dev))
            self.bias_rho = Parameter(torch.empty(n_out, device=dev))
        else:
            self.register_parameter("bias_mu", None)
            self.register_parameter("bias_rho", None)
        self.math = _default_math()
        self.kl_convention = "reference"
        self._kl_cache = None
        self.reset_parameters()

    def reset_parameters(self):
        self.W_mu.data.normal_(*self.posterior_mu_initial)
        self.W_rho.data.normal_(*self.posterior_rho_initial)
        if self.use_bias:
            self.bias_mu.data.normal_(*self.posterior_mu_initial)
            self.bias_rho.data.normal_(*self.posterior_rho_initial)

    # -- engine plumbing ------------------------------------------------------
    def _conv_geometry(self):
        return None

    def _versions(self):
        """What a cached KL scalar depends on: the parameters' versions AND the KL settings (changing
        kl_convention or the prior after a forward must not return the old value)."""
        ps = (self.W_mu, self.W_rho, self.bias_mu, self.bias_rho)
        return tuple((p._version, p.data_ptr()) if p is not None else None for p in ps) + (
            self.kl_convention, float(self.prior_mu), float(self.prior_sigma))

    def _cfg(self, sample):
        return {
            "conv": self._conv_geometry(),
            "variant": self._variant,
            "sample": bool(sample),
            "prior_mu": float(self.prior_mu),
            "prior_sigma": float(self.prior_sigma),
            "math": L.MATH_BY_NAME[self.math],
            "kl_convention": L.KL_BY_NAME[self.kl_convention],
            "act": L.ACT_NONE,
            "owner": self,
        }

    def forward(self, x, sample=True):
        stochastic = bool(self.training or sample)      # BBB/BBBConv.py:62, BBB_LRT/BBBConv.py:77
        y, kl = Fn.BayesLayerFn.apply(x, self.W_mu, self.W_rho, self.bias_mu, self.bias_rho,
                                      self._cfg(stochastic))
        self._kl_cache = (kl, self._versions(), torch.is_grad_enabled())
        return y

    def kl_loss(self):
        """0-dim tensor, differentiable w.r.t. mu and rho.  Normally the scalar the
        fused forward kernel just produced; recomputed by the stand-alone KL kernel
        if no forward preceded it or the parameters changed since (the reference
        would raise AttributeError / use a stale sigma there -- SURVEY D7)."""
        c = self._kl_cache
        if c is not None and c[1] == self._versions() and (c[2] or not torch.is_grad_enabled()):
            return c[0]
        return Fn.KLFn.apply(self.W_mu, self.W_rho, self.bias_mu, self.bias_rho, float(self.prior_mu),
                             float(self.prior_sigma), L.KL_BY_NAME[self.kl_convention])

    @property
    def W_sigma(self):
        """The reference caches log1p(exp(W_rho)) as a forward side effect
        (BBB/BBBConv.py:64); kept as a read-only view for code that inspects it."""
        return torch.log1p(torch.exp(self.W_rho))

    @W_sigma.setter
    def W_sigma(self, value):
        pass                                             # the reference assigns it in forward; derived here

    @property
    def bias_sigma(self):
        return torch.log1p(torch.exp(self.bias_rho)) if self.use_bias else None

    @bias_sigma.setter
    def bias_sigma(self, value):
        pass


class _ConvMixin:
    def _init_conv(self, in_channels, out_channels, kernel_size, stride, padding, dilation, bias, priors):
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = _pair(kernel_size)
        self.stride = stride
        self.padding = padding
        self.dilation = dilation
        self.groups = 1
        self._setup((out_channels, in_channels, *self.kernel_size), out_channels, bias, priors)

    def _conv_geometry(self):
        return (_pair(self.stride), _pair(self.padding), _pair(self.dilation))


class BBBConv2d(_ConvMixin, _BayesLayer):
    """layers/BBB/BBBConv.py:14 -- weight-space sampling conv."""
    _variant = L.VARIANT_BBB

    def __init__(self, in_channels, out_channels, kernel_size,
                 stride=1, padding=0, dilation=1, bias=True, priors=None):
        super().__init__()
        self._init_conv(in_channels, out_channels, kernel_size, stride, padding, dilation, bias, priors)


class BBBLRTConv2d(_ConvMixin, _BayesLayer):
    """layers/BBB_LRT/BBBConv.py:16 -- local-reparameterisation conv."""
    _variant = L.VARIANT_LRT
    _params_on_device = False

    def __init__(self, in_channels, out_channels, kernel_size, stride=1,
                 padding=0, dilation=1, bias=True, priors=None):
        super().__init__()
        self._init_conv(in_channels, out_channels, kernel_size, stride, padding, dilation, bias, priors)


class _LinearMixin:
    def _init_linear(self, in_features, out_features, bias, priors):
        self.in_features = in_features
        self.out_features = out_features
        self._setup((out_features, in_features), out_features, bias, priors)


class BBBLinear(_LinearMixin, _BayesLayer):
    """layers/BBB/BBBLinear.py:14."""
    _variant = L.VARIANT_BBB

    def __init__(self, in_features, out_features, bias=True, priors=None):
        super().__init__()
        self._init_linear(in_features, out_features, bias, priors)


class BBBLRTLinear(_LinearMixin, _BayesLayer):
    """layers/BBB_LRT/BBBLinear.py:16."""
    _variant = L.VARIANT_LRT
    _params_on_device = False

    def __init__(self, in_features, out_features, bias=True, priors=None):
        super().__init__()
        self._init_linear(in_features, out_features, bias, priors)
