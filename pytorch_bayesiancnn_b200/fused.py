"""Fused execution of a ModuleWrapper's children (SURVEY.md 8f row f2).

The reference's model files interleave the Bayesian layers with ``nn.Softplus`` /
``nn.ReLU``, ``nn.MaxPool2d(2, 2)`` and ``FlattenLayer`` children
(BayesianAlexNet.py:34-53).  ``ModuleWrapper.forward`` (layers/misc.py:16-18) just
calls them in order; here the same child list is pattern-matched into runs of
``[Bayesian layer, activation?, 2x2 max-pool?, flatten*]`` and each run becomes ONE
``bbb_layer_forward_fused`` call (weight-prep kernel + tcgen05 GEMM kernel whose
epilogue applies the activation and the pool and writes the packed bf16 format the
next layer's TMA loads).  The model files stay unmodified; anything that does not
match (other pools, other modules, autograd needed) falls back to the plain
child-by-child path.
"""
from __future__ import annotations

import ctypes as C

import torch
from torch import nn

from . import _lib as L
from . import functional as Fn


class _Step:
    __slots__ = ("layer", "act", "pool", "conv", "in_shape", "in_layout", "prev_hw", "out_layout", "out_chw",
                 "eps_shape", "linear", "batch")

    def desc(self, phase=0, fold=None):
        """The layer call's descriptor (ModuleWrapper calls its children with sample=True: SURVEY D6)."""
        m = self.layer
        return Fn.make_desc((self.batch,) + self.in_shape, tuple(m.W_mu.shape), self.conv, m._variant, True,
                            m.use_bias, m.prior_mu, m.prior_sigma, L.MATH_BF16_TC, L.KL_BY_NAME[m.kl_convention],
                            self.act, pool=self.pool, phase=phase, fold=fold)

    def noise(self):
        """The layer call's noise, drawn exactly as the per-layer path draws it."""
        m, (cout, oh, ow) = self.layer, self.eps_shape
        y_shape = (self.batch, cout) if self.linear else (self.batch, cout, oh, ow)
        return Fn.draw_noise(m._variant, m.W_mu.shape, m.bias_mu.shape if m.use_bias else None, y_shape,
                             m.W_mu.device)


def _act_code(m):
    if isinstance(m, nn.Softplus) and m.beta == 1 and m.threshold == 20:
        return L.ACT_SOFTPLUS
    if isinstance(m, nn.ReLU):
        return L.ACT_RELU
    return None


def _is_pool22(m):
    def two(v):
        return v == 2 or v == (2, 2)
    return (isinstance(m, nn.MaxPool2d) and two(m.kernel_size) and two(m.stride) and m.padding in (0, (0, 0))
            and m.dilation in (1, (1, 1)) and not m.ceil_mode and not m.return_indices)


def plan(children, x_shape, fold=None):
    """Return the list of fused steps for this child list and input shape, or None.
    ``fold`` = (rows per MC sample, Philox stream stride): x_shape[0] is then the FOLDED batch (samples x rows)."""
    from .modules import _BayesLayer, FlattenLayer
    if len(x_shape) != 4:
        return None
    batch, c, h, w = x_shape
    state = ("nchw", c, h, w)
    steps = []
    i, n = 0, len(children)
    while i < n:
        m = children[i]
        if not isinstance(m, _BayesLayer) or m.math not in ("bf16", "auto"):
            return None
        st = _Step()
        st.layer = m
        st.batch = batch
        st.conv = m._conv_geometry()
        st.linear = st.conv is None
        lay, c, h, w = state
        if st.linear:
            if lay != "packed" or m.in_features != c * h * w:
                return None
            st.prev_hw = h * w
            st.in_shape = (c * h * w, 1, 1)
            cout, oh, ow = m.out_features, 1, 1
        else:
            if m.in_channels != c:
                return None
            if st.conv[2] != (1, 1):            # dilation
                return None
            oh, ow = Fn.out_hw(h, w, *m.kernel_size, st.conv)
            if oh < 1 or ow < 1:
                return None
            if lay == "packed" and (h * w > 64 or c % 64):
                return None
            st.prev_hw = 1
            st.in_shape = (c, h, w)
            cout = m.out_channels
        st.in_layout = L.LAYOUT_NCHW_F32 if lay == "nchw" else L.LAYOUT_PACKED_BF16
        st.eps_shape = (cout, oh, ow)
        i += 1
        st.act = L.ACT_NONE
        if i < n and _act_code(children[i]) is not None:
            st.act = _act_code(children[i])
            i += 1
        st.pool = False
        if i < n and isinstance(children[i], nn.MaxPool2d):
            if not _is_pool22(children[i]) or st.linear or oh % 2 or ow % 2:
                return None
            st.pool = True
            oh, ow = oh // 2, ow // 2
            i += 1
        while i < n and isinstance(children[i], FlattenLayer):
            if children[i].num_features != cout * oh * ow:
                return None            # the reference's view(-1, F) would fold the batch (SURVEY D2): not fused
            i += 1
        st.out_chw = (cout, oh, ow)
        state = ("packed", cout, oh, ow)
        steps.append(st)
    if not steps:
        return None
    last = steps[-1]
    last.out_layout = L.LAYOUT_ROWMAJOR_F32 if last.out_chw[1] * last.out_chw[2] == 1 else L.LAYOUT_NCHW_F32
    for st in steps[:-1]:
        st.out_layout = L.LAYOUT_PACKED_BF16
        if st.out_chw[0] % 64:                  # tiled packed format: whole 64-channel blocks per pixel
            return None
    # the engine has the last word (same checks bbb_layer_forward_fused makes, host-only): run() must not
    # discover an unsupported shape after noise was drawn and prep kernels were enqueued on side streams
    lib = L.lib()
    for st in steps:
        d = st.desc(fold=fold)
        rc = lib.bbb_fused_supported(C.byref(d), st.in_layout, _in_pitch(st), st.prev_hw, st.out_layout, _out_pitch(st))
        if rc == L.E_UNSUPPORTED:               # not fusable, the caller runs child by child
            return None
        L.check(rc, "bbb_fused_supported")
    return steps


def _in_pitch(st):
    cin, h, w = st.in_shape
    return 0 if st.in_layout == L.LAYOUT_NCHW_F32 else cin * h * w


def _out_pitch(st):
    cout, oh, ow = st.out_chw
    return cout * oh * ow if st.out_layout == L.LAYOUT_PACKED_BF16 else 0


_side_streams: dict = {}
_direct: dict = {}                  # run()'s keyword arguments inside a direct_output block


class direct_output:
    """``with fused.direct_output(buf): logits, kls = net(x)`` -- a fused chain entered inside writes its final fp32
    logits straight into ``buf`` ([B, C], contiguous) and returns the per-layer KL scalars UN-summed (the caller's
    kernel sums them: bbb_mc_exchange), so the Monte-Carlo step has no copy and no aten reduction behind the chain.
    ``.used`` tells whether a fused chain really took the buffer (non-fusable nets ignore the hook)."""

    def __init__(self, out, kl_buf=None):
        """``kl_buf``: optional fp32 device vector the per-layer KL scalars are written to (its first n entries are
        returned) instead of a tensor allocated by the chain -- a stable address for a kernel captured separately."""
        self.out, self.used, self.kl_buf = out, False, kl_buf

    def __enter__(self):
        self.prev = dict(_direct)
        _direct.update(out=self.out, terms=True, owner=self, kls_out=self.kl_buf)
        return self

    def __exit__(self, *exc):
        _direct.clear()
        _direct.update(self.prev)
        return False


def _side_stream(dev, i=0):
    st = _side_streams.get((dev.index, i))
    if st is None:
        st = _side_streams[(dev.index, i)] = torch.cuda.Stream(device=dev)
    return st


_PREP_CHAINS = 3        # serial side streams the parameter preps are dealt over (see run)


def run(steps, x: torch.Tensor, *, out=None, terms=False, owner=None, fold=None, kls_out=None):
    """Execute a planned chain.  Returns (network output fp32, summed KL 0-dim tensor); with ``terms`` the per-layer
    KL scalars un-summed instead of their sum, and ``owner.used`` is set.  ``out``: a [B, C] fp32 buffer the last
    layer writes its output into when it can; ``fold``: as in plan(); ``kls_out``: a vector the per-layer KL scalars
    are written to.  ``ModuleWrapper`` passes the keywords of the enclosing ``direct_output`` block.

    The parameter-only half of every layer (softplus / eps / bf16 operand tiles / KL) runs on side
    streams (parallel branches of a captured graph), joined to the GEMM chain by events, so only the
    first layer's prep is on the activation critical path.  The preps are issued in layer order over
    a few serial chains (3: layers 1,4 / 2,5 / 3) rather than all at once: six concurrent prep
    grids fill the machine and the first layer's prep -- the one the GEMM chain is waiting for -- was
    scheduled last (measured with tools/timeline.py: first GEMM at 24 us instead of ~20).  The KL sum
    depends on the preps only and runs on the side as well."""
    dev = x.device
    kls = kls_out[:len(steps)] if kls_out is not None else torch.empty(len(steps), dtype=torch.float32, device=dev)
    snap = Fn.noise_snapshot()
    main = torch.cuda.current_stream(dev)
    chains = [_side_stream(dev, c) for c in range(min(_PREP_CHAINS, len(steps)))]
    forked = False
    try:
        if fold is not None and Fn.external_eps_active():
            raise L.EngineError("MC-sample folding draws its noise in-kernel (no external eps)")
        noise = [st.noise() for st in steps]
        for side in chains:
            side.wait_stream(main)
        forked = True
        # The FIRST layer's prep stays on the main stream, right in front of its GEMM kernel: launched with programmatic
        # serialization the GEMM kernel's CTAs start while the prep runs and stage their input images meanwhile
        # (conv_s4_tc.cuh); only its weight producer waits for the prep.  The other preps go to the side chains.
        events = [None] * len(steps)
        run_step(steps[0], None, None, None, 0, kl=kls[0], noise=noise[0], phase=L.FUSED_PREP_ONLY, fold=fold)
        ev0 = torch.cuda.Event()
        ev0.record(main)
        for i in range(1, len(steps)):
            side = chains[(i - 1) % len(chains)]
            with torch.cuda.stream(side):
                run_step(steps[i], None, None, None, 0, kl=kls[i], noise=noise[i], phase=L.FUSED_PREP_ONLY, fold=fold)
                ev = torch.cuda.Event()
                ev.record(side)
                events[i] = ev
        for side in chains[1:]:
            chains[0].wait_stream(side)
        if not terms:
            with torch.cuda.stream(chains[0]):
                chains[0].wait_event(ev0)
                kl_total = kls.sum()
        cur, cur_sq, cur_pitch = x.contiguous().float(), None, 0
        last = steps[-1]
        take = (out is not None and last.out_layout == L.LAYOUT_ROWMAJOR_F32 and out.is_contiguous()
                and out.dtype == torch.float32 and tuple(out.shape) == (last.batch, last.out_chw[0]))
        for i, st in enumerate(steps):
            nxt = steps[i + 1].layer if i + 1 < len(steps) else None
            y_into = out if (take and i == len(steps) - 1) else None
            if events[i] is not None:
                main.wait_event(events[i])
            cur, cur_sq, cur_pitch = run_step(st, nxt, cur, cur_sq, cur_pitch, kl=kls[i], noise=noise[i],
                                              phase=L.FUSED_SKIP_PREP, y_into=y_into, fold=fold)
        if terms:
            kl_total = kls
            if owner is not None:
                owner.used = True
    except BaseException:
        Fn.noise_restore(snap)                 # a retry / fallback sees the stream ids and eps queue it would have seen
        raise
    finally:
        if forked:                             # ALWAYS re-join the forked side streams: `kls` and the layer workspaces are
            for side in chains[1:]:            # written there, and an active graph capture must not be left with dangling forks
                chains[0].wait_stream(side)
            main.wait_stream(chains[0])
    return cur, kl_total


def run_step(st, nxt, cur, cur_sq, cur_pitch, kl=None, noise=None, phase=0, y_into=None, fold=None):
    """One fused layer call: (y, y_sq, pitch) = step(cur, cur_sq).  phase: 0 = prep + GEMM,
    FUSED_PREP_ONLY / FUSED_SKIP_PREP = one half (see include/bbb_b200.h)."""
    lib = L.lib()
    m = st.layer
    dev = m.W_mu.device
    B = st.batch                                    # (packed inputs carry rows padded to the 128-row tile)
    cin, h, w = st.in_shape
    d = st.desc(phase, fold)
    in_pitch = cur_pitch if st.in_layout == L.LAYOUT_NCHW_F32 else cin * h * w
    cout, oh, ow = st.out_chw
    if phase == L.FUSED_PREP_ONLY:
        pitch, y, y_sq = cout * oh * ow if st.out_layout == L.LAYOUT_PACKED_BF16 else 0, None, None
    elif st.out_layout == L.LAYOUT_PACKED_BF16:
        pitch = cout * oh * ow                   # tiled packed: [ceil(B/128)][F/64][planes][128 x 64] bf16
        planes = 2 if (nxt is not None and nxt._variant == L.VARIANT_LRT) else 1
        y = torch.empty((B + 127) // 128 * 128, pitch * planes, dtype=torch.bfloat16, device=dev)
        y_sq = y.view(-1)[128 * 64:] if planes == 2 else None      # x^2 blocks interleaved behind the x blocks
    elif st.out_layout == L.LAYOUT_ROWMAJOR_F32:
        pitch, y, y_sq = 0, (y_into if y_into is not None else torch.empty(B, cout, dtype=torch.float32, device=dev)), None
    else:
        pitch, y, y_sq = 0, torch.empty(B, cout, oh, ow, dtype=torch.float32, device=dev), None
    if kl is None:
        kl = torch.empty((), dtype=torch.float32, device=dev)
    if noise is None:
        noise = st.noise()
    eps_a, eps_b, seed, stream_id, base = noise
    ws = Fn.workspace(dev, d, m)
    rc = lib.bbb_layer_forward_fused(
        C.byref(d), Fn._ptr(cur), Fn._ptr(cur_sq), st.in_layout, in_pitch, st.prev_hw,
        Fn._ptr(m.W_mu), Fn._ptr(m.W_rho), Fn._ptr(m.bias_mu), Fn._ptr(m.bias_rho),
        Fn._ptr(y), Fn._ptr(y_sq), st.out_layout, pitch, Fn._ptr(kl), Fn._ptr(eps_a), Fn._ptr(eps_b),
        C.c_uint64(seed), C.c_uint64(stream_id), Fn._ptr(base), Fn._ptr(ws), C.c_size_t(ws.numel()),
        Fn._stream(dev))
    L.check(rc, "bbb_layer_forward_fused")
    if phase != L.FUSED_SKIP_PREP:
        m._kl_cache = (kl, m._versions(), torch.is_grad_enabled())
    return y, y_sq, pitch
