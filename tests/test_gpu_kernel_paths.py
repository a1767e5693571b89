"""Kernel paths that BBBAlexNet does not reach, against float64 references.

(A) The fused tcgen05 chain on synthetic child lists: the gather kernel's pooled packed epilogue, the NCHW-flatten
permutation of a linear layer fed by a map larger than 1x1 (prev_hw > 1), the stride-4 first-layer kernel with 1 and 4
input channels, another window and a tall input, the tap-GEMM on stride 2, 1x1 and non-square kernels, 64-pixel and
non-square maps, two linear steps in a row, and every launch configuration the tap-GEMM can select.  Each case runs
under the CFG priors (sigma ~ 0.0067) and under a noise-dominated set (sigma ~ 0.31 > |mu|), and is checked three ways:
against a float64 walk of the child list (the 1e-2 bf16 bar), against the same walk rounded to bf16 where the kernels
round (a tight bar: only the fp32 accumulation order differs), and in-kernel Philox against the same streams fed as
external eps.

(B) The tensor-core backward at model shapes: batch chunking of the wgrad (equal and ragged chunks), the stride-4
11x11 dgrad, the shapes that fall back to the CUDA-core kernels, each contraction alone against float64 of its
operands rounded the way the kernel rounds them, and the stream_base branch."""
import ctypes
from collections import namedtuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch import nn

from tests.util import CFG_PRIORS, scale_err
from tests.test_gpu_parity import _grad_case, _lrt_eps_like, dev  # noqa: F401  (fixture)

BF16_TOL = 1e-2
KL_TOL = 1e-5
NOISY_PRIORS = dict(CFG_PRIORS, posterior_rho_initial=(-1, 0.1))
PRIORS = {"cfg": CFG_PRIORS, "noisy": NOISY_PRIORS}

# bbb_debug_fused_config codes
S4, GATHER, TAP = 0, 1, 2
WEIGHT_PREP, S4_PREP, TAP_PREP, TAP_PREP_CONV = 0, 1, 2, 3


# --------------------------------------------------------------------------- #
# the case table
# --------------------------------------------------------------------------- #
def _conv(cin, cout, k, s=1, p=0):
    return ("conv", cin, cout, k, s, p)


def _lin(fin, fout):
    return ("lin", fin, fout)


def _flat(n):
    return ("flat", n)


RELU, SOFTPLUS, POOL = ("relu",), ("softplus",), ("pool",)

NET_GATHER = [_conv(3, 64, 3, 1, 1), RELU, POOL, _conv(64, 128, 3, 1, 1), RELU, POOL, _flat(512), _lin(512, 10)]
NET_HW64 = [_conv(3, 64, 3, 1, 1), SOFTPLUS, POOL, _conv(64, 64, 3, 2, 1), _conv(64, 128, 1), _flat(2048),
            _lin(2048, 100)]
NET_S4_CIN1 = [_conv(1, 64, 11, 4, 5), RELU, POOL, _conv(64, 128, 3, 1, 1), POOL, _flat(512), _lin(512, 10)]
NET_S4_CIN4 = [_conv(4, 64, 11, 4, 5), RELU, POOL, _conv(64, 64, 3, 1, 1), _flat(2048), _lin(2048, 10)]
NET_S4_K7 = [_conv(3, 64, 7, 4, 3), POOL, _conv(64, 64, 3, 1, 1), _flat(1024), _lin(1024, 10)]
NET_NONSQUARE = [_conv(3, 64, 3, 1, 1), POOL, _conv(64, 128, (3, 1), 1, (1, 0)), _flat(4096), _lin(4096, 10)]
NET_TWO_LINEARS = [_conv(3, 64, 3, 1, 1), POOL, _flat(1024), _lin(1024, 256), SOFTPLUS, _lin(256, 10)]
NET_ONE_STEP = [_conv(3, 64, 3, 1, 1), RELU, POOL]

# per step: (kernel, BN, CTAs per SM, pool, prep kernel) on a 148-SM B200
G_POOL = (GATHER, 64, 0, True, WEIGHT_PREP)
S4_POOL = (S4, 64, 1, True, S4_PREP)
LINEAR = (TAP, 64, 1, False, TAP_PREP)

Case = namedtuple("Case", "name net x_shape wide expect")
CASES = [
    Case("gather-pool-prevhw4-b129", NET_GATHER, (129, 3, 8, 8), False, [G_POOL, (TAP, 64, 1, True, TAP_PREP_CONV), LINEAR]),
    Case("gather-pool-prevhw4-b1", NET_GATHER, (1, 3, 8, 8), False, [G_POOL, (TAP, 64, 1, True, TAP_PREP_CONV), LINEAR]),
    # 160 CTAs of 64 columns: two per SM
    Case("gather-pool-prevhw4-b600", NET_GATHER, (600, 3, 8, 8), False, [G_POOL, (TAP, 64, 2, True, TAP_PREP_CONV), LINEAR]),
    # 96 CTAs of 128 columns cover 60 % of the SMs: the grid rule takes the wide tile
    Case("gather-pool-prevhw4-b700", NET_GATHER, (700, 3, 8, 8), False, [G_POOL, (TAP, 128, 1, True, TAP_PREP_CONV), LINEAR]),
    Case("gather-pool-prevhw4-b37-wide", NET_GATHER, (37, 3, 8, 8), True, [G_POOL, (TAP, 128, 1, True, TAP_PREP_CONV), LINEAR]),
    Case("hw64-s2-1x1-b1200", NET_HW64, (1200, 3, 16, 16), False,
         [G_POOL, (TAP, 64, 2, False, TAP_PREP_CONV), (TAP, 128, 1, False, TAP_PREP), LINEAR]),
    Case("s4-cin1-b37", NET_S4_CIN1, (37, 1, 32, 32), False, [S4_POOL, (TAP, 64, 1, True, TAP_PREP_CONV), LINEAR]),
    Case("s4-cin4-tall-b50", NET_S4_CIN4, (50, 4, 64, 32), False, [S4_POOL, (TAP, 64, 1, False, TAP_PREP_CONV), LINEAR]),
    Case("s4-k7-b20", NET_S4_K7, (20, 3, 32, 32), False, [S4_POOL, (TAP, 64, 1, False, TAP_PREP_CONV), LINEAR]),
    Case("non-square-b64-wide", NET_NONSQUARE, (64, 3, 8, 16), True, [G_POOL, (TAP, 128, 1, False, TAP_PREP_CONV), LINEAR]),
    Case("non-square-b127", NET_NONSQUARE, (127, 3, 8, 16), False, [G_POOL, (TAP, 64, 1, False, TAP_PREP_CONV), LINEAR]),
    Case("two-linears-b127", NET_TWO_LINEARS, (127, 3, 8, 8), False, [G_POOL, LINEAR, LINEAR]),
    Case("one-step-b5", NET_ONE_STEP, (5, 3, 8, 8), False, [G_POOL]),
]
CASE_IDS = [c.name for c in CASES]

# what the table must reach between its cases: every kernel the fused chain can run its steps on, every tap-GEMM
# configuration (BN 64 with one and two CTAs per SM, BN 128), each with and without the pool where it exists, and both
# tap prep kernels.  A conv step behind the pool always has a window (prep_conv); a 1x1 / linear step takes tap_prep.
REQUIRED = {
    S4_POOL, G_POOL,
    (TAP, 64, 1, True, TAP_PREP_CONV), (TAP, 64, 1, False, TAP_PREP_CONV), (TAP, 64, 1, False, TAP_PREP),
    (TAP, 64, 2, True, TAP_PREP_CONV), (TAP, 64, 2, False, TAP_PREP_CONV),
    (TAP, 128, 1, True, TAP_PREP_CONV), (TAP, 128, 1, False, TAP_PREP_CONV), (TAP, 128, 1, False, TAP_PREP),
}


def _build_net(spec, variant, priors, seed=0):
    """A ModuleWrapper whose children are the package's own classes, in the order of ``spec``."""
    import pytorch_bayesiancnn_b200 as bbb
    torch.manual_seed(seed)
    net = bbb.ModuleWrapper()
    for i, item in enumerate(spec):
        kind = item[0]
        if kind == "conv":
            cls = bbb.BBB_LRT_Conv2d if variant == "lrt" else bbb.BBB_Conv2d
            m = cls(item[1], item[2], item[3], stride=item[4], padding=item[5], priors=priors)
        elif kind == "lin":
            cls = bbb.BBB_LRT_Linear if variant == "lrt" else bbb.BBB_Linear
            m = cls(item[1], item[2], priors=priors)
        elif kind == "relu":
            m = nn.ReLU()
        elif kind == "softplus":
            m = nn.Softplus()
        elif kind == "pool":
            m = nn.MaxPool2d(2, 2)
        else:
            m = bbb.FlattenLayer(item[1])
        net.add_module(f"m{i}", m)
    return net


def _launch_config(st, n_sm, wide):
    """(kernel, BN, CTAs per SM, pool, prep kernel) that bbb_layer_forward_fused launches for a planned step."""
    from pytorch_bayesiancnn_b200 import _lib as L, fused
    fn = L.lib().bbb_debug_fused_config
    fn.argtypes = [ctypes.POINTER(L.LayerDesc)] + [ctypes.c_int32] * 7 + [ctypes.POINTER(ctypes.c_int32)]
    fn.restype = ctypes.c_int
    out = (ctypes.c_int32 * 4)()
    d = st.desc()
    rc = fn(ctypes.byref(d), st.in_layout, fused._in_pitch(st), st.prev_hw, st.out_layout, fused._out_pitch(st),
            n_sm, int(wide), out)
    L.check(rc, "bbb_debug_fused_config")
    return (out[0], out[1], out[2], bool(st.pool), out[3])


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()                                   # plan() and the launch query are host logic of the engine


def test_case_table_reaches_every_fused_launch_configuration(built):
    """Plans every case (no GPU needed) and asks the engine what each step would launch on a 148-SM B200: each case
    gets the configuration the table claims, and between them the cases reach every entry of REQUIRED, the BN-128
    tile both by the grid rule and forced by bbb_set_wide_tiles, with and without the pool, a linear step fed by a
    map larger than 1x1 and the gather kernel's pooled packed epilogue."""
    from pytorch_bayesiancnn_b200 import fused, _lib as L
    seen, wide_by = set(), set()
    prev_hw_gt1 = gather_packed = False
    for case in CASES:
        for variant in ("lrt", "bbb"):
            net = _build_net(case.net, variant, CFG_PRIORS)
            steps = fused.plan(list(net.children()), case.x_shape)
            assert steps is not None, (case.name, variant)
            got = [_launch_config(st, 148, case.wide) for st in steps]
            assert got == case.expect, (case.name, variant, got)
            for st, cfg in zip(steps, got):
                seen.add(cfg)
                if cfg[1] == 128:
                    by_rule = _launch_config(st, 148, False)[1] == 128
                    wide_by.add((cfg[3], "grid" if by_rule else "forced"))
                prev_hw_gt1 |= cfg[0] == TAP and st.prev_hw > 1
                gather_packed |= cfg[0] == GATHER and st.pool and st.out_layout == L.LAYOUT_PACKED_BF16
    assert REQUIRED <= seen, REQUIRED - seen
    assert wide_by == {(True, "grid"), (True, "forced"), (False, "grid"), (False, "forced")}, wide_by
    assert prev_hw_gt1 and gather_packed


# --------------------------------------------------------------------------- #
# float64 references of a child list
# --------------------------------------------------------------------------- #
def _bf16(t):
    return t.float().to(torch.bfloat16).double()


def _params(m):
    return [None if p is None else p.detach().double().cpu() for p in (m.W_mu, m.W_rho, m.bias_mu, m.bias_rho)]


def _ref_walk(net, x, eps, rounded, s4_first=False):
    """(logits, KL) of the child list in float64 on identical eps.  ``rounded``: round what the kernels round -- the
    input image, the BBB weight W = mu + eps*sigma (formed in fp32), the LRT mu and sigma^2, and every packed
    activation x and its square plane, both rounded from the fp32 value (fwd_tc.cuh / fused_tc.cuh: bf16(v), bf16(v*v)).
    The stride-4 kernel squares the rounded image (conv_s4_tc.cuh: bf16(bf16(x)^2)); ``s4_first`` says it runs."""
    from oracle import bbb_oracle as O
    h = x.double()
    first = True
    kl = 0.0
    q = list(eps)
    for m in net.children():
        if hasattr(m, "W_mu"):
            mu, rho, bmu, brho = _params(m)
            conv = m._conv_geometry()
            contract = (lambda a, w: F.linear(a, w)) if conv is None else (lambda a, w: F.conv2d(a, w, None, *conv))
            sig = torch.log1p(torch.exp(rho))
            bshape = (1, -1) if conv is None else (1, -1, 1, 1)
            if rounded:
                xin = _bf16(h)
                x2 = _bf16(xin * xin) if (first and s4_first) else _bf16(h * h)
            else:
                xin, x2 = h, h * h
            if m._variant == 0:                                  # BBB: W = mu + eps * sigma, one contraction
                ew, eb = q.pop(0).double(), q.pop(0).double()
                W = mu + ew * sig
                b = bmu + eb * torch.log1p(torch.exp(brho))
                h = contract(xin, _bf16(W) if rounded else W) + b.view(bshape)
            else:                                                # LRT: mean + sqrt(var) * eps of the output
                e = q.pop(0).double()
                s2 = sig * sig
                mean = contract(xin, _bf16(mu) if rounded else mu) + bmu.view(bshape)
                var = 1e-16 + contract(x2, _bf16(s2) if rounded else s2) + (torch.log1p(torch.exp(brho)) ** 2).view(bshape)
                h = mean + var.sqrt() * e
            kl = kl + float(O.kl_loss(mu, rho, bmu, brho, m.prior_mu, m.prior_sigma))
            first = False
        elif isinstance(m, nn.ReLU):
            h = F.relu(h)
        elif isinstance(m, nn.Softplus):
            h = F.softplus(h)
        elif isinstance(m, nn.MaxPool2d):
            h = F.max_pool2d(h, 2, 2)
        else:
            h = h.reshape(-1, m.num_features)
    assert not q
    return h, kl


def _eps_shapes(net, x_shape):
    """The eps the reference draws, in its order: BBB the weight then the bias eps, LRT one eps of the output (before the
    pool); walked on a meta tensor."""
    shapes = []
    h = torch.empty(x_shape, device="meta")
    for m in net.children():
        if hasattr(m, "W_mu"):
            conv = m._conv_geometry()
            w = torch.empty(m.W_mu.shape, device="meta")
            h = F.linear(h, w) if conv is None else F.conv2d(h, w, None, *conv)
            shapes += [tuple(m.W_mu.shape), tuple(m.bias_mu.shape)] if m._variant == 0 else [tuple(h.shape)]
        elif isinstance(m, nn.MaxPool2d):
            h = F.max_pool2d(h, 2, 2)
        elif hasattr(m, "num_features"):
            h = h.reshape(-1, m.num_features)
    return shapes


def _philox_eps(bbb, net, x_shape, seed, ctr, dev):
    """The eps the layers draw in-kernel from streams ctr, ctr+1, ... as external eps: LRT in NHWC element order of the
    pre-pool output, BBB the weights then the bias at offset |W|."""
    eps, shapes, i = [], _eps_shapes(net, x_shape), 0
    for k, m in enumerate([m for m in net.children() if hasattr(m, "W_mu")]):
        if m._variant == 0:
            nw = m.W_mu.numel()
            eps += [bbb.philox_normal(nw, seed, ctr + k, 0, device=dev).view(m.W_mu.shape),
                    bbb.philox_normal(m.bias_mu.numel(), seed, ctr + k, nw, device=dev)]
            i += 2
        else:
            eps.append(_lrt_eps_like(bbb, shapes[i], seed, ctr + k, dev))
            i += 1
    return eps


class _wide_tiles:
    def __init__(self, on):
        self.on = on

    def __enter__(self):
        from pytorch_bayesiancnn_b200 import _lib as L
        self.prev = L.lib().bbb_set_wide_tiles(int(self.on))

    def __exit__(self, *exc):
        from pytorch_bayesiancnn_b200 import _lib as L
        L.lib().bbb_set_wide_tiles(self.prev)
        return False


# Tight bar of the bf16-rounding reference (scale-relative, logits).  Measured on a B200 (1000 W power limit) over every
# case, both variants and both prior sets: worst 1.65e-3 (hw64-s2-1x1-b1200, bbb, CFG priors), 8.4e-4 for LRT, <= 6.8e-4
# in every other case; the unrounded float64 walk sits at 5.9e-4 - 7.2e-3 on the same runs.  What remains is the fp32
# accumulation order, plus an intermediate activation that lands on the other side of a bf16 rounding boundary now and
# then, which is why the largest batches measure the most.
TIGHT_TOL = 3e-3


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["lrt", "bbb"])
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_fused_case(dev, case, variant):
    """One table case under both prior sets: (1) external eps vs the float64 walk, 1e-2 bar, KL 1e-5, the fused plan
    really ran and each step got the launch configuration the table claims; (2) vs the float64 walk rounded where the
    kernels round (TIGHT_TOL); (3) in-kernel Philox == the same streams fed as external eps (1e-6)."""
    import pytorch_bayesiancnn_b200 as bbb
    torch.set_num_threads(max(1, torch.get_num_threads()))
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    s4_first = case.expect[0][0] == S4
    for pname, priors in PRIORS.items():
        net = _build_net(case.net, variant, priors, seed=len(case.name)).to(dev).train()
        net.set_flag("math", "auto")
        g = torch.Generator().manual_seed(3)
        x = torch.randn(case.x_shape, generator=g)
        eps = [torch.randn(s, generator=g) for s in _eps_shapes(net, case.x_shape)]
        with _wide_tiles(case.wide):
            with torch.no_grad(), bbb.external_eps(eps):
                logits, kl = net(x.to(dev))
            steps = net._fused_plans[tuple(case.x_shape)]
            assert steps is not None, case.name                      # it really took the fused path
            assert [_launch_config(st, n_sm, case.wide) for st in steps] == case.expect, (case.name, n_sm)
            ref, refkl = _ref_walk(net, x, eps, rounded=False)
            tight, _ = _ref_walk(net, x, eps, rounded=True, s4_first=s4_first)
            e1, e2 = scale_err(logits, ref), scale_err(logits, tight)
            # (3) in-kernel Philox
            seed, ctr = 1234 + len(case.name), 77
            bbb.manual_seed(seed, ctr)
            with torch.no_grad():
                y1, _ = net(x.to(dev))
            with torch.no_grad(), bbb.external_eps(_philox_eps(bbb, net, case.x_shape, seed, ctr, dev)):
                y2, _ = net(x.to(dev))
            e3 = scale_err(y1, y2)
        print(f"fused {case.name} {variant} {pname}: vs float64 {e1:.3e}, vs bf16-rounded float64 {e2:.3e}, "
              f"philox vs external {e3:.3e}")
        assert e1 < BF16_TOL, (case.name, variant, pname, e1)
        assert abs(float(kl) - refkl) <= KL_TOL * abs(refkl), (case.name, variant, pname, float(kl), refkl)
        assert e2 < TIGHT_TOL, (case.name, variant, pname, e2)
        assert e3 < 1e-6, (case.name, variant, pname, e3)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in CASES if c.expect[0][0] == S4], ids=lambda c: c.name)
def test_fused_s4_mc_folding_equals_sample_loop(dev, case):
    """LRT chains whose first layer is the stride-4 kernel (the only first-layer kernel that folds MC samples into the
    batch): S samples folded into one pass == one pass per sample, with samples sharing 128-row tiles."""
    from pytorch_bayesiancnn_b200 import mc
    net = _build_net(case.net, "lrt", NOISY_PRIORS).to(dev).train()
    net.set_flag("math", "auto")
    x = torch.randn(case.x_shape, device=dev)
    a = mc.MCForward(net, x, 5, want_uncertainty=True, seed=11, num_classes=10, fold=True)
    b = mc.MCForward(net, x, 5, want_uncertainty=True, seed=11, num_classes=10, fold=False)
    assert a.fold_steps is not None and b.fold_steps is None
    a(x), b(x)
    torch.cuda.synchronize()
    e = float((a.logits - b.logits).abs().max() / b.logits.abs().max())
    print(f"mc fold {case.name}: folded vs per-sample {e:.3e}")
    assert e <= 1e-6, (case.name, e)


# --------------------------------------------------------------------------- #
# (B) tensor-core backward at model shapes
# --------------------------------------------------------------------------- #
# (conv?, layer shape, input shape): conv (cin, cout, k, stride, padding), linear (in, out)
GRAD_SHAPES = {
    "alexnet-conv1-b512": (True, (3, 64, 11, 4, 5), (512, 3, 32, 32)),       # 4 equal wgrad chunks, stride-4 dgrad
    "lenet-conv1-b64": (True, (3, 6, 5, 1, 0), (64, 3, 32, 32)),             # chunks 6 x 10 + 4
    "3conv3fc-conv1-b20": (True, (1, 32, 5, 1, 2), (20, 1, 32, 32)),         # chunks 8 + 8 + 4
    "alexnet-conv3-b512": (True, (192, 384, 3, 1, 1), (512, 192, 2, 2)),
    "stride-remainder-b64": (True, (8, 16, 3, 2, 1), (64, 8, 34, 36)),       # (H+2p-k) % s = 1 both ways; 26 + 26 + 12
    "linear-512-1000-b2048": (False, (512, 1000), (2048, 512)),
    "pad-over-window": (True, (4, 8, 3, 1, 3), (6, 4, 6, 6)),               # p > k-1: dgrad falls back
    "linear-b20000": (False, (32, 16), (20000, 32)),                        # wgrad reduction too long: E_UNSUPPORTED
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GRAD_SHAPES))
def test_backward_tc_model_shapes(dev, name):
    """math='auto' and 'tf32', both variants, Philox and external eps, with and without bias, against torch autograd
    through the oracle, with the bars of the toy-shape backward tests (2e-2 bf16, 3e-3 tf32)."""
    torch.set_num_threads(max(1, torch.get_num_threads()))
    conv, shape, x_shape = GRAD_SHAPES[name]
    worst = {}
    for math, tol_y, tol_g in (("auto", 1e-2, 2e-2), ("tf32", 1e-3, 3e-3)):
        for variant in ("bbb", "lrt"):
            for bias in (True, False):
                for use_philox in (True, False):
                    e = _grad_case(dev, variant, conv, bias, use_philox, math=math, tol_y=tol_y, tol_g=tol_g,
                                   shape=shape, x_shape=x_shape)
                    worst[math] = max(worst.get(math, 0.0), e)
    print(f"backward {name}: worst gradient scale err {worst}")


def _tf32(t):
    """cvt.rna.tf32.f32: round to nearest, ties away from zero, to a 10-bit mantissa (finite inputs)."""
    b = t.float().contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32).double()


# Per-contraction bar (scale-relative).  Measured on a B200: worst 2.3e-5 (AlexNet conv1 wgrad, tf32; bf16 1.0e-5),
# dgrad <= 9.2e-6.  Skipping the last wgrad chunk of any chunked shape fails it by orders of magnitude.
CONTRACT_TOL = 6e-5


@pytest.mark.gpu
@pytest.mark.parametrize("math", ["bf16", "tf32"])
def test_tc_contractions_tight(dev, math):
    """functional._tc_wgrad / _tc_dgrad alone against float64 of their operands rounded the way the kernel rounds them
    (bf16: round to nearest even; tf32: cvt.rna).  What remains is fp32 accumulation over <= 8192 terms per chunk plus
    the fp32 sum of the chunks, so a dropped or doubled chunk or a wrong [:kh, :kw] crop fails at any size."""
    from pytorch_bayesiancnn_b200 import functional as Fn, _lib as L
    torch.set_num_threads(max(1, torch.get_num_threads()))
    code = L.MATH_BF16_TC if math == "bf16" else L.MATH_TF32_TC
    rnd = _bf16 if math == "bf16" else _tf32
    g = torch.Generator().manual_seed(23)
    for name, (conv, shape, x_shape) in GRAD_SHAPES.items():
        x = torch.randn(x_shape, generator=g)
        if conv:
            cin, cout, k, s, p = shape
            geom = ((s, s), (p, p), (1, 1))
            oh, ow = Fn.out_hw(x_shape[2], x_shape[3], k, k, geom)
            gy = torch.randn(x_shape[0], cout, oh, ow, generator=g)
            w = torch.randn(cout, cin, k, k, generator=g)
            ref_w = torch.nn.grad.conv2d_weight(rnd(x), w.shape, rnd(gy), s, p)
            ref_x = torch.nn.grad.conv2d_input(x.shape, rnd(w), rnd(gy), s, p)
        else:
            geom = None
            gy = torch.randn(x_shape[0], shape[1], generator=g)
            w = torch.randn(shape[1], shape[0], generator=g)
            ref_w = rnd(gy).t() @ rnd(x)
            ref_x = rnd(gy) @ rnd(w)
        xd, gd, wd = x.to(dev), gy.to(dev), w.to(dev)
        if name == "linear-b20000":                 # the reduction over 20000 rows does not fit the kernel's table
            with pytest.raises(L.EngineError) as err:
                Fn._tc_wgrad(xd, gd, geom, w.shape, code)
            assert err.value.code == L.E_UNSUPPORTED
            ew = float("nan")
        else:
            gw = Fn._tc_wgrad(xd, gd, geom, w.shape, code)
            assert tuple(gw.shape) == tuple(w.shape), name
            ew = scale_err(gw, ref_w)
        gx = Fn._tc_dgrad(gd, wd, geom, x.shape, code)
        if name == "pad-over-window":               # p > k-1: no zero-inserted correlation, the caller falls back
            assert gx is None
            ex = float("nan")
        else:
            assert tuple(gx.shape) == tuple(x.shape), name
            ex = scale_err(gx, ref_x)
        print(f"contraction {name} {math}: wgrad {ew:.3e} dgrad {ex:.3e}")
        assert not ew >= CONTRACT_TOL, (name, math, "wgrad", ew)
        assert not ex >= CONTRACT_TOL, (name, math, "dgrad", ex)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["lrt", "bbb"])
def test_backward_tc_under_stream_base(dev, variant):
    """Inside stream_base(base) a layer call takes stream id base + 0; the tensor-core backward regenerates its eps from
    that absolute id.  Same forward and gradients as the call made with the absolute stream id directly."""
    import pytorch_bayesiancnn_b200 as bbb
    from pytorch_bayesiancnn_b200 import functional as Fn
    cls = bbb.BBB_LRT_Conv2d if variant == "lrt" else bbb.BBB_Conv2d
    torch.manual_seed(2)
    layer = cls(16, 64, 3, stride=2, padding=1, priors=NOISY_PRIORS).to(dev).train()
    x = torch.randn(96, 16, 12, 12, device=dev)
    gout = None
    out = []
    for use_base in (True, False):
        layer.zero_grad()
        xg = x.clone().requires_grad_(True)
        bbb.manual_seed(99, 0)
        if use_base:
            with Fn.stream_base(torch.tensor([5], dtype=torch.int64, device=dev)):
                y = layer(xg)
        else:
            bbb.manual_seed(99, 5)
            y = layer(xg)
        if gout is None:
            gout = torch.randn(y.shape, generator=torch.Generator().manual_seed(1)).to(dev)
        (y * gout).sum().backward()
        out.append([y.detach().clone(), xg.grad.clone(), layer.W_mu.grad.clone(), layer.W_rho.grad.clone(),
                    layer.bias_rho.grad.clone()])
    for name, a, b in zip(("y", "x", "W_mu", "W_rho", "bias_rho"), *out):
        assert scale_err(a, b) < 1e-6, (variant, name, scale_err(a, b))
