"""Parity of the CUDA path against the oracle and the reference-generated golden
fixtures, through the drop-in layer API (-> ctypes -> C ABI).  Needs a GPU.

Tolerances (BASELINE.json north_star): 1e-3 relative to the output scale for the
fp32 path, 1e-2 for bf16; the fp32 CUDA-core path is held to 2e-5 here because it
is IEEE fp32 end to end.  KL: 1e-5 relative on the scalar."""
import numpy as np
import pytest
import torch

from tests.util import (CFG_PRIORS, DEF_PRIORS, build_layer_from_case, case_names, load_case,
                        load_params_into, scale_err)

pytestmark = pytest.mark.gpu
FP32_TOL = 2e-5
KL_TOL = 1e-5


@pytest.fixture(scope="module")
def dev():
    import __graft_entry__ as g
    g.build()
    return torch.device("cuda:0")


def test_layer_cases_external_eps(golden_layers, dev):
    import pytorch_bayesiancnn_b200 as bbb
    for name in case_names(golden_layers):
        c = load_case(golden_layers, name)
        layer = build_layer_from_case(name, c, dev).train()
        eps = [c["eps_w"]] + ([c["eps_b"]] if "eps_b" in c else []) if "_bbb_" in name else [c["eps_y"]]
        with torch.no_grad(), bbb.external_eps(eps):
            y = layer(c["x"].to(dev))
            kl = layer.kl_loss()
        assert y.shape == c["y"].shape, name
        assert scale_err(y, c["y"]) < FP32_TOL, (name, scale_err(y, c["y"]))
        assert abs(float(kl) - float(c["kl"])) <= KL_TOL * abs(float(c["kl"])), (name, float(kl), float(c["kl"]))
        layer.eval()
        with torch.no_grad():
            ym = layer(c["x"].to(dev), sample=False)
        assert scale_err(ym, c["y_mean"]) < FP32_TOL, name


def test_model_cases_external_eps(golden_models, dev):
    import pytorch_bayesiancnn_b200 as bbb
    from pytorch_bayesiancnn_b200 import models as M
    from oracle import bbb_oracle as O
    cls = {"alexnet": M.BBBAlexNet, "lenet": M.BBBLeNet, "3conv3fc": M.BBB3Conv3FC}
    for name in case_names(golden_models):
        c = load_case(golden_models, name)
        key, inputs, outputs, variant, act, batch = [str(v) for v in c["meta"]]
        inputs, outputs, batch = int(inputs), int(outputs), int(batch)
        params = O.init_params(key, outputs, inputs, CFG_PRIORS, seed=123)
        net = load_params_into(cls[key](outputs, inputs, CFG_PRIORS, variant, act), params).to(dev).train()
        eps = O.draw_eps_like_reference(O.eps_shapes(key, outputs, inputs, variant, batch), seed=7)
        with torch.no_grad(), bbb.external_eps(eps):
            logits, kl = net(c["x"].to(dev))
        e = scale_err(logits, c["logits"])
        assert e < 1e-4, (name, e)           # 6-layer chain of fp32 kernels
        assert abs(float(kl) - float(c["kl"])) <= KL_TOL * abs(float(c["kl"])), (name, float(kl), float(c["kl"]))


def test_philox_stream_matches_host_restatement(dev):
    import pytorch_bayesiancnn_b200 as bbb
    from oracle import bbb_oracle as O
    for (n, seed, stream, off) in [(1000, 1, 0, 0), (4099, 0xDEADBEEFCAFE, (3 << 32) + 5, 7), (257, 42, 9, 1 << 33)]:
        z = bbb.philox_normal(n, seed, stream, off, device=dev).cpu().numpy()
        ref = O.philox_normal(n, seed, stream, off)
        assert np.abs(z - ref).max() < 2e-4, (n, seed)     # device uses __logf/__sincosf
    z = bbb.philox_normal(1 << 20, 123, 4, device=dev)
    assert abs(float(z.mean())) < 5e-3 and abs(float(z.std()) - 1) < 5e-3


def _lrt_eps_like(bbb, y, seed, stream, dev):
    """The activation noise an LRT kernel draws for output y (a tensor or a shape): Philox element index is the
    NHWC-flat index of y (include/bbb_b200.h), so fill(numel).view(B,OH,OW,C).permute(0,3,1,2)."""
    shape = tuple(y.shape) if torch.is_tensor(y) else tuple(y)
    z = bbb.philox_normal(int(np.prod(shape)), seed, stream, 0, device=dev)
    if len(shape) == 4:
        B, C, H, W = shape
        return z.view(B, H, W, C).permute(0, 3, 1, 2).contiguous()
    return z.view(shape)


def test_in_kernel_philox_equals_external_draw(golden_layers, dev):
    """The eps a kernel draws itself == bbb_philox_normal_fill of the same (seed, stream):
    run once with in-kernel Philox, once feeding that stream as external eps."""
    import pytorch_bayesiancnn_b200 as bbb
    for name in case_names(golden_layers):
        c = load_case(golden_layers, name)
        layer = build_layer_from_case(name, c, dev).train()
        x = c["x"].to(dev)
        seed, ctr = 99, 1234
        bbb.manual_seed(seed, ctr)
        with torch.no_grad():
            y1 = layer(x)
        if "_bbb_" in name:
            nw = layer.W_mu.numel()
            eps = [bbb.philox_normal(nw, seed, ctr, 0, device=dev).view_as(layer.W_mu)]
            if layer.use_bias:
                eps.append(bbb.philox_normal(layer.bias_mu.numel(), seed, ctr, nw, device=dev))
        else:
            eps = [_lrt_eps_like(bbb, y1, seed, ctr, dev)]
        with torch.no_grad(), bbb.external_eps(eps):
            y2 = layer(x)
        assert scale_err(y1, y2) < 1e-6, name


def test_moments_bbb_and_lrt_agree(dev):
    """Both variants have E[y] = x(*)mu + b_mu, Var[y] = x^2(*)sigma^2 + sigma_b^2
    (SURVEY.md section 4): check the in-kernel Philox sampling against the oracle moments."""
    import pytorch_bayesiancnn_b200 as bbb
    from oracle import bbb_oracle as O
    g = torch.Generator().manual_seed(5)
    x = torch.randn(4, 3, 6, 6, generator=g)
    S = 3000
    for cls in (bbb.BBB_Conv2d, bbb.BBB_LRT_Conv2d):
        torch.manual_seed(1)
        layer = cls(3, 5, 3, padding=1, priors=DEF_PRIORS).to(dev).train()
        mu, var = O.lrt_moments(x, layer.W_mu.detach().cpu(), layer.W_rho.detach().cpu(),
                                layer.bias_mu.detach().cpu(), layer.bias_rho.detach().cpu(), (1, 1, 1))
        bbb.manual_seed(7)
        xs = x.to(dev)
        acc = torch.zeros_like(mu, device=dev, dtype=torch.float64)
        acc2 = torch.zeros_like(acc)
        with torch.no_grad():
            for _ in range(S):
                y = layer(xs).double()
                acc += y; acc2 += y * y
        m = (acc / S).cpu(); v = (acc2 / S).cpu() - m * m
        sd = var.sqrt().double()
        assert ((m - mu.double()).abs() / sd).max() < 6.0 / np.sqrt(S) * 1.5
        assert ((v / var.double()) - 1).abs().max() < 0.25


def test_kl_standalone_and_conventions(dev):
    import pytorch_bayesiancnn_b200 as bbb
    from oracle import bbb_oracle as O
    torch.manual_seed(3)
    layer = bbb.BBB_LRT_Linear(513, 77, priors=CFG_PRIORS).to(dev)
    p = [t.detach().cpu() for t in (layer.W_mu, layer.W_rho, layer.bias_mu, layer.bias_rho)]
    ref = float(O.kl_loss(*p, 0.0, 0.1))
    got = float(layer.kl_loss())                       # no forward yet: stand-alone kernel (SURVEY D7)
    assert abs(got - ref) <= KL_TOL * abs(ref)
    layer.set_flag("kl_convention", "textbook")
    tb = float(O.kl_textbook(*p, 0.0, 0.1))
    assert abs(float(layer.kl_loss()) - tb) <= KL_TOL * abs(tb)
    layer.set_flag("kl_convention", "reference")
    # stale-cache guard: parameters change after a forward -> kl_loss recomputes
    with torch.no_grad():
        layer(torch.randn(4, 513, device=dev))
        k1 = float(layer.kl_loss())
        layer.W_rho.add_(0.5)
        k2 = float(layer.kl_loss())
    ref2 = float(O.kl_loss(p[0], p[1] + 0.5, p[2], p[3], 0.0, 0.1))
    assert abs(k1 - ref) <= KL_TOL * abs(ref) and abs(k2 - ref2) <= KL_TOL * abs(ref2)


def test_kl_independent_of_input_and_eps(dev):
    """SURVEY D11."""
    import pytorch_bayesiancnn_b200 as bbb
    torch.manual_seed(0)
    layer = bbb.BBB_Conv2d(3, 8, 3, padding=1, priors=CFG_PRIORS).to(dev).train()
    vals = []
    with torch.no_grad():
        for i in range(3):
            layer(torch.randn(2 + i, 3, 8, 8, device=dev))
            vals.append(float(layer.kl_loss()))
    assert vals[0] == vals[1] == vals[2]


def test_mc_combine_matches_oracle(dev):
    import pytorch_bayesiancnn_b200 as bbb
    from oracle import bbb_oracle as O
    g = torch.Generator().manual_seed(2)
    for (S, B, C) in [(1, 5, 10), (7, 33, 10), (25, 16, 100)]:
        logits = torch.randn(S, B, C, generator=g) * 3
        out, mom = bbb.mc_combine(logits.to(dev), want_moments=True)
        ref = O.mc_combine(list(logits))
        assert (out.cpu() - ref).abs().max() < 2e-5
        pred, epi, ale, ent = O.uncertainty(list(logits))
        p1, p2, sl = [m.double().cpu() / S for m in mom]
        assert (sl - pred).abs().max() < 1e-5
        assert ((p2 - p1 * p1) - epi).abs().max() < 1e-6       # epistemic = E[p^2] - pbar^2
        assert ((p1 - p2) - ale).abs().max() < 1e-6            # aleatoric = pbar - E[p^2]


def test_full_size_properties_alexnet_b512(dev):
    """BASELINE-size run (BBBAlexNet, B=512) through size-independent properties:
    seed determinism, stream independence, KL == stand-alone KL, finite output,
    batch-slice consistency of the deterministic path."""
    import pytorch_bayesiancnn_b200 as bbb
    from pytorch_bayesiancnn_b200.models import BBBAlexNet
    for variant in ("bbb", "lrt"):
        torch.manual_seed(0)
        net = BBBAlexNet(10, 3, CFG_PRIORS, variant, "softplus").to(dev).train()
        x = torch.randn(512, 3, 32, 32, device=dev)
        with torch.no_grad():
            bbb.manual_seed(5); a, kla = net(x)
            bbb.manual_seed(5); b, klb = net(x)
            bbb.manual_seed(6); c, _ = net(x)
            assert torch.equal(a, b) and float(kla) == float(klb)
            assert not torch.equal(a, c) and torch.isfinite(a).all()
            kl_sa = sum(float(bbb.functional.KLFn.apply(m.W_mu, m.W_rho, m.bias_mu, m.bias_rho, 0.0, 0.1, 0))
                        for m in net.modules() if hasattr(m, "W_mu"))
            assert abs(kl_sa - float(kla)) <= 1e-6 * abs(kl_sa)
            # deterministic path: a batch slice gives the same rows
            net.set_flag("math", "fp32")
            net.eval()
            h = x
            h2 = x[:7]
            for m in net.children():
                h = m(h, sample=False) if hasattr(m, "W_mu") else m(h)
                h2 = m(h2, sample=False) if hasattr(m, "W_mu") else m(h2)
            assert scale_err(h[:7], h2) < 1e-6


def test_errors_are_loud(dev):
    import pytorch_bayesiancnn_b200 as bbb
    layer = bbb.BBB_Conv2d(3, 4, 3).to(dev)
    with pytest.raises(bbb.EngineError):
        layer(torch.randn(1, 3, 8, 8))                  # CPU tensor: no fallback
    with pytest.raises(bbb.EngineError):
        layer(torch.randn(1, 5, 8, 8, device=dev))      # channel mismatch
    with pytest.raises(bbb.EngineError):
        layer(torch.randn(1, 3, 2, 2, device=dev))      # kernel larger than input


# --------------------------------------------------------------------------- #
# tcgen05 path (math='bf16'): bf16 operands, fp32 accumulate -> 1e-2 bar
# --------------------------------------------------------------------------- #
BF16_TOL = 1e-2


def test_tc_layer_cases_external_eps(golden_layers, dev):
    import pytorch_bayesiancnn_b200 as bbb
    worst = 0.0
    for name in case_names(golden_layers):
        c = load_case(golden_layers, name)
        layer = build_layer_from_case(name, c, dev).train()
        layer.set_flag("math", "bf16")
        eps = [c["eps_w"]] + ([c["eps_b"]] if "eps_b" in c else []) if "_bbb_" in name else [c["eps_y"]]
        with torch.no_grad(), bbb.external_eps(eps):
            y = layer(c["x"].to(dev))
            kl = layer.kl_loss()
        e = scale_err(y, c["y"])
        worst = max(worst, e)
        assert e < BF16_TOL, (name, e)
        assert abs(float(kl) - float(c["kl"])) <= KL_TOL * abs(float(c["kl"])), (name, float(kl), float(c["kl"]))
        layer.eval()
        with torch.no_grad():
            ym = layer(c["x"].to(dev), sample=False)
        assert scale_err(ym, c["y_mean"]) < BF16_TOL, name
    print("tc layer cases worst scale err", worst)


def test_tc_alexnet_layer_shapes_b512(dev):
    """Every BBBAlexNet layer geometry at the BASELINE batch (512), both variants,
    tcgen05 path vs the oracle on identical eps."""
    import pytorch_bayesiancnn_b200 as bbb
    from oracle import bbb_oracle as O
    torch.set_num_threads(max(1, (torch.get_num_threads())))
    geoms = [(3, 64, 11, 4, 5, 32), (64, 192, 5, 1, 2, 4), (192, 384, 3, 1, 1, 2), (384, 256, 3, 1, 1, 2),
             (256, 128, 3, 1, 1, 2)]
    g = torch.Generator().manual_seed(11)
    for variant, cls in (("bbb", bbb.BBB_Conv2d), ("lrt", bbb.BBB_LRT_Conv2d)):
        for (cin, cout, k, s, p, hw) in geoms:
            torch.manual_seed(cin)
            layer = cls(cin, cout, k, stride=s, padding=p, priors=CFG_PRIORS).to(dev).train()
            layer.set_flag("math", "bf16")
            x = torch.rand(512, cin, hw, hw, generator=g) * 2
            P = [t.detach().cpu() for t in (layer.W_mu, layer.W_rho, layer.bias_mu, layer.bias_rho)]
            ho = (hw + 2 * p - k) // s + 1
            if variant == "bbb":
                eps = [torch.randn(P[0].shape, generator=g), torch.randn(cout, generator=g)]
                ref = O.bbb_forward(x, *P, eps[0], eps[1], (s, p, 1))
            else:
                eps = [torch.randn(512, cout, ho, ho, generator=g)]
                ref = O.lrt_forward(x, *P, eps[0], (s, p, 1))
            with torch.no_grad(), bbb.external_eps(eps):
                y = layer(x.to(dev))
                kl = float(layer.kl_loss())
            e = scale_err(y, ref)
            refkl = float(O.kl_loss(*P, 0.0, 0.1))
            assert e < BF16_TOL, (variant, cin, cout, e)
            assert abs(kl - refkl) <= KL_TOL * abs(refkl)
            # and the IEEE-fp32 CUDA-core path on the same inputs
            layer.set_flag("math", "fp32")
            with torch.no_grad(), bbb.external_eps(eps):
                y32 = layer(x.to(dev))
            assert scale_err(y32, ref) < FP32_TOL, (variant, cin, cout, scale_err(y32, ref))


def test_tc_model_cases_external_eps(golden_models, dev):
    import pytorch_bayesiancnn_b200 as bbb
    from pytorch_bayesiancnn_b200 import models as M
    from oracle import bbb_oracle as O
    cls = {"alexnet": M.BBBAlexNet, "lenet": M.BBBLeNet, "3conv3fc": M.BBB3Conv3FC}
    for name in case_names(golden_models):
        c = load_case(golden_models, name)
        key, inputs, outputs, variant, act, batch = [str(v) for v in c["meta"]]
        inputs, outputs, batch = int(inputs), int(outputs), int(batch)
        params = O.init_params(key, outputs, inputs, CFG_PRIORS, seed=123)
        net = load_params_into(cls[key](outputs, inputs, CFG_PRIORS, variant, act), params).to(dev).train()
        net.set_flag("math", "bf16")
        eps = O.draw_eps_like_reference(O.eps_shapes(key, outputs, inputs, variant, batch), seed=7)
        with torch.no_grad(), bbb.external_eps(eps):
            logits, kl = net(c["x"].to(dev))
        e = scale_err(logits, c["logits"])
        print(name, "bf16 chain scale err", e)
        assert e < BF16_TOL, (name, e)          # north_star bar: 1e-2 for the whole bf16 model (measured 4-8e-3)
        assert abs(float(kl) - float(c["kl"])) <= KL_TOL * abs(float(c["kl"])), (name, float(kl), float(c["kl"]))


def test_tc_philox_equals_external_draw(dev):
    import pytorch_bayesiancnn_b200 as bbb
    for cls in (bbb.BBB_Conv2d, bbb.BBB_LRT_Conv2d):
        torch.manual_seed(4)
        layer = cls(16, 96, 3, padding=1, priors=CFG_PRIORS).to(dev).train()
        layer.set_flag("math", "bf16")
        x = torch.randn(40, 16, 6, 6, device=dev)
        bbb.manual_seed(77, 5)
        with torch.no_grad():
            y1 = layer(x)
        if cls is bbb.BBB_Conv2d:
            nw = layer.W_mu.numel()
            eps = [bbb.philox_normal(nw, 77, 5, 0, device=dev).view_as(layer.W_mu),
                   bbb.philox_normal(96, 77, 5, nw, device=dev)]
        else:
            eps = [_lrt_eps_like(bbb, y1, 77, 5, dev)]
        with torch.no_grad(), bbb.external_eps(eps):
            y2 = layer(x)
        assert scale_err(y1, y2) < 1e-6


# --------------------------------------------------------------------------- #
# fused chain (activation + pool in the epilogue, packed bf16 between layers)
# --------------------------------------------------------------------------- #
def _alexnet(variant, classes, dev, act="softplus"):
    from pytorch_bayesiancnn_b200 import models as M
    from oracle import bbb_oracle as O
    params = O.init_params("alexnet", classes, 3, CFG_PRIORS, seed=123)
    net = load_params_into(M.BBBAlexNet(classes, 3, CFG_PRIORS, variant, act), params).to(dev).train()
    net.set_flag("math", "bf16")
    return net, params


def test_fused_chain_vs_oracle_external_eps(dev):
    """Whole BBBAlexNet through the fused tcgen05 chain vs the oracle on identical eps,
    at a batch that is not a multiple of the 128-row tile and at the BASELINE batch."""
    import pytorch_bayesiancnn_b200 as bbb
    from oracle import bbb_oracle as O
    for variant in ("lrt", "bbb"):
        for (batch, classes, act) in ((37, 10, "softplus"), (512, 10, "softplus"), (130, 100, "relu")):
            net, params = _alexnet(variant, classes, dev, act)
            assert net._try_fused is not None
            x = torch.randn(batch, 3, 32, 32, generator=torch.Generator().manual_seed(1))
            eps = O.draw_eps_like_reference(O.eps_shapes("alexnet", classes, 3, variant, batch), seed=9)
            ref, refkl = O.net_forward("alexnet", params, x, eps, variant, act, 0.0, 0.1, classes)
            with torch.no_grad(), bbb.external_eps(eps):
                logits, kl = net(x.to(dev))
            assert net._fused_plans[(batch, 3, 32, 32)] is not None   # it really took the fused path
            e = scale_err(logits, ref)
            print("fused", variant, batch, classes, act, "scale err", e)
            assert e < BF16_TOL, (variant, batch, e)
            assert abs(float(kl) - float(refkl)) <= KL_TOL * abs(float(refkl))


def test_fused_equals_unfused_same_philox(dev):
    import pytorch_bayesiancnn_b200 as bbb
    for variant in ("lrt", "bbb"):
        net, _ = _alexnet(variant, 10, dev)
        x = torch.randn(256, 3, 32, 32, device=dev)
        with torch.no_grad():
            bbb.manual_seed(3); a, kla = net(x)
            net.set_flag("fuse", False)
            bbb.manual_seed(3); b, klb = net(x)
            net.set_flag("fuse", True)
            bbb.manual_seed(3); c, _ = net(x)
        assert torch.equal(a, c)
        assert scale_err(a, b) < BF16_TOL, (variant, scale_err(a, b))   # same noise, bf16 inter-layer rounding only
        assert abs(float(kla) - float(klb)) <= 1e-6 * abs(float(klb))      # same terms, different summation order


# --------------------------------------------------------------------------- #
# backward (SURVEY.md Appendix A) vs torch autograd through the oracle
# --------------------------------------------------------------------------- #
def _grad_case(dev, variant, conv, bias, use_philox, math="fp32", tol_y=FP32_TOL, tol_g=1e-4, shape=None, x_shape=None):
    """One layer's forward + backward against torch autograd through the oracle.  ``shape``: the layer's constructor
    arguments, (cin, cout, k, stride, padding) of a conv or (in, out) of a linear layer, and ``x_shape`` its input;
    by default a 5->7 k3 s2 p1 conv on 6x5x9x8 and a 37->11 linear layer on 9 rows.  Returns the worst gradient error."""
    import pytorch_bayesiancnn_b200 as bbb
    from oracle import bbb_oracle as O
    g = torch.Generator().manual_seed(17)
    if conv:
        cin, cout, k, s, p = shape or (5, 7, 3, 2, 1)
        cls = bbb.BBB_LRT_Conv2d if variant == "lrt" else bbb.BBB_Conv2d
        layer = cls(cin, cout, k, stride=s, padding=p, bias=bias, priors=DEF_PRIORS)
        x = torch.randn(x_shape or (6, 5, 9, 8), generator=g)
        geom = ((s, s), (p, p), (1, 1))
    else:
        fin, fout = shape or (37, 11)
        cls = bbb.BBB_LRT_Linear if variant == "lrt" else bbb.BBB_Linear
        layer = cls(fin, fout, bias=bias, priors=DEF_PRIORS)
        x = torch.randn(x_shape or (9, fin), generator=g)
        geom = None
    layer = layer.to(dev).train()
    layer.set_flag("math", math)
    P = [p.detach().cpu().clone().requires_grad_(True) if p is not None else None
         for p in (layer.W_mu, layer.W_rho, layer.bias_mu, layer.bias_rho)]
    xr = x.clone().requires_grad_(True)
    xg = x.to(dev).requires_grad_(True)
    # ours
    if use_philox:
        bbb.manual_seed(21, 4)
        y = layer(xg)
        if variant == "lrt":
            eps = [_lrt_eps_like(bbb, y, 21, 4, dev).cpu()]
        else:
            nw = layer.W_mu.numel()
            eps = [bbb.philox_normal(nw, 21, 4, 0, device=dev).view_as(layer.W_mu).cpu()]
            if bias:
                eps.append(bbb.philox_normal(layer.bias_mu.numel(), 21, 4, nw, device=dev).cpu())
    else:
        if variant == "lrt":
            with torch.no_grad():
                yshape = layer(xg).shape
            eps = [torch.randn(yshape, generator=g)]
        else:
            eps = [torch.randn(layer.W_mu.shape, generator=g)] + ([torch.randn(layer.bias_mu.shape, generator=g)] if bias else [])
        with bbb.external_eps(eps):
            y = layer(xg)
    kl = layer.kl_loss()
    gout = torch.randn(y.shape, generator=g)
    loss = (y * gout.to(dev)).sum() + 0.37 * kl
    loss.backward()
    # oracle
    if variant == "lrt":
        yr = O.lrt_forward(xr, P[0], P[1], P[2], P[3], eps[0], geom)
    else:
        yr = O.bbb_forward(xr, P[0], P[1], P[2], P[3], eps[0], eps[1] if bias else None, geom)
    klr = O.kl_loss(P[0], P[1], P[2], P[3], 0.0, 0.1)
    ((yr * gout).sum() + 0.37 * klr).backward()
    assert scale_err(y, yr) < tol_y, (variant, conv, bias, use_philox, "y", math, scale_err(y, yr))
    got = [xg.grad, layer.W_mu.grad, layer.W_rho.grad] + ([layer.bias_mu.grad, layer.bias_rho.grad] if bias else [])
    ref = [xr.grad, P[0].grad, P[1].grad] + ([P[2].grad, P[3].grad] if bias else [])
    worst = 0.0
    for name, a, b_ in zip(("x", "W_mu", "W_rho", "bias_mu", "bias_rho"), got, ref):
        assert a is not None, name
        e = scale_err(a, b_)
        assert e < tol_g, (variant, conv, bias, use_philox, name, math, e)
        worst = max(worst, e)
    return worst


def test_backward_matches_oracle_autograd(dev):
    for variant in ("bbb", "lrt"):
        for conv in (True, False):
            for bias in (True, False):
                for use_philox in (False, True):
                    _grad_case(dev, variant, conv, bias, use_philox)


def test_backward_tensor_core_path_matches_oracle_autograd(dev):
    """math='auto': forward AND backward contractions on tcgen05 (wgrad / dgrad as role-swapped calls of the layer
    kernel, bf16 operands, fp32 accumulate) against torch autograd through the oracle: the bf16 bar."""
    for variant in ("bbb", "lrt"):
        for conv in (True, False):
            for bias in (True, False):
                _grad_case(dev, variant, conv, bias, True, math="auto", tol_y=1e-2, tol_g=2e-2)


def test_training_step_runs_and_reduces_loss(dev):
    """main_bayesian.train_model's inner loop (main_bayesian.py:38-58) on our layers: Adam on mu/rho."""
    import pytorch_bayesiancnn_b200 as bbb
    from pytorch_bayesiancnn_b200.models import BBBLeNet
    torch.manual_seed(0)
    net = BBBLeNet(10, 3, CFG_PRIORS, "lrt", "softplus").to(dev).train()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    x = torch.randn(64, 3, 32, 32, device=dev)
    yl = torch.randint(0, 10, (64,), device=dev)
    losses = []
    bbb.manual_seed(1)
    for it in range(30):
        opt.zero_grad()
        out, kl = net(x)
        loss = torch.nn.functional.nll_loss(torch.log_softmax(out, 1), yl) * 50000 + 0.1 * kl   # metrics.py:14
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert all(torch.isfinite(p.grad).all() for p in net.parameters())
    assert losses[-1] < losses[0]
