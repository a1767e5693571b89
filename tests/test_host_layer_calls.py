"""What goes into a layer call, checked without a GPU: the descriptor both paths into the engine build
(functional.make_desc), the noise they draw (functional.draw_noise) and the error code that marks a shape as
unsupported rather than wrong."""
import ctypes

import pytest
import torch

from tests.util import CFG_PRIORS

F32_01 = ctypes.c_float(0.1).value

# bbb_layer_desc fields batch .. pool_s of every step of BBBAlexNet(lrt, softplus) planned for (512, 3, 32, 32)
ALEXNET_LRT_STEPS = [
    (512, 3, 32, 32, 64, 11, 11, 4, 4, 5, 5, 1, 1, 1, 1, 1, 0, 1, 0, 1, 2, 2),
    (512, 64, 4, 4, 192, 5, 5, 1, 1, 2, 2, 1, 1, 1, 1, 1, 0, 1, 0, 1, 2, 2),
    (512, 192, 2, 2, 384, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 1, 0, 1, 0, 0),
    (512, 384, 2, 2, 256, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 1, 0, 1, 0, 0),
    (512, 256, 2, 2, 128, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 1, 0, 1, 2, 2),
    (512, 128, 1, 1, 10, 1, 1, 1, 1, 0, 0, 1, 1, 1, 1, 1, 0, 1, 0, 0, 0, 0),
]
VARIANT_FIELD = 13


@pytest.fixture(scope="module", autouse=True)
def built():
    import __graft_entry__ as g
    g.build()                                   # plan() asks the engine (host-only checks) whether a step fuses


def _fields(d):
    from pytorch_bayesiancnn_b200 import _lib as L
    return tuple(getattr(d, n) for n, _ in L.LayerDesc._fields_[:-3]) + tuple(d.reserved) + (d.prior_mu, d.prior_sigma)


class _Stop(Exception):
    pass


@pytest.mark.parametrize("variant", ["lrt", "bbb"])
@pytest.mark.parametrize("fold", [None, (512, 1 << 40)], ids=["unfolded", "folded"])
def test_fused_chain_descriptors(monkeypatch, variant, fold):
    """plan() checks each step with the phase-0 descriptor; run_step() launches the prep and GEMM halves with the
    same descriptor and the phase in reserved[0].  Folding packs (rows, stride lo, stride hi) into reserved[1..3]."""
    from pytorch_bayesiancnn_b200 import fused, functional as Fn, _lib as L
    from pytorch_bayesiancnn_b200.models import BBBAlexNet
    net = BBBAlexNet(10, 3, CFG_PRIORS, variant, "softplus")
    seen, stop = [], [False]
    real = Fn.make_desc

    def spy(*a, **k):
        d = real(*a, **k)
        seen.append(_fields(d))
        if stop[0]:
            raise _Stop                         # run_step() is stopped before it allocates or launches anything
        return d

    monkeypatch.setattr(Fn, "make_desc", spy)
    steps = fused.plan(list(net.children()), (512, 3, 32, 32), fold)
    assert steps is not None and len(seen) == len(steps) == 6
    stop[0] = True
    for phase in (L.FUSED_PREP_ONLY, L.FUSED_SKIP_PREP):
        for st in steps:
            with pytest.raises(_Stop):
                fused.run_step(st, None, None, None, 0, phase=phase, fold=fold)
    packed = (512, 0, 256) if fold else (0, 0, 0)
    vcode = L.VARIANT_LRT if variant == "lrt" else L.VARIANT_BBB
    expect = []
    for phase in (0, L.FUSED_PREP_ONLY, L.FUSED_SKIP_PREP):
        for row in ALEXNET_LRT_STEPS:
            row = row[:VARIANT_FIELD] + (vcode,) + row[VARIANT_FIELD + 1:]
            expect.append(row + (phase,) + packed + (0.0, F32_01))
    assert seen == expect


def test_per_layer_descriptors():
    from pytorch_bayesiancnn_b200 import functional as Fn, _lib as L
    conv = Fn.make_desc((8, 3, 32, 32), (16, 3, 5, 3), ((2, 1), (1, 2), (1, 2)), L.VARIANT_LRT, True, True,
                        0.0, 0.1, L.MATH_BF16_TC, L.KL_TEXTBOOK, L.ACT_RELU)
    assert _fields(conv) == (8, 3, 32, 32, 16, 5, 3, 2, 1, 1, 2, 1, 2, 1, 1, 1, 0, 1, 1, 2, 0, 0, 0, 0, 0, 0,
                             0.0, F32_01)
    lin = Fn.make_desc((8, 400), (120, 400), None, L.VARIANT_BBB, False, False, 0.5, 0.2)
    assert _fields(lin) == (8, 400, 1, 1, 120, 1, 1, 1, 1, 0, 0, 1, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                            0.5, ctypes.c_float(0.2).value)
    # the stride's low word is stored as a signed int32
    d = Fn.make_desc((8, 400), (120, 400), None, L.VARIANT_LRT, True, True, 0.0, 0.1, pool=True,
                     phase=L.FUSED_SKIP_PREP, fold=(3, (5 << 32) | 0xFFFFFFFE))
    assert (d.pool_k, d.pool_s, tuple(d.reserved)) == (2, 2, (L.FUSED_SKIP_PREP, 3, -2, 5))


def _eps(*shapes):
    return [torch.full(s, float(i)) for i, s in enumerate(shapes)]


def test_noise_draw_pops_external_eps_in_reference_order():
    from pytorch_bayesiancnn_b200 import functional as Fn, _lib as L
    cpu = torch.device("cpu")
    cases = [   # (variant, weight, bias, output, what the reference draws)
        (L.VARIANT_BBB, (4, 3, 5, 5), (4,), (2, 4, 6, 6), [(4, 3, 5, 5), (4,)]),
        (L.VARIANT_BBB, (7, 9), None, (2, 7), [(7, 9)]),
        (L.VARIANT_LRT, (4, 3, 5, 5), (4,), (2, 4, 6, 6), [(2, 4, 6, 6)]),
        (L.VARIANT_LRT, (7, 9), (7,), (2, 7), [(2, 7)]),
    ]
    for variant, w, b, y, drawn in cases:
        q = _eps(*drawn)
        with Fn.external_eps(q):
            eps_a, eps_b, seed, stream_id, base = Fn.draw_noise(variant, w, b, y, cpu)
        assert torch.equal(eps_a, q[0]) and (seed, stream_id, base) == (0, 0, None)
        assert (eps_b is None) if len(drawn) == 1 else torch.equal(eps_b, q[1])
    # the fused chain's steps draw BBBAlexNet's eps in the reference's order
    from oracle import bbb_oracle as O
    from pytorch_bayesiancnn_b200 import fused
    from pytorch_bayesiancnn_b200.models import BBBAlexNet
    for variant in ("lrt", "bbb"):
        steps = fused.plan(list(BBBAlexNet(10, 3, CFG_PRIORS, variant, "softplus").children()), (8, 3, 32, 32))
        q = _eps(*O.eps_shapes("alexnet", 10, 3, variant, 8))
        with Fn.external_eps(q):
            got = [e for st in steps for e in st.noise()[:2] if e is not None]
        assert len(got) == len(q) and all(torch.equal(a.cpu(), e) for a, e in zip(got, q))   # BBB params may be on cuda:0


def test_noise_draw_rejects_a_wrong_shape_and_an_exhausted_queue():
    from pytorch_bayesiancnn_b200 import functional as Fn, _lib as L
    cpu = torch.device("cpu")
    with pytest.raises(RuntimeError, match=r"expected shape \(4, 3, 5, 5\), got \(4, 3, 5, 4\)"):
        with Fn.external_eps(_eps((4, 3, 5, 4), (4,))):
            Fn.draw_noise(L.VARIANT_BBB, (4, 3, 5, 5), (4,), (2, 4, 6, 6), cpu)
    with pytest.raises(RuntimeError, match="queue exhausted"):
        with Fn.external_eps(_eps((4, 3, 5, 5))):
            Fn.draw_noise(L.VARIANT_BBB, (4, 3, 5, 5), (4,), (2, 4, 6, 6), cpu)


def test_noise_draw_takes_consecutive_philox_streams():
    from pytorch_bayesiancnn_b200 import functional as Fn, _lib as L
    cpu = torch.device("cpu")
    with Fn.mc_sample(3, seed=77, offset=10):
        first = Fn.noise_snapshot()[0]
        draws = [Fn.draw_noise(L.VARIANT_BBB, (4, 3, 5, 5), (4,), (2, 4, 6, 6), cpu),
                 Fn.draw_noise(L.VARIANT_LRT, (7, 9), None, (2, 7), cpu)]
        assert draws == [(None, None, 77, first, None), (None, None, 77, first + 1, None)]
        base = torch.zeros(1, dtype=torch.int64)
        with Fn.stream_base(base):
            a = Fn.draw_noise(L.VARIANT_LRT, (7, 9), None, (2, 7), cpu)
            b = Fn.draw_noise(L.VARIANT_LRT, (7, 9), None, (2, 7), cpu)
        assert a[2:4] == (77, 0) and b[2:4] == (77, 1) and a[4] is base and b[4] is base


def test_engine_errors_carry_their_code():
    """An unsupported shape (BBB_E_UNSUPPORTED) is told apart from a failure by EngineError.code, not by its text."""
    import torch.nn as nn
    from pytorch_bayesiancnn_b200 import fused, _lib as L
    from pytorch_bayesiancnn_b200.models import BBBAlexNet, BBBLeNet, BBB3Conv3FC
    from pytorch_bayesiancnn_b200.modules import ModuleWrapper, BBBLRTConv2d
    steps = fused.plan(list(BBBAlexNet(10, 3, CFG_PRIORS, "lrt", "softplus").children()), (8, 3, 32, 32))
    d = steps[0].desc()
    d.math = L.MATH_FP32
    rc = L.lib().bbb_fused_supported(ctypes.byref(d), steps[0].in_layout, 0, 1, steps[0].out_layout, 4096)
    assert rc == L.E_UNSUPPORTED
    with pytest.raises(L.EngineError) as e:
        L.check(rc, "bbb_fused_supported")
    assert e.value.code == -2
    assert str(e.value) == "bbb_fused_supported failed (code -2): the fused chain exists on the tcgen05 (bf16) path only"
    assert L.EngineError("host-side check").code is None
    for net, shape in ((BBB3Conv3FC(10, 1, CFG_PRIORS), (8, 1, 32, 32)), (BBBLeNet(10, 3, CFG_PRIORS), (8, 3, 32, 32))):
        net.set_flag("math", "bf16")
        assert fused.plan(list(net.children()), shape) is None

    class Wide(ModuleWrapper):      # 16 pixels x 8 channel blocks: more than the tap-GEMM kernel takes per tile
        def __init__(self):
            super().__init__()
            self.conv1 = BBBLRTConv2d(3, 512, 5, stride=4, padding=2, priors=CFG_PRIORS)
            self.pool1 = nn.MaxPool2d(2, 2)
            self.conv2 = BBBLRTConv2d(512, 64, 3, padding=1, priors=CFG_PRIORS)

    assert fused.plan(list(Wide().children()), (8, 3, 32, 32)) is None
    assert b"tap-GEMM" in L.lib().bbb_last_error()
