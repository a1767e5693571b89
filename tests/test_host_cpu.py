"""Host-side logic that runs without a GPU: the layer surface, state_dict keys,
the C-ABI library loads and exports every declared symbol, errors are loud."""
import ctypes
import os
import re

import pytest
import torch

from tests.conftest import ROOT
from tests.util import CFG_PRIORS


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    return g.LIB


def test_library_exports_every_declared_symbol(built):
    hdr = open(os.path.join(ROOT, "include", "bbb_b200.h")).read()
    hdr_nc = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(bbb_[a-z0-9_]+)\s*\(", hdr_nc))
    assert len(declared) >= 12
    lib = ctypes.CDLL(built)
    for name in declared:
        assert hasattr(lib, name), name
    from pytorch_bayesiancnn_b200 import _lib
    assert declared == set(_lib.SYMBOLS)
    lib.bbb_abi_version.restype = ctypes.c_int32
    assert lib.bbb_abi_version() == 2
    assert ctypes.sizeof(_lib.LayerDesc) == 4 * 26 + 8


def test_header_enums_match_the_python_mirror_and_tile_policy_is_host_only(built):
    """The enum values ctypes passes are the header's; bbb_set_wide_tiles is a host-side switch (no GPU needed)."""
    from pytorch_bayesiancnn_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "bbb_b200.h")).read()
    val = lambda name: int(re.search(name + r"\s*=\s*(-?\d+)", hdr).group(1))
    assert (val("BBB_MATH_FP32"), val("BBB_MATH_BF16_TC"), val("BBB_MATH_AUTO"), val("BBB_MATH_TF32_TC")) == \
        (_lib.MATH_FP32, _lib.MATH_BF16_TC, _lib.MATH_AUTO, _lib.MATH_TF32_TC)
    assert (val("BBB_MC_MOMENTS"), val("BBB_MC_NORMALIZED")) == (_lib.MC_MOMENTS, _lib.MC_NORMALIZED)
    assert val("BBB_E_UNSUPPORTED") == _lib.E_UNSUPPORTED
    assert set(_lib.MATH_BY_NAME) == {"fp32", "bf16", "tf32", "auto"}
    lib = _lib.lib()
    prev = lib.bbb_set_wide_tiles(1)
    assert lib.bbb_set_wide_tiles(prev) == 1 and lib.bbb_set_wide_tiles(prev) == prev


def test_invalid_calls_return_error_codes_without_gpu(built):
    from pytorch_bayesiancnn_b200 import _lib
    lib = _lib.lib()
    assert lib.bbb_kl_forward(None, None, 0, None, None, 0, 0.0, 0.1, 0, None, None, 0, None) == -1
    assert b"NULL" in lib.bbb_last_error()
    d = _lib.LayerDesc()
    assert lib.bbb_conv2d_forward(ctypes.byref(d), None, None, None, None, None, None, None, None, None, None,
                                  0, 0, None, None, 0, None) == -1
    assert b"geometry" in lib.bbb_last_error()


def test_layer_surface_and_state_dict_keys():
    import layers
    c = layers.BBB_Conv2d(3, 8, 5, stride=2, padding=1, bias=True, priors=None)
    assert list(c.state_dict().keys()) == ["W_mu", "W_rho", "bias_mu", "bias_rho"]
    assert c.kernel_size == (5, 5) and c.groups == 1 and c.use_bias and c.prior_sigma == 0.1
    assert tuple(c.W_mu.shape) == (8, 3, 5, 5)
    n = layers.BBB_LRT_Linear(7, 3, bias=False)
    assert n.bias_mu is None and list(n.state_dict().keys()) == ["W_mu", "W_rho"]
    r = layers.BBB_Conv2d(3, 4, (3, 5))
    assert r.kernel_size == (3, 5)
    # reset_parameters follows the priors (BBB/BBBConv.py:53-59)
    big = layers.BBB_LRT_Linear(400, 300, priors=CFG_PRIORS)
    assert abs(float(big.W_rho.mean()) + 5) < 0.01 and abs(float(big.W_mu.std()) - 0.1) < 0.01


def test_module_wrapper_and_flatten():
    import layers

    class Net(layers.ModuleWrapper):
        def __init__(self):
            super().__init__()
            self.flatten = layers.FlattenLayer(12)
            self.id = torch.nn.Identity()

    net = Net()
    x = torch.arange(48.0).view(4, 3, 2, 2)
    y, kl = net(x)
    assert y.shape == (4, 12) and kl == 0.0
    assert layers.FlattenLayer(24)(x).shape == (2, 24)       # no shape check, like the reference (SURVEY D2)
    net.set_flag("math", "bf16")
    assert net.math == "bf16" and net.flatten.math == "bf16"


def test_table_models_match_reference_structure():
    from pytorch_bayesiancnn_b200.models import BBBAlexNet, BBBLeNet, BBB3Conv3FC, get_model
    a = BBBAlexNet(10, 3, CFG_PRIORS, "lrt", "softplus")
    assert [k for k, _ in a.named_children()] == ["conv1", "act1", "pool1", "conv2", "act2", "pool2", "conv3", "act3",
                                                  "conv4", "act4", "conv5", "act5", "pool3", "flatten", "classifier"]
    assert sum(p.numel() for p in a.parameters()) == 2 * 2175946
    assert sum(p.numel() for p in BBBLeNet(10, 3, None, "bbb", "relu").parameters()) == 2 * 62006
    assert sum(p.numel() for p in BBB3Conv3FC(10, 1, None).parameters()) == 2 * 1781034
    assert a.num_classes == 10
    with pytest.raises(ValueError):
        BBBAlexNet(10, 3, None, "nope")
    with pytest.raises(ValueError):
        get_model("resnet", 3, 10, None, "lrt", "relu")


def test_cpu_tensors_fail_loudly(built):
    import layers
    from pytorch_bayesiancnn_b200 import EngineError
    lin = layers.BBB_Linear(4, 2)
    if lin.W_mu.is_cuda:
        pytest.skip("GPU present")
    with pytest.raises(EngineError, match="no CPU fallback"):
        lin(torch.randn(3, 4))
    with pytest.raises(EngineError):
        lin.kl_loss()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "pytorch_bayesiancnn_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "oracle" not in src.replace("# checker", ""), f
    for f in ("layers/__init__.py",):
        assert "oracle" not in open(os.path.join(ROOT, f)).read()


def test_fused_planner_matches_reference_child_lists():
    """fused.plan() pattern-matches the (unmodified) child list of the model files."""
    from pytorch_bayesiancnn_b200 import fused, _lib as L
    from pytorch_bayesiancnn_b200.models import BBBAlexNet, BBBLeNet, BBB3Conv3FC
    for variant in ("lrt", "bbb"):
        net = BBBAlexNet(10, 3, CFG_PRIORS, variant, "softplus")
        net.set_flag("math", "bf16")
        steps = fused.plan(list(net.children()), (512, 3, 32, 32))
        assert steps is not None and len(steps) == 6
        assert [s.pool for s in steps] == [True, True, False, False, True, False]
        assert [s.act for s in steps] == [L.ACT_SOFTPLUS] * 5 + [L.ACT_NONE]
        assert [s.out_chw for s in steps] == [(64, 4, 4), (192, 2, 2), (384, 2, 2), (256, 2, 2), (128, 1, 1), (10, 1, 1)]
        assert steps[0].in_layout == L.LAYOUT_NCHW_F32 and all(s.in_layout == L.LAYOUT_PACKED_BF16 for s in steps[1:])
        assert steps[-1].out_layout == L.LAYOUT_ROWMAJOR_F32 and steps[-1].linear and steps[-1].prev_hw == 1
    # 3x3 stride-2 pools (Bayesian3Conv3FC.py:38) and 6-channel maps (LeNet) are not fusable -> plain path
    n3 = BBB3Conv3FC(10, 1, CFG_PRIORS); n3.set_flag("math", "bf16")
    assert fused.plan(list(n3.children()), (8, 1, 32, 32)) is None
    nl = BBBLeNet(10, 3, CFG_PRIORS); nl.set_flag("math", "bf16")
    assert fused.plan(list(nl.children()), (8, 3, 32, 32)) is None
    # set_flag invalidates cached plans (a net first run in fp32 must still fuse after switching to bf16)
    net.__dict__["_fused_plans"] = {(8, 3, 32, 32): None}
    net.set_flag("math", "bf16")
    assert "_fused_plans" not in net.__dict__
    # the default math is 'auto' (tensor-core path where the shape fits): a plain drop-in user gets the fused chain;
    # 'fp32' (exact-arithmetic CUDA-core kernels) is never fused
    na = BBBAlexNet(10, 3, CFG_PRIORS)
    assert na.conv1.math == "auto" and fused.plan(list(na.children()), (8, 3, 32, 32)) is not None
    na.set_flag("math", "fp32")
    assert fused.plan(list(na.children()), (8, 3, 32, 32)) is None


def test_workspace_slot_context_nests_and_restores():
    """Layer workspaces are keyed per slot so that forwards replayed concurrently on different streams never
    share prepared operand tiles / KL counters (functional.workspace_slot, GraphedForward(ws_slot=...))."""
    import inspect
    from pytorch_bayesiancnn_b200 import functional as Fn
    from pytorch_bayesiancnn_b200.graph import GraphedForward
    assert Fn._ws_slot == 0
    with Fn.workspace_slot(2):
        assert Fn._ws_slot == 2
        with Fn.workspace_slot(5):
            assert Fn._ws_slot == 5
        assert Fn._ws_slot == 2
    assert Fn._ws_slot == 0
    try:
        with Fn.workspace_slot(3):
            raise RuntimeError("boom")
    except RuntimeError:
        pass
    assert Fn._ws_slot == 0
    sig = inspect.signature(GraphedForward.__init__).parameters
    assert "static_inputs" in sig and "ws_slot" in sig and sig["ws_slot"].default == 0
