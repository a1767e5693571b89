"""The reference's UNMODIFIED model files (models/BayesianModels/*.py) as consumers of this repo's `layers` package,
checked against what tests/golden/make_golden.py recorded from the reference itself (tests/golden/dropin.*): the names
the files import from `layers`, the child list they build (as `layers` exports / torch.nn types), the state_dict keys
and shapes (so their checkpoints load here), and one of their forwards, run here on the engine."""
import json
import os

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN
from tests.util import CFG_PRIORS, load_case, load_params_into, scale_err

with open(os.path.join(GOLDEN, "dropin.json")) as f:
    DROPIN = json.load(f)


def _child(name, m):
    import layers
    for export in DROPIN["layers_imports"]:
        if type(m) is getattr(layers, export):
            return f"{name} layers.{export}"
    return f"{name} nn.{type(m).__name__}"


def test_reference_model_files_build_on_our_layers():
    import layers
    import pytorch_bayesiancnn_b200 as bbb
    from pytorch_bayesiancnn_b200 import models as ours
    assert all(hasattr(layers, n) for n in DROPIN["layers_imports"])
    assert len(DROPIN["nets"]) == 6
    for case, rec in DROPIN["nets"].items():
        cls = getattr(ours, rec["class"])
        net = cls(10, rec["inputs"], CFG_PRIORS, rec["variant"], "softplus")
        assert isinstance(net, bbb.ModuleWrapper)
        assert [_child(n, m) for n, m in net.named_children()] == rec["children"], case
        sd = net.state_dict()
        assert [f"{k} {'x'.join(map(str, v.shape))}" for k, v in sd.items()] == rec["state_dict"], case
        ckpt = {}                                                   # a checkpoint of the reference's layout loads strictly
        for line in rec["state_dict"]:
            k, shape = line.split(" ")
            ckpt[k] = torch.randn([int(d) for d in shape.split("x")])
        net.load_state_dict(ckpt)
        assert all(torch.equal(net.state_dict()[k].cpu(), v) for k, v in ckpt.items()), case
        with pytest.raises(ValueError):
            cls(10, rec["inputs"], CFG_PRIORS, "nope")
        with pytest.raises(ValueError):
            cls(10, rec["inputs"], CFG_PRIORS, rec["variant"], "nope")


@pytest.mark.gpu
def test_reference_model_files_run_on_the_engine():
    """BBBLeNet with bbb layers and relu, recorded by the reference on its CPU layers, against the same net on the engine
    with the reference's parameters and eps: the fp32 kernels at the whole-model bar; the default math with in-kernel
    noise runs and is finite."""
    import __graft_entry__ as g
    g.build()
    import pytorch_bayesiancnn_b200 as bbb
    from pytorch_bayesiancnn_b200.models import BBBLeNet
    from oracle import bbb_oracle as O
    dev = torch.device("cuda:0")
    with np.load(os.path.join(GOLDEN, "dropin.npz")) as z:
        c = load_case(z, "lenet_bbb_relu")
    key, inputs, outputs, variant, act, batch = [str(v) for v in c["meta"]]
    inputs, outputs, batch = int(inputs), int(outputs), int(batch)
    params = O.init_params(key, outputs, inputs, CFG_PRIORS, seed=123)
    sums = [float(p[k].double().sum()) for p in params for k in ("W_mu", "W_rho", "bias_mu", "bias_rho")]
    np.testing.assert_allclose(sums, c["param_sums"], rtol=0, atol=0)
    net = load_params_into(BBBLeNet(outputs, inputs, CFG_PRIORS, variant, act), params).to(dev).train()
    eps = O.draw_eps_like_reference(O.eps_shapes(key, outputs, inputs, variant, batch), seed=7)
    with torch.no_grad(), bbb.external_eps(eps):
        logits, kl = net(c["x"].to(dev))
    assert scale_err(logits, c["logits"]) < 1e-4
    assert abs(float(kl) - float(c["kl"])) <= 1e-5 * abs(float(c["kl"]))
    net.set_flag("math", "auto")
    with torch.no_grad():
        out, kl = net(torch.randn(batch, inputs, 32, 32, device=dev))
    assert out.shape == (batch, outputs) and kl.dim() == 0 and torch.isfinite(out).all()
