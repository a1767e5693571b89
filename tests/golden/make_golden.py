"""Generate golden fixtures by running the UNMODIFIED reference project.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py <PyTorch-BayesianCNN checkout>

Imports the reference checkout given on the command line (read-only, never
copied into this repo), runs its layers / models on seeded inputs, recovers the
eps it drew by seed-replay of the global CPU generator (SURVEY.md 8c), and
writes small files next to this script.  The test-suite only reads the fixtures;
this script is committed so they are reproducible.

Fixtures (each file stays below 1 MB)
  layers_<kind>_<variant>.npz : per-layer cases (x, params, eps, y, kl) for
                conv/lin x bbb/lrt
  models.npz  : the three model files, both variants: x, logits, kl, and float64
                checksums of every parameter (params are re-drawn from the seed
                by oracle.init_params; the checksums prove the re-draw matches)
  dropin.json : what the model files need from the ``layers`` package (the names
                they import, their child list as ``layers`` exports / torch.nn
                types, state_dict keys and shapes), for the drop-in tests
  dropin.npz  : BBBLeNet, bbb layers, relu -- the one activation / variant pair of
                LeNet that models.npz lacks: x, logits, kl, parameter checksums
"""
import ast
import glob
import json
import os
import sys

sys.dont_write_bytecode = True
if len(sys.argv) != 2:
    raise SystemExit(__doc__)
REF = os.path.abspath(sys.argv[1])
HERE = os.path.dirname(os.path.abspath(__file__))
# the reference's layer files do `sys.path.append("..")` and import top-level
# `metrics`; run with the reference root first on sys.path, like `cd reference`.
sys.path.insert(0, REF)
os.chdir(REF)

import numpy as np
import torch

import layers as ref_layers                      # noqa: E402  (the reference's)
from models.BayesianModels.BayesianAlexNet import BBBAlexNet        # noqa: E402
from models.BayesianModels.BayesianLeNet import BBBLeNet            # noqa: E402
from models.BayesianModels.Bayesian3Conv3FC import BBB3Conv3FC      # noqa: E402
import config_bayesian as cfg                   # noqa: E402

torch.set_num_threads(1)        # oneDNN single-thread: deterministic reduction order

DEFAULT_PRIORS = None           # layer default: rho ~ N(-3, 0.1)
CFG_PRIORS = cfg.priors         # config_bayesian.py:4-9: rho ~ N(-5, 0.1)

# name, kind, variant, ctor args, ctor kwargs, x shape, priors, x distribution
LAYER_CASES = [
    ("conv_bbb_k3",      "conv", "bbb", (3, 8, 3),   dict(stride=1, padding=1),            (2, 3, 8, 8),   DEFAULT_PRIORS, "randn"),
    ("conv_bbb_k5s2",    "conv", "bbb", (4, 6, 5),   dict(stride=2, padding=2),            (3, 4, 11, 9),  CFG_PRIORS,     "rand"),
    ("conv_bbb_dil",     "conv", "bbb", (2, 5, 3),   dict(stride=1, padding=2, dilation=2), (2, 2, 9, 9),  DEFAULT_PRIORS, "randn"),
    ("conv_bbb_nobias",  "conv", "bbb", (3, 4, 3),   dict(padding=0, bias=False),          (2, 3, 6, 6),   DEFAULT_PRIORS, "randn"),
    ("conv_bbb_rect",    "conv", "bbb", (3, 4, (3, 5)), dict(padding=1),                   (2, 3, 7, 9),   DEFAULT_PRIORS, "randn"),
    ("conv_bbb_alex1",   "conv", "bbb", (3, 64, 11), dict(stride=4, padding=5),            (2, 3, 32, 32), CFG_PRIORS,     "rand"),
    ("conv_lrt_k3",      "conv", "lrt", (3, 8, 3),   dict(stride=1, padding=1),            (2, 3, 8, 8),   DEFAULT_PRIORS, "randn"),
    ("conv_lrt_k5s2",    "conv", "lrt", (4, 6, 5),   dict(stride=2, padding=2),            (3, 4, 11, 9),  CFG_PRIORS,     "rand"),
    ("conv_lrt_dil",     "conv", "lrt", (2, 5, 3),   dict(stride=1, padding=2, dilation=2), (2, 2, 9, 9),  DEFAULT_PRIORS, "randn"),
    ("conv_lrt_nobias",  "conv", "lrt", (3, 4, 3),   dict(padding=0, bias=False),          (2, 3, 6, 6),   DEFAULT_PRIORS, "randn"),
    ("conv_lrt_alex1",   "conv", "lrt", (3, 64, 11), dict(stride=4, padding=5),            (2, 3, 32, 32), CFG_PRIORS,     "rand"),
    ("conv_lrt_alex3",   "conv", "lrt", (48, 96, 3), dict(padding=1),                      (2, 48, 2, 2), CFG_PRIORS,     "rand"),
    ("lin_bbb_small",    "lin",  "bbb", (7, 5),      dict(),                               (3, 7),         DEFAULT_PRIORS, "randn"),
    ("lin_bbb_cls",      "lin",  "bbb", (128, 10),   dict(),                               (16, 128),      CFG_PRIORS,     "rand"),
    ("lin_bbb_nobias",   "lin",  "bbb", (33, 17),    dict(bias=False),                     (5, 33),        DEFAULT_PRIORS, "randn"),
    ("lin_lrt_small",    "lin",  "lrt", (7, 5),      dict(),                               (3, 7),         DEFAULT_PRIORS, "randn"),
    ("lin_lrt_cls",      "lin",  "lrt", (128, 10),   dict(),                               (16, 128),      CFG_PRIORS,     "rand"),
    ("lin_lrt_fc",       "lin",  "lrt", (400, 120),  dict(),                               (4, 400),       CFG_PRIORS,     "randn"),
    ("lin_lrt_nobias",   "lin",  "lrt", (33, 17),    dict(bias=False),                     (5, 33),        DEFAULT_PRIORS, "randn"),
]

MODEL_CASES = [
    # name, class, arch key, inputs, outputs, variant, act, batch
    ("alexnet_bbb",  BBBAlexNet,  "alexnet",  3, 10,  "bbb", "softplus", 4),
    ("alexnet_lrt",  BBBAlexNet,  "alexnet",  3, 10,  "lrt", "softplus", 4),
    ("alexnet100_lrt", BBBAlexNet, "alexnet", 3, 100, "lrt", "relu",     2),
    ("lenet_bbb",    BBBLeNet,    "lenet",    3, 10,  "bbb", "softplus", 4),
    ("lenet_lrt",    BBBLeNet,    "lenet",    3, 10,  "lrt", "relu",     4),
    ("3conv3fc_bbb", BBB3Conv3FC, "3conv3fc", 1, 10,  "bbb", "softplus", 3),
    ("3conv3fc_lrt", BBB3Conv3FC, "3conv3fc", 1, 10,  "lrt", "softplus", 3),
]
PARAM_SEED, X_SEED, EPS_SEED = 123, 0, 7


def make_x(shape, dist, seed):
    g = torch.Generator().manual_seed(seed)
    if dist == "rand":
        return torch.rand(shape, generator=g)
    return torch.randn(shape, generator=g)


def layer_case(name, kind, variant, args, kwargs, xshape, priors, dist, out):
    mods = {("conv", "bbb"): ref_layers.BBB_Conv2d, ("conv", "lrt"): ref_layers.BBB_LRT_Conv2d,
            ("lin", "bbb"): ref_layers.BBB_Linear, ("lin", "lrt"): ref_layers.BBB_LRT_Linear}
    torch.manual_seed(PARAM_SEED)
    layer = mods[(kind, variant)](*args, priors=priors, **kwargs)
    layer.train()
    x = make_x(xshape, dist, X_SEED)
    with torch.no_grad():
        torch.manual_seed(EPS_SEED)
        y = layer(x)
        kl = layer.kl_loss()
        # seed-replay: re-issue the same draws (BBB/BBBConv.py:63,68; BBB_LRT/BBBConv.py:78)
        torch.manual_seed(EPS_SEED)
        if variant == "bbb":
            eps_w = torch.empty(layer.W_mu.size()).normal_(0, 1)
            eps_b = torch.empty(layer.bias_mu.size()).normal_(0, 1) if layer.use_bias else None
        else:
            eps_y = torch.empty(y.size()).normal_(0, 1)
        # deterministic (mean-only) path: forward(x, sample=False) in eval mode
        layer.eval()
        y_mean = layer(x, sample=False)
    pre = name + "/"
    out[pre + "x"] = x.numpy()
    out[pre + "W_mu"] = layer.W_mu.detach().numpy()
    out[pre + "W_rho"] = layer.W_rho.detach().numpy()
    if layer.use_bias:
        out[pre + "bias_mu"] = layer.bias_mu.detach().numpy()
        out[pre + "bias_rho"] = layer.bias_rho.detach().numpy()
    if variant == "bbb":
        out[pre + "eps_w"] = eps_w.numpy()
        if eps_b is not None:
            out[pre + "eps_b"] = eps_b.numpy()
    else:
        out[pre + "eps_y"] = eps_y.numpy()
    out[pre + "y"] = y.numpy()
    out[pre + "y_mean"] = y_mean.numpy()
    out[pre + "kl"] = np.float32(kl.item())
    out[pre + "prior"] = np.array([layer.prior_mu, layer.prior_sigma], np.float64)
    if kind == "conv":
        def pair(v):
            return list(v) if isinstance(v, tuple) else [v, v]
        out[pre + "conv"] = np.array(pair(layer.stride) + pair(layer.padding) + pair(layer.dilation), np.int64)


def model_case(name, cls, key, inputs, outputs, variant, act, batch, out):
    torch.manual_seed(PARAM_SEED)
    net = cls(outputs, inputs, CFG_PRIORS, variant, act)
    net.train()
    x = make_x((batch, inputs, 32, 32), "randn", X_SEED)
    with torch.no_grad():
        torch.manual_seed(EPS_SEED)
        logits, kl = net(x)
    pre = name + "/"
    out[pre + "x"] = x.numpy()
    out[pre + "logits"] = logits.numpy()
    out[pre + "kl"] = np.float32(float(kl))
    out[pre + "meta"] = np.array([key, str(inputs), str(outputs), variant, act, str(batch)])
    sums = [float(p.detach().double().sum()) for _, p in net.named_parameters()]
    out[pre + "param_sums"] = np.array(sums, np.float64)
    out[pre + "param_names"] = np.array([n for n, _ in net.named_parameters()])


def layers_export(m):
    """The name under which the reference's ``layers`` package exports type(m), else the torch.nn type name."""
    for name in ref_layers.__all__ if hasattr(ref_layers, "__all__") else dir(ref_layers):
        if type(m) is getattr(ref_layers, name):
            return "layers." + name
    return "nn." + type(m).__name__


def dropin_structure():
    imports = set()
    for f in sorted(glob.glob(os.path.join(REF, "models", "BayesianModels", "*.py"))):
        for node in ast.walk(ast.parse(open(f).read())):
            if isinstance(node, ast.ImportFrom) and node.module == "layers":
                imports.update(a.name for a in node.names)
    nets = {}
    for cls, key, inputs in ((BBBAlexNet, "alexnet", 3), (BBBLeNet, "lenet", 3), (BBB3Conv3FC, "3conv3fc", 1)):
        for variant in ("lrt", "bbb"):
            net = cls(10, inputs, CFG_PRIORS, variant, "softplus")
            assert isinstance(net, ref_layers.ModuleWrapper)
            nets[f"{key}_{variant}"] = {
                "class": cls.__name__, "inputs": inputs, "variant": variant,
                "children": [f"{n} {layers_export(m)}" for n, m in net.named_children()],
                "state_dict": [f"{k} {'x'.join(map(str, v.shape))}" for k, v in net.state_dict().items()]}
        for bad in (dict(layer_type="nope"), dict(activation_type="nope")):
            try:
                cls(10, inputs, CFG_PRIORS, **bad)
            except ValueError:
                continue
            raise AssertionError(f"{cls.__name__}({bad}) did not raise ValueError")    # tests/test_dropin.py assumes it
    return {"layers_imports": sorted(imports), "nets": nets}


def main():
    lay = {}
    for c in LAYER_CASES:
        layer_case(*c, lay)
    for part in sorted({k.split("/")[0].rsplit("_", 1)[0] for k in lay}):       # conv_bbb, conv_lrt, lin_bbb, lin_lrt
        np.savez_compressed(os.path.join(HERE, f"layers_{part}.npz"),
                            **{k: v for k, v in lay.items() if k.split("/")[0].rsplit("_", 1)[0] == part})
    mod = {}
    for c in MODEL_CASES:
        model_case(*c, mod)
    np.savez_compressed(os.path.join(HERE, "models.npz"), **mod)
    drop = {}
    model_case("lenet_bbb_relu", BBBLeNet, "lenet", 3, 10, "bbb", "relu", 5, drop)
    np.savez_compressed(os.path.join(HERE, "dropin.npz"), **drop)
    with open(os.path.join(HERE, "dropin.json"), "w") as f:
        json.dump(dropin_structure(), f, indent=1)
        f.write("\n")
    for f in sorted(glob.glob(os.path.join(HERE, "*.npz")) + glob.glob(os.path.join(HERE, "*.json"))):
        print(os.path.basename(f), os.path.getsize(f))
    print("torch", torch.__version__)


if __name__ == "__main__":
    main()
