"""Shared helpers for the parity tests (tests only; may import the oracle)."""
import numpy as np
import torch

CFG_PRIORS = {"prior_mu": 0, "prior_sigma": 0.1,
              "posterior_mu_initial": (0, 0.1), "posterior_rho_initial": (-5, 0.1)}
DEF_PRIORS = {"prior_mu": 0, "prior_sigma": 0.1,
              "posterior_mu_initial": (0, 0.1), "posterior_rho_initial": (-3, 0.1)}


def case_names(g):
    return sorted({k.split("/")[0] for k in g})


def load_case(g, name):
    d = {k.split("/", 1)[1]: g[k] for k in g if k.startswith(name + "/")}
    return {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) and v.dtype == np.float32 and v.ndim > 0 else v)
            for k, v in d.items()}


def scale_err(a: torch.Tensor, ref: torch.Tensor) -> float:
    """|a - ref|_max / |ref|_max -- the scale-relative error of SURVEY.md D9."""
    a, ref = a.detach().double().cpu(), ref.detach().double().cpu()
    return float((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def build_layer_from_case(name, c, device):
    """Instantiate OUR layer class for a golden layer case and load its params."""
    import pytorch_bayesiancnn_b200 as bbb
    bias = "bias_mu" in c
    priors = {"prior_mu": float(c["prior"][0]), "prior_sigma": float(c["prior"][1]),
              "posterior_mu_initial": (0, 0.1), "posterior_rho_initial": (-3, 0.1)}
    lrt = "_lrt_" in name
    W = c["W_mu"]
    if "conv" in c:
        s = [int(v) for v in c["conv"]]
        cls = bbb.BBB_LRT_Conv2d if lrt else bbb.BBB_Conv2d
        layer = cls(W.shape[1], W.shape[0], (W.shape[2], W.shape[3]), stride=(s[0], s[1]), padding=(s[2], s[3]),
                    dilation=(s[4], s[5]), bias=bias, priors=priors)
    else:
        cls = bbb.BBB_LRT_Linear if lrt else bbb.BBB_Linear
        layer = cls(W.shape[1], W.shape[0], bias=bias, priors=priors)
    with torch.no_grad():
        layer.W_mu.copy_(c["W_mu"]); layer.W_rho.copy_(c["W_rho"])
        if bias:
            layer.bias_mu.copy_(c["bias_mu"]); layer.bias_rho.copy_(c["bias_rho"])
    layer.set_flag("math", "fp32")            # exact-arithmetic kernels unless the test asks for the tensor-core path
    return layer.to(device)


def load_params_into(net, params):
    layers = [m for m in net.children() if hasattr(m, "W_mu")]
    assert len(layers) == len(params)
    with torch.no_grad():
        for m, p in zip(layers, params):
            m.W_mu.copy_(p["W_mu"]); m.W_rho.copy_(p["W_rho"])
            m.bias_mu.copy_(p["bias_mu"]); m.bias_rho.copy_(p["bias_rho"])
    net.set_flag("math", "fp32")                  # exact-arithmetic kernels unless the test asks for the tensor-core path
    return net
