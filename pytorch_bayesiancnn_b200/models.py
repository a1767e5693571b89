"""The three Bayesian architectures of the reference, as data.

The reference's model files (models/BayesianModels/BayesianAlexNet.py:8-53,
BayesianLeNet.py:8-49, Bayesian3Conv3FC.py:7-55) are constructor-only and run
UNCHANGED on top of this repo's ``layers`` package (tests/test_dropin.py checks
these tables against what those files build).  The package does not ship them, so the
benchmark and GPU tests build the same networks from the tables below: same
child names in the same order (=> same state_dict keys, same ModuleWrapper
iteration order), same constructor signature.
"""
from __future__ import annotations

from torch import nn

from .modules import (BBBConv2d, BBBLinear, BBBLRTConv2d, BBBLRTLinear, FlattenLayer, ModuleWrapper)

# child name -> spec.  c: (cout, k, stride, pad); p: (k, stride); f: flatten features; l: out features
_ARCH = {
    "alexnet": (("conv1", "c", (64, 11, 4, 5)), ("act1", "a"), ("pool1", "p", (2, 2)),
                ("conv2", "c", (192, 5, 1, 2)), ("act2", "a"), ("pool2", "p", (2, 2)),
                ("conv3", "c", (384, 3, 1, 1)), ("act3", "a"),
                ("conv4", "c", (256, 3, 1, 1)), ("act4", "a"),
                ("conv5", "c", (128, 3, 1, 1)), ("act5", "a"), ("pool3", "p", (2, 2)),
                ("flatten", "f", 128), ("classifier", "l", None)),
    "lenet": (("conv1", "c", (6, 5, 1, 0)), ("act1", "a"), ("pool1", "p", (2, 2)),
              ("conv2", "c", (16, 5, 1, 0)), ("act2", "a"), ("pool2", "p", (2, 2)),
              ("flatten", "f", 400), ("fc1", "l", 120), ("act3", "a"),
              ("fc2", "l", 84), ("act4", "a"), ("fc3", "l", None)),
    "3conv3fc": (("conv1", "c", (32, 5, 1, 2)), ("act1", "a"), ("pool1", "p", (3, 2)),
                 ("conv2", "c", (64, 5, 1, 2)), ("act2", "a"), ("pool2", "p", (3, 2)),
                 ("conv3", "c", (128, 5, 1, 1)), ("act3", "a"), ("pool3", "p", (3, 2)),
                 ("flatten", "f", 512), ("fc1", "l", 1000), ("act4", "a"),
                 ("fc2", "l", 1000), ("act5", "a"), ("fc3", "l", None)),
}


class _TableNet(ModuleWrapper):
    _key = None

    def __init__(self, outputs, inputs, priors, layer_type="lrt", activation_type="softplus"):
        super().__init__()
        self.num_classes = outputs
        self.layer_type = layer_type
        self.priors = priors
        if layer_type == "lrt":
            conv_cls, lin_cls = BBBLRTConv2d, BBBLRTLinear
        elif layer_type == "bbb":
            conv_cls, lin_cls = BBBConv2d, BBBLinear
        else:
            raise ValueError("Undefined layer_type")
        if activation_type == "softplus":
            self.act = nn.Softplus
        elif activation_type == "relu":
            self.act = nn.ReLU
        else:
            raise ValueError("Only softplus or relu supported")
        width = inputs
        for spec in _ARCH[self._key]:
            name, kind = spec[0], spec[1]
            if kind == "c":
                cout, k, s, p = spec[2]
                mod = conv_cls(width, cout, k, stride=s, padding=p, bias=True, priors=priors)
                width = cout
            elif kind == "a":
                mod = self.act()
            elif kind == "p":
                mod = nn.MaxPool2d(kernel_size=spec[2][0], stride=spec[2][1])
            elif kind == "f":
                mod = FlattenLayer(spec[2])
                width = spec[2]
            else:
                fout = outputs if spec[2] is None else spec[2]
                mod = lin_cls(width, fout, bias=True, priors=priors)
                width = fout
            setattr(self, name, mod)


class BBBAlexNet(_TableNet):
    _key = "alexnet"


class BBBLeNet(_TableNet):
    _key = "lenet"


class BBB3Conv3FC(_TableNet):
    _key = "3conv3fc"


def get_model(net_type, inputs, outputs, priors, layer_type, activation_type):
    """main_bayesian.py:22-30 (getModel)."""
    table = {"lenet": BBBLeNet, "alexnet": BBBAlexNet, "3conv3fc": BBB3Conv3FC}
    if net_type not in table:
        raise ValueError("Network should be either [LeNet / AlexNet / 3Conv3FC")
    return table[net_type](outputs, inputs, priors, layer_type, activation_type)
