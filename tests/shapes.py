"""Shared test helpers: rebuild what the golden fixtures do not store, without the reference: the deterministic
state_dicts of the single-layer fixtures (shapes are those of the reference constructors used in
tests/golden/make_golden.py) and the input frames of the VToonify fixtures."""
import os

import numpy as np
import torch

from oracle import vt_oracle as O
from vtoonify_b200.weights import det_inputs, det_state_dict

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
K4 = O.make_kernel([1, 3, 3, 1])
VTOONIFY_CASES = {"a": (2, 32, 32), "b": (1, 48, 40)}      # (B, H, W) of the vtoonify_{d,t} golden cases


def vtoonify_frames(g, case):
    """Input frame batch ``x`` of a vtoonify_{d,t} golden case, redrawn from the seed make_golden.py used; the fixture
    keeps every 16th value of it to check the redraw."""
    B, H, W = VTOONIFY_CASES[case]
    x = det_inputs(B, H, W, seed=ord(case))[0]
    assert np.array_equal(x.reshape(-1)[::16].numpy(), g[f"{case}_x_every16"]), \
        f"det_inputs no longer redraws the frames of golden case {case}"
    return x


def _styled_conv_template(cin, cout, up):
    t = {"conv.weight": torch.empty(1, cout, cin, 3, 3), "conv.modulation.weight": torch.empty(cin, 512),
         "conv.modulation.bias": torch.empty(cin)}
    if up:
        t["conv.blur.kernel"] = K4 * 4
    t["noise.weight"] = torch.empty(1)
    t["activate.bias"] = torch.empty(cout)
    return t


def _convlayer(prefix, fin):
    return {prefix + "0.weight": torch.empty(fin, fin, 3, 3), prefix + "1.bias": torch.empty(fin)}


def layer_template(kind, name):
    if kind == "StyledConv":
        cin, cout, up = {"sc_plain": (32, 64, False), "sc_up": (64, 32, True), "sc_plain512": (512, 512, False)}[name]
        return _styled_conv_template(cin, cout, up)
    if kind == "ToRGB":
        return {"upsample.kernel": K4 * 4, "conv.weight": torch.empty(1, 3, 64, 1, 1),
                "conv.modulation.weight": torch.empty(64, 512), "conv.modulation.bias": torch.empty(64),
                "bias": torch.empty(1, 3, 1, 1)}
    if kind == "ModulatedConv2dDown":
        return {"weight": torch.empty(1, 32, 32, 3, 3), "blur.kernel": K4, "modulation.weight": torch.empty(32, 512),
                "modulation.bias": torch.empty(32)}
    if kind == "AdaResBlock":
        t = {}
        t.update(_convlayer("conv.", 64)); t.update(_convlayer("conv2.", 64))
        for n in ("norm.", "norm2."):
            t[n + "style.weight"] = torch.empty(128, 512); t[n + "style.bias"] = torch.empty(128)
        return t
    if kind == "Fusion":
        return {"conv.weight": torch.empty(32, 64, 3, 3), "conv.bias": torch.empty(32),
                "norm.style.weight": torch.empty(128, 128), "norm.style.bias": torch.empty(128),
                "conv2.weight": torch.empty(1, 64, 3, 3), "conv2.bias": torch.empty(1),
                "linear.0.weight": torch.empty(64, 1), "linear.0.bias": torch.empty(64),
                "linear.2.weight": torch.empty(128, 64), "linear.2.bias": torch.empty(128)}
    if kind == "EqualLinear":
        return {"weight": torch.empty(512, 512), "bias": torch.empty(512)}
    if kind == "Generator32":
        t = {}
        for i in (1, 2):
            t[f"style.{i}.weight"] = torch.empty(512, 512); t[f"style.{i}.bias"] = torch.empty(512)
        t["input.input"] = torch.empty(1, 512, 4, 4)
        for k, v in _styled_conv_template(512, 512, False).items():
            t["conv1." + k] = v
        t.update({"to_rgb1.bias": torch.empty(1, 3, 1, 1), "to_rgb1.conv.weight": torch.empty(1, 3, 512, 1, 1),
                  "to_rgb1.conv.modulation.weight": torch.empty(512, 512), "to_rgb1.conv.modulation.bias": torch.empty(512)})
        for lv in range(3):
            for k, v in _styled_conv_template(512, 512, True).items():
                t[f"convs.{2 * lv}." + k] = v
            for k, v in _styled_conv_template(512, 512, False).items():
                t[f"convs.{2 * lv + 1}." + k] = v
            t.update({f"to_rgbs.{lv}.bias": torch.empty(1, 3, 1, 1), f"to_rgbs.{lv}.upsample.kernel": K4 * 4,
                      f"to_rgbs.{lv}.conv.weight": torch.empty(1, 3, 512, 1, 1),
                      f"to_rgbs.{lv}.conv.modulation.weight": torch.empty(512, 512),
                      f"to_rgbs.{lv}.conv.modulation.bias": torch.empty(512)})
        for i in range(7):
            r = (i + 5) // 2
            t[f"noises.noise_{i}"] = torch.empty(1, 1, 2 ** r, 2 ** r)
        return t
    raise KeyError(kind)


def layer_state_dict(kind, name):
    seed = 3 if kind == "Generator32" else 7
    return det_state_dict(layer_template(kind, name), seed=seed)
