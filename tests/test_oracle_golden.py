"""CPU: pin oracle/vt_oracle.py against outputs of the unmodified reference (tests/golden/*.npz, produced by
tests/golden/make_golden.py from the reference's op_cpu path)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import vt_oracle as O
from vtoonify_b200.weights import det_state_dict
from tests.shapes import GOLDEN, layer_state_dict, vtoonify_frames

torch.set_grad_enabled(False)


def T(a):
    return torch.from_numpy(np.asarray(a))


def assert_close(a, b, atol, what):
    err = (a - b).abs().max().item()
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    assert err <= atol, f"{what}: max abs err {err:.3e} > {atol:.1e}"


def test_upfirdn2d_golden(golden):
    g = golden("ops")
    for i in range(int(g["n_upfirdn"])):
        cfg = json.loads(str(g[f"u{i}_cfg"]))
        up = tuple(cfg["up"]) if isinstance(cfg["up"], list) else cfg["up"]
        down = tuple(cfg["down"]) if isinstance(cfg["down"], list) else cfg["down"]
        y = O.upfirdn2d(T(g[f"u{i}_x"]), T(g[f"u{i}_k"]), up, down, tuple(cfg["pad"]))
        assert_close(y, T(g[f"u{i}_y"]), 2e-6, f"upfirdn2d case {i} {cfg}")


def test_fused_leaky_relu_golden(golden):
    g = golden("ops")
    assert torch.equal(O.fused_leaky_relu(T(g["f0_x"]), T(g["f0_b"])), T(g["f0_y"]))
    assert torch.equal(O.fused_leaky_relu(T(g["f1_x"]), T(g["f1_b"])), T(g["f1_y"]))
    assert torch.equal(O.fused_leaky_relu(T(g["f2_x"]), None, 0.2, 1.0), T(g["f2_y"]))
    assert torch.equal(O.fused_leaky_relu(T(g["f3_x"]), T(g["f3_b"]), 0.1, 0.5), T(g["f3_y"]))


@pytest.mark.parametrize("name,up", [("sc_plain", False), ("sc_up", True), ("sc_plain512", False)])
def test_styled_conv_golden(golden, name, up):
    g = golden("layers")
    sd = layer_state_dict("StyledConv", name)
    y = O.styled_conv(T(g[name + "_x"]), T(g[name + "_s"]), sd, "", T(g[name + "_noise"]), upsample=up)
    assert_close(y, T(g[name + "_y"]), 2e-5, name)
    yc = O.modulated_conv2d(T(g[name + "_x"]), T(g[name + "_s"]), sd, "conv.", upsample=up)
    assert_close(yc, T(g[name + "_yconv"]), 2e-5, name + " conv")


def test_to_rgb_golden(golden):
    g = golden("layers")
    sd = layer_state_dict("ToRGB", "rgb")
    assert_close(O.to_rgb(T(g["rgb_x"]), T(g["rgb_s"]), sd, "", T(g["rgb_skip"])), T(g["rgb_y"]), 1e-5, "to_rgb+skip")
    assert_close(O.to_rgb(T(g["rgb_x"]), T(g["rgb_s"]), sd, ""), T(g["rgb_y_noskip"]), 1e-5, "to_rgb")


def test_modconv_down_golden(golden):
    g = golden("layers")
    sd = layer_state_dict("ModulatedConv2dDown", "mcd")
    y = O.modulated_conv2d(T(g["mcd_x"]), T(g["mcd_s"]), sd, "", downsample=True)
    assert_close(y, T(g["mcd_y"]), 2e-5, "modconv down")


def test_adares_fusion_linear_golden(golden):
    g = golden("layers")
    sd = layer_state_dict("AdaResBlock", "ada")
    assert_close(O.ada_res_block(T(g["ada_x"]), T(g["ada_s"]), 0.6, sd, "", 2), T(g["ada_y"]), 2e-5, "AdaResBlock")
    sd = layer_state_dict("EqualLinear", "el")
    assert_close(O.equal_linear(T(g["el_x"]), sd["weight"], sd["bias"], 0.01, True), T(g["el_y"]), 1e-5, "EqualLinear")
    assert_close(O.pixel_norm(T(g["el_x"])), T(g["pn_y"]), 1e-6, "PixelNorm")


def test_generator_golden(golden):
    g = golden("generator32")
    sd = layer_state_dict("Generator32", "gen")
    noises = [sd[f"noises.noise_{i}"] for i in range(7)]
    y = O.generator_forward(sd, T(g["latent"]), noises)
    assert_close(y, T(g["y"]), 5e-5, "Generator(32)")
    # z -> w through the mapping MLP (PixelNorm + n_mlp EqualLinear(lr_mul 0.01, fused_lrelu)), model.py:409-417
    w = O.pixel_norm(T(g["z"]))
    for i in (1, 2):
        w = O.equal_linear(w, sd[f"style.{i}.weight"], sd[f"style.{i}.bias"], 0.01, True)
    y2 = O.generator_forward(sd, w.unsqueeze(1).repeat(1, 8, 1), noises)
    assert_close(y2, T(g["y_from_z"]), 5e-5, "Generator(32) from z")


@pytest.mark.parametrize("tag,backbone", [("d", "dualstylegan"), ("t", "toonify")])
def test_vtoonify_golden(golden, tag, backbone):
    g = golden(f"vtoonify_{tag}")
    keys = json.load(open(os.path.join(GOLDEN, f"state_dict_keys_{tag}.json")))
    sd = det_state_dict({k: torch.empty(v) for k, v in keys.items()}, seed=0)
    # FIR buffers are architecture constants, not random (weights.py keeps the template value)
    for k in sd:
        if k.endswith("blur.kernel") or k.endswith("upsample.kernel"):
            sd[k] = O.make_kernel([1, 3, 3, 1]) * 4
    for case in ("a", "b"):
        x, style = vtoonify_frames(g, case), T(g[f"{case}_style"])
        if backbone == "dualstylegan":
            y, masks = O.vtoonify_forward(sd, x, style, 0.5, backbone, return_mask=True)
            for i, m in enumerate(masks):
                assert_close(m, T(g[f"{case}_mask{i}"]), 5e-5, f"{tag}/{case} mask {i}")
        else:
            y = O.vtoonify_forward(sd, x, style, 0.5, backbone)
        ref = T(g[f"{case}_y"])
        assert_close(y, ref, 1e-4, f"VToonify-{tag} case {case} (ref rms {ref.pow(2).mean().sqrt():.3f})")


def test_frame_transforms():
    g = torch.Generator().manual_seed(0)
    u8 = torch.randint(0, 256, (2, 5, 7, 3), generator=g, dtype=torch.uint8)
    f = O.frame_u8_to_f32(u8)
    ref = ((u8.numpy().astype(np.float32) / 255.0) - 0.5) / 0.5
    assert np.array_equal(f.permute(0, 2, 3, 1).numpy(), ref)
    img = torch.randn((2, 3, 5, 7), generator=g) * 1.5
    out = O.tensor2frame_u8(img, swap_rb=True).numpy()
    c = np.clip(img.numpy(), -1, 1).transpose(0, 2, 3, 1)
    ref8 = ((c + 1.0) * 127.5).astype(np.uint8)[..., ::-1]
    assert np.array_equal(out, ref8)


def test_psp_encoder_golden(golden):
    """a10: pSp GradualStyleEncoder(50, 'ir_se') restated functionally vs the reference module's output."""
    g = golden("psp")
    keys = json.load(open(os.path.join(GOLDEN, "state_dict_keys_psp.json")))
    sd = det_state_dict({k: torch.empty(v, dtype=torch.long if k.endswith("num_batches_tracked") else torch.float32)
                         for k, v in keys.items()}, seed=11)
    y = O.psp_forward(sd, T(g["x"]).float())
    ref = T(g["y"])
    assert_close(y, ref, 1e-4 * ref.abs().max().item(), "pSp encoder")


def test_bisenet_parsing_golden(golden):
    """Next row (f): BiSeNet parsing maps of the frame loop (2x bilinear up-sampling, BiSeNet, nearest back to frame size),
    restated functionally from the state_dict, vs the reference module's output."""
    g = golden("bisenet")
    keys = json.load(open(os.path.join(GOLDEN, "state_dict_keys_bisenet.json")))
    sd = det_state_dict({k: torch.empty(v, dtype=torch.long if k.endswith("num_batches_tracked") else torch.float32)
                         for k, v in keys.items()}, seed=21)
    y = O.parsing_for_vtoonify(sd, T(g["x"]).float())
    ref = T(g["x_p"])
    assert tuple(y.shape) == (2, 19, 64, 96)
    assert_close(y, ref, 1e-4 * ref.abs().max().item(), "BiSeNet parsing maps")


def test_frame_prefilter_resize_matches_opencv(golden):
    """f3: the oracle's integer restatement of cv2.sepFilter2D / cv2.resize (style_transfer.py:124-130) is bit-exact with the
    OpenCV outputs stored by tests/golden/make_golden_frames.py"""
    g = golden("frame_prep")
    for i in range(int(g["n_cases"])):
        f = g[f"c{i}_frame"]
        scale, w, h, top, bottom, left, right = g[f"c{i}_params"]
        cur = f
        if f"c{i}_blur1" in g.files:
            cur = O.sep_filter_1331_u8(cur)
            assert np.array_equal(cur, g[f"c{i}_blur1"]), f"case {i}: first blur differs from cv2.sepFilter2D"
        if f"c{i}_blur2" in g.files:
            cur = O.sep_filter_1331_u8(cur)
            assert np.array_equal(cur, g[f"c{i}_blur2"]), f"case {i}: second blur differs"
        assert np.array_equal(O.resize_linear_u8(cur, int(w), int(h)), g[f"c{i}_resized"]), f"case {i}: resize differs from cv2.resize"
        out = O.prefilter_resize_crop(f, float(scale), (int(w), int(h)), (int(top), int(bottom), int(left), int(right)))
        assert np.array_equal(out, g[f"c{i}_out"])
