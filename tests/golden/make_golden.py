"""Generate tests/golden/*.npz by running the UNMODIFIED reference (williamyang1991/VToonify) on CPU
through its sanctioned ``model/stylegan/op_cpu`` path (model/stylegan/op_cpu/readme.md), with the deterministic
weights of vtoonify_b200/weights.py.  Needs a checkout of the reference; the tests only read the stored fixtures:

    python tests/golden/make_golden.py <path to a VToonify checkout>

The fixtures pin oracle/vt_oracle.py (tests/test_oracle_golden.py) and the CUDA path (tests/test_gpu_*.py).
"""
import importlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
if len(sys.argv) != 2:
    sys.exit(__doc__)
sys.path.insert(0, os.path.abspath(sys.argv[1]))

op_cpu = importlib.import_module("model.stylegan.op_cpu")
sys.modules["model.stylegan.op"] = op_cpu            # what op_cpu/readme.md prescribes, without editing files
from model.stylegan import model as ref_model         # noqa: E402
from model import dualstylegan as ref_dual            # noqa: E402
from model.vtoonify import VToonify as RefVToonify    # noqa: E402
from model.vtoonify import Fusion as RefFusion        # noqa: E402

from vtoonify_b200.weights import det_inputs, det_state_dict  # noqa: E402

torch.set_grad_enabled(False)


def save(name, **arrays):
    arrays = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrays.items()}
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"{name}.npz  {os.path.getsize(path) / 1024:.0f} KiB")


def gen(seed):
    g = torch.Generator()
    g.manual_seed(seed)
    return g


# ---------------------------------------------------------------------------------------------- a1
UPFIRDN_CASES = [
    # (B, C, H, W, kernel, up, down, pad)   kernel: "1331" separable sum-1 (x gain) or "rand_khxkw"
    (2, 3, 9, 11, "1331x4", 1, 1, (1, 1)),          # Blur after up-conv (mode 1)
    (2, 3, 8, 10, "1331x4", 2, 1, (2, 1)),          # Upsample (ToRGB skip, mode 3)
    (1, 4, 12, 16, "1331", 1, 2, (1, 1)),           # Downsample (mode 5)
    (1, 2, 10, 10, "1331", 1, 1, (2, 2)),           # Blur before down-conv
    (1, 2, 7, 9, "1331x4", 2, 1, (-1, 3)),          # negative pad = crop
    (1, 2, 16, 13, "rand_3x5", (2, 1), (1, 2), (1, 2, 0, 3)),   # per-axis up/down, 4-tuple pad, asymmetric kernel
    (1, 1, 6, 6, "rand_1x12", (2, 1), 1, (6, 5, 0, 0)),        # simple_augment-style 1x12 wavelet row filter
    (1, 3, 5, 4, "rand_4x4", 3, 2, (2, 3, 1, -1)),              # up=3, down=2, mixed-sign pads
    (3, 1, 1, 1, "rand_2x2", 1, 1, (1, 1)),                     # 1x1 input
]


def make_kernel_spec(spec, g):
    if spec.startswith("1331"):
        k = ref_model.make_kernel([1, 3, 3, 1])
        if spec.endswith("x4"):
            k = k * 4
        return k
    kh, kw = spec.split("_")[1].split("x")
    return torch.randn((int(kh), int(kw)), generator=g)


def golden_ops():
    out = {}
    for i, (B, C, H, W, ks, up, down, pad) in enumerate(UPFIRDN_CASES):
        g = gen(100 + i)
        x = torch.randn((B, C, H, W), generator=g)
        k = make_kernel_spec(ks, g)
        y = op_cpu.upfirdn2d(x, k, up=up, down=down, pad=pad)
        out[f"u{i}_x"], out[f"u{i}_k"], out[f"u{i}_y"] = x, k, y
        out[f"u{i}_cfg"] = np.array(json.dumps({"up": up, "down": down, "pad": pad}))
    out["n_upfirdn"] = len(UPFIRDN_CASES)
    # a2
    g = gen(200)
    x4 = torch.randn((2, 5, 6, 7), generator=g); b5 = torch.randn(5, generator=g)
    x2 = torch.randn((3, 8), generator=g); b8 = torch.randn(8, generator=g)
    out["f0_x"], out["f0_b"], out["f0_y"] = x4, b5, op_cpu.fused_leaky_relu(x4, b5)
    out["f1_x"], out["f1_b"], out["f1_y"] = x2, b8, op_cpu.fused_leaky_relu(x2, b8)
    out["f2_x"], out["f2_y"] = x4, op_cpu.fused_leaky_relu(x4, None, 0.2, 1.0)
    out["f3_x"], out["f3_b"], out["f3_y"] = x4, b5, op_cpu.fused_leaky_relu(x4, b5, negative_slope=0.1, scale=0.5)
    save("ops", **out)


# ---------------------------------------------------------------------------------------------- a3-a5, a7
def golden_layers():
    out = {}
    B = 2
    # StyledConv plain / up, ToRGB with skip — small channel counts, per-sample styles, real noise
    for name, (cin, cout, up, hw) in {"sc_plain": (32, 64, False, (12, 10)), "sc_up": (64, 32, True, (6, 5)),
                                       "sc_plain512": (512, 512, False, (4, 4))}.items():
        m = ref_model.StyledConv(cin, cout, 3, 512, upsample=up).eval()
        m.load_state_dict(det_state_dict(m, seed=7))
        g = gen(hash(name) % 1000)
        x = torch.randn((B, cin, *hw), generator=g)
        s = torch.randn((B, 512), generator=g)
        oh, ow = (hw[0] * 2, hw[1] * 2) if up else hw
        noise = torch.randn((B, 1, oh, ow), generator=g)
        out[name + "_x"], out[name + "_s"], out[name + "_noise"] = x, s, noise
        out[name + "_y"] = m(x, s, noise=noise)
        out[name + "_yconv"] = m.conv(x, s)
    m = ref_model.ToRGB(64, 512).eval()
    m.load_state_dict(det_state_dict(m, seed=7))
    g = gen(31)
    x = torch.randn((B, 64, 8, 12), generator=g); s = torch.randn((B, 512), generator=g)
    skip = torch.randn((B, 3, 4, 6), generator=g)
    out["rgb_x"], out["rgb_s"], out["rgb_skip"] = x, s, skip
    out["rgb_y"], out["rgb_y_noskip"] = m(x, s, skip), m(x, s)
    # ModulatedConv2d downsample branch
    m = ref_model.ModulatedConv2d(32, 32, 3, 512, downsample=True).eval()
    m.load_state_dict(det_state_dict(m, seed=7))
    x = torch.randn((B, 32, 10, 12), generator=g)
    out["mcd_x"], out["mcd_s"], out["mcd_y"] = x, s, m(x, s)
    # AdaResBlock (dilated) and Fusion
    m = ref_dual.AdaResBlock(64, dilation=2).eval()
    m.load_state_dict(det_state_dict(m, seed=7))
    x = torch.randn((B, 64, 9, 8), generator=g); s = torch.randn((B, 512), generator=g)
    out["ada_x"], out["ada_s"], out["ada_y"] = x, s, m(x, s, 0.6)
    m = RefFusion(32, 32, 32).eval()
    m.load_state_dict(det_state_dict(m, seed=7))
    fg = torch.randn((B, 32, 8, 8), generator=g); fe = torch.randn((B, 32, 8, 8), generator=g)
    fo, me = m(fg, fe, 0.5)
    out["fus_fg"], out["fus_fe"], out["fus_out"], out["fus_m"] = fg, fe, fo, me
    # EqualLinear / style MLP
    m = ref_model.EqualLinear(512, 512, lr_mul=0.01, activation="fused_lrelu").eval()
    m.load_state_dict(det_state_dict(m, seed=7))
    z = torch.randn((5, 512), generator=g)
    out["el_x"], out["el_y"] = z, m(z)
    out["pn_y"] = ref_model.PixelNorm()(z)
    save("layers", **out)


# ---------------------------------------------------------------------------------------------- a6
def golden_vtoonify():
    for backbone, tag in (("dualstylegan", "d"), ("toonify", "t")):
        m = RefVToonify(backbone=backbone).eval()
        keys = {k: list(v.shape) for k, v in m.state_dict().items()}
        with open(os.path.join(HERE, f"state_dict_keys_{tag}.json"), "w") as f:
            json.dump(keys, f, indent=0)
        m.load_state_dict(det_state_dict(m, seed=0), strict=True)
        out = {}
        for case, (B, H, W) in {"a": (2, 32, 32), "b": (1, 48, 40)}.items():
            x, style = det_inputs(B, H, W, seed=ord(case))
            if case == "a":   # per-sample distinct styles exercise the per-sample weight path
                style = style + 0.25 * torch.randn(style.shape, generator=gen(5))
            if backbone == "dualstylegan":
                y, masks = m(x, style, d_s=0.5, return_mask=True)
                for i, mk in enumerate(masks):
                    out[f"{case}_mask{i}"] = mk
            else:
                y = m(x, style, d_s=0.5)
            # x is not stored (it would push the file past 1 MB): tests/shapes.vtoonify_frames() redraws it from the same
            # seed and checks the redraw against every 16th value
            out[f"{case}_x_every16"], out[f"{case}_style"], out[f"{case}_y"] = x.reshape(-1)[::16], style, y
            print(tag, case, tuple(y.shape), "rms %.3f max %.3f" % (y.pow(2).mean().sqrt(), y.abs().max()))
        # zplus2wplus
        z = torch.randn((1, 18, 512), generator=gen(9))
        out["zplus"], out["wplus"] = z, m.zplus2wplus(z)
        save(f"vtoonify_{tag}", **out)


def golden_generator():
    m = ref_model.Generator(32, 512, 2).eval()
    m.load_state_dict(det_state_dict(m, seed=3))
    g = gen(77)
    latent = torch.randn((2, m.n_latent, 512), generator=g)
    img, _ = m([latent], input_is_latent=True, randomize_noise=False)
    z = torch.randn((2, 512), generator=g)
    img_z, _ = m([z], randomize_noise=False)
    save("generator32", latent=latent, y=img, z=z, y_from_z=img_z)
    print("generator32 rms %.3f" % img.pow(2).mean().sqrt())


def golden_psp():
    from argparse import Namespace
    from model.encoder.encoders.psp_encoders import GradualStyleEncoder
    m = GradualStyleEncoder(50, "ir_se", Namespace(input_nc=3, n_styles=18)).eval()
    keys = {k: list(v.shape) for k, v in m.state_dict().items()}
    with open(os.path.join(HERE, "state_dict_keys_psp.json"), "w") as f:
        json.dump(keys, f, indent=0)
    m.load_state_dict(det_state_dict(m, seed=11), strict=True)
    x = (torch.rand((1, 3, 256, 256), generator=gen(21)) * 2 - 1).half().float()   # stored as fp16, exactly reproducible
    y = m(x)
    print("psp", tuple(y.shape), "rms %.3f" % y.pow(2).mean().sqrt())
    save("psp", x=x.half(), y=y)


def golden_bisenet():
    """Face-parsing maps as the frame loop builds them (style_transfer.py:171-174). The reference constructor downloads
    ResNet-18 weights; here model_zoo.load_url is stubbed (no network) and every tensor comes from det_state_dict."""
    import torch.nn.functional as F
    import torch.utils.model_zoo as mz
    mz.load_url = lambda *a, **k: {}
    from model.bisenet.model import BiSeNet
    m = BiSeNet(n_classes=19).eval()
    keys = {k: list(v.shape) for k, v in m.state_dict().items()}
    with open(os.path.join(HERE, "state_dict_keys_bisenet.json"), "w") as f:
        json.dump(keys, f, indent=0)
    m.load_state_dict(det_state_dict(m, seed=21), strict=True)
    x = (torch.rand((2, 3, 64, 96), generator=gen(3)) * 2 - 1).half().float()
    x_p = F.interpolate(m(2 * F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=False))[0], scale_factor=0.5,
                        recompute_scale_factor=False)
    print("bisenet", tuple(x_p.shape), "rms %.3f" % x_p.pow(2).mean().sqrt())
    save("bisenet", x=x.half(), x_p=x_p)


if __name__ == "__main__":
    golden_ops()
    golden_layers()
    golden_generator()
    golden_vtoonify()
    golden_psp()
    golden_bisenet()
