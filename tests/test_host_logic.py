"""CPU: host-side logic — state_dict contract, deterministic weights, tap tables, frame sharding, product/oracle separation."""
import json
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("tag,backbone", [("d", "dualstylegan"), ("t", "toonify")])
def test_state_dict_contract(tag, backbone):
    """Same keys, order and shapes as the reference constructor (SURVEY App. A) => load_state_dict(ckpt['g_ema']) strict."""
    from vtoonify_b200.vtoonify import VToonify
    keys = json.load(open(os.path.join(ROOT, "tests", "golden", f"state_dict_keys_{tag}.json")))
    sd = VToonify(backbone=backbone).state_dict()
    assert list(sd.keys()) == list(keys.keys())
    for k, v in sd.items():
        assert list(v.shape) == keys[k], k
    assert len(sd) == {"d": 399, "t": 229}[tag]


def test_generator_constructor_defaults_match_reference_init():
    from vtoonify_b200.stylegan import Generator, ModulatedConv2d
    g = Generator(64, 512, 2)
    assert g.n_latent == 10 and g.num_layers == 9 and len(g.convs) == 8 and len(g.to_rgbs) == 4
    m = ModulatedConv2d(8, 8, 3, 512, upsample=True)
    assert m.blur.pad == (1, 1) and torch.allclose(m.blur.kernel.sum(), torch.tensor(4.0))
    assert torch.all(m.modulation.bias == 1) and m.scale == pytest.approx(1 / np.sqrt(72))
    d = ModulatedConv2d(8, 8, 3, 512, downsample=True)
    assert d.blur.pad == (2, 2) and torch.allclose(d.blur.kernel.sum(), torch.tensor(1.0))


def test_det_weights_reproducible_and_scaled():
    from vtoonify_b200.weights import det_inputs, det_state_dict
    t = {"a.conv.weight": torch.empty(1, 4, 4, 3, 3), "a.conv.modulation.bias": torch.empty(4),
         "enc.weight": torch.empty(8, 4, 3, 3), "x.blur.kernel": torch.ones(4, 4)}
    s1, s2, s3 = det_state_dict(t, 0), det_state_dict(t, 0), det_state_dict(t, 1)
    assert all(torch.equal(s1[k], s2[k]) for k in t)
    assert not torch.equal(s1["enc.weight"], s3["enc.weight"])
    assert torch.equal(s1["x.blur.kernel"], torch.ones(4, 4))
    assert abs(s1["a.conv.modulation.bias"].mean().item() - 1.0) < 0.3
    x, s = det_inputs(2, 16, 8)
    assert x.shape == (2, 22, 16, 8) and s.shape == (2, 18, 512) and torch.equal(s[0], s[1])
    assert x[:, :3].abs().max() <= 1.0


def test_conv_tap_tables_reproduce_conv2d_indexing():
    """ops.conv_taps/conv_out_size describe F.conv2d exactly (checked by evaluating the tap table in numpy)."""
    from vtoonify_b200 import ops
    g = torch.Generator().manual_seed(0)
    for k, stride, pad, dil in [(3, 1, 1, 1), (3, 2, 1, 1), (3, 1, 4, 4), (1, 1, 0, 1), (3, 1, 2, 2), (3, 2, 0, 1)]:
        x = torch.randn((1, 2, 9, 11), generator=g); w = torch.randn((3, 2, k, k), generator=g)
        ref = F.conv2d(x, w, stride=stride, padding=pad, dilation=dil)
        Ho, Wo = ops.conv_out_size(9, k, stride, pad, dil), ops.conv_out_size(11, k, stride, pad, dil)
        assert ref.shape[2:] == (Ho, Wo)
        out = torch.zeros((1, 3, Ho, Wo))
        for dy, dx, tw in ops.conv_taps(k, pad, dil):
            ky, kx = tw // k, tw % k
            for oy in range(Ho):
                for ox in range(Wo):
                    iy, ix = oy * stride + dy, ox * stride + dx
                    if 0 <= iy < 9 and 0 <= ix < 11:
                        out[0, :, oy, ox] += w[:, :, ky, kx] @ x[0, :, iy, ix]
        assert (out - ref).abs().max() < 1e-5


def test_polyphase_taps_reproduce_conv_transpose():
    g = torch.Generator().manual_seed(1)
    x = torch.randn((1, 2, 4, 5), generator=g); w = torch.randn((3, 2, 3, 3), generator=g)   # [Cout, Cin, k, k]
    ref = F.conv_transpose2d(x, w.transpose(0, 1), stride=2)
    H, W = 4, 5
    out = torch.zeros((1, 3, 2 * H + 1, 2 * W + 1))
    for py in (0, 1):
        for px in (0, 1):
            taps = [(-(ky - py) // 2, -(kx - px) // 2, ky * 3 + kx) for ky in range(py, 3, 2) for kx in range(px, 3, 2)]
            Ho, Wo = (H + 1 if py == 0 else H), (W + 1 if px == 0 else W)
            for oy in range(Ho):
                for ox in range(Wo):
                    for dy, dx, tw in taps:
                        iy, ix = oy + dy, ox + dx
                        if 0 <= iy < H and 0 <= ix < W:
                            out[0, :, 2 * oy + py, 2 * ox + px] += w[:, :, tw // 3, tw % 3] @ x[0, :, iy, ix]
    assert (out - ref).abs().max() < 1e-5


def test_round_robin_sharding():
    from vtoonify_b200.frame_loop import merge_order, shard_indices
    for n, world in [(225, 8), (7, 2), (3, 4), (8, 8)]:
        shards = [shard_indices(n, r, world) for r in range(world)]
        assert sorted(i for s in shards for i in s) == list(range(n))
        assert max(len(s) for s in shards) - min(len(s) for s in shards) <= 1
        order = merge_order(n, world)
        assert [shards[r][j] for r, j in order] == list(range(n))


def test_product_never_imports_oracle():
    """The shipped package must not route through oracle/ or /root/reference (parity claims depend on it)."""
    pkg = os.path.join(ROOT, "vtoonify_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "/root/reference" not in src, f


def test_ops_reject_cpu_tensors_without_gpu():
    from vtoonify_b200 import _lib, ops
    with pytest.raises(_lib.VtError, match="no CPU fallback"):
        ops.fused_bias_act(torch.zeros(1, 2, 3, 3), None, 0.2, 1.0)
    with pytest.raises(_lib.VtError):
        ops.to_nhwc(torch.zeros(1, 2, 3, 3))


def test_psp_state_dict_contract():
    """a10: GradualStyleEncoder(50, 'ir_se') has the reference's 621 keys/shapes (load_psp_standalone loads it strict)."""
    from argparse import Namespace
    from vtoonify_b200.psp import GradualStyleEncoder, get_blocks
    keys = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_keys_psp.json")))
    sd = GradualStyleEncoder(50, "ir_se", Namespace(input_nc=3, n_styles=18)).state_dict()
    assert list(sd.keys()) == list(keys.keys()) and len(sd) == 621
    assert all(list(sd[k].shape) == keys[k] for k in keys)
    cfg = get_blocks(50)
    assert len(cfg) == 24 and [i for i, c in enumerate(cfg) if c[2] == 2] == [0, 3, 7, 21]


def test_precision_and_algorithm_switches():
    """Host-side configuration: the product precision is the split-bf16 mode (the one that meets the 1e-3 bar); the up-conv
    formulation is chosen per layer by input channels; unknown names fail loudly."""
    import pytest
    from vtoonify_b200 import ops
    assert ops.DEFAULT_PRECISION == "bf16x3" and ops.get_precision() == "bf16x3"
    old = ops.set_precision("tf32")
    try:
        assert old == "bf16x3" and ops.get_precision() == "tf32"
        assert ops.scale_fusable() is False            # f_E * m_E fusion needs the operand-transform warps of the bf16x3 mode
    finally:
        ops.set_precision(ops.DEFAULT_PRECISION)
    assert ops.scale_fusable() is True
    with pytest.raises(ValueError):
        ops.set_precision("fp16")
    with pytest.raises(KeyError):
        ops.set_option("no_such_option", 1)
    thr = ops.get_option("fold_upconv")
    assert ops.use_folded_upconv(64) and ops.use_folded_upconv(int(thr)) and not ops.use_folded_upconv(512)
    ops.set_option("fold_upconv", True)
    try:
        assert ops.use_folded_upconv(512)
    finally:
        ops.set_option("fold_upconv", thr)


def test_bisenet_state_dict_keys_and_host_algebra():
    """Next row (f): the BiSeNet module has the reference's 191 keys / shapes, and its host-side weight algebra is exact:
    (1) the stride-2 7x7 stem equals a stride-1 4x4 convolution over the space-to-depth tensor with the re-indexed weights
    and tap list the module feeds to the tensor-core kernel, (2) conv + eval BatchNorm equals the folded conv + bias."""
    import json
    import torch
    import torch.nn.functional as F
    from vtoonify_b200.bisenet import BiSeNet, S2D_TAPS, fold_bn, s2d_stem_weight
    from vtoonify_b200.psp import BatchNorm2d
    m = BiSeNet(19)
    keys = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_keys_bisenet.json")))
    sd = m.state_dict()
    assert list(sd.keys()) == list(keys.keys()) and all(list(sd[k].shape) == keys[k] for k in keys)

    g = torch.Generator().manual_seed(0)
    for (H, W) in ((12, 16), (11, 15)):                       # even and odd sizes (zero rows beyond X)
        x = torch.randn((2, 3, H, W), generator=g)
        w7 = torch.randn((5, 3, 7, 7), generator=g)
        ref = F.conv2d(x, w7, stride=2, padding=3)
        Ho, Wo = (H + 1) // 2, (W + 1) // 2
        xp = F.pad(x, (0, 2 * Wo - W, 0, 2 * Ho - H))
        z = torch.stack([xp[:, :, py::2, px::2] for py in (0, 1) for px in (0, 1)], dim=1).reshape(2, 12, Ho, Wo)
        w4 = s2d_stem_weight(w7)
        # evaluate exactly what the kernel is asked for: out[oy,ox] = sum_t sum_c z[oy+dy_t, ox+dx_t, c] * w4[:, c, slab_t]
        zp = F.pad(z, (2, 2, 2, 2))
        out = torch.zeros_like(ref)
        for dy, dx, t in S2D_TAPS:
            patch = zp[:, :, 2 + dy:2 + dy + Ho, 2 + dx:2 + dx + Wo]
            out += torch.einsum("bchw,nc->bnhw", patch, w4[:, :, t // 4, t % 4])
        assert out.shape == ref.shape and (out - ref).abs().max().item() <= 1e-4

    bn = BatchNorm2d(6)
    bn.weight.data = torch.randn(6, generator=g); bn.bias.data = torch.randn(6, generator=g)
    bn.running_mean = torch.randn(6, generator=g); bn.running_var = torch.rand(6, generator=g) + 0.5
    w = torch.randn((6, 4, 3, 3), generator=g); x = torch.randn((1, 4, 9, 9), generator=g)
    ref = F.batch_norm(F.conv2d(x, w, padding=1), bn.running_mean, bn.running_var, bn.weight, bn.bias, False, 0.0, 1e-5)
    wf, bf = fold_bn(w, bn)
    assert (F.conv2d(x, wf, bf, padding=1) - ref).abs().max().item() <= 1e-5
