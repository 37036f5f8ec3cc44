"""GPU parity of VToonify.forward (D and T backbones) against the reference outputs in tests/golden."""
import json
import os

import numpy as np
import pytest
import torch

from tests.shapes import GOLDEN, vtoonify_frames

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

TOL = {"fp32": 2e-4, "bf16x3": 1e-3, "tf32": 2e-2}     # max-abs error as a fraction of max(1, ref rms); measured values are printed.
# bf16x3 is the product path: 1e-3 per pixel is the north_star bar (BASELINE.json); tf32 is the opt-in fast mode.


def T(a):
    return torch.from_numpy(np.asarray(a))


@pytest.fixture(scope="module", params=["d", "t"])
def model(request):
    from vtoonify_b200.vtoonify import VToonify
    from vtoonify_b200.weights import det_state_dict
    backbone = {"d": "dualstylegan", "t": "toonify"}[request.param]
    m = VToonify(backbone=backbone).eval()
    keys = json.load(open(os.path.join(GOLDEN, f"state_dict_keys_{request.param}.json")))
    sd = m.state_dict()
    assert list(sd.keys()) == list(keys.keys())
    assert all(list(sd[k].shape) == keys[k] for k in keys)
    m.load_state_dict(det_state_dict(m, seed=0), strict=True)
    return request.param, m.cuda()


@pytest.mark.parametrize("prec", ["fp32", "bf16x3", "tf32"])
def test_forward_golden(golden, model, prec):
    from vtoonify_b200 import ops
    tag, m = model
    g = golden(f"vtoonify_{tag}")
    ops.set_precision(prec)
    try:
        for case in ("a", "b"):
            x, style = vtoonify_frames(g, case).cuda(), T(g[f"{case}_style"]).cuda()
            if tag == "d":
                y, masks = m(x, style, d_s=0.5, return_mask=True)
                for i, mk in enumerate(masks):
                    e = (mk.cpu() - T(g[f"{case}_mask{i}"])).abs().max().item()
                    assert e <= {"fp32": 1e-4, "bf16x3": 5e-4, "tf32": 3e-2}[prec], f"mask {i}: {e}"
            else:
                y = m(x, style, d_s=0.5)
            ref = T(g[f"{case}_y"])
            assert tuple(y.shape) == tuple(ref.shape)
            err = (y.cpu().double() - ref.double()).abs().max().item()
            rms = ref.pow(2).mean().sqrt().item()
            print(f"VToonify-{tag} case {case} [{prec}]: max|err| {err:.3e}, ref rms {rms:.3f}, err/rms {err / rms:.2e}")
            assert err <= TOL[prec] * max(1.0, rms)
    finally:
        ops.set_precision(ops.DEFAULT_PRECISION)


def test_aux_paths(golden, model):
    tag, m = model
    g = golden(f"vtoonify_{tag}")
    w = m.zplus2wplus(T(g["zplus"]).cuda())
    assert (w.cpu() - T(g["wplus"])).abs().max().item() <= 5e-5
    x, style = vtoonify_frames(g, "b").cuda(), T(g["b_style"]).cuda()
    feat, skip = m(x, style, d_s=0.5, return_feat=True)
    assert feat.shape == (1, 512, 6, 5) and skip.shape == (1, 3, 6, 5)
    # 2-D style ([B, 512]) path of forward (model/vtoonify.py:212-216)
    y = m(x, style[:, 0], d_s=0.5)
    assert y.shape == (1, 3, 192, 160) and torch.isfinite(y).all()
    # batch independence: frames are independent units (multi-GPU sharding relies on it)
    xa, sa = vtoonify_frames(g, "a").cuda(), T(g["a_style"]).cuda()
    y2 = m(xa, sa, d_s=0.5)
    y0 = m(xa[:1], sa[:1], d_s=0.5)
    assert (y2[:1] - y0).abs().max().item() <= 1e-5


def test_style_cache(golden, model):
    """Per-style caching (one video = one style): identical results with and without cache hits, for shared (expanded or
    repeated) and per-sample styles; in-place edits of the style tensor and reloaded weights invalidate the cache."""
    from vtoonify_b200 import _lib
    from vtoonify_b200.weights import det_state_dict
    tag, m = model
    g = golden(f"vtoonify_{tag}")
    x = vtoonify_frames(g, "a").cuda()                                         # B = 2
    style = T(g["a_style"])[:1].repeat(2, 1, 1).cuda()              # one video, one style: both rows carry the same code
    y_first = m(x, style, d_s=0.5)
    n0 = _lib.launch_count()
    y_hit = m(x, style, d_s=0.5)
    n_hit = _lib.launch_count() - n0
    assert torch.equal(y_first, y_hit)
    s_exp = style[:1].expand(2, -1, -1)                              # the frame loop's stride-0 form: no device comparison needed
    n0 = _lib.launch_count()
    y_exp = m(x, s_exp, d_s=0.5)
    n_miss = _lib.launch_count() - n0
    assert torch.equal(y_first, y_exp)
    assert n_hit < n_miss, f"a cache hit must launch fewer kernels ({n_hit} vs {n_miss})"
    # per-sample styles: row 1 differs -> per-sample weights; each row equals its own single-sample run
    s2 = style.clone()
    s2[1] = s2[1] * 0.5 + 0.1
    y2 = m(x, s2, d_s=0.5)
    assert (y2[0:1] - m(x[0:1], s2[0:1], d_s=0.5)).abs().max().item() <= 1e-5
    assert (y2[1:2] - m(x[1:2], s2[1:2], d_s=0.5)).abs().max().item() <= 1e-5
    assert (y2[1] - y_first[1]).abs().max().item() > 1e-3
    # in-place edit of a cached style tensor (version bump) must not serve stale weights
    s3 = style.clone()
    ya = m(x, s3, d_s=0.5)
    s3.mul_(0.5)
    yb = m(x, s3, d_s=0.5)
    assert (ya - yb).abs().max().item() > 1e-3
    assert torch.equal(yb, m(x, s3.clone(), d_s=0.5))
    # a different d_s with the same style object
    yd = m(x, style, d_s=0.25) if tag == "d" else None
    if yd is not None:
        assert (yd - y_first).abs().max().item() > 1e-4
    # reloading (different) weights invalidates everything
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    m.load_state_dict({k: v.cuda() for k, v in det_state_dict(m, seed=1).items()}, strict=True)
    y_new = m(x, style, d_s=0.5)
    assert (y_new - y_first).abs().max().item() > 1e-3
    m.load_state_dict(sd0, strict=True)
    assert torch.equal(m(x, style, d_s=0.5), y_first)
