"""GPU parity of the pSp style encoder (SURVEY §8 row a10) against the reference output in tests/golden/psp.npz."""
import json
import os
from argparse import Namespace

import numpy as np
import pytest
import torch

from tests.shapes import GOLDEN

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


@pytest.mark.parametrize("prec,tol", [("fp32", 2e-4), ("bf16x3", 2e-4), ("tf32", 3e-2)])
def test_psp_encoder(golden, prec, tol):
    from vtoonify_b200 import ops
    from vtoonify_b200.psp import GradualStyleEncoder
    from vtoonify_b200.weights import det_state_dict
    g = golden("psp")
    m = GradualStyleEncoder(50, "ir_se", Namespace(input_nc=3, n_styles=18)).eval()
    keys = json.load(open(os.path.join(GOLDEN, "state_dict_keys_psp.json")))
    sd = m.state_dict()
    assert list(sd.keys()) == list(keys.keys()) and all(list(sd[k].shape) == keys[k] for k in keys)
    m.load_state_dict(det_state_dict(m, seed=11), strict=True)
    m.cuda()
    ops.set_precision(prec)
    try:
        y = m(torch.from_numpy(g["x"]).float().cuda())
    finally:
        ops.set_precision(ops.DEFAULT_PRECISION)
    ref = torch.from_numpy(g["y"])
    assert tuple(y.shape) == (1, 18, 512)
    err = (y.cpu() - ref).abs().max().item()
    rms = ref.pow(2).mean().sqrt().item()
    print(f"pSp encoder [{prec}]: max|err| {err:.3e}, ref rms {rms:.2f}, err/rms {err / rms:.2e}")
    assert err <= tol * rms
