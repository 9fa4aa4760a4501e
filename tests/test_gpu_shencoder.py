"""GPU parity: nerf2mesh_b200.shencoder vs the reference CUDA kernel (its outputs stored in tests/golden/sh.npz,
tests/golden/make_golden.py) and the float64 oracle.  The kernel evaluates the same polynomials through a recurrence, so the bar is the float
tolerance north_star states (<= 1e-3 relative); observed agreement is ~1e-6."""
import os

import numpy as np
import pytest
import torch

import cases
from nerf2mesh_b200.shencoder import SHEncoder, sh_encode
from oracle import sh_oracle

pytestmark = pytest.mark.gpu

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sh.npz"))


@pytest.mark.parametrize("degree", [1, 2, 3, 4, 5, 6, 7, 8])
def test_sh_forward_and_grad(degree):
    v = cases.sh_case().cuda()
    o0, dy0 = torch.from_numpy(GOLD[f"o{degree}"]).cuda(), torch.from_numpy(GOLD[f"dy{degree}"]).cuda()
    vr = v.clone().requires_grad_(True)
    o1 = sh_encode(vr, degree, True)
    scale = o0.abs().max().item()
    assert (o0 - o1).abs().max().item() <= 1e-5 * scale
    oo, go = sh_oracle.sh_encode(v.cpu().numpy(), degree, True)
    assert np.abs(oo - o1.detach().cpu().numpy()).max() <= 1e-5 * scale
    # backward = grad . dy_dx  (shencoder.cu:359-382)
    g = torch.randn_like(o1)
    o1.backward(g)
    expect = torch.einsum("bc,bdc->bd", g, dy0.view(-1, 3, degree * degree))
    gs = expect.abs().max().item() + 1e-12
    assert (vr.grad - expect).abs().max().item() <= 2e-5 * gs
    expect64 = np.einsum("bc,bdc->bd", g.cpu().numpy().astype(np.float64), go.reshape(-1, 3, degree * degree))
    assert np.abs(vr.grad.cpu().numpy() - expect64).max() <= 2e-5 * gs


def test_sh_module():
    enc = SHEncoder(degree=4)
    d = torch.randn(100, 3, device="cuda") * 3
    y = enc(d)
    assert y.shape == (100, 16)
    assert torch.allclose(y[:, 0], torch.full((100,), 0.28209479177387814, device="cuda"))
    with pytest.raises(RuntimeError):
        sh_encode(torch.randn(4, 3, device="cuda"), 9)
