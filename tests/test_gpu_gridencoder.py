"""GPU parity: nerf2mesh_b200.gridencoder (through the C ABI) vs the reference's CUDA kernels
(their outputs stored under tests/golden/: reference_ops.json digests and grid_<case>.npz, tests/golden/make_golden.py)
and vs the float64 CPU oracle.  Bar: forward + dy_dx BIT-EXACT (fp32 and fp16);
table gradients (order-nondeterministic atomics in both) within 1e-3 relative of the tensor
scale and within 1e-5 relative of the float64 oracle for fp32."""
import json
import os

import numpy as np
import pytest
import torch

import cases
import refcall
from nerf2mesh_b200._lib import call, ptr, stream
from nerf2mesh_b200.gridencoder import GridEncoder, grid_encode
from oracle import grid_oracle

pytestmark = pytest.mark.gpu

GOLD_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
with open(os.path.join(GOLD_DIR, "reference_ops.json")) as _f:
    GOLD = json.load(_f)


def gold_rows(rows, vals, shape):
    """the reference's table gradient, stored as its non-zero rows"""
    t = torch.zeros(shape, dtype=torch.float32)
    t[torch.from_numpy(rows).long()] = torch.from_numpy(vals).float()
    return t.cuda()


def ours_fwd(inputs, emb, offsets, S, H, max_level, gridtype, align, interp, calc):
    B, D = inputs.shape
    L = offsets.shape[0] - 1
    C = emb.shape[1]
    out = torch.zeros(L, B, C, device="cuda", dtype=emb.dtype)
    dy = torch.zeros(B, L * D * C, device="cuda", dtype=emb.dtype) if calc else None
    call("n2m_grid_encode_forward", ptr(inputs), ptr(emb), ptr(offsets), ptr(out), B, D, C, L, max_level, S, H,
         ptr(dy), gridtype, int(align), interp, 1 if emb.dtype == torch.float16 else 0, stream())
    return out, dy


def ours_bwd(grad, inputs, emb, offsets, S, H, max_level, gridtype, align, interp, dy):
    B, D = inputs.shape
    L = offsets.shape[0] - 1
    C = emb.shape[1]
    gemb = torch.zeros_like(emb)
    ginp = torch.zeros(B, D, device="cuda", dtype=emb.dtype) if dy is not None else None
    call("n2m_grid_encode_backward", ptr(grad), ptr(inputs), ptr(emb), ptr(offsets), ptr(gemb), B, D, C, L, max_level,
         S, H, ptr(dy), ptr(ginp), gridtype, int(align), interp, 1 if emb.dtype == torch.float16 else 0, stream())
    return gemb, ginp


@pytest.mark.parametrize("name", cases.GRID_CASES)
@pytest.mark.parametrize("partial", [False, True])
def test_forward_bit_exact(name, partial):
    c = cases.grid_case(name)
    g = GOLD[f"grid_forward/{name}/{partial}"]
    inputs, emb, offsets = c["inputs"].cuda(), c["embeddings"].cuda(), c["offsets"].cuda()
    L = c["L"]
    max_level = L // 2 if partial else L
    o1, dy1 = ours_fwd(inputs, emb, offsets, c["S"], c["H"], max_level, c["gridtype"], c["align"], c["interp"], True)
    assert refcall.digest(o1) == g["outputs"], "outputs differ"
    assert refcall.digest(dy1) == g["dy_dx"], "dy_dx differ"
    assert o1.abs().max() > 0


@pytest.mark.parametrize("name", cases.GRID_CASES)
def test_backward_vs_reference_and_oracle(name):
    c = cases.grid_case(name)
    inputs, emb, offsets = c["inputs"].cuda(), c["embeddings"].cuda(), c["offsets"].cuda()
    L, B, C = c["L"], c["B"], c["C"]
    g = torch.Generator().manual_seed(2)
    grad = torch.randn(L, B, C, generator=g).cuda().to(emb.dtype)
    _, dy = ours_fwd(inputs, emb, offsets, c["S"], c["H"], L, c["gridtype"], c["align"], c["interp"], True)
    ref = np.load(os.path.join(GOLD_DIR, f"grid_{name}.npz"))
    ge0 = gold_rows(ref["gemb_rows"], ref["gemb_vals"], tuple(emb.shape))
    ge1, gi1 = ours_bwd(grad, inputs, emb, offsets, c["S"], c["H"], L, c["gridtype"], c["align"], c["interp"], dy)
    assert refcall.digest(gi1) == GOLD[f"grid_backward/{name}"]["ginp"]          # deterministic: bit-exact
    scale = ge0.float().abs().max().item()
    tol = (2e-3 if c["half"] else 1e-5) * scale       # fp16 atomics round per add; order differs run to run
    assert (ge0.float() - ge1.float()).abs().max().item() <= tol
    # float64 oracle (order-independent sum)
    geo, gio = grid_oracle.grid_encode_backward(grad.cpu(), inputs.cpu(), c["offsets"].numpy(), emb.shape[0], c["S"], c["H"],
                                                L, c["gridtype"], c["align"], c["interp"], dy.cpu())
    # the oracle evaluates exp2 exactly; the kernels use ex2.approx (as the reference does), which moves
    # the finest levels' fractional position by ~1e-4 => compare at north_star's 1e-3 (4e-3 for fp16 atomics)
    assert (geo - ge1.double().cpu()).abs().max().item() <= (4e-3 if c["half"] else 1e-3) * scale
    if not c["half"]:
        assert (gio.float() - gi1.cpu().float()).abs().max().item() <= 1e-3 * gio.abs().max().item()


@pytest.mark.parametrize("name", ["density_c1", "color_c2_f32", "tiled_smooth_c4", "d2_c8"])
def test_total_variation(name):
    c = cases.grid_case(name)
    inputs, emb, offsets = c["inputs"].cuda(), c["embeddings"].float().cuda(), c["offsets"].cuda()
    B, D, C, L = c["B"], c["D"], c["C"], c["L"]
    ref = np.load(os.path.join(GOLD_DIR, f"grid_{name}.npz"))
    g0 = gold_rows(ref["tv_rows"], ref["tv_vals"], tuple(emb.shape))
    g1 = torch.zeros_like(emb)
    call("n2m_grad_total_variation", ptr(inputs), ptr(emb), ptr(g1), ptr(offsets), 1e-3, B, D, C, L, c["S"], c["H"],
         c["gridtype"], int(c["align"]), stream())
    scale = g0.abs().max().item()
    assert scale > 0
    assert (g0 - g1).abs().max().item() <= 1e-5 * scale
    go = grid_oracle.grad_total_variation(inputs.cpu(), emb.cpu(), c["offsets"].numpy(), 1e-3, c["S"], c["H"], c["gridtype"], c["align"])
    # vs the float64 oracle: the TV term is piecewise constant in the sample's cell, and the kernels'
    # ex2.approx level scale (same as the reference's) can move a sample that sits within ~1e-4 of a
    # cell boundary at the finest levels into the neighbouring cell; allow a handful of such rows.
    err = (go - g1.double().cpu()).abs().amax(-1)
    bad = (err > 1e-3 * scale).sum().item()
    touched = (go.abs().amax(-1) > 0).sum().item()
    assert bad <= max(4, 0.01 * touched), f"{bad} of {touched} rows differ" 


def test_module_autograd_and_amp():
    """GridEncoder module: forward under autocast uses the fp16 table iff C is even (grid.py:45-46);
    gradients flow to the fp32 Parameter; matches the float64 oracle."""
    torch.manual_seed(0)
    for C in (1, 2):
        enc = GridEncoder(level_dim=C, desired_resolution=2048).cuda()
        x = (torch.rand(500, 3, device="cuda") * 2 - 1)
        with torch.autocast("cuda", dtype=torch.float16):
            y = enc(x, bound=1)
        assert y.dtype == (torch.float16 if C == 2 else torch.float32) and y.shape == (500, 16 * C)
        y.float().square().sum().backward()
        assert enc.embeddings.grad is not None and enc.embeddings.grad.dtype == torch.float32
        assert enc.embeddings.grad.abs().sum() > 0
        y32 = enc(x, bound=1)
        ref, _ = grid_oracle.grid_encode_forward(((x + 1) / 2).cpu(), enc.embeddings.detach().cpu(), enc.offsets.cpu().numpy(),
                                                 float(np.log2(enc.per_level_scale)), 16)
        ref = ref.permute(1, 0, 2).reshape(500, -1)
        assert (y32.cpu() - ref).abs().max().item() <= 1e-3 * ref.abs().max().item()
        enc.grad_total_variation(1e-4, x, 1)


def test_error_paths():
    enc = GridEncoder(level_dim=2).cuda()
    x = torch.rand(10, 3, device="cuda")
    with pytest.raises(RuntimeError):
        grid_encode(x, torch.zeros(enc.embeddings.shape[0], 3, device="cuda"), enc.offsets, 2.0, 16)   # C = 3 unsupported
    with pytest.raises(RuntimeError):
        grid_encode(x.cpu(), enc.embeddings, enc.offsets, 2.0, 16)                                    # not CUDA
    with pytest.raises(ValueError):
        GridEncoder(level_dim=2).cuda().grad_total_variation(1e-4, x, 1)                              # no grad yet
    e = grid_encode(torch.zeros(0, 3, device="cuda"), enc.embeddings, enc.offsets, 2.0, 16)
    assert e.shape == (0, 32)
