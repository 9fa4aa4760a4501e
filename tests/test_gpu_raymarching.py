"""GPU parity: nerf2mesh_b200.raymarching (through the C ABI) vs the reference's own CUDA kernels on identical inputs, through
their outputs stored under tests/golden/ (reference_ops.json: digests of the reference's outputs, tests/golden/make_golden.py).
Bar: bit-exact sample counts, M, and per-ray sample values (integers AND floats -- the arithmetic is reproduced op for op);
composite is bit-exact too."""
import json
import os

import pytest
import torch

import cases
import refcall
from nerf2mesh_b200 import raymarching as rm

pytestmark = pytest.mark.gpu

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_ops.json")) as _f:
    GOLD = json.load(_f)
D = refcall.digest


def cu(x):
    return x.cuda() if torch.is_tensor(x) else x


@pytest.mark.parametrize("name", cases.MARCH_CASES)
def test_near_far_bit_exact(name):
    c = cases.march_case(name)
    ro, rd, aabb = cu(c["rays_o"]), cu(c["rays_d"]), cu(c["aabb"])
    ro = torch.cat([ro, torch.tensor(cases.NEAR_FAR_EXTRA_O, device="cuda")])
    rd = torch.cat([rd, torch.tensor(cases.NEAR_FAR_EXTRA_D, device="cuda")])
    n1, f1 = rm.near_far_from_aabb(ro, rd, aabb, c["min_near"])
    g = GOLD[f"near_far/{name}"]
    assert D(n1) == g["nears"] and D(f1) == g["fars"]


@pytest.mark.parametrize("name", cases.MARCH_CASES)
def test_march_rays_train_bit_exact(name):
    c = cases.march_case(name)
    g = GOLD[f"march_train/{name}"]
    ro, rd, bits, aabb = cu(c["rays_o"]), cu(c["rays_d"]), cu(c["bits"]), cu(c["aabb"])
    nears, fars = rm.near_far_from_aabb(ro, rd, aabb, c["min_near"])
    noises = cu(c["noises"])
    # the wrapper's RNG replaced by the same noises: call the C ABI protocol directly
    from nerf2mesh_b200._lib import call, ptr, stream
    N = ro.shape[0]
    for use_slab in (True, False):
        counter = torch.zeros(1, dtype=torch.int32, device="cuda")
        rays = torch.empty(N, 2, dtype=torch.int32, device="cuda")
        tbuf = torch.empty(N * c["max_steps"] * 2, device="cuda") if use_slab else None
        args = (ptr(ro), ptr(rd), ptr(bits), c["bound"], int(c["contract"]), c["dt_gamma"], c["max_steps"], N,
                c["C"], c["H"], ptr(nears), ptr(fars))
        call("n2m_march_rays_train", *args, None, None, None, ptr(rays), ptr(counter), ptr(noises), ptr(tbuf), stream())
        M = int(counter.item())
        assert M == g["M"], f"M differs: {M} vs {g['M']}"
        assert M > 0
        # counts bit-exact; our offsets are the exclusive scan in ray order
        assert D(rays[:, 1]) == g["counts"]
        cnt = rays[:, 1].long()
        assert torch.equal(rays[:, 0].long(), torch.cumsum(cnt, 0) - cnt)
        x1 = torch.zeros(M, 3, device="cuda"); d1 = torch.zeros(M, 3, device="cuda"); t1 = torch.zeros(M, 2, device="cuda")
        call("n2m_march_rays_train", *args, ptr(x1), ptr(d1), ptr(t1), ptr(rays), ptr(counter), ptr(noises), ptr(tbuf), stream())
        torch.cuda.synchronize()
        for b, nm in ((x1, "xyzs"), (d1, "dirs"), (t1, "ts")):
            assert D(refcall.by_ray(b, rays)) == g[nm], f"{nm} differ (slab={use_slab})"


def test_march_wrapper_matches_abi():
    c = cases.march_case("lego_converged")
    ro, rd, bits, aabb = cu(c["rays_o"]), cu(c["rays_d"]), cu(c["bits"]), cu(c["aabb"])
    nears, fars = rm.near_far_from_aabb(ro, rd, aabb, c["min_near"])
    xyzs, dirs, ts, rays = rm.march_rays_train(ro, rd, c["bound"], c["contract"], bits, c["C"], c["H"], nears, fars,
                                               False, c["dt_gamma"], c["max_steps"])
    M = xyzs.shape[0]
    assert M == int(rays[:, 1].sum()) and dirs.shape == (M, 3) and ts.shape == (M, 2) and rays.dtype == torch.int32
    assert (ts[:, 1] > 0).all() and (xyzs.abs() <= c["bound"]).all()
    flat = rm.flatten_rays(rays, M)
    assert torch.equal(dirs, rd[flat.long()])
    # empty input
    e = torch.zeros(0, 3, device="cuda")
    x, d, t, r = rm.march_rays_train(e, e, 1.0, False, bits, 1, 128, torch.zeros(0, device="cuda"), torch.zeros(0, device="cuda"))
    assert x.shape == (0, 3) and r.shape == (0, 2)


@pytest.mark.parametrize("alpha_mode", [False, True])
@pytest.mark.parametrize("T_thresh", [1e-4, 1e-2])
def test_composite_train_bit_exact(alpha_mode, T_thresh):
    c = cases.composite_case()
    g = GOLD[f"composite/{alpha_mode}/{T_thresh}"]
    sig = cu(c["sigmas"]); rgb = cu(c["rgbs"]); ts = cu(c["ts"]); rays = cu(c["rays"])
    if alpha_mode:
        sig = (sig / sig.max()).clamp(0, 0.999)
    w1, ws1, d1, i1 = rm.composite_rays_train(sig, rgb, ts, rays, T_thresh, alpha_mode)
    for b, k in ((w1, "w"), (ws1, "ws"), (d1, "d"), (i1, "im")):
        assert D(b) == g[k], k
    gw, gws, gd, gi = cu(c["grad_weights"]), cu(c["grad_weights_sum"]), cu(c["grad_depth"]), cu(c["grad_image"])
    sig_r = sig.clone().requires_grad_(True); rgb_r = rgb.clone().requires_grad_(True)
    w, ws, d, im = rm.composite_rays_train(sig_r, rgb_r, ts, rays, T_thresh, alpha_mode)
    torch.autograd.backward([w, ws, d, im], [gw, gws, gd, gi])
    assert D(sig_r.grad) == g["gs"] and D(rgb_r.grad) == g["gr"]


def test_composite_rays_beyond_M_zeroed():
    """rays whose slice exceeds M produce zeros (raymarching.cu:521-528)."""
    c = cases.composite_case(N=16)
    g = GOLD["composite_beyond_M"]
    sig = cu(c["sigmas"]); rgb = cu(c["rgbs"]); ts = cu(c["ts"]); rays = cu(c["rays"]).clone()
    rays[-1, 1] += 1000
    w1, ws1, d1, i1 = rm.composite_rays_train(sig, rgb, ts, rays, 1e-4, False)
    assert D(ws1) == g["ws"] and D(i1) == g["im"] and D(w1) == g["w"]
    assert ws1[-1] == 0


@pytest.mark.parametrize("name", cases.INFERENCE_CASES)
def test_inference_loop_bit_exact(name):
    """The eval loop of renderer.py:764-802 driven with our operators on the sigmas / rgbs the reference's loop saw."""
    g = GOLD[f"inference/{name}"]
    ws, depth, image, rays_t, trace = refcall.inference_loop(cases.march_case(name))
    assert len(trace) == g["rounds"]
    assert refcall.trace_digest(trace) == g["trace"]          # every round's samples
    for a, k in ((ws, "ws"), (depth, "depth"), (image, "image"), (rays_t, "rays_t")):
        assert D(a) == g[k], k


def test_packbits_morton_flatten_exact():
    g = GOLD["packbits_morton_flatten"]
    grid, coords, rays = cases.packbits_morton_flatten_case()
    grid, coords, rays = grid.cuda(), coords.cuda(), rays.cuda()
    for thresh in cases.PACKBITS_THRESH:
        b1 = rm.packbits(grid, thresh)
        assert D(b1) == g[f"packbits/{thresh}"]
        # in-place variant + unaligned view
        buf = torch.zeros(grid.numel() // 8 + 8, dtype=torch.uint8, device="cuda")
        out = rm.packbits(grid, thresh, buf[1:1 + grid.numel() // 8])
        assert torch.equal(out, b1)
    i1 = rm.morton3D(coords)
    assert D(i1) == g["morton3D"]
    c1 = rm.morton3D_invert(i1)
    assert torch.equal(c1, coords)
    assert D(c1) == g["morton3D_invert"]
    assert D(rm.flatten_rays(rays, int(rays[:, 1].sum()))) == g["flatten_rays"]


def test_sph_from_ray_close():
    ro, rd = cases.rays(500, seed=9)
    ro, rd = ro.cuda() * 0.2, rd.cuda()
    c0 = torch.tensor(GOLD["sph_from_ray"], device="cuda")
    c1 = rm.sph_from_ray(ro, rd, 4.0)
    assert torch.allclose(c0, c1, atol=1e-6, rtol=0)
