"""Deterministic input builders shared by tests/golden/make_golden.py, the CPU oracle tests and the
GPU parity tests.  Everything is generated from seeds with CPU generators, so inputs are identical
on every machine; only OUTPUTS of the reference kernels are stored under tests/golden/."""
import zlib

import numpy as np
import torch

from nerf2mesh_b200 import synthetic as S

AABB1 = [-1.0, -1.0, -1.0, 1.0, 1.0, 1.0]


def rays(N, seed=0, radius=S.LEGO_RADIUS):
    g = torch.Generator().manual_seed(seed)
    poses = S.orbit_cameras(100, radius=radius, seed=seed)
    ro, rd, _, _ = S.sample_rays(poses, S.lego_intrinsics(), 800, 800, N, g)
    return ro, rd


def march_case(name):
    """-> dict(rays_o, rays_d, bits, bound, contract, C, H, dt_gamma, max_steps, min_near, aabb, noises)"""
    cfgs = {
        # lego recipe: bound 1, one cascade, dt_gamma 0
        "lego_converged": dict(N=512, regime="converged", bound=1.0, C=1, dt_gamma=0.0, contract=False, perturb=True, radius=S.LEGO_RADIUS),
        "lego_cold": dict(N=128, regime="cold", bound=1.0, C=1, dt_gamma=0.0, contract=False, perturb=False, radius=S.LEGO_RADIUS),
        "lego_mid": dict(N=256, regime="mid", bound=1.0, C=1, dt_gamma=0.0, contract=False, perturb=True, radius=S.LEGO_RADIUS),
        # garden-like: bound 16 => 5 cascades, dt_gamma 1/256, cameras inside the volume
        "garden_cascades": dict(N=384, regime="converged", bound=16.0, C=5, dt_gamma=1.0 / 256, contract=False, perturb=True, radius=1.2),
        # contraction path (sdf + bound > 1): query bound 2 => 2 cascades
        "contract": dict(N=256, regime="converged", bound=4.0, C=2, dt_gamma=1.0 / 256, contract=True, perturb=True, radius=1.5),
        # non power-of-two bound
        "bound1p5": dict(N=256, regime="converged", bound=1.5, C=2, dt_gamma=1.0 / 128, contract=False, perturb=True, radius=2.5),
    }
    c = cfgs[name]
    H = 128
    ro, rd = rays(c["N"], seed=zlib.crc32(name.encode()) % 1000, radius=c["radius"])
    grid, bits, bricks = S.occupancy_regime(c["regime"], H=H, cascades=c["C"], bound=min(c["bound"], 2.0 ** (c["C"] - 1)))
    g = torch.Generator().manual_seed(7)
    noises = torch.rand(c["N"], generator=g) if c["perturb"] else torch.zeros(c["N"])
    b = c["bound"]
    return dict(rays_o=ro, rays_d=rd, bits=bits, bound=b, contract=c["contract"], C=c["C"], H=H,
                dt_gamma=c["dt_gamma"], max_steps=1024, min_near=0.05, aabb=torch.tensor([-b, -b, -b, b, b, b]),
                noises=noises, bricks=bricks)


MARCH_CASES = ["lego_converged", "lego_cold", "lego_mid", "garden_cascades", "contract", "bound1p5"]
INFERENCE_CASES = ["lego_converged", "garden_cascades", "contract"]
# degenerate rays appended to a march case's rays for near_far: axis-parallel (zero components) and guaranteed misses
NEAR_FAR_EXTRA_O = [[0.0, 0.0, 3.0], [5.0, 5.0, 5.0], [0.2, 0.1, 0.0]]
NEAR_FAR_EXTRA_D = [[0.0, 0.0, -1.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]
PACKBITS_THRESH = [0.0, 0.37, 10.0]


def packbits_morton_flatten_case():
    """-> (density grid [2, 64^3], morton coordinates [5000, 3] int32, rays [300, 2] int32 (offset, count))"""
    g = torch.Generator().manual_seed(0)
    grid = torch.rand(2, 64 ** 3, generator=g) * 2 - 0.5
    grid[0, :100] = -1.0
    coords = torch.randint(0, 128, (5000, 3), generator=g, dtype=torch.int32)
    cnt = torch.randint(0, 50, (300,), generator=g)
    off = torch.cumsum(cnt, 0) - cnt
    return grid, coords, torch.stack([off, cnt], -1).int()


def grid_case(name):
    """-> dict(inputs [B,D] in [0,1] (some OOB), embeddings, offsets, S, H, ...)"""
    from oracle.grid_oracle import level_offsets
    cfgs = {
        "density_c1": dict(D=3, C=1, L=16, desired=2048, log2T=19, gridtype=0, align=False, interp=0, half=False, B=300),
        "color_c2_half": dict(D=3, C=2, L=16, desired=2048, log2T=19, gridtype=0, align=False, interp=0, half=True, B=300),
        "color_c2_f32": dict(D=3, C=2, L=16, desired=2048, log2T=19, gridtype=0, align=False, interp=0, half=False, B=300),
        "garden_c2": dict(D=3, C=2, L=16, desired=32768, log2T=19, gridtype=0, align=False, interp=0, half=True, B=200),
        "tiled_smooth_c4": dict(D=3, C=4, L=8, desired=256, log2T=16, gridtype=1, align=True, interp=1, half=False, B=200),
        "d2_c8": dict(D=2, C=8, L=6, desired=512, log2T=14, gridtype=0, align=False, interp=0, half=False, B=200),
        "d4_c2": dict(D=4, C=2, L=4, desired=64, log2T=14, gridtype=0, align=False, interp=1, half=True, B=100),
    }
    c = cfgs[name]
    pls = float(np.exp2(np.log2(c["desired"] / 16) / (c["L"] - 1)))
    offsets = level_offsets(c["D"], c["L"], pls, 16, c["log2T"], c["align"])
    g = torch.Generator().manual_seed(11)
    emb = torch.rand(int(offsets[-1]), c["C"], generator=g) * 2e-1 - 1e-1     # wider than the 1e-4 init: exercises rounding
    inputs = torch.rand(c["B"], c["D"], generator=g)
    inputs[::17] = inputs[::17] * 1.2 - 0.1                               # a few out-of-range samples
    inputs[5] = 0.0; inputs[6] = 1.0                                      # exact edges
    if c["half"]:
        emb = emb.half()
    return dict(inputs=inputs, embeddings=emb, offsets=torch.from_numpy(offsets), S=float(np.log2(pls)), H=16,
                per_level_scale=pls, **c)


GRID_CASES = ["density_c1", "color_c2_half", "color_c2_f32", "garden_c2", "tiled_smooth_c4", "d2_c8", "d4_c2"]


def composite_case(seed=3, N=64, max_cnt=96, sigma_scale=40.0):
    g = torch.Generator().manual_seed(seed)
    cnt = torch.randint(0, max_cnt, (N,), generator=g)
    cnt[::9] = 0
    off = torch.cumsum(cnt, 0) - cnt
    M = int(cnt.sum())
    rays_t = torch.stack([off, cnt], -1).int()
    dt = torch.full((M,), 0.0034)
    t = torch.zeros(M)
    for n in range(N):
        k = int(cnt[n])
        if k:
            t0 = 2.0 + torch.rand(1, generator=g).item()
            t[off[n]:off[n] + k] = t0 + 0.0034 * torch.arange(1, k + 1)
    ts = torch.stack([t, dt], -1)
    sigmas = torch.rand(M, generator=g) ** 4 * sigma_scale       # some rays terminate early, some do not
    rgbs = torch.rand(M, 3, generator=g)
    grads = dict(grad_weights=torch.randn(M, generator=g) * 0.1, grad_weights_sum=torch.randn(N, generator=g),
                 grad_depth=torch.randn(N, generator=g) * 0.1, grad_image=torch.randn(N, 3, generator=g))
    return dict(sigmas=sigmas, rgbs=rgbs, ts=ts, rays=rays_t, M=M, N=N, **grads)


def sh_case(B=128, seed=5):
    g = torch.Generator().manual_seed(seed)
    v = torch.randn(B, 3, generator=g)
    v = v / v.norm(dim=-1, keepdim=True)
    v[0] = torch.tensor([0.0, 0.0, 1.0]); v[1] = torch.tensor([1.0, 0.0, 0.0]); v[2] = torch.tensor([0.0, -1.0, 0.0])
    return v
