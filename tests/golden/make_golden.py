"""Generate tests/golden/*.npz and tests/golden/reference_ops.json by running the UNMODIFIED
reference CUDA kernels (oracle/_ref, built from the reference tree by oracle/build_ref.py) on a B200:

    python tests/golden/make_golden.py OUT_DIR        # then copy OUT_DIR/* to tests/golden/

Inputs are regenerated from seeds by tests/cases.py (identical on every machine); only the
reference's OUTPUTS are stored.  The CPU tests pin oracle/ against these vectors; the GPU tests
check nerf2mesh_b200 against them, so that they need neither the reference tree nor its kernels."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cases      # noqa: E402
import refcall    # noqa: E402
from oracle.build_ref import load_ref   # noqa: E402


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    rm = load_ref("_ref_raymarching"); ge = load_ref("_ref_gridencoder"); sh = load_ref("_ref_shencoder")
    cu = lambda t: t.cuda()

    # ---- raymarching -------------------------------------------------------------------------
    for name in cases.MARCH_CASES:
        c = cases.march_case(name)
        ro, rd, bits, aabb = cu(c["rays_o"]), cu(c["rays_d"]), cu(c["bits"]), cu(c["aabb"])
        nears, fars = refcall.near_far(rm, ro, rd, aabb, c["min_near"])
        xyzs, dirs, ts, rays = refcall.march_train(rm, ro, rd, bits, c["bound"], c["contract"], c["dt_gamma"],
                                                   c["max_steps"], c["C"], c["H"], nears, fars, cu(c["noises"]))
        x = refcall.by_ray(xyzs, rays); t = refcall.by_ray(ts, rays)
        keep = min(len(x), 4096)
        np.savez_compressed(os.path.join(out_dir, f"march_{name}.npz"), nears=nears.cpu().numpy(), fars=fars.cpu().numpy(),
                            counts=rays[:, 1].cpu().numpy(), xyzs_head=x[:keep], ts_head=t[:keep],
                            xyzs_sum=x.astype(np.float64).sum(0), ts_sum=t.astype(np.float64).sum(0))
    # ---- compositing --------------------------------------------------------------------------
    c = cases.composite_case()
    sig, rgb, ts, rays = cu(c["sigmas"]), cu(c["rgbs"]), cu(c["ts"]), cu(c["rays"])
    out = {}
    for T in (1e-4, 1e-2):
        w, ws, d, im = refcall.composite_fwd(rm, sig, rgb, ts, rays, T, False)
        gs, gr = refcall.composite_bwd(rm, cu(c["grad_weights"]), cu(c["grad_weights_sum"]), cu(c["grad_depth"]), cu(c["grad_image"]),
                                       sig, rgb, ts, rays, ws, d, im, T, False)
        for k, v in dict(w=w, ws=ws, d=d, im=im, gs=gs, gr=gr).items():
            out[f"{k}_{T}"] = v.cpu().numpy()
    np.savez_compressed(os.path.join(out_dir, "composite.npz"), **out)
    # ---- grid encoder -------------------------------------------------------------------------
    for name in cases.GRID_CASES:
        c = cases.grid_case(name)
        inputs, emb, offsets = cu(c["inputs"]), cu(c["embeddings"]), cu(c["offsets"])
        o, dy = refcall.grid_fwd(ge, inputs, emb, offsets, c["S"], c["H"], c["L"], c["gridtype"], c["align"], c["interp"], True)
        g = torch.Generator().manual_seed(2)
        grad = torch.randn(c["L"], c["B"], c["C"], generator=g).cuda().to(emb.dtype)
        gemb, ginp = refcall.grid_bwd(ge, grad, inputs, emb, offsets, c["S"], c["H"], c["L"], c["gridtype"], c["align"], c["interp"], dy)
        nz = gemb.float().abs().sum(-1).nonzero().flatten()
        extra = {}
        if not c["half"]:
            gtv = torch.zeros_like(emb)
            ge.grad_total_variation(inputs, emb, gtv, offsets, 1e-3, c["B"], c["D"], c["C"], c["L"], c["S"], c["H"], c["gridtype"], c["align"])
            nzt = gtv.abs().sum(-1).nonzero().flatten()
            extra = dict(tv_rows=nzt.cpu().numpy(), tv_vals=gtv[nzt].cpu().numpy())
        np.savez_compressed(os.path.join(out_dir, f"grid_{name}.npz"), outputs=o.float().cpu().numpy(), dy_dx=dy.float().cpu().numpy(),
                            gemb_rows=nz.cpu().numpy(), gemb_vals=gemb[nz].float().cpu().numpy(), ginp=ginp.float().cpu().numpy(), **extra)
    # ---- SH ----------------------------------------------------------------------------------
    v = cu(cases.sh_case())
    out = {}
    for deg in range(1, 9):
        o, dy = refcall.sh_fwd(sh, v, deg, True)
        out[f"o{deg}"] = o.cpu().numpy(); out[f"dy{deg}"] = dy.cpu().numpy()
    np.savez_compressed(os.path.join(out_dir, "sh.npz"), **out)
    with open(os.path.join(out_dir, "reference_ops.json"), "w") as f:
        json.dump(reference_ops(rm, ge), f, indent=1, sort_keys=True)
    # ---- the reference's model, trainer and stage-1 composition (oracle/ref_stage.py) ------------------------------------------
    import tempfile
    import test_gpu_reference_parity
    import test_gpu_stage0
    import test_gpu_stage1
    G = refcall.Golden()
    with tempfile.TemporaryDirectory() as tmp:
        test_gpu_reference_parity.reference_outputs(G, tmp)
    test_gpu_stage0.reference_outputs(G)
    G.save(os.path.join(out_dir, "reference_model.npz"))
    G = refcall.Golden()
    test_gpu_stage1.reference_outputs(G)
    G.save(os.path.join(out_dir, "reference_stage1.npz"))
    torch.cuda.synchronize()
    print("golden written to", out_dir, sorted(os.listdir(out_dir)))


def reference_ops(rm, ge):
    """Digests (refcall.digest) of every reference output the GPU tests require bit-exact, on the inputs those tests build
    (tests/test_gpu_raymarching.py, tests/test_gpu_gridencoder.py), plus the few small outputs they compare with a tolerance."""
    D = refcall.digest
    cu = lambda t: t.cuda()
    res = {}
    for name in cases.MARCH_CASES:
        c = cases.march_case(name)
        ro, rd, bits, aabb = cu(c["rays_o"]), cu(c["rays_d"]), cu(c["bits"]), cu(c["aabb"])
        ro_x = torch.cat([ro, torch.tensor(cases.NEAR_FAR_EXTRA_O, device="cuda")])
        rd_x = torch.cat([rd, torch.tensor(cases.NEAR_FAR_EXTRA_D, device="cuda")])
        n0, f0 = refcall.near_far(rm, ro_x, rd_x, aabb, c["min_near"])
        res[f"near_far/{name}"] = dict(nears=D(n0), fars=D(f0))
        nears, fars = refcall.near_far(rm, ro, rd, aabb, c["min_near"])
        x0, d0, t0, r0 = refcall.march_train(rm, ro, rd, bits, c["bound"], c["contract"], c["dt_gamma"], c["max_steps"], c["C"], c["H"],
                                             nears, fars, cu(c["noises"]))
        res[f"march_train/{name}"] = dict(M=int(x0.shape[0]), counts=D(r0[:, 1]), xyzs=D(refcall.by_ray(x0, r0)),
                                          dirs=D(refcall.by_ray(d0, r0)), ts=D(refcall.by_ray(t0, r0)))
    for name in cases.INFERENCE_CASES:
        ws, depth, image, rays_t, trace = refcall.inference_loop(cases.march_case(name), rm)
        res[f"inference/{name}"] = dict(ws=D(ws), depth=D(depth), image=D(image), rays_t=D(rays_t), rounds=len(trace),
                                        trace=refcall.trace_digest(trace))
    for alpha_mode in (False, True):
        for T in (1e-4, 1e-2):
            c = cases.composite_case()
            sig, rgb, ts, rays = cu(c["sigmas"]), cu(c["rgbs"]), cu(c["ts"]), cu(c["rays"])
            if alpha_mode:
                sig = (sig / sig.max()).clamp(0, 0.999)
            w, ws, d, im = refcall.composite_fwd(rm, sig, rgb, ts, rays, T, alpha_mode)
            gs, gr = refcall.composite_bwd(rm, cu(c["grad_weights"]), cu(c["grad_weights_sum"]), cu(c["grad_depth"]), cu(c["grad_image"]),
                                           sig, rgb, ts, rays, ws, d, im, T, alpha_mode)
            res[f"composite/{alpha_mode}/{T}"] = dict(w=D(w), ws=D(ws), d=D(d), im=D(im), gs=D(gs), gr=D(gr))
    c = cases.composite_case(N=16)
    rays = cu(c["rays"]).clone()
    rays[-1, 1] += 1000
    w, ws, d, im = refcall.composite_fwd(rm, cu(c["sigmas"]), cu(c["rgbs"]), cu(c["ts"]), rays, 1e-4, False)
    res["composite_beyond_M"] = dict(w=D(w), ws=D(ws), im=D(im))
    grid, coords, rays = cases.packbits_morton_flatten_case()
    grid, coords, rays = cu(grid), cu(coords), cu(rays)
    out = {}
    for thresh in cases.PACKBITS_THRESH:
        b0 = torch.empty(grid.numel() // 8, dtype=torch.uint8, device="cuda")
        rm.packbits(grid, grid.numel() // 8, thresh, b0)
        out[f"packbits/{thresh}"] = D(b0)
    i0 = torch.empty(coords.shape[0], dtype=torch.int32, device="cuda")
    rm.morton3D(coords, coords.shape[0], i0)
    c0 = torch.empty(coords.shape[0], 3, dtype=torch.int32, device="cuda")
    rm.morton3D_invert(i0, coords.shape[0], c0)
    M = int(rays[:, 1].sum())
    f0 = torch.zeros(M, dtype=torch.int32, device="cuda")
    rm.flatten_rays(rays, rays.shape[0], M, f0)
    res["packbits_morton_flatten"] = dict(out, morton3D=D(i0), morton3D_invert=D(c0), flatten_rays=D(f0))
    ro, rd = cases.rays(500, seed=9)
    ro, rd = ro.cuda() * 0.2, rd.cuda()
    c0 = torch.empty(500, 2, device="cuda")
    rm.sph_from_ray(ro, rd, 4.0, 500, c0)
    res["sph_from_ray"] = c0.cpu().tolist()
    for name in cases.GRID_CASES:
        c = cases.grid_case(name)
        inputs, emb, offsets = cu(c["inputs"]), cu(c["embeddings"]), cu(c["offsets"])
        for partial in (False, True):
            max_level = c["L"] // 2 if partial else c["L"]
            o, dy = refcall.grid_fwd(ge, inputs, emb, offsets, c["S"], c["H"], max_level, c["gridtype"], c["align"], c["interp"], True)
            res[f"grid_forward/{name}/{partial}"] = dict(outputs=D(o), dy_dx=D(dy))
        o, dy = refcall.grid_fwd(ge, inputs, emb, offsets, c["S"], c["H"], c["L"], c["gridtype"], c["align"], c["interp"], True)
        g = torch.Generator().manual_seed(2)
        grad = torch.randn(c["L"], c["B"], c["C"], generator=g).cuda().to(emb.dtype)
        _, ginp = refcall.grid_bwd(ge, grad, inputs, emb, offsets, c["S"], c["H"], c["L"], c["gridtype"], c["align"], c["interp"], dy)
        res[f"grid_backward/{name}"] = dict(ginp=D(ginp))
    return res


if __name__ == "__main__":
    main(sys.argv[1])
