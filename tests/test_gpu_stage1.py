"""GPU: the fused stage-1 texture step (nerf2mesh_b200/stage1.py over csrc/raster.cu, csrc/stage1.cu and the stage-0 tensor-core
kernels) against the reference's render_stage1 arithmetic composed from the UNMODIFIED reference model (`NeRFNetwork.rgb`,
network.py:170-189, over the reference's grid-encoder kernels) and torch ops, following nerf/renderer.py:824-907 and
nerf/utils.py:703-712 line by line -- with this repo's rasterize / interpolate standing in for nvdiffrast (itself checked against the
CPU oracle in test_gpu_raster.py), without dr.antialias and with this repo's antialias (csrc/antialias.cu, checked against its CPU oracle
in test_gpu_antialias.py) in the place of the library's, including the image-loss gradient it sends to the vertices.

The reference's results are stored in tests/golden/reference_stage1.npz (refcall.Golden: scalars, digests, and for every large tensor its
values at stored rows -- a seeded sample, or for the sparse colour-table gradient a sample of the rows it reaches -- with its full-tensor
size, max |.| and norm); `reference_outputs()` below regenerates them where the
reference is available (tests/golden/make_golden.py).  A comparison with a sampled tensor is made on its stored rows."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import refcall

from nerf2mesh_b200 import raster as dr
from nerf2mesh_b200 import synthetic as S
from nerf2mesh_b200.stage0 import MLP_LAYOUT, Stage0Config, Stage0Trainer
from nerf2mesh_b200.stage1 import Stage1Trainer
from nerf2mesh_b200.train_synthetic import full_image_rays
from oracle import raster_oracle as R

pytestmark = pytest.mark.gpu

GOLD_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_stage1.npz")
K_IMG, K_GRAD = 768, 1024
COLOR_GRADS = ["encoder_color.embeddings"] + [n for n, _ in MLP_LAYOUT if not n.startswith("sigma")]
STAGE1_CASES = [(2, False), (1, False), (2, True), (1, True)]
_GOLD = []


def gold():
    if not _GOLD:
        _GOLD.append(refcall.Golden(GOLD_PATH))
    return _GOLD[0]


def _setup(h0=96, w0=96, ssaa=2, steps=30, antialias=False, subdiv=4, seeded=False, **s1_kw):
    N = 1024
    cfg = Stage0Config(bound=1.0, num_rays=N, max_samples=N * 256)
    t0 = Stage0Trainer(cfg, seed=5)
    grid, bits, bricks = S.occupancy_regime("converged")
    t0.set_occupancy(bits, grid)
    g = torch.Generator().manual_seed(0)
    poses = S.orbit_cameras(100, seed=0)
    if seeded:          # parameters that depend on a seed alone, for the comparisons with stored reference results
        refcall.seeded_state(t0)
        steps = 0
    for it in range(steps):       # non-trivial colour parameters
        ro, rd, _, _ = S.sample_rays(poses, S.lego_intrinsics(), 800, 800, N, g)
        t0.step(ro, rd, S.render_bricks(ro, rd, bricks), torch.rand(N, 3, generator=g), torch.rand(N, generator=g), use_graph=False)
    v, f = R.icosphere(subdiv)
    cam = np.array([1.5, 1.1, 0.9]) * 1.6
    pose = torch.from_numpy(S.look_at_pose(cam).astype(np.float32))
    intr = S.lego_intrinsics(h0, w0)
    _, rays_d = full_image_rays(pose, intr, h0, w0)
    # projection matching the pinhole rays: fovy from the focal length, OpenGL clip space; nvdiffrast row 0 = bottom, the dataset's row 0 = top:
    # flip y in the projection (as the reference's provider does in its mvp)
    mvp = R.perspective_mvp(cam, fovy=2 * np.arctan(0.5 * h0 / intr[1]), aspect=w0 / h0)
    mvp[1] *= -1
    s1 = Stage1Trainer(t0, torch.from_numpy(v), torch.from_numpy(f), h0, w0, ssaa=ssaa, antialias=antialias, **s1_kw)
    gt = torch.rand(h0 * w0, 4, generator=g); gt[:, 3] = (gt[:, 3] > 0.5).float()
    bg = torch.rand(h0 * w0, 3, generator=g)
    return t0, s1, torch.from_numpy(mvp), rays_d.cuda(), gt.cuda(), bg.cuda()


def _reference_stage1(ns, ref_stage, t0, s1, mvp, rays_d, gt, bg, lambda_mask=0.1, antialias=False):
    """render_stage1 (renderer.py:824-907) + the stage-1 loss (utils.py:703-712) with the unmodified reference model"""
    opt = ref_stage.default_opt(bound=1.0, dt_gamma=0.0, adaptive_num_rays=False)
    model = ns.make_model(opt)
    model.load_state_dict(t0.export_reference_state(), strict=True)
    model.cuda().train()
    h0, w0, ssaa = s1.h0, s1.w0, s1.ssaa
    h, w = h0 * ssaa, w0 * ssaa
    dirs = rays_d.view(h0, w0, 3)
    dirs = F.interpolate(dirs.permute(2, 0, 1)[None], (h, w), mode="nearest")[0].permute(1, 2, 0).reshape(-1, 3).contiguous()   # scale_img_hwc(mag='nearest')
    dirs = dirs / torch.sqrt(torch.clamp((dirs * dirs).sum(-1, keepdim=True), min=1e-20))
    vertices = s1.vertices.clone().requires_grad_(antialias)        # the leaf standing in for self.vertices + self.vertices_offsets
    vclip = torch.matmul(F.pad(vertices, pad=(0, 1), mode="constant", value=1.0), torch.transpose(mvp.cuda(), 0, 1)).float().unsqueeze(0)
    glctx = dr.RasterizeCudaContext()
    rast, _ = dr.rasterize(glctx, vclip, s1.triangles, (h, w))
    xyzs, _ = dr.interpolate(vertices.unsqueeze(0), rast, s1.triangles)
    mask, _ = dr.interpolate(torch.ones_like(vertices[:, :1]).unsqueeze(0), rast, s1.triangles)
    mask_flatten = (mask > 0).view(-1).detach()
    xyzs = xyzs.view(-1, 3)
    rgbs = torch.zeros(h * w, 3, device="cuda", dtype=torch.float32)
    with torch.autocast("cuda", dtype=torch.float16):
        mask_rgbs, _ = model.rgb(xyzs[mask_flatten].detach(), dirs[mask_flatten], None, "full")
    rgbs[mask_flatten] = mask_rgbs.float()
    rgbs = rgbs.view(1, h, w, 3)
    alphas = mask.float()
    if antialias:          # renderer.py:886-887
        alphas = dr.antialias(alphas, rast, vclip, s1.triangles, pos_gradient_boost=1.0).squeeze(0).clamp(0, 1)
        rgbs = dr.antialias(rgbs, rast, vclip, s1.triangles, pos_gradient_boost=1.0).squeeze(0).clamp(0, 1)
    else:
        alphas = alphas.squeeze(0).clamp(0, 1); rgbs = rgbs.squeeze(0).clamp(0, 1)         # dr.antialias omitted on both sides
    image = alphas * rgbs
    T = 1 - alphas

    def down(x):       # scale_img_hwc(x, (h0, w0)): bilinear minification
        return F.interpolate(x.permute(2, 0, 1)[None], (h0, w0), mode="bilinear")[0].permute(1, 2, 0).contiguous()

    if ssaa > 1:
        image, T = down(image), down(T)
    image = image + T * bg.view(h0, w0, 3)
    ws = (1 - T).view(-1)
    gt_mask = gt[:, 3:]
    gt_rgb = gt[:, :3] * gt_mask + bg * (1 - gt_mask)
    loss = ((image.view(-1, 3) - gt_rgb) ** 2).mean(-1) + lambda_mask * (ws - gt_mask.squeeze(1)) ** 2
    loss = loss.mean()
    scaler = torch.amp.GradScaler("cuda", init_scale=float(t0.opt_state[0].item()))
    scaler.scale(loss).backward()
    inv = 1.0 / float(t0.opt_state[0].item())
    grads = {n: p.grad * inv for n, p in model.named_parameters() if p.grad is not None}
    return dict(image=image.view(-1, 3).detach(), ws=ws.detach(), loss=float(loss), grads=grads, covered=int(mask_flatten.sum()), rast=rast,
                grad_vertices=None if vertices.grad is None else vertices.grad * inv)


def _ref_ns():
    from oracle import ref_stage
    if not ref_stage.staged():
        pytest.skip("reference Python files not staged")
    return ref_stage, ref_stage.load("ref")


def _step_setup(ssaa, antialias):
    # antialias only sees the edges of the foreground pixel's own triangle: on the 5120-face sphere (facets a few pixels wide, slivers at
    # the limb) it blends a handful of outline pixels (3-5 measured), so the antialiased cases use the 320-face sphere
    t0, s1, mvp, rays_d, gt, bg = _setup(ssaa=ssaa, antialias=antialias, subdiv=2 if antialias else 4, seeded=True)
    t0.opt_state[0] = 4096.0
    return t0, s1, mvp, rays_d, gt, bg


def _reference_step(G, ssaa, antialias):
    P = f"step/{ssaa}/{antialias}/"
    ref_stage, ns = _ref_ns()
    t0, s1, mvp, rays_d, gt, bg = _step_setup(ssaa, antialias)
    ref = _reference_stage1(ns, ref_stage, t0, s1, mvp, rays_d, gt, bg, antialias=antialias)
    G.put(P + "covered", ref["covered"]); G.put(P + "rast", refcall.digest(ref["rast"])); G.put(P + "loss", ref["loss"])
    G.put(P + "image", ref["image"], K_IMG); G.put(P + "ws", ref["ws"], K_IMG)
    if antialias:
        G.put(P + "grad_vertices", ref["grad_vertices"].cpu().numpy())
    for name in COLOR_GRADS:          # the colour table's gradient is sparse: stored at a sample of the rows it reaches
        g, key = ref["grads"][name], P + f"grad/{name}"
        G.put(key, g, index=refcall.support_rows(g, k=K_GRAD, key=key) if name == "encoder_color.embeddings" else refcall.sample_index(g.numel(), K_GRAD, key))


@pytest.mark.parametrize("ssaa,antialias", STAGE1_CASES)
def test_stage1_step_matches_reference_composition(ssaa, antialias):
    P = f"step/{ssaa}/{antialias}/"
    G = gold()
    t0, s1, mvp, rays_d, gt, bg = _step_setup(ssaa, antialias)
    t0.gtable.zero_(); t0.g_mlp.zero_()
    s1.forward(mvp, rays_d)
    s1.loss_backward(gt, bg)
    torch.cuda.synchronize()
    covered = G[P + "covered"]
    assert s1.counters[2].item() == 0 and s1.counters[1].item() == covered and covered > 0.1 * s1.h * s1.w
    assert refcall.digest(s1.rast) == G[P + "rast"]
    a, r = G.take(P + "image", s1.image)
    assert (a - r).abs().max().item() <= 2e-3
    a, r = G.take(P + "ws", s1.weights_sum)
    assert (a - r).abs().max().item() <= (1e-5 if antialias else 1e-6)
    if antialias:
        # the silhouette pixels changed, and the loss reaches the vertices through them (the reference's only path to vertices_offsets)
        assert ((s1.aa[:, 3] - s1.rgba[:, 3]).abs() > 1e-3).sum().item() > 30
        gv, rv = s1.vertex_gradient().double().flatten().cpu(), torch.from_numpy(G[P + "grad_vertices"]).double().flatten()
        assert rv.abs().max().item() > 0
        cos = (torch.dot(gv, rv) / (gv.norm() * rv.norm() + 1e-300)).item()
        assert cos > 0.999 and ((gv - rv).norm() / rv.norm()).item() <= 3e-2, (cos, ((gv - rv).norm() / rv.norm()).item())
    ref_loss = G[P + "loss"]
    assert abs(s1.read_loss() - ref_loss) <= 1e-3 * abs(ref_loss)
    g = t0.export_reference_grads()
    assert t0.opt_state[3].item() == 0
    for name in COLOR_GRADS:
        assert G[P + f"grad/{name}:absmax"] > 0, name
        e = G.cmp(P + f"grad/{name}", g[name])
        assert e["cos"] > 0.9995 and e["rel_l2"] <= 3e-2, (name, e)
    # the density branch receives no gradient in stage 1
    assert g["encoder.embeddings"].abs().max().item() == 0
    assert g["sigma_net.net.0.weight"].abs().max().item() == 0 and g["sigma_net.net.1.weight"].abs().max().item() == 0
    # and a full optimizer step runs
    before = t0.mlp.clone()
    s1.step(mvp, rays_d, gt, bg)
    torch.cuda.synchronize()
    assert not torch.equal(before, t0.mlp) and torch.isfinite(t0.mlp).all()


def test_graph_replayed_step_equals_eager_step():
    """Stage1Trainer.step(use_graph=True): the step captured once per view and replayed == the eager step from the same state (up to the
    order of the fp32 atomics of the scatter)."""
    t0, s1, mvp, rays_d, gt, bg = _setup(ssaa=2, antialias=True, subdiv=2, steps=8)
    mvp = mvp.cuda()
    s1.step(mvp, rays_d, gt, bg)                                   # warm-up (eager): lazily created buffers exist afterwards
    names = ["table", "color_master", "mlp", "m_table", "v_table", "m_mlp", "v_mlp", "wpack", "opt_state", "g_mlp"]
    snap = {n: getattr(t0, n).clone() for n in names}
    snap_g = [g.clone() for g in t0.gtables]

    def restore():
        for n in names:
            getattr(t0, n).copy_(snap[n])
        for g, s in zip(t0.gtables, snap_g):
            g.copy_(s)

    s1.step(mvp, rays_d, gt, bg)
    torch.cuda.synchronize()
    eager = {n: getattr(t0, n).clone() for n in ("table", "color_master", "mlp", "opt_state")}
    loss_e = s1.read_loss()
    restore()
    s1.step(mvp, rays_d, gt, bg, use_graph=True)                   # capture + first replay
    torch.cuda.synchronize()
    assert len(s1._graphs) == 1
    assert abs(s1.read_loss() - loss_e) <= 1e-6 * abs(loss_e)
    for n, e in eager.items():
        a = getattr(t0, n)
        if n == "table":          # {float density, half2 colour} entries: compare the fp32 density features (stage 1 leaves them untouched)
            a, e = a.view(torch.float32).reshape(-1, 2)[:, 0], e.view(torch.float32).reshape(-1, 2)[:, 0]
            assert torch.equal(a, e)
            continue
        assert (a.float() - e.float()).abs().max().item() <= 1e-5 * max(1.0, e.float().abs().max().item()), n
    restore()
    s1.step(mvp, rays_d, gt, bg, use_graph=True)                   # pure replay
    torch.cuda.synchronize()
    assert len(s1._graphs) == 1 and abs(s1.read_loss() - loss_e) <= 1e-6 * abs(loss_e)


LAM_LAP, LAM_OFF, LR_V = 0.01, 0.1, 1e-3


def _vertex_setup():
    t0, s1, mvp, rays_d, gt, bg = _setup(ssaa=2, antialias=True, subdiv=2, seeded=True, lr_vert=LR_V, lambda_lap=LAM_LAP, lambda_offsets=LAM_OFF)
    t0.opt_state[0] = 4096.0
    g = torch.Generator(device="cuda").manual_seed(3)
    s1.offsets.copy_(torch.randn(s1.offsets.shape, device="cuda", generator=g) * 2e-3)
    s1.vertices.copy_(s1.base_vertices + s1.offsets)
    return t0, s1, mvp, rays_d, gt, bg


def _reference_vertex_offsets(G):
    """image loss + its gradient w.r.t. the vertices (reference composition), and the regularisers through the reference's own
    laplacian_smooth_loss with their gradient w.r.t. the offsets by autograd"""
    ref_stage, ns = _ref_ns()
    t0, s1, mvp, rays_d, gt, bg = _vertex_setup()
    ref = _reference_stage1(ns, ref_stage, t0, s1, mvp, rays_d, gt, bg, antialias=True)
    off = s1.offsets.clone().requires_grad_(True)
    reg = LAM_LAP * ns.utils.laplacian_smooth_loss(s1.base_vertices + off, s1.triangles) + LAM_OFF * (off ** 2).sum(-1).mean()
    reg.backward()
    G.put("vertex/loss", ref["loss"]); G.put("vertex/grad_vertices", ref["grad_vertices"].cpu().numpy())
    G.put("vertex/reg", float(reg)); G.put("vertex/grad_reg", off.grad.cpu().numpy())


def test_vertex_offset_optimizer_matches_autograd_and_torch_adam():
    """lr_vert > 0: the `vertices_offsets` group of the reference's stage 1 (renderer.py:160,180; regularisers utils.py:750-779).  The total
    gradient = image loss through dr.antialias (reference composition) + lambda_lap * laplacian_smooth_loss (the reference's own function)
    + lambda_offsets * mean(sum(offsets^2)) by autograd; the update = torch.optim.Adam(lr_vert, eps=1e-15) on that gradient."""
    G = gold()
    lr_v = LR_V
    t0, s1, mvp, rays_d, gt, bg = _vertex_setup()
    off_old = s1.offsets.clone()
    ref_loss, reg = G["vertex/loss"], G["vertex/reg"]
    ref_gv = torch.from_numpy(G["vertex/grad_vertices"]).cuda()
    off_grad = torch.from_numpy(G["vertex/grad_reg"]).cuda()
    t0.gtable.zero_(); t0.g_mlp.zero_()
    s1.step(mvp, rays_d, gt, bg)
    torch.cuda.synchronize()
    assert t0.opt_state[3].item() == 0
    assert abs(s1.read_loss() - (ref_loss + reg)) <= 1e-3 * abs(ref_loss + reg)
    img_part = s1.vertex_gradient()
    reg_part = s1.grad_offsets - img_part
    assert ((reg_part - off_grad).norm() / off_grad.norm()).item() <= 1e-4, ((reg_part - off_grad).norm() / off_grad.norm()).item()
    tot_ref = ref_gv + off_grad
    rel = ((s1.grad_offsets - tot_ref).norm() / tot_ref.norm()).item()
    assert rel <= 3e-2, rel
    assert img_part.abs().max().item() > 0 and (ref_gv.norm() / off_grad.norm()).item() > 1e-3      # both parts matter in the sum
    # Adam: torch's optimizer fed with OUR gradients, two steps (fresh state, as the reference's stage-1 trainer starts)
    p = torch.nn.Parameter(off_old.clone())
    opt = torch.optim.Adam([p], lr=lr_v, eps=1e-15)
    p.grad = s1.grad_offsets.clone(); opt.step()
    assert (s1.offsets - p.data).abs().max().item() <= 1e-3 * lr_v, (s1.offsets - p.data).abs().max().item()
    assert torch.equal(s1.vertices, s1.base_vertices + s1.offsets) and s1.vert_state[0].item() == 1
    s1.step(mvp, rays_d, gt, bg)
    torch.cuda.synchronize()
    p.grad = s1.grad_offsets.clone(); opt.step()
    assert (s1.offsets - p.data).abs().max().item() <= 2e-3 * lr_v
    assert s1.vert_state[0].item() == 2
    # a skipped step (found_inf) leaves the group untouched
    before = s1.offsets.clone()
    s1.forward(mvp, rays_d); s1.loss_backward(gt, bg)
    s1.grad_vclip[0, 0] = float("inf")
    from nerf2mesh_b200._lib import call, ptr, stream
    call("n2m_s1_vert_check", ptr(s1.grad_vclip), s1.vertices.shape[0], ptr(t0.opt_state), stream())
    scale = t0.opt_state[0].item()
    t0.adam(between=s1._vertex_step)
    torch.cuda.synchronize()
    assert torch.equal(s1.offsets, before) and s1.vert_state[0].item() == 2 and t0.opt_state[0].item() == 0.5 * scale


def reference_outputs(G):
    """run the reference side of the tests above that have one (needs oracle/_ref and the staged reference Python files) into G"""
    for ssaa, antialias in STAGE1_CASES:
        _reference_step(G, ssaa, antialias)
    _reference_vertex_offsets(G)
