"""GPU parity of the FUSED stage-0 train path (include/n2m_b200_fused.h) against
  * the operator-level kernels (themselves bit-exact vs the reference CUDA kernels), and
  * the CPU train oracle (oracle/train_oracle.py, autocast-fp16 emulation),
on a small seeded batch.  Tolerances: integers bit-exact; fp32 stages bit-exact or 1e-6; stages that
carry fp16 (as the reference's autocast does) at north_star's 1e-3 of the tensor scale for forward
values and 2e-2 for fp16-accumulated gradients (the reference's own fp16 atomics have that spread)."""
import numpy as np
import pytest
import torch

import cases
from nerf2mesh_b200 import raymarching as rm
from nerf2mesh_b200 import synthetic as S
from nerf2mesh_b200.gridencoder import grid_encode
from nerf2mesh_b200.stage0 import MLP_LAYOUT, Stage0Config, Stage0Trainer

pytestmark = pytest.mark.gpu

N = 96


def make(shading="full", seed=0, lambda_tv=1e-8, N=N):
    cfg = Stage0Config(bound=1.0, num_rays=N, max_samples=N * 256, lambda_tv=lambda_tv)
    tr = Stage0Trainer(cfg, seed=seed)
    grid, bits, bricks = S.occupancy_regime("converged")
    tr.set_occupancy(bits, grid)
    ro, rd = cases.rays(N, seed=3)
    gt = S.render_bricks(ro, rd, bricks)
    g = torch.Generator().manual_seed(5)
    bg = torch.rand(N, 3, generator=g)
    noises = torch.rand(N, generator=g)
    return tr, dict(ro=ro, rd=rd, gt=gt, bg=bg, noises=noises, bits=bits, bricks=bricks)


def stage(tr, b):
    tr.rays_o.copy_(b["ro"]); tr.rays_d.copy_(b["rd"]); tr.gt.copy_(b["gt"]); tr.bg.copy_(b["bg"]); tr.noises.copy_(b["noises"])


def untile(t, M):
    """tile images [ntiles][8 chunks][128 rows][8] fp16 -> [M, 64] float"""
    nt = (M + 127) // 128
    x = t[: nt * 128 * 64].view(nt, 8, 128, 8).permute(0, 2, 1, 3).reshape(nt * 128, 64)
    return x[:M].float()


def oracle_field(tr, bound=1.0):
    from oracle import train_oracle as T
    f = T.OracleField(bound)
    st = tr.export_reference_state()
    with torch.no_grad():
        f.encoder.embeddings.copy_(st["encoder.embeddings"].cpu())
        f.encoder_color.embeddings.copy_(st["encoder_color.embeddings"].cpu())
        for name, _ in MLP_LAYOUT:
            mod, _, idx, _ = name.split(".")
            getattr(f, mod).net[int(idx)].weight.copy_(st[name].cpu())
    return f, T


def test_march_and_encode_match_operator_kernels():
    tr, b = make()
    stage(tr, b)
    tr.march(); tr.encode_fwd()
    torch.cuda.synchronize()
    c = tr.cfg
    nears, fars = rm.near_far_from_aabb(tr.rays_o, tr.rays_d, tr.aabb, c.min_near)
    from nerf2mesh_b200._lib import call, ptr, stream
    counter = torch.zeros(1, dtype=torch.int32, device="cuda"); rays = torch.empty(N, 2, dtype=torch.int32, device="cuda")
    tbuf = torch.empty(N * c.max_steps * 2, device="cuda")
    args = (ptr(tr.rays_o), ptr(tr.rays_d), ptr(tr.density_bitfield), c.real_bound, 0, c.dt_gamma, c.max_steps, N, c.cascade, c.grid_size, ptr(nears), ptr(fars))
    call("n2m_march_rays_train", *args, None, None, None, ptr(rays), ptr(counter), ptr(tr.noises), ptr(tbuf), stream())
    M = int(counter.item())
    xyzs = torch.zeros(M, 3, device="cuda"); dirs = torch.zeros(M, 3, device="cuda"); ts = torch.zeros(M, 2, device="cuda")
    call("n2m_march_rays_train", *args, ptr(xyzs), ptr(dirs), ptr(ts), ptr(rays), ptr(counter), ptr(tr.noises), ptr(tbuf), stream())
    assert tr.counters[0].item() == M and tr.counters[1].item() == M and tr.counters[2].item() == 0 and M > 1000
    assert torch.equal(tr.rays, rays)
    assert torch.equal(tr.recs[:M, 2], ts[:, 0]) and torch.equal(tr.recs[:M, 1], ts[:, 1])
    enc = untile(tr.enc_tiles, M)
    assert torch.equal(enc[:, 0:3], xyzs.half().float())
    d = dirs / torch.sqrt(torch.clamp((dirs * dirs).sum(-1, keepdim=True), min=1e-20))
    assert torch.equal(enc[:, 51:54], d.half().float())
    assert enc[:, 54:].abs().max() == 0
    st = tr.export_reference_state()
    x01 = (xyzs + 1.0) / 2.0
    e_d = grid_encode(x01, st["encoder.embeddings"], tr.offsets, c.per_level_scale, 16)
    assert torch.equal(enc[:, 3:19], e_d.half().float())                     # fp32 path: bit-exact then one fp16 rounding
    with torch.autocast("cuda", dtype=torch.float16):
        e_c = grid_encode(x01, st["encoder_color.embeddings"], tr.offsets, c.per_level_scale, 16)
    # colour features: fp32 accumulation here vs the reference's per-corner fp16 accumulation
    assert (enc[:, 19:51] - e_c.float()).abs().max().item() <= 3e-3 * e_c.float().abs().max().item()


@pytest.mark.parametrize("shading", ["full", "diffuse"])
def test_forward_loss_and_gradients_match_train_oracle(shading):
    tr, b = make(shading)
    f, T = oracle_field(tr)
    stage(tr, b)
    tr._fill_params(shading == "full", True)
    tr.forward_backward()
    torch.cuda.synchronize()
    M = int(tr.counters[1].item())
    cfg = dict(bound=1.0, C=1, H=128)
    out = T.render_train(f, b["ro"], b["rd"], b["bits"], cfg, b["noises"], b["bg"], shading, amp=True)
    assert out["num_points"] == M
    loss = T.train_loss(out, b["gt"], b["bg"], tr.cfg.lambda_mask, tr.cfg.lambda_specular)
    loss.backward()
    # forward values
    sig = tr.out[:M, 0].cpu(); rgb = tr.out[:M, 1:].cpu()
    assert (sig - out["sigmas"].detach()).abs().max().item() <= 2e-3 * out["sigmas"].abs().max().item()
    assert (rgb - out["rgbs"].detach().float()).abs().max().item() <= 2e-3
    assert (tr.image.cpu() - out["image"].detach()).abs().max().item() <= 1e-3
    assert (tr.weights_sum.cpu() - out["weights_sum"].detach()).abs().max().item() <= 1e-3
    assert abs(tr.read_loss() - loss.item()) <= 1e-3 * abs(loss.item())
    # gradients (un-scaled)
    g = tr.export_reference_grads()
    ref = {"encoder.embeddings": f.encoder.embeddings.grad, "encoder_color.embeddings": f.encoder_color.embeddings.grad}
    for name, _ in MLP_LAYOUT:
        mod, _, idx, _ = name.split(".")
        ref[name] = getattr(f, mod).net[int(idx)].weight.grad
    # TV gradient is added by the fused scatter; add it to the oracle's density-table gradient
    from oracle import grid_oracle
    x01 = (out["xyzs"] + 1.0) / 2.0
    ref["encoder.embeddings"] = ref["encoder.embeddings"] + grid_oracle.grad_total_variation(
        x01, f.encoder.embeddings.detach(), f.offsets, tr.cfg.lambda_tv, f.S, f.H).float()
    for name, r in ref.items():
        if r is None:
            assert shading == "diffuse" and name.startswith("specular")
            continue
        a = g[name].cpu().double().flatten(); r = r.double().flatten()
        scale = r.abs().max().item()
        assert scale > 0, name
        err = (a - r).abs().max().item()
        cos = torch.dot(a, r) / (a.norm() * r.norm() + 1e-300)
        assert err <= 3e-2 * scale and cos > 0.999, f"{name}: err {err:.3e} scale {scale:.3e} cos {cos:.6f}"


def test_adam_matches_torch_and_graph_replay():
    tr, b = make()
    stage(tr, b)
    tr.forward_backward()
    g = tr.export_reference_grads()
    before = tr.export_reference_state()
    tr.adam()
    after = tr.export_reference_state()
    torch.cuda.synchronize()
    assert tr.opt_state[2].item() == 1 and tr.opt_state[3].item() == 0
    assert tr.gtable.abs().max().item() == 0 and tr.g_mlp.abs().max().item() == 0
    for name in g:
        p = before[name].clone().requires_grad_(True)
        opt = torch.optim.Adam([p], lr=tr.cfg.lr, eps=tr.cfg.eps)
        p.grad = g[name].clone()
        opt.step()
        d_ref = (p.detach() - before[name]); d = (after[name] - before[name])
        assert (d - d_ref).abs().max().item() <= 1e-4 * d_ref.abs().max().item() + 1e-9, name
    # fp16 working copy of the colour table == half(master)
    tab_c = tr.table.view(torch.float16).view(-1, 4)[:, 2:4].float()
    assert torch.equal(tab_c, after["encoder_color.embeddings"].half().float())
    # a second trainer: eager vs CUDA-graph steps give the same loss trajectory
    losses = []
    for use_graph in (False, True):
        t2, b2 = make(seed=1)
        ls = []
        for it in range(3):
            t2.step(b2["ro"], b2["rd"], b2["gt"], b2["bg"], b2["noises"], use_graph=use_graph)
            ls.append(t2.read_loss())
        losses.append(ls)
    assert np.allclose(losses[0], losses[1], rtol=1e-3), losses
    assert losses[0][2] < losses[0][0]          # it trains


def test_overflow_drops_rays_and_inf_skips_step():
    cfg = Stage0Config(bound=1.0, num_rays=N, max_samples=1024)
    tr = Stage0Trainer(cfg)
    _, bits, bricks = S.occupancy_regime("cold")
    tr.set_occupancy(bits)
    ro, rd = cases.rays(N, seed=3)
    tr.rays_o.copy_(ro); tr.rays_d.copy_(rd); tr.gt.copy_(S.render_bricks(ro, rd, bricks)); tr.bg.fill_(1.0)
    tr.forward_backward()
    torch.cuda.synchronize()
    assert tr.counters[0].item() > 1024 and tr.counters[1].item() == 1024 and tr.counters[2].item() == 1
    assert torch.isfinite(tr.gtable).all() and torch.isfinite(tr.image).all()
    # force an overflow: absurd loss scale -> inf in fp16 gradients -> step skipped, scale halved
    tr.gtable.zero_(); tr.g_mlp.zero_()
    tr.opt_state[0] = 1e30
    before = tr.mlp.clone()
    tr.forward_backward(); tr.adam()
    torch.cuda.synchronize()
    assert torch.equal(before, tr.mlp) and tr.opt_state[2].item() == 0
    assert tr.opt_state[0].item() == pytest.approx(5e29, rel=1e-3)


@pytest.mark.parametrize("name", cases.MARCH_CASES)
def test_warp_marcher_equals_serial_marcher(name):
    """The warp-per-ray marcher must reproduce the sequential marcher bit for bit (counts and (t, dt) of every
    sample), for every marching configuration incl. cascades, dt_gamma > 0 and contraction."""
    from nerf2mesh_b200._lib import call
    c = cases.march_case(name)
    Nr = c["rays_o"].shape[0]
    cfg = Stage0Config(bound=c["bound"], contract=c["contract"], dt_gamma=c["dt_gamma"], num_rays=Nr, max_samples=Nr * 1024)
    assert cfg.cascade == c["C"]
    tr = Stage0Trainer(cfg)
    tr.set_occupancy(c["bits"])
    tr.rays_o.copy_(c["rays_o"]); tr.rays_d.copy_(c["rays_d"]); tr.noises.copy_(c["noises"])
    res = []
    for serial in (1, 0):
        call("n2m_s0_set_serial_march", serial)
        tr.recs.zero_()
        tr.march()
        torch.cuda.synchronize()
        res.append((tr.counters.clone(), tr.rays.clone(), tr.recs.clone()))
    call("n2m_s0_set_serial_march", 0)
    (c0, r0, s0), (c1, r1, s1) = res
    assert torch.equal(c0, c1) and c0[0].item() > 0
    assert torch.equal(r0, r1)
    M = int(c0[1].item())
    assert torch.equal(s0[:M], s1[:M])


@pytest.mark.parametrize("shading,n_rays,nparts", [("full", 192, 1), ("diffuse", 192, 1), ("full", 3072, 1), ("full", 3072, 2)])
def test_fused_backward_equals_two_kernel_backward(shading, n_rays, nparts):
    """k_s0_bwd_fused (MLP backward + scatter in one warp-specialised persistent launch, feature gradients handed over in shared
    memory) vs k_mlp_bwd followed by k_s0_encode_bwd: same table / weight gradients up to the order of the fp32 atomics; 3072 rays give
    every CTA several tiles (both buffers and both barrier phases are exercised), two parts exercise the boundary-tile row masks."""
    tr, b = make(shading, N=n_rays)
    tr.nparts = nparts
    stage(tr, b)
    tr._fill_params(shading == "full", True)
    res = []
    for fused in (False, True):
        tr.fused_bwd = fused
        tr.gtable.zero_(); tr.g_mlp.zero_(); tr.opt_state[3] = 0
        tr.forward_backward()
        torch.cuda.synchronize()
        res.append({k: v.clone() for k, v in tr.export_reference_grads().items()})
        assert tr.opt_state[3].item() == 0
    M = int(tr.counters[1].item())
    assert M > 128 * (148 if n_rays > 1000 else 1)
    for name in res[0]:
        a, r = res[1][name].double(), res[0][name].double()
        assert r.abs().max().item() > 0 or (shading == "diffuse" and name.startswith("specular")), name
        assert (a - r).abs().max().item() <= 1e-4 * r.abs().max().item() + 1e-12, name
    # the inf flag is raised by the fused kernel too
    tr.gtable.zero_(); tr.g_mlp.zero_()
    tr.opt_state[0] = 1e30
    tr.forward_backward()
    torch.cuda.synchronize()
    assert tr.opt_state[3].item() == 1


def test_update_density_grid_matches_reference_composition():
    """Stage0Trainer.update_density_grid vs the reference's update_extra_state arithmetic (renderer.py:1074-1149)
    composed from torch + the (bit-exact) operator-level encoder, same random jitter (one [H^3, 3] draw per cascade in the
    reference's meshgrid order).  The comparison against the UNMODIFIED reference method is in test_gpu_reference_parity.py."""
    import torch.nn.functional as Fnn
    from nerf2mesh_b200 import raymarching as rm
    tr, b = make()
    c = tr.cfg
    H = c.grid_size
    st = tr.export_reference_state()
    tr.density_grid.zero_()
    torch.manual_seed(123)
    tr.update_density_grid(decay=0.95, density_thresh=10.0)
    torch.cuda.synchronize()
    # reference composition (renderer.py:1095-1118)
    torch.manual_seed(123)
    ax = torch.arange(H, dtype=torch.int32, device="cuda")
    xx, yy, zz = torch.meshgrid(ax, ax, ax, indexing="ij")
    coords = torch.cat([xx.reshape(-1, 1), yy.reshape(-1, 1), zz.reshape(-1, 1)], dim=-1)
    indices = rm.morton3D(coords).long()
    xyz = 2 * coords.float() / (H - 1) - 1
    hgs = 1.0 / H
    xyz = xyz * (1.0 - hgs)
    xyz += (torch.rand_like(xyz) * 2 - 1) * hgs
    sig = torch.empty(H ** 3, device="cuda")
    for a0 in range(0, H ** 3, 1 << 19):
        x = xyz[a0:a0 + (1 << 19)]
        enc = grid_encode((x + 1) / 2, st["encoder.embeddings"], tr.offsets, c.per_level_scale, 16)
        with torch.autocast("cuda", dtype=torch.float16):
            h = Fnn.linear(torch.cat([x, enc], -1), st["sigma_net.net.0.weight"]).relu()
            h = Fnn.linear(h, st["sigma_net.net.1.weight"])
        sig[a0:a0 + (1 << 19)] = torch.exp(h[:, 0].float())
    grid = torch.zeros(1, H ** 3, device="cuda")
    grid[0, indices] = sig                                   # max(0 * decay, sigma)
    assert (tr.density_grid - grid).abs().max().item() <= 2e-3 * grid.abs().max().item()
    mean = tr.density_grid.clamp(min=0).mean().item()
    assert abs(tr.mean_density.item() - mean) < 1e-6
    assert torch.equal(tr.density_bitfield, rm.packbits(tr.density_grid, min(mean, 10.0)))      # on-device threshold == host threshold
    occ = (tr.density_grid > min(mean, 10.0)).float().mean().item()
    assert 0.05 < occ < 0.95


def test_render_equals_training_forward():
    """chunked render(early_stop=False) == the training forward on the same rays (host chunking / padding logic), and the renderer with
    the device-side alive-ray bookkeeping (csrc/render.cu) == that image up to the order in which the transmittance is accumulated; the
    parity of render() against the reference's inference loop is test_evaluation_render_matches_reference_inference_loop in
    test_gpu_reference_parity.py"""
    tr, b = make()
    stage(tr, b)
    tr.noises.zero_()
    tr.forward_backward()
    img0 = tr.image.clone(); ws0 = tr.weights_sum.clone(); dep0 = tr.depth.clone()
    img, ws, dep = tr.render(b["ro"].cuda(), b["rd"].cuda(), bg_color=b["bg"].cuda(), early_stop=False)
    assert torch.equal(img, img0) and torch.equal(ws, ws0)
    # ragged call: more rays than one chunk, white background
    ro2 = torch.cat([b["ro"], b["ro"][:10]]).cuda(); rd2 = torch.cat([b["rd"], b["rd"][:10]]).cuda()
    img2, ws2, _ = tr.render(ro2, rd2, bg_color=1.0, early_stop=False)
    assert img2.shape == (N + 10, 3) and torch.equal(img2[:10], img2[N:])
    assert torch.isfinite(img2).all()
    # per-ray background tensor with a ragged last chunk
    bgt = torch.rand(N + 10, 3, device="cuda")
    img3, _, _ = tr.render(ro2, rd2, bg_color=bgt, early_stop=False)
    assert torch.allclose(img3 - (1 - ws2)[:, None] * bgt, img2 - (1 - ws2)[:, None], atol=1e-6)
    # ---- device-side alive-ray renderer: one chunk, several ragged chunks, and a schedule too short to finish (extra rounds) ----
    assert (ws0 > 0.5).float().mean().item() > 0.05
    for kw in (dict(), dict(chunk=40), dict(chunk=32)):
        e_img, e_ws, e_dep = tr.render(b["ro"].cuda(), b["rd"].cuda(), bg_color=b["bg"].cuda(), **kw)
        assert (e_img - img0).abs().max().item() <= 2e-4, (kw, (e_img - img0).abs().max().item())
        assert (e_ws - ws0).abs().max().item() <= 2e-4 and (e_dep - dep0).abs().max().item() <= 2e-4 * max(1.0, dep0.abs().max().item())
    rounds_default = tr.render_rounds
    assert rounds_default == len(tr.RENDER_SCHEDULE)
    tr.RENDER_SCHEDULE = (2, 2)
    try:
        e_img, e_ws, _ = tr.render(ro2, rd2, bg_color=bgt)
        assert tr.render_rounds > 2                                  # rays were left alive: the read-back triggered further rounds
    finally:
        del tr.RENDER_SCHEDULE                                       # back to the class default
    assert (e_img - img3).abs().max().item() <= 2e-4 and (e_ws - ws2).abs().max().item() <= 2e-4
    # early termination is real: the rounds evaluate fewer sample rows than the march emitted for the whole batch
    assert torch.isfinite(e_img).all()


@pytest.mark.parametrize("nparts", [2, 4, 8])
def test_ray_range_parts_equal_whole_batch(nparts):
    """include/n2m_b200_fused.h "Ray-range parts": the per-part chains (concurrent streams, boundary tiles computed by
    both neighbours with row masks) give the same forward values exactly and the same loss / gradients up to fp32
    atomic summation order."""
    tr, b = make()
    tr.fused_bwd = False          # the two-kernel backward leaves the feature gradients in denc_tiles, compared below
    stage(tr, b)
    tr.forward_backward()
    torch.cuda.synchronize()
    M = int(tr.counters[1].item())
    bounds = tr.counters[4:13].cpu().tolist()
    assert bounds[0] == 0 and bounds[8] == M and all(bounds[i] <= bounds[i + 1] for i in range(8))
    for e in range(8):
        assert bounds[e] == int(tr.rays[N * e // 8, 0].item())
    assert any(x % 128 for x in bounds[1:8])                 # boundaries really fall inside tiles
    ref = dict(out=tr.out[:M].clone(), dout=tr.dout[:M].clone(), image=tr.image.clone(), ws=tr.weights_sum.clone(),
               loss=tr.read_loss(), enc=untile(tr.enc_tiles, M), denc=untile(tr.denc_tiles, M))
    g_ref = tr.export_reference_grads()
    tr.gtable.zero_(); tr.g_mlp.zero_()
    tr.enc_tiles.zero_(); tr.denc_tiles.zero_(); tr.out.zero_(); tr.dout.zero_()
    tr.nparts = nparts
    tr.forward_backward()
    torch.cuda.synchronize()
    assert torch.equal(untile(tr.enc_tiles, M), ref["enc"])
    assert torch.equal(tr.out[:M], ref["out"])
    assert torch.equal(tr.image, ref["image"]) and torch.equal(tr.weights_sum, ref["ws"])
    assert torch.equal(tr.dout[:M], ref["dout"])
    assert torch.equal(untile(tr.denc_tiles, M), ref["denc"])
    assert abs(tr.read_loss() - ref["loss"]) <= 1e-5 * abs(ref["loss"])
    g = tr.export_reference_grads()
    for name in g_ref:
        a, r = g[name].double(), g_ref[name].double()
        assert (a - r).abs().max().item() <= 1e-4 * r.abs().max().item() + 1e-12, name
    # and a graph-captured multi-stream step trains like the single-stream one
    losses = []
    for P_ in (1, nparts):
        t2, b2 = make(seed=1)
        t2.nparts = P_
        ls = []
        for it in range(3):
            t2.step(b2["ro"], b2["rd"], b2["gt"], b2["bg"], b2["noises"], use_graph=True)
            ls.append(t2.read_loss())
        losses.append(ls)
    assert np.allclose(losses[0], losses[1], rtol=1e-3), losses


def _operator_march(tr, Nr):
    """xyzs, dirs, ts, rays of the operator-level marcher (bit-exact vs the reference kernel, test_gpu_raymarching) on the
    trainer's staged rays / noises / bitfield."""
    from nerf2mesh_b200._lib import call, ptr, stream
    c = tr.cfg
    nears, fars = rm.near_far_from_aabb(tr.rays_o, tr.rays_d, tr.aabb, c.min_near)
    counter = torch.zeros(1, dtype=torch.int32, device="cuda"); rays = torch.empty(Nr, 2, dtype=torch.int32, device="cuda")
    tbuf = torch.empty(Nr * c.max_steps * 2, device="cuda")
    args = (ptr(tr.rays_o), ptr(tr.rays_d), ptr(tr.density_bitfield), c.real_bound, int(c.contract), c.dt_gamma, c.max_steps, Nr,
            c.cascade, c.grid_size, ptr(nears), ptr(fars))
    call("n2m_march_rays_train", *args, None, None, None, ptr(rays), ptr(counter), ptr(tr.noises), ptr(tbuf), stream())
    M = int(counter.item())
    xyzs = torch.zeros(M, 3, device="cuda"); dirs = torch.zeros(M, 3, device="cuda"); ts = torch.zeros(M, 2, device="cuda")
    call("n2m_march_rays_train", *args, ptr(xyzs), ptr(dirs), ptr(ts), ptr(rays), ptr(counter), ptr(tr.noises), ptr(tbuf), stream())
    torch.cuda.synchronize()
    return xyzs, dirs, ts, rays, M


@pytest.mark.parametrize("name,lambda_entropy", [("lego_converged", 1e-2), ("garden_cascades", 1e-3)])
def test_entropy_and_cascades_through_the_fused_step(name, lambda_entropy):
    """The garden recipe's extras through the fused path (scripts/runall_360_outdoor.sh, SURVEY.md section 8d config 4):
    bound 16 => 5 cascades and a 32768-resolution grid, dt_gamma 1/256, entropy regulariser on weights and weights_sum
    (utils.py:728-733, with the reference's grad_weights folding, raymarching.cu:676), TV weight x10 outside the unit cube
    (utils.py:815-821).  Samples are taken from the operator-level marcher (asserted identical to the fused one), everything
    behind it is checked against the train oracle."""
    c = cases.march_case(name)
    Nr = 96
    cfg = Stage0Config(bound=c["bound"], dt_gamma=c["dt_gamma"], num_rays=Nr, max_samples=Nr * 1024, lambda_entropy=lambda_entropy)
    assert cfg.cascade == c["C"]
    tr = Stage0Trainer(cfg, seed=2)
    tr.tv_fallback_points = 0       # this scene has no sample outside the unit cube: the reference's outer TV call would fall back to random
    #                                 points (grid.py:181-183; covered by test_tv_random_point_fallback), which the train oracle does not model
    tr.set_occupancy(c["bits"])
    ro, rd = c["rays_o"][:Nr].contiguous(), c["rays_d"][:Nr].contiguous()
    gt = S.render_bricks(ro, rd, c["bricks"])
    g = torch.Generator().manual_seed(11)
    bg = torch.rand(Nr, 3, generator=g)
    stage(tr, dict(ro=ro, rd=rd, gt=gt, bg=bg, noises=c["noises"][:Nr]))
    st = tr.export_reference_state()
    # some opacity, so that rays terminate and the weights spread over (0, 1); |x| reaches `bound`, keep exp() in range
    st["sigma_net.net.1.weight"] = st["sigma_net.net.1.weight"] * (30.0 if c["bound"] <= 1 else 4.0)
    tr.load_reference_state(st)
    tr._fill_params(True, True)
    tr.forward_backward()
    torch.cuda.synchronize()
    M = int(tr.counters[1].item())
    xyzs, dirs, ts, rays, M_op = _operator_march(tr, Nr)
    assert M_op == M and tr.counters[2].item() == 0 and M > 1000
    assert torch.equal(tr.rays, rays) and torch.equal(tr.recs[:M, 2], ts[:, 0]) and torch.equal(tr.recs[:M, 1], ts[:, 1])

    f, T = oracle_field(tr, c["bound"])
    d = dirs / torch.sqrt(torch.clamp((dirs * dirs).sum(-1, keepdim=True), min=1e-20))
    sigmas, rgbs, specs = f(xyzs.cpu(), d.cpu(), "full", True)
    weights, ws, depth, image = T._CompositeRef.apply(sigmas.float(), rgbs.float(), ts.cpu(), rays.cpu().numpy(), 1e-4)
    image = image + (1 - ws).unsqueeze(-1) * bg
    out = dict(image=image, weights_sum=ws, weights=weights, speculars=specs)
    loss = T.train_loss(out, gt, bg, cfg.lambda_mask, cfg.lambda_specular, lambda_entropy=lambda_entropy)
    loss.backward()
    assert (tr.out[:M, 0].cpu() - sigmas.detach()).abs().max().item() <= 2e-3 * sigmas.abs().max().item()
    assert (tr.image.cpu() - image.detach()).abs().max().item() <= 1e-3
    assert (tr.weights_sum.cpu() - ws.detach()).abs().max().item() <= 1e-3
    assert 0.05 < ws.mean().item() < 0.99
    assert abs(tr.read_loss() - loss.item()) <= 1e-3 * abs(loss.item())
    # gradients; TV on the density table: weight inside the unit cube, 10 x outside when bound > 1
    from oracle import grid_oracle
    ref = {"encoder.embeddings": f.encoder.embeddings.grad.clone(), "encoder_color.embeddings": f.encoder_color.embeddings.grad}
    for nm, _ in MLP_LAYOUT:
        mod, _, idx, _ = nm.split(".")
        ref[nm] = getattr(f, mod).net[int(idx)].weight.grad
    xc = xyzs.cpu()
    inner = xc.abs().amax(-1) <= 1
    groups = [(xc, cfg.lambda_tv)] if c["bound"] <= 1 else [(xc[inner], cfg.lambda_tv), (xc[~inner], cfg.lambda_tv * 10)]
    for pts, lam in groups:
        if pts.shape[0]:
            x01 = (pts + c["bound"]) / (2 * c["bound"])
            ref["encoder.embeddings"] += grid_oracle.grad_total_variation(x01, f.encoder.embeddings.detach(), f.offsets, lam, f.S, f.H).float()
    gq = tr.export_reference_grads()
    for nm, r in ref.items():
        a = gq[nm].cpu().double().flatten(); r = r.double().flatten()
        scale = r.abs().max().item()
        assert scale > 0, nm
        err = (a - r).abs().max().item()
        cos = torch.dot(a, r) / (a.norm() * r.norm() + 1e-300)
        assert err <= 3e-2 * scale and cos > 0.999, f"{nm}: err {err:.3e} scale {scale:.3e} cos {cos:.6f}"
    # the entropy term is really in there: without it the sigma_net gradient differs
    tr.gtable.zero_(); tr.g_mlp.zero_()
    tr.cfg.lambda_entropy = 0.0
    tr._fill_params(True, True)
    tr.forward_backward()
    g0 = tr.export_reference_grads()["sigma_net.net.0.weight"].cpu()
    assert (g0 - gq["sigma_net.net.0.weight"].cpu()).abs().max().item() > 1e-3 * g0.abs().max().item()


def test_reference_state_dict_and_checkpoint_schema(tmp_path):
    """export_reference_state() carries exactly the stage-0 NeRFNetwork.state_dict() keys (renderer.py:92-117, grid.py:135-140,
    network.py:66-75) and the checkpoint has the fields Trainer.load_checkpoint reads (utils.py:1423-1470); round trip."""
    tr, b = make()
    st = tr.export_reference_state()
    expect = {"aabb_train", "aabb_infer", "density_grid", "density_bitfield", "encoder.offsets", "encoder.embeddings",
              "encoder_color.offsets", "encoder_color.embeddings"} | {n for n, _ in MLP_LAYOUT}
    assert set(st) == expect
    assert st["encoder.embeddings"].shape == (tr.rows, 1) and st["encoder_color.embeddings"].shape == (tr.rows, 2)
    assert st["encoder.offsets"].dtype == torch.int32 and st["encoder.offsets"].numel() == 17 and int(st["encoder.offsets"][-1]) == tr.rows
    assert st["aabb_train"].tolist() == [-1, -1, -1, 1, 1, 1]
    assert st["density_grid"].shape == (1, 128 ** 3) and st["density_bitfield"].dtype == torch.uint8
    stage(tr, b)
    tr.step(use_graph=False)
    path = tmp_path / "ngp_stage0_ep0001.pth"
    tr.save_reference_checkpoint(str(path), epoch=1)
    ck = torch.load(str(path), weights_only=False)
    assert {"epoch", "global_step", "stats", "stage", "mean_density", "model"} <= set(ck) and ck["global_step"] == 1 and ck["stage"] == 0
    t2 = Stage0Trainer(tr.cfg, seed=123)
    t2.load_reference_state(ck["model"])
    s2 = t2.export_reference_state()
    for k, v in tr.export_reference_state().items():
        assert torch.equal(v, s2[k]), k


def _tv_fallback_points():
    tr, b = make(N=96)
    stage(tr, b)
    tr.tv_fallback_points = 20000
    tr.march()
    torch.cuda.synchronize()
    pts = torch.zeros(tr.tv_fallback_points, 3, device="cuda")
    tr.gtable.zero_()
    tr.tv_random(dump=pts)                      # test hook: unconditional, weight lambda_tv
    torch.cuda.synchronize()
    return tr, pts


def reference_outputs(G):
    """the REFERENCE kernel's TV gradient at the fallback points (tests/golden/make_golden.py; needs oracle/_ref)"""
    import numpy as np
    import refcall
    from oracle.build_ref import load_ref
    tr, pts = _tv_fallback_points()
    st = tr.export_reference_state()
    emb = st["encoder.embeddings"].contiguous()
    grad = torch.zeros_like(emb)
    S_ = float(np.log2(tr.cfg.per_level_scale))
    load_ref("_ref_gridencoder").grad_total_variation(pts, emb, grad, tr.offsets, tr.cfg.lambda_tv, pts.shape[0], 3, 1, 16, S_, 16, 0, False)
    torch.cuda.synchronize()
    G.put("tv_fallback/points", refcall.digest(pts))
    G.put("tv_fallback/grad", grad, index=refcall.support_rows(grad, k=2048, key="tv_fallback/grad"))


def test_tv_random_point_fallback():
    """GridEncoder.grad_total_variation's fallback (grid.py:181-183, reached from utils.py:815-823 when a TV call gets no sample): the
    fused path evaluates the same TV gradient at its own hash-generated points; fed to the REFERENCE kernel, those points give the same
    gradient (stored in tests/golden/reference_model.npz, on a seeded sample of the rows it reaches).  And the fallback fires exactly for
    the groups the TV pass counted as empty."""
    import os
    import refcall
    tr, pts = _tv_fallback_points()
    assert pts.min().item() >= 0 and pts.max().item() < 1 and abs(pts.mean().item() - 0.5) < 0.01
    ours = tr.export_reference_grads()["encoder.embeddings"]
    G = refcall.Golden(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_model.npz"))
    assert refcall.digest(pts) == G["tv_fallback/points"], "the stored reference gradient belongs to another point set"
    scale = G["tv_fallback/grad:absmax"]
    assert scale > 0
    a, r = G.take("tv_fallback/grad", ours)
    assert (a - r).abs().max().item() <= 1e-4 * scale, ((a - r).abs().max().item(), scale)
    # a new point set every optimizer step
    pts2 = torch.zeros_like(pts)
    tr.opt_state[2] += 1
    tr.tv_random(dump=pts2)
    assert not torch.equal(pts, pts2)
    # bound 1, samples present: the single TV call is populated -> no fallback
    tr.gtable.zero_()
    tr.tv()
    base = tr.gtable.clone()
    assert tr.counters[3].item() == tr.counters[1].item() and tr.counters[15].item() == 0
    tr.gtable.zero_(); tr.counters[3] = 0            # pretend the batch marched nothing: the fallback adds its gradient
    tr.tv_random()
    assert tr.gtable[:, 0].abs().max().item() > 0 and base[:, 0].abs().max().item() > 0
    tr.gtable.zero_(); tr.counters[3] = 5
    tr.tv_random()
    assert tr.gtable.abs().max().item() == 0


@pytest.mark.parametrize("shading,n_rays", [("full", 96), ("diffuse", 96), ("full", 4096)])
def test_fused_forward_equals_two_kernel_forward(shading, n_rays):
    """k_s0_fwd_fused (gather groups -> shared-memory tile image -> tcgen05 MLP rounds, TMA store of the image for the backward) vs
    k_s0_encode_fwd followed by k_mlp_fwd: bit-identical tile images and outputs (same per-sample arithmetic); 4096 rays give every CTA
    several tiles per gather group (buffer reuse, both barrier phases, the bulk-store read fence)."""
    tr, b = make(shading, N=n_rays)
    stage(tr, b)
    tr._fill_params(shading == "full", True)
    tr.march()
    res = []
    for fused in (False, True):
        tr.enc_tiles.zero_(); tr.out.zero_(); tr.loss_acc.zero_()
        if fused:
            tr.fwd_fused()
        else:
            tr.encode_fwd(); tr.mlp_fwd()
        torch.cuda.synchronize()
        res.append((tr.enc_tiles.clone(), tr.out.clone(), tr.loss_acc[1].item()))
    M = int(tr.counters[1].item())
    assert M > (128 * 296 * 2 if n_rays > 1000 else 1000)
    nt = (M + 127) // 128
    assert torch.equal(res[0][0][: nt * 128 * 64], res[1][0][: nt * 128 * 64])
    assert torch.equal(res[0][1][:M], res[1][1][:M])
    assert abs(res[0][2] - res[1][2]) <= 1e-5 * max(abs(res[0][2]), 1e-12)
    # and a whole step through the fused forward (+ fused backward) trains like the default path
    losses = []
    for ff in (False, True):
        t2, b2 = make(seed=1, N=n_rays if n_rays < 1000 else 512)
        t2.nparts = 1
        t2.fused_fwd = ff; t2.fused_bwd = ff
        ls = []
        for it in range(3):
            t2.step(b2["ro"], b2["rd"], b2["gt"], b2["bg"], b2["noises"], use_graph=True)
            ls.append(t2.read_loss())
        losses.append(ls)
    assert np.allclose(losses[0], losses[1], rtol=1e-3), losses
