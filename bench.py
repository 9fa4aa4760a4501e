#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native stage-0 train step (BASELINE.json metric:
ray-samples/sec of one full train step, device-timed).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (default workload: lego_stage0_converged)
    python bench.py --workload garden_stage0                        # BASELINE config 4 (bound 16, 5 cascades, entropy, cam near/far)
    python bench.py --workload lego_stage1                          # BASELINE config 5 (rasterize + texture-MLP step; pixels/s)
    python bench.py --impl reference [--steps K] [--warmup W]      # CPU restatement of the reference step on the host cores
    torchrun --nproc-per-node N bench.py --gpus N ...              # one rank per GPU (NCCL)

One "step" = one optimizer step of the fused pipeline on one batch of 4096 synthetic rays (march -> hash-grid encode -> tcgen05
MLPs -> composite + loss -> backward -> TV -> Adam).  `value` = samples of all ranks / max-over-ranks device time with the batch
already resident in HBM; `e2e` = the same through Stage0Trainer.step() with pinned-host batches (H2D inside the timed region) and a
D2H read of the loss every step.  Also in the line: `roofline` (dominant kernel, timed live with CUDA events, cold L2),
`cpu_baseline` (oracle port on the host cores, bounded sample), `reference_cuda` (the UNMODIFIED reference model + trainer over the
reference's own kernels, same box, same batches), `psnr` (ours vs that reference after the same short training run).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NUM_RAYS = 4096
ALG_BYTES = {"encode_fwd": 1053, "fwd_fused": 1053, "encode_bwd": 1024, "bwd_fused": 1024, "step": 2077}      # SURVEY.md section 8(d), bytes per sample

WORKLOADS = {
    # BASELINE config 2: lego recipe (readme.md:64): bound 1, dt_gamma 0, RGBA targets + mask loss, TV 1e-8
    "lego_stage0_converged": dict(bound=1.0, dt_gamma=0.0, lambda_entropy=0.0, radius=None, alpha=True, cam_nf=False, cap=128),
    # BASELINE config 4: garden recipe (scripts/runall_360_outdoor.sh:2): bound 16 => 5 cascades, dt_gamma 1/256, per-view camera
    # near/far, entropy regulariser 1e-3, RGB targets, TV with the 10x outer weight (utils.py:815-821)
    "garden_stage0": dict(bound=16.0, dt_gamma=1.0 / 256, lambda_entropy=1e-3, radius=1.2, alpha=False, cam_nf=True, cap=320),
}


DUMP_MAX_ELEMS = 1 << 20      # per array: larger outputs are dumped as a fixed seeded sample of this many entries (<= 64 MB in all)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array as <out_dir>/<name>.npy (float32, float64 kept); an array of more than DUMP_MAX_ELEMS entries is
    replaced by its entries at a sorted sample of flat indices seeded by the name, the same in every run, so that two builds can be
    compared output for output."""
    import zlib
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = torch.as_tensor(a).detach().reshape(-1).cpu()
        a = a.double() if a.dtype == torch.float64 else a.float()
        if a.numel() > DUMP_MAX_ELEMS:
            g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
            idx = torch.randperm(a.numel(), generator=g)[:DUMP_MAX_ELEMS].sort().values
            a = a[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), a.numpy())


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            pk = json.load(f)
        return float(pk["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` capture of this command
    (profiles/ncu_traffic.json, written by profiles/summarize_ncu.py), or None when that kernel was not captured."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)
        e = t["kernels"].get(kernel)
        return None if e is None else {"bytes": e["dram_bytes"], "capture": t.get("capture")}
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe).  NVML is polled in-process about every
    millisecond (a timed region of a few dozen sub-millisecond steps is shorter than one `nvidia-smi -lms 100` period); if NVML
    cannot be loaded the nvidia-smi loop is the fallback."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.mx, self.reasons, self.proc = index, [], [], set(), None
        self._stop_evt = threading.Event()
        self._nv = None
        try:                                   # NVML start-up (tens of ms) happens here, before the timed region
            import pynvml as nv
            nv.nvmlInit()
            self._h = nv.nvmlDeviceGetHandleByIndex(index)
            self.mx.append(int(nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)))
            self._nv = nv
        except Exception:
            self._nv = None

    def _run_nvml(self):
        nv, h = self._nv, self._h
        if nv is None:
            raise RuntimeError("NVML unavailable")
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop_evt.is_set():
            self.sm.append(int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            mask = int(get_reasons(h))
            for bit, name in self.REASONS.items():
                if mask & bit:
                    self.reasons.add(name)
            time.sleep(0.001)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                      "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            if r and r[0].isdigit():
                self.sm.append(int(r[0]))
            if len(r) > 1 and r[1].isdigit():
                self.mx.append(int(r[1]))
            for i in range(4):
                if len(r) >= 6 and r[2 + i].lower().startswith("active"):
                    self.reasons.add(names[i])

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            try:
                self._run_smi()
            except Exception:
                pass

    def stop(self):
        self._stop_evt.set()
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2.0)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# synthetic workloads (no datasets are available): SURVEY.md section 8(d)
# ------------------------------------------------------------------------------------------------
_SCENES = {}


def scene(workload):
    from nerf2mesh_b200 import synthetic as S
    if workload not in _SCENES:
        w = WORKLOADS[workload]
        _SCENES[workload] = S.garden_scene(bound=w["bound"]) if w["bound"] > 1 else S.occupancy_regime("converged")
    return _SCENES[workload]


def make_batches(n_batches, seed, pin, workload="lego_stage0_converged"):
    from nerf2mesh_b200 import synthetic as S
    w = WORKLOADS[workload]
    grid, bits, bricks = scene(workload)
    radius = w["radius"] or S.LEGO_RADIUS
    poses = S.orbit_cameras(100, radius=radius, seed=0)
    intr = S.lego_intrinsics()
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n_batches):
        ro, rd, _, _ = S.sample_rays(poses, intr, 800, 800, NUM_RAYS, g)
        gt = S.render_bricks(ro, rd, bricks)
        if not w["alpha"]:
            gt = (gt[:, :3] * gt[:, 3:] + (1 - gt[:, 3:])).contiguous()          # RGB images: white where nothing is hit
        bg = torch.rand(NUM_RAYS, 3, generator=g)
        noises = torch.rand(NUM_RAYS, generator=g)
        b = dict(ro=ro, rd=rd, gt=gt, bg=bg, noises=noises)
        if w["cam_nf"]:
            d = ro.norm(dim=-1)
            b["cnf"] = torch.stack([(d - 1.1).clamp(min=0.05), d + 14.0], -1).contiguous()
        if pin:
            b = {k: v.pin_memory() for k, v in b.items()}
        out.append(b)
    return out, grid, bits


def make_trainer(workload):
    from nerf2mesh_b200.stage0 import Stage0Config, Stage0Trainer
    w = WORKLOADS[workload]
    cfg = Stage0Config(bound=w["bound"], dt_gamma=w["dt_gamma"], lambda_entropy=w["lambda_entropy"], num_rays=NUM_RAYS,
                       max_samples=NUM_RAYS * w["cap"])
    tr = Stage0Trainer(cfg, seed=0)
    tr.use_cam_near_far = w["cam_nf"]
    return tr


# ------------------------------------------------------------------------------------------------
# CPU arm: the repo's PyTorch restatement of the reference step (the reference has no CPU path, SURVEY.md section 8c)
# ------------------------------------------------------------------------------------------------
def cpu_step_rate(steps, warmup, budget_s=150.0):
    """Times the CPU restatement of the lego train step (oracle/train_oracle.py) on a bounded sample of the 4096-ray batch: the
    thread count and the sample size are calibrated first with 8-ray steps (more threads are not always faster for the index-heavy
    torch ops), then the sample is sized so that (warmup + steps) steps end within `budget_s` -- up to the full 4096 rays."""
    from oracle import train_oracle as T
    torch.manual_seed(0)
    batches, grid, bits = make_batches(1, 123, False)
    cfg = dict(bound=1.0, C=1, H=128)
    ncpu = os.cpu_count() or 1

    def fresh():
        f = T.OracleField(1.0)
        return f, torch.optim.Adam(f.parameters(), lr=1e-2, eps=1e-15)

    def one(f, opt, b):
        t0 = time.perf_counter()
        _, out = T.train_step(f, opt, b["ro"], b["rd"], b["gt"], bits, cfg, b["noises"], b["bg"], "full", True)
        return time.perf_counter() - t0, out["num_points"]

    b8 = {k: v[:8] for k, v in batches[0].items()}
    best = None
    for nt in sorted({ncpu, min(ncpu, 32), min(ncpu, 8)}, reverse=True):
        torch.set_num_threads(nt)
        f, opt = fresh()
        one(f, opt, b8)                                   # first call at this setting: thread-pool start-up
        dt, _ = one(f, opt, b8)
        if best is None or dt < best[0]:
            best = (dt, nt)
    t8, threads = best
    torch.set_num_threads(threads)
    per_step = budget_s / max(steps + warmup, 1)
    rays = int(max(8, min(NUM_RAYS, 8 * per_step / max(t8, 1e-3))))        # t8 / 8 over-estimates the per-ray cost (fixed overheads)
    b = {k: v[:rays] for k, v in batches[0].items()}
    f, opt = fresh()
    samples, t_total = 0, 0.0
    for it in range(warmup + steps):
        dt, m = one(f, opt, b)
        if it >= warmup:
            samples += m; t_total += dt
    return samples / t_total, t_total / max(steps, 1), threads, rays


def cpu_baseline_dict(v, threads, rays, what):
    return {"value": v, "unit": "samples/s", "cores": os.cpu_count(), "threads_used": threads, "kind": "port",
            "sample": f"{rays} of the {NUM_RAYS} rays of one lego batch per step, full train step (oracle/train_oracle.py: march, "
                      f"hash-grid encode, autocast-emulated MLPs, composite, loss, backward, TV, Adam), {what}; torch threads "
                      f"calibrated over {{all, 32, 8}} -> {threads} of {os.cpu_count()} host threads"}


def run_reference(args):
    """`--impl reference`: the reference has no CPU implementation of this path (SURVEY.md section 8c), so this arm times the
    CPU restatement (oracle port) with the host threads that serve it best, on a bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    v, sec, threads, rays = cpu_step_rate(steps, warmup, budget_s=float(args.cpu_budget_s))
    line = {"impl": "reference", "metric": "ray-samples/sec (train step)", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "config": {"workload": "lego_stage0_converged", "rays_per_batch": NUM_RAYS, "rays_per_timed_step": rays},
            "cpu_baseline": cpu_baseline_dict(v, threads, rays, f"{warmup} warm-up + {steps} timed steps"),
            "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# same-box GPU baseline: the UNMODIFIED reference model + Trainer over the reference's own kernels (oracle/ref_stage.py)
# ------------------------------------------------------------------------------------------------
def reference_cuda_leg(workload, dev_batches, state, steps=10, warmup=3):
    try:
        from oracle import ref_stage
        if not ref_stage.staged():
            return {"unavailable": "reference Python files not staged (oracle/_ref/py)"}
        w = WORKLOADS[workload]
        ns = ref_stage.load("ref")
        opt = ref_stage.default_opt(bound=w["bound"], dt_gamma=w["dt_gamma"], lambda_entropy=w["lambda_entropy"], adaptive_num_rays=False,
                                    num_rays=NUM_RAYS, enable_cam_near_far=w["cam_nf"])
        model = ns.make_model(opt)
        model.load_state_dict({k: v.clone() for k, v in state.items()}, strict=True)
        model.cuda().train()
        rt = ns.utils.Trainer("ngp", opt, model, device=torch.device("cuda"), workspace=None, mute=True,
                              optimizer=lambda m: torch.optim.Adam(m.get_params(opt.lr), eps=1e-15),
                              criterion=torch.nn.MSELoss(reduction="none"), ema_decay=None, fp16=True, use_checkpoint="scratch",
                              use_tensorboardX=False, scheduler_update_every_step=True)
        rt.global_step = 2000
        samples, ms = 0, 0.0
        for it in range(warmup + steps):
            b = dev_batches[it % len(dev_batches)]
            data = dict(rays_o=b["ro"], rays_d=b["rd"], index=[0], images=b["gt"])
            if "cnf" in b:
                data["cam_near_far"] = b["cnf"]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rt.optimizer.zero_grad()                                  # nerf/utils.py:1163-1177
            _, _, loss = rt.train_step(data)
            rt.scaler.scale(loss).backward()
            rt.post_train_step()
            rt.scaler.step(rt.optimizer)
            rt.scaler.update()
            e1.record()
            torch.cuda.synchronize()
            if it >= warmup:
                ms += e0.elapsed_time(e1)
                samples += int(rt.tmp_xyzs.shape[0])
        del rt, model
        torch.cuda.empty_cache()
        return {"value": samples / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms / steps, "steps": steps,
                "what": "unmodified nerf/network.py + nerf/renderer.py + nerf/utils.py (Trainer.train_step, post_train_step, "
                        "GradScaler, torch.optim.Adam) over the reference's own CUDA kernels built for sm_100a, same batches, "
                        "device-resident inputs, CUDA events"}
    except Exception as e:      # noqa: BLE001
        return {"unavailable": repr(e)[:300]}


def psnr_leg(iters, eval_res=100, eval_views=2, seed=0):
    """BASELINE.json 'PSNR vs ref': the lego recipe (readme.md:64: 4096 rays, density-grid update every 16 steps, diffuse shading for
    the first third, lr warm-up + decay) for `iters` steps on the analytic scene -- once with this repo's fused trainer, once with the
    reference's kernels in the reference's composition (oracle/ref_pipeline.py) on the same batch stream -- then PSNR of held-out
    views against the analytic ground truth."""
    try:
        from nerf2mesh_b200 import synthetic as S
        from nerf2mesh_b200.stage0 import Stage0Config, Stage0Trainer
        from nerf2mesh_b200.train_synthetic import full_image_rays, lr_at, psnr
        from oracle import ref_pipeline as RP
        dev = "cuda"
        bricks = S.make_bricks()
        poses = S.orbit_cameras(100, seed=0)
        test_poses = S.orbit_cameras(eval_views, seed=12345)
        intr = S.lego_intrinsics()
        diffuse_until = iters // 3
        res = {}
        for which in ("ours", "reference"):
            torch.manual_seed(seed)
            g = torch.Generator().manual_seed(seed + 1)
            if which == "ours":
                tr = Stage0Trainer(Stage0Config(bound=1.0, num_rays=NUM_RAYS, max_samples=NUM_RAYS * 640), seed=seed)
                tr.density_grid.zero_()
                init = tr.export_reference_state()
            else:
                tr = RP.RefTrainer(1.0)
                tr.field.load_reference_state(init)
            t0 = time.time()
            for it in range(iters):
                if it % 16 == 0:
                    tr.update_density_grid() if which == "ours" else tr.update_extra_state()
                ro, rd, _, _ = S.sample_rays(poses, intr, 800, 800, NUM_RAYS, g)
                gt = S.render_bricks(ro, rd, bricks); bg = torch.rand(NUM_RAYS, 3, generator=g); noises = torch.rand(NUM_RAYS, generator=g)
                sh = "diffuse" if it < diffuse_until else "full"
                if which == "ours":
                    tr.step(ro, rd, gt, bg, noises, shading=sh, lr=lr_at(it, iters))
                else:
                    tr.step(ro.to(dev), rd.to(dev), gt.to(dev), bg.to(dev), sh, lr_at(it, iters))
            torch.cuda.synchronize()
            secs = time.time() - t0
            vals = []
            for k in range(eval_views):
                ro, rd = full_image_rays(test_poses[k], intr / (800 // eval_res), eval_res, eval_res)
                gtv = S.render_bricks(ro, rd, bricks)
                gt_rgb = gtv[:, :3] * gtv[:, 3:] + (1 - gtv[:, 3:])
                if which == "ours":
                    img, _, _ = tr.render(ro.to(dev), rd.to(dev), bg_color=1.0, shading="full")
                else:
                    img = tr.render_eval(ro.to(dev), rd.to(dev), 1.0, "full")
                vals.append(psnr(img.clamp(0, 1).cpu(), gt_rgb))
            res[which] = {"psnr_db": sum(vals) / len(vals), "train_seconds": secs}
            if which == "ours":
                over, max_m = tr.check_capacity(grow=False)
                res[which]["overflowed_steps"] = over
                # evaluation renderer on a full 800 x 800 view of this model: device-side alive-ray rounds (csrc/render.cu) against
                # the all-samples path (every marched sample through the training kernels), CUDA events, second call of each
                ro, rd = full_image_rays(test_poses[0], intr, 800, 800)
                ro, rd = ro.to(dev), rd.to(dev)
                ev = {"rays": int(ro.shape[0])}
                for name, kw in (("alive_rounds", {}), ("all_samples", {"early_stop": False})):
                    a_img, _, _ = tr.render(ro, rd, bg_color=1.0, **kw)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); a_img, _, _ = tr.render(ro, rd, bg_color=1.0, **kw); e1.record()
                    torch.cuda.synchronize()
                    ev[name + "_ms"] = e0.elapsed_time(e1)
                    if name == "alive_rounds":
                        ev["sample_rows_evaluated"] = int(tr.render_rows); first = a_img
                    else:
                        ev["max_abs_diff"] = float((a_img - first).abs().max().item())
                res["eval_render"] = ev
            del tr
            torch.cuda.empty_cache()
        res["iters"] = iters
        res["delta_db"] = res["ours"]["psnr_db"] - res["reference"]["psnr_db"]
        res["what"] = (f"lego recipe, {iters} steps of 4096 rays on the analytic bricks scene (host-synthesised batches, same stream for "
                       f"both), {eval_views} held-out {eval_res}x{eval_res} views vs analytic ground truth; reference = its own kernels in "
                       "its own composition (oracle/ref_pipeline.py)")
        return res
    except Exception as e:      # noqa: BLE001
        return {"unavailable": repr(e)[:300]}


def dp_divergence_check(workload, mode, rank, world, rays=512, steps=4):
    """N > 1: the fused data-parallel optimizer actually used (`mode`: nvls / peer) against the library baseline (NCCL all-reduce +
    replicated Adam) on small identical replicas: after `steps` steps every rank must hold bit-identical parameters, and they must agree
    with the NCCL path up to the summation order of the reduction."""
    import torch.distributed as dist
    from nerf2mesh_b200 import synthetic as S
    from nerf2mesh_b200.parallel import GradSync, make_grad_sync
    from nerf2mesh_b200.stage0 import Stage0Config, Stage0Trainer
    if mode == "nccl":
        return {"mode": "nccl", "note": "library path in use; nothing to compare"}
    w = WORKLOADS[workload]
    grid, bits, bricks = scene(workload)
    g = torch.Generator().manual_seed(77 + rank)
    poses = S.orbit_cameras(100, radius=w["radius"] or S.LEGO_RADIUS, seed=0)
    ro, rd, _, _ = S.sample_rays(poses, S.lego_intrinsics(), 800, 800, rays, g)
    gt = S.render_bricks(ro, rd, bricks)
    if not w["alpha"]:
        gt = (gt[:, :3] * gt[:, 3:] + (1 - gt[:, 3:])).contiguous()
    bg = torch.rand(rays, 3, generator=g); noises = torch.rand(rays, generator=g)
    res = {}
    for which in (mode, "nccl"):
        cfg = Stage0Config(bound=w["bound"], dt_gamma=w["dt_gamma"], lambda_entropy=w["lambda_entropy"], num_rays=rays, max_samples=rays * 1024)
        t = Stage0Trainer(cfg, seed=0)
        t.set_occupancy(bits, grid)
        sync = GradSync(t) if which == "nccl" else make_grad_sync(t, which)[0]
        for it in range(steps):
            t.step(ro, rd, gt, bg, noises, grad_sync=sync, use_graph=False)
        torch.cuda.synchronize()
        st = t.export_reference_state()
        res[which] = torch.cat([st[k].reshape(-1) for k in ("encoder.embeddings", "encoder_color.embeddings", "color_net.net.0.weight", "sigma_net.net.0.weight")])
        del t, sync
        torch.cuda.empty_cache()
        dist.barrier()
    mine = res[mode]
    ref0 = mine.clone()
    dist.broadcast(ref0, src=0)
    spread = (mine - ref0).abs().max().reshape(1)
    dist.all_reduce(spread, op=dist.ReduceOp.MAX)
    moved = (res["nccl"] - res["nccl"].mean()).abs().max().item()
    return {"mode": mode, "steps": steps, "rays_per_rank": rays, "replicas_bit_identical": bool(spread.item() == 0.0),
            "max_abs_diff_vs_nccl": (mine - res["nccl"]).abs().max().item(), "param_spread": moved,
            "rel_diff_vs_nccl": (mine - res["nccl"]).abs().max().item() / max(moved, 1e-12)}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (nerf2mesh_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from nerf2mesh_b200 import _lib

    workload = args.workload
    tr = make_trainer(workload)
    tr.nparts = args.parts
    tr.fused_bwd = bool(args.fused_bwd)
    tr.fused_fwd = bool(args.fused_fwd)
    tr.defer_zero = bool(args.defer_zero)
    tr.prefetch_at = args.prefetch_at
    if tr.fused_fwd:
        tr.nparts = 1
    sync, dp_used = None, args.dp
    if world > 1:
        from nerf2mesh_b200.parallel import make_grad_sync
        sync, dp_used = make_grad_sync(tr, args.dp)
    n_batches = 8
    host_batches, grid, bits = make_batches(n_batches, 1000 + rank, True, workload)
    dev_batches = [{k: v.cuda(non_blocking=True) for k, v in b.items()} for b in host_batches]
    tr.set_occupancy(bits, grid)
    m_total = torch.zeros(1, dtype=torch.int64, device="cuda")
    K, W = args.steps, args.warmup

    def tup(b):
        return (b["ro"], b["rd"], b["gt"], b["bg"], b["noises"]) + ((b["cnf"],) if "cnf" in b else ())

    def one_step(batches, it):
        # the next batch is handed over too: its H2D copy + march overlap this step on a side stream
        b = batches[it % n_batches]
        nb = None if args.no_prefetch else tup(batches[(it + 1) % n_batches])
        tr.step(b["ro"], b["rd"], b["gt"], b["bg"], b["noises"], shading="full", use_graph=not args.no_graph, grad_sync=sync,
                next_batch=nb, cam_near_far=b.get("cnf"))
        m_total.add_(tr.counters[1])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- launches per step (eager, counted by the library) ----
    l0 = _lib.launch_count()
    b0 = dev_batches[0]
    tr.step(b0["ro"], b0["rd"], b0["gt"], b0["bg"], b0["noises"], use_graph=False, grad_sync=sync, cam_near_far=b0.get("cnf"))
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - l0
    state0 = tr.export_reference_state() if (rank == 0 and world == 1 and not args.skip_reference) else None

    # ---- leg 1: device-resident inputs ----
    for it in range(W):
        one_step(dev_batches, it)
    barrier()
    m_total.zero_()
    sampler = ClockSampler(local); sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for it in range(K):
        one_step(dev_batches, W + it)
    e1.record()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs:          # what the last timed step returned: its loss, render, sample count and updated parameters
        # every rank exports: under the sharded optimizers export_reference_state() gathers the colour masters (a collective)
        outputs = {"loss": torch.tensor([tr.read_loss()], dtype=torch.float64), "image": tr.image, "weights_sum": tr.weights_sum,
                   "depth": tr.depth, "num_samples": tr.counters[1:2], **tr.export_reference_state()}
        if rank == 0:
            dump_outputs(args.dump_outputs, outputs)
        del outputs
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    samples = m_total.clone().float()
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(samples, op=dist.ReduceOp.SUM)
    ms_total = ms.item(); samples_total = samples.item()
    value = samples_total / (ms_total * 1e-3)
    overflow_steps, max_m = tr.check_capacity(grow=False)

    # ---- leg 2: end to end (pinned host -> device inside the timed region, loss read back every step) ----
    tr.drop_prefetch()
    for it in range(4):                     # untimed: (slot, parity) graph variants this leg's phase needs
        one_step(host_batches, n_batches - 4 + it)
    tr.drop_prefetch()
    barrier()
    m_total.zero_()
    loss_host = torch.zeros(4).pin_memory(); cnt_host = torch.zeros(4, dtype=torch.int32).pin_memory()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    f0.record()
    e2e_samples = 0
    for it in range(K):
        one_step(host_batches, it)
        loss_host.copy_(tr.loss_acc, non_blocking=True); cnt_host.copy_(tr.counters[:4], non_blocking=True)
        torch.cuda.current_stream().synchronize()            # the user-visible result of the step
        e2e_samples += int(cnt_host[1])
    f1.record()
    barrier()
    ms2 = torch.tensor([f0.elapsed_time(f1)], device="cuda"); s2 = torch.tensor([float(e2e_samples)], device="cuda")
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX); dist.all_reduce(s2, op=dist.ReduceOp.SUM)
    e2e_value = s2.item() / (ms2.item() * 1e-3)
    h2d = sum(v.numel() * v.element_size() for v in host_batches[0].values())
    d2h = loss_host.numel() * 4 + cnt_host.numel() * 4

    # ---- per-stage device times (eager, CUDA events on the launching stream, L2 flushed before each) -> roofline ----
    tr.drop_prefetch()
    torch.cuda.synchronize()
    stages = ["march"] + (["fwd_fused", "tv"] if tr.fused_fwd else ["encode_fwd", "tv", "mlp_fwd"]) + ["composite_loss"] + \
             (["bwd_fused"] if tr.fused_bwd else ["mlp_bwd", "encode_bwd"]) + ["adam"]
    acc = {s: 0.0 for s in stages}
    reps = 5
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda")     # > 126 MB L2
    for r in range(reps):
        b = dev_batches[r % n_batches]
        tr.slots[tr.cur].load(b["ro"], b["rd"], b["gt"], b["bg"], b["noises"], b.get("cnf"))
        tr.loss_acc.zero_()
        for s in stages:
            flush.fill_(0.0)
            a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); getattr(tr, s)(); z.record()
            torch.cuda.synchronize()
            acc[s] += a.elapsed_time(z) / reps
    M_last = int(tr.counters[1].item())
    # density-grid update (every 16 steps in the reference, utils.py:1155-1156): timed on its own, the analytic occupancy is restored
    keep_bits, keep_grid = tr.density_bitfield.clone(), tr.density_grid.clone()
    upd_ms = 0.0
    for r in range(3):
        a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); tr.update_density_grid(); z.record()
        torch.cuda.synchronize()
        if r > 0:
            upd_ms += a.elapsed_time(z) / 2
    tr.set_occupancy(keep_bits, keep_grid)
    peak, peak_kind = load_peaks()
    dom = max(("fwd_fused" if tr.fused_fwd else "encode_fwd", "bwd_fused" if tr.fused_bwd else "encode_bwd"), key=lambda s: acc[s])
    achieved = ALG_BYTES[dom] * M_last / (acc[dom] * 1e-3) / 1e9
    kname = {"encode_fwd": "k_s0_encode_fwd", "encode_bwd": "k_s0_encode_bwd", "bwd_fused": "k_s0_bwd_fused", "fwd_fused": "k_s0_fwd_fused"}[dom]
    traffic = ncu_traffic(kname)
    roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None if traffic is None else traffic["bytes"],
                "traffic_capture": None if traffic is None else traffic["capture"], "alg_bytes_per_sample": ALG_BYTES[dom],
                "samples_per_launch": M_last, "kernel_ms": acc[dom], "stage_ms_cold_l2": {k: round(v, 4) for k, v in acc.items()},
                "step_frac_of_hbm": ALG_BYTES["step"] * value / 1e9 / peak}

    dp_check, dp_stage_ms = None, None
    if world > 1:
        if getattr(sync, "fused", False):       # device time of the fused reduce-scatter + Adam + all-gather stage alone (eager, max over ranks)
            t_dp = 0.0
            for r in range(5):
                barrier()
                a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); sync.run(tr.parity); z.record()
                torch.cuda.synchronize()
                t_dp += a.elapsed_time(z) / 5
            t_dp = torch.tensor([t_dp], device="cuda")
            dist.all_reduce(t_dp, op=dist.ReduceOp.MAX)
            dp_stage_ms = t_dp.item()
        dp_check = dp_divergence_check(workload, dp_used, rank, world)

    if rank == 0:
        cpu = None
        if world == 1 and not args.skip_cpu:
            v, sec, threads, rays = cpu_step_rate(1, 1, budget_s=30.0)
            cpu = cpu_baseline_dict(v, threads, rays, "1 warm-up + 1 timed step")
        refc = None
        if state0 is not None:
            del flush
            torch.cuda.empty_cache()
            refc = reference_cuda_leg(workload, dev_batches, state0)
        ps = None
        if world == 1 and args.psnr_iters > 0 and workload == "lego_stage0_converged":
            ps = psnr_leg(args.psnr_iters)
        step_ms = ms_total / K
        line = {"metric": "ray-samples/sec (train step)", "value": value, "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp16",
                "data": "synthetic",
                "config": {"workload": workload, "rays_per_batch": NUM_RAYS, "global_rays": NUM_RAYS * world,
                           "samples_per_step": samples_total / K, "parallelism": f"dp{world}" + ("" if world == 1 else f"-{dp_used}"),
                           "cuda_graph": not args.no_graph, "ray_range_parts": int(tr.nparts), "fused_bwd": bool(tr.fused_bwd), "fused_fwd": bool(tr.fused_fwd), "defer_zero": bool(tr.defer_zero), "prefetch_at": tr.prefetch_at,
                           "march_prefetch": not args.no_prefetch, **{k: v for k, v in WORKLOADS[workload].items() if k != "cap"},
                           "sample_capacity": tr.Mcap, "capacity_overflow_steps": overflow_steps, "max_samples_seen": max_m,
                           "l2": "inputs cycle over 8 batches; tables+grads+Adam state (0.6 GB touched per step) exceed the 126 MB L2"},
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms2.item() / K},
                "gpu_launches": int(launches_per_step * K), "launches_per_step": int(launches_per_step),
                "roofline": roofline, "cpu_baseline": cpu,
                "density_update": {"ms_per_call": upd_ms, "every_steps": 16, "cells": int(tr.density_grid.numel()),
                                   "value_with_update": samples_total / K / ((step_ms + upd_ms / 16) * 1e-3)},
                "reference_cuda": refc, "psnr": ps, "dp_check": dp_check, "dp_stage_ms": dp_stage_ms}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# stage-1 workload (BASELINE config 5)
# ------------------------------------------------------------------------------------------------
def run_stage1(args):
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device")
    import numpy as np
    from nerf2mesh_b200 import synthetic as S
    from nerf2mesh_b200.stage0 import Stage0Config, Stage0Trainer
    from nerf2mesh_b200.stage1 import Stage1Trainer
    from nerf2mesh_b200.train_synthetic import full_image_rays
    R = S                                            # mesh / projection builders (host-side input synthesis)
    h0 = w0 = 800
    t0 = Stage0Trainer(Stage0Config(bound=1.0, num_rays=1024, max_samples=1024 * 128), seed=0)
    v, f = R.icosphere(7)                                         # 327 680 faces ~ the reference's decimate target 3e5 (main.py:101)
    lr_vert = float(args.lr_vert) if args.antialias else 0.0           # the vertex offsets are trained through dr.antialias only
    s1 = Stage1Trainer(t0, torch.from_numpy(v), torch.from_numpy(f), h0, w0, ssaa=2, antialias=bool(args.antialias), lr_vert=lr_vert)
    g = torch.Generator().manual_seed(0)
    views = []
    for k in range(8):
        cam = S.orbit_cameras(8, radius=2.35, seed=3)[k, :3, 3].numpy().astype(np.float64)      # the sphere covers ~40 % of the view
        pose = torch.from_numpy(S.look_at_pose(cam).astype(np.float32))
        intr = S.lego_intrinsics(h0, w0)
        _, rd = full_image_rays(pose, intr, h0, w0)
        mvp = R.perspective_mvp(cam, fovy=2 * np.arctan(0.5 * h0 / intr[1]), aspect=w0 / h0); mvp[1] *= -1
        gt = torch.rand(h0 * w0, 4, generator=g); gt[:, 3] = 1.0
        views.append((torch.from_numpy(mvp).cuda(), rd.cuda(), gt.cuda(), torch.rand(h0 * w0, 3, generator=g).cuda()))
    K, W = args.steps, max(args.warmup, 17)            # every view's graph is captured during warm-up
    ug = not args.no_graph
    for it in range(W):
        s1.step(*views[it % 8], use_graph=ug)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cov = torch.zeros(1, dtype=torch.int64, device="cuda")
    e0.record()
    for it in range(K):
        s1.step(*views[(W + it) % 8], use_graph=ug)
        cov.add_(s1.counters[1])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K
    if args.dump_outputs:          # what the last timed step returned: its loss, image, coverage and updated parameters
        dump_outputs(args.dump_outputs, {"loss": torch.tensor([s1.read_loss()], dtype=torch.float64), "image": s1.image,
                                         "weights_sum": s1.weights_sum, "covered_pixels": s1.counters[1:2], "vertex_offsets": s1.offsets,
                                         **t0.export_reference_state()})
    # rasterize + points alone
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for it in range(10):
        s1.forward(*views[it % 8][:2])
    r1.record()
    torch.cuda.synchronize()
    from nerf2mesh_b200 import raster as dr
    glctx = dr.RasterizeCudaContext()
    vclip = torch.nn.functional.pad(s1.vertices, (0, 1), value=1.0) @ views[0][0].T
    q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dr.rasterize(glctx, vclip[None], s1.triangles, (s1.h, s1.w))
    q0.record()
    for it in range(10):
        dr.rasterize(glctx, vclip[None], s1.triangles, (s1.h, s1.w))
    q1.record()
    torch.cuda.synchronize()
    aa_ms = None
    if s1.antialias:          # the antialias operator alone (4 channels): forward, backward (colour + vertex gradients)
        th = s1.topology
        from nerf2mesh_b200._lib import call, ptr, stream
        a0, a1, a2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a0.record()
        for it in range(10):
            call("n2m_antialias_forward", ptr(s1.rgba), ptr(s1.rast), ptr(s1.vclip), ptr(s1.triangles), ptr(th.keys), ptr(th.opp), th.slots, s1.h, s1.w, 4,
                 ptr(s1.aa), stream())
        a1.record()
        for it in range(10):
            call("n2m_antialias_backward", ptr(s1.rgba), ptr(s1.rast), ptr(s1.vclip), ptr(s1.triangles), ptr(th.keys), ptr(th.opp), th.slots, s1.h, s1.w, 4,
                 ptr(s1.d_aa), 1.0, ptr(s1.g_rgba), ptr(s1.grad_vclip), stream())
        a2.record()
        torch.cuda.synchronize()
        aa_ms = {"forward": a0.elapsed_time(a1) / 10, "backward": a1.elapsed_time(a2) / 10,
                 "blended_pixels": int(((s1.aa - s1.rgba).abs().amax(1) > 0).sum().item())}
    hi = s1.h * s1.w
    line = {"metric": "pixels/sec (stage-1 texture step: rasterize + interpolate + colour MLPs fwd/bwd + Adam)",
            "value": hi / (ms * 1e-3), "unit": "super-sampled pixels/s", "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "config": {"workload": "lego_stage1", "mesh_faces": int(f.shape[0]), "image": [h0, w0], "ssaa": 2, "raster": [s1.h, s1.w],
                       "covered_pixels_per_step": cov.item() / K, "antialias": bool(s1.antialias), "cuda_graph": ug,
                       "lr_vert": lr_vert, "lambda_lap": s1.lambda_lap, "lambda_offsets": s1.lambda_offsets},
            "antialias_ms": aa_ms,
            "rasterize_ms": q0.elapsed_time(q1) / 10, "rasterize_pixels_per_s": hi / (q0.elapsed_time(q1) / 10 * 1e-3),
            "forward_ms": r0.elapsed_time(r1) / 10}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="lego_stage0_converged", choices=list(WORKLOADS) + ["lego_stage1"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-prefetch", action="store_true", help="do not overlap the next batch's march with this step")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="--impl reference: wall-clock budget of the whole CPU run")
    ap.add_argument("--skip-reference", action="store_true", help="skip the same-box reference-CUDA leg")
    ap.add_argument("--psnr-iters", type=int, default=300, help="training steps of the PSNR-vs-reference pair (0 = skip)")
    ap.add_argument("--lr-vert", type=float, default=1e-4, help="lego_stage1 with --antialias 1: learning rate of the vertex-offset group (main.py:49; 0 = vertices fixed)")
    ap.add_argument("--antialias", type=int, default=1, help="lego_stage1: 1 = dr.antialias on (rgbs, alphas) as the reference does (renderer.py:886-887)")
    ap.add_argument("--prefetch-at", default="optimizer", choices=["optimizer", "start"],
                    help="where the next batch's march is released on the side stream: under the optimizer stage or under the forward pass")
    ap.add_argument("--defer-zero", type=int, default=1, help="1: the gradient table is zeroed on a side stream under the next step instead of by the optimizer kernel")
    ap.add_argument("--fused-fwd", type=int, default=0, help="1: gather + MLP forward as one warp-specialised launch (implies --parts 1)")
    ap.add_argument("--fused-bwd", type=int, default=1, help="1: MLP backward + scatter as one warp-specialised launch (csrc/fused.cu)")
    ap.add_argument("--parts", type=int, default=2, choices=[1, 2, 4, 8],
                    help="ray-range parts run as concurrent gather->MLP->composite->MLP'->scatter chains on forked streams")
    ap.add_argument("--dp", default="auto", choices=["auto", "nvls", "peer", "nccl"],
                    help="N > 1: 'nvls' = reduce-scatter inside the NVSwitch (multimem) + sharded Adam + multicast all-gather, 'peer' = the "
                         "same with P2P loads / stores over NVLink, 'nccl' = all-reduce + replicated Adam, 'auto' = first that sets up")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arms")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "lego_stage1":
        run_stage1(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
