"""Thin drivers for the UNMODIFIED reference CUDA kernels in oracle/_ref (raw pybind backends),
following the call protocol of the reference's Python wrappers (raymarching.py / grid.py /
sphere_harmonics.py), and the digests under which their bit-exact outputs are stored in
tests/golden/.  Test infrastructure only."""
import hashlib
import json
import zlib

import numpy as np
import torch


def digest(x):
    """sha256 of an array's dtype, shape and bytes: equal digests <=> bit-identical arrays"""
    a = np.ascontiguousarray(x.detach().cpu().numpy() if torch.is_tensor(x) else x)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def trace_digest(trace):
    """one digest of a sequence of (xyzs, ts) rounds"""
    return hashlib.sha256("".join(digest(x) + digest(t) for x, t in trace).encode()).hexdigest()


def sample_index(n, k, key):
    """k sorted flat indices out of n, the same for every run and every array of n entries stored under `key` (all n if n <= k)"""
    if n <= k:
        return torch.arange(n)
    g = torch.Generator().manual_seed(zlib.crc32(key.encode()))
    return torch.randperm(n, generator=g)[:k].sort().values


def sample(x, k, key):
    """float64 entries of x at sample_index(x.numel(), k, key)"""
    flat = x.detach().reshape(-1).double().cpu()
    return flat[sample_index(flat.numel(), k, key)].numpy()


def support_rows(*xs, k, key):
    """flat indices of a seeded sample of k entries (all, if fewer) among those where any of the tensors xs is non-zero: the rows
    that carry a sparse tensor's values"""
    nz = torch.zeros(xs[0].numel(), dtype=torch.bool, device=xs[0].device)
    for x in xs:
        nz |= x.detach().reshape(-1) != 0
    pool = nz.nonzero().flatten().cpu()
    return pool[sample_index(pool.numel(), k, key)]


class Golden:
    """Stored reference outputs: large tensors as a sample of their entries (`key`) plus their full-tensor max |.| and L2 norm
    (`key:absmax`, `key:norm`); scalars and digests as they are.  A sample is either seeded (sample_index) or taken at given flat
    indices, stored as `key:index` (rows where a sparse tensor is non-zero).  `put` records (generation), `take` / `cmp` read."""

    def __init__(self, path=None):
        self.d = {}
        if path is not None:
            z = np.load(path)
            meta = json.loads(str(z["meta"]))
            for k, (dt, off, shape) in meta["arrays"].items():
                n = int(np.prod(shape))
                self.d[k] = z[dt][off:off + n].reshape(shape)
            for k in [k for k in self.d if k.endswith(":index")]:
                self.d[k] = np.cumsum(self.d[k], dtype=np.int64)            # stored as differences (indices are sorted)
            self.d.update({k: np.asarray(v) for k, v in meta["scalars"].items() if not k.endswith(":index_of")})
            for k, v in meta["scalars"].items():
                if k.endswith(":index_of"):          # an index set stored once under another key
                    self.d[k[:-len("_of")]] = self.d[v]

    def put(self, key, x, k=None, index=None):
        if k is None and index is None:
            self.d[key] = np.asarray(x)
            return
        if index is None:
            self.d[key] = sample(x, k, key).astype(np.float32)
        else:
            self.d[key] = x.detach().reshape(-1).float().cpu()[index].numpy()
            self.d[key + ":index"] = np.asarray(index, dtype=np.int32)
        xd = x.detach().double()
        self.d[key + ":numel"] = np.int64(x.numel())
        self.d[key + ":absmax"] = np.float64(xd.abs().max().item() if xd.numel() else 0.0)
        self.d[key + ":norm"] = np.float64(xd.norm().item())

    def __getitem__(self, key):
        v = self.d[key]
        return v.item() if v.ndim == 0 else v

    def take(self, key, ours):
        """(our entries at the stored sample's positions, the stored sample), float64"""
        r = torch.from_numpy(self.d[key]).double()
        assert ours.numel() == self[key + ":numel"], (key, tuple(ours.shape), self[key + ":numel"])
        if key + ":index" in self.d:
            idx = torch.from_numpy(self.d[key + ":index"]).long()
            return ours.detach().reshape(-1).double().cpu()[idx], r
        return torch.from_numpy(sample(ours, r.numel(), key)), r

    def cmp(self, key, ours):
        """max error over the sample relative to the full tensor's max |.|, relative L2 error and cosine on the sample"""
        a, r = self.take(key, ours)
        scale = self[key + ":absmax"]
        return dict(max_err_of_scale=(a - r).abs().max().item() / max(scale, 1e-300),
                    rel_l2=((a - r).norm() / max(r.norm().item(), 1e-300)).item(),
                    cos=(torch.dot(a, r) / (a.norm() * r.norm() + 1e-300)).item(), scale=scale)

    def save(self, path):
        """one .npz: the arrays of each dtype concatenated into one entry named after the dtype (their places in `meta`), sorted index
        sets stored once (`key:index_of` names the key holding an identical set) and as differences; scalars and strings in `meta`"""
        layout, scalars, seen, blobs = {}, {}, {}, {}
        for k, v in sorted(self.d.items()):
            if v.ndim == 0:
                scalars[k] = v.item()
                continue
            if k.endswith(":index"):
                h = digest(v.astype(np.int64))
                if h in seen:
                    scalars[k + "_of"] = seen[h]
                    continue
                seen[h] = k
                v = np.diff(v.astype(np.int64), prepend=0).astype(np.int32)
            parts = blobs.setdefault(v.dtype.name, [])
            layout[k] = [v.dtype.name, sum(p.size for p in parts), list(v.shape)]
            parts.append(v.reshape(-1))
        np.savez_compressed(path, meta=np.asarray(json.dumps({"arrays": layout, "scalars": scalars}, sort_keys=True)),
                            **{dt: np.concatenate(parts) for dt, parts in blobs.items()})


def seeded_state(tr, seed=11):
    """Give a Stage0Trainer parameters that depend on `seed` alone, so that reference results stored for them hold in every run.  A
    trained state cannot be reproduced: the fused backward accumulates with atomics, and Adam's normalised step turns their rounding
    differences into different parameters within a few steps.  The trainer's initialisation, with the hash-grid tables drawn from
    U(-0.5, 0.5) and the density output layer scaled by 8, gives non-trivial densities (e^-3 .. e^3 and beyond), colours and gradients."""
    st = tr.export_reference_state()
    g = torch.Generator().manual_seed(seed)
    for k in ("encoder.embeddings", "encoder_color.embeddings"):
        st[k] = torch.rand(st[k].shape, generator=g) - 0.5
    st["sigma_net.net.1.weight"] = st["sigma_net.net.1.weight"] * 8.0
    tr.load_reference_state(st)


def inference_loop(c, ref=None):
    """The eval loop of renderer.py:764-802 (march_rays / composite_rays over the alive rays) on a march case, with a deterministic
    stand-in for the network; `ref` = the reference's raymarching backend, None = nerf2mesh_b200.raymarching.
    -> (ws, depth, image, rays_t, [(xyzs, ts) per round])"""
    from nerf2mesh_b200 import raymarching as rm
    ro, rd, bits, aabb = c["rays_o"].cuda(), c["rays_d"].cuda(), c["bits"].cuda(), c["aabb"].cuda()
    N = ro.shape[0]
    nears, fars = near_far(ref, ro, rd, aabb, c["min_near"]) if ref is not None else rm.near_far_from_aabb(ro, rd, aabb, c["min_near"])

    def field(xyzs):
        s = (xyzs.sum(-1) * 37.0).sin().abs() * 30.0
        return s, (xyzs * 0.5 + 0.5).clamp(0, 1)

    ws = torch.zeros(N, device="cuda"); depth = torch.zeros(N, device="cuda"); image = torch.zeros(N, 3, device="cuda")
    alive = torch.arange(N, dtype=torch.int32, device="cuda"); rays_t = nears.clone()
    step = 0
    trace = []
    while step < 256:
        n_alive = alive.shape[0]
        if n_alive <= 0:
            break
        n_step = max(min(N // n_alive, 8), 1)
        if ref is not None:
            M = n_alive * n_step
            xyzs = torch.zeros(M, 3, device="cuda"); dirs = torch.zeros(M, 3, device="cuda"); ts = torch.zeros(M, 2, device="cuda")
            noises = torch.zeros(n_alive, device="cuda")
            ref.march_rays(n_alive, n_step, alive, rays_t, ro, rd, c["bound"], c["contract"], c["dt_gamma"],
                           c["max_steps"], c["C"], c["H"], bits, nears, fars, xyzs, dirs, ts, noises)
            s, col = field(xyzs)
            ref.composite_rays(n_alive, n_step, 1e-2, False, alive, rays_t, s, col, ts, ws, depth, image)
        else:
            xyzs, dirs, ts = rm.march_rays(n_alive, n_step, alive, rays_t, ro, rd, c["bound"], c["contract"], bits,
                                           c["C"], c["H"], nears, fars, False, c["dt_gamma"], c["max_steps"])
            s, col = field(xyzs)
            rm.composite_rays(n_alive, n_step, alive, rays_t, s, col, ts, ws, depth, image, 1e-2, False)
        trace.append((xyzs.clone(), ts.clone()))
        alive = alive[alive >= 0]
        step += n_step
    return ws, depth, image, rays_t, trace


def near_far(ref, rays_o, rays_d, aabb, min_near):
    N = rays_o.shape[0]
    nears = torch.empty(N, device="cuda"); fars = torch.empty(N, device="cuda")
    ref.near_far_from_aabb(rays_o, rays_d, aabb, N, min_near, nears, fars)
    return nears, fars


def march_train(ref, rays_o, rays_d, bits, bound, contract, dt_gamma, max_steps, C, H, nears, fars, noises):
    """raymarching.py:229-241: counting pass, .item(), output pass."""
    N = rays_o.shape[0]
    counter = torch.zeros(1, dtype=torch.int32, device="cuda")
    rays = torch.empty(N, 2, dtype=torch.int32, device="cuda")
    ref.march_rays_train(rays_o, rays_d, bits, bound, contract, dt_gamma, max_steps, N, C, H, nears, fars,
                         None, None, None, rays, counter, noises)
    M = int(counter.item())
    xyzs = torch.zeros(M, 3, device="cuda"); dirs = torch.zeros(M, 3, device="cuda"); ts = torch.zeros(M, 2, device="cuda")
    ref.march_rays_train(rays_o, rays_d, bits, bound, contract, dt_gamma, max_steps, N, C, H, nears, fars,
                         xyzs, dirs, ts, rays, counter, noises)
    return xyzs, dirs, ts, rays


def by_ray(x, rays):
    """Reorder per-sample rows into ray order (the reference's offsets follow atomic order)."""
    rays = rays.cpu().numpy()
    x = x.cpu().numpy()
    parts = [x[o:o + c] for o, c in rays]
    return np.concatenate(parts, 0) if parts else x[:0]


def composite_fwd(ref, sigmas, rgbs, ts, rays, T_thresh, alpha_mode):
    M, N = sigmas.shape[0], rays.shape[0]
    weights = torch.zeros(M, device="cuda"); ws = torch.empty(N, device="cuda")
    depth = torch.empty(N, device="cuda"); image = torch.empty(N, 3, device="cuda")
    ref.composite_rays_train_forward(sigmas, rgbs, ts, rays, M, N, T_thresh, alpha_mode, weights, ws, depth, image)
    return weights, ws, depth, image


def composite_bwd(ref, gw, gws, gd, gi, sigmas, rgbs, ts, rays, ws, depth, image, T_thresh, alpha_mode):
    M, N = sigmas.shape[0], rays.shape[0]
    gs = torch.zeros_like(sigmas); gr = torch.zeros_like(rgbs)
    ref.composite_rays_train_backward(gw, gws, gd, gi, sigmas, rgbs, ts, rays, ws, depth, image, M, N, T_thresh,
                                      alpha_mode, gs, gr)
    return gs, gr


def grid_fwd(ref, inputs, emb, offsets, S, H, max_level, gridtype, align, interp, calc_dy_dx):
    B, D = inputs.shape
    L = offsets.shape[0] - 1
    C = emb.shape[1]
    out = torch.zeros(L, B, C, device="cuda", dtype=emb.dtype)
    dy = torch.zeros(B, L * D * C, device="cuda", dtype=emb.dtype) if calc_dy_dx else None
    ref.grid_encode_forward(inputs, emb, offsets, out, B, D, C, L, max_level, S, H, dy, gridtype, align, interp)
    return out, dy


def grid_bwd(ref, grad, inputs, emb, offsets, S, H, max_level, gridtype, align, interp, dy_dx):
    B, D = inputs.shape
    L = offsets.shape[0] - 1
    C = emb.shape[1]
    gemb = torch.zeros_like(emb)
    ginp = torch.zeros(B, D, device="cuda", dtype=emb.dtype) if dy_dx is not None else None
    ref.grid_encode_backward(grad, inputs, emb, offsets, gemb, B, D, C, L, max_level, S, H, dy_dx, ginp, gridtype, align, interp)
    return gemb, ginp


def sh_fwd(ref, inputs, degree, calc):
    B = inputs.shape[0]
    out = torch.empty(B, degree * degree, device="cuda")
    dy = torch.empty(B, 3 * degree * degree, device="cuda") if calc else None
    ref.sh_encode_forward(inputs, out, B, 3, degree, dy)
    return out, dy
