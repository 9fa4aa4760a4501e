"""CPU: host-side logic and the C ABI surface (no kernel is launched)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    names = []
    for h in sorted(f for f in os.listdir(os.path.join(ROOT, "include")) if f.endswith(".h")):
        src = open(os.path.join(ROOT, "include", h)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names += re.findall(r"\b(n2m_[a-zA-Z0-9_]+)\s*\(", src)
    return sorted(set(names))


def test_headers_are_plain_c(tmp_path):
    """the drop-in boundary is a C ABI: every header under include/ must compile as C99 on its own (no C++ types, no torch types)"""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        import pytest
        pytest.skip("gcc not available")
    for h in sorted(f for f in os.listdir(os.path.join(ROOT, "include")) if f.endswith(".h")):
        r = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-x", "c", os.path.join(ROOT, "include", h)],
                           capture_output=True, text=True)
        assert r.returncode == 0, (h, r.stderr[:500])
        code = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", h)).read(), flags=re.S)        # declarations without the comments
        assert "at::" not in code and "torch" not in code and "std::" not in code


def test_library_exports_every_declared_symbol():
    from nerf2mesh_b200 import _lib
    syms = declared_symbols()
    assert len(syms) >= 30
    for s in syms:
        assert hasattr(_lib.lib, s), f"libn2m_b200.so does not export {s}"
    assert _lib.lib.n2m_version() == 100
    # loading leaves no error message: checked in a fresh interpreter, since tests that run earlier in this one provoke errors on purpose
    r = subprocess.run([sys.executable, "-c", "from nerf2mesh_b200 import _lib; print(repr(_lib.last_error()))"], cwd=ROOT,
                       capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "''", (r.stdout, r.stderr[-500:])


def test_bindings_cover_the_headers():
    from nerf2mesh_b200 import _lib, mesh, parallel, raster, sampler, stage0, stage1  # noqa: F401  (register the fused / data-parallel signatures)
    bound = set(_lib.SIGNATURES) | {"n2m_last_error", "n2m_version", "n2m_launch_count", "n2m_s0_wpack_bytes",
                                   "n2m_s0_mlp_param_count", "n2m_s0_init", "n2m_dp_ctx_bytes", "n2m_antialias_topology_slots"}
    assert set(declared_symbols()) <= bound, set(declared_symbols()) - bound


def test_params_struct_matches_header():
    from nerf2mesh_b200.stage0 import S0Params
    hdr = open(os.path.join(ROOT, "include", "n2m_b200_fused.h")).read()
    body = hdr[hdr.index("typedef struct {"):hdr.index("} n2m_s0_params;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"(float|uint32_t)\s+([a-z0-9_A-Z]+);", body)
    assert [n for _, n in fields] == [n for n, _ in S0Params._fields_]
    assert ctypes.sizeof(S0Params) == 4 * len(fields)


def test_morton_spread_equals_reference_form():
    def ref(v):
        v = (v * 0x00010001) & 0xFF0000FF; v = (v * 0x00000101) & 0x0F00F00F
        v = (v * 0x00000011) & 0xC30C30C3; v = (v * 0x00000005) & 0x49249249
        return v & 0xFFFFFFFF

    def ours(v):
        v &= 0x7FF
        v = (v | (v << 16)) & 0x070000FF; v = (v | (v << 8)) & 0x0700F00F
        v = (v | (v << 4)) & 0x430C30C3; v = (v | (v << 2)) & 0x49249249
        return v & 0xFFFFFFFF
    assert all(ref(v) == ours(v) for v in range(2048))
    from oracle import raymarching_oracle as R
    c = np.random.default_rng(0).integers(0, 128, (1000, 3))
    m = R.morton3D(c)
    assert np.array_equal(R.morton3D_invert(m), c)
    from nerf2mesh_b200.synthetic import _morton_np
    assert np.array_equal(_morton_np(c), m.astype(np.int64))


def test_level_offsets_match_oracle_and_survey():
    from nerf2mesh_b200.gridencoder.grid import GridEncoder, level_offsets
    from oracle import grid_oracle
    for bound, total in ((1, 6119864), (16, 6837544)):          # SURVEY.md appendix C
        pls = float(np.exp2(np.log2(2048 * bound / 16) / 15))
        a = level_offsets(3, 16, pls, 16, 19, False)
        b = grid_oracle.level_offsets(3, 16, pls, 16, 19, False)
        assert np.array_equal(a, b) and int(a[-1]) == total
    enc = GridEncoder(level_dim=2, desired_resolution=2048)
    assert enc.embeddings.shape == (6119864, 2) and enc.output_dim == 32
    assert enc.embeddings.abs().max() <= 1e-4
    assert "GridEncoder" in repr(enc)


def test_packbits_oracle_and_synthetic_agree():
    from nerf2mesh_b200 import synthetic as S
    from oracle import raymarching_oracle as R
    g = torch.rand(2, 4096)
    assert np.array_equal(S.packbits_host(g, 0.3).numpy(), R.packbits(g.numpy(), 0.3))
    grid, bits, _ = S.occupancy_regime("converged", H=32)
    assert bits.numel() == 32 ** 3 // 8 and 0.02 < grid.mean() < 0.5


def test_stage0_config_mirrors_renderer():
    from nerf2mesh_b200.stage0 import Stage0Config
    c = Stage0Config(bound=16.0)
    assert c.cascade == 5 and abs(c.per_level_scale - 1.662476) < 1e-5            # SURVEY.md appendix C
    c = Stage0Config(bound=4.0, contract=True)
    assert c.bound == 2.0 and c.cascade == 2 and c.real_bound == 4.0              # renderer.py:74-82
    assert Stage0Config(num_rays=100, max_samples=1000).max_samples == 1024


def test_drop_in_module_names():
    import nerf2mesh_b200
    rm, ge, sh = nerf2mesh_b200.install()
    import gridencoder
    import raymarching
    import shencoder
    for n in ("near_far_from_aabb", "sph_from_ray", "morton3D", "morton3D_invert", "packbits", "flatten_rays",
              "march_rays_train", "composite_rays_train", "march_rays", "composite_rays"):
        assert callable(getattr(raymarching, n))
    assert gridencoder.GridEncoder is ge.GridEncoder and shencoder.SHEncoder is sh.SHEncoder


def test_peer_adam_slices_cover_rows_and_stay_aligned():
    """PeerAdam row slices: disjoint cover of the table, slice length a multiple of 4 so that the float2 colour
    moments stored behind the density moments are 8-byte aligned (6119864 rows / 8 ranks = 764983 is odd)."""
    from nerf2mesh_b200.parallel import slice_rows
    from nerf2mesh_b200.gridencoder.grid import level_offsets
    rows = int(level_offsets(3, 16, float(np.exp2(np.log2(2048 / 16) / 15)), 16, 19, False)[-1])
    for R in (rows, 1, 7, 1000003):
        for W in range(1, 9):
            per = slice_rows(R, W)
            assert per % 4 == 0 and per * W >= R
            lo = [min(R, r * per) for r in range(W)]
            hi = [min(R, (r + 1) * per) for r in range(W)]
            assert lo[0] == 0 and hi[-1] == R and all(hi[r] == lo[r + 1] for r in range(W - 1))


def test_step_orchestration_call_sequence(monkeypatch):
    """Stage0Trainer's per-step orchestration (ray-range parts, TV fork, split optimizer, fused backward) with the CUDA layer mocked
    out: the sequence of C-ABI calls on every path, no GPU needed.  Guards the host logic that the GPU tests only exercise on a B200."""
    import types
    import nerf2mesh_b200.stage0 as S0

    calls = []
    monkeypatch.setattr(S0, "call", lambda name, *a: calls.append((name, a)))
    monkeypatch.setattr(S0, "ptr", lambda t: 0)
    monkeypatch.setattr(S0, "stream", lambda: 0)

    class FakeStream:
        def wait_stream(self, o): pass
        def wait_event(self, e): pass
        def synchronize(self): pass

    class FakeEvent:
        def record(self, s=None): pass

    class Ctx:
        def __init__(self, s): pass
        def __enter__(self): return self
        def __exit__(self, *a): return False

    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: FakeStream())
    monkeypatch.setattr(torch.cuda, "Stream", lambda *a, **k: FakeStream())
    monkeypatch.setattr(torch.cuda, "Event", lambda *a, **k: FakeEvent())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: Ctx(s))

    class T:
        def zero_(self): return self
        def __getitem__(self, k): return self
        def data_ptr(self): return 0

    tr = object.__new__(S0.Stage0Trainer)
    tr.cfg = types.SimpleNamespace(lambda_tv=1e-8, eps=1e-15, num_levels=16)
    slot = types.SimpleNamespace(**{k: T() for k in ("rays_o", "rays_d", "gt", "bg", "noises", "rays", "counters", "tbuf", "recs", "cam_nf")}, has_alpha=True)
    tr.slots, tr.cur = [slot, slot], 0
    for k in ("table", "offsets", "enc_tiles", "opt_state", "wpack", "out", "dout", "image", "weights_sum", "depth", "denc_tiles",
              "color_master", "m_table", "v_table", "mlp", "m_mlp", "v_mlp", "loss_acc"):
        setattr(tr, k, T())
    tr.gtables, tr.g_mlps, tr.defer_zero, tr._zero_stream = [T(), T()], [T()], False, None
    tr.params = S0.S0Params(); tr.Mcap, tr.N, tr.rows, tr.parity, tr.device = 128, 4, 160, 0, "cpu"
    tr._tv_overlap, tr._tv_stream, tr._part_streams = True, None, []
    tr._adam_stream = None
    tr.fused_bwd, tr.fused_fwd, tr.tv_fallback_points, tr._graphs = False, False, 1000, {}

    tv = ["n2m_s0_tv", "n2m_s0_tv_random"]
    chain = ["n2m_s0_encode_fwd_part", "n2m_s0_mlp_fwd_part", "n2m_s0_composite_loss_part", "n2m_s0_mlp_bwd_part", "n2m_s0_encode_bwd_part"]
    fchain = chain[:3] + ["n2m_s0_bwd_fused_part"]
    adam = ["n2m_s0_adam_head", "n2m_s0_adam_mlp", "n2m_s0_adam_tables", "n2m_s0_adam_post"]

    def names():
        return [n for n, _ in calls]

    tr.nparts = 1
    tr._compute_then_adam()
    assert names() == [chain[0]] + tv + chain[1:] + adam
    for P_ in (2, 4):
        calls.clear(); tr.nparts = P_
        tr._compute_then_adam()
        assert names() == tv + chain * P_ + adam
        parts = [a[-3:-1] for n, a in calls if n == "n2m_s0_mlp_bwd_part"]
        assert parts == [(k, P_) for k in range(P_)]
    # MLP backward + scatter as ONE launch (csrc/fused.cu)
    calls.clear(); tr.fused_bwd, tr.nparts = True, 1
    tr._compute_then_adam()
    assert names() == [chain[0]] + tv + fchain[1:] + adam
    calls.clear(); tr.nparts = 2
    tr._compute_then_adam()
    assert names() == tv + fchain * 2 + adam
    # gather + MLP forward as one launch (whole batch only)
    calls.clear(); tr.fused_fwd, tr.nparts = True, 1
    tr._compute_then_adam()
    assert names() == tv + ["n2m_s0_fwd_fused", chain[2], "n2m_s0_bwd_fused_part"] + adam
    tr.nparts = 2
    import pytest
    with pytest.raises(RuntimeError):
        tr._compute()
    tr.fused_fwd = False
    # TV inside the scatter kernel (tv mode 0): no TV launch, the fallback probe follows the scatter; not available with the fused backward
    calls.clear(); tr.fused_bwd, tr.nparts = False, 1
    tr.tv_overlap = False
    assert names() == ["n2m_s0_set_tv_mode"]
    calls.clear()
    tr._compute_then_adam()
    assert names() == chain + ["n2m_s0_tv_random"] + adam
    tr.fused_bwd = True
    import pytest
    with pytest.raises(RuntimeError):
        tr._compute()
    # deferred zeroing of the gradient table: same launches, the optimizer variant that leaves the rows alone
    calls.clear(); tr.defer_zero, tr.fused_bwd = True, False
    tr._compute_then_adam()
    assert names() == chain + ["n2m_s0_tv_random"] + adam[:2] + ["n2m_s0_adam_tables_keep", adam[3]]
    tr.defer_zero = False
    # lambda_tv == 0: no TV work at all
    calls.clear(); tr.fused_bwd = False; tr.cfg.lambda_tv = 0.0
    tr._compute_then_adam()
    assert names() == chain + adam


def test_step_prefetch_ordering(monkeypatch):
    """step(next_batch=...): with prefetch_at == "optimizer" the step is launched as compute | optimizer with an event between them and the
    side stream marches the next batch only after that event (and after the slot's previous reader); with "start" the step is one launch and
    the march waits for the start mark only.  CUDA layer mocked: streams / events record what was enqueued where."""
    import types
    import nerf2mesh_b200.stage0 as S0

    log = []
    cur = {"s": "main"}

    class FakeStream:
        def __init__(self, name): self.name = name
        def wait_stream(self, o): log.append((self.name, "wait_stream", o.name))
        def wait_event(self, e): log.append((self.name, "wait_event", e.tag))
        def synchronize(self): pass

    class FakeEvent:
        n = 0
        def __init__(self): FakeEvent.n += 1; self.tag = None
        def record(self, s=None):
            self.tag = f"ev{FakeEvent.n}@{(s.name if s is not None else cur['s'])}:{len(log)}"
            log.append((s.name if s is not None else cur["s"], "record", self.tag))

    class Ctx:
        def __init__(self, s): self.s = s
        def __enter__(self): self.prev = cur["s"]; cur["s"] = self.s.name
        def __exit__(self, *a): cur["s"] = self.prev; return False

    streams = {"main": FakeStream("main")}
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: streams.setdefault(cur["s"], FakeStream(cur["s"])))
    made = []
    def mk(*a, **k):
        s = FakeStream(f"side{len(made)}"); s.priority = k.get("priority", 0); made.append(s); streams[s.name] = s; return s
    monkeypatch.setattr(torch.cuda, "Stream", mk)
    monkeypatch.setattr(torch.cuda, "Event", lambda *a, **k: FakeEvent())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: Ctx(s))

    def trainer(mode):
        tr = object.__new__(S0.Stage0Trainer)
        tr.prefetch_at, tr.defer_zero, tr.parity, tr.cur, tr.global_step, tr.device = mode, True, 0, 0, 0, "cpu"
        tr._prefetched, tr._side, tr._ev_done, tr._ev_march = None, None, [None, None], [None, None]
        tr.params = S0.S0Params(); tr.params.shading_full = 1; tr.params.gt_has_alpha = 1
        slot = types.SimpleNamespace(has_alpha=True, load=lambda *a: log.append((cur["s"], "load", None)))
        tr.slots = [slot, slot]
        tr._run = lambda name, fn, g: log.append((cur["s"], "run", name))
        return tr

    batch = (None,) * 4
    # ---- optimizer mode, two consecutive steps ----
    tr = trainer("optimizer")
    tr.step(*batch, next_batch=batch)
    runs = [(s, n) for s, k, n in log if k == "run"]
    assert runs == [("main", "march"), ("main", "compute_sg"), ("main", "adam_sg"), ("side0", "march")]
    assert made[0].priority == -1
    i_mid = next(i for i, e in enumerate(log) if e[1] == "record" and i > log.index(("main", "run", "compute_sg")))
    assert i_mid < log.index(("main", "run", "adam_sg"))                       # the mark sits between the two launches
    mid_tag = log[i_mid][2]
    i_load = log.index(("side0", "load", None))
    i_wait_mid = log.index(("side0", "wait_event", mid_tag))
    assert i_load < i_wait_mid < log.index(("side0", "run", "march"))          # staged at once, marched after the mark
    assert tr._prefetched == 1 and tr.parity == 1
    log.clear()
    tr.step(*batch, next_batch=batch)                                          # consumes the prefetched slot: no march on main
    runs = [(s, n) for s, k, n in log if k == "run"]
    assert runs == [("main", "compute_sg"), ("main", "adam_sg"), ("side0", "march")]
    assert log[0][:2] == ("main", "wait_event")                                # main waits for the prefetched march first
    assert sum(1 for e in log if e[0] == "side0" and e[1] == "wait_event") == 3   # previous reader of the slot, start mark, mid mark
    # ---- start mode: one launch, normal-priority stream, no mid mark ----
    log.clear(); made.clear()
    tr = trainer("start")
    tr.step(*batch, next_batch=batch)
    runs = [(s, n) for s, k, n in log if k == "run"]
    assert runs == [("main", "march"), ("main", "compute+adam"), ("side0", "march")]
    assert made[0].priority == 0
    assert sum(1 for e in log if e[0] == "side0" and e[1] == "wait_event") == 1
    # ---- no prefetch: one launch whatever the mode ----
    log.clear()
    tr = trainer("optimizer")
    tr.step(*batch)
    assert [(s, n) for s, k, n in log if k == "run"] == [("main", "march"), ("main", "compute+adam")]


def test_stage1_step_call_sequences(monkeypatch):
    """Stage1Trainer._step_body with the CUDA layer mocked: plain, antialiased, and antialiased with the vertex-offset group (the check
    before the optimizer head, the group's update between the table sweep and the GradScaler update)"""
    import types
    import nerf2mesh_b200.stage0 as S0
    import nerf2mesh_b200.stage1 as S1
    import nerf2mesh_b200.raster as RA

    calls = []
    rec = lambda name, *a: calls.append(name)
    for mod in (S0, S1, RA):
        monkeypatch.setattr(mod, "call", rec)
    for mod in (S0, S1, RA):
        monkeypatch.setattr(mod, "stream", lambda: 0)

    def fake_rasterize(glctx, pos, tri, resolution, **kw):          # the wrapper itself refuses host tensors: there is no CPU path
        calls.append("n2m_rasterize")
        return torch.zeros(1, resolution[0], resolution[1], 4), None
    monkeypatch.setattr(RA, "rasterize", fake_rasterize)

    class FakeStream:
        def wait_stream(self, o): pass
    class Ctx:
        def __init__(self, s): pass
        def __enter__(self): return self
        def __exit__(self, *a): return False
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: FakeStream())
    monkeypatch.setattr(torch.cuda, "Stream", lambda *a, **k: FakeStream())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: Ctx(s))

    t0 = object.__new__(S0.Stage0Trainer)
    t0.device = "cpu"
    t0.cfg = types.SimpleNamespace(eps=1e-15)
    for k in ("table", "offsets", "opt_state", "wpack", "color_master", "m_table", "v_table", "mlp", "m_mlp", "v_mlp"):
        setattr(t0, k, torch.zeros(8))
    t0.gtables, t0.g_mlps, t0.parity, t0.rows, t0._adam_stream, t0.fused_bwd, t0.global_step = [torch.zeros(8)] * 2, [torch.zeros(8)], 0, 8, None, True, 0
    t0.params = S0.S0Params()

    def make(**kw):
        monkeypatch.setattr(RA, "TopologyHash", lambda tri: types.SimpleNamespace(keys=torch.zeros(4, dtype=torch.int64), opp=torch.zeros(4, 2, dtype=torch.int32), slots=4, tri=tri))
        return S1.Stage1Trainer(t0, torch.rand(5, 3), torch.tensor([[0, 1, 2], [2, 3, 4]]), 4, 4, ssaa=2, **kw)

    mvp, rd, gt, bg = torch.eye(4), torch.rand(16, 3), torch.rand(16, 4), torch.rand(16, 3)
    fwd = ["n2m_rasterize", "n2m_s1_points", "n2m_s0_encode_points", "n2m_s0_mlp_fwd"]
    adam = ["n2m_s0_adam_head", "n2m_s0_adam_mlp", "n2m_s0_adam_tables", "n2m_s0_adam_post"]
    s1 = make()
    s1.step(mvp, rd, gt, bg)
    assert calls == fwd + ["n2m_s1_loss", "n2m_s0_bwd_fused_part"] + adam and t0.global_step == 1
    calls.clear()
    s1 = make(antialias=True)
    s1.step(mvp, rd, gt, bg)
    aa_f, aa_b = ["n2m_s1_rgba", "n2m_antialias_forward"], ["n2m_s1_loss_aa", "n2m_antialias_backward", "n2m_s1_dout"]
    assert calls == fwd + aa_f + aa_b + ["n2m_s0_bwd_fused_part"] + adam
    calls.clear()
    s1 = make(antialias=True, lr_vert=1e-4)
    s1.step(mvp, rd, gt, bg)
    assert calls == fwd + aa_f + aa_b + ["n2m_s0_bwd_fused_part", "n2m_s1_vert_check"] + adam[:3] + ["n2m_s1_vert_step", adam[3]]
    assert s1.vert_state[1].item() == pytest_approx(1e-4)
    # the image loss reaches the vertices through antialias only
    try:
        make(lr_vert=1e-4)
        assert False
    except ValueError:
        pass
    # graph mode insists on a device-resident mvp (the graph is keyed by its address)
    s1._warm = True
    try:
        s1.step(mvp, rd, gt, bg, use_graph=True)
        assert False
    except RuntimeError as e:
        assert "use_graph" in str(e)


def pytest_approx(x):
    import pytest
    return pytest.approx(x, rel=1e-6)


def test_render_chunking_and_round_continuation(monkeypatch):
    """Stage0Trainer.render (device-side alive-ray rounds) with the CUDA layer mocked: one begin / rounds / finish per chunk, further rounds
    while the control block reports rays alive, row and round diagnostics summed over the chunks"""
    import types
    import nerf2mesh_b200.stage0 as S0

    log = []
    alive_script = []          # values ctl[10] takes after successive `rounds` calls

    tr = object.__new__(S0.Stage0Trainer)
    tr.device = "cpu"
    tr.params = S0.S0Params()
    tr.aabb = torch.zeros(6); tr.density_bitfield = torch.zeros(8, dtype=torch.uint8)
    tr.table = tr.offsets = tr.wpack = torch.zeros(8)
    tr._prefetched = None
    tr.drop_prefetch = lambda: None

    def fake_call(name, *a):
        log.append((name, a))
        if name == "n2m_s0_render_begin":
            tr._render_buf["ctl"].zero_()
        if name == "n2m_s0_render_rounds":
            ctl = tr._render_buf["ctl"]
            ctl[10] = alive_script.pop(0) if alive_script else 0
            ctl[12] += int(a[6]); ctl[13] += 100
    monkeypatch.setattr(S0, "call", fake_call)
    monkeypatch.setattr(S0, "stream", lambda: 0)

    ro, rd = torch.rand(100, 3), torch.rand(100, 3)
    img, ws, dep = tr.render(ro, rd, bg_color=1.0, chunk=40)                      # 3 ragged chunks: 40, 40, 20
    names = [n for n, _ in log]
    assert names == ["n2m_s0_render_begin", "n2m_s0_render_rounds", "n2m_s0_render_finish"] * 3
    assert [a[5] for n, a in log if n == "n2m_s0_render_begin"] == [40, 40, 20]
    assert img.shape == (100, 3) and ws.shape == (100,) and dep.shape == (100,)
    assert tr.render_rounds == len(tr.RENDER_SCHEDULE) and tr.render_rows == 300
    rb = tr._render_buf
    assert rb["cap"] % 128 == 0 and rb["cap"] >= 40 * 16
    # a schedule that leaves rays alive: the read-back triggers further rounds before the background mix
    log.clear(); alive_script[:] = [7, 3, 0]
    tr.render(ro[:30], rd[:30], bg_color=torch.rand(30, 3), chunk=40)
    assert [n for n, _ in log] == ["n2m_s0_render_begin"] + ["n2m_s0_render_rounds"] * 3 + ["n2m_s0_render_finish"]
    assert tr.render_rounds == len(tr.RENDER_SCHEDULE) + 2 + 2 and tr.render_rows == 300
    fin = log[-1][1]
    assert fin[2] is not None and fin[4] == 30                                    # per-ray background pointer, ray count
    # shading flag reaches the kernels' parameter block
    tr.render(ro[:10], rd[:10], shading="diffuse")
    assert rb["params"].shading_full == 0
