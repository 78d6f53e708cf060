#!/usr/bin/env python
"""Benchmark of the SelfRecon hot path on B200 (BASELINE.json metric, config[1]).

One "step" = one pass of the hot path over one synthetic 512x512 frame:
  ray part : OptimizeSurfacePs (training thresholds: dthr 5e-5, 0.5 px angle, times=10) on every
             silhouette ray of the frame, then shading (grad f, cardinal rays, rendcond, RenderNet);
  MC part  : discretizeSDF = coarse-to-fine 257^3 SDF grid (Seg3dLossless, ladder 33..257) + MC.
`value` = rays/s over the ray part (whole job, all GPUs), `mc_voxels_per_sec` = 257^3 / MC part.
Inputs are resident in HBM for `value`; `e2e` repeats the step through the reference-facing
drop-in API with pinned host buffers, H2D/D2H inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
Under torchrun (N>1) every rank renders its own frame (weak scaling, no data-path collective).
--dump-outputs writes what the last timed step computed (rank 0) as DIR/<name>.npy: the inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_S, F_D, F_R = 3.933184e6, 1.746944e6, 1.871872e6  # FLOP per point (SURVEY.md section 8)
RATIO = {"sdfRatio": 1.0, "deformerRatio": 1.0, "renderRatio": 1.0}
GRID_N = 257


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor=d["bf16_tflops"], tensor_sustained=d.get("bf16_tflops_sustained"),
                    src="measured")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.rows = []
        self.stop = False
        self.index = index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop:
            try:
                o = subprocess.check_output(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                             "--format=csv,noheader,nounits"], timeout=5).decode()
                self.rows.append([x.strip() for x in o.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=3)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons}


# --------------------------------------------------------------------------------------------------
def build_scene(dev, frame_seed, H=512, W=512):
    from selfreconcode_b200 import synth
    sdf = synth.make_sdf().to(dev)
    tr = synth.make_translator().to(dev)
    sk = synth.make_skinner().to(dev)
    rn = synth.make_render().to(dev)
    comp = synth.CompositeDeformer([tr, sk]).to(dev)
    poses, trans, dcond = [t.to(dev) for t in synth.make_frame_params(100 + frame_seed, 1)]
    conds = [dcond, [poses, trans]]
    cam = synth.camera(H, W)

    def sdf_fn(p):
        return sdf.forward_fused(p.to(dev), RATIO, False, False)[0].view(-1)

    def def_fn(p, b):
        return comp.forward_fused(p.to(dev), conds, b.to(dev), RATIO)[0]

    rays = synth.make_rays(cam, 1, sdf_fn, def_fn, seed=7 + frame_seed)
    return dict(sdf=sdf, comp=comp, rn=rn, conds=conds, cam=cam, rays=rays,
                ang=synth.ang_threshold(cam, 0.5), synth=synth)


def make_engine(sc, dev):
    from selfreconcode_b200 import enable_dropin
    enable_dropin()
    from MCAcc import Seg3dLossless
    sdf = sc["sdf"]

    def query_func(points):
        # discretizeSDF's closure (network.py:293-295) only needs the SDF value: the sdf-only last
        # layer skips the 256-d feature the reference computes and throws away here
        return sdf.forward_fused(points.reshape(-1, 3), RATIO, False, False)[0].reshape(1, 1, -1)

    eng = Seg3dLossless(query_func=query_func, b_min=[-1.0, -1.0, -1.0], b_max=[1.0, 1.0, 1.0],
                        resolutions=sc["synth"].MC_LADDER_257, align_corners=False, balance_value=0.0,
                        use_cuda_impl=True).to(dev)
    return eng


def ray_part(sc, rays, init, bi, stats=None):
    """trace + shade through the product ops (device tensors in / out)."""
    from selfreconcode_b200 import ops
    sdf, comp, rn = sc["sdf"], sc["comp"], sc["rn"]
    tr, sk = comp.defs
    sdf_only = sdf.fused_sdf_only()
    sdf_only.set_pe_weights([1.0] * 6)
    dnet = tr.fused(RATIO)
    lbs = sk.lbs_state()
    lbs.set_pose(sc["conds"][1][0], sc["conds"][1][1])
    cam_pos = sc["cam"]["cam_pos"]
    pts, conv, counters = ops.trace_surface_points(sdf_only, dnet, lbs, cam_pos, rays, init, bi, sc["conds"][0],
                                                   5e-5, sc["ang"], 3.05, 1.0, 10, return_counters=True)
    full = sdf.fused()
    full.set_pe_weights([1.0] * 6)
    if ops.TC_ENABLED and pts.shape[0] >= ops.TC_MIN_POINTS:
        n, cr, rgb, _, _ = ops.shade_and_render_tc(full, dnet, lbs, rn.fused(RATIO), pts, rays, bi, sc["conds"][0])
    else:
        n, cr, feat, _, _ = ops.shade_geometry(full, dnet, lbs, pts, rays, bi, sc["conds"][0], nfeat=256)
        rgb = ops.render_forward(rn.fused(RATIO), pts, n, cr, feat)
    if stats is not None:
        stats["counters"] = counters
    return pts, conv, rgb


def mc_part(sc, eng):
    import MCGpu
    grid = eng.forward()
    v, f = MCGpu.mc_gpu(grid[0, 0].permute(2, 1, 0).contiguous(), eng.spacing_x, eng.spacing_y, eng.spacing_z,
                        eng.bx, eng.by, eng.bz, 0.0)
    return grid, v, f


DUMP_BUDGET = 60 << 20   # array bytes written by --dump-outputs in all: under 64 MB with the .npy headers


def dump_outputs(path, outs, budget=DUMP_BUDGET):
    """Writes each tensor of `outs` as path/<name>.npy: floating point as float32, integer and bool as float64 (exact
    for indices).  The budget is shared out smallest tensor first; a tensor larger than its share is replaced by a fixed
    sample of its elements (flattened, chosen by a seeded permutation of its size, kept in index order), so the same
    shapes always give the same sample."""
    os.makedirs(path, exist_ok=True)
    dtype = lambda t: torch.float32 if t.is_floating_point() else torch.float64
    order = sorted(outs, key=lambda k: outs[k].numel() * dtype(outs[k]).itemsize)
    for i, name in enumerate(order):
        t = outs[name].detach()
        dt = dtype(t)
        n = budget // (len(order) - i) // dt.itemsize
        budget -= min(n, t.numel()) * dt.itemsize
        if t.numel() > n:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:n].sort()[0]
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.to(dt).cpu().numpy())


def layer_roofline(dev, M, launches=24):
    """Live timing of the dominant kernel: one 512x512 softplus layer of the tracer on M rows
    (tc_layer_pair_kernel), CUDA events on the launching stream, rotating operand buffers so that no
    launch finds its rows in L2 (4 x (in + out) > 126 MB).  Bias and outputs are allocated once: the
    timed region holds nothing but the layer launches."""
    import ctypes as C
    from selfreconcode_b200 import ops, _lib
    from selfreconcode_b200._lib import SR_ACT_SOFTPLUS100
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(3)
    w = torch.randn(512, 512, device=dev, generator=g) / 22.6
    b = torch.zeros(512, device=dev)
    W = ops.tc_pack_weights(w)
    As = [ops.tc_pack_rows(torch.randn(M, 512, device=dev, generator=g)) for _ in range(4)]
    outs = [torch.empty_like(As[0]) for _ in range(4)]
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t: C.c_void_p(t.data_ptr())

    def launch(i):
        rc = lib.sr_tc_linear(vp(As[i & 3]), vp(W), vp(b), M, 512, 512, 512, SR_ACT_SOFTPLUS100, 1, vp(outs[i & 3]),
                              512, 1.0, None, 0, 0, None, 0, 0, 512, None, None, 0, 0, 1.0, None, st)
        assert rc == 0, rc

    for i in range(4):
        launch(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(launches):
        launch(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / launches
    return ms, 2.0 * M * 512 * 512


def ray_part_api(sc, rays, init, bi):
    """Same work through the reference-facing drop-in API (utils.OptimizeSurfacePs, ...)."""
    import utils
    sdf, comp, rn = sc["sdf"], sc["comp"], sc["rn"]
    cam_pos = sc["cam"]["cam_pos"].to(rays.device)
    pts, conv = utils.OptimizeSurfacePs(cam_pos, rays, init, bi, sdf, RATIO, comp, sc["conds"], dthreshold=5e-5,
                                        athreshold=sc["ang"], w1=3.05, w2=1., times=10)
    _, _, rgb = utils.shade_rays(sdf, comp, rn, pts, rays, sc["conds"], bi, RATIO)
    return pts, conv, rgb


# --------------------------------------------------------------------------------------------------
# BASELINE configs[0]: the reference's own CPU-runnable case -- one 128x128 frame, 4-layer / 64-wide SDF, identity
# deformer, 65^3 (64^3 cells) coarse-to-fine grid + MC.  Small enough that the oracle runs the WHOLE case in about a
# second, so the GPU arm and the CPU arm are timed and compared on identical inputs inside the default bench run.
def config0_part(dev, threads):
    from selfreconcode_b200 import synth, ops, enable_dropin
    from oracle import oracle as O
    from oracle import c_api
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    enable_dropin()
    from MCAcc import Seg3dLossless
    import MCGpu
    torch.set_num_threads(threads)
    sdf = synth.make_sdf(seed=40, hidden=64, n_hidden=4, feat=0, skip_in=(), perturb=0.0, bias=0.4)   # r in [0.37, 1.02]
    cam = synth.camera(128, 128)
    sp = helpers.sdf_params(sdf)
    sdf_fn = lambda p: O.sdf_forward(sp, p, 6, 1.0, skip_in=())[0]
    ident = lambda p, b: p
    with torch.no_grad():
        rays = synth.make_rays(cam, 1, lambda p: sdf_fn(p).view(-1), ident, seed=3, jitter=1e-3)
    ang = synth.ang_threshold(cam, 0.5)
    n = rays["rays"].shape[0]
    # ---- CPU arm (oracle = the reference's algorithm on host cores), whole case
    sens = {"eps_f": 5e-6, "eps_a": 2e-4}
    t0 = time.perf_counter()
    po, co, _ = O.optimize_surface_ps(cam["cam_pos"], rays["rays"], rays["init_pts"], rays["batch_inds"], sdf_fn, ident,
                                      5e-5, ang, 3.05, 1.0, 10, sensitivity=sens)
    t_ray_cpu = time.perf_counter() - t0
    t0 = time.perf_counter()
    with torch.no_grad():
        grid_o, calc_o = O.seg3d_forward(lambda q: sdf_fn(q).view(-1), [-1.2] * 3, [1.2] * 3, synth.MC_LADDER_65, 0.0)
    spc, org = O.mc_world_params([-1.2] * 3, [1.2] * 3, (65, 65, 65))
    vo, fo = c_api.marching_cubes(grid_o.permute(2, 1, 0).contiguous().numpy(), helpers.mc_tri_table(), 0.0, spc, org)
    t_mc_cpu = time.perf_counter() - t0
    # ---- GPU arm
    sdf_d = sdf.to(dev)
    net = sdf_d.fused()
    net.set_pe_weights([1.0] * 6)
    r_d, i_d, b_d = rays["rays"].to(dev), rays["init_pts"].to(dev), rays["batch_inds"].to(dev)
    cp = cam["cam_pos"].to(dev)
    eng = Seg3dLossless(query_func=lambda points: sdf_d.forward_fused(points.reshape(-1, 3), 1.0, False, False)[0]
                        .reshape(1, 1, -1), b_min=[-1.2] * 3, b_max=[1.2] * 3, resolutions=synth.MC_LADDER_65,
                        align_corners=False, balance_value=0.0, use_cuda_impl=True).to(dev)

    def gpu_rays():
        return ops.trace_surface_points(net, None, None, cp, r_d, i_d, b_d, None, 5e-5, ang, 3.05, 1.0, 10, mode="reverse")

    def gpu_mc():
        g = eng.forward()
        v, f = MCGpu.mc_gpu(g[0, 0].permute(2, 1, 0).contiguous(), eng.spacing_x, eng.spacing_y, eng.spacing_z, eng.bx,
                            eng.by, eng.bz, 0.0)
        return g, v, f

    for _ in range(3):
        gpu_rays()
        gpu_mc()
    torch.cuda.synchronize()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    tr, tm = [], []
    for _ in range(5):
        a, b, c = ev(), ev(), ev()
        a.record()
        pg, cg = gpu_rays()
        b.record()
        g, vg, fg = gpu_mc()
        c.record()
        torch.cuda.synchronize()
        tr.append(a.elapsed_time(b))
        tm.append(b.elapsed_time(c))
    ok = ~sens["sensitive"].numpy()
    dp = np.abs(pg.cpu().numpy() - po.numpy()).max(1)
    mm = cg.cpu().numpy() != co.numpy()
    gg, gc = g[0, 0].cpu().numpy(), grid_o.numpy()
    sm = (gg > 0) != (gc > 0)
    return {"workload": "config[0]: one 128x128 frame (%d silhouette rays), 4x64 SDF, identity deformer, trace times=10, "
                        "65^3 coarse-to-fine grid + MC" % n,
            "gpu": {"rays_per_sec": n / (float(np.mean(tr)) * 1e-3), "ms_rays": float(np.mean(tr)),
                    "mc_voxels_per_sec": 65 ** 3 / (float(np.mean(tm)) * 1e-3), "ms_mc": float(np.mean(tm)),
                    "engine": "fused fp32 FFMA (templated on width 64 / no skip / identity deformer)"},
            "cpu_reference": {"rays_per_sec": n / t_ray_cpu, "mc_voxels_per_sec": 65 ** 3 / t_mc_cpu, "cores": threads,
                              "kind": "port"},
            "parity": {"rays": int(n), "rays_decision_sensitive": int((~ok).sum()),
                       "conv_mismatch_insensitive": int((mm & ok).sum()), "conv_mismatch_all": int(mm.sum()),
                       "pts_max_abs_err_insensitive": float(dp[ok].max()) if ok.any() else 0.0,
                       "queried_gpu": int(eng.last_num_queried), "queried_oracle": int(calc_o.sum()),
                       "sign_mismatch": int(sm.sum()),
                       "sign_mismatch_outside_fp32_band": int((sm & (np.abs(gc) >= 1e-5)).sum()),
                       "mc_faces_gpu": int(fg.shape[0]), "mc_faces_oracle": int(fo.shape[0]),
                       "mc_mesh_identical": bool(fg.shape[0] == fo.shape[0] and np.array_equal(fg.cpu().numpy(), fo) and
                                                 np.abs(vg.cpu().numpy() - vo).max() < 1e-5)}}


# --------------------------------------------------------------------------------------------------
# Training step (BASELINE configs[2] / [3]): batch of 4 frames per GPU, SMPL LBS + FastMinv on, eikonal + colour +
# normal + def_regu + offset losses (config.conf loss_coarse), implicit differentiation, ONE NCCL all-reduce of all
# gradients, Adam step -- train.py:160-171 with the per-point work on the tensor-core training engine.
TRAIN_FRAMES = 4
TRAIN_RAYS = 2048 * TRAIN_FRAMES      # config.conf sample_pix_num per frame


def build_train(sc, dev, rank, world):
    from selfreconcode_b200 import synth, parallel
    from model.optim import OptimNetwork
    from model.CameraMine import RectifiedPerspectiveCameras
    import types
    H = W = 512
    data = synth.SyntheticDataset(TRAIN_FRAMES, H, W, seed=50 + rank).to(dev)
    fids = torch.arange(TRAIN_FRAMES, device=dev)
    poses, trans, dcond, _ = data.get_grad_parameters(fids, dev)
    sdf, comp, rn = sc["sdf"], sc["comp"], sc["rn"]
    with torch.no_grad():
        rays = synth.make_rays(sc["cam"], TRAIN_FRAMES,
                               lambda p: sdf.forward_fused(p.to(dev), RATIO, False, False)[0].view(-1),
                               lambda p, b: comp.forward_fused(p.to(dev), [dcond, [poses, trans]], b.to(dev), RATIO)[0],
                               seed=31 + rank, jitter=3e-4)
    g = torch.Generator().manual_seed(77 + rank)
    sel = torch.randperm(rays["rays"].shape[0], generator=g)[:int(TRAIN_RAYS * 1.3)].sort()[0]
    f, pp, R, T, _, _ = data.get_camera_parameters(TRAIN_FRAMES, dev)
    cams = RectifiedPerspectiveCameras(f.detach(), pp.detach(), R, T.detach(), image_size=[(W, H)])
    # The seed of the real pipeline (rasterised deformed template, network.py:485-493) puts D(start) on the PIXEL's own
    # ray.  Setup-only stand-in: Gauss-Newton on {f(p) = 0, (D(p) - c) x v_pixel = 0} from the synthetic surface point,
    # on top of the fused value / gradient / Jacobian kernels; rays that settle are kept.
    bi_a, ri_a, ci_a = rays["batch_inds"][sel].to(dev), rays["rows"][sel].to(dev), rays["cols"][sel].to(dev)
    pix = torch.stack([ci_a, ri_a, torch.ones_like(ci_a)], dim=1).float()
    dc = [dcond.detach(), [poses.detach(), trans.detach()]]
    with torch.no_grad():
        v = cams.view_rays(pix)
        c = cams.cam_pos().view(1, 3)
        p = rays["pstar"][sel].to(dev).clone()
        vx = torch.zeros(p.shape[0], 3, 3, device=dev)
        vx[:, 0, 1], vx[:, 0, 2], vx[:, 1, 0] = -v[:, 2], v[:, 1], v[:, 2]
        vx[:, 1, 2], vx[:, 2, 0], vx[:, 2, 1] = -v[:, 0], -v[:, 1], v[:, 0]
        for _ in range(12):
            fv, gf, _ = sdf.forward_fused(p, RATIO, want_grad=True, want_feat=False)
            d, J, _ = comp.forward_fused(p, dc, bi_a, RATIO, want_jac=True)
            res = torch.cat([fv.view(-1, 1), torch.linalg.cross(v, d - c, dim=1)], dim=1)
            B = torch.cat([gf.view(-1, 1, 3), vx @ J], dim=1)
            step = torch.linalg.solve(B.transpose(1, 2) @ B + 1e-9 * torch.eye(3, device=dev), B.transpose(1, 2) @ res.unsqueeze(-1))
            p = p - step.squeeze(-1).clamp(-0.05, 0.05)
        fv = sdf.forward_fused(p, RATIO, False, False)[0].view(-1)
        d = comp.forward_fused(p, dc, bi_a, RATIO)[0]
        u = d - c
        ang = torch.asin(torch.linalg.cross(u, v, dim=1).norm(dim=1) / u.norm(dim=1)) * 180.0 / np.pi
        ok = (fv.abs() < 2e-5) & (ang < 0.3 * synth.ang_threshold(sc["cam"], 0.5))
    keep = torch.nonzero(ok).view(-1)[:TRAIN_RAYS]
    assert keep.numel() > 0.6 * TRAIN_RAYS, "seed solve settled on %d of %d rays" % (keep.numel(), TRAIN_RAYS)
    # half of the seeds sit on the solution (converge at the first test: they carry the colour / normal / implicit-
    # differentiation load), half are jittered by 2e-4 and exercise the tracer's iterations
    jit = 2e-4 * torch.randn(keep.numel(), 3, generator=g).to(dev)
    jit[::2] = 0.0
    seeds = dict(bi=bi_a[keep], ri=ri_a[keep], ci=ci_a[keep], init=p[keep] + jit)
    holder = types.SimpleNamespace(rasterizer=types.SimpleNamespace(cameras=cams))
    conf = synth.reference_config().get_config("loss_coarse")
    net = OptimNetwork(sdf, comp, None, holder, rn, conf=conf)
    net.dataset = data
    params = [q for q in list(sdf.parameters()) + list(comp.parameters()) + list(rn.parameters()) +
              list(data.parameters()) if q.requires_grad]
    # lr = 0: Adam runs in full (and bumps every parameter's version, so the engines re-fold / re-pack each step as in
    # real training) but the synthetic seeds stay on the surface they were solved for
    opt = torch.optim.Adam(params, lr=0.0)
    ar = parallel.GradAllReduce(params, timed=True)
    img = (torch.rand(TRAIN_FRAMES, H, W, 3, generator=g) * 2 - 1).to(dev)
    nrm = torch.nn.functional.normalize(torch.randn(TRAIN_FRAMES, H, W, 3, generator=g), dim=-1).to(dev)
    extra = rays["pstar"][torch.randperm(rays["pstar"].shape[0], generator=g)[:4096]].to(dev)
    return dict(net=net, opt=opt, ar=ar, fids=fids, datas={"img": img, "normal": nrm}, extra=extra, params=params,
                n_rays=int(keep.numel()), **seeds)


def train_step(tr, events=None):
    net, opt = tr["net"], tr["opt"]
    mark = (lambda i: events[i].record()) if events is not None else (lambda i: None)
    mark(0)
    opt.zero_grad(set_to_none=True)
    loss = net.forward_rays(tr["datas"], tr["bi"], tr["ri"], tr["ci"], tr["init"].clone(), RATIO, tr["fids"],
                            extra_points=tr["extra"])
    mark(1)
    loss.backward()
    mark(2)
    net.propagateTmpPsGrad(tr["fids"], RATIO)
    mark(3)
    nbytes = tr["ar"]()
    mark(4)
    opt.step()
    mark(5)
    return loss, nbytes


def train_part(sc, dev, rank, world, dist, steps, warmup):
    """-> dict for the JSON line (`train`): training rays/s of the whole job with the gradient all-reduce inside the
    timed region, per-phase device times, the collective's own time / bytes, and the tensor roofline of the dominant
    training kernel (weight-gradient GEMM of the def_regu block)."""
    from selfreconcode_b200 import ops
    tr = build_train(sc, dev, rank, world)
    saved = [q.detach().clone() for q in tr["params"]]      # the scene is shared with the rendering / parity legs
    for _ in range(max(warmup, 3)):
        train_step(tr)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    phases, ar_ms, total = [], [], []
    ops.LAUNCHES = 0
    for _ in range(steps):
        e = [ev() for _ in range(6)]
        loss, nbytes = train_step(tr, e)
        torch.cuda.synchronize()
        phases.append([e[i].elapsed_time(e[i + 1]) for i in range(5)])
        total.append(e[0].elapsed_time(e[5]))
        ar_ms.append(tr["ar"].collective_ms())
    info = dict(tr["net"].info)
    t = torch.tensor([float(np.mean(total))], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    ph = np.mean(np.array(phases), axis=0)
    with torch.no_grad():
        for q, v in zip(tr["params"], saved):
            q.copy_(v)
    nr = torch.tensor([float(tr["n_rays"])], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(nr)
    return {"metric": "training_rays_per_sec", "value": nr.item() / (ms * 1e-3), "unit": "rays/s",
            "ms_per_step": ms, "frames_per_gpu": TRAIN_FRAMES, "rays_per_gpu": tr["n_rays"],
            "rays_converged": int(info["rayInfo"][1]),
            "ms_forward_incl_trace": float(ph[0]), "ms_backward": float(ph[1]), "ms_propagate": float(ph[2]),
            "ms_allreduce_incl_flatten": float(ph[3]), "ms_optimizer": float(ph[4]),
            "allreduce": {"collective_ms": float(np.mean(ar_ms)), "bytes": int(nbytes), "op": "one NCCL all-reduce "
                          "(sum, then /world) of every gradient: MLPs + per-frame poses / trans / latent codes"},
            "loss": float(loss.item()), "losses": {k: float(v) for k, v in info.items() if k.endswith("_loss")},
            "workload": "config[2]/[3] shape: %d frames of 512x512 per GPU, %d sampled silhouette rays, LBS + FastMinv, "
                        "eikonal + colour + normal (weighted) + def_regu (device singular values) + offset losses, "
                        "propagateTmpPsGrad, Adam; frames sharded across ranks (weak scaling)" % (TRAIN_FRAMES, TRAIN_RAYS)}


def wgrad_roofline(dev, M=98304 * 4):
    """Dominant training kernel timed alone: the 512x512 weight-gradient GEMM over the def_regu block's rows
    (4 frames x 2 x 12 288 points x 4 rows), CUDA events on the launching stream, 3 MMAs per product."""
    import ctypes as C
    from selfreconcode_b200 import ops, _lib
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(5)
    D = ops.tc_pack_rows(torch.randn(M, 512, device=dev, generator=g))
    X = ops.tc_pack_rows(torch.randn(M, 512, device=dev, generator=g))
    part = torch.empty((lib.sr_tc_wgrad_partial_bytes(M, 512, 512, None),), dtype=torch.uint8, device=dev)
    dW = torch.empty(512, 512, device=dev)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t: C.c_void_p(t.data_ptr())
    for _ in range(3):
        lib.sr_tc_wgrad(vp(D), 512, vp(X), 512, M, vp(part), vp(dW), 512, 512, 512, st)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        lib.sr_tc_wgrad(vp(D), 512, vp(X), 512, M, vp(part), vp(dW), 512, 512, 512, st)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    return ms, 2.0 * M * 512 * 512


# --------------------------------------------------------------------------------------------------
def cpu_reference_sample(n_rays, threads, seed=0, with_mc=True, rays=None, keep=False):
    """The oracle (CPU port of the reference path) on a bounded sample of the same workload.
    `rays` = the GPU arm's own ray set (CPU tensors): same inputs, so `keep=True` results can be compared
    element by element with the GPU's (parity_report)."""
    from selfreconcode_b200 import synth
    from oracle import oracle as O
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    torch.set_num_threads(threads)
    sdf = synth.make_sdf()
    tr = synth.make_translator()
    sk = synth.make_skinner()
    rn = synth.make_render()
    poses, trans, dcond = synth.make_frame_params(100 + seed, 1)
    sp = helpers.sdf_params(sdf)
    tp = helpers.plain_params(tr)
    rp = helpers.wn_params(rn)
    A, _ = O.bone_transforms(poses, sk.Js, synth.SMPL_PARENTS, sk.init_pose)
    lbs = dict(ws=sk.ws, bmin=sk.b_min.view(3), bmax=sk.b_max.view(3), A=A, trans=trans)
    sdf_fn = lambda p: O.sdf_forward(sp, p, 6, 1.0)[0]
    def_fn = lambda p, b: O.composite_deform(tp, 6, 1.0, dcond, lbs, p, b)[0]
    cam = synth.camera(512, 512)
    if rays is None:
        with torch.no_grad():
            rays = synth.make_rays(cam, 1, lambda p: sdf_fn(p).view(-1), def_fn, seed=7 + seed, max_rays=n_rays)
    elif n_rays is not None and n_rays < rays["rays"].shape[0]:
        g = torch.Generator().manual_seed(11)
        sel = torch.randperm(rays["rays"].shape[0], generator=g)[:n_rays].sort()[0]
        rays = {k: v[sel] for k, v in rays.items() if torch.is_tensor(v) and v.shape[0] == rays["rays"].shape[0]}
    bi = rays["batch_inds"]
    ang_thr = synth.ang_threshold(cam, 0.5)
    t0 = time.perf_counter()
    sens = {"eps_f": 4e-5, "eps_a": 1e-3} if keep else None     # the tensor-core engine's error bounds (ops.TC_EPS_*)
    pts, conv, _ = O.optimize_surface_ps(cam["cam_pos"], rays["rays"], rays["init_pts"], bi, sdf_fn, def_fn,
                                         5e-5, ang_thr, 3.05, 1.0, 10, sensitivity=sens)
    s, g, feat = O.sdf_value_and_grad(sp, pts, 6, 1.0)
    nx = g / g.norm(dim=1, keepdim=True)
    cr, ds, J, ok = O.cardinal_rays(lambda p: def_fn(p, bi), pts, rays["rays"])
    with torch.no_grad():
        rgb = O.render_forward(rp, pts, nx, cr, feat, 4, 1.0)
    t_ray = time.perf_counter() - t0
    out = {"rays": int(pts.shape[0]), "ray_seconds": t_ray, "rays_per_sec": pts.shape[0] / t_ray}
    if keep:
        u = ds - cam["cam_pos"].view(1, 3)
        ang = torch.asin(torch.linalg.cross(u, rays["rays"]).norm(dim=1) / u.norm(dim=1)) * 180.0 / np.pi
        out["keep"] = dict(pts=pts, conv=conv, rgb=rgb, f=s, ang=ang, ang_thr=ang_thr, sensitive=sens["sensitive"])
    if with_mc:
        from oracle import c_api
        t0 = time.perf_counter()
        with torch.no_grad():
            grid, calc = O.seg3d_forward(lambda q: sdf_fn(q).view(-1), [-1.0] * 3, [1.0] * 3,
                                         synth.MC_LADDER_257, 0.0)
        spc, org = O.mc_world_params([-1.0] * 3, [1.0] * 3, (257, 257, 257))
        vo, fo = c_api.marching_cubes(grid.permute(2, 1, 0).contiguous().numpy(), helpers.mc_tri_table(), 0.0,
                                      spc, org)
        t_mc = time.perf_counter() - t0
        out.update({"mc_grid": 257, "mc_seconds": t_mc, "mc_voxels_per_sec": 257 ** 3 / t_mc,
                    "mc_queried": int(calc.sum())})
        if keep:
            out["keep"].update(grid=grid, calc=calc, verts=vo, faces=fo)
    return out


def parity_report(gpu, cpu, band=1e-5):
    """GPU arm vs the oracle on the SAME inputs at the benchmark's own sizes (BASELINE config[1]); counts only,
    printed in the JSON line and asserted by tests/test_gpu_round2.py.

    Rays.  OptimizeSurfacePs is a decision-driven iteration (sign(f) in the loss gradient, two threshold tests):
    a ray whose reference trajectory comes within the engine's error bound of a decision may legitimately take
    another branch, after which its points are unrelated.  The oracle marks those rays (`sensitive`, see
    oracle.optimize_surface_ps); the bar applies to all the others: identical convergence mask, points and colours
    elementwise |a-b| <= 1e-4*|b| + 1e-4*mean|b|.  The same figures over ALL rays are reported beside them.
    Grid.  Queried-voxel sets, sign pattern and MC mesh; a sign may only differ where the oracle's own value is inside
    fp32 evaluation noise (|f| < band): two correct fp32 evaluations of an 8x512 MLP differ there."""
    rep = {}
    pg, pc = gpu["pts"].double().cpu().numpy(), cpu["pts"].double().numpy()
    rg, rc = gpu["rgb"].double().cpu().numpy(), cpu["rgb"].double().numpy()
    cg, cc = gpu["conv"].cpu().numpy().astype(bool), cpu["conv"].numpy().astype(bool)
    sens = cpu["sensitive"].numpy().astype(bool)
    ok = ~sens
    tol_p = 1e-4 * np.abs(pc) + 1e-4 * np.abs(pc).mean()
    tol_c = 1e-4 * np.abs(rc) + 1e-4 * np.abs(rc).mean()
    bad_p = (np.abs(pg - pc) > tol_p).any(1)
    bad_c = (np.abs(rg - rc) > tol_c).any(1)
    rep["rays"] = int(pc.shape[0])
    rep["rays_decision_sensitive"] = int(sens.sum())
    rep["converged_gpu"], rep["converged_oracle"] = int(cg.sum()), int(cc.sum())
    rep["conv_mismatch_all"] = int((cg != cc).sum())
    rep["conv_mismatch_insensitive"] = int(((cg != cc) & ok).sum())
    rep["pts_rays_over_tol_all"] = int(bad_p.sum())
    rep["pts_rays_over_tol_insensitive"] = int((bad_p & ok).sum())
    rep["pts_max_abs_err_insensitive"] = float(np.abs(pg - pc)[ok].max()) if ok.any() else 0.0
    both = cg & cc
    rep["pts_max_abs_err_converged_in_both"] = float(np.abs(pg - pc)[both].max()) if both.any() else 0.0
    rep["rgb_rays_over_tol_insensitive"] = int((bad_c & ok).sum())
    rep["rgb_max_abs_err_insensitive"] = float(np.abs(rg - rc)[ok].max()) if ok.any() else 0.0
    if "grid" in cpu and "grid" in gpu:
        gg, gc = gpu["grid"].cpu().numpy(), cpu["grid"].numpy()
        qg, qc = gpu["calc"].cpu().numpy().astype(bool), cpu["calc"].numpy().astype(bool)
        rep["queried_gpu"], rep["queried_oracle"] = int(qg.sum()), int(qc.sum())
        rep["queried_set_mismatch"] = int((qg != qc).sum())
        sm = (gg > 0.0) != (gc > 0.0)
        rep["sign_mismatch"] = int(sm.sum())
        rep["sign_mismatch_outside_fp32_band"] = int((sm & (np.abs(gc) >= band)).sum())
        qb = qg & qc
        rep["queried_value_max_abs_err"] = float(np.abs(gg.astype(np.float64) - gc)[qb].max())
        fg, fc = gpu["faces"].cpu().numpy(), cpu["faces"]
        rep["mc_faces_gpu"], rep["mc_faces_oracle"] = int(fg.shape[0]), int(fc.shape[0])
        rep["mc_verts_gpu"], rep["mc_verts_oracle"] = int(gpu["verts"].shape[0]), int(cpu["verts"].shape[0])
        rep["mc_mesh_identical"] = bool(fg.shape == fc.shape and np.array_equal(fg, fc))
        if "verts_on_oracle_grid" in gpu:     # the product's MC run on the ORACLE's grid: integer parity proper
            v2, f2 = gpu["verts_on_oracle_grid"].cpu().numpy(), gpu["faces_on_oracle_grid"].cpu().numpy()
            rep["mc_on_oracle_grid_faces_identical"] = bool(f2.shape == fc.shape and np.array_equal(f2, fc))
            rep["mc_on_oracle_grid_verts_identical"] = bool(v2.shape == cpu["verts"].shape and
                                                            np.array_equal(v2, cpu["verts"]))
    return rep


def pick_threads():
    """Thread count at which the CPU port is fastest on this host (the matrices are small: beyond a
    few dozen threads torch's intra-op pool only adds contention -- measured 128 -> 32 threads: 10x)."""
    ncpu = os.cpu_count() or 1
    best, best_v = 1, 0.0
    for t in sorted({min(t, ncpu) for t in (8, 16, 32, 64, ncpu)}):
        v = cpu_reference_sample(1024, t, with_mc=False)["rays_per_sec"]
        if v > best_v:
            best, best_v = t, v
    return best


def bench_config(n_rays, world):
    """The `config` object both arms print (the reference arm runs a bounded sample OF THIS workload)."""
    return {"workload": "config[1]: one 512x512 synthetic frame per GPU, %d silhouette rays, 8x512 SDF + "
                        "Deformer(MLP+LBS 129x225x65) + RenderNet; trace times=10 dthr=5e-5; 257^3 "
                        "coarse-to-fine grid + MC" % n_rays,
            "rays_per_frame": n_rays, "mc_grid": GRID_N, "l2": "256 MiB flush between timed regions",
            "parallelism": "frames sharded, dp%d, no data-path collective" % world}


def frame_ray_count():
    from selfreconcode_b200 import synth
    return int(synth.sphere_pixels(synth.camera(512, 512))[0].shape[0])


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (oracle port) on host cores.  Same config / metric as the GPU
    arm; every step is a bounded sample of that frame's rays (the whole frame takes ~25 s per step on the
    host), plus ONE untimed-in-`value` pass of the same 257^3 grid + MC for the voxel figure."""
    if rank != 0:
        return
    threads = pick_threads()
    n = 8192
    for _ in range(args.warmup if args.warmup < 2 else 1):
        cpu_reference_sample(512, threads, with_mc=False)
    vals, ts = [], []
    for _ in range(args.steps):
        r = cpu_reference_sample(n, threads, with_mc=False)
        vals.append(r["rays_per_sec"])
        ts.append(r["ray_seconds"])
    v = float(np.mean(vals))
    mc = cpu_reference_sample(256, threads, with_mc=True)
    line = {"impl": "reference", "metric": "rays_per_sec", "value": v, "unit": "rays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(ts)),
            "mc_voxels_per_sec": mc["mc_voxels_per_sec"], "mc_queried_voxels": mc["mc_queried"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(frame_ray_count(), max(world, 1)),
            "cpu_baseline": {"value": v, "unit": "rays/s", "cores": threads, "kind": "port",
                             "sample": "%d of the frame's rays per step: OptimizeSurfacePs(times=10) + shading "
                                       "through oracle/oracle.py (torch fp32 CPU); the 257^3 coarse-to-fine grid + MC "
                                       "once (mc_voxels_per_sec)" % n},
            "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step section")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's results (ray points, convergence mask, colours, SDF grid, "
                         "mesh) as DIR/<name>.npy, %d MiB at most" % (DUMP_BUDGET >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    assert torch.cuda.is_available(), "bench.py needs a GPU (the product has no CPU path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)
    from selfreconcode_b200 import _lib, ops
    _lib.load()
    sc = build_scene(dev, frame_seed=rank)
    eng = make_engine(sc, dev)
    R = sc["rays"]
    n_rays = R["rays"].shape[0]
    rays_d, init_d, bi_d = R["rays"].to(dev), R["init_pts"].to(dev), R["batch_inds"].to(dev)
    rays_h, init_h, bi_h = R["rays"].pin_memory(), R["init_pts"].pin_memory(), R["batch_inds"].pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up
    for _ in range(max(args.warmup, 3)):
        ray_part(sc, rays_d, init_d, bi_d)
        mc_part(sc, eng)
    torch.cuda.synchronize()
    ops.LAUNCHES = 0
    ev = lambda: torch.cuda.Event(enable_timing=True)
    ray_ms, mc_ms, trace_ms = [], [], []
    stats = {}
    barrier()
    with ClockSampler(local) as clk:
        t_wall0 = time.perf_counter()
        for _ in range(args.steps):
            flush.zero_()
            e0, e1, e2, e3 = ev(), ev(), ev(), ev()
            e0.record()
            pts, conv, rgb = ray_part(sc, rays_d, init_d, bi_d, stats)
            e1.record()
            flush.zero_()
            e2.record()
            grid, v, f = mc_part(sc, eng)
            e3.record()
            torch.cuda.synchronize()
            ray_ms.append(e0.elapsed_time(e1))
            mc_ms.append(e2.elapsed_time(e3))
        barrier()
        t_wall = time.perf_counter() - t_wall0
    launches = ops.LAUNCHES
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"ray_points": pts, "ray_converged": conv, "ray_rgb": rgb, "sdf_grid": grid,
                                         "mesh_vertices": v, "mesh_faces": f})
    # second number: weights change every step (a training loop): weight-norm fold + tensor-core weight packing
    # + an eager (not graph-replayed) trace are inside the timed region
    refold_ms = []
    for _ in range(args.steps):
        flush.zero_()
        for m in (sc["sdf"], sc["comp"].defs[0], sc["rn"]):
            with torch.no_grad():
                next(iter(m.parameters())).add_(0.0)      # bumps Tensor._version like optimizer.step(): refold in place
        a, b = ev(), ev()
        a.record()
        ray_part(sc, rays_d, init_d, bi_d)
        b.record()
        torch.cuda.synchronize()
        refold_ms.append(a.elapsed_time(b))
    ray_part(sc, rays_d, init_d, bi_d)   # back to the steady state (graph captured again)
    ray_part(sc, rays_d, init_d, bi_d)
    torch.cuda.synchronize()
    # per-kernel timing of the dominant kernel (trace_kernel): events around the 11 launches
    tk = []
    for _ in range(3):
        flush.zero_()
        a, b = ev(), ev()
        sdf_only = sc["sdf"].fused_sdf_only()
        dnet = sc["comp"].defs[0].fused(RATIO)
        lbs = sc["comp"].defs[1].lbs_state()
        a.record()
        _, _, counters = ops.trace_surface_points(sdf_only, dnet, lbs, sc["cam"]["cam_pos"], rays_d, init_d, bi_d,
                                                  sc["conds"][0], 5e-5, sc["ang"], 3.05, 1.0, 10,
                                                  return_counters=True)
        trace_mode = "tc" if (ops.TC_ENABLED and n_rays >= ops.TC_MIN_POINTS) else "reverse"
        b.record()
        torch.cuda.synchronize()
        tk.append(a.elapsed_time(b))
    cnt = counters.cpu().tolist()
    ray_iters = sum(cnt[1:11])
    trace_flops = (n_rays + 3.0 * ray_iters) * (F_S + F_D)  # algorithmic: (1+3k) per ray
    # MC sweep kernels alone (classify + scan + emit) on the last grid
    sd = grid[0, 0].permute(2, 1, 0).contiguous()
    mk = []
    for _ in range(5):
        flush.zero_()
        a, b = ev(), ev()
        a.record()
        vv, ff = ops.marching_cubes(sd, 1, 1, 1, 0, 0, 0, 0.0)
        b.record()
        torch.cuda.synchronize()
        mk.append(a.elapsed_time(b))
    mc_bytes = 4.0 * GRID_N ** 3 + 12.0 * vv.shape[0] + 24.0 * ff.shape[0]

    # ---- e2e: host buffers in, results out, through the drop-in API
    e2e_ms = []
    for i in range(args.steps + 1):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r_d = rays_h.to(dev, non_blocking=True)
        i_d = init_h.to(dev, non_blocking=True)
        b_d = bi_h.to(dev, non_blocking=True)
        pts, conv, rgb = ray_part_api(sc, r_d, i_d, b_d)
        rgb_h = rgb.cpu()
        conv_h = conv.cpu()
        torch.cuda.synchronize()
        if i > 0:
            e2e_ms.append(1e3 * (time.perf_counter() - t0))
    h2d = rays_h.numel() * 4 + init_h.numel() * 4 + bi_h.numel() * 8
    d2h = rgb_h.numel() * 4 + conv_h.numel()

    train = None
    if not args.no_train:
        train = train_part(sc, dev, rank, world, dist, args.steps, args.warmup)
        train_launches = ops.LAUNCHES
        # the scene's parameters moved (Adam): nothing below depends on their values

    t_ray = torch.tensor([float(np.mean(ray_ms)), float(np.mean(mc_ms)), float(np.mean(e2e_ms)),
                          float(n_rays)], device=dev, dtype=torch.float64)
    if dist is not None:
        mx = t_ray.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t_ray.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ray_t, mc_t, e2e_t, total_rays = mx[0].item(), mx[1].item(), mx[2].item(), sm[3].item()
    else:
        ray_t, mc_t, e2e_t, total_rays = t_ray[0].item(), t_ray[1].item(), t_ray[2].item(), float(n_rays)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    pk = peaks()
    layer_ms, layer_flops = layer_roofline(dev, n_rays)
    layer_tf = layer_flops / (layer_ms * 1e-3) / 1e12
    trace_s = float(np.mean(tk)) * 1e-3
    mc_s = float(np.mean(mk)) * 1e-3
    line = {
        "metric": "rays_per_sec", "value": total_rays / (ray_t * 1e-3), "unit": "rays/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ray_t + mc_t, "ms_ray_part": ray_t, "ms_mc_part": mc_t,
        "ms_ray_part_refold": float(np.mean(refold_ms)),
        "rays_per_sec_refold": n_rays / (float(np.mean(refold_ms)) * 1e-3),
        "mc_voxels_per_sec": world * GRID_N ** 3 / (mc_t * 1e-3),
        "mc_queried_voxels": int(eng.last_num_queried), "mc_vertices": int(v.shape[0]), "mc_faces": int(f.shape[0]),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(n_rays, world),
        "e2e": {"value": total_rays / (e2e_t * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "ms": e2e_t},
        "gpu_launches": int(launches),
        "roofline": {"kernel": "tc_layer_pair_kernel<softplus,1> (tcgen05 cta_group::2 split-BF16 GEMM layer 512x512 of "
                               "the tracer, M = rays of the frame; ~300 such launches per trace)",
                     "bound": "tensor", "achieved": layer_tf, "peak": pk["tensor"], "unit": "TFLOP/s",
                     "frac": layer_tf / pk["tensor"],
                     # dram__bytes_read.sum + dram__bytes_write.sum of one launch at M = 50 333 from the
                     # ncu --set full capture in profiles/r01c_summary.md (algorithmic: 103 MB in + 103 MB out)
                     "traffic": 159.3e6 if n_rays == 50333 else None,
                     "peak_source": pk["src"] + " bf16 cuBLAS burst", "ms_per_launch": layer_ms,
                     "mma_terms": 3, "tensor_pipe_frac": 3.0 * layer_tf / pk["tensor"],
                     "note": "achieved = algorithmic fp32 FLOPs of one layer launch (2*M*512*512, SURVEY 8d: 0.524 "
                             "MFLOP per point per hidden layer) / its average duration, CUDA events over %d "
                             "back-to-back launches on cold operands; the split-BF16 scheme issues 3 bf16 MMAs per "
                             "fp32 product, so the executed tensor rate is 3x that (tensor_pipe_frac) and the "
                             "ceiling of `frac` is 1/3" % 24,
                     "trace": {"ms": trace_s * 1e3, "ray_iterations": int(ray_iters), "engine": trace_mode,
                               "algorithmic_tflops_fwd_mode_count": trace_flops / trace_s / 1e12,
                               "executed_tflops_fp32_equiv": 2.0 * ray_iters * (F_S + F_D) / trace_s / 1e12,
                               "note": "SURVEY 8d counts a traced ray as (1+3k) network evaluations (forward-mode "
                                       "tangents, what the reference's autograd costs); this implementation runs "
                                       "one forward + one reverse sweep per iteration (2k+1 evaluations)"}},
        "roofline_mc": {"kernel": "mc_sign+mc_classify+mc_scan+mc_emit", "bound": "hbm",
                        "achieved": mc_bytes / mc_s / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                        "frac": mc_bytes / mc_s / 1e9 / pk["hbm"],
                        # ncu capture of the four kernels (profiles/r01c_summary.md); algorithmic = mc_bytes
                        "traffic": 92.6e6 if GRID_N == 257 else None, "algorithmic_bytes": mc_bytes,
                        "ms": mc_s * 1e3,
                        "peak_source": pk["src"]},
        "clocks": clk.summary(),
        "wall_s_timed_region": t_wall,
    }
    if train is not None:
        wg_ms, wg_flops = wgrad_roofline(dev)
        wg_tf = wg_flops / (wg_ms * 1e-3) / 1e12
        train["gpu_launches_own_kernels_per_step"] = int(train_launches // args.steps)
        train["roofline"] = {"kernel": "tc_wgrad_kernel (tcgen05 MN-major split-BF16 GEMM dW = delta^T x, 512x512 over "
                                       "393 216 rows: the def_regu block's translator layers)", "bound": "tensor",
                             "achieved": wg_tf, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": wg_tf / pk["tensor"],
                             "ms_per_launch": wg_ms, "mma_terms": 3, "tensor_pipe_frac": 3.0 * wg_tf / pk["tensor"],
                             "traffic": None, "peak_source": pk["src"] + " bf16 cuBLAS burst"}
        line["train"] = train
    if not args.no_cpu_baseline and world == 1:
        threads = pick_threads()
        cb = cpu_reference_sample(None, threads, with_mc=True, rays={k: v for k, v in R.items()}, keep=True)
        # parity at the benchmark's own size: the GPU results of one more (untimed) step vs the oracle's
        pts_g, conv_g, rgb_g = ray_part(sc, rays_d, init_d, bi_d)
        grid_g, v_g, f_g = mc_part(sc, eng)
        import MCGpu
        og = cb["keep"]["grid"].to(dev)
        v_o, f_o = MCGpu.mc_gpu(og.permute(2, 1, 0).contiguous(), eng.spacing_x, eng.spacing_y, eng.spacing_z,
                                eng.bx, eng.by, eng.bz, 0.0)
        line["parity"] = parity_report(dict(pts=pts_g, conv=conv_g, rgb=rgb_g, grid=grid_g[0, 0],
                                            calc=eng.last_calculated, verts=v_g, faces=f_g,
                                            verts_on_oracle_grid=v_o, faces_on_oracle_grid=f_o), cb["keep"])
        line["config0"] = config0_part(dev, threads)
        line["cpu_baseline"] = {"value": cb["rays_per_sec"], "unit": "rays/s", "cores": threads, "kind": "port",
                                "sample": "all rays of the same frame (trace times=10 + shading) and the same 257^3 "
                                          "coarse-to-fine grid + MC through oracle/ (torch fp32 CPU + C)",
                                "mc_voxels_per_sec": cb.get("mc_voxels_per_sec"), "mc_grid": cb.get("mc_grid"),
                                "ray_seconds": cb["ray_seconds"], "mc_seconds": cb.get("mc_seconds")}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
