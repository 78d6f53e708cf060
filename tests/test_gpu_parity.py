"""GPU parity tests (run on the B200 box: `pytest -m gpu`).

Every test calls the product through its C-ABI wrappers / drop-in modules and compares with
  (1) the golden vectors recorded from the unmodified reference (tests/golden/),
  (2) the CPU oracle on the same seeded inputs,
  (3) the outputs of the reference's own CUDA kernels on the same seeded inputs, recorded on a B200
      (tests/golden/ref_kernels.npz, written by oracle/make_golden_ref.py).
Bars: bit-exact for integer / index work (MC faces and vertex ids, sampler corner indices,
masks away from thresholds, boundary flags); 1e-4 norm-wise relative for floating point
(the north star's tolerance), tighter where the arithmetic allows it.
"""
import numpy as np
import pytest
import torch

from helpers import (RATIO, SMPL_PARENTS, build_render, build_sdf_full, build_sdf_small,
                     build_skinner, build_translator, dropin, golden, mc_tri_table, plain_params,
                     norm_err, rel_err, sdf_params, sha256, wn_params)

pytestmark = pytest.mark.gpu
FP_TOL = 1e-4


def helpers_root():
    import helpers
    return helpers.ROOT


def _sampled(g, key):
    """(flat indices, values) of a reference output stored as a seeded sample of its elements."""
    return g[key + "_idx"], g[key + "_val"]


# Inputs of the comparisons with the reference's CUDA kernels (oracle/make_golden_ref.py runs the same functions).
def _minv_ab_inputs():
    """50 000 matrices; the backward kernel is compared on 512 of them (`rows`) with gradients `gr`."""
    ms = torch.randn(50000, 3, 3, generator=torch.Generator().manual_seed(1))
    rows = torch.randperm(ms.shape[0], generator=torch.Generator().manual_seed(2))[:512].sort()[0]
    gr = torch.randn(512, 3, 3, generator=torch.Generator().manual_seed(3))
    return ms, rows, gr


def _interp_ab_inputs():
    g = torch.Generator().manual_seed(6)
    x = torch.randn(1, 1, 33, 41, 17, generator=g)
    y = torch.randn(1, 1, 65, 81, 33, generator=g)      # output gradient for the backward kernel
    return x, y


def _grid_sampler_ab_inputs():
    g = torch.Generator().manual_seed(5)
    inp = torch.rand(1, 24, 9, 17, 11, generator=g)
    grid = (torch.rand(1, 1, 1, 3000, 3, generator=g) - 0.5) * 2.2
    go = torch.randn(1, 24, 1, 1, 3000, generator=g)
    ggi, ggg = torch.randn(inp.shape, generator=g), torch.randn(grid.shape, generator=g)
    return inp, grid, go, ggi, ggg


# ------------------------------------------------------------------------------------------------
# FastMinv
# ------------------------------------------------------------------------------------------------
def test_minv3x3_forward_backward(cuda_dev):
    dropin()
    import FastMinv
    from oracle import c_api
    g = torch.Generator().manual_seed(0)
    for n in (1, 7, 10000, 100003):
        ms = torch.randn(n, 3, 3, generator=g)
        ms[::97] *= 1e-2  # near-singular rows exercise the |det|<1e-4 mask
        inv, chk = FastMinv.Fast3x3Minv(ms.to(cuda_dev))
        io, co = c_api.minv3x3(ms.numpy())
        det = torch.linalg.det(ms.double()).abs().numpy()
        safe = np.abs(det - 1e-4) > 1e-6
        assert np.array_equal(chk.cpu().numpy()[safe], co[safe])
        ok = co & chk.cpu().numpy()
        if ok.any():  # compare adjugates (inverse * det): insensitive to near-singular scaling
            # (2x2 minors cancel: agreement is to the conditioning of the minors, ~1e-4 at worst)
            assert rel_err(inv.cpu().numpy()[ok] * det[ok, None, None], io[ok] * det[ok, None, None]) < 5e-4
        assert (inv.cpu().numpy()[~chk.cpu().numpy()] == 0).all()
        # property from the reference's own check script (FastMinv/check.py:18-19)
        good = chk & (torch.from_numpy(det).to(cuda_dev) > 1e-2)
        if good.any():
            err = (inv[good].double() @ ms.to(cuda_dev)[good].double() - torch.eye(3, device=cuda_dev, dtype=torch.float64)).norm(dim=(1, 2))
            assert err.max().item() < 1e-3
        gr = torch.randn(n, 3, 3, generator=g)
        bo = FastMinv.Fast3x3Minv_backward(gr.to(cuda_dev), inv)
        ref = -(inv.transpose(1, 2) @ gr.to(cuda_dev) @ inv.transpose(1, 2))
        assert rel_err(bo.cpu().numpy(), ref.cpu().numpy()) < 1e-5
    # float64 + error behaviour
    md = torch.randn(33, 3, 3, dtype=torch.float64, generator=g).to(cuda_dev)
    invd, _ = FastMinv.Fast3x3Minv(md)
    assert torch.allclose(invd, torch.linalg.inv(md), atol=1e-9)
    with pytest.raises(RuntimeError):
        FastMinv.Fast3x3Minv(torch.randn(4, 3, 3))
    with pytest.raises(RuntimeError):
        FastMinv.Fast3x3Minv(md.transpose(1, 2))
    inv0, chk0 = FastMinv.Fast3x3Minv(torch.empty(0, 3, 3, device=cuda_dev))
    assert inv0.shape == (0, 3, 3) and chk0.shape == (0,)


def _minv_adjugate_err(inv, ms, ok):
    """rel_err of inverse * |det| * sign(det) against the float64 adjugate over the invertible rows `ok`."""
    det = torch.linalg.det(ms.double()).view(-1, 1, 1)
    adj = (torch.linalg.inv(ms.double()) * det).cpu().numpy()
    return rel_err((inv.double() * det.abs() * torch.sign(det)).cpu().numpy()[ok], adj[ok])


def test_minv3x3_matches_reference_kernel(cuda_dev):
    ref = golden("ref_kernels.npz")
    dropin()
    import FastMinv
    ms, _, gr = _minv_ab_inputs()
    ms = ms.to(cuda_dev)
    a, ac = FastMinv.Fast3x3Minv(ms)
    torch.cuda.synchronize()
    bc = np.unpackbits(ref["minv_mask"])[:ms.shape[0]].astype(bool)
    assert np.array_equal(ac.cpu().numpy(), bc), "singularity mask identical to the reference kernel"
    # floating point: the 2x2 minors cancel, and FMA contraction differs between the two builds, so
    # the two kernels agree to the conditioning of the minors, not to the last bit: both must be
    # equally close to the float64 adjugate (the reference kernel's distance is stored).
    m = ac.cpu().numpy()  # invertible ones (the others are zeroed by both kernels)
    assert (a[~ac] == 0).all()
    ea = _minv_adjugate_err(a, ms, m)
    eb = float(ref["minv_adj_err"])
    assert ea < 5e-4 and eb < 5e-4 and ea < 2 * eb + 1e-6
    # same inputs to both backward kernels: the reference kernel's inverses of 512 of the matrices
    bo = FastMinv.Fast3x3Minv_backward(gr.to(cuda_dev), torch.from_numpy(ref["minv_bwd_inv"]).to(cuda_dev))
    assert rel_err(bo.cpu().numpy(), ref["minv_bwd"]) < 1e-6


# ------------------------------------------------------------------------------------------------
# Marching cubes
# ------------------------------------------------------------------------------------------------
def _test_grid(n, seed, aniso=False):
    g = torch.Generator().manual_seed(seed)
    shape = (n, n + 6, n - 4) if aniso else (n, n, n)
    ax = [torch.linspace(-1, 1, s) for s in shape]
    xx, yy, zz = torch.meshgrid(ax, indexing="ij")
    f = torch.sqrt(xx * xx + yy * yy + zz * zz) - 0.62 + 0.07 * torch.sin(6 * xx) * torch.cos(5 * yy) \
        + 0.02 * torch.randn(shape, generator=g)
    return f.contiguous()


def test_mc_exact_vs_oracle(cuda_dev):
    dropin()
    import MCGpu
    from oracle import c_api
    tt = mc_tri_table()
    for n, aniso, iso in ((9, False, 0.0), (33, True, 0.0), (65, False, 0.013), (40, True, -0.05)):
        grid = _test_grid(n, n, aniso)
        step, org = (0.031, 0.027, 0.05), (-1.0, -0.9, -0.7)
        v, f = MCGpu.mc_gpu(grid.to(cuda_dev), *step, *org, iso)
        vo, fo = c_api.marching_cubes(grid.numpy(), tt, iso, step, org)
        assert v.dtype == torch.float32 and f.dtype == torch.int64
        assert np.array_equal(f.cpu().numpy(), fo), "face indices (canonical order) must be identical"
        assert np.array_equal(v.cpu().numpy(), vo), "vertex positions are bit-exact (double division + fmaf)"
    # word-boundary shapes of the sign bit-plane (nz = 2, 32, 33, 64, 65, 97) on dense random-sign grids:
    # every cell is active, every edge flag and every k -> k+1 word crossing is exercised
    g = torch.Generator().manual_seed(99)
    for shape in ((2, 2, 2), (3, 2, 33), (2, 5, 32), (4, 3, 64), (3, 4, 65), (5, 5, 97), (9, 7, 31)):
        grid = (torch.rand(shape, generator=g) - 0.5).contiguous()
        v, f = MCGpu.mc_gpu(grid.to(cuda_dev), 1, 1, 1, 0, 0, 0, 0.0)
        vo, fo = c_api.marching_cubes(grid.numpy(), tt)
        assert np.array_equal(f.cpu().numpy(), fo), shape
        assert np.array_equal(v.cpu().numpy(), vo), shape
    # surface touching the +x/+y/+z boundary layer -> -1 indices exactly where the oracle has them
    grid = _test_grid(17, 5)
    grid[-1] = -1.0
    v, f = MCGpu.mc_gpu(grid.to(cuda_dev), 1, 1, 1, 0, 0, 0, 0.0)
    vo, fo = c_api.marching_cubes(grid.numpy(), tt)
    assert (fo == -1).any()
    assert np.array_equal(f.cpu().numpy(), fo) and np.array_equal(v.cpu().numpy(), vo)
    # empty / legacy error convention
    v, f = MCGpu.mc_gpu(torch.ones(8, 8, 8, device=cuda_dev))
    assert v.shape == (0, 3) and f.shape == (0, 3)
    assert MCGpu.mc_gpu(torch.ones(8, 8, 8, device=cuda_dev, dtype=torch.float64)) == []
    with pytest.raises(RuntimeError):
        MCGpu.mc_gpu(torch.ones(8, 8, 8))


def _canon(v, f):
    """canonical form of a mesh with race-ordered ids: sort vertices lexicographically, remap and
    sort faces (cyclic order inside a face is kept: it is table-driven in both implementations)."""
    v = np.asarray(v)
    f = np.asarray(f)
    order = np.lexsort((v[:, 2], v[:, 1], v[:, 0]))
    inv = np.empty_like(order)
    inv[order] = np.arange(len(order))
    f2 = np.where(f >= 0, inv[np.clip(f, 0, None)], -1)
    f2 = f2[np.lexsort((f2[:, 2], f2[:, 1], f2[:, 0]))]
    return v[order], f2


MC_AB_CASES = ((33, True), (129, False))
MC_AB_ARGS = (0.0078125, 0.0078125, 0.0078125, -1.0, -1.0, -1.0, 0.0)


def test_mc_matches_reference_kernel(cuda_dev):
    ref = golden("ref_kernels.npz")
    dropin()
    import MCGpu
    for n, aniso in MC_AB_CASES:
        grid = _test_grid(n, 100 + n, aniso).to(cuda_dev)
        v, f = MCGpu.mc_gpu(grid, *MC_AB_ARGS)
        assert (v.shape[0], f.shape[0]) == (int(ref["mc%d_nv" % n]), int(ref["mc%d_nf" % n]))
        cv, cf = _canon(v.cpu().numpy(), f.cpu().numpy())
        assert sha256(cv) == ref["mc%d_v_sha" % n], "vertex positions bit-identical to the reference kernel"
        assert sha256(cf) == ref["mc%d_f_sha" % n], "faces identical after canonicalising the race-ordered ids"


def test_mc_full_size_properties(cuda_dev):
    """257^3 (the BASELINE grid): a closed surface must come out watertight."""
    dropin()
    import MCGpu
    n = 257
    ax = torch.linspace(-1, 1, n, device=cuda_dev)
    xx, yy, zz = torch.meshgrid([ax] * 3, indexing="ij")
    grid = (torch.sqrt(xx * xx + yy * yy + zz * zz) - 0.6 + 0.05 * torch.sin(9 * xx) * torch.sin(7 * yy)).contiguous()
    v, f = MCGpu.mc_gpu(grid, 2.0 / n, 2.0 / n, 2.0 / n, -1.0, -1.0, -1.0, 0.0)
    assert (f >= 0).all() and f.max().item() == v.shape[0] - 1
    e = torch.cat([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]], 0)
    key = torch.minimum(e[:, 0], e[:, 1]) * v.shape[0] + torch.maximum(e[:, 0], e[:, 1])
    _, cnt = torch.unique(key, return_counts=True)
    assert (cnt == 2).all(), "every edge shared by exactly two triangles"
    assert v.shape[0] - cnt.numel() + f.shape[0] == 2, "Euler characteristic of a sphere"
    # determinism: same call, same bytes
    v2, f2 = MCGpu.mc_gpu(grid, 2.0 / n, 2.0 / n, 2.0 / n, -1.0, -1.0, -1.0, 0.0)
    assert torch.equal(v, v2) and torch.equal(f, f2)


# ------------------------------------------------------------------------------------------------
# interp2x_boundary3d
# ------------------------------------------------------------------------------------------------
def test_interp2x3d(cuda_dev):
    dropin()
    import interp2x_boundary3d as op
    from oracle import c_api
    g = torch.Generator().manual_seed(2)
    for shape in ((3, 4, 5), (9, 9, 9), (17, 21, 9), (1, 1, 1)):
        x = torch.randn(1, 1, *shape, generator=g)
        out, bnd = op.forward(x.to(cuda_dev), 0.1)
        oo, bo = c_api.interp2x3d(x[0, 0].numpy(), 0.1)
        assert np.array_equal(out[0, 0].cpu().numpy(), oo)
        assert np.array_equal(bnd[0, 0].cpu().numpy(), bo)
        ref = torch.nn.functional.interpolate(x, size=out.shape[2:], mode="trilinear", align_corners=True)
        assert torch.allclose(out.cpu(), ref, atol=1e-6)
        # adjoint test: <A x, y> == <x, A^T y>
        y = torch.randn(out.shape, generator=g).to(cuda_dev)
        gin = op.backward(y)
        assert abs((out * y).sum().item() - (x.to(cuda_dev) * gin).sum().item()) < 1e-3 * max(1.0, out.numel() ** 0.5)
    # against the reference kernel
    ref = golden("ref_kernels.npz")
    x, y = _interp_ab_inputs()
    a, ab = op.forward(x.to(cuda_dev), 0.0)
    assert sha256(a) == ref["i2x_out_sha"] and sha256(ab) == ref["i2x_bnd_sha"]
    idx, want = _sampled(ref, "i2x_bwd")
    assert np.allclose(op.backward(y.to(cuda_dev)).cpu().numpy().reshape(-1)[idx], want, rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------------
# GridSamplerMine
# ------------------------------------------------------------------------------------------------
def test_grid_sampler_forward_exact_and_indices(cuda_dev):
    from selfreconcode_b200 import ops
    from oracle import c_api
    g = torch.Generator().manual_seed(3)
    inp = torch.rand(1, 24, 7, 13, 9, generator=g)
    grid = (torch.rand(1, 1, 1, 4000, 3, generator=g) - 0.5) * 2.3  # beyond [-1,1]: border clipping
    out, cidx = ops.grid_sample3d_forward(inp.to(cuda_dev), grid.to(cuda_dev), want_corner_idx=True)
    oo, co = c_api.grid_sample3d(inp[0].numpy(), grid.view(-1, 3).numpy())
    assert np.array_equal(cidx[0].cpu().numpy(), co), "skinning (corner) indices are bit-exact"
    assert np.array_equal(out.view(24, -1).cpu().numpy(), oo), "forward values are bit-exact"
    ref = torch.nn.functional.grid_sample(inp, grid, mode="bilinear", padding_mode="border", align_corners=False)
    assert torch.allclose(out.cpu(), ref, atol=1e-6)
    # strided (non-contiguous) input, as the reference's TensorInfo path allows
    big = torch.rand(1, 24, 7, 13, 18, generator=g).to(cuda_dev)
    view = big[..., ::2]
    o2 = ops.grid_sample3d_forward(view, grid.to(cuda_dev))
    assert torch.equal(o2, ops.grid_sample3d_forward(view.contiguous(), grid.to(cuda_dev)))


def test_grid_sampler_gradcheck_first_and_second_order(cuda_dev):
    """The reference's own check (MCAcc/check_grid_sampler_mine.py:5-16), in float64."""
    dropin()
    from MCAcc.grid_sampler_mine import GridSamplerMine3dFunction, GridSamplerMine3dBackwardFunction
    g = torch.Generator().manual_seed(4)
    inp = torch.randn(1, 5, 15, 15, 15, dtype=torch.float64, generator=g).to(cuda_dev).requires_grad_(True)
    grid = ((torch.rand(1, 1, 1, 10, 3, dtype=torch.float64, generator=g) - 0.5) * 2.2).to(cuda_dev).requires_grad_(True)
    assert torch.autograd.gradcheck(GridSamplerMine3dFunction.apply, (inp, grid))
    go = torch.randn(1, 5, 1, 1, 10, dtype=torch.float64, generator=g).to(cuda_dev).requires_grad_(True)
    assert torch.autograd.gradcheck(GridSamplerMine3dBackwardFunction.apply, (inp, grid, go))


def test_grid_sampler_matches_reference_kernels(cuda_dev):
    ref = golden("ref_kernels.npz")
    dropin()
    import GridSamplerMine as op
    inp, grid, go, ggi, ggg = [t.to(cuda_dev) for t in _grid_sampler_ab_inputs()]
    a = op.forward(inp, grid, 0, 1)
    assert sha256(a) == ref["gs_fwd_sha"], "forward bit-identical to the reference kernel"
    gi, gg = op.backward(inp, grid, go, 0, 1)
    for x, key, atol, rtol in ((gi, "gs_gi", 1e-5, 1e-5), (gg, "gs_gg", 2e-4, 1e-4)):
        idx, want = _sampled(ref, key)
        assert np.allclose(x.cpu().numpy().reshape(-1)[idx], want, rtol=rtol, atol=atol), key
    o = op.dbackward(ggi, ggg, inp, grid, go, 0, 1)
    for i, x in enumerate(o):
        # rel_err's floor (mean |reference|) is taken over the whole reference output
        idx, want = _sampled(ref, "gs_dd%d" % i)
        err = np.abs(x.cpu().numpy().reshape(-1)[idx].astype(np.float64) - want) / (np.abs(want) + ref["gs_dd%d_absmean" % i])
        assert err.max() < 1e-4, i


# ------------------------------------------------------------------------------------------------
# Fused fields vs golden (reference) and oracle
# ------------------------------------------------------------------------------------------------
def test_sdf_small_vs_golden(cuda_dev):
    g = golden("sdf_small.npz")
    net = build_sdf_small(g).to(cuda_dev)
    pts = torch.from_numpy(g["pts"]).to(cuda_dev)
    for r in (1.0, 0.4):
        s, gr, ft = net.forward_fused(pts, r, want_grad=True, want_feat=True)
        assert rel_err(s.cpu().numpy(), g["sdf_r%g" % r]) < FP_TOL
        assert rel_err(gr.cpu().numpy(), g["grad_r%g" % r]) < FP_TOL
        assert rel_err(ft.cpu().numpy(), g["feat_r%g" % r]) < FP_TOL
        # module surface: forward() under no_grad sets rendcond like the reference
        with torch.no_grad():
            y = net(pts, r)
        assert y.shape == (pts.shape[0], 1) and net.rendcond.shape == (pts.shape[0], 16)
        assert rel_err(y.cpu().numpy(), g["sdf_r%g" % r]) < FP_TOL
    with pytest.raises(RuntimeError):
        net(pts.cpu(), 1.0)


def test_sdf_full_vs_golden_and_autograd_path(cuda_dev):
    g = golden("sdf_full.npz")
    net = build_sdf_full(g).to(cuda_dev)
    pts = torch.from_numpy(g["pts"]).to(cuda_dev)
    s, gr, ft = net.forward_fused(pts, RATIO, want_grad=True, want_feat=True)
    assert rel_err(s.cpu().numpy(), g["sdf"]) < FP_TOL
    assert rel_err(gr.cpu().numpy(), g["grad"]) < FP_TOL
    assert rel_err(ft.cpu().numpy(), g["feat"]) < FP_TOL
    s1, _, _ = net.forward_fused(pts, RATIO, want_grad=False, want_feat=False)  # sdf-only last layer
    assert rel_err(s1.cpu().numpy(), g["sdf"]) < FP_TOL
    # training path (autograd, torch ops on the GPU) agrees with the fused path
    p = pts.clone().requires_grad_(True)
    y = net(p, RATIO)
    (ga,) = torch.autograd.grad(y, p, torch.ones_like(y), create_graph=True)
    assert rel_err(y.detach().cpu().numpy(), s.cpu().numpy()) < FP_TOL
    assert rel_err(ga.detach().cpu().numpy(), gr.cpu().numpy()) < FP_TOL
    # ragged sizes: tile tails (P not a multiple of 16 / 64), P = 1
    for P in (1, 15, 17, 63, 65, 96):
        a, b, _ = net.forward_fused(pts[:P], RATIO, want_grad=True, want_feat=False)
        assert torch.equal(a, s[:P]) and torch.equal(b, gr[:P])
    # refold after an in-place parameter update (optimizer step)
    with torch.no_grad():
        net.lin8.bias.add_(0.125)
    s2, _, _ = net.forward_fused(pts, RATIO, want_grad=False, want_feat=False)
    assert torch.allclose(s2, s + 0.125, atol=1e-6)


def _deform_modules(g, dev):
    dropin()
    from model.Deformer import CompositeDeformer
    tr = build_translator(g)
    sk = build_skinner(g)
    comp = CompositeDeformer([tr, sk]).to(dev)
    conds = [torch.from_numpy(g["dcond"]).to(dev),
             [torch.from_numpy(g["poses"]).to(dev), torch.from_numpy(g["trans"]).to(dev)]]
    return comp, conds


def test_deformer_vs_golden(cuda_dev):
    g = golden("deform.npz")
    comp, conds = _deform_modules(g, cuda_dev)
    np.testing.assert_allclose(comp.defs[1].init_pose.cpu().numpy(), g["init_pose_inv"], atol=1e-6)
    pts = torch.from_numpy(g["pts"]).to(cuda_dev)
    bi = torch.from_numpy(g["batch_inds"]).to(cuda_dev)
    d, J, ci = comp.forward_fused(pts, conds, bi, RATIO, want_jac=True, want_corner_idx=True)
    assert rel_err(d.cpu().numpy(), g["d"]) < FP_TOL
    assert rel_err(comp.defs[0].offset.cpu().numpy(), g["offset"]) < FP_TOL
    assert rel_err(J.cpu().numpy(), g["jac"]) < FP_TOL
    d0, _, _ = comp.forward_fused(pts, conds, bi, RATIO, want_jac=False)
    assert rel_err(d0.cpu().numpy(), g["d"]) < FP_TOL
    # LBS corner ("skinning") indices: bit-exact against the sampler oracle at the same p'
    from oracle import c_api
    pp = pts + comp.defs[0].offset
    nps = 2. * (pp - comp.defs[1].b_min) / (comp.defs[1].b_max - comp.defs[1].b_min) - 1.
    _, co = c_api.grid_sample3d(g["ws"][0], nps.cpu().numpy())
    assert np.array_equal(ci.cpu().numpy(), co)
    # posed skeleton + module forward (no grad) + autograd path agreement
    pj = comp.defs[1].posedSkeleton(conds[1])
    assert rel_err(pj.cpu().numpy(), g["posed"]) < 1e-5
    with torch.no_grad():
        dm = comp(pts, conds, bi, ratio=RATIO)
    assert torch.equal(dm, d)
    p = pts.clone().requires_grad_(True)
    da = comp(p, conds, bi, ratio=RATIO)
    assert rel_err(da.detach().cpu().numpy(), g["d"]) < FP_TOL
    from utils import compute_Jacobian
    Ja = compute_Jacobian(p, da, True, False)
    assert rel_err(Ja.cpu().numpy(), g["jac"]) < FP_TOL
    # mesh mode (batch_inds=None): [N,V,3] points, frame = leading index
    N = conds[0].shape[0]
    mesh = pts[:30].unsqueeze(0).expand(N, 30, 3).contiguous()
    with torch.no_grad():
        dmesh = comp(mesh, conds, ratio=RATIO)
    for b in range(N):
        db, _, _ = comp.forward_fused(pts[:30], conds, torch.full((30,), b, device=cuda_dev), RATIO)
        assert torch.allclose(dmesh[b], db, atol=1e-6)


def test_render_vs_golden(cuda_dev):
    g = golden("render.npz")
    rn = build_render(g).to(cuda_dev)
    args = [torch.from_numpy(g[k]).to(cuda_dev) for k in ("pts", "normals", "views", "feat")]
    with torch.no_grad():
        rgb = rn(*args, RATIO)
    assert rel_err(rgb.cpu().numpy(), g["rgb"]) < FP_TOL
    args[0].requires_grad_(True)
    rgb_a = rn(*args, RATIO)  # autograd path
    assert rel_err(rgb_a.detach().cpu().numpy(), g["rgb"]) < FP_TOL


def test_cardinal_rays_and_shade_geometry(cuda_dev):
    g, c, gs = golden("deform.npz"), golden("cardinal.npz"), golden("sdf_full.npz")
    comp, conds = _deform_modules(g, cuda_dev)
    sdf = build_sdf_full(gs).to(cuda_dev)
    pts = torch.from_numpy(g["pts"]).to(cuda_dev)
    bi = torch.from_numpy(g["batch_inds"]).to(cuda_dev)
    rays = torch.from_numpy(c["rays"]).to(cuda_dev)
    dropin()
    import utils
    cr, ds = utils.compute_cardinal_rays(comp, pts, rays, conds, bi, RATIO, 'test')
    assert rel_err(cr.cpu().numpy(), c["crays"]) < FP_TOL
    assert rel_err(ds.cpu().numpy(), c["ds"]) < FP_TOL
    from selfreconcode_b200 import ops
    lbs = comp.defs[1].lbs_state()
    lbs.set_pose(conds[1][0], conds[1][1])
    n, cr2, ft, dp, ok = ops.shade_geometry(sdf.fused(), comp.defs[0].fused(RATIO), lbs, pts, rays, bi,
                                            conds[0], nfeat=256, want_dpos=True)
    assert rel_err(cr2.cpu().numpy(), c["crays"]) < FP_TOL
    assert rel_err(dp.cpu().numpy(), c["ds"]) < FP_TOL
    s, gr, f2 = sdf.forward_fused(pts, RATIO, want_grad=True, want_feat=True)
    nn = gr / gr.norm(dim=1, keepdim=True)
    assert rel_err(n.cpu().numpy(), nn.cpu().numpy()) < 1e-5
    assert torch.allclose(ft, f2, atol=1e-6)
    assert ok.all()


def test_deformed_normals_vs_golden(cuda_dev):
    """utils.compute_deformed_normals (utils/utils.py:132-153) on the fused kernels vs the reference's values."""
    g, n, gs = golden("deform.npz"), golden("normals.npz"), golden("sdf_full.npz")
    comp, conds = _deform_modules(g, cuda_dev)
    sdf = build_sdf_full(gs).to(cuda_dev)
    pts = torch.from_numpy(g["pts"]).to(cuda_dev)
    bi = torch.from_numpy(g["batch_inds"]).to(cuda_dev)
    dropin()
    import utils
    nx, ds = utils.compute_deformed_normals(sdf, comp, pts, conds, bi, RATIO, 'test')
    assert rel_err(nx.cpu().numpy(), n["normals"]) < FP_TOL
    assert rel_err(ds.cpu().numpy(), n["ds"]) < FP_TOL
    # the autograd ('train') phase goes through the same math
    p = pts.clone().requires_grad_(True)
    nx2, _ = utils.compute_deformed_normals(sdf, comp, p, conds, bi, RATIO, 'train')
    assert rel_err(nx2.detach().cpu().numpy(), n["normals"]) < FP_TOL


def test_trace_vs_golden(cuda_dev):
    t, g, gs = golden("trace.npz"), golden("deform.npz"), golden("sdf_full.npz")
    comp, conds = _deform_modules(g, cuda_dev)
    sdf = build_sdf_full(gs).to(cuda_dev)
    dropin()
    import utils
    rays, start = torch.from_numpy(t["rays"]).to(cuda_dev), torch.from_numpy(t["start"]).to(cuda_dev)
    bi, cam = torch.from_numpy(t["batch_inds"]).to(cuda_dev), torch.from_numpy(t["cam_pos"]).to(cuda_dev)
    for name, (dth, times) in {"train": (5e-5, 10), "infer": (1e-4, 30)}.items():
        p, conv = utils.OptimizeSurfacePs(cam, rays, start.clone(), bi, sdf, RATIO, comp, conds,
                                          dthreshold=dth, athreshold=float(t["athreshold"]), w1=3.05,
                                          w2=1., times=times)
        assert p.shape == start.shape and conv.dtype == torch.bool
        assert (conv.cpu().numpy() != t["conv_" + name]).sum() <= 2
        assert np.abs(p.cpu().numpy() - t["pts_" + name]).max() < 1e-4 * 0.7  # |p| ~ 0.7
    # empty ray set
    p0, c0 = utils.OptimizeSurfacePs(cam, rays[:0], start[:0].clone(), bi[:0], sdf, RATIO, comp, conds)
    assert p0.shape == (0, 3) and c0.shape == (0,)
    # the two engines (reverse-mode sweeps = default, forward-mode tangents) agree with the
    # reference and with each other; identity deformer (BASELINE config 1) through both
    from selfreconcode_b200 import ops
    sdf_only = sdf.fused_sdf_only()
    dnet = comp.defs[0].fused(RATIO)
    lbs = comp.defs[1].lbs_state()
    lbs.set_pose(conds[1][0], conds[1][1])
    res = {}
    # identity deformer: aim the rays at the start points themselves so the problem stays local
    rays_id = torch.nn.functional.normalize(start - cam.view(1, 3), dim=1)
    for mode in ("reverse", "forward", "tc"):
        p, conv, cnt = ops.trace_surface_points(sdf_only, dnet, lbs, cam, rays, start, bi, conds[0], 5e-5,
                                                float(t["athreshold"]), 3.05, 1.0, 10, return_counters=True,
                                                mode=mode)
        assert np.abs(p.cpu().numpy() - t["pts_train"]).max() < 7e-5
        res[mode] = (p, cnt)
        pi, ci = ops.trace_surface_points(sdf_only, None, None, cam, rays_id, start, bi, None, 5e-5, 0.05,
                                          3.05, 1.0, 10, mode=mode)
        res[mode + "_id"] = pi
    assert torch.equal(res["reverse"][1], res["forward"][1]), "same active-set sizes per iteration"
    assert (res["tc"][0] - res["reverse"][0]).abs().max().item() < 7e-5   # tensor-core engine (1e-4 rel bar)
    assert (res["tc_id"] - res["reverse_id"]).abs().max().item() < 7e-5
    assert (res["reverse"][0] - res["forward"][0]).abs().max().item() < 2e-6
    assert (res["reverse_id"] - res["forward_id"]).abs().max().item() < 5e-6
    # identity deformer against the oracle
    from oracle import oracle as O
    sp = [(a.cpu(), b.cpu(), c.cpu()) for a, b, c in sdf_params(sdf)]
    po, co, _ = O.optimize_surface_ps(cam.cpu(), rays_id.cpu(), start.cpu(), bi.cpu(),
                                      lambda q: O.sdf_forward(sp, q, 6, 1.0)[0], lambda q, b: q, 5e-5, 0.05,
                                      3.05, 1.0, 10)
    assert np.abs(res["reverse_id"].cpu().numpy() - po.numpy()).max() < 7e-5


def test_seg3d_gather_scatter_match_the_torch_sequence(cuda_dev):
    """lattice -> world arithmetic of batch_eval (seg3d_lossless.py:99-101): identical bits to the
    torch op sequence; scatter: write-back, conflict mask and count."""
    from selfreconcode_b200 import ops
    g = torch.Generator().manual_seed(4)
    D, H, W = 17, 21, 15
    fD, fH, fW = 65, 81, 57
    sz, sy, sx = 4, 4, 4
    bmin, bmax = [-0.9, -1.3, -0.5], [0.9, 0.95, 0.52]
    lin = torch.randperm(D * H * W, generator=g)[:2000].sort()[0].to(cuda_dev)
    grid = torch.randn(D * H * W, generator=g).to(cuda_dev)
    calc = torch.zeros((fD, fH, fW), dtype=torch.bool, device=cuda_dev)
    pts, interp = ops.seg3d_gather(lin, (H, W), (sz, sy, sx), calc, bmin, bmax, grid)
    z, y, x = lin // (H * W), (lin // W) % H, lin % W
    coords = torch.stack([x * sx, y * sy, z * sz], dim=1)
    res = torch.tensor([fW, fH, fD], device=cuda_dev)
    step = 1.0 / res.float()
    c2 = coords.float() / res + step / 2
    lo, hi = torch.tensor(bmin, device=cuda_dev), torch.tensor(bmax, device=cuda_dev)
    want = c2 * (hi - lo) + lo
    assert torch.equal(pts, want)
    assert torch.equal(interp, grid[lin])
    ref_calc = torch.zeros_like(calc)
    ref_calc[coords[:, 2], coords[:, 1], coords[:, 0]] = True
    assert torch.equal(calc, ref_calc)
    vals = torch.randn(lin.numel(), generator=g).to(cuda_dev)
    before = grid.clone()
    conflict, ncf = ops.seg3d_scatter(lin, vals, interp, 0.05, grid)
    want_c = (interp - 0.05) * (vals - 0.05) < 0
    assert int(ncf.item()) == int(want_c.sum())
    ref_mask = torch.zeros(D * H * W, dtype=torch.bool, device=cuda_dev)
    ref_mask[lin[want_c]] = True
    assert torch.equal(conflict, ref_mask)
    before[lin] = vals
    assert torch.equal(grid, before)


def test_tc_pair_kernel_matches_single_cta_kernel(cuda_dev, monkeypatch):
    """cta_group::2 kernel vs the single-CTA kernel: same operands, same MMA terms and order."""
    import subprocess, sys, os, json
    code = (
        "import torch, json, sys; sys.path.insert(0, %r); from selfreconcode_b200 import ops; "
        "from selfreconcode_b200._lib import SR_ACT_SOFTPLUS100; torch.manual_seed(0); "
        "M=777; x=torch.randn(M,512,device='cuda'); w=torch.randn(512,512,device='cuda')/22.6; "
        "b=torch.randn(512,device='cuda')*0.01; A=ops.tc_pack_rows(x); W=ops.tc_pack_weights(w); "
        "o=ops.tc_linear(A,W,b,M,512,512,512,SR_ACT_SOFTPLUS100,want_out=True)[1]; "
        "print(json.dumps(dict(s=float(o.double().sum()), a=float(o.double().abs().sum()), m=float(o.max()))))"
    ) % helpers_root()
    outs = []
    for pair in ("1", "0"):
        env = dict(os.environ, SELFRECON_B200_TC_PAIR=pair)
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=240)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append(json.loads(r.stdout.strip().splitlines()[-1]))
    for k in outs[0]:
        assert abs(outs[0][k] - outs[1][k]) <= 1e-6 * abs(outs[1][k]), outs


def test_seg3d_lossless_vs_golden_and_mc(cuda_dev):
    dropin()
    from MCAcc import Seg3dLossless
    import MCGpu

    def query(points):
        q = points.reshape(-1, 3)
        val = q.norm(dim=1) - 0.55 + 0.08 * torch.sin(7.0 * q[:, 0]) * torch.cos(5.0 * q[:, 1]) + 0.05 * q[:, 2]
        return val.reshape(1, 1, -1)

    for name, bmin, bmax in (("seg3d.npz", [-1.0] * 3, [1.0] * 3),
                             ("seg3d_aniso.npz", [-0.9, -1.3, -0.5], [0.9, 0.9, 0.5])):
        g = golden(name)
        shape = tuple(int(v) for v in g["shape"])
        n = int(np.prod(shape))
        q_ref = np.unpackbits(g["queried"])[:n].astype(bool).reshape(shape)
        sign_ref = np.unpackbits(g["sign"])[:n].astype(bool).reshape(shape)
        ladder = [tuple(int(v) for v in r) for r in g["ladder"]]
        eng = Seg3dLossless(query_func=query, b_min=bmin, b_max=bmax, resolutions=ladder,
                            align_corners=False, balance_value=0.0, use_cuda_impl=False).to(cuda_dev)
        grid = eng.forward()
        assert tuple(grid.shape) == (1, 1) + shape
        gnp = grid[0, 0].cpu().numpy()
        assert eng.last_num_queried == q_ref.sum(), "same number of function evaluations as the reference"
        np.testing.assert_allclose(gnp[q_ref], g["values_at_queried"], atol=2e-6)
        assert np.array_equal(gnp > 0.0, sign_ref), "sign pattern (what MC consumes) identical"
        np.testing.assert_allclose(gnp.reshape(-1)[g["interp_idx"]], g["interp_val"], atol=2e-6)
        v, f = MCGpu.mc_gpu(grid[0, 0].permute(2, 1, 0).contiguous(), eng.spacing_x, eng.spacing_y,
                            eng.spacing_z, eng.bx, eng.by, eng.bz, 0.0)
        assert v.shape[0] > 100
        if name == "seg3d.npz":  # closed surface inside the box (the anisotropic box clips it)
            assert (f >= 0).all()


# ------------------------------------------------------------------------------------------------
# Tensor-core engine (tcgen05, split-BF16 operands, fp32 accumulation in TMEM)
# ------------------------------------------------------------------------------------------------
def test_tc_linear_split_bf16_matches_fp64(cuda_dev):
    from selfreconcode_b200 import ops
    from selfreconcode_b200._lib import SR_ACT_NONE, SR_ACT_SOFTPLUS100, SR_ACT_RELU
    g = torch.Generator().manual_seed(7)
    for M, K, N in ((300, 64, 512), (1000, 512, 512), (129, 192, 473)):
        x = torch.randn(M, K, generator=g).to(cuda_dev)
        w = (torch.randn(N, K, generator=g) / K ** 0.5).to(cuda_dev)
        b = (0.1 * torch.randn(N, generator=g)).to(cuda_dev)
        A = ops.tc_pack_rows(x)
        W = ops.tc_pack_weights(w)
        ref = (x.double() @ w.double().t() + b.double())
        _, out, _ = ops.tc_linear(A, W, b, M, N, K, N, SR_ACT_NONE, want_out=True)
        err = norm_err(out.cpu().numpy(), ref.cpu().numpy())
        f32 = norm_err((x @ w.t() + b).cpu().numpy(), ref.cpu().numpy())
        assert err < 1e-5, (M, K, N, err, f32)   # fp32-class accuracy (fp32 itself: ~1e-6) from six bf16 products
        # chained: hidden layer (softplus) written in the tiled layout, consumed by a second layer
        w2 = (torch.randn(3, N, generator=g) / N ** 0.5).to(cuda_dev)
        b2 = torch.zeros(3, device=cuda_dev)
        A1, _, _ = ops.tc_linear(A, W, b, M, N, K, N, SR_ACT_SOFTPLUS100, K_next=(N + 31) // 32 * 32)
        _, out2, _ = ops.tc_linear(A1, ops.tc_pack_weights(w2), b2, M, 3, (N + 31) // 32 * 32, 3, SR_ACT_NONE,
                                   want_out=True)
        h = torch.nn.functional.softplus(ref, beta=100)
        ref2 = h @ w2.double().t()
        assert norm_err(out2.cpu().numpy(), ref2.cpu().numpy()) < 1e-5
    # forward-mode tangent rows (4 rows per point: value, d/dx, d/dy, d/dz)
    P, K, N = 64, 64, 256
    x = torch.randn(P * 4, K, generator=g).to(cuda_dev)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(cuda_dev)
    b = (0.05 * torch.randn(N, generator=g)).to(cuda_dev)
    _, out, _ = ops.tc_linear(ops.tc_pack_rows(x), ops.tc_pack_weights(w), b, P * 4, N, K, N, SR_ACT_RELU, ch=4,
                              want_out=True)
    z = (x.double() @ w.double().t()).view(P, 4, N)
    zv = z[:, 0] + b.double()
    exp = torch.cat([torch.relu(zv)[:, None], (zv > 0).double()[:, None] * z[:, 1:]], 1).view(P * 4, N)
    assert norm_err(out.cpu().numpy(), exp.cpu().numpy()) < 1e-5


def test_tc_mlp_matches_ffma_engine_and_golden(cuda_dev):
    """Whole SDF / translator stacks on the tensor-core engine vs the FFMA engine vs the reference."""
    from selfreconcode_b200 import ops
    g = golden("sdf_full.npz")
    net = build_sdf_full(g).to(cuda_dev)
    pts = torch.from_numpy(g["pts"]).to(cuda_dev)
    fused = net.fused()
    fused.set_pe_weights([1.0] * 6)
    out = ops.tc_mlp_forward(fused, pts, ch=1)                      # [P, 257]
    assert rel_err(out[:, :1].cpu().numpy(), g["sdf"]) < FP_TOL
    assert rel_err(out[:, 1:].cpu().numpy(), g["feat"]) < FP_TOL
    out4 = ops.tc_mlp_forward(fused, pts, ch=4, n_out=1).view(-1, 4)  # value + d/dp
    assert rel_err(out4[:, 0].cpu().numpy(), g["sdf"].reshape(-1)) < FP_TOL
    assert rel_err(out4[:, 1:].cpu().numpy(), g["grad"]) < FP_TOL
    s, gr, _ = net.forward_fused(pts, RATIO, want_grad=True, want_feat=False)
    # engine-to-engine: the tensor core accumulates in fp32 with truncation (not round-to-nearest),
    # ~200 accumulate events per output per layer -> a small systematic offset vs the FFMA engine
    assert rel_err(out4[:, 0].cpu().numpy(), s.view(-1).cpu().numpy()) < FP_TOL
    # large ragged batch: the two engines agree point by point
    big = (torch.rand(70001, 3, generator=torch.Generator().manual_seed(3)) - 0.5).to(cuda_dev) * 1.6
    a = ops.tc_mlp_forward(net.fused_sdf_only(), big, ch=1, n_out=1).view(-1)
    b, _, _ = ops.sdf_forward(net.fused_sdf_only(), big, False, 0)
    assert (a - b).abs().max().item() < 6e-5
    # translator (ReLU, conditioning gather)
    gd = golden("deform.npz")
    tr = build_translator(gd).to(cuda_dev)
    p2 = torch.from_numpy(gd["pts"]).to(cuda_dev)
    bi = torch.from_numpy(gd["batch_inds"]).to(cuda_dev)
    dc = torch.from_numpy(gd["dcond"]).to(cuda_dev)
    off = ops.tc_mlp_forward(tr.fused(RATIO), p2, ch=1, conds=dc, batch_inds=bi)
    assert rel_err(off.cpu().numpy(), gd["offset"]) < FP_TOL


def test_tc_shade_and_render_match_ffma_engine(cuda_dev):
    from selfreconcode_b200 import ops
    g, c, gs, gr = golden("deform.npz"), golden("cardinal.npz"), golden("sdf_full.npz"), golden("render.npz")
    comp, conds = _deform_modules(g, cuda_dev)
    sdf = build_sdf_full(gs).to(cuda_dev)
    rn = build_render(gr).to(cuda_dev)
    pts = torch.from_numpy(g["pts"]).to(cuda_dev)
    bi = torch.from_numpy(g["batch_inds"]).to(cuda_dev)
    rays = torch.from_numpy(c["rays"]).to(cuda_dev)
    lbs = comp.defs[1].lbs_state()
    lbs.set_pose(conds[1][0], conds[1][1])
    full, dnet, rnet = sdf.fused(), comp.defs[0].fused(RATIO), rn.fused(RATIO)
    n, cr, rgb, dp, ok = ops.shade_and_render_tc(full, dnet, lbs, rnet, pts, rays, bi, conds[0])
    assert rel_err(cr.cpu().numpy(), c["crays"]) < FP_TOL            # reference (golden)
    assert rel_err(dp.cpu().numpy(), c["ds"]) < FP_TOL
    n2, cr2, ft, _, _ = ops.shade_geometry(full, dnet, lbs, pts, rays, bi, conds[0], nfeat=256)
    rgb2 = ops.render_forward(rnet, pts, n2, cr2, ft)
    assert rel_err(n.cpu().numpy(), n2.cpu().numpy()) < FP_TOL
    assert rel_err(rgb.cpu().numpy(), rgb2.cpu().numpy()) < 2 * FP_TOL
    assert ok.all()
