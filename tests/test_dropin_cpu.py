"""CPU: host-side behaviour of the drop-in modules -- names, state_dict keys, initialisation
identical to the reference, and loud failure without a GPU (no CPU fallback)."""
import numpy as np
import pytest
import torch

from helpers import dropin, golden, sha256


def test_import_surface():
    dropin()
    import FastMinv, MCGpu, GridSamplerMine, interp2x_boundary3d, interp2x_boundary2d  # noqa
    import MCAcc, utils, model  # noqa
    assert callable(FastMinv.Fast3x3Minv) and callable(FastMinv.Fast3x3Minv_backward)
    assert callable(MCGpu.mc_gpu) and callable(MCGpu.mc_init)
    for m in (GridSamplerMine,):
        assert callable(m.forward) and callable(m.backward) and callable(m.dbackward)
    assert callable(interp2x_boundary3d.forward) and callable(interp2x_boundary3d.backward)
    for name in ("Seg3dLossless", "create_grid3D", "GridSamplerMine3dFunction"):
        assert hasattr(MCAcc, name)
    for name in ("OptimizeSurfacePs", "FindSurfacePs", "compute_Jacobian", "compute_cardinal_rays",
                 "compute_deformed_normals", "FastDiff3x3MinvFunction", "annealing_weights",
                 "sample_points", "GMRobustError", "quat2mat", "compute_netRender_color"):
        assert hasattr(utils, name), name
    for name in ("getTmpSdf", "ImplicitNetwork", "MLPTranslator", "LBSkinner", "CompositeDeformer",
                 "RenderingNetwork_view_norm"):
        assert hasattr(model, name), name


def test_state_dict_keys_follow_the_reference():
    dropin()
    from model.network import getTmpSdf
    from model.Deformer import MLPTranslator
    from model.RenderNet import RenderingNetwork_view_norm
    sdf = getTmpSdf("cpu", 6)
    keys = set(sdf.state_dict().keys())
    assert keys == {"lin%d.%s" % (l, k) for l in range(9) for k in ("bias", "weight_g", "weight_v")}
    assert sdf.lin3.weight_v.shape == (473, 512) and sdf.lin4.weight_v.shape == (512, 512)
    assert sdf.lin8.weight_v.shape == (257, 512) and sdf.lin0.weight_v.shape == (512, 39)
    tr = MLPTranslator(128, 6)
    assert set(tr.state_dict().keys()) == {"lin%d.%s" % (l, k) for l in range(5) for k in ("bias", "weight")}
    assert tr.lin0.weight.shape == (512, 167)
    rn = RenderingNetwork_view_norm(256, 'idr', 9, 3, [512] * 4, multires_v=4)
    assert rn.lin0.weight_v.shape == (512, 289)
    n_sdf = sum(p.numel() for p in sdf.parameters())
    n_tr = sum(p.numel() for p in tr.parameters())
    n_rn = sum(p.numel() for p in rn.parameters())
    assert (n_sdf, n_tr, n_rn) == (1975220, 875523, 940038)   # SURVEY.md section 8


def test_no_cpu_fallback():
    dropin()
    from model.network import getTmpSdf
    import FastMinv, MCGpu
    sdf = getTmpSdf("cpu", 6)
    with pytest.raises(RuntimeError):
        sdf(torch.zeros(4, 3), 1.0)
    with pytest.raises(RuntimeError):
        FastMinv.Fast3x3Minv(torch.eye(3).view(1, 3, 3))
    with pytest.raises(RuntimeError):
        MCGpu.mc_gpu(torch.zeros(4, 4, 4))


def test_initialisation_is_identical_to_the_reference_classes():
    """Against digests of the reference's own getTmpSdf / MLPTranslator under the same seeds
    (tests/golden/ref_init.npz, oracle/make_golden_ref.py)."""
    from selfreconcode_b200 import synth  # drop-in classes under their package path
    ref = golden("ref_init.npz")
    torch.manual_seed(0)
    sdf = synth.ImplicitNetwork(256, 3, 1, [512] * 8, geometric_init=True, bias=0.78, skip_in=[4],
                                weight_norm=True, multires=6)
    torch.manual_seed(1)
    tr = synth.MLPTranslator(128, 6)
    for name, m in (("sdf", sdf), ("tr", tr)):
        items = sorted(m.state_dict().items())
        assert [k for k, _ in items] == list(ref[name + "_keys"])
        for (k, v), want in zip(items, ref[name + "_sha"]):
            assert sha256(v) == want, k


def test_synthetic_workload_is_reproducible():
    from selfreconcode_b200 import synth
    cam = synth.camera(128, 128)
    assert torch.allclose(cam["cam_pos"], torch.tensor([0.0, 0.0, -2.5]))
    rows, cols, pts = synth.sphere_pixels(cam, 0.6)
    assert 2500 < rows.numel() < 3500 and torch.allclose(pts.norm(dim=1), torch.full((pts.shape[0],), 0.6), atol=1e-5)
    cam512 = synth.camera(512, 512)
    r2, _, _ = synth.sphere_pixels(cam512, 0.6)
    assert 45000 < r2.numel() < 55000          # ~19% of a 512^2 frame (SURVEY.md 8d)
    assert 0.005 < synth.ang_threshold(cam512, 0.5) < 0.06
    p1 = synth.make_frame_params(3, 2)
    p2 = synth.make_frame_params(3, 2)
    assert all(torch.equal(a, b) for a, b in zip(p1, p2))
    sk = synth.make_skinner(resolution=(9, 13, 7))
    assert sk.ws.shape == (1, 24, 7, 13, 9) and torch.allclose(sk.ws.sum(1), torch.ones(1, 7, 13, 9), atol=1e-5)
    assert sk.init_pose.shape == (24, 4, 4)
