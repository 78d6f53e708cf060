"""CPU: the C restatement (oracle/oracle_c.c) against independent references -- torch ops with the
same semantics, algebraic properties, and the reference's own triangulation table (stored under tests/golden/)."""
import numpy as np
import torch

from helpers import golden, mc_tri_table
from oracle import c_api


def test_minv_property_and_mask():
    g = torch.Generator().manual_seed(0)
    ms = torch.randn(10000, 3, 3, generator=g)      # the size of FastMinv/check.py:7
    ms[::50] *= 1e-2
    inv, chk = c_api.minv3x3(ms.numpy())
    det = torch.linalg.det(ms.double()).abs().numpy()
    safe = np.abs(det - 1e-4) > 1e-6
    assert np.array_equal(chk[safe], (det >= 1e-4)[safe])
    assert (inv[~chk] == 0).all()
    good = chk & (det > 1e-2)
    err = np.linalg.norm(inv[good].astype(np.float64) @ ms.numpy()[good].astype(np.float64) - np.eye(3), axis=(1, 2))
    assert err.max() < 1e-3
    gr = torch.randn(100, 3, 3, generator=g).numpy()
    out = c_api.minv3x3_bwd(gr, inv[:100])
    ref = -(np.transpose(inv[:100], (0, 2, 1)) @ gr @ np.transpose(inv[:100], (0, 2, 1)))
    np.testing.assert_allclose(out, ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())


def test_minv_backward_is_the_vjp_of_inverse():
    m = torch.randn(20, 3, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(1)).requires_grad_(True)
    inv = torch.linalg.inv(m)
    go = torch.randn(20, 3, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(2))
    (gm,) = torch.autograd.grad(inv, m, go)
    out = c_api.minv3x3_bwd(go.float().numpy(), inv.detach().float().numpy())
    np.testing.assert_allclose(out, gm.numpy(), rtol=1e-3, atol=1e-3 * np.abs(gm.numpy()).max())


def test_interp2x_matches_torch_interpolate():
    g = torch.Generator().manual_seed(3)
    for shape in ((2, 3, 4), (9, 9, 9), (15, 21, 9)):
        x = torch.randn(*shape, generator=g)
        out, bnd = c_api.interp2x3d(x.numpy(), 0.2)
        size = tuple(2 * s - 1 for s in shape)
        ref = torch.nn.functional.interpolate(x[None, None], size=size, mode="trilinear", align_corners=True)[0, 0]
        np.testing.assert_allclose(out, ref.numpy(), atol=1e-6)
        valid = torch.nn.functional.interpolate((x > 0.2).float()[None, None], size=size, mode="trilinear",
                                                align_corners=True)[0, 0]
        assert np.array_equal(bnd, ((valid > 0) & (valid < 1)).numpy())   # seg3d_lossless.py:273-282


def test_grid_sample_matches_torch_and_clips_at_border():
    g = torch.Generator().manual_seed(4)
    inp = torch.rand(24, 7, 13, 9, generator=g)
    grid = (torch.rand(5000, 3, generator=g) - 0.5) * 2.4
    out, cidx = c_api.grid_sample3d(inp.numpy(), grid.numpy())
    ref = torch.nn.functional.grid_sample(inp[None], grid.view(1, 1, 1, -1, 3), mode="bilinear",
                                          padding_mode="border", align_corners=False).view(24, -1)
    np.testing.assert_allclose(out, ref.numpy(), atol=1e-6)
    assert cidx[:, 0].min() >= 0 and cidx[:, 0].max() <= 8
    assert cidx[:, 1].max() <= 12 and cidx[:, 2].max() <= 6
    # indices equal floor of the clipped un-normalised coordinate computed in float64
    x = np.clip(((grid[:, 0].double().numpy() + 1) * 9 - 1) / 2, 0, 8)
    far = np.abs(x - np.round(x)) > 1e-4
    assert np.array_equal(cidx[far, 0], np.floor(x[far]).astype(np.int32))


def _sphere(n, shape=None):
    shape = shape or (n, n, n)
    ax = [np.linspace(-1, 1, s, dtype=np.float32) for s in shape]
    xx, yy, zz = np.meshgrid(*ax, indexing="ij")
    return (np.sqrt(xx * xx + yy * yy + zz * zz) - 0.63 + 0.05 * np.sin(5 * xx) * np.cos(4 * yy)).astype(np.float32)


def test_mc_closed_surface_properties():
    tt = mc_tri_table()
    for shape in ((17, 17, 17), (24, 31, 19)):
        sdf = _sphere(0, shape)
        v, f = c_api.marching_cubes(sdf, tt, 0.0, (0.1, 0.2, 0.3), (1.0, 2.0, 3.0))
        assert f.min() >= 0 and f.max() == len(v) - 1
        e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
        key = np.minimum(e[:, 0], e[:, 1]) * len(v) + np.maximum(e[:, 0], e[:, 1])
        _, cnt = np.unique(key, return_counts=True)
        assert (cnt == 2).all()
        assert len(v) - len(cnt) + len(f) == 2
        # directed edges appear once each way -> consistently oriented
        dkey = e[:, 0] * len(v) + e[:, 1]
        assert len(np.unique(dkey)) == len(dkey)
        # every vertex sits on a grid edge: exactly one fractional coordinate (grid units)
        gu = (v - np.array([1.0, 2.0, 3.0], np.float32)) / np.array([0.1, 0.2, 0.3], np.float32)
        frac = np.abs(gu - np.round(gu)) > 1e-3
        assert (frac.sum(1) <= 1).all()
        # the reversed winding (CudaKernels.cu:492-505) makes normals point out of the solid
        tri = v[f]
        nrm = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
        ctr = tri.mean(1) - (np.array([1.0, 2.0, 3.0]) + 0.5 * (np.array(shape) - 1) * np.array([0.1, 0.2, 0.3]))
        assert ((nrm * ctr).sum(1) > 0).mean() > 0.95


def test_mc_boundary_layer_gives_minus_one():
    sdf = _sphere(12)
    sdf[-1, :, :] = -1.0   # inside region touches the +x boundary layer
    v, f = c_api.marching_cubes(sdf, mc_tri_table())
    assert (f == -1).any()


def test_packed_table_matches_reference_source_when_available():
    """The reference's MCGpu/CudaKernels.cu table, stored in tests/golden/ref_mc_table.npz."""
    tab = golden("ref_mc_table.npz")["table"].astype(np.int32)
    assert tab.shape == (256, 16) and np.array_equal(tab, mc_tri_table())
