"""Shared helpers for the tests: golden loading, seeded module rebuilds, comparisons."""
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

RATIO = {"sdfRatio": 1.0, "deformerRatio": 0.8, "renderRatio": 1.0}
SMPL_PARENTS = np.array([0, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 20, 21])


def golden(name):
    return np.load(os.path.join(GOLDEN, name))


def checksum(module):
    s = a = 0.0
    for _, p in sorted(module.state_dict().items()):
        s += float(p.double().sum())
        a += float(p.double().abs().sum())
    return np.array([s, a], dtype=np.float64)


def perturb(module, scale, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in module.parameters():
            p.add_(scale * torch.randn(p.shape, generator=g))


def dropin():
    import selfreconcode_b200
    selfreconcode_b200.enable_dropin()


def build_sdf_full(g):
    """Rebuilds the full-size SDF of tests/golden/sdf_full.npz from its seed; checks the checksum."""
    dropin()
    from model.network import getTmpSdf
    torch.manual_seed(int(g["seed"]))
    net = getTmpSdf("cpu", 6, bias=float(g["bias"]))
    perturb(net, float(g["perturb"]), int(g["perturb_seed"]))
    np.testing.assert_allclose(checksum(net), g["checksum"], rtol=1e-12)
    return net


def build_sdf_small(g):
    dropin()
    from model.network import ImplicitNetwork
    net = ImplicitNetwork(16, 3, 1, [64, 64, 64, 64], geometric_init=True, bias=0.6, skip_in=[2],
                          weight_norm=True, multires=6)
    sd = {k[2:].replace("__", "."): torch.from_numpy(g[k]) for k in g.files if k.startswith("p_")}
    net.load_state_dict(sd)
    return net


def build_translator(g):
    dropin()
    from model.Deformer import MLPTranslator
    torch.manual_seed(int(g["seed"]))
    tr = MLPTranslator(128, 6)
    perturb(tr, float(g["perturb"]), int(g["perturb_seed"]))
    np.testing.assert_allclose(checksum(tr), g["checksum"], rtol=1e-12)
    return tr


def build_skinner(g):
    dropin()
    from model.Deformer import LBSkinner
    return LBSkinner(torch.from_numpy(g["ws"]), g["bmin"].tolist(), g["bmax"].tolist(),
                     torch.from_numpy(g["Js"]), SMPL_PARENTS, init_pose=g["apose"])


def build_render(g):
    dropin()
    from model.RenderNet import RenderingNetwork_view_norm
    torch.manual_seed(int(g["seed"]))
    rn = RenderingNetwork_view_norm(256, 'idr', 9, 3, [512] * 4, weight_norm=True, multires_v=4,
                                    multires_n=0)
    np.testing.assert_allclose(checksum(rn), g["checksum"], rtol=1e-12)
    return rn


def sdf_params(net):
    """(v, g, b) per layer for oracle.sdf_forward from a (drop-in or reference) ImplicitNetwork."""
    out = []
    for l in range(net.num_layers - 1):
        lin = getattr(net, "lin" + str(l))
        out.append((lin.weight_v.detach(), lin.weight_g.detach(), lin.bias.detach()))
    return out


def plain_params(net):
    return [(getattr(net, "lin" + str(l)).weight.detach(), getattr(net, "lin" + str(l)).bias.detach())
            for l in range(net.num_layers - 1)]


def wn_params(net):
    out = []
    for l in range(net.num_layers - 1):
        lin = getattr(net, "lin" + str(l))
        out.append((lin.weight_v.detach(), lin.weight_g.detach(), lin.bias.detach()))
    return out


def norm_err(a, b):
    """max |a-b| / max |b| (norm-wise; round 1's bar, kept for quantities whose elements cancel)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def elem_err(a, b):
    """ELEMENTWISE relative error with a floor: max_i |a_i - b_i| / (|b_i| + mean|b|).  `< 1e-4` reads
    |a-b| <= 1e-4*|b| + 1e-4*mean|b| for every element -- the north star's "1e-4 rel fp32" with the floor
    an fp32 evaluation needs for elements that cancel to ~0."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if b.size == 0:
        return 0.0
    floor = max(float(np.abs(b).mean()), 1e-30)
    return float((np.abs(a - b) / (np.abs(b) + floor)).max())


rel_err = elem_err   # the parity bar of every floating-point test


def sha256(a):
    """Digest of an array's dtype, shape and bytes: a bit-exact comparison against a stored fixture without storing
    the array itself."""
    import hashlib
    a = np.ascontiguousarray(a.detach().cpu().numpy() if torch.is_tensor(a) else a)
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def mc_tri_table():
    """The 256x16 triangulation as an int array, decoded from the product's packed table so the
    C oracle and the kernel are checked against one another AND (test_mc_tables) against the
    algebraic properties of the classic table."""
    import re
    src = open(os.path.join(ROOT, "selfreconcode_b200", "csrc", "marching_cubes.cu")).read()
    body = src[src.index("kTriPacked[256]"):]
    body = body[:body.index("};")]
    vals = [int(x, 16) for x in re.findall(r"0x([0-9a-f]{16})ULL", body)]
    assert len(vals) == 256
    tab = -np.ones((256, 16), dtype=np.int32)
    for c, v in enumerate(vals):
        for k in range(16):
            nib = (v >> (4 * k)) & 0xF
            tab[c, k] = -1 if nib == 0xF else nib
    return tab
