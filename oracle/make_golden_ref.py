"""TEST INFRASTRUCTURE -- fixtures that let the comparisons with the reference run without the reference.

    python oracle/make_golden_ref.py python [OUT_DIR]     (needs the reference tree, CPU)
    python oracle/make_golden_ref.py kernels [OUT_DIR]    (needs oracle/_ref/ from oracle/build.py and a B200)

OUT_DIR defaults to tests/golden/.

  ref_init.npz      the reference's own getTmpSdf / MLPTranslator initialised under fixed seeds (reference Python
                    imported on CPU through oracle/ref_shim.py): state_dict keys and a SHA-256 of every tensor
                    (tests/test_dropin_cpu.py requires bit-identical initialisation).
  ref_mc_table.npz  the 256 x 16 triangulation table parsed from the reference's MCGpu/CudaKernels.cu
                    (tests/test_oracle_c.py checks the product's packed table against it).
  ref_kernels.npz   outputs of the reference's CUDA extensions FastMinv, MCGpu, interp2x_boundary3d and
                    GridSamplerMine on the seeded inputs of tests/test_gpu_parity.py.  Outputs compared bit for bit
                    are stored as SHA-256 digests (helpers.sha256); outputs compared to a tolerance as a seeded sample
                    of 2048 elements (`<key>_idx`, `<key>_val`) plus, where the bar is relative, the mean |value|
                    of the whole output (`<key>_absmean`).
"""
import os
import re
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers  # noqa: E402

N_SAMPLE = 2048


def _sample(out, key, t, seed, absmean=False):
    flat = t.detach().cpu().numpy().reshape(-1)
    idx = np.sort(np.random.RandomState(seed).choice(flat.size, size=min(N_SAMPLE, flat.size), replace=False))
    out[key + "_idx"] = idx.astype(np.int32)
    out[key + "_val"] = flat[idx]
    if absmean:
        out[key + "_absmean"] = np.float64(np.abs(flat.astype(np.float64)).mean())


def make_python(out_dir):
    import ref_shim
    ref = ref_shim.load_reference()
    out = {}
    torch.manual_seed(0)
    sdf = ref.network.getTmpSdf("cpu", 6, bias=0.78)
    torch.manual_seed(1)
    tr = ref.Deformer.MLPTranslator(128, 6)
    for name, m in (("sdf", sdf), ("tr", tr)):
        items = sorted(m.state_dict().items())
        out[name + "_keys"] = np.array([k for k, _ in items])
        out[name + "_sha"] = np.array([helpers.sha256(v) for _, v in items])
    np.savez_compressed(os.path.join(out_dir, "ref_init.npz"), **out)
    src = open(os.path.join(ref_shim.REF_ROOT, "MCGpu", "CudaKernels.cu")).read()
    i = src.index("a2iTriangleConnectionTable[256][16]")
    rows = re.findall(r"\{([^{}]*)\}", src[src.index("{", i) + 1:src.index("};", i)])
    tab = np.array([[int(x) for x in r.split(",")] for r in rows], dtype=np.int8)
    assert tab.shape == (256, 16)
    np.savez_compressed(os.path.join(out_dir, "ref_mc_table.npz"), table=tab)
    print("ref_init: %d + %d tensors; ref_mc_table: %s" % (len(out["sdf_keys"]), len(out["tr_keys"]), tab.shape))


def make_kernels(out_dir):
    from oracle import build
    import test_gpu_parity as T
    dev = torch.device("cuda:0")
    ext = {n: build.load_ref(n) for n in build.REF_EXTS}
    missing = [n for n, m in ext.items() if m is None]
    assert not missing, "oracle/_ref/ lacks %s (python oracle/build.py)" % missing
    out = {}
    # ---- FastMinv
    ms, rows, gr = T._minv_ab_inputs()
    ms = ms.to(dev)
    b, bc = ext["FastMinv"].Fast3x3Minv(ms)
    assert (b[~bc] == 0).all()
    out["minv_mask"] = np.packbits(bc.cpu().numpy())
    out["minv_adj_err"] = np.float64(T._minv_adjugate_err(b, ms, bc.cpu().numpy()))
    inv = b[rows.to(dev)].contiguous()
    out["minv_bwd_inv"] = inv.cpu().numpy()
    out["minv_bwd"] = ext["FastMinv"].Fast3x3Minv_backward(gr.to(dev), inv).cpu().numpy()
    # ---- MCGpu (race-ordered ids: digests of the canonical form)
    for n, aniso in T.MC_AB_CASES:
        v, f = ext["MCGpu"].mc_gpu(T._test_grid(n, 100 + n, aniso).to(dev), *T.MC_AB_ARGS)
        cv, cf = T._canon(v.cpu().numpy(), f.cpu().numpy())
        out["mc%d_nv" % n], out["mc%d_nf" % n] = cv.shape[0], cf.shape[0]
        out["mc%d_v_sha" % n], out["mc%d_f_sha" % n] = helpers.sha256(cv), helpers.sha256(cf)
    # ---- interp2x_boundary3d
    x, y = T._interp_ab_inputs()
    a, ab = ext["interp2x_boundary3d"].forward(x.to(dev), 0.0)
    assert a.shape == y.shape
    out["i2x_out_sha"], out["i2x_bnd_sha"] = helpers.sha256(a), helpers.sha256(ab)
    _sample(out, "i2x_bwd", ext["interp2x_boundary3d"].backward(y.to(dev)), 1)
    # ---- GridSamplerMine
    r = ext["GridSamplerMine"]
    inp, grid, go, ggi, ggg = [t.to(dev) for t in T._grid_sampler_ab_inputs()]
    a = r.forward(inp, grid, 0, 1)
    assert a.shape == go.shape
    out["gs_fwd_sha"] = helpers.sha256(a)
    gi, gg = r.backward(inp, grid, go, 0, 1)
    _sample(out, "gs_gi", gi, 2)
    _sample(out, "gs_gg", gg, 3)
    for i, t in enumerate(r.dbackward(ggi, ggg, inp, grid, go, 0, 1)):
        _sample(out, "gs_dd%d" % i, t, 4 + i, absmean=True)
    torch.cuda.synchronize()
    np.savez_compressed(os.path.join(out_dir, "ref_kernels.npz"), **out)
    print("ref_kernels: %d arrays, device %s" % (len(out), torch.cuda.get_device_name(dev)))


if __name__ == "__main__":
    what = sys.argv[1]
    out_dir = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    {"python": make_python, "kernels": make_kernels}[what](out_dir)
