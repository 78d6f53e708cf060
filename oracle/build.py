"""TEST INFRASTRUCTURE -- builds the checker's native pieces.

  build_c()    gcc: oracle/oracle_c.c -> oracle/liboracle_c.so  (CPU restatement, bit-level ops)
  build_ref()  nvcc/g++ through torch.utils.cpp_extension: the reference's OWN CUDA extensions,
               compiled from the sources where they lie under /root/reference, outputs only
               into oracle/_ref/ (git-ignored).  They are the "kernel to beat" (tools/ref_ab_bench.py) and
               the source of the recorded parity fixture tests/golden/ref_kernels.npz (oracle/make_golden_ref.py).
               GridSamplerMine needs `input.type()` -> `input.scalar_type()` at
               MCAcc/cuda/GridSamplerMineKernel.cu:931,963,1001 for torch 2.x; the patch is
               applied to a temporary copy under /tmp, never to the repo or the reference.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
REF_OUT = os.path.join(HERE, "_ref")


def build_c(force=False):
    src = os.path.join(HERE, "oracle_c.c")
    out = os.path.join(HERE, "liboracle_c.so")
    if not force and os.path.exists(out) and os.path.getmtime(out) >= os.path.getmtime(src):
        return out
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", src, "-o", out, "-lm"])
    return out


REF_EXTS = {
    "FastMinv": ("FastMinv", ["M3x3Inv.cpp", "Matrix3x3InvKernels.cu"]),
    "MCGpu": ("MCGpu", ["MCGpu.cpp", "CudaKernels.cu"]),
    "interp2x_boundary3d": ("MCAcc/cuda", ["interp2x_boundary3d.cpp", "interp2x_boundary3d_kernel.cu"]),
    "GridSamplerMine": ("MCAcc/cuda", ["GridSamplerMine.cpp", "GridSamplerMineKernel.cu"]),
}


def build_ref(verbose=False):
    """Returns {name: path-to-.so}.  No-op (returns what exists) when /root/reference is absent."""
    os.makedirs(REF_OUT, exist_ok=True)
    have = {n: os.path.join(REF_OUT, n + ".so") for n in REF_EXTS
            if os.path.exists(os.path.join(REF_OUT, n + ".so"))}
    if not os.path.isdir(REF) or len(have) == len(REF_EXTS):
        return have
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")
    from torch.utils import cpp_extension
    for name, (sub, files) in REF_EXTS.items():
        if name in have:
            continue
        srcdir = os.path.join(REF, sub)
        srcs = [os.path.join(srcdir, f) for f in files]
        if name == "GridSamplerMine":
            tmp = "/tmp/_ref_gridsampler_src"
            shutil.rmtree(tmp, ignore_errors=True)
            os.makedirs(tmp)
            srcs = []
            for f in files:
                txt = open(os.path.join(srcdir, f)).read()
                if f.endswith(".cu"):
                    txt = txt.replace("AT_DISPATCH_FLOATING_TYPES_AND_HALF(input.type(),",
                                      "AT_DISPATCH_FLOATING_TYPES_AND_HALF(input.scalar_type(),")
                dst = os.path.join(tmp, f)
                open(dst, "w").write(txt)
                srcs.append(dst)
        bdir = os.path.join("/tmp", "_ref_build_" + name)
        os.makedirs(bdir, exist_ok=True)
        try:
            cpp_extension.load(name=name, sources=srcs, build_directory=bdir, verbose=verbose,
                               extra_include_paths=[srcdir], is_python_module=False,
                               extra_cuda_cflags=["-gencode", "arch=compute_100a,code=sm_100a", "-O3"],
                               with_cuda=True)
            shutil.copy(os.path.join(bdir, name + ".so"), os.path.join(REF_OUT, name + ".so"))
            have[name] = os.path.join(REF_OUT, name + ".so")
        except Exception as e:  # unbuildable here -> say so
            sys.stderr.write("[oracle/_ref] could not build %s: %s\n" % (name, str(e)[:400]))
    return have


def load_ref(name):
    """Imports a built reference extension from oracle/_ref (GPU box or here)."""
    import importlib.util
    import torch  # noqa: F401  (the extension links against libtorch)
    path = os.path.join(REF_OUT, name + ".so")
    if not os.path.exists(path):
        return None
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    print(build_c(force=True))
    print(build_ref(verbose="-v" in sys.argv))
