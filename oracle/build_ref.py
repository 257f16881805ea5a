"""Build the reference's OWN native CUDA ops (unmodified sources, read in place from the reference checkout) into oracle/_ref/,
where `python -m oracle.make_golden ref_kernels` runs them on a GPU and records the outputs that tests/test_ref_kernels_gpu.py
compares the product's kernels against (SURVEY.md section 8c).

    python -m oracle.build_ref            # -> oracle/_ref/{ref_ctc2d,ref_deform_conv,ref_deform_pool}.so

TEST INFRASTRUCTURE, never on the product path.  Nothing is copied from the reference: nvcc / g++ read the sources in
place; the only additions are the force-included oracle/ref_shim/compat.h (AT_CHECK -> TORCH_CHECK, the
DeprecatedTypeProperties overload AT_DISPATCH needs) and an empty <THC/THC.h>.  The build needs the reference checkout
(MEGREADER_REFERENCE) and the torch headers; oracle/_ref/ is git-ignored.  load(name) returns the pybind module or None when
the .so is absent.
"""
import importlib.util
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")
SHIM = os.path.join(HERE, "ref_shim")
REF = os.environ.get("MEGREADER_REFERENCE", "/root/reference")

# The reference launches its 2D-CTC kernels with 1024 threads per block (ctc2d_cuda_kernel.cu:16 CUDA_NUM_THREADS); the
# fp64 instantiations need more than 64 registers per thread when compiled for sm_100 and then fail to launch ("too many
# resources requested").  Capping the register count is a compiler flag, not a source change.
EXTRA_NVCC = {"ref_ctc2d": ["--maxrregcount=64"]}

OPS = {
    # name: sources relative to the reference root
    "ref_ctc2d": ["ops/ctc_2d/csrc/ctc2d.cpp", "ops/ctc_2d/csrc/cuda/ctc2d_cuda.cu",
                  "ops/ctc_2d/csrc/cuda/ctc2d_cuda_kernel.cu"],
    "ref_deform_conv": ["assets/ops/dcn/src/deform_conv_cuda.cpp", "assets/ops/dcn/src/deform_conv_cuda_kernel.cu"],
    "ref_deform_pool": ["assets/ops/dcn/src/deform_pool_cuda.cpp", "assets/ops/dcn/src/deform_pool_cuda_kernel.cu"],
}


def so_path(name):
    return os.path.join(OUT, name + ".so")


def build(verbose=False):
    """Compile every op whose .so is missing.  Returns {name: path}; raises if the reference tree is absent."""
    if not os.path.isdir(REF):
        raise RuntimeError("reference tree %s not present: oracle/_ref can only be built in the build container" % REF)
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")
    from torch.utils import cpp_extension
    compat = os.path.join(SHIM, "compat.h")
    built = {}
    for name, rel in OPS.items():
        dst = so_path(name)
        srcs = [os.path.join(REF, r) for r in rel]
        if os.path.exists(dst) and all(os.path.getmtime(dst) >= os.path.getmtime(s) for s in srcs + [compat]):
            built[name] = dst
            continue
        bdir = os.path.join(OUT, "_build_" + name)
        os.makedirs(bdir, exist_ok=True)
        inc = [SHIM, os.path.join(REF, os.path.dirname(rel[0]))]
        cpp_extension.load(name=name, sources=srcs, extra_include_paths=inc, build_directory=bdir, verbose=verbose,
                           extra_cflags=["-O2", "-DWITH_CUDA", "-include", compat, "-w"],
                           extra_cuda_cflags=["-O2", "-DWITH_CUDA", "-include", compat, "-w", "-DCUDA_HAS_FP16=1",
                                              "-D__CUDA_NO_HALF_OPERATORS__", "-D__CUDA_NO_HALF_CONVERSIONS__",
                                              "-D__CUDA_NO_HALF2_OPERATORS__"] + EXTRA_NVCC.get(name, []),
                           is_python_module=False)
        os.replace(os.path.join(bdir, name + ".so"), dst)
        built[name] = dst
    return built


def load(name):
    """Import a prebuilt reference op (pybind module), or None when it was not built."""
    path = so_path(name)
    if not os.path.exists(path):
        return None
    import torch  # noqa: F401  (the extension links against libtorch)
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    for k, v in build(verbose="-v" in sys.argv).items():
        print(k, v)
