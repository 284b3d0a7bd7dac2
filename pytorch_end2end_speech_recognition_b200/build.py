"""In-tree build of the CUDA library (sm_100a only) with plain nvcc.

The C-ABI library has no PyTorch dependency, so it is compiled directly:
    nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -shared -Xcompiler -fPIC ...
The result lives next to the sources (``lib/libb200ctc.so``): it is git-ignored but
travels to the GPU box with the repo snapshot.
"""

import os
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_DIR = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "lib")
LIB_DEFAULT = os.path.join(LIB_DIR, "libb200ctc.so")       # what build_library() builds
LIB_PATH = os.environ.get("B200CTC_LIB") or LIB_DEFAULT    # what the package loads; B200CTC_LIB: a developer variant

SOURCES = ["api.cu", "plan.cu", "softmax_rows.cu", "lattice.cu", "narrow_grads.cu", "greedy.cu", "beam.cu", "eval.cu",
           "ngram_lm.cu"]

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC",
    "-Xcompiler", "-fvisibility=hidden",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    cuda_home = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    cand = os.path.join(cuda_home, "bin", "nvcc")
    return cand if os.path.exists(cand) else "nvcc"


def _source_hash(deps, flags):
    """Content hash of everything the library is built from (sources, header, flags): file times do not
    survive the snapshot copy to the GPU box, contents do."""
    import hashlib
    h = hashlib.sha1(" ".join(flags).encode())
    for d in sorted(deps):
        h.update(os.path.basename(d).encode())
        with open(d, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _stale(target, deps, flags=()):
    if not os.path.exists(target):
        return True
    try:
        with open(target + ".srchash") as f:
            return f.read().strip() != _source_hash(deps, flags)
    except OSError:
        return True


def _link(objs, out):
    # the link step names the architecture too: without it nvcc adds an (empty) sm_52 device-link stub.  Every
    # build, variants included, is named libb200ctc.so (SONAME): the extension's dependency on libb200ctc.so then
    # resolves to whichever copy the process loaded first, so B200CTC_LIB redirects the whole process.
    subprocess.run([_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xlinker", "-soname=libb200ctc.so",
                    "-o", out] + objs + ["-Xcompiler", "-fPIC"], check=True)


def build_library(force=False, verbose=False, extra_flags=(), lib_path=None):
    """Compile csrc/*.cu into lib/libb200ctc.so (no-op when up to date).  ``extra_flags`` /
    ``lib_path`` build a developer variant next to it (tools/trace_lattice.py: -DB200CTC_TRACE).
    B200CTC_LIB never names the output: it selects what is loaded, not what is built."""
    os.makedirs(LIB_DIR, exist_ok=True)
    if lib_path is not None:
        return _build_variant(list(extra_flags), lib_path, verbose)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(REPO_DIR, "include", "b200ctc.h")]
    if not force and not _stale(LIB_DEFAULT, deps, NVCC_FLAGS):
        return LIB_DEFAULT
    objs = []
    for src in SOURCES:
        obj = os.path.join(LIB_DIR, src.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + ["-I", os.path.join(REPO_DIR, "include"), "-I", CSRC,
                                        "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), file=sys.stderr)
        subprocess.run(cmd, check=True)
        objs.append(obj)
    _link(objs, LIB_DEFAULT)
    with open(LIB_DEFAULT + ".srchash", "w") as f:
        f.write(_source_hash(deps, NVCC_FLAGS))
    return LIB_DEFAULT


def _build_variant(extra_flags, lib_path, verbose):
    objs = []
    tag = os.path.basename(lib_path).replace(".so", "")
    for src in SOURCES:
        obj = os.path.join(LIB_DIR, "%s_%s" % (tag, src.replace(".cu", ".o")))
        cmd = [_nvcc()] + NVCC_FLAGS + extra_flags + ["-I", os.path.join(REPO_DIR, "include"), "-I", CSRC,
                                                      "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.run(cmd, check=True)
        objs.append(obj)
    _link(objs, lib_path)
    return lib_path


EXT_NAME = "b200ctc_torch"
EXT_DIR = os.path.join(LIB_DIR, "torch_ext")


def extension_path():
    import sysconfig
    return os.path.join(EXT_DIR, EXT_NAME + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))


def build_extension(force=False, verbose=False):
    """Compile csrc/torch_binding.cpp -- the thin PyTorch C++ extension over the C ABI -- in-tree with the host
    compiler against this interpreter's torch headers, linked to the in-tree lib/libb200ctc.so (rpath $ORIGIN/..).
    Returns the path of the extension module; a no-op when its source hash is unchanged."""
    import sysconfig
    import torch
    build_library()
    os.makedirs(EXT_DIR, exist_ok=True)
    src = os.path.join(CSRC, "torch_binding.cpp")
    out = extension_path()
    deps = [src, os.path.join(REPO_DIR, "include", "b200ctc.h")]
    flags = ["torch=" + torch.__version__, "py=" + sys.version.split()[0]]
    if not force and not _stale(out, deps, flags):
        return out
    from torch.utils import cpp_extension
    cuda_home = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    inc = ["-I" + p for p in cpp_extension.include_paths()] + ["-I" + os.path.join(cuda_home, "include"),
           "-I" + sysconfig.get_paths()["include"], "-I" + os.path.join(REPO_DIR, "include")]
    torch_lib = os.path.join(os.path.dirname(torch.__file__), "lib")
    abi = "-D_GLIBCXX_USE_CXX11_ABI=%d" % int(torch._C._GLIBCXX_USE_CXX11_ABI)
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", abi, "-DTORCH_EXTENSION_NAME=" + EXT_NAME,
           "-DTORCH_API_INCLUDE_EXTENSION_H", src, "-o", out] + inc + [
           "-L" + LIB_DIR, "-lb200ctc", "-Wl,-rpath,$ORIGIN/..",
           "-L" + torch_lib, "-ltorch", "-ltorch_cpu", "-ltorch_cuda", "-lc10", "-lc10_cuda", "-ltorch_python",
           "-Wl,-rpath," + torch_lib, "-L" + os.path.join(cuda_home, "lib64"), "-lcudart"]
    if verbose:
        print(" ".join(cmd), file=sys.stderr)
    subprocess.run(cmd, check=True)
    with open(out + ".srchash", "w") as f:
        f.write(_source_hash(deps, flags))
    return out


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
    if "--ext" in sys.argv:
        print(build_extension(force="--force" in sys.argv, verbose="-v" in sys.argv))
