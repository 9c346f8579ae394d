"""Build the torch/pybind layer (di_hpc_b200/csrc_torch/*.cpp) in-tree as ``di_hpc_b200/_lib/hpc_rl_utils_b200*.so``.
It contains no kernels and links against libhpc_rll_b200.so (rpath $ORIGIN):
  ext.cpp       list-of-tensor host work of the padding ops + the reference's 11 padding binding names
  fast_ops.cpp  C++ ``torch::autograd::Function`` per op -- what the nn.Modules of hpc_rll.rl_utils call
  legacy.cpp    the reference's 19 hot-path ``hpc_rl_utils`` binding names (tensor-list signatures)
  network.cpp   the reference's ``hpc_torch_utils_network`` ScatterConnection names, in the submodule ``_network``
The top-level packages ``hpc_rl_utils`` and ``hpc_torch_utils_network`` re-export this module (and its ``_network``
submodule) under the reference's names.

    python -m di_hpc_b200.build_torch_ext
"""
import glob
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
SRC_DIR = os.path.join(HERE, "csrc_torch")
SRCS = [os.path.join(SRC_DIR, f) for f in ("ext.cpp", "fast_ops.cpp", "legacy.cpp", "network.cpp")]
OBJ_DIR = os.path.join(HERE, "_lib", "obj")
OUT_DIR = os.path.join(HERE, "_lib")
NAME = "hpc_rl_utils_b200"


def target():
    return os.path.join(OUT_DIR, NAME + sysconfig.get_config_var("EXT_SUFFIX"))


def build(force: bool = False) -> str:
    import concurrent.futures as cf
    from . import build as core
    lib = core.build()
    out = target()
    hdrs = [os.path.join(SRC_DIR, "common.h"), os.path.join(os.path.dirname(HERE), "include", "hpc_rll_b200.h")]
    hdr_m = max(os.path.getmtime(h) for h in hdrs)
    os.makedirs(OBJ_DIR, exist_ok=True)
    objs = [os.path.join(OBJ_DIR, "torch_" + os.path.basename(s)[:-4] + ".o") for s in SRCS]
    stale = [(s, o) for s, o in zip(SRCS, objs)
             if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hdr_m)]
    if not stale and os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(o) for o in objs):
        return out
    import torch
    from torch.utils import cpp_extension as ce
    inc = ce.include_paths(device_type="cuda") + [os.path.join(os.path.dirname(HERE), "include"),
                                                  sysconfig.get_paths()["include"]]
    libdirs = ce.library_paths(device_type="cuda")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    flags = ["-O2", "-std=c++17", "-fPIC", "-DTORCH_EXTENSION_NAME=" + NAME, "-DTORCH_API_INCLUDE_EXTENSION_H",
             "-D_GLIBCXX_USE_CXX11_ABI=%d" % int(torch._C._GLIBCXX_USE_CXX11_ABI)] + ["-I" + i for i in inc]

    def compile_one(so):
        r = subprocess.run([cxx] + flags + ["-c", so[0], "-o", so[1]], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("compiling %s failed:\n%s\n%s" % (so[0], r.stdout[-3000:], r.stderr[-8000:]))

    if stale:
        with cf.ThreadPoolExecutor(max_workers=len(stale)) as ex:
            list(ex.map(compile_one, stale))
    cmd = [cxx, "-shared"] + objs + ["-o", out]
    cmd += ["-L" + d for d in libdirs] + ["-L" + OUT_DIR]
    cmd += ["-lc10", "-lc10_cuda", "-ltorch_cpu", "-ltorch_cuda", "-ltorch", "-ltorch_python", "-lhpc_rll_b200",
            "-Wl,-rpath,$ORIGIN"] + ["-Wl,-rpath," + d for d in libdirs]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("linking %s failed:\n%s\n%s" % (NAME, r.stdout[-3000:], r.stderr[-6000:]))
    assert os.path.exists(lib)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
