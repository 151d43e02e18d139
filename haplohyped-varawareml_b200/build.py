"""In-tree build of the native pieces (no JIT cache: the built .so files travel with the repo).

  csrc/*.cu            -> libhaplo_b200.so      (nvcc, sm_100a only, -lineinfo)
  csrc/parse_vcf_pybind.cpp -> parse_vcf.<abi>.so   (the reference's module name, cpp/parse_vcf.cpp:116)
"""
from __future__ import annotations

import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
OBJ = os.path.join(HERE, "_obj")
LIB = os.path.join(HERE, "libhaplo_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CU_SOURCES = ["hb_tokenize.cu", "hb_sites.cu", "hb_walk.cu", "hb_gt.cu", "hb_inflate.cu", "hb_hap.cu", "hb_synth.cu", "hb_api.cu",
              "hb_store.cu", "hb_bcf.cu", "hb_tabix.cu", "hb_index.cu"]


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        raise RuntimeError("native build failed: " + cmd[0])
    return r.stdout + r.stderr


def pybind_module_path() -> str:
    return os.path.join(HERE, "parse_vcf" + sysconfig.get_config_var("EXT_SUFFIX"))


def build_all(verbose: bool = False, force: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(ROOT, "include", "haplo_b200.h"))
    objs = []
    for src in CU_SOURCES:
        s = os.path.join(CSRC, src)
        if not os.path.exists(s):
            continue
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or _newer(o, [s] + headers):
            out = _run([NVCC, *ARCH, "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC,-O3", "-Xptxas", "-v",
                        "-c", s, "-o", o])
            if verbose:
                print(out)
        objs.append(o)
    if force or _newer(LIB, objs):
        _run([NVCC, *ARCH, "-shared", "-o", LIB, *objs, "-lz", "-lpthread"])
    mod = pybind_module_path()
    src = os.path.join(CSRC, "parse_vcf_pybind.cpp")
    if os.path.exists(src) and (force or _newer(mod, [src, LIB] + headers)):
        import pybind11
        _run(["g++", "-O2", "-shared", "-fPIC", "-std=c++17", "-I" + pybind11.get_include(),
              "-I" + sysconfig.get_paths()["include"], "-I" + os.path.join(ROOT, "include"), src, "-o", mod,
              "-L" + HERE, "-lhaplo_b200", "-Wl,-rpath,$ORIGIN"])
    return LIB


if __name__ == "__main__":
    print(build_all(verbose="-v" in sys.argv, force="-f" in sys.argv))
