"""Build recipe of lib/libbnbp.so (hand-written sm_100a kernels + the C ABI).  In-tree, so the
built library travels to the GPU box with the repository snapshot.  The sweep kernel family is
instantiated one (T, VEC, RMAX) per translation unit and compiled in parallel."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
# BNBP_BUILD_TAG: an alternative build next to the product library (kernel-tuning A/B runs pick it with BNBP_LIB)
_TAG = os.environ.get("BNBP_BUILD_TAG", "")
OBJDIR = os.path.join(LIBDIR, "obj" + ("_" + _TAG if _TAG else ""))
LIB = os.path.join(LIBDIR, "libbnbp" + ("_" + _TAG if _TAG else "") + ".so")
SPEC_SRC = os.path.join(CSRC, "bnbp_spec.cuh")           # compiled at run time by NVRTC ...
SPEC_EMBED = os.path.join(CSRC, "bnbp_spec_embed.inc")   # ... from this generated raw-string copy
ONCHIP_SRC = os.path.join(CSRC, "bnbp_onchip.cuh")       # the on-chip multi-sweep kernel, appended behind it
ONCHIP_EMBED = os.path.join(CSRC, "bnbp_onchip_embed.inc")
HEADERS = [os.path.join(CSRC, "bnbp_kernels.cuh"), os.path.join(CSRC, "bnbp_sweep.cuh"),
           os.path.join(CSRC, "bnbp_variants.h"), os.path.join(CSRC, "bnbp_jit.h"), SPEC_SRC, ONCHIP_SRC,
           os.path.join(CSRC, "bnbp_dense.h"), os.path.join(CSRC, "bnbp_dense.cuh"),
           os.path.join(CSRC, "bnbp_dense_tc.cuh"), os.path.join(CSRC, "bnbp_lw.cuh"),
           os.path.join(CSRC, "bnbp_logev.cuh"), os.path.join(os.path.dirname(HERE), "include", "bnbp.h")]
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
# host-only units: rebuilt when the drop-in headers they wrap change
HOST_HEADERS = {"bnbp_netfile.cpp": [os.path.join(INCLUDE, "bayesian", "graph.hpp"),
                                     os.path.join(INCLUDE, "bayesian", "serializer", "bif.hpp"),
                                     os.path.join(INCLUDE, "bayesian", "serializer", "dsc.hpp"),
                                     os.path.join(INCLUDE, "bayesian", "serializer", "text_scanner.hpp"),
                                     os.path.join(INCLUDE, "bnbp.h")]}


def embed_spec_header() -> None:
    """bnbp_spec.cuh / bnbp_onchip.cuh -> *_embed.inc (C++ raw string literals #included by bnbp_jit.cu)."""
    for src, dst in ((SPEC_SRC, SPEC_EMBED), (ONCHIP_SRC, ONCHIP_EMBED)):
        text = open(src).read()
        assert ')BNBPSPEC"' not in text
        out = 'R"BNBPSPEC(' + text + ')BNBPSPEC"\n'
        if not os.path.exists(dst) or open(dst).read() != out:
            with open(dst, "w") as f:
                f.write(out)


def sweep_variants():
    """(T, VEC, RMAX, KNET) instantiations: the X-macro list in csrc/bnbp_variants.h, the same
    list bnbp_api.cu dispatches over."""
    import re
    txt = open(os.path.join(CSRC, "bnbp_variants.h")).read()
    trip = re.findall(r"X\(T,\s*(\d+),\s*(\d+),\s*(\d+)\)", txt)
    return [(t, int(v), int(r), int(k)) for t in ("double", "float") for (v, r, k) in trip]

NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-I", INCLUDE]


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: libbnbp cannot be built")
    return p


def _env():
    env = dict(os.environ)
    env.pop("CC", None)     # the image exports a CC wrapper nvcc should not pick up
    env.pop("CXX", None)
    return env


def _units():
    units = [(os.path.join(CSRC, "bnbp_api.cu"), os.path.join(OBJDIR, "bnbp_api.o"), []),
             (os.path.join(CSRC, "bnbp_jit.cu"), os.path.join(OBJDIR, "bnbp_jit.o"), []),
             (os.path.join(CSRC, "bnbp_dense_inst.cu"), os.path.join(OBJDIR, "bnbp_dense.o"), []),
             (os.path.join(CSRC, "bnbp_dense_tc_inst.cu"), os.path.join(OBJDIR, "bnbp_dense_tc.o"), []),
             (os.path.join(CSRC, "bnbp_netfile.cpp"), os.path.join(OBJDIR, "bnbp_netfile.o"), [])]
    for t, v, r, k in sweep_variants():
        units.append((os.path.join(CSRC, "bnbp_sweep_inst.cu"),
                      os.path.join(OBJDIR, f"sweep_{t}_v{v}_r{r}_k{k}.o"),
                      [f"-DBNBP_T={t}", f"-DBNBP_VEC={v}", f"-DBNBP_RMAX={r}", f"-DBNBP_KNET={k}"]))
    return units


def _stale(obj: str, src: str) -> bool:
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    deps = HOST_HEADERS.get(os.path.basename(src), HEADERS)
    return any(os.path.getmtime(f) > t for f in [src] + deps)


def build(force: bool = False, verbose: bool = False, extra=()) -> str:
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = nvcc_path()
    embed_spec_header()
    todo = [(s, o, d) for (s, o, d) in _units() if force or _stale(o, s)]

    def compile_one(u):
        src, obj, defs = u
        tune = [f"-DBNBP_GEN_MINB={os.environ['BNBP_GEN_MINB']}"] if os.environ.get("BNBP_GEN_MINB") else []
        cmd = [nvcc, *NVCC_FLAGS, *extra, *defs, *tune, "-c", "-o", obj, src]
        r = subprocess.run(cmd, env=_env(), capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {os.path.basename(obj)}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stdout.write(f"[bnbp build] {os.path.basename(obj)}\n{r.stderr}")
        return obj

    if todo:
        with ThreadPoolExecutor(max_workers=max(1, min(len(todo), os.cpu_count() or 4))) as ex:
            list(ex.map(compile_one, todo))
    objs = [o for (_, o, _) in _units()]
    for f in os.listdir(OBJDIR):                      # drop objects of variants that no longer exist
        if os.path.join(OBJDIR, f) not in objs:
            os.remove(os.path.join(OBJDIR, f))
    if todo or not os.path.exists(LIB):
        cmd = [nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a",
               "-o", LIB, *objs, "-ldl"]      # NCCL (the communicators libbnbp owns, SURVEY 8e) is bound at first use: bnbp_api.cu
        subprocess.run(cmd, check=True, env=_env())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True,
                extra=["-Xptxas", "-v"] if "--ptxas" in sys.argv else ()))
