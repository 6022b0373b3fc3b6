"""Build libnerfmeshes_b200.so in-tree with nvcc for sm_100a (no GPU needed: nvcc cross-compiles).

    python -m nerfmeshes_b200.build [--force]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(OUT_DIR, "libnerfmeshes_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr"]
COMMON += os.environ.get("NM_NVCC_EXTRA", "").split()        # bring-up aid: extra -D switches for A/B builds (use with --force)
# per-file extra flags: the light render stages keep a*b+c as two roundings, like the reference's separate torch ops
SOURCES = {
    "nm_program.cu": [],
    "nm_mlp_tc.cu": [],
    "nm_mlp_simt.cu": [],
    "nm_render.cu": ["-fmad=false"],
    "nm_mc.cu": ["-fmad=false"],
    "nm_metrics.cu": ["-fmad=false"],
    "nm_train.cu": [],
    "nm_gemm_tc.cu": [],
    "nm_objwriter.cu": [],
    "nm_api.cu": [],
}


def _stale(obj, deps):
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(OUT_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "nerfmeshes_b200.h"))
    objs, jobs = [], []
    for src, extra in SOURCES.items():
        s = os.path.join(CSRC, src)
        o = os.path.join(OUT_DIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers + [__file__]):
            jobs.append((src, [NVCC] + ARCH + COMMON + extra + ["-c", s, "-o", o]))

    def run(job):
        name, cmd = job
        r = subprocess.run(cmd, capture_output=True, text=True)
        return name, r

    logs = []
    with ThreadPoolExecutor(max_workers=6) as ex:
        for name, r in ex.map(run, jobs):
            logs.append(f"== {name}\n{r.stderr}")
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError(f"nvcc failed on {name}")
    if jobs or force or _stale(LIB, objs):
        cmd = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    with open(os.path.join(OUT_DIR, "ptxas.log"), "a" if not force else "w") as f:
        f.write("\n".join(logs))
    if verbose:
        print("\n".join(logs))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
