"""Build recipe for the C-ABI shared library (nvcc, sm_100a only, in-tree output).

`python dl-dkd_b200/build.py` or `__graft_entry__.build()`.  The .so is git-ignored but travels
to the GPU box with the repo snapshot; nothing is JIT-compiled at run time.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdkd_b200.so")
SOURCES = ["dkd_api.cu", "dkd_prep.cu", "dkd_score_f32.cu", "dkd_exact_umma.cu", "dkd_score_bf16.cu", "dkd_rank.cu", "dkd_train.cu", "dkd_encoder.cu", "dkd_moments.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--shared", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default",
]


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(HERE, "..", "include", "dkd_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:  # compile translation units in parallel
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
               "-Xcompiler", "-fPIC", "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose:
            print(out)
    link = [nvcc, "--shared", "-o", LIB] + objs
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
