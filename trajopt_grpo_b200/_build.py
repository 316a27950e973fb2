"""In-tree build of the C-ABI library (nvcc, sm_100a only).

    python -m trajopt_grpo_b200._build [--force]

Produces trajopt_grpo_b200/libtrajopt_grpo_b200.so next to this file; the .so is
git-ignored but travels with the repo snapshot to the GPU box.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "obj")
LIB = os.path.join(HERE, "libtrajopt_grpo_b200.so")
SOURCES = ["tg_api.cu", "tg_rollout.cu", "tg_rollout_tc256.cu", "tg_advantage.cu", "tg_update.cu", "tg_update_tc.cu", "tg_update_tcw.cu", "tg_order.cu", "tg_export.cu", "tg_minibatch.cu", "tg_selftest.cu", "tg_env_dynamics.cu", "tg_comm.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "trajopt_grpo.h"))
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    nvcc = _nvcc()
    jobs = []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s.replace(".cu", ".o"))
        if force or _stale(obj, [src] + headers):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        with open(obj + ".log", "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=min(4, len(jobs))) as ex:
            logs = list(ex.map(compile_one, jobs))
        if verbose:
            for l in logs:
                print(l)
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in srcs]
    if jobs or force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-lcudart", "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
