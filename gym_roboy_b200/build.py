"""In-tree build of the CUDA library (nvcc, sm_100a only).

    python -m gym_roboy_b200.build        # -> gym_roboy_b200/_lib/libroboy_b200.so

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels with the tree.
"""
import os
import subprocess
import sys

_PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_PKG, "csrc")
LIB_DIR = os.path.join(_PKG, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libroboy_b200.so")
SOURCES = ("roboy_kernels.cu", "roboy_generic.cu", "roboy_policy.cu", "roboy_policy_tc.cu", "roboy_policy_generic.cu", "roboy_policy_eval.cu",
           "roboy_ppo.cu", "roboy_capi.cu")
HEADERS = ("roboy_kernels.cuh", "roboy_generic.cuh", "generic_env.cuh", "roboy_policy.cuh", "policy_common.cuh", "policy_generic.cuh", "step_rare.cuh", "msj_math.cuh", "philox.cuh", "dlpack_min.h", os.path.join("..", "..", "include", "roboy_b200.h"))

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",  # numpy never fuses a multiply and an add; neither may we (bit-exact done mask)
    "-Xcompiler", "-fPIC,-ffp-contract=off",
    "-shared",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return "nvcc"


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > built for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    """Compile libroboy_b200.so if missing or older than its sources; returns its path.  The translation units are
    compiled in parallel (one nvcc per .cu) and linked into one shared library."""
    if not force and not is_stale():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(LIB_DIR, exist_ok=True)
    obj_dir = os.path.join(os.path.dirname(_PKG), "build", "obj")
    os.makedirs(obj_dir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else [])

    def compile_one(src):
        obj = os.path.join(obj_dir, os.path.splitext(src)[0] + ".o")
        cmd = [_nvcc()] + flags + ["-c", "-o", obj, os.path.join(CSRC, src)]
        proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        return obj, cmd, proc

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    for obj, cmd, proc in results:
        if verbose or proc.returncode != 0:
            sys.stderr.write(proc.stdout)
        if proc.returncode != 0:
            raise RuntimeError("nvcc failed (exit {}): {}".format(proc.returncode, " ".join(cmd)))
    link = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-o", LIB_PATH] + [r[0] for r in results]
    proc = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or proc.returncode != 0:
        sys.stderr.write(proc.stdout)
    if proc.returncode != 0:
        raise RuntimeError("link failed (exit {}): {}".format(proc.returncode, " ".join(link)))
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
