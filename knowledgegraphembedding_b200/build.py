"""Build libkge_b200.so in-tree with nvcc for sm_100a (no torch extension machinery, plain C ABI)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libkge_b200.so")
SOURCES = ["kge_train.cu", "kge_optim.cu", "kge_eval.cu", "kge_eval_gemm.cu", "kge_eval_topk.cu", "kge_eval_relation.cu",
           "kge_eval_candidates.cu", "kge_eval_path.cu", "kge_sampler.cu", "kge_peer.cu", "kge_train_inst.cu"]
HEADERS = ["kge_common.cuh", "kge_rows.cuh", "kge_adam.cuh", "kge_eval_tile.cuh", "kge_train_args.cuh",
           "kge_train_kernels.cuh",
           "kge_train_split.cuh", "kge_train_launch.cuh", "kge_math.h", os.path.join("..", "..", "include", "kge_b200.h")]
# (source, object suffix, extra flags): the train-path kernels are instantiated once per model (model ids of
# include/kge_b200.h), one translation unit each, so that the five sets compile in parallel
UNITS = [(s, "", []) for s in SOURCES if s != "kge_train_inst.cu"] + \
        [("kge_train_inst.cu", "_m%d" % i, ["-DKGE_TU_MODEL=%d" % i]) for i in range(5)]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-diag-suppress", "1886"]
OBJ_DIR = os.path.join(CSRC, "build")


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libkge_b200.so cannot be built (there is no fallback path)")


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def _object_stale(src, obj):
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in [src] + HEADERS)


def build(force=False, verbose=False, variant=None, extra_flags=()):
    """Compile every CUDA source (one nvcc process per file, in parallel) and link csrc/libkge_b200.so; returns the
    path.  Objects are kept under csrc/build/ so that an edit recompiles only the files it touches.
    variant / extra_flags (A/B experiments): build csrc/libkge_b200_<variant>.so with extra nvcc flags from its own object
    directory; KGE_LIB=<path> makes _lib.py load it."""
    lib_path, obj_dir = LIB, OBJ_DIR
    if variant:
        lib_path = os.path.join(CSRC, "libkge_b200_%s.so" % variant)
        obj_dir = os.path.join(CSRC, "build", variant)
        force = True
    if not force and not is_stale():
        return lib_path
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(obj_dir, exist_ok=True)
    nvcc = _nvcc()
    jobs, objs = [], []
    for src, suffix, extra in UNITS:
        obj = os.path.join(obj_dir, src.replace(".cu", suffix + ".o"))
        objs.append(obj)
        if force or _object_stale(src, obj):
            jobs.append((src + suffix, [nvcc] + NVCC_FLAGS + list(extra_flags) + extra + (["-Xptxas", "-v"] if verbose else []) +
                         ["-c", src, "-o", obj]))

    def run(job):
        return job[0], subprocess.run(job[1], cwd=CSRC, capture_output=True, text=True)

    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as pool:
        for src, res in pool.map(run, jobs):
            if res.returncode != 0:
                raise RuntimeError("nvcc failed on %s:\n%s%s" % (src, res.stdout, res.stderr))
            if verbose:
                print(res.stderr)
    res = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib_path] + objs,
                         cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    return lib_path


if __name__ == "__main__":
    print(build(force=True, verbose=True))
