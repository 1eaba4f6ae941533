"""In-tree nvcc build of libneuralbody_b200.so (sm_100a only; no JIT cache, no torch headers).

The shared object lands next to this file so it travels with the repo snapshot to the
GPU box (it is git-ignored, not gpurun-ignored)."""
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libneuralbody_b200.so")
SOURCES = ["nb_capi.cu", "nb_render_f32.cu", "nb_render_tc_list.cu", "nb_tc_probe.cu", "nb_tc_probe2.cu", "nb_tc_bench.cu", "nb_render_bwd.cu", "nb_train.cu", "nb_sample_pdf.cu", "nb_mcubes.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]
OBJ_DIR = os.path.join(HERE, "build")


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libneuralbody_b200.so")


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(HERE, "..", "include", "neuralbody_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False, defines=(), out=None):
    """Compile every CUDA source of the package for sm_100a (one nvcc per file, in parallel) and link one shared library.
    `defines` / `out`: an A/B variant (e.g. defines=("NB_LIST_CLUSTER=1",), out="libnb_c1.so" -> select it with NB_LIB_PATH)."""
    if out is None and not force and not _stale():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    nvcc = find_nvcc()
    obj_dir = OBJ_DIR if out is None else OBJ_DIR + "_" + os.path.splitext(out)[0]
    lib_path = LIB_PATH if out is None else os.path.join(HERE, out)
    os.makedirs(obj_dir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-D" + d for d in defines] + (["-Xptxas", "-v"] if verbose else []) + \
              ["-c", "-o", obj, os.path.join(CSRC, src)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s%s" % (src, res.stdout, res.stderr))
        return obj, res.stderr

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        done = list(ex.map(compile_one, SOURCES))
    if verbose:
        for _, log in done:
            print(log)
    res = subprocess.run([nvcc, "--shared", "-o", lib_path] + [o for o, _ in done], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    return lib_path
