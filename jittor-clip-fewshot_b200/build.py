"""Builds libjclip_b200.so (the C-ABI library declared in include/jclip_b200.h) in-tree with nvcc.

sm_100a only: the GEMM uses tcgen05 / TMEM / TMA, which do not exist on any other target.  The library
is linked against the static CUDA runtime and resolves cuTensorMapEncodeTiled through
cudaGetDriverEntryPoint, so it has no load-time dependency beyond libstdc++ / libc and travels as a
single file.

    python jittor-clip-fewshot_b200/build.py [--force] [--verbose]
"""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
OBJ_DIR = CSRC / "build"
LIB_PATH = PKG_DIR / "libjclip_b200.so"
SOURCES = ["api.cu", "gemm.cu", "attention.cu", "attention_tc.cu", "rowwise.cu", "mta.cu", "head.cu", "tta.cu", "train.cu"]
HEADERS = [CSRC / "kernels.h", CSRC / "ptx.cuh", PKG_DIR.parent / "include" / "jclip_b200.h"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
]


def find_nvcc():
    cand = [os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"]
    for c in cand:
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _stale(target, deps):
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(d.stat().st_mtime > t for d in deps)


def build_variant(out_path, defines):
    """A/B experiments: the same library with extra -D macros, built out of tree objects into `out_path`
    (load it with JCB_LIB_PATH=...).  Not used by the product build."""
    nvcc = find_nvcc()
    vdir = OBJ_DIR / ("variant_" + Path(out_path).stem)
    vdir.mkdir(parents=True, exist_ok=True)
    flags = NVCC_FLAGS + [f"-D{d}" for d in defines]

    def one(src):
        o = vdir / (Path(src).stem + ".o")
        r = subprocess.run([nvcc] + flags + ["-c", str(CSRC / src), "-o", str(o)], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        return o

    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(one, SOURCES))
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(out_path)] + \
          [str(o) for o in objs] + ["-cudart", "static", "-lpthread", "-ldl", "-lrt"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return Path(out_path)


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a and link the shared library.  Returns the library path."""
    nvcc = find_nvcc()
    OBJ_DIR.mkdir(parents=True, exist_ok=True)
    jobs = []
    for src in SOURCES:
        s = CSRC / src
        o = OBJ_DIR / (s.stem + ".o")
        if force or _stale(o, [s] + HEADERS):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + ["-c", str(s), "-o", str(o)]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        return s, r

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for s, r in ex.map(compile_one, jobs):
            if verbose and (r.stdout or r.stderr):
                print(r.stdout + r.stderr, file=sys.stderr)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {s.name}:\n{r.stdout}\n{r.stderr}")
    objs = [OBJ_DIR / (Path(s).stem + ".o") for s in SOURCES]
    if force or jobs or _stale(LIB_PATH, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(LIB_PATH)] + \
              [str(o) for o in objs] + ["-cudart", "static", "-lpthread", "-ldl", "-lrt"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB_PATH


if __name__ == "__main__":
    if "--variant" in sys.argv:      # python build.py --variant out.so -DNAME=VALUE ...
        i = sys.argv.index("--variant")
        print(build_variant(sys.argv[i + 1], [a[2:] for a in sys.argv[i + 2:] if a.startswith("-D")]))
    else:
        p = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
        print(p)
