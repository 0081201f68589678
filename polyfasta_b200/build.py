"""Builds polyfasta_b200/libpolyfasta_b200.so in-tree with nvcc for sm_100a (no torch extension machinery:
the library is a plain C-ABI shared object loaded with ctypes)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libpolyfasta_b200.so")
CU = ["pfa_api.cu", "pfa_encode.cu", "pfa_sites.cu", "pfa_codon.cu", "pfa_pairwise.cu", "pfa_finalize.cu", "pfa_batch.cu", "pfa_xchg.cu", "pfa_ingest.cu", "pfa_windows.cu", "pfa_divergence.cu", "pfa_haplotypes.cu"]
CPP = ["pfa_fasta.cpp", "pfa_codon_rules.cpp", "pfa_pack.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--fmad=false",
              "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-deprecated-declarations", "-diag-suppress", "128", "-Xptxas", "-v"]
# (nvcc --split-compile=0 halves the build time again but costs the site scan 0.8 % -- measured, not used)


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build(force=False, verbose=False):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "polyfasta_b200.h"))
    objs = []
    logs = []
    todo = []
    for src in CU + CPP:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src + ".o")
        objs.append(o)
        if force or _newer(o, [s] + headers):
            todo.append((src, [nvcc] + NVCC_FLAGS + ["-c", s, "-o", o]))

    def compile_one(item):
        src, cmd = item
        p = subprocess.run(cmd, capture_output=True, text=True)
        return src, cmd, p

    # the translation units are independent: compile them side by side (the template-heavy scan kernels dominate)
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=max(1, min(len(todo), os.cpu_count() or 1))) as ex:
        for src, cmd, p in ex.map(compile_one, todo):
            logs.append("$ " + " ".join(cmd) + "\n" + p.stdout + p.stderr)
            if p.returncode != 0:
                sys.stderr.write(logs[-1])
                raise RuntimeError("nvcc failed on " + src)
    if force or _newer(SO, objs):
        cmd = [nvcc, "-shared", "-o", SO] + objs + ["-lcudart"]
        p = subprocess.run(cmd, capture_output=True, text=True)
        if p.returncode != 0:
            sys.stderr.write(p.stdout + p.stderr)
            raise RuntimeError("link failed")
    if logs:
        with open(os.path.join(objdir, "nvcc.log"), "w") as f:
            f.write("\n".join(logs))
        if verbose:
            print("\n".join(logs))
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
