"""Builds multilinear_b200/libmultilinear_b200.so with nvcc for sm_100a (in-tree, no JIT cache)."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libmultilinear_b200.so")
SOURCES = ["core.cu", "field_ops.cu", "ntt.cu", "merkle.cu", "fri.cu", "sumcheck.cu", "mle.cu", "prover.cu", "chain.cu", "peer.cu", "shard.cu", "pcs_shard.cu", "bpcs_shard.cu", "wsumcheck_shard.cu", "fri_shard.cu", "bfri_shard.cu", "plan.cu", "bplan.cu"]
# instrumentation (integer-pipe speed-of-light loops for bench.py / tools): its own library, not part of the product ABI
INSTR_OUT = os.path.join(HERE, "libmlb_instr.so")
INSTR_SOURCES = ["microbench.cu"]
HEADERS = ["field.cuh", "sha256.cuh", "reduce.cuh", "transcript.cuh", "internal.h", "handles.h", "prover_internal.h", "peer.h", "pcs_shard.h", "plan.h", os.path.join("..", "..", "include", "multilinear_b200.h"),
           os.path.join("..", "..", "include", "multilinear_b200_instr.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC", "-diag-suppress", "177",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")


def needs_build():
    if not os.path.exists(OUT) or not os.path.exists(INSTR_OUT):
        return True
    t = min(os.path.getmtime(OUT), os.path.getmtime(INSTR_OUT))
    deps = [os.path.join(CSRC, f) for f in SOURCES + INSTR_SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    nvcc = _nvcc()
    extra = os.environ.get("MLB_EXTRA_NVCC_FLAGS", "").split()  # experiments only (e.g. -DMLB_MERKLE_LEAF_SPECIALISED)
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES + INSTR_SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    objs, instr_objs = [], []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out.decode(errors="replace"))
            raise RuntimeError("nvcc failed on %s" % src)
        (instr_objs if src in INSTR_SOURCES else objs).append(obj)
    cmd = [nvcc, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.check_call(cmd)
    cmd = [nvcc, "-shared", "-o", INSTR_OUT] + instr_objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-L", HERE,
           "-lmultilinear_b200", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
