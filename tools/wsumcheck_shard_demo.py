"""The width-w System sumcheck sharded over N GPUs, one process per GPU (torchrun): ml_wsumcheck_shard_* with the arenas
connected through CUDA IPC records all-gathered over torch.distributed; the data path is peer stores + device flags.

    torchrun --nproc-per-node N tools/wsumcheck_shard_demo.py <n_vars> <width> [reps]

Every process generates the whole synthetic trace (seed 0x5C) on its GPU and passes a pointer to its own row block.  Rank 0
compares the result with the single-GPU handle (ml_wsumcheck_build_dev + compute_polynomials); every rank's result must agree."""
import ctypes as C
import hashlib
import json
import random
import sys

from shard_harness import Ranks

from multilinear_b200 import api as ml
from multilinear_b200 import load

nv = int(sys.argv[1]) if len(sys.argv) > 1 else 16
width = int(sys.argv[2]) if len(sys.argv) > 2 else 4
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
h = 1 << nv
ranks = Ranks()
world, rank = ranks.world, ranks.rank
L = load()
degree = 2
rng = random.Random(0x5C)
terms = [(3, []), (5, [0] * degree), (7, [width - 1, 0]), (11, [rng.randrange(width)])]
sh = ranks.connect(ml.ShardedWideSumcheck.one_rank(rank, world, ranks.local, width, nv))
sh.set_composition(terms)
trace = ml.synthetic_elements_dev(0x5C, h * width)
block = trace.ptr.value + rank * (h // world) * width * 16
row_point = ml.to_ints(ml.synthetic_elements_dev(0x5C0001, nv).elems())


def run():
    t = ml.Transcript()
    res = sh.compute_sumcheck_polynomials_dev(row_point, [block], degree, t, 42)
    return res, t.random()


ms, (res, tr) = ranks.timed(sh, run, reps)
agree = ranks.agree(hashlib.sha256(repr(res).encode() + tr).digest())

if rank == 0:
    rp = ml.as_elems(row_point)
    hd = C.c_void_p()
    ml.check(L.ml_wsumcheck_build_dev(ml._p(rp), C.c_size_t(nv), trace.ptr, C.c_size_t(width), C.c_size_t(h), None, C.byref(hd)))
    g = ml.WideSumcheckTables(hd, width)
    g.set_composition(terms)
    t1 = ml.Transcript()
    single = g.compute_sumcheck_polynomials(degree, t1, 42)
    line = {"workload": "wsumcheck_shard", "n_gpus": world, "n_vars": nv, "width": width, "composition_degree": degree, "call_ms": ms,
            "arena_bytes_per_rank": sh.arena_bytes(), "results_agree": agree,
            "matches_single_gpu": bool(single == res and t1.random() == tr)}
    print(json.dumps(line), flush=True)
ranks.close(sh)
