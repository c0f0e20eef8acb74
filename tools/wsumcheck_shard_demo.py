"""The width-w System sumcheck sharded over N GPUs, one process per GPU (torchrun): ml_wsumcheck_shard_* with the arenas
connected through CUDA IPC records all-gathered over torch.distributed; the data path is peer stores + device flags.

    torchrun --nproc-per-node N tools/wsumcheck_shard_demo.py <n_vars> <width> [reps]

Every process generates the whole synthetic trace (seed 0x5C) on its GPU and passes a pointer to its own row block.  Rank 0
compares the result with the single-GPU handle (ml_wsumcheck_build_dev + compute_polynomials); every rank's result must agree."""
import ctypes as C
import hashlib
import json
import os
import random
import sys

sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
import torch
import torch.distributed as dist

from multilinear_b200 import api as ml
from multilinear_b200 import load

nv = int(sys.argv[1]) if len(sys.argv) > 1 else 16
width = int(sys.argv[2]) if len(sys.argv) > 2 else 4
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
h = 1 << nv
world, rank, local = int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
ml.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
L = load()


def barrier():
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()


degree = 2
rng = random.Random(0x5C)
terms = [(3, []), (5, [0] * degree), (7, [width - 1, 0]), (11, [rng.randrange(width)])]
sh = ml.ShardedWideSumcheck.one_rank(rank, world, local, width, nv)
if world > 1:
    sh.connect_over(dist, dev)
else:
    sh.connect(sh.export())
sh.set_composition(terms)
trace = ml.synthetic_elements_dev(0x5C, h * width)
block = trace.ptr.value + rank * (h // world) * width * 16
row_point = ml.to_ints(ml.synthetic_elements_dev(0x5C0001, nv).elems())
torch.cuda.synchronize()
stream = torch.cuda.ExternalStream(sh.stream(0), device=dev)


def run():
    t = ml.Transcript()
    res = sh.compute_sumcheck_polynomials_dev(row_point, [block], degree, t, 42)
    return res, t.random()


barrier()
run()  # warm-up
barrier()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record(stream)
for _ in range(reps):
    res, tr = run()
e1.record(stream)
barrier()
ms = e0.elapsed_time(e1) / reps
digest = hashlib.sha256(repr(res).encode() + tr).digest()
mine = torch.tensor(list(digest), dtype=torch.uint8, device=dev)
agree = True
if world > 1:
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    d0 = mine.clone()
    dist.broadcast(d0, 0)
    flag = torch.tensor([int(torch.equal(mine, d0))], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    agree = bool(int(flag[0]))

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
barrier()
sh.free()
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
