"""BatchedPCSProof::prove sharded over N GPUs, one process per GPU (torchrun): ml_shard_* with the arenas connected through CUDA
IPC records all-gathered over torch.distributed — the only collective; the data path is NVLink stores + device flags.

    torchrun --nproc-per-node N tools/sharded_prove_demo.py <n_vars> <n_polys> [check] [reps]

`check`: rank 0 also proves on its own GPU with the unsharded prover (ml_batched_pcs_prove_dev) and compares the proof bytes
(sizes that fit one GPU); with `oracle` it compares against the CPU oracle instead (small sizes)."""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
from shard_harness import Ranks

from multilinear_b200 import api as ml
from multilinear_b200 import load

nv = int(sys.argv[1]) if len(sys.argv) > 1 else 16
B = int(sys.argv[2]) if len(sys.argv) > 2 else 8
check = sys.argv[3] if len(sys.argv) > 3 else "gpu"
reps = int(sys.argv[4]) if len(sys.argv) > 4 else 3
n = 1 << nv
ranks = Ranks()
world, rank, dev = ranks.world, ranks.rank, ranks.dev
L = load()


def poly(j):
    t = torch.empty(16 * n, dtype=torch.uint8, device=dev)
    ml.check(L.ml_synthetic_elements_dev(C.c_uint64(5000 + j), C.c_size_t(n), C.c_void_p(t.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return t


sh = ranks.connect(ml.ShardedBatchedProver.one_rank(rank, world, ranks.local, B, nv))
mine = [poly(j) for j in sh.local_polys()]
ptrs = [t.data_ptr() for t in mine]
torch.cuda.synchronize()

# the claim: evaluation point from the synthetic generator, outputs computed by each owner and all-gathered
inputs = ml.synthetic_elements_dev(0xC1A1, nv).elems()
outs_local = np.zeros((B, 16), dtype=np.uint8)
for j, t in zip(sh.local_polys(), mine):
    ob = (C.c_uint8 * 16)()
    ml.check(L.ml_mle_evals_evaluate_dev(C.c_void_p(t.data_ptr()), C.c_size_t(n), C.c_void_p(inputs.ctypes.data), C.c_size_t(nv), ob, None))
    outs_local[j] = np.frombuffer(bytes(ob), dtype=np.uint8)
if world > 1:
    g = torch.from_numpy(outs_local).to(dev).to(torch.int32)
    dist.all_reduce(g)  # rows are disjoint across ranks
    outputs = g.to(torch.uint8).cpu().numpy()
else:
    outputs = outs_local

commit_ms, root = ranks.timed(sh, lambda: sh.batch_commit_dev(ptrs), reps)
commit_phases = sh.phase_ms()
state = {}


def prove():
    t = ml.Transcript()
    p = sh.prove_dev(inputs, outputs, ptrs, t)
    state["t"] = t.random()
    return p


prove_ms, proof = ranks.timed(sh, prove, reps)
prove_phases = sh.phase_ms()
transcripts_agree = ranks.agree(state["t"])  # every rank's transcript must end in rank 0's final state

fixture = None
try:
    fx = json.load(open(os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "batch_root_64x2p22.json")))
    if fx["n_polys"] == B and fx["log_n"] == nv:
        fixture = fx["root"] == root.hex()
except Exception:  # noqa: BLE001
    pass

if rank == 0:
    blob = proof.fri_proof.serialize()
    line = {"workload": "sharded_batched_pcs_prove", "n_gpus": world, "polys": B, "n_vars": nv, "commit_ms": commit_ms, "prove_ms": prove_ms,
            "commit_melem_per_s": B * n / (commit_ms * 1e-3) / 1e6, "root": root.hex(), "root_matches_oracle_fixture": fixture,
            "proof_bytes": len(blob), "proof_sha256": hashlib.sha256(blob).hexdigest(), "verifies": proof.verify(ml.Transcript()) == 0,
            "transcripts_agree": transcripts_agree, "arena_bytes_per_rank": L.ml_shard_arena_bytes(sh.h),
            "rank0_commit_phase_ms": dict(zip(["S0_encode_pack", "S1_row_subtree", "S2_batch_root"], commit_phases)),
            "rank0_prove_phase_ms": dict(zip(["S0_encode_pack", "S1_row_subtree", "S2_root_rho", "S2_fingerprint_partials", "S3_reduce", "S4_wait_matrix",
                                              "chain_incl_first_fold", "openings_proof"], prove_phases))}
    if check == "oracle":
        from oracle.binding import Oracle
        O = Oracle(threads=os.cpu_count() or 1)
        polys = [O.synthetic(5000 + j, n) for j in range(B)]
        ot = O.transcript()
        op, st = O.batched_pcs_prove(inputs, outputs, polys, ot)
        line["matches_oracle"] = bool(st == 0 and op.fri.blob == blob and ot.random() == state["t"] and
                                      [c for nz in proof.sumcheck_polynomials for c in nz] == op.sumcheck)
    elif check == "gpu" and B * n * 16 * 5 < 150e9:
        allp = [poly(j) for j in range(B)]
        torch.cuda.synchronize()
        pa = (C.c_void_p * B)(*[t.data_ptr() for t in allp])
        t1 = ml.Transcript()
        h = C.c_void_p()
        ml.check(L.ml_batched_pcs_prove_dev(C.c_void_p(inputs.ctypes.data), C.c_size_t(nv), C.c_void_p(outputs.ctypes.data), C.c_size_t(B), pa, C.c_size_t(n),
                                            t1.h, None, C.byref(h)))
        single = ml.PCSProof(h, batched=True)
        line["matches_single_gpu_prover"] = bool(single.fri_proof.serialize() == blob and t1.random() == state["t"])
        del single, allp
    print(json.dumps(line), flush=True)
del proof
ranks.close(sh)
