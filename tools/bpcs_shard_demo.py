"""BatchedPCSProof::prove with every polynomial split by block over N GPUs, one process per GPU (torchrun): ml_bpcs_shard_* with
the arenas connected through CUDA IPC records all-gathered over torch.distributed — the only collective; the data path is NVLink
stores + device flags.

    torchrun --nproc-per-node N tools/bpcs_shard_demo.py <n_vars> <n_polys> [check] [reps]

Every process generates the whole synthetic polynomials (seeds 0xB200 + j) on its GPU and passes pointers to its own blocks.
`check`: `oracle` compares the proof with the CPU oracle's (small sizes); `gpu` with the unsharded prover on rank 0's GPU."""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np
from shard_harness import Ranks

from multilinear_b200 import api as ml
from multilinear_b200 import load

nv = int(sys.argv[1]) if len(sys.argv) > 1 else 14
B = int(sys.argv[2]) if len(sys.argv) > 2 else 10
check = sys.argv[3] if len(sys.argv) > 3 else "gpu"
reps = int(sys.argv[4]) if len(sys.argv) > 4 else 3
n = 1 << nv
ranks = Ranks()
world, rank = ranks.world, ranks.rank
L = load()
sh = ranks.connect(ml.BlockShardedBatchedProver.one_rank(rank, world, ranks.local, B, nv))
evals = [ml.synthetic_elements_dev(0xB200 + j, n) for j in range(B)]
blocks = [e.ptr.value + rank * (n // world) * 16 for e in evals]
inputs = ml.synthetic_elements_dev(0xC1A1, nv).elems()
outs = bytearray()
for e in evals:
    ob = (C.c_uint8 * 16)()
    ml.check(L.ml_mle_evals_evaluate_dev(e.ptr, C.c_size_t(n), C.c_void_p(inputs.ctypes.data), C.c_size_t(nv), ob, None))
    outs += bytes(ob)
outputs = np.frombuffer(bytes(outs), dtype=np.uint8).reshape(B, 16)
state = {}


def prove():
    t = ml.Transcript()
    p = sh.prove_dev(inputs, outputs, blocks, t)
    state["t"] = t.random()
    return p


ms, proof = ranks.timed(sh, prove, reps)
phases = sh.phase_ms()
agree = ranks.agree(state["t"])

if rank == 0:
    blob = proof.fri_proof.serialize()
    line = {"workload": "bpcs_shard_prove", "n_gpus": world, "n_vars": nv, "n_polys": B, "prove_ms": ms, "proof_bytes": len(blob),
            "proof_sha256": hashlib.sha256(blob).hexdigest(), "verifies": proof.verify(ml.Transcript()) == 0, "transcripts_agree": agree,
            "arena_bytes_per_rank": sh.arena_bytes(),
            "rank0_phase_ms": dict(zip(["S0_encode_exchange", "S1_combine_batch_tree", "S2_S3_root_tables", "sharded_rounds", "tail_chain",
                                          "openings_proof"], phases))}
    if check == "oracle":
        from oracle.binding import Oracle
        O = Oracle(threads=os.cpu_count() or 1)
        ot = O.transcript()
        op, st = O.batched_pcs_prove(inputs, outputs, [e.elems() for e in evals], ot)
        line["matches_oracle"] = bool(st == 0 and op.fri.blob == blob and ot.random() == state["t"] and
                                      [c for nz in proof.sumcheck_polynomials for c in nz] == op.sumcheck)
    elif check == "gpu":
        t1 = ml.Transcript()
        ptrs = (C.c_void_p * B)(*[e.ptr.value for e in evals])
        h = C.c_void_p()
        ml.check(L.ml_batched_pcs_prove_dev(ml._p(inputs), ml._sz(nv), ml._p(outputs), ml._sz(B), ptrs, ml._sz(n), t1.h, None, C.byref(h)))
        single = ml.PCSProof(h, batched=True)
        line["matches_single_gpu_prover"] = bool(single.fri_proof.serialize() == blob and t1.random() == state["t"])
        del single
    print(json.dumps(line), flush=True)
del proof
ranks.close(sh)
