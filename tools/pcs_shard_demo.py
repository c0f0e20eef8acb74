"""PCSProof::prove of one polynomial sharded over N GPUs, one process per GPU (torchrun): ml_pcs_shard_* with the arenas
connected through CUDA IPC records all-gathered over torch.distributed — the only collective; the data path is NVLink stores +
device flags.

    torchrun --nproc-per-node N tools/pcs_shard_demo.py <n_vars> [check] [reps]

Every process generates the whole synthetic polynomial (seed 0xB200) on its GPU and passes a pointer to its own block.
`check`: `oracle` compares the proof with the CPU oracle's (small sizes); `gpu` with the unsharded prover on rank 0's GPU."""
import ctypes as C
import hashlib
import json
import os
import sys

from shard_harness import Ranks

from multilinear_b200 import api as ml
from multilinear_b200 import load

nv = int(sys.argv[1]) if len(sys.argv) > 1 else 14
check = sys.argv[2] if len(sys.argv) > 2 else "gpu"
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
n = 1 << nv
ranks = Ranks()
world, rank = ranks.world, ranks.rank
L = load()
sh = ranks.connect(ml.ShardedPCSProver.one_rank(rank, world, ranks.local, nv))
evals = ml.synthetic_elements_dev(0xB200, n)
block = evals.ptr.value + rank * (n // world) * 16
inputs = ml.synthetic_elements_dev(0xC1A1, nv).elems()
ob = (C.c_uint8 * 16)()
ml.check(L.ml_mle_evals_evaluate_dev(evals.ptr, C.c_size_t(n), C.c_void_p(inputs.ctypes.data), C.c_size_t(nv), ob, None))
output = int.from_bytes(bytes(ob), "little")
state = {}


def prove():
    t = ml.Transcript()
    p = sh.prove_dev(inputs, output, [block], t)
    state["t"] = t.random()
    return p


ms, proof = ranks.timed(sh, prove, reps)
phases = sh.phase_ms()
agree = ranks.agree(state["t"])

if rank == 0:
    blob = proof.fri_proof.serialize()
    line = {"workload": "pcs_shard_prove", "n_gpus": world, "n_vars": nv, "prove_ms": ms, "proof_bytes": len(blob),
            "proof_sha256": hashlib.sha256(blob).hexdigest(), "verifies": proof.verify(ml.Transcript()) == 0, "transcripts_agree": agree,
            "arena_bytes_per_rank": sh.arena_bytes(),
            "rank0_phase_ms": dict(zip(["S0_encode_exchange_tables", "S1_combine", "sharded_rounds", "tail_chain", "openings_proof"], phases))}
    if check == "oracle":
        from oracle.binding import Oracle
        O = Oracle(threads=os.cpu_count() or 1)
        ev = evals.elems()
        ot = O.transcript()
        op, st = O.pcs_prove(inputs, output, ev, ot)
        line["matches_oracle"] = bool(st == 0 and op.fri.blob == blob and ot.random() == state["t"] and
                                      [c for nz in proof.sumcheck_polynomials for c in nz] == op.sumcheck)
    elif check == "gpu":
        t1 = ml.Transcript()
        single = ml.PCSProof.prove_dev(inputs, output, evals, n, t1)
        line["matches_single_gpu_prover"] = bool(single.fri_proof.serialize() == blob and t1.random() == state["t"])
        del single
    print(json.dumps(line), flush=True)
del proof
ranks.close(sh)
