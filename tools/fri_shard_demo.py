"""reed_solomon + FriProof::prove of one polynomial sharded over N GPUs, one process per GPU (torchrun): ml_fri_shard_* with the
arenas connected through CUDA IPC records all-gathered over torch.distributed — the only collective; the data path is NVLink
stores + device flags.

    torchrun --nproc-per-node N tools/fri_shard_demo.py <log_n> [check] [reps]

Every process generates all 2^log_n synthetic coefficients (seed 0xF21) on its GPU and passes a pointer to its own block.
`check`: `oracle` compares the proof with the CPU oracle's (small sizes); `gpu` with the unsharded prover on rank 0's GPU."""
import ctypes as C
import hashlib
import json
import os
import sys

from shard_harness import Ranks

from multilinear_b200 import api as ml
from multilinear_b200 import load

log_n = int(sys.argv[1]) if len(sys.argv) > 1 else 14
check = sys.argv[2] if len(sys.argv) > 2 else "gpu"
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
n = 1 << log_n
ranks = Ranks()
world, rank = ranks.world, ranks.rank
L = load()
sh = ranks.connect(ml.ShardedFriProver.one_rank(rank, world, ranks.local, log_n))
coeffs = ml.synthetic_elements_dev(0xF21, n)
block = coeffs.ptr.value + rank * (n // world) * 16
state = {}


def prove():
    t = ml.Transcript()
    p = sh.rs_prove_dev([block], t)
    state["t"] = t.random()
    return p


ms, proof = ranks.timed(sh, prove, reps)
phases = sh.phase_ms()
agree = ranks.agree(state["t"])

if rank == 0:
    blob = proof.serialize()
    line = {"workload": "fri_shard_prove", "n_gpus": world, "log_n": log_n, "prove_ms": ms, "proof_bytes": len(blob),
            "proof_sha256": hashlib.sha256(blob).hexdigest(), "verifies": proof.verify() == 0, "transcripts_agree": agree,
            "arena_bytes_per_rank": sh.arena_bytes(),
            "rank0_phase_ms": dict(zip(["S0_transpose_encode_exchange", "S1_combine", "sharded_rounds", "tail_chain", "openings_proof"], phases))}
    if check == "oracle":
        from oracle.binding import Oracle, fe_ints
        O = Oracle(threads=os.cpu_count() or 1)
        c = coeffs.elems()
        gp = O.pow2_generator_powers(log_n + 1)
        ot = O.transcript()
        op, st = O.fri_prove(O.reed_solomon(c, fe_ints(gp[1:2])[0]), gp, ot)
        line["matches_oracle"] = bool(st == 0 and op.blob == blob and ot.random() == state["t"])
    elif check == "gpu":
        t1 = ml.Transcript()
        h = C.c_void_p()
        ml.check(L.ml_rs_fri_prove_dev(coeffs.ptr, C.c_size_t(n), t1.h, None, C.byref(h)))
        single = ml.FriProof(h)
        line["matches_single_gpu_prover"] = bool(single.serialize() == blob and t1.random() == state["t"])
        del single
    print(json.dumps(line), flush=True)
del proof
ranks.close(sh)
