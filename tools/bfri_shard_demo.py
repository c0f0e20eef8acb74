"""reed_solomon of B polynomials + BatchedFriProof::prove sharded by block over N GPUs, one process per GPU (torchrun):
ml_bfri_shard_* with the arenas connected through CUDA IPC records all-gathered over torch.distributed — the only collective; the
data path is NVLink stores + device flags.

    torchrun --nproc-per-node N tools/bfri_shard_demo.py <log_n> [n_codes] [check] [reps]

Every process generates all B x 2^log_n synthetic coefficients (seeds 0xBF0 + j) on its GPU and passes pointers to its own blocks.
`check`: `oracle` compares the proof with the CPU oracle's (small sizes); `gpu` with the unsharded prover (ml_batched_fri_prove)
on rank 0's GPU."""
import hashlib
import json
import os
import sys

from shard_harness import Ranks

from multilinear_b200 import api as ml

log_n = int(sys.argv[1]) if len(sys.argv) > 1 else 14
B = int(sys.argv[2]) if len(sys.argv) > 2 else 4
check = sys.argv[3] if len(sys.argv) > 3 else "gpu"
reps = int(sys.argv[4]) if len(sys.argv) > 4 else 3
n = 1 << log_n
ranks = Ranks()
world, rank = ranks.world, ranks.rank
sh = ranks.connect(ml.ShardedBatchedFriProver.one_rank(rank, world, ranks.local, B, log_n))
coeffs = [ml.synthetic_elements_dev(0xBF0 + j, n) for j in range(B)]
blocks = [c.ptr.value + rank * (n // world) * 16 for c in coeffs]
state = {}


def prove():
    t = ml.Transcript()
    p = sh.rs_prove_dev(blocks, t)
    state["t"] = t.random()
    return p


ms, proof = ranks.timed(sh, prove, reps)
phases = sh.phase_ms()
agree = ranks.agree(state["t"])

if rank == 0:
    blob = proof.serialize()
    line = {"workload": "bfri_shard_prove", "n_gpus": world, "n_codes": B, "log_n": log_n, "prove_ms": ms, "proof_bytes": len(blob),
            "proof_sha256": hashlib.sha256(blob).hexdigest(), "verifies": proof.verify() == 0, "transcripts_agree": agree,
            "arena_bytes_per_rank": sh.arena_bytes(),
            "rank0_phase_ms": dict(zip(["S0_transpose_encode_exchange", "S1_combine_batch_tree", "S2_batch_root", "sharded_rounds",
                                        "tail_chain", "openings_proof"], phases))}
    host = [c.elems() for c in coeffs]
    if check == "oracle":
        from oracle.binding import Oracle, fe_ints
        O = Oracle(threads=os.cpu_count() or 1)
        gp = O.pow2_generator_powers(log_n + 1)
        gen = fe_ints(gp[1:2])[0]
        ot = O.transcript()
        op, st = O.batched_fri_prove([O.reed_solomon(c, gen) for c in host], gp, ot)
        line["matches_oracle"] = bool(st == 0 and op.blob == blob and ot.random() == state["t"])
    elif check == "gpu":
        gp = ml.pow_2_generator_powers(log_n + 1)
        gen = ml.to_ints(gp[1:2])[0]
        t1 = ml.Transcript()
        single = ml.BatchedFriProof.prove([ml.reed_solomon(c, gen) for c in host], gp, t1)
        line["matches_single_gpu_prover"] = bool(single.serialize() == blob and t1.random() == state["t"])
        del single
    print(json.dumps(line), flush=True)
del proof
ranks.close(sh)
