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

sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
import torch
import torch.distributed as dist

from multilinear_b200 import api as ml

log_n = int(sys.argv[1]) if len(sys.argv) > 1 else 14
B = int(sys.argv[2]) if len(sys.argv) > 2 else 4
check = sys.argv[3] if len(sys.argv) > 3 else "gpu"
reps = int(sys.argv[4]) if len(sys.argv) > 4 else 3
n = 1 << log_n
world, rank, local = int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
ml.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)


def barrier():
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()


sh = ml.ShardedBatchedFriProver.one_rank(rank, world, local, B, log_n)
if world > 1:
    sh.connect_over(dist, dev)
else:
    sh.connect(sh.export())
coeffs = [ml.synthetic_elements_dev(0xBF0 + j, n) for j in range(B)]
blocks = [c.ptr.value + rank * (n // world) * 16 for c in coeffs]
torch.cuda.synchronize()
stream = torch.cuda.ExternalStream(sh.stream(0), device=dev)
state = {}


def prove():
    t = ml.Transcript()
    p = sh.rs_prove_dev(blocks, t)
    state["t"] = t.random()
    return p


barrier()
prove()  # warm-up
barrier()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record(stream)
for _ in range(reps):
    proof = prove()
e1.record(stream)
barrier()
ms = e0.elapsed_time(e1) / reps
phases = sh.phase_ms()
tr = torch.tensor(list(state["t"]), dtype=torch.uint8, device=dev)
agree = True
if world > 1:
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    tr0 = tr.clone()
    dist.broadcast(tr0, 0)
    flag = torch.tensor([int(torch.equal(tr, tr0))], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    agree = bool(int(flag[0]))

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
barrier()
sh.free()
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
