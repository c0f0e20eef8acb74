"""ml_bpcs_shard_* timing in one process (single-process handles over real GPUs).

    python tools/bpcs_shard_bench.py --out DIR [--shapes 10x20,3x24,64x22] [--reps 10] [--gpus 1,2,4,8]

For every shape B x n_vars (B synthetic polynomials, seeds 0xB200 + j, generated on every GPU used) and every G in --gpus that the
box has: BatchedPCSProof::prove through a G-rank ml_bpcs_shard handle on devices 0 .. G-1, alternating call by call with the
unsharded ml_batched_pcs_prove_dev on device 0 and, where G divides B and G >= 2, with the by-polynomial ml_shard_* handle on the
same devices.  Every call is bracketed by CUDA events on every rank's stream (plus a device synchronise); a call's time is the
maximum over its ranks.  One warm-up call per variant; medians of --reps; the proof bytes of all provers are compared.  The
shapes are the crate's batched_pcs_verify_test size (10 x 2^20), a few large polynomials (3 x 2^24) and bench.py's batch
(64 x 2^22).  Writes DIR/r4_bpcs_shard_timing.json; GPU name, power limit and SM clock are read in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

import torch
from shard_harness import gpu_info, timed

from multilinear_b200 import api as ml
from multilinear_b200 import load

L_ = load()


def unsharded(inputs, outputs, bufs, n, stream):
    ptrs = (C.c_void_p * len(bufs))(*[b.ptr.value for b in bufs])
    h = C.c_void_p()
    t = ml.Transcript()
    ml.check(L_.ml_batched_pcs_prove_dev(ml._p(inputs), ml._sz(inputs.shape[0]), ml._p(outputs), ml._sz(len(bufs)), ptrs, ml._sz(n), t.h,
                                         C.c_void_p(stream.cuda_stream), C.byref(h)))
    proof = ml.PCSProof(h, batched=True)  # owns the handle its fri_proof borrows
    return proof.fri_proof.serialize()


def blob_of(proof):
    return proof.fri_proof.serialize()


def shape_run(B, nv, gs, reps):
    n = 1 << nv
    G_max = max(gs)
    polys = {}
    for d in range(G_max):
        ml.set_device(d)
        polys[d] = [ml.synthetic_elements_dev(0xB200 + j, n) for j in range(B)]
        torch.cuda.synchronize(d)
    ml.set_device(0)
    inputs = ml.synthetic_elements_dev(0xB2000001, nv).elems()
    outputs = ml.synthetic_elements_dev(0xB2000002, B).elems()  # any claim: the provers do not check it
    s0 = torch.cuda.Stream(device=0)
    variants = {"unsharded_1gpu": ([(0, s0)], lambda: unsharded(inputs, outputs, polys[0], n, s0))}
    handles = []
    for G in gs:
        sh = ml.BlockShardedBatchedProver.single_process(list(range(G)), B, nv)
        handles.append(sh)
        st = [(d, torch.cuda.ExternalStream(sh.stream(d), device=d)) for d in range(G)]
        ptrs = [polys[g][j].ptr.value + g * (n // G) * 16 for g in range(G) for j in range(B)]
        variants["bpcs_shard_G%d" % G] = (st, lambda sh=sh, ptrs=ptrs: blob_of(sh.prove_dev(inputs, outputs, ptrs, ml.Transcript())))
        if G >= 2 and B % G == 0:
            ps = ml.ShardedBatchedProver.single_process(list(range(G)), B, nv)
            handles.append(ps)
            st2 = [(d, torch.cuda.ExternalStream(ps.stream(d), device=d)) for d in range(G)]
            lp = [polys[g][j].ptr.value for g, j in zip([r for r in range(G) for _ in range(B // G)], ps.local_polys())]
            variants["ml_shard_G%d" % G] = (st2, lambda ps=ps, lp=lp: blob_of(ps.prove_dev(inputs, outputs, lp, ml.Transcript())))
    blobs, times = {}, {k: [] for k in variants}
    for k, (st, fn) in variants.items():  # warm-up, and the bytes to compare
        blobs[k] = fn()
        for d, _ in st:
            torch.cuda.synchronize(d)
    for _ in range(reps):
        for k, (st, fn) in variants.items():
            times[k].append(timed(st, fn)[1])
    ref = blobs["unsharded_1gpu"]
    row = {"n_polys": B, "n_vars": nv, "median_ms": {k: statistics.median(v) for k, v in times.items()},
           "all_ms": times, "same_bytes_as_unsharded": {k: blobs[k] == ref for k in variants}}
    if "bpcs_shard_G1" in row["median_ms"]:
        row["G1_over_unsharded"] = row["median_ms"]["bpcs_shard_G1"] / row["median_ms"]["unsharded_1gpu"]
    for h in handles:
        h.free()
    del polys
    for d in range(G_max):
        torch.cuda.synchronize(d)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default="10x20,3x24,64x22")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--gpus", default="1,2,4,8")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bpcs_shard_bench: no GPU")
    gs = [int(x) for x in args.gpus.split(",") if int(x) <= torch.cuda.device_count()]
    res = {"workload": "bpcs_shard_prove_timing", "reps": args.reps, "gpus": gpu_info(), "device_count": torch.cuda.device_count(),
           "ranks_measured": gs, "results": []}
    for sh in args.shapes.split(","):
        B, nv = (int(x) for x in sh.split("x"))
        row = shape_run(B, nv, gs, args.reps)
        print(json.dumps({k: row[k] for k in row if k != "all_ms"}), flush=True)
        res["results"].append(row)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r4_bpcs_shard_timing.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
