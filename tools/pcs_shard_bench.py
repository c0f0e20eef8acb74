"""ml_pcs_shard_* measurements in one process (single-process handles over real GPUs).

    python tools/pcs_shard_bench.py --out DIR [--log-n 24] [--reps 10] [--gpus 1,2,4,8] [--big 30,31]

Timing: PCSProof::prove of synthetic(0xB200, 2^log_n) with G = 1, 2, 4, 8 ranks, alternating call by call with the unsharded
ml_pcs_prove_dev on the same inputs (device 0).  Every call is bracketed by CUDA events on every rank's stream; a call's time is
the maximum over its ranks.  One warm-up call per variant; the proof bytes of both provers are compared.  The inputs are 256 MB
per GPU (larger than the 126 MB L2).
Largest size: n_vars 30 (and 31 if it fits) on 8 GPUs, the full synthetic polynomial generated on every GPU and block pointers
passed in; the claim is sum_b eq(inputs[0:L], b) * MLE(block_b)(inputs[L:]); the proof must verify.  Reports the arena and the
peak stream-ordered pool bytes per rank.
Writes DIR/r3_pcs_shard_timing.json and DIR/r3_pcs_shard_largest.json; GPU name, power limit and SM clock are read in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch

from multilinear_b200 import api as ml
from multilinear_b200 import load

L_ = load()
M = (1 << 128) - 45 * (1 << 40) + 1  # the field modulus


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout
        return [l.strip() for l in out.splitlines() if l.strip()]
    except Exception as e:  # noqa: BLE001
        return ["nvidia-smi unavailable: %s" % e]


def pool_stats(dev):
    ml.set_device(dev)
    r, u = C.c_uint64(), C.c_uint64()
    ml.check(L_.ml_pool_stats(C.byref(r), C.byref(u)))
    return r.value, u.value


def synthetic_on(dev, seed, n):
    ml.set_device(dev)
    b = ml.synthetic_elements_dev(seed, n)
    torch.cuda.synchronize(dev)
    return b


def mle_dev(buf_ptr, n, args):
    a = ml.as_elems(args)
    ob = (C.c_uint8 * 16)()
    ml.check(L_.ml_mle_evals_evaluate_dev(C.c_void_p(buf_ptr), C.c_size_t(n), C.c_void_p(a.ctypes.data), C.c_size_t(a.shape[0]), ob, None))
    return int.from_bytes(bytes(ob), "little")


def eq_weight(pts, b, L):
    """eq(inputs[0:L], b): bit L-1-t of b <-> inputs[t] (the block index is the top L bits of the evaluation index)"""
    w = 1
    for t in range(L):
        p = pts[t]
        w = w * (p if (b >> (L - 1 - t)) & 1 else (1 - p) % M) % M
    return w


def timing(args, info):
    nv, n = args.log_n, 1 << args.log_n
    gs = [int(x) for x in args.gpus.split(",") if int(x) <= torch.cuda.device_count()]
    evals = {d: synthetic_on(d, 0xB200, n) for d in range(max(gs))}
    inputs = ml.synthetic_elements_dev(0xB2000001, nv).elems()
    ml.set_device(0)
    output = mle_dev(evals[0].ptr.value, n, inputs)
    res = {"workload": "pcs_shard_prove_timing", "n_vars": nv, "reps": args.reps, "gpus": info, "results": []}
    for G in gs:
        sh = ml.ShardedPCSProver.single_process(list(range(G)), nv)
        blocks = [evals[g].ptr.value + g * (n // G) * 16 for g in range(G)]
        streams = [torch.cuda.ExternalStream(sh.stream(g), device=torch.device("cuda", g)) for g in range(G)]
        single_stream = torch.cuda.Stream(device=torch.device("cuda", 0))

        def sharded():
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(G)]
            for g in range(G):
                ev[g][0].record(streams[g])
            t = ml.Transcript()
            p = sh.prove_dev(inputs, output, blocks, t)
            for g in range(G):
                ev[g][1].record(streams[g])
            for g in range(G):
                torch.cuda.synchronize(g)
            return max(a.elapsed_time(b) for a, b in ev), p, t.random()

        def single():
            ml.set_device(0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(single_stream)
            t = ml.Transcript()
            p = ml.PCSProof.prove_dev(inputs, output, evals[0], n, t, stream=single_stream.cuda_stream)
            b.record(single_stream)
            torch.cuda.synchronize(0)
            return a.elapsed_time(b), p, t.random()

        _, p1, r1 = sharded()
        _, p2, r2 = single()
        same = p1.fri_proof.serialize() == p2.fri_proof.serialize() and r1 == r2 and p1.sumcheck_polynomials == p2.sumcheck_polynomials
        del p1, p2
        ts, tu, phases = [], [], []
        for _ in range(args.reps):
            ms, p, _ = sharded()
            ts.append(ms)
            phases.append(sh.phase_ms())
            del p
            ms, p, _ = single()
            tu.append(ms)
            del p
        names = ["S0_encode_exchange_tables", "S1_combine", "sharded_rounds", "tail_chain", "openings_proof"]
        med_phases = {k: statistics.median(ph[i] for ph in phases) for i, k in enumerate(names) if all(len(ph) > i for ph in phases)}
        row = {"G": G, "sharded_ms_median": statistics.median(ts), "sharded_ms_min": min(ts), "sharded_ms_all": ts,
               "single_gpu_ms_median": statistics.median(tu), "single_gpu_ms_min": min(tu), "single_gpu_ms_all": tu,
               "speedup_median": statistics.median(tu) / statistics.median(ts), "rank0_phase_ms_median": med_phases,
               "proof_equals_single_gpu": same, "arena_bytes_per_rank": sh.arena_bytes()}
        print(json.dumps(row), flush=True)
        res["results"].append(row)
        sh.free()
    for b in evals.values():
        b.free()
    return res


def largest(args, info):
    G, L = 8, 3
    out = {"workload": "pcs_shard_prove_largest", "G": G, "gpus": info, "results": []}
    if torch.cuda.device_count() < G:
        out["skipped"] = "needs %d GPUs, this box has %d" % (G, torch.cuda.device_count())
        return out
    for nv in [int(x) for x in args.big.split(",") if x]:
        n = 1 << nv
        row = {"n_vars": nv}
        try:
            sh = ml.ShardedPCSProver.single_process(list(range(G)), nv)
        except ml.MlError as e:
            row["error"] = str(e)
            out["results"].append(row)
            print(json.dumps(row), flush=True)
            break
        evals = []
        try:
            for d in range(G):
                evals.append(synthetic_on(d, 0xB200, n))
            inputs = ml.synthetic_elements_dev(0xB2000001, nv).elems()
            pts = ml.to_ints(inputs)
            claim = 0
            for b in range(G):
                ml.set_device(b)
                part = mle_dev(evals[b].ptr.value + b * (n // G) * 16, n // G, inputs[L:])
                claim = (claim + eq_weight(pts, b, L) * part) % M
            blocks = [evals[g].ptr.value + g * (n // G) * 16 for g in range(G)]
            t0 = time.time()
            t = ml.Transcript()
            p = sh.prove_dev(inputs, claim, blocks, t)
            row["wall_s"] = time.time() - t0
            row["rank0_phase_ms"] = dict(zip(["S0_encode_exchange_tables", "S1_combine", "sharded_rounds", "tail_chain", "openings_proof"], sh.phase_ms()))
            row["verifies"] = p.verify(ml.Transcript()) == 0
            row["arena_bytes_per_rank"] = sh.arena_bytes()
            row["pool_reserved_bytes_per_rank"] = [pool_stats(d)[0] for d in range(G)]
            row["device_used_bytes_per_rank"] = [torch.cuda.mem_get_info(d)[1] - torch.cuda.mem_get_info(d)[0] for d in range(G)]
            row["input_bytes_per_rank"] = 16 * n
            del p
        except ml.MlError as e:
            row["error"] = str(e)
        for b in evals:
            b.free()
        sh.free()
        out["results"].append(row)
        print(json.dumps(row), flush=True)
        if "error" in row:
            break
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--log-n", type=int, default=24, dest="log_n")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--big", default="30,31")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this benchmark measures on the device only")
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    res = timing(args, info)
    with open(os.path.join(args.out, "r3_pcs_shard_timing.json"), "w") as f:
        json.dump(res, f, indent=1)
    if args.big:
        big = largest(args, gpu_info())
        with open(os.path.join(args.out, "r3_pcs_shard_largest.json"), "w") as f:
            json.dump(big, f, indent=1)


if __name__ == "__main__":
    main()
