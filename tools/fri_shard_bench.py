"""ml_fri_shard_* measurements in one process (single-process handles over real GPUs).

    python tools/fri_shard_bench.py --out DIR [--reps 10] [--runs 1:24,2:24,4:24,8:24,2:27,4:27,8:27,8:30]

Each run G:log_n is reed_solomon + FriProof::prove of synthetic(0xF21, 2^log_n) coefficients with G ranks, one device each; runs
whose G exceeds the box's GPUs are skipped.  Every call is bracketed by CUDA events on every rank's stream; a call's time is the
maximum over its ranks.  Where the code fits one GPU (log_n <= 27) the unsharded ml_rs_fri_prove_dev runs on device 0 on the
same coefficients, alternating call by call with the sharded prover, and the proof bytes and transcripts of both are compared
on every call.  One warm-up call per prover.  The coefficients are 256 MB and more per GPU (larger than the 126 MB L2).
log_n 30 does not fit one GPU: it runs sharded only and its proof must verify.  Reports the phase marks of rank 0, the arena
bytes and the stream-ordered pool bytes reserved per rank (the pools keep what they reserved, so this bounds the peak).
Writes DIR/r6_fri_shard_timing.json; GPU name, power limit and SM clocks are read in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch

from multilinear_b200 import api as ml
from multilinear_b200 import load

L_ = load()
PHASES = ["S0_transpose_encode_exchange", "S1_combine", "sharded_rounds", "tail_chain", "openings_proof"]
SINGLE_MAX_LOG_N = 27


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout
        return [l.strip() for l in out.splitlines() if l.strip()]
    except Exception as e:  # noqa: BLE001
        return ["nvidia-smi unavailable: %s" % e]


def pool_reserved(dev):
    ml.set_device(dev)
    r, u = C.c_uint64(), C.c_uint64()
    ml.check(L_.ml_pool_stats(C.byref(r), C.byref(u)))
    return r.value


def run(G, log_n, reps):
    n = 1 << log_n
    coeffs = []
    for d in range(G):  # the whole polynomial on every device; rank d reads its block
        ml.set_device(d)
        coeffs.append(ml.synthetic_elements_dev(0xF21, n))
        torch.cuda.synchronize(d)
    row = {"G": G, "log_n": log_n}
    sh = ml.ShardedFriProver.single_process(list(range(G)), log_n)
    blocks = [coeffs[g].ptr.value + g * (n // G) * 16 for g in range(G)]
    streams = [torch.cuda.ExternalStream(sh.stream(g), device=torch.device("cuda", g)) for g in range(G)]
    single_stream = torch.cuda.Stream(device=torch.device("cuda", 0))

    def sharded():
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(G)]
        for g in range(G):
            ev[g][0].record(streams[g])
        t = ml.Transcript()
        p = sh.rs_prove_dev(blocks, t)
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
        h = C.c_void_p()
        ml.check(L_.ml_rs_fri_prove_dev(coeffs[0].ptr, C.c_size_t(n), t.h, C.c_void_p(single_stream.cuda_stream), C.byref(h)))
        b.record(single_stream)
        torch.cuda.synchronize(0)
        return a.elapsed_time(b), ml.FriProof(h), t.random()

    compare = log_n <= SINGLE_MAX_LOG_N
    _, p, _ = sharded()  # warm-up
    row["verifies"] = p.verify() == 0
    del p
    if compare:
        single()
    ts, tu, phases, same = [], [], [], []
    for _ in range(reps):
        ms, p, r = sharded()
        ts.append(ms)
        phases.append(sh.phase_ms())
        if compare:
            ms1, p1, r1 = single()
            tu.append(ms1)
            same.append(p.serialize() == p1.serialize() and r == r1)
            del p1
        del p
    row["sharded_ms_median"], row["sharded_ms_min"], row["sharded_ms_all"] = statistics.median(ts), min(ts), ts
    if compare:
        row["single_gpu_ms_median"], row["single_gpu_ms_min"], row["single_gpu_ms_all"] = statistics.median(tu), min(tu), tu
        row["speedup_median"] = statistics.median(tu) / statistics.median(ts)
        row["proof_equals_single_gpu_every_call"] = all(same)
    row["rank0_phase_ms_median"] = {k: statistics.median(ph[i] for ph in phases) for i, k in enumerate(PHASES) if all(len(ph) > i for ph in phases)}
    row["arena_bytes_per_rank"] = sh.arena_bytes()
    row["pool_reserved_bytes_per_rank"] = [pool_reserved(d) for d in range(G)]
    row["coefficient_bytes_per_gpu"] = 16 * n
    sh.free()
    for b in coeffs:
        b.free()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--runs", default="1:24,2:24,4:24,8:24,2:27,4:27,8:27,8:30")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this benchmark measures on the device only")
    os.makedirs(args.out, exist_ok=True)
    res = {"workload": "fri_shard_rs_prove_timing", "reps": args.reps, "gpus": gpu_info(), "results": [], "skipped": []}
    for spec in args.runs.split(","):
        G, log_n = (int(x) for x in spec.split(":"))
        if G > torch.cuda.device_count():
            res["skipped"].append({"G": G, "log_n": log_n, "reason": "needs %d GPUs, this box has %d" % (G, torch.cuda.device_count())})
            continue
        try:
            row = run(G, log_n, args.reps)
        except ml.MlError as e:
            row = {"G": G, "log_n": log_n, "error": str(e)}
        print(json.dumps(row), flush=True)
        res["results"].append(row)
    res["gpus_after"] = gpu_info()
    with open(os.path.join(args.out, "r6_fri_shard_timing.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
