"""ml_bfri_shard_* measurements in one process (single-process handles over real GPUs).

    python tools/bfri_shard_bench.py --out DIR [--reps 10] [--shapes 64:22,8:24] [--worlds 2,4,8]

Shapes B:log_n are B polynomials of 2^log_n synthetic coefficients (seeds 0xBF5000 + j) and their RS codes, the shape of the
reference's batched_fri_benchmark (reed_solomon of each polynomial, then BatchedFriProof::prove).  64:22 is BASELINE config 5's
batch.  Per shape, on device 0:
  - host entry: ml_bfri_shard_prove on a G = 1 handle against ml_batched_fri_prove, both from the same page-locked host codes
    (copies included), alternating call by call; every call is bracketed by CUDA events on the stream the call runs on, and the
    proof bytes and transcripts of both are compared on every call;
  - ml_bfri_shard_prove_dev on a G = 1 handle from device-resident codes alone, with rank 0's phase marks.
Then rs_prove_dev from device-resident coefficients with G = 2, 4, 8 ranks on separate GPUs where the box has them (skipped
otherwise); a call's time is the maximum over its ranks' streams and its bytes must equal the G = 1 handle's.  One warm-up call
per prover; medians of --reps.  The codes are 8 GB (64:22) and 4 GB (8:24), far larger than the 126 MB L2.
Writes DIR/r7_bfri_shard_timing.json; GPU name, power limit and SM clocks are read in the same run."""
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
PHASES = ["S0_transpose_encode_exchange", "S1_combine_batch_tree", "S2_batch_root", "sharded_rounds", "tail_chain", "openings_proof"]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout
        return [l.strip() for l in out.splitlines() if l.strip()]
    except Exception as e:  # noqa: BLE001
        return ["nvidia-smi unavailable: %s" % e]


def timed(streams, fn):
    """fn() under CUDA events on every (device, stream); returns (result, max ms over the streams)"""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in streams]
    for (d, s), (a, _) in zip(streams, ev):
        a.record(s)
    out = fn()
    for (d, s), (_, b) in zip(streams, ev):
        b.record(s)
    for d, _ in streams:
        torch.cuda.synchronize(d)
    return out, max(a.elapsed_time(b) for a, b in ev)


def med(xs):
    return {"median": statistics.median(xs), "min": min(xs), "all": xs}


def shape(B, log_n, reps, worlds):
    n = 1 << log_n
    ml.set_device(0)
    dev0 = torch.device("cuda", 0)
    row = {"B": B, "log_n": log_n, "code_bytes_total": B * 2 * n * 16}
    gp = ml.pow_2_generator_powers(log_n + 1)
    gen = ml.to_ints(gp[1:2])[0]
    coeffs_dev = [ml.synthetic_elements_dev(0xBF5000 + j, n) for j in range(B)]
    codes = [ml.reed_solomon(c.elems(), gen) for c in coeffs_dev]
    for c in codes:  # page-locked, so both host entries upload at pinned-memory speed
        ml.check(L_.ml_host_register(C.c_void_p(c.ctypes.data), C.c_size_t(c.nbytes)))
    ptrs = (C.c_void_p * B)(*[c.ctypes.data for c in codes])

    # --- host entry, G = 1, against ml_batched_fri_prove (alternating)
    sh = ml.ShardedBatchedFriProver.single_process([0], B, log_n)
    s_sh = torch.cuda.ExternalStream(sh.stream(0), device=dev0)
    s_lib = torch.cuda.Stream(device=dev0)

    def host_sharded():
        t = ml.Transcript()
        h = C.c_void_p()
        ml.check(L_.ml_bfri_shard_prove(sh.h, ptrs, C.c_size_t(B), C.c_size_t(2 * n), None, C.c_size_t(0), t.h, C.byref(h)))
        return ml.FriProof(h, batched=True), t.random()

    def host_single():
        ml.check(L_.ml_set_thread_stream(C.c_void_p(s_lib.cuda_stream), C.c_int(1)))
        try:
            t = ml.Transcript()
            h = C.c_void_p()
            ml.check(L_.ml_batched_fri_prove(ptrs, C.c_size_t(B), C.c_size_t(2 * n), None, C.c_size_t(0), t.h, C.byref(h)))
            return ml.FriProof(h, batched=True), t.random()
        finally:
            ml.check(L_.ml_set_thread_stream(None, C.c_int(0)))

    (p, _), _ = timed([(0, s_sh)], host_sharded)  # warm-up
    row["verifies"] = p.verify() == 0
    ref_blob = p.serialize()
    del p
    timed([(0, s_lib)], host_single)
    ts, tu, same = [], [], []
    for _ in range(reps):
        (p, r), ms = timed([(0, s_sh)], host_sharded)
        (p1, r1), ms1 = timed([(0, s_lib)], host_single)
        ts.append(ms)
        tu.append(ms1)
        same.append(p.serialize() == p1.serialize() == ref_blob and r == r1)
        del p, p1
    row["host_entry_g1_ms"], row["ml_batched_fri_prove_ms"] = med(ts), med(tu)
    row["host_entry_g1_over_unsharded"] = statistics.median(ts) / statistics.median(tu)
    row["proof_equals_unsharded_every_call"] = all(same)

    # --- prove_dev, G = 1, from device-resident codes
    codes_dev = [ml.DeviceBuffer.from_host(c) for c in codes]
    for c in codes:
        ml.check(L_.ml_host_unregister(C.c_void_p(c.ctypes.data)))
    del codes
    blocks = [c.ptr.value for c in codes_dev]

    def dev_sharded():
        t = ml.Transcript()
        return sh.prove_dev(blocks, t), t.random()

    timed([(0, s_sh)], dev_sharded)
    td, phases, same = [], [], []
    for _ in range(reps):
        (p, _), ms = timed([(0, s_sh)], dev_sharded)
        td.append(ms)
        phases.append(sh.phase_ms())
        same.append(p.serialize() == ref_blob)
        del p
    row["prove_dev_g1_ms"] = med(td)
    row["prove_dev_g1_proof_equals_every_call"] = all(same)
    row["prove_dev_g1_rank0_phase_ms_median"] = {k: statistics.median(ph[i] for ph in phases) for i, k in enumerate(PHASES)
                                                 if all(len(ph) > i for ph in phases)}
    row["arena_bytes_g1"] = sh.arena_bytes()
    sh.free()
    for c in codes_dev:
        c.free()
    host_coeffs = [c.elems() for c in coeffs_dev]
    for c in coeffs_dev:
        c.free()
    del coeffs_dev

    # --- rs_prove_dev over G separate GPUs
    row["multi_gpu"] = []
    for G in worlds:
        if G > torch.cuda.device_count():
            row["multi_gpu"].append({"G": G, "measured": False, "reason": "needs %d GPUs, this box has %d" % (G, torch.cuda.device_count())})
            continue
        bufs = []
        for g in range(G):  # rank g's blocks only
            ml.set_device(g)
            bufs.append([ml.DeviceBuffer.from_host(c[g * (n // G):(g + 1) * (n // G)]) for c in host_coeffs])
        msh = ml.ShardedBatchedFriProver.single_process(list(range(G)), B, log_n)
        streams = [(g, torch.cuda.ExternalStream(msh.stream(g), device=torch.device("cuda", g))) for g in range(G)]
        ptrs_g = [b.ptr.value for g in range(G) for b in bufs[g]]

        def multi():
            t = ml.Transcript()
            return msh.rs_prove_dev(ptrs_g, t)

        timed(streams, multi)
        tm, phases, same = [], [], []
        for _ in range(reps):
            p, ms = timed(streams, multi)
            tm.append(ms)
            phases.append(msh.phase_ms())
            same.append(p.serialize() == ref_blob)
            del p
        mrow = {"G": G, "measured": True, "rs_prove_dev_ms": med(tm), "proof_equals_g1_every_call": all(same),
                "arena_bytes_per_rank": msh.arena_bytes(),
                "rank0_phase_ms_median": {k: statistics.median(ph[i] for ph in phases) for i, k in enumerate(PHASES)
                                          if all(len(ph) > i for ph in phases)}}
        msh.free()
        for g in range(G):
            for b in bufs[g]:
                b.free()
        row["multi_gpu"].append(mrow)
    ml.set_device(0)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--shapes", default="64:22,8:24")
    ap.add_argument("--worlds", default="2,4,8")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this benchmark measures on the device only")
    os.makedirs(args.out, exist_ok=True)
    worlds = [int(x) for x in args.worlds.split(",") if x]
    res = {"workload": "bfri_shard_timing", "reps": args.reps, "gpus": gpu_info(), "results": []}
    for spec in args.shapes.split(","):
        B, log_n = (int(x) for x in spec.split(":"))
        row = shape(B, log_n, args.reps, worlds)
        print(json.dumps(row), flush=True)
        res["results"].append(row)
    res["gpus_after"] = gpu_info()
    with open(os.path.join(args.out, "r7_bfri_shard_timing.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
