"""Timing of the stream-ordered provers (ml_prove_plan_*) against the blocking ml_rs_fri_prove_dev, on one GPU.

    python tools/prove_plan_bench.py [--out profiles/r8_prove_plan_timing.json] [--log-n 24 20] [--reps 12]

At each size (log_n coefficients, code of 2^(log_n+1) elements; inputs generated on the device, 256 MiB at 2^24, larger than
the 126 MB L2) it records, with the card's name, power limit and clocks read in the same run:
  - serial latency: rs_fri_prove_async + one stream synchronise vs ml_rs_fri_prove_dev, alternating, CUDA events and host clock,
    medians of --reps;
  - the device time of fri_query_indices_kernel and fri_proof_write_kernel, from torch.profiler in a run of their own;
  - throughput: K plans on K streams driven by one host thread vs K host threads each blocking in ml_rs_fri_prove_dev on its own
    stream, K in 1 2 4 6 8, proofs/s over --reps proofs per stream;
  - graph replay: host time of the enqueue alone and device time per proof, one captured rs_fri_prove_async replayed vs the
    eager call.
Every async proof timed is compared once per size with the blocking proof's bytes and transcript."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch

from multilinear_b200 import api as ml
from multilinear_b200 import load
from shard_harness import gpu_info

_vp, _sz = C.c_void_p, C.c_size_t


def synthetic(seed, n, stream):
    t = torch.empty(16 * n, dtype=torch.uint8, device="cuda")
    ml.check(load().ml_synthetic_elements_dev(C.c_uint64(seed), _sz(n), _vp(t.data_ptr()), _vp(stream.cuda_stream)))
    return t


class AsyncSlot:
    """one plan with its output buffers on one stream; `state` is the starting transcript state kept in HBM"""

    def __init__(self, log_n, stream, seed):
        self.plan = ml.ProvePlan.create(log_n + 1, False)
        self.stream = stream
        self.coeffs = synthetic(seed, 1 << log_n, stream)
        self.state = torch.frombuffer(bytearray(ml.Transcript().export()), dtype=torch.uint8).cuda()
        self.tr = torch.empty(112, dtype=torch.uint8, device="cuda")
        self.proof = torch.empty(self.plan.proof_bytes, dtype=torch.uint8, device="cuda")
        self.status = torch.empty(4, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()

    def enqueue(self):
        with torch.cuda.stream(self.stream):
            self.tr[:104].copy_(self.state)   # a fresh transcript for every proof (a device-to-device copy)
        self.plan.rs_fri_prove_async(self.coeffs.data_ptr(), self.tr.data_ptr(), self.proof.data_ptr(), self.status.data_ptr(),
                                     self.stream.cuda_stream)


def blocking_prove(coeffs, n, stream):
    t, h = ml.Transcript(), _vp()
    ml.check(load().ml_rs_fri_prove_dev(_vp(coeffs.data_ptr()), _sz(n), t.h, _vp(stream.cuda_stream), C.byref(h)))
    return ml.FriProof(h), t


def check_equal(slot, log_n):
    slot.stream.synchronize()
    p, t = blocking_prove(slot.coeffs, 1 << log_n, slot.stream)
    assert int(slot.status.cpu()[0]) == 0
    assert bytes(slot.proof.cpu().numpy()) == p.serialize(), "async proof differs from the blocking one"
    assert bytes(slot.tr[:104].cpu().numpy()) == t.export(), "async transcript differs from the blocking one"


def serial_latency(log_n, reps):
    s = torch.cuda.Stream()
    slot = AsyncSlot(log_n, s, 11)
    slot.enqueue()
    check_equal(slot, log_n)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {"async_ms": [], "async_host_ms": [], "blocking_ms": [], "blocking_host_ms": []}
    for _ in range(reps):
        for kind in ("async", "blocking"):
            s.synchronize()
            h0 = time.perf_counter()
            ev0.record(s)
            if kind == "async":
                slot.enqueue()
            else:
                blocking_prove(slot.coeffs, 1 << log_n, s)
            ev1.record(s)
            ev1.synchronize()
            res[kind + "_host_ms"].append((time.perf_counter() - h0) * 1e3)
            res[kind + "_ms"].append(ev0.elapsed_time(ev1))
    out = {k + "_median": statistics.median(v) for k, v in res.items()}
    out["reps"] = reps
    slot.plan.free()
    return out


def kernel_costs(log_n, reps=5):
    from torch.profiler import ProfilerActivity, profile
    s = torch.cuda.Stream()
    slot = AsyncSlot(log_n, s, 12)
    slot.enqueue()
    s.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            slot.enqueue()
        s.synchronize()
    out = {}
    for e in prof.key_averages():
        for name in ("fri_query_indices_kernel", "fri_proof_write_kernel", "chain_tail_kernel"):
            if name in e.key:
                total = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                out[name + "_us"] = total / max(e.count, 1)
                out[name + "_count"] = e.count
    slot.plan.free()
    return out


def throughput(log_n, ks, reps):
    out = {}
    n = 1 << log_n
    for k in ks:
        streams = [torch.cuda.Stream() for _ in range(k)]
        slots = [AsyncSlot(log_n, streams[i], 100 + i) for i in range(k)]
        for sl in slots:   # warm-up and correctness of every plan
            sl.enqueue()
        for sl in slots:
            check_equal(sl, log_n)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            for sl in slots:
                sl.enqueue()
        torch.cuda.synchronize()
        one_thread = k * reps / (time.perf_counter() - t0)
        errors = []

        def worker(i):
            try:
                for _ in range(reps):
                    blocking_prove(slots[i].coeffs, n, streams[i])
            except Exception as e:  # noqa: BLE001
                errors.append(repr(e))
        for i in range(k):   # warm-up of the blocking path on every stream
            blocking_prove(slots[i].coeffs, n, streams[i])
        torch.cuda.synchronize()
        threads = [threading.Thread(target=worker, args=(i,)) for i in range(k)]
        t0 = time.perf_counter()
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        torch.cuda.synchronize()
        k_threads = k * reps / (time.perf_counter() - t0)
        out[str(k)] = {"one_thread_async_proofs_per_s": one_thread, "k_threads_blocking_proofs_per_s": k_threads,
                       "one_thread_async_ms_per_proof": 1e3 / one_thread, "k_threads_blocking_ms_per_proof": 1e3 / k_threads,
                       "errors": errors}
        for sl in slots:
            sl.plan.free()
    return out


def graph_replay(log_n, reps):
    s = torch.cuda.Stream()
    slot = AsyncSlot(log_n, s, 13)
    slot.enqueue()
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s, capture_error_mode="global"):
        slot.plan.rs_fri_prove_async(slot.coeffs.data_ptr(), slot.tr.data_ptr(), slot.proof.data_ptr(), slot.status.data_ptr(), s.cuda_stream)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {}
    for kind in ("eager", "graph", "eager", "graph"):
        host = []
        s.synchronize()
        ev0.record(s)
        for _ in range(reps):
            with torch.cuda.stream(s):
                slot.tr[:104].copy_(slot.state)
            h0 = time.perf_counter()
            if kind == "graph":
                with torch.cuda.stream(s):
                    g.replay()
            else:
                slot.plan.rs_fri_prove_async(slot.coeffs.data_ptr(), slot.tr.data_ptr(), slot.proof.data_ptr(), slot.status.data_ptr(),
                                             s.cuda_stream)
            host.append((time.perf_counter() - h0) * 1e3)
        ev1.record(s)
        ev1.synchronize()
        res[kind + "_host_enqueue_ms_median"] = statistics.median(host)
        res[kind + "_device_ms_per_proof"] = ev0.elapsed_time(ev1) / reps
    check_equal(slot, log_n)   # the last replay's proof
    del g
    slot.plan.free()
    res["reps"] = reps
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r8_prove_plan_timing.json"))
    ap.add_argument("--log-n", type=int, nargs="+", default=[24, 20])
    ap.add_argument("--reps", type=int, default=12)
    ap.add_argument("--ks", type=int, nargs="+", default=[1, 2, 4, 6, 8])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    ml.set_device(0)
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0), "sizes": {}}
    for log_n in args.log_n:
        r = {"log_n": log_n, "code_elements": 1 << (log_n + 1)}
        r["serial"] = serial_latency(log_n, args.reps)
        r["kernels"] = kernel_costs(log_n)
        r["throughput"] = throughput(log_n, args.ks, args.reps)
        r["graph"] = graph_replay(log_n, args.reps)
        res["sizes"][str(log_n)] = r
        print(json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
