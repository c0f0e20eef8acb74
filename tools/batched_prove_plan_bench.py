"""Timing of the stream-ordered batched provers (ml_batched_prove_plan_*) against their blocking twins, on one GPU.

    python tools/batched_prove_plan_bench.py [--out profiles/r9_batched_prove_plan_timing.json] [--reps 12]

With the card's name, power limit and clocks read in the same run, it records (inputs generated on the device; every working set
is larger than the 126 MB L2):
  - serial latency, async call + one stream synchronise vs the blocking twin, alternating, CUDA events on the stream and host
    clock, medians of --reps:
      64 x 2^22 evaluations, PCS kind, vs ml_batched_pcs_prove_dev;
      64 x 2^23 and 8 x 2^25 codes, CODES kind, vs ml_bfri_shard_prove_dev at one rank (the device-resident blocking batched FRI
      prover);
  - ms per proof with K = 1, 2, 4 PCS plans at 64 x 2^22 in flight on K streams from one host thread (the plans share the inputs);
  - host time of the enqueue, eager call vs replay of a captured graph of the same call;
  - the device time of batch_root_kernel and bfri_proof_write_kernel, from torch.profiler in a profiled pass after the timed ones.
Every timed async proof is compared once per shape with the blocking proof's bytes and transcript."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

from multilinear_b200 import api as ml
from multilinear_b200 import load
from shard_harness import gpu_info

_vp, _sz = C.c_void_p, C.c_size_t


def synthetic(seed, n):
    t = torch.empty(16 * n, dtype=torch.uint8, device="cuda")
    ml.check(load().ml_synthetic_elements_dev(C.c_uint64(seed), _sz(n), _vp(t.data_ptr()), _vp(torch.cuda.current_stream().cuda_stream)))
    return t


def rs_codes(B, D, seed):
    """B RS codes of 2^D elements from synthetic coefficients, in HBM"""
    gen = np.frombuffer(int(ml.pow_2_generator(D)).to_bytes(16, "little"), dtype=np.uint8).copy()
    out = []
    for j in range(B):
        c = synthetic(seed + j, 1 << (D - 1))
        code = torch.empty(16 << D, dtype=torch.uint8, device="cuda")
        ml.check(load().ml_reed_solomon_dev(_vp(c.data_ptr()), _sz(1 << (D - 1)), _vp(gen.ctypes.data), _vp(code.data_ptr()),
                                            _vp(torch.cuda.current_stream().cuda_stream)))
        out.append(code)
    torch.cuda.synchronize()
    return out


class Shape:
    """one batched prove: its inputs in HBM, a plan with its output buffers on `stream`, and the blocking twin"""

    def __init__(self, kind, B, D, stream, inputs=None):
        self.kind, self.B, self.D, self.stream = kind, B, D, stream
        if inputs is None:
            if kind == "pcs":
                inputs = ([synthetic(5000 + j, 1 << (D - 1)) for j in range(B)], synthetic(0xB2000001, D - 1), synthetic(0xB2000002, B))
            else:
                inputs = (rs_codes(B, D, 0xC0DE), None, None)
        self.inputs = inputs
        self.bufs, self.points, self.claims = inputs
        self.ptrs = [b.data_ptr() for b in self.bufs]
        self.plan = ml.BatchedProvePlan.create(D, B, kind)
        self.state = torch.frombuffer(bytearray(ml.Transcript().export()), dtype=torch.uint8).cuda()
        self.tr = torch.empty(112, dtype=torch.uint8, device="cuda")
        self.proof = torch.empty(self.plan.proof_bytes, dtype=torch.uint8, device="cuda")
        self.sc = torch.empty(32 * D, dtype=torch.uint8, device="cuda")
        self.status = torch.empty(4, dtype=torch.int32, device="cuda")
        self.shard = None
        if kind == "pcs":   # the blocking twin takes the claim from host memory
            self.host_points, self.host_claims = self.points.cpu().numpy(), self.claims.cpu().numpy()
        torch.cuda.synchronize()

    def enqueue(self):
        with torch.cuda.stream(self.stream):
            self.tr[:104].copy_(self.state)   # a fresh transcript for every proof (a device-to-device copy)
        s = self.stream.cuda_stream
        if self.kind == "pcs":
            self.plan.batched_pcs_prove_async(self.points.data_ptr(), self.claims.data_ptr(), self.ptrs, self.tr.data_ptr(), self.proof.data_ptr(),
                                              self.sc.data_ptr(), self.status.data_ptr(), s)
        else:
            self.plan.batched_fri_prove_async(self.ptrs, self.tr.data_ptr(), self.proof.data_ptr(), self.status.data_ptr(), s)

    def blocking(self):
        t = ml.Transcript()
        if self.kind == "pcs":
            pts, cl = self.host_points, self.host_claims
            arr, h = (C.c_void_p * self.B)(*self.ptrs), _vp()
            ml.check(load().ml_batched_pcs_prove_dev(_vp(pts.ctypes.data), _sz(self.D - 1), _vp(cl.ctypes.data), _sz(self.B), arr,
                                                     _sz(1 << (self.D - 1)), t.h, _vp(self.stream.cuda_stream), C.byref(h)))
            return ml.PCSProof(h, batched=True), t   # owns the batched FriProof
        if self.shard is None:
            self.shard = ml.ShardedBatchedFriProver.single_process([torch.cuda.current_device()], self.B, self.D - 1)
        return self.shard.prove_dev(self.ptrs, t), t

    def check(self):
        self.enqueue()
        self.stream.synchronize()
        p, t = self.blocking()
        blob = p.fri_proof.serialize() if self.kind == "pcs" else p.serialize()
        assert int(self.status.cpu()[0]) == 0
        assert bytes(self.proof.cpu().numpy()) == blob, "async proof differs from the blocking one"
        assert bytes(self.tr[:104].cpu().numpy()) == t.export(), "async transcript differs from the blocking one"

    def free(self):
        self.plan.free()
        if self.shard is not None:
            self.shard.free()


def med(xs):
    return round(statistics.median(xs), 4)


def serial_latency(sh, reps):
    sh.check()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {"async_ms": [], "async_host_ms": [], "blocking_ms": [], "blocking_host_ms": []}
    for _ in range(reps):
        sh.stream.synchronize()
        t0 = time.perf_counter()
        ev0.record(sh.stream)
        sh.enqueue()
        ev1.record(sh.stream)
        sh.stream.synchronize()
        res["async_host_ms"].append(1e3 * (time.perf_counter() - t0))
        res["async_ms"].append(ev0.elapsed_time(ev1))
        t0 = time.perf_counter()
        ev0.record(sh.stream)
        sh.blocking()
        ev1.record(sh.stream)
        sh.stream.synchronize()
        res["blocking_host_ms"].append(1e3 * (time.perf_counter() - t0))
        res["blocking_ms"].append(ev0.elapsed_time(ev1))
    out = {k: med(v) for k, v in res.items()}
    out["reps"] = reps
    return out


def in_flight(base, K, reps):
    shapes = [base] + [Shape(base.kind, base.B, base.D, torch.cuda.Stream(), base.inputs) for _ in range(K - 1)]
    for s in shapes:
        s.enqueue()
    torch.cuda.synchronize()
    per = []
    for _ in range(reps):
        t0 = time.perf_counter()
        for s in shapes:
            s.enqueue()
        torch.cuda.synchronize()
        per.append(1e3 * (time.perf_counter() - t0) / K)
    for s in shapes[1:]:
        s.free()
    return {"K": K, "ms_per_proof": med(per), "reps": reps}


def graph_enqueue(sh, reps):
    sh.enqueue()
    sh.stream.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=sh.stream, capture_error_mode="global"):
        sh.enqueue()
    torch.cuda.synchronize()
    eager, replay = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        sh.enqueue()
        eager.append(1e3 * (time.perf_counter() - t0))
        sh.stream.synchronize()
        t0 = time.perf_counter()
        with torch.cuda.stream(sh.stream):
            g.replay()
        replay.append(1e3 * (time.perf_counter() - t0))
        sh.stream.synchronize()
    assert int(sh.status.cpu()[0]) == 0
    del g
    return {"eager_enqueue_host_ms": med(eager), "graph_replay_host_ms": med(replay), "reps": reps}


def kernel_times(sh):
    from torch.profiler import ProfilerActivity, profile
    sh.enqueue()
    sh.stream.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            sh.enqueue()
        sh.stream.synchronize()
    out = {}
    for e in prof.key_averages():
        for name in ("batch_root_kernel", "bfri_proof_write_kernel", "fri_query_indices_kernel", "ptr_table_kernel"):
            if name in e.key:
                out[name + "_us"] = round(e.device_time_total / max(e.count, 1), 2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=12)
    a = ap.parse_args()
    res = {"gpu": gpu_info(), "serial": {}, "in_flight": [], "graph": None, "kernels": None, "errors": []}
    pcs = Shape("pcs", 64, 23, torch.cuda.Stream())
    res["serial"]["pcs_64x2^22"] = serial_latency(pcs, a.reps)
    print("pcs", res["serial"]["pcs_64x2^22"], flush=True)
    for K in (1, 2, 4):
        try:
            res["in_flight"].append(in_flight(pcs, K, a.reps))
            print(res["in_flight"][-1], flush=True)
        except Exception as e:  # noqa: BLE001  (memory bounds K)
            res["errors"].append("in_flight K=%d: %s" % (K, e))
    res["graph"] = graph_enqueue(pcs, a.reps)
    print(res["graph"], flush=True)
    res["kernels"] = kernel_times(pcs)
    print(res["kernels"], flush=True)
    pcs.free()
    del pcs
    torch.cuda.empty_cache()
    for B, D in ((64, 23), (8, 25)):
        sh = Shape("codes", B, D, torch.cuda.Stream())
        key = "codes_%dx2^%d" % (B, D)
        res["serial"][key] = serial_latency(sh, a.reps)
        print(key, res["serial"][key], flush=True)
        sh.free()
        del sh
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
