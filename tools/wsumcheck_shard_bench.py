"""ml_wsumcheck_shard_* timing in one process (single-process handles over real GPUs).

    python tools/wsumcheck_shard_bench.py --out DIR [--shapes 20x4x2,24x1x1,26x8x2] [--reps 10] [--gpus 1,2,4,8]

A shape is n_vars x width x composition_degree over a synthetic trace (seed 0x5C, generated on every GPU used): 2^20 x 4 at
degree 2 is the reference's sumcheck_high_bench (the pythagorean composition), 2^24 x 1 with x[0] at degree 1 is BASELINE
config 4, 2^26 x 8 at degree 2 a wide trace.  For every G in --gpus that the box has, a G-rank handle on devices 0 .. G-1
alternates call by call with the single-GPU path on device 0 (ml_wsumcheck_build_dev + set_composition +
ml_wsumcheck_compute_polynomials; the sharded calls include their set_composition too).  Every call is bracketed by CUDA
events on every rank's stream (plus a device synchronise); a call's time is the maximum over its ranks.  One warm-up call per
variant; medians of --reps; the results of all variants are compared.  Writes DIR/wsumcheck_shard_timing.json; GPU name, power
limit and SM clock are read in the same run."""
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
from oracle.pyref import M

L_ = load()


def composition(width, degree):
    if width == 1 and degree == 1:
        return [(1, [0])]  # config 4: the PCS composition
    if width == 4 and degree == 2:
        c = 0x1234567  # sumcheck_high_bench: mask0 * (x0^2 + x1^2 - x2^2) + mask1 * (x0 + x1 - x3)
        m0, m1 = (1 - c) % M, c
        return [(m0, [0, 0]), (m0, [1, 1]), ((-m0) % M, [2, 2]), (m1, [0]), (m1, [1]), ((-m1) % M, [3])]
    return [(3, []), (5, [0] * degree), (7, [width - 1] * degree), (11, [width // 2])]


def single(row_point, buf, width, h, terms, degree, stream):
    rp = ml.as_elems(row_point)
    hd = C.c_void_p()
    ml.check(L_.ml_wsumcheck_build_dev(ml._p(rp), ml._sz(rp.shape[0]), buf.ptr, ml._sz(width), ml._sz(h), C.c_void_p(stream.cuda_stream), C.byref(hd)))
    g = ml.WideSumcheckTables(hd, width)
    g.set_composition(terms)
    t = ml.Transcript()
    res = g.compute_sumcheck_polynomials(degree, t, 42)
    del g
    return res, t.random()


def sharded(sh, row_point, ptrs, terms, degree):
    sh.set_composition(terms)
    t = ml.Transcript()
    return sh.compute_sumcheck_polynomials_dev(row_point, ptrs, degree, t, 42), t.random()


def shape_run(nv, width, degree, gs, reps):
    h = 1 << nv
    traces = {}
    for d in range(max(gs)):
        ml.set_device(d)
        traces[d] = ml.synthetic_elements_dev(0x5C, h * width)
        torch.cuda.synchronize(d)
    ml.set_device(0)
    row_point = ml.to_ints(ml.synthetic_elements_dev(0x5C0001, nv).elems())
    terms = composition(width, degree)
    s0 = torch.cuda.Stream(device=0)
    variants = {"single_gpu": ([(0, s0)], lambda: single(row_point, traces[0], width, h, terms, degree, s0))}
    handles = []
    for G in gs:
        sh = ml.ShardedWideSumcheck.single_process(list(range(G)), width, nv)
        handles.append(sh)
        st = [(d, torch.cuda.ExternalStream(sh.stream(d), device=d)) for d in range(G)]
        ptrs = [traces[g].ptr.value + g * (h // G) * width * 16 for g in range(G)]
        variants["wsumcheck_shard_G%d" % G] = (st, lambda sh=sh, ptrs=ptrs: sharded(sh, row_point, ptrs, terms, degree))
    results, times = {}, {k: [] for k in variants}
    for k, (st, fn) in variants.items():  # warm-up, and the results to compare
        results[k] = fn()
        for d, _ in st:
            torch.cuda.synchronize(d)
    for _ in range(reps):
        for k, (st, fn) in variants.items():
            times[k].append(timed(st, fn)[1])
    ref = results["single_gpu"]
    row = {"n_vars": nv, "width": width, "composition_degree": degree, "median_ms": {k: statistics.median(v) for k, v in times.items()},
           "all_ms": times, "same_result_as_single_gpu": {k: results[k] == ref for k in variants}}
    if "wsumcheck_shard_G1" in row["median_ms"]:
        row["G1_over_single_gpu"] = row["median_ms"]["wsumcheck_shard_G1"] / row["median_ms"]["single_gpu"]
    for sh in handles:
        sh.free()
    del traces
    for d in range(max(gs)):
        torch.cuda.synchronize(d)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default="20x4x2,24x1x1,26x8x2")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--gpus", default="1,2,4,8")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("wsumcheck_shard_bench: no GPU")
    gs = [int(x) for x in args.gpus.split(",") if int(x) <= torch.cuda.device_count()]
    res = {"workload": "wsumcheck_shard_timing", "reps": args.reps, "gpus": gpu_info(), "device_count": torch.cuda.device_count(),
           "ranks_measured": gs, "results": []}
    for shp in args.shapes.split(","):
        nv, width, degree = (int(x) for x in shp.split("x"))
        row = shape_run(nv, width, degree, gs, args.reps)
        print(json.dumps({k: row[k] for k in row if k != "all_ms"}), flush=True)
        res["results"].append(row)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "wsumcheck_shard_timing.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
