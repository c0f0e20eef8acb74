#!/usr/bin/env python
"""bench.py — PCS commit throughput on B200 (BASELINE.json metric), one process per GPU.

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): commit to a polynomial of
2^24 coefficients = reed_solomon (RS-encode NTT to 2^25, src/fri/mod.rs:19-28) + FriProverData::fold
(Merkle commit of every FRI layer, transcript challenges, all 24 folds; src/fri/mod.rs:136-145).
A "step" is one such commit on synthetic random field elements.

  value : Melem/s = n_gpus * 2^24 / t, inputs resident in HBM, CUDA events on the launch stream, max over ranks
  e2e   : the same metric through the host-pointer C ABI (ml_rs_fri_prove: pinned host coefficients -> H2D ->
          RS-encode + FriProof::prove incl. the 128 query openings -> proof back on the host)
  --impl reference : the CPU oracle (C restatement of the reference; the Rust crate cannot be built here)
          on all host threads, same metric, bounded sample.

N > 1: launched by torchrun; every rank commits its own polynomial (weak scaling, independent units, no
data-path collective); only timing is reduced over NCCL.
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# dram__bytes_read.sum + dram__bytes_write.sum of the group's largest launch, from the committed ncu --set full capture
# profiles/r1_ncu_top_kernels_v4.txt (second part):
#   merkle_leaf_subtree (2^24 leaves): 889.8 MB read + 952.1 MB written (algorithmic: 1543.5 MB)
#   ntt_rs_encode: sum of the three passes, 1881.4 MB read (incl. the 512 MB inter-pass twiddle matrix) + 1764.9 MB written —
#   the group is timed as one unit (algorithmic: 805.3 MB; the two intermediate round trips are the four-step schedule)
DRAM_TRAFFIC = {"merkle_leaf_subtree": 889808640 + 952099328, "ntt_rs_encode": 1881384448 + 1764900096}
METRIC = "pcs_commit_melem_per_s"
UNIT = "Melem/s"
PROF_NAMES = ["ntt_rs_encode", "merkle_leaf_subtree", "merkle_nodes", "merkle_top", "fri_fold", "sumcheck_sums", "sumcheck_fold",
              "mobius", "eq_table", "bit_reverse", "query_gather", "fused_tail", "transcript_step"]


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler(threading.Thread):
    """samples SM clock and throttle reasons of one GPU through NVML while the timed region runs"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8)),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4))}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def workload_config(args):
    """the `config` object of the JSON line: a function of the command line only, identical for both arms"""
    P = max(1, args.polys_per_gpu)
    return {"workload": "pcs_commit_rs_merkle_fri_fold", "log_n": args.log_n, "blowup": 2, "polys_per_gpu": P,
            "step": "one commit of each of the %d resident polynomials of 2^%d coefficients per GPU" % (P, args.log_n),
            "l2": "inputs larger than L2 (256 MiB coefficients, 512 MiB code per commit)",
            "parallelism": "independent commits: %d streams per GPU, no data-path collective" % P}


def cpu_commit_rate(oracle_mod, log_n, threads, steps, warmup, seed=0xB200, keep=None):
    """Melem/s of the CPU oracle for reed_solomon + FriProverData::fold at 2^log_n coefficients; keep (a dict) receives the
    roots, last element and final transcript state of the last commit (the parity check of the bench line)"""
    from oracle.binding import fe_ints
    O = oracle_mod.Oracle(threads=threads)
    n = 1 << log_n
    coeffs = O.synthetic(seed, n)
    gp = O.pow2_generator_powers(log_n + 1)  # the reference's callers pass gen_pows in (src/fri/mod.rs:136)
    gen = fe_ints(gp[1:2])[0]
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        code = O.reed_solomon(coeffs, gen)
        tr = O.transcript()
        f, st = O.fri_fold(gp, code, tr)
        dt = time.perf_counter() - t0
        assert st == 0 and f.last_element() is not None
        if keep is not None:
            keep.update(roots=f.roots(), last=f.last_element(), transcript=tr.random(), log_n=log_n, seed=seed)
        del f
        if it >= warmup:
            times.append(dt)
    mean = sum(times) / len(times)
    return n / mean / 1e6, mean


def pick_cpu_sample(oracle_mod, threads, total_steps, budget_s):
    """largest log_n in {20, 22, 24} whose (warmup+steps) run fits the time budget, from one timed 2^18 commit"""
    _, t18 = cpu_commit_rate(oracle_mod, 18, threads, 1, 0)
    for log_n in (24, 22, 20):
        est = t18 * (1 << (log_n - 18)) * (log_n + 1) / 19.0
        if est * total_steps <= budget_s:
            return log_n
    return 18


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port) on all host threads; rank 0 only"""
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    from oracle import binding
    binding.build()
    threads = os.cpu_count() or 1
    log_n = pick_cpu_sample(binding, threads, args.steps + args.warmup, 150.0)
    kept = {}
    rate, mean = cpu_commit_rate(binding, log_n, threads, args.steps, args.warmup, keep=kept)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(kept["roots"], kept["last"], kept["transcript"])])
    sample = "reed_solomon + FriProverData::fold of one 2^%d-coefficient polynomial per step (workload is 2^%d)" % (log_n, args.log_n)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u128", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "sample_log_n": log_n,
                         "note": "CPU oracle = C restatement of the reference, OpenMP over all host threads (the Rust crate cannot be "
                                 "built here: no cargo, no winter-math/sha2 sources); the reference itself is single-threaded"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def run_batched_commit(torch, ml, L, dist, world, rank, local_rank, n_polys, log_n, reps=3):
    """BASELINE configs[4]: BatchedPCSProof::prove of n_polys polynomials of 2^log_n evaluations, sharded by polynomial for the
    encode and by leaf range for hashing / fingerprints / first fold / openings (ml_shard_*, csrc/shard.cu).  One process per GPU;
    the arenas are connected through CUDA IPC records all-gathered once over torch.distributed; on the data path the only
    exchange is kernels storing into peer HBM over NVLink plus device-side flags (no NCCL, no host barrier).
    Strong scaling (the batch is fixed): `ms` = commit phase (batch root, the north-star's "batched commits"), `prove_ms` = the
    whole proof.  Reported beside the headline metric, not as it."""
    import hashlib
    import numpy as np
    if n_polys % world or (1 << log_n) % world:
        return None
    n = 1 << log_n
    dev = torch.device("cuda", local_rank)
    sh = ml.ShardedBatchedProver.one_rank(rank, world, local_rank, n_polys, log_n)
    if world > 1:
        sh.connect_over(dist, dev)
    mine = []
    for j in sh.local_polys():
        t = torch.empty(16 * n, dtype=torch.uint8, device=dev)
        ml.check(L.ml_synthetic_elements_dev(C.c_uint64(5000 + j), C.c_size_t(n), C.c_void_p(t.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        mine.append(t)
    ptrs = [t.data_ptr() for t in mine]
    inputs = ml.synthetic_elements_dev(0xC1A1, log_n).elems()
    outs = np.zeros((n_polys, 16), dtype=np.uint8)
    for j, t in zip(sh.local_polys(), mine):
        ob = (C.c_uint8 * 16)()
        ml.check(L.ml_mle_evals_evaluate_dev(C.c_void_p(t.data_ptr()), C.c_size_t(n), C.c_void_p(inputs.ctypes.data), C.c_size_t(log_n), ob, None))
        outs[j] = np.frombuffer(bytes(ob), dtype=np.uint8)
    if world > 1:
        g = torch.from_numpy(outs).to(dev).to(torch.int32)
        dist.all_reduce(g)  # rows are disjoint across ranks
        outs = g.to(torch.uint8).cpu().numpy()
    stream = torch.cuda.ExternalStream(sh.stream(0), device=dev)

    def sync():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def timed(fn):
        sync()  # ranks enter together: a peer that is late by more than MLB_SHARD_TIMEOUT_S would read as ML_ERR_PEER
        launches0 = ml.kernel_launches()
        out = fn()  # warm-up: tables, pools
        per_call = ml.kernel_launches() - launches0
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            out = fn()
        e1.record(stream)
        sync()
        ms = e0.elapsed_time(e1) / reps
        if dist is not None:
            tt = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt[0])
        return ms, out, per_call

    commit_ms, root, commit_launches = timed(lambda: sh.batch_commit_dev(ptrs))
    prove_ms, proof, prove_launches = timed(lambda: sh.prove_dev(inputs, outs, ptrs, ml.Transcript()))
    fixture_ok = None
    try:  # the oracle's root for exactly this workload (tests/golden/gen_batch_root.py)
        fx = json.load(open(os.path.join(ROOT, "tests", "golden", "batch_root_64x2p22.json")))
        if fx["n_polys"] == n_polys and fx["log_n"] == log_n:
            fixture_ok = bool(fx["root"] == root.hex())
    except Exception:  # noqa: BLE001
        pass
    res = {"workload": "batched_pcs_prove_%dx2^%d" % (n_polys, log_n), "api": "ml_shard_batch_commit_dev / ml_shard_batched_pcs_prove_dev",
           "exchange": "none" if world == 1 else "kernels store into peer HBM over NVLink (CUDA IPC arenas) + device flags; no NCCL on the data path",
           "launches_per_commit_per_rank": commit_launches, "launches_per_prove_per_rank": prove_launches,
           "root": root.hex(), "root_matches_oracle_fixture": fixture_ok, "unit": UNIT, "scaling": "strong", "n_gpus": world}
    if proof is not None:
        blob = proof.fri_proof.serialize()
        res["proof_sha256"] = hashlib.sha256(blob).hexdigest()
        res["proof_verifies"] = proof.verify(ml.Transcript()) == 0
    # the numbers last: the driver keeps the tail of the line
    res["prove_ms"] = prove_ms
    res["prove_value"] = n_polys * n / (prove_ms * 1e-3) / 1e6
    res["ms"] = commit_ms
    res["value"] = n_polys * n / (commit_ms * 1e-3) / 1e6
    del proof
    sync()
    sh.free()
    del mine
    torch.cuda.empty_cache()
    return res


def run_other_configs(torch, ml, L, threads):
    """BASELINE configs[0], [1], [3] beside the headline (configs[2]): three numbers each — device-resident rate (CUDA events),
    end-to-end rate through the host-pointer C ABI (wall clock, copies included), the CPU oracle on all host threads — and a
    bit-exact comparison of the CUDA result with the oracle's on the same inputs."""
    import numpy as np
    from oracle.binding import Oracle
    O = Oracle(threads=threads)
    out = {}

    def gpu_ms(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def wall_ms(fn, reps=3):
        fn()
        best = None
        for _ in range(reps):
            t0 = time.perf_counter()
            r = fn()
            dt = (time.perf_counter() - t0) * 1e3
            best = dt if best is None or dt < best else best
        return best, r

    def rate(n, ms):
        return n / (ms * 1e-3) / 1e6

    # ---- configs[1]: forward + inverse NTT, one polynomial of 2^20 coefficients, blowup 2
    n = 1 << 20
    hc = O.synthetic(0xB200, n)
    g21 = ml.pow_2_generator(21)
    gb = (C.c_uint8 * 16)(*g21.to_bytes(16, "little"))
    dc, dcode, dback = ml.DeviceBuffer.from_host(hc), ml.DeviceBuffer(32 * n), ml.DeviceBuffer(32 * n)

    def ntt_dev():
        ml.check(L.ml_reed_solomon_dev(dc.ptr, C.c_size_t(n), gb, dcode.ptr, None))
        ml.check(L.ml_intt_dev(dcode.ptr, C.c_size_t(2 * n), gb, dback.ptr, None))

    d_ms = gpu_ms(ntt_dev, reps=10)
    e_ms, (code, back) = wall_ms(lambda: (lambda c: (c, ml.intt(c, g21)))(ml.reed_solomon(hc, g21)))
    t0 = time.perf_counter()
    ocode = O.reed_solomon(hc, g21)
    oback = O.intt(ocode, g21)
    c_ms = (time.perf_counter() - t0) * 1e3
    out["ntt_2p20_blowup2_fwd_inv"] = {"value": rate(n, d_ms), "e2e": rate(n, e_ms), "cpu": rate(n, c_ms), "unit": UNIT, "device_ms": d_ms,
                                       "bit_exact": bool(np.array_equal(code, ocode) and np.array_equal(back, oback))}
    del dc, dcode, dback

    # ---- configs[3]: sumcheck over a 2^24-entry multilinear extension product, all rounds
    nv = 24
    n = 1 << nv
    ev = O.synthetic(0xB200, n)
    inp = O.synthetic(0xB2000001, nv)
    claim = O.mle_evals_evaluate(ev, inp)
    dev = ml.DeviceBuffer.from_host(ev)

    def sc_dev():
        h = C.c_void_p()
        ml.check(L.ml_sumcheck_build_tables_for_pcs_dev(C.c_void_p(inp.ctypes.data), C.c_size_t(nv), dev.ptr, C.c_size_t(n), None, C.byref(h)))
        return ml.SumcheckTables(h).compute_sumcheck_polynomials(1, ml.Transcript(), claim)

    d_ms = gpu_ms(sc_dev)
    e_ms, got = wall_ms(lambda: ml.SumcheckTables.build_tables_for_pcs(inp, ev).compute_sumcheck_polynomials(1, ml.Transcript(), claim), reps=2)
    t0 = time.perf_counter()
    want = O.sumcheck_build(inp, ev).compute_sumcheck_polynomials(1, O.transcript(), claim)
    c_ms = (time.perf_counter() - t0) * 1e3
    out["sumcheck_2p24_all_rounds"] = {"value": rate(n, d_ms), "e2e": rate(n, e_ms), "cpu": rate(n, c_ms), "unit": UNIT, "device_ms": d_ms,
                                       "bit_exact": bool(got == want)}
    del dev

    # ---- configs[0]: the reference's own end-to-end example (multilinear_pcs_bench_test: n_vars 20, evals 7i+3, inputs i)
    nv = 20
    n = 1 << nv
    ev1 = ml.from_i64([7 * i + 3 for i in range(n)])
    in1 = ml.from_i64(range(nv))
    out1 = ml.MultilinearPolynomialEvals(ev1).evaluate(ml.to_ints(in1))
    d1 = ml.DeviceBuffer.from_host(ev1)
    d_ms = gpu_ms(lambda: ml.PCSProof.prove_dev(in1, out1, d1, n, ml.Transcript(), None))
    e_ms, proof = wall_ms(lambda: ml.PCSProof.prove(in1, out1, ev1, ml.Transcript()))
    t0 = time.perf_counter()
    op, st = O.pcs_prove(in1, out1, ev1, O.transcript())
    c_ms = (time.perf_counter() - t0) * 1e3
    out["pcs_prove_reference_example_nvars20"] = {"value": rate(n, d_ms), "e2e": rate(n, e_ms), "cpu": rate(n, c_ms), "unit": UNIT, "device_ms": d_ms,
                                                  "bit_exact": bool(st == 0 and proof.fri_proof.serialize() == op.fri.blob)}
    out["cpu_threads"] = threads
    return out


def pin_to_gpu_numa_node(local_rank):
    """N > 1: run this rank's host threads (and so its pinned allocations, first touch) on the NUMA node its GPU hangs off; with all
    ranks on node 0 the eight ranks' 2 GiB-per-step host reads share one memory controller (round 1: e2e efficiency 0.74 at N = 8)"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:  # NVML prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return {"node": node, "pinned": False}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return {"node": node, "pinned": False}
        os.sched_setaffinity(0, allowed)
        return {"node": node, "pinned": True, "cpus": len(allowed)}
    except Exception as e:  # noqa: BLE001
        return {"pinned": False, "error": str(e)[:120]}


def dump_outputs(out_dir, results):
    """writes what the last timed step returned for each of the P polynomials (FriProverData's layer roots, last element, final
    transcript state) as <out_dir>/<name>.npy.  All three are byte strings: every byte is stored as one float32 value, so any
    changed bit stays a difference of at least 1 under a tolerance comparison."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"fri_layer_roots": [b"".join(roots) for roots, _, _ in results],  # (P, log_n, 32)
              "last_element": [last.to_bytes(16, "little") for _, last, _ in results],  # (P, 16), little-endian field element
              "transcript_state": [tr for _, _, tr in results]}  # (P, 32)
    for name, rows in arrays.items():
        a = np.array([np.frombuffer(r, dtype=np.uint8) for r in rows], dtype=np.float32)
        if name == "fri_layer_roots":
            a = a.reshape(len(rows), -1, 32)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch
    from multilinear_b200 import api as ml
    from multilinear_b200 import load
    L = load()
    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the CUDA path has no CPU fallback")
    numa = pin_to_gpu_numa_node(local_rank) if (world > 1 and not os.environ.get("MLB_NO_NUMA_PIN")) else None
    torch.cuda.set_device(local_rank)
    ml.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    n = 1 << args.log_n
    P = max(1, args.polys_per_gpu)
    # P independent polynomials per GPU, resident in HBM before the timed region; each is committed on its own
    # stream by its own host thread so the latency-bound phases of one commit (tree tops, fused tail, transcript
    # steps) overlap the throughput-bound kernels of the others
    coeffs = [ml.synthetic_elements_dev(0xB200 + rank * 64 + j, n) for j in range(P)]
    streams = []
    for _ in range(P):
        h = C.c_void_p()
        ml.check(L.ml_stream_create(C.byref(h)))
        streams.append(h)
    ml.synchronize()
    results = [None] * P

    def commit(j):
        t = ml.Transcript()
        f = ml.FriProverData.fold_from_coeffs_dev(coeffs[j], n, t, streams[j].value)
        out = (f.fold_roots(), f.last_element, t.random())
        del f  # the handle (all layers, ~3.5 GB at 2^24) returns to the stream-ordered pool
        return out

    def worker(j, steps):
        ml.set_device(local_rank)  # the CUDA current device is per host thread
        for _ in range(steps):
            results[j] = commit(j)

    def run_steps(steps, which=None):
        js = list(range(P)) if which is None else which
        if len(js) == 1:
            worker(js[0], steps)
            return
        ts = [threading.Thread(target=worker, args=(j, steps)) for j in js]
        for t in ts:
            t.start()
        for t in ts:
            t.join()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    L.ml_profile_enable(0)
    run_steps(args.warmup)
    sampler = ClockSampler(local_rank)
    barrier()
    launches0 = ml.kernel_launches()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()  # legacy default stream: ordered against the (blocking) worker streams
    run_steps(args.steps)
    e1.record()
    barrier()
    sampler.stop_flag = True
    ms = e0.elapsed_time(e1) / args.steps
    launches = ml.kernel_launches() - launches0
    roots, last, tr0 = results[0]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, results)  # before the serial pass below overwrites results[0]

    # ---- serial pass of the same workload (one commit at a time) with per-kernel CUDA-event timing: per-kernel
    # durations are only well defined when commits do not share the GPU
    ser_steps = max(2, min(args.steps, 5))
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    run_steps(ser_steps, which=[0])  # plain serial pass: the latency of one commit
    s1.record()
    barrier()
    ms_serial = s0.elapsed_time(s1) / ser_steps
    launches_serial = None
    l0 = ml.kernel_launches()
    L.ml_profile_reset()
    L.ml_profile_enable(1)
    barrier()
    run_steps(ser_steps, which=[0])  # the same pass with every kernel group bracketed by CUDA events (adds ≈0.5 ms per commit)
    barrier()
    launches_serial = (ml.kernel_launches() - l0) / ser_steps
    L.ml_profile_enable(0)
    kernels = {}
    for i, name in enumerate(PROF_NAMES):
        t, cnt, by = C.c_double(0), C.c_uint64(0), C.c_double(0)
        L.ml_profile_get(C.c_int(i), C.byref(t), C.byref(cnt), C.byref(by))
        if cnt.value:
            kernels[name] = {"ms_per_commit": t.value / ser_steps, "launches_per_commit": cnt.value / ser_steps,
                             "alg_bytes_per_commit": by.value / ser_steps,
                             "achieved_gbs": by.value / (t.value * 1e-3) / 1e9 if t.value > 0 else None}
            t2, c2, b2 = C.c_double(0), C.c_uint64(0), C.c_double(0)
            L.ml_profile_get_max(C.c_int(i), C.byref(t2), C.byref(c2), C.byref(b2))
            kernels[name]["largest_launch"] = {"ms": t2.value, "alg_bytes": b2.value, "samples": c2.value}
    L.ml_profile_reset()

    # ---- full PCSProof::prove (src/fri/multilinear_pcs.rs:90-136) at the same size, one at a time, with the per-kernel table:
    # the HBM-bound kernels of the path (Moebius transform, eq table, sumcheck fold + sums) are not part of a bare commit, so
    # their achieved bandwidth is measured here; reported beside the headline, not as it
    pcs_prove = None
    try:
        nv = args.log_n
        pts = ml.from_i64(range(5, 5 + nv))
        ob = (C.c_uint8 * 16)()
        ml.check(L.ml_mle_evals_evaluate_dev(coeffs[0].ptr, C.c_size_t(n), C.c_void_p(pts.ctypes.data), C.c_size_t(nv), ob, None))
        claim = int.from_bytes(bytes(ob), "little")
        pr = ml.PCSProof.prove_dev(pts, claim, coeffs[0], n, ml.Transcript(), streams[0].value)  # warm-up
        ok = pr.verify(ml.Transcript()) == 0
        del pr
        L.ml_profile_reset()
        L.ml_profile_enable(1)
        torch.cuda.synchronize()  # rank-local leg: no cross-rank barrier inside the try block
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        reps = 3
        for _ in range(reps):
            pr = ml.PCSProof.prove_dev(pts, claim, coeffs[0], n, ml.Transcript(), streams[0].value)
            del pr
        p1.record()
        torch.cuda.synchronize()  # rank-local leg: no cross-rank barrier inside the try block
        L.ml_profile_enable(0)
        pk = {}
        for i, name in enumerate(PROF_NAMES):
            t, cnt, by = C.c_double(0), C.c_uint64(0), C.c_double(0)
            L.ml_profile_get(C.c_int(i), C.byref(t), C.byref(cnt), C.byref(by))
            if cnt.value and name in ("mobius", "eq_table", "sumcheck_sums", "sumcheck_fold", "fri_fold"):
                gbs = by.value / (t.value * 1e-3) / 1e9 if t.value > 0 else None
                pk[name] = {"ms_per_prove": t.value / reps, "alg_bytes_per_prove": by.value / reps, "achieved_gbs": gbs}
        L.ml_profile_reset()
        pcs_prove = {"workload": "PCSProof::prove n_vars=%d (Moebius + RS-encode + Merkle + sumcheck rounds + FRI folds + 128 queries)" % nv,
                     "ms": p0.elapsed_time(p1) / reps, "verifies": bool(ok), "hbm_bound_kernels": pk}
    except Exception as e:  # noqa: BLE001
        pcs_prove = {"error": str(e)[:300]}

    # ---- e2e through the host-pointer C ABI (pinned host input, proof back on the host), same P-way pipelining
    e2e_steps = max(1, min(args.steps, 5))
    PE = args.e2e_polys if args.e2e_polys > 0 else (12 if world == 1 else 8)
    while len(streams) < PE:
        h = C.c_void_p()
        ml.check(L.ml_stream_create(C.byref(h)))
        streams.append(h)
    pinned = []
    for j in range(PE):
        hp = C.c_void_p()
        ml.check(L.ml_host_alloc_pinned(C.c_size_t(16 * n), C.byref(hp)))
        ml.check(L.ml_dev_download(hp, coeffs[j % P].ptr, C.c_size_t(16 * n)))
        pinned.append(hp)
    e2e_out = [None] * PE

    e2e_phase = [[0.0, 0.0] for _ in range(PE)]  # seconds inside the C-ABI prove call / reading the proof back out

    host_bufs = pinned  # switched to pageable arrays for the second end-to-end figure

    def e2e_worker(j, steps):
        ml.set_device(local_rank)
        ml.check(L.ml_set_thread_stream(streams[j], C.c_int(1)))
        for _ in range(steps):
            t = ml.Transcript()
            h = C.c_void_p()
            t0 = time.perf_counter()
            ml.check(L.ml_rs_fri_prove(host_bufs[j], C.c_size_t(n), t.h, C.byref(h)))
            t1 = time.perf_counter()
            proof = ml.FriProof(h)
            e2e_out[j] = (proof.commitments, proof.last_elem, len(proof.serialize()))
            del proof
            e2e_phase[j][0] += t1 - t0
            e2e_phase[j][1] += time.perf_counter() - t1

    def e2e_run(steps):
        ts = [threading.Thread(target=e2e_worker, args=(j, steps)) for j in range(PE)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()

    # raw pinned host -> device bandwidth of this box (explains the e2e figure: 256 MiB of coefficients per commit)
    h2d_gbs = None
    try:
        scratch = ml.DeviceBuffer(16 * n)
        hb0, hb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = None
        for _ in range(3):
            torch.cuda.synchronize()
            hb0.record()
            ml.check(L.ml_dev_upload(scratch.ptr, pinned[0], C.c_size_t(16 * n)))
            hb1.record()
            torch.cuda.synchronize()
            dt = hb0.elapsed_time(hb1)
            best = dt if best is None or dt < best else best
        h2d_gbs = 16 * n / (best * 1e-3) / 1e9
        del scratch
    except Exception:  # noqa: BLE001
        pass
    e2e_run(1)  # warm-up
    for ph in e2e_phase:
        ph[0] = ph[1] = 0.0
    barrier()
    t0 = time.perf_counter()
    e2e_run(e2e_steps)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    blob_len = e2e_out[0][2]
    e2e_ok = e2e_out[0][0] == roots and e2e_out[0][1] == last
    e2e_call_ms = 1e3 * sum(p[0] for p in e2e_phase) / (PE * e2e_steps)
    e2e_read_ms = 1e3 * sum(p[1] for p in e2e_phase) / (PE * e2e_steps)

    # ---- the same end-to-end leg from PAGEABLE host memory (what a drop-in caller's Vec<Field128> is): plain numpy arrays, never
    # page-locked; the library stages them through its pinned ring (csrc/prover.cu staged_upload)
    e2e_pageable = None
    try:
        import numpy as np
        arrays = []
        for j in range(PE):
            a = np.empty(16 * n, dtype=np.uint8)
            C.memmove(a.ctypes.data, pinned[j], 16 * n)
            arrays.append(a)
        host_bufs = [C.c_void_p(a.ctypes.data) for a in arrays]
        e2e_run(1)
        barrier()
        pg_steps = max(1, min(e2e_steps, 3))
        t0 = time.perf_counter()
        e2e_run(pg_steps)
        torch.cuda.synchronize()
        pg_s = (time.perf_counter() - t0) / pg_steps
        pg_ok = e2e_out[0][0] == roots and e2e_out[0][1] == last
        e2e_pageable = {"seconds_per_step": pg_s, "steps": pg_steps, "ok": bool(pg_ok)}
        host_bufs = pinned
        del arrays
    except Exception as e:  # noqa: BLE001
        e2e_pageable = {"error": str(e)[:200]}
    for hp in pinned:
        L.ml_host_free_pinned(hp)

    batched = None
    if not args.no_batched:
        # secondary leg: never let it take the headline line down (e.g. a box without peer access between two GPUs);
        # every rank takes the same branch because the failure modes are collective (IPC mapping, NCCL)
        try:
            batched = run_batched_commit(torch, ml, L, dist, world, rank, local_rank, args.batched_polys, args.batched_log_n)
        except Exception as e:  # noqa: BLE001
            batched = {"workload": "batched_pcs_prove_%dx2^%d" % (args.batched_polys, args.batched_log_n), "error": str(e)[:300]}

    # max over ranks
    if dist is not None:
        pg = e2e_pageable.get("seconds_per_step", 0.0) if e2e_pageable else 0.0
        tt = torch.tensor([ms, e2e_s, pg], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, e2e_s = float(tt[0]), float(tt[1])
        if e2e_pageable and "seconds_per_step" in e2e_pageable:
            e2e_pageable["seconds_per_step"] = float(tt[2])
        ll = torch.tensor([launches], device="cuda", dtype=torch.int64)
        dist.all_reduce(ll)
        launches = int(ll[0])

    if rank == 0:
        value = world * P * n / (ms * 1e-3) / 1e6
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
        dom = max(kernels.items(), key=lambda kv: kv[1]["ms_per_commit"]) if kernels else (None, None)
        roofline = None
        if dom[0]:
            k = dom[1]
            # the launch on the first FRI layer (2^24 leaves) carries half of the group's work: report that launch
            per_launch_bytes = k["largest_launch"]["alg_bytes"]
            per_launch_ms = k["largest_launch"]["ms"]
            ach = per_launch_bytes / (per_launch_ms * 1e-3) / 1e9
            roofline = {"bound": "hbm", "kernel": dom[0], "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                        "traffic": DRAM_TRAFFIC.get(dom[0]), "peak_source": peak_src, "share_of_step": k["ms_per_commit"] / ms_serial,
                        "launches_per_commit": k["launches_per_commit"], "launch_ms": per_launch_ms, "launch_alg_bytes": per_launch_bytes,
                        "group_achieved": k["achieved_gbs"],
                        "note": "SHA-256 hashing is integer-pipe (alu) bound, not HBM bound (int_pipe_frac = time at the measured "
                                "integer speed of light / actual); per-kernel times come from the serial pass of this run"}
        ntt = kernels.get("ntt_rs_encode")
        extra = {}
        if ntt:
            extra["ntt_roofline"] = {"bound": "hbm", "achieved": ntt["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s",
                                     "frac": ntt["achieved_gbs"] / hbm_peak, "alg_bytes": ntt["alg_bytes_per_commit"], "ms": ntt["ms_per_commit"]}
        # integer-pipe speed of light measured on this GPU (no HBM traffic)
        try:
            sol = {}
            for what, nn, it in (("sha_leaf", 148 * 2048, 32), ("sha_node", 148 * 2048, 32), ("butterfly", 148 * 2048, 128)):
                mms, work = ml.microbench(what, nn, it)
                sol[what + "_per_s"] = work / (mms * 1e-3)
            extra["int_pipe"] = sol
            if dom[0] == "merkle_leaf_subtree":
                leaves = 2.0 * n  # sum over the fold chain of leaves handled by the leaf/subtree kernel
                ideal_ms = (leaves / sol["sha_leaf_per_s"] + leaves * 0.875 / sol["sha_node_per_s"]) * 1e3
                roofline["int_pipe_frac"] = ideal_ms / dom[1]["ms_per_commit"]
        except Exception as e:  # noqa: BLE001
            extra["int_pipe_error"] = str(e)

        cpu_baseline = None
        other_configs = None
        parity_at_size, parity_detail = None, None
        if world == 1 and not args.no_cpu_baseline:
            from oracle import binding
            binding.build()
            threads = os.cpu_count() or 1
            log_s = pick_cpu_sample(binding, threads, 2, 25.0)
            kept = {}
            rate, mean = cpu_commit_rate(binding, log_s, threads, 1, 1, keep=kept)
            cpu_baseline = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                            "sample": "reed_solomon + FriProverData::fold at 2^%d coefficients, %.2f s per commit, all host threads (OpenMP)" % (log_s, mean)}
            # parity at size: the oracle's commit of the same polynomial (seed 0xB200 = this rank's polynomial 0) against the
            # CUDA path's: every layer root, the last element and the final transcript state
            if log_s == args.log_n:
                g_roots, g_last, g_tr = roots, last, tr0
            else:  # the CPU sample had to be smaller than the workload: commit that size on the GPU too
                tt = ml.Transcript()
                ff = ml.FriProverData.fold_from_coeffs_dev(ml.synthetic_elements_dev(0xB200, 1 << log_s), 1 << log_s, tt, streams[0].value)
                g_roots, g_last, g_tr = ff.fold_roots(), ff.last_element, tt.random()
                del ff
            try:
                other_configs = run_other_configs(torch, ml, L, threads)
            except Exception as e:  # noqa: BLE001
                other_configs = {"error": str(e)[:300]}
            parity_at_size = bool(g_roots == kept["roots"] and g_last == kept["last"] and g_tr == kept["transcript"])
            parity_detail = {"log_n": log_s, "seed": "0xB200", "roots_compared": len(kept["roots"]), "last_element": g_last == kept["last"],
                             "transcript": g_tr == kept["transcript"], "checker": "oracle/oracle.c (CPU restatement; unpinned against the Rust crate)"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u128", "data": "synthetic",
            "config": workload_config(args),
            "serial": {"ms_per_commit": ms_serial, "value": world * n / (ms_serial * 1e-3) / 1e6, "unit": UNIT, "launches_per_commit": launches_serial,
                       "note": "one commit at a time on one stream (latency-bound phases exposed); floor analysis in profiles/r2_serial_latency.txt"},
            "roofline": roofline, "cpu_baseline": cpu_baseline,
            "e2e": {"value": world * PE * n / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": 16 * n * PE, "d2h_bytes_per_step": blob_len * PE,
                    "polys_in_flight": PE, "numa": numa,
                    "ms_per_step": e2e_s * 1e3, "steps": e2e_steps, "includes": "128 query openings + proof serialisation", "matches_device_run": bool(e2e_ok),
                    "host_memory": "pinned (ml_host_alloc_pinned)", "pinned_h2d_gbs": h2d_gbs, "prove_call_ms_mean": e2e_call_ms,
                    "proof_readout_ms_mean": e2e_read_ms,
                    "pageable": None if not e2e_pageable or "seconds_per_step" not in e2e_pageable else {
                        "value": world * PE * n / e2e_pageable["seconds_per_step"] / 1e6, "unit": UNIT,
                        "ms_per_step": e2e_pageable["seconds_per_step"] * 1e3, "steps": e2e_pageable["steps"],
                        "matches_device_run": e2e_pageable["ok"],
                        "host_memory": "pageable (numpy arrays, as a caller's Vec<Field128>); staged by the library: 4 host threads, "
                                       "4 MiB pinned slots"}},
            "gpu_launches": launches, "clocks": sampler.result(), "kernels": kernels,
        }
        if other_configs is not None:
            line["e2e"]["other_configs"] = other_configs
        if parity_at_size is not None:
            if roofline is not None:  # driver-preserved key (config must stay identical to the reference arm's)
                roofline["parity_at_size"] = parity_at_size
            if line["cpu_baseline"] is not None:
                line["cpu_baseline"]["parity_at_size"] = parity_at_size
            line["parity"] = parity_detail
        if pcs_prove is not None:
            if "hbm_bound_kernels" in pcs_prove:
                for v in pcs_prove["hbm_bound_kernels"].values():
                    v["frac_of_hbm_peak"] = v["achieved_gbs"] / hbm_peak if v["achieved_gbs"] else None
            line["pcs_prove"] = pcs_prove
        line.update(extra)
        if batched is not None:  # last key: the driver keeps the tail of the line
            line["batched_commit"] = batched
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-n", type=int, default=24, dest="log_n")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--polys-per-gpu", type=int, default=6, dest="polys_per_gpu",
                    help="independent polynomials committed concurrently per GPU (one stream + host thread each)")
    ap.add_argument("--no-batched", action="store_true", help="skip the sharded batched-commit leg (BASELINE configs[4])")
    ap.add_argument("--batched-polys", type=int, default=64, dest="batched_polys")
    ap.add_argument("--batched-log-n", type=int, default=22, dest="batched_log_n")
    ap.add_argument("--e2e-polys", type=int, default=0, dest="e2e_polys",
                    help="concurrent commits in the end-to-end leg (more in flight hides the PCIe copies); default 12 on one GPU "
                         "(measured 1708 / 1727 / 1775 Melem/s at 6 / 8 / 12), 8 per rank under torchrun")
    ap.add_argument("--dump-outputs", default=None, dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's polynomials) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
