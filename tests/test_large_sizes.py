"""The NTT, Möbius and PCS-encode kernels against the CPU oracle at the sizes where their pass plans change (2^26 to 2^29).

ntt_launch (csrc/ntt.cu) splits a transform of 2^log_n elements into (log_n + 8) / 9 passes: three for log_n 18-27, four from 28
up, with the radices (7, 7, 7, 7) at 28 and (8, 7, 7, 7) at 29.  An inter-pass twiddle matrix larger than 1 GiB is not built:
from pass 0 of log_n 27 on, the store multiplies by the two-level root tables instead (the inverse pass 0 by the 1/N-scaled
table).  mobius_launch (csrc/mle.cu) runs a 12-bit pass, then 1, 2 or 3 column passes (n 13-20, 21-28, 29 and up).  The
provers at n_vars >= 27, and every rank of a sharded prover at n_vars 30/31, encode into a domain of 2^28 or more, so these
are the paths the largest proofs run.

Every comparison is element for element or byte for byte.  The oracle needs tens of seconds to a few minutes per call at
these sizes on the host's cores, and the 2^29 cases hold several 8 GiB arrays in host memory at once.
"""
import ctypes as C
import gc
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GiB = 1 << 30


@pytest.fixture(scope="module")
def big_oracle():
    from oracle import binding
    binding.build()
    return binding.Oracle(threads=os.cpu_count() or 1)


@pytest.fixture
def need_gpu_bytes():
    """need_gpu_bytes(n): skip unless n bytes of device memory are free now.  The GPU may be shared; a large case must not
    fail with ML_ERR_ALLOC because of another process's allocations."""
    import torch

    def need(n):
        free, _ = torch.cuda.mem_get_info()
        if free < n:
            pytest.skip("needs %.1f GiB of free device memory (%d bytes); %.1f GiB are free" % (n / GiB, n, free / GiB))
    return need


@pytest.fixture(autouse=True)
def release_pools(ml):
    """every case starts with the library's device pools empty, also after a failed case"""
    yield
    gc.collect()
    ml.check(ml.load().ml_release_pools())


def assert_elems_equal(got, want, what):
    """(n, 16) arrays equal element for element.  On a mismatch, report the first differing index and how many differ: a
    pass-index bug moves whole runs of elements, a twiddle bug spoils most of them.  Compared in chunks so that no
    full-size boolean temporary is made."""
    assert got.shape == want.shape, "%s: shape %s, want %s" % (what, got.shape, want.shape)
    g, w = got.reshape(-1, 16).view(np.uint64), want.reshape(-1, 16).view(np.uint64)
    n, chunk = g.shape[0], 1 << 22
    first, count = None, 0
    for s in range(0, n, chunk):
        a, b = g[s:s + chunk], w[s:s + chunk]
        if np.array_equal(a, b):
            continue
        bad = np.flatnonzero((a != b).any(axis=1))
        count += bad.size
        if first is None:
            first = s + int(bad[0])
    assert count == 0, "%s: %d of %d elements differ, the first at index %d" % (what, count, n, first)


def gen_bytes(g):
    return (C.c_uint8 * 16)(*g.to_bytes(16, "little"))


# ------------------------------------------------------------------ NTT: three- and four-pass plans
@pytest.mark.parametrize("log_n", [26, 27, 28])
def test_ntt_intt_vs_oracle(ml, big_oracle, need_gpu_bytes, log_n):
    """26: (9, 9, 8) with twiddle tables.  27: (9, 9, 9), pass 0 without a table, forward and inverse.  28: (7, 7, 7, 7), the
    first four-pass plan, pass 0 without a table and two middle digits in the last pass's output index."""
    O, L = big_oracle, ml.load()
    n = 1 << log_n
    need_gpu_bytes(4 * 16 * n)  # input, output, one scratch array, slack for the root tables and pools
    seed = 0x2600 + log_n
    g = ml.pow_2_generator(log_n)
    x = O.synthetic(seed, n)
    dx = ml.synthetic_elements_dev(seed, n)
    dy = ml.DeviceBuffer(16 * n)
    ml.check(L.ml_ntt_dev(dx.ptr, C.c_size_t(n), gen_bytes(g), dy.ptr, None))
    assert_elems_equal(dy.elems(), O.ntt(x, g), "ntt 2^%d" % log_n)
    # dy now holds O.ntt(x), and O.intt(O.ntt(x)) is x: x is the oracle's answer without a second oracle transform
    ml.check(L.ml_intt_dev(dy.ptr, C.c_size_t(n), gen_bytes(g), dx.ptr, None))
    assert_elems_equal(dx.elems(), x, "intt 2^%d" % log_n)
    dx.free()
    dy.free()


def test_reed_solomon_2p27_into_2p28_vs_oracle(ml, big_oracle, need_gpu_bytes):
    """2^27 coefficients into a domain of 2^28: the (7, 7, 7, 7) plan whose pass 0 reads only the live half"""
    O, L = big_oracle, ml.load()
    n = 1 << 27
    need_gpu_bytes(6 * 16 * n)
    g = ml.pow_2_generator(28)
    c = O.synthetic(0x2701, n)
    dc = ml.synthetic_elements_dev(0x2701, n)
    dcode = ml.DeviceBuffer(32 * n)
    ml.check(L.ml_reed_solomon_dev(dc.ptr, C.c_size_t(n), gen_bytes(g), dcode.ptr, None))
    dc.free()
    assert_elems_equal(dcode.elems(), O.reed_solomon(c, g), "reed_solomon 2^27 -> 2^28")
    dcode.free()


# ------------------------------------------------------------------ PCS encode as the provers run it
@pytest.mark.parametrize("log_n", [27, 28])
def test_pcs_encode_vs_oracle(ml, big_oracle, need_gpu_bytes, log_n):
    """ml_pcs_encode_dev = reed_solomon(bit_reverse(to_coefficient(evals))) (multilinear_pcs.rs:101-107): Möbius with two
    column passes, then the bit reversal fused into the load of NTT pass 0 under the (7, 7, 7, 7) plan (domain 2^28) and the
    (8, 7, 7, 7) plan (domain 2^29), the first four-pass plan with unequal radices"""
    O, L = big_oracle, ml.load()
    n = 1 << log_n
    need_gpu_bytes(7 * 16 * n)  # evals, code (2n), Möbius scratch, NTT scratch (2n), slack
    seed = 0xE0C0 + log_n
    devals = ml.synthetic_elements_dev(seed, n)
    dcode = ml.DeviceBuffer(32 * n)
    ml.check(L.ml_pcs_encode_dev(devals.ptr, C.c_size_t(n), dcode.ptr, None))
    devals.free()
    got = dcode.elems()
    dcode.free()
    coeffs = O.bit_reverse(O.to_coefficient(O.synthetic(seed, n)))
    want = O.reed_solomon(coeffs, O.pow2_generator(log_n + 1))
    del coeffs
    assert_elems_equal(got, want, "pcs encode 2^%d -> 2^%d" % (log_n, log_n + 1))


# ------------------------------------------------------------------ Möbius: two and three column passes
@pytest.mark.parametrize("log_n", [21, 24, 28, 29])
def test_mobius_vs_oracle(ml, big_oracle, need_gpu_bytes, log_n):
    """to_coefficient (subtracting) and to_evaluation (adding) of the same evaluations: 21, 24 and 28 run two column passes
    after the 12-bit pass, 29 runs three (the to_coefficient of every proof at n_vars >= 29)"""
    O, L = big_oracle, ml.load()
    n = 1 << log_n
    need_gpu_bytes(3 * 16 * n)
    seed = 0x30B1 + log_n
    x = O.synthetic(seed, n)
    dx = ml.synthetic_elements_dev(seed, n)
    dout = ml.DeviceBuffer(16 * n)
    ml.check(L.ml_mle_to_coefficient_dev(dx.ptr, C.c_size_t(n), dout.ptr, None))
    assert_elems_equal(dout.elems(), O.to_coefficient(x), "to_coefficient 2^%d" % log_n)
    ml.check(L.ml_mle_to_evaluation_dev(dx.ptr, C.c_size_t(n), dout.ptr, None))
    assert_elems_equal(dout.elems(), O.to_evaluation(x), "to_evaluation 2^%d" % log_n)
    dx.free()
    dout.free()


# ------------------------------------------------------------------ whole provers
def test_pcs_prove_n_vars_27_vs_oracle(ml, big_oracle, need_gpu_bytes):
    """PCSProof::prove at n_vars 27 on one GPU: a four-pass encode into 2^28, trees of 2^27 leaves and the fold chain from
    2^28.  Proof bytes, sumcheck coefficients, transcript state and verification equal the oracle's."""
    O = big_oracle
    nv = 27
    need_gpu_bytes(40 * GiB)
    ev = O.synthetic(0x27B200, 1 << nv)
    inp = O.synthetic(0x27B201, nv)
    out = O.mle_evals_evaluate(ev, inp)
    t, ot = ml.Transcript(), O.transcript()
    proof = ml.PCSProof.prove(inp, out, ev, t)
    blob, sumcheck, final = proof.fri_proof.serialize(), [c for nz in proof.sumcheck_polynomials for c in nz], t.random()
    assert proof.verify(ml.Transcript()) == 0
    del proof
    gc.collect()
    ml.check(ml.load().ml_release_pools())  # the oracle's proof needs host memory only, but the device is shared
    oproof, st = O.pcs_prove(inp, out, ev, ot)
    assert st == 0
    assert len(blob) == len(oproof.fri.blob) and blob == oproof.fri.blob
    assert sumcheck == oproof.sumcheck
    assert final == ot.random()
    assert oproof.verify(O.transcript()) == 0


def test_sharded_two_ranks_n_vars_28_equals_unsharded(ml, big_oracle, need_gpu_bytes):
    """ShardedPCSProver with two virtual ranks at n_vars 28 against PCSProof.prove_dev: each rank encodes its 2^27 block
    into a local code of 2^28 (four passes), and the combine runs at N = 2^29.  The provers run one after the other; only host
    bytes are kept between them."""
    nv, n = 28, 1 << 28
    need_gpu_bytes(80 * GiB)
    L = ml.load()
    evals = ml.synthetic_elements_dev(0x28B200, n)
    inp = big_oracle.synthetic(0x28B201, nv)
    outb = np.empty(16, dtype=np.uint8)
    ml.check(L.ml_mle_evals_evaluate_dev(evals.ptr, C.c_size_t(n), C.c_void_p(inp.ctypes.data), C.c_size_t(nv),
                                         C.c_void_p(outb.ctypes.data), None))
    out = int.from_bytes(outb.tobytes(), "little")
    t1 = ml.Transcript()
    single = ml.PCSProof.prove_dev(inp, out, evals, n, t1)
    want_blob, want_sc, want_t = single.fri_proof.serialize(), single.sumcheck_polynomials, t1.random()
    assert single.verify(ml.Transcript()) == 0
    del single
    gc.collect()
    ml.check(L.ml_release_pools())
    sh = ml.ShardedPCSProver.single_process([0, 0], nv)
    t = ml.Transcript()
    proof = sh.prove_dev(inp, out, [evals.ptr.value, evals.ptr.value + (n // 2) * 16], t)
    assert proof.fri_proof.serialize() == want_blob
    assert proof.sumcheck_polynomials == want_sc and t.random() == want_t
    del proof
    sh.free()
    evals.free()


# ------------------------------------------------------------------ the table-free twiddle path at every size
NO_WTAB_CHILD = r"""
import json, os, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from multilinear_b200 import api as ml
from oracle.binding import Oracle
O = Oracle(threads=os.cpu_count() or 1)
ran, bad = [], []
def cmp(what, got, want):
    ran.append(what)
    if not np.array_equal(got, want):
        d = np.flatnonzero((got != want).any(axis=1))
        bad.append({"case": what, "first": int(d[0]), "count": int(d.size)})
for log_n in range(13, 25):
    n = 1 << log_n
    g = ml.pow_2_generator(log_n)
    x = O.synthetic(0x7A00 + log_n, n)
    y = ml.ntt(x, g)
    cmp("ntt %d" % log_n, y, O.ntt(x, g))
    cmp("intt %d" % log_n, ml.intt(y, g), O.intt(y, g))
    c = x[:n // 2]
    cmp("reed_solomon %d" % log_n, ml.reed_solomon(c, g), O.reed_solomon(c, g))
for nv in (14, 20):
    ev, inp = O.synthetic(0x7B00 + nv, 1 << nv), O.synthetic(0x7C00 + nv, nv)
    out = O.mle_evals_evaluate(ev, inp)
    t, ot = ml.Transcript(), O.transcript()
    p = ml.PCSProof.prove(inp, out, ev, t)
    op, st = O.pcs_prove(inp, out, ev, ot)
    ran.append("pcs_prove %d" % nv)
    same = (st == 0 and p.fri_proof.serialize() == op.fri.blob and [c for nz in p.sumcheck_polynomials for c in nz] == op.sumcheck
            and t.random() == ot.random() and p.verify(ml.Transcript()) == 0)
    if not same:
        bad.append({"case": "pcs_prove %d" % nv})
print(json.dumps({"no_wtab": os.environ.get("MLB_NTT_NO_WTAB"), "ran": ran, "bad": bad}))
"""


def test_table_free_twiddles_all_sizes_vs_oracle(ml):
    """MLB_NTT_NO_WTAB sends every inter-pass twiddle through the two-level root tables, the path that sizes >= 2^27 take
    without it (and that any size takes when a table's allocation fails).  The switch is read once per process, so a child
    process runs ntt, intt and reed_solomon for domains 2^13-2^24 and PCSProof.prove at n_vars 14 and 20 against the
    oracle."""
    env = dict(os.environ, MLB_NTT_NO_WTAB="1")
    p = subprocess.run([sys.executable, "-c", NO_WTAB_CHILD, ROOT], capture_output=True, text=True, timeout=1200, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    res = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert res["no_wtab"] == "1"
    assert len(res["ran"]) == 3 * 12 + 2
    assert res["bad"] == []
