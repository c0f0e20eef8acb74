"""ml_wsumcheck_shard_*: the width-w System sumcheck sharded over G ranks by row block (csrc/wsumcheck_shard.cu).  Every
coefficient, every challenge and the final transcript must equal the single-GPU handle's and the oracle's, whatever the number
of ranks."""
import ctypes as C
import random

import numpy as np
import pytest

from oracle import pyref as P
from oracle.binding import fe_arr

M = P.M


def _null_handle(ml, width=1, n_vars=4):
    return ml.ShardedWideSumcheck(C.c_void_p(None), 1, [0], width, n_vars)


# ------------------------------------------------------------------ argument checks (no GPU needed: they come before any device)
def test_create_rejects_bad_arguments(ml):
    for world in (3, 32):
        with pytest.raises(ml.MlError) as e:
            ml.ShardedWideSumcheck.single_process([0] * world, 4, 12)
        assert e.value.code == 8, world  # ML_ERR_ARG
    for world, log_g in ((2, 1), (4, 2), (8, 3), (16, 4)):
        with pytest.raises(ml.MlError) as e:
            ml.ShardedWideSumcheck.single_process([0] * world, 4, log_g - 1)
        assert e.value.code == 2, world  # ML_ERR_SIZE
    with pytest.raises(ml.MlError) as e:
        ml.ShardedWideSumcheck.single_process([0], 4, 0)
    assert e.value.code == 2
    for width in (0, 17):
        with pytest.raises(ml.MlError) as e:
            ml.ShardedWideSumcheck.single_process([0, 0], width, 8)
        assert e.value.code == 8, width


def test_composition_degree_above_3_rejected_before_any_device(ml):
    sh = _null_handle(ml)
    with pytest.raises(ml.MlError) as e:
        sh.compute_sumcheck_polynomials_dev([1, 2, 3, 4], [0], 4, ml.Transcript(), 0)
    assert e.value.code == 8 and "composition_degree" in str(e.value)
    sh.h = None


def test_create_without_gpu_fails_loudly(ml):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(ml.MlError) as e:
        ml.ShardedWideSumcheck.single_process([0, 0], 4, 6)
    assert e.value.code in (6, 7)  # no device: no CPU fallback


# ------------------------------------------------------------------ helpers
def terms_for(width, degree, rng):
    """a composition of total degree `degree` with a constant term and repeated columns"""
    terms = [(rng.randrange(M), [])]
    if degree >= 1:
        terms += [(rng.randrange(M), [rng.randrange(width) for _ in range(degree)]), (rng.randrange(M), [width - 1] * degree),
                  ((M - rng.randrange(1, 100)) % M, [0])]
    return terms


def single_dev(ml, row_point, buf, width, h):
    """ml_wsumcheck_build_dev over a whole trace already in HBM"""
    rp = ml.as_elems(row_point)
    hd = C.c_void_p()
    ml.check(ml.load().ml_wsumcheck_build_dev(ml._p(rp), ml._sz(rp.shape[0]), buf.ptr, ml._sz(width), ml._sz(h), None, C.byref(hd)))
    return ml.WideSumcheckTables(hd, width)


def blocks_of(buf, world, h, width):
    return [buf.ptr.value + g * (h // world) * width * 16 for g in range(world)]


# ------------------------------------------------------------------ virtual ranks on one GPU
CASES = [(1, 1, 1, 0), (1, 12, 4, 2), (1, 13, 5, 3), (1, 17, 16, 1), (1, 20, 1, 0),
         (2, 1, 4, 1), (2, 12, 16, 3), (2, 13, 1, 2), (2, 17, 5, 0),
         (4, 2, 5, 2), (4, 12, 1, 1), (4, 13, 16, 0), (4, 20, 4, 3),
         (8, 3, 16, 3), (8, 12, 5, 0), (8, 13, 4, 1), (8, 17, 1, 2),
         (16, 4, 1, 1), (16, 12, 4, 3), (16, 13, 16, 2), (16, 20, 5, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("world,nv,width,degree", CASES)
def test_virtual_ranks_vs_oracle_and_single_gpu(ml, oracle, world, nv, width, degree):
    rng = random.Random(world * 1000 + nv * 10 + width)
    h = 1 << nv
    matrix = oracle.synthetic(7000 + world + 3 * nv + 11 * width, h * width)
    row_point = fe_arr([rng.randrange(M) for _ in range(nv)])
    terms, s = terms_for(width, degree, rng), rng.randrange(M)
    sh = ml.ShardedWideSumcheck.single_process([0] * world, width, nv)
    sh.set_composition(terms)
    t, ot, gt = ml.Transcript(), oracle.transcript(), ml.Transcript()
    got = sh.compute_sumcheck_polynomials(row_point, matrix, degree, t, s)
    o = oracle.wsumcheck_build(row_point, matrix, width)
    o.set_composition(terms)
    want = o.compute_sumcheck_polynomials(degree, ot, s)
    g = ml.WideSumcheckTables.build(row_point, matrix, width)
    g.set_composition(terms)
    single = g.compute_sumcheck_polynomials(degree, gt, s)
    assert got == want == single
    assert len(got[0]) == nv * (degree + 1) and len(got[1]) == nv
    assert t.random() == ot.random() == gt.random()
    # the same handle again, then with other terms
    t2 = ml.Transcript()
    assert sh.compute_sumcheck_polynomials(row_point, matrix, degree, t2, s) == got and t2.random() == t.random()
    terms2 = terms_for(width, degree, random.Random(rng.randrange(1 << 30)))
    sh.set_composition(terms2)
    g2 = ml.WideSumcheckTables.build(row_point, matrix, width)
    g2.set_composition(terms2)
    t3, gt3 = ml.Transcript(), ml.Transcript()
    assert sh.compute_sumcheck_polynomials(row_point, matrix, degree, t3, s) == g2.compute_sumcheck_polynomials(degree, gt3, s)
    assert t3.random() == gt3.random()
    sh.free()


@pytest.mark.gpu
@pytest.mark.parametrize("log_height", [13, 20])
def test_reference_sumcheck_test_world8(ml, oracle, log_height):
    """the reference's sumcheck_test / sumcheck_high_bench (sumcheck.rs:342-398): pythagorean trace of width 4, degree 2, sum 0"""
    from test_oracle import pythagorean_system, verify_sumcheck_debug
    matrix, row_point, terms, ot = pythagorean_system(oracle, log_height)
    t = ml.Transcript()
    assert t.next_challenge() == oracle.transcript().next_challenge()  # the same transcript state as pythagorean_system leaves
    sh = ml.ShardedWideSumcheck.single_process([0] * 8, 4, log_height)
    sh.set_composition(terms)
    pols, rs = sh.compute_sumcheck_polynomials(row_point, matrix, 2, t, 0)
    o = oracle.wsumcheck_build(row_point, matrix, 4)
    o.set_composition(terms)
    assert (pols, rs) == o.compute_sumcheck_polynomials(2, ot, 0)
    assert t.random() == ot.random()
    assert verify_sumcheck_debug(oracle, oracle.transcript(), pols, 3, 0, matrix, 4, row_point, terms) == rs
    sh.free()


@pytest.mark.gpu
def test_config4_at_size_equals_pcs_tables(ml):
    """BASELINE config 4: 2^24 x 1 with the composition x[0] (degree 1) is the PCS sumcheck of SumcheckTables"""
    nv, h = 24, 1 << 24
    buf = ml.synthetic_elements_dev(0xC4, h)
    evals = buf.elems()
    row_point = ml.to_ints(ml.synthetic_elements_dev(0xC40001, nv).elems())
    s = 12345
    sh = ml.ShardedWideSumcheck.single_process([0] * 8, 1, nv)
    sh.set_composition([(1, [0])])
    t = ml.Transcript()
    got = sh.compute_sumcheck_polynomials_dev(row_point, blocks_of(buf, 8, h, 1), 1, t, s)
    pcs = ml.SumcheckTables.build_tables_for_pcs(row_point, evals)
    t1 = ml.Transcript()
    assert got == pcs.compute_sumcheck_polynomials(1, t1, s)
    assert t.random() == t1.random()
    sh.free()


@pytest.mark.gpu
def test_width16_n22_world8_equals_single_gpu(ml):
    nv, w, h = 22, 16, 1 << 22
    buf = ml.synthetic_elements_dev(0x16, h * w)
    row_point = ml.to_ints(ml.synthetic_elements_dev(0x160001, nv).elems())
    rng = random.Random(16)
    terms, s = terms_for(w, 3, rng), rng.randrange(M)
    sh = ml.ShardedWideSumcheck.single_process([0] * 8, w, nv)
    sh.set_composition(terms)
    t = ml.Transcript()
    got = sh.compute_sumcheck_polynomials_dev(row_point, blocks_of(buf, 8, h, w), 3, t, s)
    g = single_dev(ml, row_point, buf, w, h)
    g.set_composition(terms)
    t1 = ml.Transcript()
    assert got == g.compute_sumcheck_polynomials(3, t1, s) and t.random() == t1.random()
    sh.free()


@pytest.mark.gpu
def test_snark_test_sharded_sumcheck_then_sharded_pcs(ml, oracle):
    """snark_test (multilinear_pcs.rs:279-316) with both provers sharded over 4 ranks on the same row blocks: the proof and the
    final transcript equal the unsharded sequence (test_snark_test_system_sumcheck_then_pcs), and the verifier accepts them"""
    from test_oracle import PYTHAGOREAN
    log_h, world = 16, 4
    rows = list(PYTHAGOREAN)
    while len(rows) < 1 << log_h:
        rows = rows + rows
    evals = fe_arr(rows)
    buf = ml.DeviceBuffer.from_host(evals)
    blocks = blocks_of(buf, world, 1 << log_h, 1)
    terms = [(0, [])]
    # unsharded
    t1 = ml.Transcript()
    c = t1.next_challenge()
    row_point = fe_arr([c] * log_h)
    g = ml.WideSumcheckTables.build(row_point, evals, 1)
    g.set_composition(terms)
    gp, grs = g.compute_sumcheck_polynomials(1, t1, 0)
    inputs = fe_arr(grs)
    out = ml.MultilinearPolynomialEvals(evals).evaluate(grs)
    want = ml.PCSProof.prove(inputs, out, evals, t1)
    # sharded
    t = ml.Transcript()
    assert t.next_challenge() == c
    sw = ml.ShardedWideSumcheck.single_process([0] * world, 1, log_h)
    sw.set_composition(terms)
    sp, srs = sw.compute_sumcheck_polynomials_dev(row_point, blocks, 1, t, 0)
    assert (sp, srs) == (gp, grs) and not any(sp)
    sp_pcs = ml.ShardedPCSProver.single_process([0] * world, log_h)
    proof = sp_pcs.prove_dev(fe_arr(srs), out, blocks, t)
    assert proof.fri_proof.serialize() == want.fri_proof.serialize() and t.random() == t1.random()
    ot = oracle.transcript()
    ot.next_challenge()
    o = oracle.wsumcheck_build(row_point, evals, 1)
    o.set_composition(terms)
    assert o.compute_sumcheck_polynomials(1, ot, 0) == (sp, srs)
    oproof, st = oracle.pcs_prove(inputs, out, evals, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob and t.random() == ot.random()
    vt = ml.Transcript()
    assert vt.next_challenge() == c
    for k in range(log_h):
        for cf in sp[2 * k:2 * k + 2]:
            vt.absorb(int(cf).to_bytes(16, "little"))
        assert vt.next_challenge() == srs[k]
    assert proof.verify(vt) == 0
    sw.free()
    sp_pcs.free()


@pytest.mark.gpu
def test_arena_bytes_bound(ml):
    w, nv, world = 16, 24, 8
    sh = ml.ShardedWideSumcheck.single_process([0] * world, w, nv)
    tail = 4096 * (w + 1) * 16
    assert sh.arena_bytes() <= (w + 1) * 16 * (1 << nv) // world + tail + (1 << 20)
    sh.free()


@pytest.mark.gpu
def test_misuse(ml):
    nv, w = 14, 4
    matrix = fe_arr([(i * 7 + 1) % M for i in range((1 << nv) * w)])
    row_point = fe_arr(list(range(1, nv + 1)))
    one = ml.ShardedWideSumcheck.one_rank(0, 2, 0, w, nv)
    with pytest.raises(ml.MlError) as e:  # not connected
        one.compute_sumcheck_polynomials_dev(row_point, [0], 1, ml.Transcript(), 0)
    assert e.value.code == 8 and "connect" in str(e.value)
    with pytest.raises(ml.MlError) as e:  # host rows need a handle that hosts every rank
        one.compute_sumcheck_polynomials(row_point, matrix, 1, ml.Transcript(), 0)
    assert e.value.code == 8 and "every rank" in str(e.value)
    one.free()
    sh = ml.ShardedWideSumcheck.single_process([0, 0], w, nv)
    with pytest.raises(ml.MlError) as e:  # n_vars differs from the handle's
        sh.compute_sumcheck_polynomials(row_point[:nv - 1], matrix[:(w << (nv - 1))], 1, ml.Transcript(), 0)
    assert e.value.code == 2
    with pytest.raises(ml.MlError) as e:  # composition column out of range
        sh.set_composition([(1, [w])])
    assert e.value.code == 3
    sh.free()


# ------------------------------------------------------------------ real GPUs
def _gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
def test_single_process_two_devices(ml, oracle):
    if _gpus() < 2:
        pytest.skip("needs two GPUs")
    nv, w, deg = 15, 5, 3
    rng = random.Random(2)
    matrix = oracle.synthetic(77, (1 << nv) * w)
    row_point = fe_arr([rng.randrange(M) for _ in range(nv)])
    terms = terms_for(w, deg, rng)
    sh = ml.ShardedWideSumcheck.single_process([0, 1], w, nv)
    sh.set_composition(terms)
    t, gt = ml.Transcript(), ml.Transcript()
    got = sh.compute_sumcheck_polynomials(row_point, matrix, deg, t, 5)
    g = ml.WideSumcheckTables.build(row_point, matrix, w)
    g.set_composition(terms)
    assert got == g.compute_sumcheck_polynomials(deg, gt, 5) and t.random() == gt.random()
    sh.free()


@pytest.mark.gpu
def test_two_processes_two_gpus(ml):
    """one process per GPU (CUDA IPC arenas, peer stores, device flags): rank 0's result equals the single-GPU handle's and both
    processes get the same result"""
    import json
    import os
    import socket
    import subprocess
    import sys
    if _gpus() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tools", "wsumcheck_shard_demo.py"), "16", "4", "2"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    line = [json.loads(l) for l in p.stdout.splitlines() if l.startswith("{") and "wsumcheck_shard" in l][-1]
    assert line["n_gpus"] == 2 and line["matches_single_gpu"] is True and line["results_agree"] is True
