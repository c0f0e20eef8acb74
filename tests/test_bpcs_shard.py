"""ml_bpcs_shard_*: one BatchedPCSProof::prove with every polynomial split by block over G ranks (csrc/bpcs_shard.cu).  The proof
must be byte-identical to the unsharded prover's and the oracle's for any batch size and any number of ranks."""
import ctypes as C
import json
import os
import random
import struct

import numpy as np
import pytest

from oracle import pyref as P
from oracle.binding import fe_arr

M = P.M
HERE = os.path.dirname(os.path.abspath(__file__))


# ------------------------------------------------------------------ argument checks (no GPU needed: they come before any device)
def test_create_rejects_bad_world_batch_and_small_sizes(ml):
    for world in (3, 6, 32):
        with pytest.raises(ml.MlError) as e:
            ml.BlockShardedBatchedProver.single_process([0] * world, 10, 12)
        assert e.value.code == 8, world  # ML_ERR_ARG
    with pytest.raises(ml.MlError) as e:
        ml.BlockShardedBatchedProver.single_process([0, 0], 0, 12)
    assert e.value.code == 2  # ML_ERR_SIZE
    for world, log_g in ((2, 1), (4, 2), (8, 3), (16, 4)):
        with pytest.raises(ml.MlError) as e:
            ml.BlockShardedBatchedProver.single_process([0] * world, 3, 2 * log_g - 1)
        assert e.value.code == 2, world
    with pytest.raises(ml.MlError) as e:
        ml.BlockShardedBatchedProver.single_process([0], 1, 0)
    assert e.value.code == 2


def test_create_without_gpu_fails_loudly(ml):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(ml.MlError) as e:
        ml.BlockShardedBatchedProver.single_process([0, 0], 10, 6)
    assert e.value.code == 6  # ML_ERR_CUDA: no CPU fallback


# ------------------------------------------------------------------ virtual ranks on one GPU
def claim(oracle, world, B, nv):
    rng = random.Random(world * 10000 + B * 100 + nv)
    polys = [oracle.synthetic(7000 + 131 * world + 17 * B + nv + 1000 * j, 1 << nv) for j in range(B)]
    inp = fe_arr([rng.randrange(M) for _ in range(nv)])
    outs = fe_arr([oracle.mle_evals_evaluate(p, inp) for p in polys])
    return polys, inp, outs


def _grid():
    cases = []
    for L in range(5):
        lo = max(2, 2 * L)  # n_vars = 1 has no folded layer to open: the reference returns None there (test below)
        for B in (1, 2, 3, 5, 10, 17):
            for nv in sorted({lo, min(14, lo + 3 + B % 4), 14}):
                cases.append((1 << L, B, nv))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("world,B,nv", _grid())
def test_virtual_ranks_vs_oracle(ml, oracle, world, B, nv):
    polys, inp, outs = claim(oracle, world, B, nv)
    sh = ml.BlockShardedBatchedProver.single_process([0] * world, B, nv)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = sh.prove(inp, outs, polys, t)
    oproof, st = oracle.batched_pcs_prove(inp, outs, polys, ot)
    assert st == 0
    blob = proof.fri_proof.serialize()
    assert blob == oproof.fri.blob
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck
    assert t.random() == ot.random()
    assert proof.verify(ml.Transcript()) == 0
    t1 = ml.Transcript()
    single = ml.BatchedPCSProof.prove(inp, outs, polys, t1)
    assert single.fri_proof.serialize() == blob and t1.random() == ot.random()
    t2 = ml.Transcript()  # a second call on the same handle gives the same bytes
    again = sh.prove(inp, outs, polys, t2)
    assert again.fri_proof.serialize() == blob and t2.random() == ot.random()
    sh.free()


@pytest.mark.gpu
def test_n_vars_1_fails_like_the_unsharded_prover(ml, oracle):
    """n_vars = 1 (domain 4): the first fold is the last element, so BatchedFriProverData::open_query_at has no folded layer and
    the reference returns None; the handle accepts the size but its prove reports ML_ERR_OUT_OF_RANGE like ml_batched_pcs_prove"""
    polys, inp, outs = claim(oracle, 1, 2, 1)
    _, st = oracle.batched_pcs_prove(inp, outs, polys, oracle.transcript())
    assert st == 3
    with pytest.raises(ml.MlError) as e:
        ml.BatchedPCSProof.prove(inp, outs, polys, ml.Transcript())
    assert e.value.code == 3
    sh = ml.BlockShardedBatchedProver.single_process([0], 2, 1)
    with pytest.raises(ml.MlError) as e:
        sh.prove(inp, outs, polys, ml.Transcript())
    assert e.value.code == 3
    sh.free()


def reference_claim(ml, nv=20, B=10):
    """batched_pcs_verify_test's inputs (batched_pcs.rs:262-306): evals (3j + 5i) % 100 for polynomial i, inputs 0 .. n_vars-1"""
    j = np.arange(1 << nv, dtype=np.int64)
    polys = [ml.from_i64(((3 * j + 5 * i) % 100).tolist()) for i in range(B)]
    inp = ml.from_i64(range(nv))
    outs = fe_arr([ml.MultilinearPolynomialEvals(p).evaluate(ml.to_ints(inp)) for p in polys])
    return polys, inp, outs


@pytest.mark.gpu
@pytest.mark.parametrize("world", [4, 8])
def test_reference_batched_pcs_verify_inputs(ml, oracle, world):
    polys, inp, outs = reference_claim(ml)
    sh = ml.BlockShardedBatchedProver.single_process([0] * world, len(polys), 20)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = sh.prove(inp, outs, polys, t)
    oproof, st = oracle.batched_pcs_prove(inp, outs, polys, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck and t.random() == ot.random()
    assert proof.verify(ml.Transcript()) == 0
    sh.free()


def _dev_polys(ml, seeds, n):
    import torch
    from multilinear_b200 import load
    L, out = load(), []
    for s in seeds:
        t = torch.empty(16 * n, dtype=torch.uint8, device="cuda")
        ml.check(L.ml_synthetic_elements_dev(C.c_uint64(s), C.c_size_t(n), C.c_void_p(t.data_ptr()),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        out.append(t)
    torch.cuda.synchronize()
    return out


def unsharded_dev(ml, inp, outs, bufs, n, t):
    from multilinear_b200 import load
    ptrs = (C.c_void_p * len(bufs))(*[b.data_ptr() for b in bufs])
    h = C.c_void_p()
    ml.check(load().ml_batched_pcs_prove_dev(ml._p(inp), ml._sz(inp.shape[0]), ml._p(outs), ml._sz(len(bufs)), ptrs, ml._sz(n), t.h,
                                             None, C.byref(h)))
    return ml.PCSProof(h, batched=True)


def sharded_dev(ml, sh, inp, outs, bufs, n, world, t):
    ptrs = [b.data_ptr() + g * (n // world) * 16 for g in range(world) for b in bufs]
    return sh.prove_dev(inp, outs, ptrs, t)


def _batch_commitment(proof):
    out = np.empty(32, dtype=np.uint8)
    from multilinear_b200 import load
    load().ml_bfri_proof_batch_commitment(proof.fri_proof.h, out.ctypes.data_as(C.c_void_p))
    return out.tobytes()


@pytest.mark.gpu
def test_at_size_64x2p22_world8_batch_root(ml):
    """64 polynomials of 2^22 evaluations (bench.py's seeds 5000 + j) with 8 virtual ranks: the batch commitment equals the
    committed Merkle::batch_commit root, and the proof bytes equal the unsharded prover's (any claim: the prover does not check it)"""
    import torch
    nv, B, world = 22, 64, 8
    n = 1 << nv
    fx = json.load(open(os.path.join(HERE, "golden", "batch_root_64x2p22.json")))
    assert fx["n_polys"] == B and fx["log_n"] == nv
    bufs = _dev_polys(ml, [5000 + j for j in range(B)], n)
    inp = ml.synthetic_elements_dev(0xB2000001, nv).elems()
    outs = ml.synthetic_elements_dev(0xB2000002, B).elems()
    sh = ml.BlockShardedBatchedProver.single_process([0] * world, B, nv)
    t = ml.Transcript()
    proof = sharded_dev(ml, sh, inp, outs, bufs, n, world, t)
    assert _batch_commitment(proof).hex() == fx["root"]
    sh.free()
    t1 = ml.Transcript()
    single = unsharded_dev(ml, inp, outs, bufs, n, t1)
    assert proof.fri_proof.serialize() == single.fri_proof.serialize() and t.random() == t1.random()
    assert proof.sumcheck_polynomials == single.sumcheck_polynomials
    del bufs
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_at_size_b3_n24_world8_equals_unsharded(ml):
    nv, B, world = 24, 3, 8
    n = 1 << nv
    bufs = _dev_polys(ml, [0xB200 + j for j in range(B)], n)
    inp = ml.synthetic_elements_dev(0xB2000001, nv).elems()
    outs = ml.synthetic_elements_dev(0xB2000003, B).elems()  # any claim: the prover does not check it
    t1 = ml.Transcript()
    single = unsharded_dev(ml, inp, outs, bufs, n, t1)
    sh = ml.BlockShardedBatchedProver.single_process([0] * world, B, nv)
    t = ml.Transcript()
    proof = sharded_dev(ml, sh, inp, outs, bufs, n, world, t)
    assert proof.fri_proof.serialize() == single.fri_proof.serialize()
    assert proof.sumcheck_polynomials == single.sumcheck_polynomials and t.random() == t1.random()
    sh.free()


# ------------------------------------------------------------------ failure cases
def first_batch_path(blob):
    """(value, path, index) of query 0's layer-0 batch opening, parsed from the serialized BatchedFriProof"""
    o = 32
    nc = struct.unpack_from("<Q", blob, o)[0]
    o += 8 + 32 * nc + 8  # commitments, number of queries
    nb = struct.unpack_from("<Q", blob, o)[0]
    o += 8
    value = b""
    for _ in range(2 * nb):
        assert struct.unpack_from("<Q", blob, o)[0] == 16
        value += blob[o + 8:o + 24]
        o += 24
    depth = struct.unpack_from("<Q", blob, o)[0]
    o += 8
    path, index = [], 0
    for i in range(depth):
        d = struct.unpack_from("<I", blob, o + 32)[0]
        path.append((blob[o:o + 32], d))
        index |= (d == 0) << i
        o += 36
    return value, path, index


@pytest.mark.gpu
def test_wrong_claim_and_flipped_openings(ml, oracle):
    world, B, nv = 4, 5, 10
    polys, inp, outs = claim(oracle, world, B, nv)
    sh = ml.BlockShardedBatchedProver.single_process([0] * world, B, nv)
    ints = ml.to_ints(outs)
    wrong = fe_arr([(x + 1) % M if j == 2 else x for j, x in enumerate(ints)])
    tw, t1 = ml.Transcript(), ml.Transcript()
    pw = sh.prove(inp, wrong, polys, tw)
    single = ml.BatchedPCSProof.prove(inp, wrong, polys, t1)
    assert pw.fri_proof.serialize() == single.fri_proof.serialize() and tw.random() == t1.random()
    assert pw.verify(ml.Transcript()) == 107  # ML_V_SUMCHECK
    proof = sh.prove(inp, outs, polys, ml.Transcript())
    blob = proof.fri_proof.serialize()
    root = blob[:32]
    value, path, index = first_batch_path(blob)
    assert len(value) == 32 * B and len(path) == nv
    assert ml.path_verify(value, path, root, index) == 0
    bad = bytearray(value)
    bad[32 * (B - 1) + 5] ^= 1  # one byte of the last code's minus-value
    assert ml.path_verify(bytes(bad), path, root, index) != 0
    for lvl in (0, nv - 1):  # a digest in the owner's segment subtree, and one in the top tree
        d = bytearray(path[lvl][0])
        d[0] ^= 0x80
        bp = list(path)
        bp[lvl] = (bytes(d), path[lvl][1])
        assert ml.path_verify(value, bp, root, index) != 0
    sh.free()


@pytest.mark.gpu
def test_misuse(ml, oracle):
    polys, inp, outs = claim(oracle, 2, 3, 8)
    sh = ml.BlockShardedBatchedProver.single_process([0, 0], 3, 8)
    with pytest.raises(ml.MlError) as e:  # the claim has 7 variables, the handle 8
        sh.prove_dev(inp[:7], outs, [0] * 6, ml.Transcript())
    assert e.value.code == 2
    with pytest.raises(ml.MlError) as e:  # two outputs, the handle three polynomials
        sh.prove_dev(inp, outs[:2], [0] * 4, ml.Transcript())
    assert e.value.code == 2
    with pytest.raises(ml.MlError) as e:
        sh.prove(inp, outs, [p[:128] for p in polys], ml.Transcript())
    assert e.value.code == 2
    sh.free()
    one = ml.BlockShardedBatchedProver.one_rank(1, 2, 0, 3, 8)
    with pytest.raises(ml.MlError) as e:  # peers never connected
        one.prove_dev(inp, outs, [0] * 3, ml.Transcript())
    assert e.value.code == 8
    with pytest.raises(ml.MlError) as e:  # the host entry needs every rank in this process
        one.prove(inp, outs, polys, ml.Transcript())
    assert e.value.code == 8 and "every rank" in str(e.value)
    one.free()


# ------------------------------------------------------------------ real GPUs
def _gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
def test_single_process_two_devices(ml, oracle):
    if _gpus() < 2:
        pytest.skip("needs two GPUs")
    polys, inp, outs = claim(oracle, 2, 3, 12)
    sh = ml.BlockShardedBatchedProver.single_process([0, 1], 3, 12)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = sh.prove(inp, outs, polys, t)
    oproof, st = oracle.batched_pcs_prove(inp, outs, polys, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob and t.random() == ot.random()
    sh.free()


@pytest.mark.gpu
def test_world8_on_8_devices_b10_n20(ml, oracle):
    if _gpus() < 8:
        pytest.skip("needs eight GPUs")
    polys, inp, outs = reference_claim(ml)
    sh = ml.BlockShardedBatchedProver.single_process(list(range(8)), 10, 20)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = sh.prove(inp, outs, polys, t)
    oproof, st = oracle.batched_pcs_prove(inp, outs, polys, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob and t.random() == ot.random()
    assert proof.verify(ml.Transcript()) == 0
    sh.free()


@pytest.mark.gpu
def test_two_processes_two_gpus_vs_oracle(ml):
    """one process per GPU (CUDA IPC arenas, NVLink stores, device flags): 3 polynomials at n_vars 14 equal the oracle's proof
    and both transcripts end in the same state"""
    import socket
    import subprocess
    import sys
    if _gpus() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(HERE)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tools", "bpcs_shard_demo.py"), "14", "3", "oracle", "2"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
