"""ml_pcs_shard_*: one PCSProof::prove sharded over G ranks (csrc/pcs_shard.cu).  The proof must be byte-identical to the
unsharded prover's and the oracle's, whatever the number of ranks."""
import hashlib
import random

import numpy as np
import pytest

from oracle import pyref as P
from oracle.binding import fe_arr

M = P.M


# ------------------------------------------------------------------ argument checks (no GPU needed: they come before any device)
def test_create_rejects_bad_world_and_small_sizes(ml):
    for world in (3, 32):
        with pytest.raises(ml.MlError) as e:
            ml.ShardedPCSProver.single_process([0] * world, 12)
        assert e.value.code == 8, world  # ML_ERR_ARG
    for world, log_g in ((2, 1), (4, 2), (8, 3), (16, 4)):
        with pytest.raises(ml.MlError) as e:
            ml.ShardedPCSProver.single_process([0] * world, 2 * log_g - 1)
        assert e.value.code == 2, world  # ML_ERR_SIZE
    with pytest.raises(ml.MlError) as e:
        ml.ShardedPCSProver.single_process([0], 0)
    assert e.value.code == 2


def test_create_without_gpu_fails_loudly(ml):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(ml.MlError) as e:
        ml.ShardedPCSProver.single_process([0, 0], 6)
    assert e.value.code in (6, 7)  # no device: no CPU fallback


# ------------------------------------------------------------------ virtual ranks on one GPU
def claim(oracle, world, nv):
    rng = random.Random(world * 100 + nv)
    ev = oracle.synthetic(4000 + 17 * world + nv, 1 << nv)
    inp = fe_arr([rng.randrange(M) for _ in range(nv)])
    return ev, inp, oracle.mle_evals_evaluate(ev, inp)


@pytest.mark.gpu
@pytest.mark.parametrize("world,nv", [(1, 1), (1, 6), (2, 2), (2, 9), (2, 20), (4, 4), (4, 12), (4, 20), (8, 6), (8, 14), (16, 8), (16, 13),
                                      (16, 20)])
def test_virtual_ranks_vs_oracle(ml, oracle, world, nv):
    ev, inp, out = claim(oracle, world, nv)
    sh = ml.ShardedPCSProver.single_process([0] * world, nv)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = sh.prove(inp, out, ev, t)
    oproof, st = oracle.pcs_prove(inp, out, ev, ot)
    assert st == 0
    blob = proof.fri_proof.serialize()
    assert blob == oproof.fri.blob
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck
    assert t.random() == ot.random()
    assert proof.verify(ml.Transcript()) == 0
    t1 = ml.Transcript()
    assert ml.PCSProof.prove(inp, out, ev, t1).fri_proof.serialize() == blob and t1.random() == ot.random()
    t2 = ml.Transcript()  # a second call on the same handle gives the same bytes
    assert sh.prove(inp, out, ev, t2).fri_proof.serialize() == blob and t2.random() == ot.random()
    sh.free()


@pytest.mark.gpu
def test_reference_inputs_n20_world8(ml, oracle):
    """multilinear_pcs_bench_test's inputs (multilinear_pcs.rs:211-228): n_vars 20, evals 7i+3, inputs i"""
    nv = 20
    ev = ml.from_i64([7 * i + 3 for i in range(1 << nv)])
    inp = ml.from_i64(range(nv))
    out = ml.MultilinearPolynomialEvals(ev).evaluate(ml.to_ints(inp))
    sh = ml.ShardedPCSProver.single_process([0] * 8, nv)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = sh.prove(inp, out, ev, t)
    oproof, st = oracle.pcs_prove(inp, out, ev, ot)
    assert st == 0 and hashlib.sha256(proof.fri_proof.serialize()).digest() == hashlib.sha256(oproof.fri.blob).digest()
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck and t.random() == ot.random()
    assert proof.verify(ml.Transcript()) == 0
    sh.free()


def at_size_n24_equals_unsharded(ml, world):
    nv, n = 24, 1 << 24
    evals = ml.synthetic_elements_dev(0xB200, n)
    inp = ml.synthetic_elements_dev(0xB2000001, nv).elems()
    out = ml.MultilinearPolynomialEvals(evals.elems()).evaluate(ml.to_ints(inp))
    t1 = ml.Transcript()
    single = ml.PCSProof.prove_dev(inp, out, evals, n, t1)
    sh = ml.ShardedPCSProver.single_process([0] * world, nv)
    t = ml.Transcript()
    proof = sh.prove_dev(inp, out, [evals.ptr.value + g * (n // world) * 16 for g in range(world)], t)
    assert proof.fri_proof.serialize() == single.fri_proof.serialize()
    assert proof.sumcheck_polynomials == single.sumcheck_polynomials and t.random() == t1.random()
    sh.free()


@pytest.mark.gpu
def test_at_size_n24_world8_equals_unsharded(ml):
    """n_vars 24 with 8 virtual ranks: the same bytes as the unsharded CUDA prover (itself pinned to the oracle at this size by
    test_atsize_pcs_prove_n_vars_24)"""
    at_size_n24_equals_unsharded(ml, 8)


@pytest.mark.gpu
def test_at_size_n24_world16_equals_unsharded(ml):
    """the same with 16 virtual ranks: the combine kernel for G = 16 and the tail chain from layer 4 at a realistic size"""
    at_size_n24_equals_unsharded(ml, 16)


@pytest.mark.gpu
def test_dev_entry_and_wrong_claim(ml, oracle):
    """_dev with block pointers into one buffer; a wrong claimed output gives the unsharded prover's bytes, and the verifier
    rejects both with the same status"""
    world, nv = 4, 10
    ev, inp, out = claim(oracle, world, nv)
    buf = ml.DeviceBuffer.from_host(ev)
    blocks = [buf.ptr.value + g * ((1 << nv) // world) * 16 for g in range(world)]
    sh = ml.ShardedPCSProver.single_process([0] * world, nv)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = sh.prove_dev(inp, out, blocks, t)
    oproof, st = oracle.pcs_prove(inp, out, ev, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob and t.random() == ot.random()
    wrong = (out + 1) % M
    tw, t1 = ml.Transcript(), ml.Transcript()
    pw = sh.prove_dev(inp, wrong, blocks, tw)
    single = ml.PCSProof.prove(inp, wrong, ev, t1)
    assert pw.fri_proof.serialize() == single.fri_proof.serialize() and tw.random() == t1.random()
    assert pw.sumcheck_polynomials == single.sumcheck_polynomials
    vs = pw.verify(ml.Transcript())
    assert vs != 0 and vs == single.verify(ml.Transcript())
    sh.free()


@pytest.mark.gpu
def test_misuse(ml, oracle):
    ev, inp, out = claim(oracle, 2, 8)
    sh = ml.ShardedPCSProver.single_process([0, 0], 8)
    with pytest.raises(ml.MlError) as e:  # the claim has 7 variables, the handle 8
        sh.prove_dev(inp[:7], out, [0, 0], ml.Transcript())
    assert e.value.code == 2
    with pytest.raises(ml.MlError) as e:
        sh.prove(inp, out, ev[:128], ml.Transcript())
    assert e.value.code == 2
    sh.free()
    one = ml.ShardedPCSProver.one_rank(1, 2, 0, 8)
    with pytest.raises(ml.MlError) as e:  # peers never connected
        one.prove_dev(inp, out, [0], ml.Transcript())
    assert e.value.code == 8
    with pytest.raises(ml.MlError) as e:  # the host entry needs every rank in this process
        one.prove(inp, out, ev, ml.Transcript())
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
    ev, inp, out = claim(oracle, 2, 12)
    sh = ml.ShardedPCSProver.single_process([0, 1], 12)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = sh.prove(inp, out, ev, t)
    oproof, st = oracle.pcs_prove(inp, out, ev, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob and t.random() == ot.random()
    sh.free()


@pytest.mark.gpu
def test_world8_on_8_devices_n20(ml, oracle):
    if _gpus() < 8:
        pytest.skip("needs eight GPUs")
    ev, inp, out = claim(oracle, 8, 20)
    sh = ml.ShardedPCSProver.single_process(list(range(8)), 20)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = sh.prove(inp, out, ev, t)
    oproof, st = oracle.pcs_prove(inp, out, ev, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob and t.random() == ot.random()
    assert proof.verify(ml.Transcript()) == 0
    sh.free()


@pytest.mark.gpu
def test_two_processes_two_gpus_vs_oracle(ml):
    """one process per GPU (CUDA IPC arenas, NVLink stores, device flags): the proof equals the oracle's at n_vars 14 and both
    transcripts end in the same state"""
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
           "--master-port", str(port), os.path.join(root, "tools", "pcs_shard_demo.py"), "14", "oracle", "2"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    line = [json.loads(l) for l in p.stdout.splitlines() if l.startswith("{") and "pcs_shard_prove" in l][-1]
    assert line["n_gpus"] == 2 and line["matches_oracle"] is True and line["verifies"] is True and line["transcripts_agree"] is True
