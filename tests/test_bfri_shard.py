"""ml_bfri_shard_*: one BatchedFriProof::prove of B codes, each split by block over G ranks (csrc/bfri_shard.cu), from the
polynomials' coefficients (reed_solomon of each + prove) or from their codes.  The proof must be byte-identical to the unsharded
prover's and the oracle's, whatever the number of ranks and codes."""
import hashlib
import time

import pytest

from oracle.binding import fe_ints


# ------------------------------------------------------------------ argument checks (no GPU needed: they come before any device)
def test_create_rejects_bad_world_batch_and_small_sizes(ml):
    for world in (3, 32):
        with pytest.raises(ml.MlError) as e:
            ml.ShardedBatchedFriProver.single_process([0] * world, 2, 12)
        assert e.value.code == 8, world  # ML_ERR_ARG
    for world, log_g in ((2, 1), (4, 2), (8, 3), (16, 4)):
        with pytest.raises(ml.MlError) as e:
            ml.ShardedBatchedFriProver.single_process([0] * world, 2, 2 * log_g - 1)
        assert e.value.code == 2, world  # ML_ERR_SIZE
    with pytest.raises(ml.MlError) as e:
        ml.ShardedBatchedFriProver.single_process([0, 0], 0, 8)
    assert e.value.code == 2
    with pytest.raises(ml.MlError) as e:
        ml.ShardedBatchedFriProver.single_process([0], 2, 0)
    assert e.value.code == 2


def test_create_without_gpu_fails_loudly(ml):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(ml.MlError) as e:
        ml.ShardedBatchedFriProver.single_process([0, 0], 3, 6)
    assert e.value.code in (6, 7)  # no device: no CPU fallback


# ------------------------------------------------------------------ virtual ranks on one GPU
_ORACLE = {}


def rs_case(oracle, B, log_n):
    """coefficients of B polynomials, gen_pows of the code domain, their codes, and the oracle's proof blob and final challenge
    (cached: the same shape is proved at every number of ranks)"""
    key = (B, log_n)
    if key not in _ORACLE:
        cs = [oracle.synthetic(0xBF000 + 64 * log_n + j, 1 << log_n) for j in range(B)]
        gp = oracle.pow2_generator_powers(log_n + 1)
        gen = fe_ints(gp[1:2])[0]
        codes = [oracle.reed_solomon(c, gen) for c in cs]
        ot = oracle.transcript()
        oproof, st = oracle.batched_fri_prove(codes, gp, ot)
        assert st == 0
        _ORACLE.clear()  # keep one shape's arrays at a time
        _ORACLE[key] = (cs, gp, codes, oproof.blob, ot.random())
    return _ORACLE[key]


def _cases():
    out = []
    for world in (1, 2, 4, 8, 16):
        lo = max(2, 2 * (world.bit_length() - 1))
        for B in (1, 2, 3, 5, 17):
            for log_n in sorted({lo, 13}):
                out.append((B, log_n, world))
    out += [(B, 20, world) for B in (1, 3) for world in (1, 2, 4, 8, 16)]
    return sorted(out)  # grouped by shape, so the oracle runs once per shape


@pytest.mark.gpu
@pytest.mark.parametrize("B,log_n,world", _cases())
def test_virtual_ranks_vs_oracle(ml, oracle, B, log_n, world):
    cs, gp, codes, oblob, orand = rs_case(oracle, B, log_n)
    sh = ml.ShardedBatchedFriProver.single_process([0] * world, B, log_n)
    t = ml.Transcript()
    proof = sh.rs_prove(cs, t)
    blob = proof.serialize()
    assert blob == oblob and t.random() == orand
    assert proof.verify() == 0
    t1 = ml.Transcript()
    assert ml.BatchedFriProof.prove(codes, gp, t1).serialize() == blob and t1.random() == orand
    t2 = ml.Transcript()  # the same codes through the code entry
    assert sh.prove(codes, gp, t2).serialize() == blob and t2.random() == orand
    t3 = ml.Transcript()  # a second call on the same handle gives the same bytes
    assert sh.rs_prove(cs, t3).serialize() == blob and t3.random() == orand
    sh.free()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_golden_bfri_log6_b4(ml, golden, world):
    """the crate's batched FRI test inputs (4 codes of 128 elements): the golden proof at every number of ranks"""
    g = golden["bfri_log6_b4"]
    gp = ml.pow_2_generator_powers(7)
    gen = ml.to_ints(gp[1:2])[0]
    coeffs = [ml.from_i64([7 * i + 3 + 100 * j for i in range(64)]) for j in range(4)]
    codes = [ml.reed_solomon(c, gen) for c in coeffs]
    sh = ml.ShardedBatchedFriProver.single_process([0] * world, 4, 6)
    for proof in (sh.rs_prove(coeffs, ml.Transcript()), sh.prove(codes, gp, ml.Transcript())):
        assert proof.batch_commitment.hex() == g["batch_commitment"]
        assert [c.hex() for c in proof.commitments] == g["commitments"]
        assert str(proof.last_elem) == g["last_elem"]
        assert hashlib.sha256(proof.serialize()).hexdigest() == g["blob_sha"] and proof.verify() == 0
    sh.free()


@pytest.mark.gpu
def test_transcript_with_history(ml, oracle):
    """a transcript that has absorbed something before the proof: the sharded prover continues from its state"""
    B, log_n = 3, 10
    cs, gp, codes, _, _ = rs_case(oracle, B, log_n)
    sh = ml.ShardedBatchedFriProver.single_process([0] * 4, B, log_n)
    for entry in ("rs", "code"):
        t, t1 = ml.Transcript(), ml.Transcript()
        t.absorb(b"earlier messages")
        t1.absorb(b"earlier messages")
        p = sh.rs_prove(cs, t) if entry == "rs" else sh.prove(codes, None, t)
        single = ml.BatchedFriProof.prove(codes, gp, t1)
        assert p.serialize() == single.serialize() and t.random() == t1.random(), entry
    sh.free()


@pytest.mark.gpu
def test_dev_entries_read_only(ml, oracle):
    """_dev entries with block pointers into one buffer per polynomial; the caller's blocks are left as they were"""
    world, B, log_n = 4, 3, 11
    cs, gp, codes, oblob, orand = rs_case(oracle, B, log_n)
    cbufs, kbufs = [ml.DeviceBuffer.from_host(c) for c in cs], [ml.DeviceBuffer.from_host(k) for k in codes]
    sh = ml.ShardedBatchedFriProver.single_process([0] * world, B, log_n)
    t, t2 = ml.Transcript(), ml.Transcript()
    p = sh.rs_prove_dev([cbufs[j].ptr.value + g * ((1 << log_n) // world) * 16 for g in range(world) for j in range(B)], t)
    p2 = sh.prove_dev([kbufs[j].ptr.value + g * ((2 << log_n) // world) * 16 for g in range(world) for j in range(B)], t2)
    assert p.serialize() == oblob == p2.serialize() and t.random() == orand == t2.random()
    assert all((b.elems() == c).all() for b, c in zip(cbufs, cs)) and all((b.elems() == k).all() for b, k in zip(kbufs, codes))
    sh.free()


@pytest.mark.gpu
def test_not_an_rs_code(ml, oracle):
    """one junk code among valid ones: the same status as ml_batched_fri_prove, at once (not after the peer timeout), and the
    handle proves valid codes correctly afterwards"""
    world, B, log_n = 4, 3, 8
    cs, gp, codes, oblob, orand = rs_case(oracle, B, log_n)
    bad = [codes[0], oracle.synthetic(0xBAD, 2 << log_n), codes[2]]
    with pytest.raises(ml.MlError) as e1:
        ml.BatchedFriProof.prove(bad, gp, ml.Transcript())
    sh = ml.ShardedBatchedFriProver.single_process([0] * world, B, log_n)
    t0 = time.time()
    with pytest.raises(ml.MlError) as e:
        sh.prove(bad, gp, ml.Transcript())
    elapsed = time.time() - t0
    assert e.value.code == e1.value.code == 4  # ML_ERR_NOT_RS_CODE
    assert elapsed < 5.0, elapsed  # the peer timeout is 20 s
    t = ml.Transcript()
    assert sh.prove(codes, gp, t).serialize() == oblob and t.random() == orand
    sh.free()


@pytest.mark.gpu
def test_misuse(ml, oracle):
    B, log_n = 2, 8
    cs, gp, codes, _, _ = rs_case(oracle, B, log_n)
    sh = ml.ShardedBatchedFriProver.single_process([0, 0], B, log_n)
    with pytest.raises(ml.MlError) as e:  # 128 coefficients, the handle 256
        sh.rs_prove([c[:128] for c in cs], ml.Transcript())
    assert e.value.code == 2
    with pytest.raises(ml.MlError) as e:  # codes of 256 elements, the handle 512
        sh.prove([k[:256] for k in codes], gp, ml.Transcript())
    assert e.value.code == 2
    with pytest.raises(ml.MlError) as e:  # three codes, the handle two
        sh.prove(codes + codes[:1], gp, ml.Transcript())
    assert e.value.code == 2
    with pytest.raises(ml.MlError) as e:
        sh.rs_prove(cs[:1], ml.Transcript())
    assert e.value.code == 2
    for bad in (gp[:256], gp.copy()):
        if len(bad) == len(gp):
            bad[1] = bad[2]  # a probed position: not the domain generator
        with pytest.raises(ml.MlError) as e1:
            ml.FriProof.prove(codes[0], bad, ml.Transcript())
        with pytest.raises(ml.MlError) as e:
            sh.prove(codes, bad, ml.Transcript())
        assert e.value.code == e1.value.code and e.value.code in (2, 5)  # ML_ERR_SIZE / ML_ERR_GENERATOR
    sh.free()
    one = ml.ShardedBatchedFriProver.one_rank(1, 2, 0, B, log_n)
    with pytest.raises(ml.MlError) as e:  # peers never connected
        one.rs_prove_dev([0] * B, ml.Transcript())
    assert e.value.code == 8
    with pytest.raises(ml.MlError) as e:
        one.prove_dev([0] * B, ml.Transcript())
    assert e.value.code == 8
    for call in (lambda: one.rs_prove(cs, ml.Transcript()), lambda: one.prove(codes, gp, ml.Transcript())):
        with pytest.raises(ml.MlError) as e:  # the host entries need every rank in this process
            call()
        assert e.value.code == 8 and "every rank" in str(e.value)
    one.free()


@pytest.mark.gpu
def test_log_n_1_fails_like_the_unsharded_prover(ml, oracle):
    """a domain of 4 elements has no folded layer to open: the same status as ml_batched_fri_prove"""
    cs = [oracle.synthetic(0xB1 + j, 2) for j in range(2)]
    gp = oracle.pow2_generator_powers(2)
    codes = [oracle.reed_solomon(c, fe_ints(gp[1:2])[0]) for c in cs]
    with pytest.raises(ml.MlError) as e1:
        ml.BatchedFriProof.prove(codes, gp, ml.Transcript())
    sh = ml.ShardedBatchedFriProver.single_process([0], 2, 1)
    for call in (lambda: sh.rs_prove(cs, ml.Transcript()), lambda: sh.prove(codes, gp, ml.Transcript())):
        with pytest.raises(ml.MlError) as e:
            call()
        assert e.value.code == e1.value.code == 3  # ML_ERR_OUT_OF_RANGE
    sh.free()


@pytest.mark.gpu
def test_at_size_64x2p22_world8_equals_unsharded(ml):
    """BASELINE config 5's shape: 64 polynomials of 2^22 coefficients with 8 virtual ranks give the bytes of ml_batched_fri_prove
    on their RS codes (which it takes from the host)"""
    log_n, B, world = 22, 64, 8
    n = 1 << log_n
    coeffs = [ml.synthetic_elements_dev(0xBF5000 + j, n) for j in range(B)]
    sh = ml.ShardedBatchedFriProver.single_process([0] * world, B, log_n)
    t = ml.Transcript()
    proof = sh.rs_prove_dev([coeffs[j].ptr.value + g * (n // world) * 16 for g in range(world) for j in range(B)], t)
    blob = proof.serialize()
    assert proof.verify() == 0
    del proof
    sh.free()
    gp = ml.pow_2_generator_powers(log_n + 1)
    gen = ml.to_ints(gp[1:2])[0]
    host = [c.elems() for c in coeffs]
    del coeffs
    t1 = ml.Transcript()
    single = ml.BatchedFriProof.prove([ml.reed_solomon(c, gen) for c in host], gp, t1)
    assert single.serialize() == blob and t1.random() == t.random()


@pytest.mark.gpu
@pytest.mark.parametrize("world,B,log_n", [(1, 4, 12), (2, 4, 12), (4, 4, 12), (8, 4, 12), (16, 4, 12), (8, 64, 20)])
def test_arena_below_batched_pcs(ml, world, B, log_n):
    """no sumcheck tables, and the transposed coefficients share layer 0's space"""
    bfri = ml.ShardedBatchedFriProver.single_process([0] * world, B, log_n)
    bpcs = ml.BlockShardedBatchedProver.single_process([0] * world, B, log_n)
    assert bfri.arena_bytes() < bpcs.arena_bytes()
    bfri.free()
    bpcs.free()


# ------------------------------------------------------------------ real GPUs
def _gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
def test_single_process_two_devices(ml, oracle):
    if _gpus() < 2:
        pytest.skip("needs two GPUs")
    B, log_n = 3, 12
    cs, gp, codes, oblob, orand = rs_case(oracle, B, log_n)
    sh = ml.ShardedBatchedFriProver.single_process([0, 1], B, log_n)
    t, t2 = ml.Transcript(), ml.Transcript()
    assert sh.rs_prove(cs, t).serialize() == oblob and t.random() == orand
    assert sh.prove(codes, gp, t2).serialize() == oblob and t2.random() == orand
    sh.free()


@pytest.mark.gpu
def test_world8_on_8_devices_n20(ml, oracle):
    if _gpus() < 8:
        pytest.skip("needs eight GPUs")
    B, log_n = 3, 20
    cs, gp, codes, oblob, orand = rs_case(oracle, B, log_n)
    sh = ml.ShardedBatchedFriProver.single_process(list(range(8)), B, log_n)
    t = ml.Transcript()
    proof = sh.rs_prove(cs, t)
    assert proof.serialize() == oblob and t.random() == orand and proof.verify() == 0
    sh.free()


@pytest.mark.gpu
def test_two_processes_two_gpus_vs_oracle(ml):
    """one process per GPU (CUDA IPC arenas, NVLink stores, device flags): the proof of 5 codes equals the oracle's at log_n 12
    and both transcripts end in the same state"""
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
           "--master-port", str(port), os.path.join(root, "tools", "bfri_shard_demo.py"), "12", "5", "oracle", "2"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    line = [json.loads(l) for l in p.stdout.splitlines() if l.startswith("{") and "bfri_shard_prove" in l][-1]
    assert line["n_gpus"] == 2 and line["matches_oracle"] is True and line["verifies"] is True and line["transcripts_agree"] is True
