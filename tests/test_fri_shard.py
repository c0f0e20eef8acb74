"""ml_fri_shard_*: one FriProof::prove sharded over G ranks (csrc/fri_shard.cu), from coefficients (reed_solomon + prove) or from
a code.  The proof must be byte-identical to the unsharded prover's and the oracle's, whatever the number of ranks."""
import ctypes as C
import hashlib
import time

import pytest

from oracle.binding import fe_ints


# ------------------------------------------------------------------ argument checks (no GPU needed: they come before any device)
def test_create_rejects_bad_world_and_small_sizes(ml):
    for world in (3, 32):
        with pytest.raises(ml.MlError) as e:
            ml.ShardedFriProver.single_process([0] * world, 12)
        assert e.value.code == 8, world  # ML_ERR_ARG
    for world, log_g in ((2, 1), (4, 2), (8, 3), (16, 4)):
        with pytest.raises(ml.MlError) as e:
            ml.ShardedFriProver.single_process([0] * world, 2 * log_g - 1)
        assert e.value.code == 2, world  # ML_ERR_SIZE
    with pytest.raises(ml.MlError) as e:
        ml.ShardedFriProver.single_process([0], 0)
    assert e.value.code == 2


def test_create_without_gpu_fails_loudly(ml):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(ml.MlError) as e:
        ml.ShardedFriProver.single_process([0, 0], 6)
    assert e.value.code in (6, 7)  # no device: no CPU fallback


# ------------------------------------------------------------------ virtual ranks on one GPU
def rs_case(oracle, seed, log_n):
    """coefficients, gen_pows of the code domain, and the code reed_solomon(c, g)"""
    c = oracle.synthetic(seed, 1 << log_n)
    gp = oracle.pow2_generator_powers(log_n + 1)
    return c, gp, oracle.reed_solomon(c, fe_ints(gp[1:2])[0])


@pytest.mark.gpu
@pytest.mark.parametrize("world,log_n", [(1, 1), (1, 6), (2, 2), (2, 9), (2, 20), (4, 4), (4, 12), (4, 20), (8, 6), (8, 14), (16, 8), (16, 13),
                                         (16, 20)])
def test_virtual_ranks_vs_oracle(ml, oracle, world, log_n):
    c, gp, code = rs_case(oracle, 6000 + 17 * world + log_n, log_n)
    ot = oracle.transcript()
    oproof, st = oracle.fri_prove(code, gp, ot)
    assert st == 0
    sh = ml.ShardedFriProver.single_process([0] * world, log_n)
    t = ml.Transcript()
    proof = sh.rs_prove(c, t)
    blob = proof.serialize()
    assert blob == oproof.blob and t.random() == ot.random()
    assert proof.verify() == 0
    t1 = ml.Transcript()
    assert ml.FriProof.prove_from_coeffs(c, t1).serialize() == blob and t1.random() == ot.random()
    t2 = ml.Transcript()  # the same code through the code entry
    assert sh.prove(code, gp, t2).serialize() == blob and t2.random() == ot.random()
    t3 = ml.Transcript()
    assert ml.FriProof.prove(code, gp, t3).serialize() == blob and t3.random() == ot.random()
    t4 = ml.Transcript()  # a second call on the same handle gives the same bytes
    assert sh.rs_prove(c, t4).serialize() == blob and t4.random() == ot.random()
    sh.free()


@pytest.mark.gpu
def test_transcript_with_history(ml, oracle):
    """a transcript that has absorbed something before the proof: the sharded prover continues from its state"""
    c, gp, code = rs_case(oracle, 77, 10)
    sh = ml.ShardedFriProver.single_process([0] * 4, 10)
    for entry in ("rs", "code"):
        t, t1 = ml.Transcript(), ml.Transcript()
        t.absorb(b"earlier messages")
        t1.absorb(b"earlier messages")
        p = sh.rs_prove(c, t) if entry == "rs" else sh.prove(code, None, t)
        single = ml.FriProof.prove_from_coeffs(c, t1)
        assert p.serialize() == single.serialize() and t.random() == t1.random(), entry
    sh.free()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4, 8, 16])
def test_reference_inputs_log10(ml, golden, world):
    """prove_and_verify_test's inputs (coefficients 7i+3, 2^10 of them): the golden proof at every number of ranks"""
    g = golden["fri_log10"]
    vals = ml.from_i64([7 * i + 3 for i in range(1 << 10)])
    gp = ml.pow_2_generator_powers(11)
    code = ml.reed_solomon(vals, ml.to_ints(gp[1:2])[0])
    sh = ml.ShardedFriProver.single_process([0] * world, 10)
    for proof in (sh.rs_prove(vals, ml.Transcript()), sh.prove(code, gp, ml.Transcript())):
        assert [c.hex() for c in proof.commitments] == g["commitments"]
        assert str(proof.last_elem) == g["last_elem"] and proof.last_random.hex() == g["last_random"]
        blob = proof.serialize()
        assert len(blob) == g["blob_len"] and hashlib.sha256(blob).hexdigest() == g["blob_sha"]
        assert proof.verify() == 0
    sh.free()


def at_size_n24_equals_unsharded(ml, world):
    log_n, n = 24, 1 << 24
    coeffs = ml.synthetic_elements_dev(0xF21, n)
    t1 = ml.Transcript()
    h = C.c_void_p()
    ml.check(ml.load().ml_rs_fri_prove_dev(coeffs.ptr, C.c_size_t(n), t1.h, None, C.byref(h)))
    single = ml.FriProof(h)
    ml.synchronize()
    sh = ml.ShardedFriProver.single_process([0] * world, log_n)
    t = ml.Transcript()
    proof = sh.rs_prove_dev([coeffs.ptr.value + g * (n // world) * 16 for g in range(world)], t)
    assert proof.serialize() == single.serialize() and t.random() == t1.random()
    assert proof.verify() == 0
    sh.free()


@pytest.mark.gpu
def test_at_size_n24_world8_equals_unsharded(ml):
    """2^24 coefficients (the headline size) with 8 virtual ranks: the same bytes as ml_rs_fri_prove_dev"""
    at_size_n24_equals_unsharded(ml, 8)


@pytest.mark.gpu
def test_at_size_n24_world16_equals_unsharded(ml):
    """the same with 16 virtual ranks: the G = 16 transpose and combine, and the tail chain from layer 4 at a realistic size"""
    at_size_n24_equals_unsharded(ml, 16)


@pytest.mark.gpu
def test_dev_entries_read_only(ml, oracle):
    """_dev entries with block pointers into one buffer each; the caller's blocks are left as they were"""
    world, log_n = 4, 11
    c, gp, code = rs_case(oracle, 91, log_n)
    cbuf, kbuf = ml.DeviceBuffer.from_host(c), ml.DeviceBuffer.from_host(code)
    sh = ml.ShardedFriProver.single_process([0] * world, log_n)
    ot = oracle.transcript()
    oproof, st = oracle.fri_prove(code, gp, ot)
    t, t2 = ml.Transcript(), ml.Transcript()
    p = sh.rs_prove_dev([cbuf.ptr.value + g * ((1 << log_n) // world) * 16 for g in range(world)], t)
    p2 = sh.prove_dev([kbuf.ptr.value + g * ((2 << log_n) // world) * 16 for g in range(world)], t2)
    assert st == 0 and p.serialize() == oproof.blob == p2.serialize() and t.random() == ot.random() == t2.random()
    assert (cbuf.elems() == c).all() and (kbuf.elems() == code).all()
    sh.free()


@pytest.mark.gpu
def test_not_an_rs_code(ml, oracle):
    """random elements are not an RS code: the same status as ml_fri_prove, at once (not after the peer timeout), and the handle
    proves a valid code correctly afterwards"""
    world, log_n = 4, 8
    junk = oracle.synthetic(0xBAD, 2 << log_n)
    gp = oracle.pow2_generator_powers(log_n + 1)
    with pytest.raises(ml.MlError) as e1:
        ml.FriProof.prove(junk, gp, ml.Transcript())
    sh = ml.ShardedFriProver.single_process([0] * world, log_n)
    t0 = time.time()
    with pytest.raises(ml.MlError) as e:
        sh.prove(junk, gp, ml.Transcript())
    elapsed = time.time() - t0
    assert e.value.code == e1.value.code == 4  # ML_ERR_NOT_RS_CODE
    assert elapsed < 5.0, elapsed  # the peer timeout is 20 s
    c, gp, code = rs_case(oracle, 12, log_n)
    ot = oracle.transcript()
    oproof, st = oracle.fri_prove(code, gp, ot)
    t = ml.Transcript()
    assert st == 0 and sh.prove(code, gp, t).serialize() == oproof.blob and t.random() == ot.random()
    sh.free()


@pytest.mark.gpu
def test_misuse(ml, oracle):
    log_n = 8
    c, gp, code = rs_case(oracle, 5, log_n)
    sh = ml.ShardedFriProver.single_process([0, 0], log_n)
    with pytest.raises(ml.MlError) as e:  # 128 coefficients, the handle 256
        sh.rs_prove(c[:128], ml.Transcript())
    assert e.value.code == 2
    with pytest.raises(ml.MlError) as e:  # a code of 256 elements, the handle 512
        sh.prove(code[:256], gp, ml.Transcript())
    assert e.value.code == 2
    for bad in (gp[:256], gp.copy()):
        if len(bad) == len(gp):
            bad[1] = bad[2]  # a probed position: not the domain generator
        with pytest.raises(ml.MlError) as e1:
            ml.FriProof.prove(code, bad, ml.Transcript())
        with pytest.raises(ml.MlError) as e:
            sh.prove(code, bad, ml.Transcript())
        assert e.value.code == e1.value.code and e.value.code in (2, 5)  # ML_ERR_SIZE / ML_ERR_GENERATOR
    sh.free()
    one = ml.ShardedFriProver.one_rank(1, 2, 0, log_n)
    with pytest.raises(ml.MlError) as e:  # peers never connected
        one.rs_prove_dev([0], ml.Transcript())
    assert e.value.code == 8
    with pytest.raises(ml.MlError) as e:
        one.prove_dev([0], ml.Transcript())
    assert e.value.code == 8
    for call in (lambda: one.rs_prove(c, ml.Transcript()), lambda: one.prove(code, gp, ml.Transcript())):
        with pytest.raises(ml.MlError) as e:  # the host entries need every rank in this process
            call()
        assert e.value.code == 8 and "every rank" in str(e.value)
    one.free()


@pytest.mark.gpu
@pytest.mark.parametrize("world,log_n", [(1, 12), (2, 12), (4, 12), (8, 12), (16, 12), (8, 20)])
def test_arena_holds_no_tables(ml, world, log_n):
    fri = ml.ShardedFriProver.single_process([0] * world, log_n)
    pcs = ml.ShardedPCSProver.single_process([0] * world, log_n)
    assert fri.arena_bytes() < pcs.arena_bytes()
    fri.free()
    pcs.free()


# ------------------------------------------------------------------ real GPUs
def _gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
def test_single_process_two_devices(ml, oracle):
    if _gpus() < 2:
        pytest.skip("needs two GPUs")
    c, gp, code = rs_case(oracle, 21, 12)
    sh = ml.ShardedFriProver.single_process([0, 1], 12)
    ot = oracle.transcript()
    oproof, st = oracle.fri_prove(code, gp, ot)
    t, t2 = ml.Transcript(), ml.Transcript()
    assert st == 0 and sh.rs_prove(c, t).serialize() == oproof.blob and t.random() == ot.random()
    assert sh.prove(code, gp, t2).serialize() == oproof.blob and t2.random() == ot.random()
    sh.free()


@pytest.mark.gpu
def test_world8_on_8_devices_n20(ml, oracle):
    if _gpus() < 8:
        pytest.skip("needs eight GPUs")
    c, gp, code = rs_case(oracle, 22, 20)
    sh = ml.ShardedFriProver.single_process(list(range(8)), 20)
    ot = oracle.transcript()
    oproof, st = oracle.fri_prove(code, gp, ot)
    t = ml.Transcript()
    proof = sh.rs_prove(c, t)
    assert st == 0 and proof.serialize() == oproof.blob and t.random() == ot.random()
    assert proof.verify() == 0
    sh.free()


@pytest.mark.gpu
def test_two_processes_two_gpus_vs_oracle(ml):
    """one process per GPU (CUDA IPC arenas, NVLink stores, device flags): the proof equals the oracle's at log_n 14 and both
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
           "--master-port", str(port), os.path.join(root, "tools", "fri_shard_demo.py"), "14", "oracle", "2"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    line = [json.loads(l) for l in p.stdout.splitlines() if l.startswith("{") and "fri_shard_prove" in l][-1]
    assert line["n_gpus"] == 2 and line["matches_oracle"] is True and line["verifies"] is True and line["transcripts_agree"] is True
