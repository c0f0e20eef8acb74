"""Stream-ordered batched provers (ml_batched_prove_plan_*, ml_batched_fri_prove_async, ml_batched_rs_fri_prove_async,
ml_batched_pcs_prove_async) and the batched proof reader (ml_bfri_proof_deserialize).

Each async call must leave in device memory exactly what its blocking twin returns: the BatchedFriProof bincode blob of
ml_bfri_proof_serialize, the PCS sumcheck coefficients and the final transcript state.  The device proof writer
(bfri_proof_write_kernel) and write_bfri_proof in csrc/prover.cu state the wire format twice; the parity tests pin the two against
each other at the smallest domain, around the fold chain's tail boundary (the first fold's output reaches 2^12 at 2^13) and at
2^20, for one to seventeen codes, and against the CPU oracle.  Capture into a CUDA graph in global mode is the check that an
enqueue never synchronises, allocates or copies from pageable host memory."""
import ctypes as C
import hashlib
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle.binding import fe_arr, fe_ints
from test_dev_entries import IN_OFF, OUT_OFF, Region, Strm

gpu = pytest.mark.gpu
_sz, _vp = C.c_size_t, C.c_void_p
ML_OK, ML_ERR_SIZE, ML_ERR_NOT_RS_CODE, ML_ERR_CUDA, ML_ERR_ARG = 0, 2, 4, 6, 8
PREFIX = b"stream-ordered batched prove: a transcript that has absorbed something"   # the state starts mid-block
ORACLE_MAX_TOTAL = 1 << 21   # B * N up to this many elements is also checked against the CPU oracle
KINDS = ["codes", "rs", "pcs"]
HERE = os.path.dirname(os.path.abspath(__file__))


def _p(a):
    return _vp(a.ctypes.data)


def _fe(x):
    return np.frombuffer(int(x).to_bytes(16, "little"), dtype=np.uint8).copy()


def _v_codes():
    """the ML_V_* verification codes, read from the header"""
    import re
    text = open(os.path.join(os.path.dirname(HERE), "include", "multilinear_b200.h")).read()
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"\b(ML_V_\w+)\s*=\s*(\d+)", text)}


# ------------------------------------------------------------------ no GPU: the batched proof reader
def _oracle_bfri(oracle, D, B, seed, prefix=b""):
    """an oracle-made BatchedFriProof of B codes of 2^D elements: (blob, oracle proof)"""
    gp = oracle.pow2_generator_powers(D)
    gen = fe_ints(gp[1:2])[0]
    codes = [oracle.reed_solomon(oracle.synthetic(seed + j, 1 << (D - 1)), gen) for j in range(B)]
    t = oracle.transcript()
    t.absorb(prefix)
    op, st = oracle.batched_fri_prove(codes, gp, t)
    assert st == 0
    return op.blob


@pytest.mark.parametrize("D,B", [(3, 1), (4, 2), (6, 3), (9, 5)])
def test_deserialize_oracle_proofs(ml, oracle, D, B):
    """oracle-made batched proofs read back: they verify, and serializing them again gives the same bytes"""
    blob = _oracle_bfri(oracle, D, B, 100 * D + B)
    p = ml.BatchedFriProof.deserialize(blob)
    assert p.verify() == 0
    assert p.serialize() == blob
    assert len(p.commitments) == D - 2


def _bproof_len(D, B):
    """the blob length the plans write: 32 + header(D-1) + 128 (16 + 48 B + 36 (D-1) + query(D-1)) + 56"""
    def path_offset(d, j):
        return 8 + 56 * j + 36 * (j * (d - 1) - j * (j - 1) // 2)

    def query_bytes(d):
        return path_offset(d, d - 1)
    return 32 + 16 + 32 * (D - 2) + 128 * (16 + 48 * B + 36 * (D - 1) + query_bytes(D - 1)) + 56


@pytest.mark.parametrize("D", [3, 4, 6, 9])
@pytest.mark.parametrize("B", [1, 2, 3, 5])
def test_blob_length_formula(oracle, D, B):
    assert len(_oracle_bfri(oracle, D, B, 7 * D + B)) == _bproof_len(D, B)


def _offsets(D, B):
    """byte offsets inside a batched blob: first query, the first batch value of query 0, its first batch sibling, last_random"""
    q0 = 32 + 16 + 32 * (D - 2)
    return {"nq": q0 - 8, "value0": q0 + 8 + 8, "sibling0": q0 + 8 + 48 * B + 8, "last_random": _bproof_len(D, B) - 32}


def test_deserialize_tampered(ml, oracle):
    V = _v_codes()
    D, B = 6, 3
    blob = bytearray(_oracle_bfri(oracle, D, B, 4242))
    off = _offsets(D, B)
    assert int.from_bytes(blob[off["nq"]:off["nq"] + 8], "little") == 128

    def verify(b):
        return ml.BatchedFriProof.deserialize(bytes(b)).verify()

    assert verify(blob) == V["ML_V_OK"]
    b = bytearray(blob)
    b[off["last_random"]] ^= 1
    assert verify(b) == V["ML_V_LAST_RANDOM"]
    b = bytearray(blob)
    b[off["value0"]] ^= 1   # an opened batch value (its low byte: the element stays canonical)
    assert verify(b) == V["ML_V_INCLUSION_HASH"]
    b = bytearray(blob)
    b[off["sibling0"]] ^= 1   # a sibling digest of the batch path
    assert verify(b) == V["ML_V_INCLUSION_HASH"]
    # one query fewer: the count and the bytes of the last query go
    q0 = off["nq"] + 8
    qlen = (len(blob) - q0 - 56) // 128
    b = bytearray(blob[:q0 + 127 * qlen] + blob[q0 + 128 * qlen:])
    b[off["nq"]:off["nq"] + 8] = (127).to_bytes(8, "little")
    assert verify(b) == V["ML_V_WRONG_NUM_QUERIES"]


def test_deserialize_malformed(ml, oracle):
    L = ml.load()
    D, B = 5, 2
    blob = _oracle_bfri(oracle, D, B, 77)
    off = _offsets(D, B)

    def status(b):
        a = np.frombuffer(bytes(b) or b"\0", dtype=np.uint8).copy()
        h = _vp()
        st = L.ml_bfri_proof_deserialize(_p(a), _sz(len(b)), C.byref(h))
        if st == ML_OK:
            L.ml_bfri_proof_free(h)
        return st

    assert status(blob) == ML_OK
    for bad in (b"", blob[:1], blob[:-1], blob[:len(blob) // 2], blob + b"\0", blob + blob):
        assert status(bad) == ML_ERR_ARG, len(bad)
    b = bytearray(blob)   # a batch value length prefix other than 16
    b[off["value0"] - 8] = 15
    assert status(b) == ML_ERR_ARG
    b = bytearray(blob)   # a direction above 1 (the first batch path entry's)
    b[off["sibling0"] + 32] = 2
    assert status(b) == ML_ERR_ARG
    b = bytearray(blob)   # a non-canonical batch value: all ones is above the modulus
    b[off["value0"]:off["value0"] + 16] = b"\xff" * 16
    assert status(b) == ML_ERR_ARG
    b = bytearray(blob)   # a non-canonical last element
    b[off["last_random"] - 16:off["last_random"]] = b"\xff" * 16
    assert status(b) == ML_ERR_ARG


def test_plan_create_without_a_device():
    """with no device visible, creating a plan fails with ML_ERR_CUDA (run in a child process that sees no GPU)"""
    root = os.path.dirname(HERE)
    code = ("import ctypes, multilinear_b200 as m; L = m.load(); h = ctypes.c_void_p(); "
            "print(L.ml_batched_prove_plan_create(ctypes.c_size_t(12), ctypes.c_size_t(3), 1, ctypes.byref(h)), h.value)")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    assert out.stdout.split() == [str(ML_ERR_CUDA), "None"]


# ------------------------------------------------------------------ fixtures and helpers (GPU)
@pytest.fixture(params=["null", "ml_stream", "torch"])
def stream_kind(request, ml):
    import torch
    L = ml.load()
    created = None
    if request.param == "null":
        s = Strm("null", torch.cuda.default_stream(), None)
    elif request.param == "ml_stream":
        p = _vp()
        ml.check(L.ml_stream_create(C.byref(p)))
        created = p.value
        s = Strm("ml_stream", torch.cuda.ExternalStream(created), created)
    else:
        ts = torch.cuda.Stream()
        s = Strm("torch", ts, ts.cuda_stream)
    yield s
    s.ts.synchronize()
    if created:
        ml.check(L.ml_stream_synchronize(_vp(created)))
        ml.check(L.ml_stream_destroy(_vp(created)))


def _torch_strm():
    import torch
    ts = torch.cuda.Stream()
    return Strm("torch", ts, ts.cuda_stream)


class BCase:
    """the inputs of one batched prove of B codes of 2^D elements: codes (codes), coefficients (rs) or evaluations + claim (pcs)"""

    def __init__(self, ml, oracle, kind, D, B, seed, prefix=PREFIX):
        N = 1 << D
        self.kind, self.D, self.B, self.N, self.nv, self.prefix = kind, D, B, N, D - 1, prefix
        rng = random.Random(seed)
        self.gen = ml.pow_2_generator(D)
        polys = [oracle.synthetic(seed * 131 + j, N // 2) for j in range(B)]
        if kind == "codes":
            self.data = [ml.reed_solomon(c, self.gen) for c in polys]
        else:
            self.data = polys
        if kind == "pcs":
            self.inputs = fe_arr([rng.randrange(1 << 127) for _ in range(self.nv)])
            self.outputs = fe_arr([oracle.mle_evals_evaluate(p, self.inputs) for p in polys])

    def codes(self, ml):
        return self.data if self.kind == "codes" else [ml.reed_solomon(c, self.gen) for c in self.data]


def start(t, case):
    t.absorb(case.prefix)
    return t


def blocking(ml, case, strm):
    """the blocking twin on the same inputs: (blob, final transcript state, sumcheck coefficients as bytes or None)"""
    import torch
    L, t = ml.load(), start(ml.Transcript(), case)
    if case.kind != "pcs":
        proof = ml.BatchedFriProof.prove(case.codes(ml), None, t)
        return proof.serialize(), t.export(), None
    with torch.cuda.stream(strm.ts):
        bufs = [torch.from_numpy(np.ascontiguousarray(e).reshape(-1).copy()).cuda() for e in case.data]
    ptrs = (C.c_void_p * case.B)(*[b.data_ptr() for b in bufs])
    h = _vp()
    ml.check(L.ml_batched_pcs_prove_dev(_p(case.inputs), _sz(case.nv), _p(case.outputs), _sz(case.B), ptrs, _sz(case.N // 2), t.h,
                                        strm.arg, C.byref(h)))
    strm.ts.synchronize()
    proof = ml.PCSProof(h, batched=True)
    assert proof.verify(start(ml.Transcript(), case)) == 0
    sc = fe_arr([c for nz in proof.sumcheck_polynomials for c in nz]).tobytes()
    return proof.fri_proof.serialize(), t.export(), sc


class AsyncCall:
    """the buffers of one async call, each at a 16-byte offset between canary bytes; `enqueue` only enqueues"""

    def __init__(self, ml, strm, plan, case, seed=0):
        self.ml, self.strm, self.plan, self.case = ml, strm, plan, case
        state = np.frombuffer(start(ml.Transcript(), case).export(), dtype=np.uint8)
        self.tr = Region(strm, 104, OUT_OFF, state, seed)
        self.proof = Region(strm, plan.proof_bytes, OUT_OFF, seed=seed + 1)
        self.status = Region(strm, 4, OUT_OFF, np.full(4, 0x5A, dtype=np.uint8), seed + 2)
        self.data = [Region(strm, d.size, IN_OFF, d, seed + 10 + j) for j, d in enumerate(case.data)]
        self.ins = list(self.data)
        self.outs = [self.tr, self.proof, self.status]
        if case.kind == "pcs":
            self.inp = Region(strm, 16 * case.nv, IN_OFF, case.inputs, seed + 4)
            self.out = Region(strm, 16 * case.B, IN_OFF, case.outputs, seed + 5)
            self.sc = Region(strm, 32 * case.nv, OUT_OFF, seed=seed + 6)
            self.ins += [self.inp, self.out]
            self.outs.append(self.sc)

    def enqueue(self):
        c, s, ptrs = self.case, self.strm.handle, [r.ptr for r in self.data]
        if c.kind == "codes":
            self.plan.batched_fri_prove_async(ptrs, self.tr.ptr, self.proof.ptr, self.status.ptr, s)
        elif c.kind == "rs":
            self.plan.batched_rs_fri_prove_async(ptrs, self.tr.ptr, self.proof.ptr, self.status.ptr, s)
        else:
            self.plan.batched_pcs_prove_async(self.inp.ptr, self.out.ptr, ptrs, self.tr.ptr, self.proof.ptr, self.sc.ptr, self.status.ptr, s)
        return self

    def results(self):
        """(status, blob, final transcript state, sumcheck bytes or None); canaries intact, inputs unchanged"""
        for r in self.ins:
            r.result(unchanged=True)
        status = int(np.frombuffer(self.status.result().tobytes(), dtype=np.int32)[0])
        sc = self.sc.result().tobytes() if self.case.kind == "pcs" else None
        return status, self.proof.result().tobytes(), self.tr.result().tobytes(), sc

    def unchanged(self):
        for r in self.ins + self.outs:
            r.result(unchanged=True)


def oracle_result(ml, oracle, case):
    """(blob, final random, sumcheck coefficients as ints or None) of the CPU oracle"""
    ot = start(oracle.transcript(), case)
    if case.kind == "pcs":
        op, st = oracle.batched_pcs_prove(case.inputs, case.outputs, case.data, ot)
        assert st == 0
        return op.fri.blob, ot.random(), op.sumcheck
    gp = oracle.pow2_generator_powers(case.D)
    op, st = oracle.batched_fri_prove(case.codes(ml), gp, ot)
    assert st == 0
    return op.blob, ot.random(), None


def check_against_blocking(got, want):
    status, blob, state, sc = got
    wblob, wstate, wsc = want
    assert status == ML_OK
    assert blob == wblob, "async blob differs from ml_bfri_proof_serialize of the blocking proof"
    assert state == wstate, "final transcript differs from the blocking call's"
    assert sc == wsc


# ------------------------------------------------------------------ 1. parity with the blocking twins and the oracle
# every D and every B appears: the smallest domain with one and many codes, the tail boundary (D = 13: the first fold's output is
# 2^12) on both sides, and 2^20
GRID = [(3, 1), (3, 17), (4, 2), (5, 3), (12, 17), (13, 1), (13, 3), (14, 2), (20, 2)]


@gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("D,B", GRID)
def test_async_equals_blocking_and_oracle(ml, oracle, kind, D, B):
    strm = _torch_strm()
    plan = ml.BatchedProvePlan.create(D, B, kind)
    assert plan.proof_bytes == _bproof_len(D, B)
    assert plan.device_bytes >= 32 * (1 << D) + (16 * B << D if kind != "codes" else 0)
    case = BCase(ml, oracle, kind, D, B, 100 * D + B + 7 * KINDS.index(kind))
    want = blocking(ml, case, strm)
    got = AsyncCall(ml, strm, plan, case).enqueue().results()
    check_against_blocking(got, want)
    blob, state = got[1], got[2]
    assert ml.BatchedFriProof.deserialize(blob).serialize() == blob   # (verification starts from a fresh transcript: golden tests)
    if B << D <= ORACLE_MAX_TOTAL:
        oblob, orandom, osc = oracle_result(ml, oracle, case)
        assert blob == oblob, "async blob differs from the oracle's"
        assert ml.Transcript.import_(state).random() == orandom
        if osc is not None:
            assert fe_ints(np.frombuffer(got[3], dtype=np.uint8).reshape(-1, 16)) == osc
    plan.free()


# ------------------------------------------------------------------ 2. golden vectors
class _Given:
    """a case built from given inputs (the crate's test vectors)"""

    def __init__(self, kind, D, data, gen=None, inputs=None, outputs=None):
        self.kind, self.D, self.B, self.N, self.nv, self.prefix = kind, D, len(data), 1 << D, D - 1, b""
        self.data, self.gen, self.inputs, self.outputs = data, gen, inputs, outputs

    def codes(self, ml):
        return self.data if self.kind == "codes" else [ml.reed_solomon(c, self.gen) for c in self.data]


@gpu
def test_golden_bfri_log6_b4(ml, golden):
    """the crate's batched FRI test inputs (4 codes of 128 elements), from codes and from coefficients"""
    g = golden["bfri_log6_b4"]
    gen = ml.pow_2_generator(7)
    coeffs = [ml.from_i64([7 * i + 3 + 100 * j for i in range(64)]) for j in range(4)]
    strm = _torch_strm()
    for kind in ("codes", "rs"):
        data = [ml.reed_solomon(c, gen) for c in coeffs] if kind == "codes" else coeffs
        case = _Given(kind, 7, data, gen)
        plan = ml.BatchedProvePlan.create(7, 4, kind)
        status, blob, _, _ = AsyncCall(ml, strm, plan, case).enqueue().results()
        assert status == ML_OK
        assert hashlib.sha256(blob).hexdigest() == g["blob_sha"], kind
        p = ml.BatchedFriProof.deserialize(blob)
        assert p.batch_commitment.hex() == g["batch_commitment"]
        assert [c.hex() for c in p.commitments] == g["commitments"] and str(p.last_elem) == g["last_elem"]
        assert p.verify() == 0
        plan.free()


@gpu
def test_golden_bpcs_nv6_b10(ml, golden):
    g = golden["bpcs_nv6_b10"]
    nv, B = 6, 10
    polys = [fe_arr([(j * 3 + i * 5) % 100 for j in range(1 << nv)]) for i in range(B)]
    inputs = ml.from_i64(range(nv))
    outputs = [ml.MultilinearPolynomialEvals(p).evaluate(ml.to_ints(inputs)) for p in polys]
    assert [str(o) for o in outputs] == g["outputs"]
    case = _Given("pcs", nv + 1, polys, inputs=inputs, outputs=fe_arr(outputs))
    strm = _torch_strm()
    plan = ml.BatchedProvePlan.create(nv + 1, B, "pcs")
    status, blob, _, sc = AsyncCall(ml, strm, plan, case).enqueue().results()
    assert status == ML_OK
    assert hashlib.sha256(blob).hexdigest() == g["blob_sha"]
    coeffs = fe_ints(np.frombuffer(sc, dtype=np.uint8).reshape(-1, 16))
    assert [[str(coeffs[2 * i]), str(coeffs[2 * i + 1])] for i in range(nv)] == g["sumcheck"]
    assert ml.BatchedFriProof.deserialize(blob).batch_commitment.hex() == g["batch_commitment"]
    plan.free()


# ------------------------------------------------------------------ 3. at size
def _dev_polys(ml, seeds, n):
    import torch
    L, out = ml.load(), []
    for s in seeds:
        t = torch.empty(16 * n, dtype=torch.uint8, device="cuda")
        ml.check(L.ml_synthetic_elements_dev(C.c_uint64(s), C.c_size_t(n), C.c_void_p(t.data_ptr()),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        out.append(t)
    torch.cuda.synchronize()
    return out


def _dev_bytes(ml, raw):
    import torch
    return torch.from_numpy(np.frombuffer(bytes(raw), dtype=np.uint8).copy()).cuda()


def _run_async_raw(ml, plan, kind, ptrs, inp=None, outs=None, nv=0):
    """one async call on the current torch stream over raw device buffers: (status, blob, transcript, sumcheck bytes or None)"""
    import torch
    s = torch.cuda.current_stream()
    tr = _dev_bytes(ml, ml.Transcript().export())
    proof = torch.empty(plan.proof_bytes, dtype=torch.uint8, device="cuda")
    status = torch.full((4,), 0x5A, dtype=torch.uint8, device="cuda")
    sc = torch.empty(32 * nv if kind == "pcs" else 16, dtype=torch.uint8, device="cuda")
    if kind == "codes":
        plan.batched_fri_prove_async(ptrs, tr.data_ptr(), proof.data_ptr(), status.data_ptr(), s.cuda_stream)
    elif kind == "rs":
        plan.batched_rs_fri_prove_async(ptrs, tr.data_ptr(), proof.data_ptr(), status.data_ptr(), s.cuda_stream)
    else:
        plan.batched_pcs_prove_async(inp.data_ptr(), outs.data_ptr(), ptrs, tr.data_ptr(), proof.data_ptr(), sc.data_ptr(),
                                     status.data_ptr(), s.cuda_stream)
    s.synchronize()
    st = int(np.frombuffer(status.cpu().numpy().tobytes(), dtype=np.int32)[0])
    return st, proof.cpu().numpy().tobytes(), tr.cpu().numpy().tobytes(), sc.cpu().numpy().tobytes() if kind == "pcs" else None


@gpu
def test_at_size_config5_64x2p22_pcs(ml):
    """BASELINE config 5: 64 polynomials of 2^22 evaluations (seeds 5000 + j), PCS kind at D = 23.  The batch commitment equals the
    committed Merkle::batch_commit root; blob, sumcheck and transcript equal ml_batched_pcs_prove_dev's (any claim: the prover
    does not check it)"""
    import torch
    nv, B = 22, 64
    n = 1 << nv
    fx = json.load(open(os.path.join(HERE, "golden", "batch_root_64x2p22.json")))
    assert fx["n_polys"] == B and fx["log_n"] == nv
    bufs = _dev_polys(ml, [5000 + j for j in range(B)], n)
    inp = ml.synthetic_elements_dev(0xB2000001, nv).elems()
    outs = ml.synthetic_elements_dev(0xB2000002, B).elems()
    plan = ml.BatchedProvePlan.create(nv + 1, B, "pcs")
    st, blob, state, sc = _run_async_raw(ml, plan, "pcs", [b.data_ptr() for b in bufs], _dev_bytes(ml, inp.tobytes()),
                                         _dev_bytes(ml, outs.tobytes()), nv)
    plan.free()
    assert st == ML_OK
    assert blob[:32].hex() == fx["root"]
    t = ml.Transcript()
    ptrs = (C.c_void_p * B)(*[b.data_ptr() for b in bufs])
    h = _vp()
    ml.check(ml.load().ml_batched_pcs_prove_dev(_p(inp), _sz(nv), _p(outs), _sz(B), ptrs, _sz(n), t.h, None, C.byref(h)))
    proof = ml.PCSProof(h, batched=True)
    assert blob == proof.fri_proof.serialize() and state == t.export()
    assert sc == fe_arr([c for nz in proof.sumcheck_polynomials for c in nz]).tobytes()
    del bufs, proof
    torch.cuda.empty_cache()


@gpu
def test_at_size_8x2p24_codes(ml):
    """8 codes of 2^24 (the RS codes of 2^23 coefficients, seeds 0xB24 + j), CODES kind against ml_batched_fri_prove"""
    import torch
    B, D = 8, 24
    coeffs = _dev_polys(ml, [0xB24 + j for j in range(B)], 1 << (D - 1))
    gen = ml.pow_2_generator(D)
    L = ml.load()
    codes = []
    for c in coeffs:   # the RS codes, through the device reed_solomon entry
        out = torch.empty(16 << D, dtype=torch.uint8, device="cuda")
        ml.check(L.ml_reed_solomon_dev(_vp(c.data_ptr()), _sz(1 << (D - 1)), _p(fe_arr([gen])), _vp(out.data_ptr()), _vp(None)))
        codes.append(out)
    torch.cuda.synchronize()
    plan = ml.BatchedProvePlan.create(D, B, "codes")
    st, blob, state, _ = _run_async_raw(ml, plan, "codes", [c.data_ptr() for c in codes])
    plan.free()
    assert st == ML_OK
    host = [c.cpu().numpy().reshape(-1, 16) for c in codes]
    t = ml.Transcript()
    want = ml.BatchedFriProof.prove(host, None, t)
    assert blob == want.serialize() and state == t.export()
    del codes, coeffs
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ 4. streams and buffers
@gpu
def test_every_stream_kind(ml, oracle, stream_kind):
    """NULL stream, an ml_stream_create stream and a torch stream; canaries around every buffer survive, inputs are unchanged"""
    D, B = 6, 3
    for kind in KINDS:
        case = BCase(ml, oracle, kind, D, B, 500 + KINDS.index(kind))
        plan = ml.BatchedProvePlan.create(D, B, kind)
        want = blocking(ml, case, stream_kind)
        check_against_blocking(AsyncCall(ml, stream_kind, plan, case).enqueue().results(), want)
        plan.free()


# ------------------------------------------------------------------ 5. graph capture
@gpu
def test_graph_capture_global_mode(ml, oracle):
    """one call of each kind (three plans) captured into one graph in global mode: any synchronisation, cudaMalloc or pageable
    copy inside the calls fails the capture.  Three replays with new contents in the same input buffers and reset transcripts."""
    import torch
    D, B = 13, 3
    plans = {k: ml.BatchedProvePlan.create(D, B, k) for k in KINDS}
    side = torch.cuda.Stream()
    strm = Strm("torch", side, side.cuda_stream)
    calls = {k: AsyncCall(ml, strm, plans[k], BCase(ml, oracle, k, D, B, 600 + i)) for i, k in enumerate(KINDS)}
    with torch.cuda.stream(side):   # eager warm-up: every kernel of every call is loaded before capture
        for c in calls.values():
            c.enqueue()
    side.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side, capture_error_mode="global"):
        for c in calls.values():
            c.enqueue()
    torch.cuda.synchronize()

    def write(region, arr):
        t = torch.from_numpy(np.ascontiguousarray(arr).reshape(-1).view(np.uint8).copy()).cuda()
        region.t[region.off:region.off + t.numel()].copy_(t)
        region.image[region.off:region.off + t.numel()] = t.cpu().numpy()

    for rep in range(3):
        cases = {k: BCase(ml, oracle, k, D, B, 700 + 10 * rep + i) for i, k in enumerate(KINDS)}
        with torch.cuda.stream(side):
            for k, c in calls.items():
                for r, d in zip(c.data, cases[k].data):
                    write(r, d)
                if k == "pcs":
                    write(c.inp, cases[k].inputs)
                    write(c.out, cases[k].outputs)
                write(c.tr, np.frombuffer(start(ml.Transcript(), cases[k]).export(), dtype=np.uint8))
            g.replay()
        side.synchronize()
        for k, c in calls.items():
            c.case = cases[k]
            check_against_blocking(c.results(), blocking(ml, cases[k], strm))
    del g
    for p in plans.values():
        p.free()


# ------------------------------------------------------------------ 6. one thread, several proofs in flight
@gpu
def test_one_thread_plans_in_flight(ml, oracle):
    import torch
    D, B = 12, 3
    kinds = ["codes", "rs", "pcs", "rs"]
    calls = []
    for i, k in enumerate(kinds):
        calls.append(AsyncCall(ml, _torch_strm(), ml.BatchedProvePlan.create(D, B, k), BCase(ml, oracle, k, D, B, 800 + i)))
    for c in calls:   # inputs are written on each stream; make them complete before the enqueue burst
        c.strm.ts.synchronize()
    for c in calls:
        c.enqueue()
    torch.cuda.synchronize()
    for c in calls:
        check_against_blocking(c.results(), blocking(ml, c.case, c.strm))
        c.plan.free()


# ------------------------------------------------------------------ 7. not an RS code
@gpu
def test_not_an_rs_code_then_a_valid_one(ml, oracle):
    import torch
    D, B = 8, 2
    strm = _torch_strm()
    plan = ml.BatchedProvePlan.create(D, B, "codes")
    bad = BCase(ml, oracle, "codes", D, B, 900)
    bad.data = [bad.data[0], oracle.synthetic(901, 1 << D)]   # random data: the batch's last fold is not constant
    status = AsyncCall(ml, strm, plan, bad).enqueue().results()[0]
    torch.cuda.synchronize()   # raises on a CUDA error
    assert status == ML_ERR_NOT_RS_CODE
    good = BCase(ml, oracle, "codes", D, B, 902)
    check_against_blocking(AsyncCall(ml, strm, plan, good).enqueue().results(), blocking(ml, good, strm))
    plan.free()


# ------------------------------------------------------------------ 8. rejections
@gpu
def test_rejections_enqueue_nothing(ml, oracle):
    L = ml.load()
    D, B = 8, 3
    strm = _torch_strm()
    plans = {k: ml.BatchedProvePlan.create(D, B, k) for k in KINDS}
    c = AsyncCall(ml, strm, plans["codes"], BCase(ml, oracle, "codes", D, B, 950))
    r = AsyncCall(ml, strm, plans["rs"], BCase(ml, oracle, "rs", D, B, 951))
    q = AsyncCall(ml, strm, plans["pcs"], BCase(ml, oracle, "pcs", D, B, 952))
    s = strm.arg
    arr = lambda ptrs: (C.c_void_p * max(len(ptrs), 1))(*ptrs)   # noqa: E731
    cp, rp, qp = [x.ptr for x in c.data], [x.ptr for x in r.data], [x.ptr for x in q.data]

    def fa(ptrs, tr, proof, status, plan=plans["codes"]):
        return L.ml_batched_fri_prove_async(plan.h if plan else None, arr(ptrs) if ptrs is not None else None, _vp(tr), _vp(proof),
                                            _vp(status), s)

    def ra(ptrs, tr, proof, status, plan=plans["rs"]):
        return L.ml_batched_rs_fri_prove_async(plan.h, arr(ptrs), _vp(tr), _vp(proof), _vp(status), s)

    def pa(inp, out, ptrs, tr, proof, sc, status, plan=plans["pcs"]):
        return L.ml_batched_pcs_prove_async(plan.h, _vp(inp), _vp(out), arr(ptrs), _vp(tr), _vp(proof), _vp(sc), _vp(status), s)

    ok = (c.tr.ptr, c.proof.ptr, c.status.ptr)
    qok = (q.tr.ptr, q.proof.ptr, q.sc.ptr, q.status.ptr)
    cases = [
        ("null plan", fa(cp, *ok, plan=None)),
        ("null code array", fa(None, *ok)),
        ("null code in the array", fa([cp[0], None, cp[2]], *ok)),
        ("null transcript", fa(cp, None, c.proof.ptr, c.status.ptr)),
        ("null proof", ra(rp, r.tr.ptr, None, r.status.ptr)),
        ("null status", fa(cp, c.tr.ptr, c.proof.ptr, None)),
        ("null inputs", pa(None, q.out.ptr, qp, *qok)),
        ("null sumcheck", pa(q.inp.ptr, q.out.ptr, qp, q.tr.ptr, q.proof.ptr, None, q.status.ptr)),
        ("misaligned code", fa([cp[0], cp[1] + 8, cp[2]], *ok)),
        ("misaligned proof", fa(cp, c.tr.ptr, c.proof.ptr + 4, c.status.ptr)),
        ("misaligned outputs", pa(q.inp.ptr, q.out.ptr + 8, qp, *qok)),
        ("proof overlaps the last code", fa(cp, c.tr.ptr, cp[2] + 16 * 8, c.status.ptr)),
        ("transcript inside a coefficient buffer", ra(rp, rp[1] + 32, r.proof.ptr, r.status.ptr)),
        ("status inside the evals", pa(q.inp.ptr, q.out.ptr, qp, q.tr.ptr, q.proof.ptr, q.sc.ptr, qp[0] + 16)),
        ("sumcheck overlaps the claim", pa(q.inp.ptr, q.out.ptr, qp, q.tr.ptr, q.proof.ptr, q.out.ptr, q.status.ptr)),
        ("status inside the proof", fa(cp, c.tr.ptr, c.proof.ptr, c.proof.ptr + 64)),
        ("codes call on an rs plan", fa(rp, r.tr.ptr, r.proof.ptr, r.status.ptr, plan=plans["rs"])),
        ("rs call on a pcs plan", ra(qp, q.tr.ptr, q.proof.ptr, q.status.ptr, plan=plans["pcs"])),
        ("pcs call on a codes plan", pa(q.inp.ptr, q.out.ptr, qp, *qok, plan=plans["codes"])),
    ]
    for name, st in cases:
        assert st == ML_ERR_ARG, (name, st)
    for call in (c, r, q):
        call.unchanged()   # nothing was enqueued: outputs, canaries and the transcripts as they were
    for ld, nc in ((2, 1), (41, 1), (12, 0), (12, (1 << 20) + 1)):
        h = _vp()
        assert L.ml_batched_prove_plan_create(_sz(ld), _sz(nc), 0, C.byref(h)) == ML_ERR_SIZE and not h.value, (ld, nc)
    for p in plans.values():
        p.free()


@gpu
def test_plan_used_under_another_device(ml, oracle):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    L = ml.load()
    strm = _torch_strm()
    plan = ml.BatchedProvePlan.create(8, 2, "codes")
    c = AsyncCall(ml, strm, plan, BCase(ml, oracle, "codes", 8, 2, 990))
    ptrs = (C.c_void_p * 2)(*[x.ptr for x in c.data])
    ml.set_device(1)
    try:
        st = L.ml_batched_fri_prove_async(plan.h, ptrs, _vp(c.tr.ptr), _vp(c.proof.ptr), _vp(c.status.ptr), _vp(None))
    finally:
        ml.set_device(0)
    assert st == ML_ERR_ARG
    c.unchanged()
    plan.free()
