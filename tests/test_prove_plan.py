"""Stream-ordered provers (ml_prove_plan_*, ml_rs_fri_prove_async, ml_fri_prove_async, ml_pcs_prove_async) and the transcript
state they take in device memory (ml_transcript_state_bytes, ml_transcript_export, ml_transcript_import).

Each async call must leave in device memory exactly what its blocking twin returns: the FriProof bincode blob of
ml_fri_proof_serialize, the PCS sumcheck coefficients and the final transcript state.  The device proof writer and Writer in
csrc/prover.cu state the wire format twice; the parity tests pin the two against each other at every size where the chain's
plan changes (the smallest domain, the tail kernel's boundary at 2^12, the chunked folds, the headline 2^25), and against the CPU
oracle.  Capture into a CUDA graph in global mode is the check that an enqueue never synchronises, allocates or copies from
pageable host memory."""
import ctypes as C
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
PREFIX = b"stream-ordered prove: a transcript that has absorbed something"   # the state starts mid-block
ORACLE_MAX_LOG = 21
SIZES = [2, 3, 4, 12, 13, 14, 20, 25]
KINDS = ["rs", "fri", "pcs"]


def _p(a):
    return _vp(a.ctypes.data)


def _fe(x):
    return np.frombuffer(int(x).to_bytes(16, "little"), dtype=np.uint8).copy()


# ------------------------------------------------------------------ no GPU
def test_transcript_state_bytes(ml):
    assert ml.load().ml_transcript_state_bytes() == 104


def test_transcript_export_import_round_trip(ml):
    L = ml.load()
    for n in (0, 5, 63, 64, 100, 200):
        t = ml.Transcript()
        t.absorb(bytes(range(256))[:n])
        raw = (C.c_uint8 * 104)()
        ml.check(L.ml_transcript_export(t.h, raw))
        h = _vp()
        ml.check(L.ml_transcript_import(raw, C.byref(h)))
        u = ml.Transcript(h)
        assert bytes(raw) == t.export() == u.export()
        assert u.random() == t.random()
        assert u.next_challenge() == t.next_challenge()
        for step in (b"abc", b"\x00" * 70, bytes(range(17))):   # both copies continue identically
            t.absorb(step)
            u.absorb(step)
            assert u.random() == t.random() and u.next_challenge() == t.next_challenge()
        v = ml.Transcript.import_(t.export())
        assert v.export() == t.export()
    with pytest.raises(ml.SizeMismatch):
        ml.Transcript.import_(b"\x00" * 103)


def test_plan_create_without_a_device():
    """with no device visible, creating a plan fails with ML_ERR_CUDA (run in a child process that sees no GPU)"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import ctypes, multilinear_b200 as m; L = m.load(); h = ctypes.c_void_p(); "
            "print(L.ml_prove_plan_create(ctypes.c_size_t(12), 0, ctypes.byref(h)), h.value)")
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


_PLANS = {}


def plan_for(ml, log_domain, pcs):
    """plans are reused across tests (one per size and kind): creation builds tables and allocates once"""
    key = (log_domain, pcs)
    if key not in _PLANS:
        if log_domain >= 20:   # keep at most one large plan alive
            _PLANS.clear()
        _PLANS[key] = ml.ProvePlan.create(log_domain, pcs)
    return _PLANS[key]


class Case:
    """the inputs of one prove: coefficients (rs), a code (fri) or evaluations + claim (pcs), of a domain of 2^D"""

    def __init__(self, oracle, kind, D, seed, reference_inputs=False, prefix=PREFIX):
        N = 1 << D
        self.kind, self.D, self.N, self.nv, self.prefix = kind, D, N, D - 1, prefix
        rng = random.Random(seed)
        if kind == "rs":
            self.data = oracle.synthetic(seed, N // 2)
        elif kind == "fri":
            gp = oracle.pow2_generator_powers(D)
            self.data = oracle.reed_solomon(oracle.synthetic(seed, N // 2), fe_ints(gp[1:2])[0])
        else:
            if reference_inputs:   # the reference's own PCS test inputs: evals 7i + 3, inputs i
                self.data = fe_arr([7 * i + 3 for i in range(N // 2)])
                self.inputs = fe_arr(list(range(self.nv)))
            else:
                self.data = oracle.synthetic(seed, N // 2)
                self.inputs = fe_arr([rng.randrange(1 << 127) for _ in range(self.nv)])
            self.output = oracle.mle_evals_evaluate(self.data, self.inputs)


def start(t, case):
    """the transcript every prove of `case` starts from (ml_fri_verify starts from a fresh one: proofs it checks use prefix b"")"""
    t.absorb(case.prefix)
    return t


def blocking(ml, case, strm):
    """the blocking `_dev` twin on the same inputs: (blob, final transcript state, sumcheck coefficients as bytes or None)"""
    import torch
    L, t, h = ml.load(), start(ml.Transcript(), case), _vp()
    with torch.cuda.stream(strm.ts):
        d = torch.from_numpy(np.ascontiguousarray(case.data).reshape(-1).copy()).cuda()
    if case.kind == "rs":
        ml.check(L.ml_rs_fri_prove_dev(_vp(d.data_ptr()), _sz(case.N // 2), t.h, strm.arg, C.byref(h)))
        return ml.FriProof(h).serialize(), t.export(), None
    if case.kind == "fri":
        ml.check(L.ml_fri_prove_dev(_vp(d.data_ptr()), _sz(case.N), t.h, strm.arg, C.byref(h)))
        return ml.FriProof(h).serialize(), t.export(), None
    ml.check(L.ml_pcs_prove_dev(_p(case.inputs), _sz(case.nv), _p(_fe(case.output)), _vp(d.data_ptr()), _sz(case.N // 2), t.h, strm.arg,
                                C.byref(h)))
    proof = ml.PCSProof(h)
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
        self.data = Region(strm, case.data.size, IN_OFF, case.data, seed + 3)
        self.ins = [self.data]
        if case.kind == "pcs":
            self.inp = Region(strm, 16 * case.nv, IN_OFF, case.inputs, seed + 4)
            self.out = Region(strm, 16, IN_OFF, _fe(case.output), seed + 5)
            self.sc = Region(strm, 32 * case.nv, OUT_OFF, seed=seed + 6)
            self.ins += [self.inp, self.out]

    def enqueue(self):
        c, s = self.case, self.strm.handle
        if c.kind == "rs":
            self.plan.rs_fri_prove_async(self.data.ptr, self.tr.ptr, self.proof.ptr, self.status.ptr, s)
        elif c.kind == "fri":
            self.plan.fri_prove_async(self.data.ptr, self.tr.ptr, self.proof.ptr, self.status.ptr, s)
        else:
            self.plan.pcs_prove_async(self.inp.ptr, self.out.ptr, self.data.ptr, self.tr.ptr, self.proof.ptr, self.sc.ptr, self.status.ptr, s)
        return self

    def results(self):
        """(status, blob, final transcript state, sumcheck bytes or None); canaries intact, inputs unchanged"""
        for r in self.ins:
            r.result(unchanged=True)
        status = int(np.frombuffer(self.status.result().tobytes(), dtype=np.int32)[0])
        sc = self.sc.result().tobytes() if self.case.kind == "pcs" else None
        return status, self.proof.result().tobytes(), self.tr.result().tobytes(), sc


def oracle_result(oracle, case):
    """(blob, final random, sumcheck coefficients as ints or None) of the CPU oracle"""
    ot = start(oracle.transcript(), case)
    if case.kind == "pcs":
        op, st = oracle.pcs_prove(case.inputs, case.output, case.data, ot)
        assert st == 0
        return op.fri.blob, ot.random(), op.sumcheck
    gp = oracle.pow2_generator_powers(case.D)
    code = case.data if case.kind == "fri" else oracle.reed_solomon(case.data, fe_ints(gp[1:2])[0])
    op, st = oracle.fri_prove(code, gp, ot)
    assert st == 0
    return op.blob, ot.random(), None


def check_against_blocking(ml, case, got, want):
    status, blob, state, sc = got
    wblob, wstate, wsc = want
    assert status == ML_OK
    assert blob == wblob, "async blob differs from ml_fri_proof_serialize of the blocking proof"
    assert state == wstate, "final transcript differs from the blocking call's"
    assert sc == wsc


# ------------------------------------------------------------------ 1. parity across sizes
@gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("log_domain", SIZES)
def test_async_equals_blocking_and_oracle(ml, oracle, kind, log_domain):
    strm = _torch_strm()
    plan = plan_for(ml, log_domain, kind == "pcs")
    N = 1 << log_domain
    assert plan.proof_bytes > 0 and plan.device_bytes >= (96 if kind != "pcs" else 112) * N
    case = Case(oracle, kind, log_domain, 4000 + 10 * log_domain + KINDS.index(kind), prefix=b"")
    want = blocking(ml, case, strm)
    got = AsyncCall(ml, strm, plan, case).enqueue().results()
    check_against_blocking(ml, case, got, want)
    blob, state = got[1], got[2]
    assert len(blob) == plan.proof_bytes
    if kind != "pcs":   # a PCS proof's FRI part is checked by ml_pcs_verify in blocking()
        assert ml.FriProof.deserialize(blob).verify() == 0
    if log_domain <= ORACLE_MAX_LOG or (log_domain == 25 and kind == "rs"):   # 2^25 against the oracle once
        oblob, orandom, osc = oracle_result(oracle, case)
        assert blob == oblob, "async blob differs from the oracle's"
        assert ml.Transcript.import_(state).random() == orandom
        if osc is not None:
            assert fe_ints(np.frombuffer(got[3], dtype=np.uint8).reshape(-1, 16)) == osc


@gpu
def test_pcs_reference_inputs(ml, oracle):
    """PCSProof::prove on the reference's own inputs: n_vars 20, evals 7i + 3, inputs i"""
    strm = _torch_strm()
    case = Case(oracle, "pcs", 21, 0, reference_inputs=True)
    plan = plan_for(ml, 21, True)
    got = AsyncCall(ml, strm, plan, case).enqueue().results()
    check_against_blocking(ml, case, got, blocking(ml, case, strm))
    oblob, orandom, osc = oracle_result(oracle, case)
    assert got[1] == oblob and ml.Transcript.import_(got[2]).random() == orandom
    assert fe_ints(np.frombuffer(got[3], dtype=np.uint8).reshape(-1, 16)) == osc


# ------------------------------------------------------------------ 2. streams and buffers
@gpu
@pytest.mark.parametrize("log_domain", [4, 13])
def test_every_stream_kind(ml, oracle, stream_kind, log_domain):
    """NULL stream, an ml_stream_create stream and a torch stream; canaries around every buffer survive, inputs are unchanged"""
    for kind in KINDS:
        case = Case(oracle, kind, log_domain, 5000 + log_domain)
        plan = plan_for(ml, log_domain, True)   # a PCS plan proves FRI as well
        want = blocking(ml, case, stream_kind)
        check_against_blocking(ml, case, AsyncCall(ml, stream_kind, plan, case).enqueue().results(), want)


# ------------------------------------------------------------------ 3. graph capture
@gpu
def test_graph_capture_global_mode(ml, oracle):
    """one rs_fri_prove_async and one pcs_prove_async (two plans) captured into one graph in global mode: any synchronisation,
    cudaMalloc or pageable copy inside the calls fails the capture.  Three replays with rewritten inputs and reset transcripts."""
    import torch
    D = 13
    p_rs, p_pcs = ml.ProvePlan.create(D, False), ml.ProvePlan.create(D, True)
    side = torch.cuda.Stream()
    strm = Strm("torch", side, side.cuda_stream)
    rs0, pcs0 = Case(oracle, "rs", D, 6000), Case(oracle, "pcs", D, 6001)
    a, b = AsyncCall(ml, strm, p_rs, rs0), AsyncCall(ml, strm, p_pcs, pcs0)
    with torch.cuda.stream(side):   # eager warm-up: every kernel of both calls is loaded before capture
        a.enqueue()
        b.enqueue()
    side.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side, capture_error_mode="global"):
        p_rs.rs_fri_prove_async(a.data.ptr, a.tr.ptr, a.proof.ptr, a.status.ptr, side.cuda_stream)
        p_pcs.pcs_prove_async(b.inp.ptr, b.out.ptr, b.data.ptr, b.tr.ptr, b.proof.ptr, b.sc.ptr, b.status.ptr, side.cuda_stream)
    state = torch.from_numpy(np.frombuffer(start(ml.Transcript(), rs0).export(), dtype=np.uint8).copy()).cuda()
    torch.cuda.synchronize()

    def write(region, arr):
        t = torch.from_numpy(np.ascontiguousarray(arr).reshape(-1).view(np.uint8).copy()).cuda()
        region.t[region.off:region.off + t.numel()].copy_(t)
        region.image[region.off:region.off + t.numel()] = t.cpu().numpy()

    for rep in range(3):
        rs, pcs = Case(oracle, "rs", D, 6100 + rep), Case(oracle, "pcs", D, 6200 + rep)
        with torch.cuda.stream(side):
            write(a.data, rs.data)
            write(b.data, pcs.data)
            write(b.inp, pcs.inputs)
            write(b.out, _fe(pcs.output))
            a.tr.t[a.tr.off:a.tr.off + 104].copy_(state)
            b.tr.t[b.tr.off:b.tr.off + 104].copy_(state)
            g.replay()
        side.synchronize()
        a.case, b.case = rs, pcs
        check_against_blocking(ml, rs, a.results(), blocking(ml, rs, strm))
        check_against_blocking(ml, pcs, b.results(), blocking(ml, pcs, strm))
    del g
    p_rs.free()
    p_pcs.free()


# ------------------------------------------------------------------ 4. one thread, many proofs in flight
@gpu
def test_one_thread_six_plans_in_flight(ml, oracle):
    import torch
    D = 14
    plans = [ml.ProvePlan.create(D, False) for _ in range(6)]
    calls = []
    for i, p in enumerate(plans):
        strm = _torch_strm()
        calls.append(AsyncCall(ml, strm, p, Case(oracle, "rs" if i % 2 == 0 else "fri", D, 7000 + i)))
    for c in calls:   # inputs are written on each stream; make them complete before the enqueue burst
        c.strm.ts.synchronize()
    for c in calls:
        c.enqueue()
    torch.cuda.synchronize()
    for c in calls:
        check_against_blocking(ml, c.case, c.results(), blocking(ml, c.case, c.strm))
    for p in plans:
        p.free()


# ------------------------------------------------------------------ 5. not an RS code
@gpu
def test_not_an_rs_code_then_a_valid_one(ml, oracle):
    import torch
    D = 8
    strm = _torch_strm()
    plan = ml.ProvePlan.create(D, False)
    bad = Case(oracle, "fri", D, 8000)
    bad.data = oracle.synthetic(8001, 1 << D)   # random data: its last fold is not constant
    status = AsyncCall(ml, strm, plan, bad).enqueue().results()[0]
    torch.cuda.synchronize()   # raises on a CUDA error
    assert status == ML_ERR_NOT_RS_CODE
    good = Case(oracle, "fri", D, 8002)
    check_against_blocking(ml, good, AsyncCall(ml, strm, plan, good).enqueue().results(), blocking(ml, good, strm))
    plan.free()


# ------------------------------------------------------------------ 6. rejections
@gpu
def test_rejections_enqueue_nothing(ml, oracle):
    L = ml.load()
    D = 8
    strm = _torch_strm()
    fri_plan, pcs_plan = ml.ProvePlan.create(D, False), ml.ProvePlan.create(D, True)
    code, pcs = Case(oracle, "fri", D, 9000), Case(oracle, "pcs", D, 9001)
    c = AsyncCall(ml, strm, fri_plan, code)
    q = AsyncCall(ml, strm, pcs_plan, pcs)
    s = strm.arg
    fa = lambda *a: L.ml_fri_prove_async(fri_plan.h, *[_vp(x) for x in a], s)   # noqa: E731
    ra = lambda *a: L.ml_rs_fri_prove_async(fri_plan.h, *[_vp(x) for x in a], s)   # noqa: E731
    cases = [
        ("null code", fa(None, c.tr.ptr, c.proof.ptr, c.status.ptr)),
        ("null transcript", fa(c.data.ptr, None, c.proof.ptr, c.status.ptr)),
        ("null proof", ra(c.data.ptr, c.tr.ptr, None, c.status.ptr)),
        ("null status", fa(c.data.ptr, c.tr.ptr, c.proof.ptr, None)),
        ("null plan", L.ml_fri_prove_async(None, _vp(c.data.ptr), _vp(c.tr.ptr), _vp(c.proof.ptr), _vp(c.status.ptr), s)),
        ("misaligned code", fa(c.data.ptr + 8, c.tr.ptr, c.proof.ptr, c.status.ptr)),
        ("misaligned proof", fa(c.data.ptr, c.tr.ptr, c.proof.ptr + 4, c.status.ptr)),
        ("proof overlaps the code", fa(c.data.ptr, c.tr.ptr, c.data.ptr + 16 * 8, c.status.ptr)),
        ("transcript inside the coefficients", ra(c.data.ptr, c.data.ptr + 32, c.proof.ptr, c.status.ptr)),
        ("pcs on an fri plan", L.ml_pcs_prove_async(fri_plan.h, _vp(q.inp.ptr), _vp(q.out.ptr), _vp(q.data.ptr), _vp(c.tr.ptr),
                                                    _vp(c.proof.ptr), _vp(q.sc.ptr), _vp(c.status.ptr), s)),
        ("sumcheck overlaps the evals", L.ml_pcs_prove_async(pcs_plan.h, _vp(q.inp.ptr), _vp(q.out.ptr), _vp(q.data.ptr), _vp(q.tr.ptr),
                                                             _vp(q.proof.ptr), _vp(q.data.ptr + 16), _vp(q.status.ptr), s)),
    ]
    for name, st in cases:
        assert st == ML_ERR_ARG, (name, st)
    for r in (c.tr, c.proof, c.status, c.data, q.tr, q.proof, q.status, q.sc, q.data, q.inp, q.out):
        r.result(unchanged=True)   # nothing was enqueued: outputs, canaries and the transcript as they were
    for bad in (0, 1, 41, 64):
        h = _vp()
        assert L.ml_prove_plan_create(_sz(bad), 0, C.byref(h)) == ML_ERR_SIZE and not h.value
    fri_plan.free()
    pcs_plan.free()


@gpu
def test_plan_used_under_another_device(ml, oracle):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    L = ml.load()
    strm = _torch_strm()
    plan = ml.ProvePlan.create(8, False)
    c = AsyncCall(ml, strm, plan, Case(oracle, "fri", 8, 9100))
    ml.set_device(1)
    try:
        st = L.ml_fri_prove_async(plan.h, _vp(c.data.ptr), _vp(c.tr.ptr), _vp(c.proof.ptr), _vp(c.status.ptr), _vp(None))
    finally:
        ml.set_device(0)
    assert st == ML_ERR_ARG
    for r in (c.tr, c.proof, c.status):
        r.result(unchanged=True)
    plan.free()
