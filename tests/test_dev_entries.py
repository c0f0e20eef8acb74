"""The `_dev` entry points (device pointers and a stream, include/multilinear_b200.h) against the CPU oracle, the way a Rust
caller with its data already in HBM uses them:

  - on every kind of stream that reaches the library: NULL (the legacy stream), a stream from ml_stream_create (its own pool)
    and a caller-owned torch stream (the default pool), with the input written on that stream;
  - with every element buffer at a 16-byte-aligned offset inside a larger allocation, between canary bytes that must survive
    the call; inputs the header calls copied or only read must be unchanged;
  - with handles made on a caller stream used afterwards through the host methods, which run on the library stream;
  - with the status of every rejected input equal to the host-pointer twin's;
  - with in == out for every entry that has separate element input and output buffers, pinning the aliasing rule the
    header states.

It also holds the small host-side controls (thread stream, host registration, pinned memory, pools, accessors) next to a
prove compared with the oracle, and the coverage guard: every symbol the header declares must be named by a test or be
called by an api.py function a test uses."""
import ast
import ctypes as C
import os
import random
import re

import numpy as np
import pytest

from oracle import pyref as P
from oracle.binding import fe_arr, fe_ints
from test_abi import ROOT, declared_symbols

M = P.M
gpu = pytest.mark.gpu
_sz, _vp = C.c_size_t, C.c_void_p
IN_OFF, OUT_OFF, TAIL = 48, 16, 64   # byte offsets of inputs / outputs inside their allocations; canary bytes after them
ML_ERR_NOT_POW2, ML_ERR_SIZE, ML_ERR_NOT_RS_CODE, ML_ERR_GENERATOR, ML_ERR_ARG = 1, 2, 4, 5, 8


def _p(a):
    return _vp(a.ctypes.data)


def _fe(x):
    return np.frombuffer(int(x).to_bytes(16, "little"), dtype=np.uint8).copy()


class Strm:
    """one stream of the three kinds: `arg` is what the entry points take, `ts` the torch view used to write and read"""

    def __init__(self, kind, ts, handle):
        self.kind, self.ts, self.handle, self.kept = kind, ts, handle, []

    @property
    def arg(self):
        return _vp(self.handle)

    def keep(self, obj, free_name):
        """a handle made on this stream: freed before the stream is destroyed, whatever the test's outcome"""
        self.kept.append((obj, free_name))
        return obj


@pytest.fixture(params=["null", "ml_stream", "torch"])
def strm(request, ml):
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
    for obj, free_name in s.kept:
        if obj.h is not None and obj.h.value and getattr(obj, "owned", True):
            getattr(L, free_name)(obj.h)
        obj.h, obj.owned = None, False
    if created:
        ml.check(L.ml_stream_synchronize(_vp(created)))
        ml.check(L.ml_stream_destroy(_vp(created)))


class Region:
    """nbytes at byte offset `off` of a device allocation whose every other byte is a canary; `data` (if given) fills the start
    of the region, the rest of it holds canary bytes too.  Written and read on the test's stream."""

    def __init__(self, strm, nbytes, off, data=None, seed=0):
        import torch
        rng = np.random.default_rng(seed * 1000003 + nbytes + off)
        self.image = rng.integers(0, 256, off + nbytes + TAIL, dtype=np.uint8)
        if data is not None:
            d = np.ascontiguousarray(data).reshape(-1).view(np.uint8)
            self.image[off:off + d.size] = d
        self.strm, self.off, self.nbytes = strm, off, nbytes
        with torch.cuda.stream(strm.ts):
            self.t = torch.from_numpy(self.image.copy()).cuda()

    @property
    def ptr(self):
        return self.t.data_ptr() + self.off

    def result(self, unchanged=False):
        """the region after the call, as (n, 16) elements when it holds whole elements; the canaries around it must be intact,
        and with `unchanged` the region itself too"""
        import torch
        with torch.cuda.stream(self.strm.ts):
            got = self.t.cpu().numpy()
        o, n = self.off, self.nbytes
        assert np.array_equal(got[:o], self.image[:o]), "canary before the buffer overwritten"
        assert np.array_equal(got[o + n:], self.image[o + n:]), "canary after the buffer overwritten"
        body = got[o:o + n]
        if unchanged:
            assert np.array_equal(body, self.image[o:o + n]), "an input the call only reads was changed"
        return body.reshape(-1, 16) if n % 16 == 0 else body


_CACHE = {}


def cached(key, fn):
    """oracle results shared by the three stream cases of one size"""
    if key not in _CACHE:
        _CACHE[key] = fn()
    return _CACHE[key]


def rs_code(oracle, c, seed):
    """an RS code of 2^c elements and the domain generator's powers"""
    gp = oracle.pow2_generator_powers(c)
    return oracle.reed_solomon(oracle.synthetic(seed, 1 << (c - 1)), fe_ints(gp[1:2])[0]), gp


def pairs_of(code):
    """ReedSolomonPairs (code[i], code[i + n/2]) as (n/2, 32) bytes: the leaves of commit_rs_code (src/fri/mod.rs:45-55)"""
    h = code.shape[0] // 2
    return np.ascontiguousarray(np.concatenate([code[:h], code[h:]], axis=1))


# ------------------------------------------------------------------ NTT / INTT / RS, generator powers
@gpu
@pytest.mark.parametrize("log_n", [0, 1, 12, 13, 18])
def test_ntt_intt_rs_dev(ml, oracle, strm, log_n):
    L, n = ml.load(), 1 << log_n
    x = oracle.synthetic(300 + log_n, n)
    for inverse in (False, True):
        g, g2 = ml.pow_2_generator(log_n), ml.pow_2_generator(log_n + 1)
        if inverse:
            g, g2 = P.inv(g), P.inv(g2)
        cases = [("ml_ntt_dev", g, n, oracle.ntt(x, g) if n > 1 else x),
                 ("ml_intt_dev", g, n, oracle.intt(x, g) if n > 1 else x),
                 ("ml_reed_solomon_dev", g2, 2 * n, oracle.reed_solomon(x, g2))]
        for name, gen, n_out, want in cases:
            a, b, gb = Region(strm, 16 * n, IN_OFF, x), Region(strm, 16 * n_out, OUT_OFF), _fe(gen)
            ml.check(getattr(L, name)(_vp(a.ptr), _sz(n), _p(gb), _vp(b.ptr), strm.arg))
            assert np.array_equal(b.result(), want), (name, inverse)
            a.result(unchanged=True)


@gpu
@pytest.mark.parametrize("log_n", [0, 1, 12, 13, 20])
def test_pow2_generator_powers_dev(ml, oracle, strm, log_n):
    b = Region(strm, 16 << log_n, OUT_OFF)
    ml.check(ml.load().ml_pow2_generator_powers_dev(C.c_uint64(log_n), _vp(b.ptr), strm.arg))
    assert np.array_equal(b.result(), cached(("powers", log_n), lambda: oracle.pow2_generator_powers(log_n)))


# ------------------------------------------------------------------ Moebius transforms, PCS encode, evaluation
@gpu
@pytest.mark.parametrize("log_n", [0, 1, 12, 13, 20, 21])
def test_mle_transforms_and_pcs_encode_dev(ml, oracle, strm, log_n):
    L, n = ml.load(), 1 << log_n

    def want():
        x = oracle.synthetic(400 + log_n, n)
        c = oracle.to_coefficient(x)
        return x, c, oracle.to_evaluation(x), oracle.reed_solomon(oracle.bit_reverse(c), oracle.pow2_generator(log_n + 1))
    x, coeffs, evals, code = cached(("mle", log_n), want)
    for name, n_out, w in (("ml_mle_to_coefficient_dev", n, coeffs), ("ml_mle_to_evaluation_dev", n, evals), ("ml_pcs_encode_dev", 2 * n, code)):
        a, b = Region(strm, 16 * n, IN_OFF, x), Region(strm, 16 * n_out, OUT_OFF)
        ml.check(getattr(L, name)(_vp(a.ptr), _sz(n), _vp(b.ptr), strm.arg))
        assert np.array_equal(b.result(), w), name
        a.result(unchanged=True)


@gpu
@pytest.mark.parametrize("length", [1, 2, 1 << 11, 1 << 12, 1 << 13, 6])
def test_mle_evals_evaluate_dev(ml, oracle, strm, length):
    nv = (length - 1).bit_length()   # the evaluations are padded to the next power of two (polynomials.rs:165-187)
    rng = random.Random(length)
    ev = oracle.synthetic(500 + length, length)
    xs = [rng.randrange(M) for _ in range(nv)]
    args = fe_arr(xs) if nv else np.zeros((1, 16), dtype=np.uint8)
    if length == 6:
        want = P.mle_evals_evaluate(fe_ints(ev), xs)
    else:
        want = oracle.mle_evals_evaluate(ev, args) if nv else fe_ints(ev)[0]
    a, out = Region(strm, 16 * length, IN_OFF, ev), np.zeros(16, dtype=np.uint8)
    ml.check(ml.load().ml_mle_evals_evaluate_dev(_vp(a.ptr), _sz(length), _p(args), _sz(nv), _p(out), strm.arg))
    assert fe_ints(out)[0] == want
    a.result(unchanged=True)


# ------------------------------------------------------------------ FRI
def _open_all(f, of, idx, n_leaves):
    cur, cur_n = idx, n_leaves
    for j, (value, path) in enumerate(f.open_query_at(idx)):
        assert (value, path) == of.tree(j).open(cur), j
        cur_n //= 2
        cur = cur % cur_n if cur_n else 0


@gpu
@pytest.mark.parametrize("log_code", [2, 12, 13, 14])
def test_fri_init_dev_then_host_fold_steps(ml, oracle, strm, log_code):
    """ml_fri_init_dev on the test's stream copies the code; fold_step, tree_data and open_query_at then run on the library
    stream: every root, tree, opening, the last element and the transcript equal the oracle's (src/fri/mod.rs:58-174)"""
    L, N, log_n = ml.load(), 1 << log_code, log_code - 1
    code, gp = rs_code(oracle, log_code, 600 + log_code)
    a = Region(strm, 16 * N, IN_OFF, code)
    t, ot = ml.Transcript(), oracle.transcript()
    h = _vp()
    ml.check(L.ml_fri_init_dev(_vp(a.ptr), _sz(N), t.h, strm.arg, C.byref(h)))
    f = strm.keep(ml.FriProverData(h), "ml_fri_free")
    a.result(unchanged=True)
    of = oracle.fri_init(code, ot)
    for k in range(log_n):
        r = t.next_challenge()
        assert r == ot.next_challenge()
        f.fold_step(gp, k, r, t)
        assert of.fold_step(gp, k, r, ot) == 0
    assert f.num_trees() == of.num_trees() == log_n
    assert f.fold_roots() == of.roots() and f.last_element == of.last_element() is not None
    for j in range(f.num_trees()):
        assert np.array_equal(f.tree_data(j), of.tree_data(j)), j
        for x, y in zip(f.tree(j).layers, of.tree(j).layers()):
            assert np.array_equal(x, y), j
    assert t.random() == ot.random()
    _open_all(f, of, (12345 * log_code) % (N // 2), N // 2)


FOLD_SIZES = [2, 12, 13, 14, 21]


@gpu
@pytest.mark.parametrize("log_code", FOLD_SIZES)
def test_fri_fold_dev_and_rs_fri_fold_dev(ml, oracle, strm, log_code):
    """the commit phase from a device code (ml_fri_fold_dev) and from device coefficients (ml_rs_fri_fold_dev): roots, last
    element and transcript equal the oracle's FriProverData::fold (src/fri/mod.rs:136-145); the handles answer tree_data and
    open_query_at on the library stream like the oracle's trees"""
    L, N = ml.load(), 1 << log_code

    def want():
        code, gp = rs_code(oracle, log_code, 700 + log_code)
        ot = oracle.transcript()
        of, st = oracle.fri_fold(gp, code, ot)
        assert st == 0
        return code, of, ot.random()
    code, of, final = cached(("fold", log_code), want)
    coeffs = cached(("coeffs", log_code), lambda: oracle.synthetic(700 + log_code, N // 2))
    idx = (777 * log_code) % (N // 2)
    for name, data, n in (("ml_fri_fold_dev", code, N), ("ml_rs_fri_fold_dev", coeffs, N // 2)):
        a, t, h = Region(strm, 16 * n, IN_OFF, data), ml.Transcript(), _vp()
        ml.check(getattr(L, name)(_vp(a.ptr), _sz(n), t.h, strm.arg, C.byref(h)))
        f = strm.keep(ml.FriProverData(h), "ml_fri_free")
        a.result(unchanged=True)
        assert f.fold_roots() == of.roots() and len(f.fold_roots()) == log_code - 1, name
        assert f.last_element == of.last_element() is not None and t.random() == final, name
        last = f.num_trees() - 1
        assert np.array_equal(f.tree_data(last), of.tree_data(last)), name
        _open_all(f, of, idx, N // 2)


@gpu
@pytest.mark.parametrize("log_code", FOLD_SIZES)
def test_fri_prove_dev_and_rs_fri_prove_dev(ml, oracle, strm, log_code):
    """FriProof::prove from a device code and reed_solomon + prove from device coefficients: the proof bytes and the final
    transcript equal the oracle's (src/fri/mod.rs:261-285), and the proof verifies"""
    L, N = ml.load(), 1 << log_code

    def want():
        code, gp = rs_code(oracle, log_code, 800 + log_code)
        ot = oracle.transcript()
        op, st = oracle.fri_prove(code, gp, ot)
        assert st == 0
        return code, op.blob, ot.random()
    code, blob, final = cached(("prove", log_code), want)
    coeffs = cached(("pcoeffs", log_code), lambda: oracle.synthetic(800 + log_code, N // 2))
    for name, data, n in (("ml_fri_prove_dev", code, N), ("ml_rs_fri_prove_dev", coeffs, N // 2)):
        a, t, h = Region(strm, 16 * n, IN_OFF, data), ml.Transcript(), _vp()
        ml.check(getattr(L, name)(_vp(a.ptr), _sz(n), t.h, strm.arg, C.byref(h)))
        proof = ml.FriProof(h)
        a.result(unchanged=True)
        assert proof.serialize() == blob and t.random() == final, name
        assert proof.verify() == 0, name


@gpu
def test_dev_errors_match_host_twins(ml, oracle, strm):
    """a length that is not a power of two, a code of length 2 (last_element is None), a code that is not an RS code and a
    wrong generator: every `_dev` entry returns what its host-pointer twin returns"""
    L = ml.load()

    def dev(name, data, n, *mid):
        a, h = Region(strm, 16 * max(data.shape[0], 1), IN_OFF, data), _vp()
        if name.startswith(("ml_fri", "ml_rs_fri")):
            st = getattr(L, name)(_vp(a.ptr), _sz(n), ml.Transcript().h, strm.arg, C.byref(h))
            free = "ml_fri_proof_free" if "prove" in name else "ml_fri_free"
            if h.value:
                getattr(L, free)(h)
        else:
            out = Region(strm, 32 * max(n, 1), OUT_OFF)
            st = getattr(L, name)(_vp(a.ptr), _sz(n), *mid, _vp(out.ptr), strm.arg)
            out.result()
        a.result(unchanged=True)
        return st

    def host(name, data, n, *mid):
        h = _vp()
        if name == "ml_fri_prove":
            st = L.ml_fri_prove(_p(data), _sz(n), None, _sz(0), ml.Transcript().h, C.byref(h))
        elif name == "ml_fri_fold":
            st = L.ml_fri_fold(None, _sz(0), _p(data), _sz(n), ml.Transcript().h, C.byref(h))
        elif name in ("ml_fri_init", "ml_rs_fri_prove"):
            st = getattr(L, name)(_p(data), _sz(n), ml.Transcript().h, C.byref(h))
        else:
            out = np.empty((2 * max(n, 1), 16), dtype=np.uint8)
            return getattr(L, name)(_p(data), _sz(n), *mid, _p(out))
        if h.value:
            (L.ml_fri_proof_free if "prove" in name else L.ml_fri_free)(h)
        return st

    x12, x24 = oracle.synthetic(1, 12), oracle.synthetic(2, 24)
    gb, bad_gen = _fe(ml.pow_2_generator(3)), _fe(12345)
    code2, _ = rs_code(oracle, 1, 3)
    not_rs = oracle.synthetic(4, 1 << 8)   # random data is not a codeword
    x8 = oracle.synthetic(5, 8)
    cases = [  # (dev entry, host twin, data, n, extra arguments, expected status)
        ("ml_ntt_dev", "ml_ntt", x12, 12, (_p(gb),), ML_ERR_NOT_POW2),
        ("ml_intt_dev", "ml_intt", x12, 12, (_p(gb),), ML_ERR_NOT_POW2),
        ("ml_reed_solomon_dev", "ml_reed_solomon", x12, 12, (_p(gb),), ML_ERR_NOT_POW2),
        ("ml_fri_init_dev", "ml_fri_init", x24, 24, (), ML_ERR_NOT_POW2),
        ("ml_fri_fold_dev", "ml_fri_fold", x24, 24, (), ML_ERR_NOT_POW2),
        ("ml_fri_prove_dev", "ml_fri_prove", x24, 24, (), ML_ERR_NOT_POW2),
        ("ml_rs_fri_prove_dev", "ml_rs_fri_prove", x12, 12, (), ML_ERR_NOT_POW2),
        ("ml_rs_fri_fold_dev", "ml_rs_fri_prove", x12, 12, (), ML_ERR_NOT_POW2),
        ("ml_fri_fold_dev", "ml_fri_fold", code2, 2, (), None),
        ("ml_fri_prove_dev", "ml_fri_prove", code2, 2, (), None),
        ("ml_rs_fri_fold_dev", "ml_rs_fri_prove", code2[:1], 1, (), None),
        ("ml_fri_prove_dev", "ml_fri_prove", not_rs, 1 << 8, (), ML_ERR_NOT_RS_CODE),
        ("ml_fri_fold_dev", "ml_fri_fold", not_rs, 1 << 8, (), ML_ERR_NOT_RS_CODE),
        ("ml_ntt_dev", "ml_ntt", x8, 8, (_p(bad_gen),), ML_ERR_GENERATOR),
        ("ml_intt_dev", "ml_intt", x8, 8, (_p(bad_gen),), ML_ERR_GENERATOR),
        ("ml_reed_solomon_dev", "ml_reed_solomon", x8, 8, (_p(bad_gen),), ML_ERR_GENERATOR),
    ]
    for d, hname, data, n, mid, want in cases:
        sd, sh = dev(d, data, n, *mid), host(hname, data, n, *mid)
        assert sd == sh != 0, (d, n, sd, sh)
        assert want is None or sd == want, (d, n, sd)
    # a code of length 2 has no fold round: init gives a handle without a last element, as the host twin does
    a, t, h = Region(strm, 32, IN_OFF, code2), ml.Transcript(), _vp()
    ml.check(L.ml_fri_init_dev(_vp(a.ptr), _sz(2), t.h, strm.arg, C.byref(h)))
    f = strm.keep(ml.FriProverData(h), "ml_fri_free")
    fh = ml.FriProverData.init(code2, ml.Transcript())
    assert f.last_element is None and fh.last_element is None and f.fold_roots() == fh.fold_roots()


# ------------------------------------------------------------------ sumcheck tables, PCS, width-w tables
@gpu
@pytest.mark.parametrize("nv", [1, 12, 13, 20])
def test_sumcheck_build_tables_for_pcs_dev(ml, oracle, strm, nv):
    """tables built from device evaluations on the test's stream, then partial_sum / fold / compute_sumcheck_polynomials on
    the library stream: tables, partial sums and every round equal the oracle's (sumcheck.rs:128-247)"""
    L, n = ml.load(), 1 << nv
    rng = random.Random(nv)
    ev = oracle.synthetic(900 + nv, n)
    inp = fe_arr([rng.randrange(M) for _ in range(nv)])

    def build():
        a, h = Region(strm, 16 * n, IN_OFF, ev), _vp()
        ml.check(L.ml_sumcheck_build_tables_for_pcs_dev(_p(inp), _sz(nv), _vp(a.ptr), _sz(n), strm.arg, C.byref(h)))
        a.result(unchanged=True)
        return strm.keep(ml.SumcheckTables(h), "ml_sumcheck_free")
    s, os_ = build(), oracle.sumcheck_build(inp, ev)
    for x, y in zip(s.tables(), os_.tables()):
        assert np.array_equal(x, y)
    for r in (1, 2, rng.randrange(M)):
        assert s.partial_sum(r) == os_.partial_sum(r)
    rr = rng.randrange(M)
    s.fold(rr)
    os_.fold(rr)
    assert s.height == os_.height() == n // 2
    for x, y in zip(s.tables(), os_.tables()):
        assert np.array_equal(x, y)
    claim = oracle.mle_evals_evaluate(ev, inp)
    s2, os2 = build(), oracle.sumcheck_build(inp, ev)
    t, ot = ml.Transcript(), oracle.transcript()
    assert s2.compute_sumcheck_polynomials(1, t, claim) == os2.compute_sumcheck_polynomials(1, ot, claim)
    assert t.random() == ot.random()


@gpu
@pytest.mark.parametrize("nv", [5, 13])
def test_pcs_prove_dev(ml, oracle, strm, nv):
    L, n = ml.load(), 1 << nv
    rng = random.Random(nv)
    ev = oracle.synthetic(1000 + nv, n)
    inp = fe_arr([rng.randrange(M) for _ in range(nv)])
    out = oracle.mle_evals_evaluate(ev, inp)
    a, t, ot, h, ob = Region(strm, 16 * n, IN_OFF, ev), ml.Transcript(), oracle.transcript(), _vp(), _fe(out)
    ml.check(L.ml_pcs_prove_dev(_p(inp), _sz(nv), _p(ob), _vp(a.ptr), _sz(n), t.h, strm.arg, C.byref(h)))
    proof = ml.PCSProof(h)
    a.result(unchanged=True)
    oproof, st = oracle.pcs_prove(inp, out, ev, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck and t.random() == ot.random()
    assert proof.verify(ml.Transcript()) == 0


@gpu
@pytest.mark.parametrize("nv", [5, 13])
def test_batched_pcs_prove_dev(ml, oracle, strm, nv):
    L, n, B = ml.load(), 1 << nv, 3
    rng = random.Random(nv)
    polys = [oracle.synthetic(1100 + 10 * nv + j, n) for j in range(B)]
    inp = fe_arr([rng.randrange(M) for _ in range(nv)])
    outs = fe_arr([oracle.mle_evals_evaluate(p, inp) for p in polys])
    regions = [Region(strm, 16 * n, IN_OFF + 16 * j, p, seed=j) for j, p in enumerate(polys)]
    ptrs = (C.c_void_p * B)(*[r.ptr for r in regions])
    t, ot, h = ml.Transcript(), oracle.transcript(), _vp()
    ml.check(L.ml_batched_pcs_prove_dev(_p(inp), _sz(nv), _p(outs), _sz(B), ptrs, _sz(n), t.h, strm.arg, C.byref(h)))
    proof = ml.PCSProof(h, batched=True)
    for r in regions:
        r.result(unchanged=True)
    oproof, st = oracle.batched_pcs_prove(inp, outs, polys, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck and t.random() == ot.random()
    assert proof.verify(ml.Transcript()) == 0


@gpu
@pytest.mark.parametrize("nv", [5, 13])
def test_wsumcheck_build_dev(ml, oracle, strm, nv):
    """width-w tables from a device trace; the handle's methods run on the stream it was built on"""
    L, w, n = ml.load(), 3, 1 << nv
    matrix, row_point = oracle.synthetic(1200 + nv, w << nv), oracle.synthetic(1300 + nv, nv)
    terms = [(7, [0, 1, 2]), (M - 3, [2, 2]), (11, []), (5, [1])]
    a, h = Region(strm, 16 * w * n, IN_OFF, matrix), _vp()
    ml.check(L.ml_wsumcheck_build_dev(_p(row_point), _sz(nv), _vp(a.ptr), _sz(w), _sz(n), strm.arg, C.byref(h)))
    g = strm.keep(ml.WideSumcheckTables(h, w), "ml_wsumcheck_free")
    a.result(unchanged=True)
    assert L.ml_wsumcheck_width(g.h) == w and g.height == n
    o = oracle.wsumcheck_build(row_point, matrix, w)
    g.set_composition(terms)
    o.set_composition(terms)
    for x, y in zip(g.tables(), o.tables()):
        assert np.array_equal(x, y)
    for r in (5, M - 2):
        assert g.partial_sum(r) == o.partial_sum(r)
    t, ot = ml.Transcript(), oracle.transcript()
    assert g.compute_sumcheck_polynomials(3, t, 99) == o.compute_sumcheck_polynomials(3, ot, 99)
    assert t.random() == ot.random()


# ------------------------------------------------------------------ Merkle building blocks
@gpu
@pytest.mark.parametrize("leaves", [1, 8, 4096, 8192])
def test_merkle_commit_rs_code_dev(ml, oracle, strm, leaves):
    """the tree keeps the caller's code: layers, root and openings (which read the code again) equal the oracle's"""
    L = ml.load()
    code = oracle.synthetic(1400 + leaves, 2 * leaves)
    om = oracle.merkle_commit(pairs_of(code))
    a, h = Region(strm, 32 * leaves, IN_OFF, code), _vp()
    ml.check(L.ml_merkle_commit_rs_code_dev(_vp(a.ptr), _sz(2 * leaves), strm.arg, C.byref(h)))
    m = strm.keep(ml.Merkle(h, 32), "ml_merkle_free")
    assert m.root() == om.root()
    for x, y in zip(m.layers, om.layers()):
        assert np.array_equal(x, y)
    for idx in sorted({0, leaves - 1, leaves // 3}):
        assert m.open(idx) == om.open(idx), idx
    a.result(unchanged=True)


@gpu
@pytest.mark.parametrize("leaves", [1, 8, 4096, 8192])
def test_batched_leaf_subtree_and_pack_pairs_dev(ml, oracle, strm, leaves):
    """one rank's share of Merkle::batch_commit (merkle_tree/mod.rs:110-131): subtree roots to the host and to HBM, the top
    levels over the roots of two leaf ranges, and the two pair layouts of the exchange"""
    L, B = ml.load(), 3
    codes = [oracle.synthetic(1500 + 7 * leaves + j, 2 * leaves) for j in range(B)]
    pairs = [pairs_of(c) for c in codes]
    want = oracle.merkle_batch_commit(pairs).root()
    regions = [Region(strm, 32 * leaves, IN_OFF + 16 * j, p, seed=j) for j, p in enumerate(pairs)]
    ptrs = (C.c_void_p * B)(*[r.ptr for r in regions])
    root = np.zeros(32, dtype=np.uint8)
    ml.check(L.ml_batched_leaf_subtree_dev(ptrs, _sz(B), _sz(leaves), strm.arg, _p(root)))
    assert root.tobytes() == want
    rd = Region(strm, 32, OUT_OFF)
    ml.check(L.ml_batched_leaf_subtree_root_dev(ptrs, _sz(B), _sz(leaves), _vp(rd.ptr), strm.arg))
    assert rd.result().tobytes() == want
    if leaves > 1:   # subtree roots of the two halves (pointers into the middle of the pair buffers), then the top level
        half = leaves // 2
        roots = np.zeros((2, 32), dtype=np.uint8)
        for k in range(2):
            sub = (C.c_void_p * B)(*[r.ptr + 32 * half * k for r in regions])
            ml.check(L.ml_batched_leaf_subtree_dev(sub, _sz(B), _sz(half), strm.arg, _p(roots[k])))
        top = np.zeros(32, dtype=np.uint8)
        ml.check(L.ml_merkle_top_from_roots(_p(roots), _sz(2), _p(top)))
        assert top.tobytes() == want
    for r in regions:
        r.result(unchanged=True)
    # pack: pair i of local polynomial 1 (of 2) goes to [dest][1][i % rows], dest = i / rows
    n_ranks = 2 if leaves > 1 else 1
    rows = leaves // n_ranks
    a = Region(strm, 32 * leaves, IN_OFF, codes[0])
    out = Region(strm, 2 * 32 * leaves, OUT_OFF)
    ml.check(L.ml_pack_pairs_dev(_vp(a.ptr), _sz(2 * leaves), _sz(n_ranks), _sz(2), _sz(1), _vp(out.ptr), strm.arg))
    expect = out.image[OUT_OFF:OUT_OFF + 64 * leaves].reshape(n_ranks, 2, rows, 32).copy()
    expect[:, 1] = pairs[0].reshape(n_ranks, rows, 32)
    assert np.array_equal(out.result().reshape(-1), expect.reshape(-1))
    # the same pairs stored into each rank's receive buffer [global polynomial][row][32 B], here global polynomial 1 of 2
    recv = [Region(strm, 2 * 32 * rows, OUT_OFF + 16 * g, seed=10 + g) for g in range(n_ranks)]
    bases = (C.c_void_p * n_ranks)(*[r.ptr for r in recv])
    ml.check(L.ml_pack_pairs_peer_dev(_vp(a.ptr), _sz(2 * leaves), _sz(n_ranks), _sz(1), bases, C.c_uint(0), strm.arg))
    for g, r in enumerate(recv):
        e = r.image[r.off:r.off + r.nbytes].reshape(2, rows, 32).copy()
        e[1] = pairs[0][g * rows:(g + 1) * rows]
        assert np.array_equal(r.result().reshape(-1), e.reshape(-1)), g
    a.result(unchanged=True)


# ------------------------------------------------------------------ aliasing: in == out
@gpu
@pytest.mark.parametrize("log_n", [10, 14])   # one pass / several passes of the NTT and of the Moebius transform
def test_in_place_rules(ml, oracle, strm, log_n):
    """the aliasing rule the header states for each entry with separate element input and output buffers: in place is allowed
    for the transforms (the buffer holds the larger of input and output; the RS and PCS encodes read the first n elements) and
    rejected with ML_ERR_ARG for the pair packing, whose output overlaps its input"""
    L, n = ml.load(), 1 << log_n
    x = oracle.synthetic(1600 + log_n, n)
    g, g2 = ml.pow_2_generator(log_n), ml.pow_2_generator(log_n + 1)
    c = oracle.to_coefficient(x)
    cases = [("ml_ntt_dev", (_fe(g),), n, oracle.ntt(x, g)),
             ("ml_intt_dev", (_fe(g),), n, oracle.intt(x, g)),
             ("ml_reed_solomon_dev", (_fe(g2),), 2 * n, oracle.reed_solomon(x, g2)),
             ("ml_mle_to_coefficient_dev", (), n, c),
             ("ml_mle_to_evaluation_dev", (), n, oracle.to_evaluation(x)),
             ("ml_pcs_encode_dev", (), 2 * n, oracle.reed_solomon(oracle.bit_reverse(c), g2))]
    for name, gen, n_out, want in cases:
        a = Region(strm, 16 * n_out, OUT_OFF, x)
        ml.check(getattr(L, name)(_vp(a.ptr), _sz(n), *[_p(v) for v in gen], _vp(a.ptr), strm.arg))
        assert np.array_equal(a.result(), want), name
    a = Region(strm, 16 * 2 * n, OUT_OFF, x)
    for out_ptr in (a.ptr, a.ptr + 16 * n - 32):   # the same buffer, and an output that starts inside the input
        assert L.ml_pack_pairs_dev(_vp(a.ptr), _sz(n), _sz(1), _sz(1), _sz(0), _vp(out_ptr), strm.arg) == ML_ERR_ARG
        assert b"overlap" in L.ml_last_error()
        bases = (C.c_void_p * 1)(out_ptr)
        assert L.ml_pack_pairs_peer_dev(_vp(a.ptr), _sz(n), _sz(1), _sz(0), bases, C.c_uint(0), strm.arg) == ML_ERR_ARG
        assert b"overlap" in L.ml_last_error()
    a.result(unchanged=True)
    # the subtree root may be written over the first pair of its input: it is stored after the tree is complete
    pairs = pairs_of(x)
    want = oracle.merkle_batch_commit([pairs]).root()
    r = Region(strm, 16 * n, IN_OFF, pairs)
    ptrs = (C.c_void_p * 1)(r.ptr)
    ml.check(L.ml_batched_leaf_subtree_root_dev(ptrs, _sz(1), _sz(n // 2), _vp(r.ptr), strm.arg))
    assert r.result()[:2].tobytes() == want


# ------------------------------------------------------------------ host-side controls
@gpu
def test_host_controls_keep_the_proof(ml, oracle):
    """thread stream, registered and pinned host inputs, pool trimming and the release threshold: each leaves the proof
    bytes, the sumcheck and the transcript equal to the oracle's"""
    L, nv = ml.load(), 12
    n = 1 << nv
    rng = random.Random(77)
    ev = oracle.synthetic(1700, n)
    inp = fe_arr([rng.randrange(M) for _ in range(nv)])
    out = oracle.mle_evals_evaluate(ev, inp)
    ot = oracle.transcript()
    oproof, st = oracle.pcs_prove(inp, out, ev, ot)
    assert st == 0
    want = (oproof.fri.blob, oproof.sumcheck, ot.random())

    def prove(evals):
        t = ml.Transcript()
        p = ml.PCSProof.prove(inp, out, evals, t)
        return p.fri_proof.serialize(), [c for nz in p.sumcheck_polynomials for c in nz], t.random()
    assert prove(ev) == want
    s = _vp()
    ml.check(L.ml_stream_create(C.byref(s)))
    ml.check(L.ml_set_thread_stream(s, C.c_int(1)))
    try:
        assert prove(ev) == want
    finally:
        ml.check(L.ml_set_thread_stream(None, C.c_int(0)))
        ml.check(L.ml_stream_synchronize(s))
        ml.check(L.ml_stream_destroy(s))
    reg = ml.elems_empty(n)
    reg[:] = ev
    ml.check(L.ml_host_register(_p(reg), _sz(reg.nbytes)))
    try:
        assert prove(reg) == want
    finally:
        ml.check(L.ml_host_unregister(_p(reg)))
    pinned = _vp()
    ml.check(L.ml_host_alloc_pinned(_sz(16 * n), C.byref(pinned)))
    try:
        host = np.ctypeslib.as_array((C.c_uint8 * (16 * n)).from_address(pinned.value)).reshape(n, 16)
        host[:] = ev
        assert prove(host) == want
        del host
    finally:
        ml.check(L.ml_host_free_pinned(pinned))

    def stats():
        r, u = C.c_uint64(0), C.c_uint64(0)
        ml.check(L.ml_pool_stats(C.byref(r), C.byref(u)))
        return r.value, u.value
    ml.synchronize()
    r0, _ = stats()
    ml.check(L.ml_trim_pools(_sz(0)))
    r1, u1 = stats()
    assert r1 <= r0 and u1 <= r1
    assert prove(ev) == want
    ml.check(L.ml_set_pool_release_threshold(C.c_uint64(0)))
    try:
        assert prove(ev) == want
    finally:
        ml.check(L.ml_set_pool_release_threshold(C.c_uint64(2**64 - 1)))


@gpu
def test_accessors_and_device_controls(ml, oracle):
    import torch
    L = ml.load()
    dev = torch.cuda.current_device()
    ml.check(L.ml_set_device(C.c_int(dev)))
    name = C.create_string_buffer(256)
    ml.check(L.ml_device_name(name, _sz(256)))
    assert name.value.decode() == torch.cuda.get_device_name(dev)
    k0 = ml.kernel_launches()
    ml.pow_2_generator_powers(5)
    assert ml.kernel_launches() > k0
    B, log_n = 3, 4
    gen = ml.pow_2_generator(log_n + 1)
    codes = [oracle.reed_solomon(oracle.synthetic(1800 + j, 1 << log_n), gen) for j in range(B)]
    d = ml.BatchedFriProverData.init(codes, ml.Transcript())
    assert L.ml_bfri_num_codes(d.h) == B
    sh = ml.ShardedBatchedProver.single_process([dev, dev], 2, 4)
    # two virtual ranks on one GPU: ranks that share a device share its streams (csrc/shard.cu)
    assert L.ml_shard_num_local(sh.h) == 2 and sh.stream(0) and sh.stream(1) == sh.stream(0)
    sh.free()
    one = ml.ShardedBatchedProver.one_rank(1, 2, dev, 2, 4)
    assert L.ml_shard_num_local(one.h) == 1
    one.free()
    p, handle = _vp(), np.zeros(64, dtype=np.uint8)
    ml.check(L.ml_ipc_alloc(_sz(4096), C.byref(p), _p(handle)))
    try:
        assert p.value and handle.any()
    finally:
        ml.check(L.ml_ipc_free(p))


# ------------------------------------------------------------------ the coverage guard (no GPU)
# entries whose test needs a second process: a CUDA IPC handle cannot be opened by the process that made it
UNTESTED_HERE = {
    "ml_ipc_open": "maps a peer process's buffer; exercised by the two-GPU sharded tests (tools/sharded_prove_demo.py)",
    "ml_ipc_close": "unmaps what ml_ipc_open mapped; exercised by the two-GPU sharded tests (tools/sharded_prove_demo.py)",
}


def _test_sources():
    out = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, "tests")):
        for f in sorted(files):
            if f.endswith(".py") or (os.path.basename(dirpath) == "cpp" and f.endswith(".cpp")):
                with open(os.path.join(dirpath, f), errors="replace") as fh:
                    out.append(fh.read())
    return "\n".join(out)


def api_symbols(declared):
    """{name a test would use: declared symbols it reaches} for every function and method of multilinear_b200/api.py.
    Names built from a prefix resolve: string constants of a function are joined to the ml_ prefixes it holds and to the
    _PREFIX of its class and of every subclass; a function also reaches what the api.py functions it calls reach.  A method
    is used as `.name` (a call or a property); __init__ / __del__ and the class's other dunders are used with the class name."""
    tree = ast.parse(open(os.path.join(ROOT, "multilinear_b200", "api.py")).read())
    classes = {c.name: c for c in tree.body if isinstance(c, ast.ClassDef)}
    prefix = {}
    for c in classes.values():
        for st in c.body:
            if isinstance(st, ast.Assign):
                tgts = st.targets[0].elts if isinstance(st.targets[0], ast.Tuple) else st.targets
                vals = st.value.elts if isinstance(st.value, ast.Tuple) else [st.value]
                for tg, v in zip(tgts, vals):
                    if isinstance(tg, ast.Name) and tg.id == "_PREFIX" and isinstance(v, ast.Constant) and v.value:
                        prefix[c.name] = v.value

    def family(name):
        out = {name}
        for c in classes.values():
            if c.name not in out and any(isinstance(b, ast.Name) and b.id in out for b in c.bases):
                out |= family(c.name)
        return out

    funcs = []   # (use pattern, function node, owning class or None)
    for node in tree.body:
        if isinstance(node, ast.FunctionDef):
            funcs.append((r"\b%s\(" % node.name, node, None))
        elif isinstance(node, ast.ClassDef):
            for st in node.body:
                if isinstance(st, ast.FunctionDef):
                    use = r"\b%s\b" % node.name if st.name.startswith("__") else r"\.%s\b" % st.name
                    funcs.append((use, st, node.name))
    direct, refs = {}, {}
    for i, (_, fn, owner) in enumerate(funcs):
        strs = {n.value for n in ast.walk(fn) if isinstance(n, ast.Constant) and isinstance(n.value, str)}
        names = {n.attr for n in ast.walk(fn) if isinstance(n, ast.Attribute)} | {n.id for n in ast.walk(fn) if isinstance(n, ast.Name)}
        pre = {s for s in strs if s.startswith("ml_")} | {prefix[c] for c in (family(owner) if owner else ()) if c in prefix}
        direct[i] = {s for s in strs | names if s in declared} | {p + j + s for p in pre for s in strs for j in ("", "_") if p + j + s in declared}
        refs[i] = {k for k, (_, other, _) in enumerate(funcs) if other.name in names and k != i}
    reach = {}
    for i in direct:
        seen, todo, syms = {i}, [i], set()
        while todo:
            k = todo.pop()
            syms |= direct[k]
            todo += [r for r in refs[k] if r not in seen]
            seen |= refs[k]
        reach[i] = syms
    return [(funcs[i][0], reach[i]) for i in reach]


def uncovered_symbols():
    declared = set(declared_symbols())
    src = _test_sources()
    covered = {s for s in declared if re.search(r"\b%s\b" % s, src)}
    for use, syms in api_symbols(declared):
        if re.search(use, src):
            covered |= syms
    return sorted(declared - covered - set(UNTESTED_HERE))


def test_every_declared_symbol_has_a_test():
    """every entry of include/multilinear_b200.h is named by a file under tests/ or called by an api.py function or method a
    test uses (UNTESTED_HERE lists the exceptions and why)"""
    assert set(UNTESTED_HERE) <= set(declared_symbols())
    missing = uncovered_symbols()
    assert not missing, "declared in include/multilinear_b200.h but no test reaches them: %s" % ", ".join(missing)
