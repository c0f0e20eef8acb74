"""Both sumchecks over the whole argument space the C ABI accepts, bit for bit against the oracle.

The width-w System sumcheck (ml_wsumcheck_*) takes one of three paths per call:
  - device chain, composition_degree 0..3 (td = degree + 1 <= 4): per round wsumcheck_points_kernel<TD, NARROW> (NARROW: the
    4-way select chain for width <= 4, the indexed row above), wchain_finish_kernel and the fold, until the tables have 2^12
    rows; then wchain_tail_kernel<4> (width <= 4) or <16> runs every remaining round in one CTA.  So n_vars 12 runs the tail
    only, n_vars 13 one chain round and the tail, and n_vars 19 (half = 2^18 > 256 * 592 threads) the points kernel's
    grid-stride loop;
  - host rounds, composition_degree 4..15: one wsumcheck_partial_kernel launch per point, host interpolation on up to 17 points;
  - host rounds for td <= 4 (MLB_WSUMCHECK_HOST_ROUNDS, read once per process): wsumcheck_points_launch.
The PCS tables (ml_sumcheck_*) run every round on the device at composition_degree 1 and host rounds at any other degree.
The sharded handle (ml_wsumcheck_shard_*) runs the same points, finish, fold and tail kernels on every rank after a
width-dependent transpose of the row blocks.

Each case asserts, unless its comment says otherwise: coefficients, challenges and the final transcript equal the oracle's,
the handle's height ends at 1, and, where the declared degree is at least the composition's degree and the claim is the true
sum over the hypercube, the reference's verifier (verify_sumcheck_debug) accepts.
"""
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle import pyref as P
from oracle.binding import fe_arr, fe_ints
from test_oracle import eval_terms, verify_sumcheck_debug
from test_wsumcheck_shard import terms_for

M = P.M
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ML_ERR_OUT_OF_RANGE, ML_ERR_ARG = 3, 8


# ------------------------------------------------------------------ helpers
def true_sum(oracle, row_point, matrix, width, terms):
    """sum over the hypercube of comp(row) * eq(row_point, row): partial_sum(0) + partial_sum(1) of a fresh handle"""
    o = oracle.wsumcheck_build(row_point, matrix, width)
    o.set_composition(terms)
    return (o.partial_sum(0) + o.partial_sum(1)) % M


def oracle_prove(oracle, row_point, matrix, width, terms, degree, s, transcript=None):
    o = oracle.wsumcheck_build(row_point, matrix, width)
    o.set_composition(terms)
    ot = transcript or oracle.transcript()
    got = o.compute_sumcheck_polynomials(degree, ot, s)
    assert o.height() == 1
    return got, ot.random()


def check_wide(ml, oracle, nv, width, degree, terms, s=None, matrix=None, row_point=None, seed=0, verify=True):
    """one ml_wsumcheck_* proof against the oracle (and the verifier when `verify`); returns (coeffs, randoms, transcript)"""
    rng = random.Random(seed)
    if matrix is None:
        matrix = oracle.synthetic(0x5C00 + seed, width << nv)
    if row_point is None:
        row_point = fe_arr([rng.randrange(M) for _ in range(nv)])
    claim = true_sum(oracle, row_point, matrix, width, terms) if s is None else s
    want, want_random = oracle_prove(oracle, row_point, matrix, width, terms, degree, claim)
    g = ml.WideSumcheckTables.build(row_point, matrix, width)
    g.set_composition(terms)
    t = ml.Transcript()
    got = g.compute_sumcheck_polynomials(degree, t, claim)
    assert got == want
    assert len(got[0]) == nv * (degree + 1) and len(got[1]) == nv
    assert t.random() == want_random
    assert g.height == 1
    if verify and nv >= 1:
        assert s is None, "the verifier accepts the true sum only"
        assert verify_sumcheck_debug(oracle, oracle.transcript(), got[0], degree + 1, claim, matrix, width, row_point, terms) == got[1]
    return got[0], got[1], t.random()


def chain_id(nv, width, degree):
    """the path a ml_wsumcheck_compute_polynomials call takes, as a test id"""
    if nv == 0:
        where = "no-rounds"
    elif degree >= 4:
        return "host-td%d_w%d_nv%d" % (degree + 1, width, nv)
    elif nv <= 12:
        where = "tail"
    elif nv < 19:
        where = "chain+tail"
    else:
        where = "grid-stride+tail"
    return "chain-%s-td%d_w%d_nv%d_%s" % ("narrow" if width <= 4 else "wide", degree + 1, width, nv, where)


# ------------------------------------------------------------------ A. width-w, device chain (td 1..4)
A_CASES = ([(nv, w, (w - 1 + nv - 12) % 4) for nv in (12, 13) for w in range(1, 17)]
           + [(0, 1, 0), (0, 16, 3), (1, 3, 2), (1, 5, 1), (1, 16, 3), (2, 4, 3), (2, 9, 0), (2, 2, 1)]
           + [(19, 2, 3), (19, 4, 2), (19, 5, 3), (19, 16, 1)])


@pytest.mark.gpu
@pytest.mark.parametrize("nv,width,degree", A_CASES, ids=[chain_id(*c) for c in A_CASES])
def test_device_chain_every_width(ml, oracle, nv, width, degree):
    rng = random.Random(nv * 100 + width)
    check_wide(ml, oracle, nv, width, degree, terms_for(width, degree, rng), seed=nv * 100 + width)


# ------------------------------------------------------------------ B. width-w, host rounds (td 5..16)
B_WIDTHS = [1, 3, 4, 5, 16]
B_CASES = ([(5, B_WIDTHS[i % 5], d) for i, d in enumerate(range(4, 16))]
           + [(13, 16, 4), (13, 3, 9), (13, 5, 15), (0, 3, 7), (1, 16, 15), (1, 1, 5)])


@pytest.mark.gpu
@pytest.mark.parametrize("nv,width,degree", B_CASES, ids=[chain_id(*c) for c in B_CASES])
def test_host_rounds_every_degree(ml, oracle, nv, width, degree):
    rng = random.Random(1000 + nv * 100 + degree)
    check_wide(ml, oracle, nv, width, degree, terms_for(width, degree, rng), seed=1000 + degree)


@pytest.mark.gpu
def test_composition_degree_16_rejected(ml, oracle):
    matrix, row_point = oracle.synthetic(1, 4 << 5), oracle.synthetic(2, 5)
    g = ml.WideSumcheckTables.build(row_point, matrix, 4)
    g.set_composition([(1, [0])])
    with pytest.raises(ml.MlError) as e:
        g.compute_sumcheck_polynomials(16, ml.Transcript(), 0)
    assert e.value.code == ML_ERR_ARG
    assert g.height == 1 << 5
    check_wide(ml, oracle, 5, 4, 15, [(1, [0] * 15)], matrix=matrix, row_point=row_point)  # degree 15 is the largest accepted


# ------------------------------------------------------------------ C. host rounds for td <= 4 (a child with the switch set)
HOST_ROUNDS_CHILD = r"""
import json, os, sys
sys.path.insert(0, sys.argv[1])
from multilinear_b200 import api as ml
from oracle.binding import Oracle
O = Oracle()
out = []
for c in json.load(sys.stdin):
    nv, w = c["n_vars"], c["width"]
    g = ml.WideSumcheckTables.build(O.synthetic(c["seed"] + 1, nv), O.synthetic(c["seed"], w << nv), w)
    g.set_composition([(k, cs) for k, cs in c["terms"]])
    t = ml.Transcript()
    co, rs = g.compute_sumcheck_polynomials(c["degree"], t, c["sum"])
    out.append({"coeffs": co, "rs": rs, "random": t.random().hex(), "height": g.height})
print(json.dumps({"host_rounds": os.environ.get("MLB_WSUMCHECK_HOST_ROUNDS"), "results": out}))
"""


@pytest.mark.gpu
def test_host_rounds_switch_equals_device_chain(ml, oracle):
    """MLB_WSUMCHECK_HOST_ROUNDS sends td 1..4 through wsumcheck_points_launch (its TD = 4 default case included) with the
    transcript on the host.  A child process runs td 1..4 x widths {1, 3, 4, 5, 16} at n_vars 13 with the switch set; each
    result equals this process's device chain and the oracle, and the verifier accepts it."""
    nv, cases = 13, []
    for degree in range(4):
        for w in (1, 3, 4, 5, 16):
            seed = 0x4800 + 16 * degree + w
            rng = random.Random(seed)
            terms = terms_for(w, degree, rng)
            matrix, row_point = oracle.synthetic(seed, w << nv), oracle.synthetic(seed + 1, nv)
            cases.append({"n_vars": nv, "width": w, "degree": degree, "seed": seed, "terms": terms,
                          "sum": true_sum(oracle, row_point, matrix, w, terms)})
    env = dict(os.environ, MLB_WSUMCHECK_HOST_ROUNDS="1")
    p = subprocess.run([sys.executable, "-c", HOST_ROUNDS_CHILD, ROOT], input=json.dumps(cases), capture_output=True, text=True,
                       timeout=600, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    res = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert res["host_rounds"] == "1" and len(res["results"]) == len(cases)
    for c, child in zip(cases, res["results"]):
        w, degree = c["width"], c["degree"]
        matrix, row_point = oracle.synthetic(c["seed"], w << nv), oracle.synthetic(c["seed"] + 1, nv)
        co, rs, rnd = check_wide(ml, oracle, nv, w, degree, c["terms"], matrix=matrix, row_point=row_point)
        assert (child["coeffs"], child["rs"], child["random"], child["height"]) == (co, rs, rnd.hex(), 1), (w, degree)


# ------------------------------------------------------------------ D. composition shapes
def _every_column(w):
    return [(3 + j, [j]) for j in range(w)] + [(M - 7, [0, w - 1])]


SHAPES = {  # name -> (terms(width), declared degree, verifier applies)
    "no-terms": (lambda w: [], 2, True),
    "constant-only": (lambda w: [(0xC0FFEE, [])], 0, True),
    "zero-coefficients": (lambda w: [(0, [0, w - 1, 1 % w]), (0, []), (5, [w - 1]), (0, [0])], 3, True),
    "coefficient-M-1": (lambda w: [(M - 1, [0, w - 1, 0]), (M - 1, []), (M - 1, [w // 2])], 3, True),
    "every-column": (_every_column, 2, True),
    "term-longer-than-degree": (lambda w: [(9, [w - 1] * 6), (4, [0])], 2, False),
}
D_CASES = [(name, w, nv) for name in SHAPES for w in (4, 16) for nv in (13,)] + [("x0^16-declared-15", 4, 5), ("x0^16-declared-15", 16, 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,width,nv", D_CASES,
                         ids=["%s_%s" % (n, chain_id(nv, w, SHAPES[n][1] if n in SHAPES else 15)) for n, w, nv in D_CASES])
def test_composition_shapes(ml, oracle, name, width, nv):
    if name in SHAPES:
        make, degree, verify = SHAPES[name]
        terms = make(width)
    else:  # degree 16 under a declared 15: host rounds on 17 points; parity only (the round polynomial is too short)
        terms, degree, verify = [(0xABCDEF, [0] * 16)], 15, False
    rng = random.Random(7)
    row_point = fe_arr([rng.randrange(M) for _ in range(nv)])
    matrix = oracle.synthetic(0xD00 + width, width << nv)
    s = None if verify else true_sum(oracle, row_point, matrix, width, terms)
    check_wide(ml, oracle, nv, width, degree, terms, s=s, matrix=matrix, row_point=row_point, verify=verify)


def full_composition(width, seed):
    """exactly W_MAX_TERMS = 64 terms with W_MAX_COLS = 256 column references (four each: degree 4), every column used"""
    rng = random.Random(seed)
    cols = [j % width for j in range(256)]
    rng.shuffle(cols)
    return [(rng.randrange(M), cols[4 * t:4 * t + 4]) for t in range(64)]


@pytest.mark.gpu
@pytest.mark.parametrize("width", [4, 16], ids=["narrow-w4", "wide-w16"])
@pytest.mark.parametrize("degree", [4, 3], ids=["host-td5-verified", "chain-td4-full-shared-arrays"])
def test_composition_limits(ml, oracle, width, degree):
    """64 terms, 256 references: at the declared degree 4 (host rounds) the verifier accepts; at 3 the device chain and the
    tail run with their shared term arrays full (parity with the oracle only)"""
    terms = full_composition(width, width)
    nv = 13
    matrix, row_point = oracle.synthetic(0xF00 + width, width << nv), oracle.synthetic(0xF80 + width, nv)
    s = None if degree == 4 else true_sum(oracle, row_point, matrix, width, terms)
    check_wide(ml, oracle, nv, width, degree, terms, s=s, matrix=matrix, row_point=row_point, verify=degree == 4)


@pytest.mark.gpu
@pytest.mark.parametrize("width", [4, 16])
def test_composition_rejections_keep_the_previous_one(ml, oracle, width):
    nv, degree = 13, 3
    matrix, row_point = oracle.synthetic(0xE00 + width, width << nv), oracle.synthetic(0xE80 + width, nv)
    good = terms_for(width, degree, random.Random(width))
    too_many_terms = [(1, [t % width]) for t in range(65)]
    too_many_refs = full_composition(width, 1)[:63] + [(1, [0] * 5)]
    assert sum(len(c) for _, c in too_many_refs) == 257 and len(too_many_refs) == 64
    bad_column = [(1, [0]), (2, [width - 1, width])]
    g = ml.WideSumcheckTables.build(row_point, matrix, width)
    g.set_composition(good)
    for bad, code in ((too_many_terms, ML_ERR_ARG), (too_many_refs, ML_ERR_ARG), (bad_column, ML_ERR_OUT_OF_RANGE)):
        with pytest.raises(ml.MlError) as e:
            g.set_composition(bad)
        assert e.value.code == code
    t = ml.Transcript()
    got = g.compute_sumcheck_polynomials(degree, t, 5)
    assert (got, t.random()) == oracle_prove(oracle, row_point, matrix, width, good, degree, 5)


# ------------------------------------------------------------------ E. values and points
@pytest.mark.gpu
@pytest.mark.parametrize("width,nv", [(1, 9), (3, 9), (4, 9), (5, 9), (16, 9), (3, 1)])
def test_partial_sum_at_every_kind_of_point(ml, oracle, width, nv):
    """wsumcheck_partial_kernel: r = 1 is its is_one branch, r = 0 keeps only the low rows"""
    rng = random.Random(width)
    matrix, row_point = oracle.synthetic(0xA00 + width, width << nv), fe_arr([rng.randrange(M) for _ in range(nv)])
    terms = terms_for(width, 3, rng)
    o = oracle.wsumcheck_build(row_point, matrix, width)
    o.set_composition(terms)
    g = ml.WideSumcheckTables.build(row_point, matrix, width)
    g.set_composition(terms)
    for r in (0, 1, 2, 3, 4, 5, 16, M - 1, rng.randrange(M)):
        assert g.partial_sum(r) == o.partial_sum(r), r


def _special_trace(oracle, kind, width, nv):
    h = 1 << nv
    if kind == "all-M-1":
        return np.ascontiguousarray(np.tile(fe_arr([M - 1]), (h * width, 1)))
    if kind == "all-zero":
        return np.zeros((h * width, 16), dtype=np.uint8)
    half = oracle.synthetic(0xB00 + width, (h // 2) * width)  # "equal-fold-pairs": rows i and i + h/2 agree
    return np.ascontiguousarray(np.concatenate([half, half]))


E_CASES = [(kind, w, d) for kind in ("all-M-1", "all-zero", "equal-fold-pairs") for w, d in ((4, 3), (16, 2), (5, 6))]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,width,degree", E_CASES, ids=["%s_%s" % (k, chain_id(13, w, d)) for k, w, d in E_CASES])
def test_special_traces(ml, oracle, kind, width, degree):
    nv = 13
    check_wide(ml, oracle, nv, width, degree, terms_for(width, degree, random.Random(width + degree)),
               matrix=_special_trace(oracle, kind, width, nv), seed=width)


@pytest.mark.gpu
@pytest.mark.parametrize("width,degree", [(4, 3), (16, 1), (3, 5)])
def test_row_point_with_0_1_and_M_minus_1(ml, oracle, width, degree):
    """the eq table then has whole zero halves; the verifier still accepts"""
    nv = 13
    rng = random.Random(degree)
    row_point = fe_arr([0, 1, M - 1] + [rng.randrange(M) for _ in range(nv - 6)] + [M - 1, 1, 0])
    check_wide(ml, oracle, nv, width, degree, terms_for(width, degree, rng), row_point=row_point, seed=degree)


@pytest.mark.gpu
@pytest.mark.parametrize("claim", [0, M - 1], ids=["claim-0", "claim-M-1"])
@pytest.mark.parametrize("width,degree", [(4, 2), (16, 3), (5, 7)])
def test_claims_0_and_M_minus_1(ml, oracle, claim, width, degree):
    """a wrong claim is proved like any other (parity with the oracle only)"""
    check_wide(ml, oracle, 13, width, degree, terms_for(width, degree, random.Random(width)), s=claim, seed=width, verify=False)


# ------------------------------------------------------------------ F. PCS tables (ml_sumcheck_*)
def pcs_inputs(oracle, nv, seed):
    ev = oracle.synthetic(0x9C00 + seed, 1 << nv)
    inp = oracle.synthetic(0x9D00 + seed, nv)
    return ev, inp, oracle.mle_evals_evaluate(ev, inp) if nv else fe_ints(ev)[0]


F_CASES = [(cd, nv) for cd in (0, 2, 3, 4, 7, 15) for nv in (0, 1, 5, 13, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("cd,nv", F_CASES, ids=["pcs-%s-cd%d_nv%d" % ("host" if cd != 1 else "chain", cd, nv) for cd, nv in F_CASES])
def test_pcs_tables_every_composition_degree(ml, oracle, cd, nv):
    """compute_sumcheck_polynomials off the PCS degree (host transcript, one partial_sum launch per point); for degree >= 1 the
    PCS verifier's replay (delta(inputs, rs) * f(rs) == pol(r_last)) accepts the true claim"""
    ev, inp, claim = pcs_inputs(oracle, nv, 16 * cd + nv)
    s, os_ = ml.SumcheckTables.build_tables_for_pcs(inp, ev), oracle.sumcheck_build(inp, ev)
    t, ot = ml.Transcript(), oracle.transcript()
    got = s.compute_sumcheck_polynomials(cd, t, claim)
    assert got == os_.compute_sumcheck_polynomials(cd, ot, claim)
    assert t.random() == ot.random() and s.height == 1
    td = cd + 1
    coeffs, rs = got
    assert len(coeffs) == nv * td and len(rs) == nv
    for a, b in zip(s.tables(), os_.tables()):
        assert np.array_equal(a, b)
    if cd >= 1 and nv >= 1:
        polys = [coeffs[td * k:td * (k + 1)] for k in range(nv)]
        last = oracle.mle_evals_evaluate(ev, fe_arr(rs))
        assert P._sumcheck_replay(polys, claim, fe_ints(inp), rs, last)
        assert not P._sumcheck_replay(polys, (claim + 1) % M, fe_ints(inp), rs, last)


@pytest.mark.gpu
@pytest.mark.parametrize("nv", [1, 13])
def test_pcs_single_round_every_total_degree(ml, oracle, nv):
    for td in range(1, 17):
        ev, inp, claim = pcs_inputs(oracle, nv, td)
        s, os_ = ml.SumcheckTables.build_tables_for_pcs(inp, ev), oracle.sumcheck_build(inp, ev)
        t, ot = ml.Transcript(), oracle.transcript()
        assert s.compute_sumcheck_polynomial(td, claim, t) == os_.compute_sumcheck_polynomial(td, claim, ot), td
        assert t.random() == ot.random() and s.height == os_.height() == 1 << (nv - 1)
        for a, b in zip(s.tables(), os_.tables()):
            assert np.array_equal(a, b), td


@pytest.mark.gpu
def test_pcs_degree_limits(ml, oracle):
    """total_degree 0 (the reference panics) and 17, composition_degree 16: ML_ERR_ARG, and the handle is untouched"""
    ev, inp, claim = pcs_inputs(oracle, 6, 0)
    s = ml.SumcheckTables.build_tables_for_pcs(inp, ev)
    before = s.tables()
    t = ml.Transcript()
    for td in (0, 17):
        with pytest.raises(ml.MlError) as e:
            s.compute_sumcheck_polynomial(td, claim, t)
        assert e.value.code == ML_ERR_ARG, td
    with pytest.raises(ml.MlError) as e:
        s.compute_sumcheck_polynomials(16, t, claim)
    assert e.value.code == ML_ERR_ARG
    assert s.height == 1 << 6 and all(np.array_equal(a, b) for a, b in zip(s.tables(), before))
    assert t.random() == ml.Transcript().random()


# ------------------------------------------------------------------ G. sharded width-w (virtual ranks on one GPU)
G_CASES = [(G, nv, w, (i + j) % 4) for j, w in enumerate((2, 3, 7, 8, 9, 15)) for G in (2, 8)
           for i, nv in enumerate((max(1, G.bit_length() - 1), 13, 17))] + [(16, 13, 7, 2)]


def _shard_id(G, nv, w, d):
    return "shard-G%d-%s-td%d_w%d_nv%d_%s" % (G, "narrow" if w <= 4 else "wide", d + 1, w, nv, "rounds+gather+tail" if nv > 12 else "tail")


def check_sharded(ml, oracle, G, nv, w, degree, terms, seed):
    rng = random.Random(seed)
    matrix = oracle.synthetic(0x6000 + seed, w << nv)
    row_point = fe_arr([rng.randrange(M) for _ in range(nv)])
    s = rng.randrange(M)
    sh = ml.ShardedWideSumcheck.single_process([0] * G, w, nv)
    try:
        sh.set_composition(terms)
        t = ml.Transcript()
        got = sh.compute_sumcheck_polynomials(row_point, matrix, degree, t, s)
        g = ml.WideSumcheckTables.build(row_point, matrix, w)
        g.set_composition(terms)
        gt = ml.Transcript()
        assert got == g.compute_sumcheck_polynomials(degree, gt, s)
        assert (got, t.random()) == oracle_prove(oracle, row_point, matrix, w, terms, degree, s)
        assert gt.random() == t.random()
    finally:
        sh.free()


@pytest.mark.gpu
@pytest.mark.parametrize("G,nv,width,degree", G_CASES, ids=[_shard_id(*c) for c in G_CASES])
def test_sharded_widths_vs_single_gpu_and_oracle(ml, oracle, G, nv, width, degree):
    seed = G * 1000 + nv * 20 + width
    check_sharded(ml, oracle, G, nv, width, degree, terms_for(width, degree, random.Random(seed)), seed)


@pytest.mark.gpu
@pytest.mark.parametrize("width", [4, 16])
def test_sharded_full_composition(ml, oracle, width):
    """64 terms and 256 references in every rank's arena, G = 4, declared degree 3"""
    check_sharded(ml, oracle, 4, 15, width, 3, full_composition(width, 40 + width), 40 + width)


# ------------------------------------------------------------------ H. the oracle above degree 3 (no GPU)
def restated_wsumcheck(row_point, matrix, width, terms, degree, s, coeffs, rs):
    """System sumcheck (sumcheck.rs:147-247) in Python big ints, checking a prover's coefficients and challenges round by round:
    partial sums at 1..td, the round polynomial through (0, s - p(1)), (1, p(1)) .. (td, p(td)) (checked by evaluation: a
    polynomial of degree <= td through td + 1 points is the interpolant), the transcript, the fold.  Returns the transcript."""
    nv = len(row_point)
    h, w, td = 1 << nv, width, degree + 1
    mat = list(matrix)
    delta = []
    for idx in range(h):  # Mask::evaluate (evaluation.rs:56-73)
        p = 1
        for i in range(nv):
            pt = row_point[nv - 1 - i]
            p = p * (pt if (idx >> i) & 1 else 1 - pt) % M
        delta.append(p)
    t, prev = P.Transcript(), s
    for k in range(nv):
        off = h >> 1
        evals = [0] * (td + 1)
        for r in range(1, td + 1):
            acc = 0
            for i in range(off):
                row = [((1 - r) * mat[i * w + j] + r * mat[(i + off) * w + j]) % M for j in range(w)]
                acc += eval_terms(terms, row) * (((1 - r) * delta[i] + r * delta[i + off]) % M)
            evals[r] = acc % M
        evals[0] = (prev - evals[1]) % M
        pol = [evals[0]] + coeffs[k * td:(k + 1) * td]
        assert [P.poly_eval(pol, x) for x in range(td + 1)] == evals, "round %d" % k
        for c in pol[1:]:
            t.absorb(P.to_bytes(c))
        r = t.next_challenge()
        assert r == rs[k], "round %d" % k
        prev = P.poly_eval(pol, r)
        for i in range(off):
            delta[i] = ((1 - r) * delta[i] + r * delta[i + off]) % M
            for j in range(w):
                mat[i * w + j] = ((1 - r) * mat[i * w + j] + r * mat[(i + off) * w + j]) % M
        h = off
    return t


@pytest.mark.parametrize("width", [1, 3, 16])
def test_oracle_above_degree_3_vs_python_restatement(oracle, width):
    nv = 3
    for degree in range(4, 16):
        rng = random.Random(100 * width + degree)
        terms = terms_for(width, degree, rng)
        matrix, row_point = oracle.synthetic(0x3300 + degree, width << nv), fe_arr([rng.randrange(M) for _ in range(nv)])
        s = true_sum(oracle, row_point, matrix, width, terms)
        ot = oracle.transcript()
        (coeffs, rs), _ = oracle_prove(oracle, row_point, matrix, width, terms, degree, s, ot)
        assert len(coeffs) == nv * (degree + 1)
        t = restated_wsumcheck(fe_ints(row_point), fe_ints(matrix), width, terms, degree, s, coeffs, rs)
        assert t.random() == ot.random(), degree
        assert verify_sumcheck_debug(oracle, oracle.transcript(), coeffs, degree + 1, s, matrix, width, row_point, terms) == rs


def test_oracle_refuses_total_degree_0(oracle):
    """the reference indexes evals[1] of a one-point round (sumcheck.rs:188) and panics; the oracle refuses the call and leaves
    the tables and the transcript as they were"""
    ev, inp = oracle.synthetic(5, 1 << 4), oracle.synthetic(6, 4)
    s = oracle.sumcheck_build(inp, ev)
    before = s.tables()
    t = oracle.transcript()
    with pytest.raises(ValueError):
        s.compute_sumcheck_polynomial(0, 7, t)
    assert s.height() == 1 << 4 and all(np.array_equal(a, b) for a, b in zip(s.tables(), before))
    assert t.random() == oracle.transcript().random()
    with pytest.raises(IndexError):
        P.SumcheckTables(fe_ints(inp), fe_ints(ev)).compute_sumcheck_polynomial(0, 7, P.Transcript())
    assert s.compute_sumcheck_polynomial(1, 7, t)[0] == P.SumcheckTables(fe_ints(inp), fe_ints(ev)).compute_sumcheck_polynomial(
        1, 7, P.Transcript())[0]

