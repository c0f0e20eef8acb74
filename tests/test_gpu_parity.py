"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the golden vectors.  Bit-exact: every
quantity on this path is integer / byte data (SURVEY.md §8)."""
import hashlib
import random

import numpy as np
import pytest

from oracle import pyref as P
from oracle.binding import fe_arr, fe_ints

pytestmark = pytest.mark.gpu
M = P.M


def sha(b):
    return hashlib.sha256(b).hexdigest()


EDGE = [0, 1, 2, M - 1, M - 2, 2**64 - 1, 2**64, 2**64 + 1, 2**127, 2**96 - 1, 45 * 2**40 - 1, 45 * 2**40, 2**128 - 2**46 - 7, M - 2**40]


# ------------------------------------------------------------------ field
def test_field_ops_edge_and_random(ml, oracle):
    rng = random.Random(21)
    xs = [x for x in EDGE for _ in EDGE] + [rng.randrange(M) for _ in range(1 << 16)]
    ys = [y for _ in EDGE for y in EDGE] + [rng.randrange(M) for _ in range(1 << 16)]
    a, b = fe_arr(xs), fe_arr(ys)
    for op, pyop in (("mul", lambda x, y: x * y % M), ("add", lambda x, y: (x + y) % M), ("sub", lambda x, y: (x - y) % M)):
        got = getattr(ml, op)(a, b)
        assert np.array_equal(got, oracle.vec(op, a, b)), op
        assert fe_ints(got[:len(EDGE) ** 2]) == [pyop(x, y) for x, y in zip(xs[:len(EDGE) ** 2], ys[:len(EDGE) ** 2])]


def test_field_mul_large_random(ml, oracle):
    a, b = oracle.synthetic(1, 1 << 20), oracle.synthetic(2, 1 << 20)
    assert np.array_equal(ml.mul(a, b), oracle.vec("mul", a, b))
    # products whose high limbs are all-ones stress the carry chains
    near = fe_arr([M - 1 - i for i in range(4096)])
    assert np.array_equal(ml.mul(near, near[::-1].copy()), oracle.vec("mul", near, near[::-1].copy()))


@pytest.mark.parametrize("variant", [1, 2])
def test_field_reduce_wide_adversarial(ml, variant):
    """fe_reduce_wide on 256-bit patterns that exercise every carry / wrap path of both folds: all-ones limbs, low half
    near 0 / near 2^128 / around M, high half tiny / huge, second-fold wrap candidates, plus random values"""
    rng = random.Random(99 + variant)
    two128, c = 1 << 128, (1 << 128) - M
    los = [0, 1, 2, c - 1, c, c + 1, M - 1, M, M + 1, two128 - 1, two128 - 2, two128 - c, two128 - c - 1, two128 - (1 << 92), two128 - (1 << 46),
           (1 << 96) - 1, (1 << 64), (1 << 32) - 1, 0xFFFFFFFF00000000FFFFFFFF00000000]
    his = [0, 1, 2, 45, (1 << 14) - 1, (1 << 32) - 1, (1 << 32), (1 << 46) - 1, (1 << 64) - 1, (1 << 88) - 45, (1 << 96) - 1, M >> 1, M - 1, M,
           two128 - 1, two128 - 2, two128 - (1 << 40), 0xFFFFFFFF00000000FFFFFFFF00000000, 0x00000000FFFFFFFF00000000FFFFFFFF]
    vals = [(h << 128) | l for h in his for l in los]
    # values whose first fold lands just below / above a multiple of 2^128 (wrap candidates of the second fold)
    for h in his:
        t = h * c
        for d in (-2, -1, 0, 1, 2, c, -c):
            l = (-(t) + d) % two128
            vals.append((h << 128) | l)
    vals += [(M - 1) ** 2, (M - 1) * (M - 2), (two128 - 1) ** 2 % (1 << 256), (1 << 256) - 1, (1 << 255), (1 << 256) - (1 << 128)]
    vals += [rng.getrandbits(256) for _ in range(20000)]
    vals += [(rng.getrandbits(128) << 128) | rng.choice([0, 1, two128 - 1, rng.getrandbits(20), two128 - 1 - rng.getrandbits(20)]) for _ in range(20000)]
    got = ml.from_wide(vals, variant)
    bad = [(hex(v), g) for v, g in zip(vals, got) if g != v % M]
    assert not bad, bad[:3]


def test_field_inv_pow_from_i64(ml, oracle):
    rng = random.Random(22)
    xs = EDGE + [rng.randrange(M) for _ in range(500)]
    assert ml.to_ints(ml.inv(xs)) == [P.inv(x) for x in xs]  # inv(0) = 0
    e = rng.randrange(M)
    assert ml.to_ints(ml.pow_(xs, e)) == [pow(x, e, M) for x in xs]
    vals = [-1, -7, 0, 1, 2**40, -2**63, 2**63 - 1, -45 * 2**40]
    assert ml.to_ints(ml.from_i64(vals)) == [P.from_i64(v) for v in vals]


def test_synthetic_generator_matches_oracle(ml, oracle):
    buf = ml.synthetic_elements_dev(0xB200, 5000)
    ml.synchronize()
    assert np.array_equal(buf.elems(), oracle.synthetic(0xB200, 5000))


# ------------------------------------------------------------------ NTT
def test_ntt_golden(ml, golden):
    e = ml.ntt(list(range(8)), ml.pow_2_generator(3))
    assert [str(x) for x in ml.to_ints(e)] == golden["ntt8"]
    coeffs = ml.from_i64(range(1 << 10))
    assert sha(ml.ntt(coeffs, ml.pow_2_generator(10)).tobytes()) == golden["ntt_1024_sha"]
    assert sha(ml.reed_solomon(coeffs, ml.pow_2_generator(11)).tobytes()) == golden["rs_1024_sha"]


@pytest.mark.parametrize("log_n", list(range(0, 24)))
def test_ntt_intt_rs_all_sizes(ml, oracle, log_n):
    n = 1 << log_n
    x = oracle.synthetic(100 + log_n, n)
    g = ml.pow_2_generator(log_n)
    want = oracle.ntt(x, g) if n > 1 else x
    got = ml.ntt(x, g)
    assert np.array_equal(got, want)
    assert np.array_equal(ml.intt(got, g), x)  # intt_test, src/ntt/mod.rs:192-201
    if n > 1:
        assert np.array_equal(ml.intt(got, g), oracle.intt(want, g))
    g2 = ml.pow_2_generator(log_n + 1)
    assert np.array_equal(ml.reed_solomon(x, g2), oracle.reed_solomon(x, g2))


def test_ntt_inverse_generator_and_errors(ml, oracle):
    x = oracle.synthetic(7, 1 << 13)
    g = ml.pow_2_generator(13)
    ginv = P.inv(g)
    assert np.array_equal(ml.ntt(x, ginv), oracle.ntt(x, ginv))
    assert np.array_equal(ml.intt(x, ginv), oracle.intt(x, ginv))
    with pytest.raises(ml.NotPowerOfTwo):
        ml.ntt(oracle.synthetic(1, 12), g)
    with pytest.raises(ml.MlError):
        ml.ntt(x, 12345)  # not a root of unity of that order


def test_bit_reverse_and_powers(ml, oracle):
    for n in (1, 2, 8, 1 << 12, 1 << 15):
        x = oracle.synthetic(n, n)
        assert np.array_equal(ml.bit_reverse_permutation(x), oracle.bit_reverse(x))
    x = oracle.synthetic(3, 12)  # trailing_zeros(12) = 2: only the first 4 entries move
    assert np.array_equal(ml.bit_reverse_permutation(x), oracle.bit_reverse(x))
    for log in (0, 1, 5, 12, 13, 17):
        assert np.array_equal(ml.pow_2_generator_powers(log), oracle.pow2_generator_powers(log))


def test_polynomial_evaluate(ml, oracle):
    rng = random.Random(5)
    for n in (1, 5, 4096, 10000):
        c = oracle.synthetic(n, n)
        x = rng.randrange(M)
        assert ml.polynomial_evaluate(c, x) == P.poly_eval(fe_ints(c), x)


# ------------------------------------------------------------------ multilinear polynomials
def test_mle_transforms(ml, oracle, golden):
    e6 = ml.MultilinearPolynomialEvals([0, 1, 4, 8, 9, 3])
    c6 = e6.to_coefficient()
    assert [str(x) for x in ml.to_ints(c6.coeffs)] == golden["mle_conv6"]
    assert np.array_equal(c6.to_evaluation().evals, e6.evals)  # multilinear_conversion_test
    for log_n in (0, 1, 3, 11, 12, 13, 16, 20, 21, 22):
        x = oracle.synthetic(40 + log_n, 1 << log_n)
        c = ml.MultilinearPolynomialEvals(x).to_coefficient()
        assert np.array_equal(c.coeffs, oracle.to_coefficient(x)), log_n
        assert np.array_equal(c.to_evaluation().evals, x)


def test_mle_evaluate(ml, oracle):
    rng = random.Random(9)
    for nv in (0, 1, 4, 12, 13, 15):
        ev = oracle.synthetic(60 + nv, 1 << nv)
        args = fe_arr([rng.randrange(M) for _ in range(nv)]) if nv else np.zeros((0, 16), dtype=np.uint8)
        want = oracle.mle_evals_evaluate(ev, args) if nv else fe_ints(ev)[0]
        assert ml.MultilinearPolynomialEvals(ev).evaluate(ml.to_ints(args)) == want
        co = oracle.to_coefficient(ev)
        assert ml.MultilinearPolynomial(co).evaluate(ml.to_ints(args)) == want
    e6 = ml.MultilinearPolynomialEvals([0, 1, 4, 8, 9, 3])  # len 6 -> next_power_of_two = 8 = 2^3
    args = [rng.randrange(M) for _ in range(3)]
    assert e6.evaluate(args) == P.mle_evals_evaluate([0, 1, 4, 8, 9, 3], args)
    with pytest.raises(ml.SizeMismatch):
        e6.evaluate(args[:2])


# ------------------------------------------------------------------ Merkle
def test_merkle_reference_tests(ml, golden):
    d0 = np.array([[0], [8], [4], [1], [5], [7], [6], [1]], dtype=np.uint8)
    d1 = np.array([[1], [3], [2], [3], [2], [1], [2], [3]], dtype=np.uint8)
    m = ml.Merkle.commit(d0)
    assert m.root().hex() == golden["merkle_test_root"]
    value, path = m.open(5)
    assert value == bytes([7]) and ml.path_verify(value, path, m.root(), 5) == 0  # merkle_test
    assert m.open(8) is None
    mb = ml.Merkle.batch_commit([d0, d1])
    assert mb.root().hex() == golden["batched_merkle_test_root"]
    v5, p5 = mb.batch_open(5)
    assert v5 == bytes([7, 1]) and ml.path_verify(v5, p5, mb.root(), 5) == 0
    v2, p2 = mb.batch_open(2)
    assert v2 == bytes([4, 2]) and ml.path_verify(v2, p2, mb.root(), 2) == 0 and ml.path_verify(v2, p2, mb.root(), 1) != 0
    vec = [[[0, 4], [8, 2], [4, 9], [1, 3], [5, 7], [7, 2], [6, 8], [1, 5]], [[9, 3], [2, 7], [6, 1], [3, 8], [4, 2], [8, 5], [1, 9], [7, 4]],
           [[3, 6], [5, 1], [8, 3], [2, 9], [7, 5], [1, 8], [4, 3], [6, 2]], [[7, 1], [3, 9], [5, 2], [8, 6], [1, 4], [9, 7], [2, 5], [4, 8]]]
    mv = ml.Merkle.batch_commit([np.array(b, dtype=np.uint8) for b in vec])
    assert mv.root().hex() == golden["batched_merkle_with_vectors_test_root"]
    with pytest.raises(ml.NotPowerOfTwo):
        ml.Merkle.commit(d0[:6])
    with pytest.raises(ml.SizeMismatch):
        ml.Merkle.batch_commit([])


@pytest.mark.parametrize("n_items,item_bytes", [(1, 32), (2, 32), (8, 7), (64, 55), (64, 56), (1024, 64), (4096, 100), (16384, 32)])
def test_merkle_generic_items(ml, oracle, n_items, item_bytes):
    rng = np.random.default_rng(n_items + item_bytes)
    data = rng.integers(0, 256, size=(n_items, item_bytes), dtype=np.uint8)
    m, om = ml.Merkle.commit(data), oracle.merkle_commit(data)
    assert m.root() == om.root()
    for a, b in zip(m.layers, om.layers()):
        assert np.array_equal(a, b)
    for idx in {0, n_items - 1, n_items // 3}:
        assert m.open(idx) == om.open(idx)


# ------------------------------------------------------------------ FRI
def test_fri_golden(ml, golden):
    g = golden["fri_log10"]
    vals = ml.from_i64([7 * i + 3 for i in range(1 << 10)])
    gp = ml.pow_2_generator_powers(11)
    code = ml.reed_solomon(vals, ml.to_ints(gp[1:2])[0])
    t = ml.Transcript()
    proof = ml.FriProof.prove(code, gp, t)
    assert [c.hex() for c in proof.commitments] == g["commitments"]
    assert str(proof.last_elem) == g["last_elem"] and proof.last_random.hex() == g["last_random"]
    blob = proof.serialize()
    assert len(blob) == g["blob_len"] and sha(blob) == g["blob_sha"]
    assert proof.verify() == 0  # prove_and_verify_test
    t2 = ml.Transcript()
    p2 = ml.FriProof.prove_from_coeffs(vals, t2)  # fused reed_solomon + prove
    assert p2.serialize() == blob and t2.random() == t.random()


@pytest.mark.parametrize("log_n", [1, 2, 3, 4, 7, 12, 13, 16])
def test_fri_stepwise_vs_oracle(ml, oracle, log_n):
    n = 1 << log_n  # message length; code has 2n elements
    coeffs = oracle.synthetic(70 + log_n, n)
    gp = oracle.pow2_generator_powers(log_n + 1)
    code = oracle.reed_solomon(coeffs, fe_ints(gp[1:2])[0])
    t, ot = ml.Transcript(), oracle.transcript()
    f, of = ml.FriProverData.init(code, t), oracle.fri_init(code, ot)
    for k in range(log_n):
        r = t.next_challenge()
        assert r == ot.next_challenge()
        f.fold_step(gp, k, r, t)
        assert of.fold_step(gp, k, r, ot) == 0
    assert f.num_trees() == of.num_trees() == log_n
    assert f.fold_roots() == of.roots() and f.last_element == of.last_element() and f.last_element is not None
    for j in range(f.num_trees()):
        assert np.array_equal(f.tree_data(j), of.tree_data(j)), j
        for a, b in zip(f.tree(j).layers, of.tree(j).layers()):
            assert np.array_equal(a, b)
    assert t.random() == ot.random()
    idx = (12345 * log_n) % n
    q = f.open_query_at(idx)
    cur, cur_n = idx, n
    for j, (value, path) in enumerate(q):
        assert (value, path) == of.tree(j).open(cur)
        cur_n //= 2
        cur = cur % cur_n if cur_n else 0


def test_fri_prove_vs_oracle_and_errors(ml, oracle):
    log_n = 14
    coeffs = oracle.synthetic(5, 1 << log_n)
    gp = oracle.pow2_generator_powers(log_n + 1)
    code = oracle.reed_solomon(coeffs, fe_ints(gp[1:2])[0])
    t, ot = ml.Transcript(), oracle.transcript()
    proof = ml.FriProof.prove(code, gp, t)
    oproof, st = oracle.fri_prove(code, gp, ot)
    assert st == 0 and proof.serialize() == oproof.blob and proof.verify() == 0 and t.random() == ot.random()
    bad = oracle.synthetic(6, 1 << 8)  # random data is not a codeword: assert "not an RS code"
    with pytest.raises(ml.NotRsCode):
        ml.FriProof.prove(bad, None, ml.Transcript())
    with pytest.raises(ml.NotPowerOfTwo):
        ml.FriProverData.init(oracle.synthetic(1, 24), ml.Transcript())
    with pytest.raises(ml.SizeMismatch):
        ml.FriProof.prove(code, gp[:100], ml.Transcript())


def test_fri_verifier_rejects_tampered_proofs(ml, oracle):
    """every FriProofError of the reference's verifier (src/fri/mod.rs:251-258, 287-340) is reachable through the C ABI:
    a proof is serialised, one field is changed, and the re-read proof must fail with the matching ML_V_* code"""
    from multilinear_b200._lib import MlError
    log_n = 9
    coeffs = oracle.synthetic(41, 1 << log_n)
    proof = ml.FriProof.prove_from_coeffs(coeffs, ml.Transcript())
    blob = bytearray(proof.serialize())
    assert ml.FriProof.deserialize(blob).verify() == 0 and ml.FriProof.deserialize(blob).serialize() == bytes(blob)
    nc = int.from_bytes(blob[0:8], "little")
    assert nc == log_n
    q0 = 8 + 32 * nc + 8                       # first query: u64 path count, then per path: pair (2 x 24 B), u64 len, len x 36 B
    sizes = []
    off = q0 + 8
    for j in range(nc):
        ln = int.from_bytes(blob[off + 48:off + 56], "little")
        sizes.append(56 + 36 * ln)
        off += sizes[-1]
    qlen = off - q0                            # all 128 queries have the same byte length
    # ML_V_INCLUSION_HASH (104): one byte of a sibling digest on the first path of the first query
    b = bytearray(blob); b[q0 + 8 + 56 + 5] ^= 1
    assert ml.FriProof.deserialize(b).verify() == 104
    # ... or of an opened value
    b = bytearray(blob); b[q0 + 8 + 8 + 3] ^= 1
    assert ml.FriProof.deserialize(b).verify() == 104
    # ML_V_INCLUSION_INDEX (105): two valid openings swapped — the hashes match their roots, the transcript asks for other indices
    b = bytearray(blob)
    a0, a1 = bytes(b[q0:q0 + qlen]), bytes(b[q0 + qlen:q0 + 2 * qlen])
    if a0 != a1:
        b[q0:q0 + qlen], b[q0 + qlen:q0 + 2 * qlen] = a1, a0
        assert ml.FriProof.deserialize(b).verify() == 105
    # ML_V_LAST_RANDOM (106): the recorded final transcript state
    b = bytearray(blob); b[-1] ^= 0x80
    assert ml.FriProof.deserialize(b).verify() == 106
    # a different last element: it is absorbed before the indices are drawn, so the openings no longer match the indices asked
    # for (105), or — should an index survive — the fold consistency check (101)
    b = bytearray(blob); b[-32 - 16] ^= 1
    assert ml.FriProof.deserialize(b).verify() in (101, 105)
    # a changed commitment changes every later challenge: rejected (which check fires first depends on the layer)
    b = bytearray(blob); b[8 + 32 * 2 + 7] ^= 1
    assert ml.FriProof.deserialize(b).verify() in (101, 104, 105)
    # ML_V_WRONG_NUM_PATHS (103): the commitment list is one short of the paths
    b = bytearray(blob[:8 + 32 * (nc - 1)] + blob[8 + 32 * nc:]); b[0:8] = (nc - 1).to_bytes(8, "little")
    assert ml.FriProof.deserialize(b).verify() == 103
    # ML_V_WRONG_NUM_QUERIES (102): 127 queries
    b = bytearray(blob[:q0 - 8] + (127).to_bytes(8, "little") + blob[q0 + qlen:])
    assert ml.FriProof.deserialize(b).verify() == 102
    with pytest.raises(MlError):
        ml.FriProof.deserialize(blob[:-3])     # truncated blob
    with pytest.raises(MlError):
        ml.FriProof.deserialize(bytes(blob) + b"\x00")


def test_univariate_interpolation_reference_test(ml, oracle):
    """interpolation_test (src/polynomials.rs:197-204) and PolynomialEvals::interpolate against the oracle"""
    evals = ml.PolynomialEvals(ml.from_i64([0, 1, 4, 8, 9, 3]))
    pol = evals.interpolate()
    assert np.array_equal(pol.evaluate_over_domain().evals, evals.evals)
    assert np.array_equal(pol.coeffs, oracle.interpolate(evals.evals))
    for n in (1, 2, 3, 4, 17, 64):
        e = oracle.synthetic(600 + n, n)
        c = ml.PolynomialEvals(e).interpolate()
        assert np.array_equal(c.coeffs, oracle.interpolate(e)), n
        assert np.array_equal(c.evaluate_over_domain().evals, e)
        assert c.evaluate(n - 1) == fe_ints(e)[n - 1]
    big = oracle.synthetic(5, 3000)
    got = ml.UnivariatePolynomial(big).evaluate_over_domain().evals
    for i in (0, 1, 2999):
        assert fe_ints(got[i:i + 1])[0] == P.poly_eval(fe_ints(big), i)


# ------------------------------------------------------------------ sumcheck
@pytest.mark.parametrize("nv", [1, 2, 5, 12, 13, 16])
def test_sumcheck_tables_and_rounds(ml, oracle, nv):
    rng = random.Random(nv)
    ev = oracle.synthetic(80 + nv, 1 << nv)
    inp = fe_arr([rng.randrange(M) for _ in range(nv)])
    s, os_ = ml.SumcheckTables.build_tables_for_pcs(inp, ev), oracle.sumcheck_build(inp, ev)
    for a, b in zip(s.tables(), os_.tables()):
        assert np.array_equal(a, b)
    for r in (1, 2, 3, rng.randrange(M)):
        assert s.partial_sum(r) == os_.partial_sum(r)
    claim = oracle.mle_evals_evaluate(ev, inp)
    t, ot = ml.Transcript(), oracle.transcript()
    nz, r, prev = s.compute_sumcheck_polynomial(2, claim, t)
    onz, orr, oprev = os_.compute_sumcheck_polynomial(2, claim, ot)
    assert (nz, r, prev) == (onz, orr, oprev) and s.height == os_.height()
    for a, b in zip(s.tables(), os_.tables()):
        assert np.array_equal(a, b)
    rr = rng.randrange(M)
    if s.height > 1:
        s.fold(rr), os_.fold(rr)
        for a, b in zip(s.tables(), os_.tables()):
            assert np.array_equal(a, b)
    s2, os2 = ml.SumcheckTables.build_tables_for_pcs(inp, ev), oracle.sumcheck_build(inp, ev)
    t, ot = ml.Transcript(), oracle.transcript()
    assert s2.compute_sumcheck_polynomials(1, t, claim) == os2.compute_sumcheck_polynomials(1, ot, claim)
    assert t.random() == ot.random()


def test_sumcheck_general_degree_and_errors(ml, oracle):
    ev = oracle.synthetic(3, 1 << 6)
    inp = fe_arr(list(range(3, 9)))
    s, os_ = ml.SumcheckTables.build_tables_for_pcs(inp, ev), oracle.sumcheck_build(inp, ev)
    t, ot = ml.Transcript(), oracle.transcript()
    assert s.compute_sumcheck_polynomial(3, 12345, t) == os_.compute_sumcheck_polynomial(3, 12345, ot)
    with pytest.raises(ml.SizeMismatch):
        ml.SumcheckTables.build_tables_for_pcs(inp[:5], ev)


# ------------------------------------------------------------------ PCS
def test_pcs_golden(ml, golden):
    g = golden["pcs_nv8"]
    nv = 8
    evals = ml.MultilinearPolynomialEvals(ml.from_i64([7 * i + 3 for i in range(1 << nv)]))
    inputs = ml.from_i64(range(nv))
    out = evals.evaluate(ml.to_ints(inputs))
    assert str(out) == g["output"]
    t = ml.Transcript()
    proof = ml.PCSProof.prove(inputs, out, evals, t)
    assert proof.fri_proof.commitments[0].hex() == g["root0"] and str(proof.fri_proof.last_elem) == g["last_elem"]
    assert [[str(c) for c in nz] for nz in proof.sumcheck_polynomials] == g["sumcheck"]
    assert sha(proof.fri_proof.serialize()) == g["blob_sha"] and t.random().hex() == g["final_random"]
    assert proof.verify(ml.Transcript()) == 0


@pytest.mark.parametrize("nv", [1, 2, 3, 9, 13, 16])
def test_pcs_prove_vs_oracle(ml, oracle, nv):
    rng = random.Random(nv)
    ev = oracle.synthetic(90 + nv, 1 << nv)
    inp = fe_arr([rng.randrange(M) for _ in range(nv)])
    out = oracle.mle_evals_evaluate(ev, inp)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = ml.PCSProof.prove(inp, out, ev, t)
    oproof, st = oracle.pcs_prove(inp, out, ev, ot)
    assert st == 0
    assert proof.fri_proof.serialize() == oproof.fri.blob
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck
    assert t.random() == ot.random()
    assert proof.verify(ml.Transcript()) == 0 and oproof.verify(oracle.transcript()) == 0
    wrong = ml.PCSProof.prove(inp, (out + 1) % M, ev, ml.Transcript())  # a false claim must not verify
    assert wrong.verify(ml.Transcript()) == 107


def test_pcs_reference_test_inputs_n20(ml, oracle):
    """multilinear_pcs_bench_test (multilinear_pcs.rs:211-228): n_vars = 20, evals 7i+3, inputs i — BASELINE config 1"""
    nv = 20
    ev = ml.from_i64([7 * i + 3 for i in range(1 << nv)])
    inp = ml.from_i64(range(nv))
    out = ml.MultilinearPolynomialEvals(ev).evaluate(ml.to_ints(inp))
    t, ot = ml.Transcript(), oracle.transcript()
    proof = ml.PCSProof.prove(inp, out, ev, t)
    assert proof.verify(ml.Transcript()) == 0
    oproof, st = oracle.pcs_prove(inp, out, ev, ot)
    assert st == 0 and hashlib.sha256(proof.fri_proof.serialize()).digest() == hashlib.sha256(oproof.fri.blob).digest()
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck and t.random() == ot.random()


# ------------------------------------------------------------------ batched
def test_batched_golden(ml, golden):
    g = golden["bfri_log6_b4"]
    gp = ml.pow_2_generator_powers(7)
    gen = ml.to_ints(gp[1:2])[0]
    codes = [ml.reed_solomon(ml.from_i64([7 * i + 3 + 100 * j for i in range(64)]), gen) for j in range(4)]
    proof = ml.BatchedFriProof.prove(codes, gp, ml.Transcript())
    assert proof.batch_commitment.hex() == g["batch_commitment"] and [c.hex() for c in proof.commitments] == g["commitments"]
    assert str(proof.last_elem) == g["last_elem"] and sha(proof.serialize()) == g["blob_sha"] and proof.verify() == 0

    g = golden["bpcs_nv6_b10"]
    nv, B = 6, 10
    polys = [fe_arr([(j * 3 + i * 5) % 100 for j in range(1 << nv)]) for i in range(B)]
    inputs = ml.from_i64(range(nv))
    outputs = [ml.MultilinearPolynomialEvals(p).evaluate(ml.to_ints(inputs)) for p in polys]
    assert [str(o) for o in outputs] == g["outputs"]
    proof = ml.BatchedPCSProof.prove(inputs, outputs, polys, ml.Transcript())
    assert proof.fri_proof.batch_commitment.hex() == g["batch_commitment"]
    assert [[str(c) for c in nz] for nz in proof.sumcheck_polynomials] == g["sumcheck"]
    assert sha(proof.fri_proof.serialize()) == g["blob_sha"] and proof.verify(ml.Transcript()) == 0


def test_batched_fri_prover_data_stepwise(ml, oracle):
    """BatchedFriProverData::{init, batched_fold_step, fold, open_query_at} (batched_fri.rs:41-225) one call at a time with the
    host transcript, as `fold` (:183-205) sequences them: roots, last element, transcript and openings must equal those of the
    one-call prover (whose proof is compared with the oracle's)"""
    log_n, B = 7, 5
    n = 1 << (log_n + 1)
    gp = oracle.pow2_generator_powers(log_n + 1)
    gen = fe_ints(gp[1:2])[0]
    codes = [oracle.reed_solomon(oracle.synthetic(4000 + j, 1 << log_n), gen) for j in range(B)]
    t = ml.Transcript()
    d = ml.BatchedFriProverData.init(codes, t)
    r = t.next_challenge()
    d.batched_fold_step(gp, r, t)
    for k in range(1, log_n):
        r = t.next_challenge()
        d.fri_data.fold_step(gp, k, r, t)
    t2 = ml.Transcript()
    d2 = ml.BatchedFriProverData.fold(gp, codes, t2)      # the same on the device transcript
    assert d.fri_data.fold_roots() == d2.fri_data.fold_roots() and d.fri_data.last_element == d2.fri_data.last_element is not None
    assert d.batch_root() == d2.batch_root() and d.fingerprint_r == d2.fingerprint_r and t.random() == t2.random()
    ot = oracle.transcript()
    oproof, st = oracle.batched_fri_prove(codes, gp, ot)
    assert st == 0
    proof = ml.BatchedFriProof.prove(codes, gp, ml.Transcript())
    assert proof.serialize() == oproof.blob
    assert proof.batch_commitment == d.batch_root() and proof.commitments == d.fri_data.fold_roots() and proof.last_elem == d.fri_data.last_element
    bp, paths = d.open_query_at(37)
    bp2, paths2 = d2.open_query_at(37)
    assert (bp, paths) == (bp2, paths2) and len(bp[0]) == 32 * B and len(bp[1]) == log_n and len(paths) == log_n - 1
    assert ml.path_verify(bp[0], bp[1], d.batch_root(), 37) == 0
    sub = 37 % (n // 4)
    assert paths == d.fri_data.open_query_at(sub)          # :217-218
    with pytest.raises(ml.MlError):
        d.open_query_at(n // 2)


@pytest.mark.parametrize("nv,B", [(2, 1), (3, 2), (5, 3), (10, 7), (12, 64), (14, 5)])
def test_batched_pcs_vs_oracle(ml, oracle, nv, B):
    rng = random.Random(nv * 100 + B)
    polys = [oracle.synthetic(1000 * B + j, 1 << nv) for j in range(B)]
    inp = fe_arr([rng.randrange(M) for _ in range(nv)])
    outs = fe_arr([oracle.mle_evals_evaluate(p, inp) for p in polys])
    t, ot = ml.Transcript(), oracle.transcript()
    proof = ml.BatchedPCSProof.prove(inp, outs, polys, t)
    oproof, st = oracle.batched_pcs_prove(inp, outs, polys, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck
    assert t.random() == ot.random() and proof.verify(ml.Transcript()) == 0


# ------------------------------------------------------------------ width-w sumcheck tables (System path, SURVEY §8f row 4)
@pytest.mark.parametrize("log_height", [4, 7, 13])
def test_wide_sumcheck_reference_sumcheck_test(ml, oracle, log_height):
    """the reference's sumcheck_test / sumcheck_high_bench (sumcheck.rs:342-398): pythagorean trace (width 4), two
    constraints under the constraint mask, sum 0; bit-exact against the oracle, and accepted by verify_sumcheck_debug"""
    from test_oracle import pythagorean_system, verify_sumcheck_debug
    matrix, row_point, terms, ot = pythagorean_system(oracle, log_height)
    o = oracle.wsumcheck_build(row_point, matrix, 4)
    o.set_composition(terms)
    g = ml.WideSumcheckTables.build(row_point, matrix, 4)
    g.set_composition(terms)
    gm, gd = g.tables()
    om, od = o.tables()
    assert np.array_equal(gm, om) and np.array_equal(gd, od)
    for r in (1, 2, 3, 0, M - 1, 123456789):
        assert g.partial_sum(r) == o.partial_sum(r)
    t = ml.Transcript()
    gp, grs = g.compute_sumcheck_polynomials(2, t, 0)
    op, ors = o.compute_sumcheck_polynomials(2, ot, 0)
    assert gp == op and grs == ors and g.height == 1
    assert t.random() == ot.random()
    assert verify_sumcheck_debug(oracle, oracle.transcript(), gp, 3, 0, matrix, 4, row_point, terms) == grs


def test_wide_sumcheck_fold_random_and_errors(ml, oracle):
    from multilinear_b200._lib import MlError
    nv, w = 9, 5
    matrix = oracle.synthetic(31, w << nv)
    row_point = oracle.synthetic(32, nv)
    terms = [(7, [0, 1, 2]), (M - 3, [4, 4]), (11, []), (5, [3])]  # degree 3, with a constant term
    o = oracle.wsumcheck_build(row_point, matrix, w)
    g = ml.WideSumcheckTables.build(row_point, matrix, w)
    o.set_composition(terms)
    g.set_composition(terms)
    for r in (5, M - 2, 1 << 100):
        assert g.partial_sum(r) == o.partial_sum(r)
        g.fold(r)
        o.fold(r)
        gm, gd = g.tables()
        om, od = o.tables()
        assert np.array_equal(gm, om) and np.array_equal(gd, od)
    t, ot = ml.Transcript(), oracle.transcript()
    assert g.compute_sumcheck_polynomials(3, t, 99) == o.compute_sumcheck_polynomials(3, ot, 99)
    with pytest.raises(MlError):
        g.set_composition([(1, [w])])  # column out of range
    with pytest.raises(MlError):
        ml.WideSumcheckTables.build(row_point, matrix[:w * 100], w)  # height not 2^n_vars


def test_snark_test_system_sumcheck_then_pcs(ml, oracle):
    """the reference's snark_test (src/fri/multilinear_pcs.rs:279-316): System sumcheck over a width-1 trace with the
    zero constraint, then PCSProof::prove at the sumcheck's random point on the SAME transcript; the verifier replays the
    sumcheck (verify_with_evaluations, sumcheck.rs:92-124) and verifies the PCS proof.  2^16 rows (the reference uses 2^20)."""
    from test_oracle import PYTHAGOREAN
    log_h = 16
    rows = list(PYTHAGOREAN)
    while len(rows) < 1 << log_h:
        rows = rows + rows
    evals = fe_arr(rows)                                   # Trace::new(trace, 1)
    t, ot = ml.Transcript(), oracle.transcript()
    c = ot.next_challenge()                                # ChallengeSet::new: every challenge equals this value
    assert t.next_challenge() == c
    row_point = fe_arr([c] * log_h)
    terms = [(0, [])]                                      # constraint_mask = [1], Expr = 0, degree 1 (:262-267)
    g = ml.WideSumcheckTables.build(row_point, evals, 1)
    o = oracle.wsumcheck_build(row_point, evals, 1)
    g.set_composition(terms)
    o.set_composition(terms)
    gp, grs = g.compute_sumcheck_polynomials(1, t, 0)
    op, ors = o.compute_sumcheck_polynomials(1, ot, 0)
    assert gp == op and grs == ors and not any(gp)
    inputs = fe_arr(grs)
    out = ml.MultilinearPolynomialEvals(evals).evaluate(grs)
    assert out == oracle.mle_evals_evaluate(evals, inputs)
    proof = ml.PCSProof.prove(inputs, out, evals, t)
    oproof, st = oracle.pcs_prove(inputs, out, evals, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob
    assert t.random() == ot.random()
    # verifier side: fresh transcript, replay the sumcheck absorbs / challenges, then the PCS verifier
    vt = ml.Transcript()
    assert vt.next_challenge() == c
    pol_r = 0
    for k in range(log_h):
        for cf in gp[2 * k:2 * k + 2]:
            vt.absorb(int(cf).to_bytes(16, "little"))
        assert vt.next_challenge() == grs[k]
    assert ml.delta_evaluate(row_point, inputs) * 0 % M == pol_r   # delta * composition == pol(r): 0 == 0
    assert proof.verify(vt) == 0


# ------------------------------------------------------------------ sharded batched commit (config 5), single GPU
@pytest.mark.parametrize("mode", ["serial", "pipelined", "p2p"])
def test_sharded_batch_commit_single_gpu(ml, oracle, mode):
    import torch
    from multilinear_b200.sharded import CudaBackend, sharded_batch_commit
    n, B = 1 << 10, 5
    polys = [oracle.synthetic(2000 + j, n) for j in range(B)]
    local = [torch.from_numpy(p.reshape(-1).copy()).cuda() for p in polys]
    root = sharded_batch_commit(local, n, B, CudaBackend(), None, mode=mode)  # p2p degrades to pipelined on one rank
    g = oracle.pow2_generator(11)
    datas = []
    for p in polys:
        code = oracle.reed_solomon(oracle.bit_reverse(oracle.to_coefficient(p)), g)
        datas.append(np.concatenate([code[:n], code[n:]], axis=1))
    assert root == oracle.merkle_batch_commit(datas).root()


# ------------------------------------------------------------------ sharded BatchedPCSProof::prove (ml_shard_*, config 5)
@pytest.mark.parametrize("world,nv,B", [(1, 6, 3), (2, 6, 4), (2, 10, 6), (4, 12, 8), (8, 13, 16), (8, 16, 8), (8, 4, 8), (16, 5, 16), (1, 2, 1)])
def test_sharded_batched_pcs_prove_virtual_ranks_vs_oracle(ml, oracle, world, nv, B):
    """G ranks hosted by one process on ONE GPU (virtual ranks, phases enqueued in lock step): the proof bytes, the sumcheck
    polynomials and the transcript equal the oracle's BatchedPCSProof::prove; so does the unsharded CUDA prover's proof"""
    rng = random.Random(world * 1000 + nv * 10 + B)
    polys = [oracle.synthetic(3000 * B + j, 1 << nv) for j in range(B)]
    inp = fe_arr([rng.randrange(M) for _ in range(nv)])
    outs = fe_arr([oracle.mle_evals_evaluate(p, inp) for p in polys])
    sh = ml.ShardedBatchedProver.single_process([0] * world, B, nv)
    t, ot = ml.Transcript(), oracle.transcript()
    proof = sh.prove(inp, outs, polys, t)
    oproof, st = oracle.batched_pcs_prove(inp, outs, polys, ot)
    assert st == 0 and proof.fri_proof.serialize() == oproof.fri.blob
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck
    assert t.random() == ot.random() and proof.verify(ml.Transcript()) == 0
    # a second call on the same handle (epoch 2) gives the same bytes
    t2 = ml.Transcript()
    assert sh.prove(inp, outs, polys, t2).fri_proof.serialize() == oproof.fri.blob and t2.random() == ot.random()
    sh.free()


def test_sharded_batch_commit_root_and_errors(ml, oracle):
    import ctypes as C
    from multilinear_b200._lib import MlError
    nv, B, world = 11, 8, 4
    n = 1 << nv
    polys = [oracle.synthetic(7000 + j, n) for j in range(B)]
    g = oracle.pow2_generator(nv + 1)
    datas = []
    for p in polys:
        code = oracle.reed_solomon(oracle.bit_reverse(oracle.to_coefficient(p)), g)
        datas.append(np.concatenate([code[:n], code[n:]], axis=1))
    want = oracle.merkle_batch_commit(datas).root()
    sh = ml.ShardedBatchedProver.single_process([0] * world, B, nv)
    bufs = [ml.DeviceBuffer.from_host(polys[j]) for j in sh.local_polys()]
    assert sh.batch_commit_dev([b.ptr.value for b in bufs]) == want
    assert sh.batch_commit_dev([b.ptr.value for b in bufs]) == want
    sh.free()
    with pytest.raises(MlError):
        ml.ShardedBatchedProver.single_process([0] * 3, B, nv)      # world must be a power of two
    with pytest.raises(MlError):
        ml.ShardedBatchedProver.single_process([0] * 4, 6, nv)      # polynomials must split evenly
    one = ml.ShardedBatchedProver.one_rank(1, 2, 0, 4, 6)           # a rank whose peers were never connected refuses to run
    with pytest.raises(MlError):
        one.batch_commit_dev([0, 0])
    one.free()


# ------------------------------------------------------------------ oracle parity AT the BASELINE sizes (configs 2-5)
# The oracle needs seconds per case on the box's host cores (all threads); every comparison is bit-exact.
@pytest.fixture(scope="module")
def big_oracle():
    import os
    from oracle import binding
    binding.build()
    return binding.Oracle(threads=os.cpu_count() or 1)


def test_atsize_config3_commit_2p24_roots_last_transcript(ml, big_oracle):
    """BASELINE configs[2]: reed_solomon + FriProverData::fold of 2^24 coefficients (seed 0xB200, bench.py's polynomial 0):
    all 24 layer roots, the last element and the final transcript state equal the oracle's (src/fri/mod.rs:136-145)"""
    O = big_oracle
    n = 1 << 24
    coeffs = O.synthetic(0xB200, n)
    gp = O.pow2_generator_powers(25)
    code = O.reed_solomon(coeffs, fe_ints(gp[1:2])[0])
    ot = O.transcript()
    of, st = O.fri_fold(gp, code, ot)
    assert st == 0
    dev = ml.synthetic_elements_dev(0xB200, n)
    t = ml.Transcript()
    f = ml.FriProverData.fold_from_coeffs_dev(dev, n, t)
    roots = f.fold_roots()
    assert len(roots) == 24 and roots == of.roots()
    assert f.last_element == of.last_element() and f.last_element is not None
    assert t.random() == ot.random()
    # the code itself (2^25 evaluations, the (9, 8, 8) pass plan) equals the oracle's, element for element
    assert np.array_equal(ml.reed_solomon(coeffs, ml.pow_2_generator(25)), code)


def test_atsize_config2_ntt_2p20_blowup2_forward_inverse(ml, big_oracle):
    """BASELINE configs[1]: standalone forward + inverse NTT, one polynomial of 2^20 coefficients with blowup 2"""
    O = big_oracle
    n = 1 << 20
    c = O.synthetic(0xB200, n)
    g = ml.pow_2_generator(21)
    code = ml.reed_solomon(c, g)
    want = O.reed_solomon(c, g)
    assert np.array_equal(code, want)
    back = ml.intt(code, g)
    assert np.array_equal(back, O.intt(want, g))
    assert np.array_equal(back[:n], c) and not back[n:].any()


def test_atsize_config4_sumcheck_2p24_all_rounds(ml, big_oracle):
    """BASELINE configs[3]: sumcheck over a 2^24-entry multilinear extension product f * eq (composition x[0]), all 24 rounds:
    every (c1, c2), every challenge and the transcript equal the oracle's (sumcheck.rs:147-202)"""
    O = big_oracle
    nv = 24
    ev = O.synthetic(0xB200, 1 << nv)
    inp = O.synthetic(0xB2000001, nv)
    claim = O.mle_evals_evaluate(ev, inp)
    assert ml.MultilinearPolynomialEvals(ev).evaluate(ml.to_ints(inp)) == claim
    t, ot = ml.Transcript(), O.transcript()
    s, os_ = ml.SumcheckTables.build_tables_for_pcs(inp, ev), O.sumcheck_build(inp, ev)
    got = s.compute_sumcheck_polynomials(1, t, claim)
    want = os_.compute_sumcheck_polynomials(1, ot, claim)
    assert len(got[0]) == 2 * nv and got == want
    assert t.random() == ot.random()


def test_atsize_pcs_prove_n_vars_24(ml, big_oracle):
    """PCSProof::prove at the metric's size (n_vars = 24): proof bytes, sumcheck polynomials and transcript equal the oracle's"""
    O = big_oracle
    nv = 24
    ev = O.synthetic(0xB200, 1 << nv)
    inp = O.synthetic(0xB2000001, nv)
    out = O.mle_evals_evaluate(ev, inp)
    t, ot = ml.Transcript(), O.transcript()
    proof = ml.PCSProof.prove(inp, out, ev, t)
    oproof, st = O.pcs_prove(inp, out, ev, ot)
    assert st == 0 and hashlib.sha256(proof.fri_proof.serialize()).digest() == hashlib.sha256(oproof.fri.blob).digest()
    assert [c for nz in proof.sumcheck_polynomials for c in nz] == oproof.sumcheck and t.random() == ot.random()
    assert proof.verify(ml.Transcript()) == 0


def oracle_batch_root_by_ranges(O, seeds, n, n_ranges=8):
    """Merkle::batch_commit root over the RS codes of polys synthetic(seed, n), computed range by range to bound memory:
    the tree over all leaves equals the tree over the roots of equal leaf ranges (merkle_tree/mod.rs:118-129)"""
    g = O.pow2_generator((n.bit_length() - 1) + 1)
    codes = [O.reed_solomon(O.bit_reverse(O.to_coefficient(O.synthetic(s, n))), g) for s in seeds]
    rows = n // n_ranges
    roots = []
    for r in range(n_ranges):
        datas = [np.concatenate([c[r * rows:(r + 1) * rows], c[n + r * rows:n + (r + 1) * rows]], axis=1) for c in codes]
        roots.append(O.merkle_batch_commit(datas).root())
    while len(roots) > 1:
        roots = [hashlib.sha256(roots[i] + roots[i + 1]).digest() for i in range(0, len(roots), 2)]
    return roots[0]


def test_atsize_config5_batch_root_64x2p22(ml, big_oracle):
    """BASELINE configs[4]: batch root of 64 polynomials of 2^22 evaluations (bench.py's seeds 5000 + j) equals the oracle's
    Merkle::batch_commit over the 64 RS codes; the committed fixture (tests/golden/gen_batch_root.py) must agree with both"""
    import json
    import os
    import torch
    from multilinear_b200.sharded import CudaBackend, sharded_batch_commit
    n, B = 1 << 22, 64
    want = oracle_batch_root_by_ranges(big_oracle, [5000 + j for j in range(B)], n)
    import ctypes as C
    from multilinear_b200 import load
    L = load()
    local = []
    for j in range(B):
        t = torch.empty(16 * n, dtype=torch.uint8, device="cuda")
        ml.check(L.ml_synthetic_elements_dev(C.c_uint64(5000 + j), C.c_size_t(n), C.c_void_p(t.data_ptr()),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        local.append(t)
    root = sharded_batch_commit(local, n, B, CudaBackend(), None, mode="serial")
    assert root == want
    # the C-ABI sharded prover with 8 virtual ranks on this GPU: same root through leaf-range subtrees + top levels
    sh = ml.ShardedBatchedProver.single_process([0] * 8, B, 22)
    assert sh.batch_commit_dev([local[j].data_ptr() for j in sh.local_polys()]) == want
    sh.free()
    fx = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "batch_root_64x2p22.json")))
    assert fx["root"] == want.hex() and fx["n_polys"] == B and fx["log_n"] == 22


# ------------------------------------------------------------------ full-size properties (BASELINE sizes; size-independent checks)
def test_fullsize_ntt_roundtrip_and_linearity_2p24(ml):
    n = 1 << 24
    a = ml.synthetic_elements_dev(11, n).elems()
    b = ml.synthetic_elements_dev(12, n).elems()
    g = ml.pow_2_generator(24)
    fa = ml.ntt(a, g)
    assert np.array_equal(ml.intt(fa, g), a)               # intt(ntt(p)) == p at the reference's benchmark size (ntt/mod.rs:182-201)
    fb = ml.ntt(b, g)
    assert np.array_equal(ml.ntt(ml.add(a, b), g), ml.add(fa, fb))  # linearity
    # X[0] = sum of coefficients, X[N/2] = alternating sum
    s = ml.polynomial_evaluate(a, 1)
    assert ml.to_ints(fa[0:1])[0] == s
    assert ml.to_ints(fa[n // 2:n // 2 + 1])[0] == ml.polynomial_evaluate(a, M - 1)


def test_fullsize_rs_code_is_evaluation_of_the_polynomial_2p24(ml):
    n = 1 << 24
    c = ml.synthetic_elements_dev(13, n).elems()
    g = ml.pow_2_generator(25)
    code = ml.reed_solomon(c, g)
    for k in (0, 1, 12345, (1 << 24) + 7, (1 << 25) - 1):   # code[k] = p(g^k)
        assert ml.to_ints(code[k:k + 1])[0] == ml.polynomial_evaluate(c, pow(g, k, M))
    # even-indexed evaluations are the size-n transform with the squared generator
    assert np.array_equal(code[::2], ml.ntt(c, ml.pow_2_generator(24)))


def test_fullsize_commit_prove_verify_2p22(ml):
    n = 1 << 22
    coeffs = ml.synthetic_elements_dev(14, n).elems()
    t = ml.Transcript()
    proof = ml.FriProof.prove_from_coeffs(coeffs, t)
    assert len(proof.commitments) == 22 and proof.verify() == 0   # accepted by the restated reference verifier
    # the last element of a correct fold chain is the evaluation f(r_0..r_{v-1}) of the multilinear extension whose
    # coefficients (in the reference's bit-reversed order) were encoded: check through a PCS proof at the same size
    nv = 22
    evals = ml.synthetic_elements_dev(15, n).elems()
    inp = ml.from_i64(range(3, 3 + nv))
    out = ml.MultilinearPolynomialEvals(evals).evaluate(ml.to_ints(inp))
    p = ml.PCSProof.prove(inp, out, evals, ml.Transcript())
    assert p.verify(ml.Transcript()) == 0


def test_maxsize_ntt_roundtrip_2p27_device_resident(ml):
    """2^27 elements (2 GiB per array), device resident: the (9, 9, 9) three-pass plan, whose pass 0 has no twiddle table.
    intt(ntt(x)) == x and intt(reed_solomon(c)) == c || 0, compared through Merkle roots (a checksum of checksums) so
    nothing but 32 bytes crosses PCIe.  The oracle comparisons at this size and the four-pass plans are in test_large_sizes.py."""
    import ctypes as C
    from multilinear_b200 import load
    L = load()
    log_n = 27
    n = 1 << log_n
    g = ml.pow_2_generator(log_n)
    gb = (C.c_uint8 * 16)(*g.to_bytes(16, "little"))
    x = ml.synthetic_elements_dev(21, n)
    y = ml.DeviceBuffer(16 * n)
    z = ml.DeviceBuffer(16 * n)
    ml.check(L.ml_ntt_dev(x.ptr, C.c_size_t(n), gb, y.ptr, None))
    ml.check(L.ml_intt_dev(y.ptr, C.c_size_t(n), gb, z.ptr, None))
    rx = ml.Merkle.commit_rs_code_dev(x, n).root()
    assert ml.Merkle.commit_rs_code_dev(z, n).root() == rx
    assert ml.Merkle.commit_rs_code_dev(y, n).root() != rx
    # RS encode of the first half (2^26 coefficients -> 2^27 evaluations), inverted, gives the coefficients and a zero half
    ml.check(L.ml_reed_solomon_dev(x.ptr, C.c_size_t(n // 2), gb, y.ptr, None))
    ml.check(L.ml_intt_dev(y.ptr, C.c_size_t(n), gb, z.ptr, None))
    head = z.to_host(16 * 4096).reshape(-1, 16)
    assert np.array_equal(head, x.to_host(16 * 4096).reshape(-1, 16))
    ml.check(L.ml_dev_download(C.c_void_p(head.ctypes.data), C.c_void_p(z.ptr.value + 16 * (n - 4096)), C.c_size_t(16 * 4096)))
    assert not head.any()
    for b in (x, y, z):
        b.free()


# ------------------------------------------------------------------ the reference's own tests on the C++ host mirror
def test_cpp_reference_tests(ml):
    import subprocess
    import __graft_entry__ as g
    exe = g.build_cpp_tests()
    p = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "all reference tests passed" in p.stdout


def test_c_example_pcs_prove(ml, golden):
    """examples/pcs_prove.c (plain C11 over the C ABI): the PCS golden vector at n_vars = 8 and an accepted proof"""
    import subprocess
    import __graft_entry__ as g
    exe = g.build_c_example()
    p = subprocess.run([exe, "8"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout + p.stderr
    assert "root_0 623d135873c76f2306354b0d146b44c42c649d3060eaa022b0c0a96a4e051de2" in p.stdout   # SURVEY.md §8c PCS vector
    assert "accepted" in p.stdout


def test_sharded_batch_commit_two_gpus_all_exchange_modes(ml):
    """config 5 on two ranks over NCCL / NVLink peer stores (skipped on a one-GPU box): every exchange mode must give the
    root of the single-GPU tree over all codes"""
    import json
    import os
    import socket
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tools", "sharded_commit_demo.py"), "16", "8", "serial,pipelined,p2p"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    lines = [json.loads(l) for l in p.stdout.splitlines() if l.startswith("{") and "batched_commit" in l]
    assert [l["mode"] for l in lines] == ["serial", "pipelined", "p2p"]
    assert all(l["matches_single_gpu"] is True and l["n_gpus"] == 2 for l in lines)
    assert len({l["root"] for l in lines}) == 1


def test_sharded_prove_two_processes_two_gpus_vs_oracle(ml):
    """ml_shard_* with one process per GPU (CUDA IPC arenas, NVLink stores, device flags) on two ranks: the proof equals the CPU
    oracle's BatchedPCSProof::prove byte for byte and both transcripts end in the same state.  Skipped on a one-GPU box: ranks
    that wait on each other must not share a GPU; the same protocol runs there as virtual ranks in lock step (tests above)."""
    import json
    import os
    import socket
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "tools", "sharded_prove_demo.py"), "14", "8", "oracle", "2"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    line = [json.loads(l) for l in p.stdout.splitlines() if l.startswith("{") and "sharded_batched_pcs_prove" in l][-1]
    assert line["n_gpus"] == 2 and line["matches_oracle"] is True and line["verifies"] is True and line["transcripts_agree"] is True
