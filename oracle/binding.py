"""ORACLE — TEST INFRASTRUCTURE ONLY.  ctypes binding of oracle/liboracle.so.

May be imported only from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product never imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

u8p = C.POINTER(C.c_uint8)


def build(force=False):
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("oracle.c", "sha256.c", "field.h", "sha256.h", "oracle.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(so):
            build()
        L = C.CDLL(so)
        vp, sz, i32 = C.c_void_p, C.c_size_t, C.c_int
        ptr_fns = ["or_transcript_new", "or_transcript_clone", "or_merkle_commit", "or_merkle_batch_commit", "or_fri_init",
                   "or_fri_fold", "or_fri_tree", "or_fri_prove", "or_sumcheck_build_tables_for_pcs", "or_wsumcheck_build", "or_pcs_prove",
                   "or_pcs_proof_fri", "or_batched_fri_prove", "or_batched_pcs_prove", "or_bpcs_proof_fri"]
        for f in ptr_fns:
            getattr(L, f).restype = vp
        for f in ["or_merkle_num_layers", "or_merkle_layer_len", "or_fri_num_trees", "or_fri_proof_serialized_len",
                  "or_fri_proof_num_commitments", "or_sumcheck_height", "or_wsumcheck_height", "or_pcs_proof_num_rounds",
                  "or_bfri_proof_serialized_len", "or_bfri_proof_num_commitments", "or_bpcs_proof_num_rounds"]:
            getattr(L, f).restype = sz
        # every pointer/size argument is passed explicitly typed by the helpers below
        _LIB = L
    return _LIB


def buf(a):
    """ctypes void* of a C-contiguous numpy array (kept alive by the caller)."""
    assert a.flags["C_CONTIGUOUS"]
    return C.c_void_p(a.ctypes.data)


def fe_arr(ints):
    """list of python ints -> (n,16) uint8 array of LE field elements"""
    out = np.empty((len(ints), 16), dtype=np.uint8)
    for i, x in enumerate(ints):
        out[i] = np.frombuffer(int(x).to_bytes(16, "little"), dtype=np.uint8)
    return out


def fe_ints(a):
    a = np.ascontiguousarray(a).reshape(-1, 16)
    return [int.from_bytes(a[i].tobytes(), "little") for i in range(a.shape[0])]


def fe1(x):
    return np.frombuffer(int(x).to_bytes(16, "little"), dtype=np.uint8).copy()


def fe_int(a):
    return int.from_bytes(np.ascontiguousarray(a).tobytes()[:16], "little")


def aligned_empty(nbytes, align=64):
    raw = np.empty(nbytes + align, dtype=np.uint8)
    off = (-raw.ctypes.data) % align
    return raw[off:off + nbytes]


def elems_empty(n):
    return aligned_empty(16 * n).reshape(n, 16)


sz = C.c_size_t


class Oracle:
    """Thin, typed convenience layer used by the tests and the CPU-baseline leg."""

    def __init__(self, threads=1):
        self.L = lib()
        self.L.or_set_threads(C.c_int(threads))

    def set_threads(self, n):
        self.L.or_set_threads(C.c_int(n))

    # --- field
    def binop(self, name, a, b):
        out = np.empty(16, dtype=np.uint8)
        xa, xb = fe1(a), fe1(b)
        getattr(self.L, "or_fe_" + name)(buf(xa), buf(xb), buf(out))
        return fe_int(out)

    def vec(self, name, a, b):
        out = elems_empty(a.shape[0])
        getattr(self.L, "or_fe_%s_vec" % name)(buf(a), buf(b), sz(a.shape[0]), buf(out))
        return out

    def synthetic(self, seed, n):
        out = elems_empty(n)
        self.L.or_synthetic_elements(C.c_uint64(seed), sz(n), buf(out))
        return out

    def from_i64(self, v):
        out = np.empty(16, dtype=np.uint8)
        self.L.or_fe_from_i64(C.c_int64(v), buf(out))
        return fe_int(out)

    # --- ntt
    def pow2_generator(self, log_size):
        out = np.empty(16, dtype=np.uint8)
        st = self.L.or_pow2_generator(C.c_uint64(log_size), buf(out))
        return None if st else fe_int(out)

    def pow2_generator_powers(self, log_size):
        out = elems_empty(1 << log_size)
        st = self.L.or_pow2_generator_powers(C.c_uint64(log_size), buf(out))
        return None if st else out

    def ntt(self, coeffs, gen):
        out = elems_empty(coeffs.shape[0])
        g = fe1(gen)
        st = self.L.or_ntt(buf(coeffs), sz(coeffs.shape[0]), buf(g), buf(out))
        assert st == 0, st
        return out

    def intt(self, evals, gen):
        out = elems_empty(evals.shape[0])
        g = fe1(gen)
        st = self.L.or_intt(buf(evals), sz(evals.shape[0]), buf(g), buf(out))
        assert st == 0, st
        return out

    def reed_solomon(self, coeffs, gen):
        out = elems_empty(2 * coeffs.shape[0])
        g = fe1(gen)
        st = self.L.or_reed_solomon(buf(coeffs), sz(coeffs.shape[0]), buf(g), buf(out))
        assert st == 0, st
        return out

    def interpolate(self, evals):
        out = elems_empty(evals.shape[0])
        self.L.or_interpolate(buf(evals), sz(evals.shape[0]), buf(out))
        return out

    def bit_reverse(self, a):
        a = np.ascontiguousarray(a).copy()
        self.L.or_bit_reverse_permutation(buf(a), sz(a.shape[0]), sz(a.shape[1]))
        return a

    # --- mle
    def to_coefficient(self, evals):
        out = elems_empty(evals.shape[0])
        self.L.or_mle_to_coefficient(buf(evals), sz(evals.shape[0]), buf(out))
        return out

    def to_evaluation(self, coeffs):
        out = elems_empty(coeffs.shape[0])
        self.L.or_mle_to_evaluation(buf(coeffs), sz(coeffs.shape[0]), buf(out))
        return out

    def mle_evals_evaluate(self, evals, args):
        out = np.empty(16, dtype=np.uint8)
        st = self.L.or_mle_evals_evaluate(buf(evals), sz(evals.shape[0]), buf(args), sz(args.shape[0]), buf(out))
        assert st == 0, st
        return fe_int(out)

    def mle_coeffs_evaluate(self, coeffs, args):
        out = np.empty(16, dtype=np.uint8)
        st = self.L.or_mle_coeffs_evaluate(buf(coeffs), sz(coeffs.shape[0]), buf(args), sz(args.shape[0]), buf(out))
        assert st == 0, st
        return fe_int(out)

    # --- sha / transcript
    def sha256(self, data):
        d = np.frombuffer(bytes(data), dtype=np.uint8) if len(data) else np.zeros(1, dtype=np.uint8)
        out = np.empty(32, dtype=np.uint8)
        self.L.or_sha256_oneshot(buf(d), sz(len(data)), buf(out))
        return out.tobytes()

    def transcript(self):
        return OrTranscript(self.L)

    # --- merkle
    def merkle_commit(self, data):
        """data: (n_items, item_bytes) uint8"""
        data = np.ascontiguousarray(data)
        h = self.L.or_merkle_commit(buf(data), sz(data.shape[1]), sz(data.shape[0]))
        return OrMerkle(self.L, h, data.shape[1]) if h else None

    def merkle_batch_commit(self, datas):
        datas = [np.ascontiguousarray(d) for d in datas]
        ptrs = (C.c_void_p * len(datas))(*[d.ctypes.data for d in datas])
        h = self.L.or_merkle_batch_commit(ptrs, sz(len(datas)), sz(datas[0].shape[1]), sz(datas[0].shape[0]))
        return OrMerkle(self.L, h, datas[0].shape[1] * len(datas)) if h else None


class OrTranscript:
    def __init__(self, L, h=None):
        self.L = L
        self.h = C.c_void_p(h if h is not None else L.or_transcript_new())

    def clone(self):
        return OrTranscript(self.L, self.L.or_transcript_clone(self.h))

    def absorb(self, b):
        b = bytes(b)
        d = np.frombuffer(b, dtype=np.uint8) if b else np.zeros(1, dtype=np.uint8)
        self.L.or_transcript_absorb(self.h, buf(d), sz(len(b)))

    def random(self):
        out = np.empty(32, dtype=np.uint8)
        self.L.or_transcript_random(self.h, buf(out))
        return out.tobytes()

    def next_challenge(self):
        out = np.empty(16, dtype=np.uint8)
        self.L.or_transcript_next_challenge(self.h, buf(out))
        return fe_int(out)

    def __del__(self):
        try:
            self.L.or_transcript_free(self.h)
        except Exception:
            pass


class OrMerkle:
    def __init__(self, L, h, value_bytes, owned=True):
        self.L, self.h, self.value_bytes, self.owned = L, C.c_void_p(h), value_bytes, owned

    def root(self):
        out = np.empty(32, dtype=np.uint8)
        self.L.or_merkle_root(self.h, buf(out))
        return out.tobytes()

    def layers(self):
        res = []
        for l in range(self.L.or_merkle_num_layers(self.h)):
            n = self.L.or_merkle_layer_len(self.h, sz(l))
            out = np.empty((n, 32), dtype=np.uint8)
            self.L.or_merkle_layer(self.h, sz(l), buf(out))
            res.append(out)
        return res

    def open(self, index):
        value = np.empty(self.value_bytes, dtype=np.uint8)
        digs = np.empty((64, 32), dtype=np.uint8)
        dirs = np.empty(64, dtype=np.uint8)
        n = sz(0)
        st = self.L.or_merkle_open(self.h, sz(index), buf(value), buf(digs), buf(dirs), C.byref(n))
        if st:
            return None
        return value.tobytes(), [(digs[i].tobytes(), int(dirs[i])) for i in range(n.value)]

    def __del__(self):
        if self.owned:
            try:
                self.L.or_merkle_free(self.h)
            except Exception:
                pass


def _blob(L, h, prefix):
    n = getattr(L, prefix + "_serialized_len")(h)
    out = np.empty(max(n, 1), dtype=np.uint8)
    getattr(L, prefix + "_serialize")(h, buf(out))
    return out[:n].tobytes()


class OrFriProof:
    """commitments / last_elem / last_random / blob of an or_fri_proof (borrowed or owned)."""

    def __init__(self, L, h, owned=True, prefix="or_fri_proof", free="or_fri_proof_free"):
        self.L, self.h, self.owned, self._free = L, C.c_void_p(h), owned, free
        n = getattr(L, prefix + "_num_commitments")(self.h)
        c = np.empty((max(n, 1), 32), dtype=np.uint8)
        getattr(L, prefix + "_commitments")(self.h, buf(c))
        self.commitments = [c[i].tobytes() for i in range(n)]
        le, lr = np.empty(16, dtype=np.uint8), np.empty(32, dtype=np.uint8)
        getattr(L, prefix + "_last")(self.h, buf(le), buf(lr))
        self.last_elem, self.last_random = fe_int(le), lr.tobytes()
        self.blob = _blob(L, self.h, prefix)
        if prefix == "or_bfri_proof":
            bc = np.empty(32, dtype=np.uint8)
            L.or_bfri_proof_batch_commitment(self.h, buf(bc))
            self.batch_commitment = bc.tobytes()

    def verify(self):
        return self.L.or_fri_verify(self.h) if self._free == "or_fri_proof_free" else self.L.or_batched_fri_verify(self.h)

    def __del__(self):
        if self.owned:
            try:
                getattr(self.L, self._free)(self.h)
            except Exception:
                pass


class OrFri:
    """FriProverData (src/fri/mod.rs:10-14) handle."""

    def __init__(self, L, h):
        self.L, self.h = L, C.c_void_p(h)

    def fold_step(self, gen_pows, k, r, t):
        rb = fe1(r)
        return self.L.or_fri_fold_step(self.h, buf(gen_pows), sz(gen_pows.shape[0]), sz(k), buf(rb), t.h)

    def num_trees(self):
        return self.L.or_fri_num_trees(self.h)

    def roots(self):
        n = self.num_trees()
        out = np.empty((max(n, 1), 32), dtype=np.uint8)
        self.L.or_fri_fold_roots(self.h, buf(out))
        return [out[i].tobytes() for i in range(n)]

    def tree(self, i):
        return OrMerkle(self.L, self.L.or_fri_tree(self.h, sz(i)), 32, owned=False)

    def tree_data(self, i):
        n = self.L.or_merkle_layer_len(C.c_void_p(self.L.or_fri_tree(self.h, sz(i))), sz(0))
        out = np.empty((n, 32), dtype=np.uint8)
        self.L.or_fri_tree_data(self.h, sz(i), buf(out))
        return out

    def last_element(self):
        out = np.empty(16, dtype=np.uint8)
        return fe_int(out) if self.L.or_fri_last_element(self.h, buf(out)) else None

    def __del__(self):
        try:
            self.L.or_fri_free(self.h)
        except Exception:
            pass



def composition_arrays(terms):
    """[(coef int, [cols...]), ...] -> (coefs (n,16) u8, lens u32, cols u32): the sparse-polynomial form of a composition"""
    coefs = fe_arr([c for c, _ in terms]) if terms else np.empty((0, 16), dtype=np.uint8)
    lens = np.array([len(cs) for _, cs in terms], dtype=np.uint32)
    cols = np.array([c for _, cs in terms for c in cs] or [0], dtype=np.uint32)
    return np.ascontiguousarray(coefs), np.ascontiguousarray(lens), np.ascontiguousarray(cols)


class OrWSumcheck:
    """width-w SumcheckTables (System path), composition = sparse polynomial over the row"""

    def __init__(self, L, h, width):
        self.L, self.h, self.width = L, C.c_void_p(h), width

    def height(self):
        return self.L.or_wsumcheck_height(self.h)

    def set_composition(self, terms):
        coefs, lens, cols = composition_arrays(terms)
        assert self.L.or_wsumcheck_set_composition(self.h, sz(len(terms)), buf(coefs), buf(lens), buf(cols)) == 0

    def tables(self):
        n = self.height()
        m, d = elems_empty(n * self.width), elems_empty(n)
        self.L.or_wsumcheck_tables(self.h, buf(m), buf(d))
        return m, d

    def partial_sum(self, r):
        out, rb = np.empty(16, dtype=np.uint8), fe1(r)
        self.L.or_wsumcheck_partial_sum(self.h, buf(rb), buf(out))
        return fe_int(out)

    def fold(self, r):
        rb = fe1(r)
        self.L.or_wsumcheck_fold(self.h, buf(rb))

    def compute_sumcheck_polynomials(self, composition_degree, t, s):
        n = (self.height()).bit_length() - 1
        td = composition_degree + 1
        sb, co, rs = fe1(s), np.empty((max(n, 1) * td, 16), dtype=np.uint8), np.empty((max(n, 1), 16), dtype=np.uint8)
        self.L.or_wsumcheck_compute_polynomials(self.h, sz(composition_degree), t.h, buf(sb), buf(co), buf(rs))
        return fe_ints(co[:n * td]), fe_ints(rs[:n])

    def __del__(self):
        try:
            self.L.or_wsumcheck_free(self.h)
        except Exception:
            pass


class OrSumcheck:
    def __init__(self, L, h):
        self.L, self.h = L, C.c_void_p(h)

    def height(self):
        return self.L.or_sumcheck_height(self.h)

    def tables(self):
        n = self.height()
        m, d = elems_empty(n), elems_empty(n)
        self.L.or_sumcheck_tables(self.h, buf(m), buf(d))
        return m, d

    def partial_sum(self, r):
        out, rb = np.empty(16, dtype=np.uint8), fe1(r)
        self.L.or_sumcheck_partial_sum(self.h, buf(rb), buf(out))
        return fe_int(out)

    def fold(self, r):
        rb = fe1(r)
        self.L.or_sumcheck_fold(self.h, buf(rb))

    def compute_sumcheck_polynomial(self, total_degree, previous_sum, t):
        prev, co, r = fe1(previous_sum), np.empty((max(total_degree, 1), 16), dtype=np.uint8), np.empty(16, dtype=np.uint8)
        st = self.L.or_sumcheck_compute_polynomial(self.h, sz(total_degree), buf(prev), t.h, buf(co), buf(r))
        if st:
            raise ValueError("or_sumcheck_compute_polynomial: status %d (total_degree %d)" % (st, total_degree))
        return fe_ints(co[:total_degree]), fe_int(r), fe_int(prev)

    def compute_sumcheck_polynomials(self, composition_degree, t, s):
        n = (self.height()).bit_length() - 1
        td = composition_degree + 1
        sb, co, rs = fe1(s), np.empty((max(n, 1) * td, 16), dtype=np.uint8), np.empty((max(n, 1), 16), dtype=np.uint8)
        self.L.or_sumcheck_compute_polynomials(self.h, sz(composition_degree), t.h, buf(sb), buf(co), buf(rs))
        return fe_ints(co[:n * td]), fe_ints(rs[:n])

    def __del__(self):
        try:
            self.L.or_sumcheck_free(self.h)
        except Exception:
            pass


class OrPcsProof:
    def __init__(self, L, h, batched=False):
        self.L, self.h, self.batched = L, C.c_void_p(h), batched
        p = "or_bpcs_proof" if batched else "or_pcs_proof"
        fri_h = getattr(L, p + "_fri")(self.h)
        self.fri = OrFriProof(L, fri_h, owned=False, prefix="or_bfri_proof" if batched else "or_fri_proof",
                              free="or_bfri_proof_free" if batched else "or_fri_proof_free")
        n = getattr(L, p + "_num_rounds")(self.h)
        co = np.empty((max(n, 1) * 2, 16), dtype=np.uint8)
        getattr(L, p + "_sumcheck_coeffs")(self.h, buf(co))
        self.sumcheck = fe_ints(co[:2 * n])

    def verify(self, t):
        return (self.L.or_batched_pcs_verify if self.batched else self.L.or_pcs_verify)(self.h, t.h)

    def __del__(self):
        try:
            (self.L.or_bpcs_proof_free if self.batched else self.L.or_pcs_proof_free)(self.h)
        except Exception:
            pass


def _ptr_array(arrs):
    return (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])


def _ext(cls):
    def fri_init(self, code, t):
        h = self.L.or_fri_init(buf(code), sz(code.shape[0]), t.h)
        return OrFri(self.L, h) if h else None

    def fri_fold(self, gen_pows, code, t):
        st = C.c_int(0)
        h = self.L.or_fri_fold(buf(gen_pows), sz(gen_pows.shape[0]), buf(code), sz(code.shape[0]), t.h, C.byref(st))
        return (OrFri(self.L, h) if h else None), st.value

    def fri_prove(self, code, gen_pows, t):
        st = C.c_int(0)
        h = self.L.or_fri_prove(buf(code), sz(code.shape[0]), buf(gen_pows), sz(gen_pows.shape[0]), t.h, C.byref(st))
        return (OrFriProof(self.L, h) if h else None), st.value

    def sumcheck_build(self, inputs, evals):
        h = self.L.or_sumcheck_build_tables_for_pcs(buf(inputs), sz(inputs.shape[0]), buf(evals), sz(evals.shape[0]))
        return OrSumcheck(self.L, h) if h else None

    def wsumcheck_build(self, row_point, matrix, width):
        """matrix: (height*width, 16) row-major trace; row_point: (n_vars, 16)"""
        height = matrix.shape[0] // width
        h = self.L.or_wsumcheck_build(buf(row_point), sz(row_point.shape[0]), buf(matrix), sz(width), sz(height))
        return OrWSumcheck(self.L, h, width) if h else None

    def trace_evaluate(self, matrix, width, points):
        height = matrix.shape[0] // width
        out = np.empty((width, 16), dtype=np.uint8)
        self.L.or_trace_evaluate(buf(matrix), sz(width), sz(height), buf(points), buf(out))
        return fe_ints(out)

    def mask_evaluate(self, index, points):
        out = np.empty(16, dtype=np.uint8)
        self.L.or_mask_evaluate(sz(index), sz(points.shape[0]), buf(points), buf(out))
        return fe_int(out)

    def delta_evaluate(self, data, points):
        out = np.empty(16, dtype=np.uint8)
        self.L.or_delta_evaluate(buf(data), buf(points), sz(data.shape[0]), buf(out))
        return fe_int(out)

    def pcs_prove(self, inputs, output, evals, t):
        st, ob = C.c_int(0), fe1(output)
        h = self.L.or_pcs_prove(buf(inputs), sz(inputs.shape[0]), buf(ob), buf(evals), sz(evals.shape[0]), t.h, C.byref(st))
        return (OrPcsProof(self.L, h) if h else None), st.value

    def fingerprint(self, r, coeffs):
        out, rb = np.empty(16, dtype=np.uint8), fe1(r)
        self.L.or_fingerprint(buf(rb), buf(coeffs), sz(coeffs.shape[0]), buf(out))
        return fe_int(out)

    def batched_fri_prove(self, codes, gen_pows, t):
        st = C.c_int(0)
        ptrs = _ptr_array(codes)
        h = self.L.or_batched_fri_prove(ptrs, sz(len(codes)), sz(codes[0].shape[0]), buf(gen_pows), sz(gen_pows.shape[0]),
                                        t.h, C.byref(st))
        if not h:
            return None, st.value
        return OrFriProof(self.L, h, prefix="or_bfri_proof", free="or_bfri_proof_free"), st.value

    def batched_pcs_prove(self, inputs, outputs, polys, t):
        st = C.c_int(0)
        ptrs = _ptr_array(polys)
        h = self.L.or_batched_pcs_prove(buf(inputs), sz(inputs.shape[0]), buf(outputs), sz(len(polys)), ptrs,
                                        sz(polys[0].shape[0]), t.h, C.byref(st))
        return (OrPcsProof(self.L, h, batched=True) if h else None), st.value

    for f in (fri_init, fri_fold, fri_prove, sumcheck_build, wsumcheck_build, trace_evaluate, mask_evaluate, delta_evaluate, pcs_prove, fingerprint, batched_fri_prove,
              batched_pcs_prove):
        setattr(cls, f.__name__, f)


_ext(Oracle)
