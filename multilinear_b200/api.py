"""Host-side mirror of the reference's public interface for the PCS hot path, on top of the C ABI.

Names, argument meaning and error behaviour follow fr34za/multilinear (citations relative to /root/reference/):
the reference's panics become exceptions (NotPowerOfTwo, SizeMismatch, NotRsCode), `None` stays `None`.
Field elements cross as (n, 16) uint8 numpy arrays of little-endian canonical u128 (src/field.rs:33-38);
helpers convert from / to Python ints.  All array work runs in the CUDA library — nothing here computes on the CPU
beyond packing bytes.
"""
import ctypes as C

import numpy as np

from ._lib import MlError, NotPowerOfTwo, NotRsCode, SizeMismatch, check, load  # noqa: F401

M = 340282366920938463463374557953744961537  # src/ntt/mod.rs:35
LOG_BLOWUP = 1      # src/fri/mod.rs:16
NUM_QUERIES = 128   # src/fri/mod.rs:17
_sz = C.c_size_t


# ----------------------------------------------------------------------------- element packing
def _p(a):
    return C.c_void_p(a.ctypes.data)


def aligned_empty(nbytes, align=64):
    raw = np.empty(nbytes + align, dtype=np.uint8)
    off = (-raw.ctypes.data) % align
    return raw[off:off + nbytes]


def elems_empty(n):
    return aligned_empty(16 * n).reshape(n, 16)


def as_elems(x):
    """ints / (n,16) uint8 array -> aligned C-contiguous (n,16) uint8 array"""
    if isinstance(x, np.ndarray) and x.dtype == np.uint8:
        x = x.reshape(-1, 16)
        if x.flags["C_CONTIGUOUS"] and x.ctypes.data % 16 == 0:
            return x
        out = elems_empty(x.shape[0])
        out[:] = x
        return out
    xs = list(x)
    out = elems_empty(len(xs))
    for i, v in enumerate(xs):
        out[i] = np.frombuffer(int(v).to_bytes(16, "little"), dtype=np.uint8)
    return out


def to_ints(a):
    a = np.ascontiguousarray(a).reshape(-1, 16)
    return [int.from_bytes(a[i].tobytes(), "little") for i in range(a.shape[0])]


def _fe1(x):
    if isinstance(x, np.ndarray):
        return np.ascontiguousarray(x.reshape(16)).copy()
    return np.frombuffer(int(x).to_bytes(16, "little"), dtype=np.uint8).copy()


def _int(a):
    return int.from_bytes(np.ascontiguousarray(a).tobytes()[:16], "little")


def from_wide(values, variant=2):
    """256-bit integers -> v mod M through the device reduction (fe_reduce_wide_v1 / _v2)"""
    vs = list(values)
    buf = aligned_empty(32 * max(len(vs), 1))
    for i, v in enumerate(vs):
        buf[32 * i:32 * i + 32] = np.frombuffer(int(v).to_bytes(32, "little"), dtype=np.uint8)
    out = elems_empty(len(vs))
    check(load().ml_fe_from_wide_vec(_p(buf), _sz(len(vs)), C.c_int(variant), _p(out)))
    return to_ints(out)


def from_i64(values):
    """Field128::from(i64) for a list of ints (src/field.rs:150-154), on the GPU"""
    v = np.asarray(list(values), dtype=np.int64)
    out = elems_empty(len(v))
    check(load().ml_fe_from_i64_vec(_p(v), _sz(len(v)), _p(out)))
    return out


def _vec(name, a, b=None):
    a = as_elems(a)
    out = elems_empty(a.shape[0])
    if b is None:
        check(getattr(load(), name)(_p(a), _sz(a.shape[0]), _p(out)))
    else:
        b = as_elems(b)
        check(getattr(load(), name)(_p(a), _p(b), _sz(a.shape[0]), _p(out)))
    return out


def add(a, b):
    return _vec("ml_fe_add_vec", a, b)


def sub(a, b):
    return _vec("ml_fe_sub_vec", a, b)


def mul(a, b):
    return _vec("ml_fe_mul_vec", a, b)


def inv(a):
    return _vec("ml_fe_inv_vec", a)


def pow_(a, e):
    a = as_elems(a)
    out, eb = elems_empty(a.shape[0]), np.frombuffer(int(e).to_bytes(16, "little"), dtype=np.uint8).copy()
    check(load().ml_fe_pow_vec(_p(a), _p(eb), _sz(a.shape[0]), _p(out)))
    return out


# ----------------------------------------------------------------------------- device helpers
def device_count():
    n = C.c_int(0)
    check(load().ml_device_count(C.byref(n)))
    return n.value


def set_device(i):
    check(load().ml_set_device(C.c_int(i)))


def synchronize():
    check(load().ml_synchronize())


def kernel_launches():
    return int(load().ml_kernel_launches())


class DeviceBuffer:
    """Raw HBM allocation for callers that keep data resident between calls."""

    def __init__(self, nbytes):
        self.nbytes = nbytes
        p = C.c_void_p()
        check(load().ml_dev_alloc(_sz(nbytes), C.byref(p)))
        self.ptr = p

    @staticmethod
    def from_host(arr):
        arr = np.ascontiguousarray(arr)
        b = DeviceBuffer(arr.nbytes)
        check(load().ml_dev_upload(b.ptr, _p(arr), _sz(arr.nbytes)))
        return b

    def to_host(self, nbytes=None):
        n = self.nbytes if nbytes is None else nbytes
        out = aligned_empty(n)
        check(load().ml_dev_download(_p(out), self.ptr, _sz(n)))
        return out

    def elems(self):
        return self.to_host().reshape(-1, 16)

    def free(self):
        if self.ptr:
            load().ml_dev_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def synthetic_elements_dev(seed, n, stream=None):
    b = DeviceBuffer(16 * n)
    check(load().ml_synthetic_elements_dev(C.c_uint64(seed), _sz(n), b.ptr, C.c_void_p(stream)))
    return b


# ----------------------------------------------------------------------------- NTT (src/ntt/mod.rs)
def pow_2_generator(log_size):
    out = np.empty(16, dtype=np.uint8)
    st = load().ml_pow2_generator(C.c_uint64(log_size), _p(out))
    if st == 3:
        return None
    check(st)
    return _int(out)


def pow_2_generator_powers(log_size):
    if log_size > 40:
        return None
    out = elems_empty(1 << log_size)
    check(load().ml_pow2_generator_powers(C.c_uint64(log_size), _p(out)))
    return out


def bit_reverse_permutation(values):
    v = as_elems(values).copy()
    check(load().ml_bit_reverse_permutation(_p(v), _sz(v.shape[0]), _sz(16)))
    return v


def ntt(coeffs, gen):
    """Polynomial::ntt (src/ntt/mod.rs:69-110)"""
    c, g = as_elems(coeffs), _fe1(gen)
    out = elems_empty(c.shape[0])
    check(load().ml_ntt(_p(c), _sz(c.shape[0]), _p(g), _p(out)))
    return out


def intt(evals, gen):
    """LagrangePolynomial::intt (src/ntt/mod.rs:132-173)"""
    e, g = as_elems(evals), _fe1(gen)
    out = elems_empty(e.shape[0])
    check(load().ml_intt(_p(e), _sz(e.shape[0]), _p(g), _p(out)))
    return out


def reed_solomon(coeffs, gen):
    """reed_solomon (src/fri/mod.rs:19-28)"""
    c, g = as_elems(coeffs), _fe1(gen)
    out = elems_empty(c.shape[0] << LOG_BLOWUP)
    check(load().ml_reed_solomon(_p(c), _sz(c.shape[0]), _p(g), _p(out)))
    return out


def polynomial_evaluate(coeffs, x):
    c, xb, out = as_elems(coeffs), _fe1(x), np.empty(16, dtype=np.uint8)
    check(load().ml_poly_evaluate(_p(c), _sz(c.shape[0]), _p(xb), _p(out)))
    return _int(out)


# ----------------------------------------------------------------------------- multilinear polynomials (src/polynomials.rs)
class PolynomialEvals:
    """src/polynomials.rs:45-86 — evaluations over the domain 0..n-1"""

    def __init__(self, evals):
        self.evals = as_elems(evals)

    def interpolate(self):
        out = elems_empty(self.evals.shape[0])
        check(load().ml_poly_interpolate(_p(self.evals), _sz(self.evals.shape[0]), _p(out)))
        return UnivariatePolynomial(out)


class UnivariatePolynomial:
    """src/polynomials.rs:3-28 (`Polynomial<F>` of that module)"""

    def __init__(self, coeffs):
        self.coeffs = as_elems(coeffs)

    def evaluate(self, x):
        return polynomial_evaluate(self.coeffs, x)

    def evaluate_over_domain(self):
        out = elems_empty(self.coeffs.shape[0])
        check(load().ml_poly_evaluate_over_domain(_p(self.coeffs), _sz(self.coeffs.shape[0]), _p(out)))
        return PolynomialEvals(out)


class MultilinearPolynomialEvals:
    def __init__(self, evals):
        self.evals = as_elems(evals)

    def to_coefficient(self):
        out = elems_empty(self.evals.shape[0])
        check(load().ml_mle_to_coefficient(_p(self.evals), _sz(self.evals.shape[0]), _p(out)))
        return MultilinearPolynomial(out)

    def evaluate(self, args):
        a, out = as_elems(args), np.empty(16, dtype=np.uint8)
        check(load().ml_mle_evals_evaluate(_p(self.evals), _sz(self.evals.shape[0]), _p(a), _sz(a.shape[0]), _p(out)))
        return _int(out)


class MultilinearPolynomial:
    def __init__(self, coeffs):
        self.coeffs = as_elems(coeffs)

    def to_evaluation(self):
        out = elems_empty(self.coeffs.shape[0])
        check(load().ml_mle_to_evaluation(_p(self.coeffs), _sz(self.coeffs.shape[0]), _p(out)))
        return MultilinearPolynomialEvals(out)

    def evaluate(self, args):
        a, out = as_elems(args), np.empty(16, dtype=np.uint8)
        check(load().ml_mle_coeffs_evaluate(_p(self.coeffs), _sz(self.coeffs.shape[0]), _p(a), _sz(a.shape[0]), _p(out)))
        return _int(out)


# ----------------------------------------------------------------------------- transcript (src/transcript.rs)
class Transcript:
    def __init__(self, _h=None):
        if _h is None:
            _h = C.c_void_p()
            check(load().ml_transcript_new(C.byref(_h)))
        self.h = _h

    def clone(self):
        h = C.c_void_p()
        check(load().ml_transcript_clone(self.h, C.byref(h)))
        return Transcript(h)

    def absorb(self, values):
        b = bytes(values)
        d = np.frombuffer(b, dtype=np.uint8) if b else np.zeros(1, dtype=np.uint8)
        check(load().ml_transcript_absorb(self.h, _p(d), _sz(len(b))))

    def random(self):
        out = np.empty(32, dtype=np.uint8)
        check(load().ml_transcript_random(self.h, _p(out)))
        return out.tobytes()

    def next_challenge(self):
        out = np.empty(16, dtype=np.uint8)
        check(load().ml_transcript_next_challenge(self.h, _p(out)))
        return _int(out)

    def __del__(self):
        try:
            load().ml_transcript_free(self.h)
        except Exception:
            pass


# ----------------------------------------------------------------------------- Merkle (src/merkle_tree/mod.rs)
class Merkle:
    def __init__(self, h, value_bytes, owned=True):
        self.h, self.value_bytes, self.owned = h, value_bytes, owned

    @staticmethod
    def commit(data):
        """data: (n_items, item_bytes) uint8 — Merkle::commit (:65-85)"""
        d = np.ascontiguousarray(data, dtype=np.uint8)
        h = C.c_void_p()
        check(load().ml_merkle_commit(_p(d), _sz(d.shape[1]), _sz(d.shape[0]), C.byref(h)))
        return Merkle(h, d.shape[1])

    @staticmethod
    def batch_commit(datas):
        """datas: list of (n_items, item_bytes) uint8 — Merkle::batch_commit (:92-131)"""
        ds = [np.ascontiguousarray(d, dtype=np.uint8) for d in datas]
        if not ds:
            raise SizeMismatch(2, "Data must not be empty")
        if any(d.shape != ds[0].shape for d in ds):
            raise SizeMismatch(2, "All batches must have the same length")
        ptrs = (C.c_void_p * len(ds))(*[d.ctypes.data for d in ds])
        h = C.c_void_p()
        check(load().ml_merkle_batch_commit(ptrs, _sz(len(ds)), _sz(ds[0].shape[1]), _sz(ds[0].shape[0]), C.byref(h)))
        return Merkle(h, ds[0].shape[1] * len(ds))

    @staticmethod
    def commit_rs_code_dev(code_buf, n, stream=None):
        h = C.c_void_p()
        check(load().ml_merkle_commit_rs_code_dev(code_buf.ptr, _sz(n), C.c_void_p(stream), C.byref(h)))
        m = Merkle(h, 32)
        m._keep = code_buf
        return m

    def root(self):
        out = np.empty(32, dtype=np.uint8)
        check(load().ml_merkle_root(self.h, _p(out)))
        return out.tobytes()

    @property
    def layers(self):
        L = load()
        res = []
        for l in range(L.ml_merkle_num_layers(self.h)):
            n = L.ml_merkle_layer_len(self.h, _sz(l))
            out = np.empty((n, 32), dtype=np.uint8)
            check(L.ml_merkle_layer(self.h, _sz(l), _p(out)))
            res.append(out)
        return res

    def open(self, index):
        """-> (value bytes, [(digest, direction)]) or None (:31-58, :134-175)"""
        value = np.empty(max(self.value_bytes, 1), dtype=np.uint8)
        digs, dirs, n = np.empty((64, 32), dtype=np.uint8), np.empty(64, dtype=np.uint8), _sz(0)
        st = load().ml_merkle_open(self.h, _sz(index), _p(value), _p(digs), _p(dirs), C.byref(n))
        if st == 3:
            return None
        check(st)
        return value[:self.value_bytes].tobytes(), [(digs[i].tobytes(), int(dirs[i])) for i in range(n.value)]

    batch_open = open

    def __del__(self):
        if self.owned:
            try:
                load().ml_merkle_free(self.h)
            except Exception:
                pass


def path_verify(value, path, root, index):
    """MerkleInclusionPath::verify / batch_verify (:216-293); returns 0 or an ML_V_* code"""
    v = np.frombuffer(bytes(value), dtype=np.uint8)
    digs = np.frombuffer(b"".join(d for d, _ in path), dtype=np.uint8) if path else np.zeros(1, dtype=np.uint8)
    dirs = np.array([d for _, d in path] or [0], dtype=np.uint8)
    r = np.frombuffer(bytes(root), dtype=np.uint8)
    return load().ml_merkle_path_verify(_p(v), _sz(len(value)), _p(digs), _p(dirs), _sz(len(path)), _p(r), _sz(index))


# ----------------------------------------------------------------------------- FRI (src/fri/mod.rs)
class FriProof:
    def __init__(self, h, owned=True, batched=False):
        self.h, self.owned, self.batched = h, owned, batched
        L, p = load(), ("ml_bfri_proof" if batched else "ml_fri_proof")
        n = getattr(L, p + "_num_commitments")(self.h)
        c = np.empty((max(n, 1), 32), dtype=np.uint8)
        check(getattr(L, p + "_commitments")(self.h, _p(c)))
        self.commitments = [c[i].tobytes() for i in range(n)]
        le, lr = np.empty(16, dtype=np.uint8), np.empty(32, dtype=np.uint8)
        check(getattr(L, p + "_last")(self.h, _p(le), _p(lr)))
        self.last_elem, self.last_random = _int(le), lr.tobytes()
        if batched:
            bc = np.empty(32, dtype=np.uint8)
            check(L.ml_bfri_proof_batch_commitment(self.h, _p(bc)))
            self.batch_commitment = bc.tobytes()

    @staticmethod
    def prove(code, gen_pows, transcript):
        """FriProof::prove (:261-285)"""
        c = as_elems(code)
        gp = as_elems(gen_pows) if gen_pows is not None else None
        h = C.c_void_p()
        check(load().ml_fri_prove(_p(c), _sz(c.shape[0]), _p(gp) if gp is not None else None,
                                  _sz(gp.shape[0] if gp is not None else 0), transcript.h, C.byref(h)))
        return FriProof(h)

    @staticmethod
    def prove_from_coeffs(coeffs, transcript):
        """reed_solomon + FriProof::prove with the code kept in HBM (ml_rs_fri_prove)"""
        c = as_elems(coeffs)
        h = C.c_void_p()
        check(load().ml_rs_fri_prove(_p(c), _sz(c.shape[0]), transcript.h, C.byref(h)))
        return FriProof(h)

    @staticmethod
    def deserialize(blob):
        """a FriProof from its bincode bytes (fri/mod.rs:367-397) — e.g. one made by the Rust crate"""
        b = np.frombuffer(bytes(blob), dtype=np.uint8).copy()
        h = C.c_void_p()
        check(load().ml_fri_proof_deserialize(_p(b), _sz(len(b)), C.byref(h)))
        return FriProof(h)

    def verify(self):
        return load().ml_batched_fri_verify(self.h) if self.batched else load().ml_fri_verify(self.h)

    def serialize(self):
        L, p = load(), ("ml_bfri_proof" if self.batched else "ml_fri_proof")
        n = getattr(L, p + "_serialized_len")(self.h)
        out = np.empty(max(n, 1), dtype=np.uint8)
        check(getattr(L, p + "_serialize")(self.h, _p(out)))
        return out[:n].tobytes()

    def __del__(self):
        if self.owned:
            try:
                (load().ml_bfri_proof_free if self.batched else load().ml_fri_proof_free)(self.h)
            except Exception:
                pass


class FriProverData:
    def __init__(self, h, owned=True, keep=None):
        self.h, self.owned, self._keep = h, owned, keep  # keep: the owner of a borrowed handle

    @staticmethod
    def init(code, transcript):
        c = as_elems(code)
        h = C.c_void_p()
        check(load().ml_fri_init(_p(c), _sz(c.shape[0]), transcript.h, C.byref(h)))
        return FriProverData(h)

    def fold_step(self, gen_pows, k, r, transcript):
        gp = as_elems(gen_pows) if gen_pows is not None else None
        rb = _fe1(r)
        check(load().ml_fri_fold_step(self.h, _p(gp) if gp is not None else None, _sz(gp.shape[0] if gp is not None else 0),
                                      _sz(k), _p(rb), transcript.h))

    @staticmethod
    def fold(gen_pows, code, transcript):
        c = as_elems(code)
        gp = as_elems(gen_pows) if gen_pows is not None else None
        h = C.c_void_p()
        check(load().ml_fri_fold(_p(gp) if gp is not None else None, _sz(gp.shape[0] if gp is not None else 0), _p(c),
                                 _sz(c.shape[0]), transcript.h, C.byref(h)))
        return FriProverData(h)

    @staticmethod
    def fold_from_coeffs_dev(coeffs_buf, n, transcript, stream=None):
        h = C.c_void_p()
        check(load().ml_rs_fri_fold_dev(coeffs_buf.ptr, _sz(n), transcript.h, C.c_void_p(stream), C.byref(h)))
        return FriProverData(h)

    def num_trees(self):
        return load().ml_fri_num_trees(self.h)

    def fold_roots(self):
        n = self.num_trees()
        out = np.empty((max(n, 1), 32), dtype=np.uint8)
        check(load().ml_fri_fold_roots(self.h, _p(out)))
        return [out[i].tobytes() for i in range(n)]

    def tree(self, i):
        h = C.c_void_p()
        check(load().ml_fri_tree(self.h, _sz(i), C.byref(h)))
        return Merkle(h, 32, owned=False)

    def tree_data(self, i):
        n = load().ml_merkle_layer_len(self.tree(i).h, _sz(0))
        out = np.empty((n, 32), dtype=np.uint8)
        check(load().ml_fri_tree_data(self.h, _sz(i), _p(out)))
        return out

    @property
    def last_element(self):
        out, some = np.empty(16, dtype=np.uint8), C.c_int(0)
        check(load().ml_fri_last_element(self.h, _p(out), C.byref(some)))
        return _int(out) if some.value else None

    def open_query_at(self, index):
        nt = self.num_trees()
        values, digs = np.empty((nt, 32), dtype=np.uint8), np.empty((nt * 48 + 1, 32), dtype=np.uint8)
        dirs, lens = np.empty(nt * 48 + 1, dtype=np.uint8), (C.c_size_t * max(nt, 1))()
        check(load().ml_fri_open_query_at(self.h, _sz(index), _p(values), _p(digs), _p(dirs), lens))
        paths, off = [], 0
        for j in range(nt):
            n = lens[j]
            paths.append((values[j].tobytes(), [(digs[off + i].tobytes(), int(dirs[off + i])) for i in range(n)]))
            off += n
        return paths

    def __del__(self):
        try:
            if self.owned:
                load().ml_fri_free(self.h)
        except Exception:
            pass


class BatchedFriProverData:
    """BatchedFriProverData (src/fri/batched_fri.rs:9-14, 41-225) step by step"""

    def __init__(self, h, n_codes, n):
        self.h, self.n_codes, self.n = h, n_codes, n

    @staticmethod
    def _codes(codes):
        cs = [as_elems(c) for c in codes]
        return cs, (C.c_void_p * len(cs))(*[c.ctypes.data for c in cs])

    @staticmethod
    def init(codes, transcript):
        cs, ptrs = BatchedFriProverData._codes(codes)
        h = C.c_void_p()
        check(load().ml_bfri_init(ptrs, _sz(len(cs)), _sz(cs[0].shape[0] if cs else 0), transcript.h, C.byref(h)))
        return BatchedFriProverData(h, len(cs), cs[0].shape[0])

    @staticmethod
    def fold(gen_pows, codes, transcript):
        cs, ptrs = BatchedFriProverData._codes(codes)
        gp = as_elems(gen_pows) if gen_pows is not None else None
        h = C.c_void_p()
        check(load().ml_bfri_fold(_p(gp) if gp is not None else None, _sz(gp.shape[0] if gp is not None else 0), ptrs, _sz(len(cs)),
                                  _sz(cs[0].shape[0] if cs else 0), transcript.h, C.byref(h)))
        return BatchedFriProverData(h, len(cs), cs[0].shape[0])

    def batched_fold_step(self, gen_pows, r, transcript):
        gp = as_elems(gen_pows) if gen_pows is not None else None
        rb = _fe1(r)
        check(load().ml_bfri_batched_fold_step(self.h, _p(gp) if gp is not None else None, _sz(gp.shape[0] if gp is not None else 0), _p(rb), transcript.h))

    @property
    def fri_data(self):
        load().ml_bfri_fri_data.restype = C.c_void_p
        return FriProverData(C.c_void_p(load().ml_bfri_fri_data(self.h)), owned=False, keep=self)

    @property
    def fingerprint_r(self):
        out = np.empty(16, dtype=np.uint8)
        check(load().ml_bfri_fingerprint_r(self.h, _p(out)))
        return _int(out)

    def batch_root(self):
        load().ml_bfri_batch_layer.restype = C.c_void_p
        return Merkle(C.c_void_p(load().ml_bfri_batch_layer(self.h)), 32 * self.n_codes, owned=False).root()

    def open_query_at(self, index):
        nt = self.fri_data.num_trees()
        depth = max((self.n // 2).bit_length() - 1, 0)
        bvals, bdigs = np.empty((self.n_codes, 32), dtype=np.uint8), np.empty((depth + 1, 32), dtype=np.uint8)
        bdirs, blen = np.empty(depth + 1, dtype=np.uint8), C.c_size_t(0)
        values, digs = np.empty((max(nt, 1), 32), dtype=np.uint8), np.empty((nt * 48 + 1, 32), dtype=np.uint8)
        dirs, lens = np.empty(nt * 48 + 1, dtype=np.uint8), (C.c_size_t * max(nt, 1))()
        check(load().ml_bfri_open_query_at(self.h, _sz(index), _p(bvals), _p(bdigs), _p(bdirs), C.byref(blen), _p(values), _p(digs), _p(dirs), lens))
        batch_path = (bvals.tobytes(), [(bdigs[i].tobytes(), int(bdirs[i])) for i in range(blen.value)])
        paths, off = [], 0
        for j in range(nt):
            k = lens[j]
            paths.append((values[j].tobytes(), [(digs[off + i].tobytes(), int(dirs[off + i])) for i in range(k)]))
            off += k
        return batch_path, paths

    def __del__(self):
        try:
            load().ml_bfri_free(self.h)
        except Exception:
            pass


# ----------------------------------------------------------------------------- sumcheck (src/constraint_system/sumcheck.rs:127-277)
class SumcheckTables:
    def __init__(self, h):
        self.h = h

    @staticmethod
    def build_tables_for_pcs(inputs, poly):
        i, e = as_elems(inputs), (poly.evals if isinstance(poly, MultilinearPolynomialEvals) else as_elems(poly))
        h = C.c_void_p()
        check(load().ml_sumcheck_build_tables_for_pcs(_p(i), _sz(i.shape[0]), _p(e), _sz(e.shape[0]), C.byref(h)))
        return SumcheckTables(h)

    @property
    def height(self):
        return load().ml_sumcheck_height(self.h)

    def tables(self):
        n = self.height
        m, d = elems_empty(n), elems_empty(n)
        check(load().ml_sumcheck_tables(self.h, _p(m), _p(d)))
        return m, d

    def partial_sum(self, r):
        rb, out = _fe1(r), np.empty(16, dtype=np.uint8)
        check(load().ml_sumcheck_partial_sum(self.h, _p(rb), _p(out)))
        return _int(out)

    def fold(self, r):
        rb = _fe1(r)
        check(load().ml_sumcheck_fold(self.h, _p(rb)))

    def compute_sumcheck_polynomial(self, total_degree, previous_sum, transcript):
        """-> (nonzero_coeffs, r, new previous_sum)  (:174-202)"""
        prev, co, r = _fe1(previous_sum), np.empty((max(total_degree, 1), 16), dtype=np.uint8), np.empty(16, dtype=np.uint8)
        check(load().ml_sumcheck_compute_polynomial(self.h, _sz(total_degree), _p(prev), transcript.h, _p(co), _p(r)))
        return to_ints(co[:total_degree]), _int(r), _int(prev)

    def compute_sumcheck_polynomials(self, composition_degree, transcript, s):
        """-> (flat nonzero coeffs, randoms)  (:147-172)"""
        n, td = self.height.bit_length() - 1, composition_degree + 1
        sb, co, rs = _fe1(s), np.empty((max(n, 1) * td, 16), dtype=np.uint8), np.empty((max(n, 1), 16), dtype=np.uint8)
        check(load().ml_sumcheck_compute_polynomials(self.h, _sz(composition_degree), transcript.h, _p(sb), _p(co), _p(rs)))
        return to_ints(co[:n * td]), to_ints(rs[:n])

    def __del__(self):
        try:
            load().ml_sumcheck_free(self.h)
        except Exception:
            pass


class WideSumcheckTables:
    """SumcheckTables of arbitrary trace width as built by System::build_tables (src/constraint_system/sumcheck.rs:22-38).
    The composition closure of the reference (`&impl Fn(&[F]) -> F`) is given as the sparse polynomial it computes over a
    row: a list of (coefficient, [column, column, ...]) terms."""

    def __init__(self, h, width):
        self.h, self.width = h, width

    @staticmethod
    def build(row_point, matrix, width):
        """matrix: (height*width) elements, row-major; row_point: n_vars elements (ChallengeSet::row)"""
        rp, m = as_elems(row_point), as_elems(matrix)
        h = C.c_void_p()
        check(load().ml_wsumcheck_build(_p(rp), _sz(rp.shape[0]), _p(m), _sz(width), _sz(m.shape[0] // width), C.byref(h)))
        return WideSumcheckTables(h, width)

    def set_composition(self, terms):
        coefs = as_elems([c for c, _ in terms]) if terms else elems_empty(1)[:0]
        lens = np.ascontiguousarray([len(cs) for _, cs in terms], dtype=np.uint32)
        cols = np.ascontiguousarray([c for _, cs in terms for c in cs] or [0], dtype=np.uint32)
        check(load().ml_wsumcheck_set_composition(self.h, _sz(len(terms)), _p(coefs), _p(lens), _p(cols)))

    @property
    def height(self):
        return load().ml_wsumcheck_height(self.h)

    def tables(self):
        n = self.height
        m, d = elems_empty(n * self.width), elems_empty(n)
        check(load().ml_wsumcheck_tables(self.h, _p(m), _p(d)))
        return m, d

    def partial_sum(self, r):
        rb, out = _fe1(r), np.empty(16, dtype=np.uint8)
        check(load().ml_wsumcheck_partial_sum(self.h, _p(rb), _p(out)))
        return _int(out)

    def fold(self, r):
        rb = _fe1(r)
        check(load().ml_wsumcheck_fold(self.h, _p(rb)))

    def compute_sumcheck_polynomials(self, composition_degree, transcript, s):
        """-> (flat nonzero coeffs, randoms)  (:147-202)"""
        n, td = self.height.bit_length() - 1, composition_degree + 1
        sb, co, rs = _fe1(s), np.empty((max(n, 1) * td, 16), dtype=np.uint8), np.empty((max(n, 1), 16), dtype=np.uint8)
        check(load().ml_wsumcheck_compute_polynomials(self.h, _sz(composition_degree), transcript.h, _p(sb), _p(co), _p(rs)))
        return to_ints(co[:n * td]), to_ints(rs[:n])

    def __del__(self):
        try:
            load().ml_wsumcheck_free(self.h)
        except Exception:
            pass


def delta_evaluate(data, points):
    d, p, out = as_elems(data), as_elems(points), np.empty(16, dtype=np.uint8)
    check(load().ml_delta_evaluate(_p(d), _p(p), _sz(d.shape[0]), _p(out)))
    return _int(out)


# ----------------------------------------------------------------------------- PCS (src/fri/multilinear_pcs.rs, batched_*.rs)
class PCSProof:
    def __init__(self, h, batched=False):
        self.h, self.batched = h, batched
        L, p = load(), ("ml_bpcs_proof" if batched else "ml_pcs_proof")
        self.fri_proof = FriProof(C.c_void_p(getattr(L, p + "_fri")(self.h)), owned=False, batched=batched)
        n = getattr(L, p + "_num_rounds")(self.h)
        co = np.empty((max(n, 1) * 2, 16), dtype=np.uint8)
        check(getattr(L, p + "_sumcheck_coeffs")(self.h, _p(co)))
        flat = to_ints(co[:2 * n])
        self.sumcheck_polynomials = [flat[2 * i:2 * i + 2] for i in range(n)]

    @staticmethod
    def prove(inputs, output, poly, transcript):
        """PCSProof::prove (:90-136)"""
        i, o = as_elems(inputs), _fe1(output)
        e = poly.evals if isinstance(poly, MultilinearPolynomialEvals) else as_elems(poly)
        h = C.c_void_p()
        check(load().ml_pcs_prove(_p(i), _sz(i.shape[0]), _p(o), _p(e), _sz(e.shape[0]), transcript.h, C.byref(h)))
        return PCSProof(h)

    @staticmethod
    def prove_dev(inputs, output, evals_buf, n, transcript, stream=None):
        i, o = as_elems(inputs), _fe1(output)
        h = C.c_void_p()
        check(load().ml_pcs_prove_dev(_p(i), _sz(i.shape[0]), _p(o), evals_buf.ptr, _sz(n), transcript.h, C.c_void_p(stream), C.byref(h)))
        return PCSProof(h)

    def verify(self, transcript):
        return (load().ml_batched_pcs_verify if self.batched else load().ml_pcs_verify)(self.h, transcript.h)

    def __del__(self):
        try:
            (load().ml_bpcs_proof_free if self.batched else load().ml_pcs_proof_free)(self.h)
        except Exception:
            pass


class BatchedFriProof:
    @staticmethod
    def prove(codes, gen_pows, transcript):
        """BatchedFriProof::prove (batched_fri.rs:286-318)"""
        cs = [as_elems(c) for c in codes]
        if not cs:
            raise SizeMismatch(2, "Codes must not be empty")
        if any(c.shape != cs[0].shape for c in cs):
            raise SizeMismatch(2, "All codes must have the same size")
        gp = as_elems(gen_pows) if gen_pows is not None else None
        ptrs = (C.c_void_p * len(cs))(*[c.ctypes.data for c in cs])
        h = C.c_void_p()
        check(load().ml_batched_fri_prove(ptrs, _sz(len(cs)), _sz(cs[0].shape[0]), _p(gp) if gp is not None else None,
                                          _sz(gp.shape[0] if gp is not None else 0), transcript.h, C.byref(h)))
        return FriProof(h, batched=True)


def fingerprint(r, coeffs):
    rb, c, out = _fe1(r), as_elems(coeffs), np.empty(16, dtype=np.uint8)
    check(load().ml_fingerprint(_p(rb), _p(c), _sz(c.shape[0]), _p(out)))
    return _int(out)


class BatchedPCSProof:
    @staticmethod
    def prove(claim_inputs, claim_outputs, polys, transcript):
        """BatchedPCSProof::prove (batched_pcs.rs:130-180); claim = (inputs, outputs)"""
        i, o = as_elems(claim_inputs), as_elems(claim_outputs)
        ps = [p.evals if isinstance(p, MultilinearPolynomialEvals) else as_elems(p) for p in polys]
        ptrs = (C.c_void_p * len(ps))(*[p.ctypes.data for p in ps])
        h = C.c_void_p()
        check(load().ml_batched_pcs_prove(_p(i), _sz(i.shape[0]), _p(o), _sz(len(ps)), ptrs, _sz(ps[0].shape[0] if ps else 0),
                                          transcript.h, C.byref(h)))
        return PCSProof(h, batched=True)


class ShardedBatchedProver:
    """BatchedPCSProof::prove sharded over the GPUs of one box (ml_shard_*, csrc/shard.cu).  A handle hosts the ranks of one
    process: all of them (single_process; devices may repeat = virtual ranks on one GPU) or one (one_rank; the records of all
    processes are all-gathered by the caller's transport and passed to connect)."""

    def __init__(self, h, world, local_ranks, n_polys, n_vars):
        self.h, self.world, self.local_ranks, self.n_polys, self.n_vars = h, world, list(local_ranks), n_polys, n_vars

    @staticmethod
    def _create(world, ranks, devices, n_polys, n_vars):
        h = C.c_void_p()
        ra, da = (C.c_int * len(ranks))(*ranks), (C.c_int * len(devices))(*devices)
        check(load().ml_shard_create(C.c_int(world), C.c_int(len(ranks)), ra, da, _sz(n_polys), _sz(n_vars), C.byref(h)))
        return ShardedBatchedProver(h, world, ranks, n_polys, n_vars)

    @staticmethod
    def single_process(devices, n_polys, n_vars):
        return ShardedBatchedProver._create(len(devices), list(range(len(devices))), list(devices), n_polys, n_vars)

    @staticmethod
    def one_rank(rank, world, device, n_polys, n_vars):
        return ShardedBatchedProver._create(world, [rank], [device], n_polys, n_vars)

    def export(self):
        out = np.empty(72 * len(self.local_ranks), dtype=np.uint8)
        check(load().ml_shard_export(self.h, _p(out)))
        return out.tobytes()

    def connect(self, records):
        buf = np.frombuffer(bytes(records), dtype=np.uint8).copy()
        check(load().ml_shard_connect(self.h, _p(buf), _sz(len(buf) // 72)))

    def connect_over(self, dist, device):
        """all-gather the IPC records over a torch.distributed process group (the only use of the collective library)"""
        import torch
        mine = torch.tensor(list(self.export()), dtype=torch.uint8, device=device)
        allr = [torch.empty_like(mine) for _ in range(dist.get_world_size())]
        dist.all_gather(allr, mine)
        self.connect(b"".join(bytes(r.cpu().numpy().tobytes()) for r in allr))

    def stream(self, local_index=0):
        return load().ml_shard_stream(self.h, C.c_int(local_index))

    def phase_ms(self):
        """device time between the phase marks of the last call (instrumentation, multilinear_b200_instr.h)"""
        out = (C.c_double * 16)()
        n = load().ml_shard_phase_ms(self.h, out, C.c_int(16))
        return [out[i] for i in range(n)]

    def local_polys(self):
        """global polynomial indices in the order local_evals must be given: for each local rank, rank, rank + world, ..."""
        return [r + l * self.world for r in self.local_ranks for l in range(self.n_polys // self.world)]

    def batch_commit_dev(self, local_evals_ptrs):
        ptrs = (C.c_void_p * len(local_evals_ptrs))(*local_evals_ptrs)
        root = np.empty(32, dtype=np.uint8)
        check(load().ml_shard_batch_commit_dev(self.h, ptrs, _p(root)))
        return root.tobytes()

    def prove_dev(self, claim_inputs, claim_outputs, local_evals_ptrs, transcript):
        i, o = as_elems(claim_inputs), as_elems(claim_outputs)
        ptrs = (C.c_void_p * len(local_evals_ptrs))(*local_evals_ptrs)
        h = C.c_void_p()
        check(load().ml_shard_batched_pcs_prove_dev(self.h, _p(i), _sz(i.shape[0]), _p(o), _sz(o.shape[0]), ptrs, transcript.h, C.byref(h)))
        return PCSProof(h, batched=True) if h.value else None

    def prove(self, claim_inputs, claim_outputs, polys, transcript):
        """host arrays for all polynomials (needs a single-process handle) — the drop-in for batched_pcs.rs:130"""
        i, o = as_elems(claim_inputs), as_elems(claim_outputs)
        ps = [p.evals if isinstance(p, MultilinearPolynomialEvals) else as_elems(p) for p in polys]
        ptrs = (C.c_void_p * len(ps))(*[p.ctypes.data for p in ps])
        h = C.c_void_p()
        check(load().ml_shard_batched_pcs_prove(self.h, _p(i), _sz(i.shape[0]), _p(o), _sz(len(ps)), ptrs, transcript.h, C.byref(h)))
        return PCSProof(h, batched=True)

    def free(self):
        if self.h is not None and self.h.value:
            load().ml_shard_free(self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class BlockShardedBatchedProver:
    """BatchedPCSProof::prove with every polynomial split by block over the GPUs of one box (ml_bpcs_shard_*,
    csrc/bpcs_shard.cu).  Rank g holds the block evals_j[g*n/G, (g+1)*n/G) of every polynomial j, so any batch size works on any
    power-of-two G.  Handles as for ShardedPCSProver: single_process (devices may repeat = virtual ranks on one GPU) or one_rank
    with connect / connect_over.  The proof is an ordinary batched PCSProof, byte-identical to BatchedPCSProof.prove's."""

    def __init__(self, h, world, local_ranks, n_polys, n_vars):
        self.h, self.world, self.local_ranks, self.n_polys, self.n_vars = h, world, list(local_ranks), n_polys, n_vars

    @staticmethod
    def _create(world, ranks, devices, n_polys, n_vars):
        h = C.c_void_p()
        ra, da = (C.c_int * len(ranks))(*ranks), (C.c_int * len(devices))(*devices)
        check(load().ml_bpcs_shard_create(C.c_int(world), C.c_int(len(ranks)), ra, da, _sz(n_polys), _sz(n_vars), C.byref(h)))
        return BlockShardedBatchedProver(h, world, ranks, n_polys, n_vars)

    @staticmethod
    def single_process(devices, n_polys, n_vars):
        return BlockShardedBatchedProver._create(len(devices), list(range(len(devices))), list(devices), n_polys, n_vars)

    @staticmethod
    def one_rank(rank, world, device, n_polys, n_vars):
        return BlockShardedBatchedProver._create(world, [rank], [device], n_polys, n_vars)

    def export(self):
        out = np.empty(72 * len(self.local_ranks), dtype=np.uint8)
        check(load().ml_bpcs_shard_export(self.h, _p(out)))
        return out.tobytes()

    def connect(self, records):
        buf = np.frombuffer(bytes(records), dtype=np.uint8).copy()
        check(load().ml_bpcs_shard_connect(self.h, _p(buf), _sz(len(buf) // 72)))

    def connect_over(self, dist, device):
        """all-gather the IPC records over a torch.distributed process group (the only use of the collective library)"""
        import torch
        mine = torch.tensor(list(self.export()), dtype=torch.uint8, device=device)
        allr = [torch.empty_like(mine) for _ in range(dist.get_world_size())]
        dist.all_gather(allr, mine)
        self.connect(b"".join(bytes(r.cpu().numpy().tobytes()) for r in allr))

    def stream(self, local_index=0):
        return load().ml_bpcs_shard_stream(self.h, C.c_int(local_index))

    def arena_bytes(self):
        return load().ml_bpcs_shard_arena_bytes(self.h)

    def phase_ms(self):
        """device time between the phase marks of the last call (instrumentation, multilinear_b200_instr.h)"""
        out = (C.c_double * 16)()
        n = load().ml_bpcs_shard_phase_ms(self.h, out, C.c_int(16))
        return [out[i] for i in range(n)]

    def prove_dev(self, inputs, outputs, local_evals_ptrs, transcript):
        """local_evals_ptrs[i * n_polys + j]: device pointer to local rank i's block (n/G evaluations) of polynomial j;
        None unless rank 0 is local"""
        i, o = as_elems(inputs), as_elems(outputs)
        ptrs = (C.c_void_p * len(local_evals_ptrs))(*local_evals_ptrs)
        h = C.c_void_p()
        check(load().ml_bpcs_shard_prove_dev(self.h, _p(i), _sz(i.shape[0]), _p(o), _sz(o.shape[0]), ptrs, transcript.h, C.byref(h)))
        return PCSProof(h, batched=True) if h.value else None

    def prove(self, inputs, outputs, polys, transcript):
        """host evaluations (needs a single-process handle) — the drop-in for batched_pcs.rs:130"""
        i, o = as_elems(inputs), as_elems(outputs)
        ps = [p.evals if isinstance(p, MultilinearPolynomialEvals) else as_elems(p) for p in polys]
        ptrs = (C.c_void_p * len(ps))(*[p.ctypes.data for p in ps])
        h = C.c_void_p()
        check(load().ml_bpcs_shard_prove(self.h, _p(i), _sz(i.shape[0]), _p(o), _sz(len(ps)), ptrs, _sz(ps[0].shape[0] if ps else 0),
                                         transcript.h, C.byref(h)))
        return PCSProof(h, batched=True)

    def free(self):
        if self.h is not None and self.h.value:
            load().ml_bpcs_shard_free(self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class ShardedPCSProver:
    """PCSProof::prove of one polynomial sharded over the GPUs of one box (ml_pcs_shard_*, csrc/pcs_shard.cu).  Rank g holds the
    block evals[g*n/G, (g+1)*n/G).  A handle hosts the ranks of one process: all of them (single_process; devices may repeat =
    virtual ranks on one GPU) or one (one_rank; the records of all processes are all-gathered by the caller's transport and
    passed to connect).  The proof is an ordinary PCSProof, byte-identical to PCSProof.prove's."""

    def __init__(self, h, world, local_ranks, n_vars):
        self.h, self.world, self.local_ranks, self.n_vars = h, world, list(local_ranks), n_vars

    @staticmethod
    def _create(world, ranks, devices, n_vars):
        h = C.c_void_p()
        ra, da = (C.c_int * len(ranks))(*ranks), (C.c_int * len(devices))(*devices)
        check(load().ml_pcs_shard_create(C.c_int(world), C.c_int(len(ranks)), ra, da, _sz(n_vars), C.byref(h)))
        return ShardedPCSProver(h, world, ranks, n_vars)

    @staticmethod
    def single_process(devices, n_vars):
        return ShardedPCSProver._create(len(devices), list(range(len(devices))), list(devices), n_vars)

    @staticmethod
    def one_rank(rank, world, device, n_vars):
        return ShardedPCSProver._create(world, [rank], [device], n_vars)

    def export(self):
        out = np.empty(72 * len(self.local_ranks), dtype=np.uint8)
        check(load().ml_pcs_shard_export(self.h, _p(out)))
        return out.tobytes()

    def connect(self, records):
        buf = np.frombuffer(bytes(records), dtype=np.uint8).copy()
        check(load().ml_pcs_shard_connect(self.h, _p(buf), _sz(len(buf) // 72)))

    def connect_over(self, dist, device):
        """all-gather the IPC records over a torch.distributed process group (the only use of the collective library)"""
        import torch
        mine = torch.tensor(list(self.export()), dtype=torch.uint8, device=device)
        allr = [torch.empty_like(mine) for _ in range(dist.get_world_size())]
        dist.all_gather(allr, mine)
        self.connect(b"".join(bytes(r.cpu().numpy().tobytes()) for r in allr))

    def stream(self, local_index=0):
        return load().ml_pcs_shard_stream(self.h, C.c_int(local_index))

    def arena_bytes(self):
        return load().ml_pcs_shard_arena_bytes(self.h)

    def phase_ms(self):
        """device time between the phase marks of the last call (instrumentation, multilinear_b200_instr.h)"""
        out = (C.c_double * 16)()
        n = load().ml_pcs_shard_phase_ms(self.h, out, C.c_int(16))
        return [out[i] for i in range(n)]

    def prove_dev(self, inputs, output, local_evals_ptrs, transcript):
        """local_evals_ptrs[i]: device pointer to local rank i's block of n/G evaluations; None unless rank 0 is local"""
        i, o = as_elems(inputs), _fe1(output)
        ptrs = (C.c_void_p * len(local_evals_ptrs))(*local_evals_ptrs)
        h = C.c_void_p()
        check(load().ml_pcs_shard_prove_dev(self.h, _p(i), _sz(i.shape[0]), _p(o), ptrs, transcript.h, C.byref(h)))
        return PCSProof(h) if h.value else None

    def prove(self, inputs, output, poly, transcript):
        """host evaluations (needs a single-process handle) — the drop-in for multilinear_pcs.rs:90"""
        i, o = as_elems(inputs), _fe1(output)
        e = poly.evals if isinstance(poly, MultilinearPolynomialEvals) else as_elems(poly)
        h = C.c_void_p()
        check(load().ml_pcs_shard_prove(self.h, _p(i), _sz(i.shape[0]), _p(o), _p(e), _sz(e.shape[0]), transcript.h, C.byref(h)))
        return PCSProof(h)

    def free(self):
        if self.h is not None and self.h.value:
            load().ml_pcs_shard_free(self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class ShardedFriProver:
    """FriProof::prove of one polynomial sharded over the GPUs of one box (ml_fri_shard_*, csrc/fri_shard.cu), from its 2^log_n
    coefficients (reed_solomon + prove) or from its code of 2^(log_n+1) elements.  Rank g holds the block coeffs[g*n/G, (g+1)*n/G)
    or code[g*N/G, (g+1)*N/G).  Handles as for ShardedPCSProver.  The proof is an ordinary FriProof, byte-identical to
    FriProof.prove_from_coeffs's / FriProof.prove's."""

    def __init__(self, h, world, local_ranks, log_n):
        self.h, self.world, self.local_ranks, self.log_n = h, world, list(local_ranks), log_n

    @staticmethod
    def _create(world, ranks, devices, log_n):
        h = C.c_void_p()
        ra, da = (C.c_int * len(ranks))(*ranks), (C.c_int * len(devices))(*devices)
        check(load().ml_fri_shard_create(C.c_int(world), C.c_int(len(ranks)), ra, da, _sz(log_n), C.byref(h)))
        return ShardedFriProver(h, world, ranks, log_n)

    @staticmethod
    def single_process(devices, log_n):
        return ShardedFriProver._create(len(devices), list(range(len(devices))), list(devices), log_n)

    @staticmethod
    def one_rank(rank, world, device, log_n):
        return ShardedFriProver._create(world, [rank], [device], log_n)

    def export(self):
        out = np.empty(72 * len(self.local_ranks), dtype=np.uint8)
        check(load().ml_fri_shard_export(self.h, _p(out)))
        return out.tobytes()

    def connect(self, records):
        buf = np.frombuffer(bytes(records), dtype=np.uint8).copy()
        check(load().ml_fri_shard_connect(self.h, _p(buf), _sz(len(buf) // 72)))

    def connect_over(self, dist, device):
        """all-gather the IPC records over a torch.distributed process group (the only use of the collective library)"""
        import torch
        mine = torch.tensor(list(self.export()), dtype=torch.uint8, device=device)
        allr = [torch.empty_like(mine) for _ in range(dist.get_world_size())]
        dist.all_gather(allr, mine)
        self.connect(b"".join(bytes(r.cpu().numpy().tobytes()) for r in allr))

    def stream(self, local_index=0):
        return load().ml_fri_shard_stream(self.h, C.c_int(local_index))

    def arena_bytes(self):
        return load().ml_fri_shard_arena_bytes(self.h)

    def phase_ms(self):
        """device time between the phase marks of the last call (instrumentation, multilinear_b200_instr.h)"""
        out = (C.c_double * 16)()
        n = load().ml_fri_shard_phase_ms(self.h, out, C.c_int(16))
        return [out[i] for i in range(n)]

    def rs_prove_dev(self, local_coeffs_ptrs, transcript):
        """local_coeffs_ptrs[i]: device pointer to local rank i's block of n/G coefficients; None unless rank 0 is local"""
        ptrs = (C.c_void_p * len(local_coeffs_ptrs))(*local_coeffs_ptrs)
        h = C.c_void_p()
        check(load().ml_fri_shard_rs_prove_dev(self.h, ptrs, transcript.h, C.byref(h)))
        return FriProof(h) if h.value else None

    def prove_dev(self, local_code_ptrs, transcript):
        """local_code_ptrs[i]: device pointer to local rank i's block of N/G code elements; None unless rank 0 is local"""
        ptrs = (C.c_void_p * len(local_code_ptrs))(*local_code_ptrs)
        h = C.c_void_p()
        check(load().ml_fri_shard_prove_dev(self.h, ptrs, transcript.h, C.byref(h)))
        return FriProof(h) if h.value else None

    def rs_prove(self, coeffs, transcript):
        """host coefficients (needs a single-process handle): reed_solomon + FriProof::prove"""
        c = as_elems(coeffs)
        h = C.c_void_p()
        check(load().ml_fri_shard_rs_prove(self.h, _p(c), _sz(c.shape[0]), transcript.h, C.byref(h)))
        return FriProof(h)

    def prove(self, code, gen_pows, transcript):
        """host code (needs a single-process handle) — the drop-in for fri/mod.rs:261"""
        c = as_elems(code)
        gp = as_elems(gen_pows) if gen_pows is not None else None
        h = C.c_void_p()
        check(load().ml_fri_shard_prove(self.h, _p(c), _sz(c.shape[0]), _p(gp) if gp is not None else None,
                                        _sz(gp.shape[0] if gp is not None else 0), transcript.h, C.byref(h)))
        return FriProof(h)

    def free(self):
        if self.h is not None and self.h.value:
            load().ml_fri_shard_free(self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class ShardedBatchedFriProver:
    """BatchedFriProof::prove of B codes sharded by block over the GPUs of one box (ml_bfri_shard_*, csrc/bfri_shard.cu), from the
    2^log_n coefficients of each polynomial (reed_solomon of each + prove) or from their codes of 2^(log_n+1) elements.  Rank g
    holds block g of every polynomial: coeffs_j[g*n/G, (g+1)*n/G) or code_j[g*N/G, (g+1)*N/G).  Handles as for ShardedPCSProver.
    The proof is an ordinary batched FriProof, byte-identical to BatchedFriProof.prove's."""

    def __init__(self, h, world, local_ranks, n_codes, log_n):
        self.h, self.world, self.local_ranks, self.n_codes, self.log_n = h, world, list(local_ranks), n_codes, log_n

    @staticmethod
    def _create(world, ranks, devices, n_codes, log_n):
        h = C.c_void_p()
        ra, da = (C.c_int * len(ranks))(*ranks), (C.c_int * len(devices))(*devices)
        check(load().ml_bfri_shard_create(C.c_int(world), C.c_int(len(ranks)), ra, da, _sz(n_codes), _sz(log_n), C.byref(h)))
        return ShardedBatchedFriProver(h, world, ranks, n_codes, log_n)

    @staticmethod
    def single_process(devices, n_codes, log_n):
        return ShardedBatchedFriProver._create(len(devices), list(range(len(devices))), list(devices), n_codes, log_n)

    @staticmethod
    def one_rank(rank, world, device, n_codes, log_n):
        return ShardedBatchedFriProver._create(world, [rank], [device], n_codes, log_n)

    def export(self):
        out = np.empty(72 * len(self.local_ranks), dtype=np.uint8)
        check(load().ml_bfri_shard_export(self.h, _p(out)))
        return out.tobytes()

    def connect(self, records):
        buf = np.frombuffer(bytes(records), dtype=np.uint8).copy()
        check(load().ml_bfri_shard_connect(self.h, _p(buf), _sz(len(buf) // 72)))

    def connect_over(self, dist, device):
        """all-gather the IPC records over a torch.distributed process group (the only use of the collective library)"""
        import torch
        mine = torch.tensor(list(self.export()), dtype=torch.uint8, device=device)
        allr = [torch.empty_like(mine) for _ in range(dist.get_world_size())]
        dist.all_gather(allr, mine)
        self.connect(b"".join(bytes(r.cpu().numpy().tobytes()) for r in allr))

    def stream(self, local_index=0):
        return load().ml_bfri_shard_stream(self.h, C.c_int(local_index))

    def arena_bytes(self):
        return load().ml_bfri_shard_arena_bytes(self.h)

    def phase_ms(self):
        """device time between the phase marks of the last call (instrumentation, multilinear_b200_instr.h)"""
        out = (C.c_double * 16)()
        n = load().ml_bfri_shard_phase_ms(self.h, out, C.c_int(16))
        return [out[i] for i in range(n)]

    def rs_prove_dev(self, local_coeffs_ptrs, transcript):
        """local_coeffs_ptrs[i * n_codes + j]: device pointer to local rank i's block (n/G coefficients) of polynomial j;
        None unless rank 0 is local"""
        ptrs = (C.c_void_p * len(local_coeffs_ptrs))(*local_coeffs_ptrs)
        h = C.c_void_p()
        check(load().ml_bfri_shard_rs_prove_dev(self.h, ptrs, transcript.h, C.byref(h)))
        return FriProof(h, batched=True) if h.value else None

    def prove_dev(self, local_codes_ptrs, transcript):
        """local_codes_ptrs[i * n_codes + j]: device pointer to local rank i's block (N/G elements) of code j; None unless rank 0
        is local"""
        ptrs = (C.c_void_p * len(local_codes_ptrs))(*local_codes_ptrs)
        h = C.c_void_p()
        check(load().ml_bfri_shard_prove_dev(self.h, ptrs, transcript.h, C.byref(h)))
        return FriProof(h, batched=True) if h.value else None

    @staticmethod
    def _arrays(xs):
        cs = [as_elems(x) for x in xs]
        if any(c.shape != cs[0].shape for c in cs):
            raise SizeMismatch(2, "All codes must have the same size")
        return cs, (C.c_void_p * len(cs))(*[c.ctypes.data for c in cs]), (cs[0].shape[0] if cs else 0)

    def rs_prove(self, coeffs_list, transcript):
        """host coefficients, one array per polynomial (needs a single-process handle): reed_solomon of each + BatchedFriProof::prove"""
        cs, ptrs, n = self._arrays(coeffs_list)
        h = C.c_void_p()
        check(load().ml_bfri_shard_rs_prove(self.h, ptrs, _sz(len(cs)), _sz(n), transcript.h, C.byref(h)))
        return FriProof(h, batched=True)

    def prove(self, codes, gen_pows, transcript):
        """host codes (needs a single-process handle) — the drop-in for batched_fri.rs:286"""
        cs, ptrs, n = self._arrays(codes)
        gp = as_elems(gen_pows) if gen_pows is not None else None
        h = C.c_void_p()
        check(load().ml_bfri_shard_prove(self.h, ptrs, _sz(len(cs)), _sz(n), _p(gp) if gp is not None else None,
                                         _sz(gp.shape[0] if gp is not None else 0), transcript.h, C.byref(h)))
        return FriProof(h, batched=True)

    def free(self):
        if self.h is not None and self.h.value:
            load().ml_bfri_shard_free(self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class ShardedWideSumcheck:
    """The width-w System sumcheck over the GPUs of one box (ml_wsumcheck_shard_*, csrc/wsumcheck_shard.cu).  Rank g holds the row
    block matrix[g*h/G, (g+1)*h/G) of the row-major trace.  Handles as for ShardedPCSProver.  One call equals
    WideSumcheckTables.build + set_composition + compute_sumcheck_polynomials exactly, and every process gets the whole result."""

    def __init__(self, h, world, local_ranks, width, n_vars):
        self.h, self.world, self.local_ranks, self.width, self.n_vars = h, world, list(local_ranks), width, n_vars

    @staticmethod
    def _create(world, ranks, devices, width, n_vars):
        h = C.c_void_p()
        ra, da = (C.c_int * len(ranks))(*ranks), (C.c_int * len(devices))(*devices)
        check(load().ml_wsumcheck_shard_create(C.c_int(world), C.c_int(len(ranks)), ra, da, _sz(width), _sz(n_vars), C.byref(h)))
        return ShardedWideSumcheck(h, world, ranks, width, n_vars)

    @staticmethod
    def single_process(devices, width, n_vars):
        return ShardedWideSumcheck._create(len(devices), list(range(len(devices))), list(devices), width, n_vars)

    @staticmethod
    def one_rank(rank, world, device, width, n_vars):
        return ShardedWideSumcheck._create(world, [rank], [device], width, n_vars)

    def export(self):
        out = np.empty(72 * len(self.local_ranks), dtype=np.uint8)
        check(load().ml_wsumcheck_shard_export(self.h, _p(out)))
        return out.tobytes()

    def connect(self, records):
        buf = np.frombuffer(bytes(records), dtype=np.uint8).copy()
        check(load().ml_wsumcheck_shard_connect(self.h, _p(buf), _sz(len(buf) // 72)))

    def connect_over(self, dist, device):
        """all-gather the IPC records over a torch.distributed process group"""
        import torch
        mine = torch.tensor(list(self.export()), dtype=torch.uint8, device=device)
        allr = [torch.empty_like(mine) for _ in range(dist.get_world_size())]
        dist.all_gather(allr, mine)
        self.connect(b"".join(bytes(r.cpu().numpy().tobytes()) for r in allr))

    def stream(self, local_index=0):
        return load().ml_wsumcheck_shard_stream(self.h, C.c_int(local_index))

    def arena_bytes(self):
        return load().ml_wsumcheck_shard_arena_bytes(self.h)

    def set_composition(self, terms):
        """terms: [(coefficient, [column, ...]), ...] as for WideSumcheckTables.set_composition"""
        coefs = as_elems([c for c, _ in terms]) if terms else elems_empty(1)[:0]
        lens = np.ascontiguousarray([len(cs) for _, cs in terms], dtype=np.uint32)
        cols = np.ascontiguousarray([c for _, cs in terms for c in cs] or [0], dtype=np.uint32)
        check(load().ml_wsumcheck_shard_set_composition(self.h, _sz(len(terms)), _p(coefs), _p(lens), _p(cols)))

    def _outputs(self, composition_degree):
        n, td = self.n_vars, composition_degree + 1
        return n, td, np.empty((max(n, 1) * td, 16), dtype=np.uint8), np.empty((max(n, 1), 16), dtype=np.uint8)

    def compute_sumcheck_polynomials_dev(self, row_point, local_blocks_ptrs, composition_degree, transcript, s):
        """local_blocks_ptrs[i]: device pointer to local rank i's row block -> (flat nonzero coeffs, randoms)"""
        rp, sb = as_elems(row_point), _fe1(s)
        n, td, co, rs = self._outputs(composition_degree)
        ptrs = (C.c_void_p * len(local_blocks_ptrs))(*local_blocks_ptrs)
        check(load().ml_wsumcheck_shard_compute_polynomials_dev(self.h, _p(rp), _sz(rp.shape[0]), ptrs, _sz(composition_degree), transcript.h,
                                                                _p(sb), _p(co), _p(rs)))
        return to_ints(co[:n * td]), to_ints(rs[:n])

    def compute_sumcheck_polynomials(self, row_point, matrix, composition_degree, transcript, s):
        """host rows (needs a single-process handle) -> (flat nonzero coeffs, randoms)"""
        rp, m, sb = as_elems(row_point), as_elems(matrix), _fe1(s)
        n, td, co, rs = self._outputs(composition_degree)
        check(load().ml_wsumcheck_shard_compute_polynomials(self.h, _p(rp), _sz(rp.shape[0]), _p(m), _sz(self.width), _sz(m.shape[0] // self.width),
                                                            _sz(composition_degree), transcript.h, _p(sb), _p(co), _p(rs)))
        return to_ints(co[:n * td]), to_ints(rs[:n])

    def free(self):
        if self.h is not None and self.h.value:
            load().ml_wsumcheck_shard_free(self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


_INSTR = None


def microbench(what, n, iters):
    """integer-pipe speed-of-light loops (instrumentation library libmlb_instr.so, include/multilinear_b200_instr.h)"""
    global _INSTR
    if _INSTR is None:
        import os
        load()  # the instrumentation library links against the product library
        _INSTR = C.CDLL(os.path.join(os.path.dirname(os.path.abspath(__file__)), "libmlb_instr.so"))
    ms, work = C.c_double(0), C.c_double(0)
    check(_INSTR.ml_microbench(what.encode(), _sz(n), C.c_int(iters), C.byref(ms), C.byref(work)))
    return ms.value, work.value
