"""ctypes loader for libmultilinear_b200.so (the C ABI declared in include/multilinear_b200.h).

There is no CPU fallback: if the shared library is missing it is built with nvcc; if that fails, or a
compute entry point finds no sm_100 device, the call raises.
"""
import ctypes as C
import os

from . import build as _build

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

ML_OK = 0
ERR_NAMES = {1: "ML_ERR_NOT_POW2", 2: "ML_ERR_SIZE", 3: "ML_ERR_OUT_OF_RANGE", 4: "ML_ERR_NOT_RS_CODE", 5: "ML_ERR_GENERATOR",
             6: "ML_ERR_CUDA", 7: "ML_ERR_ALLOC", 8: "ML_ERR_ARG", 9: "ML_ERR_PEER"}


class MlError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s (%d): %s" % (ERR_NAMES.get(code, "ML_ERR"), code, msg))
        self.code = code


class NotPowerOfTwo(MlError):
    """the reference's assert!(n.is_power_of_two()) panics"""


class SizeMismatch(MlError):
    pass


class NotRsCode(MlError):
    """assert!(..., "not an RS code") — src/fri/mod.rs:119-122"""


_EXC = {1: NotPowerOfTwo, 2: SizeMismatch, 4: NotRsCode}

_SIZE_T_FUNCS = ["ml_merkle_num_layers", "ml_merkle_layer_len", "ml_fri_num_trees", "ml_fri_proof_num_commitments",
                 "ml_fri_proof_serialized_len", "ml_sumcheck_height", "ml_wsumcheck_height", "ml_wsumcheck_width", "ml_pcs_proof_num_rounds", "ml_bfri_proof_num_commitments",
                 "ml_bfri_proof_serialized_len", "ml_bpcs_proof_num_rounds", "ml_shard_record_bytes", "ml_shard_arena_bytes", "ml_bfri_num_codes",
                 "ml_pcs_shard_arena_bytes", "ml_bpcs_shard_arena_bytes", "ml_wsumcheck_shard_arena_bytes",
                 "ml_fri_shard_arena_bytes", "ml_bfri_shard_arena_bytes"]
_PTR_FUNCS = ["ml_pcs_proof_fri", "ml_bpcs_proof_fri", "ml_shard_stream", "ml_bfri_fri_data", "ml_bfri_batch_layer", "ml_pcs_shard_stream", "ml_bpcs_shard_stream", "ml_wsumcheck_shard_stream",
              "ml_fri_shard_stream", "ml_bfri_shard_stream"]
_VOID_FUNCS = ["ml_transcript_free", "ml_merkle_free", "ml_fri_free", "ml_fri_proof_free", "ml_sumcheck_free", "ml_wsumcheck_free", "ml_pcs_proof_free",
               "ml_bfri_proof_free", "ml_bpcs_proof_free", "ml_shard_free", "ml_bfri_free", "ml_pcs_shard_free", "ml_bpcs_shard_free", "ml_wsumcheck_shard_free",
               "ml_fri_shard_free", "ml_bfri_shard_free"]


def lib_path():
    return os.path.join(_HERE, "libmultilinear_b200.so")


def load():
    global _LIB
    if _LIB is None:
        path = lib_path()
        if not os.path.exists(path):
            _build.build()  # raises if nvcc is unavailable
        L = C.CDLL(path)
        L.ml_last_error.restype = C.c_char_p
        L.ml_version.restype = C.c_char_p
        L.ml_kernel_launches.restype = C.c_uint64
        for f in _SIZE_T_FUNCS:
            getattr(L, f).restype = C.c_size_t
        for f in _PTR_FUNCS:
            getattr(L, f).restype = C.c_void_p
        for f in _VOID_FUNCS:
            getattr(L, f).restype = None
        _LIB = L
    return _LIB


def check(code):
    """status -> exception (mirrors the reference's panics / None)"""
    if code != ML_OK:
        msg = load().ml_last_error().decode(errors="replace")
        raise _EXC.get(code, MlError)(code, msg)
    return code
