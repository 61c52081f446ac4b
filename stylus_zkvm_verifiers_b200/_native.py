"""ctypes binding of libzkv_b200.so (the C ABI of include/zkv.h).  There is no CPU fallback: a missing
library or a missing CUDA device is an error, never a silent software path."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("ZKV_LIB") or os.path.join(HERE, "libzkv_b200.so")   # ZKV_LIB: alternative build of the same library (tuning experiments)

ZKV_OK, ZKV_INVALID_INITIALIZATION, ZKV_INVALID_PROOF_DATA, ZKV_SELECTOR_MISMATCH, ZKV_VERIFICATION_FAILED = range(5)
ZKV_ERR_ARG, ZKV_ERR_CUDA, ZKV_ERR_STATE = -1, -2, -3
ZKV_VM_RISC0, ZKV_VM_SP1 = 0, 1
TUNE = {"overlap": 0, "normalised_lines": 1, "miller_segments": 2, "final_exp_stages": 3, "layout": 4}     # ZKV_TUNE_* of zkv.h
ZKV_TUNE_QUERY = -1

_P = C.c_void_p
_SIGS = {
    "zkv_last_error": (C.c_char_p, []),
    "zkv_device_count": (C.c_int, []),
    "zkv_vk_load": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, C.c_int, _P, C.c_int, C.POINTER(_P)]),
    "zkv_vk_load_risc0": (C.c_int, [_P, C.c_int, C.POINTER(_P)]),
    "zkv_vk_load_sp1": (C.c_int, [_P, C.c_int, C.POINTER(_P)]),
    "zkv_vk_free": (None, [_P]),
    "zkv_groth16_verify_batch": (C.c_int, [_P, _P, _P, C.c_int, C.c_size_t, _P]),
    "zkv_vkset_create": (C.c_int, [_P, C.c_int, _P, C.c_int, C.POINTER(_P)]),
    "zkv_vkset_destroy": (None, [_P]),
    "zkv_groth16_verify_batch_keys": (C.c_int, [_P, _P, _P, _P, _P, C.c_size_t, _P]),
    "zkv_groth16_verify_batch_keys_device": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_size_t, _P, _P]),
    "zkv_risc0_create": (C.c_int, [_P, _P, C.c_int, C.POINTER(_P)]),
    "zkv_risc0_destroy": (None, [_P]),
    "zkv_risc0_initialize": (C.c_int, [_P, _P, _P]),
    "zkv_risc0_is_initialized": (C.c_int, [_P]),
    "zkv_risc0_get_selector": (C.c_int, [_P, _P]),
    "zkv_risc0_get_control_root": (C.c_int, [_P, _P, _P]),
    "zkv_risc0_get_bn254_control_id": (C.c_int, [_P, _P]),
    "zkv_risc0_get_verifier_key_digest": (C.c_int, [_P, _P]),
    "zkv_risc0_verify_batch": (C.c_int, [_P, _P, _P, _P, _P, C.c_size_t, _P]),
    "zkv_risc0_verify_integrity_batch": (C.c_int, [_P, _P, _P, _P, C.c_size_t, _P]),
    "zkv_risc0_verify": (C.c_int, [_P, _P, C.c_size_t, _P, _P, _P]),
    "zkv_risc0_verify_integrity": (C.c_int, [_P, _P, C.c_size_t, _P, _P]),
    "zkv_sp1_create": (C.c_int, [_P, _P, C.c_int, C.POINTER(_P)]),
    "zkv_sp1_destroy": (None, [_P]),
    "zkv_sp1_verifier_hash": (C.c_int, [_P, _P]),
    "zkv_sp1_version": (C.c_char_p, [_P]),
    "zkv_sp1_verify_batch": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "zkv_sp1_verify_proof": (C.c_int, [_P, _P, _P, C.c_size_t, _P, C.c_size_t, _P]),
    "zkv_risc0_verify_batch_device": (C.c_int, [_P, C.c_int, _P, _P, _P, C.c_size_t, _P, _P]),
    "zkv_sp1_verify_batch_device": (C.c_int, [_P, C.c_int, _P, _P, C.c_size_t, _P, C.c_size_t, _P, _P]),
    "zkv_pairing4_batch": (C.c_int, [_P, _P, _P, C.c_size_t, _P, _P, _P]),
    "zkv_pairing4_batch_device": (C.c_int, [_P, C.c_int, _P, _P, C.c_size_t, _P, _P, _P]),
    "zkv_ec_pairing_batch": (C.c_int, [_P, C.c_int, C.c_size_t, _P, _P, _P, C.c_int]),
    "zkv_ec_pairing": (C.c_int, [_P, C.c_size_t, _P, _P, C.c_int]),
    "zkv_ec_add_batch": (C.c_int, [_P, C.c_size_t, _P, _P, C.c_int]),
    "zkv_ec_mul_batch": (C.c_int, [_P, C.c_size_t, _P, _P, C.c_int]),
    "zkv_g2_mul_batch": (C.c_int, [_P, C.c_int, _P, C.c_size_t, _P, _P, C.c_int]),
    "zkv_vk_x_batch": (C.c_int, [_P, _P, C.c_int, C.c_size_t, _P]),
    "zkv_fp_mul_batch": (C.c_int, [_P, _P, C.c_size_t, _P, C.c_int]),
    "zkv_fp12_op_batch": (C.c_int, [C.c_int, _P, _P, C.c_size_t, _P, C.c_int]),
    "zkv_g2_check_batch": (C.c_int, [_P, C.c_size_t, _P, C.c_int]),
    "zkv_last_stage_ms": (C.c_int, [_P, C.c_int, _P, C.c_int]),
    "zkv_risc0_vk": (_P, [_P]),
    "zkv_sp1_vk": (_P, [_P]),
    "zkv_vk_tune": (C.c_int, [_P, C.c_int, C.c_int]),
    "zkv_launch_count": (C.c_ulonglong, []),
    "zkv_wave_proofs": (C.c_longlong, [C.c_int, C.c_int]),
    "zkv_imad_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "zkv_self_test": (C.c_int, [C.c_int]),
    "zkv_host_alloc": (C.c_void_p, [C.c_size_t]),
    "zkv_host_free": (None, [C.c_void_p]),
    "zkv_test_parallel_copy": (None, [C.c_void_p, C.c_void_p, C.c_size_t]),
}
EXPORTS = tuple(_SIGS)

_lib = None


class ZkvError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libzkv_b200 error %d: %s" % (code, msg))
        self.code = code


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a). This package has no CPU fallback." % SO_PATH)
        L = C.CDLL(SO_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        # known-answer self test of the production kernels, once per process (zkv.h: zkv_self_test): a build whose kernels mis-verify the
        # reference's golden proofs must not be used.  Runs on this process's own device (torchrun: LOCAL_RANK).
        nd = L.zkv_device_count()
        if nd > 0 and not os.environ.get("ZKV_SKIP_SELFTEST"):
            dev = int(os.environ.get("LOCAL_RANK", "0"))
            rc = L.zkv_self_test(dev if 0 <= dev < nd else 0)
            if rc != 0:
                raise ZkvError(rc, (L.zkv_last_error() or b"").decode())
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise ZkvError(rc, (lib().zkv_last_error() or b"").decode())


def buf(b):
    """bytes / bytearray / numpy array -> something ctypes accepts for a void* parameter"""
    if isinstance(b, (bytes, bytearray)):
        return C.cast(C.c_char_p(bytes(b)), _P) if not isinstance(b, bytes) else C.cast(C.c_char_p(b), _P)
    return C.c_void_p(b.ctypes.data)
