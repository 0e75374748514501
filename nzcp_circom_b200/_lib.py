"""ctypes binding of libnzcp_prover.so (the C ABI declared in include/nzcp_prover.h).

There is no fallback of any kind: if the shared library is missing or a CUDA device is absent the calls raise.
Build the library with `python -c "import __graft_entry__ as g; g.build()"` (or `make -C nzcp_circom_b200/csrc`).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NZCP_LIB_PATH") or os.path.join(_HERE, "libnzcp_prover.so")   # override: tuning variants

NZCP_OK = 0
NZCP_E_ARG, NZCP_E_FORMAT, NZCP_E_NOT_GROTH16, NZCP_E_CURVE = -1, -2, -3, -4
NZCP_E_WITNESS_LEN, NZCP_E_CUDA, NZCP_E_RANGE, NZCP_E_INTERNAL = -5, -6, -7, -8


class NzcpError(RuntimeError):
    """Mirrors the `Error` snarkjs rejects its promise with; `.code` is the NZCP_E_* value."""

    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


class ZkeyInfo(C.Structure):
    _fields_ = [("n_vars", C.c_uint32), ("n_public", C.c_uint32), ("domain_size", C.c_uint32),
                ("power", C.c_uint32), ("n_coefs", C.c_uint64),
                ("alpha1", C.c_uint8 * 64), ("beta1", C.c_uint8 * 64), ("delta1", C.c_uint8 * 64),
                ("beta2", C.c_uint8 * 128), ("gamma2", C.c_uint8 * 128), ("delta2", C.c_uint8 * 128),
                ("device_bytes", C.c_uint64)]


class ZkeyCheck(C.Structure):
    _fields_ = [("n_vars", C.c_uint32), ("n_public", C.c_uint32), ("domain_size", C.c_uint32),
                ("n_constraints", C.c_uint32), ("n_coefs", C.c_uint64), ("bad_coef_values", C.c_uint64),
                ("bad_coef_indices", C.c_uint64), ("off_curve", C.c_uint64 * 6), ("infinity", C.c_uint64 * 6),
                ("header_moduli_ok", C.c_uint32), ("header_points_ok", C.c_uint32), ("public_rows_ok", C.c_uint32),
                ("ok", C.c_uint32)]


class Proof(C.Structure):
    _fields_ = [("pi_a", C.c_uint8 * 64), ("pi_b", C.c_uint8 * 128), ("pi_c", C.c_uint8 * 64)]


class ProveDebug(C.Structure):
    _fields_ = [("msm_a", C.c_uint8 * 64), ("msm_b1", C.c_uint8 * 64), ("msm_b2", C.c_uint8 * 128),
                ("msm_c", C.c_uint8 * 64), ("msm_h", C.c_uint8 * 64), ("h_scalars", C.c_void_p),
                ("stage_ms", C.c_float * 8), ("sort_ms", C.c_float * 2), ("accumulate_ms", C.c_float * 5),
                ("n_entries", C.c_uint32 * 2), ("total_ms", C.c_float)]


class VerifyClaim(C.Structure):
    _fields_ = [("step", C.c_int32), ("record", C.c_int32), ("a", C.c_uint8 * 64), ("b", C.c_uint8 * 64),
                ("c", C.c_uint8 * 128), ("d", C.c_uint8 * 128)]


class Contribution(C.Structure):
    _fields_ = [("hash", C.c_uint8 * 64), ("type", C.c_uint32), ("num_iterations_exp", C.c_uint32),
                ("name_len", C.c_uint32), ("beacon_hash_len", C.c_uint32), ("name", C.c_uint8 * 256),
                ("beacon_hash", C.c_uint8 * 256)]


class VerifyReport(C.Structure):
    _fields_ = [("failed_step", C.c_int32), ("failed_record", C.c_int32), ("message", C.c_char * 256),
                ("n_contributions", C.c_uint32), ("n_claims", C.c_uint32), ("cs_hash", C.c_uint8 * 64)]


class PtauContribution(C.Structure):
    _fields_ = [("response_hash", C.c_uint8 * 64), ("next_challenge", C.c_uint8 * 64), ("type", C.c_uint32),
                ("num_iterations_exp", C.c_uint32), ("name_len", C.c_uint32), ("beacon_hash_len", C.c_uint32),
                ("name", C.c_uint8 * 256), ("beacon_hash", C.c_uint8 * 256)]


class PtauVerifyReport(C.Structure):
    _fields_ = [("failed_step", C.c_int32), ("failed_record", C.c_int32), ("message", C.c_char * 256),
                ("n_contributions", C.c_uint32), ("n_claims", C.c_uint32), ("prepared", C.c_uint32),
                ("next_challenge", C.c_uint8 * 64)]


# every symbol include/nzcp_prover.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_U8P = C.c_void_p          # raw byte pointers are passed as addresses / buffers
SIGNATURES = {
    "nzcp_last_error": (C.c_char_p, []),
    "nzcp_device_count": (C.c_int, []),
    "nzcp_zkey_load": (C.c_int, [_U8P, C.c_size_t, C.c_int, C.POINTER(_P)]),
    "nzcp_zkey_info_get": (C.c_int, [_P, C.POINTER(ZkeyInfo)]),
    "nzcp_zkey_free": (None, [_P]),
    "nzcp_prover_create": (C.c_int, [_P, C.POINTER(_P)]),
    "nzcp_prover_create_mode": (C.c_int, [_P, C.c_int, C.POINTER(_P)]),
    "nzcp_prover_free": (None, [_P]),
    "nzcp_prove": (C.c_int, [_P, _U8P, C.c_size_t, _U8P, _U8P, C.POINTER(Proof), C.POINTER(ProveDebug)]),
    "nzcp_prove_batch": (C.c_int, [_P, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t, _U8P, _U8P,
                                   C.POINTER(Proof), C.c_int, C.POINTER(C.c_int)]),
    "nzcp_prove_witness": (C.c_int, [_P, _U8P, C.c_uint32, _U8P, _U8P, C.POINTER(Proof), C.POINTER(ProveDebug)]),
    "nzcp_prove_device": (C.c_int, [_P, _P, _U8P, _U8P, C.POINTER(Proof), C.POINTER(ProveDebug)]),
    "nzcp_prover_witness_buffer": (_P, [_P]),
    "nzcp_prover_launch_count": (C.c_uint64, [_P]),
    "nzcp_ntt": (C.c_int, [_U8P, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "nzcp_ntt_coset": (C.c_int, [_U8P, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "nzcp_msm": (C.c_int, [_U8P, _U8P, C.c_size_t, C.c_int, C.c_int, C.c_int, _U8P, C.POINTER(C.c_float)]),
    "nzcp_zkey_selfcheck": (C.c_int, [_U8P, C.c_size_t, C.c_int, C.POINTER(ZkeyCheck)]),
    "nzcp_zkey_new_size": (C.c_int, [_U8P, C.c_size_t, _U8P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "nzcp_zkey_new": (C.c_int, [_U8P, C.c_size_t, _U8P, C.c_size_t, C.c_int, _U8P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "nzcp_ptau_prepare_size": (C.c_int, [_U8P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "nzcp_ptau_prepare": (C.c_int, [_U8P, C.c_size_t, C.c_int, _U8P, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_float)]),
    "nzcp_ptau_new_size": (C.c_int, [C.c_uint32, C.POINTER(C.c_size_t)]),
    "nzcp_ptau_new": (C.c_int, [C.c_uint32, _U8P, C.c_size_t, C.POINTER(C.c_size_t), _U8P]),
    "nzcp_ptau_contribute_size": (C.c_int, [_U8P, C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "nzcp_ptau_contribute": (C.c_int, [_U8P, C.c_size_t, C.c_char_p, _U8P, C.c_size_t, _U8P, C.c_int, _U8P, C.c_size_t,
                                       C.POINTER(C.c_size_t), _U8P, C.POINTER(C.c_float)]),
    "nzcp_ptau_beacon": (C.c_int, [_U8P, C.c_size_t, C.c_char_p, _U8P, C.c_size_t, C.c_uint32, C.c_int, _U8P, C.c_size_t,
                                   C.POINTER(C.c_size_t), _U8P, C.POINTER(C.c_float)]),
    "nzcp_zkey_contribute_size": (C.c_int, [_U8P, C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "nzcp_zkey_contribute": (C.c_int, [_U8P, C.c_size_t, C.c_char_p, _U8P, C.c_size_t, _U8P, C.c_int, _U8P, C.c_size_t,
                                       C.POINTER(C.c_size_t), _U8P, C.POINTER(C.c_float)]),
    "nzcp_zkey_beacon": (C.c_int, [_U8P, C.c_size_t, C.c_char_p, _U8P, C.c_size_t, C.c_uint32, C.c_int, _U8P, C.c_size_t,
                                   C.POINTER(C.c_size_t), _U8P, C.POINTER(C.c_float)]),
    "nzcp_zkey_circuit_hash": (C.c_int, [_U8P, C.c_size_t, _U8P, C.c_size_t, C.c_int, _U8P, C.POINTER(C.c_float)]),
    "nzcp_zkey_verify_size": (C.c_int, [_U8P, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "nzcp_zkey_verify_from_init": (C.c_int, [_U8P, C.c_size_t, _U8P, C.c_size_t, _U8P, C.c_size_t, _U8P, C.c_int,
                                             C.POINTER(VerifyClaim), C.c_size_t, C.POINTER(Contribution), C.c_size_t,
                                             C.POINTER(VerifyReport), C.POINTER(C.c_float)]),
    "nzcp_zkey_verify_from_r1cs": (C.c_int, [_U8P, C.c_size_t, _U8P, C.c_size_t, _U8P, C.c_size_t, _U8P, C.c_int,
                                             C.POINTER(VerifyClaim), C.c_size_t, C.POINTER(Contribution), C.c_size_t,
                                             C.POINTER(VerifyReport), C.POINTER(C.c_float)]),
    "nzcp_ptau_verify_size": (C.c_int, [_U8P, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "nzcp_ptau_verify": (C.c_int, [_U8P, C.c_size_t, _U8P, C.c_int, C.POINTER(VerifyClaim), C.c_size_t,
                                   C.POINTER(PtauContribution), C.c_size_t, C.POINTER(PtauVerifyReport),
                                   C.POINTER(C.c_float)]),
    "nzcp_msm_plan_create": (C.c_int, [_U8P, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_P),
                                       C.POINTER(C.c_float)]),
    "nzcp_msm_plan_free": (None, [_P]),
    "nzcp_msm_plan_run": (C.c_int, [_P, _U8P, C.c_size_t, _U8P, C.POINTER(C.c_float)]),
    "nzcp_msm_plan_accumulate_ms": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "nzcp_msm_plan_run_partial": (C.c_int, [_P, _U8P, C.c_size_t, _P, C.POINTER(C.c_float)]),
    "nzcp_msm_sum_partials": (C.c_int, [_P, C.c_size_t, C.c_int, C.c_int, _U8P]),
    "nzcp_msm_var": (C.c_int, [_U8P, _U8P, C.c_size_t, C.c_int, C.c_int, C.c_int, _U8P, C.POINTER(C.c_float)]),
    "nzcp_selftest": (C.c_int, [C.c_int, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint32)]),
    "nzcp_field_op": (C.c_int, [C.c_int, C.c_int, _U8P, _U8P, _U8P, C.c_size_t, C.c_int]),
    "nzcp_arith_op": (C.c_int, [C.c_int, _U8P, _U8P, C.c_size_t, C.c_int]),
    "nzcp_curve_op": (C.c_int, [C.c_int, C.c_int, _U8P, _U8P, _U8P, C.c_size_t, C.c_int]),
    "nzcp_intpipe_modes": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "nzcp_intpipe_bench": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "nzcp_pipe_probe": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "nzcp_host_field_op": (C.c_int, [C.c_int, C.c_int, _U8P, _U8P, _U8P, C.c_size_t]),
    "nzcp_host_scalar_mul": (C.c_int, [C.c_int, _U8P, _U8P, _U8P]),
    "nzcp_host_root_of_unity": (C.c_int, [C.c_int, _U8P]),
    "nzcp_host_ptau_prepare": (C.c_int, [_U8P, C.c_size_t, _U8P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "nzcp_host_zkey_contribute": (C.c_int, [_U8P, C.c_size_t, C.c_char_p, _U8P, C.c_size_t, _U8P, _U8P, C.c_size_t,
                                            C.c_uint32, _U8P, C.c_size_t, C.POINTER(C.c_size_t), _U8P]),
    "nzcp_host_ptau_contribute": (C.c_int, [_U8P, C.c_size_t, C.c_char_p, _U8P, C.c_size_t, _U8P, _U8P, C.c_size_t,
                                            C.c_uint32, _U8P, C.c_size_t, C.POINTER(C.c_size_t), _U8P]),
    "nzcp_host_ptau_verify": (C.c_int, [_U8P, C.c_size_t, _U8P, C.POINTER(VerifyClaim), C.c_size_t,
                                        C.POINTER(PtauContribution), C.c_size_t, C.POINTER(PtauVerifyReport)]),
    "nzcp_host_zkey_circuit_hash": (C.c_int, [_U8P, C.c_size_t, _U8P, C.c_size_t, _U8P]),
    "nzcp_host_msm_sim": (C.c_int, [_U8P, _U8P, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, _U8P]),
    "nzcp_tuning_set": (C.c_int, [C.c_char_p, C.c_int]),
    "nzcp_synth_points": (C.c_int, [C.c_uint64, C.c_size_t, C.c_int, C.c_int, _U8P]),
    "nzcp_synth_create": (C.c_int, [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(_P)]),
    "nzcp_synth_free": (None, [_P]),
    "nzcp_synth_dims": (C.c_int, [_P, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                  C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
    "nzcp_synth_zkey_size": (C.c_size_t, [_P]),
    "nzcp_synth_r1cs_size": (C.c_size_t, [_P]),
    "nzcp_synth_wtns_size": (C.c_size_t, [_P]),
    "nzcp_synth_write_zkey": (C.c_int, [_P, _U8P, C.c_int, _U8P, C.c_size_t]),
    "nzcp_synth_write_r1cs": (C.c_int, [_P, _U8P, C.c_size_t]),
    "nzcp_synth_write_wtns": (C.c_int, [_P, C.c_uint64, _U8P, C.c_size_t]),
}

_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libnzcp_prover.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'`. "
            "nzcp_circom_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here == header and library out of sync
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code):
    if code != NZCP_OK:
        msg = load().nzcp_last_error()
        raise NzcpError(code, msg.decode() if msg else "nzcp error %d" % code)


def addr(buf):
    """Address of a bytes / bytearray / memoryview / numpy array / ctypes buffer, without copying."""
    if buf is None:
        return None
    if isinstance(buf, int):
        return buf
    if isinstance(buf, bytes):
        return C.cast(C.c_char_p(buf), C.c_void_p).value
    if hasattr(buf, "ctypes"):            # numpy
        return buf.ctypes.data
    if hasattr(buf, "data_ptr"):          # torch tensor
        return buf.data_ptr()
    if isinstance(buf, C.Array):
        return C.addressof(buf)
    mv = memoryview(buf)
    if mv.readonly:
        raise TypeError("need a writable or bytes buffer")
    return C.addressof((C.c_char * mv.nbytes).from_buffer(mv))
