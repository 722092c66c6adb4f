"""ctypes binding of libb200zk.so (include/b200zk.h).  Fails loudly when the
library is missing or no CUDA device is present: there is no CPU fallback."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200zk.so")

PARTIAL_BYTES = 1344
B2Z_OK, B2Z_EINVAL, B2Z_ESIZE, B2Z_ECUDA, B2Z_ENOMEM = 0, 1, 2, 3, 4
STATUS_NAMES = {0: "B2Z_OK", 1: "B2Z_EINVAL", 2: "B2Z_ESIZE", 3: "B2Z_ECUDA", 4: "B2Z_ENOMEM"}

u64p = ctypes.POINTER(ctypes.c_uint64)
u32p = ctypes.POINTER(ctypes.c_uint32)
u8p = ctypes.POINTER(ctypes.c_uint8)
i32p = ctypes.POINTER(ctypes.c_int32)
vp = ctypes.c_void_p


class PkDesc(ctypes.Structure):
    _fields_ = [
        ("num_variables", ctypes.c_uint64), ("num_instance", ctypes.c_uint64), ("log_domain", ctypes.c_uint32),
        ("a_query", vp), ("a_inf", vp), ("b_g1_query", vp), ("b_g1_inf", vp),
        ("b_g2_query", vp), ("b_g2_inf", vp), ("h_query", vp), ("h_inf", vp),
        ("l_query", vp), ("l_inf", vp),
        ("alpha_g1", vp), ("beta_g1", vp), ("delta_g1", vp), ("beta_g2", vp), ("delta_g2", vp),
    ]


class VkDesc(ctypes.Structure):
    _fields_ = [("num_instance", ctypes.c_uint64), ("alpha_g1", vp), ("beta_g2", vp), ("gamma_g2", vp),
                ("delta_g2", vp), ("gamma_abc_g1", vp), ("gamma_abc_inf", vp)]


class SetupDesc(ctypes.Structure):
    _fields_ = [("alpha", vp), ("beta", vp), ("gamma", vp), ("delta", vp), ("tau", vp),
                ("g1_generator", vp), ("g2_generator", vp)]


class VkOut(ctypes.Structure):
    _fields_ = [("alpha_g1", ctypes.c_uint64 * 12), ("beta_g2", ctypes.c_uint64 * 24), ("gamma_g2", ctypes.c_uint64 * 24),
                ("delta_g2", ctypes.c_uint64 * 24), ("gamma_abc_g1", vp), ("gamma_abc_inf", vp)]


class PkArrays(ctypes.Structure):
    _fields_ = [
        ("num_variables", ctypes.c_uint64), ("num_instance", ctypes.c_uint64), ("log_domain", ctypes.c_uint32),
        ("a_query", vp), ("a_inf", vp), ("b_g1_query", vp), ("b_g1_inf", vp),
        ("b_g2_query", vp), ("b_g2_inf", vp), ("h_query", vp), ("h_inf", vp),
        ("l_query", vp), ("l_inf", vp),
        ("alpha_g1", ctypes.c_uint64 * 12), ("beta_g1", ctypes.c_uint64 * 12), ("delta_g1", ctypes.c_uint64 * 12),
        ("beta_g2", ctypes.c_uint64 * 24), ("delta_g2", ctypes.c_uint64 * 24),
    ]


class PoseidonDesc(ctypes.Structure):
    _fields_ = [("full_rounds", ctypes.c_uint32), ("partial_rounds", ctypes.c_uint32), ("alpha", ctypes.c_uint64),
                ("width", ctypes.c_uint32), ("rate", ctypes.c_uint32), ("capacity", ctypes.c_uint32),
                ("ark", vp), ("mds", vp)]


class PrimeCheck(ctypes.Structure):
    _fields_ = [("j", ctypes.c_uint64), ("digest", ctypes.c_uint8 * 32), ("is_prime", ctypes.c_int32),
                ("quotient", ctypes.c_uint64 * 4), ("remainder", ctypes.c_uint64), ("a", ctypes.c_uint64 * 4)]


# name -> (restype, argtypes); the test-suite checks this table against include/b200zk.h
SIGNATURES = {
    "b2z_ctx_create": (ctypes.c_int32, [ctypes.c_int, ctypes.POINTER(vp)]),
    "b2z_ctx_destroy": (None, [vp]),
    "b2z_last_error": (ctypes.c_char_p, [vp]),
    "b2z_ntt_fr": (ctypes.c_int32, [vp, vp, ctypes.c_uint32, ctypes.c_int, vp]),
    "b2z_witness_map": (ctypes.c_int32, [vp, vp, vp, vp, ctypes.c_uint32, vp]),
    "b2z_msm_g1": (ctypes.c_int32, [vp, vp, vp, vp, ctypes.c_uint64, vp]),
    "b2z_msm_g2": (ctypes.c_int32, [vp, vp, vp, vp, ctypes.c_uint64, vp]),
    "b2z_pk_upload": (ctypes.c_int32, [vp, ctypes.POINTER(PkDesc), ctypes.POINTER(vp)]),
    "b2z_pk_free": (None, [vp, vp]),
    "b2z_groth16_prove": (ctypes.c_int32, [vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "b2z_r1cs_upload": (ctypes.c_int32, [vp, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64] + [vp] * 9 + [ctypes.POINTER(vp)]),
    "b2z_r1cs_free": (None, [vp, vp]),
    "b2z_r1cs_eval": (ctypes.c_int32, [vp, vp, vp, vp, vp, vp]),
    "b2z_spmv_fr": (ctypes.c_int32, [vp, ctypes.c_uint64, ctypes.c_uint64, vp, vp, vp, vp, vp]),
    "b2z_witness_map_from_matrices": (ctypes.c_int32, [vp, vp, vp, vp]),
    "b2z_groth16_prove_r1cs": (ctypes.c_int32, [vp, vp, vp, vp, vp, vp, vp]),
    "b2z_pk_upload_slice": (ctypes.c_int32, [vp, ctypes.POINTER(PkDesc), ctypes.c_uint32, ctypes.c_uint32,
                                             ctypes.c_uint32, ctypes.POINTER(vp)]),
    "b2z_pk_upload_shard": (ctypes.c_int32, [vp, ctypes.POINTER(PkDesc), ctypes.c_uint32, ctypes.c_uint32,
                                             ctypes.POINTER(vp)]),
    "b2z_groth16_prove_partial": (ctypes.c_int32, [vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "b2z_groth16_prove_partial_r1cs": (ctypes.c_int32, [vp, vp, vp, vp, vp, vp, vp]),
    "b2z_groth16_combine": (ctypes.c_int32, [vp, ctypes.c_uint32, vp]),
    "b2z_groth16_prove_device": (ctypes.c_int32, [vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "b2z_fixed_base_mul_g1": (ctypes.c_int32, [vp, vp, ctypes.c_uint64, vp, vp]),
    "b2z_fixed_base_mul_g2": (ctypes.c_int32, [vp, vp, ctypes.c_uint64, vp, vp]),
    "b2z_groth16_setup": (ctypes.c_int32, [vp, vp, ctypes.POINTER(SetupDesc), ctypes.POINTER(vp), ctypes.POINTER(VkOut)]),
    "b2z_groth16_setup_shard": (ctypes.c_int32, [vp, vp, ctypes.POINTER(SetupDesc), ctypes.c_uint32, ctypes.c_uint32,
                                                 ctypes.POINTER(vp), ctypes.POINTER(VkOut)]),
    "b2z_pk_download": (ctypes.c_int32, [vp, vp, ctypes.POINTER(PkArrays)]),
    "b2z_profile_enable": (ctypes.c_int32, [vp, ctypes.c_int]),
    "b2z_profile_read": (ctypes.c_int32, [vp, vp, vp, vp, ctypes.c_int]),
    "b2z_profile_spans": (ctypes.c_int, [vp, ctypes.c_int, vp, vp, vp]),
    "b2z_kernel_launches": (ctypes.c_uint64, [vp]),
    "b2z_measure_int_peak": (ctypes.c_int32, [vp, vp, vp]),
    "b2z_groth16_shard_begin": (ctypes.c_int32, [vp, vp, vp, vp, vp, vp]),
    "b2z_r1cs_coset_evals": (ctypes.c_int32, [vp, vp, ctypes.c_uint32, vp, vp]),
    "b2z_groth16_shard_finish": (ctypes.c_int32, [vp, vp, vp, vp, vp, vp]),
    "b2z_groth16_prepare_verifying_key": (ctypes.c_int32, [ctypes.POINTER(VkDesc), vp, ctypes.c_uint64,
                                                            ctypes.POINTER(ctypes.c_uint64)]),
    "b2z_groth16_verify_with_processed_vk": (ctypes.c_int32, [vp, ctypes.c_uint64, vp, ctypes.c_uint64, vp,
                                                               ctypes.POINTER(ctypes.c_int32)]),
    "b2z_groth16_verify_batch": (ctypes.c_int32, [vp, vp, ctypes.c_uint64, vp, ctypes.c_uint64, vp, ctypes.c_uint64,
                                                   vp]),
    "b2z_dist_shared_bytes": (ctypes.c_uint64, [ctypes.c_uint32]),
    "b2z_dist_combine_shared": (ctypes.c_int32, [vp, ctypes.c_uint32, ctypes.c_uint32, ctypes.POINTER(ctypes.c_uint32), vp,
                                                  vp]),
    "b2z_dist_create": (ctypes.c_int32, [vp, vp, vp, ctypes.c_uint32, ctypes.c_uint32, vp, ctypes.POINTER(vp)]),
    "b2z_dist_destroy": (None, [vp, vp]),
    "b2z_dist_export": (ctypes.c_int32, [vp, vp, vp, ctypes.POINTER(vp)]),
    "b2z_dist_attach": (ctypes.c_int32, [vp, vp, ctypes.c_uint32, vp, vp]),
    "b2z_dist_prove": (ctypes.c_int32, [vp, vp, vp, ctypes.c_int, vp, vp, vp]),
    "b2z_host_register": (ctypes.c_int32, [vp, vp, ctypes.c_uint64]),
    "b2z_host_unregister": (ctypes.c_int32, [vp, vp]),
    "b2z_fr_lagrange_at": (ctypes.c_int32, [ctypes.c_uint32, vp, ctypes.c_uint64, ctypes.c_uint32, vp]),
    "b2z_fr_geometric": (ctypes.c_int32, [vp, vp, ctypes.c_uint64, ctypes.c_uint32, vp]),
    "b2z_fr_lincomb3": (ctypes.c_int32, [ctypes.c_uint64, vp, vp, vp, vp, vp, vp, ctypes.c_uint32, vp]),
    "b2z_fr_into_bigint": (ctypes.c_int32, [ctypes.c_uint64, vp, ctypes.c_uint32, vp]),
    "b2z_poseidon_hash": (ctypes.c_int32, [ctypes.POINTER(PoseidonDesc), vp, ctypes.c_uint64, vp]),
    "b2z_matrix_circuit_num_variables": (ctypes.c_uint64, [ctypes.POINTER(PoseidonDesc), ctypes.c_uint32]),
    "b2z_matrix_circuit_witness": (ctypes.c_int32, [ctypes.POINTER(PoseidonDesc), ctypes.c_uint32, vp, vp,
                                                    ctypes.c_uint32, vp, ctypes.c_uint64]),
    "b2z_fibonacci_witness": (ctypes.c_int32, [vp, vp, ctypes.c_uint64, vp]),
    "b2z_modpow_witnesses": (ctypes.c_int32, [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32,
                                              vp, vp, vp, ctypes.POINTER(ctypes.c_uint64)]),
    "b2z_prime_search": (ctypes.c_int32, [vp, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32,
                                          ctypes.c_uint32, ctypes.POINTER(PrimeCheck), ctypes.POINTER(ctypes.c_int32)]),
    "b2z_sha256": (None, [vp, ctypes.c_uint64, vp]),
    "b2z_host_field_op": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, vp, vp, vp]),
    "b2z_host_fq_inv_gcd": (ctypes.c_int, [vp, vp]),
    "b2z_host_accum_affine": (ctypes.c_int, [ctypes.c_int, vp, vp, vp, ctypes.c_uint32, ctypes.c_uint32,
                                              ctypes.c_uint32, vp]),
    "b2z_host_point_sum": (ctypes.c_int, [ctypes.c_int, vp, vp, ctypes.c_uint32, vp]),
    "b2z_host_msm_digits": (ctypes.c_uint32, [vp, ctypes.c_uint32, vp]),
    "b2z_host_msm_window_bits": (ctypes.c_uint32, [ctypes.c_uint64, ctypes.c_int]),
    "b2z_host_planes_horner": (ctypes.c_int, [ctypes.c_int, vp, ctypes.c_uint32, ctypes.c_uint32, vp]),
    "b2z_host_verify_one": (ctypes.c_int32, [vp, ctypes.c_uint64, vp, ctypes.c_uint64, vp, ctypes.POINTER(ctypes.c_int32)]),
    "b2z_host_pairing_op": (ctypes.c_int, [ctypes.c_int, vp, vp, vp, vp]),
}

_lib = None


class B2zError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("%s: %s" % (STATUS_NAMES.get(status, status), message))
        self.status = status


def lib():
    """The loaded library; raises if libb200zk.so has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libb200zk.so is missing (%s): build it with `python zksnark-finalproject_b200/build.py` "
                "or __graft_entry__.build(); there is no CPU fallback" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib
