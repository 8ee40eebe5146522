"""ctypes declarations for include/eg_b200.h (the C ABI of libeg_b200.so)."""
import ctypes as C
import os
import pathlib

PKG = pathlib.Path(__file__).resolve().parent
DEFAULT_LIB = PKG / "libeg_b200.so"

SUCCESS, ERR_INVALID_ARG, ERR_INVALID_ELEMENT, ERR_IDENTITY_KEY, ERR_NO_RECEIVER, ERR_NO_DEVICE, ERR_CUDA, \
    ERR_OUT_OF_MEMORY, ERR_LEN_MISMATCH, ERR_NCCL = range(10)
STATUS_NAMES = ["SUCCESS", "ERR_INVALID_ARG", "ERR_INVALID_ELEMENT", "ERR_IDENTITY_KEY", "ERR_NO_RECEIVER",
                "ERR_NO_DEVICE", "ERR_CUDA", "ERR_OUT_OF_MEMORY", "ERR_LEN_MISMATCH", "ERR_NCCL"]
COMM_ID_BYTES = 128
WIRE_CIPHERTEXT, WIRE_DECRYPTION, WIRE_LOG_EQUALITY_PROOF, WIRE_COMMITMENT_EQUIV_PROOF, WIRE_RING_PROOF, WIRE_POSSESSION_PROOF, \
    WIRE_SUMSQ_PROOF = range(7)

V_OK, V_MALFORMED, V_CHALLENGE_MISMATCH, V_CHOICE_SUM, V_CHOICE_RANGE, V_QV_CREDIT_RANGE, V_QV_CREDIT_EQUIV, \
    V_MALFORMED_PARTICIPANT_KEYS = range(8)
V_QV_VARIANT_BASE = 16


class Range(C.Structure):
    _fields_ = [("n_rings", C.c_uint32), ("reserved", C.c_uint32), ("size", C.c_uint64 * 64), ("step", C.c_uint64 * 64)]

    @property
    def rings(self):
        return [(self.size[i], self.step[i]) for i in range(self.n_rings)]

    @property
    def rings_size(self):
        return sum(self.size[i] for i in range(self.n_rings))


class QvParams(C.Structure):
    _fields_ = [("options", C.c_uint32), ("reserved", C.c_uint32), ("credits", C.c_uint64), ("vote_range", Range),
                ("credit_range", Range)]


class KeySet(C.Structure):
    _fields_ = [("shares", C.c_uint32), ("threshold", C.c_uint32), ("shared_key", C.c_uint8 * 32),
                ("participant_keys", (C.c_uint8 * 32) * 64)]


P8 = C.c_void_p   # byte buffers are passed as raw addresses (host numpy arrays or device pointers)

PROTOTYPES = {
    "eg_ctx_create": (C.c_int32, [C.c_int, C.POINTER(C.c_void_p)]),
    "eg_ctx_create_multi": (C.c_int32, [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    "eg_comm_unique_id": (C.c_int32, [P8]),
    "eg_ctx_attach_comm": (C.c_int32, [C.c_void_p, P8, C.c_int, C.c_int]),
    "eg_ctx_comm_info": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "eg_ctx_destroy": (None, [C.c_void_p]),
    "eg_last_error": (C.c_char_p, [C.c_void_p]),
    "eg_version": (C.c_char_p, []),
    "eg_ctx_set_receiver": (C.c_int32, [C.c_void_p, P8]),
    "eg_ctx_set_blinding_base": (C.c_int32, [C.c_void_p, P8]),
    "eg_verify_commitment_equiv_batch": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_size_t, P8, P8, P8, P8]),
    "eg_verify_possession_batch": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_uint32, C.c_size_t, P8, P8, P8]),
    "eg_base64url_chars": (C.c_size_t, [C.c_size_t]),
    "eg_base64url_decode_batch": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_size_t, P8, P8, P8]),
    "eg_base64url_encode_batch": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_size_t, P8, P8]),
    "eg_base64url_decode_batch_dev": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_size_t, P8, P8, P8]),
    "eg_base64url_encode_batch_dev": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_size_t, P8, P8]),
    "eg_wire_fields": (C.c_size_t, [C.c_int, C.c_uint32]),
    "eg_wire_decode_batch": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_size_t, P8, P8, P8]),
    "eg_wire_encode_batch": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_size_t, P8, P8]),
    "eg_elements_validate": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8]),
    "eg_scalars_validate": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8]),
    "eg_scalars_from_wide": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8]),
    "eg_double_mul_generator_batch": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, P8, P8, P8]),
    "eg_mul_generator_batch": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, P8]),
    "eg_ciphertexts_sum": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_size_t, P8, P8, P8]),
    "eg_ciphertexts_sum_dev": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_size_t, P8, P8, P8]),
    "eg_verify_zero_batch": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, P8]),
    "eg_verify_bool_batch": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, P8]),
    "eg_verify_choice_batch": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint32, C.c_int, P8, P8, P8, P8, P8]),
    "eg_verify_bool_batch_dev": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, P8]),
    "eg_verify_choice_batch_dev": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint32, C.c_int, P8, P8, P8, P8, P8]),
    "eg_range_optimal": (C.c_int32, [C.c_uint64, C.POINTER(Range)]),
    "eg_range_display": (C.c_size_t, [C.POINTER(Range), C.c_char_p, C.c_size_t]),
    "eg_verify_range_batch": (C.c_int32, [C.c_void_p, C.POINTER(Range), C.c_char_p, C.c_size_t, P8, P8, P8, P8]),
    "eg_verify_range_batch_dev": (C.c_int32, [C.c_void_p, C.POINTER(Range), C.c_char_p, C.c_size_t, P8, P8, P8, P8]),
    "eg_qv_params_new": (C.c_int32, [C.c_uint32, C.c_uint64, C.POINTER(QvParams)]),
    "eg_qv_ballot_size": (C.c_size_t, [C.POINTER(QvParams)]),
    "eg_verify_qv_batch": (C.c_int32, [C.c_void_p, C.POINTER(QvParams), C.c_size_t, P8, P8, P8]),
    "eg_verify_sumsq_batch": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_uint32, C.c_size_t, P8, P8, P8, P8]),
    "eg_verify_decryption_batch": (C.c_int32, [C.c_void_p, C.c_char_p, P8, C.c_size_t, P8, P8, P8, P8]),
    "eg_verify_shares_batch": (C.c_int32, [C.c_void_p, C.POINTER(KeySet), C.c_size_t, C.c_uint32, C.POINTER(C.c_uint32), P8, P8, P8, P8]),
    "eg_keysets_validate_batch": (C.c_int32, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_size_t, P8, P8, P8]),
    "eg_dlog_table_create": (C.c_int32, [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_void_p)]),
    "eg_dlog_table_destroy": (None, [C.c_void_p]),
    "eg_combine_decrypt_batch": (C.c_int32, [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_size_t, C.c_uint32, P8, P8, C.c_void_p, P8, P8]),
    "eg_verify_qv_batch_dev": (C.c_int32, [C.c_void_p, C.POINTER(QvParams), C.c_size_t, P8, P8, P8]),
    "eg_verify_shares_batch_dev": (C.c_int32, [C.c_void_p, C.POINTER(KeySet), C.c_size_t, C.c_uint32, C.POINTER(C.c_uint32), P8, P8, P8, P8]),
    "eg_combine_decrypt_batch_dev": (C.c_int32, [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_size_t, C.c_uint32, P8, P8, C.c_void_p, P8, P8]),
    "eg_encrypt_bool_batch_dev": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, P8, C.c_uint64, P8, P8]),
    "eg_encrypt_choice_batch_dev": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint32, C.c_int, P8, P8, P8, C.c_uint64, P8, P8, P8]),
    "eg_encrypt_range_batch_dev": (C.c_int32, [C.c_void_p, C.POINTER(Range), C.c_char_p, C.c_size_t, P8, P8, P8, C.c_uint64, P8, P8, P8]),
    "eg_multi_mul_batch": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint32, P8, P8, P8, P8]),
    "eg_ciphertexts_lincomb_batch": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint32, P8, P8, P8, P8]),
    "eg_encrypt_batch": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, P8]),
    "eg_encrypt_zero_batch": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, P8]),
    "eg_encrypt_bool_batch": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, P8, P8]),
    "eg_encrypt_choice_batch": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint32, C.c_int, P8, P8, P8, P8, P8]),
    "eg_encrypt_batch_seeded": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, C.c_uint64, P8]),
    "eg_encrypt_zero_batch_seeded": (C.c_int32, [C.c_void_p, C.c_size_t, P8, C.c_uint64, P8, P8]),
    "eg_encrypt_bool_batch_seeded": (C.c_int32, [C.c_void_p, C.c_size_t, P8, P8, C.c_uint64, P8, P8]),
    "eg_encrypt_choice_batch_seeded": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint32, C.c_int, P8, P8, C.c_uint64, P8, P8, P8]),
    "eg_encrypt_range_batch_seeded": (C.c_int32, [C.c_void_p, C.POINTER(Range), C.c_char_p, C.c_size_t, P8, P8, C.c_uint64, P8, P8, P8]),
    "eg_encrypt_qv_batch_seeded": (C.c_int32, [C.c_void_p, C.POINTER(QvParams), C.c_size_t, P8, P8, C.c_uint64, P8]),
    "eg_ctx_set_prover_mode": (C.c_int32, [C.c_void_p, C.c_int]),
    "eg_range_prover_draws": (C.c_size_t, [C.POINTER(Range)]),
    "eg_encrypt_range_batch": (C.c_int32, [C.c_void_p, C.POINTER(Range), C.c_char_p, C.c_size_t, P8, P8, P8, P8, P8]),
    "eg_prove_range_batch": (C.c_int32, [C.c_void_p, C.POINTER(Range), C.c_char_p, C.c_size_t, P8, P8, P8, P8, P8, P8]),
    "eg_prove_range_batch_seeded": (C.c_int32, [C.c_void_p, C.POINTER(Range), C.c_char_p, C.c_size_t, P8, P8, P8, C.c_uint64, P8, P8, P8]),
    "eg_qv_prover_draws": (C.c_size_t, [C.POINTER(QvParams)]),
    "eg_encrypt_qv_batch": (C.c_int32, [C.c_void_p, C.POINTER(QvParams), C.c_size_t, P8, P8, P8]),
    "eg_decrypt_batch": (C.c_int32, [C.c_void_p, P8, C.c_size_t, P8, C.c_void_p, P8, P8, P8]),
    "eg_decrypt_share_batch": (C.c_int32, [C.c_void_p, C.POINTER(KeySet), C.c_uint32, P8, C.c_size_t, P8, P8, P8, P8, P8]),
    "eg_decrypt_share_batch_seeded": (C.c_int32, [C.c_void_p, C.POINTER(KeySet), C.c_uint32, P8, C.c_size_t, P8, P8, C.c_uint64, P8, P8, P8]),
    "eg_decrypt_share_batch_dev": (C.c_int32, [C.c_void_p, C.POINTER(KeySet), C.c_uint32, P8, C.c_size_t, P8, P8, P8, C.c_uint64, P8, P8,
                                               P8]),
    "eg_prove_decryption_batch": (C.c_int32, [C.c_void_p, C.c_char_p, P8, C.c_size_t, P8, P8, P8, P8, P8]),
    "eg_prove_decryption_batch_seeded": (C.c_int32, [C.c_void_p, C.c_char_p, P8, C.c_size_t, P8, P8, C.c_uint64, P8, P8, P8]),
    "eg_kernel_launch_count": (C.c_uint64, [C.c_void_p]),
    "eg_last_timings": (C.c_int32, [C.c_void_p, C.POINTER(C.c_float * 5)]),
    "eg_ctx_stream": (C.c_void_p, [C.c_void_p]),
    "eg_last_commit_stats": (C.c_int32, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_float)]),
    "eg_last_kernel_stats": (C.c_int32, [C.c_void_p, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_float)]),
    "eg_selftest_field": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint64, C.POINTER(C.c_uint64)]),
    "eg_ctx_set_chunk_items": (C.c_int32, [C.c_void_p, C.c_size_t]),
    "eg_ctx_set_ring_mode": (C.c_int32, [C.c_void_p, C.c_int]),
    "eg_ctx_set_key_table_min": (C.c_int32, [C.c_void_p, C.c_size_t]),
}


def load(path=None):
    """Loads the C-ABI library.  Fails loudly when it has not been built: there is no fallback."""
    # EG_B200_LIB selects another build of the same CUDA library (A/B tuning runs); there is still no CPU fallback:
    # only an explicit `path` (the test harness) may name the CPU-compiled hostsim library.
    explicit = path is not None
    path = pathlib.Path(path) if path else pathlib.Path(os.environ.get("EG_B200_LIB", DEFAULT_LIB))
    if not path.exists():
        raise RuntimeError(f"{path} is missing: build it with `python -m elastic_elgamal_b200.build` "
                           "(the engine has no CPU fallback)")
    lib = C.CDLL(str(path))
    missing = []
    for name, (res, args) in PROTOTYPES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            missing.append(name)
            continue
        fn.restype = res
        fn.argtypes = args
    if missing:
        raise RuntimeError(f"{path} does not export: {', '.join(missing)}")
    if not explicit and b"sm_100a" not in lib.eg_version():
        raise RuntimeError(f"{path} is not a CUDA sm_100a build ({lib.eg_version().decode()}): the engine has no CPU path")
    return lib
