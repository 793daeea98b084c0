"""ctypes binding of libvrfs_b200.so (include/vrfs_b200.h).  Loading fails loudly when the library has
not been built; there is no Python / CPU implementation behind these calls."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VRFS_B200_LIB") or os.path.join(HERE, "libvrfs_b200.so")

OK, INVALID_DATA, CUDA_ERROR, BAD_ARG, UNSUPPORTED = range(5)
STATUS_NAMES = {0: "VRFS_OK", 1: "VRFS_INVALID_DATA", 2: "VRFS_CUDA_ERROR", 3: "VRFS_BAD_ARG", 4: "VRFS_UNSUPPORTED"}

# every symbol include/vrfs_b200.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "vrfs_abi_version", "vrfs_ctx_create", "vrfs_ctx_destroy", "vrfs_ctx_sync", "vrfs_last_error", "vrfs_ctx_stream",
    "vrfs_ctx_launch_count", "vrfs_ctx_enable_kernel_timing", "vrfs_ctx_kernel_timings", "vrfs_suite_challenge_len", "vrfs_suite_hash_len", "vrfs_suite_point_enc_len",
    "vrfs_secret_from_seed_batch", "vrfs_data_to_point_batch", "vrfs_output_batch", "vrfs_point_to_hash_batch",
    "vrfs_point_encode_batch", "vrfs_point_decode_batch", "vrfs_nonce_batch",
    "vrfs_ietf_prove_batch", "vrfs_ietf_verify_batch", "vrfs_ietf_verify_batch_dev",
    "vrfs_public_keys_prepare", "vrfs_public_keys_release", "vrfs_ietf_verify_prepared_batch", "vrfs_ietf_verify_prepared_batch_dev",
    "vrfs_public_keys_prepare_encoded", "vrfs_ietf_verify_prepared_wire_batch",
    "vrfs_inputs_prepare", "vrfs_inputs_release", "vrfs_ietf_verify_prepared_io_batch", "vrfs_ietf_verify_prepared_io_batch_dev",
    "vrfs_ietf_verify_prepared_io_wire_batch",
    "vrfs_pedersen_prove_batch", "vrfs_pedersen_verify_batch",
    "vrfs_suite_ietf_signature_len", "vrfs_point_decode_checked_batch", "vrfs_subgroup_check_batch", "vrfs_ietf_sign_wire_batch", "vrfs_ietf_verify_wire_batch",
    "vrfs_suite_pedersen_signature_len", "vrfs_pedersen_sign_wire_batch", "vrfs_pedersen_verify_wire_batch",
    "vrfs_msm_g1_bls12_381", "vrfs_msm_g1_bls12_381_ex", "vrfs_msm_g1_prepare", "vrfs_msm_g1_prepare_ex", "vrfs_msm_g1_prepared", "vrfs_msm_g1_prepared_partial", "vrfs_msm_g1_release", "vrfs_msm_g1_partial", "vrfs_g1_sum_partials", "vrfs_measure_mac32_peak",
    "vrfs_ctx_debug_read_staging", "vrfs_suite_pedersen_proof_len", "vrfs_pedersen_prove_compressed_batch", "vrfs_pedersen_verify_compressed_batch",
    "vrfs_ctx_peer_export", "vrfs_ctx_peer_connect", "vrfs_ctx_peer_set_timeout_ms", "vrfs_ctx_peer_world", "vrfs_msm_g1_prepared_allgather", "vrfs_ring_commit_rows_allgather",
    "vrfs_ctx_create_multi", "vrfs_mctx_destroy", "vrfs_mctx_device_count", "vrfs_mctx_device_ctx", "vrfs_mctx_last_error", "vrfs_mctx_launch_count",
    "vrfs_multi_ietf_verify_batch", "vrfs_multi_msm_g1_prepare", "vrfs_multi_msm_g1_prepared", "vrfs_multi_ring_commit", "vrfs_multi_msm_g1_release",
    "vrfs_pairing_product_batch", "vrfs_kzg_batch_verify", "vrfs_pedersen_batch_verify", "vrfs_pedersen_batch_verify_wire",
    "vrfs_host_alloc", "vrfs_host_free", "vrfs_host_register", "vrfs_host_unregister",
    "vrfs_ring_fixed_columns", "vrfs_ring_commit", "vrfs_ring_commit_delta", "vrfs_ring_commit_rows_partial", "vrfs_fr_fft_batch", "vrfs_fq381_inv_batch", "vrfs_g1_compress_batch", "vrfs_g1_decompress_batch",
]

_lib = None


class VrfsError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {msg}")
        self.status = status


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -m ark_ec_vrfs_b200.build` "
                              "(there is no CPU fallback)")
        _lib = C.CDLL(LIB_PATH)
        _lib.vrfs_last_error.restype = C.c_char_p
        _lib.vrfs_ctx_stream.restype = C.c_void_p
        _lib.vrfs_ctx_launch_count.restype = C.c_uint64
        _lib.vrfs_mctx_launch_count.restype = C.c_uint64
        _lib.vrfs_mctx_last_error.restype = C.c_char_p
        _lib.vrfs_mctx_device_ctx.restype = C.c_void_p
    return _lib
