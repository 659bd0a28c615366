"""ctypes loader for libbpperm_cuda.so (the C ABI in include/bpperm.h).

There is no CPU fallback: if the shared library is missing, or no sm_100 device is
visible, the product path raises.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# BPPERM_LIB: another build of the same library (tuning variants, tools/build_variants.sh); never a fallback
LIB_PATH = os.environ.get("BPPERM_LIB") or os.path.join(_HERE, "libbpperm_cuda.so")

# every symbol include/bpperm.h declares (tests check that the .so exports all of them)
SYMBOLS = [
    "bpp_init", "bpp_free", "bpp_set_stream", "bpp_synchronize", "bpp_strerror", "bpp_last_error",
    "bpp_launch_count", "bpp_device_info", "bpp_points_upload", "bpp_points_from_uniform", "bpp_points_compress", "bpp_points_free", "bpp_points_len",
    "bpp_comm_unique_id", "bpp_comm_init", "bpp_comm_free", "bpp_comm_info", "bpp_comm_all_gather_dev", "bpp_msm_sharded_dev", "bpp_msm_sharded_submit_dev", "bpp_msm_sharded_wait", "bpp_acp_batch_gather_accept",
    "bpp_msm_vartime", "bpp_msm_vartime_host", "bpp_points_precompute", "bpp_msm_vartime_batch", "bpp_msm_vartime_batch_dev", "bpp_msm_multi", "bpp_msm_multi_indexed", "bpp_msm_multi_dev", "bpp_msm_multi_indexed_dev", "bpp_msm_mixed", "bpp_msm_mixed_dev", "bpp_msm_vartime_dev", "bpp_msm_partial_dev", "bpp_msm_submit_dev", "bpp_msm_submit_partial_dev", "bpp_msm_wait", "bpp_msm_wait_previous",
    "bpp_points_sum_compress_dev", "bpp_set_window_bits", "bpp_set_msm_groups", "bpp_set_msm_partition", "bpp_set_msm_tile", "bpp_set_msm_trace", "bpp_msm_trace_dump", "bpp_bench_imad_peak", "bpp_device_clock_khz", "bpp_bench_pipe_probe", "bpp_set_profiling",
    "bpp_last_phase_ms", "bpp_last_op_counts", "bpp_test_op",
    "bpp_inner_product", "bpp_hadamard_V", "bpp_vm_mult", "bpp_mv_mult", "bpp_exp_iter", "bpp_scalar_powers",
    "bpp_scalar_exp", "bpp_scalar_invert", "bpp_scalar_from_wide", "bpp_scalar_reduce",
    "bpp_vecpoly3_special_inner_product", "bpp_vecpoly3_eval", "bpp_poly6_eval",
    "bpp_circuit_create", "bpp_circuit_create_shuffle", "bpp_circuit_free", "bpp_gens_create", "bpp_gens_free", "bpp_acproof_proof_len", "bpp_acproof_proof_len_mode", "bpp_acproof_wire_len", "bpp_acproof_to_wire", "bpp_acproof_from_wire",
    "bpp_acproof_prove_batch", "bpp_acproof_verify_batch", "bpp_acp_batch_create", "bpp_acp_batch_free",
    "bpp_acp_batch_upload_witness", "bpp_acp_batch_commit", "bpp_acp_batch_upload_commitments", "bpp_acp_batch_gen_shuffle_witness", "bpp_acp_batch_prove", "bpp_acp_batch_download_proofs",
    "bpp_acp_batch_upload_proofs", "bpp_acp_batch_verify", "bpp_acp_batch_download_accept",
    "bpp_acp_batch_time_commit_msm", "bpp_acp_batch_set_host_transcripts", "bpp_transcript_script", "bpp_ipa_fold_generators", "bpp_acp_batch_set_batch_rlc", "bpp_acp_batch_set_priority_split",
    "bpp_transcript_new", "bpp_transcript_append_message", "bpp_transcript_challenge_bytes",
    "bpp_ipa_proof_len", "bpp_ipa_batch_create", "bpp_ipa_batch_free", "bpp_ipa_batch_prove", "bpp_ipa_batch_verify",
    "bpp_ipa_batch_verify_combined", "bpp_ipa_batch_gather_accept", "bpp_ipa_batch_download_weights",
]

_lib = None


class BppError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"bpperm status {status}: {msg}")
        self.status = status


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing - build it with `python -c 'import __graft_entry__ as g; g.build()'`; "
            "this backend has no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    c = ctypes
    vp, sz, u8p = c.c_void_p, c.c_size_t, c.c_char_p
    lib.bpp_init.argtypes = [c.c_int, c.POINTER(vp)]
    lib.bpp_free.argtypes = [vp]
    lib.bpp_free.restype = None
    lib.bpp_set_stream.argtypes = [vp, vp]
    lib.bpp_synchronize.argtypes = [vp]
    lib.bpp_strerror.argtypes = [c.c_int]
    lib.bpp_strerror.restype = c.c_char_p
    lib.bpp_last_error.argtypes = [vp]
    lib.bpp_last_error.restype = c.c_char_p
    lib.bpp_launch_count.argtypes = [vp]
    lib.bpp_launch_count.restype = c.c_uint64
    lib.bpp_device_info.argtypes = [vp, c.POINTER(c.c_int), c.POINTER(c.c_int), c.POINTER(c.c_int), c.POINTER(sz)]
    lib.bpp_points_upload.argtypes = [vp, c.c_int, u8p, sz, c.POINTER(vp)]
    lib.bpp_points_from_uniform.argtypes = [vp, u8p, sz, c.POINTER(vp)]
    lib.bpp_points_compress.argtypes = [vp, vp, sz, sz, c.c_char_p]
    lib.bpp_points_free.argtypes = [vp, vp]
    lib.bpp_points_free.restype = None
    lib.bpp_points_len.argtypes = [vp]
    lib.bpp_points_len.restype = sz
    lib.bpp_msm_vartime.argtypes = [vp, u8p, sz, vp, sz, sz, c.c_char_p, c.c_char_p]
    lib.bpp_msm_vartime_host.argtypes = [vp, u8p, sz, c.c_int, u8p, sz, c.c_char_p]
    lib.bpp_comm_unique_id.argtypes = [c.c_char_p]
    lib.bpp_comm_init.argtypes = [vp, c.c_int, c.c_int, u8p]
    lib.bpp_comm_free.argtypes = [vp]
    lib.bpp_comm_info.argtypes = [vp, c.POINTER(c.c_int), c.POINTER(c.c_int)]
    lib.bpp_comm_all_gather_dev.argtypes = [vp, vp, sz, vp]
    lib.bpp_msm_sharded_dev.argtypes = [vp, vp, vp, sz, sz, vp]
    lib.bpp_msm_sharded_submit_dev.argtypes = [vp, vp, vp, sz, sz, vp]
    lib.bpp_msm_sharded_wait.argtypes = [vp]
    lib.bpp_acp_batch_gather_accept.argtypes = [vp, sz, c.c_char_p]
    lib.bpp_points_precompute.argtypes = [vp, vp, c.c_int]
    lib.bpp_msm_vartime_batch.argtypes = [vp, u8p, sz, vp, sz, sz, c.c_char_p]
    lib.bpp_msm_vartime_batch_dev.argtypes = [vp, vp, sz, vp, sz, sz, vp]
    u32p = c.POINTER(c.c_uint32)
    lib.bpp_msm_multi.argtypes = [vp, sz, u32p, u8p, u8p, c.c_char_p, c.c_char_p]
    lib.bpp_msm_multi_indexed.argtypes = [vp, sz, u32p, u8p, vp, u32p, c.c_char_p]
    lib.bpp_msm_multi_dev.argtypes = [vp, sz, u32p, vp, vp, vp, vp]
    lib.bpp_msm_multi_indexed_dev.argtypes = [vp, sz, u32p, vp, vp, vp, vp]
    lib.bpp_msm_mixed.argtypes = [vp, sz, vp, sz, sz, u8p, u32p, u8p, u8p, c.c_char_p, c.c_char_p]
    lib.bpp_msm_mixed_dev.argtypes = [vp, sz, vp, sz, sz, vp, u32p, vp, vp, vp, vp]
    lib.bpp_msm_vartime_dev.argtypes = [vp, vp, vp, sz, sz, vp]
    lib.bpp_msm_partial_dev.argtypes = [vp, vp, vp, sz, sz, vp]
    lib.bpp_msm_submit_dev.argtypes = [vp, vp, vp, sz, sz, vp]
    lib.bpp_msm_submit_partial_dev.argtypes = [vp, vp, vp, sz, sz, vp]
    lib.bpp_msm_wait.argtypes = [vp]
    lib.bpp_msm_wait_previous.argtypes = [vp]
    lib.bpp_points_sum_compress_dev.argtypes = [vp, vp, sz, vp]
    lib.bpp_set_window_bits.argtypes = [vp, c.c_int]
    lib.bpp_set_msm_groups.argtypes = [vp, c.c_int]
    lib.bpp_set_msm_tile.argtypes = [vp, c.c_int]
    lib.bpp_set_msm_partition.argtypes = [vp, c.POINTER(c.c_int), c.c_int]
    lib.bpp_set_msm_trace.argtypes = [vp, c.c_int]
    lib.bpp_msm_trace_dump.argtypes = [vp, c.c_char_p, sz]
    lib.bpp_device_clock_khz.argtypes = [vp]
    lib.bpp_bench_imad_peak.argtypes = [vp, c.c_int, c.POINTER(c.c_double), c.POINTER(c.c_double)]
    lib.bpp_bench_pipe_probe.argtypes = [vp, c.c_int, c.c_int, c.POINTER(c.c_double)]
    lib.bpp_set_profiling.argtypes = [vp, c.c_int]
    lib.bpp_last_phase_ms.argtypes = [vp, c.POINTER(c.c_float)]
    lib.bpp_last_op_counts.argtypes = [vp, c.POINTER(c.c_uint64), c.POINTER(c.c_uint64), c.POINTER(c.c_uint64)]
    lib.bpp_test_op.argtypes = [vp, c.c_int, u8p, u8p, c.c_char_p, sz]
    lib.bpp_inner_product.argtypes = [vp, u8p, sz, u8p, sz, c.c_char_p]
    lib.bpp_hadamard_V.argtypes = [vp, u8p, sz, u8p, sz, c.c_char_p]
    lib.bpp_vm_mult.argtypes = [vp, u8p, sz, u8p, sz, sz, c.c_char_p]
    lib.bpp_mv_mult.argtypes = [vp, u8p, sz, sz, u8p, sz, c.c_char_p]
    lib.bpp_exp_iter.argtypes = [vp, u8p, sz, c.c_char_p]
    lib.bpp_scalar_powers.argtypes = [vp, u8p, sz, sz, c.c_char_p]
    lib.bpp_scalar_exp.argtypes = [vp, u8p, c.c_uint32, c.c_char_p]
    lib.bpp_scalar_invert.argtypes = [vp, u8p, sz, c.c_char_p]
    lib.bpp_scalar_from_wide.argtypes = [vp, u8p, sz, c.c_char_p]
    lib.bpp_scalar_reduce.argtypes = [vp, u8p, sz, c.c_char_p]
    lib.bpp_vecpoly3_special_inner_product.argtypes = [vp, u8p, u8p, sz, c.c_char_p]
    lib.bpp_vecpoly3_eval.argtypes = [vp, u8p, sz, u8p, c.c_char_p]
    lib.bpp_poly6_eval.argtypes = [vp, u8p, u8p, c.c_char_p]
    u32p = c.POINTER(c.c_uint32)
    lib.bpp_circuit_create.argtypes = [vp, sz, sz, sz, u32p, u32p, u32p, u8p, u8p, c.POINTER(vp)]
    lib.bpp_circuit_create_shuffle.argtypes = [vp, sz, c.POINTER(vp)]
    lib.bpp_acp_batch_gen_shuffle_witness.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.bpp_circuit_free.argtypes = [vp, vp]
    lib.bpp_circuit_free.restype = None
    lib.bpp_gens_create.argtypes = [vp, u8p, u8p, u8p, u8p, sz, c.c_int, c.POINTER(vp)]
    lib.bpp_gens_free.argtypes = [vp, vp]
    lib.bpp_gens_free.restype = None
    lib.bpp_acproof_proof_len.argtypes = [sz]
    lib.bpp_acproof_wire_len.restype = sz
    lib.bpp_acproof_wire_len.argtypes = [sz, c.c_int]
    lib.bpp_acproof_to_wire.argtypes = [sz, c.c_int, sz, u8p, c.c_char_p]
    lib.bpp_acproof_from_wire.argtypes = [sz, c.c_int, sz, u8p, sz, c.c_char_p, c.c_char_p]
    lib.bpp_acproof_proof_len.restype = sz
    lib.bpp_acproof_proof_len_mode.argtypes = [sz, c.c_int]
    lib.bpp_acproof_proof_len_mode.restype = sz
    lib.bpp_acproof_prove_batch.argtypes = [vp, vp, vp, c.c_int, sz, u8p, u8p, u8p, u8p, u8p, u8p, u8p, sz, c.c_char_p]
    lib.bpp_acproof_verify_batch.argtypes = [vp, vp, vp, c.c_int, sz, u8p, u8p, u8p, sz, u8p, c.c_char_p]
    lib.bpp_acp_batch_create.argtypes = [vp, vp, vp, c.c_int, sz, u8p, sz, c.POINTER(vp)]
    lib.bpp_acp_batch_free.argtypes = [vp]
    lib.bpp_acp_batch_free.restype = None
    # host buffers as void*: bytes objects or raw addresses of pinned memory
    lib.bpp_acp_batch_upload_witness.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.bpp_acp_batch_commit.argtypes = [vp, vp, vp]
    lib.bpp_acp_batch_upload_commitments.argtypes = [vp, vp]
    lib.bpp_acp_batch_prove.argtypes = [vp]
    lib.bpp_acp_batch_download_proofs.argtypes = [vp, vp]
    lib.bpp_acp_batch_upload_proofs.argtypes = [vp, vp, vp]
    lib.bpp_acp_batch_verify.argtypes = [vp, u8p]
    lib.bpp_acp_batch_download_accept.argtypes = [vp, vp]
    lib.bpp_acp_batch_set_host_transcripts.argtypes = [vp, c.c_int]
    lib.bpp_acp_batch_set_batch_rlc.argtypes = [vp, c.c_int]
    lib.bpp_acp_batch_set_priority_split.argtypes = [vp, c.c_int]
    lib.bpp_ipa_fold_generators.argtypes = [vp, vp, sz, sz, u8p, u8p, sz, c.c_char_p, c.POINTER(c.c_float)]
    lib.bpp_transcript_script.argtypes = [vp, u8p, sz, c.c_char_p, sz]
    lib.bpp_acp_batch_time_commit_msm.argtypes = [vp, c.c_int, c.POINTER(c.c_float), c.POINTER(c.c_uint64),
                                                  c.POINTER(c.c_uint64)]
    # transcripts (host only) and the stand-alone inner-product batch; in/out buffers as char* (ctypes string buffers)
    lib.bpp_transcript_new.argtypes = [u8p, sz, c.c_char_p]
    lib.bpp_transcript_append_message.argtypes = [c.c_char_p, u8p, sz, u8p, sz]
    lib.bpp_transcript_challenge_bytes.argtypes = [c.c_char_p, u8p, sz, c.c_char_p, sz]
    lib.bpp_ipa_proof_len.argtypes = [sz]
    lib.bpp_ipa_proof_len.restype = sz
    lib.bpp_ipa_batch_create.argtypes = [vp, vp, sz, sz, sz, sz, sz, c.POINTER(vp)]
    lib.bpp_ipa_batch_free.argtypes = [vp]
    lib.bpp_ipa_batch_free.restype = None
    lib.bpp_ipa_batch_prove.argtypes = [vp, u8p, u8p, u8p, u8p, u8p, c.c_char_p, c.c_char_p]
    lib.bpp_ipa_batch_verify.argtypes = [vp, u8p, u8p, u8p, u8p, u8p, c.c_char_p, c.c_char_p]
    lib.bpp_ipa_batch_verify_combined.argtypes = [vp, u8p, u8p, u8p, u8p, u8p, u8p, c.c_char_p, c.c_char_p]
    lib.bpp_ipa_batch_gather_accept.argtypes = [vp, sz, c.c_char_p]
    lib.bpp_ipa_batch_download_weights.argtypes = [vp, c.c_char_p]
    _lib = lib
    return lib
