//! Raw bindings to include/bpperm.h (hand-written, bindgen-free).  Status codes: 0 = ok, negative = error
//! (`bpp_strerror`).  Every pointer is caller-owned; the library never frees caller memory.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int};

#[repr(C)] pub struct bpp_ctx { _p: [u8; 0] }
#[repr(C)] pub struct bpp_points { _p: [u8; 0] }
#[repr(C)] pub struct bpp_circuit { _p: [u8; 0] }
#[repr(C)] pub struct bpp_gens { _p: [u8; 0] }
#[repr(C)] pub struct bpp_acp_batch { _p: [u8; 0] }
#[repr(C)] pub struct bpp_ipa_batch { _p: [u8; 0] }

pub const BPP_OK: c_int = 0;
pub const BPP_ERR_LENGTH_MISMATCH: c_int = -4;
pub const BPP_FMT_COMPRESSED: c_int = 0; // 32 B RFC 9496 encodings
pub const BPP_FMT_AFFINE: c_int = 1;     // 64 B (x, y) canonical little endian
pub const BPP_FMT_DALEK_XYZT: c_int = 2; // 160 B EdwardsPoint { X, Y, Z, T: FieldElement51([u64; 5]) }
pub const MODE_REFERENCE: c_int = 0;
pub const MODE_REFERENCE_FIXED: c_int = 1;
pub const MODE_FIXED: c_int = 2;
/// merlin Transcript state across the ABI: 25 Keccak lanes + pos | pos_begin << 8 | cur_flags << 16, little-endian u64
pub const BPP_TRANSCRIPT_BYTES: usize = 208;

extern "C" {
    pub fn bpp_init(device: c_int, out: *mut *mut bpp_ctx) -> c_int;
    pub fn bpp_free(ctx: *mut bpp_ctx);
    pub fn bpp_strerror(status: c_int) -> *const c_char;
    pub fn bpp_last_error(ctx: *mut bpp_ctx) -> *const c_char;
    pub fn bpp_synchronize(ctx: *mut bpp_ctx) -> c_int;

    pub fn bpp_points_upload(ctx: *mut bpp_ctx, fmt: c_int, pts: *const u8, n: usize, out: *mut *mut bpp_points) -> c_int;
    pub fn bpp_points_free(ctx: *mut bpp_ctx, p: *mut bpp_points);
    pub fn bpp_points_len(p: *const bpp_points) -> usize;
    pub fn bpp_msm_vartime(ctx: *mut bpp_ctx, scalars: *const u8, n_scalars: usize, points: *const bpp_points, off: usize,
                           n: usize, out_compressed: *mut u8, out_ext: *mut u8) -> c_int;
    pub fn bpp_msm_vartime_host(ctx: *mut bpp_ctx, scalars: *const u8, n_scalars: usize, fmt: c_int, pts: *const u8,
                                n_points: usize, out_compressed: *mut u8) -> c_int;

    // device-pointer forms: scalars / results already in HBM (pointers from the caller's CUDA allocator)
    pub fn bpp_set_stream(ctx: *mut bpp_ctx, cuda_stream: *mut core::ffi::c_void) -> c_int;
    pub fn bpp_msm_vartime_dev(ctx: *mut bpp_ctx, d_scalars: *const core::ffi::c_void, points: *const bpp_points, off: usize,
                               n: usize, d_out: *mut core::ffi::c_void) -> c_int;
    // throughput form: submit without joining, up to two MSMs in flight; results valid after bpp_msm_wait
    pub fn bpp_msm_submit_dev(ctx: *mut bpp_ctx, d_scalars: *const core::ffi::c_void, points: *const bpp_points, off: usize,
                              n: usize, d_out: *mut core::ffi::c_void) -> c_int;
    pub fn bpp_msm_wait(ctx: *mut bpp_ctx) -> c_int;
    pub fn bpp_msm_wait_previous(ctx: *mut bpp_ctx) -> c_int;
    pub fn bpp_msm_partial_dev(ctx: *mut bpp_ctx, d_scalars: *const core::ffi::c_void, points: *const bpp_points, off: usize,
                               n: usize, d_partial: *mut core::ffi::c_void) -> c_int;
    pub fn bpp_points_sum_compress_dev(ctx: *mut bpp_ctx, d_partials: *const core::ffi::c_void, g: usize,
                                       d_out32: *mut core::ffi::c_void) -> c_int;
    // long-lived point sets: window table once, then small MSMs and `count` MSMs per launch without buckets or doublings
    pub fn bpp_points_precompute(ctx: *mut bpp_ctx, points: *mut bpp_points, window_bits: c_int) -> c_int;
    pub fn bpp_msm_vartime_batch(ctx: *mut bpp_ctx, scalars: *const u8, count: usize, points: *mut bpp_points, off: usize, n: usize,
                                 out32: *mut u8) -> c_int;
    pub fn bpp_msm_vartime_batch_dev(ctx: *mut bpp_ctx, d_scalars: *const core::ffi::c_void, count: usize, points: *mut bpp_points,
                                     off: usize, n: usize, d_out32: *mut core::ffi::c_void) -> c_int;
    // many independent MSMs over caller points: MSM j takes the next sizes[j] terms (sizes: host memory)
    pub fn bpp_msm_multi(ctx: *mut bpp_ctx, count: usize, sizes: *const u32, scalars: *const u8, points_enc: *const u8,
                         out32: *mut u8, ok: *mut u8) -> c_int;
    pub fn bpp_msm_multi_indexed(ctx: *mut bpp_ctx, count: usize, sizes: *const u32, scalars: *const u8,
                                 points: *const bpp_points, index: *const u32, out32: *mut u8) -> c_int;
    pub fn bpp_msm_multi_dev(ctx: *mut bpp_ctx, count: usize, sizes: *const u32, d_scalars: *const core::ffi::c_void,
                             d_points_enc: *const core::ffi::c_void, d_out32: *mut core::ffi::c_void,
                             d_ok: *mut core::ffi::c_void) -> c_int;
    pub fn bpp_msm_multi_indexed_dev(ctx: *mut bpp_ctx, count: usize, sizes: *const u32, d_scalars: *const core::ffi::c_void,
                                     points: *const bpp_points, d_index: *const core::ffi::c_void,
                                     d_out32: *mut core::ffi::c_void) -> c_int;
    // multi-GPU: one process per GPU, NCCL inside the library
    pub fn bpp_comm_unique_id(id: *mut u8) -> c_int;                      // 128 bytes, made on rank 0
    pub fn bpp_comm_init(ctx: *mut bpp_ctx, nranks: c_int, rank: c_int, id: *const u8) -> c_int;
    pub fn bpp_comm_free(ctx: *mut bpp_ctx) -> c_int;
    pub fn bpp_comm_info(ctx: *mut bpp_ctx, nranks: *mut c_int, rank: *mut c_int) -> c_int;
    pub fn bpp_comm_all_gather_dev(ctx: *mut bpp_ctx, d_send: *const core::ffi::c_void, bytes_per_rank: usize,
                                   d_recv: *mut core::ffi::c_void) -> c_int;
    pub fn bpp_msm_sharded_dev(ctx: *mut bpp_ctx, d_scalars: *const core::ffi::c_void, points: *const bpp_points, off: usize,
                               n: usize, d_out32: *mut core::ffi::c_void) -> c_int;
    pub fn bpp_msm_sharded_submit_dev(ctx: *mut bpp_ctx, d_scalars: *const core::ffi::c_void, points: *const bpp_points, off: usize,
                                      n: usize, d_out32: *mut core::ffi::c_void) -> c_int;
    pub fn bpp_msm_sharded_wait(ctx: *mut bpp_ctx) -> c_int;
    // result-neutral tuning hooks
    pub fn bpp_set_window_bits(ctx: *mut bpp_ctx, c: c_int) -> c_int;
    pub fn bpp_set_msm_groups(ctx: *mut bpp_ctx, groups: c_int) -> c_int;
    pub fn bpp_set_msm_partition(ctx: *mut bpp_ctx, sizes: *const c_int, count: c_int) -> c_int;

    pub fn bpp_inner_product(ctx: *mut bpp_ctx, a: *const u8, la: usize, b: *const u8, lb: usize, out: *mut u8) -> c_int;
    pub fn bpp_hadamard_V(ctx: *mut bpp_ctx, a: *const u8, la: usize, b: *const u8, lb: usize, out: *mut u8) -> c_int;
    pub fn bpp_vm_mult(ctx: *mut bpp_ctx, a: *const u8, la: usize, b: *const u8, rows: usize, cols: usize, out: *mut u8) -> c_int;
    pub fn bpp_mv_mult(ctx: *mut bpp_ctx, a: *const u8, rows: usize, cols: usize, b: *const u8, lb: usize, out: *mut u8) -> c_int;
    pub fn bpp_exp_iter(ctx: *mut bpp_ctx, x: *const u8, count: usize, out: *mut u8) -> c_int;
    pub fn bpp_scalar_exp(ctx: *mut bpp_ctx, x: *const u8, pow: u32, out: *mut u8) -> c_int;
    pub fn bpp_scalar_invert(ctx: *mut bpp_ctx, a: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn bpp_scalar_powers(ctx: *mut bpp_ctx, x: *const u8, first: usize, count: usize, out: *mut u8) -> c_int;
    pub fn bpp_scalar_reduce(ctx: *mut bpp_ctx, in32: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn bpp_scalar_from_wide(ctx: *mut bpp_ctx, in64: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn bpp_vecpoly3_special_inner_product(ctx: *mut bpp_ctx, lhs: *const u8, rhs: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn bpp_vecpoly3_eval(ctx: *mut bpp_ctx, coeffs: *const u8, n: usize, x: *const u8, out: *mut u8) -> c_int;
    pub fn bpp_poly6_eval(ctx: *mut bpp_ctx, t1_t6: *const u8, x: *const u8, out: *mut u8) -> c_int;

    pub fn bpp_circuit_create(ctx: *mut bpp_ctx, n: usize, q: usize, m: usize, nnz: *const u32, wire: *const u32,
                              constraint: *const u32, coeff: *const u8, c_vec: *const u8, out: *mut *mut bpp_circuit) -> c_int;
    /// weights.rs:130-204 replaced: the corrected k-card shuffle circuit built inside the library
    pub fn bpp_circuit_create_shuffle(ctx: *mut bpp_ctx, k: usize, out: *mut *mut bpp_circuit) -> c_int;
    pub fn bpp_circuit_free(ctx: *mut bpp_ctx, c: *mut bpp_circuit);
    pub fn bpp_gens_create(ctx: *mut bpp_ctx, g: *const u8, h: *const u8, g_vec: *const u8, h_vec: *const u8, n: usize,
                           window_bits: c_int, out: *mut *mut bpp_gens) -> c_int;
    pub fn bpp_gens_free(ctx: *mut bpp_ctx, g: *mut bpp_gens);
    pub fn bpp_acproof_proof_len_mode(n: usize, mode: c_int) -> usize;
    // wire records: version byte + proof bytes (mode 2 = bulletproofs R1CSProof::to_bytes, one-phase); no context needed
    pub fn bpp_acproof_wire_len(n: usize, mode: c_int) -> usize;
    pub fn bpp_acproof_to_wire(n: usize, mode: c_int, count: usize, proofs: *const u8, wire_out: *mut u8) -> c_int;
    pub fn bpp_acproof_from_wire(n: usize, mode: c_int, count: usize, wire: *const u8, wire_len: usize,
                                 proofs_out: *mut u8, status: *mut u8) -> c_int;
    /// v: count x m x 32 compressed commitments - required in modes 1 and 2 (bound to every transcript), null in mode 0
    pub fn bpp_acproof_prove_batch(ctx: *mut bpp_ctx, cir: *const bpp_circuit, gens: *const bpp_gens, mode: c_int, count: usize,
                                   a_l: *const u8, a_r: *const u8, a_o: *const u8, gamma: *const u8, seeds: *const u8,
                                   v: *const u8, label: *const u8, label_len: usize, proofs_out: *mut u8) -> c_int;
    pub fn bpp_acproof_verify_batch(ctx: *mut bpp_ctx, cir: *const bpp_circuit, gens: *const bpp_gens, mode: c_int, count: usize,
                                    proofs: *const u8, v: *const u8, label: *const u8, label_len: usize,
                                    verifier_seed: *const u8, accept: *mut u8) -> c_int;
    pub fn bpp_acp_batch_create(ctx: *mut bpp_ctx, cir: *const bpp_circuit, gens: *const bpp_gens, mode: c_int, count: usize,
                                label: *const u8, label_len: usize, out: *mut *mut bpp_acp_batch) -> c_int;
    pub fn bpp_acp_batch_free(b: *mut bpp_acp_batch);
    pub fn bpp_acp_batch_upload_witness(b: *mut bpp_acp_batch, a_l: *const u8, a_r: *const u8, a_o: *const u8,
                                        gamma: *const u8, seeds: *const u8) -> c_int;
    /// weights.rs:38-113 replaced: a_L, a_R, a_O and v = deck | deck[perm] | x computed on the device
    pub fn bpp_acp_batch_gen_shuffle_witness(b: *mut bpp_acp_batch, deck: *const u8, perm: *const u32, x: *const u8,
                                             gamma: *const u8, seeds: *const u8) -> c_int;
    /// v nullable: commit to the values left by bpp_acp_batch_gen_shuffle_witness
    pub fn bpp_acp_batch_commit(b: *mut bpp_acp_batch, v: *const u8, v_out: *mut u8) -> c_int;
    pub fn bpp_acp_batch_upload_commitments(b: *mut bpp_acp_batch, v: *const u8) -> c_int;
    /// sharded batch verification: all ranks' accept bytes (nranks x per) through the library's communicator
    pub fn bpp_acp_batch_gather_accept(b: *mut bpp_acp_batch, per: usize, accept_all: *mut u8) -> c_int;
    pub fn bpp_acp_batch_prove(b: *mut bpp_acp_batch) -> c_int;
    pub fn bpp_acp_batch_download_proofs(b: *mut bpp_acp_batch, proofs_out: *mut u8) -> c_int;
    pub fn bpp_acp_batch_upload_proofs(b: *mut bpp_acp_batch, proofs: *const u8, v: *const u8) -> c_int;
    pub fn bpp_acp_batch_verify(b: *mut bpp_acp_batch, verifier_seed: *const u8) -> c_int;
    pub fn bpp_acp_batch_download_accept(b: *mut bpp_acp_batch, accept: *mut u8) -> c_int;
    pub fn bpp_acp_batch_set_host_transcripts(b: *mut bpp_acp_batch, on: c_int) -> c_int;
    pub fn bpp_acp_batch_set_batch_rlc(b: *mut bpp_acp_batch, on: c_int) -> c_int;
    pub fn bpp_acp_batch_set_priority_split(b: *mut bpp_acp_batch, on: c_int) -> c_int;

    // transcripts across the ABI (host only) and the stand-alone inner-product argument (inner_product_proof.rs)
    pub fn bpp_transcript_new(label: *const u8, label_len: usize, state: *mut u8) -> c_int;
    pub fn bpp_transcript_append_message(state: *mut u8, label: *const u8, label_len: usize, msg: *const u8, msg_len: usize) -> c_int;
    pub fn bpp_transcript_challenge_bytes(state: *mut u8, label: *const u8, label_len: usize, out: *mut u8, out_len: usize) -> c_int;
    pub fn bpp_ipa_proof_len(n: usize) -> usize;
    pub fn bpp_ipa_batch_create(ctx: *mut bpp_ctx, gens: *mut bpp_points, g_off: usize, h_off: usize, q_off: usize, n: usize,
                                count: usize, out: *mut *mut bpp_ipa_batch) -> c_int;
    pub fn bpp_ipa_batch_free(b: *mut bpp_ipa_batch);
    /// q, G_factors, H_factors nullable (= ones); transcripts: count x BPP_TRANSCRIPT_BYTES, in/out
    pub fn bpp_ipa_batch_prove(b: *mut bpp_ipa_batch, q: *const u8, g_factors: *const u8, h_factors: *const u8, a: *const u8,
                               b_vec: *const u8, transcripts: *mut u8, proofs_out: *mut u8) -> c_int;
    pub fn bpp_ipa_batch_verify(b: *mut bpp_ipa_batch, q: *const u8, g_factors: *const u8, h_factors: *const u8, p: *const u8,
                                proofs: *const u8, transcripts: *mut u8, accept: *mut u8) -> c_int;
    /// verify's decisions through one random-linear-combination MSM; verifier_seed nullable (= from the OS)
    pub fn bpp_ipa_batch_verify_combined(b: *mut bpp_ipa_batch, q: *const u8, g_factors: *const u8, h_factors: *const u8,
                                         p: *const u8, proofs: *const u8, verifier_seed: *const u8, transcripts: *mut u8,
                                         accept: *mut u8) -> c_int;
    /// sharded verification: all ranks' accept bytes (nranks x per) through the library's communicator
    pub fn bpp_ipa_batch_gather_accept(b: *mut bpp_ipa_batch, per: usize, accept_all: *mut u8) -> c_int;
    /// audit / test hook: rho_p of the last combined check (count x 32)
    pub fn bpp_ipa_batch_download_weights(b: *mut bpp_ipa_batch, rho: *mut u8) -> c_int;
}
