/* bpperm.h - C ABI of the B200 (sm_100a) backend for bulletproof-perm's hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  Every
 * entry point names the reference interface it replaces.  The reference
 * (/root/reference/bp-perm, Rust) reaches its group arithmetic through the dalek trait
 *     curve25519_dalek_ng::traits::VartimeMultiscalarMul      (circuit_lib.rs:11, lib.rs:27)
 * invoked as RistrettoPoint::vartime_multiscalar_mul(scalars, points) at
 * circuit_lib.rs:187,202,216,363,374,385,396,407,498,504,509,525,535,552,568, and its scalar
 * vector work through the free functions of util.rs / poly.rs.  INTEGRATION.md shows the Rust
 * `extern "C"` block and the `impl VartimeMultiscalarMul for GpuRistretto` that bind these symbols.
 *
 * Conventions
 *   - every function returns BPP_OK (0) or a negative bpp_status; nothing aborts or throws.
 *   - scalars are 32-byte little-endian integers with bit 255 clear (dalek `Scalar` invariant);
 *     canonical (< l) wherever a scalar is an arithmetic operand of the mod-l kernels.
 *   - compressed points are 32-byte RFC 9496 ristretto255 encodings.
 *   - "host" entry points take host pointers and include the host<->device copies;
 *     "_dev" entry points take device pointers and enqueue on the context's stream.
 *   - a context is bound to one GPU and one stream; use one context per thread.  Work is stream-ordered on that
 *     stream: a large MSM internally forks onto the library's own streams (window groups, msm_kernels.cuh) and joins
 *     back before the call's result is used, so the caller sees ordinary stream semantics; only the explicit
 *     throughput form (bpp_msm_submit_dev / bpp_msm_wait) leaves work in flight across calls.
 *   - there is no CPU fallback: without a CUDA device bpp_init fails with BPP_ERR_NO_DEVICE.
 */
#ifndef BPPERM_H
#define BPPERM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum bpp_status {
    BPP_OK = 0,
    BPP_ERR_NO_DEVICE = -1,     /* no CUDA device / wrong architecture */
    BPP_ERR_CUDA = -2,          /* a CUDA runtime call failed; see bpp_last_error() */
    BPP_ERR_INVALID_ARG = -3,   /* null pointer, zero where non-zero is required, bad enum */
    BPP_ERR_LENGTH_MISMATCH = -4, /* dalek panics when the two iterators differ in length (edwards.rs) */
    BPP_ERR_INVALID_POINT = -5, /* a compressed point failed RFC 9496 decoding (dalek: decompress() -> None) */
    BPP_ERR_SCALAR_RANGE = -6,  /* a scalar has bit 255 set */
    BPP_ERR_OOM = -7,
    BPP_ERR_VERIFICATION = -8   /* bulletproofs::ProofError::VerificationError (circuit_lib.rs:487,519,543) */
} bpp_status;

typedef struct bpp_ctx bpp_ctx;
typedef struct bpp_points bpp_points;

/* point input formats */
enum {
    BPP_FMT_COMPRESSED = 0, /* 32 B RFC 9496 encoding (CompressedRistretto) */
    BPP_FMT_AFFINE = 1,     /* 64 B: x || y, each 32-byte little-endian, any representative of the Ristretto coset */
    BPP_FMT_DALEK_XYZT = 2  /* 160 B: dalek-ng in-memory RistrettoPoint = EdwardsPoint{X,Y,Z,T: FieldElement51([u64;5])} */
};

/* ---- lifecycle ---------------------------------------------------------------------------- */
int bpp_init(int device, bpp_ctx **out);
void bpp_free(bpp_ctx *ctx);
/* Enqueue on an existing CUDA stream (a cudaStream_t passed as void*) instead of the context's own. */
int bpp_set_stream(bpp_ctx *ctx, void *cuda_stream);
int bpp_synchronize(bpp_ctx *ctx);
const char *bpp_strerror(int status);
const char *bpp_last_error(bpp_ctx *ctx);
/* Number of kernels this context has launched since creation (bench.py's `gpu_launches`). */
uint64_t bpp_launch_count(bpp_ctx *ctx);
int bpp_device_info(bpp_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem);
/* Maximum SM clock in kHz (cudaDevAttrClockRate); the IMAD.WIDE pipe limit is sm_count * 32 lanes * this. */
int bpp_device_clock_khz(bpp_ctx *ctx);

/* ---- points: upload once, reuse across MSMs (generators are static in the protocol) -------- */
/* Converts n points to the device layout (affine Niels, 96 B/point).  For BPP_FMT_COMPRESSED an
 * invalid encoding yields BPP_ERR_INVALID_POINT (dalek: decompress().unwrap() panics, circuit_lib.rs:532). */
int bpp_points_upload(bpp_ctx *ctx, int fmt, const uint8_t *pts, size_t n, bpp_points **out);
/* RistrettoPoint::from_uniform_bytes / RistrettoPoint::random(rng) (lib.rs:165-166,179-180): n x 64 uniform
 * bytes -> n points (RFC 9496 one-way map), kept on the device. */
int bpp_points_from_uniform(bpp_ctx *ctx, const uint8_t *bytes64, size_t n, bpp_points **out);
/* RistrettoPoint::compress for points[off .. off+n): n x 32 bytes to host memory. */
int bpp_points_compress(bpp_ctx *ctx, const bpp_points *points, size_t off, size_t n, uint8_t *out32);
void bpp_points_free(bpp_ctx *ctx, bpp_points *p);
size_t bpp_points_len(const bpp_points *p);

/* ---- multiscalar multiplication ------------------------------------------------------------
 * Replaces RistrettoPoint::vartime_multiscalar_mul (dalek-ng 4.1.1 traits.rs / edwards.rs
 * optional_multiscalar_mul; Straus below 190 points, Pippenger above).  Result = sum_i s_i * P_i
 * over points[off .. off+n).  out_compressed receives the canonical 32-byte encoding
 * (== result.compress().to_bytes()); out_ext (nullable) receives X,Y,Z,T as 4 x 32-byte
 * canonical little-endian field elements (128 B) for callers that keep an uncompressed point. */
int bpp_msm_vartime(bpp_ctx *ctx, const uint8_t *scalars, size_t n_scalars, const bpp_points *points, size_t off,
                    size_t n, uint8_t out_compressed[32], uint8_t *out_ext /* 128 B or NULL */);
/* One-shot form: uploads the points, runs the MSM, frees them (what a trait call with fresh
 * iterators does). */
int bpp_msm_vartime_host(bpp_ctx *ctx, const uint8_t *scalars, size_t n_scalars, int fmt, const uint8_t *pts,
                         size_t n_points, uint8_t out_compressed[32]);
/* Device-resident form: scalars already in HBM (n x 32 B), result (32 B compressed, then 128 B
 * X,Y,Z,T as raw 8x32-bit-limb field elements) written to d_out (160 B, device). Asynchronous. */
int bpp_msm_vartime_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n,
                        void *d_out);
/* Throughput form of bpp_msm_vartime_dev for a sequence of independent MSMs: submit enqueues the MSM without
 * making the caller's stream wait for it; the result is valid (in stream order on the caller's stream) after
 * bpp_msm_wait.  Up to two submitted MSMs are in flight on the library's internal streams - the dependent tail of
 * one (bucket reduction, Horner, compress) runs beside the sort and accumulate of the next; a third submit first
 * waits for the oldest.  d_scalars and d_out of a submitted MSM must stay untouched until bpp_msm_wait (or
 * bpp_synchronize / bpp_points_free / bpp_set_stream, which wait too).  Inputs are taken in stream order: work
 * queued on the caller's stream before the submit is complete before the MSM reads d_scalars. */
int bpp_msm_submit_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n,
                       void *d_out);
/* submitted form of bpp_msm_partial_dev (128-byte extended point, not compressed): the sharded multi-GPU MSM in
 * throughput form - submit(i), wait_previous, all-gather + bpp_points_sum_compress_dev of step i-1. */
int bpp_msm_submit_partial_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n,
                               void *d_partial);
int bpp_msm_wait(bpp_ctx *ctx);
/* Like bpp_msm_wait, but the MSM submitted last stays in flight: after submit(i), the results of every MSM up to
 * i-1 are valid - the form a producer/consumer loop uses (submit i, wait_previous, consume i-1). */
int bpp_msm_wait_previous(bpp_ctx *ctx);
/* Partial (uncompressed) sum for multi-GPU sharding: writes the 128-byte extended point (raw limbs)
 * to d_partial and does not compress.  bpp_points_sum_compress_dev adds g such partials (e.g. after an
 * all-gather) and compresses: d_out32 receives the 32-byte encoding. */
int bpp_msm_partial_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n,
                        void *d_partial);
int bpp_points_sum_compress_dev(bpp_ctx *ctx, const void *d_partials, size_t g, void *d_out32);
/* Override the Pippenger window width (0 = automatic). */
int bpp_set_window_bits(bpp_ctx *ctx, int c);
/* Override the number of window groups of the pipelined MSM (0 = automatic, 1 = everything in order on the
 * caller's stream, up to 8).  With more than one group the windows are processed group by group from the top:
 * the sort of the next group and the dependent tail of the previous one (fix-up, bucket reduction, Horner, the
 * doublings to the group's weight) run on internal high-priority streams beside the accumulate of the current
 * group; the call still is stream-ordered on the caller's stream.  The result bytes do not depend on it. */
int bpp_set_msm_groups(bpp_ctx *ctx, int groups);
/* Entries per accumulate tile (one thread adds one tile of the bucket-sorted entry list): 0 = by input size (32, and 64
 * from 3 M points), else 8..256.  Result-neutral tuning hook. */
int bpp_set_msm_tile(bpp_ctx *ctx, int tile_len);
/* Explicit window-group sizes, top group first (count <= 8; used when they sum to the number of windows of the
 * MSM, ignored otherwise; count = 0 clears).  A tuning hook like bpp_set_window_bits. */
int bpp_set_msm_partition(bpp_ctx *ctx, const int *sizes, int count);

/* ---- scalar-vector operators mod l: the reference's util.rs / poly.rs -------------------------------
 * All vectors are arrays of 32-byte little-endian canonical scalars in host memory.  Where the Rust
 * function panics on a dimension mismatch (util.rs:9-11,26-28,44-46,86-88) the call returns
 * BPP_ERR_LENGTH_MISMATCH. */
/* util.rs:84-94  inner_product(a, b) */
int bpp_inner_product(bpp_ctx *ctx, const uint8_t *a, size_t len_a, const uint8_t *b, size_t len_b, uint8_t out[32]);
/* util.rs:6-20  hadamard_V(a, b) */
int bpp_hadamard_V(bpp_ctx *ctx, const uint8_t *a, size_t len_a, const uint8_t *b, size_t len_b, uint8_t *out);
/* util.rs:22-38  vm_mult(a, b): out[i] = <a, b[i]>; b is rows x cols row-major, a has cols entries */
int bpp_vm_mult(bpp_ctx *ctx, const uint8_t *a, size_t len_a, const uint8_t *b, size_t rows, size_t cols, uint8_t *out);
/* util.rs:40-56  mv_mult(a, b): out[j] = sum_i a[i][j] * b[i]; a is rows x cols, b has rows entries */
int bpp_mv_mult(bpp_ctx *ctx, const uint8_t *a, size_t rows, size_t cols, const uint8_t *b, size_t len_b, uint8_t *out);
/* util.rs:63-65,139-157  exp_iter(x).take(count), exactly as coded: x^F(i) = x, x, x^2, x^3, x^5, ... */
int bpp_exp_iter(bpp_ctx *ctx, const uint8_t x[32], size_t count, uint8_t *out);
/* the standard powers x^first, x^(first+1), ... (what exp_iter is meant to produce; used by the IPA mode) */
int bpp_scalar_powers(bpp_ctx *ctx, const uint8_t x[32], size_t first, size_t count, uint8_t *out);
/* util.rs:67-82  scalar_exp(x, pow) */
int bpp_scalar_exp(bpp_ctx *ctx, const uint8_t x[32], uint32_t pow, uint8_t out[32]);
/* circuit_lib.rs:273-275  y_n.iter().map(|k| k.invert()) */
int bpp_scalar_invert(bpp_ctx *ctx, const uint8_t *a, size_t n, uint8_t *out);
/* transcript_protocol.rs:62-67 / Scalar::random: Scalar::from_bytes_mod_order_wide over n x 64 bytes */
int bpp_scalar_from_wide(bpp_ctx *ctx, const uint8_t *in64, size_t n, uint8_t *out);
/* traits.rs:7-17  reduce_scalars: Scalar::reduce over n x 32 bytes */
int bpp_scalar_reduce(bpp_ctx *ctx, const uint8_t *in32, size_t n, uint8_t *out);
/* poly.rs:39-55  VecPoly3::special_inner_product(lhs, rhs) -> Poly6 {t1..t6}; lhs/rhs are 4 x n */
int bpp_vecpoly3_special_inner_product(bpp_ctx *ctx, const uint8_t *lhs, const uint8_t *rhs, size_t n,
                                       uint8_t out_t1_t6[192]);
/* poly.rs:57-76  VecPoly3::eval / eval_ref */
int bpp_vecpoly3_eval(bpp_ctx *ctx, const uint8_t *coeffs, size_t n, const uint8_t x[32], uint8_t *out);
/* poly.rs:14-18  Poly6::eval */
int bpp_poly6_eval(bpp_ctx *ctx, const uint8_t t1_t6[192], const uint8_t x[32], uint8_t out[32]);

/* ---- multi-GPU: one process per GPU, NCCL inside the library (SURVEY 8(e), D.3) -----------------------------
 * Only what the path shards: a large MSM (points partitioned, 128-byte partial results all-gathered, summed and
 * compressed on every rank) and batch verification (proofs partitioned, accept bytes all-gathered).  Rank 0 makes the
 * id, the host program distributes it (any channel), every rank calls bpp_comm_init once; libnccl.so.2 is resolved
 * at run time.  Without a communicator every call below degrades to its single-GPU meaning. */
#define BPP_COMM_ID_BYTES 128
int bpp_comm_unique_id(uint8_t id[BPP_COMM_ID_BYTES]);
int bpp_comm_init(bpp_ctx *ctx, int nranks, int rank, const uint8_t id[BPP_COMM_ID_BYTES]);
int bpp_comm_free(bpp_ctx *ctx);
int bpp_comm_info(bpp_ctx *ctx, int *nranks, int *rank);
/* all-gather of bytes_per_rank device bytes per rank into d_recv (nranks x bytes_per_rank), on the context's stream */
int bpp_comm_all_gather_dev(bpp_ctx *ctx, const void *d_send, size_t bytes_per_rank, void *d_recv);
/* sharded vartime_multiscalar_mul: this rank's slice of scalars and points -> the full result's encoding (32 B at
 * d_out32, identical on every rank).  _submit/_wait: the throughput form (two MSMs in flight, the gather of MSM i-1
 * beside MSM i; results valid after bpp_msm_sharded_wait). */
int bpp_msm_sharded_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n, void *d_out32);
int bpp_msm_sharded_submit_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n,
                               void *d_out32);
int bpp_msm_sharded_wait(bpp_ctx *ctx);

/* ---- small and batched MSMs over a long-lived point set (SURVEY 2.3 K5) ---------------------------------
 * The reference's 15 call sites (circuit_lib.rs:187-575) multiply 2..209 points that always come from the same
 * generator set (g, h, G_vec, H_vec, lib.rs:164-180) by fresh scalars.  bpp_points_precompute attaches a fixed-base
 * window table to a point set (window_bits 4..20, 0 = 8: 2^(c-1) x ceil(256/c) entries of 96 B per point, built once);
 * from then on bpp_msm_vartime over any sub-range of up to 8192 of its points is table look-ups + mixed adds (no
 * buckets, no doublings: three short launches), and bpp_msm_vartime_batch evaluates `count` MSMs over the same
 * points[off..off+n) with count x n scalars in one launch (out32: count x 32 compressed results).  The table is built
 * on first use (c = 8) if bpp_points_precompute was not called.  _dev: scalars and results in device memory,
 * stream-ordered, no synchronisation. */
int bpp_points_precompute(bpp_ctx *ctx, bpp_points *points, int window_bits);
int bpp_msm_vartime_batch(bpp_ctx *ctx, const uint8_t *scalars, size_t count, bpp_points *points, size_t off, size_t n,
                          uint8_t *out32);
int bpp_msm_vartime_batch_dev(bpp_ctx *ctx, const void *d_scalars, size_t count, bpp_points *points, size_t off, size_t n,
                              void *d_out32);

/* ---- batched MSMs over caller points: many independent vartime_multiscalar_mul calls in one call ----------
 * MSM j has sizes[j] terms; the terms of all MSMs are stored one after another.  With T = sum sizes and
 * start_j = sum_{i<j} sizes[i], MSM j = sum_{t = start_j}^{start_j + sizes[j] - 1} s_t * P_t.  sizes is host memory (the
 * launch plan is made from it).  out32[j] is the canonical encoding of MSM j; sizes[j] == 0 gives the identity (32 zero
 * bytes).  Scalars are 32-byte little-endian with bit 255 clear; non-canonical scalars below 2^255 are accepted, as dalek
 * accepts them.  A few launches per call whatever count is, all on the context's stream; results depend on the inputs
 * only (not on the batch's composition or order).
 * Errors, host forms, before any device work: NULL pointers or count == 0, or T >= 2^31: BPP_ERR_INVALID_ARG; an
 * index[t] >= bpp_points_len(points): BPP_ERR_LENGTH_MISMATCH; a scalar with bit 255 set: BPP_ERR_SCALAR_RANGE.  The _dev
 * forms check what the host sees (NULL pointers, count, T); device data cannot make them fault: bit 255 of a scalar is read
 * as zero and an index outside the set is clamped into it (the -DBPP_DEBUG_BOUNDS build asserts instead). */
/* points as 32-byte RFC 9496 encodings (T x 32).  An undecodable encoding fails only its own MSM:
 * ok[j] = 0 and out32[j] = 32 zero bytes (dalek: optional_multiscalar_mul -> None); ok[j] = 1 otherwise. */
int bpp_msm_multi(bpp_ctx *ctx, size_t count, const uint32_t *sizes, const uint8_t *scalars /* T x 32 */,
                  const uint8_t *points_enc /* T x 32 */, uint8_t *out32 /* count x 32 */, uint8_t *ok /* count */);
/* points from a resident set: P_t = points[index[t]]; no decoding. */
int bpp_msm_multi_indexed(bpp_ctx *ctx, size_t count, const uint32_t *sizes, const uint8_t *scalars,
                          const bpp_points *points, const uint32_t *index /* T */, uint8_t *out32);
/* _dev: scalars, encodings / index, out32, ok are device pointers; stream-ordered on the context's stream, no synchronisation */
int bpp_msm_multi_dev(bpp_ctx *ctx, size_t count, const uint32_t *sizes, const void *d_scalars,
                      const void *d_points_enc, void *d_out32, void *d_ok);
int bpp_msm_multi_indexed_dev(bpp_ctx *ctx, size_t count, const uint32_t *sizes, const void *d_scalars,
                              const bpp_points *points, const void *d_index, void *d_out32);

/* ---- the arithmetic-circuit (shuffle) proof, batched ------------------------------------------------
 * Replaces the group/scalar arithmetic of ACProof::ArithmeticCircuitProof (circuit_lib.rs:133-585) for
 * `count` independent proofs that share one circuit and one generator set, driven in the reference's
 * call order (lib.rs:219-231): create -> challenge_wit_and_const -> compute_per_challenges -> commit_Ts
 * -> random_chall_x -> blinding_values -> verify.  Merlin transcripts (transcript_protocol.rs) run one
 * device thread per proof between the protocol's kernels (no host round trip; the common prefix
 * Transcript::new(label) + domain separator is hashed once on the host), or on host threads when
 * bpp_acp_batch_set_host_transcripts(b, 1) is set - same bytes either way; the prover's RNG is a ChaCha20 stream per proof (seed = 32 bytes ==
 * rand_chacha::ChaCha20Rng::from_seed), drawn in the reference's order alpha, beta, ro, s_l[], s_r[],
 * tau_1, tau_3, tau_4, tau_5, tau_6 (circuit_lib.rs:180-182,213-214,361-404).
 *   mode 0 "reference"        what the reference code computes, defects included (SURVEY A.3); its
 *                             verifier rejects every proof (circuit_lib.rs:541-544), so does this one.
 *   mode 1 "reference-fixed"  defects 2-5 corrected: an accepting protocol with l, r in the clear.
 *   mode 2 "fixed"            + standard powers y^i, z^q and l, r replaced by an inner-product proof: bulletproofs
 *                             4.0.0 InnerProductProof::create / verification_scalars (Cargo.lock:47-50; absent from
 *                             the reference, SURVEY 8 row a16) with dalek's R1CS glue (t_x, t_x_blinding, e_blinding,
 *                             w, Q = w*g, H_factors = y^-n, padding to n' = next_pow2(n)).  Needs n' generators
 *                             in bpp_gens_create.  Proof bytes: the same 8 points | t | tau_x | mu |
 *                             L_0 | R_0 | .. | L_{lg n'-1} | R_{lg n'-1} | a | b.
 * Proof bytes (the reference defines no serialisation): A_I | A_O | S | T_1 | T_3 | T_4 | T_5 | T_6 |
 * tau_x | mu | t | l[0..n) | r[0..n), 32 bytes each. */
typedef struct bpp_circuit bpp_circuit;
typedef struct bpp_gens bpp_gens;
typedef struct bpp_acp_batch bpp_acp_batch;
/* Sparse form of ACEssentials' W_L, W_R, W_O (n x Q) and W_V (m x Q) (circuit_lib.rs:66-70): triples
 * (wire, constraint, coefficient), the four matrices concatenated in that order with nnz[4] counts;
 * c_vec is the dense constant vector (Q x 32).  Constraint q: W_L a_L + W_R a_R + W_O a_O = W_V v + c. */
int bpp_circuit_create(bpp_ctx *ctx, size_t n, size_t Q, size_t m, const uint32_t nnz[4], const uint32_t *wire,
                       const uint32_t *constraint, const uint8_t *coeff, const uint8_t *c_vec, bpp_circuit **out);
/* The corrected k-card shuffle circuit, built inside the library (replaces weights.rs:130-204 create_weights, which as
 * coded only makes sense for 2-3 cards - SURVEY A.3 defects 6-9): prod_i (v_i - X) == prod_i (v_{k+i} - X) with
 * X = v[2k]; n = 2k multipliers, Q = 4k constraints, m = 2k + 1 committed values, c = 0. */
int bpp_circuit_create_shuffle(bpp_ctx *ctx, size_t k, bpp_circuit **out);
void bpp_circuit_free(bpp_ctx *ctx, bpp_circuit *c);
/* g_base, h_base, G_vec[n], H_vec[n] (circuit_lib.rs:59-65) as compressed points; builds the fixed-base
 * window tables (window_bits 4..20, 0 = default 8; 2^(c-1) entries x 96 B per generator and window: a memory/throughput
 * dial - c = 16: 48 MiB per generator, c = 18: 180 MiB, c = 19: 336 MiB) used by every commitment of the protocol. */
int bpp_gens_create(bpp_ctx *ctx, const uint8_t g[32], const uint8_t h[32], const uint8_t *G, const uint8_t *H, size_t n,
                    int window_bits, bpp_gens **out);
void bpp_gens_free(bpp_ctx *ctx, bpp_gens *g);
/* Proof wire format (the reference defines none; SURVEY 8 row f-2).  A record is one version byte followed by the
 * proof bytes above.  Mode 2: version 0 - the layout of bulletproofs 4.0.0 R1CSProof::to_bytes for a one-phase proof
 * (A_I1 A_O1 S1 | T_1 T_3 T_4 T_5 T_6 | t_x t_x_blinding e_blinding | L_0 R_0 .. | a b).  Modes 0 / 1: versions
 * 0x80 / 0x81.  from_wire is the parser a verifier runs first: like R1CSProof::from_bytes it flags (status 1 =
 * ProofError::FormatError) a wrong version byte and any non-canonical scalar field; points stay compressed, an
 * invalid point encoding is the verifier's VerificationError.  A wire_len that does not match the circuit returns
 * BPP_ERR_LENGTH_MISMATCH.  Byte handling only: no device work, no context. */
size_t bpp_acproof_wire_len(size_t n, int mode);
int bpp_acproof_to_wire(size_t n, int mode, size_t count, const uint8_t *proofs, uint8_t *wire_out);
int bpp_acproof_from_wire(size_t n, int mode, size_t count, const uint8_t *wire, size_t wire_len, uint8_t *proofs_out,
                          uint8_t *status);
size_t bpp_acproof_proof_len(size_t n);                  /* modes 0 and 1: 32 * (11 + 2n) */
size_t bpp_acproof_proof_len_mode(size_t n, int mode);    /* mode 2: 32 * (13 + 2 lg n') */
/* One-call host forms: host buffers in, host buffers out (all copies included). */
int bpp_acproof_prove_batch(bpp_ctx *ctx, const bpp_circuit *cir, const bpp_gens *gens, int mode, size_t count,
                            const uint8_t *aL, const uint8_t *aR, const uint8_t *aO /* count x n x 32 */,
                            const uint8_t *gamma /* count x m x 32 */, const uint8_t *seeds /* count x 32 */,
                            const uint8_t *V /* count x m x 32 compressed; modes 1, 2 (bound to the transcript) */,
                            const uint8_t *label, size_t label_len, uint8_t *proofs_out /* count x proof_len */);
int bpp_acproof_verify_batch(bpp_ctx *ctx, const bpp_circuit *cir, const bpp_gens *gens, int mode, size_t count,
                             const uint8_t *proofs, const uint8_t *V /* count x m x 32 compressed */,
                             const uint8_t *label, size_t label_len,
                             const uint8_t *verifier_seed /* 32 secret bytes, or NULL: drawn from the OS */,
                             uint8_t *accept /* count bytes: 1 = Ok(()), 0 = Err(VerificationError) */);
/* Staged forms (device-resident batches; used for the resident-input timing and by long-lived provers). */
int bpp_acp_batch_create(bpp_ctx *ctx, const bpp_circuit *cir, const bpp_gens *gens, int mode, size_t count,
                         const uint8_t *label, size_t label_len, bpp_acp_batch **out);
void bpp_acp_batch_free(bpp_acp_batch *b);
int bpp_acp_batch_upload_witness(bpp_acp_batch *b, const uint8_t *aL, const uint8_t *aR, const uint8_t *aO,
                                 const uint8_t *gamma, const uint8_t *seeds);
/* The shuffle witness generated on the device (replaces weights.rs:38-113 create_variables + create_a for the circuit
 * of bpp_circuit_create_shuffle): deck = k card values (k x 32, shared by the batch), perm = count x k indices into the
 * deck (proof p's output deck is deck[perm[p][i]]), x = count x 32 challenge values, gamma = count x m x 32 blindings,
 * seeds = count x 32 prover RNG seeds.  Leaves a_L, a_R, a_O, gamma and v = deck | deck[perm] | x resident
 * (bpp_acp_batch_commit with v = NULL commits to that v).  perm is not checked on the host (it may be a device
 * address) and cannot make the call fault: an index >= k is clamped to k - 1, i.e. read as the deck's last card (the
 * -DBPP_DEBUG_BOUNDS build asserts instead).  perm is not required to be a permutation; a witness built from one that
 * is not is not a shuffle, and the verifier rejects its proof. */
int bpp_acp_batch_gen_shuffle_witness(bpp_acp_batch *b, const uint8_t *deck, const uint32_t *perm, const uint8_t *x,
                                      const uint8_t *gamma, const uint8_t *seeds);
/* commit_variables (weights.rs:58-61): V_j = v_j*g + gamma_j*h with the uploaded gamma; V_out nullable; v = NULL: the
 * values left by bpp_acp_batch_gen_shuffle_witness. */
int bpp_acp_batch_commit(bpp_acp_batch *b, const uint8_t *v /* count x m x 32, nullable */, uint8_t *V_out);
/* The value commitments as the caller holds them (count x m x 32 compressed).  Modes 1 and 2 bind them to every
 * proof's transcript right after the domain separator (append_u64("m"), append_point("V") per commitment - what
 * bulletproofs 4.0.0's R1CS prover/verifier do at commit time), so the prover needs them resident before
 * bpp_acp_batch_prove: through this call or bpp_acp_batch_commit.  Mode 0 reproduces the reference, which never
 * appends them (circuit_lib.rs:178-200; SURVEY A.3 defect 12). */
int bpp_acp_batch_upload_commitments(bpp_acp_batch *b, const uint8_t *V);
int bpp_acp_batch_prove(bpp_acp_batch *b);
int bpp_acp_batch_download_proofs(bpp_acp_batch *b, uint8_t *proofs_out);
int bpp_acp_batch_upload_proofs(bpp_acp_batch *b, const uint8_t *proofs, const uint8_t *V /* nullable */);
/* verifier_seed: 32 bytes of SECRET, FRESH randomness of the verifier, or NULL to have the library draw them from
 * the operating system (getrandom).  The per-proof weight w (check 2 + w * check 3 as one MSM) and the batch weight rho
 * are challenge scalars of each proof's own transcript - which has absorbed V and every proof message - continued with
 * the remaining proof bytes, this seed and the proof's index (dalek draws its verifier weights the same way, from a
 * transcript RNG rekeyed with thread_rng).  A seed known to the prover before it fixes its proofs would still leave the
 * weights bound to every proof byte, but pass NULL or fresh randomness; a constant is for reproducible tests only. */
int bpp_acp_batch_verify(bpp_acp_batch *b, const uint8_t *verifier_seed);
int bpp_acp_batch_download_accept(bpp_acp_batch *b, uint8_t *accept);
/* Sharded batch verification (BASELINE configs[3]): every rank verified its own slice of the batch; all ranks' accept
 * bytes are all-gathered (NCCL, bpp_comm_init) into accept_all = nranks x per bytes, rank r's count bytes at r * per
 * (per >= every rank's count; the rest is zero padding).  Host buffer; synchronises. */
int bpp_acp_batch_gather_accept(bpp_acp_batch *b, size_t per, uint8_t *accept_all);
/* Verification strategy: 1 (default) = first ONE random-linear-combination MSM over the whole batch (weights from
 * the verifier seed; Pippenger over count x (m + 8) decompressed points + the shared generators), the per-proof
 * kernels only when it is not the identity, i.e. some proof is invalid; 0 = always per proof.  The accept bytes
 * are the per-proof decisions either way. */
int bpp_acp_batch_set_batch_rlc(bpp_acp_batch *b, int on);
/* Fiat-Shamir location: 0 (default) per-proof Merlin transcripts on the device, 1 on host threads. */
int bpp_acp_batch_set_host_transcripts(bpp_acp_batch *b, int on);
/* Priority split for a caller that keeps several batches in flight on several streams: with on = 1 the table-gather
 * MSMs of this batch (the launches that fill the GPU) run on an internal stream of the lowest priority, bracketed by
 * events, so that when the caller's stream is an urgent one (cudaStreamCreateWithPriority) the short dependent
 * kernels of this batch - transcripts, power chains, dot products - take SM slots ahead of the GPU-filling kernels of
 * the other batches.  Result-neutral; no effect worth having on a default-priority stream. */
int bpp_acp_batch_set_priority_split(bpp_acp_batch *b, int on);
/* K7 (SURVEY 2.3, D.3; bulletproofs 4.0.0 inner_product_proof.rs create(): G'_i = u^-1 G_i + u G_{i+n/2}) as an operator:
 * `folds` independent foldings of points[off..off+n) (n even) with scalars u_f, u_f^-1 (folds x 32 each, reduced):
 * out_enc[f][i] = compress(u_f^-1 P_i + u_f P_{i+n/2}) (host, folds x n/2 x 32, nullable); ms (nullable) = device time of
 * the folding kernel.  The prover does not use it - it folds the scalars and keeps the tabled generators
 * (DESIGN.md section 5) - it exists so the two forms can be measured against each other and checked for equality. */
int bpp_ipa_fold_generators(bpp_ctx *ctx, const bpp_points *points, size_t off, size_t n, const uint8_t *u, const uint8_t *uinv,
                            size_t folds, uint8_t *out_enc, float *ms);
/* merlin::Transcript on the device, scripted (test hook for the Merlin KAT and framing edge cases): records
 * op (1 B: 0 append_message, 1 challenge_bytes) | label_len (1 B) | label | n (4 B LE) | message (op 0);
 * the transcript is Transcript::new(first record's message) when the first record is labelled "dom-sep";
 * challenge outputs are concatenated into out (out_len = sum of the challenge lengths). */
int bpp_transcript_script(bpp_ctx *ctx, const uint8_t *script, size_t len, uint8_t *out, size_t out_len);
/* measurement hook: the A_I-shaped fixed-base MSM kernel alone, timed with CUDA events over `reps` launches */
int bpp_acp_batch_time_commit_msm(bpp_acp_batch *b, int reps, float *ms_avg, uint64_t *mixed_adds, uint64_t *full_adds);

/* ---- transcripts across the ABI (host only: no context, no device) ------------------------------------------
 * merlin 3.0.0 Transcript (the `&mut Transcript` of bulletproofs' inner_product_proof.rs) as a caller-held state of
 * BPP_TRANSCRIPT_BYTES: 26 little-endian u64, the 25 Keccak-f[1600] lanes of the STROBE-128 sponge, then
 * pos | pos_begin << 8 | cur_flags << 16.  A state no transcript could be in (pos or pos_begin beyond the rate)
 * is BPP_ERR_INVALID_ARG.  Labels are byte strings of label_len bytes (merlin's &'static [u8]). */
#define BPP_TRANSCRIPT_BYTES 208
/* Transcript::new(label) */
int bpp_transcript_new(const uint8_t *label, size_t label_len, uint8_t state[BPP_TRANSCRIPT_BYTES]);
/* Transcript::append_message(label, msg) */
int bpp_transcript_append_message(uint8_t state[BPP_TRANSCRIPT_BYTES], const uint8_t *label, size_t label_len,
                                  const uint8_t *msg, size_t msg_len);
/* Transcript::challenge_bytes(label, out) */
int bpp_transcript_challenge_bytes(uint8_t state[BPP_TRANSCRIPT_BYTES], const uint8_t *label, size_t label_len,
                                   uint8_t *out, size_t out_len);

/* ---- stand-alone inner-product argument, batched ---------------------------------------------------------------
 * bulletproofs 4.0.0 InnerProductProof::create / verify (inner_product_proof.rs; the crate keeps the module private)
 * for `count` independent proofs of length n over caller generators and caller transcripts - what a caller needs to
 * replace the 2n scalars l, r that circuit_lib.rs:464-468 sends in the clear by a proof of 2 lg n + 2 words.
 * For proof p: G = gens[g_off .. g_off + n), H = gens[h_off .. h_off + n), Q_p = q_p * gens[q_off] (every use in dalek:
 * the R1CS and range-proof verifiers take Q = w * B; an arbitrary per-proof Q is not supported).  gens is one tabled
 * point set: the c = 8 window table is built on first use unless bpp_points_precompute ran.  n is a power of two, at
 * most 8192.  Scalars are 32-byte little-endian; factor vectors are count x n x 32 (NULL = all ones), q count x 32
 * (NULL = ones), transcripts count x BPP_TRANSCRIPT_BYTES, read and written back.  Host buffers; each call ends with one
 * synchronisation.
 * Errors, before any device work: n not a power of two or > 8192, NULL arguments, count == 0: BPP_ERR_INVALID_ARG; an
 * offset range outside gens: BPP_ERR_LENGTH_MISMATCH; a scalar input >= l: BPP_ERR_SCALAR_RANGE. */
typedef struct bpp_ipa_batch bpp_ipa_batch;
/* 32 (2 lg n + 2): L_0 R_0 .. L_{lg n - 1} R_{lg n - 1} a b (InnerProductProof::to_bytes); 0 unless n is a power of two */
size_t bpp_ipa_proof_len(size_t n);
int bpp_ipa_batch_create(bpp_ctx *ctx, bpp_points *gens, size_t g_off, size_t h_off, size_t q_off, size_t n, size_t count,
                         bpp_ipa_batch **out);
void bpp_ipa_batch_free(bpp_ipa_batch *b);
/* InnerProductProof::create(transcript, Q, G_factors, H_factors, G, H, a, b): from each transcript state, the domain
 * separator ("dom-sep" "ipp v1", u64 "n") and the rounds; proofs_out count x bpp_ipa_proof_len(n); every transcript is
 * left as create leaves it. */
int bpp_ipa_batch_prove(bpp_ipa_batch *b, const uint8_t *q, const uint8_t *G_factors, const uint8_t *H_factors,
                        const uint8_t *a, const uint8_t *b_vec, uint8_t *transcripts, uint8_t *proofs_out);
/* InnerProductProof::verify(n, transcript, G_factors, H_factors, P, Q, G, H): P count x 32 compressed; accept[p] = 1 iff
 * P_p = a b Q_p + sum a s_i gf_i G_i + sum b s_i^-1 hf_i H_i - sum u_j^2 L_j - sum u_j^-2 R_j.  A proof is rejected (0,
 * not an error) when its a or b is >= l (from_bytes refuses it), an L_j or R_j is the all-zero encoding
 * (validate_and_append_point) or L_j, R_j or P fails decoding.  The transcripts of accepted proofs are left as verify
 * leaves them. */
int bpp_ipa_batch_verify(bpp_ipa_batch *b, const uint8_t *q, const uint8_t *G_factors, const uint8_t *H_factors,
                         const uint8_t *P, const uint8_t *proofs, uint8_t *transcripts, uint8_t *accept);

/* ---- measurement helpers --------------------------------------------------------------------- */
/* IMAD.WIDE.U32 peak microbenchmark: returns wide multiply-adds per second over all SMs. */
int bpp_bench_imad_peak(bpp_ctx *ctx, int iters, double *ops_per_sec, double *ms);
/* Same harness for the other instruction forms a multiplier can be built from.  mode 0: plain IMAD.WIDE.U32
 * with a 64-bit addend; 1: carry-chained IMAD.WIDE.U32 (mad.lo.cc/madc.hi.cc); 2: 32-bit IMAD; 3: IADD3.X chains;
 * 4: dependent field multiplications (reported as 72 wide multiply-adds each); 5: dependent mixed point adds (504 each).
 * Every multiply has a data-dependent operand so the assembler cannot strength-reduce the loop. */
int bpp_bench_pipe_probe(bpp_ctx *ctx, int mode, int iters, double *ops_per_sec);
/* Per-phase device time (ms) of the last bpp_msm_* call when profiling is enabled. */
enum { BPP_PHASE_RECODE = 0, BPP_PHASE_SCAN, BPP_PHASE_SCATTER, BPP_PHASE_ACCUMULATE, BPP_PHASE_REDUCE,
       BPP_PHASE_FINISH, BPP_PHASE_COUNT };
int bpp_set_profiling(bpp_ctx *ctx, int on);
/* Stage timeline of the last bpp_msm_* call (pipelined or not): with tracing on, every stage boundary records a
 * timing event on the stream that runs the stage; the dump synchronises the device and writes one line per mark,
 * "<stage>[group] <microseconds since the start mark>" ('>' = stage begins, '.' = stage done). */
int bpp_set_msm_trace(bpp_ctx *ctx, int on);
int bpp_msm_trace_dump(bpp_ctx *ctx, char *buf, size_t cap);
int bpp_last_phase_ms(bpp_ctx *ctx, float ms[BPP_PHASE_COUNT]);
/* point-add count of the last MSM: accumulate (mixed) adds, reduction (full) adds, doublings */
int bpp_last_op_counts(bpp_ctx *ctx, uint64_t *mixed_adds, uint64_t *full_adds, uint64_t *doublings);

/* ---- element-wise self-test hooks (used by tests/ to compare single operations with the oracle) */
enum { BPP_TEST_FE_MUL = 0, BPP_TEST_FE_ADD, BPP_TEST_FE_SUB, BPP_TEST_FE_INVERT, BPP_TEST_FE_CANON,
       BPP_TEST_GE_ADD, BPP_TEST_GE_DOUBLE, BPP_TEST_GE_COMPRESS_ROUNDTRIP, BPP_TEST_GE_SCALARMULT,
       BPP_TEST_FE_SQR, BPP_TEST_GE_DOUBLE_Z1 /* doubling with a compile-time Z = 1 */ };
/* a, b: n x 32-byte operands (points as compressed encodings); out: n x 32 bytes. */
int bpp_test_op(bpp_ctx *ctx, int op, const uint8_t *a, const uint8_t *b, uint8_t *out, size_t n);

#ifdef __cplusplus
}
#endif
#endif /* BPPERM_H */
