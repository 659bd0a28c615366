// transcript_kernels.cuh - the Fiat-Shamir steps of the batched shuffle prover / verifier on the
// device: one thread per proof runs that proof's Merlin transcript (merlin_dev.cuh) and writes the
// challenge scalars straight into the proof's scalar block.  Labels and order follow
// /root/reference/bp-perm/src/circuit_lib.rs:231-233 (A_I, A_O, S), :133-138 (y, z), :368-412
// (T1, T3, T4 - carrying T_3 in `reference` mode, :391 -, T5, T6), :425-432 (x); the `fixed` mode tail
// follows bulletproofs 4.0.0 r1cs/prover + inner_product_proof.rs (t_x, t_x_blinding, e_blinding,
// w, "ipp v1" domain separator, L/R -> u per round).
#pragma once
#include "acproof_kernels.cuh"
#include "merlin_dev.cuh"
#include "merlin_warp.cuh"

// Every transcript kernel exists in two forms, selected by the number of independent sponges of the launch:
//   merlin_warp  one WARP per sponge (merlin_warp.cuh): lowest latency per permutation (~2.5 us), nine 64-bit shuffles
//                per round - the form for small batches, where the sponge is the critical path;
//   merlin_tr    one THREAD per sponge (merlin_dev.cuh): ~6 us per permutation but 32 sponges per warp and no shuffles,
//                2-3 x less issue work per permutation - it only pays once the launch has enough sponges for more than
//                a warp per SM sub-partition (measured, profiles/r2c_launches_*.csv: 4096 sponges - k_tr_weights 0.94 ms
//                against 0.40 ms in the warp form, k_tr_verify 0.43 against 0.27; 8192 sponges - k_tr_vchunks 0.35
//                against 0.48).
// TR_LAUNCH picks by count (tr_warp_max sponges and below: warp form; BPP_TR_WARP_MAX overrides).
#define TR_THREADS 128
template <class T>
__device__ __forceinline__ uint32_t tr_index() { return (blockIdx.x * blockDim.x + threadIdx.x) / T::GROUP; }
template <class T>
__device__ __forceinline__ bool tr_leader() { return (threadIdx.x % T::GROUP) == 0; }
static inline uint32_t tr_warp_max() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("BPP_TR_WARP_MAX");
        v = e ? atoi(e) : 2047;
    }
    return (uint32_t)v;
}
// TR_LAUNCH_AT: the same with an explicit limit (k_ipa_challenge ends in a one-lane inversion per sponge, which a warp
// per sponge spreads over 32 x more warps: thread form from 1024 proofs - measured 17.8 against 20.2 ms per 4096-proof
// `fixed` prover).
#define TR_LAUNCH(kern, count, stream, ...) TR_LAUNCH_AT(tr_warp_max(), kern, count, stream, __VA_ARGS__)
#define TR_LAUNCH_AT(limit, kern, count, stream, ...)                                                              \
    do {                                                                                                           \
        const uint32_t tr_cnt_ = (uint32_t)(count);                                                                \
        if (tr_cnt_ <= (limit)) kern<merlin_warp><<<(tr_cnt_ + TR_THREADS / 32 - 1) / (TR_THREADS / 32), TR_THREADS, 0, stream>>>(__VA_ARGS__); \
        else kern<merlin_tr><<<(tr_cnt_ + 31) / 32, 32, 0, stream>>>(__VA_ARGS__);                                 \
    } while (0)

// The value commitments, bound to the transcript right after the domain separator (modes 1 and 2; the reference never
// appends them - SURVEY A.3 defect 12, weak Fiat-Shamir: the prover of a shuffle chooses the output-deck commitments).
// Two levels (CPU restatements: commitment_digests / append_commitments in the test tree): every chunk of TR_V_CHUNK commitments is a
// sponge of its own - Transcript::new("acp-V"), append_u64("chunk", index), append_message("V", the chunk's encodings
// concatenated), challenge_bytes("d", 32) - and the proof's transcript absorbs m under "m" and the concatenated chunk digests as one message under "Vd".  One
// serial sponge over the m = 8193 commitments of a 4096-card deck is ~2000 permutations in a row on the critical path
// of prover and verifier; the chunks run as independent warps.
#define TR_V_CHUNK 64
#define TR_V_CHUNKS(m) (((m) + TR_V_CHUNK - 1) / TR_V_CHUNK)
// vproto: the transcript after Transcript::new("acp-V").  One warp per (proof, chunk); vdig: B x chunks x 32.
template <class T>
__global__ void __launch_bounds__(TR_THREADS) k_tr_vchunks(const uint64_t *__restrict__ vproto, const uint8_t *__restrict__ V,
                                                           uint32_t m, uint32_t B, uint8_t *__restrict__ vdig) {
    const uint32_t nch = TR_V_CHUNKS(m), w = tr_index<T>();
    if (w >= B * nch) return;
    const uint32_t p = w / nch, c = w % nch;
    T t;
    t.load(vproto);
    t.append_u64(MERLIN_LABEL("chunk"), c);
    const uint8_t *v = V + 32 * ((size_t)p * m + (size_t)c * TR_V_CHUNK);
    const uint32_t cnt = min((uint32_t)TR_V_CHUNK, m - c * TR_V_CHUNK);
    t.append_message(MERLIN_LABEL("V"), v, 32 * cnt);   // the chunk's encodings as one message
    t.challenge_bytes(MERLIN_LABEL("d"), vdig + 32 * (size_t)w, 32);
}
template <class T>
__device__ __forceinline__ void tr_append_commitments(T &t, const uint8_t *vdig, uint32_t m) {
    t.append_u64(MERLIN_LABEL("m"), m);
    // the digests are contiguous per proof: one message (129 separate appends of a 4096-card deck were 129 framing
    // headers and ~520 short absorb calls in a row on the critical path of prover and verifier)
    t.append_message(MERLIN_LABEL("Vd"), vdig, 32 * TR_V_CHUNKS(m));
}

// proto: the transcript after Transcript::new(label) + arithmetic_domain_sep(n), identical for every proof (hashed
// once on the host).  pts8: B x 8 x 32 compressed (A_I, A_O, S, T1, T3, T4, T5, T6).  vdig: the chunk digests of the
// commitments (k_tr_vchunks), null in mode 0.
template <class T>
__global__ void __launch_bounds__(TR_THREADS) k_tr_prove_yz(const uint64_t *__restrict__ proto, const uint8_t *__restrict__ vdig,
                                                            const uint8_t *__restrict__ pts8, acp_layout lay,
                                                            uint32_t B, uint64_t *__restrict__ states,
                                                            uint32_t *__restrict__ blk) {
    const uint32_t p = tr_index<T>();
    if (p >= B) return;
    T t;
    t.load(proto);
    if (vdig) tr_append_commitments(t, vdig + 32 * (size_t)p * TR_V_CHUNKS(lay.m), lay.m);
    const uint8_t *pt = pts8 + 256 * (size_t)p;
    t.append_message(MERLIN_LABEL("A_I"), pt, 32);
    t.append_message(MERLIN_LABEL("A_O"), pt + 32, 32);
    t.append_message(MERLIN_LABEL("S"), pt + 64, 32);
    sc c;
    t.challenge_scalar(MERLIN_LABEL("y"), c);
    if (t.lane == 0) sc_store(ACP_PTR(blk, lay, p, lay.y), c);
    t.challenge_scalar(MERLIN_LABEL("z"), c);
    if (t.lane == 0) sc_store(ACP_PTR(blk, lay, p, lay.z), c);
    t.store(states + MERLIN_STATE_WORDS * (size_t)p);
}

template <class T>
__global__ void __launch_bounds__(TR_THREADS) k_tr_prove_x(const uint8_t *__restrict__ pts8, acp_layout lay, uint32_t B,
                                                           int mode, uint64_t *__restrict__ states,
                                                           uint32_t *__restrict__ blk) {
    const uint32_t p = tr_index<T>();
    if (p >= B) return;
    T t;
    t.load(states + MERLIN_STATE_WORDS * (size_t)p);
    const uint8_t *pt = pts8 + 256 * (size_t)p + 96;
    t.append_message(MERLIN_LABEL("T1"), pt, 32);
    t.append_message(MERLIN_LABEL("T3"), pt + 32, 32);
    t.append_message(MERLIN_LABEL("T4"), mode == 0 ? pt + 32 : pt + 64, 32);  // circuit_lib.rs:391 appends T_3 under "T4"
    t.append_message(MERLIN_LABEL("T5"), pt + 96, 32);
    t.append_message(MERLIN_LABEL("T6"), pt + 128, 32);
    sc c;
    t.challenge_scalar(MERLIN_LABEL("x"), c);
    if (t.lane == 0) sc_store(ACP_PTR(blk, lay, p, lay.x), c);
    t.store(states + MERLIN_STATE_WORDS * (size_t)p);
}

// `fixed` mode: t_x, t_x_blinding, e_blinding (contiguous canonical scalars at lay.that: in memory they ARE their
// 32-byte little-endian encodings) -> w; inner-product domain separator
template <class T>
__device__ __forceinline__ void tr_fixed_w(T &t, const uint8_t *s3, uint32_t np, sc &w) {
    t.append_message(MERLIN_LABEL("t_x"), s3, 32);
    t.append_message(MERLIN_LABEL("t_x_blinding"), s3 + 32, 32);
    t.append_message(MERLIN_LABEL("e_blinding"), s3 + 64, 32);
    t.challenge_scalar(MERLIN_LABEL("w"), w);
    t.append_message(MERLIN_LABEL("dom-sep"), (const uint8_t *)"ipp v1", 6);
    t.append_u64(MERLIN_LABEL("n"), np);
}
// Inner-product rounds of the prover, one warp per proof.  round < 0: t_x, t_x_blinding, e_blinding -> w and the
// inner-product domain separator.  round >= 0: append L_round, R_round, draw u_round and invert it (lane 0; the
// branch-free GCD of sc_invert) - u and u^-1 are left in Montgomery form at lay.u / lay.uinv for k_ipa_round.
template <class T>
__global__ void __launch_bounds__(TR_THREADS) k_ipa_challenge(const uint8_t *__restrict__ lr, acp_layout lay, uint32_t B,
                                                              int round, uint64_t *__restrict__ states,
                                                              uint32_t *__restrict__ blk) {
    const uint32_t p = tr_index<T>();
    if (p >= B) return;
    T t;
    t.load(states + MERLIN_STATE_WORDS * (size_t)p);
    sc c;
    if (round < 0) {
        tr_fixed_w(t, (const uint8_t *)ACP_PTR(blk, lay, p, lay.that), lay.np, c);
        if (t.lane == 0) sc_store(ACP_PTR(blk, lay, p, lay.wq), c);
    } else {
        const uint8_t *q = lr + 64 * ((size_t)lay.lg * p + round);
        t.append_message(MERLIN_LABEL("L"), q, 32);
        t.append_message(MERLIN_LABEL("R"), q + 32, 32);
        t.challenge_scalar(MERLIN_LABEL("u"), c);
    }
    t.store(states + MERLIN_STATE_WORDS * (size_t)p);
    if (round >= 0 && t.lane == 0) {
        sc ci;
        sc_invert(ci, c);
        sc_to_mont(c, c);
        sc_to_mont(ci, ci);
        sc_store(ACP_PTR(blk, lay, p, lay.u + round), c);
        sc_store(ACP_PTR(blk, lay, p, lay.uinv + round), ci);
    }
}

// Small batches (a single large-deck proof: every inner-product round is a chain of short dependent launches): the tail
// of a round in ONE launch instead of three (k_fb_sum_splits -> k_compress_strided -> k_ipa_challenge).  Block per proof,
// two warps: warp 0 sums the split partial sums of L_round (lane-strided additions, then five shuffle steps), warp 1
// those of R_round; lane 0 of each compresses its point (the two inverse square roots run side by side); after the
// barrier warp 0 appends both encodings to the proof's transcript, draws u_round and inverts it.
__global__ void __launch_bounds__(64) k_ipa_lr_tail(const uint32_t *__restrict__ part /* [p][2][splits] x 32 */, uint32_t splits,
                                                    uint32_t *__restrict__ lrext /* [p][2 lg] x 32 */, uint8_t *__restrict__ lr,
                                                    acp_layout lay, int round, uint64_t *__restrict__ states,
                                                    uint32_t *__restrict__ blk) {
    const uint32_t p = blockIdx.x, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    {   // the split sum spelled out, not through ge_warp_sum: that form schedules this latency-bound kernel differently and
        // was measured 1 % slower (2116 -> 2138 us of k_ipa_lr_tail per large-deck proof, B200 at 1000 W)
        const uint32_t *src = part + 32 * ((size_t)p * 2 + w) * splits;
        ge_ext acc, t;
        ge_identity(acc);
#pragma unroll 1
        for (uint32_t z = lane; z < splits; z += 32) {
            ge_load(t, src + 32 * (size_t)z);
            ge_add_noinline(acc, acc, t);
        }
#pragma unroll 1
        for (int d = 16; d >= 1; d >>= 1) {
            ge_ext o2;
#pragma unroll
            for (int i = 0; i < 8; i++) {
                o2.X.v[i] = __shfl_down_sync(0xffffffffu, acc.X.v[i], d);
                o2.Y.v[i] = __shfl_down_sync(0xffffffffu, acc.Y.v[i], d);
                o2.Z.v[i] = __shfl_down_sync(0xffffffffu, acc.Z.v[i], d);
                o2.T.v[i] = __shfl_down_sync(0xffffffffu, acc.T.v[i], d);
            }
            ge_add_noinline(acc, acc, o2);
        }
        if (lane == 0) {
            const size_t k = (size_t)p * 2 * lay.lg + 2 * (uint32_t)round + w;
            ge_store(lrext + 32 * k, acc);
            ge_compress(lr + 32 * k, acc);
        }
    }
    __syncthreads();   // both encodings are in global memory, written by this block
    if (w != 0) return;
    merlin_warp t;
    t.load(states + MERLIN_STATE_WORDS * (size_t)p);
    const uint8_t *q = lr + 64 * ((size_t)lay.lg * p + (uint32_t)round);
    t.append_message(MERLIN_LABEL("L"), q, 32);
    t.append_message(MERLIN_LABEL("R"), q + 32, 32);
    sc c;
    t.challenge_scalar(MERLIN_LABEL("u"), c);
    t.store(states + MERLIN_STATE_WORDS * (size_t)p);
    if (lane == 0) {
        sc ci;
        sc_invert(ci, c);
        sc_to_mont(c, c);
        sc_to_mont(ci, ci);
        sc_store(ACP_PTR(blk, lay, p, lay.u + round), c);
        sc_store(ACP_PTR(blk, lay, p, lay.uinv + round), ci);
    }
}

// Stand-alone inner-product batch (bpp_ipa_batch_*): the caller's transcripts, uploaded in `states`, get
// innerproduct_domain_sep(n) - dom-sep "ipp v1", u64 "n" - in place (InnerProductProof::create and
// verification_scalars both start so).
template <class T>
__global__ void __launch_bounds__(TR_THREADS) k_ipa_start(uint32_t n, uint32_t B, uint64_t *__restrict__ states) {
    const uint32_t p = tr_index<T>();
    if (p >= B) return;
    T t;
    t.load(states + MERLIN_STATE_WORDS * (size_t)p);
    t.append_message(MERLIN_LABEL("dom-sep"), (const uint8_t *)"ipp v1", 6);
    t.append_u64(MERLIN_LABEL("n"), n);
    t.store(states + MERLIN_STATE_WORDS * (size_t)p);
}
// Its verifier: verification_scalars' transcript steps on the uploaded states - the domain separator, then L_j, R_j ->
// u_j (standard form at lay.u + j) for every round.  lrp: B x (2 lg + 1) x 32 (k_ipa_unpack).  An all-zero L_j or R_j
// (validate_and_append_point refuses it) rejects the proof in k_acp_decompress_lr; the state is then left as if the
// point had been appended, which dalek does not define.
template <class T>
__global__ void __launch_bounds__(TR_THREADS) k_ipa_vtranscript(const uint8_t *__restrict__ lrp, acp_layout lay, uint32_t B,
                                                                uint64_t *__restrict__ states, uint32_t *__restrict__ blk) {
    const uint32_t p = tr_index<T>();
    if (p >= B) return;
    T t;
    t.load(states + MERLIN_STATE_WORDS * (size_t)p);
    t.append_message(MERLIN_LABEL("dom-sep"), (const uint8_t *)"ipp v1", 6);
    t.append_u64(MERLIN_LABEL("n"), lay.np);
    sc c;
#pragma unroll 1
    for (uint32_t j = 0; j < lay.lg; j++) {
        const uint8_t *q = lrp + 32 * ((size_t)(2 * lay.lg + 1) * p + 2 * j);
        t.append_message(MERLIN_LABEL("L"), q, 32);
        t.append_message(MERLIN_LABEL("R"), q + 32, 32);
        t.challenge_scalar(MERLIN_LABEL("u"), c);
        if (t.lane == 0) sc_store(ACP_PTR(blk, lay, p, lay.u + j), c);
    }
    t.store(states + MERLIN_STATE_WORDS * (size_t)p);
}

// Verifier: replays the whole transcript of one proof and leaves its final state in `states` (k_tr_weights continues
// it).  tx3 (B x 3 x 32: t_x, t_x_blinding, e_blinding, reduced) and lr are used in `fixed` mode only (lay.lg > 0).
template <class T>
__global__ void __launch_bounds__(TR_THREADS) k_tr_verify(const uint64_t *__restrict__ proto, const uint8_t *__restrict__ vdig,
                                                          const uint8_t *__restrict__ pts8,
                                                          const uint8_t *__restrict__ tx3,
                                                          const uint8_t *__restrict__ lr, acp_layout lay, uint32_t B,
                                                          int mode, uint32_t *__restrict__ blk,
                                                          uint64_t *__restrict__ states) {
    const uint32_t p = tr_index<T>();
    if (p >= B) return;
    T t;
    t.load(proto);
    if (mode != 0) tr_append_commitments(t, vdig + 32 * (size_t)p * TR_V_CHUNKS(lay.m), lay.m);
    const uint8_t *pt = pts8 + 256 * (size_t)p;
    t.append_message(MERLIN_LABEL("A_I"), pt, 32);
    t.append_message(MERLIN_LABEL("A_O"), pt + 32, 32);
    t.append_message(MERLIN_LABEL("S"), pt + 64, 32);
    sc c;
    t.challenge_scalar(MERLIN_LABEL("y"), c);
    if (t.lane == 0) sc_store(ACP_PTR(blk, lay, p, lay.y), c);
    t.challenge_scalar(MERLIN_LABEL("z"), c);
    if (t.lane == 0) sc_store(ACP_PTR(blk, lay, p, lay.z), c);
    t.append_message(MERLIN_LABEL("T1"), pt + 96, 32);
    t.append_message(MERLIN_LABEL("T3"), pt + 128, 32);
    t.append_message(MERLIN_LABEL("T4"), mode == 0 ? pt + 128 : pt + 160, 32);
    t.append_message(MERLIN_LABEL("T5"), pt + 192, 32);
    t.append_message(MERLIN_LABEL("T6"), pt + 224, 32);
    t.challenge_scalar(MERLIN_LABEL("x"), c);
    if (t.lane == 0) sc_store(ACP_PTR(blk, lay, p, lay.x), c);
    if (mode == 2) {
        tr_fixed_w(t, tx3 + 96 * (size_t)p, lay.np, c);
        if (t.lane == 0) sc_store(ACP_PTR(blk, lay, p, lay.wq), c);
#pragma unroll 1
        for (uint32_t j = 0; j < lay.lg; j++) {   // an identity encoding is rejected in k_acp_decompress_lr
            const uint8_t *q = lr + 64 * ((size_t)lay.lg * p + j);
            t.append_message(MERLIN_LABEL("L"), q, 32);
            t.append_message(MERLIN_LABEL("R"), q + 32, 32);
            t.challenge_scalar(MERLIN_LABEL("u"), c);
            if (t.lane == 0) sc_store(ACP_PTR(blk, lay, p, lay.u + j), c);
        }
    }
    t.store(states + MERLIN_STATE_WORDS * (size_t)p);
}

// Verifier weights.  The per-proof weight w (check 2 + w * check 3 as ONE multiscalar multiplication, SURVEY D.1) and
// the batch weight rho (random linear combination over the batch) must be unpredictable to whoever made the proofs:
// with a known w a prover cancels an error of check 3 against tau_x in check 2, with known rho two proofs of one batch
// carry cancelling offsets.  They are drawn like dalek's verifier draws its weights - from the proof's own transcript,
// which has absorbed the commitments and every proof message, rekeyed with the verifier's secret randomness: the final
// verifier state continues with the rest of the proof bytes (the scalars after the eight points), the verifier seed
// and the proof's index, then "w" and "rho" are challenge scalars.  So even a caller that reuses or leaks its seed
// gets weights that depend on every byte of the proof.  (bpp_acp_batch_verify draws the seed from the OS when the
// caller passes none.)  mode 0 (`reference`): w = 0, only checks 1 and 2 are live (circuit_lib.rs:577-582).
template <class T>
__global__ void __launch_bounds__(TR_THREADS) k_tr_weights(const uint64_t *__restrict__ states,
                                                           const uint8_t *__restrict__ proofs, uint32_t proof_len,
                                                           const uint8_t *__restrict__ vseed, acp_layout lay, uint32_t B,
                                                           int mode, uint32_t *__restrict__ blk) {
    const uint32_t p = tr_index<T>();
    if (p >= B) return;
    sc w, rho;
    if (mode == 0) {
        sc_set0(w);
        sc_set0(rho);
    } else {
        T t;
        t.load(states + MERLIN_STATE_WORDS * (size_t)p);
        t.append_message(MERLIN_LABEL("proof-tail"), proofs + (size_t)p * proof_len + 256, proof_len - 256);
        t.append_message(MERLIN_LABEL("verifier-seed"), vseed, 32);
        t.append_u64(MERLIN_LABEL("proof-index"), p);
        t.challenge_scalar(MERLIN_LABEL("w"), w);
        t.challenge_scalar(MERLIN_LABEL("rho"), rho);
    }
    if (tr_leader<T>()) {
        sc_store(ACP_PTR(blk, lay, p, lay.w), w);
        sc_store(ACP_PTR(blk, lay, p, lay.rho0), rho);
    }
}

// Batch weight of the stand-alone inner-product batch (bpp_ipa_batch_verify_combined), the construction of k_tr_weights:
// a copy of proof p's final verifier state (k_ipa_vtranscript; `states` is only read, so the caller's transcript never
// sees these appends) absorbs the proof's a || b and P - which dalek's verify does not absorb: without it two proofs of
// equal bytes with P + D and P - D would get equal weights under a reused seed and cancel - then the verifier seed and
// the proof's index, and draws "rho" (at lay.rho0).  lrp: k_ipa_unpack's B x (2 lg + 1) x 32, P last; proofs: the
// uploaded proofs, a || b in their last 64 bytes.
template <class T>
__global__ void __launch_bounds__(TR_THREADS) k_ipa_weights(const uint64_t *__restrict__ states, const uint8_t *__restrict__ proofs,
                                                            const uint8_t *__restrict__ lrp, const uint8_t *__restrict__ vseed,
                                                            acp_layout lay, uint32_t B, uint32_t *__restrict__ blk) {
    const uint32_t p = tr_index<T>();
    if (p >= B) return;
    // every address taken before the sponge: this form compiles without spills in both transcript forms
    const uint32_t words = 2 * lay.lg + 2;
    const uint8_t *ab = proofs + 32 * ((size_t)p * words + words - 2), *P = lrp + 32 * ((size_t)p * (words - 1) + words - 2);
    uint32_t *dst = ACP_PTR(blk, lay, p, lay.rho0);
    T t;
    t.load(states + MERLIN_STATE_WORDS * (size_t)p);
    t.append_message(MERLIN_LABEL("proof-tail"), ab, 64);
    t.append_message(MERLIN_LABEL("P"), P, 32);
    t.append_message(MERLIN_LABEL("verifier-seed"), vseed, 32);
    t.append_u64(MERLIN_LABEL("proof-index"), p);
    sc rho;
    t.challenge_scalar(MERLIN_LABEL("rho"), rho);
    if (t.lane == 0) sc_store(dst, rho);
}

// Scripted transcript for tests (one thread): script = sequence of records
//   op (1 B: 0 = append_message, 1 = challenge_bytes) | label_len (1 B) | label | n (4 B LE) | msg (op 0 only)
// starting from Transcript::new(first record's message); challenge outputs are concatenated into out.
__global__ void k_tr_script(const uint8_t *__restrict__ script, uint32_t len, uint8_t *__restrict__ out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    merlin_tr t;
    for (int i = 0; i < 25; i++) t.st[i] = 0;
    // Strobe128::new("Merlin v1.0")
    const uint8_t init[18] = {1, 168, 1, 0, 1, 96, 'S', 'T', 'R', 'O', 'B', 'E', 'v', '1', '.', '0', '.', '2'};
    for (uint32_t i = 0; i < 18; i++) t.xor_byte(i, init[i]);
    keccak_f1600_dev(t.st);
    t.pos = 0; t.pos_begin = 0; t.cur_flags = 0;
    t.meta_ad((const uint8_t *)"Merlin v1.0", 11, false);
    uint32_t o = 0, w = 0;
    while (o < len) {
        uint32_t op = script[o], ll = script[o + 1];
        const char *label = (const char *)(script + o + 2);
        o += 2 + ll;
        uint32_t n = (uint32_t)script[o] | ((uint32_t)script[o + 1] << 8) | ((uint32_t)script[o + 2] << 16) |
                     ((uint32_t)script[o + 3] << 24);
        o += 4;
        if (op == 0) {
            t.append_message(label, ll, script + o, n);
            o += n;
        } else {
            t.challenge_bytes(label, ll, out + w, n);
            w += n;
        }
    }
}
