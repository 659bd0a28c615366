// acproof_kernels.cuh - batched arithmetic-circuit (shuffle) prover / verifier kernels for sm_100a.
//
// Re-expresses the arithmetic of /root/reference/bp-perm/src/circuit_lib.rs for a batch of B
// independent proofs that share one circuit and one set of generators:
//   create                  :139-253   A_I, A_O, S commitments          -> k_acp_rng, k_fb_msm, k_compress_batch
//   compute_per_challenges  :256-302   y^n, y^-n, z^Q, z*W, l_in, sigma -> k_acp_pow, k_acp_csr, k_acp_vec1, k_acp_dots
//   commit_Ts               :304-423   l(X), r(X), t(X), T_i            -> k_acp_vec1, k_acp_dots, k_acp_tcoef, k_fb_msm
//   blinding_values         :434-476   l, r, t, tau_x, mu               -> k_acp_final, k_acp_dots2, k_acp_final2
//   verify                  :478-585   the three checks, fused into one MSM per proof (SURVEY D.1)
//                                      -> k_acp_vscal, k_fb_msm, k_dyn_window_sums, k_dyn_horner_accept
// Each proof owns one block of scalars in HBM (layout below); a kernel touches element (proof, i) from
// one thread, so all loads are 32-byte contiguous per thread and coalesced across the warp.
#pragma once
#include "ge25519.cuh"
#include "vec_kernels.cuh"

struct acp_layout {
    uint32_t n, Q, m, stride;  // stride: scalars per proof
    uint32_t np, lg;           // `fixed` mode: n padded to a power of two and its log2 (np = n, lg = 0 otherwise);
                               // yn, yninv, l, r, vG, vH hold np entries, vd holds m + 8 + 2 lg
    uint32_t aL, aR, aO, gamma;                    // witness (uploaded)
    uint32_t alpha, beta, ro, sl, sr, tau;         // prover randomness, RNG draw order (contiguous)
    uint32_t y, z, x, w;                           // challenges, verifier weight
    uint32_t yn, yninv, zq;                        // exp_iter outputs and inverses
    uint32_t zWL, zWR, zWO, zWV, zc;               // z*W_L, z*W_R, z*W_O (n each), z*W_V (m), <z_q,c> (contiguous)
    uint32_t lin, l1, r0, r1, r3;                  // vector polynomial coefficients
    uint32_t dots;                                 // 12 block-reduced dot products
    uint32_t tc, tsel, sigma;                      // t1..t6, the five committed values, delta(y,z)
    uint32_t l, r, that, taux, mu;                 // proof scalars
    uint32_t vg, vh, vG, vH, vd;                   // verifier MSM scalars: static (contiguous g,h,G,H), dynamic (m+8)
    uint32_t rho, rho0;                            // batch verification weight: as drawn (k_tr_weights), as used (k_rlc_weights)
    uint32_t wq, u, uinv, cl, pa, pb, ptab;        // `fixed` mode: challenge w, u_j / u_j^-1 (lg each), w*c_L, w*c_R,
                                                   // the proof's a and b, 3 x IPA_MAX_LG squarings for the power tables
    uint32_t stab;                                 // `fixed` mode: 2 x n' table of the s_t (ipa_kernels.cuh)
    uint32_t vr, nx;                               // shuffle-shaped circuits: a_R = v' - x as written by the witness
                                                   // kernels, v' (n - 2) and -x (1); none otherwise
};

#define ACP_PTR(base, lay, p, off) ((base) + 8 * ((size_t)(p) * (lay).stride + (off)))

// ---- RNG: ChaCha20 keystream block j of the proof's stream -> Scalar::random -----------------------
// rand_chacha::ChaCha20Rng::from_seed(seed): key = seed, 64-bit block counter, zero nonce; each
// Scalar::random consumes exactly one 64-byte block (circuit_lib.rs:180-182,213-214,361-404).
SC_INLINE uint32_t rotl32(uint32_t v, int n) { return (v << n) | (v >> (32 - n)); }
#define CHACHA_QR(a, b, c, d) \
    a += b; d = rotl32(d ^ a, 16); c += d; b = rotl32(b ^ c, 12); a += b; d = rotl32(d ^ a, 8); c += d; b = rotl32(b ^ c, 7);

__global__ void k_acp_rng(const uint32_t *__restrict__ seeds /* B x 8 */, acp_layout lay, uint32_t count,
                          uint32_t *__restrict__ blk) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (j >= count) return;
    uint32_t s[16], x[16];
    s[0] = 0x61707865u; s[1] = 0x3320646eu; s[2] = 0x79622d32u; s[3] = 0x6b206574u;
#pragma unroll
    for (int i = 0; i < 8; i++) s[4 + i] = seeds[8 * (size_t)p + i];
    s[12] = j; s[13] = 0; s[14] = 0; s[15] = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) x[i] = s[i];
#pragma unroll 1
    for (int r = 0; r < 10; r++) {
        CHACHA_QR(x[0], x[4], x[8], x[12]) CHACHA_QR(x[1], x[5], x[9], x[13])
        CHACHA_QR(x[2], x[6], x[10], x[14]) CHACHA_QR(x[3], x[7], x[11], x[15])
        CHACHA_QR(x[0], x[5], x[10], x[15]) CHACHA_QR(x[1], x[6], x[11], x[12])
        CHACHA_QR(x[2], x[7], x[8], x[13]) CHACHA_QR(x[3], x[4], x[9], x[14])
    }
#pragma unroll
    for (int i = 0; i < 16; i++) x[i] += s[i];
    sc r;
    sc_from_wide(r, x);
    sc_store(ACP_PTR(blk, lay, p, lay.alpha + j), r);
}

// staged witness [a_L (B x n) | a_R (B x n) | a_O (B x n) | gamma (B x m)] -> the proofs' scalar blocks, each value reduced
// mod l (Scalar::from_bytes_mod_order): every kernel after this one takes canonical scalars
__global__ void __launch_bounds__(128) k_acp_place_witness(const uint32_t *__restrict__ st, acp_layout lay, uint32_t B,
                                                           uint32_t *__restrict__ blk) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    const uint32_t n = lay.n, m = lay.m;
    if (i >= 3 * n + m) return;
    const uint32_t which = i < 3 * n ? i / n : 3, k = i - which * n;
    const uint32_t *src = which < 3 ? st + 8 * (((size_t)which * B + p) * n + k) : st + 8 * ((size_t)3 * B * n + (size_t)p * m + k);
    const uint32_t off = which == 0 ? lay.aL : which == 1 ? lay.aR : which == 2 ? lay.aO : lay.gamma;
    sc s;
    sc_load(s, src);
    sc_reduce256(s, s);
    sc_store(ACP_PTR(blk, lay, p, off + k), s);
}

// caller scalars in place, mod l: rows x cnt values, row r at p + r * pitch (u32).  The shuffle witness' deck, x and
// gamma and the caller's v of bpp_acp_batch_commit, which may be any 256-bit values.
__global__ void __launch_bounds__(128) k_sc_reduce_rows(uint32_t *__restrict__ p, size_t pitch, uint32_t cnt) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cnt) return;
    uint32_t *q = p + pitch * blockIdx.y + 8 * (size_t)i;
    sc s;
    sc_load(s, q);
    sc_reduce256(s, s);
    sc_store(q, s);
}

// ---- shuffle witness on the device (replaces weights.rs:38-113 create_variables / create_a for the corrected k-card
// circuit of bpp_circuit_create_shuffle; CPU restatement: shuffle_witness in the test tree) ----------------------
// v = deck | deck[perm] | x (m = 2k + 1 committed values).  Chain c (0: input deck, 1: output deck), base multiplier
// gb = c (k - 1), base value vb = c k:  a_R[gb + i] = v[vb + i + 1] - x,  a_L[gb] = v[vb] - x,  a_L[gb + i] = a_O[gb + i - 1],
// a_O[gb + i] = a_L[gb + i] a_R[gb + i]  (i < k - 1): a_O is the running product of (v[vb + t] - x), t <= i + 1.  The two
// padding multipliers 2k - 2, 2k - 1 are zero.  Block per (chain, proof): each thread multiplies up a run of consecutive
// factors, the run totals are scanned through shared memory (Hillis-Steele), so a 4096-card chain is 8 + 9 + 8
// dependent multiplications deep instead of 4095.  Products in Montgomery form until the final store.
// Both forms also write a_R in its structured form: v'[gb + i] = v[vb + i + 1] and -x (sc_sub(0, x)), so that the prover
// can commit <a_R, H> as <v', H> + (-x) H_sum (bpp_acp_batch_prove).
// perm is device data: an index >= k asserts in the debug build and is clamped to k - 1 in the product build, so that
// it reads the deck's last card instead of whatever follows the deck (device data must not fault).
#define WIT_THREADS 256
FE_INLINE uint32_t wit_card(const uint32_t *pp, uint32_t j, uint32_t k) {
    const uint32_t i = pp[j];
    BPP_ASSERT(i < k);
    return i < k ? i : k - 1;
}
SC_INLINE void acp_store_neg_x(uint32_t *blk, const acp_layout &lay, uint32_t p, const sc &x) {
    sc z, nx;
    sc_set0(z);
    sc_sub(nx, z, x);
    sc_store(ACP_PTR(blk, lay, p, lay.nx), nx);
}
__global__ void __launch_bounds__(WIT_THREADS) k_shuffle_witness(const uint32_t *__restrict__ deck /* k x 8 */,
                                                                 const uint32_t *__restrict__ perm /* B x k */,
                                                                 const uint32_t *__restrict__ xs /* B x 8 */, uint32_t k,
                                                                 acp_layout lay, uint32_t *__restrict__ blk,
                                                                 uint32_t *__restrict__ vout /* B x m x 8 */) {
    __shared__ __align__(16) uint32_t sh[2][WIT_THREADS * 8];
    const uint32_t c = blockIdx.x, p = blockIdx.y, tid = threadIdx.x;
    const uint32_t gb = c * (k - 1), vb = c * k, len = k - 1;      // factors f_i = v[vb + i + 1] - x, i < len
    const uint32_t T = blockDim.x;   // a power of two <= WIT_THREADS: 64 threads for a 52-card chain, 256 for long ones
    const uint32_t run = (len + T - 1) / T, i0 = tid * run, i1 = min(len, i0 + run);
    const uint32_t *pp = perm + (size_t)p * k;
    uint32_t *vp = vout + 8 * (size_t)p * lay.m;
    sc x, one, r2;
    sc_load(x, xs + 8 * (size_t)p);
    sc_const(one, SC_R);
    sc_const(r2, SC_R2);
    auto value = [&](uint32_t j) {      // v[vb + j], also written out
        sc v;
        BPP_ASSERT(j < k);
        sc_load(v, deck + 8 * (size_t)(c ? wit_card(pp, j, k) : j));
        sc_store(vp + 8 * (size_t)(vb + j), v);
        return v;
    };
    // pass 1: this thread's run product (Montgomery)
    sc acc = one, f, t;
    for (uint32_t i = i0; i < i1; i++) {
        f = value(i + 1);
        sc_store(ACP_PTR(blk, lay, p, lay.vr + gb + i), f);
        sc_sub(f, f, x);
        sc_store(ACP_PTR(blk, lay, p, lay.aR + gb + i), f);
        sc_mont(t, f, r2);
        sc_mont(acc, acc, t);
    }
    if (tid == 0) {                     // the chain's first value joins the first run
        f = value(0);
        sc_sub(f, f, x);
        sc_store(ACP_PTR(blk, lay, p, lay.aL + gb), f);
        sc_mont(t, f, r2);
        sc_mont(acc, acc, t);
        if (c == 0) {
            sc_store(vp + 8 * (size_t)(2 * k), x);
            acp_store_neg_x(blk, lay, p, x);
            sc z;
            sc_set0(z);
            for (uint32_t q = 2 * k - 2; q < 2 * k; q++) {
                sc_store(ACP_PTR(blk, lay, p, lay.aL + q), z);
                sc_store(ACP_PTR(blk, lay, p, lay.aR + q), z);
                sc_store(ACP_PTR(blk, lay, p, lay.aO + q), z);
            }
        }
    }
    // inclusive scan of the run products
    int cur = 0;
    sc_store(sh[0] + 8 * tid, acc);
    __syncthreads();
    for (uint32_t d = 1; d < T; d <<= 1) {
        sc a, b2;
        sc_load(a, sh[cur] + 8 * tid);
        if (tid >= d) {
            sc_load(b2, sh[cur] + 8 * (tid - d));
            sc_mont(a, a, b2);
        }
        sc_store(sh[cur ^ 1] + 8 * tid, a);
        cur ^= 1;
        __syncthreads();
    }
    // pass 2: exclusive prefix of the earlier runs, then the run again
    if (tid) sc_load(acc, sh[cur] + 8 * (tid - 1));
    else {                              // thread 0 restarts from the first value
        sc_load(f, ACP_PTR(blk, lay, p, lay.aL + gb));
        sc_mont(acc, f, r2);
    }
    for (uint32_t i = i0; i < i1; i++) {
        sc prev;
        sc_from_mont(prev, acc);
        if (i) sc_store(ACP_PTR(blk, lay, p, lay.aL + gb + i), prev);
        sc_load(f, ACP_PTR(blk, lay, p, lay.aR + gb + i));
        sc_mont(t, f, r2);
        sc_mont(acc, acc, t);
        sc_from_mont(prev, acc);
        sc_store(ACP_PTR(blk, lay, p, lay.aO + gb + i), prev);
    }
}
// Short chains, many proofs (the 52-card batch): one THREAD per (chain, proof) walks its chain serially - 2 multiplications
// per factor (f -> f R, then P <- P f R / R: the running product stays in standard form) instead of the ~13 per thread of
// the block scan above, whose log-depth only pays when a single chain has to fill the GPU (k_shuffle_witness on the
// 4096-proof 52-card batch: 510 us = 7 % of a prove + verify step; this form: 8192 threads, ~100 multiplications deep).
__global__ void __launch_bounds__(64) k_shuffle_witness_serial(const uint32_t *__restrict__ deck /* k x 8 */,
                                                               const uint32_t *__restrict__ perm /* B x k */,
                                                               const uint32_t *__restrict__ xs /* B x 8 */, uint32_t k, uint32_t B,
                                                               acp_layout lay, uint32_t *__restrict__ blk,
                                                               uint32_t *__restrict__ vout /* B x m x 8 */) {
    const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= 2 * B) return;
    const uint32_t c = id & 1u, p = id >> 1;
    const uint32_t gb = c * (k - 1), vb = c * k, len = k - 1;
    const uint32_t *pp = perm + (size_t)p * k;
    uint32_t *vp = vout + 8 * (size_t)p * lay.m;
    sc x, r2, v, f, fm, P;
    sc_load(x, xs + 8 * (size_t)p);
    sc_const(r2, SC_R2);
    sc_load(v, deck + 8 * (size_t)(c ? wit_card(pp, 0, k) : 0));
    sc_store(vp + 8 * (size_t)vb, v);
    sc_sub(P, v, x);
    sc_store(ACP_PTR(blk, lay, p, lay.aL + gb), P);
#pragma unroll 1
    for (uint32_t i = 0; i < len; i++) {
        sc_load(v, deck + 8 * (size_t)(c ? wit_card(pp, i + 1, k) : i + 1));
        sc_store(vp + 8 * (size_t)(vb + i + 1), v);
        sc_store(ACP_PTR(blk, lay, p, lay.vr + gb + i), v);
        sc_sub(f, v, x);
        sc_store(ACP_PTR(blk, lay, p, lay.aR + gb + i), f);
        if (i) sc_store(ACP_PTR(blk, lay, p, lay.aL + gb + i), P);   // a_L[gb + i] = a_O[gb + i - 1]
        sc_mont_noinline(fm, f, r2);
        sc_mont_noinline(P, P, fm);
        sc_store(ACP_PTR(blk, lay, p, lay.aO + gb + i), P);
    }
    if (c == 0) {
        sc_store(vp + 8 * (size_t)(2 * k), x);
        acp_store_neg_x(blk, lay, p, x);
        sc z;
        sc_set0(z);
        for (uint32_t q = 2 * k - 2; q < 2 * k; q++) {
            sc_store(ACP_PTR(blk, lay, p, lay.aL + q), z);
            sc_store(ACP_PTR(blk, lay, p, lay.aR + q), z);
            sc_store(ACP_PTR(blk, lay, p, lay.aO + q), z);
        }
    }
}
// gamma (B x m, staged contiguously) -> the proofs' scalar blocks
__global__ void __launch_bounds__(128) k_acp_place_gamma(const uint32_t *__restrict__ st, acp_layout lay, uint32_t *__restrict__ blk) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (i >= lay.m) return;
    const uint32_t *src = st + 8 * ((size_t)p * lay.m + i);
    uint4 lo = *reinterpret_cast<const uint4 *>(src), hi = *reinterpret_cast<const uint4 *>(src + 4);
    uint32_t *dst = ACP_PTR(blk, lay, p, lay.gamma + i);
    *reinterpret_cast<uint4 *>(dst) = lo;
    *reinterpret_cast<uint4 *>(dst + 4) = hi;
}

// wide challenge bytes (64 B each, from the host transcripts) -> scalars at a layout offset
__global__ void k_acp_put_wide(const uint32_t *__restrict__ wide /* B x per x 16 */, acp_layout lay, uint32_t off,
                               uint32_t per, uint32_t B, uint32_t *__restrict__ blk) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * per) return;
    uint32_t p = i / per, k = i - p * per;
    uint32_t w[16];
#pragma unroll
    for (int t = 0; t < 16; t++) w[t] = wide[16 * (size_t)i + t];
    sc r;
    sc_from_wide(r, w);
    sc_store(ACP_PTR(blk, lay, p, off + k), r);
}

// ---- fixed-base tables ---------------------------------------------------------------------------
// u32 per table entry.  Padding the 96-byte entries to 128 bytes (exactly two 64-byte DRAM atoms per gather instead
// of two or three; ncu shows 2.5 GB read per launch for 1.3 GB of entries) was measured: 3 % SLOWER (1.185 vs
// 1.155 ms per A_I-shaped launch) - the larger table costs more in L2/TLB reach than the atoms save.
#define FB_ENTRY_U32 24
// table[((gen * Wn + w) * half + (j - 1))] = j * 2^(c w) * P_gen as affine Niels (96 B).
// Thread per (gen, window): 2^(c w) P by doublings, then j = 1..half by repeated addition, each
// entry normalised with its own inversion (one-time cost at generator upload).
__global__ void __launch_bounds__(64) k_fb_build(const uint32_t *__restrict__ gens_niels, uint32_t n_gens, int c,
                                                 int Wn, uint32_t *__restrict__ table) {
    uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= n_gens * (uint32_t)Wn) return;
    const uint32_t gen = id / Wn, w = id - gen * Wn;
    const uint32_t half = 1u << (c - 1);
    ge_niels q;
    ge_niels_load(q, gens_niels + 24 * (size_t)gen);
    ge_ext base, run;
    ge_identity(base);
    ge_madd(base, base, q, false);
#pragma unroll 1
    for (uint32_t i = 0; i < w * (uint32_t)c; i++) ge_double_noinline(base, base);
    run = base;
    uint32_t *dst = table + FB_ENTRY_U32 * ((size_t)id * half);
#pragma unroll 1
    for (uint32_t j = 1; j <= half; j++) {
        fe zi, x, y;
        fe_invert(zi, run.Z);
        fe_mul_noinline(x, run.X, zi);
        fe_mul_noinline(y, run.Y, zi);
        ge_niels e;
        ge_affine_to_niels(e, x, y);
        ge_niels_store(dst + FB_ENTRY_U32 * (size_t)(j - 1), e);
        if (j < half) ge_add_noinline(run, run, base);
    }
}

// ---- batched fixed-base MSM ----------------------------------------------------------------------
// One block per output point.  The MSM's terms are up to 4 segments of (scalar range in the proof
// block) x (generator range); every term costs Wn table look-ups + mixed adds, no doublings and no
// buckets.  Signed digits without a carry chain: s' = s + sum_{w < Wn-1} half*2^(cw), digit_w =
// window_w(s') - half (top window unsigned), so any (term, window) can be evaluated independently.
struct fb_shape {
    uint32_t nseg;
    uint32_t sc_off[4];      // scalar offset of the segment inside the proof block
    uint32_t sc_ostride[4];  // added per output index (blockIdx.y)
    uint32_t gen[4];         // first generator of the segment
    uint32_t cnt[4];
    uint32_t outs;           // outputs per proof (gridDim.y)
    uint32_t sel_period;     // 0 = off.  IPA rounds (ipa_kernels.cuh): term k of a segment belongs to output 0 (L) or
    uint32_t sel[4];         // 1 (R) by the half of its period it lies in: sel 1 = upper half -> L, 2 = lower half -> L
};
// k_fb_msm_warp_d<C, true> only (fb_warp_d_fits), kept out of fb_shape so that the other table kernels' parameters stay
// as they were measured: segments of mask `alt` index alt_table (a table of the same width) instead of the launch's
// table, and terms with at most FB_SPARSE_MAX non-zero digits are spread over all lanes
struct fb_sparse {
    uint32_t on, alt;
    const uint32_t *alt_table;
};
struct fb_consts {
    uint32_t K[8];  // sum_{w < Wn-1} half * 2^(c w)
};
#ifndef FB_THREADS
#define FB_THREADS 128
#endif
#ifndef FB_GROUP
#define FB_GROUP 4  // windows handled per work item
#endif

// ---- pieces shared by the table kernels ----
static __host__ __device__ __forceinline__ uint32_t fb_terms(const fb_shape &sh) {
    uint32_t n = 0;
    for (uint32_t s = 0; s < sh.nseg; s++) n += sh.cnt[s];
    return n;
}
// term t -> (segment, index k inside the segment)
__device__ __forceinline__ void fb_locate_term(const fb_shape &sh, uint32_t t, uint32_t &seg, uint32_t &k) {
    seg = 0;
    k = t;
    while (seg + 1 < sh.nseg && k >= sh.cnt[seg]) { k -= sh.cnt[seg]; seg++; }
}
// whether term k of segment seg enters output o: L (o = 0) takes the upper half of each period where sel is 1, the lower
// half where sel is 2, and R the other half; every term enters when sel_period or sel is 0
__device__ __forceinline__ bool fb_term_selected(const fb_shape &sh, uint32_t seg, uint32_t k, uint32_t o) {
    if (!sh.sel_period || !sh.sel[seg]) return true;
    const bool upper = (k & (sh.sel_period - 1)) >= (sh.sel_period >> 1);
    return (upper == (o == 0)) == (sh.sel[seg] == 1);
}
__device__ __forceinline__ const uint32_t *fb_scalar(const uint32_t *blk, const acp_layout &lay, const fb_shape &sh, uint32_t p,
                                                     uint32_t o, uint32_t seg, uint32_t k) {
    return ACP_PTR(blk, lay, p, sh.sc_off[seg] + o * sh.sc_ostride[seg] + k);
}
// s[0..8) = the low 256 bits of s' = *sp + K; returns the carry out of them (s'[8] of the 9-limb form)
__device__ __forceinline__ uint32_t fb_recode(const uint32_t *sp, const uint32_t *K, uint32_t *s) {
    const uint4 lo = *reinterpret_cast<const uint4 *>(sp), hi = *reinterpret_cast<const uint4 *>(sp + 4);
    s[0] = lo.x; s[1] = lo.y; s[2] = lo.z; s[3] = lo.w; s[4] = hi.x; s[5] = hi.y; s[6] = hi.z; s[7] = hi.w;
    unsigned long long carry = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        carry += (unsigned long long)s[i] + K[i];
        s[i] = (uint32_t)carry;
        carry >>= 32;
    }
    return (uint32_t)carry;
}
// signed digit of window w from the 9 limbs of s'
__device__ __forceinline__ int fb_digit(const uint32_t *s, int c, int Wn, uint32_t w) {
    const int bit = c * (int)w, limb = bit >> 5, shf = bit & 31;
    unsigned long long v = s[limb];
    if (limb + 1 < 9) v |= (unsigned long long)s[limb + 1] << 32;
    const uint32_t u = (uint32_t)(v >> shf) & ((1u << c) - 1u);
    return w + 1 == (uint32_t)Wn ? (int)u : (int)u - (int)(1u << (c - 1));
}
// mag * 2^(c w) * P_gen (layout of k_fb_build)
__device__ __forceinline__ const uint32_t *fb_entry(const uint32_t *table, uint32_t gen, int Wn, uint32_t half, uint32_t w,
                                                    uint32_t mag) {
    return table + FB_ENTRY_U32 * (((size_t)gen * Wn + w) * half + (mag - 1));
}
// acc = the sum of the stream advance(ptr, neg) yields: (table entry, sign) pairs until it returns false.  The stream is
// software pipelined: the next entry's 96-byte gather (random access into a multi-GB table) is issued before the current
// mixed add.
template <class Advance>
__device__ __forceinline__ void fb_accumulate(ge_ext &acc, Advance &advance) {
    ge_identity(acc);
    const uint32_t *ptr = nullptr, *ptr_n = nullptr;
    bool neg = false, neg_n = false;
    bool ok = advance(ptr, neg);
    ge_niels q, qn;
    if (ok) ge_niels_load(q, ptr);
#pragma unroll 1
    while (ok) {
        bool ok_n = advance(ptr_n, neg_n);
        qn = q;
        if (ok_n) ge_niels_load(qn, ptr_n);
        ge_madd(acc, acc, q, neg);
        q = qn;
        neg = neg_n;
        ok = ok_n;
    }
}
// lane 0: the sum of the warp's 32 points, in five shuffle steps.  NOINLINE: the adds as calls (fewer registers).
template <bool NOINLINE>
__device__ __forceinline__ void ge_warp_sum(ge_ext &acc) {
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
        if (NOINLINE) ge_add_noinline(acc, acc, o2);
        else ge_add(acc, acc, o2);
    }
}
// k_fb_msm and k_fb_msm_warp: this thread's work items (term, group of FB_GROUP windows) of output o - it, it + stride,
// ... - as one stream of non-zero digits into fb_accumulate.  scalar(seg, k, term): where the term's scalar is read.
// s: the 9 words of the current term's s' - indexed by the window, so in local memory; the kernel owns the array, which
// keeps its stack frame and register allocation as they were measured.
template <class Scalar>
__device__ __forceinline__ void fb_accumulate_items(ge_ext &acc, uint32_t (&s)[9], const fb_shape &sh, const uint32_t *table, int c, int Wn,
                                                    const fb_consts &kc, uint32_t o, uint32_t total_terms, uint32_t it,
                                                    uint32_t stride, Scalar scalar) {
    const uint32_t half = 1u << (c - 1);
    const uint32_t groups = (Wn + FB_GROUP - 1) / FB_GROUP;
    const uint32_t items = total_terms * groups;
    uint32_t w = 0, w_end = 0, gen = 0;
    bool first = true;
    auto advance = [&](const uint32_t *&ptr, bool &neg) -> bool {
        for (;;) {
            if (w >= w_end) {
                if (!first) it += stride;
                first = false;
                if (it >= items) return false;
                const uint32_t term = it / groups, grp = it - term * groups;
                uint32_t seg, k;
                fb_locate_term(sh, term, seg, k);
                w = grp * FB_GROUP;
                w_end = min((uint32_t)Wn, (grp + 1) * FB_GROUP);
                if (!fb_term_selected(sh, seg, k, o)) { w = w_end; continue; }
                gen = sh.gen[seg] + k;
                s[8] = fb_recode(scalar(seg, k, term), kc.K, s);
            }
            const uint32_t ww = w++;
            const int d = fb_digit(s, c, Wn, ww);
            if (d == 0) continue;
            const uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
            BPP_ASSERT(mag >= 1 && mag <= half && ww < (uint32_t)Wn && it < items);
            ptr = fb_entry(table, gen, Wn, half, ww, mag);
            neg = d < 0;
            return true;
        }
    };
    fb_accumulate(acc, advance);
}

// ---- the table kernels ----
__global__ void __launch_bounds__(FB_THREADS) k_fb_msm(const uint32_t *__restrict__ blk, acp_layout lay, fb_shape sh,
                                                       const uint32_t *__restrict__ table, int c, int Wn, fb_consts kc,
                                                       uint32_t *__restrict__ out_ext /* [p][outs] x 32 */) {
    __shared__ __align__(16) uint32_t red[FB_THREADS][32];
    const uint32_t p = blockIdx.x, o = blockIdx.y;
    uint32_t s[9];
    ge_ext acc;
    // work items strided over the block and its gridDim.z splits
    fb_accumulate_items(acc, s, sh, table, c, Wn, kc, o, fb_terms(sh), blockIdx.z * FB_THREADS + threadIdx.x, FB_THREADS * gridDim.z,
                        [&](uint32_t seg, uint32_t k, uint32_t) { return fb_scalar(blk, lay, sh, p, o, seg, k); });
    // block tree reduction
    ge_store(&red[threadIdx.x][0], acc);
    __syncthreads();
#pragma unroll 1
    for (uint32_t dstep = FB_THREADS / 2; dstep >= 1; dstep >>= 1) {
        if (threadIdx.x < dstep) {
            ge_ext a, b;
            ge_load(a, &red[threadIdx.x][0]);
            ge_load(b, &red[threadIdx.x + dstep][0]);
            ge_add(a, a, b);
            ge_store(&red[threadIdx.x][0], a);
        }
        __syncthreads();
    }
    if (threadIdx.x < 32) {  // gridDim.z > 1: partial sums, [p][o][z], added up by k_fb_sum_splits
        uint32_t *dst = gridDim.z == 1 ? out_ext + 32 * ((size_t)p * sh.outs + o)
                                       : out_ext + 32 * (((size_t)p * gridDim.y + o) * gridDim.z + blockIdx.z);
        dst[threadIdx.x] = red[0][threadIdx.x];
    }
}
// One WARP per output point (large batches: B x outs warps fill the GPU): no shared memory, no block barrier - the
// 32 partial sums meet in five shuffle steps.  (ncu of the block-per-output form, profiles/r1_ncu_full_k_fb_msm.csv:
// barrier stalls 1.7 per issue from the 7-level shared-memory tree.)
// STAGE: the warp first copies the scalars of all its terms into shared memory (coalesced 32-byte loads, one pass), so
// that the per-item scalar fetch - every FB_GROUP mixed adds, an un-prefetched global load on which the digit extraction
// waits: 12 % of the warp stall samples in profiles/r2_ncu_full_k_fb_msm_warp.csv - becomes a shared-memory read.
// Dynamic shared memory: (FB_THREADS / 32) x total_terms x 32 B (the host picks STAGE when that fits 48 KB).
#ifndef FB_WARP_MINBLOCKS
#define FB_WARP_MINBLOCKS 4
#endif
template <bool STAGE>
__global__ void __launch_bounds__(FB_THREADS, FB_WARP_MINBLOCKS) k_fb_msm_warp(const uint32_t *__restrict__ blk, acp_layout lay, fb_shape sh,
                                                            const uint32_t *__restrict__ table, int c, int Wn, fb_consts kc,
                                                            uint32_t B, uint32_t outs /* per proof; sh.outs = pitch */,
                                                            uint32_t *__restrict__ out_ext /* [p][pitch] x 32 */) {
    extern __shared__ __align__(16) uint32_t fb_stage[];
    const uint32_t wid = blockIdx.x * (FB_THREADS / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (wid >= B * outs) return;   // whole warps leave together
    const uint32_t p = wid / outs, o = wid - p * outs;
    const uint32_t total_terms = fb_terms(sh);
    uint32_t *stage = fb_stage + 8 * (size_t)(threadIdx.x >> 5) * total_terms;
    if (STAGE) {
        for (uint32_t t = lane; t < total_terms; t += 32) {
            uint32_t seg, k;
            fb_locate_term(sh, t, seg, k);
            const uint32_t *sp = fb_scalar(blk, lay, sh, p, o, seg, k);
            const uint4 lo = *reinterpret_cast<const uint4 *>(sp), hi = *reinterpret_cast<const uint4 *>(sp + 4);
            *reinterpret_cast<uint4 *>(stage + 8 * (size_t)t) = lo;
            *reinterpret_cast<uint4 *>(stage + 8 * (size_t)t + 4) = hi;
        }
        __syncwarp();
    }
    uint32_t s[9];
    ge_ext acc;
    // work items strided over the warp
    fb_accumulate_items(acc, s, sh, table, c, Wn, kc, o, total_terms, lane, 32, [&](uint32_t seg, uint32_t k, uint32_t term) {
        return STAGE ? stage + 8 * (size_t)term : fb_scalar(blk, lay, sh, p, o, seg, k);
    });
    ge_warp_sum<false>(acc);
    if (lane == 0) ge_store(out_ext + 32 * ((size_t)p * sh.outs + o), acc);
}
// Digit-staged form of k_fb_msm_warp for the window widths whose window count is a power of two (c = 16: 16 windows,
// c = 8: 32).  The source page of the form above (profiles/r2_ncu_source_fb_msm_warp.csv.gz) shows where its issue slots
// go besides the mixed adds: ~200 of ~1200 warp instructions per add are the work-item bookkeeping (term / segment walk,
// an 8-limb s + K, a local-memory array indexed by the window, 64-bit table index arithmetic on the multiplier pipe), and
// every long-scoreboard stall (9.8 % of the samples) sits on that bookkeeping, none on the prefetched table gathers.
// Here the warp does the bookkeeping ONCE while staging: the terms selected for this output are compacted (ballot +
// popc), s' = s + K is written to shared memory - for these widths the digits of s' ARE its 16-bit / 8-bit fields - with
// the generator index beside it.  The main loop then is: one LDS.U16 (digit), one LDS (generator), a shift/or for the
// table entry - and, since the lane stride 32 is a multiple of the window count, a lane keeps the same window for its
// whole life (ww = lane mod Wn): items are single (term, window) pairs, so lanes differ by at most one mixed add
// (the 4-window items above: by four).  Dynamic shared memory: (FB_THREADS / 32) x total_terms x 36 B.
//
// SPARSE (launches with sp.on set): a term with at most FB_SPARSE_MAX non-zero digits - a small scalar, such as a
// card value of the shuffle witness, has one - would put all its work on the lanes of those windows (lanes 0 and 16 for
// a value below 2^15) while the other 30 lanes idle.  Such terms are not staged as digits: while staging, each of
// their non-zero digits becomes one word (entry << 1 | sign) of a per-warp list, compacted with ballot + popc, and the
// lanes take that list round-robin after their dense items, continuing the lane order where the dense items stop, so the
// mixed adds per lane differ by at most one (skipped zero digits aside).  Terms of an `alt` segment (their generator
// index carries FB_ALT) read sp.alt_table and always stay dense.  The list is sized for the worst case: 2 words per
// term, (FB_THREADS / 32) x total_terms x 8 B more dynamic shared memory.
#ifndef FB_STAGE_MAX_BYTES
#define FB_STAGE_MAX_BYTES (48u * 1024u)   // dynamic shared memory without an opt-in attribute
#endif
#define FB_SPARSE_MAX 2
#define FB_ALT 0x80000000u
// 32-bit words per warp of the digit-staged form's stage: s' (8 per term) and the generator index, rounded up to 16
// bytes; with SPARSE the list after them
static __host__ __device__ __forceinline__ uint32_t fb_stage_d_words(uint32_t terms, bool sparse) {
    return ((9 * terms + 3) & ~3u) + (sparse ? FB_SPARSE_MAX * terms : 0);
}
template <int C>
__device__ __forceinline__ uint32_t fb_field(const uint32_t (&s)[8], uint32_t w) {   // w: a compile-time constant after unrolling
    return C == 16 ? (s[w >> 1] >> (16 * (w & 1))) & 0xffffu : (s[w >> 2] >> (8 * (w & 3))) & 0xffu;
}
template <int C, bool SPARSE>
__global__ void __launch_bounds__(FB_THREADS, FB_WARP_MINBLOCKS) k_fb_msm_warp_d(const uint32_t *__restrict__ blk, acp_layout lay, fb_shape sh,
                                                              const uint32_t *__restrict__ table, fb_consts kc, fb_sparse sp,
                                                              uint32_t B, uint32_t outs /* per proof; sh.outs = pitch */,
                                                              uint32_t *__restrict__ out_ext /* [p][pitch] x 32 */) {
    constexpr uint32_t WN = (256 + C - 1) / C, LOG_WN = WN == 32 ? 5 : 4, HALF = 1u << (C - 1);
    static_assert((C == 16 && WN == 16) || (C == 8 && WN == 32), "window count must be a power of two dividing 32");
    extern __shared__ __align__(16) uint32_t fb_stage[];
    const uint32_t wid = blockIdx.x * (FB_THREADS / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (wid >= B * outs) return;   // whole warps leave together
    const uint32_t p = wid / outs, o = wid - p * outs;
    const uint32_t total_terms = fb_terms(sh);
    const uint32_t lt = (1u << lane) - 1u;
    // per warp: total_terms x 8 words of s', then the generator indices (region rounded up to 16 bytes), then the list
    uint32_t *stage = fb_stage + (size_t)(threadIdx.x >> 5) * fb_stage_d_words(total_terms, SPARSE);
    uint32_t *sgen = stage + 8 * (size_t)total_terms;
    uint32_t *slist = stage + fb_stage_d_words(total_terms, false);
    uint32_t n_act = 0, n_sp = 0;
    for (uint32_t t0 = 0; t0 < total_terms; t0 += 32) {
        const uint32_t t = t0 + lane;
        bool act = t < total_terms;
        uint32_t seg = 0, k = t, gen = 0;
        uint32_t s[8];
        if (act) {
            fb_locate_term(sh, t, seg, k);
            act = fb_term_selected(sh, seg, k, o);
        }
        if (act) {
            const uint32_t carry = fb_recode(fb_scalar(blk, lay, sh, p, o, seg, k), kc.K, s);
            BPP_ASSERT(carry == 0);   // s' < 2^256 (s < 2^255, K < 2^(C (WN - 1)))
            (void)carry;
            gen = sh.gen[seg] + k;
            if (SPARSE && ((sp.alt >> seg) & 1u)) gen |= FB_ALT;
        }
        if (SPARSE) {
            uint32_t nz = 0;
            if (act && !(gen & FB_ALT)) {
#pragma unroll
                for (uint32_t w = 0; w < WN; w++) nz += fb_field<C>(s, w) != (w == WN - 1 ? 0u : HALF);
            }
            const bool sp = act && !(gen & FB_ALT) && nz <= FB_SPARSE_MAX;
            static_assert(FB_SPARSE_MAX == 2, "the list positions below count terms of one and of two digits");
            const uint32_t b1 = __ballot_sync(0xffffffffu, sp && nz == 1), b2 = __ballot_sync(0xffffffffu, sp && nz == 2);
            if (sp) {
                uint32_t pos = n_sp + __popc(b1 & lt) + 2 * __popc(b2 & lt);
#pragma unroll
                for (uint32_t w = 0; w < WN; w++) {
                    const uint32_t u = fb_field<C>(s, w);
                    const int d = w == WN - 1 ? (int)u : (int)u - (int)HALF;
                    if (d != 0) {
                        const uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
                        BPP_ASSERT(pos < FB_SPARSE_MAX * total_terms);
                        slist[pos++] = ((((gen << LOG_WN) + w) << (C - 1)) + (mag - 1)) << 1 | (d < 0 ? 1u : 0u);
                    }
                }
            }
            n_sp += __popc(b1) + 2 * __popc(b2);
            act = act && !sp;
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, act);
        if (act) {
            const uint32_t idx = n_act + __popc(bal & lt);
            BPP_ASSERT(idx < total_terms);
            *reinterpret_cast<uint4 *>(stage + 8 * (size_t)idx) = make_uint4(s[0], s[1], s[2], s[3]);
            *reinterpret_cast<uint4 *>(stage + 8 * (size_t)idx + 4) = make_uint4(s[4], s[5], s[6], s[7]);
            sgen[idx] = gen;
        }
        n_act += __popc(bal);
    }
    __syncwarp();
    const uint32_t items = n_act << LOG_WN;
    const uint32_t ww = lane & (WN - 1);
    const bool top = ww == WN - 1;                      // the top window's digit is unsigned
    const uint32_t lane_entry = ww << (C - 1);          // entry = (gen * WN + ww) * HALF + mag - 1
    uint32_t it = lane;
    uint32_t js = (lane - items) & 31u;                 // list word js goes to lane (items + js) mod 32
    auto advance = [&](const uint32_t *&ptr, bool &neg) -> bool {
        for (;;) {
            if (it >= items) {
                if (!SPARSE || js >= n_sp) return false;
                const uint32_t wd = slist[js];
                js += 32;
                ptr = table + (size_t)(wd >> 1) * FB_ENTRY_U32;
                neg = wd & 1u;
                return true;
            }
            const uint32_t term = it >> LOG_WN;
            it += 32;
            uint32_t u;
            if (C == 16) u = reinterpret_cast<const uint16_t *>(stage)[(term << 4) + ww];
            else u = reinterpret_cast<const uint8_t *>(stage)[(term << 5) + ww];
            const int d = top ? (int)u : (int)u - (int)HALF;
            if (d == 0) continue;
            const uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
            const uint32_t g = sgen[term];
            const uint32_t entry = ((g << LOG_WN) << (C - 1)) + lane_entry + (mag - 1);   // the shift drops FB_ALT
            BPP_ASSERT(mag >= 1 && mag <= HALF && term < n_act);
            ptr = (SPARSE && (g & FB_ALT) ? sp.alt_table : table) + (size_t)entry * FB_ENTRY_U32;
            neg = d < 0;
            return true;
        }
    };
    ge_ext acc;
    fb_accumulate(acc, advance);
    ge_warp_sum<false>(acc);
    if (lane == 0) ge_store(out_ext + 32 * ((size_t)p * sh.outs + o), acc);
}
// whether fb_warp_launch runs shape sh in the digit-staged form: the window width has one, its stage fits and the entry
// indices fit 32 bits (31 with SPARSE: the list words carry the sign beside them; the alt table has generator 0 only)
static inline bool fb_warp_d_fits(const fb_shape &sh, const fb_sparse &sp, int c, int Wn) {
    uint64_t gen_end = 0;
    for (uint32_t k = 0; k < sh.nseg; k++) {
        const uint64_t e = ((sp.alt >> k) & 1u) ? 1 : (uint64_t)sh.gen[k] + sh.cnt[k];
        gen_end = gen_end > e ? gen_end : e;
    }
    const bool fits = ((gen_end * Wn) << (c - 1)) < (sp.on ? 1ull << 31 : 1ull << 32);
    const size_t stage_d = (size_t)(FB_THREADS / 32) * fb_stage_d_words(fb_terms(sh), sp.on != 0) * 4;
    return fits && stage_d <= FB_STAGE_MAX_BYTES && (c == 16 || c == 8);
}
// host side: the warp-per-output launch.  The digit-staged form where fb_warp_d_fits; else the scalar-staged form where
// its stage fits; else the unstaged form.  A launch with sp.on or sp.alt set only runs in the digit-staged form (the
// caller checks fb_warp_d_fits).
static inline void fb_warp_launch(const uint32_t *d_sc, const acp_layout &lay, const fb_shape &sh, const uint32_t *table, int c, int Wn,
                                  const fb_consts &kc, uint32_t B, uint32_t outs, uint32_t *d_ext, cudaStream_t st,
                                  const fb_sparse &sp = fb_sparse{}) {
    const uint32_t n_out = B * outs, terms = fb_terms(sh);
    const unsigned grid = (n_out + FB_THREADS / 32 - 1) / (FB_THREADS / 32);
    const size_t stage_d = (size_t)(FB_THREADS / 32) * fb_stage_d_words(terms, sp.on != 0) * 4,
                 stage_b = (size_t)(FB_THREADS / 32) * terms * 32;
    if (fb_warp_d_fits(sh, sp, c, Wn)) {
        if (sp.on && c == 16) k_fb_msm_warp_d<16, true><<<grid, FB_THREADS, stage_d, st>>>(d_sc, lay, sh, table, kc, sp, B, outs, d_ext);
        else if (sp.on) k_fb_msm_warp_d<8, true><<<grid, FB_THREADS, stage_d, st>>>(d_sc, lay, sh, table, kc, sp, B, outs, d_ext);
        else if (c == 16) k_fb_msm_warp_d<16, false><<<grid, FB_THREADS, stage_d, st>>>(d_sc, lay, sh, table, kc, sp, B, outs, d_ext);
        else k_fb_msm_warp_d<8, false><<<grid, FB_THREADS, stage_d, st>>>(d_sc, lay, sh, table, kc, sp, B, outs, d_ext);
    } else if (stage_b <= FB_STAGE_MAX_BYTES) {
        k_fb_msm_warp<true><<<grid, FB_THREADS, stage_b, st>>>(d_sc, lay, sh, table, c, Wn, kc, B, outs, d_ext);
    } else {
        k_fb_msm_warp<false><<<grid, FB_THREADS, 0, st>>>(d_sc, lay, sh, table, c, Wn, kc, B, outs, d_ext);
    }
}
// Few-term shapes (T_i = t_i*g + tau_i*h, V_j = v_j*g + gamma_j*h: 2 terms): one THREAD per output point
// walks its terms x windows serially - no block tree, no idle lanes.
__global__ void __launch_bounds__(128) k_fb_msm_small(const uint32_t *__restrict__ blk, acp_layout lay, fb_shape sh,
                                                      const uint32_t *__restrict__ table, int c, int Wn, fb_consts kc,
                                                      uint32_t B, uint32_t outs /* per proof; sh.outs = pitch */,
                                                      uint32_t *__restrict__ out_ext /* [p][pitch] x 32 */) {
    const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= B * outs) return;
    const uint32_t p = id / outs, o = id - p * outs;
    const uint32_t half = 1u << (c - 1);
    ge_ext acc;
    ge_identity(acc);
#pragma unroll 1
    for (uint32_t seg = 0; seg < sh.nseg; seg++) {
#pragma unroll 1
        for (uint32_t k = 0; k < sh.cnt[seg]; k++) {
            const uint32_t gen = sh.gen[seg] + k;
            uint32_t s[9];
            s[8] = fb_recode(fb_scalar(blk, lay, sh, p, o, seg, k), kc.K, s);
#pragma unroll 1
            for (uint32_t w = 0; w < (uint32_t)Wn; w++) {
                const int d = fb_digit(s, c, Wn, w);
                if (d == 0) continue;
                const uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
                ge_niels q;
                ge_niels_load(q, fb_entry(table, gen, Wn, half, w, mag));
                ge_madd(acc, acc, q, d < 0);
            }
        }
    }
    ge_store(out_ext + 32 * ((size_t)p * sh.outs + o), acc);
}

// warp per output: sum of `splits` partial points -> dst[p * pitch + o]
__global__ void __launch_bounds__(32) k_fb_sum_splits(const uint32_t *__restrict__ part, uint32_t outs, uint32_t splits,
                                                      uint32_t pitch, uint32_t *__restrict__ dst) {
    const uint32_t p = blockIdx.x, o = blockIdx.y, lane = threadIdx.x;
    const uint32_t *src = part + 32 * ((size_t)p * outs + o) * splits;
    ge_ext acc, t;
    ge_identity(acc);
#pragma unroll 1
    for (uint32_t z = lane; z < splits; z += 32) {
        ge_load(t, src + 32 * (size_t)z);
        ge_add(acc, acc, t);
    }
    ge_warp_sum<true>(acc);
    if (lane == 0) ge_store(dst + 32 * ((size_t)p * pitch + o), acc);
}

// one warp: out = the sum of the points niels[first .. first + cnt) (one-time: H_sum of bpp_acp_batch_create)
__global__ void __launch_bounds__(32) k_point_sum(const uint32_t *__restrict__ niels, uint32_t first, uint32_t cnt,
                                                  uint32_t *__restrict__ out_ext) {
    ge_ext acc;
    ge_identity(acc);
#pragma unroll 1
    for (uint32_t i = threadIdx.x; i < cnt; i += 32) {
        ge_niels q;
        ge_niels_load(q, niels + 24 * (size_t)(first + i));
        ge_madd(acc, acc, q, false);
    }
    ge_warp_sum<true>(acc);
    if (threadIdx.x == 0) ge_store(out_ext, acc);
}

// thread per point: ext (raw limbs) -> 32-byte encoding
__global__ void __launch_bounds__(128) k_compress_batch(const uint32_t *__restrict__ ext, uint32_t n,
                                                        uint8_t *__restrict__ out32) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ge_ext p;
    ge_load(p, ext + 32 * (size_t)i);
    ge_compress(out32 + 32 * (size_t)i, p);
}

// ---- per-challenge scalars -------------------------------------------------------------------------
// Three threads per proof (one per warp of the block): y_n = exp_iter(y) (n), z_q = exp_iter(z) (Q) with
// the reference's Fibonacci recurrence (util.rs:139-157), and y_n_inv.  The reference inverts every
// y_n[i] (circuit_lib.rs:273-275); since y_n[i] = y^F(i), its inverse is (y^-1)^F(i): ONE inversion, then
// the same recurrence started from y^-1 - identical values (dalek's invert(0) = 0 also falls out: the
// chain of 0 is 0).  All chains stay in Montgomery form.
#define ACP_POW_THREADS 96
__global__ void __launch_bounds__(ACP_POW_THREADS) k_acp_pow(acp_layout lay, uint32_t B, uint32_t *__restrict__ blk) {
    const uint32_t p = blockIdx.x * 32 + (threadIdx.x & 31);
    const int which = threadIdx.x >> 5;   // 0: y chain, 1: z chain, 2: y^-1 chain
    if (p >= B) return;
    sc one_m;
    sc_const(one_m, SC_R);
    const uint32_t cnt = which == 1 ? lay.Q : lay.n;
    uint32_t *dst = ACP_PTR(blk, lay, p, which == 0 ? lay.yn : which == 1 ? lay.zq : lay.yninv);
    sc base = one_m, nxt, ret;
    sc_load(nxt, ACP_PTR(blk, lay, p, which == 1 ? lay.z : lay.y));
    if (which == 2) sc_invert(nxt, nxt);
    sc_to_mont(nxt, nxt);
    // the chain stores Montgomery-form values: one dependent multiplication per step; k_acp_vec1 converts y_n and
    // y_n_inv afterwards (and uses their Montgomery forms), k_acp_pow_unmont z_q, with one thread per element
#pragma unroll 1
    for (uint32_t i = 0; i < cnt; i++) {
        ret = nxt;
        sc_mont(nxt, nxt, base);
        base = ret;
        sc_store(dst + 8 * (size_t)i, ret);
    }
}
// z_q: Montgomery form -> standard form, in place
__global__ void __launch_bounds__(128) k_acp_pow_unmont(acp_layout lay, uint32_t *__restrict__ blk) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (i >= lay.Q) return;
    uint32_t *ptr = ACP_PTR(blk, lay, p, lay.zq + i);
    sc v;
    sc_load(v, ptr);
    sc_from_mont(v, v);
    sc_store(ptr, v);
}

// CSR weights.  Row r of the concatenation [W_L (n) | W_R (n) | W_O (n) | W_V (m) | c (1)] holds
// (constraint q, coefficient) pairs; out[r] = sum coeff * z_q[q]  (vm_mult(z_q, W) of util.rs:22-38
// without the dense zero entries; <z_q, c> for the last row).  kind: 1 = +1, 2 = -1, 0 = general.
struct acp_csr {
    const uint32_t *rowptr;   // rows + 1
    const uint32_t *col;      // nnz
    const uint8_t *kind;      // nnz
    const uint32_t *coeff;    // nnz x 8 (used when kind == 0)
    uint32_t rows;
};
// rows of more than ACP_CSR_LONG entries (the shuffle circuit has one: the challenge value's row of W_V, 2k - 2
// entries) are left to k_acp_csr_long, a block per (row, proof) - one thread walking 8190 entries is 2.5 ms of a
// single-proof 4096-card prover and of its verifier (profiles/r2a_launches_large_deck.csv)
#define ACP_CSR_LONG 64
SC_INLINE void acp_csr_term(sc &acc, const acp_csr &W, const uint32_t *zq, uint32_t e) {
    sc z, t, cf;
    BPP_ASSERT(e < W.rowptr[W.rows]);
    sc_load(z, zq + 8 * (size_t)W.col[e]);
    const uint8_t k = W.kind[e];
    if (k == 1) sc_add(acc, acc, z);
    else if (k == 2) sc_sub(acc, acc, z);
    else {
        sc_load(cf, W.coeff + 8 * (size_t)e);
        sc_mul(t, cf, z);
        sc_add(acc, acc, t);
    }
}
__global__ void __launch_bounds__(128) k_acp_csr(acp_csr W, acp_layout lay, uint32_t *__restrict__ blk) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (r >= W.rows) return;
    const uint32_t e0 = W.rowptr[r], e1 = W.rowptr[r + 1];
    if (e1 - e0 > ACP_CSR_LONG) return;
    const uint32_t *zq = ACP_PTR(blk, lay, p, lay.zq);
    sc acc;
    sc_set0(acc);
    for (uint32_t e = e0; e < e1; e++) acp_csr_term(acc, W, zq, e);
    sc_store(ACP_PTR(blk, lay, p, lay.zWL + r), acc);
}
__global__ void __launch_bounds__(128) k_acp_csr_long(acp_csr W, const uint32_t *__restrict__ long_rows, acp_layout lay,
                                                      uint32_t *__restrict__ blk) {
    __shared__ __align__(16) uint32_t sh[32 * 8];
    const uint32_t r = long_rows[blockIdx.x], p = blockIdx.y;
    BPP_ASSERT(r < W.rows);
    const uint32_t *zq = ACP_PTR(blk, lay, p, lay.zq);
    sc acc, tot;
    sc_set0(acc);
    for (uint32_t e = W.rowptr[r] + threadIdx.x; e < W.rowptr[r + 1]; e += blockDim.x) acp_csr_term(acc, W, zq, e);
    block_sum_sc(tot, acc, sh);
    if (threadIdx.x == 0) sc_store(ACP_PTR(blk, lay, p, lay.zWL + r), tot);
}

// thread per (proof, i < n): l_in (prover and verifier), l1, r0, r1, r3 (prover only; circuit_lib.rs:286,313-339).
// MONT: y_n[i] and y_n_inv[i] arrive in Montgomery form from k_acp_pow and are written back in standard form here, so
// that each product y^i v or y^-i v is one Montgomery multiplication; otherwise (k_pow_fill's standard powers) they are
// taken to Montgomery form first.
template <bool PROVER, bool MONT>
__global__ void __launch_bounds__(128) k_acp_vec1(acp_layout lay, uint32_t *__restrict__ blk) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (i >= lay.n) return;
    sc yn, ynr, yir, zwr, lin, t;
    sc_load(ynr, ACP_PTR(blk, lay, p, lay.yn + i));
    sc_load(yir, ACP_PTR(blk, lay, p, lay.yninv + i));
    if (MONT) {
        sc_from_mont(yn, ynr);
        sc_store(ACP_PTR(blk, lay, p, lay.yn + i), yn);
        sc_from_mont(t, yir);
        sc_store(ACP_PTR(blk, lay, p, lay.yninv + i), t);
    } else {
        yn = ynr;
        if (PROVER) sc_to_mont(ynr, yn);
        sc_to_mont(yir, yir);
    }
    sc_load(zwr, ACP_PTR(blk, lay, p, lay.zWR + i));
    sc_mont(lin, yir, zwr);
    sc_store(ACP_PTR(blk, lay, p, lay.lin + i), lin);
    if (!PROVER) return;
    sc zwl, zwo, al, ar, srv;
    sc_load(zwl, ACP_PTR(blk, lay, p, lay.zWL + i));
    sc_load(zwo, ACP_PTR(blk, lay, p, lay.zWO + i));
    sc_load(al, ACP_PTR(blk, lay, p, lay.aL + i));
    sc_load(ar, ACP_PTR(blk, lay, p, lay.aR + i));
    sc_load(srv, ACP_PTR(blk, lay, p, lay.sr + i));
    sc_add(t, al, lin);
    sc_store(ACP_PTR(blk, lay, p, lay.l1 + i), t);
    sc_sub(t, zwo, yn);
    sc_store(ACP_PTR(blk, lay, p, lay.r0 + i), t);
    sc_mont(t, ynr, ar);
    sc_add(t, t, zwl);
    sc_store(ACP_PTR(blk, lay, p, lay.r1 + i), t);
    sc_mont(t, ynr, srv);
    sc_store(ACP_PTR(blk, lay, p, lay.r3 + i), t);
}

// block per (proof, k): dots[k] = <u_k, v_k> over n (k < 10) - the nine products of
// VecPoly3::special_inner_product (poly.rs:39-55; l2 = a_O, l3 = s_l) and sigma = <l_in, z*W_L> (:291).
// second stage (k = 10, 11): t_hat = <l, r> (n) and <z*W_V, gamma> (m) for blinding_values (:444,452).
__global__ void __launch_bounds__(128) k_acp_dots(acp_layout lay, uint32_t first, uint32_t *__restrict__ blk) {
    __shared__ __align__(16) uint32_t sh[32 * 8];
    const uint32_t k = first + blockIdx.x, p = blockIdx.y;
    uint32_t ua, vb, len = lay.n;
    switch (k) {
        case 0: ua = lay.l1; vb = lay.r0; break;
        case 1: ua = lay.l1; vb = lay.r1; break;
        case 2: ua = lay.aO; vb = lay.r0; break;
        case 3: ua = lay.aO; vb = lay.r1; break;
        case 4: ua = lay.sl; vb = lay.r0; break;
        case 5: ua = lay.l1; vb = lay.r3; break;
        case 6: ua = lay.sl; vb = lay.r1; break;
        case 7: ua = lay.aO; vb = lay.r3; break;
        case 8: ua = lay.sl; vb = lay.r3; break;
        case 9: ua = lay.lin; vb = lay.zWL; break;
        case 10: ua = lay.l; vb = lay.r; len = lay.np; break;
        default: ua = lay.zWV; vb = lay.gamma; len = lay.m; break;
    }
    sc acc, tot, r2;
    dot_partial(acc, ACP_PTR(blk, lay, p, ua), 1, ACP_PTR(blk, lay, p, vb), 1, len);
    block_sum_sc(tot, acc, sh);
    if (threadIdx.x == 0) {
        sc_const(r2, SC_R2);
        sc_mont(tot, tot, r2);
        sc_store(ACP_PTR(blk, lay, p, lay.dots + k), tot);
    }
}

// The same dot products for large batches: block per proof, one WARP per dot product (blockDim = 32 x count, dot
// first + warp): one barrier, a proof's vectors are read by the warps of one block (L1).  The
// block-per-dot form above launches 10 x B blocks of one multiplication per thread - at B = 4096 its time is block
// dispatch, not arithmetic (261 us for 4.3 M multiplications) - and stays for small batches, where a single proof's
// n = 8192 needs the blocks.
__global__ void __launch_bounds__(320, 3) k_acp_dots_warp(acp_layout lay, uint32_t first, uint32_t *__restrict__ blk) {
    const uint32_t k = first + (threadIdx.x >> 5), p = blockIdx.x, lane = threadIdx.x & 31;
    uint32_t ua, vb, len = lay.n;
    switch (k) {
        case 0: ua = lay.l1; vb = lay.r0; break;
        case 1: ua = lay.l1; vb = lay.r1; break;
        case 2: ua = lay.aO; vb = lay.r0; break;
        case 3: ua = lay.aO; vb = lay.r1; break;
        case 4: ua = lay.sl; vb = lay.r0; break;
        case 5: ua = lay.l1; vb = lay.r3; break;
        case 6: ua = lay.sl; vb = lay.r1; break;
        case 7: ua = lay.aO; vb = lay.r3; break;
        case 8: ua = lay.sl; vb = lay.r3; break;
        case 9: ua = lay.lin; vb = lay.zWL; break;
        case 10: ua = lay.l; vb = lay.r; len = lay.np; break;
        default: ua = lay.zWV; vb = lay.gamma; len = lay.m; break;
    }
    const uint32_t *a = ACP_PTR(blk, lay, p, ua), *b = ACP_PTR(blk, lay, p, vb);
    // a lane's products are summed as 512-bit integers and reduced once (sc_mont_reduce: up to SC_MAC_MAX at a time), not one
    // Montgomery reduction per product: 64 instead of 132 wide multiplies per element
    sc acc, x, y, pr, tot;
    sc_set0(acc);
    uint32_t t[16], cnt = 0;
#pragma unroll
    for (int j = 0; j < 16; j++) t[j] = 0;
    for (uint32_t i = lane; i < len; i += 32) {
        sc_load(x, a + 8 * (size_t)i);
        sc_load(y, b + 8 * (size_t)i);
        sc_mac(t, x, y);
        if (++cnt == SC_MAC_MAX) {
            sc_mont_reduce(pr, t);
            sc_add(acc, acc, pr);
#pragma unroll
            for (int j = 0; j < 16; j++) t[j] = 0;
            cnt = 0;
        }
    }
    sc_mont_reduce(pr, t);
    sc_add(acc, acc, pr);
    // the warps leave their integer sums in shared memory; the reductions mod l and out of Montgomery form (three
    // multiplications each) then run side by side in the first lanes of warp 0 instead of once per warp
    __shared__ uint32_t sums[10 * 9];
    uint32_t s9[9];
    warp_sum9(s9, acc);
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 9; i++) sums[9 * (threadIdx.x >> 5) + i] = s9[i];
    }
    __syncthreads();
    if (threadIdx.x < (blockDim.x >> 5)) {
#pragma unroll
        for (int i = 0; i < 9; i++) s9[i] = sums[9 * threadIdx.x + i];
        sc r2;
        sc_from9(tot, s9);
        sc_const(r2, SC_R2);
        sc_mont(tot, tot, r2);
        sc_store(ACP_PTR(blk, lay, p, lay.dots + first + threadIdx.x), tot);
    }
}
// host side: the form by batch size
static inline void acp_dots_launch(const acp_layout &lay, uint32_t first, uint32_t count, uint32_t B, uint32_t *blk, cudaStream_t s) {
    if (B >= 256 && count <= 10) k_acp_dots_warp<<<B, 32 * count, 0, s>>>(lay, first, blk);
    else k_acp_dots<<<dim3(count, B), 128, 0, s>>>(lay, first, blk);
}

// thread per proof: t1..t6, sigma, and the five values committed in T_1,T_3,T_4,T_5,T_6:
// mode 0 ("reference", circuit_lib.rs:362-406): t(X) evaluated at the integers 1,3,4,5,6;
// mode 1 ("reference-fixed"): the coefficients t_1,t_3,t_4,t_5,t_6.
__global__ void __launch_bounds__(64) k_acp_tcoef(acp_layout lay, uint32_t B, int mode, uint32_t *__restrict__ blk) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    sc d[10], t[6];
    for (int k = 0; k < 10; k++) sc_load(d[k], ACP_PTR(blk, lay, p, lay.dots + k));
    t[0] = d[0];
    sc_add(t[1], d[1], d[2]);
    sc_add(t[2], d[3], d[4]);
    sc_add(t[3], d[5], d[6]);
    t[4] = d[7];
    t[5] = d[8];
    for (int k = 0; k < 6; k++) sc_store(ACP_PTR(blk, lay, p, lay.tc + k), t[k]);
    sc_store(ACP_PTR(blk, lay, p, lay.sigma), d[9]);
    const int deg[5] = {1, 3, 4, 5, 6};
    for (int k = 0; k < 5; k++) {
        sc v;
        if (mode == 0) {  // Poly6::eval(deg)
            sc xx, acc;
            sc_set_u32(xx, (uint32_t)deg[k]);
            acc = t[5];
            for (int j = 4; j >= 0; j--) {
                sc_mul_noinline(acc, xx, acc);
                sc_add(acc, acc, t[j]);
            }
            sc_mul_noinline(v, xx, acc);
        } else {
            v = t[deg[k] - 1];
        }
        sc_store(ACP_PTR(blk, lay, p, lay.tsel + k), v);
    }
}

// thread per (proof, i): l = l(x), r = r(x)  (poly.rs:67-76 with l0 = 0, r2 = 0)
// x R, x^2 R, x^3 R are computed once per block (thread 0, shared memory).  Then l = x l1 + x^2 a_O + x^3 s_l and
// r - r0 = x r1 + x^3 r3 are each a sum of products x^k R * v accumulated as a 512-bit integer and reduced once
// (sc_mac, sc_mont_reduce): 5 products and 2 reductions per element instead of the 6 Montgomery multiplications of
// Horner's rule.
__global__ void __launch_bounds__(128, 10) k_acp_final(acp_layout lay, uint32_t *__restrict__ blk) {
    __shared__ __align__(16) uint32_t sh_x[3 * 8];   // x R | x^2 R | x^3 R
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (threadIdx.x == 0) {
        sc x0, r2, xr, x2r;
        sc_load(x0, ACP_PTR(blk, lay, p, lay.x));
        sc_const(r2, SC_R2);
        sc_mont(xr, x0, r2);
        sc_store(sh_x, xr);
        sc_mont(x2r, xr, xr);
        sc_store(sh_x + 8, x2r);
        sc_mont(x2r, x2r, xr);
        sc_store(sh_x + 16, x2r);
    }
    __syncthreads();
    if (i >= lay.np) return;
    sc x, a, b, c, t;
    if (i >= lay.n) {  // `fixed` mode padding (as dalek pads): l = 0, r = -y^i
        sc_set0(t);
        sc_store(ACP_PTR(blk, lay, p, lay.l + i), t);
        sc_load(a, ACP_PTR(blk, lay, p, lay.yn + i));
        sc_neg(t, a);
        sc_store(ACP_PTR(blk, lay, p, lay.r + i), t);
        return;
    }
    sc x2, x3;
    sc_load(x, sh_x);
    sc_load(x2, sh_x + 8);
    sc_load(x3, sh_x + 16);
    uint32_t w[16];
#pragma unroll
    for (int j = 0; j < 16; j++) w[j] = 0;
    sc_load(a, ACP_PTR(blk, lay, p, lay.l1 + i));
    sc_load(b, ACP_PTR(blk, lay, p, lay.aO + i));
    sc_load(c, ACP_PTR(blk, lay, p, lay.sl + i));
    sc_mac(w, x, a);
    sc_mac(w, x2, b);
    sc_mac(w, x3, c);
    sc_mont_reduce(t, w);
    sc_store(ACP_PTR(blk, lay, p, lay.l + i), t);
#pragma unroll
    for (int j = 0; j < 16; j++) w[j] = 0;
    sc_load(a, ACP_PTR(blk, lay, p, lay.r0 + i));
    sc_load(b, ACP_PTR(blk, lay, p, lay.r1 + i));
    sc_load(c, ACP_PTR(blk, lay, p, lay.r3 + i));
    sc_mac(w, x, b);
    sc_mac(w, x3, c);
    sc_mont_reduce(t, w);
    sc_add(t, t, a);
    sc_store(ACP_PTR(blk, lay, p, lay.r + i), t);
}

// thread per proof: t_hat, tau_x, mu (circuit_lib.rs:444-462).  mode 0 adds the x^2<z_q, W_V gamma> term
// five times like the reference (:452-456), mode 1 once.
__global__ void __launch_bounds__(64) k_acp_final2(acp_layout lay, uint32_t B, int mode, uint32_t *__restrict__ blk) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    sc x, xp[7], t, acc, wvg, v;
    sc_load(x, ACP_PTR(blk, lay, p, lay.x));
    sc_set_u32(xp[0], 1);
    for (int k = 1; k <= 6; k++) sc_mul_noinline(xp[k], xp[k - 1], x);
    sc_load(v, ACP_PTR(blk, lay, p, lay.dots + 10));
    sc_store(ACP_PTR(blk, lay, p, lay.that), v);
    sc_load(wvg, ACP_PTR(blk, lay, p, lay.dots + 11));
    sc_mul_noinline(wvg, wvg, xp[2]);
    const int deg[5] = {1, 3, 4, 5, 6};
    sc_set0(acc);
    for (int k = 0; k < 5; k++) {
        sc_load(v, ACP_PTR(blk, lay, p, lay.tau + k));
        sc_mul_noinline(t, v, xp[deg[k]]);
        sc_add(acc, acc, t);
        if (mode == 0) sc_add(acc, acc, wvg);
    }
    if (mode != 0) sc_add(acc, acc, wvg);
    sc_store(ACP_PTR(blk, lay, p, lay.taux), acc);
    sc_set0(acc);
    for (int k = 0; k < 3; k++) {  // mu = alpha x + beta x^2 + ro x^3 (alpha, beta, ro contiguous)
        sc_load(v, ACP_PTR(blk, lay, p, lay.alpha + k));
        sc_mul_noinline(t, v, xp[k + 1]);
        sc_add(acc, acc, t);
    }
    sc_store(ACP_PTR(blk, lay, p, lay.mu), acc);
}

// ---- proof (de)serialisation: A_I,A_O,S,T1,T3,T4,T5,T6 | tau_x, mu, t | l[n] | r[n] ------------------
__global__ void k_acp_pack(acp_layout lay, uint32_t B, const uint8_t *__restrict__ pts8 /* B x 8 x 32 */,
                           const uint32_t *__restrict__ blk, uint8_t *__restrict__ out, uint32_t proof_len) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;  // i: 32-byte word of the proof
    const uint32_t words = proof_len / 32;
    if (i >= words) return;
    uint4 lo, hi;
    if (i < 8) {
        const uint4 *s = reinterpret_cast<const uint4 *>(pts8 + 32 * ((size_t)p * 8 + i));
        lo = s[0]; hi = s[1];
    } else {
        uint32_t off = i == 8 ? lay.taux : i == 9 ? lay.mu : i == 10 ? lay.that
                     : i < 11 + lay.n ? lay.l + (i - 11) : lay.r + (i - 11 - lay.n);
        const uint4 *s = reinterpret_cast<const uint4 *>(ACP_PTR(blk, lay, p, off));
        lo = s[0]; hi = s[1];
    }
    uint4 *d = reinterpret_cast<uint4 *>(out + (size_t)p * proof_len + 32 * (size_t)i);
    d[0] = lo; d[1] = hi;
}
// proofs -> scalars into the proof block (reduced mod l: a non-canonical scalar is taken mod l, as
// dalek's arithmetic would) and the 8 compressed points into pts8
__global__ void k_acp_unpack(acp_layout lay, uint32_t B, const uint8_t *__restrict__ proofs, uint32_t proof_len,
                             uint32_t *__restrict__ blk, uint8_t *__restrict__ pts8) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    const uint32_t words = proof_len / 32;
    if (i >= words) return;
    const uint4 *s = reinterpret_cast<const uint4 *>(proofs + (size_t)p * proof_len + 32 * (size_t)i);
    uint4 lo = s[0], hi = s[1];
    if (i < 8) {
        uint4 *d = reinterpret_cast<uint4 *>(pts8 + 32 * ((size_t)p * 8 + i));
        d[0] = lo; d[1] = hi;
        return;
    }
    uint32_t off = i == 8 ? lay.taux : i == 9 ? lay.mu : i == 10 ? lay.that
                 : i < 11 + lay.n ? lay.l + (i - 11) : lay.r + (i - 11 - lay.n);
    sc v;
    v.v[0] = lo.x; v.v[1] = lo.y; v.v[2] = lo.z; v.v[3] = lo.w; v.v[4] = hi.x; v.v[5] = hi.y; v.v[6] = hi.z; v.v[7] = hi.w;
    sc_reduce256(v, v);
    sc_store(ACP_PTR(blk, lay, p, off), v);
}

// ---- verifier ------------------------------------------------------------------------------------------
// Scalars of the fused check (SURVEY D.1), w = per-proof verifier weight (w = 0 in "reference" mode,
// where only checks 1 and 2 are live: circuit_lib.rs:518,541,577-582):
//   g: t - x^2(<z_q,c> + sigma)        h: tau_x - w mu
//   G_i: w (x l_in_i - l_i)            H_i: w y_n_inv_i (x zWL_i + zWO_i - y_n_i - r_i)
//   V_j: -x^2 zWV_j     T_1,T_3..T_6: -x, -x^3 .. -x^6     A_I, A_O, S: w x, w x^2, w x^3
// accept <=> t == <l, r>  and  the MSM over these scalars is the identity.
// Per-proof factors in Montgomery form, computed once per block by two threads (shared memory): x R, x^2 R, w R, w R^2;
// the per-element products then cost 5 Montgomery multiplications per generator pair instead of the 10 of five sc_mul,
// 1 instead of 4 per commitment.
__global__ void __launch_bounds__(128) k_acp_vscal(acp_layout lay, uint32_t *__restrict__ blk) {
    __shared__ __align__(16) uint32_t sh_c[4 * 8];   // x R | x^2 R | w R | w R^2
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    const uint32_t tot = lay.n + lay.m + 1;
    if (threadIdx.x < 2) {
        sc a, r2, b;
        sc_const(r2, SC_R2);
        sc_load(a, ACP_PTR(blk, lay, p, threadIdx.x == 0 ? lay.x : lay.w));
        sc_mont(a, a, r2);                                  // x R   | w R
        sc_store(sh_c + 16 * threadIdx.x, a);
        if (threadIdx.x == 0) sc_mont(b, a, a);             // x^2 R
        else sc_mont(b, a, r2);                             // w R^2
        sc_store(sh_c + 16 * threadIdx.x + 8, b);
    }
    __syncthreads();
    if (i >= tot) return;
    sc x, w, t, u, v;
    if (i < lay.n) {
        sc xr, wr, wr2, lin, l, yi, zwl, zwo, yn, r;
        sc_load(xr, sh_c);
        sc_load(wr, sh_c + 16);
        sc_load(wr2, sh_c + 24);
        sc_load(lin, ACP_PTR(blk, lay, p, lay.lin + i));
        sc_load(l, ACP_PTR(blk, lay, p, lay.l + i));
        sc_mont(t, xr, lin);                                // x lin
        sc_sub(t, t, l);
        sc_mont(t, wr, t);                                  // w (x lin - l)
        sc_store(ACP_PTR(blk, lay, p, lay.vG + i), t);
        sc_load(yi, ACP_PTR(blk, lay, p, lay.yninv + i));
        sc_load(zwl, ACP_PTR(blk, lay, p, lay.zWL + i));
        sc_load(zwo, ACP_PTR(blk, lay, p, lay.zWO + i));
        sc_load(yn, ACP_PTR(blk, lay, p, lay.yn + i));
        sc_load(r, ACP_PTR(blk, lay, p, lay.r + i));
        sc_mont(t, xr, zwl);
        sc_add(t, t, zwo);
        sc_sub(t, t, yn);
        sc_sub(t, t, r);
        sc_mont(u, wr2, yi);                                // w y^-i R
        sc_mont(t, u, t);                                   // w y^-i (x zWL + zWO - y^i - r)
        sc_store(ACP_PTR(blk, lay, p, lay.vH + i), t);
    } else if (i < lay.n + lay.m) {
        const uint32_t j = i - lay.n;
        sc x2r;
        sc_load(x2r, sh_c + 8);
        sc_load(u, ACP_PTR(blk, lay, p, lay.zWV + j));
        sc_mont(t, x2r, u);                                 // x^2 zWV_j
        sc_neg(t, t);
        sc_store(ACP_PTR(blk, lay, p, lay.vd + j), t);
    } else {
        sc_load(x, ACP_PTR(blk, lay, p, lay.x));
        sc_load(w, ACP_PTR(blk, lay, p, lay.w));
        sc xp[7];
        sc_set_u32(xp[0], 1);
        for (int k = 1; k <= 6; k++) sc_mul_noinline(xp[k], xp[k - 1], x);
        // g
        sc_load(u, ACP_PTR(blk, lay, p, lay.zc));
        sc_load(v, ACP_PTR(blk, lay, p, lay.sigma));
        sc_add(u, u, v);
        sc_mul_noinline(u, u, xp[2]);
        sc_load(v, ACP_PTR(blk, lay, p, lay.that));
        sc_sub(t, v, u);
        sc_store(ACP_PTR(blk, lay, p, lay.vg), t);
        // h
        sc_load(u, ACP_PTR(blk, lay, p, lay.mu));
        sc_mul_noinline(u, u, w);
        sc_load(v, ACP_PTR(blk, lay, p, lay.taux));
        sc_sub(t, v, u);
        sc_store(ACP_PTR(blk, lay, p, lay.vh), t);
        const int deg[5] = {1, 3, 4, 5, 6};
        for (int k = 0; k < 5; k++) {
            sc_neg(t, xp[deg[k]]);
            sc_store(ACP_PTR(blk, lay, p, lay.vd + lay.m + k), t);
        }
        for (int k = 0; k < 3; k++) {
            sc_mul_noinline(t, w, xp[k + 1]);
            sc_store(ACP_PTR(blk, lay, p, lay.vd + lay.m + 5 + k), t);
        }
    }
}

// thread per point: compressed -> affine Niels; invalid encodings flag the proof (dalek: decompress() is
// None; the reference unwraps and panics, circuit_lib.rs:532 - here the proof is rejected).
__global__ void __launch_bounds__(128) k_acp_decompress(const uint8_t *__restrict__ V /* B x m x 32 */,
                                                        const uint8_t *__restrict__ pts8 /* B x 8 x 32 */, uint32_t m,
                                                        uint32_t B, uint32_t pitch /* points per proof in dyn */,
                                                        uint32_t *__restrict__ dyn /* B x pitch x 24 */,
                                                        uint32_t *__restrict__ bad /* B */) {
    const uint32_t per = m + 8;
    uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= B * per) return;
    const uint32_t p = id / per, k = id - p * per;
    const uint8_t *src = k < m ? V + 32 * ((size_t)p * m + k) : pts8 + 32 * ((size_t)p * 8 + (k < m + 5 ? 3 + (k - m) : k - m - 5));
    fe x, y;
    bool ok = ge_decompress(x, y, src);
    if (!ok) {
        atomicOr(&bad[p], 1u);
        fe_set0(x);
        fe_set1(y);
    }
    ge_niels q;
    ge_affine_to_niels(q, x, y);
    ge_niels_store(dyn + 24 * ((size_t)p * pitch + k), q);
}

// Dynamic-point MSM, phase 1.  Block per proof, one thread per 4-bit signed window (64 windows):
// each thread walks the proof's m+8 points and adds them into its 8 buckets (shared memory), then
// folds the buckets with the running-sum trick into the window sum.
#define DYN_C 4
#define DYN_W 64
FE_INLINE void dyn_bucket_store(uint4 *bk4, uint32_t b, uint32_t w, const ge_ext &a) {
    const fe *f[4] = {&a.X, &a.Y, &a.Z, &a.T};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        bk4[((b * 8 + 2 * k) * DYN_W) + w] = make_uint4(f[k]->v[0], f[k]->v[1], f[k]->v[2], f[k]->v[3]);
        bk4[((b * 8 + 2 * k + 1) * DYN_W) + w] = make_uint4(f[k]->v[4], f[k]->v[5], f[k]->v[6], f[k]->v[7]);
    }
}
FE_INLINE void dyn_bucket_load(ge_ext &a, const uint4 *bk4, uint32_t b, uint32_t w) {
    fe *f[4] = {&a.X, &a.Y, &a.Z, &a.T};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        uint4 lo = bk4[((b * 8 + 2 * k) * DYN_W) + w], hi = bk4[((b * 8 + 2 * k + 1) * DYN_W) + w];
        f[k]->v[0] = lo.x; f[k]->v[1] = lo.y; f[k]->v[2] = lo.z; f[k]->v[3] = lo.w;
        f[k]->v[4] = hi.x; f[k]->v[5] = hi.y; f[k]->v[6] = hi.z; f[k]->v[7] = hi.w;
    }
}
__global__ void __launch_bounds__(DYN_W) k_dyn_window_sums(const uint32_t *__restrict__ blk, acp_layout lay,
                                                           const uint32_t *__restrict__ dyn, uint32_t per,
                                                           uint32_t *__restrict__ wsum /* B x 64 x 32 */) {
    // 8 buckets per thread in local memory (per-thread interleaved, L1-resident): no shared-memory
    // occupancy limit, 128 B load + store per mixed add
    ge_ext bkt[8];
    const uint32_t p = blockIdx.x, w = threadIdx.x;
    for (int b = 0; b < 8; b++) ge_identity(bkt[b]);
    const uint32_t *scal = ACP_PTR(blk, lay, p, lay.vd);
    const uint32_t *pts = dyn + 24 * (size_t)p * per;
    // digit w of s' = s + 0x0888...8 (carry-free signed recoding, top window unsigned)
#pragma unroll 1
    for (uint32_t k = 0; k < per; k++) {
        uint32_t s[9];
        unsigned long long carry = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            uint32_t kl = (i == 7) ? 0x08888888u : 0x88888888u;
            carry += (unsigned long long)scal[8 * (size_t)k + i] + kl;
            s[i] = (uint32_t)carry;
            carry >>= 32;
        }
        s[8] = (uint32_t)carry;
        uint32_t u = (s[w >> 3] >> ((w & 7) * 4)) & 15u;
        if (w == DYN_W - 1) u += s[8] << 4;  // cannot happen for s < 2^255 (kept for safety)
        int d = (w == DYN_W - 1) ? (int)u : (int)u - 8;
        if (d == 0) continue;
        uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
        ge_niels q;
        ge_niels_load(q, pts + 24 * (size_t)k);
        ge_ext a = bkt[mag - 1];
        ge_madd(a, a, q, d < 0);
        bkt[mag - 1] = a;
    }
    ge_ext run, acc, t;
    run = bkt[7];
    acc = run;
#pragma unroll 1
    for (int b = 6; b >= 0; b--) {
        t = bkt[b];
        ge_add(run, run, t);
        ge_add(acc, acc, run);
    }
    ge_store(wsum + 32 * ((size_t)p * DYN_W + w), acc);
}

// phase 2.  Thread per proof: Horner over the 64 window sums (4 doublings each), add the fixed-base
// part, test for the identity and fold in the scalar check t == <l, r>.
FE_INLINE void dyn_horner(ge_ext &acc, const uint32_t *__restrict__ wsum, uint32_t p) {
    ge_ext t;
    ge_load(acc, wsum + 32 * ((size_t)p * DYN_W + DYN_W - 1));
#pragma unroll 1
    for (int w = DYN_W - 2; w >= 0; w--) {
#pragma unroll 1
        for (int i = 0; i < DYN_C; i++) ge_double(acc, acc);
        ge_load(t, wsum + 32 * ((size_t)p * DYN_W + w));
        ge_add(acc, acc, t);
    }
}
__global__ void __launch_bounds__(64) k_dyn_horner_accept(acp_layout lay, uint32_t B, const uint32_t *__restrict__ blk,
                                                          const uint32_t *__restrict__ wsum,
                                                          const uint32_t *__restrict__ stat_ext /* B x 32 */,
                                                          const uint32_t *__restrict__ bad, int check_t,
                                                          uint8_t *__restrict__ accept) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    ge_ext acc, t;
    dyn_horner(acc, wsum, p);
    ge_load(t, stat_ext + 32 * (size_t)p);
    ge_add(acc, acc, t);
    bool ident = fe_is_zero(acc.X) || fe_is_zero(acc.Y);  // the Ristretto identity coset
    sc that, lr;
    sc_load(that, ACP_PTR(blk, lay, p, lay.that));
    sc_load(lr, ACP_PTR(blk, lay, p, lay.dots + 10));
    accept[p] = (ident && (!check_t || sc_eq(that, lr)) && bad[p] == 0) ? 1 : 0;
}

// ---- batch verification by random linear combination ---------------------------------------------------
// Every proof's check is "one MSM is the identity" (k_acp_vscal / k_acp_vscal_fixed give its scalars).  With
// independent verifier weights rho_p, sum_p rho_p * MSM_p is ONE Pippenger MSM over the batch's
// B x per decompressed points plus the shared generators (whose scalars add up across proofs): c = 16
// windows instead of per-proof 4-bit windows, i.e. 16 mixed adds per point instead of ~64.  It is the
// identity for an all-valid batch and, for any invalid proof, a non-identity except with probability
// ~2^-252; on failure the caller falls back to the per-proof kernels, so per-proof decisions are unchanged.
// rho_p comes from the proof's own transcript rekeyed with the verifier seed (k_tr_weights, transcript_kernels.cuh);
// proofs that already failed a cheap check (bad encoding, t != <l, r>) get rho_p = 0 and are rejected here.
__global__ void k_rlc_weights(acp_layout lay, uint32_t B, int check_t, const uint32_t *__restrict__ bad,
                              uint32_t *__restrict__ blk) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    sc r;
    sc_load(r, ACP_PTR(blk, lay, p, lay.rho0));
    bool ok = bad[p] == 0;
    if (check_t) {
        sc that, lr;
        sc_load(that, ACP_PTR(blk, lay, p, lay.that));
        sc_load(lr, ACP_PTR(blk, lay, p, lay.dots + 10));
        ok = ok && sc_eq(that, lr);
    }
    if (!ok) sc_set0(r);
    sc_store(ACP_PTR(blk, lay, p, lay.rho), r);
}
// out[p * per + k] = rho_p * vd_p[k]; rho_p R is computed once per block (shared memory), so that each product is one
// Montgomery multiplication instead of the two of sc_mul
__global__ void __launch_bounds__(128) k_rlc_dyn_scalars(acp_layout lay, uint32_t per, uint32_t B, uint32_t rho_off,
                                                         const uint32_t *__restrict__ blk, uint32_t *__restrict__ out) {
    __shared__ __align__(16) uint32_t sh_rho[8];
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    sc rho, v;
    if (threadIdx.x == 0) {
        sc_load(rho, ACP_PTR(blk, lay, p, rho_off));
        sc_to_mont(rho, rho);
        sc_store(sh_rho, rho);
    }
    __syncthreads();
    if (k >= per) return;
    sc_load(rho, sh_rho);
    sc_load(v, ACP_PTR(blk, lay, p, lay.vd + k));
    sc_mont(v, v, rho);
    sc_store(out + 8 * ((size_t)p * per + k), v);
}
// Where the shared generators' scalars sit in a proof block: generator i of segment k (i < cnt[k]) at off[k] + i, the
// segments in the order of the generators' points (the shuffle: one segment g, h, G[], H[] at lay.vg; the stand-alone
// inner-product batch: vG, vH, and the Q coefficient at lay.cl).
#define RLC_MAX_SEGS 3
struct rlc_segs {
    uint32_t off[RLC_MAX_SEGS], cnt[RLC_MAX_SEGS];
};
// out[i] = sum_p rho_p * vstat_p[i] for the shared generators of `sg`; block per generator
__global__ void __launch_bounds__(128) k_rlc_stat_scalars(acp_layout lay, rlc_segs sg, uint32_t B, uint32_t rho_off,
                                                          const uint32_t *__restrict__ blk, uint32_t *__restrict__ out) {
    __shared__ __align__(16) uint32_t red[128][8];
    const uint32_t i = blockIdx.x;
    uint32_t k = 0, j = i;
    while (k + 1 < RLC_MAX_SEGS && j >= sg.cnt[k]) j -= sg.cnt[k++];
    const uint32_t src = sg.off[k] + j;
    sc acc, rho, v, rr;
    sc_set0(acc);
    sc_const(rr, SC_R2);
    for (uint32_t p = threadIdx.x; p < B; p += 128) {
        sc_load(rho, ACP_PTR(blk, lay, p, rho_off));
        sc_load(v, ACP_PTR(blk, lay, p, src));
        sc_mont(v, v, rho);      // rho * v / R; the factor R is restored once after the reduction
        sc_add(acc, acc, v);
    }
    sc_store(&red[threadIdx.x][0], acc);
    __syncthreads();
    for (uint32_t d = 64; d >= 1; d >>= 1) {
        if (threadIdx.x < d) {
            sc a, b2;
            sc_load(a, &red[threadIdx.x][0]);
            sc_load(b2, &red[threadIdx.x + d][0]);
            sc_add(a, a, b2);
            sc_store(&red[threadIdx.x][0], a);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        sc_load(acc, &red[0][0]);
        sc_mont(acc, acc, rr);
        sc_store(out + 8 * (size_t)i, acc);
    }
}
// enc32 = compressed result of the batch MSM: all-zero bytes <=> identity.  accept[p] = identity and rho_p != 0;
// flag[0] = 1 when the combination is not the identity (caller falls back to per-proof verification).
__global__ void k_rlc_accept(const uint8_t *__restrict__ enc32, acp_layout lay, uint32_t B, uint32_t rho_off,
                             const uint32_t *__restrict__ blk, uint8_t *__restrict__ accept, uint32_t *__restrict__ flag) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    uint32_t o = 0;
    for (int i = 0; i < 32; i++) o |= enc32[i];
    sc rho;
    sc_load(rho, ACP_PTR(blk, lay, p, rho_off));
    accept[p] = (o == 0 && !sc_is_zero(rho)) ? 1 : 0;
    if (p == 0) flag[0] = o == 0 ? 0u : 1u;
}
