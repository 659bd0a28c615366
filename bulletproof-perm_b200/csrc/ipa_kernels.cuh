// ipa_kernels.cuh - `fixed` protocol mode: standard powers and the inner-product argument, batched.
//
// SURVEY section 8 row a16 / north_star item (2): bulletproofs 4.0.0 `InnerProductProof::create`
// (inner_product_proof.rs; Cargo.lock:47-50, un-vendored) - absent from the reference, which sends l and r
// in the clear (circuit_lib.rs:464-468).  The CPU restatements the tests compare with live in the test tree.
//
// Formulation (SURVEY D.3, "fold the scalars, not the points"): the folded generators of round j are
//   G^(j)[i] = sum_t s_t G[i + t n_j],   H^(j)[i] = sum_t s_t^-1 y^-(i + t n_j) H[i + t n_j],
//   n_j = n' / 2^j,  s_t = prod_{k<j} u_k^(+-1)  (+ iff bit j-1-k of t is set),
// so L_j and R_j are MSMs over the ORIGINAL generators with scalars a[i^h] s_t (G side) and
// b[i^h] s_t^-1 y^-g (H side), h = n_j / 2: they run through the same fixed-base tables as the
// commitments (k_fb_msm) and no generator is ever folded.  a and b fold in place in the proof block.
#pragma once
#include <cooperative_groups.h>

#include "acproof_kernels.cuh"

#define IPA_MAX_LG 20

// ---- standard powers ---------------------------------------------------------------------------------
// Thread per proof: squarings y^(2^k), (y^-1)^(2^k), z^(2^k) (Montgomery form) into the proof block.
__global__ void __launch_bounds__(64) k_pow_table(acp_layout lay, uint32_t B, uint32_t *__restrict__ blk) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    sc y, z, yi;
    sc_load(y, ACP_PTR(blk, lay, p, lay.y));
    sc_load(z, ACP_PTR(blk, lay, p, lay.z));
    sc_invert(yi, y);
    sc_to_mont(y, y);
    sc_to_mont(yi, yi);
    sc_to_mont(z, z);
#pragma unroll 1
    for (uint32_t k = 0; k < IPA_MAX_LG; k++) {
        sc_store(ACP_PTR(blk, lay, p, lay.ptab + k), y);
        sc_store(ACP_PTR(blk, lay, p, lay.ptab + IPA_MAX_LG + k), yi);
        sc_store(ACP_PTR(blk, lay, p, lay.ptab + 2 * IPA_MAX_LG + k), z);
        sc_mont_noinline(y, y, y);
        sc_mont_noinline(yi, yi, yi);
        sc_mont_noinline(z, z, z);
    }
}
// Thread per (proof, j): y_n[i] = y^i, y_n_inv[i] = y^-i (i < n'), z_q[q] = z^(q+1) (q < Q) as products of the
// squarings selected by the exponent's bits (<= lg multiplications each, no serial chain over n).
__global__ void __launch_bounds__(128) k_pow_fill(acp_layout lay, uint32_t *__restrict__ blk) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    const uint32_t total = 2 * lay.np + lay.Q;
    if (j >= total) return;
    uint32_t which, e, dst;
    if (j < lay.np) { which = 0; e = j; dst = lay.yn + j; }
    else if (j < 2 * lay.np) { which = 1; e = j - lay.np; dst = lay.yninv + e; }
    else { which = 2; e = j - 2 * lay.np + 1; dst = lay.zq + (e - 1); }
    sc acc, t;
    sc_const(acc, SC_R);
    const uint32_t *tab = ACP_PTR(blk, lay, p, lay.ptab + which * IPA_MAX_LG);
#pragma unroll 1
    for (uint32_t k = 0; e; k++, e >>= 1)
        if (e & 1u) {
            sc_load(t, tab + 8 * (size_t)k);
            sc_mont_noinline(acc, acc, t);
        }
    sc_from_mont(acc, acc);
    sc_store(ACP_PTR(blk, lay, p, dst), acc);
}

// ---- prover rounds -----------------------------------------------------------------------------------
// A round is: [MSM over the original generators -> L_j, R_j] -> compress -> k_ipa_challenge (transcript_kernels.cuh: one
// warp per proof appends L_j, R_j, draws u_j and inverts it) -> k_ipa_round (below: everything that is parallel over the
// vector - fold a and b, extend the table of the s_t, the next round's two inner products and its MSM scalars).
//
// s table (lay.stab, 2 x n' scalars per proof, Montgomery form, double buffered by the parity of the rounds done):
// after r rounds buffer r & 1 holds s_t = prod_{k<r} (bit (r-1-k) of t ? u_k : u_k^-1) for t < 2^r, built by doubling,
// s'_{2t+b} = s_t * (b ? u_r : u_r^-1): one multiplication per entry and round instead of r per generator and round.
// The inverse is the complemented index: s_t^-1 = s_{2^r - 1 - t}.
#define IPA_ROUND_THREADS 512
SC_INLINE uint32_t *ipa_stab(uint32_t *blk, const acp_layout &lay, uint32_t p, uint32_t rounds_done) {
    return ACP_PTR(blk, lay, p, lay.stab + (rounds_done & 1u) * lay.np);
}
// One thread-block CLUSTER per proof (1 CTA up to n' = 1024, then n' / 1024 CTAs up to 8: a single 4096-card proof has
// n' = 8192 and would otherwise run each round on one SM).  round = index of the challenge just drawn (u[round],
// uinv[round] in Montgomery form), -1 before the first round (w at lay.wq drawn).  Leaves a, b folded (lay.l, lay.r),
// cl[0..1] = w <a_lo, b_hi>, w <a_hi, b_lo> and vG, vH = the next round's MSM scalars; after the last round only the
// fold happens (a, b are l[0], r[0]).  The two barriers are cluster barriers (release/acquire at cluster scope: the
// folded vectors and the table written by one CTA are read by the others); the CTAs' partial inner products meet in
// rank 0 through distributed shared memory.
// GF: the stand-alone inner-product batch (bpp_ipa_batch_*), whose G generators carry per-proof factors (dalek's G_factors,
// held at lay.yn there): the G-side MSM scalars are multiplied by them as the H side's are by lay.yninv.  k_ipa_round (the
// `fixed` mode, G_factors = 1) is the GF = false instance.
template <bool GF>
__device__ __forceinline__ void ipa_round_body(const acp_layout &lay, int round, uint32_t *__restrict__ blk) {
    namespace cg = cooperative_groups;
    __shared__ __align__(16) uint32_t sh[32 * 8];
    __shared__ __align__(16) uint32_t part[2 * 8];     // this CTA's share of the two inner products (Montgomery sums)
    cg::cluster_group cluster = cg::this_cluster();
    const uint32_t C = cluster.num_blocks(), rank = cluster.block_rank();
    const uint32_t p = blockIdx.x / C, tid = rank * blockDim.x + threadIdx.x, nt = C * blockDim.x;
    const uint32_t done = (uint32_t)(round + 1);
    uint32_t *st_new = ipa_stab(blk, lay, p, done);
    if (round < 0) {
        if (tid == 0) {
            sc one;
            sc_const(one, SC_R);
            sc_store(st_new, one);
        }
    } else {
        const uint32_t h = lay.np >> done;
        sc u, ui, lo, hi, t1, t2;
        sc_load(u, ACP_PTR(blk, lay, p, lay.u + round));
        sc_load(ui, ACP_PTR(blk, lay, p, lay.uinv + round));
        for (uint32_t i = tid; i < h; i += nt) {       // a[i] = a[i] u + u^-1 a[h+i],  b[i] = b[i] u^-1 + u b[h+i]
            sc_load(lo, ACP_PTR(blk, lay, p, lay.l + i));
            sc_load(hi, ACP_PTR(blk, lay, p, lay.l + h + i));
            sc_mont(t1, lo, u);
            sc_mont(t2, hi, ui);
            sc_add(t1, t1, t2);
            sc_store(ACP_PTR(blk, lay, p, lay.l + i), t1);
            sc_load(lo, ACP_PTR(blk, lay, p, lay.r + i));
            sc_load(hi, ACP_PTR(blk, lay, p, lay.r + h + i));
            sc_mont(t1, lo, ui);
            sc_mont(t2, hi, u);
            sc_add(t1, t1, t2);
            sc_store(ACP_PTR(blk, lay, p, lay.r + i), t1);
        }
        if (done < lay.lg) {                           // the last round's table is never read
            const uint32_t *st_old = ipa_stab(blk, lay, p, (uint32_t)round);
            for (uint32_t t = tid; t < (1u << done); t += nt) {
                sc_load(lo, st_old + 8 * (size_t)(t >> 1));
                sc_mont(t1, lo, (t & 1u) ? u : ui);
                sc_store(st_new + 8 * (size_t)t, t1);
            }
        }
    }
    if (done >= lay.lg) return;                        // uniform over the cluster
    cluster.sync();                                    // a, b, s table: visible to every CTA of the proof
    const uint32_t nj = lay.np >> done, h = nj >> 1;
    for (uint32_t which = 0; which < 2; which++) {
        const uint32_t *a = ACP_PTR(blk, lay, p, lay.l + (which ? h : 0)), *b = ACP_PTR(blk, lay, p, lay.r + (which ? 0 : h));
        sc acc, tot, x, y, pr;
        sc_set0(acc);
        for (uint32_t i = tid; i < h; i += nt) {
            sc_load(x, a + 8 * (size_t)i);
            sc_load(y, b + 8 * (size_t)i);
            sc_mont(pr, x, y);
            sc_add(acc, acc, pr);
        }
        block_sum_sc(tot, acc, sh);
        if (threadIdx.x == 0) sc_store(part + 8 * which, tot);
    }
    const uint32_t tmask = (1u << done) - 1u;
    for (uint32_t g = tid; g < lay.np; g += nt) {      // the round's MSM scalars over the original generators
        const uint32_t i = g & (nj - 1), t = g >> (lay.lg - done), ip = i ^ h;
        BPP_ASSERT(t <= tmask && ip < nj && done < lay.lg);
        sc s, sinv, a, b, yi, r;
        sc_load(s, st_new + 8 * (size_t)t);
        sc_load(sinv, st_new + 8 * (size_t)(tmask - t));
        sc_load(a, ACP_PTR(blk, lay, p, lay.l + ip));
        sc_load(b, ACP_PTR(blk, lay, p, lay.r + ip));
        sc_load(yi, ACP_PTR(blk, lay, p, lay.yninv + g));
        sc_mont(r, a, s);                              // a * s_t (s in Montgomery form -> standard result)
        if (GF) {
            sc gf;
            sc_load(gf, ACP_PTR(blk, lay, p, lay.yn + g));
            sc_mul(r, r, gf);
        }
        sc_store(ACP_PTR(blk, lay, p, lay.vG + g), r);
        sc_mont(r, b, sinv);
        sc_mul(r, r, yi);
        sc_store(ACP_PTR(blk, lay, p, lay.vH + g), r);
    }
    cluster.sync();                                    // every CTA's partial sums are in its shared memory
    if (rank == 0 && threadIdx.x < 2) {
        const uint32_t which = threadIdx.x;
        sc tot, o, w, r2;
        sc_set0(tot);
        for (uint32_t r = 0; r < C; r++) {
            const uint32_t *remote = cluster.map_shared_rank(part, r);
            sc_load(o, remote + 8 * which);
            sc_add(tot, tot, o);
        }
        sc_load(w, ACP_PTR(blk, lay, p, lay.wq));
        sc_const(r2, SC_R2);
        sc_mont(tot, tot, r2);
        sc_mul(tot, tot, w);
        sc_store(ACP_PTR(blk, lay, p, lay.cl + which), tot);
    }
    cluster.sync();                                    // no CTA leaves while rank 0 reads its shared memory
}
__global__ void __launch_bounds__(IPA_ROUND_THREADS) k_ipa_round(acp_layout lay, int round, uint32_t *__restrict__ blk) {
    ipa_round_body<false>(lay, round, blk);
}
__global__ void __launch_bounds__(IPA_ROUND_THREADS) k_ipa_round_gf(acp_layout lay, int round, uint32_t *__restrict__ blk) {
    ipa_round_body<true>(lay, round, blk);
}
// launch: cluster of `C` CTAs per proof; gf: the k_ipa_round_gf instance
static inline cudaError_t ipa_round_launch(acp_layout lay, int round, uint32_t *blk, uint32_t B, cudaStream_t s, bool gf = false) {
    const uint32_t np = lay.np;
    const unsigned threads = np >= IPA_ROUND_THREADS ? IPA_ROUND_THREADS : (np < 128 ? 128 : np);
    unsigned C = 1;
    while (C < 8 && (size_t)C * 1024 < np) C <<= 1;
    void (*kern)(acp_layout, int, uint32_t *) = gf ? k_ipa_round_gf : k_ipa_round;
    if (C == 1) {
        kern<<<B, threads, 0, s>>>(lay, round, blk);
        return cudaGetLastError();
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(B * C);
    cfg.blockDim = dim3(threads);
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, lay, round, blk);
}
// ---- K7: explicit generator folding (SURVEY 2.3 / D.3; bulletproofs 4.0.0 inner_product_proof.rs create():
// G'_i = u^-1 G_i + u G_{i + n/2}).  NOT on the prover's path - the rounds above fold the scalars and keep the original
// generators, whose window tables exist - but built as an operator so that the two forms can be measured against each
// other per round (tools/ipa_fold_compare.py, profiles/r2_ipa_fold_compare.json) and checked for equality.
// Thread per (fold f, i < half): a two-scalar Straus multiplication with signed 4-bit digits: tables of 1..8 multiples
// of both points (extended coordinates, local memory), then 64 windows of 4 doublings + up to 2 additions:
// 256 doublings + ~134 additions per folded point, against 16 (c = 16) or 32 (c = 8) mixed adds per generator and
// round in the scalar-folding form.
SC_INLINE void ipa_signed_digits4(int8_t d[64], const uint32_t s[8]) {   // s < 2^253: 64 digits in [-8, 8)
    uint32_t carry = 0;
#pragma unroll 1
    for (int i = 0; i < 64; i++) {
        uint32_t v = ((s[i >> 3] >> (4 * (i & 7))) & 15u) + carry;
        carry = v >= 8u;
        d[i] = (int8_t)((int)v - (int)(carry << 4));
    }   // the top nibble of a scalar below 2^253 is at most 1: no carry out
}
__global__ void __launch_bounds__(64) k_ipa_fold_gens(const uint32_t *__restrict__ niels /* n x 24: affine Niels */, uint32_t half,
                                                      const uint32_t *__restrict__ u /* folds x 8 */,
                                                      const uint32_t *__restrict__ uinv, uint32_t folds,
                                                      uint32_t *__restrict__ out_ext /* folds x half x 32 */) {
    const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= folds * half) return;
    const uint32_t f = id / half, i = id - f * half;
    ge_ext tab[2][8];
#pragma unroll 1
    for (int s = 0; s < 2; s++) {
        ge_niels q;
        ge_niels_load(q, niels + 24 * (size_t)(i + s * half));
        ge_identity(tab[s][0]);
        ge_madd(tab[s][0], tab[s][0], q, false);
#pragma unroll 1
        for (int k = 1; k < 8; k++) ge_madd(tab[s][k], tab[s][k - 1], q, false);
    }
    int8_t d_lo[64], d_hi[64];
    uint32_t sc8[8];
#pragma unroll
    for (int k = 0; k < 8; k++) sc8[k] = uinv[8 * (size_t)f + k];
    ipa_signed_digits4(d_lo, sc8);
#pragma unroll
    for (int k = 0; k < 8; k++) sc8[k] = u[8 * (size_t)f + k];
    ipa_signed_digits4(d_hi, sc8);
    ge_ext acc, t;
    ge_identity(acc);
#pragma unroll 1
    for (int w = 63; w >= 0; w--) {
        if (w != 63)
            for (int k = 0; k < 4; k++) ge_double_noinline(acc, acc);
        const int a = d_lo[w], b = d_hi[w];
        if (a) {
            t = tab[0][(a < 0 ? -a : a) - 1];
            if (a < 0) ge_neg(t, t);
            ge_add_noinline(acc, acc, t);
        }
        if (b) {
            t = tab[1][(b < 0 ? -b : b) - 1];
            if (b < 0) ge_neg(t, t);
            ge_add_noinline(acc, acc, t);
        }
    }
    ge_store(out_ext + 32 * (size_t)id, acc);
}

// host-transcript path: thread per proof: u_round^-1; both kept in Montgomery form at u[round], uinv[round]
__global__ void __launch_bounds__(64) k_ipa_uinv(acp_layout lay, uint32_t B, uint32_t round, uint32_t *__restrict__ blk) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    sc u, ui;
    sc_load(u, ACP_PTR(blk, lay, p, lay.u + round));   // standard form (k_acp_put_wide)
    sc_invert(ui, u);
    sc_to_mont(u, u);
    sc_to_mont(ui, ui);
    sc_store(ACP_PTR(blk, lay, p, lay.u + round), u);
    sc_store(ACP_PTR(blk, lay, p, lay.uinv + round), ui);
}
// verifier: the complete table s_i, i < n' (all lg challenges known) into buffer lg & 1 of lay.stab; block per proof
__global__ void __launch_bounds__(IPA_ROUND_THREADS) k_ipa_stable_full(acp_layout lay, uint32_t *__restrict__ blk) {
    const uint32_t p = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    if (tid == 0) {
        sc one;
        sc_const(one, SC_R);
        sc_store(ipa_stab(blk, lay, p, 0), one);
    }
    for (uint32_t r = 0; r < lay.lg; r++) {
        __syncthreads();
        sc u, ui, v, o;
        sc_load(u, ACP_PTR(blk, lay, p, lay.u + r));
        sc_load(ui, ACP_PTR(blk, lay, p, lay.uinv + r));
        const uint32_t *st_old = ipa_stab(blk, lay, p, r);
        uint32_t *st_new = ipa_stab(blk, lay, p, r + 1);
        for (uint32_t t = tid; t < (2u << r); t += nt) {
            sc_load(v, st_old + 8 * (size_t)(t >> 1));
            sc_mont(o, v, (t & 1u) ? u : ui);
            sc_store(st_new + 8 * (size_t)t, o);
        }
    }
}

// ---- proof (de)serialisation, `fixed` mode: 8 points | t_hat, tau_x, mu | (L_j, R_j) x lg | a, b -----------
__global__ void k_acp_pack_fixed(acp_layout lay, const uint8_t *__restrict__ pts8, const uint8_t *__restrict__ lr,
                                 const uint32_t *__restrict__ blk, uint8_t *__restrict__ out, uint32_t proof_len) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    const uint32_t words = proof_len / 32;
    if (i >= words) return;
    const uint4 *s;
    if (i < 8) s = reinterpret_cast<const uint4 *>(pts8 + 32 * ((size_t)p * 8 + i));
    else if (i < 11) s = reinterpret_cast<const uint4 *>(ACP_PTR(blk, lay, p, i == 8 ? lay.that : i == 9 ? lay.taux : lay.mu));
    else if (i < 11 + 2 * lay.lg) s = reinterpret_cast<const uint4 *>(lr + 32 * ((size_t)p * 2 * lay.lg + (i - 11)));
    else s = reinterpret_cast<const uint4 *>(ACP_PTR(blk, lay, p, i == 11 + 2 * lay.lg ? lay.l : lay.r));
    uint4 *d = reinterpret_cast<uint4 *>(out + (size_t)p * proof_len + 32 * (size_t)i);
    d[0] = s[0];
    d[1] = s[1];
}
// scalars are taken mod l (dalek arithmetic on a non-canonical scalar would do the same); the three transcript
// scalars are also written, reduced, to tx3 for the host
__global__ void k_acp_unpack_fixed(acp_layout lay, const uint8_t *__restrict__ proofs, uint32_t proof_len,
                                   uint32_t *__restrict__ blk, uint8_t *__restrict__ pts8, uint8_t *__restrict__ lr,
                                   uint32_t *__restrict__ tx3) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    const uint32_t words = proof_len / 32;
    if (i >= words) return;
    const uint4 *s = reinterpret_cast<const uint4 *>(proofs + (size_t)p * proof_len + 32 * (size_t)i);
    uint4 lo = s[0], hi = s[1];
    if (i < 8 || (i >= 11 && i < 11 + 2 * lay.lg)) {
        uint4 *d = i < 8 ? reinterpret_cast<uint4 *>(pts8 + 32 * ((size_t)p * 8 + i))
                         : reinterpret_cast<uint4 *>(lr + 32 * ((size_t)p * 2 * lay.lg + (i - 11)));
        d[0] = lo;
        d[1] = hi;
        return;
    }
    sc v;
    v.v[0] = lo.x; v.v[1] = lo.y; v.v[2] = lo.z; v.v[3] = lo.w; v.v[4] = hi.x; v.v[5] = hi.y; v.v[6] = hi.z; v.v[7] = hi.w;
    sc_reduce256(v, v);
    uint32_t off = i == 8 ? lay.that : i == 9 ? lay.taux : i == 10 ? lay.mu : i == 11 + 2 * lay.lg ? lay.pa : lay.pb;
    sc_store(ACP_PTR(blk, lay, p, off), v);
    if (i < 11) sc_store(tx3 + 8 * ((size_t)p * 3 + (i - 8)), v);
}

// ---- verifier ------------------------------------------------------------------------------------------------
// the verifier's 4 + lg wide challenges per proof (y, z, x, w, u_0..) -> y, z, x, wq, u[j]
__global__ void k_acp_put_wide_strided(const uint32_t *__restrict__ wide, acp_layout lay, uint32_t nch, uint32_t B,
                                       uint32_t *__restrict__ blk) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * nch) return;
    uint32_t p = i / nch, k = i - p * nch;
    uint32_t w[16];
#pragma unroll
    for (int t = 0; t < 16; t++) w[t] = wide[16 * (size_t)i + t];
    sc r;
    sc_from_wide(r, w);
    const uint32_t off = k == 0 ? lay.y : k == 1 ? lay.z : k == 2 ? lay.x : k == 3 ? lay.wq : lay.u + (k - 4);
    sc_store(ACP_PTR(blk, lay, p, off), r);
}
// thread per proof: u_j^-1 for all rounds with one inversion; u, uinv in Montgomery form; usq, uinvsq standard at
// lay.vd + first + 2 k, + 1 (`fixed` mode: first = m + 8, after the commitments and the eight proof points)
__global__ void __launch_bounds__(64) k_ipa_vprep(acp_layout lay, uint32_t B, uint32_t first, uint32_t *__restrict__ blk) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    uint32_t *u = ACP_PTR(blk, lay, p, lay.u), *ui = ACP_PTR(blk, lay, p, lay.uinv);
    sc acc, v, inv;
    sc_const(acc, SC_R);
    bool zero = false;
#pragma unroll 1
    for (uint32_t k = 0; k < lay.lg; k++) {     // prefix products (Montgomery) in uinv
        sc_store(ui + 8 * (size_t)k, acc);
        sc_load(v, u + 8 * (size_t)k);
        zero = zero || sc_is_zero(v);
        sc_to_mont(v, v);
        sc_store(u + 8 * (size_t)k, v);
        sc_mont_noinline(acc, acc, v);
    }
    sc_from_mont(v, acc);
    sc_invert(inv, v);
    sc_to_mont(inv, inv);
#pragma unroll 1
    for (int k = (int)lay.lg - 1; k >= 0; k--) {
        sc pre, r, e, sq;
        sc_load(pre, ui + 8 * (size_t)k);
        sc_mont_noinline(r, inv, pre);          // u_k^-1 (Montgomery)
        sc_load(e, u + 8 * (size_t)k);
        sc_mont_noinline(inv, inv, e);
        if (zero) sc_set0(r);                   // only if some u_k = 0: dalek's invert(0) = 0
        sc_store(ui + 8 * (size_t)k, r);
        sc_mont_noinline(sq, e, e);
        sc_from_mont(sq, sq);
        sc_store(ACP_PTR(blk, lay, p, lay.vd + first + 2 * k), sq);              // L_k: u_k^2
        sc_mont_noinline(sq, r, r);
        sc_from_mont(sq, sq);
        sc_store(ACP_PTR(blk, lay, p, lay.vd + first + 2 * k + 1), sq);          // R_k: u_k^-2
    }
}
// Scalars of the fused check (SURVEY D.1, `fixed` layout; rho = per-proof verifier weight on check 2):
//   g: rho (t - x^2(<z_q,c> + sigma)) + w (t - a b)          h: rho tau_x - mu
//   G_i: x l_in_i - a s_i                                     H_i: y^-i (x zWL_i + zWO_i - y^i - b s_i^-1)
//   V_j: -rho x^2 zWV_j   T_1,T_3..T_6: -rho x^deg   A_I, A_O, S: x, x^2, x^3   L_k: u_k^2   R_k: u_k^-2
// x R and rho x^2 R are computed once per block (thread 0, shared memory): x * t is then one Montgomery multiplication
// instead of two, -rho x^2 zWV_j one instead of six.
__global__ void __launch_bounds__(128) k_acp_vscal_fixed(acp_layout lay, uint32_t *__restrict__ blk) {
    __shared__ __align__(16) uint32_t sh_c[2 * 8];   // x R | rho x^2 R
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    const uint32_t tot = lay.np + lay.m + 1;
    if (threadIdx.x == 0) {
        sc a, b, r2;
        sc_const(r2, SC_R2);
        sc_load(a, ACP_PTR(blk, lay, p, lay.x));
        sc_mont(a, a, r2);                       // x R
        sc_store(sh_c, a);
        sc_mont(a, a, a);                        // x^2 R
        sc_load(b, ACP_PTR(blk, lay, p, lay.w));
        sc_mont(b, b, r2);                       // rho R
        sc_mont(a, a, b);                        // rho x^2 R
        sc_store(sh_c + 8, a);
    }
    __syncthreads();
    if (i >= tot) return;
    sc x, rho, t, u, v;
    sc_load(x, ACP_PTR(blk, lay, p, lay.x));
    sc_load(rho, ACP_PTR(blk, lay, p, lay.w));
    sc xr;
    sc_load(xr, sh_c);
    if (i < lay.np) {
        sc s, sinv, pa, pb, yi, yn;
        const uint32_t *st = ipa_stab(blk, lay, p, lay.lg);   // k_ipa_stable_full
        sc_load(s, st + 8 * (size_t)i);
        sc_load(sinv, st + 8 * (size_t)(lay.np - 1 - i));
        sc_load(pa, ACP_PTR(blk, lay, p, lay.pa));
        sc_load(pb, ACP_PTR(blk, lay, p, lay.pb));
        sc_load(yi, ACP_PTR(blk, lay, p, lay.yninv + i));
        sc_load(yn, ACP_PTR(blk, lay, p, lay.yn + i));
        sc_mont(u, pa, s);                       // a s_i
        sc_set0(t);
        if (i < lay.n) {
            sc_load(v, ACP_PTR(blk, lay, p, lay.lin + i));
            sc_mont(t, xr, v);                   // x l_in_i
        }
        sc_sub(t, t, u);
        sc_store(ACP_PTR(blk, lay, p, lay.vG + i), t);
        sc_mont(u, pb, sinv);                    // b / s_i
        sc_set0(t);
        if (i < lay.n) {
            sc zwl, zwo;
            sc_load(zwl, ACP_PTR(blk, lay, p, lay.zWL + i));
            sc_load(zwo, ACP_PTR(blk, lay, p, lay.zWO + i));
            sc_mont(t, xr, zwl);                 // x zWL_i
            sc_add(t, t, zwo);
        }
        sc_sub(t, t, yn);
        sc_sub(t, t, u);
        sc_mul(t, yi, t);
        sc_store(ACP_PTR(blk, lay, p, lay.vH + i), t);
    } else if (i < lay.np + lay.m) {
        const uint32_t j = i - lay.np;
        sc c;
        sc_load(c, sh_c + 8);
        sc_load(u, ACP_PTR(blk, lay, p, lay.zWV + j));
        sc_mont(t, c, u);                        // rho x^2 zWV_j
        sc_neg(t, t);
        sc_store(ACP_PTR(blk, lay, p, lay.vd + j), t);
    } else {
        sc xp[7], wq, pa, pb, that;
        sc_set_u32(xp[0], 1);
        for (int k = 1; k <= 6; k++) sc_mul_noinline(xp[k], xp[k - 1], x);
        sc_load(that, ACP_PTR(blk, lay, p, lay.that));
        sc_load(u, ACP_PTR(blk, lay, p, lay.zc));
        sc_load(v, ACP_PTR(blk, lay, p, lay.sigma));
        sc_add(u, u, v);
        sc_mul_noinline(u, u, xp[2]);
        sc_sub(t, that, u);
        sc_mul_noinline(t, t, rho);              // rho (t - x^2(zc + sigma))
        sc_load(wq, ACP_PTR(blk, lay, p, lay.wq));
        sc_load(pa, ACP_PTR(blk, lay, p, lay.pa));
        sc_load(pb, ACP_PTR(blk, lay, p, lay.pb));
        sc_mul_noinline(u, pa, pb);
        sc_sub(u, that, u);
        sc_mul_noinline(u, u, wq);               // w (t - a b)
        sc_add(t, t, u);
        sc_store(ACP_PTR(blk, lay, p, lay.vg), t);
        sc_load(u, ACP_PTR(blk, lay, p, lay.taux));
        sc_mul_noinline(u, u, rho);
        sc_load(v, ACP_PTR(blk, lay, p, lay.mu));
        sc_sub(t, u, v);
        sc_store(ACP_PTR(blk, lay, p, lay.vh), t);
        const int deg[5] = {1, 3, 4, 5, 6};
        for (int k = 0; k < 5; k++) {
            sc_mul_noinline(t, rho, xp[deg[k]]);
            sc_neg(t, t);
            sc_store(ACP_PTR(blk, lay, p, lay.vd + lay.m + k), t);
        }
        for (int k = 0; k < 3; k++) sc_store(ACP_PTR(blk, lay, p, lay.vd + lay.m + 5 + k), xp[k + 1]);
    }
}
// extra dynamic points: `cnt` encodings per proof (lr: B x cnt x 32) into slots first .. first + cnt of the proof's `per`
// dynamic points.  `fixed` mode: L_k, R_k after the commitments and the eight proof points; the stand-alone
// inner-product verifier: L_k, R_k, P.  Entries below `nonzero` reject an identity encoding (validate_and_append_point),
// every entry an invalid one (decompress() = None).
__global__ void __launch_bounds__(128) k_acp_decompress_lr(const uint8_t *__restrict__ lr, uint32_t cnt, uint32_t nonzero, uint32_t first,
                                                           uint32_t per, uint32_t B, uint32_t *__restrict__ dyn, uint32_t *__restrict__ bad) {
    uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= B * cnt) return;
    const uint32_t p = id / cnt, k = id - p * cnt;
    const uint8_t *src = lr + 32 * (size_t)id;
    uint32_t any = 0;
    for (int b = 0; b < 32; b++) any |= src[b];
    fe x, y;
    bool ok = ge_decompress(x, y, src) && (any != 0 || k >= nonzero);
    if (!ok) {
        atomicOr(&bad[p], 1u);
        fe_set0(x);
        fe_set1(y);
    }
    ge_niels q;
    ge_affine_to_niels(q, x, y);
    ge_niels_store(dyn + 24 * ((size_t)p * per + first + k), q);
}

// ---- stand-alone inner-product batch (bpp_ipa_batch_*; bulletproofs 4.0.0 inner_product_proof.rs create / verify) ----
// The proof block holds the inner-product fields of acp_layout only (ipa_make_layout, capi_acproof.cu): a, b at lay.l,
// lay.r (folded in place by the prover; lay.pa, lay.pb for the verifier), H_factors at lay.yninv, G_factors at lay.yn
// (k_ipa_round_gf), q at lay.wq - so that k_ipa_round's "w c_L" is the Q coefficient of Q = q gens[q_off] - and the
// round state u, uinv, stab, vG, vH, cl.  The verifier's dynamic scalars sit at lay.vd: u_k^2, u_k^-2 (k_ipa_vprep with
// first = 0), then -1 for P.

// contiguous staged inputs (count x n scalars each; q: count x 1) -> proof blocks.  A null a / b is skipped (verifier),
// a null factor vector or q stands for all ones.  Grid (ceil((4 n + 1) / 128), B).
__global__ void __launch_bounds__(128) k_ipa_place(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b,
                                                   const uint32_t *__restrict__ gf, const uint32_t *__restrict__ hf,
                                                   const uint32_t *__restrict__ q, acp_layout lay, uint32_t *__restrict__ blk) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y, n = lay.np;
    if (j > 4 * n) return;
    const uint32_t which = j == 4 * n ? 4 : j / n, i = j - which * n;
    const uint32_t *src = which == 0 ? a : which == 1 ? b : which == 2 ? gf : which == 3 ? hf : q;
    if (!src && which < 2) return;
    const uint32_t dst = which == 0 ? lay.l : which == 1 ? lay.r : which == 2 ? lay.yn : which == 3 ? lay.yninv : lay.wq;
    sc v;
    if (src) sc_load(v, src + 8 * ((size_t)p * (which == 4 ? 1 : n) + i));
    else sc_set_u32(v, 1);
    sc_store(ACP_PTR(blk, lay, p, dst + i), v);
}
// prover: proof p = L_0 R_0 .. L_{lg-1} R_{lg-1} a b (InnerProductProof::to_bytes); lr: B x 2 lg x 32
__global__ void __launch_bounds__(128) k_ipa_pack(acp_layout lay, const uint8_t *__restrict__ lr, const uint32_t *__restrict__ blk,
                                                  uint32_t B, uint8_t *__restrict__ out) {
    const uint32_t words = 2 * lay.lg + 2, id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= B * words) return;
    const uint32_t p = id / words, i = id - p * words;
    const uint4 *s = i < 2 * lay.lg ? reinterpret_cast<const uint4 *>(lr + 32 * ((size_t)p * 2 * lay.lg + i))
                                    : reinterpret_cast<const uint4 *>(ACP_PTR(blk, lay, p, i == 2 * lay.lg ? lay.l : lay.r));
    uint4 *d = reinterpret_cast<uint4 *>(out + 32 * (size_t)id);
    d[0] = s[0];
    d[1] = s[1];
}
// verifier: proofs (B x (2 lg + 2) x 32) and P (B x 32) -> lrp (B x (2 lg + 1) x 32: L_0 R_0 .. P) and a, b at lay.pa,
// lay.pb.  An a or b >= l rejects the proof (InnerProductProof::from_bytes refuses it): bad[p] |= 1.
__global__ void __launch_bounds__(128) k_ipa_unpack(acp_layout lay, const uint8_t *__restrict__ proofs, const uint8_t *__restrict__ P,
                                                    uint32_t B, uint32_t *__restrict__ blk, uint8_t *__restrict__ lrp,
                                                    uint32_t *__restrict__ bad) {
    const uint32_t words = 2 * lay.lg + 2, id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= B * words) return;
    const uint32_t p = id / words, i = id - p * words;
    if (i == words - 1) {   // b's thread also copies P
        const uint4 *s = reinterpret_cast<const uint4 *>(P + 32 * (size_t)p);
        uint4 *d = reinterpret_cast<uint4 *>(lrp + 32 * ((size_t)p * (words - 1) + words - 2));
        d[0] = s[0];
        d[1] = s[1];
    }
    const uint4 *s = reinterpret_cast<const uint4 *>(proofs + 32 * (size_t)id);
    const uint4 lo = s[0], hi = s[1];
    if (i < 2 * lay.lg) {
        uint4 *d = reinterpret_cast<uint4 *>(lrp + 32 * ((size_t)p * (words - 1) + i));
        d[0] = lo;
        d[1] = hi;
        return;
    }
    sc v;
    v.v[0] = lo.x; v.v[1] = lo.y; v.v[2] = lo.z; v.v[3] = lo.w; v.v[4] = hi.x; v.v[5] = hi.y; v.v[6] = hi.z; v.v[7] = hi.w;
    uint32_t l8[8], t[8];
#pragma unroll
    for (int k = 0; k < 8; k++) l8[k] = SC_L[k];
    if (!sc_sub8(t, v.v, l8)) atomicOr(&bad[p], 1u);   // no borrow: v >= l
    sc_reduce256(v, v);
    sc_store(ACP_PTR(blk, lay, p, i == 2 * lay.lg ? lay.pa : lay.pb), v);
}
// verifier scalars of  -a s_i gf_i G_i - b s_i^-1 hf_i H_i - a b q Q + sum_k (u_k^2 L_k + u_k^-2 R_k) + P  (= identity iff
// dalek's verify accepts): vG, vH (n each), cl[0] (Q), and vd[2 lg] = 1 (P).  s from k_ipa_stable_full.  Grid
// (ceil((n + 1) / 128), B).
__global__ void __launch_bounds__(128) k_ipa_vscal(acp_layout lay, uint32_t *__restrict__ blk) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y, n = lay.np;
    if (i > n) return;
    sc pa, pb, t, f;
    sc_load(pa, ACP_PTR(blk, lay, p, lay.pa));
    sc_load(pb, ACP_PTR(blk, lay, p, lay.pb));
    if (i == n) {
        sc_mul(t, pa, pb);
        sc_load(f, ACP_PTR(blk, lay, p, lay.wq));
        sc_mul(t, t, f);
        sc_neg(t, t);
        sc_store(ACP_PTR(blk, lay, p, lay.cl), t);
        sc_set_u32(t, 1);
        sc_store(ACP_PTR(blk, lay, p, lay.vd + 2 * lay.lg), t);
        return;
    }
    sc s;
    const uint32_t *st = ipa_stab(blk, lay, p, lay.lg);
    sc_load(s, st + 8 * (size_t)i);
    sc_mont(t, pa, s);                           // a s_i
    sc_load(f, ACP_PTR(blk, lay, p, lay.yn + i));
    sc_mul(t, t, f);
    sc_neg(t, t);
    sc_store(ACP_PTR(blk, lay, p, lay.vG + i), t);
    sc_load(s, st + 8 * (size_t)(n - 1 - i));
    sc_mont(t, pb, s);                           // b s_i^-1
    sc_load(f, ACP_PTR(blk, lay, p, lay.yninv + i));
    sc_mul(t, t, f);
    sc_neg(t, t);
    sc_store(ACP_PTR(blk, lay, p, lay.vH + i), t);
}
// thread per proof: the dynamic part (k_dyn_window_sums) plus the fixed-base part must be the identity, and no encoding or
// scalar may have been refused
__global__ void __launch_bounds__(64) k_ipa_accept(uint32_t B, const uint32_t *__restrict__ wsum, const uint32_t *__restrict__ stat_ext,
                                                   const uint32_t *__restrict__ bad, uint8_t *__restrict__ accept) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    ge_ext acc, t;
    dyn_horner(acc, wsum, p);
    ge_load(t, stat_ext + 32 * (size_t)p);
    ge_add(acc, acc, t);
    const bool ident = fe_is_zero(acc.X) || fe_is_zero(acc.Y);  // the Ristretto identity coset
    accept[p] = (ident && bad[p] == 0) ? 1 : 0;
}
