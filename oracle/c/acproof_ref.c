/* acproof_ref.c - CPU restatement of the reference's arithmetic-circuit (shuffle) proof.
 *
 * TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): a C restatement of
 * /root/reference/bp-perm/src/{util,poly,transcript_protocol,circuit_lib}.rs on top of dalek_ref.c,
 * structured like the reference (dense W matrices, one vartime MSM per call site, n separate
 * inversions, n variable-base scalar multiplications in verify) so that its timing is the
 * reference's CPU path.  Used as the fast checker for batches and as the timed CPU baseline of
 * bench.py; pinned against oracle/acproof.py (Python) in tests/test_oracle_acproof.py.
 * Compiled together with dalek_ref.c (single translation unit via #include).
 */
#include "dalek_ref.c"
typedef uint32_t u32;

/* ------------------------------------------------------------------ scalars mod l ------------- */
/* dalek Scalar: 32 canonical bytes; every operation unpacks, computes, repacks (scalar.rs). */
typedef struct { u64 v[4]; } sc;
static const u64 SC_Lq[4] = {0x5812631a5cf5d3edULL, 0x14def9dea2f79cd6ULL, 0, 0x1000000000000000ULL};
static const u64 SC_R2q[4] = {0xa40611e3449c0f01ULL, 0xd00e1ba768859347ULL, 0xceec73d217f5be65ULL, 0x0399411b7c309a3dULL};
static const u64 SC_Rq[4] = {0xd6ec31748d98951dULL, 0xc6ef5bf4737dcf70ULL, 0xfffffffffffffffeULL, 0x0fffffffffffffffULL};
#define SC_NPRIME64 0xd2b51da312547e1bULL /* -l^{-1} mod 2^64 */

static void sc_frombytes(sc *r, const u8 *b) { memcpy(r->v, b, 32); }
static void sc_tobytes(u8 *b, const sc *a) { memcpy(b, a->v, 32); }
static int sc_geq_l(const u64 a[4], u64 top) {
    if (top) return 1;
    for (int i = 3; i >= 0; i--) {
        if (a[i] > SC_Lq[i]) return 1;
        if (a[i] < SC_Lq[i]) return 0;
    }
    return 1;
}
static void sc_sub_l(u64 a[4]) {
    u128 borrow = 0;
    for (int i = 0; i < 4; i++) {
        u128 d = (u128)a[i] - SC_Lq[i] - (u64)borrow;
        a[i] = (u64)d;
        borrow = (d >> 64) & 1;
    }
}
static void sc_mont(sc *r, const sc *a, const sc *b) {
    u64 t[9] = {0};
    for (int i = 0; i < 4; i++) {
        u128 carry = 0;
        for (int j = 0; j < 4; j++) {
            u128 v = (u128)a->v[j] * b->v[i] + t[i + j] + (u64)carry;
            t[i + j] = (u64)v;
            carry = v >> 64;
        }
        t[i + 4] = (u64)carry;
    }
    for (int i = 0; i < 4; i++) {
        u64 m = t[i] * SC_NPRIME64;
        u128 carry = 0;
        for (int j = 0; j < 4; j++) {
            u128 v = (u128)m * SC_Lq[j] + t[i + j] + (u64)carry;
            t[i + j] = (u64)v;
            carry = v >> 64;
        }
        for (int k = i + 4; k < 9; k++) {
            carry += t[k];
            t[k] = (u64)carry;
            carry >>= 64;
        }
    }
    u64 res[4] = {t[4], t[5], t[6], t[7]};
    if (sc_geq_l(res, t[8])) sc_sub_l(res);
    memcpy(r->v, res, 32);
}
static void sc_mul(sc *r, const sc *a, const sc *b) {
    sc t, r2;
    memcpy(r2.v, SC_R2q, 32);
    sc_mont(&t, a, b);
    sc_mont(r, &t, &r2);
}
static void sc_add(sc *r, const sc *a, const sc *b) {
    u64 s[4];
    u128 c = 0;
    for (int i = 0; i < 4; i++) {
        c += (u128)a->v[i] + b->v[i];
        s[i] = (u64)c;
        c >>= 64;
    }
    if (sc_geq_l(s, (u64)c)) sc_sub_l(s);
    memcpy(r->v, s, 32);
}
static void sc_neg(sc *r, const sc *a) {
    int zero = !(a->v[0] | a->v[1] | a->v[2] | a->v[3]);
    u128 borrow = 0;
    for (int i = 0; i < 4; i++) {
        u128 d = (u128)SC_Lq[i] - a->v[i] - (u64)borrow;
        r->v[i] = zero ? 0 : (u64)d;
        borrow = (d >> 64) & 1;
    }
}
static void sc_sub(sc *r, const sc *a, const sc *b) {
    sc nb;
    sc_neg(&nb, b);
    sc_add(r, a, &nb);
}
static void sc_invert(sc *r, const sc *a) { /* a^(l-2) */
    static const u64 E[4] = {0x5812631a5cf5d3ebULL, 0x14def9dea2f79cd6ULL, 0, 0x1000000000000000ULL};
    sc am, acc, r2, one = {{1, 0, 0, 0}};
    memcpy(r2.v, SC_R2q, 32);
    sc_mont(&am, a, &r2);
    memcpy(acc.v, SC_Rq, 32);
    for (int bit = 252; bit >= 0; bit--) {
        sc_mont(&acc, &acc, &acc);
        if ((E[bit >> 6] >> (bit & 63)) & 1) sc_mont(&acc, &acc, &am);
    }
    sc_mont(r, &acc, &one);
}
static void sc_from_wide(sc *r, const u8 in[64]) { /* Scalar::from_bytes_mod_order_wide */
    sc lo, hi, k, a, b;
    memcpy(lo.v, in, 32);
    memcpy(hi.v, in + 32, 32);
    memcpy(k.v, SC_Rq, 32);
    sc_mont(&a, &lo, &k);
    memcpy(k.v, SC_R2q, 32);
    sc_mont(&b, &hi, &k);
    sc_add(r, &a, &b);
}
static void sc_from_u64(sc *r, u64 x) { r->v[0] = x; r->v[1] = r->v[2] = r->v[3] = 0; }
static void sc_from_bytes_mod_order(sc *r, const u8 *b) { u8 w[64] = {0}; memcpy(w, b, 32); sc_from_wide(r, w); }

/* ------------------------------------------------------------------ util.rs / poly.rs ---------- */
static void v_inner_product(sc *out, const sc *a, const sc *b, size_t n) { /* util.rs:84-94 */
    sc acc = {{0, 0, 0, 0}}, t;
    for (size_t i = 0; i < n; i++) { sc_mul(&t, &a[i], &b[i]); sc_add(&acc, &acc, &t); }
    *out = acc;
}
static void v_hadamard(sc *out, const sc *a, const sc *b, size_t n) { /* util.rs:6-20 (the `1 *=` included) */
    sc one = {{1, 0, 0, 0}}, t;
    for (size_t i = 0; i < n; i++) { sc_mul(&t, &a[i], &b[i]); sc_mul(&out[i], &one, &t); }
}
/* vm_mult (util.rs:22-38): copies each row into a fresh Vec, then inner_product */
static void v_vm_mult(sc *out, const sc *a, const sc *b, size_t rows, size_t cols) {
    sc *col = malloc(cols * sizeof(sc));
    for (size_t i = 0; i < rows; i++) {
        for (size_t j = 0; j < cols; j++) col[j] = b[i * cols + j];
        v_inner_product(&out[i], a, col, cols);
    }
    free(col);
}
/* mv_mult (util.rs:40-56): out[j] = sum_i a[i][j] b[i], column gathered into a fresh Vec */
static void v_mv_mult(sc *out, const sc *a, const sc *b, size_t rows, size_t cols) {
    sc *col = malloc(rows * sizeof(sc));
    for (size_t j = 0; j < cols; j++) {
        for (size_t i = 0; i < rows; i++) col[i] = a[i * cols + j];
        v_inner_product(&out[j], col, b, rows);
    }
    free(col);
}
static void v_exp_iter(sc *out, const sc *x, size_t count) { /* util.rs:63-65,139-157 (Fibonacci exponents) */
    sc base = {{1, 0, 0, 0}}, nxt = *x, ret;
    for (size_t i = 0; i < count; i++) { ret = nxt; sc_mul(&nxt, &nxt, &base); base = ret; out[i] = ret; }
}
static void v_scalar_exp(sc *out, const sc *x, int pw) { /* util.rs:75-82 */
    sc r = {{1, 0, 0, 0}};
    for (int i = 0; i < pw; i++) sc_mul(&r, &r, x);
    *out = r;
}
static void v_poly3_eval(sc *out, const sc *c0, const sc *c1, const sc *c2, const sc *c3, const sc *x, size_t n) {
    sc t;                                            /* poly.rs:57-76 */
    for (size_t i = 0; i < n; i++) {
        sc_mul(&t, x, &c3[i]); sc_add(&t, &t, &c2[i]);
        sc_mul(&t, x, &t); sc_add(&t, &t, &c1[i]);
        sc_mul(&t, x, &t); sc_add(&out[i], &t, &c0[i]);
    }
}
static void v_poly6_eval(sc *out, const sc t[6], const sc *x) { /* poly.rs:14-18 */
    sc acc = t[5];
    for (int k = 4; k >= 0; k--) { sc_mul(&acc, x, &acc); sc_add(&acc, &acc, &t[k]); }
    sc_mul(out, x, &acc);
}

/* ------------------------------------------------------------------ Merlin (merlin 3.0.0) ------ */
static u64 rol64(u64 v, int n) { return n ? (v << n) | (v >> (64 - n)) : v; }
static void keccak_f1600(u64 a[25]) {
    static const u64 RC[24] = {
        0x0000000000000001ULL, 0x0000000000008082ULL, 0x800000000000808aULL, 0x8000000080008000ULL,
        0x000000000000808bULL, 0x0000000080000001ULL, 0x8000000080008081ULL, 0x8000000000008009ULL,
        0x000000000000008aULL, 0x0000000000000088ULL, 0x0000000080008009ULL, 0x000000008000000aULL,
        0x000000008000808bULL, 0x800000000000008bULL, 0x8000000000008089ULL, 0x8000000000008003ULL,
        0x8000000000008002ULL, 0x8000000000000080ULL, 0x000000000000800aULL, 0x800000008000000aULL,
        0x8000000080008081ULL, 0x8000000000008080ULL, 0x0000000080000001ULL, 0x8000000080008008ULL};
    static const int RHO[25] = {0, 1, 62, 28, 27, 36, 44, 6, 55, 20, 3, 10, 43, 25, 39, 41, 45, 15, 21, 8, 18, 2, 61, 56, 14};
    for (int rd = 0; rd < 24; rd++) {
        u64 c[5], b[25];
        for (int x = 0; x < 5; x++) c[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
        for (int x = 0; x < 5; x++) {
            u64 d = c[(x + 4) % 5] ^ rol64(c[(x + 1) % 5], 1);
            for (int y = 0; y < 25; y += 5) a[x + y] ^= d;
        }
        for (int x = 0; x < 5; x++)
            for (int y = 0; y < 5; y++) b[y + 5 * ((2 * x + 3 * y) % 5)] = rol64(a[x + 5 * y], RHO[x + 5 * y]);
        for (int y = 0; y < 25; y += 5)
            for (int x = 0; x < 5; x++) a[x + y] = b[x + y] ^ (~b[(x + 1) % 5 + y] & b[(x + 2) % 5 + y]);
        a[0] ^= RC[rd];
    }
}
typedef struct { u8 st[200]; u8 pos, pos_begin, cur_flags; } strobe;
#define STROBE_R 166
static void strobe_permute(strobe *s) { u64 l[25]; memcpy(l, s->st, 200); keccak_f1600(l); memcpy(s->st, l, 200); }
static void strobe_run_f(strobe *s) {
    s->st[s->pos] ^= s->pos_begin; s->st[s->pos + 1] ^= 0x04; s->st[STROBE_R + 1] ^= 0x80;
    strobe_permute(s); s->pos = 0; s->pos_begin = 0;
}
static void strobe_absorb(strobe *s, const u8 *d, size_t n) {
    for (size_t i = 0; i < n; i++) { s->st[s->pos] ^= d[i]; if (++s->pos == STROBE_R) strobe_run_f(s); }
}
static void strobe_squeeze(strobe *s, u8 *d, size_t n) {
    for (size_t i = 0; i < n; i++) { d[i] = s->st[s->pos]; s->st[s->pos] = 0; if (++s->pos == STROBE_R) strobe_run_f(s); }
}
static void strobe_begin(strobe *s, u8 flags, int more) {
    if (more) return;
    u8 hdr[2] = {s->pos_begin, flags};
    s->pos_begin = s->pos + 1; s->cur_flags = flags;
    strobe_absorb(s, hdr, 2);
    if ((flags & (4 | 32)) && s->pos != 0) strobe_run_f(s);
}
static void strobe_meta_ad(strobe *s, const u8 *d, size_t n, int more) { strobe_begin(s, 16 | 2, more); strobe_absorb(s, d, n); }
static void strobe_ad(strobe *s, const u8 *d, size_t n, int more) { strobe_begin(s, 2, more); strobe_absorb(s, d, n); }
static void strobe_prf(strobe *s, u8 *d, size_t n) { strobe_begin(s, 1 | 2 | 4, 0); strobe_squeeze(s, d, n); }
static void tr_append(strobe *s, const char *label, const u8 *msg, size_t n) {
    u8 len[4] = {(u8)n, (u8)(n >> 8), (u8)(n >> 16), (u8)(n >> 24)};
    strobe_meta_ad(s, (const u8 *)label, strlen(label), 0);
    strobe_meta_ad(s, len, 4, 1);
    strobe_ad(s, msg, n, 0);
}
static void tr_new(strobe *s, const u8 *label, size_t n) {
    memset(s, 0, sizeof(*s));
    const u8 init[6] = {1, STROBE_R + 2, 1, 0, 1, 96};
    memcpy(s->st, init, 6); memcpy(s->st + 6, "STROBEv1.0.2", 12);
    strobe_permute(s);
    strobe_meta_ad(s, (const u8 *)"Merlin v1.0", 11, 0);
    tr_append(s, "dom-sep", label, n);
}
static void tr_challenge_scalar(strobe *s, const char *label, sc *out) { /* transcript_protocol.rs:62-67 */
    u8 buf[64], len[4] = {64, 0, 0, 0};
    strobe_meta_ad(s, (const u8 *)label, strlen(label), 0);
    strobe_meta_ad(s, len, 4, 1);
    strobe_prf(s, buf, 64);
    sc_from_wide(out, buf);
}
static void tr_challenge_bytes(strobe *s, const char *label, u8 *out, size_t n) {
    u8 len[4] = {(u8)n, (u8)(n >> 8), (u8)(n >> 16), (u8)(n >> 24)};
    strobe_meta_ad(s, (const u8 *)label, strlen(label), 0);
    strobe_meta_ad(s, len, 4, 1);
    strobe_prf(s, out, n);
}
static void tr_append_scalar(strobe *s, const char *label, const sc *x) { u8 b[32]; sc_tobytes(b, x); tr_append(s, label, b, 32); }
/* append_vec_scalar (transcript_protocol.rs:36-43): decimal strings + bytevec framing; no challenge is
 * drawn afterwards in the reference flow, so only its cost matters here */
static void tr_append_vec_scalar(strobe *s, const char *label, const sc *v, size_t n) {
    u8 *buf = malloc(8 + n * (8 + 80)); size_t o = 8;
    for (size_t i = 0; i < n; i++) {
        u64 w[4]; memcpy(w, v[i].v, 32);
        char dec[80]; int nd = 0;
        while (w[0] | w[1] | w[2] | w[3]) {
            u128 rem = 0;
            for (int k = 3; k >= 0; k--) { u128 cur = (rem << 64) | w[k]; w[k] = (u64)(cur / 10); rem = cur % 10; }
            dec[nd++] = (char)('0' + (int)rem);
        }
        if (!nd) dec[nd++] = '0';
        for (int k = 0; k < 8; k++) buf[o + k] = (u8)((u64)nd >> (56 - 8 * k));
        o += 8;
        for (int k = 0; k < nd; k++) buf[o++] = (u8)dec[nd - 1 - k];
    }
    for (int k = 0; k < 8; k++) buf[k] = (u8)((u64)(o - 8) >> (56 - 8 * k));
    tr_append(s, label, buf, o);
    free(buf);
}

/* ------------------------------------------------------------------ RNG: ChaCha20 stream ------- */
static u32 rotl32(u32 v, int n) { return (v << n) | (v >> (32 - n)); }
#define QR(a, b, c, d) a += b; d = rotl32(d ^ a, 16); c += d; b = rotl32(b ^ c, 12); a += b; d = rotl32(d ^ a, 8); c += d; b = rotl32(b ^ c, 7);
typedef struct { u32 key[8]; u64 ctr; } rng_t;
static void rng_scalar(rng_t *g, sc *out) { /* Scalar::random: next 64 bytes -> wide reduce */
    u32 s[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u}, x[16];
    memcpy(s + 4, g->key, 32);
    s[12] = (u32)g->ctr; s[13] = (u32)(g->ctr >> 32); s[14] = s[15] = 0;
    g->ctr++;
    memcpy(x, s, 64);
    for (int r = 0; r < 10; r++) {
        QR(x[0], x[4], x[8], x[12]) QR(x[1], x[5], x[9], x[13]) QR(x[2], x[6], x[10], x[14]) QR(x[3], x[7], x[11], x[15])
        QR(x[0], x[5], x[10], x[15]) QR(x[1], x[6], x[11], x[12]) QR(x[2], x[7], x[8], x[13]) QR(x[3], x[4], x[9], x[14])
    }
    for (int i = 0; i < 16; i++) x[i] += s[i];
    sc_from_wide(out, (const u8 *)x);
}

/* ------------------------------------------------------------------ group helpers -------------- */
static void msm_sc(ge_ext *out, const sc *scalars, const ge_ext *pts, size_t n) { /* vartime_multiscalar_mul */
    msm_dispatch(out, (const u8 *)scalars, pts, n);
}
/* `RistrettoPoint * Scalar` (circuit_lib.rs:491): dalek variable_base::mul, fixed radix-16 windows */
static void ge_scalarmul_radix16(ge_ext *out, const sc *s, const ge_ext *p) {
    ge_pniels tab[8];
    ge_ext cur = *p;
    ge_to_pniels(&tab[0], &cur);
    for (int k = 1; k < 8; k++) { ge_compl c; ge_add_pn(&c, &cur, &tab[0], 0); ge_compl_to_ext(&cur, &c); ge_to_pniels(&tab[k], &cur); }
    int8_t d[64]; u8 b[32];
    sc_tobytes(b, s);
    for (int i = 0; i < 32; i++) { d[2 * i] = b[i] & 15; d[2 * i + 1] = (b[i] >> 4) & 15; }
    for (int i = 0; i < 63; i++) { int8_t carry = (d[i] + 8) >> 4; d[i] -= carry << 4; d[i + 1] += carry; }
    ge_ext acc; ge_identity(&acc);
    for (int i = 63; i >= 0; i--) {
        if (i != 63) ge_mul_pow2(&acc, &acc, 4);
        if (d[i] > 0) { ge_compl c; ge_add_pn(&c, &acc, &tab[d[i] - 1], 0); ge_compl_to_ext(&acc, &c); }
        else if (d[i] < 0) { ge_compl c; ge_add_pn(&c, &acc, &tab[-d[i] - 1], 1); ge_compl_to_ext(&acc, &c); }
    }
    *out = acc;
}
static int ge_ristretto_eq(const ge_ext *p, const ge_ext *q) {
    fe a, b;
    fe_mul(&a, &p->X, &q->Y); fe_mul(&b, &p->Y, &q->X);
    if (fe_eq(&a, &b)) return 1;
    fe_mul(&a, &p->X, &q->X); fe_mul(&b, &p->Y, &q->Y);
    return fe_eq(&a, &b);
}

/* ------------------------------------------------------------------ the 7-step flow ------------ */
/* m as a u64 under "m", then every value commitment's encoding under "V" (oracle/acproof.py append_commitments;
 * bulletproofs 4.0.0 r1cs prover: append_point(b"V", ..) per commit(), append_u64(b"m", m)).  V_enc (m x 32 compressed
 * encodings, what a verifier is handed) is used when given, else the points are compressed here. */
#define V_CHUNK 64
static void tr_append_commitments(strobe *tr, const ge_ext *V, const u8 *V_enc, size_t m) {
    u8 mb[8], buf[32 * V_CHUNK];
    const size_t nch = (m + V_CHUNK - 1) / V_CHUNK;
    u8 *digs = (u8 *)malloc(32 * nch);
    for (int i = 0; i < 8; i++) mb[i] = (u8)((u64)m >> (8 * i));
    tr_append(tr, "m", mb, 8);
    for (size_t c = 0; c < m; c += V_CHUNK) {   /* one sponge per chunk of 64 commitments */
        strobe ch; tr_new(&ch, (const u8 *)"acp-V", 5);
        for (int i = 0; i < 8; i++) mb[i] = (u8)((u64)(c / V_CHUNK) >> (8 * i));
        tr_append(&ch, "chunk", mb, 8);
        size_t cnt = 0;
        for (size_t j = c; j < m && j < c + V_CHUNK; j++, cnt++) {
            if (V_enc) memcpy(buf + 32 * cnt, V_enc + 32 * j, 32);
            else ristretto_compress(buf + 32 * cnt, &V[j]);
        }
        tr_append(&ch, "V", buf, 32 * cnt);   /* the chunk's encodings as one message */
        tr_challenge_bytes(&ch, "d", digs + 32 * (c / V_CHUNK), 32);
    }
    tr_append(tr, "Vd", digs, 32 * nch);        /* the chunk digests, concatenated, as one message */
    free(digs);
}

/* verify :478-585 from the proof bytes alone (A_I,A_O,S,T1,T3,T4,T5,T6,tau_x,mu,t,l,r): replays the verifier's
 * transcript from those bytes (mode 1: with the commitment binding; mode 0: "T4" carries T_3's bytes), then checks
 * 1 (t == <l, r>), 2 and, in mode 1, 3.  Decoding as the library's verifier: a scalar >= l is taken mod l, an
 * undecodable point is a reject (the reference unwraps T and panics, circuit_lib.rs:532), the all-zero encoding is the
 * identity.  V: the commitments as points; V_enc, when given, is what the transcript binds.  Returns 1 for Ok(()). */
static int acp_verify(int mode, size_t n, size_t Q, size_t m, const sc *W_L, const sc *W_R, const sc *W_O, const sc *W_V,
                      const sc *cv, const ge_ext *g, const ge_ext *h, const ge_ext *G, const ge_ext *H, const u8 *po,
                      const ge_ext *V, const u8 *V_enc, const u8 *label, size_t label_len) {
    static const int DEG[5] = {1, 3, 4, 5, 6};
    static const char *TL[5] = {"T1", "T3", "T4", "T5", "T6"};
    ge_ext pts8[8];
    for (int k = 0; k < 8; k++)
        if (!ristretto_decompress(&pts8[k], po + 32 * k)) return 0;
    const ge_ext A_I = pts8[0], A_O = pts8[1], S = pts8[2];
    size_t big = 2 * n + m + 16;
    sc *sv = malloc(big * sizeof(sc)); ge_ext *pv = malloc(big * sizeof(ge_ext));
    sc tau_x, mu, that;
    sc_from_bytes_mod_order(&tau_x, po + 256); sc_from_bytes_mod_order(&mu, po + 288); sc_from_bytes_mod_order(&that, po + 320);
    sc *l = malloc(n * sizeof(sc)), *r = malloc(n * sizeof(sc));
    for (size_t i = 0; i < n; i++) { sc_from_bytes_mod_order(&l[i], po + 352 + 32 * i); sc_from_bytes_mod_order(&r[i], po + 352 + 32 * (n + i)); }
    /* ---- the transcript, as create .. random_chall_x appended it ---- */
    strobe tr; tr_new(&tr, label, label_len);
    { u8 nb[8]; for (int i = 0; i < 8; i++) nb[i] = (u8)((u64)n >> (8 * i)); tr_append(&tr, "dom-sep", (const u8 *)"acp v1", 6); tr_append(&tr, "n", nb, 8); }
    if (mode != 0) tr_append_commitments(&tr, V, V_enc, m);
    tr_append(&tr, "A_I", po, 32); tr_append(&tr, "A_O", po + 32, 32); tr_append(&tr, "S", po + 64, 32);
    sc y, z; tr_challenge_scalar(&tr, "y", &y); tr_challenge_scalar(&tr, "z", &z);
    for (int k = 0; k < 5; k++) tr_append(&tr, TL[k], (mode == 0 && k == 2) ? po + 96 + 32 : po + 96 + 32 * k, 32);
    sc x; tr_challenge_scalar(&tr, "x", &x);
    /* ---- compute_per_challenges :256-302 ---- */
    sc *y_n = malloc(n * sizeof(sc)), *y_n_inv = malloc(n * sizeof(sc)), *z_q = malloc(Q * sizeof(sc));
    sc *z_W_R = malloc(n * sizeof(sc)), *z_W_L = malloc(n * sizeof(sc)), *l_in = malloc(n * sizeof(sc));
    sc *tmp = malloc((Q > n ? Q : n) * sizeof(sc));
    v_exp_iter(y_n, &y, n);
    for (size_t i = 0; i < n; i++) sc_invert(&y_n_inv[i], &y_n[i]);
    v_exp_iter(z_q, &z, Q);
    v_vm_mult(z_W_R, z_q, W_R, n, Q);
    v_hadamard(l_in, y_n_inv, z_W_R, n);
    v_vm_mult(z_W_L, z_q, W_L, n, Q);
    sc sigma; v_inner_product(&sigma, l_in, z_W_L, n);
    sc xx, xp3; sc_mul(&xx, &x, &x); v_scalar_exp(&xp3, &x, 3);
    int result = 1;
    ge_ext *h_ = malloc(n * sizeof(ge_ext));
    for (size_t i = 0; i < n; i++) ge_scalarmul_radix16(&h_[i], &y_n_inv[i], &H[i]);           /* :491 */
    ge_ext wL, wR, wO;
    msm_sc(&wL, z_W_L, h_, n);                                                                 /* :498 */
    msm_sc(&wR, l_in, G, n);                                                                   /* :504 */
    v_vm_mult(tmp, z_q, W_O, n, Q); msm_sc(&wO, tmp, h_, n);                                   /* :509 */
    sc chk; v_inner_product(&chk, l, r, n);
    if (memcmp(chk.v, that.v, 32) != 0) result = 0;                                            /* :518 */
    if (result) {
        sc g_exp, zc; v_inner_product(&zc, z_q, cv, Q); sc_add(&zc, &zc, &sigma); sc_mul(&g_exp, &xx, &zc);
        sc *zwv = malloc(m * sizeof(sc)); v_vm_mult(zwv, z_q, W_V, m, Q);
        sv[0] = g_exp; pv[0] = *g;
        for (size_t j = 0; j < m; j++) { sc_mul(&sv[1 + j], &xx, &zwv[j]); pv[1 + j] = V[j]; }
        for (int k = 0; k < 5; k++) { v_scalar_exp(&sv[1 + m + k], &x, DEG[k]); pv[1 + m + k] = pts8[3 + k]; }
        free(zwv);
        ge_ext cand, lhs; msm_sc(&cand, sv, pv, 1 + m + 5);                                    /* :525-533 */
        sv[0] = that; sv[1] = tau_x; pv[0] = *g; pv[1] = *h; msm_sc(&lhs, sv, pv, 2);          /* :535-538 */
        if (!ge_ristretto_eq(&lhs, &cand)) result = 0;                                         /* :541 */
    }
    if (result == 1) {
        sc one = {{1, 0, 0, 0}};
        sv[0] = x; sv[1] = xx; pv[0] = A_I; pv[1] = A_O;
        for (size_t i = 0; i < n; i++) { sc_neg(&sv[2 + i], &y_n[i]); pv[2 + i] = h_[i]; }
        sv[2 + n] = x; sv[3 + n] = x; sv[4 + n] = one; sv[5 + n] = xp3;
        pv[2 + n] = wL; pv[3 + n] = wR; pv[4 + n] = wO; pv[5 + n] = S;
        ge_ext P, candP; msm_sc(&P, sv, pv, n + 6);                                            /* :552-565 */
        sv[0] = mu; pv[0] = *h; memcpy(sv + 1, l, n * 32); memcpy(sv + 1 + n, r, n * 32);
        memcpy(pv + 1, G, n * sizeof(ge_ext)); memcpy(pv + 1 + n, mode == 0 ? H : h_, n * sizeof(ge_ext));
        msm_sc(&candP, sv, pv, 1 + 2 * n);                                                     /* :568-575 */
        if (mode != 0 && !ge_ristretto_eq(&P, &candP)) result = 0;                             /* :577-582 disabled in mode 0 */
    }
    free(h_); free(sv); free(pv); free(l); free(r); free(y_n); free(y_n_inv); free(z_q); free(z_W_R); free(z_W_L);
    free(l_in); free(tmp);
    return result;
}

/* The verifier alone (acp_verify) over caller proof bytes.  V_pts: the commitments as points, or NULL to decode them
 * from V_enc (an undecodable commitment is a reject); V_enc NULL: the transcript binds the compressed V_pts. */
int orc_acp_verify(int mode, size_t n, size_t Q, size_t m, const u8 *WLb, const u8 *WRb, const u8 *WOb, const u8 *WVb,
                   const u8 *cb, const u8 *g_pt, const u8 *h_pt, const u8 *G_pts, const u8 *H_pts, const u8 *proof,
                   const u8 *V_pts, const u8 *V_enc, const u8 *label, size_t label_len) {
    orc_init();
    if (!V_pts && !V_enc) return -1;
    ge_ext *Vd = NULL;
    if (!V_pts) {
        Vd = malloc(m * sizeof(ge_ext));
        for (size_t j = 0; j < m; j++)
            if (!ristretto_decompress(&Vd[j], V_enc + 32 * j)) { free(Vd); return 0; }
    }
    int rc = acp_verify(mode, n, Q, m, (const sc *)WLb, (const sc *)WRb, (const sc *)WOb, (const sc *)WVb, (const sc *)cb,
                        (const ge_ext *)g_pt, (const ge_ext *)h_pt, (const ge_ext *)G_pts, (const ge_ext *)H_pts, proof,
                        V_pts ? (const ge_ext *)V_pts : Vd, V_enc, label, label_len);
    free(Vd);
    return rc;
}

/* lib.rs:219-231 / circuit_lib.rs:133-585.  W_* dense, row-major: W_L,W_R,W_O n x Q, W_V m x Q.
 * mode 0 = reference (defects included), 1 = reference-fixed.  Writes the proof bytes
 * (A_I,A_O,S,T1,T3,T4,T5,T6,tau_x,mu,t,l,r) and, with do_verify, returns acp_verify's decision over them:
 * 1 for Ok(()), 0 for Err(VerificationError). */
int orc_acp_prove_verify(int mode, size_t n, size_t Q, size_t m, const u8 *WLb, const u8 *WRb, const u8 *WOb,
                         const u8 *WVb, const u8 *cb, const u8 *g_pt, const u8 *h_pt, const u8 *G_pts, const u8 *H_pts,
                         const u8 *aLb, const u8 *aRb, const u8 *aOb, const u8 *gammab, const u8 *V_pts, const u8 *V_enc,
                         const u8 *seed32, const u8 *label, size_t label_len, u8 *proof_out, int do_verify) {
    orc_init();
    const sc *W_L = (const sc *)WLb, *W_R = (const sc *)WRb, *W_O = (const sc *)WOb, *W_V = (const sc *)WVb;
    const sc *cv = (const sc *)cb, *a_L = (const sc *)aLb, *a_R = (const sc *)aRb, *a_O = (const sc *)aOb;
    const sc *gamma = (const sc *)gammab;
    const ge_ext *g = (const ge_ext *)g_pt, *h = (const ge_ext *)h_pt, *G = (const ge_ext *)G_pts, *H = (const ge_ext *)H_pts;
    const ge_ext *V = (const ge_ext *)V_pts;
    rng_t rng; memcpy(rng.key, seed32, 32); rng.ctr = 0;
    strobe tr; tr_new(&tr, label, label_len);
    size_t big = 2 * n + m + 16;
    sc *sv = malloc(big * sizeof(sc)); ge_ext *pv = malloc(big * sizeof(ge_ext));
    /* ---- create :139-253 ---- */
    { u8 nb[8]; for (int i = 0; i < 8; i++) nb[i] = (u8)((u64)n >> (8 * i)); tr_append(&tr, "dom-sep", (const u8 *)"acp v1", 6); tr_append(&tr, "n", nb, 8); }
    if (mode != 0) tr_append_commitments(&tr, V, V_enc, m);   /* the reference never binds V (defect 12) */
    sc alpha, beta, ro; rng_scalar(&rng, &alpha); rng_scalar(&rng, &beta); rng_scalar(&rng, &ro);
    ge_ext A_I, A_O, S;
    sv[0] = alpha; pv[0] = *h; memcpy(sv + 1, a_L, n * 32); memcpy(pv + 1, G, n * sizeof(ge_ext));
    memcpy(sv + 1 + n, a_R, n * 32); memcpy(pv + 1 + n, H, n * sizeof(ge_ext));
    msm_sc(&A_I, sv, pv, 1 + 2 * n);
    sv[0] = beta; memcpy(sv + 1, a_O, n * 32);
    msm_sc(&A_O, sv, pv, 1 + n);
    sc *s_l = malloc(n * sizeof(sc)), *s_r = malloc(n * sizeof(sc));
    for (size_t i = 0; i < n; i++) rng_scalar(&rng, &s_l[i]);
    for (size_t i = 0; i < n; i++) rng_scalar(&rng, &s_r[i]);
    sv[0] = ro; memcpy(sv + 1, s_l, n * 32); memcpy(sv + 1 + n, s_r, n * 32);
    msm_sc(&S, sv, pv, 1 + 2 * n);
    u8 *po = proof_out;
    ristretto_compress(po, &A_I); ristretto_compress(po + 32, &A_O); ristretto_compress(po + 64, &S);
    tr_append(&tr, "A_I", po, 32); tr_append(&tr, "A_O", po + 32, 32); tr_append(&tr, "S", po + 64, 32);
    /* ---- challenge_wit_and_const :133-138 ---- */
    sc y, z; tr_challenge_scalar(&tr, "y", &y); tr_challenge_scalar(&tr, "z", &z);
    /* ---- compute_per_challenges :256-302 ---- */
    sc *y_n = malloc(n * sizeof(sc)), *y_n_inv = malloc(n * sizeof(sc)), *z_q = malloc(Q * sizeof(sc));
    sc *z_W_R = malloc(n * sizeof(sc)), *z_W_L = malloc(n * sizeof(sc)), *l_in = malloc(n * sizeof(sc));
    v_exp_iter(y_n, &y, n);
    for (size_t i = 0; i < n; i++) sc_invert(&y_n_inv[i], &y_n[i]);
    v_exp_iter(z_q, &z, Q);
    v_vm_mult(z_W_R, z_q, W_R, n, Q);
    v_hadamard(l_in, y_n_inv, z_W_R, n);
    v_vm_mult(z_W_L, z_q, W_L, n, Q);
    sc sigma; v_inner_product(&sigma, l_in, z_W_L, n);
    /* ---- commit_Ts :304-423 ---- */
    sc *l1 = malloc(n * sizeof(sc)), *r0 = malloc(n * sizeof(sc)), *r1 = malloc(n * sizeof(sc)), *r3 = malloc(n * sizeof(sc));
    sc *tmp = malloc((Q > n ? Q : n) * sizeof(sc)), *tmp2 = malloc((Q > n ? Q : n) * sizeof(sc));
    for (size_t i = 0; i < n; i++) sc_add(&l1[i], &a_L[i], &l_in[i]);
    v_vm_mult(tmp, z_q, W_O, n, Q);
    for (size_t i = 0; i < n; i++) sc_sub(&r0[i], &tmp[i], &y_n[i]);
    v_hadamard(tmp, y_n, a_R, n);
    v_vm_mult(tmp2, z_q, W_L, n, Q);
    for (size_t i = 0; i < n; i++) sc_add(&r1[i], &tmp[i], &tmp2[i]);
    v_hadamard(r3, y_n, s_r, n);
    sc t6[6], d1, d2;
    v_inner_product(&t6[0], l1, r0, n);
    v_inner_product(&d1, l1, r1, n); v_inner_product(&d2, a_O, r0, n); sc_add(&t6[1], &d1, &d2);
    v_inner_product(&d1, a_O, r1, n); v_inner_product(&d2, s_l, r0, n); sc_add(&t6[2], &d1, &d2);
    v_inner_product(&d1, l1, r3, n); v_inner_product(&d2, s_l, r1, n); sc_add(&t6[3], &d1, &d2);
    v_inner_product(&t6[4], a_O, r3, n);
    v_inner_product(&t6[5], s_l, r3, n);
    {   /* :344-356  w = W_L a_L + W_R a_R + W_O a_O and t_2: computed and discarded by the reference */
        sc *wq = malloc(Q * sizeof(sc)), *wq2 = malloc(Q * sizeof(sc)), t2;
        v_mv_mult(wq, W_L, a_L, n, Q); v_mv_mult(wq2, W_R, a_R, n, Q);
        for (size_t q = 0; q < Q; q++) sc_add(&wq[q], &wq[q], &wq2[q]);
        v_mv_mult(wq2, W_O, a_O, n, Q);
        for (size_t q = 0; q < Q; q++) sc_add(&wq[q], &wq[q], &wq2[q]);
        v_hadamard(tmp, a_R, y_n, n); v_inner_product(&t2, a_L, tmp, n);
        v_inner_product(&d1, z_q, wq, Q); sc_add(&t2, &t2, &d1); sc_add(&t2, &t2, &sigma);
        v_inner_product(&d1, a_O, y_n, n); sc_sub(&t2, &t2, &d1);
        free(wq); free(wq2);
    }
    static const int DEG[5] = {1, 3, 4, 5, 6};
    static const char *TL[5] = {"T1", "T3", "T4", "T5", "T6"};
    sc taus[5];
    for (int k = 0; k < 5; k++) {
        rng_scalar(&rng, &taus[k]);
        sc ti;
        if (mode == 0) { sc xi; sc_from_u64(&xi, (u64)DEG[k]); v_poly6_eval(&ti, t6, &xi); }
        else ti = t6[DEG[k] - 1];
        sv[0] = ti; sv[1] = taus[k]; pv[0] = *g; pv[1] = *h;
        ge_ext T; msm_sc(&T, sv, pv, 2);
        ristretto_compress(po + 96 + 32 * k, &T);
        tr_append(&tr, TL[k], (mode == 0 && k == 2) ? po + 96 + 32 : po + 96 + 32 * k, 32);
    }
    /* ---- random_chall_x :425-432 ---- */
    sc x; tr_challenge_scalar(&tr, "x", &x);
    /* ---- blinding_values :434-476 ---- */
    sc *l = malloc(n * sizeof(sc)), *r = malloc(n * sizeof(sc)), *zero = calloc(n, sizeof(sc));
    v_poly3_eval(l, zero, l1, a_O, s_l, &x, n);
    v_poly3_eval(r, r0, r1, zero, r3, &x, n);
    sc that; v_inner_product(&that, l, r, n);
    sc tau_x = {{0, 0, 0, 0}}, xx, wvg, term;
    sc_mul(&xx, &x, &x);
    sc *wvq = malloc(Q * sizeof(sc));
    for (int k = 0; k < 5; k++) {
        sc xp; v_scalar_exp(&xp, &x, DEG[k]); sc_mul(&term, &taus[k], &xp); sc_add(&tau_x, &tau_x, &term);
        if (mode == 0 || k == 0) {   /* the reference recomputes mv_mult(W_V, gamma) inside each of its 5 terms */
            v_mv_mult(wvq, W_V, gamma, m, Q); v_inner_product(&wvg, z_q, wvq, Q); sc_mul(&wvg, &xx, &wvg);
        }
        if (mode == 0) sc_add(&tau_x, &tau_x, &wvg);
    }
    if (mode != 0) sc_add(&tau_x, &tau_x, &wvg);
    sc mu, xp3; v_scalar_exp(&xp3, &x, 3);
    sc_mul(&mu, &alpha, &x); sc_mul(&term, &beta, &xx); sc_add(&mu, &mu, &term); sc_mul(&term, &ro, &xp3); sc_add(&mu, &mu, &term);
    tr_append_scalar(&tr, "TX", &tau_x); tr_append_scalar(&tr, "mu", &mu);
    tr_append_vec_scalar(&tr, "l", l, n); tr_append_vec_scalar(&tr, "r", r, n); tr_append_scalar(&tr, "t", &that);
    sc_tobytes(po + 256, &tau_x); sc_tobytes(po + 288, &mu); sc_tobytes(po + 320, &that);
    memcpy(po + 352, l, n * 32); memcpy(po + 352 + 32 * n, r, n * 32);
    free(sv); free(pv); free(s_l); free(s_r); free(y_n); free(y_n_inv); free(z_q); free(z_W_R); free(z_W_L); free(l_in);
    free(l1); free(r0); free(r1); free(r3); free(tmp); free(tmp2); free(l); free(r); free(zero); free(wvq);
    if (!do_verify) return 1;
    return acp_verify(mode, n, Q, m, W_L, W_R, W_O, W_V, cv, g, h, G, H, po, V, V_enc, label, label_len);
}

/* PedersenGens::commit (weights.rs:58-61): v*B + r*B_blinding for m values */
void orc_commit_variables(const u8 *g_pt, const u8 *h_pt, const u8 *v, const u8 *gamma, size_t m, u8 *V_pts) {
    orc_init();
    for (size_t j = 0; j < m; j++) {
        sc s[2]; ge_ext p[2] = {*(const ge_ext *)g_pt, *(const ge_ext *)h_pt};
        memcpy(s[0].v, v + 32 * j, 32); memcpy(s[1].v, gamma + 32 * j, 32);
        msm_sc((ge_ext *)V_pts + j, s, p, 2);
    }
}
void orc_scalar_ops_selftest(const u8 *a32, const u8 *b32, const u8 *w64, u8 *out /* mul|add|sub|inv|wide = 160 B */) {
    sc a, b, r;
    sc_frombytes(&a, a32); sc_frombytes(&b, b32);
    sc_mul(&r, &a, &b); sc_tobytes(out, &r);
    sc_add(&r, &a, &b); sc_tobytes(out + 32, &r);
    sc_sub(&r, &a, &b); sc_tobytes(out + 64, &r);
    sc_invert(&r, &a); sc_tobytes(out + 96, &r);
    sc_from_wide(&r, w64); sc_tobytes(out + 128, &r);
}

/* ------------------------------------------------------------------ `fixed` mode (IPA) ---------- */
/* Restatement of bulletproofs 4.0.0 inner_product_proof.rs (create / verification_scalars / verify)
 * and of the R1CS glue around it, as described in oracle/ipa.py (the reference has no IPA; PARITY
 * UNPINNED, this file == oracle/ipa.py == the CUDA path).  The prover folds the generators explicitly
 * with 2-term vartime MSMs exactly like dalek; weights come as sparse (wire, constraint, coeff)
 * triples for W_L|W_R|W_O|W_V so that the 4096-card deck fits in memory. */
static size_t next_pow2_sz(size_t n) { size_t p = 1; while (p < n) p <<= 1; return p; }
static void v_std_powers(sc *out, const sc *x, size_t count, const sc *first) {
    sc cur = *first;
    for (size_t i = 0; i < count; i++) { out[i] = cur; sc_mul(&cur, &cur, x); }
}
/* out[wire] += coeff * z_q[constraint] over one matrix's triples */
static void v_sparse_vm(sc *out, size_t rows, const sc *z_q, const u32 *wire, const u32 *cons, const sc *coeff, size_t nnz) {
    memset(out, 0, rows * sizeof(sc));
    for (size_t e = 0; e < nnz; e++) { sc t; sc_mul(&t, &coeff[e], &z_q[cons[e]]); sc_add(&out[wire[e]], &out[wire[e]], &t); }
}
static int is_zero32(const u8 *b) { u8 o = 0; for (int i = 0; i < 32; i++) o |= b[i]; return o == 0; }

size_t orc_acp_fixed_proof_len(size_t n) {
    size_t np = next_pow2_sz(n), lg = 0; while (((size_t)1 << lg) < np) lg++;
    return 32 * (13 + 2 * lg);
}

/* G_pts, H_pts: next_pow2(n) generators each.  Returns 1 accept / 0 reject (or 1 when !do_verify). */
int orc_acp_fixed_prove_verify(size_t n, size_t Q, size_t m, const u32 nnz[4], const u32 *wire, const u32 *cons,
                               const u8 *coeffb, const u8 *cb, const u8 *g_pt, const u8 *h_pt, const u8 *G_pts,
                               const u8 *H_pts, const u8 *aLb, const u8 *aRb, const u8 *aOb, const u8 *gammab,
                               const u8 *V_pts, const u8 *V_enc, const u8 *seed32, const u8 *label, size_t label_len,
                               u8 *proof, int do_prove, int do_verify) {
    orc_init();
    const size_t np = next_pow2_sz(n);
    size_t lg = 0; while (((size_t)1 << lg) < np) lg++;
    const sc *coeff = (const sc *)coeffb, *cv = (const sc *)cb;
    const sc *a_L = (const sc *)aLb, *a_R = (const sc *)aRb, *a_O = (const sc *)aOb, *gamma = (const sc *)gammab;
    const ge_ext *g = (const ge_ext *)g_pt, *h = (const ge_ext *)h_pt, *G = (const ge_ext *)G_pts, *H = (const ge_ext *)H_pts;
    const ge_ext *V = (const ge_ext *)V_pts;
    const u32 *wr[4], *cn[4]; const sc *cf[4]; size_t off = 0;
    for (int k = 0; k < 4; k++) { wr[k] = wire + off; cn[k] = cons + off; cf[k] = coeff + off; off += nnz[k]; }
    const size_t big = 2 * np + m + 2 * lg + 16;
    sc *sv = malloc(big * sizeof(sc)); ge_ext *pv = malloc(big * sizeof(ge_ext));
    sc *y_n = malloc(np * sizeof(sc)), *y_n_inv = malloc(np * sizeof(sc)), *z_q = malloc(Q * sizeof(sc));
    sc *zWL = malloc(n * sizeof(sc)), *zWR = malloc(n * sizeof(sc)), *zWO = malloc(n * sizeof(sc)), *zWV = malloc(m * sizeof(sc));
    sc *l_in = malloc(n * sizeof(sc));
    const sc one = {{1, 0, 0, 0}};
    static const int DEG[5] = {1, 3, 4, 5, 6};
    static const char *TL[5] = {"T1", "T3", "T4", "T5", "T6"};
    u8 *po = proof;
    int result = 1;
    if (do_prove) {
        rng_t rng; memcpy(rng.key, seed32, 32); rng.ctr = 0;
        strobe tr; tr_new(&tr, label, label_len);
        { u8 nb[8]; for (int i = 0; i < 8; i++) nb[i] = (u8)((u64)n >> (8 * i)); tr_append(&tr, "dom-sep", (const u8 *)"acp v1", 6); tr_append(&tr, "n", nb, 8); }
        tr_append_commitments(&tr, V, V_enc, m);
        sc alpha, beta, ro; rng_scalar(&rng, &alpha); rng_scalar(&rng, &beta); rng_scalar(&rng, &ro);
        ge_ext A_I, A_O, S;
        sv[0] = alpha; pv[0] = *h; memcpy(sv + 1, a_L, n * 32); memcpy(pv + 1, G, n * sizeof(ge_ext));
        memcpy(sv + 1 + n, a_R, n * 32); memcpy(pv + 1 + n, H, n * sizeof(ge_ext));
        msm_sc(&A_I, sv, pv, 1 + 2 * n);
        sv[0] = beta; memcpy(sv + 1, a_O, n * 32);
        msm_sc(&A_O, sv, pv, 1 + n);
        sc *s_l = malloc(n * sizeof(sc)), *s_r = malloc(n * sizeof(sc));
        for (size_t i = 0; i < n; i++) rng_scalar(&rng, &s_l[i]);
        for (size_t i = 0; i < n; i++) rng_scalar(&rng, &s_r[i]);
        sv[0] = ro; memcpy(sv + 1, s_l, n * 32); memcpy(sv + 1 + n, s_r, n * 32);
        msm_sc(&S, sv, pv, 1 + 2 * n);
        ristretto_compress(po, &A_I); ristretto_compress(po + 32, &A_O); ristretto_compress(po + 64, &S);
        tr_append(&tr, "A_I", po, 32); tr_append(&tr, "A_O", po + 32, 32); tr_append(&tr, "S", po + 64, 32);
        sc y, z, y_inv; tr_challenge_scalar(&tr, "y", &y); tr_challenge_scalar(&tr, "z", &z);
        sc_invert(&y_inv, &y);
        v_std_powers(y_n, &y, np, &one); v_std_powers(y_n_inv, &y_inv, np, &one); v_std_powers(z_q, &z, Q, &z);
        v_sparse_vm(zWL, n, z_q, wr[0], cn[0], cf[0], nnz[0]);
        v_sparse_vm(zWR, n, z_q, wr[1], cn[1], cf[1], nnz[1]);
        v_sparse_vm(zWO, n, z_q, wr[2], cn[2], cf[2], nnz[2]);
        v_sparse_vm(zWV, m, z_q, wr[3], cn[3], cf[3], nnz[3]);
        v_hadamard(l_in, y_n_inv, zWR, n);
        sc *l1 = malloc(n * sizeof(sc)), *r0 = malloc(n * sizeof(sc)), *r1 = malloc(n * sizeof(sc)), *r3 = malloc(n * sizeof(sc));
        for (size_t i = 0; i < n; i++) {
            sc t;
            sc_add(&l1[i], &a_L[i], &l_in[i]);
            sc_sub(&r0[i], &zWO[i], &y_n[i]);
            sc_mul(&t, &y_n[i], &a_R[i]); sc_add(&r1[i], &t, &zWL[i]);
            sc_mul(&r3[i], &y_n[i], &s_r[i]);
        }
        sc t6[6], d1, d2;
        v_inner_product(&t6[0], l1, r0, n);
        v_inner_product(&d1, l1, r1, n); v_inner_product(&d2, a_O, r0, n); sc_add(&t6[1], &d1, &d2);
        v_inner_product(&d1, a_O, r1, n); v_inner_product(&d2, s_l, r0, n); sc_add(&t6[2], &d1, &d2);
        v_inner_product(&d1, l1, r3, n); v_inner_product(&d2, s_l, r1, n); sc_add(&t6[3], &d1, &d2);
        v_inner_product(&t6[4], a_O, r3, n);
        v_inner_product(&t6[5], s_l, r3, n);
        sc taus[5];
        for (int k = 0; k < 5; k++) {
            rng_scalar(&rng, &taus[k]);
            sv[0] = t6[DEG[k] - 1]; sv[1] = taus[k]; pv[0] = *g; pv[1] = *h;
            ge_ext T; msm_sc(&T, sv, pv, 2);
            ristretto_compress(po + 96 + 32 * k, &T);
            tr_append(&tr, TL[k], po + 96 + 32 * k, 32);
        }
        sc x; tr_challenge_scalar(&tr, "x", &x);
        sc *a = calloc(np, sizeof(sc)), *b = malloc(np * sizeof(sc)), *zero = calloc(n, sizeof(sc));
        v_poly3_eval(a, zero, l1, a_O, s_l, &x, n);
        v_poly3_eval(b, r0, r1, zero, r3, &x, n);
        for (size_t i = n; i < np; i++) sc_neg(&b[i], &y_n[i]);
        sc that; v_inner_product(&that, a, b, np);
        sc tau_x, xx, term, wvg;
        sc_mul(&xx, &x, &x);
        v_inner_product(&wvg, zWV, gamma, m);     /* <z_q, W_V gamma> = <z W_V, gamma> */
        sc_mul(&tau_x, &xx, &wvg);
        for (int k = 0; k < 5; k++) { sc xp; v_scalar_exp(&xp, &x, DEG[k]); sc_mul(&term, &taus[k], &xp); sc_add(&tau_x, &tau_x, &term); }
        sc mu, xp3; sc_mul(&xp3, &xx, &x);
        sc_mul(&mu, &alpha, &x); sc_mul(&term, &beta, &xx); sc_add(&mu, &mu, &term); sc_mul(&term, &ro, &xp3); sc_add(&mu, &mu, &term);
        tr_append_scalar(&tr, "t_x", &that); tr_append_scalar(&tr, "t_x_blinding", &tau_x); tr_append_scalar(&tr, "e_blinding", &mu);
        sc_tobytes(po + 256, &that); sc_tobytes(po + 288, &tau_x); sc_tobytes(po + 320, &mu);
        sc w; tr_challenge_scalar(&tr, "w", &w);
        ge_ext Qp; sv[0] = w; pv[0] = *g; msm_sc(&Qp, sv, pv, 1);
        /* InnerProductProof::create with G_factors = 1, H_factors = y^-n */
        { u8 nb[8]; for (int i = 0; i < 8; i++) nb[i] = (u8)((u64)np >> (8 * i)); tr_append(&tr, "dom-sep", (const u8 *)"ipp v1", 6); tr_append(&tr, "n", nb, 8); }
        ge_ext *Gf = malloc(np * sizeof(ge_ext)), *Hf = malloc(np * sizeof(ge_ext));
        memcpy(Gf, G, np * sizeof(ge_ext)); memcpy(Hf, H, np * sizeof(ge_ext));
        size_t cur = np, round = 0;
        while (cur != 1) {
            cur /= 2;
            const int first = round == 0;
            sc c_L, c_R;
            v_inner_product(&c_L, a, b + cur, cur); v_inner_product(&c_R, a + cur, b, cur);
            /* L = <a_L o gf_R, G_R> + <b_R o hf_L, H_L> + c_L Q */
            for (size_t i = 0; i < cur; i++) {
                sv[i] = a[i]; pv[i] = Gf[cur + i];
                if (first) sc_mul(&sv[cur + i], &b[cur + i], &y_n_inv[i]); else sv[cur + i] = b[cur + i];
                pv[cur + i] = Hf[i];
            }
            sv[2 * cur] = c_L; pv[2 * cur] = Qp;
            ge_ext Lp, Rp; msm_sc(&Lp, sv, pv, 2 * cur + 1);
            for (size_t i = 0; i < cur; i++) {
                sv[i] = a[cur + i]; pv[i] = Gf[i];
                if (first) sc_mul(&sv[cur + i], &b[i], &y_n_inv[cur + i]); else sv[cur + i] = b[i];
                pv[cur + i] = Hf[cur + i];
            }
            sv[2 * cur] = c_R;
            msm_sc(&Rp, sv, pv, 2 * cur + 1);
            u8 *lr = po + 352 + 64 * round;
            ristretto_compress(lr, &Lp); ristretto_compress(lr + 32, &Rp);
            tr_append(&tr, "L", lr, 32); tr_append(&tr, "R", lr + 32, 32);
            sc u, u_inv; tr_challenge_scalar(&tr, "u", &u); sc_invert(&u_inv, &u);
            for (size_t i = 0; i < cur; i++) {
                sc t1, t2;
                sc_mul(&t1, &a[i], &u); sc_mul(&t2, &u_inv, &a[cur + i]); sc_add(&a[i], &t1, &t2);
                sc_mul(&t1, &b[i], &u_inv); sc_mul(&t2, &u, &b[cur + i]); sc_add(&b[i], &t1, &t2);
                sc s2[2]; ge_ext p2[2];
                s2[0] = u_inv; s2[1] = u; p2[0] = Gf[i]; p2[1] = Gf[cur + i];
                msm_sc(&Gf[i], s2, p2, 2);
                if (first) { sc_mul(&s2[0], &u, &y_n_inv[i]); sc_mul(&s2[1], &u_inv, &y_n_inv[cur + i]); }
                else { s2[0] = u; s2[1] = u_inv; }
                p2[0] = Hf[i]; p2[1] = Hf[cur + i];
                msm_sc(&Hf[i], s2, p2, 2);
            }
            round++;
        }
        sc_tobytes(po + 352 + 64 * lg, &a[0]); sc_tobytes(po + 384 + 64 * lg, &b[0]);
        free(s_l); free(s_r); free(l1); free(r0); free(r1); free(r3); free(a); free(b); free(zero); free(Gf); free(Hf);
    }
    if (do_verify) {
        ge_ext pts8[8], *Lp = malloc((lg + 1) * sizeof(ge_ext)), *Rp = malloc((lg + 1) * sizeof(ge_ext));
        for (int k = 0; k < 8 && result == 1; k++) if (!ristretto_decompress(&pts8[k], po + 32 * k)) result = 0;
        sc that, tau_x, mu, pa, pb;
        sc_from_bytes_mod_order(&that, po + 256); sc_from_bytes_mod_order(&tau_x, po + 288); sc_from_bytes_mod_order(&mu, po + 320);
        sc_from_bytes_mod_order(&pa, po + 352 + 64 * lg); sc_from_bytes_mod_order(&pb, po + 384 + 64 * lg);
        strobe tr; tr_new(&tr, label, label_len);
        { u8 nb[8]; for (int i = 0; i < 8; i++) nb[i] = (u8)((u64)n >> (8 * i)); tr_append(&tr, "dom-sep", (const u8 *)"acp v1", 6); tr_append(&tr, "n", nb, 8); }
        tr_append_commitments(&tr, V, V_enc, m);
        tr_append(&tr, "A_I", po, 32); tr_append(&tr, "A_O", po + 32, 32); tr_append(&tr, "S", po + 64, 32);
        sc y, z, x, w, y_inv; tr_challenge_scalar(&tr, "y", &y); tr_challenge_scalar(&tr, "z", &z);
        for (int k = 0; k < 5; k++) tr_append(&tr, TL[k], po + 96 + 32 * k, 32);
        tr_challenge_scalar(&tr, "x", &x);
        tr_append_scalar(&tr, "t_x", &that); tr_append_scalar(&tr, "t_x_blinding", &tau_x); tr_append_scalar(&tr, "e_blinding", &mu);
        tr_challenge_scalar(&tr, "w", &w);
        { u8 nb[8]; for (int i = 0; i < 8; i++) nb[i] = (u8)((u64)np >> (8 * i)); tr_append(&tr, "dom-sep", (const u8 *)"ipp v1", 6); tr_append(&tr, "n", nb, 8); }
        sc *u_sq = malloc((lg + 1) * sizeof(sc)), *u_inv_sq = malloc((lg + 1) * sizeof(sc)), *s = malloc(np * sizeof(sc));
        sc allinv = one;
        for (size_t j = 0; j < lg; j++) {
            const u8 *lr = po + 352 + 64 * j;
            if (is_zero32(lr) || is_zero32(lr + 32)) result = 0;           /* validate_and_append_point */
            if (result == 1 && (!ristretto_decompress(&Lp[j], lr) || !ristretto_decompress(&Rp[j], lr + 32))) result = 0;
            tr_append(&tr, "L", lr, 32); tr_append(&tr, "R", lr + 32, 32);
            sc u, ui; tr_challenge_scalar(&tr, "u", &u); sc_invert(&ui, &u);
            sc_mul(&u_sq[j], &u, &u); sc_mul(&u_inv_sq[j], &ui, &ui); sc_mul(&allinv, &allinv, &ui);
        }
        if (result == 1) {
            s[0] = allinv;
            for (size_t i = 1; i < np; i++) {
                size_t lg_i = 0; while (((size_t)2 << lg_i) <= i) lg_i++;
                sc_mul(&s[i], &s[i - ((size_t)1 << lg_i)], &u_sq[(lg - 1) - lg_i]);
            }
            sc_invert(&y_inv, &y);
            v_std_powers(y_n, &y, np, &one); v_std_powers(y_n_inv, &y_inv, np, &one); v_std_powers(z_q, &z, Q, &z);
            v_sparse_vm(zWL, n, z_q, wr[0], cn[0], cf[0], nnz[0]);
            v_sparse_vm(zWR, n, z_q, wr[1], cn[1], cf[1], nnz[1]);
            v_sparse_vm(zWO, n, z_q, wr[2], cn[2], cf[2], nnz[2]);
            v_sparse_vm(zWV, m, z_q, wr[3], cn[3], cf[3], nnz[3]);
            v_hadamard(l_in, y_n_inv, zWR, n);
            sc sigma, zc, xx, g_exp; v_inner_product(&sigma, l_in, zWL, n);
            sc_mul(&xx, &x, &x);
            v_inner_product(&zc, z_q, cv, Q); sc_add(&zc, &zc, &sigma); sc_mul(&g_exp, &xx, &zc);
            /* check 2 */
            sv[0] = g_exp; pv[0] = *g;
            for (size_t j = 0; j < m; j++) { sc_mul(&sv[1 + j], &xx, &zWV[j]); pv[1 + j] = V[j]; }
            for (int k = 0; k < 5; k++) { v_scalar_exp(&sv[1 + m + k], &x, DEG[k]); pv[1 + m + k] = pts8[3 + k]; }
            ge_ext cand, lhs; msm_sc(&cand, sv, pv, 1 + m + 5);
            sv[0] = that; sv[1] = tau_x; pv[0] = *g; pv[1] = *h; msm_sc(&lhs, sv, pv, 2);
            if (!ge_ristretto_eq(&lhs, &cand)) result = 0;
        }
        if (result == 1) {
            /* check 3 + InnerProductProof::verify: P + t_hat Q == a<s,G> + b<s^-1 o y^-n,H> + ab Q - sum u^2 L - sum u^-2 R */
            sc xx, xxx, t; sc_mul(&xx, &x, &x); sc_mul(&xxx, &xx, &x);
            size_t o = 0;
            sv[o] = x; pv[o++] = pts8[0]; sv[o] = xx; pv[o++] = pts8[1]; sv[o] = xxx; pv[o++] = pts8[2];
            sc_neg(&sv[o], &mu); pv[o++] = *h;
            for (size_t i = 0; i < n; i++) { sc_mul(&sv[o], &x, &l_in[i]); pv[o++] = G[i]; }
            for (size_t i = 0; i < np; i++) {
                sc inner = {{0, 0, 0, 0}};
                if (i < n) { sc_mul(&inner, &x, &zWL[i]); sc_add(&inner, &inner, &zWO[i]); }
                sc_sub(&inner, &inner, &y_n[i]);
                sc_mul(&sv[o], &y_n_inv[i], &inner); pv[o++] = H[i];
            }
            sc_mul(&sv[o], &that, &w); pv[o++] = *g;       /* t_hat Q, Q = w g */
            ge_ext P; msm_sc(&P, sv, pv, o);
            o = 0;
            for (size_t i = 0; i < np; i++) { sc_mul(&sv[o], &pa, &s[i]); pv[o++] = G[i]; }
            for (size_t i = 0; i < np; i++) { sc_mul(&t, &pb, &s[np - 1 - i]); sc_mul(&sv[o], &t, &y_n_inv[i]); pv[o++] = H[i]; }
            sc_mul(&t, &pa, &pb); sc_mul(&sv[o], &t, &w); pv[o++] = *g;
            for (size_t j = 0; j < lg; j++) { sc_neg(&sv[o], &u_sq[j]); pv[o++] = Lp[j]; }
            for (size_t j = 0; j < lg; j++) { sc_neg(&sv[o], &u_inv_sq[j]); pv[o++] = Rp[j]; }
            ge_ext rhs; msm_sc(&rhs, sv, pv, o);
            if (!ge_ristretto_eq(&P, &rhs)) result = 0;
        }
        free(Lp); free(Rp); free(u_sq); free(u_inv_sq); free(s);
    }
    free(sv); free(pv); free(y_n); free(y_n_inv); free(z_q); free(zWL); free(zWR); free(zWO); free(zWV); free(l_in);
    return result;
}
