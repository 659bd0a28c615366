// sc25519.cuh - scalar arithmetic mod l = 2^252 + 27742317777372353535851937790883648493 (sm_100a).
//
// Replaces curve25519-dalek-ng 4.1.1 `Scalar` / `Scalar52` (backend/serial/u64/scalar.rs) under the
// reference's scalar-vector operators: util.rs:6-94 (hadamard_V, vm_mult, mv_mult, exp_iter,
// scalar_exp, inner_product), poly.rs:14-76, circuit_lib.rs:269-291,313-356,441-462 and
// `Scalar::from_bytes_mod_order_wide` (transcript_protocol.rs:62-67).
//
// Representation: 8 x 32-bit limbs, canonical (< l) in memory - the same bytes dalek keeps.
// Multiplication is Montgomery with R = 2^256: mont(a, b) = a*b/R.  sc_mul() of two standard-form
// values is mont(mont(a, b), R^2); chains may stay in Montgomery form (sc_to_mont/sc_from_mont).
// Every result is fully reduced, so any evaluation order gives identical bytes.
#pragma once
#include "mp256.cuh"
#include <stdint.h>

#define SC_INLINE __device__ __forceinline__

struct sc {
    uint32_t v[8];
};

__device__ __constant__ const uint32_t SC_L[8] = {0x5cf5d3edu, 0x5812631au, 0xa2f79cd6u, 0x14def9deu,
                                                  0x00000000u, 0x00000000u, 0x00000000u, 0x10000000u};
// R mod l, R^2 mod l (R = 2^256), -l^{-1} mod 2^32
__device__ __constant__ const uint32_t SC_R[8] = {0x8d98951du, 0xd6ec3174u, 0x737dcf70u, 0xc6ef5bf4u,
                                                  0xfffffffeu, 0xffffffffu, 0xffffffffu, 0x0fffffffu};
__device__ __constant__ const uint32_t SC_R2[8] = {0x449c0f01u, 0xa40611e3u, 0x68859347u, 0xd00e1ba7u,
                                                   0x17f5be65u, 0xceec73d2u, 0x7c309a3du, 0x0399411bu};
#define SC_NPRIME 0x12547e1bu

SC_INLINE void sc_set0(sc &r) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = 0;
}
SC_INLINE void sc_set_u32(sc &r, uint32_t x) {
    sc_set0(r);
    r.v[0] = x;
}
SC_INLINE void sc_const(sc &r, const uint32_t *c) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = c[i];
}
SC_INLINE void sc_load(sc &r, const uint32_t *p) {  // 16-byte aligned
    uint4 lo = *reinterpret_cast<const uint4 *>(p);
    uint4 hi = *reinterpret_cast<const uint4 *>(p + 4);
    r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w;
    r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
}
SC_INLINE void sc_store(uint32_t *p, const sc &a) {
    *reinterpret_cast<uint4 *>(p) = make_uint4(a.v[0], a.v[1], a.v[2], a.v[3]);
    *reinterpret_cast<uint4 *>(p + 4) = make_uint4(a.v[4], a.v[5], a.v[6], a.v[7]);
}
SC_INLINE bool sc_is_zero(const sc &a) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) o |= a.v[i];
    return o == 0;
}
SC_INLINE bool sc_eq(const sc &a, const sc &b) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) o |= a.v[i] ^ b.v[i];
    return o == 0;
}

// r = a - l if a >= l else a      (a < 2l)
SC_INLINE void sc_cond_sub_l(sc &r, const uint32_t a[8], uint32_t top /* bit 256 of a */) {
    uint32_t d[8];
    long long borrow = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        long long t = (long long)a[i] - (long long)SC_L[i] + borrow;
        d[i] = (uint32_t)t;
        borrow = t >> 32;
    }
    bool ge = (top != 0) || (borrow == 0);
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = ge ? d[i] : a[i];
}

SC_INLINE void sc_add(sc &r, const sc &a, const sc &b) {  // canonical inputs
    uint32_t s[8];
    unsigned long long c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        c += (unsigned long long)a.v[i] + b.v[i];
        s[i] = (uint32_t)c;
        c >>= 32;
    }
    sc_cond_sub_l(r, s, (uint32_t)c);
}
SC_INLINE void sc_sub(sc &r, const sc &a, const sc &b) {  // canonical inputs
    uint32_t d[8];
    long long borrow = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        long long t = (long long)a.v[i] - (long long)b.v[i] + borrow;
        d[i] = (uint32_t)t;
        borrow = t >> 32;
    }
    // add l back if negative
    unsigned long long c = 0;
    uint32_t mask = borrow ? 0xffffffffu : 0u;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        c += (unsigned long long)d[i] + (SC_L[i] & mask);
        r.v[i] = (uint32_t)c;
        c >>= 32;
    }
}
SC_INLINE void sc_neg(sc &r, const sc &a) {
    sc z;
    sc_set0(z);
    sc_sub(r, z, a);
}

// Montgomery product: r = a * b / 2^256 mod l.  Needs a * b < l * 2^256 (one operand < l suffices).
// t = a*b (64 wide multiply-adds, mp_mul8); q = t_lo * (-l^-1) mod 2^256 (36); r = (t + q*l) / 2^256.  With
// l = 2^252 + delta, q*l = q*delta (8 x 4 limbs) + (q << 252); the low half of t + q*l is 0 mod 2^256 by
// construction and carries out exactly when t_lo != 0, so only the high half is assembled.  No word-serial
// dependency (the classic per-limb m_i = t_i * n' loop is one chain of ~100 dependent steps).
__device__ __constant__ const uint32_t SC_NP[8] = {0x12547e1bu, 0xd2b51da3u, 0xfdba84ffu, 0xb1a206f2u,
                                                   0xffa36beau, 0x14e75438u, 0x6fe91836u, 0x9db6c6f2u};
// sc_mont_reduce(r, t) = t / 2^256 mod l for any t < l * 2^256 (the reduction half of sc_mont): (t + q*l) / 2^256 <
// t / 2^256 + l < 2l, so one conditional subtraction makes it canonical.  A sum of up to 15 products of canonical
// scalars stays below that bound, so sums of products can be accumulated as 512-bit integers (sc_mac) and reduced once.
// SC_MAC_MAX is that count: 15 (l-1)^2 < l * 2^256 <= 16 (l-1)^2, so a 16th product of large operands can exceed it.
#define SC_MAC_MAX 15
#pragma nv_diag_suppress 550   // `dummy` receives a limb whose carry-out is all that matters
SC_INLINE void sc_mont_reduce(sc &r, const uint32_t t[16]) {
    uint32_t qf[8], u[12], np[8], dl[4];
#pragma unroll
    for (int i = 0; i < 8; i++) np[i] = SC_NP[i];
    mp_mul8_lo(qf, t, np);            // q = t_lo * (-l^-1) mod 2^256: 36 products
#pragma unroll
    for (int i = 0; i < 4; i++) dl[i] = SC_L[i];
    mp_mul8<4>(u, qf, dl);            // q * delta, 12 limbs
    // h = high half of (q*delta + (q << 252)): limbs 8..15, with the carry out of limb 7
    uint32_t w[9];                    // (q << 28) occupies limbs 7..15
    w[0] = qf[0] << 28;
#pragma unroll
    for (int k = 1; k < 8; k++) w[k] = (qf[k] << 28) | (qf[k - 1] >> 4);
    w[8] = qf[7] >> 4;
    uint32_t nz = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) nz |= t[i];
    nz = nz ? 0xffffffffu : 0u;
    uint32_t h[8], dummy = 0;
    asm("add.cc.u32 %8, %9, %10;\n\t"          // limb 7: only the carry matters
        "addc.cc.u32 %0, %11, %15;\n\t"
        "addc.cc.u32 %1, %12, %16;\n\t"
        "addc.cc.u32 %2, %13, %17;\n\t"
        "addc.cc.u32 %3, %14, %18;\n\t"
        "addc.cc.u32 %4, %19, 0;\n\t"
        "addc.cc.u32 %5, %20, 0;\n\t"
        "addc.cc.u32 %6, %21, 0;\n\t"
        "addc.u32 %7, %22, 0;"
        : "=&r"(h[0]), "=&r"(h[1]), "=&r"(h[2]), "=&r"(h[3]), "=&r"(h[4]), "=&r"(h[5]), "=&r"(h[6]), "=&r"(h[7]),
          "=&r"(dummy)
        : "r"(u[7]), "r"(w[0]), "r"(u[8]), "r"(u[9]), "r"(u[10]), "r"(u[11]), "r"(w[1]), "r"(w[2]), "r"(w[3]),
          "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]), "r"(w[8]));
    // s = t_hi + h + (t_lo != 0): the carry-in is produced by nz + nz (0xffffffff + 0xffffffff carries)
    uint32_t s8[8];
    asm("add.cc.u32 %8, %9, %9;\n\t"
        "addc.cc.u32 %0, %10, %18;\n\t"
        "addc.cc.u32 %1, %11, %19;\n\t"
        "addc.cc.u32 %2, %12, %20;\n\t"
        "addc.cc.u32 %3, %13, %21;\n\t"
        "addc.cc.u32 %4, %14, %22;\n\t"
        "addc.cc.u32 %5, %15, %23;\n\t"
        "addc.cc.u32 %6, %16, %24;\n\t"
        "addc.u32 %7, %17, %25;"
        : "=&r"(s8[0]), "=&r"(s8[1]), "=&r"(s8[2]), "=&r"(s8[3]), "=&r"(s8[4]), "=&r"(s8[5]), "=&r"(s8[6]),
          "=&r"(s8[7]), "=&r"(dummy)
        : "r"(nz), "r"(t[8]), "r"(t[9]), "r"(t[10]), "r"(t[11]), "r"(t[12]), "r"(t[13]), "r"(t[14]), "r"(t[15]),
          "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]), "r"(h[4]), "r"(h[5]), "r"(h[6]), "r"(h[7]));
    sc_cond_sub_l(r, s8, 0);          // s < 2l < 2^254
}
#pragma nv_diag_default 550
SC_INLINE void sc_mont(sc &r, const sc &a, const sc &b) {
    uint32_t t[16];
    mp_mul8<8>(t, a.v, b.v);
    sc_mont_reduce(r, t);
}
// t += a * b as a 512-bit integer (64 wide multiply-adds and one 16-limb carry chain; no reduction)
SC_INLINE void sc_mac(uint32_t t[16], const sc &a, const sc &b) {
    uint32_t p[16];
    mp_mul8<8>(p, a.v, b.v);
    asm("add.cc.u32 %0, %0, %16;\n\t"
        "addc.cc.u32 %1, %1, %17;\n\t"
        "addc.cc.u32 %2, %2, %18;\n\t"
        "addc.cc.u32 %3, %3, %19;\n\t"
        "addc.cc.u32 %4, %4, %20;\n\t"
        "addc.cc.u32 %5, %5, %21;\n\t"
        "addc.cc.u32 %6, %6, %22;\n\t"
        "addc.cc.u32 %7, %7, %23;\n\t"
        "addc.cc.u32 %8, %8, %24;\n\t"
        "addc.cc.u32 %9, %9, %25;\n\t"
        "addc.cc.u32 %10, %10, %26;\n\t"
        "addc.cc.u32 %11, %11, %27;\n\t"
        "addc.cc.u32 %12, %12, %28;\n\t"
        "addc.cc.u32 %13, %13, %29;\n\t"
        "addc.cc.u32 %14, %14, %30;\n\t"
        "addc.u32 %15, %15, %31;"
        : "+&r"(t[0]), "+&r"(t[1]), "+&r"(t[2]), "+&r"(t[3]), "+&r"(t[4]), "+&r"(t[5]), "+&r"(t[6]), "+&r"(t[7]),
          "+&r"(t[8]), "+&r"(t[9]), "+&r"(t[10]), "+&r"(t[11]), "+&r"(t[12]), "+&r"(t[13]), "+&r"(t[14]), "+&r"(t[15])
        : "r"(p[0]), "r"(p[1]), "r"(p[2]), "r"(p[3]), "r"(p[4]), "r"(p[5]), "r"(p[6]), "r"(p[7]),
          "r"(p[8]), "r"(p[9]), "r"(p[10]), "r"(p[11]), "r"(p[12]), "r"(p[13]), "r"(p[14]), "r"(p[15]));
}

SC_INLINE void sc_to_mont(sc &r, const sc &a) {
    sc k;
    sc_const(k, SC_R2);
    sc_mont(r, a, k);
}
SC_INLINE void sc_from_mont(sc &r, const sc &a) {
    sc one;
    sc_set_u32(one, 1);
    sc_mont(r, a, one);
}
// standard-form product a * b mod l
SC_INLINE void sc_mul(sc &r, const sc &a, const sc &b) {
    sc t, k;
    sc_mont(t, a, b);
    sc_const(k, SC_R2);
    sc_mont(r, t, k);
}
static __device__ __noinline__ void sc_mul_noinline(sc &r, const sc &a, const sc &b) { sc_mul(r, a, b); }
static __device__ __noinline__ void sc_mont_noinline(sc &r, const sc &a, const sc &b) { sc_mont(r, a, b); }

// Scalar::from_bytes_mod_order_wide: 512-bit little-endian value mod l
SC_INLINE void sc_from_wide(sc &r, const uint32_t w[16]) {
    sc lo, hi, k, a, b;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        lo.v[i] = w[i];
        hi.v[i] = w[8 + i];
    }
    sc_const(k, SC_R);
    sc_mont(a, lo, k);   // lo * R / R = lo mod l
    sc_const(k, SC_R2);
    sc_mont(b, hi, k);   // hi * R^2 / R = hi * 2^256 mod l
    sc_add(r, a, b);
}
// any 256-bit value -> canonical (Scalar::from_bytes_mod_order)
SC_INLINE void sc_reduce256(sc &r, const sc &a) {
    sc k;
    sc_const(k, SC_R);
    sc_mont(r, a, k);
}

// 8-limb helpers for the inversion below (one carry chain each)
SC_INLINE uint32_t sc_sub8(uint32_t *r, const uint32_t *a, const uint32_t *b) {   // r = a - b, returns the borrow (0/1)
    uint32_t bw;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7]), "=&r"(bw)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    return bw & 1u;
}
SC_INLINE void sc_add8_masked(uint32_t *r, const uint32_t *a, const uint32_t *b, uint32_t mask) {   // r = a + (b & mask)
    asm("add.cc.u32 %0, %8, %16;\n\t"
        "addc.cc.u32 %1, %9, %17;\n\t"
        "addc.cc.u32 %2, %10, %18;\n\t"
        "addc.cc.u32 %3, %11, %19;\n\t"
        "addc.cc.u32 %4, %12, %20;\n\t"
        "addc.cc.u32 %5, %13, %21;\n\t"
        "addc.cc.u32 %6, %14, %22;\n\t"
        "addc.u32 %7, %15, %23;"
        : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0] & mask), "r"(b[1] & mask), "r"(b[2] & mask), "r"(b[3] & mask), "r"(b[4] & mask), "r"(b[5] & mask),
          "r"(b[6] & mask), "r"(b[7] & mask));
}

// r = a^-1 mod l (standard form in and out); 0 -> 0, like dalek's Scalar::invert (circuit_lib.rs:273-275), which
// raises to l - 2: 253 squarings + 67 multiplications, one dependent chain (~270 us for a lone warp).  Inversion
// sits on the critical path of every proof (y^-1 before the power chains, u_j^-1 in every inner-product round), so it
// is done by division steps instead (Bernstein-Yang "safegcd", in the batched form of libsecp256k1's modinv32):
// 20 batches of 30 divsteps; a batch runs on the low 30 bits of f and g alone (about ten plain 32-bit instructions
// per step, branch-free) and yields a 2 x 2 matrix of 31-bit entries, which is then applied once to the full f, g
// (exact division by 2^30) and to d, e modulo l (division by 2^30 made exact by adding the right multiple of l):
// values as nine signed 30-bit limbs, 64-bit accumulators.  600 >= 590 divsteps always bring g to 0 for inputs
// below 2^256, leaving f = +-1 and d = +-a^-1 (d = 0 for a = 0).  ~10 K instructions instead of the ~50 K of the
// round-1 bit-serial binary GCD (508 steps of 8-limb operations): 76 -> ~20 us for a lone thread.
#define SC_INV_M30 0x3fffffff
struct sc_s30 { int32_t v[9]; };
__device__ __constant__ const int32_t SC_L30[9] = {485872621, 541690985, 796511589, 935229352, 20, 0, 0, 0, 4096};
#define SC_L_INV30 766214629u   // l^-1 mod 2^30
SC_INLINE int32_t sc_divsteps_30(int32_t zeta, uint32_t f0, uint32_t g0, int32_t t[4]) {
    uint32_t u = 1, v = 0, q = 0, r = 1, f = f0, g = g0;
#pragma unroll 1
    for (int i = 0; i < 30; i++) {
        uint32_t mask1 = (uint32_t)(zeta >> 31);            // zeta < 0
        const uint32_t mask2 = 0u - (g & 1u);               // g odd
        const uint32_t x = (f ^ mask1) - mask1, y = (u ^ mask1) - mask1, z = (v ^ mask1) - mask1;
        g += x & mask2;
        q += y & mask2;
        r += z & mask2;
        mask1 &= mask2;
        zeta = (int32_t)((uint32_t)zeta ^ mask1) - 1;
        f += g & mask1;
        u += q & mask1;
        v += r & mask1;
        g >>= 1;
        u <<= 1;
        v <<= 1;
    }
    t[0] = (int32_t)u; t[1] = (int32_t)v; t[2] = (int32_t)q; t[3] = (int32_t)r;
    return zeta;
}
SC_INLINE void sc_update_fg_30(sc_s30 &f, sc_s30 &g, const int32_t t[4]) {
    const int32_t u = t[0], v = t[1], q = t[2], r = t[3];
    long long cf = (long long)u * f.v[0] + (long long)v * g.v[0];
    long long cg = (long long)q * f.v[0] + (long long)r * g.v[0];
    cf >>= 30;
    cg >>= 30;
#pragma unroll
    for (int i = 1; i < 9; i++) {
        cf += (long long)u * f.v[i] + (long long)v * g.v[i];
        cg += (long long)q * f.v[i] + (long long)r * g.v[i];
        f.v[i - 1] = (int32_t)cf & SC_INV_M30; cf >>= 30;
        g.v[i - 1] = (int32_t)cg & SC_INV_M30; cg >>= 30;
    }
    f.v[8] = (int32_t)cf;
    g.v[8] = (int32_t)cg;
}
SC_INLINE void sc_update_de_30(sc_s30 &d, sc_s30 &e, const int32_t t[4]) {
    const int32_t u = t[0], v = t[1], q = t[2], r = t[3];
    const int32_t sd = d.v[8] >> 31, se = e.v[8] >> 31;
    int32_t md = (u & sd) + (v & se), me = (q & sd) + (r & se);
    long long cd = (long long)u * d.v[0] + (long long)v * e.v[0];
    long long ce = (long long)q * d.v[0] + (long long)r * e.v[0];
    md -= (int32_t)((SC_L_INV30 * (uint32_t)cd + (uint32_t)md) & SC_INV_M30);
    me -= (int32_t)((SC_L_INV30 * (uint32_t)ce + (uint32_t)me) & SC_INV_M30);
    cd += (long long)SC_L30[0] * md;
    ce += (long long)SC_L30[0] * me;
    cd >>= 30;
    ce >>= 30;
#pragma unroll
    for (int i = 1; i < 9; i++) {
        cd += (long long)u * d.v[i] + (long long)v * e.v[i] + (long long)SC_L30[i] * md;
        ce += (long long)q * d.v[i] + (long long)r * e.v[i] + (long long)SC_L30[i] * me;
        d.v[i - 1] = (int32_t)cd & SC_INV_M30; cd >>= 30;
        e.v[i - 1] = (int32_t)ce & SC_INV_M30; ce >>= 30;
    }
    d.v[8] = (int32_t)cd;
    e.v[8] = (int32_t)ce;
}
static __device__ __noinline__ void sc_invert(sc &r, const sc &a) {
    sc_s30 d, e, f, g;
#pragma unroll
    for (int i = 0; i < 9; i++) { d.v[i] = 0; e.v[i] = 0; f.v[i] = SC_L30[i]; }
    e.v[0] = 1;
#pragma unroll
    for (int i = 0; i < 9; i++) {   // 8 x 32 bits -> 9 x 30 bits
        const int bit = 30 * i, limb = bit >> 5, sh = bit & 31;
        unsigned long long w = a.v[limb];
        if (limb + 1 < 8) w |= (unsigned long long)a.v[limb + 1] << 32;
        g.v[i] = (int32_t)((uint32_t)(w >> sh) & SC_INV_M30);
    }
    int32_t zeta = -1;   // -(delta + 1/2), delta starts at 1/2
    int32_t t[4];
#pragma unroll 1
    for (int it = 0; it < 20; it++) {
        zeta = sc_divsteps_30(zeta, (uint32_t)f.v[0], (uint32_t)g.v[0], t);
        sc_update_de_30(d, e, t);
        sc_update_fg_30(f, g, t);
    }
    // d in (-2l, l), f = +-1: result = sign(f) * d mod l
    int32_t cond_add = d.v[8] >> 31;
    const int32_t cond_neg = f.v[8] >> 31;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        d.v[i] += SC_L30[i] & cond_add;
        d.v[i] = (d.v[i] ^ cond_neg) - cond_neg;
    }
#pragma unroll
    for (int i = 0; i < 8; i++) { d.v[i + 1] += d.v[i] >> 30; d.v[i] &= SC_INV_M30; }
    cond_add = d.v[8] >> 31;
#pragma unroll
    for (int i = 0; i < 9; i++) d.v[i] += SC_L30[i] & cond_add;
#pragma unroll
    for (int i = 0; i < 8; i++) { d.v[i + 1] += d.v[i] >> 30; d.v[i] &= SC_INV_M30; }
    // 9 x 30 bits -> 8 x 32 bits
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int bit = 32 * k, li = bit / 30, sh = bit % 30;
        unsigned long long w = (unsigned long long)(uint32_t)d.v[li] >> sh;
        w |= (unsigned long long)(uint32_t)d.v[li + 1] << (30 - sh);
        if (li + 2 < 9) w |= (unsigned long long)(uint32_t)d.v[li + 2] << (60 - sh);
        r.v[k] = (uint32_t)w;
    }
}
