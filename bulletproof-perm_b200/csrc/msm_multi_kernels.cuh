// msm_multi_kernels.cuh - `count` independent variable-base MSMs with ragged sizes in one call (bpp_msm_multi*).
//
// MSM j is sum_{t in [start_j, start_j + n_j)} s_t P_t.  Every MSM is split into its window sums
// S_w = sum_t d_{t,w} P_t (signed c-bit digits d_{t,w} of s_t) and a Horner step over them:
//   k_mm_decode      thread per term: RFC 9496 decode -> affine Niels; a bad encoding sets ITS MSM's flag only
//   k_mm_straus      small MSMs (c = 4): block per MSM, thread per window.  The block builds every term's multiples
//                    1..8 P_t in shared memory (8 mixed adds per term); window w is then n table look-ups + full adds
//   k_mm_pippenger   larger MSMs (c = MM_PIPPENGER_C): block per chunk of at most MM_CHUNK terms, thread per window,
//                    the 2^(c-1) buckets of the thread's window in local memory (as k_dyn_window_sums); running-sum fold
//   k_mm_finish      thread per MSM: adds the window sums of its chunks, Horner (c doublings per window), compress
// Digits: s' = s + K with K = sum_{w < W-1} 2^(c-1) 2^(cw); d_w = field w of s' minus 2^(c-1), the top window unsigned.
// With s < 2^255 and cW >= 256, s' < 2^256 and every |d_w| <= 2^(c-1).
#pragma once
#include "ge25519.cuh"

#define MM_THREADS_FINISH 128
#define MM_TILE 64            // terms staged in shared memory at a time (scalars s' and Niels points)
#define MM_STRAUS_MAX 32      // MSMs of up to this many terms take k_mm_straus (its table: 1 KB of shared memory per term)
#define MM_PIPPENGER_C 5      // window width of k_mm_pippenger.  Wider windows cost more than they save with the buckets in
                              // local memory: c = 6 and c = 8 were measured slower at every size (DESIGN.md 3.6)
#define MM_CHUNK 1024         // terms per k_mm_pippenger block: a longer MSM is split and k_mm_finish adds the chunks

// Host-built plan (one upload per call).
struct mm_item {              // one k_mm_straus / k_mm_pippenger block
    uint32_t t0, n;           // its terms [t0, t0 + n)
    uint32_t wofs;            // its W window sums at wsum[wofs .. wofs + W) (128 B each)
    uint32_t pad;
};
struct mm_msm {               // one k_mm_finish thread
    uint32_t wofs, items;     // window sums of its first chunk; chunk k at wofs + k W
    uint32_t c, pad;          // window width (W = ceil(256 / c)); items = 0: the empty MSM
};

__host__ __device__ __forceinline__ uint32_t mm_windows(uint32_t c) { return (256 + c - 1) / c; }

// bit `bit` .. bit + c - 1 of an 8-limb value (c <= 8)
FE_INLINE uint32_t mm_field(const uint32_t s[8], uint32_t bit, uint32_t c) {
    const uint32_t limb = bit >> 5, sh = bit & 31;
    uint64_t v = s[limb];
    if (limb + 1 < 8) v |= (uint64_t)s[limb + 1] << 32;
    return (uint32_t)(v >> sh) & ((1u << c) - 1u);
}
// signed digit of window w of s' (see the header comment)
FE_INLINE int mm_digit(const uint32_t s[8], uint32_t w, uint32_t c, uint32_t W) {
    const uint32_t u = mm_field(s, c * w, c);
    return w == W - 1 ? (int)u : (int)u - (int)(1u << (c - 1));
}

// P_t as affine Niels: niels[index ? index[t] : t].  An index outside the set asserts in the debug build and is clamped
// into range in the product build (device data must not fault).
FE_INLINE const uint32_t *mm_point(const uint32_t *niels, const uint32_t *index, uint32_t n_pts, uint32_t t) {
    uint32_t i = t;
    if (index) {
        i = index[t];
        BPP_ASSERT(i < n_pts);
        if (i >= n_pts) i = n_pts - 1;
    }
    return niels + 24 * (size_t)i;
}

// The block stages terms [t0, t0 + cnt) (cnt <= MM_TILE) of the item: s' = s + K (8 words) and the Niels point (24 words).
// Bit 255 of a scalar is read as zero (the host forms reject it before; the _dev forms cannot fault on it).
FE_INLINE void mm_stage(uint32_t (*ss)[8], uint32_t (*sq)[24], const uint32_t *__restrict__ scalars, const uint32_t *niels,
                        const uint32_t *index, uint32_t n_pts, uint32_t t0, uint32_t cnt, uint32_t c, uint32_t W) {
    for (uint32_t k = threadIdx.x; k < cnt; k += blockDim.x) {
        const uint32_t *sp = scalars + 8 * (size_t)(t0 + k);
        uint64_t carry = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            uint32_t kl = 0;   // word i of K
#pragma unroll 1
            for (uint32_t w = 0; w + 1 < W; w++) {
                const uint32_t bit = c * w + c - 1;
                if ((bit >> 5) == (uint32_t)i) kl |= 1u << (bit & 31);
            }
            const uint32_t si = i == 7 ? (sp[i] & 0x7fffffffu) : sp[i];
            carry += (uint64_t)si + kl;
            ss[k][i] = (uint32_t)carry;
            carry >>= 32;
        }
        const uint32_t *q = mm_point(niels, index, n_pts, t0 + k);
#pragma unroll
        for (int i = 0; i < 24; i += 4) *reinterpret_cast<uint4 *>(&sq[k][i]) = *reinterpret_cast<const uint4 *>(q + i);
    }
}
FE_INLINE void mm_niels_smem(ge_niels &q, const uint32_t *p) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
        q.yp.v[i] = p[i];
        q.ym.v[i] = p[8 + i];
        q.t2d.v[i] = p[16 + i];
    }
}

// msm_of: the MSM whose term range holds t (starts: count + 1 prefix sums)
FE_INLINE uint32_t mm_msm_of(const uint32_t *__restrict__ starts, uint32_t count, uint32_t t) {
    uint32_t lo = 0, hi = count;   // starts[lo] <= t < starts[hi]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (starts[mid] <= t) lo = mid;
        else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(128) k_mm_decode(const uint8_t *__restrict__ enc, uint32_t T, const uint32_t *__restrict__ starts,
                                                   uint32_t count, uint32_t *__restrict__ niels, uint32_t *__restrict__ bad) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    fe x, y;
    if (!ge_decompress(x, y, enc + 32 * (size_t)t)) {   // the identity for the arithmetic; the MSM's result is discarded
        const uint32_t j = mm_msm_of(starts, count, t);
        BPP_ASSERT(j < count && starts[j] <= t && t < starts[j + 1]);
        atomicOr(&bad[j], 1u);
        fe_set0(x);
        fe_set1(y);
    }
    ge_niels q;
    ge_affine_to_niels(q, x, y);
    ge_niels_store(niels + 24 * (size_t)t, q);
}

// Straus form, c = 4 (64 windows, one thread each).  Dynamic shared memory: max_n x 8 x 128 B of multiples.
__global__ void __launch_bounds__(64) k_mm_straus(const mm_item *__restrict__ items, const uint32_t *__restrict__ scalars,
                                                  const uint32_t *niels, const uint32_t *__restrict__ index, uint32_t n_pts,
                                                  uint32_t *__restrict__ wsum) {
    extern __shared__ __align__(16) uint32_t mm_tab[];             // [term][multiple 1..8] x 32 words (extended)
    __shared__ __align__(16) uint32_t ss[MM_STRAUS_MAX][8];
    __shared__ __align__(16) uint32_t sq[MM_STRAUS_MAX][24];
    const mm_item it = items[blockIdx.x];
    BPP_ASSERT(it.n <= MM_STRAUS_MAX);
    const uint32_t n = it.n <= MM_STRAUS_MAX ? it.n : MM_STRAUS_MAX;
    mm_stage(ss, sq, scalars, niels, index, n_pts, it.t0, n, 4, 64);
    __syncthreads();
    for (uint32_t k = threadIdx.x; k < n; k += blockDim.x) {
        ge_niels q;
        mm_niels_smem(q, sq[k]);
        ge_ext a;
        ge_identity(a);
#pragma unroll 1
        for (int m = 0; m < 8; m++) {
            ge_madd(a, a, q, false);
            ge_store(mm_tab + 32 * (8 * (size_t)k + m), a);
        }
    }
    __syncthreads();
    const uint32_t w = threadIdx.x;
    ge_ext acc, e;
    ge_identity(acc);
#pragma unroll 1
    for (uint32_t k = 0; k < n; k++) {
        const int d = mm_digit(ss[k], w, 4, 64);
        if (d == 0) continue;
        const uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
        BPP_ASSERT(mag >= 1 && mag <= 8);
        ge_load(e, mm_tab + 32 * (8 * (size_t)k + mag - 1));
        if (d < 0) {
            fe_neg(e.X, e.X);
            fe_neg(e.T, e.T);
        }
        ge_add(acc, acc, e);
    }
    ge_store(wsum + 32 * ((size_t)it.wofs + w), acc);
}

// Pippenger form: block of 64 threads per chunk, thread w < W = 52 owns window w and its 2^(C-1) = 16 buckets.
__global__ void __launch_bounds__(64) k_mm_pippenger(const mm_item *__restrict__ items, const uint32_t *__restrict__ scalars,
                                                     const uint32_t *niels, const uint32_t *__restrict__ index, uint32_t n_pts,
                                                     uint32_t *__restrict__ wsum) {
    constexpr uint32_t C = MM_PIPPENGER_C, W = (256 + C - 1) / C, B = 1u << (C - 1);
    __shared__ __align__(16) uint32_t ss[MM_TILE][8];
    __shared__ __align__(16) uint32_t sq[MM_TILE][24];
    const mm_item it = items[blockIdx.x];
    BPP_ASSERT(it.n <= MM_CHUNK);
    const uint32_t w = threadIdx.x;
    ge_ext bkt[B];
#pragma unroll 1
    for (uint32_t b = 0; b < B; b++) ge_identity(bkt[b]);
#pragma unroll 1
    for (uint32_t k0 = 0; k0 < it.n; k0 += MM_TILE) {
        const uint32_t cnt = it.n - k0 < MM_TILE ? it.n - k0 : MM_TILE;
        __syncthreads();
        mm_stage(ss, sq, scalars, niels, index, n_pts, it.t0 + k0, cnt, C, W);
        __syncthreads();
        if (w >= W) continue;
#pragma unroll 1
        for (uint32_t k = 0; k < cnt; k++) {
            const int d = mm_digit(ss[k], w, C, W);
            if (d == 0) continue;
            const uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
            BPP_ASSERT(mag >= 1 && mag <= B);
            ge_niels q;
            mm_niels_smem(q, sq[k]);
            ge_ext a = bkt[mag - 1];
            ge_madd(a, a, q, d < 0);
            bkt[mag - 1] = a;
        }
    }
    if (w >= W) return;
    ge_ext run = bkt[B - 1], acc = run, t;   // sum_b (b + 1) bkt[b] by running sums
#pragma unroll 1
    for (int b = (int)B - 2; b >= 0; b--) {
        t = bkt[b];
        ge_add(run, run, t);
        ge_add(acc, acc, run);
    }
    ge_store(wsum + 32 * ((size_t)it.wofs + w), acc);
}

// Thread per MSM: window sums of all its chunks, Horner, then the encoding (32 zero bytes and ok = 0 when one of its
// points failed to decode; the identity also encodes as 32 zero bytes).
__global__ void __launch_bounds__(MM_THREADS_FINISH) k_mm_finish(const mm_msm *__restrict__ msms, uint32_t count,
                                                                 const uint32_t *__restrict__ wsum, const uint32_t *__restrict__ bad,
                                                                 uint8_t *__restrict__ out32, uint8_t *__restrict__ ok) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const mm_msm m = msms[j];
    ge_ext acc, t;
    ge_identity(acc);
    if (m.items) {
        const uint32_t W = mm_windows(m.c);
#pragma unroll 1
        for (int w = (int)W - 1; w >= 0; w--) {
            if (w != (int)W - 1) {
#pragma unroll 1
                for (uint32_t i = 0; i + 1 < m.c; i++) ge_double_p2(acc, acc);
                ge_double(acc, acc);
            }
#pragma unroll 1
            for (uint32_t k = 0; k < m.items; k++) {
                ge_load(t, wsum + 32 * ((size_t)m.wofs + (size_t)k * W + w));
                ge_add(acc, acc, t);
            }
        }
    }
    const bool good = !bad || bad[j] == 0;
    if (good) {
        ge_compress(out32 + 32 * (size_t)j, acc);
    } else {
#pragma unroll
        for (int i = 0; i < 32; i += 4) *reinterpret_cast<uint32_t *>(out32 + 32 * (size_t)j + i) = 0u;
    }
    if (ok) ok[j] = good ? 1 : 0;
}
