// msm_kernels.cuh - GPU Pippenger for Ristretto255 on sm_100a.
//
// Replaces dalek-ng 4.1.1 `backend::serial::scalar_mul::{straus,pippenger}` behind
// `RistrettoPoint::vartime_multiscalar_mul` (reference call sites: circuit_lib.rs:187,202,216,
// 363-407,498-568).  The group result is algorithm independent and the Ristretto encoding is
// canonical, so the bytes equal dalek's for every input.
//
// Pipeline (N points, window c bits, W = ceil(256/c) windows, B = 2^(c-1) buckets per window):
//   k_digit_hist      signed-window recode, per-(window,bucket) histogram (atomics)
//   k_window_scan     exclusive scan of each window's histogram -> bucket offsets
//   k_digit_scatter   counting-sort scatter of (point index | sign) into bucket order (no bucket ids are stored:
//                     the sorted order and the offsets determine them)
//   k_bucket_accum    one thread per tile of 32 sorted entries: mixed adds (extended += affine Niels, 7M)
//   k_bucket_fixup    stitches buckets cut by tile boundaries (+ k_bucket_fixup_long for hot buckets)
//   k_node_merge_*    bucket running sums as a tree of (S, A) nodes: thread-serial merges of 8 while
//                     the GPU is full, warp-shuffle merges of 32 after that
//   k_msm_finish      last merge per window, Horner over windows (c doublings each), compress
#pragma once
#include "ge25519.cuh"
#include "vec_kernels.cuh"

#define BPP_ACC_THREADS 128

// ---- signed-window recoding ---------------------------------------------------------------
// Digits d_w in [-(2^(c-1)-1), 2^(c-1)] with sum d_w 2^(cw) = s, for s < 2^255.
// (dalek Scalar::to_radix_2w uses the same carry scheme for w <= 8.)
FE_INLINE uint32_t sc_window(const uint32_t s[8], int bit, int c) {
    int limb = bit >> 5, sh = bit & 31;
    if (limb >= 8) return 0;
    uint64_t v = s[limb];
    if (limb + 1 < 8) v |= (uint64_t)s[limb + 1] << 32;
    return (uint32_t)(v >> sh) & ((1u << c) - 1u);
}

// Windows [w_begin, w_end) are counted (a window group of the pipelined MSM); the recoding carry is
// still rippled up from window 0.
__global__ void k_digit_hist(const uint32_t *__restrict__ scalars, uint32_t n, int c, int w_begin, int w_end,
                             uint32_t *__restrict__ counts) {
    const uint32_t half = 1u << (c - 1);
    // grid-stride: the pipelined MSM launches this with a small grid (a block or two per SM) so that the sort keeps
    // few SM slots while the accumulate of the previous group runs
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t s[8];
        const uint4 *p = reinterpret_cast<const uint4 *>(scalars + 8 * (size_t)i);
        uint4 lo = __ldg(p), hi = __ldg(p + 1);
        s[0] = lo.x; s[1] = lo.y; s[2] = lo.z; s[3] = lo.w; s[4] = hi.x; s[5] = hi.y; s[6] = hi.z; s[7] = hi.w;
        uint32_t carry = 0;
        for (int w = 0; w < w_end; w++) {
            uint32_t raw = sc_window(s, w * c, c) + carry;
            carry = raw > half ? 1u : 0u;
            uint32_t mag = carry ? (1u << c) - raw : raw;
            if (mag && w >= w_begin) atomicAdd(&counts[(size_t)w * half + (mag - 1)], 1u);
        }
    }
}

// one block (1024 threads) per window: exclusive scan of B counts
// `cursor` receives the offsets again (the global-atomic scatter advances them to the bucket ends) or, with
// ends_mode, the bucket ends themselves (offset + count: the shared-memory sort never touches it).
__global__ void __launch_bounds__(1024) k_window_scan(const uint32_t *__restrict__ counts, uint32_t B,
                                                      uint32_t *__restrict__ offsets,
                                                      uint32_t *__restrict__ cursor, int ends_mode) {
    __shared__ uint32_t warp_sums[32];
    const uint32_t w = blockIdx.x;
    const uint32_t per = (B + 1023) / 1024;
    const uint32_t base = threadIdx.x * per;
    const uint32_t *cw = counts + (size_t)w * B;
    uint32_t local = 0;
    const bool vec = (per & 3u) == 0;  // B >= 4096: whole uint4 groups per thread
    if (vec) {
        const uint4 *cv = reinterpret_cast<const uint4 *>(cw + base);
        for (uint32_t k = 0; k < per / 4; k++) {
            uint4 v = cv[k];
            local += v.x + v.y + v.z + v.w;
        }
    } else {
        for (uint32_t k = 0; k < per; k++)
            if (base + k < B) local += cw[base + k];
    }
    // block exclusive scan of `local`
    uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t incl = local;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= (uint32_t)d) incl += o;
    }
    if (lane == 31) warp_sums[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        uint32_t v = warp_sums[lane];
        uint32_t iv = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, iv, d);
            if (lane >= (uint32_t)d) iv += o;
        }
        warp_sums[lane] = iv - v;
    }
    __syncthreads();
    uint32_t run = warp_sums[wid] + incl - local;
    if (vec) {
        const uint4 *cv = reinterpret_cast<const uint4 *>(cw + base);
        uint4 *ov = reinterpret_cast<uint4 *>(offsets + (size_t)w * B + base);
        uint4 *uv = reinterpret_cast<uint4 *>(cursor + (size_t)w * B + base);
        for (uint32_t k = 0; k < per / 4; k++) {
            uint4 v = cv[k], o;
            o.x = run;
            o.y = o.x + v.x;
            o.z = o.y + v.y;
            o.w = o.z + v.z;
            run = o.w + v.w;
            ov[k] = o;
            if (ends_mode) {
                o.x = o.y; o.y = o.z; o.z = o.w; o.w = run;
            }
            uv[k] = o;
        }
    } else {
        for (uint32_t k = 0; k < per; k++)
            if (base + k < B) {
                offsets[(size_t)w * B + base + k] = run;
                cursor[(size_t)w * B + base + k] = ends_mode ? run + cw[base + k] : run;
                run += cw[base + k];
            }
    }
}

__global__ void k_digit_scatter(const uint32_t *__restrict__ scalars, uint32_t n, int c, int w_begin, int w_end,
                                uint32_t *__restrict__ cursor, uint32_t *__restrict__ entries) {
    const uint32_t half = 1u << (c - 1);
    // (issuing the position atomics eight windows at a time before the first write was measured: not faster, alone
    // or beside the accumulate - profiles/r1_msm_sort.md)
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        uint32_t s[8];
        const uint4 *p = reinterpret_cast<const uint4 *>(scalars + 8 * (size_t)i);
        uint4 lo = __ldg(p), hi = __ldg(p + 1);
        s[0] = lo.x; s[1] = lo.y; s[2] = lo.z; s[3] = lo.w; s[4] = hi.x; s[5] = hi.y; s[6] = hi.z; s[7] = hi.w;
        uint32_t carry = 0;
        for (int w = 0; w < w_end; w++) {
            uint32_t raw = sc_window(s, w * c, c) + carry;
            carry = raw > half ? 1u : 0u;
            uint32_t mag = carry ? (1u << c) - raw : raw;
            if (mag && w >= w_begin) {
                BPP_ASSERT(mag <= half);
                uint32_t pos = atomicAdd(&cursor[(size_t)w * half + (mag - 1)], 1u);
                BPP_ASSERT(pos < n);
                entries[(size_t)w * n + pos] = i | (carry << 31);
            }
        }
    }
}

// (Two other sort forms were built and measured in round 1 - per-window counters in shared memory, and a two-pass sort
// with coalesced writes.  Neither beat the global-atomic form beside the accumulate; they were removed from the product
// in round 2.  Record: profiles/r1_msm_sort.md, code: tools/experiments/msm_sort_forms_2_3.patch.)

// ---- bucket accumulation: the dominant kernel ------------------------------------------------
// The bucket-sorted entry list of each window is cut into tiles of `tile_len` entries; one thread
// owns one tile, so every thread performs the same number of mixed adds (extended += affine
// Niels, 7M) whatever the bucket sizes are: no warp divergence from Poisson bucket sizes and no
// serialisation on hot buckets (repeated / small scalars).  A bucket that lies inside one tile is
// written directly; a bucket cut by a tile boundary leaves partial sums (at most two per tile:
// `head` = the run touching the tile start, `tail` = the run touching the tile end) that
// k_bucket_fixup adds up.  `niels` is the static point table (96 B per point, read-only path).
// The tile length is a launch parameter (`tile_len`): 32 entries, 64 from 3 M points (measured: half the partials
// and half the cut buckets outweigh the coarser accumulate grid only once the input is large - 2^22 points 6.15 ->
// 5.79 ms per submitted MSM, 2^21 3.12 -> 3.19 ms, 2^18 0.66 -> 0.73 ms; bpp_set_msm_tile overrides).

FE_INLINE void bucket_flush(const ge_ext &acc, uint32_t w, uint32_t b, uint32_t rs, uint32_t re, uint32_t e0,
                            uint32_t B, size_t tile, const uint32_t *__restrict__ offsets,
                            const uint32_t *__restrict__ ends, uint32_t *__restrict__ buckets,
                            uint32_t *__restrict__ partials) {
    size_t g = (size_t)w * B + b;
    BPP_ASSERT(b < B && rs < re);
    bool complete = (offsets[g] == rs) && (ends[g] == re);
    uint32_t *dst = complete ? buckets + 32 * g : partials + 32 * (2 * tile + (rs == e0 ? 0 : 1));
    ge_store(dst, acc);
}

__global__ void __launch_bounds__(BPP_ACC_THREADS, 4) k_bucket_accum(
    const uint32_t *__restrict__ niels, const uint32_t *__restrict__ entries, const uint32_t *__restrict__ offsets,
    const uint32_t *__restrict__ ends, uint32_t n, uint32_t B, uint32_t tiles_per_window, uint32_t total_tiles,
    uint32_t tile_len, uint32_t *__restrict__ buckets, uint32_t *__restrict__ partials) {
    uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x;
    if (tile >= total_tiles) return;
    const uint32_t w = tile / tiles_per_window, t = tile - w * tiles_per_window;
    const uint32_t *endw = ends + (size_t)w * B;
    const uint32_t cnt = endw[B - 1];  // entries in this window
    const uint32_t e0 = t * tile_len;
    if (e0 >= cnt) return;
    const uint32_t e1 = min(e0 + tile_len, cnt);
    const uint32_t *ew = entries + (size_t)w * n;
    // bucket of entry e0 = the first bucket whose end offset lies beyond e0 (the entry list carries no
    // bucket ids: the sorted order and the offsets determine them)
    uint32_t lo = 0, hi = B - 1;
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (endw[mid] > e0) hi = mid;
        else lo = mid + 1;
    }
    uint32_t cur = lo, cur_end = endw[lo], run_start = e0;
    ge_ext acc;
    ge_identity(acc);
    uint32_t idx = ew[e0];
    BPP_ASSERT((idx & 0x7fffffffu) < n && cnt <= n && lo < B);
    ge_niels q;
    ge_niels_load(q, niels + 24 * (size_t)(idx & 0x7fffffffu));
#pragma unroll 1
    for (uint32_t e = e0; e < e1; e++) {
        // software pipeline: fetch the next entry's point while this one is being added
        uint32_t idx_n = idx;
        ge_niels qn = q;
        if (e + 1 < e1) {
            idx_n = ew[e + 1];
            BPP_ASSERT((idx_n & 0x7fffffffu) < n);
            ge_niels_load(qn, niels + 24 * (size_t)(idx_n & 0x7fffffffu));
        }
        ge_madd(acc, acc, q, (idx >> 31) != 0);
        if (e + 1 == e1 || e + 1 == cur_end) {
            bucket_flush(acc, w, cur, run_start, e + 1, e0, B, tile, offsets, ends, buckets, partials);
            ge_identity(acc);
            run_start = e + 1;
            if (e + 1 < e1) {   // next non-empty bucket
                do {
                    cur++;
                    BPP_ASSERT(cur < B);
                    cur_end = endw[cur];
                } while (cur_end <= e + 1);
            }
        }
        idx = idx_n;
        q = qn;
    }
}

// One thread per (window, bucket): empty buckets become the identity; buckets cut by tile
// boundaries are assembled from their partial sums.  Buckets spanning more than BPP_LONG_SPAN
// tiles (hot buckets) are queued for k_bucket_fixup_long.
#define BPP_LONG_SPAN 24
__global__ void __launch_bounds__(128) k_bucket_fixup(const uint32_t *__restrict__ offsets,
                                                      const uint32_t *__restrict__ ends, uint32_t B,
                                                      uint32_t tiles_per_window, uint32_t total_buckets, uint32_t tile_len,
                                                      const uint32_t *__restrict__ partials,
                                                      uint32_t *__restrict__ buckets, uint32_t *__restrict__ long_list,
                                                      uint32_t *__restrict__ n_long) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total_buckets) return;
    const uint32_t beg = offsets[g], end = ends[g];
    if (beg == end) {
        ge_ext id;
        ge_identity(id);
        ge_store(buckets + 32 * (size_t)g, id);
        return;
    }
    const uint32_t first = beg / tile_len, last = (end - 1) / tile_len;
    BPP_ASSERT(beg < end && last < tiles_per_window);
    if (first == last) return;  // complete inside one tile: already written
    if (last - first > BPP_LONG_SPAN) {
        long_list[atomicAdd(n_long, 1u)] = g;
        return;
    }
    const size_t tbase = (size_t)(g / B) * tiles_per_window;
    ge_ext acc, t;
    ge_load(acc, partials + 32 * (2 * (tbase + first) + (beg > first * tile_len ? 1 : 0)));
#pragma unroll 1
    for (uint32_t k = first + 1; k <= last; k++) {
        ge_load(t, partials + 32 * (2 * (tbase + k)));
        ge_add(acc, acc, t);
    }
    ge_store(buckets + 32 * (size_t)g, acc);
}

// One block (128 threads) per hot bucket: strided partial sums, then a shared-memory tree.
__global__ void __launch_bounds__(128) k_bucket_fixup_long(const uint32_t *__restrict__ offsets,
                                                           const uint32_t *__restrict__ ends, uint32_t B,
                                                           uint32_t tiles_per_window, uint32_t tile_len,
                                                           const uint32_t *__restrict__ partials,
                                                           uint32_t *__restrict__ buckets,
                                                           const uint32_t *__restrict__ long_list,
                                                           const uint32_t *__restrict__ n_long) {
    __shared__ __align__(16) uint32_t sh[128][32];
    const uint32_t nl = *n_long;
    for (uint32_t i = blockIdx.x; i < nl; i += gridDim.x) {
        const uint32_t g = long_list[i];
        const uint32_t beg = offsets[g], end = ends[g];
        const uint32_t first = beg / tile_len, last = (end - 1) / tile_len;
        const size_t tbase = (size_t)(g / B) * tiles_per_window;
        ge_ext acc, t;
        ge_identity(acc);
#pragma unroll 1
        for (uint32_t k = first + 1 + threadIdx.x; k <= last; k += 128) {
            ge_load(t, partials + 32 * (2 * (tbase + k)));
            ge_add(acc, acc, t);
        }
        ge_store(&sh[threadIdx.x][0], acc);
        __syncthreads();
#pragma unroll 1
        for (uint32_t d = 64; d >= 1; d >>= 1) {
            if (threadIdx.x < d) {
                ge_load(acc, &sh[threadIdx.x][0]);
                ge_load(t, &sh[threadIdx.x + d][0]);
                ge_add(acc, acc, t);
                ge_store(&sh[threadIdx.x][0], acc);
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            ge_load(acc, &sh[0][0]);
            ge_load(t, partials + 32 * (2 * (tbase + first) + (beg > first * tile_len ? 1 : 0)));
            ge_add(acc, acc, t);
            ge_store(buckets + 32 * (size_t)g, acc);
        }
        __syncthreads();
    }
}

// ---- bucket reduction ---------------------------------------------------------------------------
// Window total = sum_b (b+1) * bucket_b.  The reduction works on NODES: a node covers a contiguous
// range [lo, lo+len) of one window's buckets and carries
//     S = sum bucket_b,          A = sum (b - lo) * bucket_b         (b in the range)
// so that total = A_root + S_root.  Merging L adjacent nodes of equal length len:
//     S' = sum_k S_k,            A' = sum_k A_k + len * sum_k k * S_k
// (sum_k k*S_k by the running-sum trick, len = 2^loglen by doublings).  A bucket is a node with
// len = 1 and A = 0.  Two kernels: a thread-serial merge of L nodes (used while there are enough
// nodes to fill the GPU) and a warp-shuffle merge of 32 nodes (short dependency chains for the
// few nodes left); k_msm_finish merges the last <= 32 nodes of every window and combines windows.
__global__ void __launch_bounds__(128) k_node_merge_serial(const uint32_t *__restrict__ inS,
                                                           const uint32_t *__restrict__ inA, uint32_t L,
                                                           uint32_t loglen, uint32_t n_out,
                                                           uint32_t *__restrict__ outS, uint32_t *__restrict__ outA) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_out) return;
    const uint32_t *ps = inS + 32 * (size_t)g * L;
    ge_ext run, acc, t;
    ge_load(run, ps + 32 * (size_t)(L - 1));
    acc = run;  // after the loop: acc = sum_k k * S_k, run = sum_k S_k
#pragma unroll 1
    for (int k = (int)L - 2; k >= 1; k--) {
        ge_load(t, ps + 32 * (size_t)k);
        ge_add(run, run, t);
        ge_add(acc, acc, run);
    }
    if (L > 1) {
        ge_load(t, ps);
        ge_add(run, run, t);
    } else {
        ge_identity(acc);
    }
#pragma unroll 1
    for (uint32_t i = 0; i < loglen; i++) ge_double(acc, acc);
    if (inA) {   // (interleaving this independent chain with the one above was measured: slower, 212 registers)
        const uint32_t *pa = inA + 32 * (size_t)g * L;
#pragma unroll 1
        for (uint32_t k = 0; k < L; k++) {
            ge_load(t, pa + 32 * (size_t)k);
            ge_add(acc, acc, t);
        }
    }
    ge_store(outS + 32 * (size_t)g, run);
    ge_store(outA + 32 * (size_t)g, acc);
}

// ---- lane-parallel ("quad") point arithmetic --------------------------------------------------------
// Everything after the first merge level is a short dependent chain of point operations on few points:
// nothing to parallelise across points, and a warp instruction costs the same for 1 or 32 active lanes.
// So the four independent field multiplications of each stage of a point operation run in four LANES:
// an aligned group of 4 lanes (a quad) holds one point, lane k of the quad holds coordinate k of
// (X, Y, Z, T).  A doubling costs one squaring + one multiplication of warp time instead of 4 + 4, a full
// addition three multiplications instead of nine; a warp carries 8 points.
FE_INLINE void fe_shfl4(fe &r, const fe &a, int k) {   // coordinate k of this lane's quad
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = __shfl_sync(0xffffffffu, a.v[i], k, 4);
}
FE_INLINE void fe_shfl_xor1(fe &r, const fe &a) {      // swap within the lane pairs (0,1) and (2,3)
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = __shfl_xor_sync(0xffffffffu, a.v[i], 1);
}
FE_INLINE void fe_pick(fe &r, const fe &a, const fe &b, bool take_a) {
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = take_a ? a.v[i] : b.v[i];
}
FE_INLINE void quad_identity(fe &v, uint32_t ql) {     // (0, 1, 1, 0)
    fe_set0(v);
    v.v[0] = (ql == 1 || ql == 2) ? 1u : 0u;
}
FE_INLINE void quad_load(fe &v, const uint32_t *node, uint32_t ql) { fe_load(v, node + 8 * ql); }
FE_INLINE void quad_store(uint32_t *node, const fe &v, uint32_t ql) { fe_store(node + 8 * ql, v); }
// last stage shared by doubling and addition: lane0 E*F, lane1 G*H, lane2 F*G, lane3 E*H
FE_INLINE void quad_finish(fe &v, const fe &E, const fe &F, const fe &G, const fe &H, uint32_t ql) {
    fe p, q, t;
    fe_pick(t, G, F, ql == 1);
    fe_pick(p, E, t, ql == 0 || ql == 3);
    fe_pick(t, G, H, ql == 2);
    fe_pick(q, F, t, ql == 0);
    fe_mul(v, p, q);
}
static __device__ __noinline__ void quad_double(fe &v, uint32_t ql) {
    fe x, y, s, in, sq, A, B, Zs, D, E, F, G, H;
    fe_shfl4(x, v, 0);
    fe_shfl4(y, v, 1);
    fe_add(s, x, y);
    fe_pick(in, s, v, ql == 3);
    fe_sqr(sq, in);
    fe_shfl4(A, sq, 0);
    fe_shfl4(B, sq, 1);
    fe_shfl4(Zs, sq, 2);
    fe_shfl4(D, sq, 3);
    fe_add(H, A, B);
    fe_sub(E, H, D);
    fe_sub(G, A, B);
    fe_dbl(Zs, Zs);
    fe_add(F, Zs, G);
    quad_finish(v, E, F, G, H, ql);
}
// v += the point cached at c (8 limbs each of Y+X, Y-X, Z, 2d*T; same address in every lane): two stages
static __device__ __noinline__ void quad_add_cached(fe &v, const uint32_t *c, uint32_t ql) {
    fe x, y, z, t, p, q, m, a, b, cc, d, E, F, G, H;
    fe_shfl4(x, v, 0);
    fe_shfl4(y, v, 1);
    fe_shfl4(z, v, 2);
    fe_shfl4(t, v, 3);
    fe_sub(a, y, x);
    fe_add(b, y, x);
    fe_pick(p, a, b, ql == 0);
    fe_pick(q, t, z, ql == 2);
    fe_pick(p, p, q, ql < 2);
    fe_load(q, c + 8 * (ql == 0 ? 1 : ql == 1 ? 0 : ql == 2 ? 3 : 2));
    fe_mul(m, p, q);
    fe_shfl4(a, m, 0);
    fe_shfl4(b, m, 1);
    fe_shfl4(cc, m, 2);
    fe_shfl4(d, m, 3);
    fe_dbl(d, d);
    fe_sub(E, b, a);
    fe_add(H, b, a);
    fe_sub(F, d, cc);
    fe_add(G, d, cc);
    quad_finish(v, E, F, G, H, ql);
}
// v += w, both in quad form: (Y1-X1)(Y2-X2) | (Y1+X1)(Y2+X2) | T1*T2 | Z1*Z2, then 2d*(T1*T2) in lane 2,
// then the four products of the last stage.
static __device__ __noinline__ void quad_add(fe &v, const fe &w, uint32_t ql) {
    fe x1, y1, x2, y2, p1, p2, a, b, m, k, cc, d, E, F, G, H;
    fe_shfl4(x1, v, 0);
    fe_shfl4(y1, v, 1);
    fe_shfl4(x2, w, 0);
    fe_shfl4(y2, w, 1);
    fe_shfl_xor1(p1, v);    // lane 2 <- T1, lane 3 <- Z1
    fe_shfl_xor1(p2, w);    // lane 2 <- T2, lane 3 <- Z2
    fe_sub(a, y1, x1);
    fe_sub(b, y2, x2);
    fe_add(m, y1, x1);
    fe_add(k, y2, x2);
    fe_pick(a, a, m, ql == 0);
    fe_pick(b, b, k, ql == 0);
    fe_pick(a, a, p1, ql < 2);
    fe_pick(b, b, p2, ql < 2);
    fe_mul(m, a, b);
    fe_const(k, GE_D2);
    fe_set1(a);
    fe_pick(k, k, a, ql == 2);
    fe_mul(m, m, k);        // lane 2: 2d*T1*T2; the other lanes multiply by one
    fe_shfl4(a, m, 0);
    fe_shfl4(b, m, 1);
    fe_shfl4(cc, m, 2);
    fe_shfl4(d, m, 3);
    fe_dbl(d, d);
    fe_sub(E, b, a);
    fe_add(H, b, a);
    fe_sub(F, d, cc);
    fe_add(G, d, cc);
    quad_finish(v, E, F, G, H, ql);
}

// Quad-serial merge of L nodes into one (same arithmetic as k_node_merge_serial, one quad per output node).
__global__ void __launch_bounds__(128) k_node_merge_quad_serial(const uint32_t *__restrict__ inS,
                                                                const uint32_t *__restrict__ inA, uint32_t L,
                                                                uint32_t loglen, uint32_t n_out,
                                                                uint32_t *__restrict__ outS, uint32_t *__restrict__ outA) {
    const uint32_t ql = threadIdx.x & 3;
    uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    const bool live = g < n_out;
    if (!live) g = n_out - 1;   // whole quads stay in step for the shuffles; only live quads store
    const uint32_t *ps = inS + 32 * (size_t)g * L, *pa = inA + 32 * (size_t)g * L;
    fe run, acc, t;
    quad_load(run, ps + 32 * (size_t)(L - 1), ql);
    acc = run;
#pragma unroll 1
    for (int k = (int)L - 2; k >= 1; k--) {
        quad_load(t, ps + 32 * (size_t)k, ql);
        quad_add(run, t, ql);
        quad_add(acc, run, ql);
    }
    quad_load(t, ps, ql);
    quad_add(run, t, ql);
#pragma unroll 1
    for (uint32_t i = 0; i < loglen; i++) quad_double(acc, ql);
#pragma unroll 1
    for (uint32_t k = 0; k < L; k++) {
        quad_load(t, pa + 32 * (size_t)k, ql);
        quad_add(acc, t, ql);
    }
    if (live) {
        quad_store(outS + 32 * (size_t)g, run, ql);
        quad_store(outA + 32 * (size_t)g, acc, ql);
    }
}

// Block merge of 32 nodes (one per quad, identity for missing ones): suffix scan of S (5 additions),
// then sum_k k*S_k and sum_k A_k as two trees riding together (5 x 2), loglen doublings, one addition.
// Partner values travel through shared memory (the 32 quads span 4 warps).  grid (T_out, W).
__global__ void __launch_bounds__(128) k_node_merge_quad_block(const uint32_t *__restrict__ inS,
                                                               const uint32_t *__restrict__ inA, uint32_t T,
                                                               uint32_t loglen, uint32_t T_out,
                                                               uint32_t *__restrict__ outS, uint32_t *__restrict__ outA) {
    __shared__ __align__(16) uint32_t shS[32][32], shA[32][32];
    const uint32_t w = blockIdx.y, g = blockIdx.x, quad = threadIdx.x >> 2, ql = threadIdx.x & 3;
    const uint32_t t = g * 32 + quad;
    fe S, A, o, oa, tmp;
    quad_identity(S, ql);
    quad_identity(A, ql);
    if (t < T) {
        quad_load(S, inS + 32 * ((size_t)w * T + t), ql);
        if (inA) quad_load(A, inA + 32 * ((size_t)w * T + t), ql);
    }
#pragma unroll 1
    for (uint32_t d = 1; d < 32; d <<= 1) {   // inclusive suffix scan: S_q = sum_{j >= q} S_j
        quad_store(&shS[quad][0], S, ql);
        __syncthreads();
        quad_load(o, &shS[(quad + d) & 31][0], ql);
        __syncthreads();
        tmp = S;
        quad_add(tmp, o, ql);
        fe_pick(S, tmp, S, quad + d < 32);
    }
    fe b = S;   // sum_k k * S_k = sum_{j = 1..31} suffix_j
    if (quad == 0) quad_identity(b, ql);
#pragma unroll 1
    for (uint32_t d = 16; d >= 1; d >>= 1) {
        quad_store(&shS[quad][0], b, ql);
        quad_store(&shA[quad][0], A, ql);
        __syncthreads();
        quad_load(o, &shS[(quad + d) & 31][0], ql);
        quad_load(oa, &shA[(quad + d) & 31][0], ql);
        __syncthreads();
        tmp = b;
        quad_add(tmp, o, ql);
        fe_pick(b, tmp, b, quad < d);
        tmp = A;
        quad_add(tmp, oa, ql);
        fe_pick(A, tmp, A, quad < d);
    }
#pragma unroll 1
    for (uint32_t i = 0; i < loglen; i++) quad_double(b, ql);
    quad_add(A, b, ql);
    if (quad == 0) {
        quad_store(outS + 32 * ((size_t)w * T_out + g), S, ql);
        quad_store(outA + 32 * ((size_t)w * T_out + g), A, ql);
    }
}

// One warp.  Lane w < W adds window w's root node (A + S = window total) and caches it; then the
// warp runs Horner over the windows in quad form (c doublings + 1 addition per window) and lane 0
// compresses.  With `do_compress` the 32-byte encoding goes to out[0..32) and the raw extended
// point to out[32..160); otherwise the raw extended point goes to out[0..128).
// `shift` extra doublings at the end place a window group at its weight 2^shift (pipelined MSM).
__global__ void __launch_bounds__(32) k_msm_finish(const uint32_t *__restrict__ inS,
                                                   const uint32_t *__restrict__ inA, int c, int W, int shift,
                                                   int do_compress, uint8_t *__restrict__ out) {
    __shared__ __align__(16) uint32_t sh[64][32];
    const uint32_t lane = threadIdx.x;
    for (uint32_t w = lane; w < (uint32_t)W; w += 32) {
        ge_ext S, A;
        ge_load(S, inS + 32 * (size_t)w);
        if (inA) {
            ge_load(A, inA + 32 * (size_t)w);
            ge_add(S, S, A);
        }
        fe yp, ym, t2d, d2;
        fe_add(yp, S.Y, S.X);
        fe_sub(ym, S.Y, S.X);
        fe_const(d2, GE_D2);
        fe_mul(t2d, S.T, d2);
        fe_store(&sh[w][0], yp);
        fe_store(&sh[w][8], ym);
        fe_store(&sh[w][16], S.Z);
        fe_store(&sh[w][24], t2d);
    }
    __syncwarp();
    fe v;
    quad_identity(v, lane & 3);   // the warp's 8 quads all run the same chain; quad 0 is the one that is read
#pragma unroll 1
    for (int k = W - 1; k >= 0; k--) {
        quad_add_cached(v, &sh[k][0], lane & 3);
        if (k > 0) {
#pragma unroll 1
            for (int i = 0; i < c; i++) quad_double(v, lane & 3);
        }
    }
#pragma unroll 1
    for (int i = 0; i < shift; i++) quad_double(v, lane & 3);
    ge_ext acc;
    fe_shfl4(acc.X, v, 0);
    fe_shfl4(acc.Y, v, 1);
    fe_shfl4(acc.Z, v, 2);
    fe_shfl4(acc.T, v, 3);
    if (lane == 0) {
        if (do_compress) {
            ge_compress(out, acc);
            ge_store(reinterpret_cast<uint32_t *>(out + 32), acc);
        } else {
            ge_store(reinterpret_cast<uint32_t *>(out), acc);
        }
    }
}

// sum of g extended points (raw limbs, 128 B each) -> compress
__global__ void __launch_bounds__(32) k_points_sum_compress(const uint32_t *__restrict__ parts, uint32_t g,
                                                            uint8_t *__restrict__ out32) {
    if (threadIdx.x != 0) return;
    ge_ext acc, t;
    ge_load(acc, parts);
#pragma unroll 1
    for (uint32_t i = 1; i < g; i++) {
        ge_load(t, parts + 32 * (size_t)i);
        ge_add(acc, acc, t);
    }
    ge_compress(out32, acc);
}

// sum of g window-group partials, written like k_msm_finish does (encoding + raw point, or raw point only)
__global__ void __launch_bounds__(32) k_points_sum_finish(const uint32_t *__restrict__ parts, uint32_t g,
                                                          int do_compress, uint8_t *__restrict__ out) {
    if (threadIdx.x != 0) return;
    ge_ext acc, t;
    ge_load(acc, parts);
#pragma unroll 1
    for (uint32_t i = 1; i < g; i++) {
        ge_load(t, parts + 32 * (size_t)i);
        ge_add(acc, acc, t);
    }
    if (do_compress) {
        ge_compress(out, acc);
        ge_store(reinterpret_cast<uint32_t *>(out + 32), acc);
    } else {
        ge_store(reinterpret_cast<uint32_t *>(out), acc);
    }
}

// ---- point ingestion ----------------------------------------------------------------------------
__global__ void k_decompress_to_niels(const uint8_t *__restrict__ in, uint32_t n, uint32_t *__restrict__ niels,
                                      uint32_t *__restrict__ n_invalid) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe x, y;
    bool ok = ge_decompress(x, y, in + 32 * (size_t)i);
    if (!ok) {
        atomicAdd(n_invalid, 1u);
        fe_set0(x);
        fe_set1(y);
    }
    ge_niels q;
    ge_affine_to_niels(q, x, y);
    ge_niels_store(niels + 24 * (size_t)i, q);
}

__global__ void k_affine_to_niels(const uint8_t *__restrict__ in, uint32_t n, uint32_t *__restrict__ niels) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe x, y;
    fe_frombytes(x, in + 64 * (size_t)i);
    fe_frombytes(y, in + 64 * (size_t)i + 32);
    ge_niels q;
    ge_affine_to_niels(q, x, y);
    ge_niels_store(niels + 24 * (size_t)i, q);
}

// dalek FieldElement51: 5 x u64 limbs radix 2^51 (limbs may exceed 51 bits by a few bits)
FE_INLINE void fe_from_radix51(fe &r, const unsigned long long *l) {
    // value = sum l_i 2^(51 i); accumulate into 9 x 32-bit limbs, then fold
    unsigned long long acc[9];
#pragma unroll
    for (int i = 0; i < 9; i++) acc[i] = 0;
#pragma unroll
    for (int i = 0; i < 5; i++) {
        int bit = 51 * i, limb = bit >> 5, sh = bit & 31;
        unsigned long long lo = l[i] << sh;                      // low 64 bits of l_i << sh
        unsigned long long hi = sh ? (l[i] >> (64 - sh)) : 0ull;  // overflow bits
        acc[limb] += lo & 0xffffffffull;
        acc[limb + 1] += lo >> 32;
        if (limb + 2 < 9) acc[limb + 2] += hi;
    }
    uint32_t t[16];
    unsigned long long carry = 0;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        carry += acc[i];
        t[i] = (uint32_t)carry;
        carry >>= 32;
    }
    t[9] = (uint32_t)carry;
#pragma unroll
    for (int i = 10; i < 16; i++) t[i] = 0;
    fe_reduce16(r, t);
}

__global__ void k_dalek_xyzt_to_niels(const unsigned long long *__restrict__ in, uint32_t n,
                                      uint32_t *__restrict__ niels) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long *p = in + 20 * (size_t)i;
    unsigned long long l[5];
    fe X, Y, Z, zi, x, y;
#pragma unroll
    for (int k = 0; k < 5; k++) l[k] = p[k];
    fe_from_radix51(X, l);
#pragma unroll
    for (int k = 0; k < 5; k++) l[k] = p[5 + k];
    fe_from_radix51(Y, l);
#pragma unroll
    for (int k = 0; k < 5; k++) l[k] = p[10 + k];
    fe_from_radix51(Z, l);
    fe_invert(zi, Z);
    fe_mul_noinline(x, X, zi);
    fe_mul_noinline(y, Y, zi);
    ge_niels q;
    ge_affine_to_niels(q, x, y);
    ge_niels_store(niels + 24 * (size_t)i, q);
}

// RistrettoPoint::from_uniform_bytes / ::random (lib.rs:165-166,179-180): 64 uniform bytes -> point
__global__ void k_from_uniform_to_niels(const uint8_t *__restrict__ in, uint32_t n, uint32_t *__restrict__ niels) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ge_ext p;
    ge_from_uniform(p, in + 64 * (size_t)i);
    fe zi, x, y;
    fe_invert(zi, p.Z);
    fe_mul_noinline(x, p.X, zi);
    fe_mul_noinline(y, p.Y, zi);
    ge_niels q;
    ge_affine_to_niels(q, x, y);
    ge_niels_store(niels + 24 * (size_t)i, q);
}

// Niels table -> compressed encodings (x = (yp - ym)/2, y = (yp + ym)/2; the common factor 2 is
// projective: (X, Y, Z, T) = (2x*2, 2y*2, 4, 2x*2y) = (2(yp-ym), 2(yp+ym), 4, (yp-ym)(yp+ym)))
__global__ void k_niels_compress(const uint32_t *__restrict__ niels, uint32_t n, uint8_t *__restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ge_niels q;
    ge_niels_load(q, niels + 24 * (size_t)i);
    fe x2, y2;
    fe_sub(x2, q.yp, q.ym);
    fe_add(y2, q.yp, q.ym);
    ge_ext p;
    fe_dbl(p.X, x2);
    fe_dbl(p.Y, y2);
    fe_set0(p.Z);
    p.Z.v[0] = 4;
    fe_mul_noinline(p.T, x2, y2);
    ge_compress(out + 32 * (size_t)i, p);
}

// ---- integer-pipe microbenchmarks --------------------------------------------------------------
// Every multiply takes one operand from ANOTHER chain's previous result, so ptxas can neither hoist
// the product out of the loop nor strength-reduce repeated accumulation into adds (an earlier version
// with loop-invariant operands was rewritten by ptxas into one IMAD.WIDE + IADD3 pairs and measured the
// alu pipe instead; the SASS of these kernels is checked in tests/test_cabi.py::test_probe_sass).
//   mode 0: plain IMAD.WIDE.U32 with 64-bit addend       (8 chains/thread, 128 per loop trip)
//   mode 1: carry-chained IMAD.WIDE.U32 (mad.lo.cc/madc.hi.cc pairs: the saturated multiplier's form)
//   mode 2: 32-bit IMAD                                   mode 3: IADD3 carry chains
//   mode 4: fe_mul chains (2 per thread; 72 IMAD.WIDE-equivalents each)
//   mode 5: ge_madd chains (1 per thread; 504 IMAD.WIDE-equivalents each)
__global__ void __launch_bounds__(256) k_imad_peak(uint32_t seed, int iters, unsigned long long *out) {
    uint32_t a[16], b[8];
    unsigned long long c[8];
#pragma unroll
    for (int u = 0; u < 16; u++) a[u] = (seed + threadIdx.x) * (2u * u + 3u) + u;
#pragma unroll
    for (int k = 0; k < 8; k++) c[k] = blockIdx.x + k + 1;
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int k = 0; k < 8; k++) b[k] = (uint32_t)(c[(k + 1) & 7] >> 7) | 1u;  // data dependent, once per trip
#pragma unroll
        for (int u = 0; u < 16; u++)
#pragma unroll
            for (int k = 0; k < 8; k++) c[k] += (unsigned long long)a[u] * b[k];  // IMAD.WIDE.U32 Rc, Ra, Rb, Rc
    }
    unsigned long long r = c[0] ^ c[1] ^ c[2] ^ c[3] ^ c[4] ^ c[5] ^ c[6] ^ c[7];
    if (r == 0x1234567812345678ull) out[0] = r;  // practically never; keeps the chains alive
}

__global__ void __launch_bounds__(256) k_pipe_probe(int mode, uint32_t seed, int iters, unsigned long long *out) {
    uint32_t a0 = seed + threadIdx.x, a1 = a0 * 3u + 1u, a2 = a0 * 5u + 2u, a3 = a0 * 7u + 3u;
    uint32_t c0 = 1 + blockIdx.x, c1 = 2, c2 = 3, c3 = 4, c4 = 5, c5 = 6, c6 = 7, c7 = 8, c8 = 0;
    uint32_t d0 = 9, d1 = 10, d2 = 11, d3 = 12, d4 = 13, d5 = 14, d6 = 15, d7 = 16, d8 = 0;
    if (mode == 1) {
#pragma unroll 1
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int u = 0; u < 8; u++) {  // 2 chains of 4 carry-linked wide multiply-adds (8 per u)
                fe_mad4(c0, c1, c2, c3, c4, c5, c6, c7, c8, a0, a1, a2, a3, d0 ^ d7);
                fe_mad4(d0, d1, d2, d3, d4, d5, d6, d7, d8, a1, a2, a3, a0, c0 ^ c7);
            }
        }
    } else if (mode == 2) {
#pragma unroll 1
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int u = 0; u < 8; u++) {  // 16 32-bit multiply-adds per u, multiplier from the other half
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(c0) : "r"(a0), "r"(d0));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(c1) : "r"(a1), "r"(d1));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(c2) : "r"(a2), "r"(d2));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(c3) : "r"(a3), "r"(d3));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(c4) : "r"(a0), "r"(d4));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(c5) : "r"(a1), "r"(d5));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(c6) : "r"(a2), "r"(d6));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(c7) : "r"(a3), "r"(d7));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(d0) : "r"(a0), "r"(c0));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(d1) : "r"(a1), "r"(c1));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(d2) : "r"(a2), "r"(c2));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(d3) : "r"(a3), "r"(c3));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(d4) : "r"(a0), "r"(c4));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(d5) : "r"(a1), "r"(c5));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(d6) : "r"(a2), "r"(c6));
                asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+&r"(d7) : "r"(a3), "r"(c7));
            }
        }
    } else if (mode == 3) {
#pragma unroll 1
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int u = 0; u < 8; u++) {  // 2 add-with-carry chains of 8 (16 adds per u), cross-fed
                asm volatile("add.cc.u32 %0,%0,%8; addc.cc.u32 %1,%1,%8; addc.cc.u32 %2,%2,%8; addc.cc.u32 %3,%3,%8;"
                             "addc.cc.u32 %4,%4,%8; addc.cc.u32 %5,%5,%8; addc.cc.u32 %6,%6,%8; addc.u32 %7,%7,%8;"
                             : "+&r"(c0), "+&r"(c1), "+&r"(c2), "+&r"(c3), "+&r"(c4), "+&r"(c5), "+&r"(c6), "+&r"(c7) : "r"(d7));
                asm volatile("add.cc.u32 %0,%0,%8; addc.cc.u32 %1,%1,%8; addc.cc.u32 %2,%2,%8; addc.cc.u32 %3,%3,%8;"
                             "addc.cc.u32 %4,%4,%8; addc.cc.u32 %5,%5,%8; addc.cc.u32 %6,%6,%8; addc.u32 %7,%7,%8;"
                             : "+&r"(d0), "+&r"(d1), "+&r"(d2), "+&r"(d3), "+&r"(d4), "+&r"(d5), "+&r"(d6), "+&r"(d7) : "r"(c7));
            }
        }
    } else if (mode == 4) {
        fe x, y;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            x.v[i] = a0 * (2u * i + 1u) + c0;
            y.v[i] = a1 * (2u * i + 3u) + i;
        }
#pragma unroll 1
        for (int it = 0; it < iters; it++) {  // 2 multiplications per trip
            fe_mul(x, x, y);
            fe_mul(y, y, x);
        }
#pragma unroll
        for (int i = 0; i < 8; i++) c1 ^= x.v[i] ^ y.v[i];
    } else {
        ge_ext p;
        ge_niels q;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            p.X.v[i] = a0 + i; p.Y.v[i] = a1 + c0 + i; p.Z.v[i] = a2 + i; p.T.v[i] = a3 + i;
            q.yp.v[i] = a0 * 3u + i; q.ym.v[i] = a1 * 5u + i; q.t2d.v[i] = a2 * 7u + i;
        }
#pragma unroll 1
        for (int it = 0; it < iters; it++) ge_madd(p, p, q, (it & 1) != 0);
#pragma unroll
        for (int i = 0; i < 8; i++) c1 ^= p.X.v[i] ^ p.Y.v[i] ^ p.Z.v[i] ^ p.T.v[i];
    }
    uint32_t r = c0 ^ c1 ^ c2 ^ c3 ^ c4 ^ c5 ^ c6 ^ c7 ^ c8 ^ d0 ^ d1 ^ d2 ^ d3 ^ d4 ^ d5 ^ d6 ^ d7 ^ d8;
    if (r == 0x12345678u) out[0] = r;  // practically never; keeps every chain alive
}

// ---- element-wise test kernels -------------------------------------------------------------------
__global__ void k_test_op(int op, const uint8_t *__restrict__ a, const uint8_t *__restrict__ b,
                          uint8_t *__restrict__ out, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *pa = a + 32 * (size_t)i, *pb = b + 32 * (size_t)i;
    uint8_t *po = out + 32 * (size_t)i;
    if (op >= BPP_TEST_SC_ADD) {   // scalars mod l (bpp_test_op checks the op code and, for SC_WARP_SUM, n % 32)
        sc x, y, r;
        uint32_t t[16];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            x.v[k] = t[k] = pa[4 * k] | (uint32_t)pa[4 * k + 1] << 8 | (uint32_t)pa[4 * k + 2] << 16 | (uint32_t)pa[4 * k + 3] << 24;
            y.v[k] = t[8 + k] = pb[4 * k] | (uint32_t)pb[4 * k + 1] << 8 | (uint32_t)pb[4 * k + 2] << 16 | (uint32_t)pb[4 * k + 3] << 24;
        }
        switch (op) {
            case BPP_TEST_SC_ADD: sc_add(r, x, y); break;
            case BPP_TEST_SC_SUB: sc_sub(r, x, y); break;
            case BPP_TEST_SC_NEG: sc_neg(r, x); break;
            case BPP_TEST_SC_MONT: sc_mont(r, x, y); break;
            case BPP_TEST_SC_MUL: sc_mul(r, x, y); break;
            case BPP_TEST_SC_INVERT: sc_invert(r, x); break;
            case BPP_TEST_SC_REDUCE256: sc_reduce256(r, x); break;
            case BPP_TEST_SC_FROM_WIDE: sc_from_wide(r, t); break;
            case BPP_TEST_SC_MONT_REDUCE: sc_mont_reduce(r, t); break;
            case BPP_TEST_SC_WARP_SUM: {   // n % 32 == 0: whole warps, each over 32 consecutive values
                uint32_t s9[9];
                warp_sum9(s9, x);
#pragma unroll
                for (int k = 0; k < 9; k++) s9[k] = __shfl_sync(0xffffffffu, s9[k], 0);
                sc_from9(r, s9);
                break;
            }
            default: {   // SC_MAC + K - 1: K products accumulated by sc_mac, one sc_mont_reduce
                const uint32_t K = (uint32_t)(op - BPP_TEST_SC_MAC) + 1;
#pragma unroll
                for (int k = 0; k < 16; k++) t[k] = 0;
                for (uint32_t j = 0; j < K; j++) {
                    const uint32_t e = (uint32_t)(((uint64_t)i + j) % n);
                    const uint8_t *qa = a + 32 * (size_t)e, *qb = b + 32 * (size_t)e;
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        x.v[k] = qa[4 * k] | (uint32_t)qa[4 * k + 1] << 8 | (uint32_t)qa[4 * k + 2] << 16 | (uint32_t)qa[4 * k + 3] << 24;
                        y.v[k] = qb[4 * k] | (uint32_t)qb[4 * k + 1] << 8 | (uint32_t)qb[4 * k + 2] << 16 | (uint32_t)qb[4 * k + 3] << 24;
                    }
                    sc_mac(t, x, y);
                }
                sc_mont_reduce(r, t);
            }
        }
#pragma unroll
        for (int k = 0; k < 32; k++) po[k] = (uint8_t)(r.v[k >> 2] >> (8 * (k & 3)));
        return;
    }
    if (op <= 4 || op == 9) {
        fe x, y, r;
        fe_frombytes(x, pa);
        fe_frombytes(y, pb);
        switch (op) {
            case 0: fe_mul(r, x, y); break;
            case 1: fe_add(r, x, y); break;
            case 2: fe_sub(r, x, y); break;
            case 3: fe_invert(r, x); break;
            case 9: fe_sqr(r, x); break;
            default: fe_copy(r, x); break;
        }
        fe_tobytes(po, r);
        return;
    }
    ge_ext P, Q, Rr;
    fe x, y;
    bool ok = ge_decompress(x, y, pa);
    P.X = x; P.Y = y; fe_set1(P.Z); fe_mul(P.T, x, y);
    P.Z.v[0] += n >> 31;  // 0 at run time; keeps Z out of ptxas' uniform datapath (see k_test_uniform_sqr)
    if (!ok) {
        for (int k = 0; k < 32; k++) po[k] = 0xff;
        return;
    }
    if (op == 5) {
        ok = ge_decompress(x, y, pb);
        Q.X = x; Q.Y = y; fe_set1(Q.Z); fe_mul(Q.T, x, y);
        if (!ok) {
            for (int k = 0; k < 32; k++) po[k] = 0xff;
            return;
        }
        ge_add(Rr, P, Q);
    } else if (op == 6) {
        ge_double(Rr, P);
    } else if (op == 10) {  // doubling with a compile-time Z = 1 (uniform-datapath code)
        fe_set1(P.Z);
        ge_double(Rr, P);
    } else if (op == 7) {
        Rr = P;
    } else {  // scalar mult: b is a 32-byte scalar, plain double-and-add via Niels
        ge_niels q;
        ge_affine_to_niels(q, P.X, P.Y);
        ge_identity(Rr);
#pragma unroll 1
        for (int bit = 255; bit >= 0; bit--) {
            ge_double(Rr, Rr);
            if ((pb[bit >> 3] >> (bit & 7)) & 1) ge_madd(Rr, Rr, q, false);
        }
    }
    ge_compress(po, Rr);
}
