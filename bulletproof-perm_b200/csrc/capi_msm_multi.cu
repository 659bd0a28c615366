// capi_msm_multi.cu - C ABI of the batched variable-base MSM (bpp_msm_multi*, include/bpperm.h): `count` independent
// vartime_multiscalar_mul calls with ragged sizes, each over its own points, in a few launches on the context's stream;
// and its mixed form (bpp_msm_mixed*), which adds a static part over a tabled point set to every MSM.
#include "bpperm_internal.hpp"
#include "msm_multi_kernels.cuh"

namespace {

// The size classes (msm_multi_kernels.cuh): the kernel and its window width from the MSM's size, with the crossover
// measured (DESIGN.md 3.6, tools/msm_multi_bench.py).
enum mm_class { MM_STRAUS = 0, MM_PIPPENGER, MM_NCLASS };
const uint32_t mm_class_c[MM_NCLASS] = {4, MM_PIPPENGER_C};
mm_class mm_class_of(uint32_t n) { return n <= MM_STRAUS_MAX ? MM_STRAUS : MM_PIPPENGER; }

inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

struct mm_plan {
    uint64_t T = 0;
    uint32_t n_items[MM_NCLASS] = {}, first[MM_NCLASS] = {}, straus_max_n = 0;
    uint64_t windows = 0;             // window sums in all (wsum slots)
    uint64_t madd = 0, add = 0, dbl = 0;   // operation counts (every digit taken as non-zero)
    size_t starts_b = 0, msms_b = 0, plan_b = 0;   // host plan: starts | msms | items
};

// Fills ctx->mm_host with starts (count + 1) | msms (count) | items, each region 256-byte aligned, and the plan.
int mm_make_plan(bpp_ctx *ctx, size_t count, const uint32_t *sizes, mm_plan &pl) {
    uint64_t T = 0;
    for (size_t j = 0; j < count; j++) T += sizes[j];
    if (T >= (1ull << 31)) return BPP_ERR_INVALID_ARG;
    pl.T = T;
    // items per class, so that each class is one contiguous launch
    for (size_t j = 0; j < count; j++) {
        if (!sizes[j]) continue;
        const mm_class k = mm_class_of(sizes[j]);
        pl.n_items[k] += k == MM_STRAUS ? 1 : (sizes[j] + MM_CHUNK - 1) / MM_CHUNK;
    }
    uint32_t n_items = 0;
    for (int k = 0; k < MM_NCLASS; k++) {
        pl.first[k] = n_items;
        n_items += pl.n_items[k];
    }
    const size_t starts_b = pl.starts_b = al256((count + 1) * 4);
    const size_t msms_b = pl.msms_b = al256(count * sizeof(mm_msm));
    const size_t bytes = pl.plan_b = starts_b + msms_b + (size_t)n_items * sizeof(mm_item);
    if (ctx->mm_host.size() < bytes) ctx->mm_host.resize(bytes);
    uint32_t *starts = reinterpret_cast<uint32_t *>(ctx->mm_host.data());
    mm_msm *msms = reinterpret_cast<mm_msm *>(ctx->mm_host.data() + starts_b);
    mm_item *items = reinterpret_cast<mm_item *>(ctx->mm_host.data() + starts_b + msms_b);
    uint32_t fill[MM_NCLASS];
    for (int k = 0; k < MM_NCLASS; k++) fill[k] = pl.first[k];
    uint64_t t = 0, wofs = 0;
    for (size_t j = 0; j < count; j++) {
        const uint32_t n = sizes[j];
        starts[j] = (uint32_t)t;
        mm_msm m = {0, 0, 4, 0};
        if (n) {
            const mm_class k = mm_class_of(n);
            const uint32_t c = mm_class_c[k], W = mm_windows(c), B = 1u << (c - 1);
            const uint32_t chunks = k == MM_STRAUS ? 1 : (n + MM_CHUNK - 1) / MM_CHUNK;
            m = {(uint32_t)wofs, chunks, c, 0};
            for (uint32_t q = 0; q < chunks; q++) {
                const uint32_t t0 = (uint32_t)t + q * MM_CHUNK, len = n - q * MM_CHUNK < MM_CHUNK ? n - q * MM_CHUNK : MM_CHUNK;
                items[fill[k]++] = {t0, k == MM_STRAUS ? n : len, (uint32_t)wofs, 0};
                wofs += W;
            }
            if (k == MM_STRAUS) {
                if (n > pl.straus_max_n) pl.straus_max_n = n;
                pl.madd += 8ull * n;
                pl.add += (uint64_t)W * n;
            } else {
                pl.madd += (uint64_t)W * n;
                pl.add += (uint64_t)chunks * W * 2 * (B - 1);
            }
            pl.add += (uint64_t)chunks * W;      // Horner (and the chunk sums)
            pl.dbl += (uint64_t)c * (W - 1);
        }
        msms[j] = m;
        t += n;
    }
    starts[count] = (uint32_t)t;
    pl.windows = wofs;
    if (wofs >= (1ull << 32)) return BPP_ERR_OOM;
    return BPP_OK;
}

// Device bytes mm_run needs after the caller's own regions.
size_t mm_bytes(const mm_plan &pl, size_t count, bool enc) {
    return (enc ? al256(pl.T * 96) : 0) + al256(pl.plan_b) + al256(count * 4) + pl.windows * 128;
}

// Enqueues a call whose plan mm_make_plan made; the arena holds mm_bytes() from byte `base` on.  enc: the T x 32
// encodings (device) or NULL; then index (T, device) selects from `points`.  st_ext (bpp_msm_mixed*): count x 128 B
// extended points, MSM j's static part, added by the finish kernel (k_mm_finish_mixed instead of k_mm_finish).
int mm_run(bpp_ctx *ctx, const mm_plan &pl, size_t count, const uint32_t *d_scalars, const uint8_t *d_enc,
           const bpp_points *points, const uint32_t *d_index, uint8_t *d_out32, uint8_t *d_ok, size_t base,
           const uint32_t *d_st_ext = nullptr) {
    const size_t niels_b = d_enc ? al256(pl.T * 96) : 0;
    uint8_t *d = ctx->d_multi + base;
    uint32_t *d_niels = reinterpret_cast<uint32_t *>(d);
    d += niels_b;
    const uint32_t *d_starts = reinterpret_cast<const uint32_t *>(d);
    const mm_msm *d_msms = reinterpret_cast<const mm_msm *>(d + pl.starts_b);
    const mm_item *d_items = reinterpret_cast<const mm_item *>(d + pl.starts_b + pl.msms_b);
    CK(ctx, cudaMemcpyAsync(d, ctx->mm_host.data(), pl.plan_b, cudaMemcpyHostToDevice, ctx->stream));
    d += al256(pl.plan_b);
    uint32_t *d_bad = reinterpret_cast<uint32_t *>(d);
    d += al256(count * 4);
    uint32_t *d_wsum = reinterpret_cast<uint32_t *>(d);
    cudaStream_t s = ctx->stream;
    const uint32_t *niels = d_enc ? d_niels : points->niels;
    const uint32_t n_pts = d_enc ? (uint32_t)pl.T : (uint32_t)points->n;
    if (d_enc) {
        CK(ctx, cudaMemsetAsync(d_bad, 0, count * 4, s));
        if (pl.T) {
            k_mm_decode<<<(unsigned)((pl.T + 127) / 128), 128, 0, s>>>(d_enc, (uint32_t)pl.T, d_starts, (uint32_t)count, d_niels, d_bad);
            LAUNCH_CHECK(ctx);
        }
    }
    if (pl.n_items[MM_STRAUS]) {
        k_mm_straus<<<pl.n_items[MM_STRAUS], 64, (size_t)pl.straus_max_n * 8 * 128, s>>>(d_items + pl.first[MM_STRAUS], d_scalars, niels,
                                                                                        d_index, n_pts, d_wsum);
        LAUNCH_CHECK(ctx);
    }
    if (pl.n_items[MM_PIPPENGER]) {
        k_mm_pippenger<<<pl.n_items[MM_PIPPENGER], 64, 0, s>>>(d_items + pl.first[MM_PIPPENGER], d_scalars, niels, d_index, n_pts,
                                                                d_wsum);
        LAUNCH_CHECK(ctx);
    }
    const unsigned fin = (unsigned)((count + MM_THREADS_FINISH - 1) / MM_THREADS_FINISH);
    if (d_st_ext)
        k_mm_finish_mixed<<<fin, MM_THREADS_FINISH, 0, s>>>(d_msms, (uint32_t)count, d_wsum, d_st_ext, d_enc ? d_bad : nullptr,
                                                            d_out32, d_ok);
    else
        k_mm_finish<<<fin, MM_THREADS_FINISH, 0, s>>>(d_msms, (uint32_t)count, d_wsum, d_enc ? d_bad : nullptr, d_out32, d_ok);
    LAUNCH_CHECK(ctx);
    ctx->n_madd = pl.madd;
    ctx->n_add = pl.add;
    ctx->n_dbl = pl.dbl;
    return BPP_OK;
}

int mm_check_common(bpp_ctx *ctx, size_t count, const uint32_t *sizes, uint64_t &T) {
    if (!ctx || !sizes || count == 0 || count >= (1ull << 31)) return BPP_ERR_INVALID_ARG;
    T = 0;
    for (size_t j = 0; j < count; j++) T += sizes[j];
    if (T >= (1ull << 31)) return BPP_ERR_INVALID_ARG;
    return BPP_OK;
}

int mm_check_scalars(const uint8_t *scalars, uint64_t T) {
    for (uint64_t i = 0; i < T; i++)
        if (scalars[32 * i + 31] & 0x80) return BPP_ERR_SCALAR_RANGE;
    return BPP_OK;
}

// ---- bpp_msm_mixed*: a static part over a tabled sub-range plus a ragged dynamic part, per MSM ----------------
// The static part is bpp_msm_vartime_batch's table-gather launches, stopped at the extended sums (count x 128 B); the
// dynamic part is mm_run's decode and window-sum kernels; k_mm_finish_mixed adds the two per MSM and compresses.

// what the host sees, both forms
int mx_check(bpp_ctx *ctx, size_t count, const bpp_points *points, size_t off, size_t n_static, const uint32_t *sizes, uint64_t &T) {
    int rc = mm_check_common(ctx, count, sizes, T);
    if (rc) return rc;
    if (!points || n_static == 0 || n_static >= (1ull << 31) || (uint64_t)count * n_static >= (1ull << 31)) return BPP_ERR_INVALID_ARG;
    if (off > points->n || n_static > points->n - off) return BPP_ERR_LENGTH_MISMATCH;
    return BPP_OK;
}

// The arena from byte `own` on: the static extended points | their split partials | mm_run's regions.
struct mx_layout {
    size_t ext_b = 0, part_b = 0, mm_b = 0;
    size_t total(size_t own) const { return own + ext_b + part_b + mm_b; }
};
int mx_prepare(bpp_ctx *ctx, size_t count, bpp_points *points, size_t n_static, const uint32_t *sizes, mm_plan &pl, mx_layout &ly) {
    int rc;
    CK(ctx, cudaSetDevice(ctx->device));
    if (!points->fb_table && (rc = bpp_points_precompute(ctx, points, 8))) return rc;
    if ((rc = mm_make_plan(ctx, count, sizes, pl))) return rc;
    ly.ext_b = al256(count * 128);
    ly.part_b = al256(msm_table_part_bytes(ctx, points, n_static, count));
    ly.mm_b = mm_bytes(pl, count, true);
    return BPP_OK;
}
// Enqueues the call; the arena holds ly.total(own) bytes.  d_st_sc: count x n_static scalars with bit 255 clear.
int mx_run(bpp_ctx *ctx, size_t count, const bpp_points *points, size_t off, size_t n_static, const uint32_t *d_st_sc,
           const mm_plan &pl, const mx_layout &ly, const uint32_t *d_dyn_sc, const uint8_t *d_enc, uint8_t *d_out32, uint8_t *d_ok,
           size_t own) {
    uint32_t *d_ext = reinterpret_cast<uint32_t *>(ctx->d_multi + own);
    uint32_t *d_part = reinterpret_cast<uint32_t *>(ctx->d_multi + own + ly.ext_b);
    uint64_t t_madd = 0, t_add = 0;
    int rc = msm_table_ext(ctx, d_st_sc, points, off, n_static, count, d_ext, d_part, &t_madd, &t_add);
    if (rc) return rc;
    if ((rc = mm_run(ctx, pl, count, d_dyn_sc, d_enc, nullptr, nullptr, d_out32, d_ok, own + ly.ext_b + ly.part_b, d_ext))) return rc;
    ctx->n_madd += t_madd;
    ctx->n_add += t_add + count;   // and the finish kernel's static + dynamic add
    return BPP_OK;
}

}  // namespace

extern "C" int bpp_msm_multi_dev(bpp_ctx *ctx, size_t count, const uint32_t *sizes, const void *d_scalars,
                                 const void *d_points_enc, void *d_out32, void *d_ok) {
    uint64_t T = 0;
    int rc = mm_check_common(ctx, count, sizes, T);
    if (rc) return rc;
    if (!d_scalars || !d_points_enc || !d_out32 || !d_ok) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    mm_plan pl;
    if ((rc = mm_make_plan(ctx, count, sizes, pl))) return rc;
    if ((rc = grow(ctx, &ctx->d_multi, &ctx->cap_multi, mm_bytes(pl, count, true)))) return rc;
    return mm_run(ctx, pl, count, (const uint32_t *)d_scalars, (const uint8_t *)d_points_enc, nullptr, nullptr,
                  (uint8_t *)d_out32, (uint8_t *)d_ok, 0);
}

extern "C" int bpp_msm_multi_indexed_dev(bpp_ctx *ctx, size_t count, const uint32_t *sizes, const void *d_scalars,
                                         const bpp_points *points, const void *d_index, void *d_out32) {
    uint64_t T = 0;
    int rc = mm_check_common(ctx, count, sizes, T);
    if (rc) return rc;
    if (!d_scalars || !points || !d_index || !d_out32) return BPP_ERR_INVALID_ARG;
    if (T && points->n == 0) return BPP_ERR_LENGTH_MISMATCH;
    CK(ctx, cudaSetDevice(ctx->device));
    mm_plan pl;
    if ((rc = mm_make_plan(ctx, count, sizes, pl))) return rc;
    if ((rc = grow(ctx, &ctx->d_multi, &ctx->cap_multi, mm_bytes(pl, count, false)))) return rc;
    return mm_run(ctx, pl, count, (const uint32_t *)d_scalars, nullptr, points, (const uint32_t *)d_index, (uint8_t *)d_out32,
                  nullptr, 0);
}

extern "C" int bpp_msm_multi(bpp_ctx *ctx, size_t count, const uint32_t *sizes, const uint8_t *scalars,
                             const uint8_t *points_enc, uint8_t *out32, uint8_t *ok) {
    uint64_t T = 0;
    int rc = mm_check_common(ctx, count, sizes, T);
    if (rc) return rc;
    if (!scalars || !points_enc || !out32 || !ok) return BPP_ERR_INVALID_ARG;
    if ((rc = mm_check_scalars(scalars, T))) return rc;
    CK(ctx, cudaSetDevice(ctx->device));
    mm_plan pl;
    if ((rc = mm_make_plan(ctx, count, sizes, pl))) return rc;
    // arena: scalars | encodings | results | ok bytes, then mm_run's regions
    const size_t sc_b = al256(T * 32), out_b = al256(count * 32), ok_b = al256(count), own = 2 * sc_b + out_b + ok_b;
    if ((rc = grow(ctx, &ctx->d_multi, &ctx->cap_multi, own + mm_bytes(pl, count, true)))) return rc;
    uint8_t *d_sc = ctx->d_multi, *d_enc = d_sc + sc_b, *d_out = d_enc + sc_b, *d_ok = d_out + out_b;
    if (T) {
        CK(ctx, cudaMemcpyAsync(d_sc, scalars, T * 32, cudaMemcpyHostToDevice, ctx->stream));
        CK(ctx, cudaMemcpyAsync(d_enc, points_enc, T * 32, cudaMemcpyHostToDevice, ctx->stream));
    }
    if ((rc = mm_run(ctx, pl, count, (const uint32_t *)d_sc, d_enc, nullptr, nullptr, d_out, d_ok, own))) return rc;
    CK(ctx, cudaMemcpyAsync(out32, d_out, count * 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaMemcpyAsync(ok, d_ok, count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return BPP_OK;
}

extern "C" int bpp_msm_multi_indexed(bpp_ctx *ctx, size_t count, const uint32_t *sizes, const uint8_t *scalars,
                                     const bpp_points *points, const uint32_t *index, uint8_t *out32) {
    uint64_t T = 0;
    int rc = mm_check_common(ctx, count, sizes, T);
    if (rc) return rc;
    if (!scalars || !points || !index || !out32) return BPP_ERR_INVALID_ARG;
    for (uint64_t t = 0; t < T; t++)
        if (index[t] >= points->n) return BPP_ERR_LENGTH_MISMATCH;
    if ((rc = mm_check_scalars(scalars, T))) return rc;
    CK(ctx, cudaSetDevice(ctx->device));
    mm_plan pl;
    if ((rc = mm_make_plan(ctx, count, sizes, pl))) return rc;
    const size_t sc_b = al256(T * 32), ix_b = al256(T * 4), out_b = al256(count * 32), own = sc_b + ix_b + out_b;
    if ((rc = grow(ctx, &ctx->d_multi, &ctx->cap_multi, own + mm_bytes(pl, count, false)))) return rc;
    uint8_t *d_sc = ctx->d_multi, *d_ix = d_sc + sc_b, *d_out = d_ix + ix_b;
    if (T) {
        CK(ctx, cudaMemcpyAsync(d_sc, scalars, T * 32, cudaMemcpyHostToDevice, ctx->stream));
        CK(ctx, cudaMemcpyAsync(d_ix, index, T * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    if ((rc = mm_run(ctx, pl, count, (const uint32_t *)d_sc, nullptr, points, (const uint32_t *)d_ix, d_out, nullptr, own))) return rc;
    CK(ctx, cudaMemcpyAsync(out32, d_out, count * 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return BPP_OK;
}

int msm_scalars_low255(bpp_ctx *ctx, const void *src, uint64_t n, void *dst) {
    k_mm_scalars_low255<<<(unsigned)((2 * n + 127) / 128), 128, 0, ctx->stream>>>((const uint4 *)src, n, (uint4 *)dst);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}
extern "C" int bpp_msm_mixed_dev(bpp_ctx *ctx, size_t count, bpp_points *points, size_t off, size_t n_static,
                                 const void *d_static_scalars, const uint32_t *sizes, const void *d_dyn_scalars,
                                 const void *d_dyn_points_enc, void *d_out32, void *d_ok) {
    uint64_t T = 0;
    if (!d_static_scalars || !d_dyn_scalars || !d_dyn_points_enc || !d_out32 || !d_ok) return BPP_ERR_INVALID_ARG;
    int rc = mx_check(ctx, count, points, off, n_static, sizes, T);
    if (rc) return rc;
    mm_plan pl;
    mx_layout ly;
    if ((rc = mx_prepare(ctx, count, points, n_static, sizes, pl, ly))) return rc;
    // arena: the static scalars with bit 255 cleared, then mx_run's regions
    const uint64_t n_sc = (uint64_t)count * n_static;
    const size_t own = al256(n_sc * 32);
    if ((rc = grow(ctx, &ctx->d_multi, &ctx->cap_multi, ly.total(own)))) return rc;
    if ((rc = msm_scalars_low255(ctx, d_static_scalars, n_sc, ctx->d_multi))) return rc;
    return mx_run(ctx, count, points, off, n_static, (const uint32_t *)ctx->d_multi, pl, ly, (const uint32_t *)d_dyn_scalars,
                  (const uint8_t *)d_dyn_points_enc, (uint8_t *)d_out32, (uint8_t *)d_ok, own);
}

extern "C" int bpp_msm_mixed(bpp_ctx *ctx, size_t count, bpp_points *points, size_t off, size_t n_static,
                             const uint8_t *static_scalars, const uint32_t *sizes, const uint8_t *dyn_scalars,
                             const uint8_t *dyn_points_enc, uint8_t *out32, uint8_t *ok) {
    uint64_t T = 0;
    if (!static_scalars || !dyn_scalars || !dyn_points_enc || !out32 || !ok) return BPP_ERR_INVALID_ARG;
    int rc = mx_check(ctx, count, points, off, n_static, sizes, T);
    if (rc) return rc;
    const uint64_t n_sc = (uint64_t)count * n_static;
    if ((rc = mm_check_scalars(static_scalars, n_sc)) || (rc = mm_check_scalars(dyn_scalars, T))) return rc;
    mm_plan pl;
    mx_layout ly;
    if ((rc = mx_prepare(ctx, count, points, n_static, sizes, pl, ly))) return rc;
    // arena: static scalars | dynamic scalars | encodings | results | ok bytes, then mx_run's regions
    const size_t st_b = al256(n_sc * 32), sc_b = al256(T * 32), out_b = al256(count * 32), ok_b = al256(count),
                 own = st_b + 2 * sc_b + out_b + ok_b;
    if ((rc = grow(ctx, &ctx->d_multi, &ctx->cap_multi, ly.total(own)))) return rc;
    uint8_t *d_st = ctx->d_multi, *d_sc = d_st + st_b, *d_enc = d_sc + sc_b, *d_out = d_enc + sc_b, *d_ok = d_out + out_b;
    CK(ctx, cudaMemcpyAsync(d_st, static_scalars, n_sc * 32, cudaMemcpyHostToDevice, ctx->stream));
    if (T) {
        CK(ctx, cudaMemcpyAsync(d_sc, dyn_scalars, T * 32, cudaMemcpyHostToDevice, ctx->stream));
        CK(ctx, cudaMemcpyAsync(d_enc, dyn_points_enc, T * 32, cudaMemcpyHostToDevice, ctx->stream));
    }
    if ((rc = mx_run(ctx, count, points, off, n_static, (const uint32_t *)d_st, pl, ly, (const uint32_t *)d_sc, d_enc, d_out, d_ok,
                     own)))
        return rc;
    CK(ctx, cudaMemcpyAsync(out32, d_out, count * 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaMemcpyAsync(ok, d_ok, count, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return BPP_OK;
}
