// capi_core.cu - C ABI (include/bpperm.h): lifecycle, point tables, the Pippenger MSM, measurement and test hooks.
// No torch, no CPU fallback.
#include "bpperm_internal.hpp"
#include "msm_kernels.cuh"

extern "C" const char *bpp_strerror(int s) {
    switch (s) {
        case BPP_OK: return "ok";
        case BPP_ERR_NO_DEVICE: return "no CUDA device (this backend has no CPU fallback)";
        case BPP_ERR_CUDA: return "CUDA runtime error";
        case BPP_ERR_INVALID_ARG: return "invalid argument";
        case BPP_ERR_LENGTH_MISMATCH: return "scalars and points differ in length";
        case BPP_ERR_INVALID_POINT: return "invalid ristretto255 encoding";
        case BPP_ERR_SCALAR_RANGE: return "scalar has bit 255 set";
        case BPP_ERR_OOM: return "out of device memory";
        case BPP_ERR_VERIFICATION: return "verification failed";
        default: return "unknown status";
    }
}

extern "C" int bpp_init(int device, bpp_ctx **out) {
    if (!out) return BPP_ERR_INVALID_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device < 0 || device >= count) {
        cudaGetLastError();
        return BPP_ERR_NO_DEVICE;
    }
    bpp_ctx *ctx = new bpp_ctx();
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return BPP_ERR_NO_DEVICE; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return BPP_ERR_NO_DEVICE; }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    ctx->total_mem = prop.totalGlobalMem;
    if (prop.major != 10) {  // the library is built for sm_100a only
        delete ctx;
        return BPP_ERR_NO_DEVICE;
    }
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return BPP_ERR_CUDA; }
    ctx->own_stream = true;
    for (int i = 0; i <= BPP_PHASE_COUNT; i++) cudaEventCreate(&ctx->ev[i]);
    if (cudaMalloc((void **)&ctx->d_out, 256) != cudaSuccess || cudaMalloc((void **)&ctx->d_flag, 256) != cudaSuccess ||
        cudaMallocHost((void **)&ctx->h_out, 256) != cudaSuccess) {
        delete ctx;
        return BPP_ERR_OOM;
    }
    *out = ctx;
    return BPP_OK;
}

extern "C" void bpp_free(bpp_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    void *ptrs[] = {ctx->d_scalars, ctx->d_out, ctx->d_stage, ctx->d_flag, ctx->d_vec, ctx->d_small, ctx->d_multi};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    for (auto &sc : ctx->scr) {
        void *sp[] = {sc.d_counts, sc.d_offsets, sc.d_cursor, sc.d_entries, sc.d_partials, sc.d_long, sc.d_nlong,
                      sc.d_buckets, sc.d_segS, sc.d_segR, sc.d_gparts};
        for (void *p : sp)
            if (p) cudaFree(p);
        if (sc.ev_done) cudaEventDestroy(sc.ev_done);
    }
    if (ctx->comm) bpp_comm_free(ctx);
    if (ctx->h_out) cudaFreeHost(ctx->h_out);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    for (int i = 0; i <= BPP_PHASE_COUNT; i++)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->pipe_ready) {
        cudaStreamDestroy(ctx->s_sort);
        cudaStreamDestroy(ctx->s_bulk[0]);
        cudaStreamDestroy(ctx->s_bulk[1]);
        cudaStreamDestroy(ctx->s_final);
        cudaEventDestroy(ctx->ev_fork);
        for (int g = 0; g < BPP_MAX_GROUPS; g++) {
            cudaStreamDestroy(ctx->s_tail[g]);
            cudaEventDestroy(ctx->ev_sorted[g]);
            cudaEventDestroy(ctx->ev_acc[g]);
            cudaEventDestroy(ctx->ev_tail[g]);
        }
    }
    delete ctx;
}

extern "C" int bpp_set_stream(bpp_ctx *ctx, void *s) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = msm_wait_pending(ctx);
    if (rc) return rc;
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = (cudaStream_t)s;
    ctx->own_stream = false;
    return BPP_OK;
}
extern "C" int bpp_synchronize(bpp_ctx *ctx) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    if (int rc = msm_wait_pending(ctx)) return rc;
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return BPP_OK;
}
extern "C" const char *bpp_last_error(bpp_ctx *ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }
extern "C" uint64_t bpp_launch_count(bpp_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" int bpp_device_info(bpp_ctx *ctx, int *sm, int *maj, int *min, size_t *mem) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    if (sm) *sm = ctx->sm_count;
    if (maj) *maj = ctx->cc_major;
    if (min) *min = ctx->cc_minor;
    if (mem) *mem = ctx->total_mem;
    return BPP_OK;
}
extern "C" int bpp_device_clock_khz(bpp_ctx *ctx) {
    if (!ctx) return 0;
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
    return khz;
}
extern "C" int bpp_set_window_bits(bpp_ctx *ctx, int c) {
    if (!ctx || (c != 0 && (c < 4 || c > 16))) return BPP_ERR_INVALID_ARG;
    ctx->forced_c = c;
    return BPP_OK;
}
extern "C" int bpp_set_msm_groups(bpp_ctx *ctx, int groups) {
    if (!ctx || groups < 0 || groups > BPP_MAX_GROUPS) return BPP_ERR_INVALID_ARG;
    ctx->forced_groups = groups;
    ctx->n_forced_part = 0;
    return BPP_OK;
}

extern "C" int bpp_set_msm_tile(bpp_ctx *ctx, int tile_len) {
    if (!ctx || (tile_len != 0 && (tile_len < 8 || tile_len > 256))) return BPP_ERR_INVALID_ARG;
    ctx->forced_tile = tile_len;
    return BPP_OK;
}

extern "C" int bpp_set_msm_partition(bpp_ctx *ctx, const int *sizes, int count) {
    if (!ctx || count < 0 || count > BPP_MAX_GROUPS || (count && !sizes)) return BPP_ERR_INVALID_ARG;
    for (int i = 0; i < count; i++)
        if (sizes[i] < 1) return BPP_ERR_INVALID_ARG;
    for (int i = 0; i < count; i++) ctx->forced_part[i] = sizes[i];
    ctx->n_forced_part = count;
    return BPP_OK;
}

extern "C" int bpp_set_msm_trace(bpp_ctx *ctx, int on) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    ctx->trace = on != 0;
    return BPP_OK;
}

extern "C" int bpp_msm_trace_dump(bpp_ctx *ctx, char *buf, size_t cap) {
    if (!ctx || !buf || cap == 0) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaDeviceSynchronize());
    std::string out;
    for (size_t i = 0; i < ctx->trace_ev.size(); i++) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ctx->trace_ev[0].second, ctx->trace_ev[i].second);
        char line[96];
        snprintf(line, sizeof line, "%s %.1f\n", ctx->trace_ev[i].first.c_str(), ms * 1000.f);
        out += line;
    }
    snprintf(buf, cap, "%s", out.c_str());
    return BPP_OK;
}

extern "C" int bpp_set_profiling(bpp_ctx *ctx, int on) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    ctx->profiling = on != 0;
    return BPP_OK;
}
extern "C" int bpp_last_phase_ms(bpp_ctx *ctx, float ms[BPP_PHASE_COUNT]) {
    if (!ctx || !ms) return BPP_ERR_INVALID_ARG;
    if (ctx->profiling && ctx->events_pending) {  // the events of the last MSM were recorded on the stream
        CK(ctx, cudaEventSynchronize(ctx->ev[BPP_PHASE_COUNT]));
        for (int i = 0; i < BPP_PHASE_COUNT; i++) cudaEventElapsedTime(&ctx->phase_ms[i], ctx->ev[i], ctx->ev[i + 1]);
        ctx->events_pending = false;
    }
    for (int i = 0; i < BPP_PHASE_COUNT; i++) ms[i] = ctx->phase_ms[i];
    return BPP_OK;
}
extern "C" int bpp_last_op_counts(bpp_ctx *ctx, uint64_t *m, uint64_t *a, uint64_t *d) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    if (m) *m = ctx->n_madd;
    if (a) *a = ctx->n_add;
    if (d) *d = ctx->n_dbl;
    return BPP_OK;
}

// ---- points ----------------------------------------------------------------------------------
static size_t fmt_bytes(int fmt) {
    switch (fmt) {
        case BPP_FMT_COMPRESSED: return 32;
        case BPP_FMT_AFFINE: return 64;
        case BPP_FMT_DALEK_XYZT: return 160;
        default: return 0;
    }
}

extern "C" int bpp_points_upload(bpp_ctx *ctx, int fmt, const uint8_t *pts, size_t n, bpp_points **out) {
    if (!ctx || !out || (!pts && n) || n >= (1ull << 31)) return BPP_ERR_INVALID_ARG;
    size_t eb = fmt_bytes(fmt);
    if (!eb) return BPP_ERR_INVALID_ARG;
    *out = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    bpp_points *p = new bpp_points();
    p->n = n;
    if (n == 0) { *out = p; return BPP_OK; }
    int rc = grow(ctx, &ctx->d_stage, &ctx->cap_stage, n * eb);
    if (rc) { delete p; return rc; }
    if (cudaMalloc((void **)&p->niels, n * 96) != cudaSuccess) {
        cudaGetLastError();
        delete p;
        return BPP_ERR_OOM;
    }
    cudaError_t e = cudaMemcpyAsync(ctx->d_stage, pts, n * eb, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(ctx->d_flag, 0, 4, ctx->stream);
    if (e != cudaSuccess) {
        ctx->last_error = cudaGetErrorString(e);
        cudaFree(p->niels);
        delete p;
        return BPP_ERR_CUDA;
    }
    unsigned blocks = (unsigned)((n + 127) / 128);
    if (fmt == BPP_FMT_COMPRESSED)
        k_decompress_to_niels<<<blocks, 128, 0, ctx->stream>>>(ctx->d_stage, (uint32_t)n, p->niels, ctx->d_flag);
    else if (fmt == BPP_FMT_AFFINE)
        k_affine_to_niels<<<blocks, 128, 0, ctx->stream>>>(ctx->d_stage, (uint32_t)n, p->niels);
    else
        k_dalek_xyzt_to_niels<<<blocks, 128, 0, ctx->stream>>>((const unsigned long long *)ctx->d_stage, (uint32_t)n,
                                                             p->niels);
    ctx->launches++;
    uint32_t bad = 0;
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(&bad, ctx->d_flag, 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        ctx->last_error = cudaGetErrorString(e);
        cudaFree(p->niels);
        delete p;
        return BPP_ERR_CUDA;
    }
    if (bad) {
        cudaFree(p->niels);
        delete p;
        return BPP_ERR_INVALID_POINT;
    }
    *out = p;
    return BPP_OK;
}

extern "C" int bpp_points_from_uniform(bpp_ctx *ctx, const uint8_t *bytes64, size_t n, bpp_points **out) {
    if (!ctx || !out || !bytes64 || n == 0 || n >= (1ull << 31)) return BPP_ERR_INVALID_ARG;
    *out = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = grow(ctx, &ctx->d_stage, &ctx->cap_stage, n * 64);
    if (rc) return rc;
    bpp_points *p = new bpp_points();
    p->n = n;
    if (cudaMalloc((void **)&p->niels, n * 96) != cudaSuccess) {
        cudaGetLastError();
        delete p;
        return BPP_ERR_OOM;
    }
    cudaError_t e = cudaMemcpyAsync(ctx->d_stage, bytes64, n * 64, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        k_from_uniform_to_niels<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(ctx->d_stage, (uint32_t)n, p->niels);
        ctx->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        ctx->last_error = cudaGetErrorString(e);
        cudaFree(p->niels);
        delete p;
        return BPP_ERR_CUDA;
    }
    *out = p;
    return BPP_OK;
}

extern "C" int bpp_points_compress(bpp_ctx *ctx, const bpp_points *points, size_t off, size_t n, uint8_t *out32) {
    if (!ctx || !points || !out32 || n == 0) return BPP_ERR_INVALID_ARG;
    if (off + n > points->n) return BPP_ERR_LENGTH_MISMATCH;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = grow(ctx, &ctx->d_stage, &ctx->cap_stage, n * 32);
    if (rc) return rc;
    k_niels_compress<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(points->niels + 24 * off, (uint32_t)n, ctx->d_stage);
    LAUNCH_CHECK(ctx);
    CK(ctx, cudaMemcpyAsync(out32, ctx->d_stage, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return BPP_OK;
}

extern "C" void bpp_points_free(bpp_ctx *ctx, bpp_points *p) {
    if (!p) return;
    if (ctx) {
        cudaSetDevice(ctx->device);
        msm_wait_pending(ctx);   // a submitted MSM may still be reading the table on the side streams
        cudaStreamSynchronize(ctx->stream);
    }
    if (p->niels) cudaFree(p->niels);
    if (p->fb_table) cudaFree(p->fb_table);
    delete p;
}
extern "C" size_t bpp_points_len(const bpp_points *p) { return p ? p->n : 0; }

// ---- MSM ---------------------------------------------------------------------------------------
static int pick_window(size_t n) {
    // Measured on B200 (tools/window_tune.py, 2^10..2^21 points, every c in 8..16): below ~2^17 points the MSM
    // is bound by its dependent chains (node merges + c*(W-1) Horner doublings), which c = 11 keeps shortest
    // once the buckets fit (c = 8 for tiny inputs); from there the accumulate's W*n mixed adds decide:
    // c = 15 below ~2^20 points, c = 16 from there (equal at 2^20; 16 keeps W*n exact for 252-bit scalars).  (Odd widths win over their even neighbours because
    // W = ceil(256/c) drops at 11, 13, 15.)
    if (n <= 1500) return 8;
    if (n <= 96000) return 11;   // crossover between 2^16 (c = 11: 0.638 vs 0.654 ms) and 2^17 (c = 15: 0.764 vs 0.795 ms)
    if (n < 1000000) return 15;
    return 16;
}

// Side streams and events of the pipelined MSM, created on first use.
static int msm_pipeline_init(bpp_ctx *ctx) {
    if (ctx->pipe_ready) return BPP_OK;
    int lo = 0, hi = 0;
    CK(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));  // hi = numerically lowest = most urgent
    // (the sort at the accumulate's priority was measured: 1.84 ms per submitted 2^20-point MSM instead of 1.71)
    CK(ctx, cudaStreamCreateWithPriority(&ctx->s_sort, cudaStreamNonBlocking, hi));
    CK(ctx, cudaStreamCreateWithPriority(&ctx->s_bulk[0], cudaStreamNonBlocking, lo));
    CK(ctx, cudaStreamCreateWithPriority(&ctx->s_bulk[1], cudaStreamNonBlocking, lo));
    CK(ctx, cudaStreamCreateWithPriority(&ctx->s_final, cudaStreamNonBlocking, hi));
    for (int g = 0; g < BPP_MAX_GROUPS; g++) {
        CK(ctx, cudaStreamCreateWithPriority(&ctx->s_tail[g], cudaStreamNonBlocking, hi));
        CK(ctx, cudaEventCreateWithFlags(&ctx->ev_sorted[g], cudaEventDisableTiming));
        CK(ctx, cudaEventCreateWithFlags(&ctx->ev_acc[g], cudaEventDisableTiming));
        CK(ctx, cudaEventCreateWithFlags(&ctx->ev_tail[g], cudaEventDisableTiming));
    }
    CK(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    ctx->pipe_ready = true;
    return BPP_OK;
}

// Window groups of an n-point MSM, top group first (sizes sum to W; one group = everything in order on the
// caller's stream).  Measured on B200 (tools/msm_groups.py, tools/msm_trace.py): the pipeline pays once the
// accumulate of one group is long enough to hide the dependent tail (fix-up, node merges, Horner) of the previous
// one; a small first group starts the accumulate early and a small last group leaves a short tail.
static int pick_partition(const bpp_ctx *ctx, size_t n, int W, bool join, int groups, int part[BPP_MAX_GROUPS]) {
    if (ctx->n_forced_part && !ctx->profiling) {
        int sum = 0;
        for (int i = 0; i < ctx->n_forced_part; i++) sum += ctx->forced_part[i];
        if (sum == W) {
            for (int i = 0; i < ctx->n_forced_part; i++) part[i] = ctx->forced_part[i];
            return ctx->n_forced_part;
        }
    }
    if (!ctx->forced_groups && !groups && !ctx->profiling && W >= 8 &&
        n >= (join ? BPP_PIPELINE_MIN_POINTS : BPP_PIPELINE_MIN_POINTS_SUBMIT)) {
        // measured best of the partitions tried at 2^18..2^22 points (profiles/r1_msm_partitions.md): an eighth of the
        // windows first and last, the rest in two halves (16 windows: 2, 6, 6, 2)
        if (!join && n >= BPP_TILE64_MIN_POINTS) {   // very large submitted MSMs: two halves (2^22: 5.81 -> 5.62 ms)
            part[0] = W / 2; part[1] = W - W / 2;
            return 2;
        }
        const int edge = W / 8, mid = W - 2 * edge;
        part[0] = edge; part[1] = (mid + 1) / 2; part[2] = mid / 2; part[3] = edge;
        return 4;
    }
    int G = ctx->forced_groups ? ctx->forced_groups : (groups ? groups : 1);
    if (G > W) G = W;
    if (G > BPP_MAX_GROUPS) G = BPP_MAX_GROUPS;
    if (ctx->profiling || G < 1) G = 1;  // the per-phase events describe the in-order pipeline
    for (int g = 0; g < G; g++) part[g] = (W - (W / G) * G > g) ? W / G + 1 : W / G;
    return G;
}

// The caller's stream waits for every MSM that was submitted and not yet waited for (keep_latest: except the one
// submitted last, which stays in flight).
int msm_wait_pending(bpp_ctx *ctx, bool keep_latest) {
    for (int i = 0; i < 2; i++) {
        bpp_ctx::msm_scratch &sc = ctx->scr[i];
        if (sc.pending && !(keep_latest && i == ctx->slot)) {
            CK(ctx, cudaStreamWaitEvent(ctx->stream, sc.ev_done, 0));
            sc.pending = false;
        }
    }
    return BPP_OK;
}

// Tuning hook (BPP_ACC_SMEM=<bytes>): unused dynamic shared memory requested by the accumulate launch, which caps its
// resident blocks per SM below the four its 128 registers allow (e.g. 60000 -> three) and so leaves register-file room
// for the sort blocks of the next window group / the next submitted MSM.  0 (default) = no cap.
static size_t msm_acc_pad_smem() {
    static long v = -1;
    if (v < 0) {
        const char *e = getenv("BPP_ACC_SMEM");
        v = e ? atol(e) : 0;
        if (v > 48 * 1024) cudaFuncSetAttribute(k_bucket_accum, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)v);
    }
    return (size_t)v;
}
// Enqueues one MSM.  join = true: the result is in d_out in stream order on the caller's stream when the call returns
// (the classic contract).  join = false (bpp_msm_submit_dev): the caller's stream is not made to wait; the result is
// valid after bpp_msm_wait, and up to two submitted MSMs are in flight (the tail of one beside the sort and
// accumulate of the next).
int msm_enqueue(bpp_ctx *ctx, const uint32_t *d_scalars, const bpp_points *pts, size_t off, size_t n, uint8_t *d_out,
                int do_compress, bool join, int groups) {
    const int c = ctx->forced_c ? ctx->forced_c : pick_window(n);
    const int W = (256 + c - 1) / c;
    const uint32_t B = 1u << (c - 1);
    const size_t WB = (size_t)W * B;
    // reduction plan (msm_kernels.cuh): level 0 merges 8 buckets per THREAD (the GPU is full: 2^(c-1)*W buckets);
    // after that few nodes are left and the work is a dependent chain, so a QUAD of lanes carries each node:
    // quad-serial merges of 8 while more than 1024 nodes per window remain, then block merges of 32 down to one root
    struct level { int kind; uint32_t L, T_in, T_out, loglen; };   // kind 0 thread-serial, 1 quad-serial, 2 quad block merge
    level plan[10];
    int n_levels = 0;
    uint32_t T = B, loglen = 0, max_T_out = 0;
    while (T > 1) {
        level lv;
        if (n_levels == 0 && T >= 64) { lv.kind = 0; lv.L = 8; lv.T_out = T / 8; }
        else if (T > 1024) { lv.kind = 1; lv.L = 8; lv.T_out = T / 8; }
        else { lv.kind = 2; lv.L = 32; lv.T_out = (T + 31) / 32; }
        lv.T_in = T;
        lv.loglen = loglen;
        plan[n_levels++] = lv;
        if (lv.T_out > max_T_out) max_T_out = lv.T_out;
        T = lv.T_out;
        loglen += lv.kind == 2 ? 5 : 3;
    }
    // node storage (S and A each): two ping-pong halves; inside a half every window owns max_T_out nodes, so the
    // window groups of the pipelined form (each at its own level at any moment) never share storage
    const size_t node_elems = (size_t)W * max_T_out * 32;
    int part[BPP_MAX_GROUPS];
    const int G = pick_partition(ctx, n, W, join, groups, part);
    int rc;
    if (G > 1 && (rc = msm_pipeline_init(ctx))) return rc;
    ctx->slot ^= 1;
    bpp_ctx::msm_scratch &sc = ctx->scr[ctx->slot];
    cudaStream_t s = ctx->stream;
    if (!sc.ev_done) {
        CK(ctx, cudaEventCreateWithFlags(&sc.ev_done, cudaEventDisableTiming));
        CK(ctx, cudaMalloc((void **)&sc.d_gparts, 128 * BPP_MAX_GROUPS));
        CK(ctx, cudaMalloc((void **)&sc.d_nlong, 4 * BPP_MAX_GROUPS));
    }
    // the slot's previous MSM (two submissions ago) must be done before its scratch is reused (or reallocated)
    if (sc.pending) {
        CK(ctx, cudaStreamWaitEvent(s, sc.ev_done, 0));
        sc.pending = false;
    }
    const uint32_t tile_len = ctx->forced_tile ? (uint32_t)ctx->forced_tile : (n >= BPP_TILE64_MIN_POINTS ? 64u : 32u);
    const uint32_t tpw = (uint32_t)((n + tile_len - 1) / tile_len);
    const size_t total_tiles = (size_t)W * tpw;
    // Hot-bucket queue: a bucket is queued when it spans more than BPP_LONG_SPAN tiles, so one window holds at most
    // tpw / BPP_LONG_SPAN + 1 of them.  Every window group owns a DISJOINT region sized for that worst case (the groups'
    // fix-up kernels run concurrently on different streams).
    const size_t long_per_window = tpw / BPP_LONG_SPAN + 1, long_total = (size_t)W * long_per_window;
    // Scratch of BOTH slots is grown together (the next call uses the other slot: without this its first use would
    // allocate - and synchronise the device - in the middle of somebody's pipeline).
    auto grow_slot = [&](bpp_ctx::msm_scratch &x) -> int {
        const bool must_grow = WB > x.cap_wb || WB > x.cap_offsets || WB > x.cap_cursor || (size_t)W * n > x.cap_entries ||
                               total_tiles * 64 > x.cap_partials || WB * 32 > x.cap_buckets || 2 * node_elems > x.cap_seg ||
                               long_total > x.cap_long;
        if (!must_grow) return BPP_OK;
        CK(ctx, cudaDeviceSynchronize());   // nothing in flight may still use what is freed below
        int r;
        if ((r = grow(ctx, &x.d_counts, &x.cap_wb, WB))) return r;
        if ((r = grow(ctx, &x.d_offsets, &x.cap_offsets, WB))) return r;
        if ((r = grow(ctx, &x.d_cursor, &x.cap_cursor, WB))) return r;
        if ((r = grow(ctx, &x.d_entries, &x.cap_entries, (size_t)W * n))) return r;
        if ((r = grow(ctx, &x.d_partials, &x.cap_partials, total_tiles * 2 * 32))) return r;
        if ((r = grow(ctx, &x.d_long, &x.cap_long, long_total))) return r;
        if ((r = grow(ctx, &x.d_buckets, &x.cap_buckets, WB * 32))) return r;
        if (2 * node_elems > x.cap_seg) {   // two ping-pong buffers in each of segS / segR
            const size_t need = 2 * node_elems;
            if (x.d_segS) cudaFree(x.d_segS);
            if (x.d_segR) cudaFree(x.d_segR);
            x.d_segS = x.d_segR = nullptr;
            x.cap_seg = 0;
            CK(ctx, cudaMalloc((void **)&x.d_segS, need * 4));
            CK(ctx, cudaMalloc((void **)&x.d_segR, need * 4));
            x.cap_seg = need;
        }
        return BPP_OK;
    };
    if ((rc = grow_slot(sc))) return rc;
    if (n >= BPP_PIPELINE_MIN_POINTS_SUBMIT && (rc = grow_slot(ctx->scr[ctx->slot ^ 1]))) return rc;

    const bool prof = ctx->profiling && G == 1;
    const uint32_t *niels = pts->niels + 24 * off;
    unsigned sb = (unsigned)((n + 255) / 256);
    // Pipelined form: the sort kernels run grid-stride on two blocks per SM.  Their threads mostly wait on the L2, and
    // the accumulate owns the whole register file (4 blocks x 128 threads x 128 registers per SM), so every resident
    // sort block displaces accumulate work; a small resident set does the same L2-bound work while holding few SM
    // slots.  Measured (submitted form): 2^21 points 3.27 -> 3.10 ms, 2^22 6.50 -> 6.14 ms, 2^20 and below unchanged.
    if (G > 1 && BPP_SORT_BLOCKS_PER_SM * (unsigned)ctx->sm_count < sb) sb = BPP_SORT_BLOCKS_PER_SM * (unsigned)ctx->sm_count;
    uint64_t red_add = 0, red_dbl = 0;
    if (prof) cudaEventRecord(ctx->ev[0], s);
    if (ctx->trace) {
        for (auto &pe : ctx->trace_ev) cudaEventDestroy(pe.second);
        ctx->trace_ev.clear();
    }
    trace_mark(ctx, s, "start", 0);
    // Pipelined form: nothing but the fork and (join) the final wait touches the caller's stream.
    //   s_sort (urgent)     sort of group 0, 1, 2, ... in order: runs ahead of the accumulates
    //   s_bulk[g & 1] (low) accumulate of group g: the work that fills the GPU; alternating streams let the last,
    //                       partly filled wave of one group run beside the first wave of the next
    //   s_tail[g] (urgent)  fix-up, bucket reduction, Horner and the doublings to the group's weight: dependent
    //                       chains that take the SM slots they need as accumulate blocks retire
    //   s_final (urgent)    sum of the group partials, compress
    cudaStream_t s_sort = G > 1 ? ctx->s_sort : s;
    if (G > 1) {
        CK(ctx, cudaEventRecord(ctx->ev_fork, s));
        CK(ctx, cudaStreamWaitEvent(s_sort, ctx->ev_fork, 0));
    }
    CK(ctx, cudaMemsetAsync(sc.d_counts, 0, WB * 4, s_sort));
    CK(ctx, cudaMemsetAsync(sc.d_nlong, 0, 4 * BPP_MAX_GROUPS, s_sort));
    // Window groups from the top down: the top group's partial needs the most doublings to reach its weight, and
    // they run beside the accumulate of the groups below.  With G == 1 every stream below is the caller's.
    int w_hi = W;
    for (int g = 0; g < G; g++) {
        const int Wg = part[g];
        const int w0 = w_hi - Wg;
        w_hi = w0;
        cudaStream_t s_tail = G > 1 ? ctx->s_tail[g] : s, s_acc = G > 1 ? ctx->s_bulk[g & 1] : s;
        uint32_t *counts = sc.d_counts + (size_t)w0 * B, *offsets = sc.d_offsets + (size_t)w0 * B;
        uint32_t *ends = sc.d_cursor + (size_t)w0 * B, *entries = sc.d_entries + (size_t)w0 * n;
        uint32_t *buckets = sc.d_buckets + (size_t)w0 * B * 32, *partials = sc.d_partials + (size_t)w0 * tpw * 64;
        uint32_t *long_list = sc.d_long + (size_t)w0 * long_per_window, *d_nlong = sc.d_nlong + g;
        const uint32_t group_tiles = (uint32_t)Wg * tpw, group_buckets = (uint32_t)Wg * B;
        // sort: recode + histogram, scan, counting-sort scatter (absolute window numbers: the recoding carry
        // ripples up from window 0)
        trace_mark(ctx, s_sort, "sort>", g);
        {
            k_digit_hist<<<sb, 256, 0, s_sort>>>(d_scalars, (uint32_t)n, c, w0, w0 + Wg, sc.d_counts);
            LAUNCH_CHECK(ctx);
            trace_mark(ctx, s_sort, "hist.", g);
            if (prof) cudaEventRecord(ctx->ev[1], s);
            k_window_scan<<<Wg, 1024, 0, s_sort>>>(counts, B, offsets, ends, 0);
            LAUNCH_CHECK(ctx);
            if (prof) cudaEventRecord(ctx->ev[2], s);
            k_digit_scatter<<<sb, 256, 0, s_sort>>>(d_scalars, (uint32_t)n, c, w0, w0 + Wg, sc.d_cursor, sc.d_entries);
            LAUNCH_CHECK(ctx);
        }
        if (prof) cudaEventRecord(ctx->ev[3], s);
        trace_mark(ctx, s_sort, "sort.", g);
        if (G > 1) {
            CK(ctx, cudaEventRecord(ctx->ev_sorted[g], s_sort));
            CK(ctx, cudaStreamWaitEvent(s_acc, ctx->ev_sorted[g], 0));
        }
        trace_mark(ctx, s_acc, "accum>", g);
        k_bucket_accum<<<(group_tiles + BPP_ACC_THREADS - 1) / BPP_ACC_THREADS, BPP_ACC_THREADS, msm_acc_pad_smem(), s_acc>>>(
            niels, entries, offsets, ends, (uint32_t)n, B, tpw, group_tiles, tile_len, buckets, partials);
        LAUNCH_CHECK(ctx);
        if (prof) cudaEventRecord(ctx->ev[4], s);
        trace_mark(ctx, s_acc, "accum.", g);
        if (G > 1) {
            CK(ctx, cudaEventRecord(ctx->ev_acc[g], s_acc));
            CK(ctx, cudaStreamWaitEvent(s_tail, ctx->ev_acc[g], 0));
        }
        trace_mark(ctx, s_tail, "tail>", g);
        k_bucket_fixup<<<(group_buckets + 127) / 128, 128, 0, s_tail>>>(offsets, ends, B, tpw, group_buckets, tile_len, partials,
                                                                       buckets, long_list, d_nlong);
        LAUNCH_CHECK(ctx);
        k_bucket_fixup_long<<<ctx->sm_count * 2, 128, 0, s_tail>>>(offsets, ends, B, tpw, tile_len, partials, buckets, long_list,
                                                                  d_nlong);
        LAUNCH_CHECK(ctx);
        trace_mark(ctx, s_tail, "fixup.", g);
        const uint32_t *curS = buckets, *curA = nullptr;
        for (int i = 0; i < n_levels; i++) {
            const level &lv = plan[i];
            uint32_t *oS = sc.d_segS + (i & 1) * node_elems + (size_t)w0 * max_T_out * 32;
            uint32_t *oA = sc.d_segR + (i & 1) * node_elems + (size_t)w0 * max_T_out * 32;
            const uint32_t n_out = (uint32_t)Wg * lv.T_out;
            if (lv.kind == 0) {
                k_node_merge_serial<<<(n_out + 127) / 128, 128, 0, s_tail>>>(curS, curA, lv.L, lv.loglen, n_out, oS, oA);
                red_add += (uint64_t)n_out * (2 * lv.L - 3 + (curA ? lv.L : 0));
                red_dbl += (uint64_t)n_out * lv.loglen;
            } else if (lv.kind == 1) {
                k_node_merge_quad_serial<<<(4 * n_out + 127) / 128, 128, 0, s_tail>>>(curS, curA, lv.L, lv.loglen, n_out, oS, oA);
                red_add += (uint64_t)n_out * (3 * lv.L - 3);
                red_dbl += (uint64_t)n_out * lv.loglen;
            } else {
                k_node_merge_quad_block<<<dim3(lv.T_out, Wg), 128, 0, s_tail>>>(curS, curA, lv.T_in, lv.loglen, lv.T_out, oS, oA);
                red_add += (uint64_t)Wg * lv.T_out * (2 * (uint64_t)lv.T_in / lv.T_out + 1);  // useful additions
                red_dbl += (uint64_t)Wg * lv.T_out * lv.loglen;
            }
            LAUNCH_CHECK(ctx);
            trace_mark(ctx, s_tail, i == 0 ? "merge0." : "merge.", g);
            curS = oS;
            curA = oA;
        }
        if (prof) cudaEventRecord(ctx->ev[5], s);
        if (G == 1) {
            k_msm_finish<<<1, 32, 0, s>>>(curS, curA, c, W, 0, do_compress, d_out);
            LAUNCH_CHECK(ctx);
        } else {
            // Horner inside the group, then c*w0 doublings to the group's weight; raw point to d_gparts[g]
            k_msm_finish<<<1, 32, 0, s_tail>>>(curS, curA, c, Wg, c * w0, 0, sc.d_gparts + 128 * g);
            LAUNCH_CHECK(ctx);
            CK(ctx, cudaEventRecord(ctx->ev_tail[g], s_tail));
        }
        trace_mark(ctx, s_tail, "finish.", g);
    }
    if (G > 1) {
        for (int g = 0; g < G; g++) CK(ctx, cudaStreamWaitEvent(ctx->s_final, ctx->ev_tail[g], 0));
        k_points_sum_finish<<<1, 32, 0, ctx->s_final>>>((const uint32_t *)sc.d_gparts, (uint32_t)G, do_compress, d_out);
        LAUNCH_CHECK(ctx);
        trace_mark(ctx, ctx->s_final, "end", 0);
        CK(ctx, cudaEventRecord(sc.ev_done, ctx->s_final));
        sc.pending = true;
        if (join && (rc = msm_wait_pending(ctx))) return rc;
    } else {
        trace_mark(ctx, s, "end", 0);
        if (!join) {   // in order on the caller's stream: nothing to wait for, but the slot's reuse rule stays uniform
            CK(ctx, cudaEventRecord(sc.ev_done, s));
        }
    }
    if (prof) { cudaEventRecord(ctx->ev[6], s); ctx->events_pending = true; }
    ctx->n_madd = (uint64_t)W * n;
    ctx->n_add = (uint64_t)W * (B < tpw ? B : tpw) /* fix-up of buckets cut by tile boundaries (upper bound) */ +
                 red_add + 2 * (uint64_t)W + (G > 1 ? G - 1 : 0);
    ctx->n_dbl = (uint64_t)c * (W - 1) + red_dbl;  // the useful Horner doublings (the grouped form spends more, off the critical path)
    return BPP_OK;
}


static int check_scalars_host(const uint8_t *scalars, size_t n) {
    for (size_t i = 0; i < n; i++)
        if (scalars[32 * i + 31] & 0x80) return BPP_ERR_SCALAR_RANGE;
    return BPP_OK;
}

static int empty_msm_result(uint8_t out32[32], uint8_t *out_ext) {
    memset(out32, 0, 32);  // identity compresses to 32 zero bytes
    if (out_ext) {
        memset(out_ext, 0, 128);
        out_ext[32] = 1;  // Y = 1
        out_ext[64] = 1;  // Z = 1
    }
    return BPP_OK;
}

extern "C" int bpp_msm_vartime_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n,
                                   void *d_out) {
    if (!ctx || !d_scalars || !points || !d_out || n == 0) return BPP_ERR_INVALID_ARG;
    if (off + n > points->n) return BPP_ERR_LENGTH_MISMATCH;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc = msm_enqueue(ctx, (const uint32_t *)d_scalars, points, off, n, (uint8_t *)d_out, 1);
    return rc;
}

extern "C" int bpp_msm_submit_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n,
                                  void *d_out) {
    if (!ctx || !d_scalars || !points || !d_out || n == 0) return BPP_ERR_INVALID_ARG;
    if (off + n > points->n) return BPP_ERR_LENGTH_MISMATCH;
    CK(ctx, cudaSetDevice(ctx->device));
    return msm_enqueue(ctx, (const uint32_t *)d_scalars, points, off, n, (uint8_t *)d_out, 1, false);
}

extern "C" int bpp_msm_submit_partial_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off,
                                          size_t n, void *d_partial) {
    if (!ctx || !d_scalars || !points || !d_partial || n == 0) return BPP_ERR_INVALID_ARG;
    if (off + n > points->n) return BPP_ERR_LENGTH_MISMATCH;
    CK(ctx, cudaSetDevice(ctx->device));
    return msm_enqueue(ctx, (const uint32_t *)d_scalars, points, off, n, (uint8_t *)d_partial, 0, false);
}

extern "C" int bpp_msm_wait(bpp_ctx *ctx) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    return msm_wait_pending(ctx);
}

extern "C" int bpp_msm_wait_previous(bpp_ctx *ctx) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    return msm_wait_pending(ctx, true);
}

extern "C" int bpp_msm_partial_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n,
                                   void *d_partial) {
    if (!ctx || !d_scalars || !points || !d_partial || n == 0) return BPP_ERR_INVALID_ARG;
    if (off + n > points->n) return BPP_ERR_LENGTH_MISMATCH;
    CK(ctx, cudaSetDevice(ctx->device));
    return msm_enqueue(ctx, (const uint32_t *)d_scalars, points, off, n, (uint8_t *)d_partial, 0);
}

extern "C" int bpp_points_sum_compress_dev(bpp_ctx *ctx, const void *d_partials, size_t g, void *d_out32) {
    if (!ctx || !d_partials || !d_out32 || g == 0) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    k_points_sum_compress<<<1, 32, 0, ctx->stream>>>((const uint32_t *)d_partials, (uint32_t)g, (uint8_t *)d_out32);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}

extern "C" int bpp_msm_vartime(bpp_ctx *ctx, const uint8_t *scalars, size_t n_scalars, const bpp_points *points,
                               size_t off, size_t n, uint8_t out32[32], uint8_t *out_ext) {
    if (!ctx || !points || !out32 || (!scalars && n)) return BPP_ERR_INVALID_ARG;
    if (n_scalars != n || off + n > points->n) return BPP_ERR_LENGTH_MISMATCH;
    if (n == 0) return empty_msm_result(out32, out_ext);
    int rc = check_scalars_host(scalars, n);
    if (rc) return rc;
    CK(ctx, cudaSetDevice(ctx->device));
    if (points->fb_table && !out_ext && n <= BPP_TABLE_MSM_MAX_POINTS)   // precomputed points: no buckets, no doublings
        return bpp_msm_vartime_batch(ctx, scalars, 1, const_cast<bpp_points *>(points), off, n, out32);
    if ((rc = grow(ctx, &ctx->d_scalars, &ctx->cap_scalars, n * 8))) return rc;
    CK(ctx, cudaMemcpyAsync(ctx->d_scalars, scalars, n * 32, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = msm_enqueue(ctx, ctx->d_scalars, points, off, n, ctx->d_out, 1))) return rc;
    CK(ctx, cudaMemcpyAsync(ctx->h_out, ctx->d_out, 160, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(out32, ctx->h_out, 32);
    if (out_ext) {
        // canonicalise the four raw field elements on the host: value mod p, little endian
        for (int k = 0; k < 4; k++) {
            // 256-bit value v (may be >= p): subtract p up to twice (v < 2^256 < 3p)
            uint32_t v[8];
            memcpy(v, ctx->h_out + 32 + 32 * k, 32);
            static const uint32_t P[8] = {0xffffffedu, 0xffffffffu, 0xffffffffu, 0xffffffffu,
                                          0xffffffffu, 0xffffffffu, 0xffffffffu, 0x7fffffffu};
            for (int round = 0; round < 2; round++) {
                uint32_t t[8];
                int64_t borrow = 0;
                for (int i = 0; i < 8; i++) {
                    int64_t d = (int64_t)v[i] - (int64_t)P[i] + borrow;
                    t[i] = (uint32_t)d;
                    borrow = d >> 32;
                }
                if (borrow == 0) memcpy(v, t, 32);
            }
            memcpy(out_ext + 32 * k, v, 32);
        }
    }
    return BPP_OK;
}

extern "C" int bpp_msm_vartime_host(bpp_ctx *ctx, const uint8_t *scalars, size_t n_scalars, int fmt, const uint8_t *pts,
                                    size_t n_points, uint8_t out32[32]) {
    if (!ctx || !out32) return BPP_ERR_INVALID_ARG;
    if (n_scalars != n_points) return BPP_ERR_LENGTH_MISMATCH;
    if (n_points == 0) return empty_msm_result(out32, nullptr);
    bpp_points *p = nullptr;
    int rc = bpp_points_upload(ctx, fmt, pts, n_points, &p);
    if (rc) return rc;
    rc = bpp_msm_vartime(ctx, scalars, n_scalars, p, 0, n_points, out32, nullptr);
    bpp_points_free(ctx, p);
    return rc;
}

// ---- multi-GPU: NCCL inside the library (SURVEY 8b / D.3 "NCCL communicator created once") --------------------
// One process per GPU; rank 0 makes a 128-byte id (bpp_comm_unique_id), the host program hands it to every rank by
// whatever channel it has, every rank calls bpp_comm_init.  libnccl.so.2 is resolved at run time (dlopen), so a
// single-GPU host needs no NCCL installed; a process that already loaded NCCL (e.g. through PyTorch) shares that copy.
#include <dlfcn.h>
#include <nccl.h>
namespace {
struct nccl_api {
    void *h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
nccl_api &nccl() {
    static nccl_api a;
    static std::once_flag once;
    std::call_once(once, [] {
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *nm : names)
            if ((a.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL))) break;
        if (!a.h) return;
        a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(a.h, "ncclGetUniqueId");
        a.CommInitRank = (decltype(a.CommInitRank))dlsym(a.h, "ncclCommInitRank");
        a.AllGather = (decltype(a.AllGather))dlsym(a.h, "ncclAllGather");
        a.CommDestroy = (decltype(a.CommDestroy))dlsym(a.h, "ncclCommDestroy");
        a.GetErrorString = (decltype(a.GetErrorString))dlsym(a.h, "ncclGetErrorString");
        a.ok = a.GetUniqueId && a.CommInitRank && a.AllGather && a.CommDestroy && a.GetErrorString;
    });
    return a;
}
}  // namespace
#define NCCL_CK(ctx, call)                                                                  \
    do {                                                                                    \
        ncclResult_t r_ = (call);                                                           \
        if (r_ != ncclSuccess) {                                                            \
            (ctx)->last_error = std::string(#call) + ": " + nccl().GetErrorString(r_);      \
            return BPP_ERR_CUDA;                                                            \
        }                                                                                   \
    } while (0)

extern "C" int bpp_comm_unique_id(uint8_t id[BPP_COMM_ID_BYTES]) {
    if (!id) return BPP_ERR_INVALID_ARG;
    static_assert(sizeof(ncclUniqueId) == BPP_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
    if (!nccl().ok) return BPP_ERR_NO_DEVICE;
    ncclUniqueId u;
    if (nccl().GetUniqueId(&u) != ncclSuccess) return BPP_ERR_CUDA;
    memcpy(id, &u, sizeof(u));
    return BPP_OK;
}
extern "C" int bpp_comm_free(bpp_ctx *ctx) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    if (!ctx->comm) return BPP_OK;
    cudaSetDevice(ctx->device);
    msm_wait_pending(ctx);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->s_comm);
    nccl().CommDestroy((ncclComm_t)ctx->comm);
    ctx->comm = nullptr;
    cudaStreamDestroy(ctx->s_comm);
    cudaEventDestroy(ctx->ev_comm_ready);
    for (int i = 0; i < 3; i++) cudaEventDestroy(ctx->ev_comm_done[i]);
    cudaFree(ctx->d_comm);
    ctx->d_comm = nullptr;
    ctx->comm_nranks = 1;
    ctx->comm_rank = 0;
    return BPP_OK;
}
extern "C" int bpp_comm_init(bpp_ctx *ctx, int nranks, int rank, const uint8_t id[BPP_COMM_ID_BYTES]) {
    if (!ctx || !id || nranks < 1 || rank < 0 || rank >= nranks) return BPP_ERR_INVALID_ARG;
    if (ctx->comm) return BPP_ERR_INVALID_ARG;   // once per context
    if (!nccl().ok) {
        ctx->last_error = "libnccl.so.2 not found (dlopen)";
        return BPP_ERR_NO_DEVICE;
    }
    CK(ctx, cudaSetDevice(ctx->device));
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    ncclComm_t c = nullptr;
    NCCL_CK(ctx, nccl().CommInitRank(&c, nranks, u, rank));
    ctx->comm = c;
    ctx->comm_rank = rank;
    ctx->comm_nranks = nranks;
    CK(ctx, cudaStreamCreateWithFlags(&ctx->s_comm, cudaStreamNonBlocking));
    CK(ctx, cudaEventCreateWithFlags(&ctx->ev_comm_ready, cudaEventDisableTiming));
    for (int i = 0; i < 3; i++) CK(ctx, cudaEventCreateWithFlags(&ctx->ev_comm_done[i], cudaEventDisableTiming));
    CK(ctx, cudaMalloc((void **)&ctx->d_comm, 3 * (size_t)(1 + nranks) * 128));
    return BPP_OK;
}
extern "C" int bpp_comm_info(bpp_ctx *ctx, int *nranks, int *rank) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    if (nranks) *nranks = ctx->comm_nranks;
    if (rank) *rank = ctx->comm_rank;
    return BPP_OK;
}
int comm_all_gather(bpp_ctx *ctx, const void *d_send, void *d_recv, size_t bytes_per_rank, cudaStream_t stream) {
    if (!ctx->comm) {   // a single rank: the gather is a copy
        if (d_send != d_recv) CK(ctx, cudaMemcpyAsync(d_recv, d_send, bytes_per_rank, cudaMemcpyDeviceToDevice, stream));
        return BPP_OK;
    }
    NCCL_CK(ctx, nccl().AllGather(d_send, d_recv, bytes_per_rank, ncclUint8, (ncclComm_t)ctx->comm, stream));
    return BPP_OK;
}
extern "C" int bpp_comm_all_gather_dev(bpp_ctx *ctx, const void *d_send, size_t bytes_per_rank, void *d_recv) {
    if (!ctx || !d_send || !d_recv || bytes_per_rank == 0) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    return comm_all_gather(ctx, d_send, d_recv, bytes_per_rank, ctx->stream);
}
static inline uint8_t *comm_part(bpp_ctx *ctx, int slot) { return ctx->d_comm + (size_t)slot * (1 + ctx->comm_nranks) * 128; }
// Sharded MSM (SURVEY 8(e)): this rank holds a slice of the points and the matching scalars; every rank reduces its
// slice to one extended point (128 B), one all-gather of those partials, every rank adds them and compresses - the
// result (32 B encoding at d_out32) is identical on all ranks.  Joined form: in stream order on the caller's stream.
extern "C" int bpp_msm_sharded_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n,
                                   void *d_out32) {
    if (!ctx || !d_scalars || !points || !d_out32 || n == 0) return BPP_ERR_INVALID_ARG;
    if (off + n > points->n) return BPP_ERR_LENGTH_MISMATCH;
    CK(ctx, cudaSetDevice(ctx->device));
    if (!ctx->comm) return msm_enqueue(ctx, (const uint32_t *)d_scalars, points, off, n, (uint8_t *)d_out32, 1);
    int rc;
    uint8_t *part = comm_part(ctx, 0);
    if ((rc = msm_enqueue(ctx, (const uint32_t *)d_scalars, points, off, n, part, 0))) return rc;
    if ((rc = comm_all_gather(ctx, part, part + 128, 128, ctx->stream))) return rc;
    k_points_sum_compress<<<1, 32, 0, ctx->stream>>>((const uint32_t *)(part + 128), (uint32_t)ctx->comm_nranks, (uint8_t *)d_out32);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}
// Throughput form for a sequence of independent sharded MSMs: two MSMs in flight per rank (bpp_msm_submit_partial_dev),
// the 128-byte all-gather + sum + compress of MSM i - 1 on the communication stream beside MSM i; d_out32 of MSM i is
// final once the caller's stream has passed the submit of MSM i + 2, or after bpp_msm_sharded_wait.  Nothing but event
// waits goes onto the caller's stream between two submits.
static int comm_gather_slot(bpp_ctx *ctx, int slot) {
    uint8_t *part = comm_part(ctx, slot);
    CK(ctx, cudaEventRecord(ctx->ev_comm_ready, ctx->stream));
    CK(ctx, cudaStreamWaitEvent(ctx->s_comm, ctx->ev_comm_ready, 0));
    int rc = comm_all_gather(ctx, part, part + 128, 128, ctx->s_comm);
    if (rc) return rc;
    k_points_sum_compress<<<1, 32, 0, ctx->s_comm>>>((const uint32_t *)(part + 128), (uint32_t)ctx->comm_nranks, ctx->d_comm_out[slot]);
    LAUNCH_CHECK(ctx);
    CK(ctx, cudaEventRecord(ctx->ev_comm_done[slot], ctx->s_comm));
    return BPP_OK;
}
extern "C" int bpp_msm_sharded_submit_dev(bpp_ctx *ctx, const void *d_scalars, const bpp_points *points, size_t off, size_t n,
                                          void *d_out32) {
    if (!ctx || !d_scalars || !points || !d_out32 || n == 0) return BPP_ERR_INVALID_ARG;
    if (off + n > points->n) return BPP_ERR_LENGTH_MISMATCH;
    CK(ctx, cudaSetDevice(ctx->device));
    if (!ctx->comm) return msm_enqueue(ctx, (const uint32_t *)d_scalars, points, off, n, (uint8_t *)d_out32, 1, false);
    int rc;
    const uint64_t i = ctx->comm_seq++;
    const int slot = (int)(i % 3);
    ctx->d_comm_out[slot] = (uint8_t *)d_out32;
    if ((rc = msm_enqueue(ctx, (const uint32_t *)d_scalars, points, off, n, comm_part(ctx, slot), 0, false))) return rc;
    if ((rc = msm_wait_pending(ctx, true))) return rc;                       // MSM i - 1 is complete on the caller's stream
    if (i >= 1 && (rc = comm_gather_slot(ctx, (int)((i - 1) % 3)))) return rc;
    if (i >= 2) CK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_comm_done[(i - 2) % 3], 0));
    return BPP_OK;
}
extern "C" int bpp_msm_sharded_wait(bpp_ctx *ctx) {
    if (!ctx) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc;
    if ((rc = msm_wait_pending(ctx))) return rc;
    if (!ctx->comm || ctx->comm_seq == 0) return BPP_OK;
    const uint64_t k = ctx->comm_seq;
    if ((rc = comm_gather_slot(ctx, (int)((k - 1) % 3)))) return rc;
    if (k >= 2) CK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_comm_done[(k - 2) % 3], 0));
    CK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_comm_done[(k - 1) % 3], 0));
    ctx->comm_seq = 0;
    return BPP_OK;
}

// ---- measurement / tests -------------------------------------------------------------------------
extern "C" int bpp_bench_imad_peak(bpp_ctx *ctx, int iters, double *ops_per_sec, double *ms_out) {
    if (!ctx || iters <= 0) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    unsigned long long *d = (unsigned long long *)ctx->d_flag;
    int blocks = ctx->sm_count * 8;
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    k_imad_peak<<<blocks, 256, 0, ctx->stream>>>(1u, iters / 8 + 1, d);  // warm-up
    LAUNCH_CHECK(ctx);
    cudaEventRecord(a, ctx->stream);
    k_imad_peak<<<blocks, 256, 0, ctx->stream>>>(7u, iters, d);
    LAUNCH_CHECK(ctx);
    cudaEventRecord(b, ctx->stream);
    CK(ctx, cudaEventSynchronize(b));
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    double ops = (double)blocks * 256.0 * (double)iters * 16.0 * 8.0;
    if (ops_per_sec) *ops_per_sec = ops / (ms * 1e-3);
    if (ms_out) *ms_out = ms;
    return BPP_OK;
}

// mode 0: plain IMAD.WIDE.U32 (64-bit accumulate); 1: carry-chained IMAD.WIDE.U32; 2: 32-bit IMAD; 3: IADD3.X chains;
// 4: fe_mul chains (counted as 72 IMAD.WIDE each); 5: ge_madd chains (504 each)
extern "C" int bpp_bench_pipe_probe(bpp_ctx *ctx, int mode, int iters, double *ops_per_sec) {
    if (!ctx || iters <= 0 || mode < 0 || mode > 5 || !ops_per_sec) return BPP_ERR_INVALID_ARG;
    if (mode == 0) return bpp_bench_imad_peak(ctx, iters, ops_per_sec, nullptr);
    CK(ctx, cudaSetDevice(ctx->device));
    unsigned long long *d = (unsigned long long *)ctx->d_flag;
    int blocks = ctx->sm_count * 8;
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    k_pipe_probe<<<blocks, 256, 0, ctx->stream>>>(mode, 1u, iters / 8 + 1, d);
    LAUNCH_CHECK(ctx);
    cudaEventRecord(a, ctx->stream);
    k_pipe_probe<<<blocks, 256, 0, ctx->stream>>>(mode, 7u, iters, d);
    LAUNCH_CHECK(ctx);
    cudaEventRecord(b, ctx->stream);
    CK(ctx, cudaEventSynchronize(b));
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    double per_iter = mode == 1 ? 64.0 : mode == 4 ? 144.0 : mode == 5 ? 504.0 : 128.0;
    *ops_per_sec = (double)blocks * 256.0 * (double)iters * per_iter / (ms * 1e-3);
    return BPP_OK;
}

extern "C" int bpp_test_op(bpp_ctx *ctx, int op, const uint8_t *a, const uint8_t *b, uint8_t *out, size_t n) {
    if (!ctx || !a || !b || !out || n == 0 || n >= (1ull << 31)) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    uint8_t *d = nullptr;
    CK(ctx, cudaMalloc((void **)&d, n * 96));
    cudaError_t e = cudaMemcpyAsync(d, a, n * 32, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + n * 32, b, n * 32, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        k_test_op<<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>(op, d, d + n * 32, d + n * 64, (uint32_t)n);
        ctx->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d + n * 64, n * 32, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess) {
        ctx->last_error = cudaGetErrorString(e);
        return BPP_ERR_CUDA;
    }
    return BPP_OK;
}

