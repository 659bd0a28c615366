// bpperm_internal.hpp - what the translation units of libbpperm_cuda.so share: the context, the error macros and the
// scratch allocator.  Not part of the C ABI (include/bpperm.h is).
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/bpperm.h"

#define BPP_MAX_GROUPS 8
#define BPP_SORT_BLOCKS_PER_SM 2u
#define BPP_TILE64_MIN_POINTS (3u << 20)
#define BPP_PIPELINE_MIN_POINTS (1u << 18)
#define BPP_PIPELINE_MIN_POINTS_SUBMIT (1u << 12)
#define BPP_TABLE_MSM_MAX_POINTS (1u << 13)   // single MSMs over precomputed points go through the table up to here

struct bpp_points {
    uint32_t *niels = nullptr;  // n x 24 u32 (96 B)
    size_t n = 0;
    // bpp_points_precompute: fixed-base window table over all n points (entry layout of acproof_kernels.cuh k_fb_build)
    uint32_t *fb_table = nullptr;
    int fb_c = 0, fb_Wn = 0;
    uint32_t fb_K[8] = {};
};

struct bpp_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0, cc_major = 0, cc_minor = 0;
    size_t total_mem = 0;
    std::string last_error;
    uint64_t launches = 0;
    int forced_c = 0;
    bool profiling = false, events_pending = false;
    cudaEvent_t ev[BPP_PHASE_COUNT + 1] = {};
    float phase_ms[BPP_PHASE_COUNT] = {};
    uint64_t n_madd = 0, n_add = 0, n_dbl = 0;
    // scratch (grown on demand)
    uint32_t *d_scalars = nullptr; size_t cap_scalars = 0;       // n x 8
    // MSM scratch: two slots, so that a submitted MSM (bpp_msm_submit_dev) can still be in its tail while the
    // next one sorts and accumulates
    struct msm_scratch {
        uint32_t *d_counts = nullptr, *d_offsets = nullptr, *d_cursor = nullptr;  // W x B each
        size_t cap_wb = 0, cap_offsets = 0, cap_cursor = 0;
        uint32_t *d_entries = nullptr; size_t cap_entries = 0;      // W x n
        uint32_t *d_partials = nullptr; size_t cap_partials = 0;    // 2 x tiles x 32
        uint32_t *d_long = nullptr; size_t cap_long = 0;            // hot-bucket queues (one region per window group)
        uint32_t *d_nlong = nullptr;                                // their counters
        uint32_t *d_buckets = nullptr; size_t cap_buckets = 0;      // W x B x 32
        uint32_t *d_segS = nullptr, *d_segR = nullptr; size_t cap_seg = 0;
        uint8_t *d_gparts = nullptr;                                // BPP_MAX_GROUPS x 128 B: window-group partials
        cudaEvent_t ev_done = nullptr;                              // recorded when the slot's MSM has written its result
        bool pending = false;                                       // the caller's stream has not waited for ev_done yet
    } scr[2];
    int slot = 0;
    uint8_t *d_out = nullptr;                                   // 160 B
    uint8_t *h_out = nullptr;                                   // pinned 160 B
    uint8_t *d_stage = nullptr; size_t cap_stage = 0;           // upload staging
    uint32_t *d_flag = nullptr;
    uint8_t *h_pinned = nullptr; size_t cap_pinned = 0;         // pinned staging for host scalars
    uint8_t *d_vec = nullptr; size_t cap_vec = 0;               // arena of the scalar-vector operators
    uint8_t *d_small = nullptr; size_t cap_small = 0;           // arena of bpp_msm_vartime_batch
    uint8_t *d_multi = nullptr; size_t cap_multi = 0;           // arena of bpp_msm_multi*
    std::vector<uint8_t> mm_host;                               // host plan of the last bpp_msm_multi* call
    // pipelined MSM: window groups on side streams (msm_pipeline_init)
    bool pipe_ready = false;
    int forced_groups = 0;
    int forced_tile = 0;                                        // tile length override (bpp_set_msm_tile), 0 = by input size
    int forced_part[BPP_MAX_GROUPS] = {}, n_forced_part = 0;    // explicit group sizes, top window group first
    cudaStream_t s_sort = nullptr, s_bulk[2] = {}, s_tail[BPP_MAX_GROUPS] = {};
    cudaEvent_t ev_fork = nullptr, ev_sorted[BPP_MAX_GROUPS] = {}, ev_acc[BPP_MAX_GROUPS] = {}, ev_tail[BPP_MAX_GROUPS] = {};
    cudaStream_t s_final = nullptr;
    // multi-GPU (bpp_comm_init): one NCCL communicator per context, created once; collectives run on s_comm or on the
    // caller's stream.  Payloads are tiny (128 B partial points, accept bytes): latency, not bandwidth.
    void *comm = nullptr;                                       // ncclComm_t
    int comm_rank = 0, comm_nranks = 1;
    cudaStream_t s_comm = nullptr;
    uint8_t *d_comm = nullptr;                                  // 3 slots x (128 B partial + nranks x 128 B gathered)
    uint8_t *d_comm_out[3] = {};                                // where each slot's result goes (caller's buffers)
    cudaEvent_t ev_comm_ready = nullptr, ev_comm_done[3] = {};
    uint64_t comm_seq = 0;                                      // sharded MSMs submitted so far
    // stage timeline of the last MSM (bpp_set_msm_trace): timing events on whichever stream ran the stage
    bool trace = false;
    std::vector<std::pair<std::string, cudaEvent_t>> trace_ev;
};

static inline void trace_mark(bpp_ctx *ctx, cudaStream_t s, const char *what, int g) {
    if (!ctx->trace) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, s);
    ctx->trace_ev.emplace_back(std::string(what) + "[" + std::to_string(g) + "]", e);
}

#define CK(ctx, call)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            (ctx)->last_error = std::string(#call) + ": " + cudaGetErrorString(e_);                \
            return e_ == cudaErrorMemoryAllocation ? BPP_ERR_OOM : BPP_ERR_CUDA;                   \
        }                                                                                          \
    } while (0)

#define LAUNCH_CHECK(ctx)                                                                          \
    do {                                                                                           \
        (ctx)->launches++;                                                                         \
        cudaError_t e_ = cudaGetLastError();                                                       \
        if (e_ != cudaSuccess) {                                                                   \
            (ctx)->last_error = std::string("kernel launch: ") + cudaGetErrorString(e_);           \
            return BPP_ERR_CUDA;                                                                   \
        }                                                                                          \
    } while (0)

template <typename T>
static int grow(bpp_ctx *ctx, T **p, size_t *cap, size_t need_elems) {
    if (need_elems <= *cap) return BPP_OK;
    if (*p) CK(ctx, cudaFree(*p));
    *p = nullptr;
    *cap = 0;
    size_t want = need_elems + need_elems / 8;
    CK(ctx, cudaMalloc((void **)p, want * sizeof(T)));
    *cap = want;
    return BPP_OK;
}

// defined in capi_core.cu
int comm_all_gather(bpp_ctx *ctx, const void *d_send, void *d_recv, size_t bytes_per_rank, cudaStream_t stream);
int msm_wait_pending(bpp_ctx *ctx, bool keep_latest = false);
// groups: number of window groups, split evenly (0 = the library's partition for n, which minimises the latency of one
// call; bpp_set_msm_groups / bpp_set_msm_partition override it)
int msm_enqueue(bpp_ctx *ctx, const uint32_t *d_scalars, const bpp_points *pts, size_t off, size_t n, uint8_t *d_out,
                int do_compress, bool join = true, int groups = 0);
// defined in capi_acproof.cu: bpp_msm_vartime_batch's table-gather MSM (`count` MSMs over pts[off, off + n), count x n
// scalars at d_sc) up to the extended sums, count x 128 B at d_ext.  d_part: msm_table_part_bytes of split partials.
// madd / add: its operation counts.  The window table must exist.  Stream-ordered on ctx->stream.
size_t msm_table_part_bytes(const bpp_ctx *ctx, const bpp_points *P, size_t n, size_t count);
int msm_table_ext(bpp_ctx *ctx, const uint32_t *d_sc, const bpp_points *P, size_t off, size_t n, size_t count, uint32_t *d_ext,
                  uint32_t *d_part, uint64_t *madd, uint64_t *add);
// defined in capi_msm_multi.cu: dst = n scalars of src with bit 255 cleared (the _dev table MSMs: device data cannot drive
// a table digit past the window's 2^(c-1) entries).  Stream-ordered on ctx->stream.
int msm_scalars_low255(bpp_ctx *ctx, const void *src, uint64_t n, void *dst);

