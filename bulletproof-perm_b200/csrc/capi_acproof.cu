// capi_acproof.cu - host driver + C ABI of the batched shuffle prover / verifier.
// The driver re-expresses the seven-step state machine of
// /root/reference/bp-perm/src/circuit_lib.rs (call order lib.rs:219-231) for B proofs in lock-step:
// one kernel launch per protocol step for the whole batch, Fiat-Shamir transcripts on host threads.
#include <functional>
#include <thread>

#include "bpperm_internal.hpp"

#include "acproof_kernels.cuh"
#include "ipa_kernels.cuh"
#include "transcript_kernels.cuh"
#include "host_merlin.hpp"


struct bpp_circuit {
    uint32_t n = 0, Q = 0, m = 0, rows = 0, nnz = 0;
    uint32_t *d_rowptr = nullptr, *d_col = nullptr, *d_coeff = nullptr;
    uint8_t *d_kind = nullptr;
    uint32_t n_long = 0, *d_long = nullptr;   // rows of more than ACP_CSR_LONG entries (k_acp_csr_long)
};

struct bpp_gens {
    uint32_t n = 0, n_gens = 0;  // gens order: g, h, G[0..n), H[0..n)
    bpp_points *pts = nullptr;   // the n_gens points and their window table (bpp_points_precompute)
    // sums of generator ranges with their own window table (acp_gens_sum: H_sum of the shuffle prover's A_I), built once
    // per (range, window width) for all batches over these generators and freed with them
    struct range_sum { uint32_t first, cnt; bpp_points *pts; };
    std::vector<range_sum> sums;
    std::mutex mu;
};

struct bpp_acp_batch {
    bpp_ctx *ctx = nullptr;
    const bpp_circuit *cir = nullptr;
    const bpp_gens *gens = nullptr;
    int mode = 1;
    uint32_t B = 0, proof_len = 0;
    acp_layout lay;
    std::vector<uint8_t> label;
    uint32_t *d_blk = nullptr, *d_seeds = nullptr, *d_wide = nullptr, *d_ext8 = nullptr, *d_dyn = nullptr,
             *d_wsum = nullptr, *d_stat = nullptr, *d_bad = nullptr, *d_vext = nullptr, *d_vseed = nullptr;
    uint8_t *d_pts8 = nullptr, *d_proofs = nullptr, *d_V = nullptr, *d_accept = nullptr;
    uint8_t *h_pts8 = nullptr, *h_wide = nullptr, *h_proofs = nullptr;  // pinned
    // `fixed` mode: L_j/R_j encodings (B x 2 lg x 32), the three transcript scalars (B x 3 x 32), fb split scratch
    uint8_t *d_lr = nullptr, *h_lr = nullptr, *h_tx3 = nullptr;
    uint32_t *d_tx3 = nullptr, *d_lrext = nullptr, *d_part = nullptr;
    uint32_t fb_splits = 1;
    // Fiat-Shamir: per-proof Merlin states on the device (default; no host round trip between kernels) or on
    // host threads (host_transcripts: the same bytes, kept as the cross-check and for hosts that want the
    // transcript in their own process)
    bool host_transcripts = false;
    uint64_t *d_tr = nullptr, *d_proto = nullptr;   // d_proto: 2 states - the proof transcripts' common prefix, Transcript::new("acp-V")
    uint8_t *d_vdig = nullptr;                      // chunk digests of the commitments (k_tr_vchunks), B x chunks x 32
    uint32_t *d_wstage = nullptr;   // witness staging (contiguous upload), allocated on first use
    // verifier fork: point decompression (IMAD-bound, fills the GPU) runs on `aux` beside the challenge-dependent
    // scalar chain (Fiat-Shamir replay, Fibonacci power chains, CSR products: serial, low occupancy)
    cudaStream_t aux = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // second side stream: the prover's absorption of the commitments (beside the commitment MSMs) and the verifier's
    // weight derivation (k_tr_weights: hashes the rest of the proof; beside the challenge-dependent scalar chain)
    cudaStream_t aux2 = nullptr;
    cudaEvent_t ev_fork2 = nullptr, ev_join2 = nullptr;
    cudaStream_t aux3 = nullptr;      // small batches: the third commitment of A_I / A_O / S side by side
    cudaEvent_t ev_join3 = nullptr;
    uint32_t *d_vwit = nullptr, *d_wgen = nullptr;   // bpp_acp_batch_gen_shuffle_witness: v (B x m), staging of its inputs
    bool have_vwit = false;
    // the resident witness came from bpp_acp_batch_gen_shuffle_witness (v', -x are in the block): A_I may take the
    // structured shape (acp_ai_shape) over H_sum = H_0 + .. + H_{n-3}, whose table hsum is (owned by the generators)
    bool shuffle_wit = false;
    const bpp_points *hsum = nullptr;
    bool have_V = false;            // commitments resident (bpp_acp_batch_commit / _upload_commitments / _upload_proofs)
    uint8_t *h_V = nullptr;         // host transcripts only: pinned copy of the commitments
    // priority split (bpp_acp_batch_set_priority_split): the table-gather MSMs (k_fb_msm) run on `bulk`, a stream of
    // the lowest priority, so that on an urgent caller's stream the short dependent kernels of this batch win the SM
    // slots against the GPU-filling kernels of a second batch in flight on another stream
    bool priority_split = false;
    cudaStream_t bulk = nullptr;
    cudaEvent_t ev_bfork = nullptr, ev_bjoin = nullptr;
    // batch verification by random linear combination (k_rlc_*): scalars of the one MSM over the batch's
    // dynamic points + the shared generators (appended to d_dyn), its compressed result, the fall-back flag
    bool batch_rlc = true;
    bool decompress_late = false;   // verifier: fork the point decompression after the transcript replay (BPP_DECOMPRESS_LATE=1)
    uint32_t *d_rlc_sc = nullptr, *d_rlc_flag = nullptr;
    uint8_t *d_rlc_out = nullptr;
    uint32_t *h_rlc_flag = nullptr;
    std::vector<bpp_host::Transcript> tr;
    // BPP_ACP_TRACE=1: stage timeline of prove / verify (timing events on the caller's stream, printed to stderr)
    bool trace = false;
    std::vector<std::pair<const char *, cudaEvent_t>> marks;
};

static uint32_t acp_next_pow2(uint32_t n) { uint32_t p = 1; while (p < n) p <<= 1; return p; }
static uint32_t acp_log2(uint32_t p) { uint32_t l = 0; while ((1u << l) < p) l++; return l; }

static void acp_mark(bpp_acp_batch *b, const char *name) {
    if (!b->trace) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, b->ctx->stream);
    b->marks.emplace_back(name, e);
}
static void acp_marks_dump(bpp_acp_batch *b, const char *what) {
    if (!b->trace || b->marks.empty()) return;
    cudaStreamSynchronize(b->ctx->stream);
    fprintf(stderr, "[acp trace] %s:", what);
    for (size_t i = 1; i < b->marks.size(); i++) {
        float ms = 0;
        cudaEventElapsedTime(&ms, b->marks[i - 1].second, b->marks[i].second);
        fprintf(stderr, " %s %.0f us |", b->marks[i].first, ms * 1e3f);
    }
    float tot = 0;
    cudaEventElapsedTime(&tot, b->marks.front().second, b->marks.back().second);
    fprintf(stderr, " total %.0f us\n", tot * 1e3f);
    for (auto &m : b->marks) cudaEventDestroy(m.second);
    b->marks.clear();
}
// the shape of bpp_circuit_create_shuffle's circuit, which bpp_acp_batch_gen_shuffle_witness needs: n = 2k, m = 2k + 1, k >= 2
static bool acp_shuffle_shaped(uint32_t n, uint32_t m) { return n >= 4 && !(n & 1u) && m == n + 1; }
static acp_layout acp_make_layout(uint32_t n_, uint32_t Q, uint32_t m, int mode) {
    acp_layout L;
    uint32_t o = 0;
    auto take = [&](uint32_t cnt) { uint32_t r = o; o += cnt; return r; };
    L.n = n_; L.Q = Q; L.m = m;
    L.np = mode == 2 ? acp_next_pow2(n_) : n_;
    L.lg = mode == 2 ? acp_log2(L.np) : 0;
    const uint32_t n = L.n, np = L.np;   // only y^n, y^-n, l, r and the verifier's G/H scalars have the padded length
    L.aL = take(n); L.aR = take(n); L.aO = take(n); L.gamma = take(m);
    L.alpha = take(1); L.beta = take(1); L.ro = take(1); L.sl = take(n); L.sr = take(n); L.tau = take(5);
    L.y = take(1); L.z = take(1); L.x = take(1); L.w = take(1); L.rho0 = take(1);   // contiguous: host transcripts place them in one go
    L.yn = take(np); L.yninv = take(np); L.zq = take(Q);
    L.zWL = take(n); L.zWR = take(n); L.zWO = take(n); L.zWV = take(m); L.zc = take(1);
    L.lin = take(n); L.l1 = take(n); L.r0 = take(n); L.r1 = take(n); L.r3 = take(n);
    L.dots = take(12); L.sigma = L.dots + 9;
    L.tc = take(6); L.tsel = take(5);
    L.l = take(np); L.r = take(np); L.that = take(1); L.taux = take(1); L.mu = take(1);
    L.vg = take(1); L.vh = take(1); L.vG = take(np); L.vH = take(np); L.vd = take(m + 8 + 2 * L.lg);
    L.wq = take(1); L.u = take(L.lg); L.uinv = take(L.lg); L.cl = take(2); L.pa = take(1); L.pb = take(1);
    L.ptab = take(mode == 2 ? 3 * IPA_MAX_LG : 0);
    L.stab = take(mode == 2 ? 2 * np : 0);
    L.rho = take(1);
    const bool shuffle = acp_shuffle_shaped(n, m);
    L.vr = take(shuffle ? n - 2 : 0); L.nx = take(shuffle ? 1 : 0);
    L.stride = (o + 3) & ~3u;
    return L;
}

// ---- circuit --------------------------------------------------------------------------------------
// Weights arrive as (wire, constraint, coefficient) triples of the four matrices concatenated in the
// order W_L, W_R, W_O, W_V - the sparse form of the reference's dense n x Q / m x Q matrices
// (ACEssentials, circuit_lib.rs:58-74; shapes SURVEY A.1) - plus the dense constant vector c (Q).
extern "C" int bpp_circuit_create(bpp_ctx *ctx, size_t n, size_t Q, size_t m, const uint32_t nnz[4], const uint32_t *wire,
                                  const uint32_t *constraint, const uint8_t *coeff, const uint8_t *c_vec,
                                  bpp_circuit **out) {
    if (!ctx || !out || !nnz || n == 0 || Q == 0 || m == 0 || !c_vec) return BPP_ERR_INVALID_ARG;
    *out = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    const uint32_t rows = (uint32_t)(3 * n + m + 1);
    const uint32_t row_base[4] = {0, (uint32_t)n, (uint32_t)(2 * n), (uint32_t)(3 * n)};
    const uint32_t row_cnt[4] = {(uint32_t)n, (uint32_t)n, (uint32_t)n, (uint32_t)m};
    size_t total = 0;
    for (int k = 0; k < 4; k++) total += nnz[k];
    if (total && (!wire || !constraint || !coeff)) return BPP_ERR_INVALID_ARG;
    static const uint8_t ONE[32] = {1};
    static const uint8_t MINUS_ONE[32] = {0xec, 0xd3, 0xf5, 0x5c, 0x1a, 0x63, 0x12, 0x58, 0xd6, 0x9c, 0xf7, 0xa2, 0xde, 0xf9, 0xde, 0x14,
                                          0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0x10};
    std::vector<uint32_t> rowptr(rows + 1, 0);
    size_t e = 0;
    for (int k = 0; k < 4; k++)
        for (uint32_t i = 0; i < nnz[k]; i++, e++) {
            if (wire[e] >= row_cnt[k] || constraint[e] >= Q) return BPP_ERR_INVALID_ARG;
            rowptr[row_base[k] + wire[e] + 1]++;
        }
    size_t c_nnz = 0;
    for (size_t q = 0; q < Q; q++) {
        bool nz = false;
        for (int b = 0; b < 32; b++) nz |= c_vec[32 * q + b] != 0;
        if (nz) c_nnz++;
    }
    rowptr[rows] = (uint32_t)c_nnz;
    for (uint32_t r = 0; r < rows; r++) rowptr[r + 1] += rowptr[r];
    const size_t all = total + c_nnz;
    std::vector<uint32_t> col(all ? all : 1), cf((all ? all : 1) * 8, 0), fill(rowptr.begin(), rowptr.end() - 1);
    std::vector<uint8_t> kind(all ? all : 1);
    auto put = [&](uint32_t row, uint32_t q, const uint8_t *v) {
        uint32_t pos = fill[row]++;
        col[pos] = q;
        kind[pos] = memcmp(v, ONE, 32) == 0 ? 1 : memcmp(v, MINUS_ONE, 32) == 0 ? 2 : 0;
        memcpy(&cf[8 * (size_t)pos], v, 32);
    };
    e = 0;
    for (int k = 0; k < 4; k++)
        for (uint32_t i = 0; i < nnz[k]; i++, e++) put(row_base[k] + wire[e], constraint[e], coeff + 32 * e);
    for (size_t q = 0; q < Q; q++) {
        bool nz = false;
        for (int b = 0; b < 32; b++) nz |= c_vec[32 * q + b] != 0;
        if (nz) put(rows - 1, (uint32_t)q, c_vec + 32 * q);
    }
    bpp_circuit *c = new bpp_circuit();
    c->n = (uint32_t)n; c->Q = (uint32_t)Q; c->m = (uint32_t)m; c->rows = rows; c->nnz = (uint32_t)all;
    cudaError_t err = cudaMalloc((void **)&c->d_rowptr, (rows + 1) * 4);
    if (err == cudaSuccess) err = cudaMalloc((void **)&c->d_col, col.size() * 4);
    if (err == cudaSuccess) err = cudaMalloc((void **)&c->d_coeff, cf.size() * 4);
    if (err == cudaSuccess) err = cudaMalloc((void **)&c->d_kind, kind.size());
    if (err == cudaSuccess) err = cudaMemcpy(c->d_rowptr, rowptr.data(), (rows + 1) * 4, cudaMemcpyHostToDevice);
    if (err == cudaSuccess) err = cudaMemcpy(c->d_col, col.data(), col.size() * 4, cudaMemcpyHostToDevice);
    if (err == cudaSuccess) err = cudaMemcpy(c->d_coeff, cf.data(), cf.size() * 4, cudaMemcpyHostToDevice);
    if (err == cudaSuccess) err = cudaMemcpy(c->d_kind, kind.data(), kind.size(), cudaMemcpyHostToDevice);
    std::vector<uint32_t> long_rows;
    for (uint32_t r = 0; r < rows; r++)
        if (rowptr[r + 1] - rowptr[r] > ACP_CSR_LONG) long_rows.push_back(r);
    c->n_long = (uint32_t)long_rows.size();
    if (err == cudaSuccess && c->n_long) err = cudaMalloc((void **)&c->d_long, long_rows.size() * 4);
    if (err == cudaSuccess && c->n_long) err = cudaMemcpy(c->d_long, long_rows.data(), long_rows.size() * 4, cudaMemcpyHostToDevice);
    if (err != cudaSuccess) {
        ctx->last_error = cudaGetErrorString(err);
        delete c;
        return BPP_ERR_CUDA;
    }
    *out = c;
    return BPP_OK;
}
// The corrected k-card shuffle circuit (SURVEY 8 row f-1; CPU restatement: shuffle_circuit in the test tree; the shape of weights.rs:130-204
// create_weights, which as coded only makes sense for 2-3 cards): prod_i (v_i - X) == prod_i (v_{k+i} - X), X = v[2k] -
// two product chains of k - 1 multipliers, one equality, two padding multipliers.  n = 2k, Q = 4k, m = 2k + 1, c = 0.
extern "C" int bpp_circuit_create_shuffle(bpp_ctx *ctx, size_t k_, bpp_circuit **out) {
    if (!ctx || !out || k_ < 2 || k_ > (1u << 24)) return BPP_ERR_INVALID_ARG;
    const uint32_t k = (uint32_t)k_;
    struct trip { uint32_t wire, q; bool minus; };
    std::vector<trip> W[4];   // W_L, W_R, W_O, W_V
    uint32_t q = 0;
    for (uint32_t c = 0; c < 2; c++) {
        const uint32_t gb = c * (k - 1), vb = c * k;
        W[0].push_back({gb, q, false}); W[3].push_back({vb, q, false}); W[3].push_back({2 * k, q, true}); q++;
        for (uint32_t i = 0; i + 1 < k; i++) {
            W[1].push_back({gb + i, q, false}); W[3].push_back({vb + i + 1, q, false}); W[3].push_back({2 * k, q, true}); q++;
        }
        for (uint32_t i = 1; i + 1 < k; i++) {
            W[0].push_back({gb + i, q, false}); W[2].push_back({gb + i - 1, q, true}); q++;
        }
    }
    W[2].push_back({k - 2, q, false}); W[2].push_back({2 * k - 3, q, true}); q++;
    W[0].push_back({2 * k - 2, q, false}); q++;
    W[0].push_back({2 * k - 1, q, false}); q++;
    static const uint8_t ONE[32] = {1};
    static const uint8_t MINUS_ONE[32] = {0xec, 0xd3, 0xf5, 0x5c, 0x1a, 0x63, 0x12, 0x58, 0xd6, 0x9c, 0xf7, 0xa2, 0xde, 0xf9, 0xde, 0x14,
                                          0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0x10};
    uint32_t nnz[4];
    std::vector<uint32_t> wire, cons;
    std::vector<uint8_t> coeff;
    for (int m = 0; m < 4; m++) {
        nnz[m] = (uint32_t)W[m].size();
        for (const trip &t : W[m]) {
            wire.push_back(t.wire);
            cons.push_back(t.q);
            coeff.insert(coeff.end(), t.minus ? MINUS_ONE : ONE, (t.minus ? MINUS_ONE : ONE) + 32);
        }
    }
    std::vector<uint8_t> cvec((size_t)4 * k * 32, 0);
    return bpp_circuit_create(ctx, 2 * (size_t)k, 4 * (size_t)k, 2 * (size_t)k + 1, nnz, wire.data(), cons.data(), coeff.data(),
                              cvec.data(), out);
}
extern "C" void bpp_circuit_free(bpp_ctx *ctx, bpp_circuit *c) {
    if (!c) return;
    if (ctx) { cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream); }
    cudaFree(c->d_rowptr); cudaFree(c->d_col); cudaFree(c->d_coeff); cudaFree(c->d_kind); cudaFree(c->d_long);
    delete c;
}

// ---- generators + fixed-base tables ---------------------------------------------------------------
// g_base, h_base, G_vec, H_vec of ACEssentials (circuit_lib.rs:58-65) as compressed points.
extern "C" int bpp_gens_create(bpp_ctx *ctx, const uint8_t g[32], const uint8_t h[32], const uint8_t *G, const uint8_t *H,
                               size_t n, int window_bits, bpp_gens **out) {
    if (!ctx || !out || !g || !h || !G || !H || n == 0) return BPP_ERR_INVALID_ARG;
    if (window_bits == 0) window_bits = 8;
    if (window_bits < 4 || window_bits > 20) return BPP_ERR_INVALID_ARG;   // 2^(c-1) entries x 96 B per (generator, window)
    *out = nullptr;
    std::vector<uint8_t> all(32 * (2 * n + 2));
    memcpy(&all[0], g, 32);
    memcpy(&all[32], h, 32);
    memcpy(&all[64], G, 32 * n);
    memcpy(&all[64 + 32 * n], H, 32 * n);
    bpp_points *pts = nullptr;
    int rc = bpp_points_upload(ctx, BPP_FMT_COMPRESSED, all.data(), 2 * n + 2, &pts);
    if (rc) return rc;
    if ((rc = bpp_points_precompute(ctx, pts, window_bits))) {
        bpp_points_free(ctx, pts);
        return rc;
    }
    bpp_gens *gs = new bpp_gens();
    gs->n = (uint32_t)n;
    gs->n_gens = (uint32_t)(2 * n + 2);
    gs->pts = pts;
    *out = gs;
    return BPP_OK;
}
extern "C" void bpp_gens_free(bpp_ctx *ctx, bpp_gens *g) {
    if (!g) return;
    for (auto &e : g->sums) bpp_points_free(ctx, e.pts);
    bpp_points_free(ctx, g->pts);
    delete g;
}

__global__ void k_compress_strided(const uint32_t *__restrict__ ext, uint32_t pitch, uint32_t first, uint32_t cnt, uint32_t B,
                                   uint8_t *__restrict__ out32);
// ---- small and batched variable-base MSMs over a long-lived point set (SURVEY 2.3 K5, 8b) ---------------------
// The reference's 15 vartime_multiscalar_mul call sites (circuit_lib.rs:187-575) have 2..209 points, always drawn from
// the same generator set, with fresh scalars per proof.  For such a set the window table of bpp_points_precompute turns
// every MSM into table look-ups and mixed adds - no buckets, no doublings, so no 253-step dependent chain - and
// bpp_msm_vartime_batch evaluates `count` of them per launch.
extern "C" int bpp_points_precompute(bpp_ctx *ctx, bpp_points *p, int window_bits) {
    if (!ctx || !p || p->n == 0) return BPP_ERR_INVALID_ARG;
    if (window_bits == 0) window_bits = 8;
    if (window_bits < 4 || window_bits > 20) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    if (p->fb_table && p->fb_c == window_bits) return BPP_OK;
    if (p->fb_table) {
        CK(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(p->fb_table);
        p->fb_table = nullptr;
    }
    const int Wn = (256 + window_bits - 1) / window_bits;
    const size_t half = (size_t)1 << (window_bits - 1), entries = p->n * Wn * half;
    if (p->n * (size_t)Wn >= (1ull << 31)) return BPP_ERR_INVALID_ARG;
    if (cudaMalloc((void **)&p->fb_table, entries * FB_ENTRY_U32 * 4) != cudaSuccess) {
        cudaGetLastError();
        p->fb_table = nullptr;
        return BPP_ERR_OOM;
    }
    const uint32_t threads = (uint32_t)(p->n * Wn);
    k_fb_build<<<(threads + 63) / 64, 64, 0, ctx->stream>>>(p->niels, (uint32_t)p->n, window_bits, Wn, p->fb_table);
    LAUNCH_CHECK(ctx);
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    p->fb_c = window_bits;
    p->fb_Wn = Wn;
    memset(p->fb_K, 0, sizeof(p->fb_K));   // K = sum_{w < Wn-1} 2^(c w + c - 1)
    for (int w = 0; w < Wn - 1; w++) {
        const int bit = window_bits * w + window_bits - 1;
        p->fb_K[bit >> 5] |= 1u << (bit & 31);
    }
    return BPP_OK;
}
// The table-gather MSM's forms: a thread per output (k_fb_msm_small; few terms, many outputs), a warp per output
// (fb_warp_launch; from 16 outputs per SM: no block tree, no barrier - as fast as a block on the A_I shape, 5 % faster
// on the `fixed` mode's prover), else a block per output (k_fb_msm), split over `splits` blocks when the outputs alone
// do not fill the GPU (k_fb_sum_splits adds the partial sums).
enum fb_form { FB_SMALL, FB_WARP, FB_BLOCK };
struct fb_plan {
    fb_form form;
    uint32_t splits;
};
// blocks per output of the block form: 4 blocks per SM in all, at least one work item per thread, at most 256
static uint32_t fb_split_count(const bpp_ctx *ctx, uint64_t outputs, uint64_t items) {
    const uint64_t want = 4ull * ctx->sm_count, cap = (items + FB_THREADS - 1) / FB_THREADS;
    uint64_t sp = outputs >= want ? 1 : (want + outputs - 1) / outputs;
    if (sp > cap) sp = cap;
    if (sp > 256) sp = 256;
    return (uint32_t)(sp ? sp : 1);
}
static fb_plan fb_choose(const bpp_ctx *ctx, uint64_t outputs, uint32_t terms, int Wn, bool small_ok, uint32_t max_splits) {
    if (small_ok && (uint64_t)terms * Wn <= 64 && outputs >= 32ull * ctx->sm_count) return {FB_SMALL, 1};
    if (outputs >= 16ull * ctx->sm_count) return {FB_WARP, 1};
    const uint32_t sp = fb_split_count(ctx, outputs, (uint64_t)terms * ((Wn + FB_GROUP - 1) / FB_GROUP));
    return {FB_BLOCK, sp < max_splits ? sp : max_splits};
}
// bpp_msm_vartime_batch: the warp or the block form
static fb_plan msm_table_plan(const bpp_ctx *ctx, const bpp_points *P, size_t n, size_t count) {
    return fb_choose(ctx, count, (uint32_t)n, P->fb_Wn, false, 256);
}
// d_sc: count x n scalars; d_out32: count x 32.  Stream-ordered, no synchronisation.
static int msm_table_run(bpp_ctx *ctx, const uint32_t *d_sc, const bpp_points *P, size_t off, size_t n, size_t count, uint8_t *d_out32,
                         uint32_t *d_ext, uint32_t *d_part, const fb_plan &pl) {
    acp_layout lay;
    memset(&lay, 0, sizeof(lay));
    lay.stride = (uint32_t)n;          // one "proof block" per MSM: its n scalars
    fb_shape sh;
    memset(&sh, 0, sizeof(sh));
    sh.nseg = 1; sh.cnt[0] = (uint32_t)n; sh.gen[0] = (uint32_t)off; sh.outs = 1;
    fb_consts kc;
    memcpy(kc.K, P->fb_K, 32);
    cudaStream_t st = ctx->stream;
    if (pl.form == FB_WARP) {
        fb_warp_launch(d_sc, lay, sh, P->fb_table, P->fb_c, P->fb_Wn, kc, (uint32_t)count, 1, d_ext, st);
        LAUNCH_CHECK(ctx);
    } else {
        k_fb_msm<<<dim3((unsigned)count, 1, pl.splits), FB_THREADS, 0, st>>>(d_sc, lay, sh, P->fb_table, P->fb_c, P->fb_Wn, kc,
                                                                           pl.splits > 1 ? d_part : d_ext);
        LAUNCH_CHECK(ctx);
        if (pl.splits > 1) {
            k_fb_sum_splits<<<dim3((unsigned)count, 1), 32, 0, st>>>(d_part, 1, pl.splits, 1, d_ext);
            LAUNCH_CHECK(ctx);
        }
    }
    k_compress_strided<<<(unsigned)((count + 127) / 128), 128, 0, st>>>(d_ext, 1, 0, 1, (uint32_t)count, d_out32);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}
extern "C" int bpp_msm_vartime_batch_dev(bpp_ctx *ctx, const void *d_scalars, size_t count, bpp_points *points, size_t off, size_t n,
                                         void *d_out32) {
    if (!ctx || !d_scalars || !points || !d_out32 || count == 0 || n == 0) return BPP_ERR_INVALID_ARG;
    if (off + n > points->n || count >= (1ull << 31)) return BPP_ERR_LENGTH_MISMATCH;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc;
    if (!points->fb_table && (rc = bpp_points_precompute(ctx, points, 8))) return rc;
    const fb_plan pl = msm_table_plan(ctx, points, n, count);
    const size_t ext_b = count * 128, part_b = pl.splits > 1 ? count * pl.splits * 128 : 0;
    if ((rc = grow(ctx, &ctx->d_small, &ctx->cap_small, ext_b + part_b))) return rc;
    return msm_table_run(ctx, (const uint32_t *)d_scalars, points, off, n, count, (uint8_t *)d_out32, (uint32_t *)ctx->d_small,
                         (uint32_t *)(ctx->d_small + ext_b), pl);
}
extern "C" int bpp_msm_vartime_batch(bpp_ctx *ctx, const uint8_t *scalars, size_t count, bpp_points *points, size_t off, size_t n,
                                     uint8_t *out32) {
    if (!ctx || !scalars || !points || !out32 || count == 0 || n == 0) return BPP_ERR_INVALID_ARG;
    if (off + n > points->n || count >= (1ull << 31)) return BPP_ERR_LENGTH_MISMATCH;
    for (size_t i = 0; i < count * n; i++)
        if (scalars[32 * i + 31] & 0x80) return BPP_ERR_SCALAR_RANGE;
    CK(ctx, cudaSetDevice(ctx->device));
    int rc;
    if (!points->fb_table && (rc = bpp_points_precompute(ctx, points, 8))) return rc;
    const fb_plan pl = msm_table_plan(ctx, points, n, count);
    const size_t sc_b = count * n * 32, ext_b = count * 128, part_b = pl.splits > 1 ? count * pl.splits * 128 : 0, out_b = count * 32;
    if ((rc = grow(ctx, &ctx->d_small, &ctx->cap_small, sc_b + ext_b + part_b + out_b))) return rc;
    uint8_t *d = ctx->d_small;
    CK(ctx, cudaMemcpyAsync(d, scalars, sc_b, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = msm_table_run(ctx, (const uint32_t *)d, points, off, n, count, d + sc_b + ext_b + part_b, (uint32_t *)(d + sc_b),
                            (uint32_t *)(d + sc_b + ext_b), pl)))
        return rc;
    CK(ctx, cudaMemcpyAsync(out32, d + sc_b + ext_b + part_b, out_b, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return BPP_OK;
}

// ---- batch object ----------------------------------------------------------------------------------
extern "C" size_t bpp_acproof_proof_len(size_t n) { return 32 * (11 + 2 * n); }
// mode 2 (`fixed`): 8 points | t_hat, tau_x, mu | (L_j, R_j) x lg | a, b
extern "C" size_t bpp_acproof_proof_len_mode(size_t n, int mode) {
    if (mode != 2) return bpp_acproof_proof_len(n);
    return 32 * (13 + 2 * (size_t)acp_log2(acp_next_pow2((uint32_t)n)));
}

// ---- proof wire format (SURVEY 8 row f-2) -----------------------------------------------------------------
// The reference defines no serialisation.  Mode 2 (`fixed`) adopts bulletproofs 4.0.0 R1CSProof::to_bytes for a
// one-phase proof (r1cs/proof.rs): version byte 0 | A_I1 A_O1 S1 | T_1 T_3 T_4 T_5 T_6 | t_x t_x_blinding e_blinding |
// L_0 R_0 .. | a b - i.e. the version byte followed by the library's own proof bytes.  Modes 0 and 1 (l, r in the
// clear: no upstream format) use the version bytes 0x80 / 0x81 the same way.  from_wire is the parser a batch
// verifier runs first: like R1CSProof::from_bytes it rejects (FormatError) a wrong version byte, a length that is
// not 1 + 32k or does not match the circuit, and any scalar field that is not canonical (>= l); points stay
// compressed - an invalid encoding is a VerificationError of the verifier, not a format error.  Pure byte handling:
// no device work, callable without a context.
static const uint8_t ACP_WIRE_VERSION[3] = {0x80, 0x81, 0x00};

static bool acp_scalar_is_canonical(const uint8_t *s) {   // little-endian s < l = 2^252 + 27742317777372353535851937790883648493
    static const uint8_t L[32] = {0xed, 0xd3, 0xf5, 0x5c, 0x1a, 0x63, 0x12, 0x58, 0xd6, 0x9c, 0xf7, 0xa2, 0xde, 0xf9, 0xde, 0x14,
                                  0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0x10};
    for (int i = 31; i >= 0; i--) {
        if (s[i] < L[i]) return true;
        if (s[i] > L[i]) return false;
    }
    return false;
}

extern "C" size_t bpp_acproof_wire_len(size_t n, int mode) { return 1 + bpp_acproof_proof_len_mode(n, mode); }

extern "C" int bpp_acproof_to_wire(size_t n, int mode, size_t count, const uint8_t *proofs, uint8_t *wire_out) {
    if (mode < 0 || mode > 2 || (count && (!proofs || !wire_out))) return BPP_ERR_INVALID_ARG;
    const size_t plen = bpp_acproof_proof_len_mode(n, mode);
    for (size_t p = 0; p < count; p++) {
        wire_out[p * (plen + 1)] = ACP_WIRE_VERSION[mode];
        memcpy(wire_out + p * (plen + 1) + 1, proofs + p * plen, plen);
    }
    return BPP_OK;
}

// wire: count records of wire_len bytes each.  status[p] = 0 ok, 1 format error (that proof's bytes in proofs_out are
// zeroed, so a verifier fed with them rejects).  Returns BPP_ERR_LENGTH_MISMATCH if wire_len itself is not the
// circuit's record length (nothing is parsed then).
extern "C" int bpp_acproof_from_wire(size_t n, int mode, size_t count, const uint8_t *wire, size_t wire_len,
                                     uint8_t *proofs_out, uint8_t *status) {
    if (mode < 0 || mode > 2 || (count && (!wire || !proofs_out || !status))) return BPP_ERR_INVALID_ARG;
    const size_t plen = bpp_acproof_proof_len_mode(n, mode);
    if (wire_len != plen + 1) return BPP_ERR_LENGTH_MISMATCH;
    const size_t words = plen / 32, lg = mode == 2 ? (words - 13) / 2 : 0;
    for (size_t p = 0; p < count; p++) {
        const uint8_t *rec = wire + p * wire_len, *body = rec + 1;
        bool ok = rec[0] == ACP_WIRE_VERSION[mode];
        for (size_t i = 8; ok && i < words; i++) {
            // scalar fields: modes 0/1 everything after the 8 points; mode 2 t_x, t_x_blinding, e_blinding and a, b
            const bool is_scalar = mode != 2 || i < 11 || i >= 11 + 2 * lg;
            if (is_scalar && !acp_scalar_is_canonical(body + 32 * i)) ok = false;
        }
        status[p] = ok ? 0 : 1;
        if (ok) memcpy(proofs_out + p * plen, body, plen);
        else memset(proofs_out + p * plen, 0, plen);
    }
    return BPP_OK;
}

extern "C" void bpp_acp_batch_free(bpp_acp_batch *b) {
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(b->ctx->stream);
    void *dev[] = {b->d_blk, b->d_seeds, b->d_wide, b->d_ext8, b->d_dyn, b->d_wsum, b->d_stat, b->d_bad, b->d_vext, b->d_vseed,
                   b->d_pts8, b->d_proofs, b->d_V, b->d_accept, b->d_lr, b->d_tx3, b->d_lrext, b->d_part, b->d_tr, b->d_proto, b->d_vdig, b->d_vwit, b->d_wgen, b->d_rlc_sc, b->d_rlc_flag, b->d_rlc_out, b->d_wstage};
    for (void *p : dev)
        if (p) cudaFree(p);
    if (b->h_pts8) cudaFreeHost(b->h_pts8);
    if (b->h_wide) cudaFreeHost(b->h_wide);
    if (b->h_proofs) cudaFreeHost(b->h_proofs);
    if (b->h_lr) cudaFreeHost(b->h_lr);
    if (b->h_tx3) cudaFreeHost(b->h_tx3);
    if (b->h_rlc_flag) cudaFreeHost(b->h_rlc_flag);
    if (b->h_V) cudaFreeHost(b->h_V);
    if (b->aux2) cudaStreamDestroy(b->aux2);
    if (b->aux3) cudaStreamDestroy(b->aux3);
    if (b->ev_join3) cudaEventDestroy(b->ev_join3);
    if (b->ev_fork2) cudaEventDestroy(b->ev_fork2);
    if (b->ev_join2) cudaEventDestroy(b->ev_join2);
    if (b->aux) cudaStreamDestroy(b->aux);
    if (b->bulk) cudaStreamDestroy(b->bulk);
    if (b->ev_bfork) cudaEventDestroy(b->ev_bfork);
    if (b->ev_bjoin) cudaEventDestroy(b->ev_bjoin);
    if (b->ev_fork) cudaEventDestroy(b->ev_fork);
    if (b->ev_join) cudaEventDestroy(b->ev_join);
    delete b;
}

static int acp_prepare_hsum(bpp_acp_batch *b);

// mode 0 = "reference" (bit-for-bit what circuit_lib.rs does, defects included; verification never
// accepts), mode 1 = "reference-fixed" (SURVEY A.3), mode 2 = "fixed" (standard powers + inner-product argument,
// ipa_kernels.cuh; needs next_pow2(n) generators).  label = the Transcript::new label (lib.rs:172: b"test").
extern "C" int bpp_acp_batch_create(bpp_ctx *ctx, const bpp_circuit *cir, const bpp_gens *gens, int mode, size_t count,
                                    const uint8_t *label, size_t label_len, bpp_acp_batch **out) {
    if (!ctx || !cir || !gens || !out || count == 0 || count > (1u << 24) || mode < 0 || mode > 2 ||
        (!label && label_len))
        return BPP_ERR_INVALID_ARG;
    if (gens->n != (mode == 2 ? acp_next_pow2(cir->n) : cir->n)) return BPP_ERR_LENGTH_MISMATCH;  // circuit_lib.rs:154-160 assert_eq!
    if (mode == 2 && acp_log2(acp_next_pow2(cir->n)) > IPA_MAX_LG) return BPP_ERR_INVALID_ARG;
    *out = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    bpp_acp_batch *b = new bpp_acp_batch();
    b->ctx = ctx; b->cir = cir; b->gens = gens; b->mode = mode; b->B = (uint32_t)count;
    b->lay = acp_make_layout(cir->n, cir->Q, cir->m, mode);
    b->proof_len = (uint32_t)bpp_acproof_proof_len_mode(cir->n, mode);
    if (const char *e = getenv("BPP_ACP_TRACE")) b->trace = e[0] == '1';
    if (const char *e = getenv("BPP_DECOMPRESS_LATE")) b->decompress_late = e[0] == '1';
    b->label.assign(label, label + label_len);
    const size_t B = count, lg = b->lay.lg, per = cir->m + 8 + 2 * lg, nch = 6 + lg;   // challenges per proof + the two weights
    // split scratch of the block form: the largest MSM's terms at 8 work items each (c = 8) whatever the table's width,
    // so that for c < 8 this, not the launch's own item count, caps the split count
    b->fb_splits = fb_split_count(ctx, B, (2 * (uint64_t)b->lay.np + 2) * 8);
    cudaError_t e = cudaMalloc((void **)&b->d_blk, B * b->lay.stride * 32);
    if (e == cudaSuccess) e = cudaMemsetAsync(b->d_blk, 0, B * b->lay.stride * 32, ctx->stream);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_seeds, B * 32);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->aux, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_join, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->aux2, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_fork2, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_join2, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->aux3, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_join3, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_tr, B * MERLIN_STATE_WORDS * 8);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_proto, 2 * MERLIN_STATE_WORDS * 8);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_vdig, B * TR_V_CHUNKS(cir->m) * 32);
    if (e == cudaSuccess) {   // Transcript::new(label) + arithmetic_domain_sep(n): identical for every proof, hashed once
        bpp_host::Transcript proto(b->label.data(), b->label.size());
        proto.arithmetic_domain_sep(cir->n);
        uint64_t st[2 * MERLIN_STATE_WORDS];
        proto.export_state(st);
        bpp_host::Transcript vproto((const uint8_t *)"acp-V", 5);
        vproto.export_state(st + MERLIN_STATE_WORDS);
        e = cudaMemcpyAsync(b->d_proto, st, sizeof(st), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_wide, B * nch * 64);
    if (e == cudaSuccess && b->fb_splits > 1) e = cudaMalloc((void **)&b->d_part, B * 8 * b->fb_splits * 128);
    if (e == cudaSuccess && lg) e = cudaMalloc((void **)&b->d_lr, B * 2 * lg * 32);
    if (e == cudaSuccess && lg) e = cudaMalloc((void **)&b->d_lrext, B * 2 * lg * 128);
    if (e == cudaSuccess && lg) e = cudaMalloc((void **)&b->d_tx3, B * 3 * 32);
    if (e == cudaSuccess && lg) e = cudaMallocHost((void **)&b->h_lr, B * 2 * lg * 32);
    if (e == cudaSuccess && lg) e = cudaMallocHost((void **)&b->h_tx3, B * 3 * 32);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_ext8, B * 8 * 128);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_dyn, (B * per + gens->n_gens) * 96);   // + the shared generators (RLC batch MSM)
    if (e == cudaSuccess) e = cudaMemcpyAsync(b->d_dyn + 24 * B * per, gens->pts->niels, (size_t)gens->n_gens * 96, cudaMemcpyDeviceToDevice,
                                              ctx->stream);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_rlc_sc, (B * per + gens->n_gens) * 32);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_rlc_flag, 64);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_rlc_out, 256);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&b->h_rlc_flag, 64);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_wsum, B * DYN_W * 128);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_stat, B * 128);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_bad, B * 4);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_vseed, 64);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_pts8, B * 8 * 32);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_proofs, B * b->proof_len);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_V, B * cir->m * 32);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_vext, B * cir->m * 128);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_accept, B);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&b->h_pts8, B * 8 * 32);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&b->h_wide, B * nch * 64);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&b->h_proofs, B * b->proof_len);
    if (e != cudaSuccess) {
        ctx->last_error = cudaGetErrorString(e);
        bool oom = e == cudaErrorMemoryAllocation;
        cudaGetLastError();
        bpp_acp_batch_free(b);
        return oom ? BPP_ERR_OOM : BPP_ERR_CUDA;
    }
    if (int rc = acp_prepare_hsum(b)) {
        bpp_acp_batch_free(b);
        return rc;
    }
    *out = b;
    return BPP_OK;
}

// Verification strategy: 1 (default) = one random-linear-combination MSM over the whole batch first, per-proof
// kernels only if it fails (some proof is invalid); 0 = always per proof.  Decisions are identical.
extern "C" int bpp_acp_batch_set_priority_split(bpp_acp_batch *b, int on) {
    if (!b) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    if (on && !b->bulk) {
        int lo = 0, hi = 0;
        CK(ctx, cudaSetDevice(ctx->device));
        CK(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CK(ctx, cudaStreamCreateWithPriority(&b->bulk, cudaStreamNonBlocking, lo));
        CK(ctx, cudaEventCreateWithFlags(&b->ev_bfork, cudaEventDisableTiming));
        CK(ctx, cudaEventCreateWithFlags(&b->ev_bjoin, cudaEventDisableTiming));
    }
    b->priority_split = on != 0;
    return BPP_OK;
}

extern "C" int bpp_acp_batch_set_batch_rlc(bpp_acp_batch *b, int on) {
    if (!b) return BPP_ERR_INVALID_ARG;
    b->batch_rlc = on != 0;
    return BPP_OK;
}

// Fiat-Shamir location: 0 (default) = per-proof Merlin transcripts on the device, 1 = on host threads.
// Both produce the same challenges; proofs and decisions are identical (tests/test_gpu_acproof.py).
extern "C" int bpp_acp_batch_set_host_transcripts(bpp_acp_batch *b, int on) {
    if (!b) return BPP_ERR_INVALID_ARG;
    b->host_transcripts = on != 0;
    return BPP_OK;
}

template <typename F>
static void acp_parallel_for(uint32_t n, F fn) {
    unsigned T = std::thread::hardware_concurrency();
    if (T == 0) T = 4;
    if (T > 32) T = 32;
    if (n < 64 || T == 1) { for (uint32_t i = 0; i < n; i++) fn(i); return; }
    std::vector<std::thread> th;
    uint32_t per = (n + T - 1) / T;
    for (unsigned t = 0; t < T; t++) {
        uint32_t lo = t * per, hi = lo + per < n ? lo + per : n;
        if (lo >= hi) break;
        th.emplace_back([=]() { for (uint32_t i = lo; i < hi; i++) fn(i); });
    }
    for (auto &x : th) x.join();
}

static fb_shape acp_shape(uint32_t outs) {
    fb_shape s;
    memset(&s, 0, sizeof(s));
    s.outs = outs;
    return s;
}
static void acp_seg(fb_shape &s, uint32_t off, uint32_t ostride, uint32_t gen, uint32_t cnt) {
    s.sc_off[s.nseg] = off; s.sc_ostride[s.nseg] = ostride; s.gen[s.nseg] = gen; s.cnt[s.nseg] = cnt;
    s.nseg++;
}
// the form acp_fb runs for this shape: the split scratch holds 8 outputs per proof, so launches with more do not split
static fb_plan acp_fb_plan(const bpp_acp_batch *b, const fb_shape &sh) {
    return fb_choose(b->ctx, (uint64_t)b->B * sh.outs, fb_terms(sh), b->gens->pts->fb_Wn, !sh.sel_period,
                     sh.outs > 8 ? 1 : b->fb_splits);
}
// A_I = alpha*h + <a_L,G> + <a_R,H>.  For a witness of bpp_acp_batch_gen_shuffle_witness, a_R[i] = v'[i] - x on the first
// n - 2 multipliers and 0 on the last two, so (the group has prime order) <a_R,H> = <v',H> + (-x) H_sum with H_sum =
// H_0 + .. + H_{n-3}: the same point.  Card values are small integers, so v' has one non-zero digit where a_R has
// Wn, and the digit-staged warp kernel spreads those digits over all lanes (fb_sparse): A_I costs (1 + n/2) x Wn
// + (n - 2) + Wn table adds per proof instead of (1 + n) x Wn for a small deck (52 cards, c = 16: 1766 instead of
// 3280).  structured: that shape, which only the digit-staged warp form runs (acp_ai_structured_ok).
static fb_shape acp_ai_shape(const bpp_acp_batch *b, bool structured, fb_sparse *sp = nullptr) {
    const acp_layout &L = b->lay;
    const uint32_t gH = 2 + b->gens->n;   // first H generator (gens order g, h, G[..], H[..])
    fb_shape sh = acp_shape(1);
    acp_seg(sh, L.alpha, 0, 1, 1); acp_seg(sh, L.aL, 0, 2, L.n);
    if (!structured) {
        acp_seg(sh, L.aR, 0, gH, L.n);
        return sh;
    }
    acp_seg(sh, L.vr, 0, gH, L.n - 2); acp_seg(sh, L.nx, 0, 0, 1);
    if (sp) *sp = fb_sparse{1, 1u << 3, b->hsum ? b->hsum->fb_table : nullptr};
    return sh;
}
static bool acp_ai_structured_ok(const bpp_acp_batch *b) {
    if (!acp_shuffle_shaped(b->lay.n, b->lay.m)) return false;
    const bpp_points &P = *b->gens->pts;
    fb_sparse sp;
    const fb_shape sh = acp_ai_shape(b, true, &sp);
    return acp_fb_plan(b, sh).form == FB_WARP && fb_warp_d_fits(sh, sp, P.fb_c, P.fb_Wn);
}
// H_sum's table for batches that can use the structured A_I, shared by every batch over the same generators: built on
// first use (one warp sums the points, the sum goes through compression and bpp_points_upload, then gets its own table
// at the generators' width), looked up under the generators' lock afterwards.
static int acp_prepare_hsum(bpp_acp_batch *b) {
    if (!acp_ai_structured_ok(b)) return BPP_OK;
    bpp_ctx *ctx = b->ctx;
    bpp_gens *g = const_cast<bpp_gens *>(b->gens);
    const uint32_t first = 2 + g->n, cnt = b->lay.n - 2;
    const int c = g->pts->fb_c;
    std::lock_guard<std::mutex> lock(g->mu);
    for (const auto &e : g->sums)
        if (e.first == first && e.cnt == cnt && e.pts->fb_c == c) {
            b->hsum = e.pts;
            return BPP_OK;
        }
    uint32_t *d = nullptr;
    CK(ctx, cudaMalloc((void **)&d, 128 + 32));
    uint8_t enc[32];
    k_point_sum<<<1, 32, 0, ctx->stream>>>(g->pts->niels, first, cnt, d);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) {
        k_compress_batch<<<1, 128, 0, ctx->stream>>>(d, 1, (uint8_t *)(d + 32));
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(enc, d + 32, 32, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess) {
        ctx->last_error = cudaGetErrorString(e);
        return BPP_ERR_CUDA;
    }
    ctx->launches += 2;
    bpp_points *pts = nullptr;
    int rc = bpp_points_upload(ctx, BPP_FMT_COMPRESSED, enc, 1, &pts);
    if (rc) return rc;
    if ((rc = bpp_points_precompute(ctx, pts, c))) {
        bpp_points_free(ctx, pts);
        return rc;
    }
    g->sums.push_back({first, cnt, pts});
    b->hsum = pts;
    return BPP_OK;
}

// The fixed-base MSM launch over B proof blocks of layout `lay` in the form `pl`: results land in dst[(p * pitch + o)]
// (raw extended points).  part: the split scratch of the block form (B x outs x pl.splits partial sums); deferred_splits:
// when given and the launch is split, the partial sums are left there for the caller's own tail kernel (their count is
// written; 1 = the result is complete in dst).
static int fb_launch(bpp_ctx *ctx, const uint32_t *blk, const acp_layout &lay, uint32_t B, const bpp_points &P, const fb_shape &sh,
                     const fb_plan &pl, uint32_t *dst, uint32_t pitch, cudaStream_t st, uint32_t *part, uint32_t *deferred_splits,
                     const fb_sparse &sp = fb_sparse{}) {
    if (deferred_splits) *deferred_splits = 1;
    if ((sp.on || sp.alt) && !(pl.form == FB_WARP && fb_warp_d_fits(sh, sp, P.fb_c, P.fb_Wn))) {
        ctx->last_error = "fixed-base MSM: a sparse / two-table shape needs the digit-staged warp form";
        return BPP_ERR_INVALID_ARG;
    }
    fb_shape s = sh;
    s.outs = pitch;  // the kernels address out_ext + 32 * (p * outs + o)
    fb_consts kc;
    memcpy(kc.K, P.fb_K, 32);
    if (pl.form == FB_SMALL) {
        const uint32_t total = B * sh.outs;
        k_fb_msm_small<<<(total + 127) / 128, 128, 0, st>>>(blk, lay, s, P.fb_table, P.fb_c, P.fb_Wn, kc, B, sh.outs, dst);
        LAUNCH_CHECK(ctx);
    } else if (pl.form == FB_WARP) {
        fb_warp_launch(blk, lay, s, P.fb_table, P.fb_c, P.fb_Wn, kc, B, sh.outs, dst, st, sp);
        LAUNCH_CHECK(ctx);
    } else {
        k_fb_msm<<<dim3(B, sh.outs, pl.splits), FB_THREADS, 0, st>>>(blk, lay, s, P.fb_table, P.fb_c, P.fb_Wn, kc,
                                                                    pl.splits > 1 ? part : dst);
        LAUNCH_CHECK(ctx);
        if (pl.splits > 1 && deferred_splits) {
            *deferred_splits = pl.splits;
        } else if (pl.splits > 1) {
            k_fb_sum_splits<<<dim3(B, sh.outs), 32, 0, st>>>(part, sh.outs, pl.splits, pitch, dst);
            LAUNCH_CHECK(ctx);
        }
    }
    return BPP_OK;
}
// fb_launch over this batch's proof blocks.  on: run on this stream instead of the context's (small batches: independent
// commitments side by side); part_region: which eighth of the split scratch to use (concurrent split launches must not
// share it).  With the priority split, the GPU-filling forms go to the low-priority stream.
static int acp_fb(bpp_acp_batch *b, const fb_shape &sh, uint32_t *dst, uint32_t pitch, cudaStream_t on = nullptr,
                  uint32_t part_region = 0, uint32_t *deferred_splits = nullptr, const fb_sparse &sp = fb_sparse{}) {
    bpp_ctx *ctx = b->ctx;
    const bpp_points &P = *b->gens->pts;
    const fb_plan pl = acp_fb_plan(b, sh);
    uint32_t *part = b->d_part + 32 * (size_t)part_region * b->B * b->fb_splits;
    if (pl.form == FB_SMALL) return fb_launch(ctx, b->d_blk, b->lay, b->B, P, sh, pl, dst, pitch, ctx->stream, part, deferred_splits, sp);
    cudaStream_t st = on ? on : ctx->stream;
    if (b->priority_split && !on) {   // the GPU-filling launch goes to the low-priority stream, bracketed by events
        st = b->bulk;
        CK(ctx, cudaEventRecord(b->ev_bfork, ctx->stream));
        CK(ctx, cudaStreamWaitEvent(st, b->ev_bfork, 0));
    }
    int rc = fb_launch(ctx, b->d_blk, b->lay, b->B, P, sh, pl, dst, pitch, st, part, deferred_splits, sp);
    if (rc) return rc;
    if (b->priority_split && !on) {
        CK(ctx, cudaEventRecord(b->ev_bjoin, st));
        CK(ctx, cudaStreamWaitEvent(ctx->stream, b->ev_bjoin, 0));
    }
    return BPP_OK;
}

__global__ void __launch_bounds__(128) k_compress_strided(const uint32_t *__restrict__ ext, uint32_t pitch, uint32_t first,
                                                          uint32_t cnt, uint32_t B, uint8_t *__restrict__ out32) {
    uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= B * cnt) return;
    uint32_t p = id / cnt, k = first + (id - p * cnt);
    ge_ext pt;
    ge_load(pt, ext + 32 * ((size_t)p * pitch + k));
    ge_compress(out32 + 32 * ((size_t)p * pitch + k), pt);
}

// witness: a_L, a_R, a_O (count x n), gamma (count x m), prover RNG seeds (count x 32)
extern "C" int bpp_acp_batch_upload_witness(bpp_acp_batch *b, const uint8_t *aL, const uint8_t *aR, const uint8_t *aO,
                                            const uint8_t *gamma, const uint8_t *seeds) {
    if (!b || !aL || !aR || !aO || !gamma || !seeds) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    // four contiguous copies at full link speed into a staging buffer, then one kernel places every scalar in
    // its proof's block (a strided 2-D copy of 3 KB rows runs at a fraction of the link rate)
    const size_t n32 = (size_t)b->lay.n * 32 * b->B, m32 = (size_t)b->lay.m * 32 * b->B;
    if (!b->d_wstage) CK(ctx, cudaMalloc((void **)&b->d_wstage, 3 * n32 + m32));
    uint8_t *st = (uint8_t *)b->d_wstage;
    CK(ctx, cudaMemcpyAsync(st, aL, n32, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaMemcpyAsync(st + n32, aR, n32, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaMemcpyAsync(st + 2 * n32, aO, n32, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaMemcpyAsync(st + 3 * n32, gamma, m32, cudaMemcpyHostToDevice, ctx->stream));
    {
        const uint32_t per = 3 * b->lay.n + b->lay.m;
        k_acp_place_witness<<<dim3((per + 127) / 128, b->B), 128, 0, ctx->stream>>>(b->d_wstage, b->lay, b->B, b->d_blk);
        LAUNCH_CHECK(ctx);
    }
    CK(ctx, cudaMemcpyAsync(b->d_seeds, seeds, (size_t)b->B * 32, cudaMemcpyHostToDevice, ctx->stream));
    b->shuffle_wit = false;
    return BPP_OK;
}

// The k-card shuffle witness generated on the device (weights.rs:38-113 create_variables + create_a for the circuit of
// bpp_circuit_create_shuffle): the caller sends what defines the shuffles - the deck, one permutation and one challenge
// value per proof - plus the blindings and RNG seeds, 4 k + 32 (m + 2) bytes per proof instead of the 32 (3 n + m + 1) of
// bpp_acp_batch_upload_witness (52 cards: 3.6 KB instead of 13.4 KB).  v = deck | deck[perm] | x stays resident for
// bpp_acp_batch_commit(b, NULL, ..).
extern "C" int bpp_acp_batch_gen_shuffle_witness(bpp_acp_batch *b, const uint8_t *deck, const uint32_t *perm, const uint8_t *x,
                                                 const uint8_t *gamma, const uint8_t *seeds) {
    if (!b || !deck || !perm || !x || !gamma || !seeds) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    const acp_layout &L = b->lay;
    if (L.n < 4 || (L.n & 1u) || L.m != L.n + 1) {
        ctx->last_error = "gen_shuffle_witness: not a shuffle circuit (n = 2k, m = 2k + 1)";
        return BPP_ERR_INVALID_ARG;
    }
    const uint32_t k = L.n / 2, B = b->B;
    const size_t m32 = (size_t)L.m * 32 * B, dk = (size_t)k * 32, pk = (size_t)B * k * 4, xb = (size_t)B * 32;
    if (!b->d_vwit) CK(ctx, cudaMalloc((void **)&b->d_vwit, m32));
    if (!b->d_wgen) CK(ctx, cudaMalloc((void **)&b->d_wgen, m32 + dk + pk + xb));
    uint8_t *st = (uint8_t *)b->d_wgen;   // gamma | deck | x | perm
    CK(ctx, cudaMemcpyAsync(st, gamma, m32, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaMemcpyAsync(st + m32, deck, dk, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaMemcpyAsync(st + m32 + dk, x, xb, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaMemcpyAsync(st + m32 + dk + xb, perm, pk, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaMemcpyAsync(b->d_seeds, seeds, (size_t)B * 32, cudaMemcpyHostToDevice, ctx->stream));
    k_acp_place_gamma<<<dim3((L.m + 127) / 128, B), 128, 0, ctx->stream>>>((const uint32_t *)st, L, b->d_blk);
    LAUNCH_CHECK(ctx);
    if (k <= 64 || (k <= 1024 && 2ull * B >= 2048)) {
        // short chains or enough of them: a thread per chain
        k_shuffle_witness_serial<<<(2 * B + 63) / 64, 64, 0, ctx->stream>>>((const uint32_t *)(st + m32), (const uint32_t *)(st + m32 + dk + xb),
                                                                           (const uint32_t *)(st + m32 + dk), k, B, L, b->d_blk, b->d_vwit);
    } else {
        unsigned wit_threads = 32;
        while (wit_threads < WIT_THREADS && wit_threads < k - 1) wit_threads <<= 1;
        k_shuffle_witness<<<dim3(2, B), wit_threads, 0, ctx->stream>>>((const uint32_t *)(st + m32), (const uint32_t *)(st + m32 + dk + xb),
                                                                      (const uint32_t *)(st + m32 + dk), k, L, b->d_blk, b->d_vwit);
    }
    LAUNCH_CHECK(ctx);
    b->have_vwit = true;
    b->shuffle_wit = true;
    return BPP_OK;
}

// commit_variables (weights.rs:58-61): V_j = v_j * g + gamma_j * h for the uploaded gamma; the compressed
// commitments are returned (count x m x 32) and also stay resident as this batch's V.  v = NULL: the values generated
// by bpp_acp_batch_gen_shuffle_witness.
extern "C" int bpp_acp_batch_commit(bpp_acp_batch *b, const uint8_t *v, uint8_t *V_out) {
    if (!b || (!v && !b->have_vwit)) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    const acp_layout &L = b->lay;
    // v is staged in the l/r area of the proof block (not yet used at this point; 2n >= m)
    if (2 * L.n < L.m) return BPP_ERR_INVALID_ARG;
    const size_t pitch = (size_t)L.stride * 32, m32 = (size_t)L.m * 32;
    CK(ctx, cudaMemcpy2DAsync((uint8_t *)b->d_blk + 32 * (size_t)L.l, pitch, v ? (const void *)v : (const void *)b->d_vwit, m32, m32, b->B,
                              v ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, ctx->stream));
    fb_shape sh = acp_shape(L.m);
    acp_seg(sh, L.l, 1, 0, 1);
    acp_seg(sh, L.gamma, 1, 1, 1);
    int rc = acp_fb(b, sh, b->d_vext, L.m);
    if (rc) return rc;
    k_compress_strided<<<(b->B * L.m + 127) / 128, 128, 0, ctx->stream>>>(b->d_vext, L.m, 0, L.m, b->B, b->d_V);
    LAUNCH_CHECK(ctx);
    if (V_out) CK(ctx, cudaMemcpyAsync(V_out, b->d_V, (size_t)b->B * L.m * 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    b->have_V = true;
    return BPP_OK;
}

// The value commitments of the batch (count x m x 32 compressed): the prover binds them to its transcript (modes 1, 2),
// the verifier needs them for check 2.
extern "C" int bpp_acp_batch_upload_commitments(bpp_acp_batch *b, const uint8_t *V) {
    if (!b || !V) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(b->d_V, V, (size_t)b->B * b->lay.m * 32, cudaMemcpyHostToDevice, ctx->stream));
    b->have_V = true;
    return BPP_OK;
}

// host transcripts: the commitments on the host (pinned), fetched from the resident copy
static int acp_fetch_commitments(bpp_acp_batch *b) {
    bpp_ctx *ctx = b->ctx;
    const size_t bytes = (size_t)b->B * b->lay.m * 32;
    if (!b->h_V) CK(ctx, cudaMallocHost((void **)&b->h_V, bytes));
    CK(ctx, cudaMemcpyAsync(b->h_V, b->d_V, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return BPP_OK;
}
static void acp_host_append_commitments(bpp_host::Transcript &t, const uint8_t *V, uint32_t m) {
    t.append_u64("m", m);
    std::vector<uint8_t> digs(32 * (size_t)TR_V_CHUNKS(m));
    for (uint32_t c = 0; c < m; c += TR_V_CHUNK) {   // two levels, see k_tr_vchunks
        bpp_host::Transcript ch((const uint8_t *)"acp-V", 5);
        ch.append_u64("chunk", c / TR_V_CHUNK);
        ch.append_message("V", V + 32 * (size_t)c, 32 * (size_t)((m - c) < TR_V_CHUNK ? (m - c) : TR_V_CHUNK));
        ch.challenge_bytes("d", digs.data() + 32 * (size_t)(c / TR_V_CHUNK), 32);
    }
    t.append_message("Vd", digs.data(), digs.size());   // the chunk digests, concatenated, as one message
}
// device transcripts: the chunk digests of the resident commitments, on the second side stream
static int acp_fork_vchunks(bpp_acp_batch *b) {
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaEventRecord(b->ev_fork2, ctx->stream));
    CK(ctx, cudaStreamWaitEvent(b->aux2, b->ev_fork2, 0));
    TR_LAUNCH(k_tr_vchunks, b->B * TR_V_CHUNKS(b->lay.m), b->aux2, b->d_proto + MERLIN_STATE_WORDS, b->d_V, b->lay.m,
                                                                                      b->B, b->d_vdig);
    LAUNCH_CHECK(ctx);
    CK(ctx, cudaEventRecord(b->ev_join2, b->aux2));
    return BPP_OK;
}

// h_wide[byte_off ..): B x per wide (64-byte) values -> scalars at layout offset `off` of every proof
static int acp_put_challenges(bpp_acp_batch *b, uint32_t off, uint32_t per, size_t byte_off = 0) {
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaMemcpyAsync((uint8_t *)b->d_wide + byte_off, b->h_wide + byte_off, (size_t)b->B * per * 64, cudaMemcpyHostToDevice,
                            ctx->stream));
    k_acp_put_wide<<<(b->B * per + 127) / 128, 128, 0, ctx->stream>>>(b->d_wide + byte_off / 4, b->lay, off, per, b->B, b->d_blk);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}

// The verifier's secret randomness (k_tr_weights): the caller's 32 bytes, or 32 bytes from the operating system when the
// caller passes NULL.  Soundness of the fused per-proof check and of the batch combination needs weights the prover
// cannot predict; they are additionally bound to every byte of each proof through its transcript.
#include <sys/random.h>
static int set_verifier_seed(bpp_ctx *ctx, uint32_t *d_vseed, const uint8_t *seed, uint8_t host_copy[32]) {
    if (seed) {
        memcpy(host_copy, seed, 32);
    } else {
        size_t got = 0;
        while (got < 32) {
            ssize_t r = getrandom(host_copy + got, 32 - got, 0);
            if (r <= 0) {
                ctx->last_error = "getrandom failed: no verifier seed";
                return BPP_ERR_INVALID_ARG;
            }
            got += (size_t)r;
        }
    }
    CK(ctx, cudaMemcpyAsync(d_vseed, host_copy, 32, cudaMemcpyHostToDevice, ctx->stream));   // pageable: staged before return
    return BPP_OK;
}
static int acp_set_verifier_seed(bpp_acp_batch *b, const uint8_t *seed, uint8_t host_copy[32]) {
    return set_verifier_seed(b->ctx, b->d_vseed, seed, host_copy);
}
// device transcripts: continue every proof's final verifier state into its weights, on the second side stream
static int acp_fork_weights(bpp_acp_batch *b) {
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaEventRecord(b->ev_fork2, ctx->stream));
    CK(ctx, cudaStreamWaitEvent(b->aux2, b->ev_fork2, 0));
    TR_LAUNCH(k_tr_weights, b->B, b->aux2, b->d_tr, b->d_proofs, b->proof_len, (const uint8_t *)b->d_vseed, b->lay,
                                                              b->B, b->mode, b->d_blk);
    LAUNCH_CHECK(ctx);
    CK(ctx, cudaEventRecord(b->ev_join2, b->aux2));
    return BPP_OK;
}
// host transcripts: the same continuation on the host; writes the wide values of w and rho to out128
static void acp_host_weights(bpp_host::Transcript &t, const uint8_t *proof, uint32_t proof_len, const uint8_t seed[32],
                             uint32_t p, int mode, uint8_t *out128) {
    if (mode == 0) { memset(out128, 0, 128); return; }
    t.append_message("proof-tail", proof + 256, proof_len - 256);
    t.append_message("verifier-seed", seed, 32);
    t.append_u64("proof-index", p);
    t.challenge_wide("w", out128);
    t.challenge_wide("rho", out128 + 64);
}

static int acp_challenge_dependent_scalars(bpp_acp_batch *b) {
    bpp_ctx *ctx = b->ctx;
    const acp_layout &L = b->lay;
    if (b->mode == 2) {   // standard powers y^i, y^-i (i < n'), z^(q+1)
        k_pow_table<<<(b->B + 63) / 64, 64, 0, ctx->stream>>>(L, b->B, b->d_blk);
        LAUNCH_CHECK(ctx);
        k_pow_fill<<<dim3((2 * L.np + L.Q + 127) / 128, b->B), 128, 0, ctx->stream>>>(L, b->d_blk);
        LAUNCH_CHECK(ctx);
    } else {
        k_acp_pow<<<(b->B + 31) / 32, ACP_POW_THREADS, 0, ctx->stream>>>(L, b->B, b->d_blk);
        LAUNCH_CHECK(ctx);
        k_acp_pow_unmont<<<dim3((2 * L.n + L.Q + 127) / 128, b->B), 128, 0, ctx->stream>>>(L, b->d_blk);
        LAUNCH_CHECK(ctx);
    }
    acp_csr W{b->cir->d_rowptr, b->cir->d_col, b->cir->d_kind, b->cir->d_coeff, b->cir->rows};
    k_acp_csr<<<dim3((W.rows + 127) / 128, b->B), 128, 0, ctx->stream>>>(W, L, b->d_blk);
    LAUNCH_CHECK(ctx);
    if (b->cir->n_long) {
        k_acp_csr_long<<<dim3(b->cir->n_long, b->B), 128, 0, ctx->stream>>>(W, b->cir->d_long, L, b->d_blk);
        LAUNCH_CHECK(ctx);
    }
    k_acp_vec1<<<dim3((L.n + 127) / 128, b->B), 128, 0, ctx->stream>>>(L, b->d_blk);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}

// The prover's inner-product rounds (scalar folding, ipa_kernels.cuh), shared by the `fixed` mode and the stand-alone
// batch.  On entry the transcripts stand after innerproduct_domain_sep and the block holds a, b (lay.l, lay.r), the
// H factors (lay.yninv), the G factors (lay.yn, io.gf only) and the Q scalar (lay.wq).  G = gens[gG ..), H = gens[gH ..),
// Q = gens[gQ].  fb(shape, dst, pitch, split_n) launches the fixed-base MSM (acp_fb's contract); host_u(j), when set,
// draws u_j on host transcripts from the compressed L_j, R_j and leaves u_j, u_j^-1 in the block.  Without it the
// transcripts are the device states io.tr: batches of up to 1023 proofs run each round's split sums, compression and
// challenge in one launch (k_ipa_lr_tail), larger ones through k_compress_strided + k_ipa_challenge.
struct ipa_rounds_io {
    uint32_t *blk, *lrext, *part;
    uint8_t *lr;        // B x 2 lg x 32: the compressed L_j, R_j
    uint64_t *tr;
    uint32_t gG, gH, gQ;
    bool gf;
};
template <class FB>
static int ipa_prove_rounds(bpp_ctx *ctx, const acp_layout &L, uint32_t B, const ipa_rounds_io &io, FB fb,
                            const std::function<int(uint32_t)> &host_u) {
    const uint32_t np = L.np, lg = L.lg;
    cudaStream_t s = ctx->stream;
    int rc;
    CK(ctx, ipa_round_launch(L, -1, io.blk, B, s, io.gf));   // s table = {1}, c_L, c_R and the MSM scalars of round 0
    ctx->launches++;
    for (uint32_t j = 0; j < lg; j++) {
        const uint32_t nj = np >> j;
        fb_shape sh = acp_shape(2);
        sh.sel_period = nj;
        acp_seg(sh, L.vG, 0, io.gG, np); sh.sel[0] = 1;    // <a_L s, G_R> for L, <a_R s, G_L> for R
        acp_seg(sh, L.vH, 0, io.gH, np); sh.sel[1] = 2;    // <b_R s^-1 y^-n, H_L> for L, <b_L .., H_R> for R
        acp_seg(sh, L.cl, 1, io.gQ, 1);  sh.sel[2] = 0;    // c_L Q, c_R Q
        // small batches with device transcripts: split sums, compression, transcript and u^-1 in one launch
        const bool fuse_tail = !host_u && B <= 1023;
        uint32_t split_n = 1;
        if ((rc = fb(sh, io.lrext + 32 * 2 * (size_t)j, 2 * lg, fuse_tail ? &split_n : nullptr))) return rc;
        if (split_n > 1) {
            k_ipa_lr_tail<<<B, 64, 0, s>>>(io.part, split_n, io.lrext, io.lr, L, (int)j, io.tr, io.blk);
            LAUNCH_CHECK(ctx);
            CK(ctx, ipa_round_launch(L, (int)j, io.blk, B, s, io.gf));
            ctx->launches++;
            continue;
        }
        k_compress_strided<<<(2 * B + 127) / 128, 128, 0, s>>>(io.lrext, 2 * lg, 2 * j, 2, B, io.lr);
        LAUNCH_CHECK(ctx);
        if (!host_u) {
            TR_LAUNCH_AT(tr_warp_max() < 1023 ? tr_warp_max() : 1023, k_ipa_challenge, B, s, io.lr, L, B, (int)j, io.tr, io.blk);
            LAUNCH_CHECK(ctx);
        } else if ((rc = host_u(j))) {
            return rc;
        }
        CK(ctx, ipa_round_launch(L, (int)j, io.blk, B, s, io.gf));   // fold a, b; s table; next round's c_L, c_R and MSM scalars
        ctx->launches++;
    }
    return BPP_OK;
}

// `fixed` mode tail of the prover (bulletproofs 4.0.0 inner_product_proof.rs create() behind dalek's R1CS glue):
// append t_x, t_x_blinding, e_blinding -> w; lg rounds of (L_j, R_j) -> u_j with a, b folded in place.
static int acp_prove_ipa(bpp_acp_batch *b) {
    bpp_ctx *ctx = b->ctx;
    const acp_layout &L = b->lay;
    const uint32_t B = b->B, np = L.np, lg = L.lg;
    cudaStream_t s = ctx->stream;
    int rc;
    if (!b->host_transcripts) {
        TR_LAUNCH_AT(tr_warp_max() < 1023 ? tr_warp_max() : 1023, k_ipa_challenge, B, s, nullptr, L, B, -1, b->d_tr, b->d_blk);
        LAUNCH_CHECK(ctx);
    } else {
        // t_hat, tau_x, mu are contiguous in the proof block
        CK(ctx, cudaMemcpy2DAsync(b->h_tx3, 96, ACP_PTR(b->d_blk, L, 0, L.that), (size_t)L.stride * 32, 96, B, cudaMemcpyDeviceToHost, s));
        CK(ctx, cudaStreamSynchronize(s));
        acp_parallel_for(B, [&](uint32_t p) {
            bpp_host::Transcript &t = b->tr[p];
            const uint8_t *sc3 = b->h_tx3 + 96 * (size_t)p;
            t.append_scalar("t_x", sc3);
            t.append_scalar("t_x_blinding", sc3 + 32);
            t.append_scalar("e_blinding", sc3 + 64);
            t.challenge_wide("w", b->h_wide + 64 * (size_t)p);
            t.append_message("dom-sep", (const uint8_t *)"ipp v1", 6);
            t.append_u64("n", np);
        });
        if ((rc = acp_put_challenges(b, L.wq, 1))) return rc;
    }
    ipa_rounds_io io;
    io.blk = b->d_blk; io.lr = b->d_lr; io.lrext = b->d_lrext; io.part = b->d_part; io.tr = b->d_tr;
    io.gG = 2; io.gH = 2 + b->gens->n; io.gQ = 0;   // Q = w g
    io.gf = false;
    auto fb = [&](const fb_shape &sh, uint32_t *dst, uint32_t pitch, uint32_t *split_n) {
        return acp_fb(b, sh, dst, pitch, nullptr, 0, split_n);
    };
    std::function<int(uint32_t)> host_u;
    if (b->host_transcripts)
        host_u = [&](uint32_t j) -> int {
            CK(ctx, cudaMemcpy2DAsync(b->h_pts8, 64, b->d_lr + 64 * (size_t)j, 64 * (size_t)lg, 64, B, cudaMemcpyDeviceToHost, s));
            CK(ctx, cudaStreamSynchronize(s));
            acp_parallel_for(B, [&](uint32_t p) {
                bpp_host::Transcript &t = b->tr[p];
                t.append_point("L", b->h_pts8 + 64 * (size_t)p);
                t.append_point("R", b->h_pts8 + 64 * (size_t)p + 32);
                t.challenge_wide("u", b->h_wide + 64 * (size_t)p);
            });
            int rc2 = acp_put_challenges(b, L.u + j, 1);
            if (rc2) return rc2;
            k_ipa_uinv<<<(B + 63) / 64, 64, 0, s>>>(L, B, j, b->d_blk);
            LAUNCH_CHECK(ctx);
            return BPP_OK;
        };
    if ((rc = ipa_prove_rounds(ctx, L, B, io, fb, host_u))) return rc;
    k_acp_pack_fixed<<<dim3((b->proof_len / 32 + 127) / 128, B), 128, 0, s>>>(L, b->d_pts8, b->d_lr, b->d_blk, b->d_proofs,
                                                                             b->proof_len);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}

// Prover: witness resident -> proofs resident (b->d_proofs).  Steps and labels follow lib.rs:219-228.
extern "C" int bpp_acp_batch_prove(bpp_acp_batch *b) {
    if (!b) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    const acp_layout &L = b->lay;
    const uint32_t B = b->B, n = L.n;
    cudaStream_t s = ctx->stream;
    int rc;
    const bool bind_V = b->mode != 0;   // `reference` mode: the reference never appends V (SURVEY A.3 defect 12)
    if (bind_V && !b->have_V) {
        ctx->last_error = "prove: the value commitments are not resident (bpp_acp_batch_commit / _upload_commitments)";
        return BPP_ERR_INVALID_ARG;
    }
    if (bind_V && !b->host_transcripts && (rc = acp_fork_vchunks(b))) return rc;   // beside the commitment MSMs
    // create(): randomness alpha,beta,ro,s_l,s_r (+ the five tau drawn later from the same stream)
    acp_mark(b, "start");
    const uint32_t nrand = 3 + 2 * n + 5;
    k_acp_rng<<<dim3((nrand + 127) / 128, B), 128, 0, s>>>(b->d_seeds, L, nrand, b->d_blk);
    LAUNCH_CHECK(ctx);
    {   // A_I = alpha*h + <a_L,G> + <a_R,H>; A_O = beta*h + <a_O,G>; S = ro*h + <s_l,G> + <s_r,H>
        // small batches (split launches that do not fill the GPU for long): the three commitments side by side on
        // three streams, each with its own part of the split scratch
        const bool side = b->fb_splits > 1 && !b->priority_split && b->aux3;
        if (side) {
            CK(ctx, cudaEventRecord(b->ev_fork, s));
            CK(ctx, cudaStreamWaitEvent(b->aux, b->ev_fork, 0));
            CK(ctx, cudaStreamWaitEvent(b->aux3, b->ev_fork, 0));
        }
        const bpp_points &P = *b->gens->pts;
        const bool structured = b->shuffle_wit && b->hsum && b->hsum->fb_c == P.fb_c && acp_ai_structured_ok(b);
        fb_sparse sp{};
        fb_shape sh = acp_ai_shape(b, structured, &sp);
        if ((rc = acp_fb(b, sh, b->d_ext8 + 0, 8, nullptr, 0, nullptr, sp))) return rc;
        const uint32_t gH = 2 + b->gens->n;   // first H generator (gens order g, h, G[..], H[..])
        sh = acp_shape(1);
        acp_seg(sh, L.beta, 0, 1, 1); acp_seg(sh, L.aO, 0, 2, n);
        if ((rc = acp_fb(b, sh, b->d_ext8 + 32, 8, side ? b->aux : nullptr, side ? 1 : 0))) return rc;
        sh = acp_shape(1);
        acp_seg(sh, L.ro, 0, 1, 1); acp_seg(sh, L.sl, 0, 2, n); acp_seg(sh, L.sr, 0, gH, n);
        if ((rc = acp_fb(b, sh, b->d_ext8 + 64, 8, side ? b->aux3 : nullptr, side ? 2 : 0))) return rc;
        if (side) {
            CK(ctx, cudaEventRecord(b->ev_join, b->aux));
            CK(ctx, cudaEventRecord(b->ev_join3, b->aux3));
            CK(ctx, cudaStreamWaitEvent(s, b->ev_join, 0));
            CK(ctx, cudaStreamWaitEvent(s, b->ev_join3, 0));
        }
    }
    acp_mark(b, "rng+A_I,A_O,S");
    k_compress_strided<<<(B * 3 + 127) / 128, 128, 0, s>>>(b->d_ext8, 8, 0, 3, B, b->d_pts8);
    LAUNCH_CHECK(ctx);
    acp_mark(b, "compress");
    // transcripts: dom-sep, A_I, A_O, S -> y, z
    if (!b->host_transcripts) {
        if (bind_V) CK(ctx, cudaStreamWaitEvent(s, b->ev_join2, 0));
        TR_LAUNCH(k_tr_prove_yz, B, s, b->d_proto, bind_V ? b->d_vdig : nullptr, b->d_pts8, L, B, b->d_tr, b->d_blk);
        LAUNCH_CHECK(ctx);
    } else {
        CK(ctx, cudaMemcpyAsync(b->h_pts8, b->d_pts8, (size_t)B * 256, cudaMemcpyDeviceToHost, s));
        if (bind_V && (rc = acp_fetch_commitments(b))) return rc;
        CK(ctx, cudaStreamSynchronize(s));
        {   // Transcript::new(label) + arithmetic_domain_sep(n) are identical for every proof: hash once, copy
            bpp_host::Transcript proto(b->label.data(), b->label.size());
            proto.arithmetic_domain_sep(n);
            b->tr.assign(B, proto);
        }
        acp_parallel_for(B, [&](uint32_t p) {
            bpp_host::Transcript &t = b->tr[p];
            const uint8_t *pt = b->h_pts8 + 256 * (size_t)p;
            if (bind_V) acp_host_append_commitments(t, b->h_V + 32 * (size_t)p * L.m, L.m);
            t.append_point("A_I", pt);
            t.append_point("A_O", pt + 32);
            t.append_point("S", pt + 64);
            t.challenge_wide("y", b->h_wide + 128 * (size_t)p);
            t.challenge_wide("z", b->h_wide + 128 * (size_t)p + 64);
        });
        if ((rc = acp_put_challenges(b, L.y, 2))) return rc;
    }
    acp_mark(b, "y,z");
    if ((rc = acp_challenge_dependent_scalars(b))) return rc;
    acp_mark(b, "scalars");
    acp_dots_launch(L, 0, 10, B, b->d_blk, s);
    LAUNCH_CHECK(ctx);
    k_acp_tcoef<<<(B + 63) / 64, 64, 0, s>>>(L, B, b->mode, b->d_blk);
    LAUNCH_CHECK(ctx);
    acp_mark(b, "dots");
    {   // T_i = t_i*g + tau_i*h for i in (1,3,4,5,6)
        fb_shape sh = acp_shape(5);
        acp_seg(sh, L.tsel, 1, 0, 1); acp_seg(sh, L.tau, 1, 1, 1);
        if ((rc = acp_fb(b, sh, b->d_ext8 + 96, 8))) return rc;
    }
    k_compress_strided<<<(B * 5 + 127) / 128, 128, 0, s>>>(b->d_ext8, 8, 3, 5, B, b->d_pts8);
    LAUNCH_CHECK(ctx);
    acp_mark(b, "T_i");
    const int mode = b->mode;
    if (!b->host_transcripts) {
        TR_LAUNCH(k_tr_prove_x, B, s, b->d_pts8, L, B, mode, b->d_tr, b->d_blk);
        LAUNCH_CHECK(ctx);
    } else {
        CK(ctx, cudaMemcpyAsync(b->h_pts8, b->d_pts8, (size_t)B * 256, cudaMemcpyDeviceToHost, s));
        CK(ctx, cudaStreamSynchronize(s));
        acp_parallel_for(B, [&](uint32_t p) {
            bpp_host::Transcript &t = b->tr[p];
            const uint8_t *pt = b->h_pts8 + 256 * (size_t)p + 96;
            t.append_point("T1", pt);
            t.append_point("T3", pt + 32);
            t.append_point("T4", mode == 0 ? pt + 32 : pt + 64);  // circuit_lib.rs:391 appends T_3 under "T4"
            t.append_point("T5", pt + 96);
            t.append_point("T6", pt + 128);
            t.challenge_wide("x", b->h_wide + 64 * (size_t)p);
        });
        if ((rc = acp_put_challenges(b, L.x, 1))) return rc;
    }
    acp_mark(b, "x");
    k_acp_final<<<dim3((L.np + 127) / 128, B), 128, 0, s>>>(L, b->d_blk);
    LAUNCH_CHECK(ctx);
    acp_dots_launch(L, 10, 2, B, b->d_blk, s);
    LAUNCH_CHECK(ctx);
    k_acp_final2<<<(B + 63) / 64, 64, 0, s>>>(L, B, b->mode, b->d_blk);
    LAUNCH_CHECK(ctx);
    acp_mark(b, "l,r,t,tau_x,mu");
    if (b->mode == 2) {
        rc = acp_prove_ipa(b);
        acp_mark(b, "inner-product rounds");
        acp_marks_dump(b, "prove");
        return rc;
    }
    k_acp_pack<<<dim3((b->proof_len / 32 + 127) / 128, B), 128, 0, s>>>(L, B, b->d_pts8, b->d_blk, b->d_proofs, b->proof_len);
    LAUNCH_CHECK(ctx);
    acp_mark(b, "pack");
    acp_marks_dump(b, "prove");
    return BPP_OK;
}

extern "C" int bpp_acp_batch_download_proofs(bpp_acp_batch *b, uint8_t *proofs_out) {
    if (!b || !proofs_out) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaMemcpyAsync(proofs_out, b->d_proofs, (size_t)b->B * b->proof_len, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return BPP_OK;
}

// proofs (count x proof_len) and commitments V (count x m x 32, compressed); V may be NULL to keep the
// resident commitments of bpp_acp_batch_commit
extern "C" int bpp_acp_batch_upload_proofs(bpp_acp_batch *b, const uint8_t *proofs, const uint8_t *V) {
    if (!b || !proofs) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(b->d_proofs, proofs, (size_t)b->B * b->proof_len, cudaMemcpyHostToDevice, ctx->stream));
    if (V) {
        CK(ctx, cudaMemcpyAsync(b->d_V, V, (size_t)b->B * b->lay.m * 32, cudaMemcpyHostToDevice, ctx->stream));
        b->have_V = true;
    }
    return BPP_OK;
}

// One MSM over the batch (see k_rlc_weights).  *decided = true when every proof's accept byte is final.
static int acp_verify_rlc(bpp_acp_batch *b, uint32_t per, int check_t, bool *decided) {
    bpp_ctx *ctx = b->ctx;
    const acp_layout &L = b->lay;
    const uint32_t B = b->B, nstat = b->gens->n_gens;
    cudaStream_t s = ctx->stream;
    *decided = false;
    const size_t N = (size_t)B * per + nstat;
    k_rlc_weights<<<(B + 127) / 128, 128, 0, s>>>(L, B, check_t, b->d_bad, b->d_blk);
    LAUNCH_CHECK(ctx);
    k_rlc_dyn_scalars<<<dim3((per + 127) / 128, B), 128, 0, s>>>(L, per, B, L.rho, b->d_blk, b->d_rlc_sc);
    LAUNCH_CHECK(ctx);
    k_rlc_stat_scalars<<<nstat, 128, 0, s>>>(L, rlc_segs{{L.vg, 0, 0}, {nstat, 0, 0}}, B, L.rho, b->d_blk, b->d_rlc_sc + 8 * (size_t)B * per);
    LAUNCH_CHECK(ctx);
    bpp_points view;
    view.niels = b->d_dyn;
    view.n = N;
    acp_mark(b, "rlc-scalars");
    // One window group: shaped for throughput, not for the latency of one call.  With several batches in flight the short
    // dependent kernels of one batch hide behind the GPU-filling kernels of another, so what counts is the SM time the
    // MSM takes: one sort, one accumulate grid without a partial wave per group, one merge + Horner chain.  Against the
    // four groups pick_partition gives 4096 x 113 + 210 points: 612 K -> 695 K proofs/s in the 52-card step with six
    // batches in flight, B200 at 1000 W (DESIGN.md section 3.2).
    int rc = msm_enqueue(ctx, b->d_rlc_sc, &view, 0, N, b->d_rlc_out, 1, true, 1);
    view.niels = nullptr;
    if (rc) return rc;
    acp_mark(b, "rlc-msm");
    k_rlc_accept<<<(B + 127) / 128, 128, 0, s>>>(b->d_rlc_out, L, B, L.rho, b->d_blk, b->d_accept, b->d_rlc_flag);
    LAUNCH_CHECK(ctx);
    CK(ctx, cudaMemcpyAsync(b->h_rlc_flag, b->d_rlc_flag, 4, cudaMemcpyDeviceToHost, s));
    acp_mark(b, "accept");
    CK(ctx, cudaStreamSynchronize(s));
    acp_marks_dump(b, "verify");
    *decided = b->h_rlc_flag[0] == 0;
    return BPP_OK;
}

// `fixed` mode verifier (bulletproofs 4.0.0 verification_scalars + the mega-check of dalek's R1CS verifier): replays the transcript including the inner-product rounds,
// then evaluates rho * check 2 + check 3 with the inner-product verification substituted for <l,G> + <r,h'>
// as ONE MSM per proof (2 n' + 2 fixed-base terms, m + 8 + 2 lg decompressed points) that must be the identity.
static int acp_verify_fixed(bpp_acp_batch *b, const uint8_t *verifier_seed) {
    bpp_ctx *ctx = b->ctx;
    const acp_layout &L = b->lay;
    const uint32_t B = b->B, n = L.n, np = L.np, m = L.m, lg = L.lg, per = m + 8 + 2 * lg, nch = 4 + lg;
    cudaStream_t s = ctx->stream;
    int rc;
    uint8_t seed[32];
    k_acp_unpack_fixed<<<dim3((b->proof_len / 32 + 127) / 128, B), 128, 0, s>>>(L, b->d_proofs, b->proof_len, b->d_blk, b->d_pts8,
                                                                               b->d_lr, b->d_tx3);
    LAUNCH_CHECK(ctx);
    // point decompression (IMAD-bound, fills the GPU) on `aux`, beside the dependent chain.  decompress_late: forked
    // only after the transcript replay - the few warps of the hashing kernels otherwise share every SM with it and take
    // three times as long (stage timeline, DESIGN.md section 3.2)
    auto fork_decompress = [&]() -> int {
        CK(ctx, cudaEventRecord(b->ev_fork, s));
        CK(ctx, cudaStreamWaitEvent(b->aux, b->ev_fork, 0));
        CK(ctx, cudaMemsetAsync(b->d_bad, 0, (size_t)B * 4, b->aux));
        k_acp_decompress<<<(B * (m + 8) + 127) / 128, 128, 0, b->aux>>>(b->d_V, b->d_pts8, m, B, per, b->d_dyn, b->d_bad);
        LAUNCH_CHECK(ctx);
        k_acp_decompress_lr<<<(B * 2 * lg + 127) / 128, 128, 0, b->aux>>>(b->d_lr, 2 * lg, 2 * lg, m + 8, per, B, b->d_dyn, b->d_bad);
        LAUNCH_CHECK(ctx);
        CK(ctx, cudaEventRecord(b->ev_join, b->aux));
        return BPP_OK;
    };
    const bool late = b->decompress_late && !b->host_transcripts;
    if (!late && (rc = fork_decompress())) return rc;
    if ((rc = acp_set_verifier_seed(b, verifier_seed, seed))) return rc;
    if (!b->host_transcripts) {
        if ((rc = acp_fork_vchunks(b))) return rc;
        CK(ctx, cudaStreamWaitEvent(s, b->ev_join2, 0));
        TR_LAUNCH(k_tr_verify, B, s, b->d_proto, b->d_vdig, b->d_pts8, (const uint8_t *)b->d_tx3, b->d_lr, L, B, 2,
                                                        b->d_blk, b->d_tr);
        LAUNCH_CHECK(ctx);
        if (late && (rc = fork_decompress())) return rc;
        if ((rc = acp_fork_weights(b))) return rc;
    } else {
        CK(ctx, cudaMemcpyAsync(b->h_pts8, b->d_pts8, (size_t)B * 256, cudaMemcpyDeviceToHost, s));
        CK(ctx, cudaMemcpyAsync(b->h_tx3, b->d_tx3, (size_t)B * 96, cudaMemcpyDeviceToHost, s));
        CK(ctx, cudaMemcpyAsync(b->h_lr, b->d_lr, (size_t)B * 64 * lg, cudaMemcpyDeviceToHost, s));
        CK(ctx, cudaMemcpyAsync(b->h_proofs, b->d_proofs, (size_t)B * b->proof_len, cudaMemcpyDeviceToHost, s));
        if ((rc = acp_fetch_commitments(b))) return rc;
        CK(ctx, cudaStreamSynchronize(s));
        bpp_host::Transcript proto(b->label.data(), b->label.size());
        proto.arithmetic_domain_sep(n);
        const size_t w_off = (size_t)B * nch * 64;   // the two weights follow the challenges in h_wide
        acp_parallel_for(B, [&](uint32_t p) {
            bpp_host::Transcript t = proto;
            const uint8_t *pt = b->h_pts8 + 256 * (size_t)p, *sc3 = b->h_tx3 + 96 * (size_t)p, *lr = b->h_lr + 64 * (size_t)lg * p;
            uint8_t *wide = b->h_wide + 64 * (size_t)nch * p;
            acp_host_append_commitments(t, b->h_V + 32 * (size_t)p * m, m);
            t.append_point("A_I", pt);
            t.append_point("A_O", pt + 32);
            t.append_point("S", pt + 64);
            t.challenge_wide("y", wide);
            t.challenge_wide("z", wide + 64);
            t.append_point("T1", pt + 96);
            t.append_point("T3", pt + 128);
            t.append_point("T4", pt + 160);
            t.append_point("T5", pt + 192);
            t.append_point("T6", pt + 224);
            t.challenge_wide("x", wide + 128);
            t.append_scalar("t_x", sc3);
            t.append_scalar("t_x_blinding", sc3 + 32);
            t.append_scalar("e_blinding", sc3 + 64);
            t.challenge_wide("w", wide + 192);
            t.append_message("dom-sep", (const uint8_t *)"ipp v1", 6);
            t.append_u64("n", np);
            for (uint32_t j = 0; j < lg; j++) {   // an identity encoding is rejected on the device (k_acp_decompress_lr)
                t.append_point("L", lr + 64 * (size_t)j);
                t.append_point("R", lr + 64 * (size_t)j + 32);
                t.challenge_wide("u", wide + 256 + 64 * (size_t)j);
            }
            acp_host_weights(t, b->h_proofs + (size_t)p * b->proof_len, b->proof_len, seed, p, 2, b->h_wide + w_off + 128 * (size_t)p);
        });
        // challenges land at y, z, x, wq and u_j; the verifier weights at w, rho0
        CK(ctx, cudaMemcpyAsync(b->d_wide, b->h_wide, (size_t)B * nch * 64, cudaMemcpyHostToDevice, s));
        k_acp_put_wide_strided<<<(B * nch + 127) / 128, 128, 0, s>>>(b->d_wide, L, nch, B, b->d_blk);
        LAUNCH_CHECK(ctx);
        if ((rc = acp_put_challenges(b, L.w, 2, w_off))) return rc;
    }
    if ((rc = acp_challenge_dependent_scalars(b))) return rc;
    acp_dots_launch(L, 9, 1, B, b->d_blk, s);   // sigma
    LAUNCH_CHECK(ctx);
    k_ipa_vprep<<<(B + 63) / 64, 64, 0, s>>>(L, B, m + 8, b->d_blk);
    LAUNCH_CHECK(ctx);
    k_ipa_stable_full<<<B, np >= IPA_ROUND_THREADS ? IPA_ROUND_THREADS : (np < 128 ? 128 : np), 0, s>>>(L, b->d_blk);
    LAUNCH_CHECK(ctx);
    if (!b->host_transcripts) CK(ctx, cudaStreamWaitEvent(s, b->ev_join2, 0));   // w, rho0 (k_tr_weights)
    k_acp_vscal_fixed<<<dim3((np + m + 1 + 127) / 128, B), 128, 0, s>>>(L, b->d_blk);
    LAUNCH_CHECK(ctx);
    CK(ctx, cudaStreamWaitEvent(s, b->ev_join, 0));   // decompressed points + bad flags (forked after the unpack)
    if (b->batch_rlc && (size_t)B * per >= 1024) {   // enough points for the bucket method to pay
        bool decided = false;
        if ((rc = acp_verify_rlc(b, per, 0, &decided))) return rc;
        if (decided) return BPP_OK;
    }
    {
        fb_shape sh = acp_shape(1);
        acp_seg(sh, L.vg, 0, 0, 2 * np + 2);
        if ((rc = acp_fb(b, sh, b->d_stat, 1))) return rc;
    }
    k_dyn_window_sums<<<B, DYN_W, 0, s>>>(b->d_blk, L, b->d_dyn, per, b->d_wsum);
    LAUNCH_CHECK(ctx);
    k_dyn_horner_accept<<<(B + 63) / 64, 64, 0, s>>>(L, B, b->d_blk, b->d_wsum, b->d_stat, b->d_bad, 0, b->d_accept);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}

// Verifier: proofs + V resident -> accept bytes resident.  Replays the transcript (A_I,A_O,S -> y,z;
// T's -> x), recomputes the challenge-dependent scalars and evaluates the checks of
// circuit_lib.rs:518 (t == <l,r>), :541 and (mode 1) :577-582 as one MSM per proof.
extern "C" int bpp_acp_batch_verify(bpp_acp_batch *b, const uint8_t *verifier_seed) {
    if (!b) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    if (!b->have_V) {
        ctx->last_error = "verify: the value commitments are not resident (bpp_acp_batch_upload_proofs with V / _upload_commitments)";
        return BPP_ERR_INVALID_ARG;
    }
    if (b->mode == 2) return acp_verify_fixed(b, verifier_seed);
    const acp_layout &L = b->lay;
    const uint32_t B = b->B, n = L.n, m = L.m, per = m + 8;
    cudaStream_t s = ctx->stream;
    int rc;
    uint8_t seed[32];
    acp_mark(b, "start");
    k_acp_unpack<<<dim3((b->proof_len / 32 + 127) / 128, B), 128, 0, s>>>(L, B, b->d_proofs, b->proof_len, b->d_blk, b->d_pts8);
    LAUNCH_CHECK(ctx);
    auto fork_decompress = [&]() -> int {   // see acp_verify_fixed
        CK(ctx, cudaEventRecord(b->ev_fork, s));
        CK(ctx, cudaStreamWaitEvent(b->aux, b->ev_fork, 0));
        CK(ctx, cudaMemsetAsync(b->d_bad, 0, (size_t)B * 4, b->aux));
        k_acp_decompress<<<(B * per + 127) / 128, 128, 0, b->aux>>>(b->d_V, b->d_pts8, m, B, per, b->d_dyn, b->d_bad);
        LAUNCH_CHECK(ctx);
        CK(ctx, cudaEventRecord(b->ev_join, b->aux));
        return BPP_OK;
    };
    const bool late = b->decompress_late && !b->host_transcripts;
    if (!late && (rc = fork_decompress())) return rc;
    if ((rc = acp_set_verifier_seed(b, verifier_seed, seed))) return rc;
    const int mode = b->mode;
    if (!b->host_transcripts) {
        if (mode != 0) {
            if ((rc = acp_fork_vchunks(b))) return rc;
            CK(ctx, cudaStreamWaitEvent(s, b->ev_join2, 0));
        }
        TR_LAUNCH(k_tr_verify, B, s, b->d_proto, b->d_vdig, b->d_pts8, nullptr, nullptr, L, B, mode, b->d_blk, b->d_tr);
        LAUNCH_CHECK(ctx);
        if (late && (rc = fork_decompress())) return rc;
        if ((rc = acp_fork_weights(b))) return rc;
    } else {
        CK(ctx, cudaMemcpyAsync(b->h_pts8, b->d_pts8, (size_t)B * 256, cudaMemcpyDeviceToHost, s));
        CK(ctx, cudaMemcpyAsync(b->h_proofs, b->d_proofs, (size_t)B * b->proof_len, cudaMemcpyDeviceToHost, s));
        if (mode != 0 && (rc = acp_fetch_commitments(b))) return rc;
        CK(ctx, cudaStreamSynchronize(s));
        bpp_host::Transcript proto(b->label.data(), b->label.size());
        proto.arithmetic_domain_sep(n);
        acp_parallel_for(B, [&](uint32_t p) {
            bpp_host::Transcript t = proto;
            const uint8_t *pt = b->h_pts8 + 256 * (size_t)p;
            uint8_t *wide = b->h_wide + 320 * (size_t)p;   // y, z, x, w, rho0
            if (mode != 0) acp_host_append_commitments(t, b->h_V + 32 * (size_t)p * m, m);
            t.append_point("A_I", pt);
            t.append_point("A_O", pt + 32);
            t.append_point("S", pt + 64);
            t.challenge_wide("y", wide);
            t.challenge_wide("z", wide + 64);
            t.append_point("T1", pt + 96);
            t.append_point("T3", pt + 128);
            t.append_point("T4", mode == 0 ? pt + 128 : pt + 160);
            t.append_point("T5", pt + 192);
            t.append_point("T6", pt + 224);
            t.challenge_wide("x", wide + 128);
            acp_host_weights(t, b->h_proofs + (size_t)p * b->proof_len, b->proof_len, seed, p, mode, wide + 192);
        });
        if ((rc = acp_put_challenges(b, L.y, 5))) return rc;
    }
    acp_mark(b, "transcript");
    if ((rc = acp_challenge_dependent_scalars(b))) return rc;
    acp_dots_launch(L, 9, 2, B, b->d_blk, s);  // sigma, <l, r>
    LAUNCH_CHECK(ctx);
    acp_mark(b, "scalars");
    if (!b->host_transcripts) CK(ctx, cudaStreamWaitEvent(s, b->ev_join2, 0));   // w, rho0 (k_tr_weights)
    acp_mark(b, "wait-weights");
    k_acp_vscal<<<dim3((n + m + 1 + 127) / 128, B), 128, 0, s>>>(L, b->d_blk);
    LAUNCH_CHECK(ctx);
    acp_mark(b, "vscal");
    CK(ctx, cudaStreamWaitEvent(s, b->ev_join, 0));   // decompressed points + bad flags (forked after the unpack)
    acp_mark(b, "wait-decompress");
    if (b->batch_rlc && mode != 0 && (size_t)B * per >= 1024) {   // `reference` mode never accepts: nothing to gain from the combined check
        bool decided = false;
        if ((rc = acp_verify_rlc(b, per, 1, &decided))) return rc;
        if (decided) return BPP_OK;
    }
    {
        fb_shape sh = acp_shape(1);
        acp_seg(sh, L.vg, 0, 0, 2 * n + 2);
        if ((rc = acp_fb(b, sh, b->d_stat, 1))) return rc;
    }
    k_dyn_window_sums<<<B, DYN_W, 0, s>>>(b->d_blk, L, b->d_dyn, per, b->d_wsum);
    LAUNCH_CHECK(ctx);
    k_dyn_horner_accept<<<(B + 63) / 64, 64, 0, s>>>(L, B, b->d_blk, b->d_wsum, b->d_stat, b->d_bad, 1, b->d_accept);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}

extern "C" int bpp_acp_batch_download_accept(bpp_acp_batch *b, uint8_t *accept) {
    if (!b || !accept) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaMemcpyAsync(accept, b->d_accept, b->B, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return BPP_OK;
}

// Measurement hook: the commitment-shaped fixed-base MSM (A_I: 1 + 2n terms per proof) alone, `reps`
// launches between CUDA events on the context's stream.  madds = point adds per launch by SURVEY 8(d)'s
// accounting (terms x windows mixed adds + the block tree reduction's full adds).
extern "C" int bpp_acp_batch_time_commit_msm(bpp_acp_batch *b, int reps, float *ms_avg, uint64_t *mixed_adds,
                                             uint64_t *full_adds) {
    if (!b || reps <= 0 || !ms_avg) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    const acp_layout &L = b->lay;
    const fb_shape sh = acp_ai_shape(b, false);   // the generic A_I shape whatever the witness
    int rc = acp_fb(b, sh, b->d_ext8, 8);  // warm-up
    if (rc) return rc;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, ctx->stream);
    for (int i = 0; i < reps; i++)
        if ((rc = acp_fb(b, sh, b->d_ext8, 8))) return rc;
    cudaEventRecord(e1, ctx->stream);
    CK(ctx, cudaEventSynchronize(e1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ms_avg = ms / reps;
    if (mixed_adds) *mixed_adds = (uint64_t)b->B * (1 + 2 * L.n) * b->gens->pts->fb_Wn;
    if (full_adds) *full_adds = (uint64_t)b->B * (acp_fb_plan(b, sh).form == FB_WARP ? 31 : FB_THREADS - 1);
    return BPP_OK;
}

// K7 as an operator (measurement + parity; see k_ipa_fold_gens): `folds` independent foldings of points[off..off+n)
// with (u_f, u_f^-1): out[f][i] = u_f^-1 P_i + u_f P_{i + n/2}.  out_enc (host, folds x n/2 x 32, nullable): compressed
// results; ms (nullable): device time of the folding kernel alone (CUDA events).
extern "C" int bpp_ipa_fold_generators(bpp_ctx *ctx, const bpp_points *points, size_t off, size_t n, const uint8_t *u,
                                       const uint8_t *uinv, size_t folds, uint8_t *out_enc, float *ms) {
    if (!ctx || !points || !u || !uinv || n < 2 || (n & 1) || folds == 0) return BPP_ERR_INVALID_ARG;
    if (off + n > points->n) return BPP_ERR_LENGTH_MISMATCH;
    for (size_t i = 0; i < folds; i++)
        if ((u[32 * i + 31] | uinv[32 * i + 31]) & 0xe0) return BPP_ERR_SCALAR_RANGE;   // reduced scalars (< 2^253)
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t half = n / 2, outs = folds * half;
    if (outs >= (1ull << 31)) return BPP_ERR_INVALID_ARG;
    int rc;
    if ((rc = grow(ctx, &ctx->d_small, &ctx->cap_small, folds * 64 + outs * 128 + outs * 32))) return rc;
    uint8_t *d_u = ctx->d_small, *d_ui = d_u + folds * 32, *d_ext = d_ui + folds * 32, *d_enc = d_ext + outs * 128;
    CK(ctx, cudaMemcpyAsync(d_u, u, folds * 32, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaMemcpyAsync(d_ui, uinv, folds * 32, cudaMemcpyHostToDevice, ctx->stream));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, ctx->stream);
    k_ipa_fold_gens<<<(unsigned)((outs + 63) / 64), 64, 0, ctx->stream>>>(points->niels + 24 * off, (uint32_t)half, (const uint32_t *)d_u,
                                                                         (const uint32_t *)d_ui, (uint32_t)folds, (uint32_t *)d_ext);
    cudaEventRecord(e1, ctx->stream);
    LAUNCH_CHECK(ctx);
    if (out_enc) {
        k_compress_strided<<<(unsigned)((outs + 127) / 128), 128, 0, ctx->stream>>>((const uint32_t *)d_ext, 1, 0, 1, (uint32_t)outs, d_enc);
        LAUNCH_CHECK(ctx);
        CK(ctx, cudaMemcpyAsync(out_enc, d_enc, outs * 32, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    if (ms) cudaEventElapsedTime(ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return BPP_OK;
}

// Sharded batch verification: this rank's `count` accept bytes, zero-padded to `per`, all-gathered over the context's
// communicator into accept_all (nranks x per, host); a single rank gets its own bytes.  Synchronises.
static int gather_accept(bpp_ctx *ctx, const uint8_t *d_accept, uint32_t count, size_t per, uint8_t *accept_all) {
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t nr = (size_t)ctx->comm_nranks;
    int rc;
    if ((rc = grow(ctx, &ctx->d_small, &ctx->cap_small, per * (nr + 1)))) return rc;
    uint8_t *mine = ctx->d_small, *all = ctx->d_small + per;
    CK(ctx, cudaMemsetAsync(mine, 0, per, ctx->stream));
    CK(ctx, cudaMemcpyAsync(mine, d_accept, count, cudaMemcpyDeviceToDevice, ctx->stream));
    if ((rc = comm_all_gather(ctx, mine, all, per, ctx->stream))) return rc;
    CK(ctx, cudaMemcpyAsync(accept_all, all, per * nr, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return BPP_OK;
}
extern "C" int bpp_acp_batch_gather_accept(bpp_acp_batch *b, size_t per, uint8_t *accept_all) {
    if (!b || !accept_all || per < b->B) return BPP_ERR_INVALID_ARG;
    return gather_accept(b->ctx, b->d_accept, b->B, per, accept_all);
}

// ---- one-call host forms (what a drop-in for create..blinding_values / verify binds) -------------------
extern "C" int bpp_acproof_prove_batch(bpp_ctx *ctx, const bpp_circuit *cir, const bpp_gens *gens, int mode, size_t count,
                                       const uint8_t *aL, const uint8_t *aR, const uint8_t *aO, const uint8_t *gamma,
                                       const uint8_t *seeds, const uint8_t *V, const uint8_t *label, size_t label_len,
                                       uint8_t *proofs_out) {
    if (mode != 0 && !V) return BPP_ERR_INVALID_ARG;   // modes 1 and 2 bind the commitments to the transcript
    bpp_acp_batch *b = nullptr;
    int rc = bpp_acp_batch_create(ctx, cir, gens, mode, count, label, label_len, &b);
    if (rc) return rc;
    rc = bpp_acp_batch_upload_witness(b, aL, aR, aO, gamma, seeds);
    if (!rc && V) rc = bpp_acp_batch_upload_commitments(b, V);
    if (!rc) rc = bpp_acp_batch_prove(b);
    if (!rc) rc = bpp_acp_batch_download_proofs(b, proofs_out);
    bpp_acp_batch_free(b);
    return rc;
}

extern "C" int bpp_acproof_verify_batch(bpp_ctx *ctx, const bpp_circuit *cir, const bpp_gens *gens, int mode, size_t count,
                                        const uint8_t *proofs, const uint8_t *V, const uint8_t *label, size_t label_len,
                                        const uint8_t *verifier_seed, uint8_t *accept) {
    if (!V) return BPP_ERR_INVALID_ARG;
    bpp_acp_batch *b = nullptr;
    int rc = bpp_acp_batch_create(ctx, cir, gens, mode, count, label, label_len, &b);
    if (rc) return rc;
    rc = bpp_acp_batch_upload_proofs(b, proofs, V);
    if (!rc) rc = bpp_acp_batch_verify(b, verifier_seed);
    if (!rc) rc = bpp_acp_batch_download_accept(b, accept);
    bpp_acp_batch_free(b);
    return rc;
}

// ---- scripted device transcript (test hook) -----------------------------------------------------------
extern "C" int bpp_transcript_script(bpp_ctx *ctx, const uint8_t *script, size_t len, uint8_t *out, size_t out_len) {
    if (!ctx || !script || len == 0 || len > (1u << 24) || (!out && out_len)) return BPP_ERR_INVALID_ARG;
    CK(ctx, cudaSetDevice(ctx->device));
    uint8_t *d = nullptr;
    CK(ctx, cudaMalloc((void **)&d, len + out_len + 64));
    cudaError_t e = cudaMemcpyAsync(d, script, len, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        k_tr_script<<<1, 32, 0, ctx->stream>>>(d, (uint32_t)len, d + len);
        ctx->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && out_len) e = cudaMemcpyAsync(out, d + len, out_len, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess) {
        ctx->last_error = cudaGetErrorString(e);
        return BPP_ERR_CUDA;
    }
    return BPP_OK;
}

// ---- transcript state across the C ABI (host only) ------------------------------------------------------------
// merlin::Transcript cannot be serialised, so a transcript crosses the ABI as BPP_TRANSCRIPT_BYTES: the 25 Keccak lanes
// and pos | pos_begin << 8 | cur_flags << 16, 26 little-endian u64 - host_merlin.hpp export_state, merlin_dev.cuh load.
static_assert(BPP_TRANSCRIPT_BYTES == 8 * MERLIN_STATE_WORDS, "transcript state layout");
static bool tr_state_ok(const uint8_t *state) {
    uint64_t w[MERLIN_STATE_WORDS];
    memcpy(w, state, sizeof(w));
    return bpp_host::Strobe128::state_valid(w);
}
extern "C" int bpp_transcript_new(const uint8_t *label, size_t label_len, uint8_t state[BPP_TRANSCRIPT_BYTES]) {
    if ((!label && label_len) || !state || label_len >= (1ull << 32)) return BPP_ERR_INVALID_ARG;
    bpp_host::Transcript t(label, label_len);
    uint64_t w[MERLIN_STATE_WORDS];
    t.export_state(w);
    memcpy(state, w, sizeof(w));
    return BPP_OK;
}
extern "C" int bpp_transcript_append_message(uint8_t state[BPP_TRANSCRIPT_BYTES], const uint8_t *label, size_t label_len,
                                             const uint8_t *msg, size_t msg_len) {
    if (!state || (!label && label_len) || (!msg && msg_len) || msg_len >= (1ull << 32)) return BPP_ERR_INVALID_ARG;
    if (!tr_state_ok(state)) return BPP_ERR_INVALID_ARG;
    uint64_t w[MERLIN_STATE_WORDS];
    memcpy(w, state, sizeof(w));
    bpp_host::Transcript t(w);
    t.append_message((const char *)label, label_len, msg, msg_len);
    t.export_state(w);
    memcpy(state, w, sizeof(w));
    return BPP_OK;
}
extern "C" int bpp_transcript_challenge_bytes(uint8_t state[BPP_TRANSCRIPT_BYTES], const uint8_t *label, size_t label_len,
                                              uint8_t *out, size_t out_len) {
    if (!state || (!label && label_len) || (!out && out_len) || out_len >= (1ull << 32)) return BPP_ERR_INVALID_ARG;
    if (!tr_state_ok(state)) return BPP_ERR_INVALID_ARG;
    uint64_t w[MERLIN_STATE_WORDS];
    memcpy(w, state, sizeof(w));
    bpp_host::Transcript t(w);
    t.challenge_bytes((const char *)label, label_len, out, out_len);
    t.export_state(w);
    memcpy(state, w, sizeof(w));
    return BPP_OK;
}

// ---- stand-alone inner-product argument, batched (bulletproofs 4.0.0 inner_product_proof.rs) -----------------------
// The prover runs the scalar-fold rounds of the `fixed` mode (ipa_prove_rounds) over a block holding only the
// inner-product fields (ipa_make_layout); the verifier evaluates dalek's verify as one MSM per proof: the 2 n + 1
// generator terms through the window table, the 2 lg n + 1 proof points through k_dyn_window_sums.  The combined form
// (bpp_ipa_batch_verify_combined) first runs one random-linear-combination MSM over the whole batch (ipa_verify_rlc).
struct bpp_ipa_batch {
    bpp_ctx *ctx = nullptr;
    bpp_points *gens = nullptr;
    uint32_t g_off = 0, h_off = 0, q_off = 0, n = 0, lg = 0, B = 0, fb_splits = 1;
    acp_layout lay;
    // d_dyn: B x (2 lg + 1) decompressed proof points; once the batch has run the combined check (ipa_rlc_alloc), followed
    // by the Niels forms of G, H and the Q base, so that it holds all of the combined MSM's points
    uint32_t *d_blk = nullptr, *d_lrext = nullptr, *d_part = nullptr, *d_stat = nullptr, *d_wsum = nullptr, *d_bad = nullptr,
             *d_dyn = nullptr;
    // combined verification: the verifier seed, the MSM's scalars (proof points, then generators), its compressed
    // result and the fall-back flag
    uint32_t *d_vseed = nullptr, *d_rlc_sc = nullptr, *d_rlc_flag = nullptr, *h_rlc_flag = nullptr;
    uint8_t *d_rlc_out = nullptr;
    uint8_t *d_in = nullptr;       // staged inputs: a | b | G factors | H factors (B x n x 32 each) | q (B x 32) | P (B x 32)
    uint8_t *d_lr = nullptr;       // B x (2 lg + 1) x 32: L_j, R_j (prover: the first 2 lg per proof, pitch 2 lg), then P
    uint8_t *d_proofs = nullptr, *d_accept = nullptr;
    uint64_t *d_tr = nullptr;
    // BPP_ACP_TRACE=1: stage timeline of prove / verify on the context's stream, printed to stderr (as bpp_acp_batch's)
    bool trace = false;
    std::vector<std::pair<const char *, cudaEvent_t>> marks;
};
static void ipa_mark(bpp_ipa_batch *b, const char *name) {
    if (!b->trace) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, b->ctx->stream);
    b->marks.emplace_back(name, e);
}
// after the call's synchronisation
static void ipa_marks_dump(bpp_ipa_batch *b, const char *what) {
    if (!b->trace || b->marks.empty()) return;
    fprintf(stderr, "[ipa trace] %s:", what);
    for (size_t i = 1; i < b->marks.size(); i++) {
        float ms = 0;
        cudaEventElapsedTime(&ms, b->marks[i - 1].second, b->marks[i].second);
        fprintf(stderr, " %s %.0f us |", b->marks[i].first, ms * 1e3f);
    }
    fprintf(stderr, "\n");
    for (auto &m : b->marks) cudaEventDestroy(m.second);
    b->marks.clear();
}

static acp_layout ipa_make_layout(uint32_t n) {
    acp_layout L;
    memset(&L, 0, sizeof(L));
    uint32_t o = 0;
    auto take = [&](uint32_t cnt) { uint32_t r = o; o += cnt; return r; };
    L.n = n; L.np = n; L.lg = acp_log2(n);
    L.l = take(n); L.r = take(n); L.yn = take(n); L.yninv = take(n); L.vG = take(n); L.vH = take(n);
    L.stab = take(2 * n);
    L.u = take(L.lg); L.uinv = take(L.lg); L.vd = take(2 * L.lg + 1);
    L.wq = take(1); L.cl = take(2); L.pa = take(1); L.pb = take(1);
    L.rho0 = take(1); L.rho = take(1);
    L.stride = (o + 3) & ~3u;
    return L;
}

extern "C" size_t bpp_ipa_proof_len(size_t n) {
    if (n == 0 || (n & (n - 1))) return 0;
    size_t lg = 0;
    while (((size_t)1 << lg) < n) lg++;
    return 32 * (2 * lg + 2);
}

extern "C" void bpp_ipa_batch_free(bpp_ipa_batch *b) {
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(b->ctx->stream);
    void *dev[] = {b->d_blk, b->d_lrext, b->d_part, b->d_stat, b->d_wsum, b->d_bad, b->d_dyn, b->d_in, b->d_lr, b->d_proofs,
                   b->d_accept, b->d_tr, b->d_vseed, b->d_rlc_sc, b->d_rlc_flag, b->d_rlc_out};
    for (void *p : dev)
        if (p) cudaFree(p);
    if (b->h_rlc_flag) cudaFreeHost(b->h_rlc_flag);
    for (auto &m : b->marks) cudaEventDestroy(m.second);
    delete b;
}

#define IPA_MAX_N 8192   // the large deck's n' (4096 cards): the largest shape the tables and tests cover
extern "C" int bpp_ipa_batch_create(bpp_ctx *ctx, bpp_points *gens, size_t g_off, size_t h_off, size_t q_off, size_t n, size_t count,
                                    bpp_ipa_batch **out) {
    if (!ctx || !gens || !out || count == 0 || count > (1u << 24) || n == 0 || n > IPA_MAX_N || (n & (n - 1)))
        return BPP_ERR_INVALID_ARG;
    *out = nullptr;
    if (g_off > gens->n || n > gens->n - g_off || h_off > gens->n || n > gens->n - h_off || q_off >= gens->n)
        return BPP_ERR_LENGTH_MISMATCH;
    CK(ctx, cudaSetDevice(ctx->device));
    bpp_ipa_batch *b = new bpp_ipa_batch();
    b->ctx = ctx; b->gens = gens;
    b->g_off = (uint32_t)g_off; b->h_off = (uint32_t)h_off; b->q_off = (uint32_t)q_off;
    b->n = (uint32_t)n; b->B = (uint32_t)count;
    b->lay = ipa_make_layout(b->n);
    b->lg = b->lay.lg;
    if (const char *e = getenv("BPP_ACP_TRACE")) b->trace = e[0] == '1';
    const size_t B = count, lg = b->lg;
    b->fb_splits = fb_split_count(ctx, B, (2 * (uint64_t)n + 2) * 8);   // as bpp_acp_batch_create sizes its scratch
    cudaError_t e = cudaMalloc((void **)&b->d_blk, B * b->lay.stride * 32);
    if (e == cudaSuccess) e = cudaMemsetAsync(b->d_blk, 0, B * b->lay.stride * 32, ctx->stream);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_in, B * (4 * n + 2) * 32);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_lr, B * (2 * lg + 1) * 32);
    if (e == cudaSuccess && lg) e = cudaMalloc((void **)&b->d_lrext, B * 2 * lg * 128);
    if (e == cudaSuccess && b->fb_splits > 1) e = cudaMalloc((void **)&b->d_part, B * 2 * b->fb_splits * 128);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_stat, B * 128);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_wsum, B * DYN_W * 128);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_bad, B * 4);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_dyn, B * (2 * lg + 1) * 96);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_proofs, B * bpp_ipa_proof_len(n));
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_accept, B);
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->d_tr, B * BPP_TRANSCRIPT_BYTES);
    if (e != cudaSuccess) {
        ctx->last_error = cudaGetErrorString(e);
        bool oom = e == cudaErrorMemoryAllocation;
        cudaGetLastError();
        bpp_ipa_batch_free(b);
        return oom ? BPP_ERR_OOM : BPP_ERR_CUDA;
    }
    *out = b;
    return BPP_OK;
}

// canonical (< l) scalars; nearly every one is decided by its top byte
static bool ipa_all_canonical(const uint8_t *s, size_t cnt) {
    for (size_t i = 0; i < cnt; i++)
        if (s[32 * i + 31] >= 0x10 && !acp_scalar_is_canonical(s + 32 * i)) return false;
    return true;
}
// the checks prove and verify share; 0 or the status to return
static int ipa_check_inputs(const bpp_ipa_batch *b, const uint8_t *q, const uint8_t *gf, const uint8_t *hf, const uint8_t *transcripts) {
    const size_t B = b->B, n = b->n;
    for (size_t p = 0; p < B; p++)
        if (!tr_state_ok(transcripts + BPP_TRANSCRIPT_BYTES * p)) return BPP_ERR_INVALID_ARG;
    if ((q && !ipa_all_canonical(q, B)) || (gf && !ipa_all_canonical(gf, B * n)) || (hf && !ipa_all_canonical(hf, B * n)))
        return BPP_ERR_SCALAR_RANGE;
    return BPP_OK;
}
// uploads q and the factors (NULL = ones) and the transcripts, places them in the proof blocks
static int ipa_upload_common(bpp_ipa_batch *b, const uint8_t *q, const uint8_t *gf, const uint8_t *hf, const uint8_t *transcripts,
                             const uint32_t *d_a, const uint32_t *d_b) {
    bpp_ctx *ctx = b->ctx;
    cudaStream_t s = ctx->stream;
    const size_t B = b->B, n = b->n, vec = B * n * 32;
    uint8_t *d_gf = b->d_in + 2 * vec, *d_hf = b->d_in + 3 * vec, *d_q = b->d_in + 4 * vec;
    if (gf) CK(ctx, cudaMemcpyAsync(d_gf, gf, vec, cudaMemcpyHostToDevice, s));
    if (hf) CK(ctx, cudaMemcpyAsync(d_hf, hf, vec, cudaMemcpyHostToDevice, s));
    if (q) CK(ctx, cudaMemcpyAsync(d_q, q, B * 32, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemcpyAsync(b->d_tr, transcripts, B * BPP_TRANSCRIPT_BYTES, cudaMemcpyHostToDevice, s));
    k_ipa_place<<<dim3((4 * b->n + 1 + 127) / 128, b->B), 128, 0, s>>>(d_a, d_b, gf ? (const uint32_t *)d_gf : nullptr,
                                                                     hf ? (const uint32_t *)d_hf : nullptr,
                                                                     q ? (const uint32_t *)d_q : nullptr, b->lay, b->d_blk);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}
static fb_plan ipa_fb_plan(const bpp_ipa_batch *b, const fb_shape &sh) {
    return fb_choose(b->ctx, (uint64_t)b->B * sh.outs, fb_terms(sh), b->gens->fb_Wn, !sh.sel_period, sh.outs > 8 ? 1 : b->fb_splits);
}

extern "C" int bpp_ipa_batch_prove(bpp_ipa_batch *b, const uint8_t *q, const uint8_t *G_factors, const uint8_t *H_factors,
                                   const uint8_t *a, const uint8_t *b_vec, uint8_t *transcripts, uint8_t *proofs_out) {
    if (!b || !a || !b_vec || !transcripts || !proofs_out) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    const size_t B = b->B, n = b->n, vec = B * n * 32;
    int rc;
    if ((rc = ipa_check_inputs(b, q, G_factors, H_factors, transcripts))) return rc;
    if (!ipa_all_canonical(a, B * n) || !ipa_all_canonical(b_vec, B * n)) return BPP_ERR_SCALAR_RANGE;
    CK(ctx, cudaSetDevice(ctx->device));
    if (!b->gens->fb_table && (rc = bpp_points_precompute(ctx, b->gens, 8))) return rc;
    cudaStream_t s = ctx->stream;
    const acp_layout &L = b->lay;
    ipa_mark(b, "start");
    CK(ctx, cudaMemcpyAsync(b->d_in, a, vec, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemcpyAsync(b->d_in + vec, b_vec, vec, cudaMemcpyHostToDevice, s));
    if ((rc = ipa_upload_common(b, q, G_factors, H_factors, transcripts, (const uint32_t *)b->d_in, (const uint32_t *)(b->d_in + vec))))
        return rc;
    ipa_mark(b, "upload");
    TR_LAUNCH(k_ipa_start, b->B, s, b->n, b->B, b->d_tr);
    LAUNCH_CHECK(ctx);
    ipa_mark(b, "dom-sep");
    if (b->lg) {
        ipa_rounds_io io;
        io.blk = b->d_blk; io.lr = b->d_lr; io.lrext = b->d_lrext; io.part = b->d_part; io.tr = b->d_tr;
        io.gG = b->g_off; io.gH = b->h_off; io.gQ = b->q_off;
        io.gf = true;
        auto fb = [&](const fb_shape &sh, uint32_t *dst, uint32_t pitch, uint32_t *split_n) {
            return fb_launch(ctx, b->d_blk, L, b->B, *b->gens, sh, ipa_fb_plan(b, sh), dst, pitch, s, b->d_part, split_n);
        };
        if ((rc = ipa_prove_rounds(ctx, L, b->B, io, fb, std::function<int(uint32_t)>()))) return rc;
    }
    ipa_mark(b, "inner-product rounds");
    const size_t plen = bpp_ipa_proof_len(n);
    k_ipa_pack<<<(unsigned)((B * (plen / 32) + 127) / 128), 128, 0, s>>>(L, b->d_lr, b->d_blk, b->B, b->d_proofs);
    LAUNCH_CHECK(ctx);
    CK(ctx, cudaMemcpyAsync(proofs_out, b->d_proofs, B * plen, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(transcripts, b->d_tr, B * BPP_TRANSCRIPT_BYTES, cudaMemcpyDeviceToHost, s));
    ipa_mark(b, "pack+download");
    CK(ctx, cudaStreamSynchronize(s));
    ipa_marks_dump(b, "prove");
    return BPP_OK;
}

// The combined check's buffers, on the batch's first combined verification (batches that only prove or only run the
// per-proof verify never pay for them): d_dyn grows by the Niels forms of G, H and the Q base, copied from the
// generators; the MSM's scalars, its result, the fall-back flag and the verifier seed.  d_rlc_sc is allocated last and
// marks the set complete.
static int ipa_rlc_alloc(bpp_ipa_batch *b) {
    if (b->d_rlc_sc) return BPP_OK;
    bpp_ctx *ctx = b->ctx;
    const size_t npts = (size_t)b->B * (2 * b->lg + 1), n = b->n, nstat = 2 * n + 1;
    const uint32_t *g = b->gens->niels;
    uint32_t *dyn = nullptr;
    CK(ctx, cudaMalloc((void **)&dyn, (npts + nstat) * 96));
    CK(ctx, cudaFree(b->d_dyn));
    b->d_dyn = dyn;
    CK(ctx, cudaMemcpyAsync(dyn + 24 * npts, g + 24 * (size_t)b->g_off, n * 96, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(ctx, cudaMemcpyAsync(dyn + 24 * (npts + n), g + 24 * (size_t)b->h_off, n * 96, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(ctx, cudaMemcpyAsync(dyn + 24 * (npts + 2 * n), g + 24 * (size_t)b->q_off, 96, cudaMemcpyDeviceToDevice, ctx->stream));
    if (!b->d_vseed) CK(ctx, cudaMalloc((void **)&b->d_vseed, 64));
    if (!b->d_rlc_flag) CK(ctx, cudaMalloc((void **)&b->d_rlc_flag, 64));
    if (!b->d_rlc_out) CK(ctx, cudaMalloc((void **)&b->d_rlc_out, 256));
    if (!b->h_rlc_flag) CK(ctx, cudaMallocHost((void **)&b->h_rlc_flag, 64));
    CK(ctx, cudaMalloc((void **)&b->d_rlc_sc, (npts + nstat) * 32));
    return BPP_OK;
}

// Below this many proof points the per-proof path is cheaper than the buckets (the shuffle verifier's rule)
#define IPA_RLC_MIN_POINTS 1024
static bool ipa_rlc_pays(const bpp_ipa_batch *b) { return (size_t)b->B * (2 * b->lg + 1) >= IPA_RLC_MIN_POINTS; }

// Verifier up to the per-proof scalars: argument checks, uploads, unpack, decompression, transcript replay, vprep, the
// s table and k_ipa_vscal.  The proofs stay staged at b->d_in.  rlc: the combined check follows (its buffers are made
// first, after the argument checks).
static int ipa_verify_scalars(bpp_ipa_batch *b, const uint8_t *q, const uint8_t *G_factors, const uint8_t *H_factors,
                              const uint8_t *P, const uint8_t *proofs, uint8_t *transcripts, uint8_t *accept, bool rlc) {
    if (!b || !P || !proofs || !transcripts || !accept) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    const size_t B = b->B, n = b->n, lg = b->lg, plen = bpp_ipa_proof_len(n), per = 2 * lg + 1;
    int rc;
    if ((rc = ipa_check_inputs(b, q, G_factors, H_factors, transcripts))) return rc;
    CK(ctx, cudaSetDevice(ctx->device));
    if (!b->gens->fb_table && (rc = bpp_points_precompute(ctx, b->gens, 8))) return rc;
    if (rlc && (rc = ipa_rlc_alloc(b))) return rc;
    cudaStream_t s = ctx->stream;
    const acp_layout &L = b->lay;
    ipa_mark(b, "start");
    // the proofs go where the prover stages a and b, P after q
    uint8_t *d_pr = b->d_in, *d_P = b->d_in + (4 * n + 1) * B * 32;
    CK(ctx, cudaMemcpyAsync(d_pr, proofs, B * plen, cudaMemcpyHostToDevice, s));
    CK(ctx, cudaMemcpyAsync(d_P, P, B * 32, cudaMemcpyHostToDevice, s));
    if ((rc = ipa_upload_common(b, q, G_factors, H_factors, transcripts, nullptr, nullptr))) return rc;
    CK(ctx, cudaMemsetAsync(b->d_bad, 0, B * 4, s));
    ipa_mark(b, "upload");
    k_ipa_unpack<<<(unsigned)((B * (plen / 32) + 127) / 128), 128, 0, s>>>(L, d_pr, d_P, b->B, b->d_blk, b->d_lr, b->d_bad);
    LAUNCH_CHECK(ctx);
    k_acp_decompress_lr<<<(unsigned)((B * per + 127) / 128), 128, 0, s>>>(b->d_lr, (uint32_t)per, 2 * b->lg, 0, (uint32_t)per, b->B,
                                                                         b->d_dyn, b->d_bad);
    LAUNCH_CHECK(ctx);
    TR_LAUNCH(k_ipa_vtranscript, b->B, s, b->d_lr, L, b->B, b->d_tr, b->d_blk);
    LAUNCH_CHECK(ctx);
    k_ipa_vprep<<<(b->B + 63) / 64, 64, 0, s>>>(L, b->B, 0, b->d_blk);
    LAUNCH_CHECK(ctx);
    k_ipa_stable_full<<<b->B, n >= IPA_ROUND_THREADS ? IPA_ROUND_THREADS : (n < 128 ? 128 : (unsigned)n), 0, s>>>(L, b->d_blk);
    LAUNCH_CHECK(ctx);
    k_ipa_vscal<<<dim3((b->n + 1 + 127) / 128, b->B), 128, 0, s>>>(L, b->d_blk);
    LAUNCH_CHECK(ctx);
    return BPP_OK;
}
// Every proof on its own: the generator terms through the window table, the proof points through k_dyn_window_sums.
static int ipa_verify_per_proof(bpp_ipa_batch *b) {
    bpp_ctx *ctx = b->ctx;
    cudaStream_t s = ctx->stream;
    const acp_layout &L = b->lay;
    int rc;
    {
        fb_shape sh = acp_shape(1);
        acp_seg(sh, L.vG, 0, b->g_off, b->n);
        acp_seg(sh, L.vH, 0, b->h_off, b->n);
        acp_seg(sh, L.cl, 0, b->q_off, 1);
        if ((rc = fb_launch(ctx, b->d_blk, L, b->B, *b->gens, sh, ipa_fb_plan(b, sh), b->d_stat, 1, s, b->d_part, nullptr))) return rc;
    }
    k_dyn_window_sums<<<b->B, DYN_W, 0, s>>>(b->d_blk, L, b->d_dyn, 2 * b->lg + 1, b->d_wsum);
    LAUNCH_CHECK(ctx);
    k_ipa_accept<<<(b->B + 63) / 64, 64, 0, s>>>(b->B, b->d_wsum, b->d_stat, b->d_bad, b->d_accept);
    LAUNCH_CHECK(ctx);
    ipa_mark(b, "check");
    return BPP_OK;
}
// accept bytes and the transcripts as the replay left them (never touched by the weights) back to the caller
static int ipa_verify_download(bpp_ipa_batch *b, uint8_t *transcripts, uint8_t *accept, const char *what) {
    bpp_ctx *ctx = b->ctx;
    cudaStream_t s = ctx->stream;
    CK(ctx, cudaMemcpyAsync(accept, b->d_accept, b->B, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaMemcpyAsync(transcripts, b->d_tr, (size_t)b->B * BPP_TRANSCRIPT_BYTES, cudaMemcpyDeviceToHost, s));
    ipa_mark(b, "download");
    CK(ctx, cudaStreamSynchronize(s));
    ipa_marks_dump(b, what);
    return BPP_OK;
}

extern "C" int bpp_ipa_batch_verify(bpp_ipa_batch *b, const uint8_t *q, const uint8_t *G_factors, const uint8_t *H_factors,
                                    const uint8_t *P, const uint8_t *proofs, uint8_t *transcripts, uint8_t *accept) {
    int rc;
    if ((rc = ipa_verify_scalars(b, q, G_factors, H_factors, P, proofs, transcripts, accept, false))) return rc;
    if ((rc = ipa_verify_per_proof(b))) return rc;
    return ipa_verify_download(b, transcripts, accept, "verify");
}

// The batch as one MSM (the shuffle verifier's acp_verify_rlc over this layout): rho_p from a copy of each proof's
// final transcript rekeyed with the verifier seed (k_ipa_weights; 0 for a proof already refused), then
// sum_p rho_p (P_p + sum_k u_k^2 L_k + u_k^-2 R_k) + sum_i (sum_p rho_p vG_p,i) G_i + (.. vH ..) H_i + (.. cl ..) Q in one
// Pippenger MSM over B (2 lg n + 1) proof points and the 2 n + 1 generators, whose scalars add up across proofs.  The
// identity accepts every proof of nonzero weight; otherwise *decided = false and the caller checks every proof on its own.
static int ipa_verify_rlc(bpp_ipa_batch *b, const uint8_t *verifier_seed, bool *decided) {
    bpp_ctx *ctx = b->ctx;
    const acp_layout &L = b->lay;
    const uint32_t B = b->B, n = b->n, per = 2 * b->lg + 1, nstat = 2 * n + 1;
    const size_t N = (size_t)B * per + nstat;
    cudaStream_t s = ctx->stream;
    *decided = false;
    int rc;
    uint8_t seed[32];
    if ((rc = set_verifier_seed(ctx, b->d_vseed, verifier_seed, seed))) return rc;
    TR_LAUNCH(k_ipa_weights, B, s, b->d_tr, b->d_in, b->d_lr, (const uint8_t *)b->d_vseed, L, B, b->d_blk);
    LAUNCH_CHECK(ctx);
    k_rlc_weights<<<(B + 127) / 128, 128, 0, s>>>(L, B, 0, b->d_bad, b->d_blk);
    LAUNCH_CHECK(ctx);
    k_rlc_dyn_scalars<<<dim3((per + 127) / 128, B), 128, 0, s>>>(L, per, B, L.rho, b->d_blk, b->d_rlc_sc);
    LAUNCH_CHECK(ctx);
    k_rlc_stat_scalars<<<nstat, 128, 0, s>>>(L, rlc_segs{{L.vG, L.vH, L.cl}, {n, n, 1}}, B, L.rho, b->d_blk,
                                             b->d_rlc_sc + 8 * (size_t)B * per);
    LAUNCH_CHECK(ctx);
    ipa_mark(b, "rlc-scalars");
    bpp_points view;
    view.niels = b->d_dyn;
    view.n = N;
    // one window group, as acp_verify_rlc: the SM time of the MSM, not the latency of one call
    rc = msm_enqueue(ctx, b->d_rlc_sc, &view, 0, N, b->d_rlc_out, 1, true, 1);
    view.niels = nullptr;
    if (rc) return rc;
    ipa_mark(b, "rlc-msm");
    k_rlc_accept<<<(B + 127) / 128, 128, 0, s>>>(b->d_rlc_out, L, B, L.rho, b->d_blk, b->d_accept, b->d_rlc_flag);
    LAUNCH_CHECK(ctx);
    CK(ctx, cudaMemcpyAsync(b->h_rlc_flag, b->d_rlc_flag, 4, cudaMemcpyDeviceToHost, s));
    CK(ctx, cudaStreamSynchronize(s));
    *decided = b->h_rlc_flag[0] == 0;
    return BPP_OK;
}

extern "C" int bpp_ipa_batch_verify_combined(bpp_ipa_batch *b, const uint8_t *q, const uint8_t *G_factors, const uint8_t *H_factors,
                                             const uint8_t *P, const uint8_t *proofs, const uint8_t *verifier_seed,
                                             uint8_t *transcripts, uint8_t *accept) {
    int rc;
    const bool rlc = b && ipa_rlc_pays(b);
    if ((rc = ipa_verify_scalars(b, q, G_factors, H_factors, P, proofs, transcripts, accept, rlc))) return rc;
    bool decided = false;
    if (rlc && (rc = ipa_verify_rlc(b, verifier_seed, &decided))) return rc;
    if (!decided && (rc = ipa_verify_per_proof(b))) return rc;
    return ipa_verify_download(b, transcripts, accept, "verify_combined");
}

// The weights rho_p as k_ipa_weights drew them in the batch's last combined check (count x 32, host)
extern "C" int bpp_ipa_batch_download_weights(bpp_ipa_batch *b, uint8_t *rho) {
    if (!b || !rho || !b->d_rlc_sc) return BPP_ERR_INVALID_ARG;
    bpp_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpy2DAsync(rho, 32, b->d_blk + 8 * (size_t)b->lay.rho0, (size_t)b->lay.stride * 32, 32, b->B,
                              cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return BPP_OK;
}

extern "C" int bpp_ipa_batch_gather_accept(bpp_ipa_batch *b, size_t per, uint8_t *accept_all) {
    if (!b || !accept_all || per < b->B) return BPP_ERR_INVALID_ARG;
    return gather_accept(b->ctx, b->d_accept, b->B, per, accept_all);
}
