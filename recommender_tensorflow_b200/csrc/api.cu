// libdeepfm_b200: C ABI (include/deepfm_b200.h) + step orchestration.
// One handle = one model instance (tables, optimizer slots, dense tower, workspaces) on one device.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <type_traits>
#include <vector>

#include <cfloat>
#include "dfm_types.cuh"
#include "embed_kernels.cuh"
#include "mlp_kernels.cuh"
#include "prims.cuh"
#include "small_mlp.cuh"
#include "fused_small.cuh"
#include "fused_rows_args.cuh"
#include "summary.cuh"
#include "tc_gemm.cuh"
#include "xchg.cuh"

#ifndef TC_BK
#define TC_BK 32   // k-block depth of the tcgen05 GEMMs (16 gives a deeper TMA ring; measured equal, smem bandwidth is the limit)
#endif

static thread_local std::string g_create_error;
struct dfm_handle;
struct EpiArgs;
static int tc_setup_once();
static int build_replay(dfm_handle* h, int64_t cap);
static RowReplay make_rr(const dfm_handle* h, int64_t upto);
template <int K> static int fused_set_attr(dfm_handle* h);
static bool tc_presplit();
// Split count of the weight-gradient GEMM (reduction over the batch).  tcgen05 aligns and TRUNCATES the products it
// folds into the fp32 TMEM accumulator: measured bias ~3e-8 x (products in the chain) relative to the accumulated
// magnitude (1.9e-5 after an 8 192-row chain of random operands, tests/test_gpu_tc_gemm.py; an fp32 reference: 3.5e-7).
// Shorter chains + round-to-nearest adds of the partials bound it; 2 048 rows keeps the partial traffic of the
// default split (one CTA per SM) and was measured equal, on the configs[2] step, to 512-row chains (which cost 0.06 ms).
static inline int tc_wgrad_splits(int64_t K, int requested) {
    const int64_t need = (K + 2047) / 2048;
    return (int)std::min<int64_t>(std::max<int64_t>(requested, need), 1024);
}
static int tc_gemm_kmajor(dfm_handle* h, const float* A_hi, const float* A_lo, int lda, const float* B_hi, const float* B_lo, int ldb,
                          float* C, int ldc, int M, int N, int K, int epi, const EpiArgs& ep, cudaStream_t st);
static int tc_gemm_mnmajor(dfm_handle* h, const float* A, int lda, const float* B, int ldb, float* Cpart, int M, int N, int K, int splits,
                           int* k_per_split_out, cudaStream_t st);

// sort + segment workspace for one list of (row key, payload) pairs
struct SegWS {
    int64_t cap = 0;
    uint32_t *keys[2] = {nullptr, nullptr}, *vals[2] = {nullptr, nullptr};
    void* sort_temp = nullptr;
    unsigned long long* flags = nullptr; void* scan_temp = nullptr; unsigned long long* seg_total = nullptr;
    SegCounts* seg_cnt = nullptr;
    uint32_t *row_start = nullptr, *row_piece0 = nullptr, *piece_start = nullptr, *urow = nullptr, *uval = nullptr, *hot_list = nullptr;
    uint32_t* pos_row = nullptr;     // sharded requester: unique-row index of every sorted position
    uint32_t* n_compact = nullptr;   // record-staged step: {lookups that go through the sort, once-only lookups} of the step
    float* piece_sum = nullptr;
    int cur = 0;     // which keys/vals buffer holds the sorted list
    const uint32_t* skeys() const { return keys[cur]; }
    const uint32_t* svals() const { return vals[cur]; }
};

struct DenseT {
    std::string name;
    int64_t off, rows, cols;
};

// alpha_t = lr sqrt(1 - beta2^t) / (1 - beta1^t) with TF's float32 running products is a deterministic function of t:
// the whole sequence (and the replay tables built from it) exists ahead of time
struct ReplayHost {
    std::vector<float> alpha;          // [cap + H + 1], alpha[0] unused
    int H = 0; bool adam = false, closed = false;
    float* d_alpha = nullptr; float4* d_T4 = nullptr; float* d_U = nullptr; float4* d_PQ = nullptr;
    ReplayTab tab{};
};

struct HostStage {          // one in-flight host batch (double buffered)
    uint8_t* d_arena = nullptr;
    size_t   cap = 0;
    cudaEvent_t copied = nullptr, done = nullptr;
    float*   h_loss = nullptr;   // pinned
    bool     busy = false;
};

struct dfm_handle {
    int dc = 0, dn = 0, K = 0, L = 0;
    int dcs = 0;                 // value slots per sample = sum of column widths (== dc without multivalent columns)
    int n_src = 0;               // source columns of crossed columns: cols[dc + s], raw data cat_data[dc + s]
    bool has_cross = false;      // a crossed column among the model columns: transform_kernel<.., CROSS = true>
    bool has_bags = false;
    // tiny-vocabulary columns reduced densely instead of through the sort (embed_kernels.cuh: tiny_reduce_kernel)
    int n_tiny = 0, n_big = 0, n_tiny_rows = 0, tiny_blocks_max = 0, tiny_group_rows = 0;
    int32_t *d_tiny_slot = nullptr, *d_key_slot = nullptr, *d_trow0 = nullptr;
    uint32_t* d_trow_grow = nullptr; float* tiny_partial = nullptr; SegCounts* d_tiny_cnt = nullptr;
    int32_t *d_slot_col = nullptr, *d_slot_j = nullptr, *d_field_slot0 = nullptr; float* inv_cnt = nullptr;
    int hidden[DFM_MAX_HIDDEN] = {0};
    int use_linear = 1, use_mf = 1, use_dnn = 1, need_emb = 1, loss_red = 0;
    dfm_optimizer od{}, ol{};
    int max_batch = 0, device = 0, rank = 0, world = 1;
    float dropout = 0.f; uint64_t dropout_seed = 0;
    int activation = 0;          // DFM_ACT_*; != ReLU: general CUDA-core tower only
    std::vector<ColDev> cols;
    std::vector<std::string> col_names;
    std::vector<uint32_t> row_off;   // [dc+1]
    uint64_t R = 0;
    int key_bits = 1;
    int emb_slots = 2;
    Table tb{};               // one record per row: w | {lin w, s1, s2, last_step} | slot1 | slot2 (dfm_types.cuh)

    ColDev* d_cols = nullptr; float* d_bounds = nullptr; uint8_t* d_voc_bytes = nullptr; int32_t* d_voc_offs = nullptr;
    longlong2* d_vtab = nullptr;     // hash tables of the table-looked-up vocabulary columns, back to back
    bool has_vtab = false;           // such a column exists: transform_kernel<.., VTAB = true>
    uint32_t* d_row_off = nullptr;

    std::vector<DenseT> dense;
    int64_t n_deep = 0, n_dense = 0;
    float *dw = nullptr, *ds1 = nullptr, *ds2 = nullptr, *dg = nullptr;

    // workspaces
    int32_t* ids = nullptr;
    SegWS ws;        // lookups of the local batch (requester side when sharded)
    SegWS ws_own;    // sharded mode: lookups received from all ranks for the rows this rank owns
    uint64_t R_loc = 0;          // rows stored on this rank (= R when world == 1)
    uint32_t Rl = 0;             // ceil(R / world): key space per owner
    uint32_t* uidx = nullptr;    // lookup -> index in the unique-row list of the local batch
    uint32_t* req_rows = nullptr;   // unique rows of the local batch as local indices at their owners (owner-major order)
    int32_t* d_counts = nullptr; int32_t* h_counts = nullptr;   // [world] unique rows per owner, [world] = total
    // state of the NEXT batch, computed ahead of time on the side stream (dfm_prefetch_batch)
    SegWS ws_next; int32_t* ids_next = nullptr; uint32_t *uidx_next = nullptr, *req_rows_next = nullptr; int32_t* d_counts_next = nullptr;
    cudaEvent_t ev_prefetch = nullptr; int prefetch_B = -1;
    cudaEvent_t ev_done[2] = {nullptr, nullptr};     // end of train step t on its stream, ring of two (t % 2)
    const void* prefetch_tag = nullptr;      // unsharded prefetch (dfm_prefetch_batch): first column pointer of the prefetched batch
    int64_t shard_n_req = 0, shard_n_recv = 0; int shard_B = 0; float shard_scale = 0.f;
    // flag-synchronised exchange over peer memory (xchg.cuh): own region + mapped peer regions
    uint8_t* xreg = nullptr; size_t xreg_bytes = 0; XchgDev xd{}; bool x_ready = false;
    void* x_opened[MAX_PEERS] = {nullptr};
    uint32_t x_epoch = 0; unsigned int* x_ticket = nullptr;      // exchange rounds so far; tickets of the producer kernels
    PeerRoute* d_xroute = nullptr; uint32_t* d_nrecv = nullptr; float* d_dense_total = nullptr; float* d_loss_part = nullptr;
    bool xchg_pending = false;
    cudaEvent_t ev_xpf_fork = nullptr, ev_xpf_done = nullptr; bool x_pf_valid = false; const void* x_pf_tag = nullptr; int x_pf_B = -1;
    cudaEvent_t ev_xfork = nullptr, ev_xjoin = nullptr; int x_B = -1; int64_t x_global_batch = 0; bool x_train = false;
    float *h0 = nullptr, *s = nullptr, *zacc = nullptr, *logits = nullptr, *dz = nullptr, *dE = nullptr;
    float* act[DFM_MAX_HIDDEN + 1] = {nullptr};
    float* dact[DFM_MAX_HIDDEN + 1] = {nullptr};
    float* splitk = nullptr; int splits = 1, k_chunk = 0;
    float* colpart = nullptr; int rows_per_chunk = 512; int num_rows_per_chunk = 128;   // numeric-gradient chunks are smaller: more CTAs
    float* head_part = nullptr; int head_blocks = 0;
    bool fused_head = false; float* head_gpart = nullptr; int fused_head_blocks = 0;
    bool tc_mlp = false; float* tc_w = nullptr; int64_t tc_off[DFM_MAX_HIDDEN] = {0}; int tc_nz[DFM_MAX_HIDDEN] = {0};
    bool small_mlp = false; SmallMlpDesc sm{}; int small_grid = 0; size_t small_smem = 0;
    float *up_partial = nullptr, *w0_partial = nullptr;
    float* d_loss = nullptr; float* d_dzsum = nullptr;
    int* d_err = nullptr;

    // step state
    int64_t step = 0, flushed_step = 0;
    // alpha_t sequence + closed-form replay tables of the non-lazy Adam (replay.cuh), one set per optimizer group
    ReplayHost rp_d, rp_l; bool rp_same = false; int64_t alpha_cap = 0;
    // fused small-tower step (fused_small.cuh): gather + FM + tower forward/backward in one kernel
    bool fused = false; size_t fused_smem = 0; int fused_grid = 0, n_numacc = 0;
    float *num_partial = nullptr, *num_scratch = nullptr; unsigned int* fused_done = nullptr;
    // record-staged step with the in-kernel optimizer for once-only rows (fused_rows.cuh)
    bool fused_rows = false; size_t fr_smem = 0; uint32_t* claim = nullptr; uint32_t claim_mask = 0; size_t claim_bytes = 0;
    // layer_summary workspace (summary.cuh), allocated on first use
    float *sum_h0 = nullptr, *sum_s = nullptr, *sum_lin = nullptr, *sum_mf = nullptr, *sum_hidden = nullptr, *sum_dnn = nullptr, *sum_logits = nullptr;
    double* sum_limits = nullptr; SummaryStats* sum_stats = nullptr; unsigned long long* sum_buckets = nullptr;
    bool claim_live = false;          // this step's claim table is filled: once-only rows are applied by fused_rows_kernel
    bool last_step_rows = false;
    bool fr_side = false;             // this step's sort runs on the side stream beside fused_rows_kernel
    // row-sharded requester on the record-staged kernel (row-buffer mode)
    bool fused_rows_rb = false; size_t fr_smem_rb = 0; uint8_t* once_lk = nullptr; bool fr_rb_live = false;

    cudaStream_t stream = nullptr, copy_stream = nullptr;
    // small tables: the sort / segment stage runs on a side stream next to the gather and the tower (see train_impl)
    cudaStream_t side_stream = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_aux_fork = nullptr, ev_aux_join = nullptr;
    bool overlap_sort = false; size_t splitk_off[DFM_MAX_HIDDEN] = {0};
    HostStage stage[2];
    int64_t host_calls = 0; int last_slot = -1;
    float* h_logits_pinned = nullptr;

    int64_t launches = 0, last_step_launches = 0;
    bool profiling = false;
    // small-batch steps replay as one CUDA graph (train_step_graphed)
    cudaGraphExec_t gexec = nullptr; int64_t graph_steps = 0, graph_rebuilds = 0;
    static constexpr int NPH = 11;
    cudaEvent_t ph_ev[NPH + 1] = {nullptr};
    float ph_ms[NPH] = {0};
    std::string err;
    int sm_count = 148;
};

static const char* kPhases[dfm_handle::NPH] = {"transform", "sort", "segments", "catchup", "gather", "mlp_fwd",
                                               "loss", "mlp_bwd", "reduce", "update", "dense"};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            char buf_[512];                                                                        \
            snprintf(buf_, sizeof buf_, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            if (h) h->err = buf_; else g_create_error = buf_;                                      \
            return DFM_ERR_CUDA;                                                                   \
        }                                                                                          \
    } while (0)

#define FAIL(code, msg)                                        \
    do {                                                       \
        if (h) h->err = (msg); else g_create_error = (msg);    \
        return (code);                                         \
    } while (0)

static inline unsigned cdiv(int64_t a, int64_t b) { return (unsigned)((a + b - 1) / b); }
static inline float __int_as_float_host(int v) { float f; memcpy(&f, &v, 4); return f; }

static int opt_slots(int kind) { return kind == DFM_OPT_ADAM ? 2 : kind == DFM_OPT_ADAGRAD ? 1 : kind == DFM_OPT_FTRL ? 2 : kind == DFM_OPT_RMSPROP ? 2 : 0; }

static OptDev make_opt(const dfm_optimizer& o, float alpha) {
    OptDev d{};
    d.kind = o.kind; d.lr = o.lr; d.b1 = o.beta1; d.b2 = o.beta2; d.eps = o.eps;
    d.omb1 = 1.0f - o.beta1;
    d.omb2 = 1.0f - o.beta2;
    d.alpha = o.kind == DFM_OPT_ADAM ? alpha : 0.f;
    d.safe_early = (o.kind == DFM_OPT_ADAM && o.beta1 < 0.95f * sqrtf(o.beta2)) ? 1 : 0;
    return d;
}

static void free_replay(ReplayHost& r) {
    if (r.d_alpha) cudaFree(r.d_alpha);
    if (r.d_T4) cudaFree(r.d_T4);
    if (r.d_U) cudaFree(r.d_U);
    if (r.d_PQ) cudaFree(r.d_PQ);
    r.d_alpha = nullptr; r.d_T4 = nullptr; r.d_U = nullptr; r.d_PQ = nullptr;
}

template <typename T>
static int dalloc(dfm_handle* h, T** p, size_t count) {
    CK(cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(count, 1) * sizeof(T)));
    return DFM_OK;
}

static int alloc_ws(dfm_handle* h, SegWS& ws, int64_t n, int K, bool with_pos_row = false) {
    ws.cap = n;
    if (with_pos_row && dalloc(h, &ws.pos_row, n)) return DFM_ERR_CUDA;
    for (int i = 0; i < 2; ++i) { if (dalloc(h, &ws.keys[i], n)) return DFM_ERR_CUDA; if (dalloc(h, &ws.vals[i], n)) return DFM_ERR_CUDA; }
    CK(cudaMalloc(&ws.sort_temp, std::max(prims::sort_temp_bytes(n), prims::onesweep_temp_bytes(n))));
    if (dalloc(h, &ws.flags, n)) return DFM_ERR_CUDA;
    CK(cudaMalloc(&ws.scan_temp, prims::scan_temp_bytes(n, 8) + 64));
    if (dalloc(h, &ws.seg_total, 1)) return DFM_ERR_CUDA;
    if (dalloc(h, &ws.seg_cnt, 1)) return DFM_ERR_CUDA;
    CK(cudaMemset(ws.seg_cnt, 0, sizeof(SegCounts)));
    if (dalloc(h, &ws.row_start, n + 1)) return DFM_ERR_CUDA;
    if (dalloc(h, &ws.row_piece0, n + 1)) return DFM_ERR_CUDA;
    if (dalloc(h, &ws.piece_start, n + 1)) return DFM_ERR_CUDA;
    if (dalloc(h, &ws.urow, n + 1)) return DFM_ERR_CUDA;
    if (dalloc(h, &ws.uval, n + 1)) return DFM_ERR_CUDA;
    if (dalloc(h, &ws.n_compact, 2)) return DFM_ERR_CUDA;
    if (dalloc(h, &ws.hot_list, (size_t)(2 * (n / 32 + 2)))) return DFM_ERR_CUDA;
    if (dalloc(h, &ws.piece_sum, (size_t)(2 * (n / 32 + 2)) * (K + 4))) return DFM_ERR_CUDA;
    return DFM_OK;
}

static void free_ws(SegWS& ws) {
    void* ptrs[] = {ws.keys[0], ws.keys[1], ws.vals[0], ws.vals[1], ws.sort_temp, ws.flags, ws.scan_temp, ws.seg_total, ws.seg_cnt,
                    ws.row_start, ws.row_piece0, ws.piece_start, ws.urow, ws.uval, ws.hot_list, ws.piece_sum, ws.pos_row, ws.n_compact};
    for (void* p : ptrs) if (p) cudaFree(p);
}

// ------------------------------------------------------------------------------------- create
extern "C" const char* dfm_version(void) { return "deepfm_b200 0.1 (sm_100a)"; }

extern "C" const char* dfm_last_error(const dfm_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

static int64_t pad32(int64_t x) { return (x + 31) / 32 * 32; }

static void free_all(dfm_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    void* ptrs[] = {h->d_cols, h->d_bounds, h->d_voc_bytes, h->d_voc_offs, h->d_vtab, h->d_row_off, h->tb.rec, h->dw,
                    h->ds1, h->ds2, h->dg, h->ids, h->h0, h->s, h->zacc, h->logits, h->dz, h->dE, h->splitk, h->colpart, h->head_part,
                    h->d_loss, h->d_dzsum, h->d_err, h->num_partial, h->num_scratch, h->fused_done, h->claim, h->once_lk, h->sum_h0, h->sum_s, h->sum_lin, h->sum_mf, h->sum_hidden, h->sum_dnn, h->sum_logits, h->sum_limits, h->sum_stats, h->sum_buckets, h->up_partial, h->w0_partial, h->tc_w, h->head_gpart, h->d_slot_col, h->d_slot_j, h->d_field_slot0, h->inv_cnt, h->uidx,
                    h->req_rows, h->d_counts};
    for (void* p : ptrs) if (p) cudaFree(p);
    free_ws(h->ws);
    free_ws(h->ws_own);
    free_replay(h->rp_d); free_replay(h->rp_l);
    if (h->h_counts) cudaFreeHost(h->h_counts);
    free_ws(h->ws_next);
    { void* np[] = {h->ids_next, h->uidx_next, h->req_rows_next, h->d_counts_next}; for (void* p : np) if (p) cudaFree(p); }
    if (h->ev_prefetch) cudaEventDestroy(h->ev_prefetch);
    if (h->gexec) cudaGraphExecDestroy(h->gexec);
    for (cudaEvent_t e : h->ev_done) if (e) cudaEventDestroy(e);
    { void* tp[] = {h->d_tiny_slot, h->d_key_slot, h->d_trow0, h->d_trow_grow, h->tiny_partial, h->d_tiny_cnt};
      for (void* p : tp) if (p) cudaFree(p); }
    for (void* p : h->x_opened) if (p) cudaIpcCloseMemHandle(p);
    { void* xp[] = {h->xreg, h->x_ticket, h->d_xroute, h->d_nrecv, h->d_dense_total, h->d_loss_part}; for (void* p : xp) if (p) cudaFree(p); }
    if (h->ev_xpf_fork) cudaEventDestroy(h->ev_xpf_fork);
    if (h->ev_xpf_done) cudaEventDestroy(h->ev_xpf_done);
    if (h->ev_xfork) cudaEventDestroy(h->ev_xfork);
    if (h->ev_xjoin) cudaEventDestroy(h->ev_xjoin);
    for (int i = 1; i <= DFM_MAX_HIDDEN; ++i) { if (h->act[i]) cudaFree(h->act[i]); if (h->dact[i]) cudaFree(h->dact[i]); }
    for (auto& s : h->stage) {
        if (s.d_arena) cudaFree(s.d_arena);
        if (s.copied) cudaEventDestroy(s.copied);
        if (s.done) cudaEventDestroy(s.done);
        if (s.h_loss) cudaFreeHost(s.h_loss);
    }
    if (h->h_logits_pinned) cudaFreeHost(h->h_logits_pinned);
    for (auto& e : h->ph_ev) if (e) cudaEventDestroy(e);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->side_stream) cudaStreamDestroy(h->side_stream);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->ev_aux_fork) cudaEventDestroy(h->ev_aux_fork);
    if (h->ev_aux_join) cudaEventDestroy(h->ev_aux_join);
    delete h;
}

extern "C" void dfm_destroy(dfm_handle* h) { free_all(h); }

// String vocabularies up to this size are scanned (embed_kernels.cuh transform_one); larger ones, and every integer
// vocabulary, are looked up through a hash table (vocab_probe).  DFM_VOCAB_PATH=scan|table forces string vocabularies
// onto one path (A/B runs and tests).
constexpr int VOCAB_SCAN_MAX = 8;

static const uint8_t* vocab_entry(const dfm_column& c, int j, int64_t* len) {
    if (c.vocab) { *len = (int64_t)strlen(c.vocab[j]); return reinterpret_cast<const uint8_t*>(c.vocab[j]); }
    *len = c.vocab_offsets[j + 1] - c.vocab_offsets[j];
    return c.vocab_data + c.vocab_offsets[j];
}

// vocabulary and identity columns (cat and src), before any CUDA call (TF-1.12 feature_column.py argument checks where
// TF has one)
static int check_vocab_columns(const dfm_config* cfg, dfm_handle* h) {
    int64_t total = 0;
    for (int f = 0; f < cfg->n_cat + cfg->n_src; ++f) {
        const dfm_column& c = f < cfg->n_cat ? cfg->cat[f] : cfg->src[f - cfg->n_cat];
        const std::string nm = c.name ? c.name : "";
        if (c.kind == DFM_COL_IDENTITY && c.has_default && (c.default_value < 0 || c.default_value >= c.num_buckets))
            FAIL(DFM_ERR_INVALID_ARG, "default_value " + std::to_string(c.default_value) + " not in range [0, " +
                                          std::to_string(c.num_buckets) + "), column_name " + nm);
        if (c.kind != DFM_COL_VOCAB) continue;
        if (c.vocab_size < 1) FAIL(DFM_ERR_INVALID_ARG, "vocabulary column " + nm + " needs vocab_size >= 1");
        if (c.num_oov < 0) FAIL(DFM_ERR_INVALID_ARG, "Invalid num_oov_buckets " + std::to_string(c.num_oov) + " in " + nm + ".");
        const bool str_voc = c.vocab || c.vocab_data || c.vocab_offsets;
        if (c.dtype == DFM_STRING) {
            if (!str_voc && c.vocab_int) FAIL(DFM_ERR_INVALID_ARG, "dtype string and vocabulary dtype int64 do not match in " + nm);
            if (!c.vocab && !(c.vocab_data && c.vocab_offsets))
                FAIL(DFM_ERR_INVALID_ARG, "string vocabulary column " + nm + " needs vocab or vocab_data + vocab_offsets");
            if (!c.vocab) {
                if (c.vocab_offsets[0] < 0) FAIL(DFM_ERR_INVALID_ARG, "vocab_offsets of " + nm + " must start at >= 0");
                for (int j = 0; j < c.vocab_size; ++j)
                    if (c.vocab_offsets[j + 1] < c.vocab_offsets[j]) FAIL(DFM_ERR_INVALID_ARG, "vocab_offsets of " + nm + " are not monotone");
            }
            for (int j = 0; j < c.vocab_size; ++j) {
                int64_t len;
                vocab_entry(c, j, &len);
                total += len;
            }
            if (total > 0x7fffffffll)
                FAIL(DFM_ERR_UNSUPPORTED, "string vocabularies hold more than 2^31 - 1 bytes (int32 device offsets)");
        } else if (c.dtype == DFM_INT32) {
            if (!c.vocab_int && str_voc) FAIL(DFM_ERR_INVALID_ARG, "dtype int32 and vocabulary dtype string do not match in " + nm);
            if (!c.vocab_int) FAIL(DFM_ERR_INVALID_ARG, "integer vocabulary column " + nm + " needs vocab_int");
        } else {
            FAIL(DFM_ERR_UNSUPPORTED, "vocabulary column " + nm + " needs string or int32 input");
        }
        if (c.has_default) {
            if (c.num_oov > 0) FAIL(DFM_ERR_INVALID_ARG, "Can't specify both num_oov_buckets and default_value in " + nm + ".");
            if (c.default_value != -1 && (c.default_value < 0 || c.default_value >= c.vocab_size))
                FAIL(DFM_ERR_INVALID_ARG, "default_value " + std::to_string(c.default_value) + " of " + nm +
                                              " must be -1 or in [0, vocab_size)");
        }
    }
    return DFM_OK;
}

// Hash tables of the table-looked-up vocabulary columns (vocab_probe): capacity = the power of two >= 2 V, placement on
// the host in vocabulary order (a deterministic layout; a repeated entry keeps its first index).  String fingerprints
// are computed on the device by the function the probe uses.
static int build_vocab_tables(dfm_handle* h, const dfm_config* cfg, const std::vector<int>& vt_cols) {
    if (vt_cols.empty()) return DFM_OK;
    const char* bits_env = getenv("DFM_VOCAB_FP_BITS");
    const int fp_bits = bits_env ? atoi(bits_env) : 64;
    const uint64_t fp_mask = fp_bits >= 64 || fp_bits <= 0 ? ~0ull : (1ull << fp_bits) - 1;
    std::vector<uint64_t> base;
    uint64_t total = 0;
    for (int f : vt_cols) {
        uint64_t cap = 2;
        while (cap < 2ull * (uint64_t)h->cols[f].voc_cnt) cap <<= 1;
        base.push_back(total);
        total += cap;
    }
    std::vector<longlong2> tab(total, make_longlong2(0, -1));
    std::vector<uint64_t> keys;
    uint64_t* d_fp = nullptr;
    for (size_t t = 0; t < vt_cols.size(); ++t) {
        const int f = vt_cols[t];
        ColDev& d = h->cols[f];
        const dfm_column& c = f < h->dc ? cfg->cat[f] : cfg->src[f - h->dc];
        const int V = d.voc_cnt;
        keys.resize(V);
        if (d.dtype == DFM_STRING) {
            if (dalloc(h, &d_fp, (size_t)V)) return DFM_ERR_CUDA;
            fingerprint_kernel<<<cdiv(V, 256), 256>>>(h->d_voc_bytes, h->d_voc_offs + d.voc_off, V, d_fp);
            CK(cudaGetLastError());
            CK(cudaMemcpy(keys.data(), d_fp, (size_t)V * 8, cudaMemcpyDeviceToHost));
            CK(cudaFree(d_fp));
            d_fp = nullptr;
            for (auto& k : keys) k &= fp_mask;
            d.fp_mask = fp_mask;
        } else {
            for (int j = 0; j < V; ++j) keys[j] = (uint64_t)c.vocab_int[j];
            d.fp_mask = ~0ull;
        }
        const uint64_t mask = (base.size() > t + 1 ? base[t + 1] : total) - base[t] - 1;
        longlong2* T = tab.data() + base[t];
        for (int j = 0; j < V; ++j) {
            uint64_t i = vocab_mix(keys[j]) & mask;
            bool dup = false;
            for (; T[i].y >= 0; i = (i + 1) & mask) {
                if ((uint64_t)T[i].x != keys[j]) continue;
                if (d.dtype != DFM_STRING) { dup = true; break; }
                int64_t la, lb;
                const uint8_t* a = vocab_entry(c, (int)T[i].y, &la);
                const uint8_t* b = vocab_entry(c, j, &lb);
                if (la == lb && memcmp(a, b, (size_t)la) == 0) { dup = true; break; }
            }
            if (!dup) T[i] = make_longlong2((long long)keys[j], j);
        }
        d.tab_mask = (uint32_t)mask;
    }
    if (dalloc(h, &h->d_vtab, (size_t)total)) return DFM_ERR_CUDA;
    CK(cudaMemcpy(h->d_vtab, tab.data(), total * sizeof(longlong2), cudaMemcpyHostToDevice));
    for (size_t t = 0; t < vt_cols.size(); ++t) h->cols[vt_cols[t]].vtab = h->d_vtab + base[t];
    h->has_vtab = true;
    return DFM_OK;
}

static int create_impl(const dfm_config* cfg, dfm_handle* h) {
    if (cfg->n_cat < 0 || cfg->n_cat > DFM_MAX_CAT || cfg->n_num < 0 || cfg->n_num > DFM_MAX_NUM || cfg->n_src < 0 ||
        cfg->n_cat + cfg->n_src > DFM_MAX_CAT)
        FAIL(DFM_ERR_INVALID_ARG, "too many feature columns");
    if (cfg->n_src > 0 && !cfg->src) FAIL(DFM_ERR_INVALID_ARG, "src is null");
    // crossed columns and their sources (TF-1.12 feature_column.py crossed_column / sparse_cross_op.cc)
    for (int s = 0; s < cfg->n_src; ++s) {
        const dfm_column& c = cfg->src[s];
        if (c.kind == DFM_COL_HASH)
            FAIL(DFM_ERR_INVALID_ARG, "categorical_column_with_hash_bucket is not supported for crossing. Hashing before crossing "
                                      "will increase probability of collision. Instead, use the feature name as a string.");
        if (c.kind == DFM_COL_RAW && c.dtype != DFM_INT32 && c.dtype != DFM_STRING)
            FAIL(DFM_ERR_INVALID_ARG, "a raw feature of a crossed column must be int32 or string (sparse_cross takes int64 / string)");
        if (c.kind != DFM_COL_RAW && c.kind != DFM_COL_BUCKETIZED && c.kind != DFM_COL_VOCAB && c.kind != DFM_COL_IDENTITY)
            FAIL(DFM_ERR_INVALID_ARG, "Unsupported key type. All keys must be either string, or categorical column except "
                                      "_HashedCategoricalColumn.");
    }
    for (int f = 0; f < cfg->n_cat; ++f) {
        const dfm_column& c = cfg->cat[f];
        if (c.kind == DFM_COL_RAW) FAIL(DFM_ERR_INVALID_ARG, "a raw column is allowed only as a source column of a cross");
        if (c.kind != DFM_COL_CROSSED) continue;
        if (c.num_buckets < 1) FAIL(DFM_ERR_INVALID_ARG, "hash_bucket_size must be > 1.");
        if (c.n_keys < 2 || !c.keys) FAIL(DFM_ERR_INVALID_ARG, "keys must be a list with length > 1.");
        if (c.n_keys > DFM_MAX_CROSS_KEYS) FAIL(DFM_ERR_UNSUPPORTED, "a crossed column has at most 8 keys");
        int64_t width = 1;
        for (int i = 0; i < c.n_keys; ++i) {
            if (c.keys[i] < 0 || c.keys[i] >= cfg->n_src) FAIL(DFM_ERR_INVALID_ARG, "crossed column key outside [0, n_src)");
            width *= std::max(1, cfg->src[c.keys[i]].width);
            if (width > 4 * DFM_MAX_CAT) FAIL(DFM_ERR_UNSUPPORTED, "too many value slots (sum of column widths)");
        }
    }
    if (int rc = check_vocab_columns(cfg, h)) return rc;
    // trainers/deep_fm.py:31-34
    if (cfg->n_cat + cfg->n_num == 0)
        FAIL(DFM_ERR_INVALID_ARG, "At least 1 feature column of categorical_columns or numeric_columns must be specified.");
    if (!(cfg->use_linear || cfg->use_mf || cfg->use_dnn))
        FAIL(DFM_ERR_INVALID_ARG, "At least 1 of linear, mf or dnn component must be used.");
    const int K = cfg->embedding_size;
    if (K < 4 || K > 128 || (K % 4) != 0 || (128 % K) != 0)
        FAIL(DFM_ERR_UNSUPPORTED, "embedding_size must be one of 4, 8, 16, 32, 64, 128");
    if (cfg->n_hidden < 0 || cfg->n_hidden > DFM_MAX_HIDDEN) FAIL(DFM_ERR_INVALID_ARG, "too many hidden layers");
    if (cfg->max_batch <= 0) FAIL(DFM_ERR_INVALID_ARG, "max_batch must be positive");
    if (cfg->max_batch > (1 << (32 - PAYLOAD_SLOT_BITS))) FAIL(DFM_ERR_UNSUPPORTED, "max_batch must be <= 2^24");
    if (cfg->world > 1 && (cfg->rank < 0 || cfg->rank >= cfg->world)) FAIL(DFM_ERR_INVALID_ARG, "rank must be in [0, world)");
    h->dc = cfg->n_cat; h->dn = cfg->n_num; h->K = K; h->L = cfg->use_dnn ? cfg->n_hidden : 0;
    for (int i = 0; i < h->L; ++i) {
        if (cfg->hidden_units[i] <= 0) FAIL(DFM_ERR_INVALID_ARG, "hidden_units must be positive");
        h->hidden[i] = cfg->hidden_units[i];
    }
    h->use_linear = cfg->use_linear != 0; h->use_mf = cfg->use_mf != 0; h->use_dnn = cfg->use_dnn != 0;
    h->need_emb = h->use_mf || h->use_dnn;
    h->loss_red = cfg->loss_reduction;
    h->od = cfg->opt_deep; h->ol = cfg->opt_linear;
    for (const dfm_optimizer* o : {&h->od, &h->ol})
        if (o->kind < DFM_OPT_ADAM || o->kind > DFM_OPT_RMSPROP) FAIL(DFM_ERR_INVALID_ARG, "unknown optimizer kind");
    h->max_batch = cfg->max_batch; h->device = cfg->device; h->rank = cfg->rank; h->world = std::max(1, cfg->world);
    if (!(cfg->dropout >= 0.f && cfg->dropout < 1.f)) FAIL(DFM_ERR_INVALID_ARG, "dropout must be in [0, 1)");
    h->dropout = cfg->dropout; h->dropout_seed = cfg->dropout_seed;
    if (cfg->activation < DFM_ACT_RELU || cfg->activation > DFM_ACT_IDENTITY) FAIL(DFM_ERR_INVALID_ARG, "activation must be one of DFM_ACT_*");
    h->activation = cfg->activation;
    CK(cudaSetDevice(h->device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->device));
    h->sm_count = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_aux_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_aux_join, cudaEventDisableTiming));

    // ---- columns
    std::vector<float> bounds;
    std::vector<uint8_t> voc_bytes;
    std::vector<int32_t> voc_offs;
    h->row_off.assign(h->dc + 1, 0);
    std::vector<int32_t> slot_col, slot_j, field_slot0;
    std::vector<int> vt_cols;        // vocabulary columns looked up through a hash table
    const char* vpath = getenv("DFM_VOCAB_PATH");
    uint64_t R = 0;
    h->n_src = cfg->n_src;
    for (int f = 0; f < h->dc + h->n_src; ++f) {
        const bool is_src = f >= h->dc;          // a source column: no table, no slots, no place in model order
        const dfm_column& c = is_src ? cfg->src[f - h->dc] : cfg->cat[f];
        ColDev d{};
        d.kind = c.kind; d.dtype = c.dtype;
        d.dflt = -1;
        d.width = std::max(1, c.width);
        if (c.kind == DFM_COL_CROSSED) {
            h->has_cross = true;
            d.width = 1;
            d.n_keys = c.n_keys;
            d.hash_key = c.hash_key ? c.hash_key : 0xDECAFCAFFEull;     // sparse_ops.py _DEFAULT_HASH_KEY
            for (int i = 0; i < c.n_keys && i < DFM_MAX_CROSS_KEYS; ++i) {      // n_keys was checked above
                d.keys[i] = (uint8_t)(h->dc + c.keys[i]);
                d.width *= std::max(1, cfg->src[c.keys[i]].width);
            }
        }
        if (!is_src) {
            if (d.width > 1) h->has_bags = true;
            for (int j = 0; j < d.width; ++j) { slot_col.push_back(f); slot_j.push_back(j); }
            field_slot0.push_back((int32_t)slot_col.size() - d.width);
        }
        uint64_t nb = 0;
        switch (c.kind) {
            case DFM_COL_CROSSED:
                nb = (uint64_t)c.num_buckets;
                break;
            case DFM_COL_RAW:
                break;
            case DFM_COL_HASH:
                if (c.num_buckets <= 0) FAIL(DFM_ERR_INVALID_ARG, "hash column needs num_buckets > 0");
                if (c.dtype == DFM_FLOAT32) FAIL(DFM_ERR_UNSUPPORTED, "hash column over float32 keys");
                nb = (uint64_t)c.num_buckets;
                break;
            case DFM_COL_IDENTITY:
                if (c.num_buckets <= 0) FAIL(DFM_ERR_INVALID_ARG, "identity column needs num_buckets > 0");
                if (c.dtype != DFM_INT32) FAIL(DFM_ERR_UNSUPPORTED, "identity column needs int32 input");
                if (c.has_default) d.dflt = (int32_t)c.default_value;      // range checked by check_vocab_columns
                nb = (uint64_t)c.num_buckets;
                break;
            case DFM_COL_BUCKETIZED:
                if (c.dtype == DFM_STRING) FAIL(DFM_ERR_INVALID_ARG, "bucketized column needs numeric input");
                d.bnd_off = (int)bounds.size(); d.bnd_cnt = c.n_boundaries;
                for (int j = 0; j < c.n_boundaries; ++j) bounds.push_back(c.boundaries[j]);
                nb = (uint64_t)c.n_boundaries + 1;
                break;
            case DFM_COL_VOCAB:       // checked by check_vocab_columns
                d.voc_off = (int)voc_offs.size(); d.voc_cnt = c.vocab_size; d.num_oov = c.num_oov;
                d.dflt = c.has_default ? (int32_t)c.default_value : -1;
                if (c.dtype == DFM_STRING) {
                    for (int j = 0; j < c.vocab_size; ++j) {
                        voc_offs.push_back((int32_t)voc_bytes.size());
                        int64_t len;
                        const uint8_t* p = vocab_entry(c, j, &len);
                        voc_bytes.insert(voc_bytes.end(), p, p + len);
                    }
                    voc_offs.push_back((int32_t)voc_bytes.size());
                }
                if (c.dtype != DFM_STRING || (vpath && !strcmp(vpath, "table")) ||
                    (!(vpath && !strcmp(vpath, "scan")) && c.vocab_size > VOCAB_SCAN_MAX))
                    vt_cols.push_back(f);
                nb = (uint64_t)c.vocab_size + (uint64_t)c.num_oov;
                break;
            default: FAIL(DFM_ERR_INVALID_ARG, "unknown column kind");
        }
        d.nb = nb;
        d.nb_rcp = nb >= 2 ? (uint64_t)(((unsigned __int128)1 << 64) / nb) : 0;
        h->cols.push_back(d);
        h->col_names.push_back(c.name ? c.name : "");
        if (is_src) continue;
        if (R > 0xffffffffull) FAIL(DFM_ERR_UNSUPPORTED, "more than 2^32 table rows on one device");
        h->row_off[f] = (uint32_t)R;
        R += nb;
    }
    if (R >= 0xfffffff0ull) FAIL(DFM_ERR_UNSUPPORTED, "more than 2^32 table rows on one device");
    h->row_off[h->dc] = (uint32_t)R;
    h->R = R;
    field_slot0.push_back((int32_t)slot_col.size());
    h->dcs = (int)slot_col.size();
    if (h->dcs > 4 * DFM_MAX_CAT) FAIL(DFM_ERR_UNSUPPORTED, "too many value slots (sum of column widths)");
    if (dalloc(h, &h->d_slot_col, slot_col.size())) return DFM_ERR_CUDA;
    if (dalloc(h, &h->d_slot_j, slot_j.size())) return DFM_ERR_CUDA;
    if (dalloc(h, &h->d_field_slot0, field_slot0.size())) return DFM_ERR_CUDA;
    if (!slot_col.empty()) {
        CK(cudaMemcpy(h->d_slot_col, slot_col.data(), slot_col.size() * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(h->d_slot_j, slot_j.data(), slot_j.size() * 4, cudaMemcpyHostToDevice));
    }
    CK(cudaMemcpy(h->d_field_slot0, field_slot0.data(), field_slot0.size() * 4, cudaMemcpyHostToDevice));
    h->Rl = (uint32_t)((R + h->world - 1) / h->world);
    h->R_loc = h->world > 1 ? (R > (uint64_t)h->rank ? (R - h->rank + h->world - 1) / h->world : 0) : R;
    if ((uint64_t)h->Rl * h->world >= 0xfffffff0ull) FAIL(DFM_ERR_UNSUPPORTED, "sharded key space exceeds 32 bits");
    h->key_bits = 1;
    const uint64_t key_max = h->world > 1 ? (uint64_t)h->Rl * h->world : R;   // keys take values 0..key_max
    while ((1ull << h->key_bits) <= key_max) ++h->key_bits;
    if (dalloc(h, &h->d_cols, h->cols.size())) return DFM_ERR_CUDA;
    if (dalloc(h, &h->d_bounds, bounds.size())) return DFM_ERR_CUDA;
    if (dalloc(h, &h->d_voc_bytes, voc_bytes.size())) return DFM_ERR_CUDA;
    if (dalloc(h, &h->d_voc_offs, voc_offs.size())) return DFM_ERR_CUDA;
    if (dalloc(h, &h->d_row_off, h->row_off.size())) return DFM_ERR_CUDA;
    if (!bounds.empty()) CK(cudaMemcpy(h->d_bounds, bounds.data(), bounds.size() * 4, cudaMemcpyHostToDevice));
    if (!voc_bytes.empty()) CK(cudaMemcpy(h->d_voc_bytes, voc_bytes.data(), voc_bytes.size(), cudaMemcpyHostToDevice));
    if (!voc_offs.empty()) CK(cudaMemcpy(h->d_voc_offs, voc_offs.data(), voc_offs.size() * 4, cudaMemcpyHostToDevice));
    if (int rc = build_vocab_tables(h, cfg, vt_cols)) return rc;
    if (!h->cols.empty()) CK(cudaMemcpy(h->d_cols, h->cols.data(), h->cols.size() * sizeof(ColDev), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->d_row_off, h->row_off.data(), h->row_off.size() * 4, cudaMemcpyHostToDevice));
    {
        const char* env = getenv("DFM_TINY");
        std::vector<int32_t> tslot, key_slot(std::max(h->dcs, 1), -1), trow0;
        std::vector<uint32_t> tgrow;
        // fused small-tower step (fused_small.cuh): its sparse optimizer rebuilds the lookup gradients on the fly, the
        // dense tiny-column reduction (which reads a dE buffer) is not used with it
        bool fused_candidate = false;
        if (cfg->use_dnn && h->activation == DFM_ACT_RELU && h->need_emb && !h->has_bags && h->L >= 1 && h->L <= SM_MAXL && K <= 32 && getenv("DFM_NO_FUSED") == nullptr &&
            getenv("DFM_NO_SMALL_MLP") == nullptr) {
            const int H1 = h->hidden[0];
            fused_candidate = (H1 == 8 || H1 == 16 || H1 == 32);
            for (int i = 0; i < h->L; ++i) fused_candidate = fused_candidate && h->hidden[i] <= SM_MAXH;
            const int D = (h->dc + h->dn) * K;
            fused_candidate = fused_candidate && D <= (256 / (H1 / 4)) * FS_NC && h->dn * (K + H1 + 2) <= 256 * FS_NUMACC &&
                              h->dc * FS_TS <= 512;
        }
        h->fused = fused_candidate;      // confirmed below once the shared-memory footprint is known
        const bool enable = h->world == 1 && !h->has_bags && !fused_candidate && !(env && atoi(env) == 0);
        for (int f = 0; f < h->dc; ++f) {
            const uint32_t nb = h->row_off[f + 1] - h->row_off[f];
            // the per-warp accumulators of all tiny rows must fit the shared-memory budget of tiny_reduce_kernel
            if (enable && nb <= (uint32_t)TINY_MAX && tgrow.size() + nb <= 4096) {
                trow0.push_back((int32_t)tgrow.size());
                for (uint32_t b = 0; b < nb; ++b) tgrow.push_back(h->row_off[f] + b);
                tslot.push_back(f);
            } else {
                key_slot[f] = h->n_big++;
            }
        }
        if (tslot.size() < 2) {       // not worth a second path
            h->n_big = h->dcs; tslot.clear(); trow0.clear(); tgrow.clear();
        }
        h->n_tiny = (int)tslot.size(); h->n_tiny_rows = (int)tgrow.size();
        trow0.push_back((int32_t)tgrow.size());
        {   // rows of the largest group of 32/LPR adjacent tiny columns = accumulator rows of one tiny_reduce block
            const int G = 32 / std::max(1, K / 4);
            for (int c0 = 0; c0 < h->n_tiny; c0 += G)
                h->tiny_group_rows = std::max(h->tiny_group_rows, trow0[std::min(h->n_tiny, c0 + G)] - trow0[c0]);
        }
        if (h->n_tiny) {
            h->tiny_blocks_max = (h->max_batch + TINY_SPB - 1) / TINY_SPB;
            if (dalloc(h, &h->d_tiny_slot, tslot.size()) || dalloc(h, &h->d_key_slot, key_slot.size()) || dalloc(h, &h->d_trow0, trow0.size()) ||
                dalloc(h, &h->d_trow_grow, tgrow.size()) || dalloc(h, &h->d_tiny_cnt, 1) ||
                dalloc(h, &h->tiny_partial, (size_t)h->tiny_blocks_max * h->n_tiny_rows * (K + 4)))
                return DFM_ERR_CUDA;
            CK(cudaMemcpy(h->d_tiny_slot, tslot.data(), tslot.size() * 4, cudaMemcpyHostToDevice));
            CK(cudaMemcpy(h->d_key_slot, key_slot.data(), key_slot.size() * 4, cudaMemcpyHostToDevice));
            CK(cudaMemcpy(h->d_trow0, trow0.data(), trow0.size() * 4, cudaMemcpyHostToDevice));
            CK(cudaMemcpy(h->d_trow_grow, tgrow.data(), tgrow.size() * 4, cudaMemcpyHostToDevice));
            SegCounts sc{};
            sc.n_rows = (uint32_t)h->n_tiny_rows;
            CK(cudaMemcpy(h->d_tiny_cnt, &sc, sizeof sc, cudaMemcpyHostToDevice));
        }
    }

    {   // With small tables every row is brought up to date at the start of the step (the literal non-lazy Adam, a few
        // microseconds for some thousand rows), so the forward pass does not wait for the list of touched rows and the
        // sort / segment kernels (small grids that leave most SMs idle) run beside the gather and the tower.
        const char* env = getenv("DFM_OVERLAP_SORT");
        h->overlap_sort = h->world == 1 && h->R_loc <= (1u << 16) && !(env && atoi(env) == 0);
    }

    // ---- tables: one record per row (see Table)
    h->emb_slots = opt_slots(h->od.kind);
    const size_t Ralloc = std::max<uint64_t>(h->R_loc, 1);
    R = h->R_loc;   // from here on: rows stored on this rank
    if (h->need_emb) {
        h->tb.lin_off = K; h->tb.s1_off = K + 4; h->tb.s2_off = 2 * K + 4;
        h->tb.stride = (K + 4 + h->emb_slots * K + 15) / 16 * 16;
    } else {
        h->tb.lin_off = 0; h->tb.s1_off = 0; h->tb.s2_off = 0; h->tb.stride = 4;
    }
    if (dalloc(h, &h->tb.rec, Ralloc * h->tb.stride)) return DFM_ERR_CUDA;
    CK(cudaMemset(h->tb.rec, 0, Ralloc * h->tb.stride * 4));

    // ---- dense parameters, packed: deep group first, then the linear group
    const int d = h->dc + h->dn, dK = d * K;
    int64_t off = 0;
    auto add = [&](const std::string& nm, int64_t rows, int64_t cols) {
        h->dense.push_back({nm, off, rows, cols});
        off += pad32(rows * cols);
    };
    if (h->need_emb && h->dn) add("num_emb", h->dn, K);
    if (h->use_dnn) {
        int in = dK;
        for (int i = 0; i < h->L; ++i) {
            add("W" + std::to_string(i), in, h->hidden[i]);
            add("b" + std::to_string(i), h->hidden[i], 1);
            in = h->hidden[i];
        }
        add("Wo", in, 1);
        add("bo", 1, 1);
    }
    h->n_deep = off;
    if (h->use_linear) {
        if (h->dn) add("num_lin", h->dn, 1);
        add("bias", 1, 1);
    }
    h->n_dense = off;
    for (float** p : {&h->dw, &h->ds1, &h->ds2, &h->dg}) {
        if (dalloc(h, p, (size_t)h->n_dense)) return DFM_ERR_CUDA;
        CK(cudaMemset(*p, 0, std::max<int64_t>(h->n_dense, 1) * 4));
    }

    // ---- workspaces
    const int64_t Bm = h->max_batch, n = Bm * std::max(h->dcs, 1);
    if (h->has_bags && dalloc(h, &h->inv_cnt, (size_t)Bm * h->dc)) return DFM_ERR_CUDA;
    CK(cudaFuncSetAttribute(transform_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 4 * DFM_MAX_CAT * 4));
    CK(cudaFuncSetAttribute(transform_kernel<32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 4 * DFM_MAX_CAT * 4));
    CK(cudaFuncSetAttribute(transform_kernel<32, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 4 * DFM_MAX_CAT * 4));
    CK(cudaFuncSetAttribute(transform_kernel<32, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 4 * DFM_MAX_CAT * 4));
    if (n >= (1ll << 31)) FAIL(DFM_ERR_UNSUPPORTED, "max_batch * n_cat must be < 2^31");
    if (dalloc(h, &h->ids, n)) return DFM_ERR_CUDA;
    if (alloc_ws(h, h->ws, n, K, h->world > 1)) return DFM_ERR_CUDA;
    if (h->world > 1) {
        // owner side: every rank may send up to its whole unique list; 2x the per-rank lookups + slack, checked at run time
        if (alloc_ws(h, h->ws_own, 2 * n + 4096, K)) return DFM_ERR_CUDA;
        if (dalloc(h, &h->uidx, n)) return DFM_ERR_CUDA;
        if (dalloc(h, &h->req_rows, n)) return DFM_ERR_CUDA;
        if (dalloc(h, &h->d_counts, (size_t)h->world + 1)) return DFM_ERR_CUDA;
        CK(cudaMallocHost(&h->h_counts, ((size_t)h->world + 1) * sizeof(int32_t)));
        h->xchg_pending = h->world <= MAX_PEERS;      // the exchange region is allocated below, once the dense size is known
    }
    if (h->fused) {       // does the fused kernel's tile fit in shared memory?
        SmallMlpDesc probe{};
        probe.L = h->L; probe.D = dK;
        int sum = 0, upc = 0;
        for (int i = 0; i < h->L; ++i) { probe.H[i] = h->hidden[i]; sum += h->hidden[i]; }
        for (int i = 0; i < h->L; ++i) upc += (int)pad32(h->hidden[i]) + (i + 1 < h->L ? (int)pad32((int64_t)h->hidden[i] * h->hidden[i + 1]) : 0);
        upc += (int)pad32(h->hidden[h->L - 1]) + 32;
        probe.up_count = upc; probe.act_stride = sum | 1;
        if (fused_smem_floats(probe, K, h->dc, h->dn) * 4 > 200 * 1024) h->fused = false;
    }
    if (h->need_emb) {
        if (!h->fused) {      // the fused step never materialises input_layer or its gradient
            if (dalloc(h, &h->h0, Bm * dK)) return DFM_ERR_CUDA;
            if (dalloc(h, &h->dE, Bm * dK)) return DFM_ERR_CUDA;
        }
        if (dalloc(h, &h->s, Bm * K)) return DFM_ERR_CUDA;
    }
    if (dalloc(h, &h->zacc, Bm)) return DFM_ERR_CUDA;
    if (dalloc(h, &h->logits, Bm)) return DFM_ERR_CUDA;
    if (dalloc(h, &h->dz, Bm)) return DFM_ERR_CUDA;
    h->act[0] = h->h0;
    int64_t max_w = 1, max_n = std::max<int64_t>(dK, 1);
    {
        int in = dK;
        for (int i = 0; i < h->L; ++i) {
            if (dalloc(h, &h->act[i + 1], Bm * h->hidden[i])) return DFM_ERR_CUDA;
            if (dalloc(h, &h->dact[i + 1], Bm * h->hidden[i])) return DFM_ERR_CUDA;
            max_w = std::max<int64_t>(max_w, (int64_t)in * h->hidden[i]);
            max_n = std::max<int64_t>(max_n, h->hidden[i]);
            in = h->hidden[i];
        }
    }
    h->splits = (int)std::min<int64_t>(64, std::max<int64_t>(1, (Bm + 1023) / 1024));
    size_t splitk_elems = (size_t)h->splits * max_w, tc_split_total = 0;
    // tensor-core tower (3xTF32 tcgen05): every hidden width a multiple of 32 and at least one >= 64
    if (h->use_dnn && h->activation == DFM_ACT_RELU && h->L >= 1 && getenv("DFM_NO_TC") == nullptr && prop.major == 10) {
        bool ok = true, big = false;
        for (int i = 0; i < h->L; ++i) { ok = ok && (h->hidden[i] % 32 == 0); big = big || h->hidden[i] >= 64; }
        if (ok && big && tc_setup_once() > 0) {
            h->tc_mlp = true;
            int64_t off_w = 0;
            int in = dK;
            for (int i = 0; i < h->L; ++i) {
                h->tc_off[i] = off_w;
                off_w += 4 * (int64_t)pad32((int64_t)in * h->hidden[i]);     // W hi, W lo, W^T hi, W^T lo
                const int m_tiles = (in + 127) / 128, n_tiles = (h->hidden[i] + 255) / 256;
                h->tc_nz[i] = tc_wgrad_splits(h->max_batch, std::max(1, std::min(128, h->sm_count / std::max(1, m_tiles * n_tiles))));
                // one region per layer: the reduction of layer i's partials runs on the side stream while layer i-1's
                // weight-gradient GEMM already writes its own
                h->splitk_off[i] = tc_split_total; tc_split_total += pad32((int64_t)h->tc_nz[i] * in * h->hidden[i]);
                in = h->hidden[i];
            }
            splitk_elems = std::max(splitk_elems, tc_split_total);
            if (dalloc(h, &h->tc_w, (size_t)off_w)) return DFM_ERR_CUDA;
        }
    }
    if (dalloc(h, &h->splitk, splitk_elems)) return DFM_ERR_CUDA;
    const int64_t chunks = (Bm + h->rows_per_chunk - 1) / h->rows_per_chunk;
    const int64_t nchunks = (Bm + h->num_rows_per_chunk - 1) / h->num_rows_per_chunk;
    if (dalloc(h, &h->colpart, std::max<size_t>((size_t)chunks * max_n, (size_t)nchunks * h->dn * (K + 1)))) return DFM_ERR_CUDA;
    h->head_blocks = (int)std::min<int64_t>(h->sm_count * 8, std::max<int64_t>(1, (Bm + 7) / 8));
    if (dalloc(h, &h->head_part, (size_t)h->head_blocks * 2)) return DFM_ERR_CUDA;
    // fused small-MLP path: every hidden layer <= 32 wide (not a real GEMM)
    if (h->use_dnn && h->activation == DFM_ACT_RELU && h->L >= 1 && h->L <= SM_MAXL && getenv("DFM_NO_SMALL_MLP") == nullptr) {
        bool ok = (h->hidden[0] == 8 || h->hidden[0] == 16 || h->hidden[0] == 32);
        int sum = 0;
        for (int i = 0; i < h->L; ++i) { ok = ok && h->hidden[i] <= SM_MAXH; sum += h->hidden[i]; }
        if (ok) {
            SmallMlpDesc& m = h->sm;
            m.L = h->L; m.D = dK;
            for (int i = 0; i < h->L; ++i) {
                m.H[i] = h->hidden[i];
                for (const DenseT& dt : h->dense) {
                    if (dt.name == "W" + std::to_string(i)) m.off_W[i] = (int)dt.off;
                    if (dt.name == "b" + std::to_string(i)) m.off_b[i] = (int)dt.off;
                }
            }
            for (const DenseT& dt : h->dense) { if (dt.name == "Wo") m.off_Wo = (int)dt.off; if (dt.name == "bo") m.off_bo = (int)dt.off; }
            m.up_begin = m.off_b[0];
            m.up_count = m.off_bo + 32 - m.off_b[0];
            m.act_stride = sum | 1;
            h->small_smem = small_mlp_fwd_smem(m);
            if (h->fused) {
                h->fused_smem = fused_smem_floats(m, K, h->dc, h->dn) * 4;
                if (h->fused_smem > 200 * 1024) FAIL(DFM_ERR_UNSUPPORTED, "internal: fused tile estimate was too small");
                h->small_mlp = true;            // (weights-in-shared-memory tower; selects the small-tower buffers below)
                h->fused_grid = 2 * h->sm_count;    // persistent, two CTAs per SM
                h->n_numacc = h->dn * (K + m.H[0] + 2);
                const size_t g = (size_t)h->fused_grid;
                if (dalloc(h, &h->up_partial, g * m.up_count)) return DFM_ERR_CUDA;
                if (dalloc(h, &h->w0_partial, g * (size_t)dK * m.H[0])) return DFM_ERR_CUDA;
                if (dalloc(h, &h->num_partial, g * (size_t)std::max(h->n_numacc, 1))) return DFM_ERR_CUDA;
                if (dalloc(h, &h->num_scratch, (size_t)std::max(h->n_numacc, 1))) return DFM_ERR_CUDA;
                if (dalloc(h, &h->fused_done, 1)) return DFM_ERR_CUDA;
                CK(cudaMemset(h->fused_done, 0, 4));
                CK(cudaFree(h->head_part)); h->head_part = nullptr;
                if (dalloc(h, &h->head_part, g * 2)) return DFM_ERR_CUDA;
                int rcf = DFM_OK;
                switch (K) {
                    case 4: rcf = fused_set_attr<4>(h); break;
                    case 8: rcf = fused_set_attr<8>(h); break;
                    case 16: rcf = fused_set_attr<16>(h); break;
                    default: rcf = fused_set_attr<32>(h); break;
                }
                if (rcf) return rcf;
                // record-staged variant: the shapes BASELINE.json names (k = 16, first hidden layer 16), unsharded
                const int rs = K + 4 + h->emb_slots * K;
                if (fused_rows_supported(K, m.H[0], h->dc, h->dn) && h->world > 1 && !h->has_bags && h->dropout == 0.f && h->need_emb &&
                    getenv("DFM_NO_FUSED_ROWS") == nullptr) {
                    h->fr_smem_rb = fused_rows_smem_bytes(m, K, h->dc, h->dn, K + 4);
                    if (h->fr_smem_rb <= 227 * 1024) {
                        h->fused_rows_rb = true;
                        CK(fused_rows_set_attr((int)h->fr_smem_rb));
                        if (dalloc(h, &h->once_lk, (size_t)h->max_batch * h->dcs)) return DFM_ERR_CUDA;
                    }
                }
                if (fused_rows_supported(K, m.H[0], h->dc, h->dn) && h->world == 1 && !h->has_bags && h->dropout == 0.f && h->need_emb &&
                    getenv("DFM_NO_FUSED_ROWS") == nullptr) {
                    h->fr_smem = fused_rows_smem_bytes(m, K, h->dc, h->dn, rs);
                    if (h->fr_smem <= 227 * 1024) {
                        h->fused_rows = true;
                        CK(fused_rows_set_attr((int)h->fr_smem));
                        uint64_t slots = 1024;
                        while (slots < (uint64_t)h->R && slots < (1ull << 26)) slots <<= 1;      // 16 MB at most: L2 resident
                        h->claim_mask = (uint32_t)(slots - 1);
                        h->claim_bytes = (size_t)(slots / 4);
                        if (dalloc(h, &h->claim, h->claim_bytes / 4)) return DFM_ERR_CUDA;
                    }
                }
            } else if (h->small_smem <= 200 * 1024) {
                h->small_mlp = true;
                const int tiles = (int)((Bm + SM_TB - 1) / SM_TB);
                h->small_grid = std::min(tiles, 2 * h->sm_count);
                if (dalloc(h, &h->up_partial, (size_t)h->small_grid * m.up_count)) return DFM_ERR_CUDA;
                if (dalloc(h, &h->w0_partial, (size_t)std::min(tiles, 4 * h->sm_count) * dK * m.H[0])) return DFM_ERR_CUDA;
                if (h->head_blocks < h->small_grid) {
                    CK(cudaFree(h->head_part)); h->head_part = nullptr;
                    if (dalloc(h, &h->head_part, (size_t)h->small_grid * 2)) return DFM_ERR_CUDA;
                }
                CK(cudaFuncSetAttribute(small_mlp_fwd_bwd_top_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->small_smem));
                CK(cudaFuncSetAttribute(small_mlp_fwd_bwd_top_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->small_smem));
                CK(cudaFuncSetAttribute(small_mlp_fwd_bwd_top_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->small_smem));
                CK(cudaFuncSetAttribute(small_mlp_bwd_input_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_mlp_bwd_smem<8>(K)));
                CK(cudaFuncSetAttribute(small_mlp_bwd_input_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_mlp_bwd_smem<16>(K)));
                CK(cudaFuncSetAttribute(small_mlp_bwd_input_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_mlp_bwd_smem<32>(K)));
            }
        }
    }
    if (h->use_dnn && h->activation == DFM_ACT_RELU && !h->small_mlp && h->L >= 1 && h->hidden[h->L - 1] % 32 == 0 && h->hidden[h->L - 1] <= 256 &&
        getenv("DFM_NO_FUSED_HEAD") == nullptr) {
        h->fused_head = true;
        h->fused_head_blocks = std::min(h->head_blocks, 2 * h->sm_count);
        if (dalloc(h, &h->head_gpart, (size_t)h->fused_head_blocks * 2 * h->hidden[h->L - 1])) return DFM_ERR_CUDA;
    }
    if (dalloc(h, &h->d_loss, 1)) return DFM_ERR_CUDA;
    if (dalloc(h, &h->d_dzsum, 1)) return DFM_ERR_CUDA;
    if (dalloc(h, &h->d_err, 1)) return DFM_ERR_CUDA;
    CK(cudaMemset(h->d_err, 0, 4));
    {
        int rc = build_replay(h, 1 << 14);
        if (rc) return rc;
    }
    for (auto& s : h->stage) {
        CK(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
        CK(cudaMallocHost(&s.h_loss, 64));
    }
    for (auto& e : h->ph_ev) CK(cudaEventCreate(&e));
    CK(cudaFuncSetAttribute(numeric_grad_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, h->num_rows_per_chunk * (DFM_MAX_NUM + 1) * 4));

    if (h->xchg_pending) {
        // exchange region (xchg.cuh): fixed-capacity segments per (source, owner), rows, dense slots, flags
        XchgDev& x = h->xd;
        x.W = h->world; x.me = h->rank; x.cap = (uint32_t)n; x.rw = K + 4; x.nd1 = (int)((h->n_dense + 1 + 3) / 4 * 4);
        size_t off = 0;
        auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
        for (int par = 0; par < 2; ++par) x.off_ids[par] = take((size_t)x.W * x.cap * 4);
        for (int par = 0; par < 2; ++par) x.off_hdr[par] = take((size_t)MAX_PEERS * 16);
        x.off_grads = take((size_t)x.W * x.cap * x.rw * 4);
        x.off_rows = take((size_t)x.cap * x.rw * 4);
        x.off_dense = take((size_t)x.W * x.nd1 * 4);
        x.off_flags = take((size_t)4 * MAX_PEERS * 4);
        h->xreg_bytes = off;
        CK(cudaMalloc(&h->xreg, off));
        CK(cudaMemset(h->xreg + x.off_hdr[0], 0, off - x.off_hdr[0] > (x.off_grads - x.off_hdr[0]) ? (x.off_grads - x.off_hdr[0]) : 0));
        CK(cudaMemset(h->xreg + x.off_dense, 0, off - x.off_dense));
        if (dalloc(h, &h->x_ticket, 16) || dalloc(h, &h->d_xroute, 1) || dalloc(h, &h->d_nrecv, 4) ||
            dalloc(h, &h->d_dense_total, (size_t)x.nd1) || dalloc(h, &h->d_loss_part, 4)) return DFM_ERR_CUDA;
        CK(cudaMemset(h->x_ticket, 0, 16 * 4));
        CK(cudaEventCreateWithFlags(&h->ev_xpf_fork, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_xpf_done, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_xfork, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_xjoin, cudaEventDisableTiming));
    }
    // optimizer slot initial values (Adagrad / FTRL accumulators start at init_acc)
    auto init_acc = [&](const dfm_optimizer& o) { return (o.kind == DFM_OPT_ADAGRAD || o.kind == DFM_OPT_FTRL || o.kind == DFM_OPT_RMSPROP) ? o.init_acc : 0.f; };
    if (init_acc(h->od) != 0.f) {
        if (h->need_emb && R)
            fill_strided_kernel<<<cdiv((int64_t)R * K, 256), 256, 0, h->stream>>>(h->tb.rec + h->tb.s1_off, R, K, h->tb.stride, init_acc(h->od));
        if (h->n_deep) fill_strided_kernel<<<cdiv(h->n_deep, 256), 256, 0, h->stream>>>(h->ds1, 1, (int)h->n_deep, 0, init_acc(h->od));
    }
    if (init_acc(h->ol) != 0.f) {
        if (R) fill_strided_kernel<<<cdiv((int64_t)R, 256), 256, 0, h->stream>>>(h->tb.rec + h->tb.lin_off + 1, R, 1, h->tb.stride, init_acc(h->ol));
        if (h->n_dense > h->n_deep)
            fill_strided_kernel<<<cdiv(h->n_dense - h->n_deep, 256), 256, 0, h->stream>>>(h->ds1 + h->n_deep, 1, (int)(h->n_dense - h->n_deep), 0, init_acc(h->ol));
    }
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    return DFM_OK;
}

extern "C" int dfm_create(const dfm_config* cfg, dfm_handle** out) {
    g_create_error.clear();
    if (!cfg || !out) { g_create_error = "null argument"; return DFM_ERR_INVALID_ARG; }
    *out = nullptr;
    dfm_handle* h = new dfm_handle();
    int rc = create_impl(cfg, h);
    if (rc != DFM_OK) {
        g_create_error = h->err;
        free_all(h);
        return rc;
    }
    *out = h;
    return DFM_OK;
}

// ------------------------------------------------------------------------------ tensor access
struct TensorRef {
    float* base; int64_t rows, row_elems, pitch;   // pitch in floats
};

static bool resolve(dfm_handle* h, const std::string& full, TensorRef& t) {
    std::string name = full, slot;
    size_t p = full.find('/');
    if (p != std::string::npos) { name = full.substr(0, p); slot = full.substr(p + 1); }
    auto slot_index = [&](int kind) -> int {
        if (slot.empty()) return 0;
        if (kind == DFM_OPT_ADAM) return slot == "m" ? 1 : slot == "v" ? 2 : -1;
        if (kind == DFM_OPT_ADAGRAD) return slot == "acc" ? 1 : -1;
        if (kind == DFM_OPT_FTRL) return slot == "acc" ? 1 : slot == "lin" ? 2 : -1;
        if (kind == DFM_OPT_RMSPROP) return slot == "rms" ? 1 : slot == "mom" ? 2 : -1;
        return -1;
    };
    if (name == "emb") {
        if (!h->need_emb) return false;
        int si = slot_index(h->od.kind);
        if (si < 0) return false;
        t = {h->tb.rec + (si == 0 ? 0 : si == 1 ? h->tb.s1_off : h->tb.s2_off), (int64_t)h->R_loc, h->K, h->tb.stride};
        return true;
    }
    if (name == "lin") {
        if (!h->use_linear) return false;
        int si = slot_index(h->ol.kind);
        if (si < 0) return false;
        t = {h->tb.rec + h->tb.lin_off + si, (int64_t)h->R_loc, 1, h->tb.stride};
        return true;
    }
    for (const DenseT& dt : h->dense) {
        if (dt.name != name) continue;
        bool deep = dt.off < h->n_deep;
        int si = slot_index(deep ? h->od.kind : h->ol.kind);
        if (si < 0) return false;
        float* b = si == 0 ? h->dw : si == 1 ? h->ds1 : h->ds2;
        t = {b + dt.off, dt.rows, dt.cols, dt.cols};
        return true;
    }
    return false;
}

extern "C" int dfm_tensor_rows(dfm_handle* h, const char* name, int64_t* rows, int64_t* row_elems) {
    if (!h || !name) return DFM_ERR_INVALID_ARG;
    TensorRef t;
    if (!resolve(h, name, t)) FAIL(DFM_ERR_NOT_FOUND, std::string("no tensor named ") + name);
    if (rows) *rows = t.rows;
    if (row_elems) *row_elems = t.row_elems;
    return DFM_OK;
}

extern "C" int dfm_flush(dfm_handle* h, void* stream);

extern "C" int dfm_set_tensor(dfm_handle* h, const char* name, int64_t row_begin, int64_t n_rows, const float* src) {
    if (!h || !name || !src) return DFM_ERR_INVALID_ARG;
    TensorRef t;
    if (!resolve(h, name, t)) FAIL(DFM_ERR_NOT_FOUND, std::string("no tensor named ") + name);
    if (row_begin < 0 || n_rows < 0 || row_begin + n_rows > t.rows) FAIL(DFM_ERR_INVALID_ARG, "row range out of bounds");
    CK(cudaSetDevice(h->device));
    int rc = dfm_flush(h, h->stream);   // rows must be current before they are overwritten piecewise
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->stream));
    if (n_rows)
        CK(cudaMemcpy2D(t.base + row_begin * t.pitch, t.pitch * 4, src, t.row_elems * 4, t.row_elems * 4, n_rows, cudaMemcpyHostToDevice));
    return DFM_OK;
}

extern "C" int dfm_get_tensor(dfm_handle* h, const char* name, int64_t row_begin, int64_t n_rows, float* dst) {
    if (!h || !name || !dst) return DFM_ERR_INVALID_ARG;
    TensorRef t;
    if (!resolve(h, name, t)) FAIL(DFM_ERR_NOT_FOUND, std::string("no tensor named ") + name);
    if (row_begin < 0 || n_rows < 0 || row_begin + n_rows > t.rows) FAIL(DFM_ERR_INVALID_ARG, "row range out of bounds");
    CK(cudaSetDevice(h->device));
    int rc = dfm_flush(h, h->stream);
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->stream));
    if (n_rows)
        CK(cudaMemcpy2D(dst, t.row_elems * 4, t.base + row_begin * t.pitch, t.pitch * 4, t.row_elems * 4, n_rows, cudaMemcpyDeviceToHost));
    return DFM_OK;
}

extern "C" int dfm_init_random(dfm_handle* h, uint64_t seed) {
    if (!h) return DFM_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    if (h->need_emb && h->R_loc) {
        uint64_t tot = h->R_loc * (uint64_t)h->K;
        init_trunc_normal_kernel<<<cdiv((int64_t)tot, 256), 256, 0, st>>>(h->tb.rec, h->R_loc, h->K, h->tb.stride,
                                                                          1.0f / sqrtf((float)h->K), seed * 0x9E3779B97F4A7C15ULL + 1,
                                                                          (uint64_t)h->world, (uint64_t)(h->world > 1 ? h->rank : 0));
    }
    int idx = 0;
    for (const DenseT& dt : h->dense) {
        ++idx;
        bool kernel = dt.name[0] == 'W' || dt.name == "num_emb";
        if (!kernel) continue;   // biases, linear weights: zeros
        float fan_in = (float)dt.rows, fan_out = (float)dt.cols;
        float lim = sqrtf(6.0f / (fan_in + fan_out));
        init_uniform_kernel<<<cdiv(dt.rows * dt.cols, 256), 256, 0, st>>>(h->dw + dt.off, dt.rows * dt.cols, lim, seed * 0xD1B54A32D192ED03ULL + idx);
    }
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    return DFM_OK;
}

// -------------------------------------------------------------------------------- step pieces
static BatchPtrs make_ptrs(const dfm_handle* h, const dfm_raw_batch* b) {
    BatchPtrs bp{};
    for (int f = 0; f < h->dc + h->n_src; ++f) {
        bp.cat[f] = b->cat_data ? b->cat_data[f] : nullptr;
        bp.off[f] = b->cat_offsets ? b->cat_offsets[f] : nullptr;
    }
    for (int j = 0; j < h->dn; ++j) bp.num[j] = b->num_data ? b->num_data[j] : nullptr;
    bp.labels = b->labels;
    return bp;
}

// identity of a batch for the prefetch paths: its first raw column pointer (a crossed column has none of its own)
static const void* batch_tag(const dfm_handle* h, const void* const* cat) {
    for (int f = 0; f < h->dc + h->n_src; ++f)
        if (h->cols[f].kind != DFM_COL_CROSSED) return cat[f];
    return nullptr;
}

static int check_batch(dfm_handle* h, const dfm_raw_batch* b, bool need_labels) {
    if (!b) FAIL(DFM_ERR_INVALID_ARG, "null batch");
    if (b->batch_size <= 0 || b->batch_size > h->max_batch) FAIL(DFM_ERR_INVALID_ARG, "batch_size outside (0, max_batch]");
    if (h->dc && !b->cat_data) FAIL(DFM_ERR_INVALID_ARG, "cat_data is null");
    for (int f = 0; f < h->dc + h->n_src; ++f) {
        if (h->cols[f].kind == DFM_COL_CROSSED) continue;           // computed from its source columns
        if (!b->cat_data[f]) FAIL(DFM_ERR_INVALID_ARG, "missing feature column: " + h->col_names[f]);
        if (h->cols[f].dtype == DFM_STRING && (!b->cat_offsets || !b->cat_offsets[f]))
            FAIL(DFM_ERR_INVALID_ARG, "missing string offsets for column: " + h->col_names[f]);
    }
    if (h->dn && !b->num_data) FAIL(DFM_ERR_INVALID_ARG, "num_data is null");
    for (int j = 0; j < h->dn; ++j)
        if (!b->num_data[j]) FAIL(DFM_ERR_INVALID_ARG, "missing numeric column");
    if (need_labels && !b->labels) FAIL(DFM_ERR_INVALID_ARG, "labels are required for a train step");
    return DFM_OK;
}

struct Phase {
    dfm_handle* h; cudaStream_t st; int idx = 0;
    Phase(dfm_handle* h_, cudaStream_t s) : h(h_), st(s) { if (h->profiling) cudaEventRecord(h->ph_ev[0], st); }
    void next() { ++idx; if (h->profiling && idx <= dfm_handle::NPH) cudaEventRecord(h->ph_ev[idx], st); }
};

template <int K>
static void launch_transform(dfm_handle* h, const BatchPtrs& bp, int B, bool with_keys, int32_t* ids_out, cudaStream_t st,
                             bool with_claim = false) {
    if (h->dc == 0) return;
    (h->has_vtab ? (h->has_cross ? transform_kernel<32, true, true> : transform_kernel<32, false, true>)
                 : (h->has_cross ? transform_kernel<32, true> : transform_kernel<32, false>))<<<cdiv(B, 32), 256, (size_t)32 * h->dcs * 4, st>>>(
        bp, h->d_cols, h->d_bounds, h->d_voc_bytes, h->d_voc_offs, B, h->dcs, h->has_bags ? h->d_slot_col : nullptr,
        h->has_bags ? h->d_slot_j : nullptr, h->d_row_off, (uint32_t)h->R, ids_out,
        with_keys ? h->ws.keys[with_claim ? 1 : 0] : nullptr, with_keys ? h->ws.vals[with_claim ? 1 : 0] : nullptr, h->d_err,
        with_keys && h->n_tiny ? h->d_key_slot : nullptr, h->n_big, with_claim ? h->claim : nullptr, h->claim_mask);
    h->launches++;
}

// dense reduction + optimizer for the tiny-vocabulary columns (no-op when the model has none)
template <int K>
static int tiny_update(dfm_handle* h, int B, const OptDev& od, const OptDev& ol, int64_t t, cudaStream_t st) {
    if (!h->n_tiny || B <= 0) return DFM_OK;
    const int blocks = (B + TINY_SPB - 1) / TINY_SPB;
    constexpr int G = 32 / (K / 4);                                   // columns per block
    const size_t smem = (size_t)8 * h->tiny_group_rows * (K + 4) * 4;
    static size_t smem_attr = 48 * 1024;
    if (smem > smem_attr) { CK(cudaFuncSetAttribute(tiny_reduce_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); smem_attr = smem; }
    tiny_reduce_kernel<K><<<dim3(blocks, (h->n_tiny + G - 1) / G), 256, smem, st>>>(h->ids, B, h->dcs, h->d_tiny_slot, h->d_trow0, h->n_tiny, h->n_tiny_rows,
                                                     h->need_emb ? h->dE : nullptr, h->dz, (h->dc + h->dn) * K, h->tiny_partial);
    tiny_update_kernel<K><<<cdiv((int64_t)h->n_tiny_rows * 32, 256), 256, 0, st>>>(h->tiny_partial, blocks, h->d_trow_grow, h->n_tiny_rows, h->tb, h->emb_slots,
                                                                                   od, ol, (bool)h->need_emb, (bool)h->use_linear, (int)t, make_rr(h, t - 1));
    h->launches += 2;
    CK(cudaGetLastError());
    return DFM_OK;
}

template <int K>
static void launch_gather(dfm_handle* h, const BatchPtrs& bp, int B, cudaStream_t st, const float* rowbuf = nullptr, int64_t upto = -1) {
    float* num_emb = nullptr; float* num_lin = nullptr; float* bias = nullptr;
    for (const DenseT& dt : h->dense) {
        if (dt.name == "num_emb") num_emb = h->dw + dt.off;
        if (dt.name == "num_lin") num_lin = h->dw + dt.off;
        if (dt.name == "bias") bias = h->dw + dt.off;
    }
    unsigned grid = std::min<unsigned>(cdiv(B, 8), (unsigned)h->sm_count * 16);
    auto kern = h->has_bags ? gather_fm_kernel<K, true> : gather_fm_kernel<K, false>;
    kern<<<grid, 256, 0, st>>>(h->ids, B, h->dc, h->dn, h->dcs, h->has_bags ? h->d_field_slot0 : nullptr,
                                              h->has_bags ? h->inv_cnt : nullptr, h->d_row_off, h->tb, bp,
                                              num_emb, num_lin, bias, h->use_linear, h->use_mf, h->need_emb, h->h0, h->s, h->zacc,
                                              rowbuf ? h->uidx : nullptr, rowbuf, K + 4, make_rr(h, rowbuf ? -1 : upto),
                                              make_opt(h->od, 0.f), make_opt(h->ol, 0.f));
    h->launches++;
}

static const DenseT* find_dense(const dfm_handle* h, const std::string& nm) {
    for (const DenseT& dt : h->dense) if (dt.name == nm) return &dt;
    return nullptr;
}

static bool vec_ok(const void* a, int lda, const void* b, int ldb, const void* c, int ldc) {
    auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    return al(a) && al(b) && al(c) && lda % 4 == 0 && ldb % 4 == 0 && ldc % 4 == 0;
}

template <bool A_KC, bool B_KC, int EPI>
static void launch_sgemm(dfm_handle* h, const float* A, int lda, const float* Bm, int ldb, float* C, int ldc, int M, int N, int Kd,
                         int splits, int k_chunk, const EpiArgs& ep, cudaStream_t st) {
    dim3 grid(cdiv(N, 128), cdiv(M, 128), splits);
    size_t stride = (size_t)M * ldc;
    if (vec_ok(A, lda, Bm, ldb, C, ldc) && k_chunk % 4 == 0)
        sgemm_kernel<A_KC, B_KC, EPI, true><<<grid, 256, 0, st>>>(A, lda, Bm, ldb, C, ldc, M, N, Kd, k_chunk, stride, ep);
    else
        sgemm_kernel<A_KC, B_KC, EPI, false><<<grid, 256, 0, st>>>(A, lda, Bm, ldb, C, ldc, M, N, Kd, k_chunk, stride, ep);
    h->launches++;
}

// out[N] = sum_b w[b] * X[b, :]  (deterministic two-level)
static void launch_colsum(dfm_handle* h, const float* X, int ldx, const float* w, int B, int N, float* out, cudaStream_t st) {
    int chunks = (int)cdiv(B, h->rows_per_chunk);
    colsum_partial_kernel<<<dim3(cdiv(N, 32), chunks), 256, 0, st>>>(X, ldx, w, B, N, h->rows_per_chunk, h->colpart);
    reduce_partials_kernel<<<cdiv(N, 256), 256, 0, st>>>(h->colpart, chunks, (size_t)N, N, out);
    h->launches += 2;
}

// (Re)builds the alpha_t sequence and the replay tables of both optimizer groups for steps < cap.
static int build_replay_group(dfm_handle* h, ReplayHost& r, const dfm_optimizer& o, int64_t cap) {
    free_replay(r);
    r = ReplayHost{};
    r.adam = o.kind == DFM_OPT_ADAM;
    if (!r.adam) return DFM_OK;
    const double b1 = (double)o.beta1, b2 = (double)o.beta2, q = sqrt(b2);
    // closed form: b1^H < 1e-10 within 4096 terms and the series in (1 - q^i) converging fast enough for 4 terms
    if (b1 > 0.0 && b1 < 1.0 && b2 > 0.0 && b2 < 1.0 && getenv("DFM_REPLAY_LOOP") == nullptr) {
        const double hh = ceil(log(1e-10) / log(b1));
        if (hh <= 4096.0 && (1.0 - q) / (1.0 - b1) <= 0.01) { r.closed = true; r.H = std::max(1, (int)hh); }
    }
    const size_t n = (size_t)cap + r.H + 1;
    r.alpha.assign(n, 0.f);
    float p1 = 1.f, p2 = 1.f;                       // TF's float32 beta1_power / beta2_power
    for (size_t t = 1; t < n; ++t) {
        p1 *= o.beta1; p2 *= o.beta2;
        r.alpha[t] = o.lr * sqrtf(1.0f - p2) / (1.0f - p1);
    }
    CK(cudaMalloc(&r.d_alpha, n * 4));
    CK(cudaMemcpy(r.d_alpha, r.alpha.data(), n * 4, cudaMemcpyHostToDevice));
    if (r.closed) {
        CK(cudaMalloc(&r.d_T4, (size_t)cap * sizeof(float4)));
        CK(cudaMalloc(&r.d_U, (size_t)cap * 12 * 4));
        std::vector<float4> pq(REPLAY_PQ_N);
        for (int g = 0; g < REPLAY_PQ_N; ++g) pq[g] = make_float4((float)pow(b1, g), (float)pow(b2, g), (float)(-expm1((double)g * log(q))), 0.f);
        CK(cudaMalloc(&r.d_PQ, sizeof(float4) * REPLAY_PQ_N));
        CK(cudaMemcpy(r.d_PQ, pq.data(), sizeof(float4) * REPLAY_PQ_N, cudaMemcpyHostToDevice));
        replay_tables_kernel<<<cdiv(cap, 128), 128, 0, h->stream>>>(r.d_alpha, (int)cap, r.H, b1, q, r.d_T4, r.d_U);
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaGetLastError());
    }
    r.tab.T4 = r.d_T4; r.tab.U = r.d_U; r.tab.alpha = r.d_alpha; r.tab.PQ = r.d_PQ;
    r.tab.l2b1 = (float)log2(b1); r.tab.l2b2 = (float)log2(b2); r.tab.lnq = (float)log(q);
    r.tab.closed = r.closed ? 1 : 0;
    return DFM_OK;
}

static int build_replay(dfm_handle* h, int64_t cap) {
    int rc = build_replay_group(h, h->rp_d, h->od, cap);
    if (rc) return rc;
    if ((rc = build_replay_group(h, h->rp_l, h->ol, cap))) return rc;
    h->rp_same = h->rp_d.adam && h->rp_l.adam && h->od.lr == h->ol.lr && h->od.beta1 == h->ol.beta1 && h->od.beta2 == h->ol.beta2 &&
                 h->od.eps == h->ol.eps;
    h->alpha_cap = cap;
    return DFM_OK;
}

static int ensure_alpha(dfm_handle* h, int64_t t) {
    if (t + 2 < h->alpha_cap) return DFM_OK;
    int64_t ncap = h->alpha_cap * 2;
    while (t + 2 >= ncap) ncap *= 2;
    // rare (capacity doubles): kernels of earlier steps may still read the tables on the caller's stream or on the
    // side stream, so wait for the whole device before they move
    CK(cudaDeviceSynchronize());
    return build_replay(h, ncap);
}

static bool any_adam(const dfm_handle* h) {
    return (h->need_emb && h->od.kind == DFM_OPT_ADAM) || (h->use_linear && h->ol.kind == DFM_OPT_ADAM);
}

static float alpha_at(const ReplayHost& r, int64_t t) { return (r.adam && t >= 0 && (size_t)t < r.alpha.size()) ? r.alpha[(size_t)t] : 0.f; }

// the replay descriptor of a kernel that must see the rows as of step `upto` (< 0 or no Adam group: nothing to replay)
static RowReplay make_rr(const dfm_handle* h, int64_t upto) {
    RowReplay rr{};
    rr.rd = h->rp_d.tab; rr.rl = h->rp_l.tab;
    rr.emb_adam = (h->need_emb && h->od.kind == DFM_OPT_ADAM) ? 1 : 0;
    rr.lin_adam = (h->use_linear && h->ol.kind == DFM_OPT_ADAM) ? 1 : 0;
    rr.same = h->rp_same ? 1 : 0;
    rr.upto = (rr.emb_adam || rr.lin_adam) ? (int)upto : -1;
    if (upto <= 0) rr.upto = -1;       // step 0: nothing has ever been applied
    return rr;
}

template <int K>
static int flush_impl(dfm_handle* h, cudaStream_t st) {
    if (!any_adam(h) || h->flushed_step == h->step || h->R_loc == 0) { h->flushed_step = h->step; return DFM_OK; }
    OptDev od = make_opt(h->od, alpha_at(h->rp_d, h->step)), ol = make_opt(h->ol, alpha_at(h->rp_l, h->step));
    unsigned grid = (unsigned)std::min<uint64_t>((h->R_loc + (256 / (K / 4)) - 1) / (256 / (K / 4)), (uint64_t)h->sm_count * 16);
    catchup_all_kernel<K><<<grid, 256, 0, st>>>(h->tb, h->R_loc, make_rr(h, h->step), od, ol, (bool)h->need_emb);
    h->launches++;
    CK(cudaGetLastError());
    h->flushed_step = h->step;
    return DFM_OK;
}

static void set_dropout(const dfm_handle* h, EpiArgs& ep, bool train, int layer) {
    if (train && h->dropout > 0.f) {
        ep.drop_keep = 1.f - h->dropout; ep.drop_inv = 1.f / (1.f - h->dropout);
        ep.drop_key = dfm_drop_key(h->dropout_seed, (uint64_t)(h->step + 1), (uint64_t)layer);
        ep.drop_row0 = (int64_t)h->rank * h->max_batch;
    }
}

template <int K>
static int forward_impl(dfm_handle* h, const BatchPtrs& bp, int B, cudaStream_t st, const float* labels, float scale,
                        float* logits_out, Phase* ph, const float* rowbuf = nullptr, int64_t upto = -1) {
    const int d = h->dc + h->dn, dK = d * K;
    launch_gather<K>(h, bp, B, st, rowbuf, upto);
    if (ph) ph->next();
    const float* hL = nullptr; int H = 0;
    const DenseT* Wo = find_dense(h, "Wo"); const DenseT* bo = find_dense(h, "bo");
    if (h->small_mlp) {
        const float* za = (h->use_linear || h->use_mf) ? h->zacc : nullptr;
        const int train = labels ? 1 : 0;
        const int grid = std::min((B + SM_TB - 1) / SM_TB, h->small_grid);
        SmallMlpDesc smd = h->sm;
        if (train && h->dropout > 0.f) {
            smd.drop_keep = 1.f - h->dropout; smd.drop_inv = 1.f / (1.f - h->dropout);
            smd.drop_seed = h->dropout_seed; smd.drop_step = (uint64_t)(h->step + 1); smd.drop_row0 = (int64_t)h->rank * h->max_batch;
        }
#define SMALL_FWD(HH) small_mlp_fwd_bwd_top_kernel<HH><<<grid, 256, h->small_smem, st>>>(smd, h->dw, h->h0, za, labels, B, scale, train, \
            h->logits, logits_out, h->dz, h->dact[1], h->up_partial, h->head_part)
        if (h->sm.H[0] == 8) SMALL_FWD(8); else if (h->sm.H[0] == 16) SMALL_FWD(16); else SMALL_FWD(32);
#undef SMALL_FWD
        h->launches++;
        if (ph) { ph->next(); }
        return DFM_OK;
    }
    if (h->use_dnn && h->tc_mlp) {
        int in = dK;
        for (int i = 0; i < h->L; ++i) {
            const DenseT* W = find_dense(h, "W" + std::to_string(i));
            const DenseT* b = find_dense(h, "b" + std::to_string(i));
            const int out = h->hidden[i];
            const int64_t wsz = pad32((int64_t)in * out);
            // tc_w layout per layer: [W^T hi | W^T lo | W hi | W lo], each pad32(in*out) floats
            float* wt = h->tc_w + h->tc_off[i];
            float* wt_lo = tc_presplit() ? wt + wsz : nullptr;
            // forward needs W^T [out, in] (K-major B operand).  The weights are split into tf32 hi/lo ONCE here (the
            // persistent GEMM is bound by shared-memory bandwidth: splitting the weight tile again in every CTA costs
            // 24 KB of shared-memory traffic per k-block against 8 KB more TMA traffic for the ready-made lo tile);
            // the activations are split in the kernel.
            tc::split_tf32_transpose_kernel<<<dim3(cdiv(out, 32), cdiv(in, 32)), dim3(32, 8), 0, st>>>(h->dw + W->off, in, out, wt, wt_lo);
            h->launches += 1;
            EpiArgs ep{}; ep.bias = h->dw + b->off;
            set_dropout(h, ep, labels != nullptr, i);
            int rc = tc_gemm_kmajor(h, h->act[i], nullptr, in, wt, wt_lo, in, h->act[i + 1], out, B, out, in, EPI_BIAS_RELU, ep, st);
            if (rc) return rc;
            in = out;
        }
        hL = h->act[h->L]; H = in;
    } else if (h->use_dnn) {
        int in = dK;
        for (int i = 0; i < h->L; ++i) {
            const DenseT* W = find_dense(h, "W" + std::to_string(i));
            const DenseT* b = find_dense(h, "b" + std::to_string(i));
            EpiArgs ep{}; ep.bias = h->dw + b->off; ep.act_kind = h->activation;
            set_dropout(h, ep, labels != nullptr, i);
            launch_sgemm<true, false, EPI_BIAS_RELU>(h, h->act[i], in, h->dw + W->off, h->hidden[i], h->act[i + 1], h->hidden[i], B,
                                                     h->hidden[i], in, 1, (in + 15) / 16 * 16, ep, st);
            in = h->hidden[i];
        }
        hL = h->act[h->L]; H = in;
    }
    if (ph) ph->next();
    const float* za = (h->use_linear || h->use_mf) ? h->zacc : nullptr;
    if (h->fused_head && labels) {
        const int grid = std::min(h->fused_head_blocks, (B + 7) / 8);
#define HEAD_BWD(NHH) head_bwd_kernel<NHH><<<grid, 256, 0, st>>>(za, hL, h->dw + Wo->off, h->dw + bo->off, labels, B, scale, h->logits, logits_out, \
                                                             h->dz, h->dact[h->L], h->head_part, h->head_gpart, h->dropout > 0.f ? 1.f / (1.f - h->dropout) : 1.f)
        switch (H / 32) {
            case 1: HEAD_BWD(1); break; case 2: HEAD_BWD(2); break; case 3: HEAD_BWD(3); break; case 4: HEAD_BWD(4); break;
            case 5: HEAD_BWD(5); break; case 6: HEAD_BWD(6); break; case 7: HEAD_BWD(7); break; default: HEAD_BWD(8); break;
        }
#undef HEAD_BWD
        h->launches++;
        return DFM_OK;
    }
    head_kernel<<<std::min(h->head_blocks, (B + 7) / 8), 256, 0, st>>>(za, hL, H, Wo ? h->dw + Wo->off : nullptr,
                                                bo ? h->dw + bo->off : nullptr, labels, B, scale, h->logits, logits_out, h->dz, h->head_part);
    h->launches++;
    return DFM_OK;
}

// sort the (key, payload) pairs in ws.keys[0]/vals[0] and derive unique rows / pieces.
// Default: one-sweep radix sort (one launch per 8-bit digit) + single-pass segment builder; n_dev != nullptr: the pair
// count lives in device memory (n is then its upper bound).  DFM_OLD_SORT=1: the multi-launch sort / scan kernels.
static int build_segments(dfm_handle* h, SegWS& ws, int64_t n, uint32_t limit, int bits, cudaStream_t st, Phase* ph,
                          const uint32_t* n_dev = nullptr) {
    static const bool old_sort = getenv("DFM_OLD_SORT") != nullptr;
    ws.cur = 0;
    if (old_sort && !n_dev && !ws.pos_row) {
        if (n > 0) ws.cur = prims::radix_sort_pairs(ws.keys, ws.vals, n, bits, ws.sort_temp, st, &h->launches);
        if (ph) ph->next();
        if (n > 0) {
            seg_flag_kernel<<<cdiv(n, 256), 256, 0, st>>>(ws.skeys(), n, limit, ws.flags, ws.seg_cnt);
            h->launches++;
            prims::exclusive_scan_u64(reinterpret_cast<const uint64_t*>(ws.flags), reinterpret_cast<uint64_t*>(ws.flags), n, ws.scan_temp,
                                      reinterpret_cast<uint64_t*>(ws.seg_total), st, &h->launches);
            seg_fill_kernel<<<cdiv(n, 256), 256, 0, st>>>(ws.skeys(), ws.svals(), n, limit, ws.flags, ws.seg_total, ws.seg_cnt, ws.row_start,
                                                          ws.row_piece0, ws.piece_start, ws.urow, ws.uval);
            h->launches++;
        } else {
            CK(cudaMemsetAsync(ws.seg_cnt, 0, sizeof(SegCounts), st));
        }
        if (ph) ph->next();
        return DFM_OK;
    }
    static const bool small_ok = getenv("DFM_NO_SMALL_SEGMENTS") == nullptr;
    if (small_ok && !n_dev && n <= SS_MAX) {         // small batches: sort + segments in one single-CTA launch
        int m = 64;
        while (m < n) m <<= 1;
        static bool attr_set = false;
        if (!attr_set) { CK(cudaFuncSetAttribute(small_segments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SS_MAX * 12)); attr_set = true; }
        small_segments_kernel<<<1, SS_THREADS, (size_t)m * 12, st>>>(ws.keys[0], ws.vals[0], (int)n, m, limit, ws.seg_cnt, ws.row_start, ws.row_piece0,
                                                                     ws.piece_start, ws.urow, ws.uval, ws.pos_row);
        h->launches++;
        if (ph) { ph->next(); ph->next(); }
        CK(cudaGetLastError());
        return DFM_OK;
    }
    if (n > 0) ws.cur = prims::onesweep_sort_pairs(ws.keys, ws.vals, n, n_dev, bits, ws.sort_temp, st, &h->launches);
    if (ph) ph->next();
    const int64_t tiles = std::max<int64_t>((n + SB_TILE - 1) / SB_TILE, 1);
    CK(cudaMemsetAsync(ws.seg_total, 0, 8, st));                          // ticket of the count kernel
    seg_count_kernel<<<(unsigned)tiles, 256, 0, st>>>(ws.skeys(), n, n_dev, limit, ws.flags, reinterpret_cast<unsigned int*>(ws.seg_total), ws.seg_cnt,
                                                      ws.row_start, ws.row_piece0, ws.piece_start);
    seg_fill_kernel2<<<(unsigned)tiles, 256, 0, st>>>(ws.skeys(), ws.svals(), n, n_dev, limit, ws.flags, ws.row_start, ws.row_piece0, ws.piece_start,
                                                      ws.urow, ws.uval, ws.pos_row);
    h->launches += 2;
    if (ph) ph->next();
    CK(cudaGetLastError());
    return DFM_OK;
}

// loss reduction + backward through the tower + numeric-feature gradients -> h->dg, h->dE
template <int K>
static int tower_backward(dfm_handle* h, const BatchPtrs& bp, int B, float scale, float* loss_out, cudaStream_t st, Phase* ph,
                          cudaStream_t aux = nullptr) {
    const int dc = h->dc, d = dc + h->dn, dK = d * K;
    // aux: side stream for the small reductions (split-K partials, bias column sums) of the tensor-core tower: they
    // depend only on the kernel just issued and fit beside the GEMM CTAs, so they leave the critical path
    if (!aux || !h->tc_mlp) aux = st;
    auto fork = [&]() -> cudaError_t {
        if (aux == st) return cudaSuccess;
        cudaError_t e = cudaEventRecord(h->ev_aux_fork, st);
        return e ? e : cudaStreamWaitEvent(aux, h->ev_aux_fork, 0);
    };
    const DenseT* bo = find_dense(h, "bo"); const DenseT* bias = find_dense(h, "bias");
    const int small_blocks = std::min((B + SM_TB - 1) / SM_TB, h->small_grid);
    const int head_blocks = h->small_mlp ? small_blocks : std::min(h->fused_head ? h->fused_head_blocks : h->head_blocks, (B + 7) / 8);
    head_final_kernel<<<1, 256, 0, st>>>(h->head_part, head_blocks, scale, h->d_loss, h->d_dzsum, loss_out,
                                         (bo && !h->small_mlp) ? h->dg + bo->off : nullptr, bias ? h->dg + bias->off : nullptr);
    h->launches++;
    if (ph) ph->next();
    // backward through the tower
    if (h->small_mlp) {
        const SmallMlpDesc& m = h->sm;
        const int tiles = (B + SM_TB - 1) / SM_TB;
        reduce_partials_kernel<<<cdiv(m.up_count, 256), 256, 0, st>>>(h->up_partial, small_blocks, (size_t)m.up_count, m.up_count, h->dg + m.up_begin);
        const int chunks = (int)cdiv(dK, SM_BC);
        const int groups = std::max(1, std::min(tiles, (4 * h->sm_count + chunks - 1) / chunks));
        dim3 grid(groups, chunks);
        const float* sv = h->use_mf ? h->s : nullptr;
#define SMALL_BWD(HH) small_mlp_bwd_input_kernel<HH><<<grid, 256, small_mlp_bwd_smem<HH>(K), st>>>(h->dw + m.off_W[0], h->h0, h->dact[1], h->dz, sv, K, B, dK, h->dE, h->w0_partial)
        if (m.H[0] == 8) SMALL_BWD(8); else if (m.H[0] == 16) SMALL_BWD(16); else SMALL_BWD(32);
#undef SMALL_BWD
        reduce_partials_kernel<<<cdiv((int64_t)dK * m.H[0], 256), 256, 0, st>>>(h->w0_partial, groups, (size_t)dK * m.H[0], (int64_t)dK * m.H[0], h->dg + m.off_W[0]);
        h->launches += 3;
    } else if (h->use_dnn) {
        const DenseT* Wo = find_dense(h, "Wo");
        const int L = h->L;
        const float* hL = h->act[L];
        const int H = L ? h->hidden[L - 1] : dK;
        if (h->fused_head) {   // head_bwd_kernel already produced dh_L', gWo and gb_L partials
            const DenseT* bL = find_dense(h, "b" + std::to_string(L - 1));
            CK(fork());
            reduce_partials_kernel<<<cdiv(H, 256), 256, 0, aux>>>(h->head_gpart, head_blocks, (size_t)2 * H, H, h->dg + Wo->off);
            reduce_partials_kernel<<<cdiv(H, 256), 256, 0, aux>>>(h->head_gpart + H, head_blocks, (size_t)2 * H, H, h->dg + bL->off);
            h->launches += 2;
        } else {
            launch_colsum(h, hL, H, h->dz, B, H, h->dg + Wo->off, st);   // gWo = h_L^T dz
        }
        if (L == 0) {
            dh_last_kernel<<<cdiv((int64_t)B * H, 256), 256, 0, st>>>(nullptr, h->dw + Wo->off, h->dz, (int64_t)B * H, H, h->dE, 1.f);
            h->launches++;
            if (h->use_mf) {
                de_fm_kernel<<<cdiv((int64_t)B * dK, 256), 256, 0, st>>>(h->h0, h->s, h->dz, (int64_t)B * dK, dK, K, h->dE, 1);
                h->launches++;
            }
        } else {
            if (!h->fused_head) {
                dh_last_kernel<<<cdiv((int64_t)B * H, 256), 256, 0, st>>>(hL, h->dw + Wo->off, h->dz, (int64_t)B * H, H, h->dact[L],
                                                                          h->dropout > 0.f ? 1.f / (1.f - h->dropout) : 1.f, h->activation);
                h->launches++;
            }
            const int splits = std::max(1, std::min(h->splits, (B + 1023) / 1024));
            const int k_chunk = ((B + splits - 1) / splits + 15) / 16 * 16;
            const int nsplit = (B + k_chunk - 1) / k_chunk;
            for (int i = L - 1; i >= 0; --i) {
                const int in = i ? h->hidden[i - 1] : dK, out = h->hidden[i];
                const DenseT* W = find_dense(h, "W" + std::to_string(i));
                const DenseT* b = find_dense(h, "b" + std::to_string(i));
                // gW_i [in,out] = act_i^T [in,B] * dh_{i+1} [B,out]   (deterministic split over the batch)
                EpiArgs none{};
                const bool tc_wgrad = h->tc_mlp && in % 32 == 0 && B >= 1024;
                int nparts = nsplit;
                float* part = h->splitk + (tc_wgrad ? h->splitk_off[i] : 0);
                cudaStream_t rs = tc_wgrad ? aux : st;      // the CUDA-core fallback shares one partial buffer: keep it in order
                if (tc_wgrad) {
                    int rc2 = tc_gemm_mnmajor(h, h->act[i], in, h->dact[i + 1], out, part, in, out, B, h->tc_nz[i], &nparts, st);
                    if (rc2) return rc2;
                    CK(fork());
                } else {
                    launch_sgemm<false, false, EPI_NONE>(h, h->act[i], in, h->dact[i + 1], out, part, out, in, out, B, nsplit, k_chunk, none, st);
                }
                reduce_partials_kernel<<<cdiv((int64_t)in * out, 256), 256, 0, rs>>>(part, nparts, (size_t)in * out, (int64_t)in * out,
                                                                                     h->dg + W->off);
                h->launches++;
                if (!(h->fused_head && i == L - 1)) launch_colsum(h, h->dact[i + 1], out, nullptr, B, out, h->dg + b->off, rs);
                // dh_i [B,in] = dh_{i+1} [B,out] * W_i^T
                if (h->tc_mlp) {
                    const float* w_hi = h->dw + W->off; const float* w_lo = nullptr;   // W [in, out] is already K-major for this GEMM
                    if (tc_presplit()) {
                        const int64_t wsz = pad32((int64_t)in * out);
                        float* sp_hi = h->tc_w + h->tc_off[i] + 2 * wsz;
                        float* sp_lo = sp_hi + wsz;
                        tc::split_tf32_kernel<<<cdiv((int64_t)in * out, 256), 256, 0, st>>>(w_hi, (int64_t)in * out, sp_hi, sp_lo);
                        h->launches++;
                        w_hi = sp_hi; w_lo = sp_lo;
                    }
                    EpiArgs ep{};
                    int rc2;
                    if (i > 0) {
                        ep.act = h->act[i]; ep.ld_act = in;
                        ep.bwd_scale = h->dropout > 0.f ? 1.f / (1.f - h->dropout) : 0.f;
                        rc2 = tc_gemm_kmajor(h, h->dact[i + 1], nullptr, out, w_hi, w_lo, out, h->dact[i], in, B, in, out, EPI_MASK, ep, st);
                    } else {
                        ep.act = h->h0; ep.ld_act = dK; ep.dz = h->dz; ep.s = h->use_mf ? h->s : nullptr; ep.K = K;
                        rc2 = tc_gemm_kmajor(h, h->dact[1], nullptr, out, w_hi, w_lo, out, h->dE, dK, B, dK, out, EPI_DE, ep, st);
                    }
                    if (rc2) return rc2;
                } else if (i > 0) {
                    EpiArgs ep{}; ep.act = h->act[i]; ep.ld_act = in; ep.act_kind = h->activation;
                    ep.bwd_scale = h->dropout > 0.f ? 1.f / (1.f - h->dropout) : 0.f;
                    launch_sgemm<true, true, EPI_MASK>(h, h->dact[i + 1], out, h->dw + W->off, out, h->dact[i], in, B, in, out, 1,
                                                       (out + 15) / 16 * 16, ep, st);
                } else {
                    EpiArgs ep{}; ep.act = h->h0; ep.ld_act = dK; ep.dz = h->dz; ep.s = h->use_mf ? h->s : nullptr; ep.K = K;
                    launch_sgemm<true, true, EPI_DE>(h, h->dact[1], out, h->dw + W->off, out, h->dE, dK, B, dK, out, 1,
                                                     (out + 15) / 16 * 16, ep, st);
                }
            }
        }
    } else if (h->use_mf) {
        de_fm_kernel<<<cdiv((int64_t)B * dK, 256), 256, 0, st>>>(h->h0, h->s, h->dz, (int64_t)B * dK, dK, K, h->dE, 0);
        h->launches++;
    }
    if (aux != st) {      // join: everything below (and the optimizer) sees the reduced gradients
        CK(cudaEventRecord(h->ev_aux_join, aux));
        CK(cudaStreamWaitEvent(st, h->ev_aux_join, 0));
    }
    // numeric-feature gradients
    if (h->dn) {
        const DenseT* ne = find_dense(h, "num_emb"); const DenseT* nl = find_dense(h, "num_lin");
        const int chunks = (int)cdiv(B, h->num_rows_per_chunk), total = h->dn * K + h->dn;
        numeric_grad_partial_kernel<<<chunks, 256, (size_t)h->num_rows_per_chunk * (h->dn + 1) * 4, st>>>(bp, h->need_emb ? h->dE : nullptr, dK, dc, h->dn, K, h->dz, B, h->num_rows_per_chunk, h->colpart);
        h->launches++;
        if (ne) { reduce_partials_kernel<<<cdiv(h->dn * K, 256), 256, 0, st>>>(h->colpart, chunks, (size_t)total, h->dn * K, h->dg + ne->off); h->launches++; }
        if (nl) { reduce_partials_kernel<<<1, 256, 0, st>>>(h->colpart + h->dn * K, chunks, (size_t)total, h->dn, h->dg + nl->off); h->launches++; }
    }
    if (ph) ph->next();
    return DFM_OK;
}

template <int K, bool BAGS>
static StageSrcPlain<K, BAGS> stage_src(const GradSrc<K, BAGS>& src) { StageSrcPlain<K, BAGS> s{}; s.s = src; return s; }
template <typename SRC>
static SRC stage_src(const SRC& src) { return src; }

// deterministic segmented reduction of the sparse gradients (+ optimizer, or gradient rows out when gsum != nullptr)
template <int K, typename SRC>
static int sparse_update(dfm_handle* h, SegWS& ws, int64_t n, const SRC& src, const OptDev& od, const OptDev& ol, int64_t t,
                         float* gsum, cudaStream_t st, Phase* ph, const PeerRoute* route = nullptr) {
    const unsigned row_grid = (unsigned)h->sm_count * 8;
    if (n > 0) {
        hot_pieces_kernel<<<row_grid, 256, 0, st>>>(ws.row_start, ws.row_piece0, ws.seg_cnt, ws.hot_list);
        piece_reduce_kernel<K, SRC><<<row_grid, 256, 0, st>>>(ws.svals(), ws.piece_start, ws.hot_list, ws.seg_cnt, src, ws.piece_sum);
        h->launches += 2;
    }
    if (ph) ph->next();
    // gradient operands of the first lookup of every row (and, applying, the table records) staged by cp.async a few
    // iterations ahead (row_apply.cuh); the plain sources gain the staging interface, the fused one has it
    using S = decltype(stage_src(src));
    const S ss = stage_src(src);
    const unsigned grid = n > 0 ? (unsigned)h->sm_count * 2 : 1;
    if (!gsum) {
        // rows are rewritten here: the non-lazy Adam decay they skipped since their last write is replayed first (to step t-1)
        const int smem = RowApplyCfg<K, S>::SMEM + ss.aux_floats() * 4;
        if (smem > 200 * 1024) FAIL(DFM_ERR_UNSUPPORTED, "internal: staged sparse apply does not fit in shared memory");
        static int attr = 0;
        if (attr < smem) { CK(cudaFuncSetAttribute(row_apply_kernel<K, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); attr = smem; }
        row_apply_kernel<K, S><<<grid, 256, smem, st>>>(ws.urow, ws.uval, ws.svals(), ws.row_start, ws.row_piece0, ws.piece_start, ws.seg_cnt, ss,
                                                        ws.piece_sum, h->tb, h->emb_slots, od, ol, (bool)h->need_emb, (bool)h->use_linear,
                                                        (int)t, make_rr(h, t - 1));
    } else {
        // requester side of the sharded step: gradient rows into gsum (collectives) or over NVLink into the owners' segments
        const int smem = RowGsumCfg<K, S>::SMEM + ss.aux_floats() * 4;
        if (smem > 200 * 1024) FAIL(DFM_ERR_UNSUPPORTED, "internal: staged gradient-row kernel does not fit in shared memory");
        static int attr = 0;
        if (attr < smem) { CK(cudaFuncSetAttribute(row_gsum_kernel<K, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); attr = smem; }
        row_gsum_kernel<K, S><<<grid, 256, smem, st>>>(ws.urow, ws.uval, ws.svals(), ws.row_start, ws.row_piece0, ws.piece_start, ws.seg_cnt, ss,
                                                       ws.piece_sum, route, gsum, h->fr_rb_live);
    }
    h->launches++;
    if (ph) ph->next();
    CK(cudaGetLastError());
    return DFM_OK;
}


struct StepOpts { OptDev od, ol; };
static StepOpts step_opts(const dfm_handle* h) {
    StepOpts o;
    const int64_t t = h->step + 1;         // alpha_t as seen by step t (TF multiplies the beta powers after each apply)
    o.od = make_opt(h->od, alpha_at(h->rp_d, t)); o.ol = make_opt(h->ol, alpha_at(h->rp_l, t));
    return o;
}
static void commit_step(dfm_handle* h, const StepOpts&, int64_t t) { h->step = t; }

// ---- fused small-tower step (fused_small.cuh)
template <int K>
static FusedArgs make_fused_args(dfm_handle* h, const BatchPtrs& bp, int B, const float* labels, float scale, float* logits_out,
                                 const float* rowbuf, int64_t upto) {
    FusedArgs a{};
    a.ids = h->ids; a.B = B; a.dc = h->dc; a.dn = h->dn; a.n_slots = h->dcs;
    a.row_off = h->d_row_off; a.tb = h->tb; a.bp = bp; a.dw = h->dw;
    const DenseT* ne = find_dense(h, "num_emb"); const DenseT* nl = find_dense(h, "num_lin"); const DenseT* bs = find_dense(h, "bias");
    a.off_num_emb = ne ? (int)ne->off : -1; a.off_num_lin = nl ? (int)nl->off : -1; a.off_bias = bs ? (int)bs->off : -1;
    a.use_linear = h->use_linear; a.use_mf = h->use_mf;
    a.m = h->sm;
    const int train = labels ? 1 : 0;
    if (train && h->dropout > 0.f) {
        a.m.drop_keep = 1.f - h->dropout; a.m.drop_inv = 1.f / (1.f - h->dropout);
        a.m.drop_seed = h->dropout_seed; a.m.drop_step = (uint64_t)(h->step + 1); a.m.drop_row0 = (int64_t)h->rank * h->max_batch;
    }
    a.labels = labels; a.scale = scale; a.train = train;
    a.rr = make_rr(h, rowbuf ? -1 : upto);
    a.od = make_opt(h->od, 0.f); a.ol = make_opt(h->ol, 0.f);
    a.uidx = rowbuf ? h->uidx : nullptr; a.rowbuf = rowbuf; a.rowbuf_stride = K + 4;
    a.logits = h->logits; a.logits_out = logits_out; a.dz_out = h->dz; a.dh1_out = h->dact[1]; a.s_out = h->s;
    a.up_partial = h->up_partial; a.w0_partial = h->w0_partial; a.num_partial = h->num_partial; a.head_part = h->head_part;
    a.D = h->sm.D; a.n_numacc = h->n_numacc;
    a.es_stride = fs_es_stride(h->sm.D);
    return a;
}

// record-staged step (fused_rows.cuh): gather + tower forward/backward + the optimizer of once-only rows in one kernel
template <int K>
static int launch_fused_rows(dfm_handle* h, const BatchPtrs& bp, int B, const float* labels, float scale, float* logits_out, int64_t upto,
                             const StepOpts* so, int64_t t, cudaStream_t st, const float* rowbuf = nullptr, float* gsum = nullptr,
                             const PeerRoute* route = nullptr) {
    if constexpr (K == 16) {
        FusedRowsArgs A{};
        A.f = make_fused_args<K>(h, bp, B, labels, scale, logits_out, rowbuf, upto);
        A.claim = (so && h->claim_live) ? h->claim : nullptr; A.claim_mask = h->claim_mask;
        A.emb_slots = rowbuf ? 0 : h->emb_slots;
        A.rowbuf_mode = rowbuf ? 1 : 0; A.once_lk = h->once_lk; A.route = route; A.gsum = gsum;
        A.rs = K + 4 + A.emb_slots * K;
        A.sst = fr_sst(h->dc, h->dn, K, A.rs);
        A.step = (int)t;
        if (so) { A.od_t = so->od; A.ol_t = so->ol; }
        A.numg_partial = h->num_partial;
        fr_layout(A, h->sm, K, h->dc, h->dn);
        fr_balance(A, h->dc, h->dn, A.f.train && (A.rowbuf_mode || A.claim != nullptr));
        const int grid = fused_rows_grid(B, h->sm_count, rowbuf ? false : h->fr_side);
        CK(fused_rows_launch(A, grid, rowbuf ? h->fr_smem_rb : h->fr_smem, st));
        h->launches++;
        return DFM_OK;
    }
    return DFM_ERR_UNSUPPORTED;
}

template <int K>
static int launch_fused(dfm_handle* h, const BatchPtrs& bp, int B, const float* labels, float scale, float* logits_out,
                        const float* rowbuf, int64_t upto, cudaStream_t st) {
    FusedArgs a = make_fused_args<K>(h, bp, B, labels, scale, logits_out, rowbuf, upto);
    const int grid = std::min((B + FS_TS - 1) / FS_TS, h->fused_grid);
    const int H1 = h->sm.H[0];
    const int need_nc = ((h->dc + h->dn) + (256 / (H1 / 4)) / K - 1) / ((256 / (H1 / 4)) / K);     // ceil(d / fields per column group)
    // NC (dW0 columns per thread) is a compile-time bound: exact instantiations for the shapes BASELINE.json names
    // (Criteo k=16 [16,..]: 10, ML-100K k=16: 7, ML-100K k=4: 2), the generic bound otherwise
#define FUSED_GO(HH, NCC)                                                                                              \
    do {                                                                                                               \
        if (rowbuf) fused_small_kernel<K, HH, true, NCC><<<grid, 256, h->fused_smem, st>>>(a);                         \
        else fused_small_kernel<K, HH, false, NCC><<<grid, 256, h->fused_smem, st>>>(a);                               \
    } while (0)
    bool done = false;
    if constexpr (K == 16) {
        if (H1 == 16 && need_nc <= 7) { FUSED_GO(16, 7); done = true; }
        else if (H1 == 16 && need_nc <= 10) { FUSED_GO(16, 10); done = true; }
    }
    if constexpr (K == 4) {
        if (H1 == 16 && need_nc <= 2) { FUSED_GO(16, 2); done = true; }
    }
    if (!done) { if (H1 == 8) FUSED_GO(8, FS_NC); else if (H1 == 16) FUSED_GO(16, FS_NC); else FUSED_GO(32, FS_NC); }
#undef FUSED_GO
    h->launches++;
    CK(cudaGetLastError());
    return DFM_OK;
}

template <int K>
static int fused_set_attr(dfm_handle* h) {
    const int smem = (int)h->fused_smem;
#define FUSED_ATTR(HH, NCC)                                                                                                            \
    CK(cudaFuncSetAttribute(fused_small_kernel<K, HH, false, NCC>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));                \
    CK(cudaFuncSetAttribute(fused_small_kernel<K, HH, true, NCC>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    FUSED_ATTR(8, FS_NC) FUSED_ATTR(16, FS_NC) FUSED_ATTR(32, FS_NC)
    if constexpr (K == 16) { FUSED_ATTR(16, 7) FUSED_ATTR(16, 10) }
    if constexpr (K == 4) { FUSED_ATTR(16, 2) }
#undef FUSED_ATTR
    return DFM_OK;
}

// per-CTA partials of the fused kernel -> dense gradient buffer, loss, dz sum (one launch)
static int launch_fused_reduce(dfm_handle* h, int B, float scale, float* loss_out, cudaStream_t st, bool rows = false) {
    const DenseT* ne = find_dense(h, "num_emb"); const DenseT* nl = find_dense(h, "num_lin"); const DenseT* bs = find_dense(h, "bias");
    FusedReduceArgs r{};
    r.up_partial = h->up_partial; r.w0_partial = h->w0_partial; r.num_partial = h->num_partial; r.head_part = h->head_part;
    r.n_cta = rows ? fused_rows_grid(B, h->sm_count, h->fr_rb_live ? false : h->fr_side) : std::min((B + FS_TS - 1) / FS_TS, h->fused_grid);
    r.up_count = h->sm.up_count; r.up_begin = h->sm.up_begin; r.off_W0 = h->sm.off_W[0]; r.w0_count = h->sm.D * h->sm.H[0];
    r.n_numacc = rows ? h->dn * h->K + h->dn : h->n_numacc;
    r.direct_num = rows ? 1 : 0;
    r.dg = h->dg; r.num_scratch = h->num_scratch; r.done = h->fused_done;
    r.dw = h->dw; r.off_num_emb = ne ? (int)ne->off : -1; r.off_num_lin = nl ? (int)nl->off : -1; r.off_bias = bs ? (int)bs->off : -1;
    r.dc = h->dc; r.dn = h->dn; r.K = h->K; r.H1 = h->sm.H[0]; r.use_mf = h->use_mf;
    r.loss_scale = scale; r.loss_out = h->d_loss; r.loss_copy = loss_out; r.dzsum_out = h->d_dzsum;
    const int total = r.up_count + r.w0_count + r.n_numacc;
    fused_reduce_kernel<<<cdiv(total, 256), 256, 0, st>>>(r);
    h->launches++;
    CK(cudaGetLastError());
    return DFM_OK;
}

template <int K, int H1>
static GradSrcFused<K, H1> fused_src(const dfm_handle* h, const float* erow) {
    GradSrcFused<K, H1> src{};
    src.dh1 = h->dact[1]; src.s = h->use_mf ? h->s : nullptr; src.dz = h->dz; src.W0 = h->dw + h->sm.off_W[0];
    src.n_slots = h->dcs; src.erow = erow; src.erow_stride = K + 4;
    src.n_w0 = h->sm.D * H1;
    return src;
}

template <int K>
static int fused_sparse_update(dfm_handle* h, SegWS& ws, int64_t n, const StepOpts& so, int64_t t, float* gsum, const float* erow,
                               cudaStream_t st, Phase* ph, const PeerRoute* route = nullptr) {
    if constexpr (K <= 32) {
        switch (h->sm.H[0]) {
            case 8: return sparse_update<K, GradSrcFused<K, 8>>(h, ws, n, fused_src<K, 8>(h, erow), so.od, so.ol, t, gsum, st, ph, route);
            case 16: return sparse_update<K, GradSrcFused<K, 16>>(h, ws, n, fused_src<K, 16>(h, erow), so.od, so.ol, t, gsum, st, ph, route);
            default: return sparse_update<K, GradSrcFused<K, 32>>(h, ws, n, fused_src<K, 32>(h, erow), so.od, so.ol, t, gsum, st, ph, route);
        }
    }
    return DFM_ERR_UNSUPPORTED;
}

template <int K>
static int train_fused(dfm_handle* h, const BatchPtrs& bp, int B, float* loss_out, float* logits_out, cudaStream_t st) {
    if constexpr (K <= 32) {
        const int64_t n = (int64_t)B * h->dcs;
        const int64_t t = h->step + 1;
        int rc = ensure_alpha(h, t);
        if (rc) return rc;
        const int64_t l0 = h->launches;
        const StepOpts so = step_opts(h);
        Phase ph(h, st);
        const bool prefetched = h->prefetch_B == B && h->dc > 0 && h->prefetch_tag == batch_tag(h, bp.cat);
        if (h->prefetch_B >= 0 && !prefetched) h->prefetch_B = -1;
        // record-staged step: once-only rows are updated inside the kernel (the claim table is filled by the transform,
        // so a prefetched batch - ids computed earlier, no claims - takes the older kernel)
        static const bool inline_ok = getenv("DFM_NO_INLINE_APPLY") == nullptr;
        const bool rows = h->fused_rows && !prefetched && inline_ok;
        if (prefetched) {
            CK(cudaStreamWaitEvent(st, h->ev_prefetch, 0));
            std::swap(h->ws, h->ws_next); std::swap(h->ids, h->ids_next);
            h->prefetch_B = -1;
        } else {
            if (rows) CK(cudaMemsetAsync(h->claim, 0, h->claim_bytes, st));
            launch_transform<K>(h, bp, B, true, h->ids, st, rows);                              // K1 (+ claim table; pairs into buffer 1)
        }
        h->claim_live = rows; h->last_step_rows = rows;
        ph.next();
        // The forward pass reads the table rows as stored and replays the deferred Adam decay in registers, so it does
        // not need the list of touched rows: sort + segments (many small dependent launches) run on the side stream
        // beside the fused kernel and are joined in front of the sparse optimizer.
        const bool side = !prefetched && n > 0 && B >= 1024 && !h->profiling;
        h->fr_side = side && rows;
        if (side) {
            CK(cudaEventRecord(h->ev_fork, st));
            CK(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
            if (rows) CK(fused_rows_compact(h->ws.keys[1], h->ws.vals[1], n, (uint32_t)h->R, h->claim, h->claim_mask, h->ws.keys[0], h->ws.vals[0],
                                            reinterpret_cast<uint32_t*>(h->ws.flags), h->ws.n_compact, h->side_stream, &h->launches));
            if ((rc = build_segments(h, h->ws, n, (uint32_t)h->R, h->key_bits, h->side_stream, nullptr, rows ? h->ws.n_compact : nullptr))) return rc;
            CK(cudaEventRecord(h->ev_join, h->side_stream));
            ph.next(); ph.next();
        } else if (!prefetched) {
            if (rows) CK(fused_rows_compact(h->ws.keys[1], h->ws.vals[1], n, (uint32_t)h->R, h->claim, h->claim_mask, h->ws.keys[0], h->ws.vals[0],
                                            reinterpret_cast<uint32_t*>(h->ws.flags), h->ws.n_compact, st, &h->launches));
            if ((rc = build_segments(h, h->ws, n, (uint32_t)h->R, h->key_bits, st, &ph, rows ? h->ws.n_compact : nullptr))) return rc;
        } else {
            ph.next(); ph.next();
        }
        ph.next();                                                                               // (no catch-up pass)
        const float scale = h->loss_red == DFM_LOSS_MEAN ? 1.0f / (float)B : 1.0f;
        if (h->fused_rows) rc = launch_fused_rows<K>(h, bp, B, bp.labels, scale, logits_out, t - 1, &so, t, st);
        else rc = launch_fused<K>(h, bp, B, bp.labels, scale, logits_out, nullptr, t - 1, st);
        if (rc) return rc;
        ph.next(); ph.next();                                                                    // gather + tower forward/backward top
        // The sparse optimizer of the repeated rows needs the per-sample vectors of the kernel above and the side stream's
        // segments, not the dense reduction: it stays on the side stream, beside fused_reduce, and is joined in front of
        // dense_apply (it reads W0).
        static const bool tail_overlap = getenv("DFM_NO_TAIL_OVERLAP") == nullptr;
        const bool side_tail = side && tail_overlap;
        if (side_tail) {
            CK(cudaEventRecord(h->ev_aux_fork, st));
            CK(cudaStreamWaitEvent(h->side_stream, h->ev_aux_fork, 0));
            if ((rc = fused_sparse_update<K>(h, h->ws, n, so, t, nullptr, nullptr, h->side_stream, nullptr))) return rc;
            CK(cudaEventRecord(h->ev_aux_join, h->side_stream));
        }
        if ((rc = launch_fused_reduce(h, B, scale, loss_out, st, h->fused_rows))) return rc;
        ph.next(); ph.next();                                                                    // loss, dense gradients
        if (!side_tail) {
            if (side) CK(cudaStreamWaitEvent(st, h->ev_join, 0));
            if ((rc = fused_sparse_update<K>(h, h->ws, n, so, t, nullptr, nullptr, st, &ph))) return rc;
        }
        h->claim_live = false;
        if (side_tail) CK(cudaStreamWaitEvent(st, h->ev_aux_join, 0));      // row_apply rebuilds gradients from W0: before the dense update
        if (h->n_dense) {
            dense_apply_kernel<<<cdiv(h->n_dense, 256), 256, 0, st>>>(h->dw, h->ds1, h->ds2, h->dg, h->n_deep, h->n_dense, so.od, so.ol);
            h->launches++;
        }
        ph.next();
        CK(cudaGetLastError());
        commit_step(h, so, t);
        if (h->ev_done[t & 1]) CK(cudaEventRecord(h->ev_done[t & 1], st));
        h->last_step_launches = h->launches - l0;
        return DFM_OK;
    }
    return DFM_ERR_UNSUPPORTED;
}

template <int K>
static int train_impl(dfm_handle* h, const BatchPtrs& bp, int B, float* loss_out, float* logits_out, cudaStream_t st) {
    if (h->world > 1) FAIL(DFM_ERR_UNSUPPORTED, "row-sharded handle: drive the step with the dfm_shard_* entry points");
    if (h->fused) return train_fused<K>(h, bp, B, loss_out, logits_out, st);
    const int dc = h->dc, d = dc + h->dn, dK = d * K;
    const int64_t n = (int64_t)B * (h->n_tiny ? h->n_big : h->dcs);      // lookups that go through the sort
    const int64_t t = h->step + 1;
    int rc = ensure_alpha(h, t);
    if (rc) return rc;
    const int64_t l0 = h->launches;
    const StepOpts so = step_opts(h);
    Phase ph(h, st);
    // ids, sort and segments of this batch may have been computed ahead of time on the side stream (dfm_prefetch_batch)
    const bool prefetched = h->prefetch_B == B && h->dc > 0 && h->prefetch_tag == batch_tag(h, bp.cat);
    if (h->prefetch_B >= 0 && !prefetched) h->prefetch_B = -1;            // a different batch arrived: drop the prefetch
    if (prefetched) {
        CK(cudaStreamWaitEvent(st, h->ev_prefetch, 0));
        std::swap(h->ws, h->ws_next); std::swap(h->ids, h->ids_next);
        h->prefetch_B = -1;
    } else {
        launch_transform<K>(h, bp, B, true, h->ids, st);                                    // K1
    }
    ph.next();
    // The gather replays the deferred non-lazy Adam decay of the rows it reads in registers (replay.cuh), so the forward
    // pass never waits for the list of touched rows: with batches large enough to matter the sort / segment stage (small
    // grids that leave most SMs idle) runs on the side stream beside the gather and the tower.
    const bool overlap = h->overlap_sort && B >= 4096 && n > 0 && !prefetched;
    if (prefetched) {
        ph.next(); ph.next();
    } else if (overlap) {
        CK(cudaEventRecord(h->ev_fork, st));
        CK(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
        if ((rc = build_segments(h, h->ws, n, (uint32_t)h->R, h->key_bits, h->side_stream, nullptr))) return rc;   // sort + segments, side stream
        CK(cudaEventRecord(h->ev_join, h->side_stream));
        ph.next(); ph.next();
    } else {
        if ((rc = build_segments(h, h->ws, n, (uint32_t)h->R, h->key_bits, st, &ph))) return rc;   // sort + segments
    }
    ph.next();
    const float scale = h->loss_red == DFM_LOSS_MEAN ? 1.0f / (float)B : 1.0f;
    if ((rc = forward_impl<K>(h, bp, B, st, bp.labels, scale, logits_out, &ph, nullptr, t - 1))) return rc;
    if ((rc = tower_backward<K>(h, bp, B, scale, loss_out, st, &ph, B >= 4096 ? h->side_stream : nullptr))) return rc;
    if (overlap) CK(cudaStreamWaitEvent(st, h->ev_join, 0));
    const bool tiny_side = h->n_tiny && B >= 4096;      // the tiny-column reduction touches other rows than the sorted path: run both at once
    if (tiny_side) {
        CK(cudaEventRecord(h->ev_aux_fork, st));
        CK(cudaStreamWaitEvent(h->side_stream, h->ev_aux_fork, 0));
        if ((rc = tiny_update<K>(h, B, so.od, so.ol, t, h->side_stream))) return rc;
        CK(cudaEventRecord(h->ev_aux_join, h->side_stream));
    }
    if (h->has_bags) {
        GradSrc<K, true> src{};
        src.dE = h->need_emb ? h->dE : nullptr; src.dz = h->dz; src.dc = dc; src.dK = dK; src.flat = nullptr; src.flat_stride = 0;
        src.n_slots = h->dcs; src.slot_field = h->d_slot_col; src.inv_cnt = h->inv_cnt;
        rc = sparse_update<K, GradSrc<K, true>>(h, h->ws, n, src, so.od, so.ol, t, nullptr, st, &ph);
    } else {
        GradSrc<K, false> src{};
        src.dE = h->need_emb ? h->dE : nullptr; src.dz = h->dz; src.dc = dc; src.dK = dK; src.flat = nullptr; src.flat_stride = 0;
        src.n_slots = h->dcs; src.slot_field = nullptr; src.inv_cnt = nullptr;
        rc = sparse_update<K, GradSrc<K, false>>(h, h->ws, n, src, so.od, so.ol, t, nullptr, st, &ph);
    }
    if (rc) return rc;
    if (tiny_side) CK(cudaStreamWaitEvent(st, h->ev_aux_join, 0));
    else if ((rc = tiny_update<K>(h, B, so.od, so.ol, t, st))) return rc;
    if (h->n_dense) {
        dense_apply_kernel<<<cdiv(h->n_dense, 256), 256, 0, st>>>(h->dw, h->ds1, h->ds2, h->dg, h->n_deep, h->n_dense, so.od, so.ol);
        h->launches++;
    }
    ph.next();
    CK(cudaGetLastError());
    commit_step(h, so, t);
    if (h->ev_done[t & 1]) CK(cudaEventRecord(h->ev_done[t & 1], st));      // dfm_prefetch_batch orders buffer reuse on these
    h->last_step_launches = h->launches - l0;
    return DFM_OK;
}

// mode == EVAL / PREDICT: forward pass alone on the rows as of the latest step (replayed in registers, nothing written)
template <int K>
static int eval_forward(dfm_handle* h, const BatchPtrs& bp, int B, float* logits_out, const float* rowbuf, cudaStream_t st) {
    if (h->fused) {
        if constexpr (K <= 32) return launch_fused<K>(h, bp, B, nullptr, 1.f, logits_out, rowbuf, h->step, st);
    }
    return forward_impl<K>(h, bp, B, st, nullptr, 1.f, logits_out, nullptr, rowbuf, h->step);
}

#define DISPATCH_K(h, CALL)                                          \
    switch ((h)->K) {                                                \
        case 4: { constexpr int KK = 4; CALL; } break;               \
        case 8: { constexpr int KK = 8; CALL; } break;               \
        case 16: { constexpr int KK = 16; CALL; } break;             \
        case 32: { constexpr int KK = 32; CALL; } break;             \
        case 64: { constexpr int KK = 64; CALL; } break;             \
        default: { constexpr int KK = 128; CALL; } break;            \
    }

// ------------------------------------------------------------------------- device entry points
extern "C" int dfm_flush(dfm_handle* h, void* stream) {
    if (!h) return DFM_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    int rc = DFM_OK;
    DISPATCH_K(h, rc = flush_impl<KK>(h, st));
    return rc;
}

extern "C" int dfm_transform(dfm_handle* h, const dfm_raw_batch* b, int32_t* ids_out, void* stream) {
    if (!h || !ids_out) return DFM_ERR_INVALID_ARG;
    int rc = check_batch(h, b, false);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    BatchPtrs bp = make_ptrs(h, b);
    launch_transform<4>(h, bp, b->batch_size, false, ids_out, st);
    CK(cudaGetLastError());
    return DFM_OK;
}

// Small batches are launch-bound (BASELINE configs[0] / [1]: ~22 kernels of a few microseconds each per step), so the
// step is replayed as ONE CUDA graph.  The per-step scalars (alpha_t, step number, replay horizon, dropout key) are plain
// kernel arguments, so every step is stream-captured through the ordinary host path - nothing executes during a capture -
// and the instantiated graph is updated in place from the capture (cudaGraphExecUpdate: same topology, new arguments)
// and launched once; only a change of topology (another batch size or path) re-instantiates.
static bool graph_step_ok(const dfm_handle* h, int B) {
    // (large batches gain too: the Criteo-shaped step 0.80 -> 0.79 ms, its host-buffer form 0.87 -> 0.82 ms, configs[2] 0.657 -> 0.640 ms)
    static const int max_b = getenv("DFM_GRAPH_MAX_BATCH") ? atoi(getenv("DFM_GRAPH_MAX_BATCH")) : 131072;
    return B <= max_b && h->world == 1 && !h->profiling && h->prefetch_B < 0 && !h->ws_next.cap;
}
static int train_step_graphed(dfm_handle* h, const BatchPtrs& bp, int B, float* loss_out, float* logits_out, cudaStream_t st) {
    int rc = ensure_alpha(h, h->step + 1);               // growth allocates and synchronises: outside the capture
    if (rc) return rc;
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        cudaGetLastError();                               // a stream that cannot be captured (legacy default stream): ordinary launches
        DISPATCH_K(h, rc = train_impl<KK>(h, bp, B, loss_out, logits_out, st));
        return rc;
    }
    DISPATCH_K(h, rc = train_impl<KK>(h, bp, B, loss_out, logits_out, st));
    cudaGraph_t g = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(st, &g);
    if (rc || ce != cudaSuccess) {
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        if (rc) return rc;
        FAIL(DFM_ERR_CUDA, "stream capture of the train step failed");
    }
    if (h->gexec) {
        cudaGraphExecUpdateResultInfo info{};
        if (cudaGraphExecUpdate(h->gexec, g, &info) != cudaSuccess) {
            cudaGetLastError();
            cudaGraphExecDestroy(h->gexec);
            h->gexec = nullptr;
        }
    }
    if (!h->gexec) {
        const cudaError_t ie = cudaGraphInstantiate(&h->gexec, g, 0);
        if (ie != cudaSuccess) { cudaGraphDestroy(g); h->gexec = nullptr; CK(ie); }
        h->graph_rebuilds++;
    }
    cudaGraphDestroy(g);
    CK(cudaGraphLaunch(h->gexec, st));
    h->graph_steps++;
    return DFM_OK;
}
extern "C" int64_t dfm_graph_steps(const dfm_handle* h) { return h ? h->graph_steps : -1; }

extern "C" int dfm_train_step(dfm_handle* h, const dfm_raw_batch* b, float* loss_out, float* logits_out, void* stream) {
    if (!h) return DFM_ERR_INVALID_ARG;
    int rc = check_batch(h, b, true);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    BatchPtrs bp = make_ptrs(h, b);
    static const bool graphs = getenv("DFM_NO_GRAPH") == nullptr;
    if (graphs && graph_step_ok(h, b->batch_size)) return train_step_graphed(h, bp, b->batch_size, loss_out, logits_out, st);
    DISPATCH_K(h, rc = train_impl<KK>(h, bp, b->batch_size, loss_out, logits_out, st));
    return rc;
}

// Input-pipeline lookahead for the unsharded step: feature transforms, sort and segments of the NEXT batch depend on
// nothing but the batch, so they can run on the side stream while the current step is still in its tower.  The
// following dfm_train_step on the same batch (same first column pointer and size) adopts the result.
extern "C" int dfm_prefetch_batch(dfm_handle* h, const dfm_raw_batch* b, void* after_stream) {
    if (!h) return DFM_ERR_INVALID_ARG;
    if (h->world > 1) FAIL(DFM_ERR_UNSUPPORTED, "row-sharded handle: no batch prefetch");
    int rc = check_batch(h, b, false);
    if (rc) return rc;
    if (h->dc == 0) return DFM_OK;
    CK(cudaSetDevice(h->device));
    const int B = b->batch_size;
    if (!h->ws_next.cap) {
        const int64_t nmax = (int64_t)h->max_batch * std::max(h->dcs, 1);
        if (alloc_ws(h, h->ws_next, nmax, h->K) || dalloc(h, &h->ids_next, (size_t)nmax)) return DFM_ERR_CUDA;
        CK(cudaEventCreateWithFlags(&h->ev_prefetch, cudaEventDisableTiming));
        for (cudaEvent_t& e : h->ev_done) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CK(cudaDeviceSynchronize());        // first use: nothing recorded yet, start from a quiet device
    } else if (h->step >= 1) {
        // the second buffer set was last read by step (latest - 1); the prefetch may overlap the latest step only
        CK(cudaStreamWaitEvent(h->side_stream, h->ev_done[(h->step - 1) & 1], 0));
    }
    if (after_stream) {
        CK(cudaEventRecord(h->ev_prefetch, (cudaStream_t)after_stream));
        CK(cudaStreamWaitEvent(h->side_stream, h->ev_prefetch, 0));
    }
    BatchPtrs bp = make_ptrs(h, b);
    const int64_t n = (int64_t)B * (h->n_tiny ? h->n_big : h->dcs);
    std::swap(h->ws, h->ws_next); std::swap(h->ids, h->ids_next);       // launches below capture the second buffer set
    DISPATCH_K(h, launch_transform<KK>(h, bp, B, true, h->ids, h->side_stream));
    rc = build_segments(h, h->ws, n, (uint32_t)h->R, h->key_bits, h->side_stream, nullptr);
    std::swap(h->ws, h->ws_next); std::swap(h->ids, h->ids_next);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev_prefetch, h->side_stream));
    h->prefetch_B = B; h->prefetch_tag = batch_tag(h, bp.cat);
    CK(cudaGetLastError());
    return DFM_OK;
}

extern "C" int dfm_forward(dfm_handle* h, const dfm_raw_batch* b, float* logits_out, void* stream) {
    if (!h || !logits_out) return DFM_ERR_INVALID_ARG;
    if (h->world > 1) FAIL(DFM_ERR_UNSUPPORTED, "row-sharded handle: use dfm_shard_requests / serve / dfm_shard_forward");
    int rc = check_batch(h, b, false);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    BatchPtrs bp = make_ptrs(h, b);
    bp.labels = nullptr;
    rc = ensure_alpha(h, h->step);
    if (rc) return rc;
    launch_transform<4>(h, bp, b->batch_size, false, h->ids, st);
    DISPATCH_K(h, rc = eval_forward<KK>(h, bp, b->batch_size, logits_out, nullptr, st));
    if (rc) return rc;
    CK(cudaGetLastError());
    return DFM_OK;
}

// ---- layer_summary side outputs (summary.cuh; trainers/model_utils.py:4-6 and its call sites in trainers/deep_fm.py)
static std::vector<double> summary_limits() {      // core/lib/histogram/histogram.cc InitDefaultBucketsInner
    std::vector<double> pos, out;
    for (double v = 1.0e-12; v < 1.0e20; v *= 1.1) pos.push_back(v);
    pos.push_back(DBL_MAX);
    for (size_t i = pos.size(); i-- > 0;) out.push_back(-pos[i]);
    out.push_back(0.0);
    out.insert(out.end(), pos.begin(), pos.end());
    return out;
}
extern "C" int dfm_summary_bucket_limits(double* limits_out, int32_t* n_out) {
    const std::vector<double> l = summary_limits();
    if (n_out) *n_out = (int32_t)l.size();
    if (limits_out) memcpy(limits_out, l.data(), l.size() * sizeof(double));
    return DFM_OK;
}
static __global__ void summary_total_kernel(const float* lin, const float* mf, const float* dnn, int B, float* out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) out[b] = (lin ? lin[b] : 0.f) + (mf ? mf[b] : 0.f) + (dnn ? dnn[b] : 0.f);
}
template <int K>
static int summary_gather(dfm_handle* h, const BatchPtrs& bp, int B, int use_linear, int use_mf, float* zacc, cudaStream_t st) {
    float* num_emb = nullptr; float* num_lin = nullptr; float* bias = nullptr;
    for (const DenseT& dt : h->dense) {
        if (dt.name == "num_emb") num_emb = h->dw + dt.off;
        if (dt.name == "num_lin") num_lin = h->dw + dt.off;
        if (dt.name == "bias") bias = h->dw + dt.off;
    }
    unsigned grid = std::min<unsigned>(cdiv(B, 8), (unsigned)h->sm_count * 16);
    auto kern = h->has_bags ? gather_fm_kernel<K, true> : gather_fm_kernel<K, false>;
    kern<<<grid, 256, 0, st>>>(h->ids, B, h->dc, h->dn, h->dcs, h->has_bags ? h->d_field_slot0 : nullptr, h->has_bags ? h->inv_cnt : nullptr,
                               h->d_row_off, h->tb, bp, num_emb, num_lin, bias, use_linear, use_mf, h->need_emb, h->sum_h0, h->sum_s, zacc,
                               nullptr, nullptr, K + 4, make_rr(h, h->step), make_opt(h->od, 0.f), make_opt(h->ol, 0.f));
    h->launches++;
    CK(cudaGetLastError());
    return DFM_OK;
}
extern "C" int dfm_layer_summary(dfm_handle* h, const dfm_raw_batch* b, int32_t train_mode, dfm_tensor_summary* out, int64_t* bucket_counts,
                                 int32_t max_tensors, int32_t* n_tensors) {
    if (!h || !out || !n_tensors) return DFM_ERR_INVALID_ARG;
    if (h->world > 1) FAIL(DFM_ERR_UNSUPPORTED, "layer summaries of a row-sharded handle are not built");
    int rc = check_batch(h, b, false);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const int B = b->batch_size, K = h->K, dK = (h->dc + h->dn) * K;
    const int T = (h->use_linear ? 1 : 0) + (h->use_mf ? 1 : 0) + (h->use_dnn ? h->L + 1 : 0) + 1;
    if (T > max_tensors) FAIL(DFM_ERR_INVALID_ARG, "dfm_layer_summary: out[] is too small for the tensors of this model");
    int hid = 0, maxdim = dK;
    for (int i = 0; i < h->L; ++i) { hid += h->hidden[i]; maxdim = std::max(maxdim, h->hidden[i]); }
    const std::vector<double> limits = summary_limits();
    const int NL = (int)limits.size();
    if (!h->sum_logits) {
        const size_t Bm = (size_t)h->max_batch;
        if (h->need_emb && dalloc(h, &h->sum_h0, Bm * dK)) return DFM_ERR_CUDA;
        if (dalloc(h, &h->sum_s, Bm * K)) return DFM_ERR_CUDA;
        if (dalloc(h, &h->sum_lin, Bm)) return DFM_ERR_CUDA;
        if (dalloc(h, &h->sum_mf, Bm)) return DFM_ERR_CUDA;
        if (h->use_dnn && dalloc(h, &h->sum_hidden, Bm * std::max(hid, 1))) return DFM_ERR_CUDA;
        if (dalloc(h, &h->sum_dnn, Bm)) return DFM_ERR_CUDA;
        if (dalloc(h, &h->sum_limits, (size_t)NL)) return DFM_ERR_CUDA;
        if (dalloc(h, &h->sum_stats, (size_t)DFM_MAX_HIDDEN + 4)) return DFM_ERR_CUDA;
        if (dalloc(h, &h->sum_buckets, (size_t)(DFM_MAX_HIDDEN + 4) * NL)) return DFM_ERR_CUDA;
        if (dalloc(h, &h->sum_logits, Bm)) return DFM_ERR_CUDA;
        CK(cudaMemcpy(h->sum_limits, limits.data(), NL * sizeof(double), cudaMemcpyHostToDevice));
    }
    BatchPtrs bp = make_ptrs(h, b);
    bp.labels = nullptr;
    rc = ensure_alpha(h, h->step + 1);
    if (rc) return rc;
    launch_transform<4>(h, bp, B, false, h->ids, st);
    if (h->use_linear) DISPATCH_K(h, rc = summary_gather<KK>(h, bp, B, 1, 0, h->sum_lin, st));
    if (rc) return rc;
    if (h->use_mf || h->use_dnn) DISPATCH_K(h, rc = summary_gather<KK>(h, bp, B, 0, h->use_mf, h->sum_mf, st));
    if (rc) return rc;
    if (h->use_dnn) {
        SummaryTowerArgs a{};
        a.h0 = h->sum_h0; a.dK = dK; a.dw = h->dw; a.L = h->L; a.B = B; a.maxdim = maxdim; a.hid_stride = hid;
        for (int i = 0; i < h->L; ++i) {
            a.H[i] = h->hidden[i];
            a.off_W[i] = (int)find_dense(h, "W" + std::to_string(i))->off; a.off_b[i] = (int)find_dense(h, "b" + std::to_string(i))->off;
        }
        a.off_Wo = (int)find_dense(h, "Wo")->off; a.off_bo = (int)find_dense(h, "bo")->off;
        if (train_mode && h->dropout > 0.f) {
            a.drop_keep = 1.f - h->dropout; a.drop_inv = 1.f / (1.f - h->dropout);
            a.drop_seed = h->dropout_seed; a.drop_step = (uint64_t)(h->step + 1); a.drop_row0 = (int64_t)h->rank * h->max_batch;
        }
        a.hidden_out = h->sum_hidden; a.dnn_logit = h->sum_dnn; a.act_kind = h->activation;
        const int smem = 4 * 2 * maxdim * 4;
        if (smem > 200 * 1024) FAIL(DFM_ERR_UNSUPPORTED, "layer summary: layer too wide for the diagnostic tower kernel");
        static int attr = 0;
        if (attr < smem) { CK(cudaFuncSetAttribute(summary_tower_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); attr = smem; }
        summary_tower_kernel<<<std::min((B + 3) / 4, h->sm_count * 8), 128, smem, st>>>(a);
        h->launches++;
    }
    summary_total_kernel<<<cdiv(B, 256), 256, 0, st>>>(h->use_linear ? h->sum_lin : nullptr, h->use_mf ? h->sum_mf : nullptr,
                                                       h->use_dnn ? h->sum_dnn : nullptr, B, h->sum_logits);
    // reduce every tensor: {fraction of zeros, HistogramProto fields}
    std::vector<SummaryStats> init((size_t)T);
    for (auto& x : init) { x.sum = 0; x.sum_sq = 0; x.num = 0; x.zeros = 0; x.min = __int_as_float_host(0x7f800000); x.max = __int_as_float_host((int)0x807fffff); }
    CK(cudaMemcpyAsync(h->sum_stats, init.data(), T * sizeof(SummaryStats), cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(h->sum_buckets, 0, (size_t)T * NL * sizeof(unsigned long long), st));
    int ti = 0;
    auto reduce = [&](const float* base, int cols, int64_t stride) {
        const int64_t n = (int64_t)B * cols;
        summary_reduce_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)h->sm_count * 8), 256, 0, st>>>(
            base, B, cols, stride, h->sum_limits, NL, h->sum_stats + ti, h->sum_buckets + (size_t)ti * NL);
        ++ti;
    };
    if (h->use_linear) reduce(h->sum_lin, 1, 1);
    if (h->use_mf) reduce(h->sum_mf, 1, 1);
    if (h->use_dnn) {
        int col = 0;
        for (int i = 0; i < h->L; ++i) { reduce(h->sum_hidden + col, h->hidden[i], hid); col += h->hidden[i]; }
        reduce(h->sum_dnn, 1, 1);
    }
    reduce(h->sum_logits, 1, 1);
    CK(cudaGetLastError());
    std::vector<SummaryStats> res((size_t)T);
    CK(cudaMemcpyAsync(res.data(), h->sum_stats, T * sizeof(SummaryStats), cudaMemcpyDeviceToHost, st));
    if (bucket_counts) CK(cudaMemcpyAsync(bucket_counts, h->sum_buckets, (size_t)T * NL * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    auto dec = [](float f) { int i; memcpy(&i, &f, 4); if (i < 0) i ^= 0x7fffffff; float r; memcpy(&r, &i, 4); return r; };
    for (int i = 0; i < T; ++i) {
        out[i].min = dec(res[i].min); out[i].max = dec(res[i].max); out[i].num = (double)res[i].num;
        out[i].sum = res[i].sum; out[i].sum_squares = res[i].sum_sq;
        out[i].zero_fraction = res[i].num ? (double)res[i].zeros / (double)res[i].num : 0.0;
    }
    *n_tensors = T;
    return DFM_OK;
}
// device copies of the summarised tensors of the last dfm_layer_summary call (tests): 0 linear, 1 mf, 2 hidden [B, sum H], 3 dnn logit, 4 logits
extern "C" int dfm_layer_summary_tensor(dfm_handle* h, int32_t which, int64_t n, float* out_host) {
    if (!h || !out_host || !h->sum_logits) return DFM_ERR_INVALID_ARG;
    const float* src = which == 0 ? h->sum_lin : which == 1 ? h->sum_mf : which == 2 ? h->sum_hidden : which == 3 ? h->sum_dnn : h->sum_logits;
    if (!src) return DFM_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpy(out_host, src, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return DFM_OK;
}

extern "C" int dfm_sync(dfm_handle* h) {
    if (!h) return DFM_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->copy_stream));
    CK(cudaStreamSynchronize(h->stream));
    int e = 0;
    CK(cudaMemcpy(&e, h->d_err, 4, cudaMemcpyDeviceToHost));
    if (h->profiling) {
        for (int i = 0; i < dfm_handle::NPH; ++i) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, h->ph_ev[i], h->ph_ev[i + 1]) == cudaSuccess) h->ph_ms[i] = ms;
            else cudaGetLastError();
        }
    }
    if (e) {
        CK(cudaMemset(h->d_err, 0, 4));
        if (e & 2) FAIL(DFM_ERR_PEER, "exchange: a peer's flag did not arrive within 4 s");
        if (e & 4) FAIL(DFM_ERR_UNSUPPORTED, "exchange: more rows for one owner than its segment / workspace holds (raise max_batch)");
        FAIL(DFM_ERR_OUT_OF_RANGE, "identity column value outside [0, num_buckets)");
    }
    return DFM_OK;
}

extern "C" int64_t dfm_global_step(const dfm_handle* h) { return h ? h->step : -1; }

// order-independent checksum (sum of the 32-bit patterns, mod 2^64) of everything the handle trains: table records
// (weights, optimizer slots, last_step) after materialising the deferred decay, and the dense parameters + slots
__global__ void checksum_kernel(const uint32_t* __restrict__ p, size_t n, unsigned long long* __restrict__ out) {
    unsigned long long acc = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) acc += p[i];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}
extern "C" int dfm_state_checksum(dfm_handle* h, uint64_t* out_host) {
    if (!h || !out_host) return DFM_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    int rc = dfm_flush(h, h->stream);
    if (rc) return rc;
    unsigned long long* d = nullptr;
    CK(cudaMalloc(&d, 8));
    CK(cudaMemsetAsync(d, 0, 8, h->stream));
    const size_t nrec = (size_t)h->R_loc * h->tb.stride;
    if (nrec) checksum_kernel<<<(unsigned)h->sm_count * 8, 256, 0, h->stream>>>(reinterpret_cast<const uint32_t*>(h->tb.rec), nrec, d);
    for (const float* p : {h->dw, h->ds1, h->ds2})
        if (h->n_dense) checksum_kernel<<<4, 256, 0, h->stream>>>(reinterpret_cast<const uint32_t*>(p), (size_t)h->n_dense, d);
    unsigned long long v = 0;
    CK(cudaMemcpyAsync(&v, d, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    cudaFree(d);
    *out_host = v;
    return DFM_OK;
}
// unique table rows touched by the last step's batch (requester-side list when sharded); synchronises the handle's stream
extern "C" int64_t dfm_last_unique_rows(dfm_handle* h) {
    if (!h) return -1;
    cudaSetDevice(h->device);
    SegCounts sc{};
    cudaDeviceSynchronize();
    if (cudaMemcpy(&sc, h->ws.seg_cnt, sizeof sc, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    int64_t once = 0;
    if (h->last_step_rows) {      // record-staged step: the sorted list holds only the rows looked up more than once
        uint32_t nc[2] = {0, 0};
        if (cudaMemcpy(nc, h->ws.n_compact, sizeof nc, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        once = nc[1];
    }
    return (int64_t)sc.n_rows + once;
}

// Restore point: variables + slots were loaded with dfm_set_tensor from a checkpoint taken at `step`
// (tables fully materialised, i.e. after dfm_flush).  Rebuilds what TF keeps in beta1_power / beta2_power /
// global_step and marks every row as current.
extern "C" int dfm_set_global_step(dfm_handle* h, int64_t step) {
    if (!h || step < 0) return DFM_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    int rc = ensure_alpha(h, step + 1);
    if (rc) return rc;
    h->step = step; h->flushed_step = step;      // alpha_t / beta powers are functions of the step (build_replay)
    if (h->R_loc) {
        fill_strided_kernel<<<cdiv((int64_t)h->R_loc, 256), 256, 0, h->stream>>>(h->tb.rec + h->tb.lin_off + 3, h->R_loc, 1, h->tb.stride,
                                                                                  __int_as_float_host((int)step));
    }
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    return DFM_OK;
}
extern "C" int64_t dfm_last_step_launches(const dfm_handle* h) { return h ? h->last_step_launches : -1; }
extern "C" int dfm_set_profiling(dfm_handle* h, int32_t on) { if (!h) return DFM_ERR_INVALID_ARG; h->profiling = on != 0; return DFM_OK; }
extern "C" float dfm_phase_ms(dfm_handle* h, const char* phase) {
    if (!h || !phase) return -1.f;
    for (int i = 0; i < dfm_handle::NPH; ++i) if (!strcmp(phase, kPhases[i])) return h->ph_ms[i];
    return -1.f;
}

// ------------------------------------------------------------------------------- row sharding
// One handle per rank; rank r owns global rows {g : g % world == r} (local index g / world).  The four
// calls below are the per-rank compute of one sharded step; the host performs the collectives
// between them (all_to_all of row ids, rows and gradient rows; all_reduce of dense gradients).
extern "C" int dfm_shard_row_width(const dfm_handle* h) { return h ? h->K + 4 : -1; }
extern "C" int dfm_num_slots(const dfm_handle* h) { return h ? h->dcs : -1; }
extern "C" int64_t dfm_dense_size(const dfm_handle* h) { return h ? h->n_dense : -1; }

template <int K>
static int shard_requests_impl(dfm_handle* h, const BatchPtrs& bp, int B, uint32_t* req_rows_out, int32_t* counts_host, cudaStream_t st) {
    const int64_t n = (int64_t)B * h->dcs;
    const int64_t t = h->step + 1;
    int rc = ensure_alpha(h, t);
    if (rc) return rc;
    h->last_step_launches = 0;
    const int64_t l0 = h->launches;
    const uint32_t W = (uint32_t)h->world, limit = W * h->Rl;
    launch_transform<K>(h, bp, B, true, h->ids, st);
    if (n > 0) { shard_rekey_kernel<<<cdiv(n, 256), 256, 0, st>>>(h->ws.keys[0], n, (uint32_t)h->R, W, h->Rl); h->launches++; }
    if ((rc = build_segments(h, h->ws, n, limit, h->key_bits, st, nullptr))) return rc;
    CK(cudaMemsetAsync(h->d_counts, 0, ((size_t)W + 1) * 4, st));
    if (n > 0) {
        shard_uniq_kernel<<<cdiv(n, 256), 256, 0, st>>>(h->ws.skeys(), h->ws.svals(), n, limit, h->Rl, W, h->dcs, h->ws.pos_row, h->uidx, h->req_rows, h->d_counts, h->once_lk);
        h->launches++;
    }
    CK(cudaMemcpyAsync(h->h_counts, h->d_counts, (size_t)W * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    int64_t U = 0;
    for (uint32_t o = 0; o < W; ++o) { counts_host[o] = h->h_counts[o]; U += h->h_counts[o]; }
    if (U && req_rows_out) CK(cudaMemcpyAsync(req_rows_out, h->req_rows, (size_t)U * 4, cudaMemcpyDeviceToDevice, st));
    h->shard_n_req = U; h->shard_B = B;
    h->last_step_launches += h->launches - l0;
    CK(cudaGetLastError());
    return DFM_OK;
}

extern "C" int dfm_shard_requests(dfm_handle* h, const dfm_raw_batch* b, uint32_t* req_rows_out_dev, int32_t* counts_host, void* stream) {
    if (!h || !counts_host) return DFM_ERR_INVALID_ARG;
    if (h->world < 2) FAIL(DFM_ERR_INVALID_ARG, "handle was not created with world > 1");
    int rc = check_batch(h, b, false);      // labels are only needed by dfm_shard_forward_backward
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    BatchPtrs bp = make_ptrs(h, b);
    DISPATCH_K(h, rc = shard_requests_impl<KK>(h, bp, b->batch_size, req_rows_out_dev, counts_host, st));
    return rc;
}

template <int K>
static int shard_serve_impl(dfm_handle* h, const uint32_t* recv_rows, int64_t n_recv, float* reply, cudaStream_t st) {
    if (n_recv > h->ws_own.cap) FAIL(DFM_ERR_UNSUPPORTED, "more row requests than the owner workspace holds (raise max_batch)");
    const int64_t l0 = h->launches;
    const int64_t t = h->step + 1;
    int bits = 1;
    while ((1ull << bits) <= h->R_loc) ++bits;
    if (n_recv > 0) {
        CK(cudaMemcpyAsync(h->ws_own.keys[0], recv_rows, (size_t)n_recv * 4, cudaMemcpyDeviceToDevice, st));
        iota_kernel<<<cdiv(n_recv, 256), 256, 0, st>>>(h->ws_own.vals[0], n_recv);
        h->launches++;
    }
    // the rows are served as of step t-1 (deferred Adam decay replayed in registers, nothing written); the sorted list
    // of the received ids is what dfm_shard_apply reduces the gradient rows by
    int rc = build_segments(h, h->ws_own, n_recv, (uint32_t)h->R_loc, bits, st, nullptr);
    if (rc) return rc;
    if (n_recv > 0) {
        const RowReplay rr = make_rr(h, t - 1);
        const OptDev od = make_opt(h->od, 0.f), ol = make_opt(h->ol, 0.f);
        shard_serve_kernel<K><<<(unsigned)h->sm_count * 8, 256, 0, st>>>(recv_rows, n_recv, h->tb, (bool)h->need_emb,
                                                                         (bool)h->use_linear, reply, K + 4, rr, od, ol);
        h->launches++;
    }
    h->shard_n_recv = n_recv;
    h->last_step_launches += h->launches - l0;
    CK(cudaGetLastError());
    return DFM_OK;
}

extern "C" int dfm_shard_serve(dfm_handle* h, const uint32_t* recv_rows_dev, int64_t n_recv, float* reply_dev, void* stream) {
    if (!h || n_recv < 0 || (n_recv > 0 && (!recv_rows_dev || !reply_dev))) return DFM_ERR_INVALID_ARG;
    if (h->world < 2) FAIL(DFM_ERR_INVALID_ARG, "handle was not created with world > 1");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    int rc = DFM_OK;
    DISPATCH_K(h, rc = shard_serve_impl<KK>(h, recv_rows_dev, n_recv, reply_dev, st));
    return rc;
}

template <int K>
static int shard_fb_impl(dfm_handle* h, const BatchPtrs& bp, int B, const float* rowbuf, int64_t global_batch, float* loss_out,
                         float* logits_out, float* gsum, float* dense_grad, cudaStream_t st, const PeerRoute* route = nullptr) {
    const int dc = h->dc, dK = (dc + h->dn) * K;
    const int64_t n = (int64_t)B * h->dcs, t = h->step + 1;
    const int64_t l0 = h->launches;
    const StepOpts so = step_opts(h);
    const float scale = h->loss_red == DFM_LOSS_MEAN ? 1.0f / (float)global_batch : 1.0f;
    int rc;
    if (h->fused) {
        if constexpr (K <= 32) {
            // record-staged kernel in row-buffer mode: the gradient rows of the rows looked up once leave from inside it
            const bool rb = h->fused_rows_rb && gsum != nullptr;
            h->fr_rb_live = rb;
            if (rb) rc = launch_fused_rows<K>(h, bp, B, bp.labels, scale, logits_out, -1, &so, t, st, rowbuf, route ? nullptr : gsum, route);
            else rc = launch_fused<K>(h, bp, B, bp.labels, scale, logits_out, rowbuf, -1, st);
            if (rc) return rc;
            if ((rc = launch_fused_reduce(h, B, scale, loss_out, st, rb))) return rc;
            rc = fused_sparse_update<K>(h, h->ws, n, so, t, gsum, rowbuf, st, nullptr, route);
            h->fr_rb_live = false;
            if (rc) return rc;
        }
    } else {
        if ((rc = forward_impl<K>(h, bp, B, st, bp.labels, scale, logits_out, nullptr, rowbuf))) return rc;
        if ((rc = tower_backward<K>(h, bp, B, scale, loss_out, st, nullptr))) return rc;
        if (h->has_bags) {
            GradSrc<K, true> src{};
            src.dE = h->need_emb ? h->dE : nullptr; src.dz = h->dz; src.dc = dc; src.dK = dK; src.flat = nullptr; src.flat_stride = 0;
            src.n_slots = h->dcs; src.slot_field = h->d_slot_col; src.inv_cnt = h->inv_cnt;
            rc = sparse_update<K, GradSrc<K, true>>(h, h->ws, n, src, so.od, so.ol, t, gsum, st, nullptr, route);
        } else {
            GradSrc<K, false> src{};
            src.dE = h->need_emb ? h->dE : nullptr; src.dz = h->dz; src.dc = dc; src.dK = dK; src.flat = nullptr; src.flat_stride = 0;
            src.n_slots = h->dcs; src.slot_field = nullptr; src.inv_cnt = nullptr;
            rc = sparse_update<K, GradSrc<K, false>>(h, h->ws, n, src, so.od, so.ol, t, gsum, st, nullptr, route);
        }
        if (rc) return rc;
    }
    if (h->n_dense && dense_grad) CK(cudaMemcpyAsync(dense_grad, h->dg, (size_t)h->n_dense * 4, cudaMemcpyDeviceToDevice, st));
    h->last_step_launches += h->launches - l0;
    return DFM_OK;
}

extern "C" int dfm_shard_forward_backward(dfm_handle* h, const dfm_raw_batch* b, const float* rowbuf_dev, int64_t global_batch,
                                          float* loss_dev, float* logits_dev, float* gsum_dev, float* dense_grad_dev, void* stream) {
    if (!h || global_batch <= 0) return DFM_ERR_INVALID_ARG;
    if (h->world < 2) FAIL(DFM_ERR_INVALID_ARG, "handle was not created with world > 1");
    int rc = check_batch(h, b, true);
    if (rc) return rc;
    if (b->batch_size != h->shard_B) FAIL(DFM_ERR_INVALID_ARG, "batch differs from the one given to dfm_shard_requests");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    BatchPtrs bp = make_ptrs(h, b);
    DISPATCH_K(h, rc = shard_fb_impl<KK>(h, bp, b->batch_size, rowbuf_dev, global_batch, loss_dev, logits_dev, gsum_dev, dense_grad_dev, st));
    return rc;
}

// mode == EVAL / PREDICT on a row-sharded model: the rows were requested and served exactly as for a train step
// (requests -> exchange -> serve -> exchange); this is the forward pass alone, no state changes.
extern "C" int dfm_shard_forward(dfm_handle* h, const dfm_raw_batch* b, const float* rowbuf_dev, float* logits_dev, void* stream) {
    if (!h || !logits_dev) return DFM_ERR_INVALID_ARG;
    if (h->world < 2) FAIL(DFM_ERR_INVALID_ARG, "handle was not created with world > 1");
    int rc = check_batch(h, b, false);
    if (rc) return rc;
    if (b->batch_size != h->shard_B) FAIL(DFM_ERR_INVALID_ARG, "batch differs from the one given to dfm_shard_requests");
    if (!rowbuf_dev) FAIL(DFM_ERR_INVALID_ARG, "rowbuf_dev is null");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    BatchPtrs bp = make_ptrs(h, b);
    bp.labels = nullptr;
    const int64_t l0 = h->launches;
    DISPATCH_K(h, rc = eval_forward<KK>(h, bp, b->batch_size, logits_dev, rowbuf_dev, st));
    h->last_step_launches += h->launches - l0;
    if (rc) return rc;
    CK(cudaGetLastError());
    return DFM_OK;
}

template <int K>
static int shard_apply_impl(dfm_handle* h, const float* grecv, const float* dense_grad, cudaStream_t st) {
    const int64_t t = h->step + 1;
    const int64_t l0 = h->launches;
    const StepOpts so = step_opts(h);
    GradSrc<K, false> src{};
    src.dE = nullptr; src.dz = nullptr; src.dc = 1; src.dK = 0; src.flat = grecv; src.flat_stride = K + 4; src.n_slots = 1;
    src.slot_field = nullptr; src.inv_cnt = nullptr;
    int rc = sparse_update<K, GradSrc<K, false>>(h, h->ws_own, h->shard_n_recv, src, so.od, so.ol, t, nullptr, st, nullptr);
    if (rc) return rc;
    if (h->n_dense) {
        dense_apply_kernel<<<cdiv(h->n_dense, 256), 256, 0, st>>>(h->dw, h->ds1, h->ds2, dense_grad ? dense_grad : h->dg, h->n_deep, h->n_dense, so.od, so.ol);
        h->launches++;
    }
    CK(cudaGetLastError());
    commit_step(h, so, t);
    h->last_step_launches += h->launches - l0;
    return DFM_OK;
}

extern "C" int dfm_shard_apply(dfm_handle* h, const float* grecv_dev, const float* dense_grad_dev, void* stream) {
    if (!h) return DFM_ERR_INVALID_ARG;
    if (h->world < 2) FAIL(DFM_ERR_INVALID_ARG, "handle was not created with world > 1");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    int rc = DFM_OK;
    DISPATCH_K(h, rc = shard_apply_impl<KK>(h, grecv_dev, dense_grad_dev, st));
    return rc;
}

// ---- flag-synchronised exchange over NVLink peer memory (xchg.cuh) ---------------------------------
extern "C" int dfm_xchg_export(dfm_handle* h, unsigned char* out /* 64 bytes */) {
    if (!h || !out) return DFM_ERR_INVALID_ARG;
    if (h->world < 2 || !h->xreg) FAIL(DFM_ERR_UNSUPPORTED, "handle has no exchange region");
    CK(cudaSetDevice(h->device));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t mh;
    CK(cudaIpcGetMemHandle(&mh, h->xreg));
    memcpy(out, &mh, 64);
    return DFM_OK;
}

// Raw device pointer of this rank's exchange region / the table of all ranks' regions.  A host that runs several
// ranks inside ONE process (the single-GPU emulation used by the tests) wires the handles together with these two
// calls; separate processes use the IPC pair, which ends in the same table.
extern "C" int dfm_xchg_buffer(dfm_handle* h, void** out) {
    if (!h || !out) return DFM_ERR_INVALID_ARG;
    if (h->world < 2 || !h->xreg) FAIL(DFM_ERR_UNSUPPORTED, "handle has no exchange region");
    *out = h->xreg;
    return DFM_OK;
}

extern "C" int dfm_xchg_set_peers(dfm_handle* h, void* const* regions /* world, rank order */) {
    if (!h || !regions) return DFM_ERR_INVALID_ARG;
    if (h->world < 2 || !h->xreg) FAIL(DFM_ERR_UNSUPPORTED, "handle has no exchange region");
    for (int p = 0; p < h->world; ++p) {
        h->xd.peer[p] = p == h->rank ? h->xreg : reinterpret_cast<uint8_t*>(regions[p]);
        if (!h->xd.peer[p]) FAIL(DFM_ERR_INVALID_ARG, "null peer region");
    }
    h->x_ready = true;
    return DFM_OK;
}

extern "C" int dfm_xchg_import(dfm_handle* h, const unsigned char* all /* world * 64 bytes, rank order */) {
    if (!h || !all) return DFM_ERR_INVALID_ARG;
    if (h->world < 2 || !h->xreg) FAIL(DFM_ERR_UNSUPPORTED, "handle has no exchange region");
    CK(cudaSetDevice(h->device));
    void* ptrs[MAX_PEERS] = {nullptr};
    for (int p = 0; p < h->world; ++p) {
        if (p == h->rank) { ptrs[p] = h->xreg; continue; }
        if (!h->x_opened[p]) {
            cudaIpcMemHandle_t mh;
            memcpy(&mh, all + (size_t)p * 64, 64);
            CK(cudaIpcOpenMemHandle(&h->x_opened[p], mh, cudaIpcMemLazyEnablePeerAccess));
        }
        ptrs[p] = h->x_opened[p];
    }
    return dfm_xchg_set_peers(h, ptrs);
}

static int xchg_wait(dfm_handle* h, int kind, cudaStream_t st) {
    xchg_wait_kernel<<<1, 32, 0, st>>>(h->xd, kind, h->x_epoch, h->d_err);
    h->launches++;
    CK(cudaGetLastError());
    return DFM_OK;
}

// phase 1: transform + owner-major unique rows of the local batch, ids pushed into the owners' regions
template <int K>
static int xchg_begin_impl(dfm_handle* h, const BatchPtrs& bp, int B, cudaStream_t st) {
    const int64_t n = (int64_t)B * h->dcs;
    int rc = ensure_alpha(h, h->step + 1);
    if (rc) return rc;
    h->last_step_launches = 0;
    const int64_t l0 = h->launches;
    const uint32_t W = (uint32_t)h->world, limit = W * h->Rl;
    launch_transform<K>(h, bp, B, true, h->ids, st);
    if (n > 0) { shard_rekey_kernel<<<cdiv(n, 256), 256, 0, st>>>(h->ws.keys[0], n, (uint32_t)h->R, W, h->Rl); h->launches++; }
    if ((rc = build_segments(h, h->ws, n, limit, h->key_bits, st, nullptr))) return rc;
    CK(cudaMemsetAsync(h->d_counts, 0, ((size_t)W + 1) * 4, st));
    if (n > 0) {
        shard_uniq_kernel<<<cdiv(n, 256), 256, 0, st>>>(h->ws.skeys(), h->ws.svals(), n, limit, h->Rl, W, h->dcs, h->ws.pos_row, h->uidx, h->req_rows, h->d_counts, h->once_lk);
        h->launches++;
    }
    h->x_epoch += 1;
    xchg_push_kernel<<<(unsigned)std::max<int64_t>(1, std::min<int64_t>(cdiv(std::max<int64_t>(n, 1), 256), (int64_t)h->sm_count * 8)), 256, 0, st>>>(
        h->xd, (int)(h->x_epoch & 1), h->x_epoch, h->req_rows, h->d_counts, h->d_xroute, h->x_ticket + 0, h->d_err);
    h->launches++;
    h->x_B = B; h->shard_B = B;
    h->last_step_launches += h->launches - l0;
    CK(cudaGetLastError());
    return DFM_OK;
}

extern "C" int dfm_xchg_train_step_next(dfm_handle* h, const dfm_raw_batch* b, const dfm_raw_batch* next_b, int64_t global_batch,
                                        float* loss_out_dev, float* logits_dev, void* stream);
// phase 2: serve the rows my peers asked for; on the side stream, sort their ids for the gradient reduction
template <int K>
static int xchg_serve_impl(dfm_handle* h, bool train, cudaStream_t st) {
    const int64_t l0 = h->launches;
    const int64_t t = h->step + 1;
    const int par = (int)(h->x_epoch & 1);
    int rc = xchg_wait(h, XF_IDS, st);
    if (rc) return rc;
    if (train) {       // owner-side sort + segments of the received ids: beside the serve / forward / backward kernels
        CK(cudaEventRecord(h->ev_xfork, st));
        CK(cudaStreamWaitEvent(h->side_stream, h->ev_xfork, 0));
        int bits = 1;
        while ((1ull << bits) <= h->R_loc) ++bits;
        xchg_owner_keys_kernel<<<(unsigned)h->sm_count * 4, 256, 0, h->side_stream>>>(h->xd, par, h->ws_own.keys[0], h->ws_own.vals[0], (uint32_t)h->ws_own.cap,
                                                                                       h->d_nrecv, h->d_err);
        h->launches++;
        if ((rc = build_segments(h, h->ws_own, h->ws_own.cap, (uint32_t)h->R_loc, bits, h->side_stream, nullptr, h->d_nrecv))) return rc;
        CK(cudaEventRecord(h->ev_xjoin, h->side_stream));
    }
    xchg_serve_kernel<K><<<(unsigned)h->sm_count * 8, 256, 0, st>>>(h->xd, par, h->x_epoch, h->tb, (bool)h->need_emb, (bool)h->use_linear,
                                                                    make_rr(h, t - 1), make_opt(h->od, 0.f), make_opt(h->ol, 0.f), h->x_ticket + 1);
    h->launches++;
    h->last_step_launches += h->launches - l0;
    CK(cudaGetLastError());
    return DFM_OK;
}

// phase 3: forward / loss / backward from the served rows; gradient rows straight into the owners' regions; dense push
template <int K>
static int xchg_fb_impl(dfm_handle* h, const BatchPtrs& bp, int B, int64_t global_batch, float* logits_out, cudaStream_t st) {
    const int64_t l0 = h->launches;
    int rc = xchg_wait(h, XF_ROWS, st);
    if (rc) return rc;
    float* rowbuf = reinterpret_cast<float*>(h->xreg + h->xd.off_rows);
    if ((rc = shard_fb_impl<K>(h, bp, B, rowbuf, global_batch, h->d_loss_part, logits_out, rowbuf /*non-null: gradient-row mode*/, nullptr, st, h->d_xroute)))
        return rc;
    xchg_signal_kernel<<<1, 32, 0, st>>>(h->xd, XF_GRADS, h->x_epoch, h->x_ticket + 2);
    xchg_dense_push_kernel<<<dim3(cdiv(h->n_dense + 1, 256), (unsigned)h->world), 256, 0, st>>>(h->xd, h->x_epoch, h->dg, (int)h->n_dense, h->d_loss_part,
                                                                                              h->x_ticket + 3);
    h->launches += 2;
    h->last_step_launches += h->launches - l0;
    CK(cudaGetLastError());
    return DFM_OK;
}

// phase 4: ordered reduction of the received gradient rows + sparse optimizer; dense all-reduce (rank order) + dense optimizer
template <int K>
static int xchg_apply_impl(dfm_handle* h, float* loss_out, cudaStream_t st) {
    const int64_t l0 = h->launches;
    const int64_t t = h->step + 1;
    const StepOpts so = step_opts(h);
    int rc = xchg_wait(h, XF_GRADS, st);
    if (rc) return rc;
    CK(cudaStreamWaitEvent(st, h->ev_xjoin, 0));
    GradSrc<K, false> src{};
    src.dE = nullptr; src.dz = nullptr; src.dc = 1; src.dK = 0; src.flat = reinterpret_cast<const float*>(h->xreg + h->xd.off_grads);
    src.flat_stride = K + 4; src.n_slots = 1; src.slot_field = nullptr; src.inv_cnt = nullptr;
    if ((rc = sparse_update<K, GradSrc<K, false>>(h, h->ws_own, h->ws_own.cap, src, so.od, so.ol, t, nullptr, st, nullptr))) return rc;
    if ((rc = xchg_wait(h, XF_DENSE, st))) return rc;
    xchg_dense_sum_kernel<<<cdiv(h->n_dense + 1, 256), 256, 0, st>>>(h->xd, (int)h->n_dense, h->d_dense_total, loss_out);
    h->launches++;
    if (h->n_dense) {
        dense_apply_kernel<<<cdiv(h->n_dense, 256), 256, 0, st>>>(h->dw, h->ds1, h->ds2, h->d_dense_total, h->n_deep, h->n_dense, so.od, so.ol);
        h->launches++;
    }
    CK(cudaGetLastError());
    commit_step(h, so, t);
    h->last_step_launches += h->launches - l0;
    return DFM_OK;
}

static int xchg_check(dfm_handle* h) {
    if (h->world < 2 || !h->xreg) FAIL(DFM_ERR_INVALID_ARG, "handle was not created with 1 < world <= 16");
    if (!h->x_ready) FAIL(DFM_ERR_INVALID_ARG, "call dfm_xchg_import / dfm_xchg_set_peers first");
    return DFM_OK;
}

extern "C" int dfm_xchg_begin(dfm_handle* h, const dfm_raw_batch* b, void* stream) {
    if (!h) return DFM_ERR_INVALID_ARG;
    int rc = xchg_check(h);
    if (rc) return rc;
    if ((rc = check_batch(h, b, false))) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    BatchPtrs bp = make_ptrs(h, b);
    DISPATCH_K(h, rc = xchg_begin_impl<KK>(h, bp, b->batch_size, st));
    return rc;
}

extern "C" int dfm_xchg_serve(dfm_handle* h, int32_t train, void* stream) {
    if (!h) return DFM_ERR_INVALID_ARG;
    int rc = xchg_check(h);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    DISPATCH_K(h, rc = xchg_serve_impl<KK>(h, train != 0, st));
    return rc;
}

extern "C" int dfm_xchg_forward_backward(dfm_handle* h, const dfm_raw_batch* b, int64_t global_batch, float* logits_dev, void* stream) {
    if (!h || global_batch <= 0) return DFM_ERR_INVALID_ARG;
    int rc = xchg_check(h);
    if (rc) return rc;
    if ((rc = check_batch(h, b, true))) return rc;
    if (b->batch_size != h->x_B) FAIL(DFM_ERR_INVALID_ARG, "batch differs from the one given to dfm_xchg_begin");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    BatchPtrs bp = make_ptrs(h, b);
    DISPATCH_K(h, rc = xchg_fb_impl<KK>(h, bp, b->batch_size, global_batch, logits_dev, st));
    return rc;
}

extern "C" int dfm_xchg_apply(dfm_handle* h, float* loss_out_dev, void* stream) {
    if (!h) return DFM_ERR_INVALID_ARG;
    int rc = xchg_check(h);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    DISPATCH_K(h, rc = xchg_apply_impl<KK>(h, loss_out_dev, st));
    return rc;
}

// mode == EVAL / PREDICT: after dfm_xchg_begin + dfm_xchg_serve(train = 0) the forward pass alone on the served rows
extern "C" int dfm_xchg_forward(dfm_handle* h, const dfm_raw_batch* b, float* logits_dev, void* stream) {
    if (!h || !logits_dev) return DFM_ERR_INVALID_ARG;
    int rc = xchg_check(h);
    if (rc) return rc;
    if ((rc = check_batch(h, b, false))) return rc;
    if (b->batch_size != h->x_B) FAIL(DFM_ERR_INVALID_ARG, "batch differs from the one given to dfm_xchg_begin");
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    BatchPtrs bp = make_ptrs(h, b);
    bp.labels = nullptr;
    const int64_t l0 = h->launches;
    if ((rc = xchg_wait(h, XF_ROWS, st))) return rc;
    DISPATCH_K(h, rc = eval_forward<KK>(h, bp, b->batch_size, logits_dev, reinterpret_cast<float*>(h->xreg + h->xd.off_rows), st));
    h->last_step_launches += h->launches - l0;
    return rc;
}

// One whole step for a one-process-per-GPU host: the four phases back to back on `stream`, nothing but kernel
// launches (no collective, no host synchronisation); the peers' kernels meet through the flags.
extern "C" int dfm_xchg_train_step(dfm_handle* h, const dfm_raw_batch* b, int64_t global_batch, float* loss_out_dev, float* logits_dev,
                                   void* stream) {
    return dfm_xchg_train_step_next(h, b, nullptr, global_batch, loss_out_dev, logits_dev, stream);
}

// The same step with the requests of the NEXT batch (transform, owner-major sort, unique rows, push of the ids: no model
// state involved) issued on the side stream as soon as this step's forward / backward has read the request buffers, i.e.
// beside this step's owner-side apply.  The next call must be given that batch (every rank alike: the exchange round was
// opened); it then skips its own begin phase.  Results are bit-identical to the unprefetched sequence.
extern "C" int dfm_xchg_train_step_next(dfm_handle* h, const dfm_raw_batch* b, const dfm_raw_batch* next_b, int64_t global_batch,
                                        float* loss_out_dev, float* logits_dev, void* stream) {
    if (!h || !b) return DFM_ERR_INVALID_ARG;
    int rc = xchg_check(h);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    if (h->x_pf_valid) {
        if (b->batch_size != h->x_pf_B || (h->dc > 0 && batch_tag(h, b->cat_data) != h->x_pf_tag))
            FAIL(DFM_ERR_INVALID_ARG, "dfm_xchg_train_step_next: the batch announced as next_batch must be trained next");
        h->x_pf_valid = false;
        CK(cudaStreamWaitEvent(st, h->ev_xpf_done, 0));
    } else if ((rc = dfm_xchg_begin(h, b, st))) {
        return rc;
    }
    if ((rc = dfm_xchg_serve(h, 1, st))) return rc;
    if ((rc = dfm_xchg_forward_backward(h, b, global_batch, logits_dev, st))) return rc;
    if (next_b) CK(cudaEventRecord(h->ev_xpf_fork, st));       // the request buffers of this step have been consumed
    if ((rc = dfm_xchg_apply(h, loss_out_dev, st))) return rc;
    if (next_b) {
        CK(cudaStreamWaitEvent(h->side_stream, h->ev_xpf_fork, 0));
        if ((rc = dfm_xchg_begin(h, next_b, h->side_stream))) return rc;
        CK(cudaEventRecord(h->ev_xpf_done, h->side_stream));
        h->x_pf_valid = true; h->x_pf_B = next_b->batch_size; h->x_pf_tag = h->dc > 0 ? batch_tag(h, next_b->cat_data) : nullptr;
    }
    return DFM_OK;
}

// --------------------------------------------------------------------------- host entry points
// Copies the raw columns of a host batch into the stage's device arena.  When the caller laid the
// columns out back to back in one (pinned) allocation this is a single cudaMemcpyAsync.
static int stage_batch(dfm_handle* h, const dfm_raw_batch* b, HostStage& sg, bool need_labels, BatchPtrs& out, size_t* h2d_bytes) {
    struct Seg { const uint8_t* p; size_t bytes; const void** dst; };
    std::vector<Seg> segs;
    const int B = b->batch_size;
    out = BatchPtrs{};
    for (int f = 0; f < h->dc + h->n_src; ++f) {
        if (h->cols[f].kind == DFM_COL_CROSSED) continue;          // no raw data of its own: the sources are staged
        const size_t nv = (size_t)B * h->cols[f].width;      // values of this column in the batch (multivalent: B * width)
        if (h->cols[f].dtype == DFM_STRING) {
            const int32_t* off = b->cat_offsets[f];
            segs.push_back({reinterpret_cast<const uint8_t*>(off), (nv + 1) * 4, reinterpret_cast<const void**>(&out.off[f])});
            size_t nbytes = (size_t)off[nv];
            segs.push_back({reinterpret_cast<const uint8_t*>(b->cat_data[f]), std::max<size_t>(nbytes, 1), &out.cat[f]});
        } else {
            segs.push_back({reinterpret_cast<const uint8_t*>(b->cat_data[f]), nv * 4, &out.cat[f]});
        }
    }
    for (int j = 0; j < h->dn; ++j)
        segs.push_back({reinterpret_cast<const uint8_t*>(b->num_data[j]), (size_t)B * 4, reinterpret_cast<const void**>(&out.num[j])});
    if (need_labels) segs.push_back({reinterpret_cast<const uint8_t*>(b->labels), (size_t)B * 4, reinterpret_cast<const void**>(&out.labels)});
    const uint8_t* lo = nullptr; const uint8_t* hi = nullptr; size_t sum = 0;
    for (const Seg& s : segs) {
        if (!lo || s.p < lo) lo = s.p;
        if (!hi || s.p + s.bytes > hi) hi = s.p + s.bytes;
        sum += (s.bytes + 255) / 256 * 256;
    }
    const size_t span = (size_t)(hi - lo);
    const bool contiguous = span <= sum + 4096;
    const size_t need = contiguous ? span + 256 : sum + 256;
    if (sg.cap < need) {
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaStreamSynchronize(h->copy_stream));
        if (sg.d_arena) CK(cudaFree(sg.d_arena));
        sg.cap = need + need / 4;
        CK(cudaMalloc(&sg.d_arena, sg.cap));
    }
    size_t bytes = 0;
    if (contiguous) {
        // keep the 16-byte phase of the host layout so aligned columns stay aligned
        size_t phase = reinterpret_cast<uintptr_t>(lo) & 255;
        CK(cudaMemcpyAsync(sg.d_arena + phase, lo, span, cudaMemcpyHostToDevice, h->copy_stream));
        for (const Seg& s : segs) *s.dst = sg.d_arena + phase + (s.p - lo);
        bytes = span;
    } else {
        size_t o = 0;
        for (const Seg& s : segs) {
            CK(cudaMemcpyAsync(sg.d_arena + o, s.p, s.bytes, cudaMemcpyHostToDevice, h->copy_stream));
            *s.dst = sg.d_arena + o;
            o += (s.bytes + 255) / 256 * 256;
            bytes += s.bytes;
        }
    }
    if (h2d_bytes) *h2d_bytes = bytes;
    return DFM_OK;
}

static int enqueue_host_step(dfm_handle* h, const dfm_raw_batch* b, int slot) {
    HostStage& sg = h->stage[slot];
    if (sg.busy) { CK(cudaEventSynchronize(sg.done)); sg.busy = false; }
    BatchPtrs bp;
    int rc = stage_batch(h, b, sg, true, bp, nullptr);
    if (rc) return rc;
    CK(cudaEventRecord(sg.copied, h->copy_stream));
    CK(cudaStreamWaitEvent(h->stream, sg.copied, 0));
    static const bool graphs = getenv("DFM_NO_GRAPH") == nullptr;
    if (graphs && graph_step_ok(h, b->batch_size)) rc = train_step_graphed(h, bp, b->batch_size, nullptr, nullptr, h->stream);
    else DISPATCH_K(h, rc = train_impl<KK>(h, bp, b->batch_size, nullptr, nullptr, h->stream));
    if (rc) return rc;
    CK(cudaMemcpyAsync(sg.h_loss, h->d_loss, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaEventRecord(sg.done, h->stream));
    sg.busy = true;
    return DFM_OK;
}

extern "C" int dfm_train_step_host_async(dfm_handle* h, const dfm_raw_batch* b, float* prev_loss) {
    if (!h) return DFM_ERR_INVALID_ARG;
    int rc = check_batch(h, b, true);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    const int slot = (int)(h->host_calls & 1);
    const int prev = h->last_slot;
    rc = enqueue_host_step(h, b, slot);
    if (rc) return rc;
    h->host_calls++;
    h->last_slot = slot;
    if (prev_loss) {
        if (prev >= 0 && prev != slot) {
            CK(cudaEventSynchronize(h->stage[prev].done));
            h->stage[prev].busy = false;
            *prev_loss = *h->stage[prev].h_loss;
        } else {
            *prev_loss = NAN;
        }
    }
    return DFM_OK;
}

extern "C" int dfm_train_step_host_drain(dfm_handle* h, float* last_loss) {
    if (!h) return DFM_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (h->last_slot < 0) { if (last_loss) *last_loss = NAN; return DFM_OK; }
    HostStage& sg = h->stage[h->last_slot];
    CK(cudaEventSynchronize(sg.done));
    sg.busy = false;
    if (last_loss) *last_loss = *sg.h_loss;
    h->last_slot = -1;
    return DFM_OK;
}

extern "C" int dfm_train_step_host(dfm_handle* h, const dfm_raw_batch* b, float* loss_out, float* logits_out) {
    if (!h) return DFM_ERR_INVALID_ARG;
    int rc = check_batch(h, b, true);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    const int slot = (int)(h->host_calls & 1);
    rc = enqueue_host_step(h, b, slot);
    if (rc) return rc;
    h->host_calls++;
    h->last_slot = -1;
    if (logits_out) CK(cudaMemcpyAsync(logits_out, h->logits, (size_t)b->batch_size * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->stage[slot].busy = false;
    if (loss_out) *loss_out = *h->stage[slot].h_loss;
    return DFM_OK;
}

extern "C" int dfm_forward_host(dfm_handle* h, const dfm_raw_batch* b, float* logits_out) {
    if (!h || !logits_out) return DFM_ERR_INVALID_ARG;
    if (h->world > 1) FAIL(DFM_ERR_UNSUPPORTED, "row-sharded handle: use dfm_shard_requests / serve / dfm_shard_forward");
    int rc = check_batch(h, b, false);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    HostStage& sg = h->stage[0];
    if (sg.busy) { CK(cudaEventSynchronize(sg.done)); sg.busy = false; }
    CK(cudaStreamSynchronize(h->stream));
    BatchPtrs bp;
    rc = stage_batch(h, b, sg, false, bp, nullptr);
    if (rc) return rc;
    CK(cudaEventRecord(sg.copied, h->copy_stream));
    CK(cudaStreamWaitEvent(h->stream, sg.copied, 0));
    rc = ensure_alpha(h, h->step);
    if (rc) return rc;
    launch_transform<4>(h, bp, b->batch_size, false, h->ids, h->stream);
    DISPATCH_K(h, rc = eval_forward<KK>(h, bp, b->batch_size, nullptr, nullptr, h->stream));
    if (rc) return rc;
    CK(cudaMemcpyAsync(logits_out, h->logits, (size_t)b->batch_size * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    return DFM_OK;
}

// ------------------------------------------------------------------- building-block test hooks
extern "C" int dfm_test_sort_pairs(uint32_t* keys_dev, uint32_t* vals_dev, int64_t n, int32_t key_bits) {
    dfm_handle* h = nullptr;
    if (n <= 0) return DFM_OK;
    uint32_t *k[2] = {keys_dev, nullptr}, *v[2] = {vals_dev, nullptr};
    void* temp = nullptr;
    CK(cudaMalloc(&k[1], n * 4));
    CK(cudaMalloc(&v[1], n * 4));
    CK(cudaMalloc(&temp, prims::sort_temp_bytes(n)));
    int cur = prims::radix_sort_pairs(k, v, n, key_bits, temp, 0, nullptr);
    if (cur == 1) {
        CK(cudaMemcpyAsync(keys_dev, k[1], n * 4, cudaMemcpyDeviceToDevice, 0));
        CK(cudaMemcpyAsync(vals_dev, v[1], n * 4, cudaMemcpyDeviceToDevice, 0));
    }
    CK(cudaDeviceSynchronize());
    cudaFree(k[1]); cudaFree(v[1]); cudaFree(temp);
    CK(cudaGetLastError());
    return DFM_OK;
}

// algo 0: multi-launch LSD sort; 1: one-sweep; 2: one-sweep with the element count in device memory (grids sized for
// a larger bound, as on the row-sharded owner side)
extern "C" int dfm_test_sort_pairs_algo(uint32_t* keys_dev, uint32_t* vals_dev, int64_t n, int32_t key_bits, int32_t algo) {
    dfm_handle* h = nullptr;
    if (n <= 0) return DFM_OK;
    if (algo == 0) return dfm_test_sort_pairs(keys_dev, vals_dev, n, key_bits);
    const int64_t n_max = algo == 2 ? n + 100000 : n;
    uint32_t *k[2] = {keys_dev, nullptr}, *v[2] = {vals_dev, nullptr};
    void* temp = nullptr; uint32_t* n_dev = nullptr;
    CK(cudaMalloc(&k[1], n * 4));
    CK(cudaMalloc(&v[1], n * 4));
    CK(cudaMalloc(&temp, prims::onesweep_temp_bytes(n_max)));
    if (algo == 2) {
        const uint32_t nn = (uint32_t)n;
        CK(cudaMalloc(&n_dev, 4));
        CK(cudaMemcpy(n_dev, &nn, 4, cudaMemcpyHostToDevice));
    }
    int cur = prims::onesweep_sort_pairs(k, v, n_max, n_dev, key_bits, temp, 0, nullptr);
    if (cur == 1) {
        CK(cudaMemcpyAsync(keys_dev, k[1], n * 4, cudaMemcpyDeviceToDevice, 0));
        CK(cudaMemcpyAsync(vals_dev, v[1], n * 4, cudaMemcpyDeviceToDevice, 0));
    }
    cudaError_t e = cudaDeviceSynchronize();
    cudaFree(k[1]); cudaFree(v[1]); cudaFree(temp); if (n_dev) cudaFree(n_dev);
    CK(e);
    CK(cudaGetLastError());
    return DFM_OK;
}

extern "C" int dfm_test_fingerprint64(const uint8_t* bytes_dev, const int32_t* offsets_dev, int64_t n, uint64_t* out_dev) {
    dfm_handle* h = nullptr;
    if (n <= 0) return DFM_OK;
    fingerprint_kernel<<<cdiv(n, 256), 256>>>(bytes_dev, offsets_dev, n, out_dev);
    CK(cudaDeviceSynchronize());
    CK(cudaGetLastError());
    return DFM_OK;
}

// test hook: non-lazy Adam replay of n independent elements (device arrays) from step last[i] to step upto
__global__ void test_replay_kernel(float* __restrict__ w, float* __restrict__ m, float* __restrict__ v, const int32_t* __restrict__ last,
                                   int64_t n, RowReplay rr, OptDev od) {
    const ReplayStep rs = replay_step_load(rr.rd, rr.upto);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 w4 = make_float4(w[i], 0.f, 0.f, 0.f), m4 = make_float4(m[i], 0.f, 0.f, 0.f), v4 = make_float4(v[i], 0.f, 0.f, 0.f);
    float4 lr = make_float4(0.f, 0.f, 0.f, __int_as_float(last[i]));
    replay_row(w4, m4, v4, lr, false, rr, rs, od, od);
    w[i] = w4.x; m[i] = m4.x; v[i] = v4.x;
}

extern "C" int dfm_test_replay(const dfm_optimizer* opt, float* w_dev, float* m_dev, float* v_dev, const int32_t* last_dev, int64_t n,
                               int32_t upto, int32_t force_loop) {
    dfm_handle* h = nullptr;
    if (!opt || n < 0 || upto < 0) return DFM_ERR_INVALID_ARG;
    if (n == 0) return DFM_OK;
    dfm_handle tmp;                          // only the stream (0) and the error string are used
    ReplayHost r;
    if (force_loop) setenv("DFM_REPLAY_LOOP", "1", 1);
    int rc = build_replay_group(&tmp, r, *opt, (int64_t)upto + 2);
    if (force_loop) unsetenv("DFM_REPLAY_LOOP");
    if (rc) { g_create_error = tmp.err; free_replay(r); return rc; }
    RowReplay rr{};
    rr.rd = r.tab; rr.rl = r.tab; rr.upto = upto; rr.emb_adam = 1; rr.lin_adam = 0; rr.same = 1;
    test_replay_kernel<<<cdiv(n, 256), 256>>>(w_dev, m_dev, v_dev, last_dev, n, rr, make_opt(*opt, 0.f));
    cudaError_t e = cudaDeviceSynchronize();
    free_replay(r);
    CK(e);
    CK(cudaGetLastError());
    return DFM_OK;
}

static bool tc_presplit() {
    static const int v = getenv("DFM_TC_PRESPLIT") ? atoi(getenv("DFM_TC_PRESPLIT")) : 1;     // 0: split the weights in every CTA (A/B runs)
    return v != 0;
}

// ------------------------------------------------------------------------- tensor-core GEMM host
// C[M,N] = A[M,K] * B[N,K]^T  (both K-major).  A_lo / B_lo == nullptr -> the operand is split into
// tf32 hi/lo inside the kernel; otherwise hi/lo were produced beforehand (weights).
static unsigned long long* g_tc_ts = nullptr;   // experiments only (DFM_TC_TS in dfm_test_tc_gemm)
static int tc_gemm_kmajor(dfm_handle* h, const float* A_hi, const float* A_lo, int lda, const float* B_hi, const float* B_lo, int ldb,
                          float* C, int ldc, int M, int N, int K, int epi, const EpiArgs& ep, cudaStream_t st) {
    static const int persist = getenv("DFM_TC_PERSIST") ? atoi(getenv("DFM_TC_PERSIST")) : 1;   // 0: one CTA per tile (A/B runs)
    const int BN = persist ? tc::P_BN : N > 128 ? 256 : 128;
    const int bk = persist ? tc::P_BK : TC_BK;
    const int ntile = (N + BN - 1) / BN;
    const int bn = std::min(BN, ((N + ntile - 1) / ntile + 15) / 16 * 16);   // equal tiles, multiple of 16 (UMMA N granularity)
    CUtensorMap ma, mal, mb, mbl;
    bool ok = tc::make_map_2d(&ma, A_hi, M, K, lda, tc::BM, bk) && tc::make_map_2d(&mal, A_lo ? A_lo : A_hi, M, K, lda, tc::BM, bk) &&
              tc::make_map_2d(&mb, B_hi, N, K, ldb, bn, bk) && tc::make_map_2d(&mbl, B_lo ? B_lo : B_hi, N, K, ldb, bn, bk);
    if (!ok) FAIL(DFM_ERR_CUDA, "cuTensorMapEncodeTiled failed");
    tc::Params p{};
    p.M = M; p.N = N; p.K = K; p.k_per_split = K; p.C = C; p.ldc = ldc; p.c_split_stride = 0; p.epi = epi; p.ep = ep;
    p.split_a = A_lo ? 0 : 1; p.split_b = B_lo ? 0 : 1;
    p.bn = bn;
    if (const char* e = getenv("DFM_TC_DBG")) p.dbg = atoi(e);
    p.ts = g_tc_ts;
    dim3 grid(cdiv(N, bn), cdiv(M, tc::BM), 1);
    if (persist) {
        static int sms = 0;
        if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); }
        const int tiles = cdiv(N, bn) * cdiv(M, tc::BM);
        tc::gemm_persist_kernel<tc::P_BK><<<std::min(tiles, sms), tc::P_THREADS, tc::PSmem<tc::P_BK>::TOTAL, st>>>(ma, mal, mb, mbl, p);
    } else if (BN == 256) tc::gemm_kernel<256, 0, TC_BK><<<grid, tc::NTHREADS, tc::Smem<256, TC_BK>::TOTAL, st>>>(ma, mal, mb, mbl, p);
    else tc::gemm_kernel<128, 0, TC_BK><<<grid, tc::NTHREADS, tc::Smem<128, TC_BK>::TOTAL, st>>>(ma, mal, mb, mbl, p);
    if (h) h->launches++;
    CK(cudaGetLastError());
    return DFM_OK;
}

// Cpartial[z][M,N] = sum over k in split z of A[k,M]^T * B[k,N]  (both MN-major, reduction over rows = batch)
static int tc_gemm_mnmajor(dfm_handle* h, const float* A, int lda, const float* B, int ldb, float* Cpart, int M, int N, int K, int splits,
                           int* k_per_split_out, cudaStream_t st) {
    if (M % 32 || N % 32) FAIL(DFM_ERR_UNSUPPORTED, "tc_gemm_mnmajor needs M, N multiples of 32");
    const int BN = N > 128 ? 256 : 128;
    CUtensorMap ma, mb;
    bool ok = tc::make_map_3d(&ma, A, K, M, lda, TC_BK, tc::BM / 32) && tc::make_map_3d(&mb, B, K, N, ldb, TC_BK, BN / 32);
    if (!ok) FAIL(DFM_ERR_CUDA, "cuTensorMapEncodeTiled failed");
    splits = tc_wgrad_splits(K, splits);
    int kps = ((K + splits - 1) / splits + TC_BK - 1) / TC_BK * TC_BK;
    int nz = (K + kps - 1) / kps;
    if (k_per_split_out) *k_per_split_out = nz;
    tc::Params p{};
    p.M = M; p.N = N; p.K = K; p.k_per_split = kps; p.C = Cpart; p.ldc = N; p.c_split_stride = (size_t)M * N; p.epi = EPI_NONE;
    p.split_a = 1; p.split_b = 1;
    p.bn = BN;
    if (const char* e = getenv("DFM_TC_DBG")) p.dbg = atoi(e);
    dim3 grid(cdiv(N, BN), cdiv(M, tc::BM), nz);
    if (BN == 256) tc::gemm_kernel<256, 1, TC_BK><<<grid, tc::NTHREADS, tc::Smem<256, TC_BK>::TOTAL, st>>>(ma, ma, mb, mb, p);
    else tc::gemm_kernel<128, 1, TC_BK><<<grid, tc::NTHREADS, tc::Smem<128, TC_BK>::TOTAL, st>>>(ma, ma, mb, mb, p);
    if (h) h->launches++;
    CK(cudaGetLastError());
    return DFM_OK;
}

static int tc_setup_once() {
    static int done = 0;
    if (done) return done;
    cudaError_t e = cudaSuccess;
    e = cudaFuncSetAttribute(tc::gemm_kernel<256, 0, TC_BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::Smem<256, TC_BK>::TOTAL); if (e) return done = -1;
    e = cudaFuncSetAttribute(tc::gemm_kernel<128, 0, TC_BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::Smem<128, TC_BK>::TOTAL); if (e) return done = -1;
    e = cudaFuncSetAttribute(tc::gemm_kernel<256, 1, TC_BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::Smem<256, TC_BK>::TOTAL); if (e) return done = -1;
    e = cudaFuncSetAttribute(tc::gemm_kernel<128, 1, TC_BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::Smem<128, TC_BK>::TOTAL); if (e) return done = -1;
    e = cudaFuncSetAttribute(tc::gemm_persist_kernel<tc::P_BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::PSmem<tc::P_BK>::TOTAL); if (e) return done = -1;
    return done = 1;
}

// test hook: mode 0: C[M,N] = A[M,K] B[N,K]^T (both split in-kernel); mode 2: same with B pre-split on the host side of
// the call; mode 1: C[M,N] = A[K,M]^T B[K,N] through `splits` deterministic partials.
extern "C" int dfm_test_tc_gemm(int32_t mode, const float* A, const float* B, float* C, int32_t M, int32_t N, int32_t K, int32_t splits) {
    dfm_handle* h = nullptr;
    if (tc_setup_once() < 0) FAIL(DFM_ERR_CUDA, "tc setup failed");
    EpiArgs ep{};
    int rc = DFM_OK;
    if (mode == 0) {
        rc = tc_gemm_kmajor(nullptr, A, nullptr, K, B, nullptr, K, C, N, M, N, K, EPI_NONE, ep, 0);
    } else if (mode == 2) {
        float *bh = nullptr, *bl = nullptr;
        CK(cudaMalloc(&bh, (size_t)N * K * 4)); CK(cudaMalloc(&bl, (size_t)N * K * 4));
        tc::split_tf32_kernel<<<cdiv((int64_t)N * K, 256), 256>>>(B, (int64_t)N * K, bh, bl);
        rc = tc_gemm_kmajor(nullptr, A, nullptr, K, bh, bl, K, C, N, M, N, K, EPI_NONE, ep, 0);
        CK(cudaDeviceSynchronize());
        if (getenv("DFM_TC_TS") && rc == DFM_OK) {
            // per-CTA phase timeline of one warm launch (ns, globaltimer), printed as a summary on stderr
            const int nct = cdiv(M, tc::BM) * 4;
            unsigned long long* ts = nullptr;
            CK(cudaMalloc(&ts, (size_t)nct * 8 * 8));
            CK(cudaMemset(ts, 0, (size_t)nct * 8 * 8));
            if (getenv("DFM_TC_FLUSH")) {     // evict the operands from L2 first (the in-step situation)
                void* junk = nullptr;
                CK(cudaMalloc(&junk, (size_t)512 << 20));
                CK(cudaMemset(junk, 1, (size_t)512 << 20));
                CK(cudaDeviceSynchronize());
                cudaFree(junk);
            }
            cudaEvent_t e0, e1;
            cudaEventCreate(&e0); cudaEventCreate(&e1);
            g_tc_ts = ts;
            cudaEventRecord(e0, 0);
            rc = tc_gemm_kmajor(nullptr, A, nullptr, K, bh, bl, K, C, N, M, N, K, EPI_NONE, ep, 0);
            cudaEventRecord(e1, 0);
            g_tc_ts = nullptr;
            CK(cudaDeviceSynchronize());
            float ems = 0.f;
            cudaEventElapsedTime(&ems, e0, e1);
            fprintf(stderr, "[tc-ts] launch %.1f us (events)%s\n", ems * 1e3, getenv("DFM_TC_FLUSH") ? " after L2 flush" : "");
            cudaEventDestroy(e0); cudaEventDestroy(e1);
            std::vector<unsigned long long> hts((size_t)nct * 8);
            CK(cudaMemcpy(hts.data(), ts, hts.size() * 8, cudaMemcpyDeviceToHost));
            cudaFree(ts);
            static const int persist = getenv("DFM_TC_PERSIST") ? atoi(getenv("DFM_TC_PERSIST")) : 1;
            if (persist) {
                double acc[8] = {0}; int n = 0;
                for (int c = 0; c < 148 && c < nct; ++c) {
                    const unsigned long long* e = &hts[(size_t)c * 8];
                    if (!e[0]) continue;
                    ++n;
                    for (int k = 0; k < 8; ++k) acc[k] += (double)e[k];
                }
                fprintf(stderr, "[tc-ts persist] M=%d N=%d K=%d ctas=%d mean cycles: total=%.0f | tma wait_empty=%.0f | mma wait_split=%.0f wait_acc_empty=%.0f | "
                                "split wait_full=%.0f busy=%.0f | epi wait_acc_full=%.0f busy=%.0f\n",
                        M, N, K, n, acc[0] / n, acc[1] / n, acc[2] / n, acc[3] / n, acc[4] / n, acc[6] / n, acc[5] / n, acc[7] / n);
            } else {
            unsigned long long t0 = ~0ull, t1 = 0; int n = 0;
            double acc[7] = {0};
            for (int c = 0; c < nct; ++c) {
                const unsigned long long* e = &hts[(size_t)c * 8];
                if (!e[0]) continue;
                ++n; t0 = std::min(t0, e[0]); t1 = std::max(t1, e[6]);
                for (int k = 1; k < 7; ++k) acc[k] += (double)(e[k] - e[0]);
            }
            fprintf(stderr, "[tc-ts] M=%d N=%d K=%d ctas=%d makespan=%.1f us | mean ns since CTA start: tma_issued=%.0f mma_issued=%.0f first_split=%.0f last_split=%.0f accum_done=%.0f end=%.0f\n",
                    M, N, K, n, (t1 - t0) * 1e-3, acc[1] / n, acc[2] / n, acc[3] / n, acc[4] / n, acc[5] / n, acc[6] / n);
            // CTAs per SM and the idle gaps between consecutive CTAs of SM 0's timeline
            std::vector<std::pair<unsigned long long, unsigned long long>> sm0;
            const unsigned long long sm_first = hts[7];
            for (int c = 0; c < nct; ++c) if (hts[(size_t)c * 8] && hts[(size_t)c * 8 + 7] == sm_first) sm0.push_back({hts[(size_t)c * 8], hts[(size_t)c * 8 + 6]});
            std::sort(sm0.begin(), sm0.end());
            fprintf(stderr, "[tc-ts] SM %llu timeline (start,end us rel.):", sm_first);
            for (auto& pr : sm0) fprintf(stderr, " (%.1f,%.1f)", (pr.first - t0) * 1e-3, (pr.second - t0) * 1e-3);
            fprintf(stderr, "\n");
            }
        }
        cudaFree(bh); cudaFree(bl);
    } else {
        float* part = nullptr;
        int nz = 0;
        const int eff = tc_wgrad_splits(K, std::max(splits, 1));
        CK(cudaMalloc(&part, (size_t)eff * M * N * 4 + 16));
        rc = tc_gemm_mnmajor(nullptr, A, M, B, N, part, M, N, K, eff, &nz, 0);
        if (rc == DFM_OK) reduce_partials_kernel<<<cdiv((int64_t)M * N, 256), 256>>>(part, nz, (size_t)M * N, (int64_t)M * N, C);
        CK(cudaDeviceSynchronize());
        cudaFree(part);
    }
    if (rc) return rc;
    CK(cudaDeviceSynchronize());
    CK(cudaGetLastError());
    return DFM_OK;
}
