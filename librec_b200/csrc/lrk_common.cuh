// Shared declarations of the B200-native LibRec MF path (handle layout, error plumbing).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <type_traits>
#include <unordered_map>
#include "../../include/librec_b200.h"

#define LRK_MAX_FACTORS 256
#define LRK_MAX_TOPN 512

struct lrk_handle_s {
    lrk_config_t cfg{};
    int k = 0;        // rec.factor.number
    int ld = 0;       // padded fp32 row length: power of two >= max(k,4); multiple of 128 above 128
    int G = 0;        // lanes cooperating on one rating (each lane owns V float4 of a row)
    int V = 1;
    int32_t U = 0, I = 0;
    int64_t nnz = 0;
    int sm_count = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t copy_stream = nullptr;          // second stream: the H2D copy of the rating values overlaps the sort of the staging
    cudaEvent_t ev_copy0 = nullptr, ev_copy1 = nullptr;

    // train CSR (device): membership for BPR sampling and the top-N train mask
    int64_t* d_rowptr = nullptr;
    int32_t* d_col = nullptr;
    // shuffled COO stream for the SGD epoch (SoA, 12 B / rating)
    int32_t* d_su = nullptr;
    int32_t* d_si = nullptr;
    float* d_sr = nullptr;
    bool has_train = false;
    void* group = nullptr;    // GroupUnits*: the stream is unit-ordered (staging_group.cuh) and the epoch runs sgd_group_epoch_kernel
    int64_t run_tiles = 0;    // 32-rating item-run tiles in the staged stream (lrk_stage_stats)
    uint32_t max_item_deg = 0;
    double hot_share = 0.0;   // largest share one item has of the train ratings (stability cap of the SGD grid)
    float* d_pnorm2 = nullptr;        // mean |p_u|^2 at the start of the epoch (curvature term of that step)
    float pnorm2_host = 0.f;          // its host copy, refreshed with every loss read-back (picks the kernel variant)
    float pnorm2_prev = 0.f;          // the value one epoch earlier (growth of the user factors, sgd_launch_gv)
    uint32_t* d_item_deg = nullptr;   // ratings per item in this handle's shard (staleness-aware step of run tiles, sgd.cuh)
    uint32_t* d_item_cum = nullptr;   // RankSGD: inclusive prefix sums of d_item_deg (negative sampling table)

    // factors: fp32 working copies (padded rows) + fp64 masters (dense rows, what Java sees)
    float *P32 = nullptr, *Q32 = nullptr, *bu32 = nullptr, *bi32 = nullptr;
    double *P64 = nullptr, *Q64 = nullptr, *bu64 = nullptr, *bi64 = nullptr;
    double mu = 0.0;
    bool has_factors = false;
    bool f64_valid = false;   // masters are in sync with the fp32 working copies

    // Safeguard of the fast SGD mode (lrk_epoch.cuh): factors are snapshotted before an epoch; a non-finite (or exploding) loss
    // rolls the epoch back and re-runs it with 4x fewer ratings in flight (sticky, relaxed again after 8 good epochs)
    float *bk_P = nullptr, *bk_Q = nullptr, *bk_bu = nullptr, *bk_bi = nullptr;
    int conc_div = 1;           // divisor of the SGD grid
    int good_epochs = 0;
    double prev_loss = -1.0;    // loss of the last accepted epoch (< 0: none yet)
    int64_t rollbacks = 0;
    int epochs_done = 0;        // accepted epochs since lrk_set_factors (picks the kernel variant of the first epochs)
    double* d_loss = nullptr;   // device accumulator
    double* h_loss = nullptr;   // pinned
    float* h_pnorm2 = nullptr;  // pinned
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    float last_epoch_ms = 0.f;
    uint64_t launches = 0;

    // top-N statistics
    int64_t topn_fast_users = 0, topn_fallback_users = 0, topn_resweep_users = 0;
    float topn_ms = 0.f;
    float topn_phase_ms[4] = {0.f, 0.f, 0.f, 0.f};
    float topn_err_ratio = 0.f;   // largest observed |fp16 sweep score - exact score| / certificate bound (must be < 1)
    // result buffers of lrk_topn, reused across calls (cudaMalloc/cudaFree of 130 MB cost 20-400 ms per call)
    int32_t *tn_users = nullptr, *tn_items = nullptr, *tn_counts = nullptr;
    double* tn_scores = nullptr;
    // tensor-core top-N state (bf16 copies, norms); see topn_tc.cuh
    void* tc = nullptr;

    void* gbpr = nullptr;     // GbprState* (sgd_gbpr.cuh)
    void* svdpp = nullptr;    // SvdppState* (sgd_svdpp.cuh)
    void* aobpr = nullptr;    // AobprState* (sgd_aobpr.cuh)
    void* als = nullptr;      // AlsState* (als.cuh): WRMF / eALS

    // reference-order (wavefront) schedule, see sgd_exact.cuh
    void* exact = nullptr;

    // single-process multi-GPU parent (multi.cuh): no device state of its own, forwards to one child per device
    void* multi = nullptr;
    bool same_process = false; // DSGD child of a multi handle: its ring neighbours live in this process (CUDA IPC cannot map them;
                               // the in-kernel ring takes their buffers by plain peer pointers instead)
    lrk_handle_s** siblings = nullptr;   // same_process: the handles of all ranks, indexed by rank
    bool score_only = false;   // scoring child of a multi handle: the train CSR is kept for the top-N mask only (no COO stream)

    // DSGD
    void* comm = nullptr;   // ncclComm_t
    int rank = 0, world = 1;
    void* dsgd = nullptr;   // DsgdState*

    // allocation bookkeeping: device buffers are reused across calls when they are large enough
    std::unordered_map<void*, size_t> caps;
    void* scratch = nullptr;      // staging workspace (temporaries of lrk_set_train_csr), grown on demand
    size_t scratch_bytes = 0;

    std::string err;
};

extern thread_local std::string g_lrk_tls_error;

static inline int lrk_fail(lrk_handle_s* h, int code, const char* what, const char* detail, const char* file, int line) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s (%s:%d)", what, detail ? detail : "", file, line);
    if (h) h->err = buf;
    g_lrk_tls_error = buf;
    return code;
}

#define LRK_CUDA(h, call)                                                                        \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess)                                                                  \
            return lrk_fail((h), e__ == cudaErrorMemoryAllocation ? LRK_ERR_NOMEM : LRK_ERR_CUDA, \
                            #call, cudaGetErrorString(e__), __FILE__, __LINE__);                 \
    } while (0)

#define LRK_REQUIRE(h, cond, msg)                                                         \
    do {                                                                                  \
        if (!(cond)) return lrk_fail((h), LRK_ERR_INVALID, "invalid argument", msg, __FILE__, __LINE__); \
    } while (0)

#define LRK_LAUNCH_CHECK(h)                  \
    do {                                     \
        (h)->launches++;                     \
        LRK_CUDA((h), cudaGetLastError());   \
    } while (0)

template <typename T>
static inline int lrk_dev_alloc(lrk_handle_s* h, T** p, size_t count) {
    if (count == 0) count = 1;
    const size_t bytes = count * sizeof(T);
    if (*p) {
        auto it = h->caps.find((void*)*p);
        if (it != h->caps.end() && it->second >= bytes) return LRK_OK;   // reuse
        if (it != h->caps.end()) h->caps.erase(it);
        cudaFree(*p);
        *p = nullptr;
    }
    LRK_CUDA(h, cudaMalloc((void**)p, bytes));
    h->caps[(void*)*p] = bytes;
    return LRK_OK;
}
template <typename T>
static inline void lrk_dev_free(T** p) {
    if (*p) { cudaFree(*p); *p = nullptr; }
}
// bump allocator over the handle's staging workspace
struct LrkScratch {
    char* base = nullptr;
    size_t used = 0, cap = 0;
    template <typename T>
    T* take(size_t count) {
        const size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
        if (used + bytes > cap) return nullptr;
        T* r = reinterpret_cast<T*>(base + used);
        used += bytes;
        return r;
    }
};
static inline int lrk_scratch_begin(lrk_handle_s* h, size_t bytes, LrkScratch* out) {
    if (h->scratch_bytes < bytes) {
        if (h->scratch) { cudaFree(h->scratch); h->scratch = nullptr; h->scratch_bytes = 0; }
        LRK_CUDA(h, cudaMalloc(&h->scratch, bytes));
        h->scratch_bytes = bytes;
    }
    out->base = (char*)h->scratch; out->used = 0; out->cap = h->scratch_bytes;
    return LRK_OK;
}

static inline int lrk_ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// What the host code needs to know about each model: one row per lrk_model value, in enum order
struct LrkModelInfo {
    double loss_scale;  // reported loss = loss_scale * the kernels' sum (the references' 0.5 of the squared error); 0: no loss (ALS)
    bool safeguard;     // the epoch runs under the rollback safeguard (lrk_epoch.cuh)
    bool damped;        // staleness-aware item step: the SGD kernels read the item degrees and mean |p_u|^2
    bool multi_gpu;     // DSGD / multi-device handle
    int biases;         // 0: none; 1: item biases (lrk_set_factors requires bi; user biases stay zero); 2: user and item biases.
                        // Predictions add b_i + p_u.q_i (+ b_u + mu) when > 0
    bool rating;        // BiasedMF / PMF: the rating is the target (item-run tiles, reference-order mode, user-group kernel)
    bool als;           // WRMF / eALS: alternating least squares on the fp64 masters (als.cuh); lrk_sgd_epoch = one ALS iteration
    bool f64_working;   // the fp64 masters are the working set: an epoch leaves them valid (lrk_model_info sets it)
};
static const LrkModelInfo k_lrk_models[] = {
    //                scale  guard  damped multi  biases rating als
    /* BiasedMF */ {0.5, true,  true,  true,  2, true,  false},
    /* PMF      */ {0.5, true,  true,  true,  0, true,  false},
    /* BPR      */ {1.0, true,  false, true,  0, false, false},
    /* RankSGD  */ {0.5, true,  true,  false, 0, false, false},
    /* GBPR     */ {1.0, false, false, false, 1, false, false},
    /* SVD++    */ {0.5, false, false, false, 2, false, false},
    /* AoBPR    */ {1.0, true,  false, false, 0, false, false},
    /* WRMF     */ {0.0, false, false, false, 0, false, true},
    /* eALS     */ {0.0, false, false, false, 0, false, true},
};
static inline bool lrk_model_known(int model) { return model >= 0 && model < (int)(sizeof k_lrk_models / sizeof k_lrk_models[0]); }
// the row of cfg.model, for cfg.update_mode: the reference-order mode works on the fp64 masters, single-GPU, without the safeguard
static inline LrkModelInfo lrk_model_info(const lrk_config_t& cfg) {
    LrkModelInfo m = k_lrk_models[cfg.model];
    m.f64_working = m.als;
    if (cfg.update_mode == LRK_UPDATE_REFERENCE_ORDER) { m.safeguard = false; m.multi_gpu = false; m.f64_working = true; }
    return m;
}
static const char* const k_lrk_single_gpu = "reference-order mode, RankSGD, GBPR, SVD++, AoBPR, WRMF and eALS are single-GPU in this build";
static inline bool lrk_has_bias(const lrk_handle_s* h) { return k_lrk_models[h->cfg.model].biases > 0; }

// Calls f(G, V) with the handle's layout (layout_for_k) as std::integral_constant arguments: a generic lambda instantiates its
// kernel for each layout, e.g. [&](auto g, auto v) { return launch_gv<decltype(g)::value, decltype(v)::value>(h, p); }
template <class F>
static int lrk_with_layout(lrk_handle_s* h, F&& f) {
    using std::integral_constant;
    switch (h->G * 100 + h->V) {
        case 101: return f(integral_constant<int, 1>{}, integral_constant<int, 1>{});
        case 201: return f(integral_constant<int, 2>{}, integral_constant<int, 1>{});
        case 401: return f(integral_constant<int, 4>{}, integral_constant<int, 1>{});
        case 801: return f(integral_constant<int, 8>{}, integral_constant<int, 1>{});
        case 1601: return f(integral_constant<int, 16>{}, integral_constant<int, 1>{});
        case 3201: return f(integral_constant<int, 32>{}, integral_constant<int, 1>{});
        case 3202: return f(integral_constant<int, 32>{}, integral_constant<int, 2>{});
        default: return lrk_fail(h, LRK_ERR_INVALID, "lrk_with_layout", "unsupported factor layout", __FILE__, __LINE__);
    }
}
