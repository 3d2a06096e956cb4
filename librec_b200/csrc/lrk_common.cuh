// Shared declarations of the B200-native LibRec MF path (handle layout, error plumbing).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <type_traits>
#include <utility>
#include "../../include/librec_b200.h"

#define LRK_MAX_FACTORS 256
#define LRK_MAX_TOPN 512

// Owning device buffer: cudaFree on destruction, reused by lrk_dev_alloc while its capacity suffices.  It converts to T*, so
// kernel arguments and parameter structs take it as they would a raw pointer.
template <typename T>
struct LrkBuf {
    T* ptr = nullptr;
    size_t cap = 0;   // bytes
    LrkBuf() = default;
    LrkBuf(LrkBuf&& o) noexcept { swap(o); }
    LrkBuf& operator=(LrkBuf&& o) noexcept { swap(o); return *this; }
    ~LrkBuf() { reset(); }
    void swap(LrkBuf& o) noexcept { std::swap(ptr, o.ptr); std::swap(cap, o.cap); }
    void reset() { if (ptr) cudaFree(ptr); ptr = nullptr; cap = 0; }
    operator T*() const { return ptr; }
};

// model states (one translation unit: lrk_api.cu includes their headers and defines ~lrk_handle_s after them)
struct GroupUnits; struct TcState; struct GbprState; struct SvdppState; struct AobprState; struct AlsState; struct ExactSchedule; struct DsgdState;
struct BprRefState;
struct MultiState;

// owning pointer of a child handle of a multi-device parent (multi.cuh): lrk_destroy selects its device, syncs and deletes it
struct LrkChildDelete { void operator()(lrk_handle_s* c) const { lrk_destroy(c); } };
using LrkChild = std::unique_ptr<lrk_handle_s, LrkChildDelete>;

struct lrk_handle_s {
    lrk_config_t cfg{};
    int k = 0;        // rec.factor.number
    int ld = 0;       // padded fp32 row length: power of two >= max(k,4); multiple of 128 above 128
    int G = 0;        // lanes cooperating on one rating (each lane owns V float4 of a row)
    int V = 1;
    int32_t U = 0, I = 0;
    int64_t nnz = 0;
    int sm_count = 0;
    size_t smem_optin = 0;    // largest dynamic shared memory a block can opt in to (cudaDevAttrMaxSharedMemoryPerBlockOptin)
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaStream_t copy_stream = nullptr;          // second stream: the H2D copy of the rating values overlaps the sort of the staging
    cudaEvent_t ev_copy0 = nullptr, ev_copy1 = nullptr;

    // train CSR (device): membership for BPR sampling and the top-N train mask
    LrkBuf<int64_t> d_rowptr;
    LrkBuf<int32_t> d_col;
    // shuffled COO stream for the SGD epoch (SoA, 12 B / rating)
    LrkBuf<int32_t> d_su;
    LrkBuf<int32_t> d_si;
    LrkBuf<float> d_sr;
    bool has_train = false;
    bool sgd_group = false;              // LRK_SGD_GROUP=1 at lrk_create: BiasedMF / PMF in atomic mode use the user-group kernel
    std::unique_ptr<GroupUnits> group;   // the stream is unit-ordered (staging_group.cuh) and the epoch runs sgd_group_epoch_kernel
    int64_t run_tiles = 0;    // 32-rating item-run tiles in the staged stream (lrk_stage_stats)
    uint32_t max_item_deg = 0;
    LrkBuf<float> d_pnorm2;           // mean |p_u|^2 at the start of the epoch (curvature term of that step)
    float pnorm2_host = 0.f;          // its host copy, refreshed with every loss read-back (picks the kernel variant)
    float pnorm2_prev = 0.f;          // the value one epoch earlier (growth of the user factors, the LRK_SGD_TRACE line)
    LrkBuf<uint32_t> d_item_deg;      // ratings per item in this handle's shard (staleness-aware step of run tiles, sgd.cuh)
    LrkBuf<uint32_t> d_item_cum;      // RankSGD: inclusive prefix sums of d_item_deg (negative sampling table)

    // factors: fp32 working copies (padded rows) + fp64 masters (dense rows, what Java sees)
    LrkBuf<float> P32, Q32, bu32, bi32;
    LrkBuf<double> P64, Q64, bu64, bi64;
    double mu = 0.0;
    bool has_factors = false;
    bool f64_valid = false;   // masters are in sync with the fp32 working copies

    // Safeguard of the fast SGD mode (lrk_epoch.cuh): factors are snapshotted before an epoch; a non-finite (or exploding) loss
    // rolls the epoch back and re-runs it with 4x fewer ratings in flight (sticky, relaxed again after 8 good epochs)
    LrkBuf<float> bk_P, bk_Q, bk_bu, bk_bi;
    int conc_div = 1;           // divisor of the SGD grid
    int good_epochs = 0;
    double prev_loss = -1.0;    // loss of the last accepted epoch (< 0: none yet)
    int64_t rollbacks = 0;
    int epochs_done = 0;        // accepted epochs since lrk_set_factors (picks the kernel variant of the first epochs)
    LrkBuf<double> d_loss;      // device accumulator
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
    LrkBuf<int32_t> tn_users, tn_items, tn_counts;
    LrkBuf<double> tn_scores;
    // heaps of the warp-per-user top-N kernel when they do not fit in shared memory (topn_exact_launch).  Not the staging arena:
    // the tie replay of the item-parallel path runs while that path holds it
    LrkBuf<char> tn_heaps;
    // tensor-core top-N state (bf16 copies, norms); see topn_tc.cuh
    std::unique_ptr<TcState> tc;

    std::unique_ptr<GbprState> gbpr;     // sgd_gbpr.cuh
    std::unique_ptr<SvdppState> svdpp;   // sgd_svdpp.cuh
    std::unique_ptr<AobprState> aobpr;   // sgd_aobpr.cuh
    std::unique_ptr<AlsState> als;       // als.cuh: WRMF / eALS

    // reference-order (wavefront) schedule, see sgd_exact.cuh
    std::unique_ptr<ExactSchedule> exact;
    // reference-order BPR: the java.util.Random state and the epoch's draw and update buffers, see sgd_bpr_exact.cuh
    std::unique_ptr<BprRefState> bprref;

    // single-process multi-GPU parent (multi.cuh): no device state of its own, forwards to one child per device
    std::unique_ptr<MultiState> multi;
    bool same_process = false; // DSGD child of a multi handle: its ring neighbours live in this process (CUDA IPC cannot map them;
                               // the in-kernel ring takes their buffers by plain peer pointers instead), and it serves top-N
    const LrkChild* siblings = nullptr;  // same_process: the handles of all ranks, indexed by rank (the parent's child table)

    // DSGD
    void* comm = nullptr;   // ncclComm_t
    int rank = 0, world = 1;
    std::unique_ptr<DsgdState> dsgd;

    LrkBuf<char> scratch;   // staging arena (lrk_scratch_begin)

    std::string err;

    // frees everything above; safe on a handle without device state (a multi-device parent, a half-created handle)
    ~lrk_handle_s();
};

extern thread_local std::string g_lrk_tls_error;

static inline int lrk_fail(lrk_handle_s* h, int code, const char* what, const char* detail, const char* file, int line) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s (%s:%d)", what, detail ? detail : "", file, line);
    if (h) h->err = buf;
    g_lrk_tls_error = buf;
    return code;
}

// A failed call also clears the runtime's last error: a non-sticky error (an out-of-memory cudaMalloc, a rejected launch
// attribute) is returned once, here, and not again by the next call on any handle that checks cudaGetLastError.
#define LRK_CUDA(h, call)                                                                        \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess) {                                                                \
            cudaGetLastError();                                                                  \
            return lrk_fail((h), e__ == cudaErrorMemoryAllocation ? LRK_ERR_NOMEM : LRK_ERR_CUDA, \
                            #call, cudaGetErrorString(e__), __FILE__, __LINE__);                 \
        }                                                                                        \
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

// at least `count` elements in *b (one when count is 0): kept when large enough, otherwise reallocated without its contents
template <typename T>
static inline int lrk_dev_alloc(lrk_handle_s* h, LrkBuf<T>* b, size_t count) {
    const size_t bytes = (count ? count : 1) * sizeof(T);
    if (b->cap >= bytes) return LRK_OK;
    b->reset();
    LRK_CUDA(h, cudaMalloc((void**)&b->ptr, bytes));
    b->cap = bytes;
    return LRK_OK;
}
// bump allocator over the handle's staging arena
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
// The staging arena serves the outermost level of one C-ABI call: a call takes it once and everything it hands out is
// overwritten by the next lrk_scratch_begin.  A helper that runs inside another helper's use of the arena keeps its
// temporaries in LrkBufs of the state it belongs to instead.
static inline int lrk_scratch_begin(lrk_handle_s* h, size_t bytes, LrkScratch* out) {
    const int rc = lrk_dev_alloc(h, &h->scratch, bytes);
    if (rc) return rc;
    out->base = h->scratch; out->used = 0; out->cap = h->scratch.cap;
    return LRK_OK;
}

static inline int lrk_ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// What the host code needs to know about each model: one row per lrk_model value, in enum order
struct LrkModelInfo {
    double loss_scale;  // reported loss = loss_scale * the kernels' sum (the references' 0.5 of the squared error); 0: no loss (ALS)
    bool safeguard;     // the epoch runs under the rollback safeguard (lrk_epoch.cuh)
    bool damped;        // staleness-aware item step: the SGD kernels read the item degrees and mean |p_u|^2
    bool dsgd;          // a DSGD rank: lrk_comm_init (process per GPU) and the DSGD children of a multi-device handle
    bool multi_device;  // lrk_create_multi with more than one device (DSGD children, or for WRMF full replicas that split the rows)
    int biases;         // 0: none; 1: item biases (lrk_set_factors requires bi; user biases stay zero); 2: user and item biases.
                        // Predictions add b_i + p_u.q_i (+ b_u + mu) when > 0
    bool rating;        // BiasedMF / PMF: the rating is the target (item-run tiles, reference-order mode, user-group kernel)
    bool als;           // WRMF / eALS: alternating least squares on the fp64 masters (als.cuh); lrk_sgd_epoch = one ALS iteration
    bool f64_working;   // the fp64 masters are the working set: an epoch leaves them valid (lrk_model_info sets it)
};
static const LrkModelInfo k_lrk_models[] = {
    //                scale  guard  damped dsgd   multi  biases rating als
    /* BiasedMF */ {0.5, true,  true,  true,  true,  2, true,  false},
    /* PMF      */ {0.5, true,  true,  true,  true,  0, true,  false},
    /* BPR      */ {1.0, true,  false, true,  true,  0, false, false},
    /* RankSGD  */ {0.5, true,  true,  false, false, 0, false, false},
    /* GBPR     */ {1.0, false, false, false, false, 1, false, false},
    /* SVD++    */ {0.5, false, false, false, false, 2, false, false},
    /* AoBPR    */ {1.0, true,  false, false, false, 0, false, false},
    /* WRMF     */ {0.0, false, false, false, true,  0, false, true},
    /* eALS     */ {0.0, false, false, false, false, 0, false, true},
};
static inline bool lrk_model_known(int model) { return model >= 0 && model < (int)(sizeof k_lrk_models / sizeof k_lrk_models[0]); }
// the row of cfg.model, for cfg.update_mode: the reference-order mode works on the fp64 masters, single-GPU, without the safeguard
static inline LrkModelInfo lrk_model_info(const lrk_config_t& cfg) {
    LrkModelInfo m = k_lrk_models[cfg.model];
    m.f64_working = m.als;
    if (cfg.update_mode == LRK_UPDATE_REFERENCE_ORDER) { m.safeguard = false; m.dsgd = false; m.multi_device = false; m.f64_working = true; }
    return m;
}
static const char* const k_lrk_single_gpu = "reference-order mode, RankSGD, GBPR, SVD++, AoBPR and eALS are single-GPU in this build; "
                                            "WRMF runs on several GPUs through lrk_create_multi only, not as a DSGD rank";
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
