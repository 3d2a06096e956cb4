// C ABI of the B200-native LibRec MF path (include/librec_b200.h).  Single translation unit:
// staging, SGD epoch, exact prediction / top-N, tensor-core top-N candidates, DSGD.
#include "lrk_common.cuh"
#include "staging.cuh"
#include "sgd.cuh"
#include "staging_group.cuh"
#include "sgd_group.cuh"
#include "sgd_exact.cuh"
#include "sgd_gbpr.cuh"
#include "sgd_svdpp.cuh"
#include "sgd_aobpr.cuh"
#include "als.cuh"
#include "lrk_epoch.cuh"
#include <chrono>
#include "topn_exact.cuh"
#include "topn_tc.cuh"
#include "dsgd.cuh"
#include "l2_probe.cuh"
#include "multi.cuh"

#include <cmath>
#include <new>

thread_local std::string g_lrk_tls_error;

static int multi_destroy(lrk_handle_s* h);
static int multi_set_train_csr(lrk_handle_s* h, int32_t U, int32_t I, const int64_t* rowptr, const int32_t* col, const double* val);
static int multi_set_factors(lrk_handle_s* h, const double* P, const double* Q, const double* bu, const double* bi, double mu);
static int multi_get_factors(lrk_handle_s* h, double* P, double* Q, double* bu, double* bi);
static int multi_sgd_epoch(lrk_handle_s* h, float lr, float reg_u, float reg_i, double reg_b, int32_t epoch_idx, double* loss_out);
static int multi_topn(lrk_handle_s* h, const int32_t* users, int32_t nq, int32_t topn, int32_t exclude_train, int32_t* out_items,
                      double* out_scores, int32_t* out_counts);
#define LRK_NOT_MULTI(h, what) LRK_REQUIRE(h, !(h)->multi, what " is not available on a multi-device handle: call lrk_get_factors and use a single-device handle")

// GBPR: train CSC (users of every item, ascending) next to the CSR -- the group draws of GBPRRecommender.java:104-116 walk an item's column
static int gbpr_stage(lrk_handle_s* h) {
    cudaStream_t st = h->stream;
    if (!h->gbpr) h->gbpr.reset(new GbprState());
    GbprState* g = h->gbpr.get();
    const int64_t nnz = h->nnz;
    const int32_t U = h->U, I = h->I;
    int rc;
    if ((rc = lrk_dev_alloc(h, &g->d_colptr, (size_t)I + 1))) return rc;
    if ((rc = lrk_dev_alloc(h, &g->d_cusers, (size_t)nnz))) return rc;
    if (nnz == 0) { LRK_CUDA(h, cudaMemsetAsync(g->d_colptr, 0, sizeof(int64_t) * ((size_t)I + 1), st)); return LRK_OK; }
    size_t tb_sort = 0, tb_scan = 0;
    int end_bit = 1;
    while (end_bit < 32 && ((int64_t)1 << end_bit) < (int64_t)I) ++end_bit;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, tb_sort, (uint32_t*)nullptr, (uint32_t*)nullptr, (int32_t*)nullptr, (int32_t*)nullptr, (int)nnz, 0, end_bit, st));
    LRK_CUDA(h, cub::DeviceScan::ExclusiveSum(nullptr, tb_scan, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)I, st));
    const size_t tb = std::max(tb_sort, tb_scan) + 256;
    LrkScratch sc;
    if ((rc = lrk_scratch_begin(h, (size_t)nnz * 16 + (size_t)I * 8 + tb + 16 * 256, &sc))) return rc;
    uint32_t *k_in = sc.take<uint32_t>((size_t)nnz), *k_out = sc.take<uint32_t>((size_t)nnz);
    int32_t* rows = sc.take<int32_t>((size_t)nnz);
    uint32_t *deg = sc.take<uint32_t>((size_t)I), *deg_ex = sc.take<uint32_t>((size_t)I);
    void* tmp = sc.take<char>(tb);
    if (!k_in || !k_out || !rows || !deg || !deg_ex || !tmp) return lrk_fail(h, LRK_ERR_NOMEM, "gbpr_stage", "scratch arena too small", __FILE__, __LINE__);
    const int nb = lrk_ceil_div(nnz, 256);
    coo_rows_kernel<<<nb, 256, 0, st>>>(h->d_rowptr, U, nnz, rows); LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaMemcpyAsync(k_in, h->d_col, sizeof(uint32_t) * (size_t)nnz, cudaMemcpyDeviceToDevice, st));
    LRK_CUDA(h, cudaMemsetAsync(deg, 0, sizeof(uint32_t) * (size_t)I, st));
    item_degree_kernel<<<nb, 256, 0, st>>>(h->d_col, nnz, deg); LRK_LAUNCH_CHECK(h);
    size_t t1 = tb;
    LRK_CUDA(h, cub::DeviceScan::ExclusiveSum(tmp, t1, deg, deg_ex, (int)I, st));
    gbpr_colptr_kernel<<<lrk_ceil_div(I, 256), 256, 0, st>>>(deg_ex, deg, I, g->d_colptr); LRK_LAUNCH_CHECK(h);
    t1 = tb;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(tmp, t1, k_in, k_out, rows, g->d_cusers.ptr, (int)nnz, 0, end_bit, st));   // stable: users ascending
    LRK_CUDA(h, cudaStreamSynchronize(st));
    return LRK_OK;
}

static int gbpr_fill(lrk_handle_s* h, GbprParams& p, float lr, float reg_u, float reg_i, double reg_b, int32_t epoch_idx) {
    GbprState* g = h->gbpr.get();
    memset(&p, 0, sizeof p);
    p.n = h->nnz; p.P = h->P32; p.Q = h->Q32; p.tP = g->tP; p.tQ = g->tQ; p.bi = h->bi32;
    p.lr = lr; p.reg_u = reg_u; p.reg_i = reg_i; p.reg_b = (float)reg_b; p.rho = g->rho; p.glen = g->glen;
    p.loss = h->d_loss; p.ld = h->ld; p.rowptr = h->d_rowptr; p.col = h->d_col; p.colptr = g->d_colptr; p.cusers = g->d_cusers;
    p.U = h->U; p.I = h->I; p.seed_lo = (uint32_t)h->cfg.seed; p.seed_hi = (uint32_t)(h->cfg.seed >> 32); p.epoch = (uint32_t)epoch_idx;
    return LRK_OK;
}

template <int G, int V>
static int gbpr_launch_gv(lrk_handle_s* h, const GbprParams& p) {
    int per_sm = 0;
    LRK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sgd_gbpr_epoch_kernel<G, V>, 256, 0));
    int64_t grid = (int64_t)h->sm_count * (per_sm < 1 ? 1 : per_sm);
    const int64_t need = ((p.n + 31) / 32 + 7) / 8;
    if (need < grid) grid = need;
    // the factor side is frozen inside an epoch; only the item biases race.  Small matrices: keep at most n/16 samples in flight
    const int64_t cap = (p.n / 16) / (8 * (int64_t)(32 / G));
    if (cap < grid) grid = cap;
    if (grid < 1) grid = 1;
    sgd_gbpr_epoch_kernel<G, V><<<(unsigned)grid, 256, 0, h->stream>>>(p);
    LRK_LAUNCH_CHECK(h);
    return LRK_OK;
}

// one GBPR iteration: GBPRRecommender.java:84-168
static int gbpr_epoch(lrk_handle_s* h, float lr, float reg_u, float reg_i, double reg_b, int32_t epoch_idx, double* loss_out) {
    GbprState* g = h->gbpr.get();
    LRK_REQUIRE(h, g != nullptr, "GBPR state missing: call lrk_set_train_csr first");
    cudaStream_t st = h->stream;
    const size_t np_ = (size_t)h->U * h->ld, nq_ = (size_t)h->I * h->ld;
    int rc;
    if ((rc = lrk_dev_alloc(h, &g->tP, np_))) return rc;
    if ((rc = lrk_dev_alloc(h, &g->tQ, nq_))) return rc;
    LRK_CUDA(h, cudaMemsetAsync(g->tP, 0, sizeof(float) * np_, st));
    LRK_CUDA(h, cudaMemsetAsync(g->tQ, 0, sizeof(float) * nq_, st));
    GbprParams p;
    gbpr_fill(h, p, lr, reg_u, reg_i, reg_b, epoch_idx);
    LrkEpoch e;
    e.enqueue = [&](int) -> int {
        if (h->nnz == 0) return LRK_OK;
        const int rc_l = lrk_with_layout(h, [&](auto G, auto V) { return gbpr_launch_gv<decltype(G)::value, decltype(V)::value>(h, p); });
        if (rc_l) return rc_l;
        gbpr_apply_kernel<<<lrk_ceil_div((int64_t)np_, 256), 256, 0, st>>>(h->P32, g->tP, (int64_t)np_); LRK_LAUNCH_CHECK(h);
        gbpr_apply_kernel<<<lrk_ceil_div((int64_t)nq_, 256), 256, 0, st>>>(h->Q32, g->tQ, (int64_t)nq_); LRK_LAUNCH_CHECK(h);
        return LRK_OK;
    };
    return lrk_epoch(h, e, loss_out);                 // no 0.5 (GBPRRecommender.java:130-165)
}

// SVD++: train values in CSR order + users by descending degree
static int svdpp_stage(lrk_handle_s* h, const double* h_val) {
    cudaStream_t st = h->stream;
    if (!h->svdpp) h->svdpp.reset(new SvdppState());
    SvdppState* g = h->svdpp.get();
    const int64_t nnz = h->nnz;
    const int32_t U = h->U;
    int rc;
    if ((rc = lrk_dev_alloc(h, &g->d_cval, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &g->d_uorder, (size_t)U))) return rc;
    if ((rc = lrk_dev_alloc(h, &g->d_counter, 1))) return rc;
    size_t tb = 0;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairsDescending(nullptr, tb, (uint32_t*)nullptr, (uint32_t*)nullptr, (int32_t*)nullptr, (int32_t*)nullptr, (int)U, 0, 32, st));
    LrkScratch sc;
    if ((rc = lrk_scratch_begin(h, (size_t)nnz * 8 + (size_t)U * 12 + tb + 16 * 256, &sc))) return rc;
    double* d_val = sc.take<double>((size_t)std::max<int64_t>(nnz, 1));
    uint32_t *deg = sc.take<uint32_t>((size_t)U), *deg2 = sc.take<uint32_t>((size_t)U);
    int32_t* ids = sc.take<int32_t>((size_t)U);
    void* tmp = sc.take<char>(tb + 16);
    if (!d_val || !deg || !deg2 || !ids || !tmp) return lrk_fail(h, LRK_ERR_NOMEM, "svdpp_stage", "scratch arena too small", __FILE__, __LINE__);
    if (nnz > 0) {
        LRK_CUDA(h, cudaMemcpyAsync(d_val, h_val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, st));
        f64_to_f32_kernel<<<lrk_ceil_div(nnz, 256), 256, 0, st>>>(d_val, g->d_cval, nnz); LRK_LAUNCH_CHECK(h);
    }
    svdpp_deg_kernel<<<lrk_ceil_div(U, 256), 256, 0, st>>>(h->d_rowptr, U, deg, ids); LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairsDescending(tmp, tb, deg, deg2, ids, g->d_uorder.ptr, (int)U, 0, 32, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    return LRK_OK;
}

template <int G, int V>
static int svdpp_launch_gv(lrk_handle_s* h, const SvdppParams& p) {
    int per_sm = 0;
    LRK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sgd_svdpp_epoch_kernel<G, V>, 256, 0));
    int64_t grid = (int64_t)h->sm_count * (per_sm < 1 ? 1 : per_sm);
    const int64_t need = ((int64_t)p.U + 8 * (32 / G) - 1) / (8 * (32 / G));
    if (need < grid) grid = need;
    // small matrices: at most ~1/16 of the users in flight (every worker holds one user's whole row)
    const int64_t cap = ((int64_t)p.U / 16) / (8 * (32 / G));
    if (cap >= 1 && cap < grid) grid = cap;
    if (grid < 1) grid = 1;
    sgd_svdpp_epoch_kernel<G, V><<<(unsigned)grid, 256, 0, h->stream>>>(p);
    LRK_LAUNCH_CHECK(h);
    return LRK_OK;
}

// one SVD++ iteration: SVDPlusPlusRecommender.java:63-109
static int svdpp_epoch(lrk_handle_s* h, float lr, float reg_u, float reg_i, double reg_b, double* loss_out) {
    SvdppState* g = h->svdpp.get();
    LRK_REQUIRE(h, g != nullptr && g->has_y, "SVD++ needs impItemFactors: lrk_set_matrix(h, \"svdpp.y\", Y) after lrk_set_factors");
    cudaStream_t st = h->stream;
    SvdppParams p;
    memset(&p, 0, sizeof p);
    p.rowptr = h->d_rowptr; p.col = h->d_col; p.cval = g->d_cval; p.uorder = g->d_uorder; p.U = h->U; p.counter = g->d_counter;
    p.P = h->P32; p.Q = h->Q32; p.Y = g->Y32; p.bu = h->bu32; p.bi = h->bi32;
    p.mu = (float)h->mu; p.lr = lr; p.reg_u = reg_u; p.reg_i = reg_i; p.reg_b = (float)reg_b; p.reg_imp = (float)g->reg_imp;
    p.loss = h->d_loss; p.ld = h->ld;
    LRK_CUDA(h, cudaMemsetAsync(g->d_counter, 0, sizeof(unsigned int), st));
    LrkEpoch e;
    e.enqueue = [&](int) -> int {
        if (h->nnz == 0) return LRK_OK;
        return lrk_with_layout(h, [&](auto G, auto V) { return svdpp_launch_gv<decltype(G)::value, decltype(V)::value>(h, p); });
    };
    return lrk_epoch(h, e, loss_out);                 // 0.5 * sum: SVDPlusPlusRecommender.java:109
}

__global__ void pairs_validate_kernel(const int32_t* __restrict__ u, const int32_t* __restrict__ i, int64_t n, int32_t U, int32_t I, int* __restrict__ flag) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n && (u[t] < 0 || u[t] >= U || i[t] < 0 || i[t] >= I)) atomicOr(flag, 1);
}

extern "C" {

const char* lrk_version(void) { return "librec_b200 0.1.0 (sm_100a; LibRec 3.0.0 MF path)"; }
int32_t lrk_abi_version(void) { return LRK_ABI_VERSION; }

int32_t lrk_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char* lrk_last_error(lrk_handle_t h) { return h ? h->err.c_str() : g_lrk_tls_error.c_str(); }

int lrk_host_alloc(void** out, uint64_t bytes) {
    if (!out) return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_host_alloc", "out is NULL", __FILE__, __LINE__);
    LRK_CUDA(nullptr, cudaMallocHost(out, bytes ? bytes : 1));
    return LRK_OK;
}
int lrk_host_free(void* p) {
    if (p) LRK_CUDA(nullptr, cudaFreeHost(p));
    return LRK_OK;
}

static void layout_for_k(int k, int* ld, int* G, int* V) {
    int l = 4;
    while (l < k && l < 128) l <<= 1;
    if (k > 128) l = ((k + 127) / 128) * 128;
    *ld = l;
    if (l <= 128) { *G = l / 4; *V = 1; } else { *G = 32; *V = l / 128; }
}

int lrk_create(const lrk_config_t* cfg, lrk_handle_t* out) {
    if (!cfg || !out) return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create", "NULL argument", __FILE__, __LINE__);
    *out = nullptr;
    if (cfg->num_factors < 1 || cfg->num_factors > LRK_MAX_FACTORS)
        return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create", "num_factors must be in 1..256", __FILE__, __LINE__);
    if (!lrk_model_known(cfg->model))
        return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create", "unknown model", __FILE__, __LINE__);
    if (cfg->model == LRK_MODEL_WRMF && cfg->num_factors > ALS_MAX_K)
        return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create", "WRMF on the device needs rec.factor.number <= 112 (the Gauss-Jordan step lives in shared memory)", __FILE__, __LINE__);
    if (cfg->update_mode < LRK_UPDATE_ATOMIC || cfg->update_mode > LRK_UPDATE_REFERENCE_ORDER)
        return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create", "unknown update_mode", __FILE__, __LINE__);
    if (cfg->update_mode == LRK_UPDATE_REFERENCE_ORDER && !k_lrk_models[cfg->model].rating)
        return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create", "reference-order mode covers BiasedMF and PMF", __FILE__, __LINE__);
    int ndev = 0;
    LRK_CUDA(nullptr, cudaGetDeviceCount(&ndev));
    if (cfg->device < 0 || cfg->device >= ndev)
        return lrk_fail(nullptr, LRK_ERR_CUDA, "lrk_create", "no such CUDA device (there is no CPU fallback)", __FILE__, __LINE__);
    cudaDeviceProp prop;
    LRK_CUDA(nullptr, cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10)
        return lrk_fail(nullptr, LRK_ERR_CUDA, "lrk_create", "device is not sm_100 (this library is built for sm_100a only)", __FILE__, __LINE__);
    lrk_handle_s* h = new (std::nothrow) lrk_handle_s();
    if (!h) return lrk_fail(nullptr, LRK_ERR_NOMEM, "lrk_create", "host allocation failed", __FILE__, __LINE__);
    h->cfg = *cfg;
    h->k = cfg->num_factors;
    layout_for_k(h->k, &h->ld, &h->G, &h->V);
    {   // the user-group kernel (LRK_SGD_GROUP=1, sgd_group.cuh) needs at least 8 lanes per rating: small k are padded to 32 columns
        const char* env = getenv("LRK_SGD_GROUP");
        h->sgd_group = env && atoi(env) != 0 && k_lrk_models[cfg->model].rating && cfg->update_mode == LRK_UPDATE_ATOMIC;
        if (h->sgd_group && h->ld < 32) { h->ld = 32; h->G = 8; h->V = 1; }
    }
    h->sm_count = prop.multiProcessorCount;
    int rc = LRK_OK;
    do {
        if (cudaSetDevice(cfg->device) != cudaSuccess) { rc = LRK_ERR_CUDA; break; }
        if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) { rc = LRK_ERR_CUDA; break; }
        h->stream = h->own_stream;
        if (cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess) { rc = LRK_ERR_CUDA; break; }
        if (lrk_dev_alloc(h, &h->d_loss, 8) != LRK_OK) { rc = LRK_ERR_NOMEM; break; }
        if (cudaMallocHost((void**)&h->h_loss, 64) != cudaSuccess) { rc = LRK_ERR_NOMEM; break; }
    } while (0);
    if (rc != LRK_OK) {
        lrk_fail(nullptr, rc, "lrk_create", cudaGetErrorString(cudaGetLastError()), __FILE__, __LINE__);
        lrk_destroy(h);
        return rc;
    }
    *out = h;
    return LRK_OK;
}

int lrk_destroy(lrk_handle_t h) {
    if (!h) return LRK_OK;
    if (h->multi) return multi_destroy(h);
    cudaSetDevice(h->cfg.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    delete h;
    return LRK_OK;
}

int lrk_set_stream(lrk_handle_t h, void* cuda_stream) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    LRK_NOT_MULTI(h, "lrk_set_stream");
    LRK_CUDA(h, cudaStreamSynchronize(h->stream));
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    return LRK_OK;
}
int lrk_synchronize(lrk_handle_t h) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    if (h->multi) { for (lrk_handle_s* c : ((MultiState*)h->multi)->child) { const int rc = lrk_synchronize(c); if (rc) return rc; } return LRK_OK; }
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    LRK_CUDA(h, cudaStreamSynchronize(h->stream));
    return LRK_OK;
}

// -------------------------------------------------------------------------------------------
int lrk_set_train_csr(lrk_handle_t h, int32_t U, int32_t I, const int64_t* rowptr, const int32_t* col, const double* val) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    LRK_REQUIRE(h, U > 0 && I > 0 && rowptr && (col || rowptr[U] == 0) && (val || rowptr[U] == 0 || h->score_only), "bad CSR arguments");
    if (h->multi) return multi_set_train_csr(h, U, I, rowptr, col, val);
    LRK_REQUIRE(h, !h->has_factors || (h->U == U && h->I == I), "CSR shape differs from the factors already set");
    const int64_t nnz = rowptr[U];
    LRK_REQUIRE(h, nnz >= 0 && nnz < (int64_t)0x7fffffffLL, "nnz out of range (the staging sorts take an int count: at most 2^31 - 1 train entries per handle)");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    if (h->world > 1) return dsgd_set_train_csr(h, U, I, rowptr, col, val);
    cudaStream_t st = h->stream;
    h->has_train = false;
    int rc;
    if ((rc = lrk_dev_alloc(h, &h->d_rowptr, (size_t)U + 1))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->d_col, (size_t)nnz))) return rc;
    if (!h->score_only) {
        if ((rc = lrk_dev_alloc(h, &h->d_su, (size_t)nnz))) return rc;
        if ((rc = lrk_dev_alloc(h, &h->d_si, (size_t)nnz))) return rc;
        if ((rc = lrk_dev_alloc(h, &h->d_sr, (size_t)nnz))) return rc;
    }
    LRK_CUDA(h, cudaMemcpyAsync(h->d_rowptr, rowptr, sizeof(int64_t) * ((size_t)U + 1), cudaMemcpyHostToDevice, st));
    LRK_CUDA(h, cudaMemcpyAsync(h->d_col, col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, st));
    h->U = U; h->I = I; h->nnz = nnz;
    if (h->score_only) {            // top-N mask only (scoring child of a multi handle; its DSGD sibling validated the shard)
        LRK_CUDA(h, cudaStreamSynchronize(st));
        h->has_train = true;
        topn_tc_invalidate(h);
        return LRK_OK;
    }
    // BiasedMF / PMF in atomic mode with LRK_SGD_GROUP=1 train with the user-group kernel over a unit-ordered stream (sgd_group.cuh);
    // everything else keeps the item-run-tile stream of sgd.cuh
    h->group.reset();
    const bool want_group = lrk_use_group_kernel(h) && group_order_supported(U, I, nnz, 1);
    rc = stage_coo_from_csr(h, h->d_rowptr, h->d_col, val, U, I, nnz, h->d_su, h->d_si, h->d_sr, /*validate=*/true,
                            want_group ? sgd_group_resident_workers(h) : 0, &h->group);
    if (rc) return rc;
    if (h->cfg.model == LRK_MODEL_RANKSGD && nnz > 0) {
        // sampling table of the negatives: inclusive prefix sums of the item degrees (RankSGDRecommender.java:47-57)
        if ((rc = lrk_dev_alloc(h, &h->d_item_cum, (size_t)I))) return rc;
        size_t tb = 0;
        LRK_CUDA(h, cub::DeviceScan::InclusiveSum(nullptr, tb, h->d_item_deg.ptr, h->d_item_cum.ptr, (int)I, st));
        LrkScratch sc;
        if ((rc = lrk_scratch_begin(h, tb + 256, &sc))) return rc;
        LRK_CUDA(h, cub::DeviceScan::InclusiveSum(sc.take<char>(tb), tb, h->d_item_deg.ptr, h->d_item_cum.ptr, (int)I, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
        h->launches++;
    }
    if (h->cfg.update_mode == LRK_UPDATE_REFERENCE_ORDER) {
        h->exact.reset();
        if ((rc = exact_build_schedule(h, &h->exact, U, I, rowptr, col, val))) return rc;
    }
    if (h->cfg.model == LRK_MODEL_GBPR && (rc = gbpr_stage(h))) return rc;
    if (h->cfg.model == LRK_MODEL_SVDPP && (rc = svdpp_stage(h, val))) return rc;
    if (k_lrk_models[h->cfg.model].als && (rc = als_stage(h, val))) return rc;
    h->has_train = true;
    topn_tc_invalidate(h);
    return LRK_OK;
}

int lrk_set_factors(lrk_handle_t h, const double* P, const double* Q, const double* bu, const double* bi, double mu) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    if (h->multi) return multi_set_factors(h, P, Q, bu, bi, mu);
    LRK_REQUIRE(h, h->has_train, "call lrk_set_train_csr first (it fixes numUsers / numItems)");
    LRK_REQUIRE(h, P && Q, "P and Q are required");
    const LrkModelInfo m = lrk_model_info(h->cfg);
    const bool biased = m.biases > 0;
    LRK_REQUIRE(h, m.biases < 2 || (bu && bi), "BiasedMF / SVD++ need userBiases and itemBiases");
    LRK_REQUIRE(h, m.biases < 1 || bi, "GBPR needs itemBiases");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    if (h->world > 1) return dsgd_set_factors(h, P, Q, bu, bi, mu);
    cudaStream_t st = h->stream;
    const int k = h->k, ld = h->ld;
    const int64_t U = h->U, I = h->I;
    int rc;
    if ((rc = lrk_dev_alloc(h, &h->P64, (size_t)U * k))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->Q64, (size_t)I * k))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->P32, (size_t)U * ld))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->Q32, (size_t)I * ld))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->bu64, (size_t)U))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->bi64, (size_t)I))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->bu32, (size_t)U))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->bi32, (size_t)I + 4))) return rc;
    LRK_CUDA(h, cudaMemcpyAsync(h->P64, P, sizeof(double) * (size_t)U * k, cudaMemcpyHostToDevice, st));
    LRK_CUDA(h, cudaMemcpyAsync(h->Q64, Q, sizeof(double) * (size_t)I * k, cudaMemcpyHostToDevice, st));
    if (biased && bu) LRK_CUDA(h, cudaMemcpyAsync(h->bu64, bu, sizeof(double) * (size_t)U, cudaMemcpyHostToDevice, st));
    else LRK_CUDA(h, cudaMemsetAsync(h->bu64, 0, sizeof(double) * (size_t)U, st));
    if (biased) LRK_CUDA(h, cudaMemcpyAsync(h->bi64, bi, sizeof(double) * (size_t)I, cudaMemcpyHostToDevice, st));
    else LRK_CUDA(h, cudaMemsetAsync(h->bi64, 0, sizeof(double) * (size_t)I, st));
    f64_to_f32_rows_kernel<<<lrk_ceil_div(U * ld, 256), 256, 0, st>>>(h->P64, h->P32, U, k, ld); LRK_LAUNCH_CHECK(h);
    f64_to_f32_rows_kernel<<<lrk_ceil_div(I * ld, 256), 256, 0, st>>>(h->Q64, h->Q32, I, k, ld); LRK_LAUNCH_CHECK(h);
    f64_to_f32_rows_kernel<<<lrk_ceil_div(U, 256), 256, 0, st>>>(h->bu64, h->bu32, U, 1, 1); LRK_LAUNCH_CHECK(h);
    f64_to_f32_rows_kernel<<<lrk_ceil_div(I, 256), 256, 0, st>>>(h->bi64, h->bi32, I, 1, 1); LRK_LAUNCH_CHECK(h);
    if (m.damped && (rc = refresh_user_norm2(h, true))) return rc;
    if (h->aobpr) h->aobpr->count = 0;                 // a new trainModel(): countIter starts at 0 (AoBPRRecommender.java:88)
    if (h->h_pnorm2) { h->pnorm2_prev = 0.f; h->pnorm2_host = *h->h_pnorm2; }
    LRK_CUDA(h, cudaStreamSynchronize(st));   // host buffers may be reused by the caller on return
    h->mu = mu;
    h->has_factors = true;
    h->f64_valid = true;
    h->prev_loss = -1.0; h->conc_div = 1; h->good_epochs = 0; h->epochs_done = 0;
    topn_tc_invalidate(h);
    return LRK_OK;
}

// bring the fp64 masters up to date with the fp32 working copies (exact widening)
static int refresh_masters(lrk_handle_s* h) {
    if (h->f64_valid) return LRK_OK;
    cudaStream_t st = h->stream;
    const int64_t U = h->U, I = h->I;
    f32_to_f64_rows_kernel<<<lrk_ceil_div(U * h->k, 256), 256, 0, st>>>(h->P32, h->P64, U, h->k, h->ld); LRK_LAUNCH_CHECK(h);
    f32_to_f64_rows_kernel<<<lrk_ceil_div(I * h->k, 256), 256, 0, st>>>(h->Q32, h->Q64, I, h->k, h->ld); LRK_LAUNCH_CHECK(h);
    if (lrk_has_bias(h)) {
        f32_to_f64_rows_kernel<<<lrk_ceil_div(U, 256), 256, 0, st>>>(h->bu32, h->bu64, U, 1, 1); LRK_LAUNCH_CHECK(h);
        f32_to_f64_rows_kernel<<<lrk_ceil_div(I, 256), 256, 0, st>>>(h->bi32, h->bi64, I, 1, 1); LRK_LAUNCH_CHECK(h);
    }
    h->f64_valid = true;
    return LRK_OK;
}

int lrk_get_factors(lrk_handle_t h, double* P, double* Q, double* bu, double* bi) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    if (h->multi) return multi_get_factors(h, P, Q, bu, bi);
    LRK_REQUIRE(h, h->has_factors, "no factors set");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    if (h->world > 1) return dsgd_get_factors(h, P, Q, bu, bi);
    int rc = refresh_masters(h);
    if (rc) return rc;
    cudaStream_t st = h->stream;
    if (P) LRK_CUDA(h, cudaMemcpyAsync(P, h->P64, sizeof(double) * (size_t)h->U * h->k, cudaMemcpyDeviceToHost, st));
    if (Q) LRK_CUDA(h, cudaMemcpyAsync(Q, h->Q64, sizeof(double) * (size_t)h->I * h->k, cudaMemcpyDeviceToHost, st));
    if (bu) LRK_CUDA(h, cudaMemcpyAsync(bu, h->bu64, sizeof(double) * (size_t)h->U, cudaMemcpyDeviceToHost, st));
    if (bi) LRK_CUDA(h, cudaMemcpyAsync(bi, h->bi64, sizeof(double) * (size_t)h->I, cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    return LRK_OK;
}

// -------------------------------------------------------------------------------------------
int lrk_sgd_epoch(lrk_handle_t h, float lr, float reg_u, float reg_i, double reg_b, int32_t epoch_idx, double* loss_out) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    if (h->multi) return multi_sgd_epoch(h, lr, reg_u, reg_i, reg_b, epoch_idx, loss_out);
    LRK_REQUIRE(h, h->has_train && h->has_factors, "set the train CSR and the factors before training");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    if (h->world > 1) return dsgd_epoch(h, lr, reg_u, reg_i, reg_b, epoch_idx, loss_out);
    if (h->cfg.model == LRK_MODEL_GBPR) return gbpr_epoch(h, lr, reg_u, reg_i, reg_b, epoch_idx, loss_out);
    if (h->cfg.model == LRK_MODEL_SVDPP) return svdpp_epoch(h, lr, reg_u, reg_i, reg_b, loss_out);
    if (k_lrk_models[h->cfg.model].als) { topn_tc_invalidate(h); return als_epoch(h, reg_u, reg_i, loss_out); }
    LrkEpoch e;
    if (h->cfg.update_mode == LRK_UPDATE_REFERENCE_ORDER) {
        // fp64 masters are the working set in this mode
        int rc = refresh_masters(h);
        if (rc) return rc;
        e.enqueue = [&](int) { return h->nnz > 0 ? exact_epoch(h, h->exact.get(), lr, reg_u, reg_i, reg_b) : (int)LRK_OK; };
        return lrk_epoch(h, e, loss_out);
    }
    // curvature estimate of the epoch: the value the last norm refresh left in pinned memory (once per epoch call, so that a
    // lrk_bpr_peek_samples between two epochs cannot change which kernel variant the next epoch picks)
    if (h->h_pnorm2) { h->pnorm2_prev = h->pnorm2_host; h->pnorm2_host = *h->h_pnorm2; }
    SgdParams sp = sgd_segment(h, sgd_params(h, lr, reg_u, reg_i, reg_b, epoch_idx), 0, h->nnz, h->Q32, h->bi32, 0);
    AobprState* ao = nullptr;
    if (h->cfg.model == LRK_MODEL_AOBPR) {
        ao = h->aobpr.get();
        LRK_REQUIRE(h, ao != nullptr, "AoBPR needs rec.item.distribution.parameter: lrk_set_param(h, \"aobpr.lambda\", value)");
        int rc_a = aobpr_prepare(h, ao);
        if (rc_a) return rc_a;
        sp.ao_rank = ao->d_rank; sp.ao_var = ao->d_var; sp.ao_cum = ao->d_cum; sp.n_entries = h->nnz;
    }
    e.saved = [&] {
        std::vector<LrkSaved> v{{h->P32, &h->bk_P, (size_t)h->U * h->ld}, {h->Q32, &h->bk_Q, (size_t)h->I * h->ld}};
        if (lrk_has_bias(h)) { v.push_back({h->bu32, &h->bk_bu, (size_t)h->U}); v.push_back({h->bi32, &h->bk_bi, (size_t)h->I}); }
        return v;
    };
    e.enqueue = [&](int attempt) -> int {
        if (h->nnz == 0) return LRK_OK;
        int rc;
        if (h->group) {
            LRK_CUDA(h, cudaMemsetAsync(h->group->d_counter, 0, sizeof(unsigned int), h->stream));
            return sgd_group_launch(h, sp, 0);
        }
        if (!ao) return sgd_launch(h, sp);
        // AoBPR: the epoch in windows of loopNumber samples, the factor rankings refreshed between them (countIter runs across
        // iterations and restarts at every refresh, AoBPRRecommender.java:92-97)
        int64_t count = ao->count, done = 0;
        while (done < h->nnz) {
            if (count % ao->loop == 0) { if ((rc = aobpr_refresh(h, ao))) return rc; count = 0; }
            const int64_t w = std::min<int64_t>(h->nnz - done, (int64_t)ao->loop - count);
            SgdParams wp = sgd_segment(h, sp, 0, w, h->Q32, h->bi32, 0);
            wp.sample_base = done;
            if ((rc = sgd_launch(h, wp))) return rc;
            done += w; count += w;
        }
        if (attempt == 0) ao->count = count;          // a rolled-back attempt replays the same windows
        return LRK_OK;
    };
    // the group kernel takes the curvature from the rows it holds; the stream kernels need mean |p_u|^2 refreshed per epoch
    e.refresh_norm = !h->group && (sp.item_deg != nullptr || h->cfg.model == LRK_MODEL_RANKSGD);
    e.rolled_back = [&]() -> int {
        if (!e.refresh_norm) return LRK_OK;
        const int rc = refresh_user_norm2(h, true);     // the restored factors' norm, visible to the host now
        if (rc) return rc;
        h->pnorm2_host = *h->h_pnorm2;
        return LRK_OK;
    };
    return lrk_epoch(h, e, loss_out);
}

int lrk_set_param(lrk_handle_t h, const char* name, double value) {
    LRK_REQUIRE(h, h != nullptr && name != nullptr, "NULL argument");
    LRK_NOT_MULTI(h, "lrk_set_param");
    if (!strcmp(name, "gbpr.rho") || !strcmp(name, "gbpr.gsize")) {
        LRK_REQUIRE(h, h->cfg.model == LRK_MODEL_GBPR, "gbpr.* parameters need a GBPR handle");
        if (!h->gbpr) h->gbpr.reset(new GbprState());
        GbprState* g = h->gbpr.get();
        if (!strcmp(name, "gbpr.rho")) g->rho = (float)value;
        else {
            LRK_REQUIRE(h, value >= 1.0 && value <= (double)LRK_GBPR_MAX_GROUP, "rec.gpbr.gsize must be in 1..8");
            g->glen = (int)value;
        }
        return LRK_OK;
    }
    if (!strcmp(name, "aobpr.lambda")) {
        LRK_REQUIRE(h, h->cfg.model == LRK_MODEL_AOBPR, "aobpr.* parameters need an AoBPR handle");
        if (!h->aobpr) h->aobpr.reset(new AobprState());
        h->aobpr->dist_param = (float)value;
        h->aobpr->I = 0;                                // the rank distribution is rebuilt at the next epoch
        return LRK_OK;
    }
    if (!strcmp(name, "svdpp.reg_imp")) {
        LRK_REQUIRE(h, h->cfg.model == LRK_MODEL_SVDPP, "svdpp.* parameters need an SVD++ handle");
        if (!h->svdpp) h->svdpp.reset(new SvdppState());
        h->svdpp->reg_imp = value;
        return LRK_OK;
    }
    return lrk_fail(h, LRK_ERR_INVALID, "lrk_set_param", "unknown parameter name", __FILE__, __LINE__);
}

int lrk_set_matrix(lrk_handle_t h, const char* name, const double* values) {
    LRK_REQUIRE(h, h != nullptr && name != nullptr && values != nullptr, "NULL argument");
    LRK_NOT_MULTI(h, "lrk_set_matrix");
    if (!strcmp(name, "eals.confidences") && h->cfg.model == LRK_MODEL_EALS) {
        LRK_REQUIRE(h, h->has_train, "call lrk_set_train_csr first (it fixes numItems)");
        LRK_CUDA(h, cudaSetDevice(h->cfg.device));
        AlsState* a = h->als.get();
        LRK_REQUIRE(h, a != nullptr, "ALS state missing");
        int rc_a;
        if ((rc_a = lrk_dev_alloc(h, &a->d_conf, (size_t)h->I))) return rc_a;
        LRK_CUDA(h, cudaMemcpyAsync(a->d_conf, values, sizeof(double) * (size_t)h->I, cudaMemcpyHostToDevice, h->stream));
        LRK_CUDA(h, cudaStreamSynchronize(h->stream));
        a->has_conf = true;
        return LRK_OK;
    }
    LRK_REQUIRE(h, !strcmp(name, "svdpp.y") && h->cfg.model == LRK_MODEL_SVDPP, "unknown matrix name for this model");
    LRK_REQUIRE(h, h->has_factors, "call lrk_set_factors first");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    if (!h->svdpp) h->svdpp.reset(new SvdppState());
    SvdppState* g = h->svdpp.get();
    cudaStream_t st = h->stream;
    const int64_t I = h->I;
    int rc;
    if ((rc = lrk_dev_alloc(h, &g->Y64, (size_t)I * h->k))) return rc;
    if ((rc = lrk_dev_alloc(h, &g->Y32, (size_t)I * h->ld))) return rc;
    LRK_CUDA(h, cudaMemcpyAsync(g->Y64, values, sizeof(double) * (size_t)I * h->k, cudaMemcpyHostToDevice, st));
    f64_to_f32_rows_kernel<<<lrk_ceil_div(I * h->ld, 256), 256, 0, st>>>(g->Y64, g->Y32, I, h->k, h->ld); LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaStreamSynchronize(st));
    g->has_y = true;
    return LRK_OK;
}

int lrk_get_matrix(lrk_handle_t h, const char* name, double* values) {
    LRK_REQUIRE(h, h != nullptr && name != nullptr && values != nullptr, "NULL argument");
    LRK_NOT_MULTI(h, "lrk_get_matrix");
    if (!strcmp(name, "eals.confidences") && h->cfg.model == LRK_MODEL_EALS) {
        AlsState* a = h->als.get();
        LRK_REQUIRE(h, a != nullptr && a->has_conf, "matrix not set");
        LRK_CUDA(h, cudaSetDevice(h->cfg.device));
        LRK_CUDA(h, cudaMemcpyAsync(values, a->d_conf, sizeof(double) * (size_t)h->I, cudaMemcpyDeviceToHost, h->stream));
        LRK_CUDA(h, cudaStreamSynchronize(h->stream));
        return LRK_OK;
    }
    LRK_REQUIRE(h, !strcmp(name, "svdpp.y") && h->cfg.model == LRK_MODEL_SVDPP, "unknown matrix name for this model");
    SvdppState* g = h->svdpp.get();
    LRK_REQUIRE(h, g != nullptr && g->has_y, "matrix not set");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = h->stream;
    const int64_t I = h->I;
    f32_to_f64_rows_kernel<<<lrk_ceil_div(I * h->k, 256), 256, 0, st>>>(g->Y32, g->Y64, I, h->k, h->ld); LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaMemcpyAsync(values, g->Y64, sizeof(double) * (size_t)I * h->k, cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    return LRK_OK;
}

int lrk_sgd_epochs(lrk_handle_t h, int32_t n_epochs, float lr, float decay, float max_lr, float reg_u, float reg_i, double reg_b,
                   int32_t first_epoch_idx, double* losses_out) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    LRK_REQUIRE(h, n_epochs >= 0 && (n_epochs == 0 || losses_out != nullptr), "bad arguments");
    float rate = lr;
    for (int32_t it = 0; it < n_epochs; ++it) {
        const int rc = lrk_sgd_epoch(h, rate, reg_u, reg_i, reg_b, first_epoch_idx + it, losses_out + it);
        if (rc) return rc;
        // updateLRate without the bold driver (MatrixFactorizationRecommender.java:131-138): float arithmetic like the reference
        if (decay > 0.f && decay < 1.f) rate *= decay;
        if (max_lr > 0.f && rate > max_lr) rate = max_lr;
    }
    return LRK_OK;
}

int lrk_stage_stats(lrk_handle_t h, int64_t out[4]) {
    LRK_REQUIRE(h, h != nullptr && out != nullptr, "NULL argument");
    if (h->multi && ((MultiState*)h->multi)->als) {            // every child stages the whole matrix: count it once
        lrk_handle_s* c = ((MultiState*)h->multi)->child[0];
        const int rc = lrk_stage_stats(c, out);
        if (rc) h->err = c->err;
        return rc;
    }
    if (h->multi) {
        int64_t acc[4] = {0, 0, 0, 0};
        for (lrk_handle_s* c : ((MultiState*)h->multi)->child) {
            int64_t v[4];
            const int rc = lrk_stage_stats(c, v);
            if (rc) { h->err = c->err; return rc; }
            acc[0] += v[0]; acc[1] += v[1]; acc[2] = std::max(acc[2], v[2]); acc[3] = v[3];
        }
        for (int i = 0; i < 4; ++i) out[i] = acc[i];
        return LRK_OK;
    }
    LRK_REQUIRE(h, h->has_train, "no train CSR");
    out[0] = h->nnz; out[1] = 32 * h->run_tiles; out[2] = (int64_t)h->max_item_deg; out[3] = LRK_RUN_MIN_DEGREE;
    return LRK_OK;
}

int lrk_debug_stream(lrk_handle_t h, int32_t* su, int32_t* si, float* sr, int32_t* units, int64_t max_units, int64_t* n_units_out) {
    LRK_REQUIRE(h, h != nullptr && n_units_out != nullptr, "NULL argument");
    LRK_NOT_MULTI(h, "lrk_debug_stream");
    LRK_REQUIRE(h, h->has_train, "no train CSR");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    cudaStream_t st = h->stream;
    GroupUnits* gu = h->group.get();
    *n_units_out = gu ? gu->n_units : 0;
    const size_t n = (size_t)h->nnz;
    if (su && n) LRK_CUDA(h, cudaMemcpyAsync(su, h->d_su, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    if (si && n) LRK_CUDA(h, cudaMemcpyAsync(si, h->d_si, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    if (sr && n) LRK_CUDA(h, cudaMemcpyAsync(sr, h->d_sr, sizeof(float) * n, cudaMemcpyDeviceToHost, st));
    if (units && gu) {
        LRK_REQUIRE(h, max_units >= gu->n_units, "units buffer too small");
        LRK_CUDA(h, cudaMemcpyAsync(units, gu->d_units, sizeof(int4) * (size_t)gu->n_units, cudaMemcpyDeviceToHost, st));
    }
    LRK_CUDA(h, cudaStreamSynchronize(st));
    return LRK_OK;
}

int lrk_sgd_safeguard_state(lrk_handle_t h, int32_t* conc_div, int64_t* rollbacks) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    if (h->multi) return lrk_sgd_safeguard_state(((MultiState*)h->multi)->child[0], conc_div, rollbacks);   // the ranks decide alike
    if (conc_div) *conc_div = h->conc_div;
    if (rollbacks) *rollbacks = h->rollbacks;
    return LRK_OK;
}
int lrk_last_epoch_ms(lrk_handle_t h, float* ms_out) {
    LRK_REQUIRE(h, h != nullptr && ms_out != nullptr, "NULL argument");
    if (h->multi && !((MultiState*)h->multi)->als) {
        *ms_out = 0.f;
        for (lrk_handle_s* c : ((MultiState*)h->multi)->child) *ms_out = std::max(*ms_out, c->last_epoch_ms);
        return LRK_OK;
    }
    *ms_out = h->last_epoch_ms;
    return LRK_OK;
}
int lrk_launch_count(lrk_handle_t h, uint64_t* out) {
    LRK_REQUIRE(h, h != nullptr && out != nullptr, "NULL argument");
    if (h->multi) {
        MultiState* ms = (MultiState*)h->multi;
        *out = 0;
        for (lrk_handle_s* c : ms->child) *out += c->launches;
        for (lrk_handle_s* c : ms->scorer) if (c) *out += c->launches;
        return LRK_OK;
    }
    *out = h->launches;
    return LRK_OK;
}

int lrk_bpr_peek_samples(lrk_handle_t h, int32_t epoch_idx, int64_t first, int64_t n, int32_t* out) {
    LRK_REQUIRE(h, h != nullptr && out != nullptr && n >= 0 && first >= 0, "bad arguments");
    LRK_NOT_MULTI(h, "lrk_bpr_peek_samples");
    LRK_REQUIRE(h, h->has_train, "no train CSR");
    LRK_REQUIRE(h, h->world == 1, "not available in DSGD mode");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    if (n == 0) return LRK_OK;
    SgdParams sp = sgd_params(h, 0.f, 0.f, 0.f, 0.0, epoch_idx);
    if (h->cfg.model == LRK_MODEL_AOBPR) {
        // the draws depend on the factor rankings: those of the current item factors (what the first window of an epoch uses)
        AobprState* ao = h->aobpr.get();
        LRK_REQUIRE(h, ao != nullptr && h->has_factors, "AoBPR: set the factors and rec.item.distribution.parameter first");
        int rc_a = aobpr_prepare(h, ao);
        if (rc_a == LRK_OK) rc_a = aobpr_refresh(h, ao);
        if (rc_a) return rc_a;
        sp.ao_rank = ao->d_rank; sp.ao_var = ao->d_var; sp.ao_cum = ao->d_cum; sp.n_entries = h->nnz;
    }
    const bool gbpr = h->cfg.model == LRK_MODEL_GBPR;
    const size_t n_out = (gbpr ? 3 + LRK_GBPR_MAX_GROUP : 3) * (size_t)n;    // GBPR: 11 ints per sample {u, i, j, group[8] padded with -1}
    LrkScratch sc;
    int rc;
    if ((rc = lrk_scratch_begin(h, sizeof(int32_t) * n_out + 256, &sc))) return rc;
    int32_t* d_out = sc.take<int32_t>(n_out);
    if (!d_out) return lrk_fail(h, LRK_ERR_NOMEM, "lrk_bpr_peek_samples", "scratch arena too small", __FILE__, __LINE__);
    if (gbpr) {
        LRK_REQUIRE(h, h->gbpr != nullptr, "GBPR state missing");
        GbprParams gp;
        gbpr_fill(h, gp, 0.f, 0.f, 0.f, 0.0, epoch_idx);
        gbpr_peek_kernel<<<lrk_ceil_div(n, 256), 256, 0, h->stream>>>(gp, first, n, d_out);
    } else if (h->cfg.model == LRK_MODEL_RANKSGD) {
        if (first + n > h->nnz) return lrk_fail(h, LRK_ERR_INVALID, "lrk_bpr_peek_samples", "RankSGD has one sample per train entry: first + n exceeds nnz", __FILE__, __LINE__);
        ranksgd_peek_kernel<<<lrk_ceil_div(n, 256), 256, 0, h->stream>>>(sp, first, n, d_out);
    } else
        bpr_peek_kernel<<<lrk_ceil_div(n, 256), 256, 0, h->stream>>>(sp, first, n, d_out);
    LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaMemcpyAsync(out, d_out, sizeof(int32_t) * n_out, cudaMemcpyDeviceToHost, h->stream));
    LRK_CUDA(h, cudaStreamSynchronize(h->stream));
    return LRK_OK;
}

// -------------------------------------------------------------------------------------------
int lrk_predict_pairs(lrk_handle_t h, const int32_t* users, const int32_t* items, int64_t n, double* out) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    LRK_NOT_MULTI(h, "lrk_predict_pairs");
    LRK_REQUIRE(h, h->cfg.model != LRK_MODEL_SVDPP, "SVD++ predictions need the per-user sum of the implicit factors: read the matrices back (lrk_get_factors, lrk_get_matrix) and use the reference predict()");
    LRK_REQUIRE(h, h->has_factors, "no factors set");
    LRK_REQUIRE(h, n >= 0 && (n == 0 || (users && items && out)), "bad arguments");
    LRK_REQUIRE(h, h->world == 1, "gather the factors with lrk_get_factors in DSGD mode");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    if (n == 0) return LRK_OK;
    int rc = refresh_masters(h);
    if (rc) return rc;
    cudaStream_t st = h->stream;
    // inputs, output and the range-check flag live in the handle's staging arena (no per-call cudaMalloc); the indices are
    // validated on the device before anything is indexed with them
    LrkScratch sc;
    if ((rc = lrk_scratch_begin(h, (size_t)n * 16 + 4 * 256, &sc))) return rc;
    int32_t *d_u = sc.take<int32_t>((size_t)n), *d_i = sc.take<int32_t>((size_t)n);
    double* d_o = sc.take<double>((size_t)n);
    int* d_flag = sc.take<int>(1);
    if (!d_u || !d_i || !d_o || !d_flag) return lrk_fail(h, LRK_ERR_NOMEM, "lrk_predict_pairs", "scratch arena too small", __FILE__, __LINE__);
    int flag = 0;
    LRK_CUDA(h, cudaMemcpyAsync(d_u, users, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    LRK_CUDA(h, cudaMemcpyAsync(d_i, items, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    LRK_CUDA(h, cudaMemsetAsync(d_flag, 0, sizeof(int), st));
    pairs_validate_kernel<<<lrk_ceil_div(n, 256), 256, 0, st>>>(d_u, d_i, n, h->U, h->I, d_flag); LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaMemcpyAsync(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    LRK_REQUIRE(h, flag == 0, "user/item index out of range");
    predict_pairs_kernel<<<lrk_ceil_div(n, 128), 128, 0, st>>>(h->P64, h->Q64, h->bu64, h->bi64, h->mu, lrk_has_bias(h), h->k, d_u, d_i, n, d_o);
    LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaMemcpyAsync(out, d_o, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    return LRK_OK;
}

int lrk_eval_rating(lrk_handle_t h, int32_t U, const int64_t* t_rowptr, const int32_t* t_col, const double* t_val,
                    double min_rate, double max_rate, double* pred_out, double* rmse_out, double* mae_out) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    LRK_NOT_MULTI(h, "lrk_eval_rating");
    LRK_REQUIRE(h, h->cfg.model != LRK_MODEL_SVDPP, "SVD++ predictions need the per-user sum of the implicit factors: read the matrices back (lrk_get_factors, lrk_get_matrix) and use the reference predict()");
    LRK_REQUIRE(h, h->has_factors, "no factors set");
    LRK_REQUIRE(h, U == h->U && t_rowptr, "test matrix must have numUsers rows");
    LRK_REQUIRE(h, h->world == 1, "gather the factors with lrk_get_factors in DSGD mode");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    const int64_t nnz = t_rowptr[U];
    if (nnz == 0) { if (rmse_out) *rmse_out = 0.0; if (mae_out) *mae_out = 0.0; return LRK_OK; }   // RMSEEvaluator.java:35-37
    LRK_REQUIRE(h, t_col && t_val, "NULL test arrays");
    int rc = refresh_masters(h);
    if (rc) return rc;
    cudaStream_t st = h->stream;
    const int nb = lrk_ceil_div(nnz, 256);
    LrkScratch sc;
    if ((rc = lrk_scratch_begin(h, sizeof(int64_t) * ((size_t)U + 1) + (size_t)nnz * 20 + sizeof(double) * ((size_t)nb * 2 + 2) + 5 * 256, &sc))) return rc;
    int64_t* d_rp = sc.take<int64_t>((size_t)U + 1);
    int32_t* d_c = sc.take<int32_t>((size_t)nnz);
    double* d_v = sc.take<double>((size_t)nnz);
    double* d_p = sc.take<double>((size_t)nnz);
    double* d_part = sc.take<double>((size_t)nb * 2 + 2);
    if (!d_rp || !d_c || !d_v || !d_p || !d_part) return lrk_fail(h, LRK_ERR_NOMEM, "lrk_eval_rating", "scratch arena too small", __FILE__, __LINE__);
    LRK_CUDA(h, cudaMemcpyAsync(d_rp, t_rowptr, sizeof(int64_t) * ((size_t)U + 1), cudaMemcpyHostToDevice, st));
    LRK_CUDA(h, cudaMemcpyAsync(d_c, t_col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, st));
    LRK_CUDA(h, cudaMemcpyAsync(d_v, t_val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, st));
    eval_rating_kernel<<<nb, 256, 0, st>>>(h->P64, h->Q64, h->bu64, h->bi64, h->mu, lrk_has_bias(h),
                                           h->k, U, d_rp, d_c, d_v, min_rate, max_rate, d_p, d_part, d_part + nb);
    eval_rating_final_kernel<<<1, 32, 0, st>>>(d_part, d_part + nb, nb, nnz, d_part + 2 * (size_t)nb);
    h->launches += 2;
    LRK_CUDA(h, cudaGetLastError());
    double res[2] = {0, 0};
    if (pred_out) LRK_CUDA(h, cudaMemcpyAsync(pred_out, d_p, sizeof(double) * (size_t)nnz, cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaMemcpyAsync(res, d_part + 2 * (size_t)nb, sizeof(double) * 2, cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    if (rmse_out) *rmse_out = res[0];
    if (mae_out) *mae_out = res[1];
    return LRK_OK;
}

// -------------------------------------------------------------------------------------------
// top-N lists of the queried users into the handle's device buffers (tn_items / tn_scores / tn_counts)
static int topn_to_device(lrk_handle_s* h, const int32_t* users, int32_t nq, int32_t topn, int32_t exclude_train) {
    LRK_REQUIRE(h, h->has_factors, "no factors set");
    LRK_REQUIRE(h, h->cfg.model != LRK_MODEL_SVDPP, "SVD++ predictions need the per-user sum of the implicit factors: read the matrices back (lrk_get_factors, lrk_get_matrix) and use the reference predict()");
    LRK_REQUIRE(h, topn > 0, "rec.recommender.ranking.topn should be more than 0!");   // AbstractRecommender.java:115-117
    LRK_REQUIRE(h, topn <= LRK_MAX_TOPN, "topn above LRK_MAX_TOPN (512)");
    LRK_REQUIRE(h, !exclude_train || h->has_train, "exclude_train needs the train CSR");
    LRK_REQUIRE(h, h->world == 1, "gather the factors with lrk_get_factors in DSGD mode; top-N shards by user block");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    h->topn_fast_users = 0; h->topn_fallback_users = 0; h->topn_ms = 0.f;
    for (int i = 0; i < 4; ++i) h->topn_phase_ms[i] = 0.f;
    h->topn_err_ratio = 0.f; h->topn_resweep_users = 0;
    if (nq == 0) return LRK_OK;
    if (users) for (int32_t c = 0; c < nq; ++c) LRK_REQUIRE(h, users[c] >= 0 && users[c] < h->U, "user index out of range");
    else LRK_REQUIRE(h, nq <= h->U, "nq exceeds numUsers");
    int rc = refresh_masters(h);
    if (rc) return rc;
    cudaStream_t st = h->stream;
    int32_t* d_users = nullptr;
    if (users) {
        if ((rc = lrk_dev_alloc(h, &h->tn_users, (size_t)nq))) return rc;
        d_users = h->tn_users;
        LRK_CUDA(h, cudaMemcpyAsync(d_users, users, sizeof(int32_t) * (size_t)nq, cudaMemcpyHostToDevice, st));
    }
    if ((rc = lrk_dev_alloc(h, &h->tn_items, (size_t)nq * topn))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->tn_scores, (size_t)nq * topn))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->tn_counts, (size_t)nq))) return rc;
    cudaEventRecord(h->ev0, st);
    const bool want_tc = h->cfg.topn_path == 2 || (h->cfg.topn_path == 0 && topn_tc_profitable(h, nq, topn));
    if (want_tc) rc = topn_tc_run(h, d_users, nq, topn, exclude_train, h->tn_items, h->tn_scores, h->tn_counts);
    else if (d_users && h->cfg.topn_path != 1 && nq <= 4 * h->sm_count && h->I >= 32768) {
        rc = topn_exact_parallel_launch(h, d_users, nq, topn, exclude_train, h->tn_items, h->tn_scores, h->tn_counts);
        h->topn_fallback_users = nq;
    } else { rc = topn_exact_launch(h, d_users, nq, topn, exclude_train, h->tn_items, h->tn_scores, h->tn_counts); h->topn_fallback_users = nq; }
    cudaEventRecord(h->ev1, st);
    return rc;
}
static int topn_lists_to_host(lrk_handle_s* h, int32_t nq, int32_t topn, int32_t* out_items, double* out_scores, int32_t* out_counts) {
    cudaStream_t st = h->stream;
    if (out_items) LRK_CUDA(h, cudaMemcpyAsync(out_items, h->tn_items, sizeof(int32_t) * (size_t)nq * topn, cudaMemcpyDeviceToHost, st));
    if (out_scores) LRK_CUDA(h, cudaMemcpyAsync(out_scores, h->tn_scores, sizeof(double) * (size_t)nq * topn, cudaMemcpyDeviceToHost, st));
    if (out_counts) LRK_CUDA(h, cudaMemcpyAsync(out_counts, h->tn_counts, sizeof(int32_t) * (size_t)nq, cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    cudaEventElapsedTime(&h->topn_ms, h->ev0, h->ev1);
    return LRK_OK;
}

int lrk_topn(lrk_handle_t h, const int32_t* users, int32_t nq, int32_t topn, int32_t exclude_train,
             int32_t* out_items, double* out_scores, int32_t* out_counts) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    LRK_REQUIRE(h, nq >= 0 && (nq == 0 || (out_items && out_scores && out_counts)), "bad arguments");
    if (h->multi) return multi_topn(h, users, nq, topn, exclude_train, out_items, out_scores, out_counts);
    int rc = topn_to_device(h, users, nq, topn, exclude_train);
    if (rc || nq == 0) return rc;
    return topn_lists_to_host(h, nq, topn, out_items, out_scores, out_counts);
}

int lrk_eval_ranking(lrk_handle_t h, int32_t topn, const int64_t* t_rowptr, const int32_t* t_col, const double* t_val,
                     int32_t* out_items, double* out_scores, int32_t* out_counts, double out_measures[8]) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    LRK_NOT_MULTI(h, "lrk_eval_ranking");
    LRK_REQUIRE(h, t_rowptr && out_measures, "NULL argument");
    LRK_REQUIRE(h, h->has_train && h->has_factors, "set the train CSR and the factors first");
    LRK_REQUIRE(h, topn >= 1 && topn <= LRK_EVAL_MAX_TOPN, "lrk_eval_ranking supports 1 <= topn <= 64");
    const int32_t U = h->U;
    const int64_t nnz = t_rowptr[U];
    LRK_REQUIRE(h, nnz == 0 || (t_col && t_val), "NULL test arrays");
    int rc = topn_to_device(h, nullptr, U, topn, /*exclude_train=*/1);      // MatrixRecommender.java:153-201
    if (rc) return rc;
    cudaStream_t st = h->stream;
    LrkScratch sc;
    const int nb = lrk_ceil_div(U, 128);
    if ((rc = lrk_scratch_begin(h, sizeof(int64_t) * ((size_t)U + 1) + (size_t)nnz * 12 + sizeof(double) * (8 * (size_t)U + 16) +
                                       sizeof(int32_t) * 2 * (size_t)h->I + 16 * 256, &sc))) return rc;
    int64_t* d_rp = sc.take<int64_t>((size_t)U + 1);
    int32_t* d_c = sc.take<int32_t>((size_t)std::max<int64_t>(nnz, 1));
    double* d_v = sc.take<double>((size_t)std::max<int64_t>(nnz, 1));
    double* d_part = sc.take<double>(8 * (size_t)U);
    double* d_out = sc.take<double>(8);
    int32_t* d_purch = sc.take<int32_t>((size_t)h->I);
    int32_t* d_reco = sc.take<int32_t>((size_t)h->I);
    if (!d_rp || !d_c || !d_v || !d_part || !d_out || !d_purch || !d_reco) return lrk_fail(h, LRK_ERR_NOMEM, "lrk_eval_ranking", "scratch arena too small", __FILE__, __LINE__);
    LRK_CUDA(h, cudaMemcpyAsync(d_rp, t_rowptr, sizeof(int64_t) * ((size_t)U + 1), cudaMemcpyHostToDevice, st));
    if (nnz > 0) {
        LRK_CUDA(h, cudaMemcpyAsync(d_c, t_col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, st));
        LRK_CUDA(h, cudaMemcpyAsync(d_v, t_val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, st));
    }
    // rec.eval.item.purchase.num = train + test column counts (MatrixRecommender.java:118-122)
    LRK_CUDA(h, cudaMemsetAsync(d_purch, 0, sizeof(int32_t) * (size_t)h->I, st));
    LRK_CUDA(h, cudaMemsetAsync(d_reco, 0, sizeof(int32_t) * (size_t)h->I, st));
    if (h->nnz > 0) { item_count_add_kernel<<<lrk_ceil_div(h->nnz, 256), 256, 0, st>>>(h->d_col, h->nnz, d_purch); LRK_LAUNCH_CHECK(h); }
    if (nnz > 0) { item_count_add_kernel<<<lrk_ceil_div(nnz, 256), 256, 0, st>>>(d_c, nnz, d_purch); LRK_LAUNCH_CHECK(h); }
    eval_ranking_kernel<<<nb, 128, 0, st>>>(U, h->I, topn, h->tn_items, h->tn_counts, d_rp, d_c, d_v, h->d_rowptr, d_purch, d_reco, d_part);
    LRK_LAUNCH_CHECK(h);
    eval_ranking_final_kernel<<<8, 256, 0, st>>>(d_part, U, d_reco, h->I, d_out);
    LRK_LAUNCH_CHECK(h);
    double res[8];
    LRK_CUDA(h, cudaMemcpyAsync(res, d_out, sizeof(double) * 8, cudaMemcpyDeviceToHost, st));
    if ((rc = topn_lists_to_host(h, U, topn, out_items, out_scores, out_counts))) return rc;
    for (int m = 0; m < 8; ++m) out_measures[m] = res[m];
    return LRK_OK;
}

int lrk_topn_phase_ms(lrk_handle_t h, float out[6]) {
    LRK_REQUIRE(h, h != nullptr && out != nullptr, "NULL argument");
    LRK_NOT_MULTI(h, "lrk_topn_phase_ms");
    for (int i = 0; i < 4; ++i) out[i] = h->topn_phase_ms[i];
    out[4] = h->topn_err_ratio;
    out[5] = (float)h->topn_resweep_users;
    return LRK_OK;
}

int lrk_topn_stats(lrk_handle_t h, int64_t* fast_users, int64_t* fallback_users, float* ms_out) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    if (h->multi) {
        int64_t a = 0, b = 0; float ms = 0.f;
        for (lrk_handle_s* c : ((MultiState*)h->multi)->scorer) if (c) { a += c->topn_fast_users; b += c->topn_fallback_users; ms = std::max(ms, c->topn_ms); }
        if (fast_users) *fast_users = a;
        if (fallback_users) *fallback_users = b;
        if (ms_out) *ms_out = ms;
        return LRK_OK;
    }
    if (fast_users) *fast_users = h->topn_fast_users;
    if (fallback_users) *fallback_users = h->topn_fallback_users;
    if (ms_out) *ms_out = h->topn_ms;
    return LRK_OK;
}

int lrk_probe_l2(lrk_handle_t h, uint64_t working_set_bytes, int32_t row_floats, double out_gbps[3]) {
    LRK_REQUIRE(h, h != nullptr && out_gbps != nullptr, "NULL argument");
    if (h->multi) h = ((MultiState*)h->multi)->child[0];
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    return l2_probe_run(h, (size_t)working_set_bytes, row_floats, out_gbps);
}

int lrk_comm_unique_id(uint8_t out[128]) { return dsgd_unique_id(out); }
int lrk_comm_init(lrk_handle_t h, int32_t rank, int32_t world, const uint8_t unique_id[128]) {
    LRK_REQUIRE(h, h != nullptr, "handle is NULL");
    LRK_NOT_MULTI(h, "lrk_comm_init");
    LRK_REQUIRE(h, lrk_model_info(h->cfg).dsgd, k_lrk_single_gpu);
    return dsgd_comm_init(h, rank, world, unique_id);
}

int lrk_create_multi(const lrk_config_t* cfg, const int32_t* devices, int32_t n_devices, lrk_handle_t* out) {
    if (!cfg || !out || !devices) return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create_multi", "NULL argument", __FILE__, __LINE__);
    *out = nullptr;
    if (n_devices < 1 || n_devices > 8) return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create_multi", "1 to 8 devices", __FILE__, __LINE__);
    for (int a = 0; a < n_devices; ++a) for (int b = a + 1; b < n_devices; ++b)
        if (devices[a] == devices[b]) return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create_multi", "a device is listed twice", __FILE__, __LINE__);
    if (n_devices > 1 && lrk_model_known(cfg->model) && !lrk_model_info(*cfg).multi_device)     // an unknown model fails in lrk_create
        return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create_multi", k_lrk_single_gpu, __FILE__, __LINE__);
    lrk_handle_s* h = new (std::nothrow) lrk_handle_s();
    MultiState* ms = new (std::nothrow) MultiState();
    if (!h || !ms) { delete h; delete ms; return lrk_fail(nullptr, LRK_ERR_NOMEM, "lrk_create_multi", "host allocation failed", __FILE__, __LINE__); }
    h->cfg = *cfg; h->cfg.device = devices[0]; h->k = cfg->num_factors; h->multi = ms;
    ms->n = n_devices; ms->devices.assign(devices, devices + n_devices);
    ms->child.assign((size_t)n_devices, nullptr); ms->scorer.assign((size_t)n_devices, nullptr);
    ms->als = n_devices > 1 && lrk_model_known(cfg->model) && !lrk_model_info(*cfg).dsgd;     // WRMF: plain children, no DSGD
    int rc = LRK_OK;
    for (int g = 0; g < n_devices && rc == LRK_OK; ++g) {
        lrk_config_t c = *cfg;
        c.device = devices[g];
        rc = lrk_create(&c, &ms->child[(size_t)g]);
        if (rc == LRK_OK && !ms->als) { ms->child[(size_t)g]->same_process = true; ms->child[(size_t)g]->siblings = ms->child.data(); }   // peer pointers instead of CUDA IPC
    }
    for (int g = 0; g < n_devices; ++g) {
        LrkWorker* w = new LrkWorker();
        w->th = std::thread([w] { w->loop(); });
        ms->workers.push_back(w);
    }
    if (rc == LRK_OK && ms->als) {
        // the row exchange copies device to device: direct peer access where the pair has it (cudaMemcpyPeerAsync stages
        // through the host otherwise), and the events of the phase split
        ms->als_ev.assign((size_t)n_devices * LRK_ALS_EVENTS, nullptr);
        for (int a = 0; a < n_devices && rc == LRK_OK; ++a) {
            if (cudaSetDevice(devices[a]) != cudaSuccess) { rc = lrk_fail(h, LRK_ERR_CUDA, "cudaSetDevice", cudaGetErrorString(cudaGetLastError()), __FILE__, __LINE__); break; }
            for (int b = 0; b < n_devices && rc == LRK_OK; ++b) {
                int can = 0;
                if (b == a || cudaDeviceCanAccessPeer(&can, devices[a], devices[b]) != cudaSuccess || !can) { cudaGetLastError(); continue; }
                const cudaError_t pe = cudaDeviceEnablePeerAccess(devices[b], 0);
                if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) rc = lrk_fail(h, LRK_ERR_CUDA, "cudaDeviceEnablePeerAccess", cudaGetErrorString(pe), __FILE__, __LINE__);
                cudaGetLastError();
            }
            for (int e = 0; e < LRK_ALS_EVENTS && rc == LRK_OK; ++e) {
                const cudaError_t ce = cudaEventCreate(&ms->als_ev[(size_t)a * LRK_ALS_EVENTS + e]);
                if (ce != cudaSuccess) rc = lrk_fail(h, LRK_ERR_CUDA, "cudaEventCreate", cudaGetErrorString(ce), __FILE__, __LINE__);
            }
        }
    } else if (rc == LRK_OK && n_devices > 1) {
        uint8_t uid[128];
        rc = lrk_comm_unique_id(uid);
        if (rc == LRK_OK) rc = multi_run(h, ms, [&](int g) { return lrk_comm_init(ms->child[(size_t)g], g, ms->n, uid); });
    }
    if (rc != LRK_OK) {
        const std::string why = h->err.empty() ? g_lrk_tls_error : h->err;
        multi_destroy(h);
        return lrk_fail(nullptr, rc, "lrk_create_multi", why.c_str(), __FILE__, __LINE__);
    }
    *out = h;
    return LRK_OK;
}

}  // extern "C"

lrk_handle_s::~lrk_handle_s() {
    dsgd.reset();                                       // the ring buffers and their IPC mappings go before the communicator
    if (comm && nccl_api()) nccl_api()->CommDestroy((ncclComm_t)comm);
    if (h_loss) cudaFreeHost(h_loss);
    if (h_pnorm2) cudaFreeHost(h_pnorm2);
    for (cudaEvent_t ev : {ev0, ev1, ev_copy0, ev_copy1}) if (ev) cudaEventDestroy(ev);
    if (copy_stream) cudaStreamDestroy(copy_stream);
    if (own_stream) cudaStreamDestroy(own_stream);
}

static int multi_destroy(lrk_handle_s* h) {
    MultiState* ms = (MultiState*)h->multi;
    // the children's communicators are destroyed together, each on its own thread
    if (!ms->workers.empty() && (int)ms->workers.size() == ms->n)
        multi_run(h, ms, [&](int g) -> int { return ms->child[(size_t)g] ? lrk_destroy(ms->child[(size_t)g]) : (int)LRK_OK; });
    else for (lrk_handle_s* c : ms->child) if (c) lrk_destroy(c);
    for (lrk_handle_s* c : ms->scorer) if (c) lrk_destroy(c);
    for (size_t e = 0; e < ms->als_ev.size(); ++e)
        if (ms->als_ev[e]) { cudaSetDevice(ms->devices[e / LRK_ALS_EVENTS]); cudaEventDestroy(ms->als_ev[e]); }
    for (LrkWorker* w : ms->workers) { w->stop(); delete w; }
    delete ms;
    h->multi = nullptr;
    delete h;
    return LRK_OK;
}

static int multi_set_train_csr(lrk_handle_s* h, int32_t U, int32_t I, const int64_t* rowptr, const int32_t* col, const double* val) {
    MultiState* ms = (MultiState*)h->multi;
    LRK_REQUIRE(h, U >= ms->n, "fewer users than devices");
    ms->U = U; ms->I = I;
    const int64_t nnz = rowptr[U];
    if (ms->als) {
        // every child stages the whole matrix; the rows are split by the estimated solve cost: the entries' rank-one updates
        // (k^2 each) plus the row's Gauss-Jordan inverse (k^3)
        LRK_REQUIRE(h, nnz >= 0 && nnz < (int64_t)0x7fffffffLL, "nnz out of range (the staging sorts take an int count: at most 2^31 - 1 train entries; every device of a WRMF multi-device handle stages all of them)");
        const double k = (double)h->k, row_cost = k * k * k;
        std::vector<int64_t> deg((size_t)I, 0);
        for (int64_t e = 0; e < nnz; ++e) {
            LRK_REQUIRE(h, col[e] >= 0 && col[e] < I, "column index out of range");
            deg[(size_t)col[e]]++;
        }
        ms->ub = multi_cost_bounds(U, ms->n, true, [&](int64_t u) { return (double)(rowptr[u + 1] - rowptr[u]) * k * k + row_cost; });
        ms->ib = multi_cost_bounds(I, ms->n, false, [&](int64_t i) { return (double)deg[(size_t)i] * k * k + row_cost; });
    } else {
        ms->ub.assign((size_t)ms->n + 1, 0);
        for (int g = 0; g <= ms->n; ++g) ms->ub[(size_t)g] = (int64_t)g * U / ms->n;
    }
    ms->rowptr.assign(rowptr, rowptr + U + 1);                 // kept for the scoring handles (top-N train mask)
    ms->col.assign(col, col + nnz);
    ms->scorer_csr = false; ms->scorer_factors = false;
    const int rc = multi_run(h, ms, [&](int g) -> int {
        if (ms->als) return lrk_set_train_csr(ms->child[(size_t)g], U, I, rowptr, col, val);
        const int64_t lo = ms->ub[(size_t)g], hi = ms->ub[(size_t)g + 1], off = rowptr[lo];
        std::vector<int64_t> rp((size_t)(hi - lo) + 1);
        for (int64_t u = lo; u <= hi; ++u) rp[(size_t)(u - lo)] = rowptr[u] - off;
        return lrk_set_train_csr(ms->child[(size_t)g], (int32_t)(hi - lo), I, rp.data(), col + off, val + off);
    });
    if (rc == LRK_OK) { h->U = U; h->I = I; h->nnz = nnz; h->has_train = true; }
    return rc;
}

static int multi_set_factors(lrk_handle_s* h, const double* P, const double* Q, const double* bu, const double* bi, double mu) {
    MultiState* ms = (MultiState*)h->multi;
    LRK_REQUIRE(h, h->has_train, "call lrk_set_train_csr first (it fixes numUsers / numItems)");
    LRK_REQUIRE(h, P && Q, "P and Q are required");
    ms->mu = mu; ms->scorer_factors = false;
    const int k = h->k;
    const int rc = multi_run(h, ms, [&](int g) {
        if (ms->als) return lrk_set_factors(ms->child[(size_t)g], P, Q, bu, bi, mu);   // full replicas
        const int64_t lo = ms->ub[(size_t)g];
        return lrk_set_factors(ms->child[(size_t)g], P + lo * k, Q, bu ? bu + lo : nullptr, bi, mu);
    });
    if (rc == LRK_OK) { h->has_factors = true; h->mu = mu; }
    return rc;
}

static int multi_get_factors(lrk_handle_s* h, double* P, double* Q, double* bu, double* bi) {
    MultiState* ms = (MultiState*)h->multi;
    LRK_REQUIRE(h, h->has_factors, "no factors set");
    if (ms->als) {                             // the replicas are equal after every iteration
        const int rc = lrk_get_factors(ms->child[0], P, Q, bu, bi);
        if (rc) h->err = ms->child[0]->err;
        return rc;
    }
    const int k = h->k;
    return multi_run(h, ms, [&](int g) {       // every rank enters the ring gather; rank 0 delivers the item side
        const int64_t lo = ms->ub[(size_t)g];
        return lrk_get_factors(ms->child[(size_t)g], P ? P + lo * k : nullptr, g == 0 ? Q : nullptr, bu ? bu + lo : nullptr, g == 0 ? bi : nullptr);
    });
}

// One WRMF iteration over the devices.  Every child holds the full train matrix and full replicas of P and Q; device g solves the
// users [ub[g], ub[g+1]) and the items [ib[g], ib[g+1]).  Per half: the Gram matrix of the fixed side on every device (each
// computes the same full sum, so nothing depends on the partition), the device's row range, then every device pulls the other
// ranges' new rows straight from their owners' replicas.  multi_run is the host barrier between the phases: a device's rows are
// final before anyone copies them, and a Gram starts only after all blocks of its side have arrived.
static int multi_als_epoch(lrk_handle_s* h, MultiState* ms, float reg_u, float reg_i, double* loss_out) {
    const auto t0 = std::chrono::steady_clock::now();
    const int k = h->k;
    auto ev = [&](int g, int e) { return ms->als_ev[(size_t)g * LRK_ALS_EVENTS + e]; };
    // the other devices' ranges of one side into device g's replica, on g's stream
    auto pull = [&](int g, bool item_side) -> int {
        lrk_handle_s* c = ms->child[(size_t)g];
        const std::vector<int64_t>& b = item_side ? ms->ib : ms->ub;
        for (int s = 0; s < ms->n; ++s) {
            const int64_t lo = b[(size_t)s], cnt = b[(size_t)s + 1] - lo;
            if (s == g || cnt == 0) continue;
            lrk_handle_s* src = ms->child[(size_t)s];
            double* dst = item_side ? c->Q64.ptr : c->P64.ptr;
            const double* from = item_side ? src->Q64.ptr : src->P64.ptr;
            LRK_CUDA(c, cudaMemcpyPeerAsync(dst + lo * k, c->cfg.device, from + lo * k, src->cfg.device, sizeof(double) * (size_t)(cnt * k), c->stream));
        }
        return LRK_OK;
    };
    int rc = multi_run(h, ms, [&](int g) -> int {
        lrk_handle_s* c = ms->child[(size_t)g];
        LRK_CUDA(c, cudaSetDevice(c->cfg.device));
        LRK_REQUIRE(c, c->als != nullptr && c->f64_valid, "ALS state missing: call lrk_set_train_csr and lrk_set_factors first");
        const int64_t lo = ms->ub[(size_t)g], hi = ms->ub[(size_t)g + 1];
        int r;
        LRK_CUDA(c, cudaEventRecord(ev(g, 0), c->stream));
        if ((r = als_wrmf_gram(c, false))) return r;
        LRK_CUDA(c, cudaEventRecord(ev(g, 1), c->stream));
        if ((r = als_wrmf_side(c, als_wrmf_params(c, false, reg_u, (int32_t)lo, (int32_t)(hi - lo))))) return r;
        LRK_CUDA(c, cudaEventRecord(ev(g, 2), c->stream));
        LRK_CUDA(c, cudaStreamSynchronize(c->stream));
        return LRK_OK;
    });
    if (rc == LRK_OK) rc = multi_run(h, ms, [&](int g) -> int {
        lrk_handle_s* c = ms->child[(size_t)g];
        LRK_CUDA(c, cudaSetDevice(c->cfg.device));
        const int64_t lo = ms->ib[(size_t)g], hi = ms->ib[(size_t)g + 1];
        int r;
        LRK_CUDA(c, cudaEventRecord(ev(g, 3), c->stream));
        if ((r = pull(g, false))) return r;
        LRK_CUDA(c, cudaEventRecord(ev(g, 4), c->stream));
        if ((r = als_wrmf_gram(c, true))) return r;
        LRK_CUDA(c, cudaEventRecord(ev(g, 5), c->stream));
        if ((r = als_wrmf_side(c, als_wrmf_params(c, true, reg_i, (int32_t)lo, (int32_t)(hi - lo))))) return r;
        LRK_CUDA(c, cudaEventRecord(ev(g, 6), c->stream));
        LRK_CUDA(c, cudaStreamSynchronize(c->stream));
        return LRK_OK;
    });
    if (rc == LRK_OK) rc = multi_run(h, ms, [&](int g) -> int {
        lrk_handle_s* c = ms->child[(size_t)g];
        LRK_CUDA(c, cudaSetDevice(c->cfg.device));
        int r;
        LRK_CUDA(c, cudaEventRecord(ev(g, 7), c->stream));
        if ((r = pull(g, true))) return r;
        LRK_CUDA(c, cudaEventRecord(ev(g, 8), c->stream));
        if ((r = als_refresh_f32(c))) return r;
        LRK_CUDA(c, cudaStreamSynchronize(c->stream));
        return LRK_OK;
    });
    if (rc) return rc;
    h->last_epoch_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (loss_out) *loss_out = 0.0;                    // trainModel never assigns `loss`
    const char* trace = getenv("LRK_ALS_TRACE");
    if (trace && atoi(trace)) {
        // per device, ms between consecutive events: Gram(Q), users, waiting for the slowest device, P exchange, Gram(P), items,
        // waiting, Q exchange
        static const char* const names[] = {"gram_q", "solve_u", "wait_p", "xchg_p", "gram_p", "solve_i", "wait_q", "xchg_q"};
        for (int g = 0; g < ms->n; ++g) {
            std::string line = "[als] device " + std::to_string(ms->devices[(size_t)g]);
            for (int e = 0; e + 1 < LRK_ALS_EVENTS; ++e) {
                float t = 0.f;
                cudaEventElapsedTime(&t, ev(g, e), ev(g, e + 1));
                char buf[48];
                snprintf(buf, sizeof buf, " %s %.3f", names[e], t);
                line += buf;
            }
            fprintf(stderr, "%s total %.3f ms\n", line.c_str(), h->last_epoch_ms);
        }
    }
    return LRK_OK;
}

static int multi_sgd_epoch(lrk_handle_s* h, float lr, float reg_u, float reg_i, double reg_b, int32_t epoch_idx, double* loss_out) {
    MultiState* ms = (MultiState*)h->multi;
    LRK_REQUIRE(h, h->has_train && h->has_factors, "set the train CSR and the factors before training");
    if (ms->als) { ms->scorer_factors = false; return multi_als_epoch(h, ms, reg_u, reg_i, loss_out); }
    std::vector<double> loss((size_t)ms->n, 0.0);
    const int rc = multi_run(h, ms, [&](int g) { return lrk_sgd_epoch(ms->child[(size_t)g], lr, reg_u, reg_i, reg_b, epoch_idx, &loss[(size_t)g]); });
    if (loss_out) *loss_out = loss[0];          // all-reduced: the same on every rank
    ms->scorer_factors = false;
    return rc;
}

// top-N: users shard by block, every device holds the full item matrix, no collective (SURVEY.md 8e)
static int multi_topn(lrk_handle_s* h, const int32_t* users, int32_t nq, int32_t topn, int32_t exclude_train, int32_t* out_items,
                      double* out_scores, int32_t* out_counts) {
    MultiState* ms = (MultiState*)h->multi;
    LRK_REQUIRE(h, h->has_factors, "no factors set");
    LRK_REQUIRE(h, topn > 0 && topn <= LRK_MAX_TOPN, "rec.recommender.ranking.topn should be more than 0!");
    if (nq == 0) return LRK_OK;
    if (users) for (int32_t c = 0; c < nq; ++c) LRK_REQUIRE(h, users[c] >= 0 && users[c] < ms->U, "user index out of range");
    else LRK_REQUIRE(h, nq <= ms->U, "nq exceeds numUsers");
    const int k = h->k;
    const bool biased = lrk_has_bias(h);
    int rc;
    if (!ms->scorer_factors) {
        ms->P.resize((size_t)ms->U * k); ms->Q.resize((size_t)ms->I * k);
        if (biased) { ms->bu.resize((size_t)ms->U); ms->bi.resize((size_t)ms->I); }
        if ((rc = multi_get_factors(h, ms->P.data(), ms->Q.data(), biased ? ms->bu.data() : nullptr, biased ? ms->bi.data() : nullptr))) return rc;
    }
    // queries by shard
    std::vector<std::vector<int32_t>> local((size_t)ms->n), pos((size_t)ms->n);
    for (int32_t c = 0; c < nq; ++c) {
        const int32_t u = users ? users[c] : c;
        int g = (int)(((int64_t)u * ms->n) / ms->U);
        while (g > 0 && u < ms->ub[(size_t)g]) --g;
        while (g + 1 < ms->n && u >= ms->ub[(size_t)g + 1]) ++g;
        local[(size_t)g].push_back((int32_t)(u - ms->ub[(size_t)g]));
        pos[(size_t)g].push_back(c);
    }
    const bool stage_csr = !ms->scorer_csr, stage_fac = !ms->scorer_factors;
    rc = multi_run(h, ms, [&](int g) -> int {
        int r = LRK_OK;
        lrk_handle_s*& sc = ms->scorer[(size_t)g];
        if (!sc) {
            lrk_config_t c = h->cfg;
            c.device = ms->devices[(size_t)g];
            if ((r = lrk_create(&c, &sc))) return r;
            sc->score_only = true;
        }
        const int64_t lo = ms->ub[(size_t)g], hi = ms->ub[(size_t)g + 1];
        if (stage_csr) {
            const int64_t off = ms->rowptr[(size_t)lo];
            std::vector<int64_t> rp((size_t)(hi - lo) + 1);
            for (int64_t u = lo; u <= hi; ++u) rp[(size_t)(u - lo)] = ms->rowptr[(size_t)u] - off;
            if ((r = lrk_set_train_csr(sc, (int32_t)(hi - lo), ms->I, rp.data(), ms->col.data() + off, nullptr))) return r;
        }
        if (stage_csr || stage_fac)
            if ((r = lrk_set_factors(sc, ms->P.data() + lo * k, ms->Q.data(), biased ? ms->bu.data() + lo : nullptr, biased ? ms->bi.data() : nullptr, ms->mu))) return r;
        const size_t m = local[(size_t)g].size();
        if (m == 0) return LRK_OK;
        std::vector<int32_t> it(m * (size_t)topn), cn(m);
        std::vector<double> sc_(m * (size_t)topn);
        if ((r = lrk_topn(sc, local[(size_t)g].data(), (int32_t)m, topn, exclude_train, it.data(), sc_.data(), cn.data()))) return r;
        for (size_t t = 0; t < m; ++t) {
            const size_t c = (size_t)pos[(size_t)g][t];
            memcpy(out_items + c * topn, it.data() + t * topn, sizeof(int32_t) * (size_t)topn);
            memcpy(out_scores + c * topn, sc_.data() + t * topn, sizeof(double) * (size_t)topn);
            out_counts[c] = cn[t];
        }
        return LRK_OK;
    }, &ms->scorer);
    if (rc == LRK_OK) { ms->scorer_csr = true; ms->scorer_factors = true; }
    return rc;
}
