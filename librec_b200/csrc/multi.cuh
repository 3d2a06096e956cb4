// Single-process multi-GPU handle (lrk_create_multi): what the Java shim uses for rec.cuda.devices=0,1,...,7.
//
// The reference drives a recommender from ONE thread of ONE JVM (job/RecommenderJob.java:121-143), so "one process per GPU" cannot
// be reached through its plugin API.  A multi handle takes and returns the FULL matrices exactly like a single-device handle and
// does the sharding inside: users are cut into n contiguous blocks, one per device; every device gets a DSGD child handle (rank g
// of an n-rank NCCL communicator created inside this process) driven by its own host thread, because the children's calls contain
// collectives that all ranks must enter together.  Training = the children's DSGD epoch (csrc/dsgd.cuh; the in-kernel ring takes the
// neighbours' buffers by peer pointers); top-N = each child scores the queried users of its block: it holds their train rows and,
// after the ring gather of lrk_get_factors, the full item matrix in its fp64 masters (SURVEY.md 8e).
//
// WRMF takes another route (`als` below): no DSGD and no communicator.  Every device gets a plain child handle that stages the FULL
// train matrix and holds full replicas of P and Q; users and, separately, items are cut into contiguous ranges of about equal
// solve cost, and one iteration solves each device's ranges and exchanges the new rows between the devices (multi_als_epoch).
// A row's solve reads only the full other side, its Gram matrix and the row's own entries, so the split changes no floating-point
// operation: the factors are bit-identical to a single device's.  Top-N: each child scores the users of its range.
//
// The multi code drives the children through the public lrk_* entry points only.
#pragma once
#include "lrk_common.cuh"
#include "als.cuh"
#include "topn_tc.cuh"
#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <new>
#include <mutex>
#include <thread>
#include <vector>

#define LRK_ALS_EVENTS 9   // per device and WRMF iteration: start, Gram(Q), users, P pull start / end, Gram(P), items, Q pull start / end

// one host thread that runs submitted jobs in order; the destructor stops and joins it
struct LrkWorker {
    std::mutex m;
    std::condition_variable cv;
    std::function<int()> job;
    bool has_job = false, done = true, quit = false;
    int rc = 0;
    std::thread th{[this] { loop(); }};   // last member: the thread starts once the state above exists
    ~LrkWorker() {
        { std::lock_guard<std::mutex> lk(m); quit = true; cv.notify_all(); }
        th.join();
    }
    void loop() {
        std::unique_lock<std::mutex> lk(m);
        for (;;) {
            cv.wait(lk, [&] { return has_job || quit; });
            if (quit) return;
            std::function<int()> j = std::move(job);
            has_job = false;
            lk.unlock();
            const int r = j();
            lk.lock();
            rc = r; done = true;
            cv.notify_all();
        }
    }
    void submit(std::function<int()> j) {
        std::lock_guard<std::mutex> lk(m);
        job = std::move(j); has_job = true; done = false;
        cv.notify_all();
    }
    int wait() {
        std::unique_lock<std::mutex> lk(m);
        cv.wait(lk, [&] { return done; });
        return rc;
    }
};

struct MultiState {
    int n = 0;
    std::vector<int32_t> devices;
    std::vector<std::unique_ptr<LrkWorker>> workers;   // one host thread per device: created before the children, stopped after them
    std::vector<LrkChild> child;          // per device: a DSGD rank, a WRMF replica (als), or with n == 1 a plain handle
    std::vector<int64_t> ub;              // n + 1 user bounds
    bool als = false;                     // WRMF on n > 1 devices: plain children with the full matrices, rows split by solve cost
    std::vector<int64_t> ib;              // als: n + 1 item bounds (a range may be empty)
    std::vector<cudaEvent_t> als_ev;      // als: LRK_ALS_EVENTS per device (the phase split of the LRK_ALS_TRACE line)
    int32_t U = 0;
    bool masters_current = false;         // every child's fp64 masters hold its factors: no epoch, set_factors or set_train_csr
                                          // since the last multi_get_factors
    MultiState(const int32_t* dev, int n_) : n(n_), devices(dev, dev + n_), child((size_t)n_) {
        for (int g = 0; g < n; ++g) workers.emplace_back(new LrkWorker());
    }
    ~MultiState() {
        // the DSGD children's communicators are destroyed together, each child on its own thread
        for (int g = 0; g < n; ++g) workers[(size_t)g]->submit([this, g] { child[(size_t)g].reset(); return (int)LRK_OK; });
        for (auto& w : workers) w->wait();
        for (size_t e = 0; e < als_ev.size(); ++e)
            if (als_ev[e]) { cudaSetDevice(devices[e / LRK_ALS_EVENTS]); cudaEventDestroy(als_ev[e]); }
    }
};

// run f(g) on every device's thread; first failing child wins, its message is copied to the parent
static int multi_run(lrk_handle_s* h, MultiState* ms, const std::function<int(int)>& f) {
    for (int g = 0; g < ms->n; ++g)
        ms->workers[(size_t)g]->submit([&f, g]() -> int {
            try { return f(g); }
            catch (const std::bad_alloc&) { return (int)LRK_ERR_NOMEM; }       // nothing may unwind through a worker thread
            catch (...) { return (int)LRK_ERR_INVALID; }
        });
    int rc = LRK_OK;
    for (int g = 0; g < ms->n; ++g) {
        const int r = ms->workers[(size_t)g]->wait();
        if (r != LRK_OK && rc == LRK_OK) {
            rc = r;
            h->err = "device " + std::to_string(ms->devices[(size_t)g]) + ": " + ms->child[(size_t)g]->err;
        }
    }
    return rc;
}

// n + 1 bounds that cut the rows [0, rows) into n contiguous ranges of about equal total cost; with `nonempty` (rows >= n) every
// range keeps at least one row
static std::vector<int64_t> multi_cost_bounds(int64_t rows, int n, bool nonempty, const std::function<double(int64_t)>& cost) {
    std::vector<int64_t> b((size_t)n + 1, rows);
    b[0] = 0;
    double total = 0.0;
    for (int64_t r = 0; r < rows; ++r) total += cost(r);
    double acc = 0.0;
    int g = 1;
    for (int64_t r = 0; r < rows && g < n; ++r) {
        while (g < n && acc >= total * g / n) b[(size_t)g++] = r;
        acc += cost(r);
    }
    if (nonempty) {
        for (int q = 1; q < n; ++q) b[(size_t)q] = std::max(b[(size_t)q], b[(size_t)q - 1] + 1);
        for (int q = n - 1; q >= 1; --q) b[(size_t)q] = std::min(b[(size_t)q], b[(size_t)q + 1] - 1);
    }
    return b;
}

static int multi_create(const lrk_config_t* cfg, const int32_t* devices, int32_t n_devices, lrk_handle_t* out) {
    if (!cfg || !out || !devices) return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create_multi", "NULL argument", __FILE__, __LINE__);
    *out = nullptr;
    if (n_devices < 1 || n_devices > 8) return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create_multi", "1 to 8 devices", __FILE__, __LINE__);
    for (int a = 0; a < n_devices; ++a) for (int b = a + 1; b < n_devices; ++b)
        if (devices[a] == devices[b]) return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create_multi", "a device is listed twice", __FILE__, __LINE__);
    if (n_devices > 1 && lrk_model_known(cfg->model) && !lrk_model_info(*cfg).multi_device)     // an unknown model fails in lrk_create
        return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_create_multi", k_lrk_single_gpu, __FILE__, __LINE__);
    std::unique_ptr<lrk_handle_s> h(new (std::nothrow) lrk_handle_s());
    if (h) h->multi.reset(new (std::nothrow) MultiState(devices, n_devices));
    if (!h || !h->multi) return lrk_fail(nullptr, LRK_ERR_NOMEM, "lrk_create_multi", "host allocation failed", __FILE__, __LINE__);
    MultiState* ms = h->multi.get();
    h->cfg = *cfg; h->cfg.device = devices[0]; h->k = cfg->num_factors;
    ms->als = n_devices > 1 && lrk_model_known(cfg->model) && !lrk_model_info(*cfg).dsgd;     // WRMF: plain children, no DSGD
    int rc = LRK_OK;
    for (int g = 0; g < n_devices && rc == LRK_OK; ++g) {
        lrk_config_t c = *cfg;
        c.device = devices[g];
        lrk_handle_s* ch = nullptr;
        rc = lrk_create(&c, &ch);
        ms->child[(size_t)g].reset(ch);
        if (rc == LRK_OK && !ms->als) { ch->same_process = true; ch->siblings = ms->child.data(); }   // peer pointers instead of CUDA IPC
    }
    if (rc == LRK_OK && ms->als) {
        // the row exchange copies device to device: direct peer access where the pair has it (cudaMemcpyPeerAsync stages
        // through the host otherwise), and the events of the phase split
        ms->als_ev.assign((size_t)n_devices * LRK_ALS_EVENTS, nullptr);
        for (int a = 0; a < n_devices && rc == LRK_OK; ++a) {
            if (cudaSetDevice(devices[a]) != cudaSuccess) { rc = lrk_fail(h.get(), LRK_ERR_CUDA, "cudaSetDevice", cudaGetErrorString(cudaGetLastError()), __FILE__, __LINE__); break; }
            for (int b = 0; b < n_devices && rc == LRK_OK; ++b) {
                int can = 0;
                if (b == a || cudaDeviceCanAccessPeer(&can, devices[a], devices[b]) != cudaSuccess || !can) { cudaGetLastError(); continue; }
                const cudaError_t pe = cudaDeviceEnablePeerAccess(devices[b], 0);
                if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) rc = lrk_fail(h.get(), LRK_ERR_CUDA, "cudaDeviceEnablePeerAccess", cudaGetErrorString(pe), __FILE__, __LINE__);
                cudaGetLastError();
            }
            for (int e = 0; e < LRK_ALS_EVENTS && rc == LRK_OK; ++e) {
                const cudaError_t ce = cudaEventCreate(&ms->als_ev[(size_t)a * LRK_ALS_EVENTS + e]);
                if (ce != cudaSuccess) rc = lrk_fail(h.get(), LRK_ERR_CUDA, "cudaEventCreate", cudaGetErrorString(ce), __FILE__, __LINE__);
            }
        }
    } else if (rc == LRK_OK && n_devices > 1) {
        uint8_t uid[128];
        rc = lrk_comm_unique_id(uid);
        if (rc == LRK_OK) rc = multi_run(h.get(), ms, [&](int g) { return lrk_comm_init(ms->child[(size_t)g].get(), g, ms->n, uid); });
    }
    if (rc != LRK_OK) {
        const std::string why = h->err.empty() ? g_lrk_tls_error : h->err;
        h.reset();
        return lrk_fail(nullptr, rc, "lrk_create_multi", why.c_str(), __FILE__, __LINE__);
    }
    *out = h.release();
    return LRK_OK;
}

static int multi_set_train_csr(lrk_handle_s* h, int32_t U, int32_t I, const int64_t* rowptr, const int32_t* col, const double* val) {
    MultiState* ms = h->multi.get();
    LRK_REQUIRE(h, U >= ms->n, "fewer users than devices");
    ms->U = U;
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
    ms->masters_current = false;
    const int rc = multi_run(h, ms, [&](int g) -> int {
        if (ms->als) return lrk_set_train_csr(ms->child[(size_t)g].get(), U, I, rowptr, col, val);
        const int64_t lo = ms->ub[(size_t)g], hi = ms->ub[(size_t)g + 1], off = rowptr[lo];
        std::vector<int64_t> rp((size_t)(hi - lo) + 1);
        for (int64_t u = lo; u <= hi; ++u) rp[(size_t)(u - lo)] = rowptr[u] - off;
        return lrk_set_train_csr(ms->child[(size_t)g].get(), (int32_t)(hi - lo), I, rp.data(), col + off, val + off);
    });
    if (rc == LRK_OK) { h->U = U; h->I = I; h->nnz = nnz; h->has_train = true; }
    return rc;
}

static int multi_set_factors(lrk_handle_s* h, const double* P, const double* Q, const double* bu, const double* bi, double mu) {
    MultiState* ms = h->multi.get();
    LRK_REQUIRE(h, h->has_train, "call lrk_set_train_csr first (it fixes numUsers / numItems)");
    LRK_REQUIRE(h, P && Q, "P and Q are required");
    ms->masters_current = false;
    const int k = h->k;
    const int rc = multi_run(h, ms, [&](int g) {
        if (ms->als) return lrk_set_factors(ms->child[(size_t)g].get(), P, Q, bu, bi, mu);   // full replicas
        const int64_t lo = ms->ub[(size_t)g];
        return lrk_set_factors(ms->child[(size_t)g].get(), P + lo * k, Q, bu ? bu + lo : nullptr, bi, mu);
    });
    if (rc == LRK_OK) { h->has_factors = true; h->mu = mu; }
    return rc;
}

// also brings every child's fp64 masters up to date (with all four outputs NULL, that is all it does)
static int multi_get_factors(lrk_handle_s* h, double* P, double* Q, double* bu, double* bi) {
    MultiState* ms = h->multi.get();
    LRK_REQUIRE(h, h->has_factors, "no factors set");
    int rc;
    if (ms->als) {                             // the replicas are equal after every iteration, and their masters always current
        rc = lrk_get_factors(ms->child[0].get(), P, Q, bu, bi);
        if (rc) h->err = ms->child[0]->err;
    } else {
        const int k = h->k;
        rc = multi_run(h, ms, [&](int g) {     // every rank enters the ring gather; rank 0 delivers the item side
            const int64_t lo = ms->ub[(size_t)g];
            return lrk_get_factors(ms->child[(size_t)g].get(), P ? P + lo * k : nullptr, g == 0 ? Q : nullptr, bu ? bu + lo : nullptr, g == 0 ? bi : nullptr);
        });
    }
    if (rc == LRK_OK) ms->masters_current = true;
    return rc;
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
        lrk_handle_s* c = ms->child[(size_t)g].get();
        const std::vector<int64_t>& b = item_side ? ms->ib : ms->ub;
        for (int s = 0; s < ms->n; ++s) {
            const int64_t lo = b[(size_t)s], cnt = b[(size_t)s + 1] - lo;
            if (s == g || cnt == 0) continue;
            lrk_handle_s* src = ms->child[(size_t)s].get();
            double* dst = item_side ? c->Q64.ptr : c->P64.ptr;
            const double* from = item_side ? src->Q64.ptr : src->P64.ptr;
            LRK_CUDA(c, cudaMemcpyPeerAsync(dst + lo * k, c->cfg.device, from + lo * k, src->cfg.device, sizeof(double) * (size_t)(cnt * k), c->stream));
        }
        return LRK_OK;
    };
    int rc = multi_run(h, ms, [&](int g) -> int {
        lrk_handle_s* c = ms->child[(size_t)g].get();
        LRK_CUDA(c, cudaSetDevice(c->cfg.device));
        LRK_REQUIRE(c, c->als != nullptr && c->f64_valid, "ALS state missing: call lrk_set_train_csr and lrk_set_factors first");
        topn_tc_invalidate(c);                        // the solve and the pulls rewrite the masters the top-N operand is built from
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
        lrk_handle_s* c = ms->child[(size_t)g].get();
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
        lrk_handle_s* c = ms->child[(size_t)g].get();
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
    MultiState* ms = h->multi.get();
    LRK_REQUIRE(h, h->has_train && h->has_factors, "set the train CSR and the factors before training");
    ms->masters_current = false;
    if (ms->als) return multi_als_epoch(h, ms, reg_u, reg_i, loss_out);
    std::vector<double> loss((size_t)ms->n, 0.0);
    const int rc = multi_run(h, ms, [&](int g) { return lrk_sgd_epoch(ms->child[(size_t)g].get(), lr, reg_u, reg_i, reg_b, epoch_idx, &loss[(size_t)g]); });
    if (loss_out) *loss_out = loss[0];          // all-reduced: the same on every rank
    return rc;
}

// top-N: users shard by block, each child scores its own users from its fp64 masters (SURVEY.md 8e)
static int multi_topn(lrk_handle_s* h, const int32_t* users, int32_t nq, int32_t topn, int32_t exclude_train, int32_t* out_items,
                      double* out_scores, int32_t* out_counts) {
    MultiState* ms = h->multi.get();
    LRK_REQUIRE(h, h->has_factors, "no factors set");
    LRK_REQUIRE(h, topn > 0 && topn <= LRK_MAX_TOPN, "rec.recommender.ranking.topn should be more than 0!");
    if (nq == 0) return LRK_OK;
    if (users) for (int32_t c = 0; c < nq; ++c) LRK_REQUIRE(h, users[c] >= 0 && users[c] < ms->U, "user index out of range");
    else LRK_REQUIRE(h, nq <= ms->U, "nq exceeds numUsers");
    int rc;
    // a DSGD child holds only its item block until the ring gather: every rank enters it, with or without queries
    if (!ms->masters_current && (rc = multi_get_factors(h, nullptr, nullptr, nullptr, nullptr))) return rc;
    // queries by shard: a DSGD child indexes its block's users from 0, a WRMF child holds all users
    std::vector<std::vector<int32_t>> local((size_t)ms->n), pos((size_t)ms->n);
    for (int32_t c = 0; c < nq; ++c) {
        const int32_t u = users ? users[c] : c;
        int g = (int)(((int64_t)u * ms->n) / ms->U);
        while (g > 0 && u < ms->ub[(size_t)g]) --g;
        while (g + 1 < ms->n && u >= ms->ub[(size_t)g + 1]) ++g;
        local[(size_t)g].push_back(ms->als ? u : (int32_t)(u - ms->ub[(size_t)g]));
        pos[(size_t)g].push_back(c);
    }
    return multi_run(h, ms, [&](int g) -> int {
        const size_t m = local[(size_t)g].size();
        if (m == 0) return LRK_OK;
        std::vector<int32_t> it(m * (size_t)topn), cn(m);
        std::vector<double> sc(m * (size_t)topn);
        const int r = lrk_topn(ms->child[(size_t)g].get(), local[(size_t)g].data(), (int32_t)m, topn, exclude_train, it.data(), sc.data(), cn.data());
        if (r) return r;
        for (size_t t = 0; t < m; ++t) {
            const size_t c = (size_t)pos[(size_t)g][t];
            memcpy(out_items + c * topn, it.data() + t * topn, sizeof(int32_t) * (size_t)topn);
            memcpy(out_scores + c * topn, sc.data() + t * topn, sizeof(double) * (size_t)topn);
            out_counts[c] = cn[t];
        }
        return LRK_OK;
    });
}

static int multi_stage_stats(lrk_handle_s* h, int64_t out[4]) {
    MultiState* ms = h->multi.get();
    if (ms->als) {                             // every child stages the whole matrix: count it once
        lrk_handle_s* c = ms->child[0].get();
        const int rc = lrk_stage_stats(c, out);
        if (rc) h->err = c->err;
        return rc;
    }
    int64_t acc[4] = {0, 0, 0, 0};
    for (const LrkChild& c : ms->child) {
        int64_t v[4];
        const int rc = lrk_stage_stats(c.get(), v);
        if (rc) { h->err = c->err; return rc; }
        acc[0] += v[0]; acc[1] += v[1]; acc[2] = std::max(acc[2], v[2]); acc[3] = v[3];
    }
    for (int i = 0; i < 4; ++i) out[i] = acc[i];
    return LRK_OK;
}

// the users of the last top-N call summed over the children, its time the slowest child's
static int multi_topn_stats(lrk_handle_s* h, int64_t* fast_users, int64_t* fallback_users, float* ms_out) {
    int64_t a = 0, b = 0; float ms = 0.f;
    for (const LrkChild& c : h->multi->child) { a += c->topn_fast_users; b += c->topn_fallback_users; ms = std::max(ms, c->topn_ms); }
    if (fast_users) *fast_users = a;
    if (fallback_users) *fallback_users = b;
    if (ms_out) *ms_out = ms;
    return LRK_OK;
}
