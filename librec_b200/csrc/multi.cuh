// Single-process multi-GPU handle (lrk_create_multi): what the Java shim uses for rec.cuda.devices=0,1,...,7.
//
// The reference drives a recommender from ONE thread of ONE JVM (job/RecommenderJob.java:121-143), so "one process per GPU" cannot
// be reached through its plugin API.  A multi handle takes and returns the FULL matrices exactly like a single-device handle and
// does the sharding inside: users are cut into n contiguous blocks, one per device; every device gets a DSGD child handle (rank g
// of an n-rank NCCL communicator created inside this process) driven by its own host thread, because the children's calls contain
// collectives that all ranks must enter together.  Training = the children's DSGD epoch (csrc/dsgd.cuh; the in-kernel ring takes the
// neighbours' buffers by peer pointers, CUDA IPC cannot map memory of the same process); top-N = one scoring
// handle per device over its user block with the full item matrix, no collective (SURVEY.md 8e).
//
// WRMF takes another route (`als` below): no DSGD and no communicator.  Every device gets a plain child handle that stages the FULL
// train matrix and holds full replicas of P and Q; users and, separately, items are cut into contiguous ranges of about equal
// solve cost, and one iteration solves each device's ranges and exchanges the new rows between the devices (multi_als_epoch in
// lrk_api.cu).  A row's solve reads only the full other side, its Gram matrix and the row's own entries, so the split changes no
// floating-point operation: the factors are bit-identical to a single device's.
#pragma once
#include "lrk_common.cuh"
#include <algorithm>
#include <condition_variable>
#include <functional>
#include <new>
#include <mutex>
#include <thread>
#include <vector>

#define LRK_ALS_EVENTS 9   // per device and WRMF iteration: start, Gram(Q), users, P pull start / end, Gram(P), items, Q pull start / end

struct LrkWorker {
    std::thread th;
    std::mutex m;
    std::condition_variable cv;
    std::function<int()> job;
    bool has_job = false, done = true, quit = false;
    int rc = 0;
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
    void stop() {
        { std::lock_guard<std::mutex> lk(m); quit = true; cv.notify_all(); }
        if (th.joinable()) th.join();
    }
};

struct MultiState {
    int n = 0;
    std::vector<int32_t> devices;
    std::vector<lrk_handle_s*> child;     // DSGD rank per device (a plain handle when n == 1)
    std::vector<lrk_handle_s*> scorer;    // top-N handle per device over its user block (created on first use)
    std::vector<LrkWorker*> workers;
    std::vector<int64_t> ub;              // n + 1 user bounds
    bool als = false;                     // WRMF on n > 1 devices: plain children with the full matrices, rows split by solve cost
    std::vector<int64_t> ib;              // als: n + 1 item bounds (a range may be empty)
    std::vector<cudaEvent_t> als_ev;      // als: LRK_ALS_EVENTS per device (the phase split of the LRK_ALS_TRACE line)
    int32_t U = 0, I = 0;
    double mu = 0.0;
    // host copies the scoring handles are staged from
    std::vector<int64_t> rowptr;
    std::vector<int32_t> col;
    std::vector<double> P, Q, bu, bi;
    bool scorer_csr = false, scorer_factors = false;
};

// run f(g) on every device's thread; first failing child wins, its message is copied to the parent
static int multi_run(lrk_handle_s* h, MultiState* ms, const std::function<int(int)>& f, const std::vector<lrk_handle_s*>* who = nullptr) {
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
            const std::vector<lrk_handle_s*>& hs = who ? *who : ms->child;
            if ((size_t)g < hs.size() && hs[(size_t)g]) h->err = "device " + std::to_string(ms->devices[(size_t)g]) + ": " + hs[(size_t)g]->err;
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
