// Reference-order SGD (LRK_UPDATE_REFERENCE_ORDER): the reference's sequential Gauss-Seidel walk
// (BiasedMFRecommender.java:68-100 / PMFSimilarityRecommender.java:59-90: one thread, CSR order,
// fp64) executed as a dependency wavefront.  Rating e=(u,i) depends only on the previous rating of
// row u and the previous rating (in CSR order) of column i, so
//      level(e) = 1 + max(level(row predecessor), level(column predecessor))
// and all ratings of one level touch pairwise distinct users AND items: they can run in any order,
// in parallel, and still produce exactly the sequential result.  One warp owns one rating and
// evaluates it in fp64 with Java's operation order (no FMA contraction: __dmul_rn/__dadd_rn), so
// the learned factors are BIT-IDENTICAL to the reference arithmetic; only the scalar epoch loss is
// summed in a different order (agrees to ~1e-13 relative).
// Levels are separated by a grid-wide barrier inside one persistent cooperative kernel.
// Throughput is bounded by the critical path (the most-rated item: 115 812 levels for the ML-20M
// shape, 914 for ml-100k), not by bandwidth -- this is the parity mode, not the fast mode.
#pragma once
#include "lrk_common.cuh"
#include <vector>

struct ExactSchedule {
    int64_t nnz = 0;
    int32_t num_levels = 0;
    int64_t max_width = 0;
    LrkBuf<int64_t> d_level_ptr;      // num_levels + 1
    LrkBuf<int32_t> d_u;
    LrkBuf<int32_t> d_i;
    LrkBuf<double> d_r;
    LrkBuf<unsigned long long> d_bar;
    unsigned long long generation = 0;   // arrivals counted by d_bar so far; lives and dies with d_bar (a re-staged schedule starts at 0)
};

struct ExactParams {
    const int64_t* __restrict__ level_ptr;
    const int32_t* __restrict__ lu;
    const int32_t* __restrict__ li;
    const double* __restrict__ lr_val;
    int32_t num_levels;
    double* P; double* Q; double* bu; double* bi;
    double mu, learn_rate, reg_u, reg_i, reg_b;
    int k;
    double* loss;
    unsigned long long* bar;
    unsigned long long bar_base;     // barrier generation offset of this launch
};

__device__ __forceinline__ double ldcg_f64(const double* p) { return __ldcg(p); }

template <bool BIASED>
__global__ void __launch_bounds__(256) sgd_reference_order_kernel(ExactParams p) {
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int64_t gwarp = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * warps_per_block;
    const int k = p.k;
    double loss_acc = 0.0;
    for (int32_t lv = 0; lv < p.num_levels; ++lv) {
        const int64_t b = p.level_ptr[lv], e = p.level_ptr[lv + 1];
        for (int64_t t = b + gwarp; t < e; t += nwarps) {
            const int32_t u = p.lu[t], i = p.li[t];
            const double r = p.lr_val[t];
            double* pu = p.P + (int64_t)u * k;
            double* qi = p.Q + (int64_t)i * k;
            // DenseVector.dot: left-to-right sum of q[f]*p[f] from 0.0 (DenseVector.java:104-111).
            // Lanes fetch 32 factors at a time; every lane then replays the same sequential sum.
            double dot = 0.0;
            for (int f0 = 0; f0 < k; f0 += 32) {
                const int f = f0 + lane;
                double uf = 0.0, itf = 0.0;
                if (f < k) { uf = ldcg_f64(pu + f); itf = ldcg_f64(qi + f); }
                const double prod = __dmul_rn(itf, uf);
                const int n = min(32, k - f0);
                for (int j = 0; j < n; ++j) dot = __dadd_rn(dot, __shfl_sync(0xffffffffu, prod, j));
            }
            double pred = dot;
            double ub = 0.0, ib = 0.0;
            if (BIASED) {
                ub = ldcg_f64(p.bu + u); ib = ldcg_f64(p.bi + i);
                pred = __dadd_rn(__dadd_rn(__dadd_rn(dot, ub), ib), p.mu);   // BiasedMFRecommender.java:119
            }
            const double err = __dsub_rn(r, pred);
            if (lane == 0) {
                loss_acc = __dadd_rn(loss_acc, __dmul_rn(err, err));
                if (BIASED) {
                    // :82-88  bias += learnRate * (error - regBias * bias) ; loss += regBias * bias * bias
                    __stcg(p.bu + u, __dadd_rn(ub, __dmul_rn(p.learn_rate, __dsub_rn(err, __dmul_rn(p.reg_b, ub)))));
                    loss_acc = __dadd_rn(loss_acc, __dmul_rn(__dmul_rn(p.reg_b, ub), ub));
                    __stcg(p.bi + i, __dadd_rn(ib, __dmul_rn(p.learn_rate, __dsub_rn(err, __dmul_rn(p.reg_b, ib)))));
                    loss_acc = __dadd_rn(loss_acc, __dmul_rn(__dmul_rn(p.reg_b, ib), ib));
                }
            }
            for (int f = lane; f < k; f += 32) {
                const double uf = ldcg_f64(pu + f), itf = ldcg_f64(qi + f);
                // :95-97  p += lr * (e*q - regU*p) ; q += lr * (e*p_old - regI*q) ; loss += regU*p*p + regI*q*q
                __stcg(pu + f, __dadd_rn(uf, __dmul_rn(p.learn_rate, __dsub_rn(__dmul_rn(err, itf), __dmul_rn(p.reg_u, uf)))));
                __stcg(qi + f, __dadd_rn(itf, __dmul_rn(p.learn_rate, __dsub_rn(__dmul_rn(err, uf), __dmul_rn(p.reg_i, itf)))));
                loss_acc = __dadd_rn(loss_acc, __dadd_rn(__dmul_rn(__dmul_rn(p.reg_u, uf), uf), __dmul_rn(__dmul_rn(p.reg_i, itf), itf)));
            }
        }
        // grid-wide barrier between levels (all CTAs are co-resident: cooperative launch)
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            atomicAdd(p.bar, 1ULL);
            const unsigned long long target = p.bar_base + (unsigned long long)(lv + 1) * gridDim.x;
            unsigned long long seen;
            do {
                asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(seen) : "l"(p.bar) : "memory");
            } while (seen < target);
        }
        __syncthreads();
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) loss_acc += __shfl_xor_sync(0xffffffffu, loss_acc, m);
    if (lane == 0) atomicAdd(p.loss, loss_acc);
}

// Host scheduling: one O(nnz) pass in CSR order computes the levels, a counting sort groups the
// ratings by level.  (Host logic, like the reference's own CSR construction; no arithmetic on ratings.)
static int exact_build_schedule(lrk_handle_s* h, std::unique_ptr<ExactSchedule>* out, int32_t U, int32_t I, const int64_t* rowptr,
                                const int32_t* col, const double* val) {
    std::unique_ptr<ExactSchedule> s(new ExactSchedule());
    const int64_t nnz = rowptr[U];
    s->nnz = nnz;
    std::vector<int32_t> row_level((size_t)U, 0), col_level((size_t)I, 0), level((size_t)nnz);
    int32_t L = 0;
    for (int32_t u = 0; u < U; ++u)
        for (int64_t e = rowptr[u]; e < rowptr[u + 1]; ++e) {
            const int32_t i = col[e];
            const int32_t l = (row_level[u] > col_level[i] ? row_level[u] : col_level[i]) + 1;
            level[(size_t)e] = l; row_level[u] = l; col_level[i] = l;
            if (l > L) L = l;
        }
    s->num_levels = L;
    std::vector<int64_t> ptr((size_t)L + 1, 0);
    for (int64_t e = 0; e < nnz; ++e) ptr[(size_t)level[(size_t)e]]++;      // ptr[l] = count of level l (1-based)
    for (int32_t l = 1; l <= L; ++l) { if (ptr[(size_t)l] > s->max_width) s->max_width = ptr[(size_t)l]; }
    // exclusive prefix: level l (1-based) occupies [start[l-1], start[l])
    std::vector<int64_t> start((size_t)L + 1, 0);
    for (int32_t l = 1; l <= L; ++l) start[(size_t)l] = start[(size_t)l - 1] + ptr[(size_t)l];
    std::vector<int64_t> cursor(start.begin(), start.end());
    std::vector<int32_t> lu((size_t)nnz), li((size_t)nnz);
    std::vector<double> lr((size_t)nnz);
    for (int32_t u = 0; u < U; ++u)
        for (int64_t e = rowptr[u]; e < rowptr[u + 1]; ++e) {
            const int64_t pos = cursor[(size_t)level[(size_t)e] - 1]++;
            lu[(size_t)pos] = u; li[(size_t)pos] = col[e]; lr[(size_t)pos] = val[e];
        }
    int rc;
    if ((rc = lrk_dev_alloc(h, &s->d_level_ptr, (size_t)L + 1))) return rc;
    if ((rc = lrk_dev_alloc(h, &s->d_u, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &s->d_i, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &s->d_r, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &s->d_bar, 1))) return rc;
    LRK_CUDA(h, cudaMemset(s->d_bar, 0, sizeof(unsigned long long)));
    LRK_CUDA(h, cudaMemcpy(s->d_level_ptr, start.data(), sizeof(int64_t) * ((size_t)L + 1), cudaMemcpyHostToDevice));
    if (nnz) LRK_CUDA(h, cudaMemcpy(s->d_u, lu.data(), sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice));
    if (nnz) LRK_CUDA(h, cudaMemcpy(s->d_i, li.data(), sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice));
    if (nnz) LRK_CUDA(h, cudaMemcpy(s->d_r, lr.data(), sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice));
    *out = std::move(s);
    return LRK_OK;
}

static int exact_epoch(lrk_handle_s* h, ExactSchedule* s, float lr, float reg_u, float reg_i, double reg_b) {
    const bool biased = h->cfg.model == LRK_MODEL_BIASEDMF;
    ExactParams p;
    memset(&p, 0, sizeof p);
    p.level_ptr = s->d_level_ptr; p.lu = s->d_u; p.li = s->d_i; p.lr_val = s->d_r; p.num_levels = s->num_levels;
    p.P = h->P64; p.Q = h->Q64; p.bu = h->bu64; p.bi = h->bi64;
    p.mu = h->mu; p.learn_rate = (double)lr; p.reg_u = (double)reg_u; p.reg_i = (double)reg_i; p.reg_b = reg_b;
    p.k = h->k; p.loss = h->d_loss; p.bar = s->d_bar; p.bar_base = s->generation;
    void* kern = biased ? (void*)sgd_reference_order_kernel<true> : (void*)sgd_reference_order_kernel<false>;
    int per_sm = 0;
    LRK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, 0));
    int64_t grid = (s->max_width + 7) / 8;                 // one warp per rating of the widest level
    const int64_t cap = (int64_t)h->sm_count * (per_sm < 1 ? 1 : per_sm);
    if (grid > cap) grid = cap;
    if (grid > h->sm_count) grid = h->sm_count;            // one CTA per SM keeps the barrier cheap
    if (grid < 1) grid = 1;
    void* args[] = {&p};
    LRK_CUDA(h, cudaLaunchCooperativeKernel(kern, dim3((unsigned)grid), dim3(256), args, 0, h->stream));
    h->launches++;
    s->generation += (unsigned long long)s->num_levels * (unsigned long long)grid;
    return LRK_OK;
}
