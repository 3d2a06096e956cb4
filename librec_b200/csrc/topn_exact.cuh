// Exact fp64 prediction and top-N kernels (sm_100a).  They reproduce the reference arithmetic
// bit for bit when given identical factors:
//   predict      recommender/MatrixFactorizationRecommender.java:104-106, cf/rating/BiasedMFRecommender.java:118-120
//   dot order    math/structure/DenseVector.java:104-111 (f = 0..k-1, from 0.0, separate multiply and add:
//                __dmul_rn/__dadd_rn keep nvcc from contracting them into an FMA, which Java never does)
//   top-N        recommender/MatrixRecommender.java:153-201 + util/Lists.java:416-468:
//                java.util.PriorityQueue min-heap of size N fed in ascending item order, an item
//                replaces the minimum only if strictly greater under Double.compareTo, result is
//                the heap ARRAY order followed by a stable descending sort.
// The heap walk is inherently sequential per user, so one warp owns a user: lanes score 32
// consecutive items in parallel (each lane a full left-to-right dot), then the warp replays the
// 32 offers in item order against the heap kept in shared memory.
// This kernel is the exact path for every catalogue and the fallback of the tensor-core
// candidate path (topn_tc.cuh) when its exactness certificate fails.
#pragma once
#include "lrk_common.cuh"

// Double.compareTo: numeric order, except -0.0 < +0.0 (NaN never reaches the heap)
__device__ __forceinline__ int jcompare(double a, double b) {
    if (a < b) return -1;
    if (a > b) return 1;
    const long long x = __double_as_longlong(a), y = __double_as_longlong(b);
    return x == y ? 0 : (x < y ? -1 : 1);
}

__device__ __forceinline__ double dot_lr_f64(const double* __restrict__ a, const double* __restrict__ b, int k) {
    double r = 0.0;
    for (int f = 0; f < k; ++f) r = __dadd_rn(r, __dmul_rn(b[f], a[f]));
    return r;
}

// predict(u,i) for explicit pairs
__global__ void predict_pairs_kernel(const double* __restrict__ P, const double* __restrict__ Q,
                                     const double* __restrict__ bu, const double* __restrict__ bi, double mu, int biased,
                                     int k, const int32_t* __restrict__ us, const int32_t* __restrict__ is, int64_t n,
                                     double* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int32_t u = us[t], i = is[t];
    double d = dot_lr_f64(P + (int64_t)u * k, Q + (int64_t)i * k, k);
    if (biased) d = __dadd_rn(__dadd_rn(__dadd_rn(d, bu[u]), bi[i]), mu);
    out[t] = d;
}

// recommendRating(DataSet): bounded prediction per test entry (MatrixRecommender.java:230-248,272-284)
// + per-block partial sums of squared / absolute error (RMSEEvaluator.java:55, MAEEvaluator.java:56).
__global__ void eval_rating_kernel(const double* __restrict__ P, const double* __restrict__ Q,
                                   const double* __restrict__ bu, const double* __restrict__ bi, double mu, int biased,
                                   int k, int32_t U, const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                   const double* __restrict__ val, double min_rate, double max_rate,
                                   double* __restrict__ pred_out, double* __restrict__ part_se, double* __restrict__ part_ae) {
    __shared__ double s_se[256], s_ae[256];
    const int64_t nnz = rowptr[U];
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double se = 0.0, ae = 0.0;
    if (e < nnz) {
        int32_t lo = 0, hi = U;   // largest u with rowptr[u] <= e
        while (hi - lo > 1) { const int32_t m = (lo + hi) >> 1; if (rowptr[m] <= e) lo = m; else hi = m; }
        const int32_t u = lo, i = col[e];
        double p = dot_lr_f64(P + (int64_t)u * k, Q + (int64_t)i * k, k);
        if (biased) p = __dadd_rn(__dadd_rn(__dadd_rn(p, bu[u]), bi[i]), mu);
        if (p > max_rate) p = max_rate; else if (p < min_rate) p = min_rate;
        if (p != p) p = mu;
        if (pred_out) pred_out[e] = p;
        const double d = val[e] - p;
        se = d * d; ae = fabs(d);
    }
    s_se[threadIdx.x] = se; s_ae[threadIdx.x] = ae;
    __syncthreads();
    for (int m = 128; m >= 1; m >>= 1) {
        if ((int)threadIdx.x < m) { s_se[threadIdx.x] += s_se[threadIdx.x + m]; s_ae[threadIdx.x] += s_ae[threadIdx.x + m]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { part_se[blockIdx.x] = s_se[0]; part_ae[blockIdx.x] = s_ae[0]; }
}
__global__ void eval_rating_final_kernel(const double* __restrict__ part_se, const double* __restrict__ part_ae, int nb,
                                         int64_t n, double* __restrict__ out2) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double se = 0.0, ae = 0.0;
        for (int b = 0; b < nb; ++b) { se += part_se[b]; ae += part_ae[b]; }
        out2[0] = n > 0 ? sqrt(se / (double)n) : 0.0;
        out2[1] = n > 0 ? ae / (double)n : 0.0;
    }
}

// ---- java.util.PriorityQueue (JDK 8) on a shared-memory array, executed by one lane ---------
struct HeapRef {
    double* v;
    int32_t* key;
};
__device__ __forceinline__ void heap_sift_up(HeapRef h, int kpos, double xv, int32_t xk) {
    while (kpos > 0) {
        const int parent = (kpos - 1) >> 1;
        if (jcompare(xv, h.v[parent]) >= 0) break;
        h.v[kpos] = h.v[parent]; h.key[kpos] = h.key[parent];
        kpos = parent;
    }
    h.v[kpos] = xv; h.key[kpos] = xk;
}
__device__ __forceinline__ void heap_sift_down(HeapRef h, int size, int kpos, double xv, int32_t xk) {
    const int half = size >> 1;
    while (kpos < half) {
        int child = (kpos << 1) + 1;
        const int right = child + 1;
        if (right < size && jcompare(h.v[child], h.v[right]) > 0) child = right;
        if (jcompare(xv, h.v[child]) <= 0) break;
        h.v[kpos] = h.v[child]; h.key[kpos] = h.key[child];
        kpos = child;
    }
    h.v[kpos] = xv; h.key[kpos] = xk;
}
// Lists.java:436-441: poll() then add(entry) on a full heap of `size` elements
__device__ __forceinline__ void heap_replace_min(HeapRef h, int size, double xv, int32_t xk) {
    const int s = size - 1;
    const double lv = h.v[s]; const int32_t lk = h.key[s];
    if (s != 0) heap_sift_down(h, s, 0, lv, lk);
    if (s == 0) { h.v[0] = xv; h.key[0] = xk; } else heap_sift_up(h, s, xv, xk);
}

#define TOPN_WARPS 8
#define TOPN_UPW 4                      // users per warp
#define TOPN_UPB (TOPN_WARPS * TOPN_UPW)  // users per block

// smem layout (doubles first): Qs[32][k+1] | Ps[UPB][k] | hv[UPB][topn] | hk[UPB][topn] (int32)
static inline size_t topn_exact_smem(int k, int topn) {
    return sizeof(double) * ((size_t)32 * (k + 1) + (size_t)TOPN_UPB * k + (size_t)TOPN_UPB * topn) +
           sizeof(int32_t) * (size_t)TOPN_UPB * topn;
}

__global__ void __launch_bounds__(TOPN_WARPS * 32) topn_exact_kernel(
    const double* __restrict__ P, const double* __restrict__ Q, const double* __restrict__ bu,
    const double* __restrict__ bi, double mu, int biased, int k, int32_t I,
    const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, int exclude_train,
    const int32_t* __restrict__ users, int32_t nq, int topn,
    int32_t* __restrict__ out_items, double* __restrict__ out_scores, int32_t* __restrict__ out_counts) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* Qs = reinterpret_cast<double*>(smem_raw);
    double* Ps = Qs + (size_t)32 * (k + 1);
    double* hv_all = Ps + (size_t)TOPN_UPB * k;
    int32_t* hk_all = reinterpret_cast<int32_t*>(hv_all + (size_t)TOPN_UPB * topn);

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int qs_ld = k + 1;
    const int32_t c0 = blockIdx.x * TOPN_UPB;   // first query slot of this block

    // stage the block's user rows
    for (int idx = threadIdx.x; idx < TOPN_UPB * k; idx += blockDim.x) {
        const int s = idx / k, f = idx - s * k;
        const int32_t c = c0 + s;
        double v = 0.0;
        if (c < nq) { const int32_t u = users ? users[c] : c; v = P[(int64_t)u * k + f]; }
        Ps[idx] = v;
    }

    int32_t uu[TOPN_UPW];
    int64_t tp[TOPN_UPW], tend[TOPN_UPW];
    int hsize[TOPN_UPW];
    double ubias[TOPN_UPW];
#pragma unroll
    for (int j = 0; j < TOPN_UPW; ++j) {
        const int32_t c = c0 + warp * TOPN_UPW + j;
        uu[j] = c < nq ? (users ? users[c] : c) : -1;
        tp[j] = 0; tend[j] = 0; hsize[j] = 0; ubias[j] = 0.0;
        if (uu[j] >= 0) {
            if (exclude_train && rowptr) { tp[j] = rowptr[uu[j]]; tend[j] = rowptr[uu[j] + 1]; }
            if (biased) ubias[j] = bu[uu[j]];
        }
    }

    for (int32_t base = 0; base < I; base += 32) {
        __syncthreads();   // previous tile fully consumed (also covers the Ps staging on the first trip)
        for (int idx = threadIdx.x; idx < 32 * k; idx += blockDim.x) {
            const int r = idx / k, f = idx - r * k;
            const int32_t it = base + r;
            Qs[r * qs_ld + f] = it < I ? Q[(int64_t)it * k + f] : 0.0;
        }
        // train columns that can fall inside this tile (issued early, consumed after the dot loop)
        int32_t tc[TOPN_UPW];
#pragma unroll
        for (int j = 0; j < TOPN_UPW; ++j) tc[j] = (tp[j] + lane < tend[j]) ? __ldg(col + tp[j] + lane) : 0x7fffffff;
        __syncthreads();

        const int32_t item = base + lane;
        double acc[TOPN_UPW];
#pragma unroll
        for (int j = 0; j < TOPN_UPW; ++j) acc[j] = 0.0;
        const double* qrow = Qs + lane * qs_ld;
        const double* prow = Ps + (size_t)(warp * TOPN_UPW) * k;
        for (int f = 0; f < k; ++f) {
            const double q = qrow[f];
#pragma unroll
            for (int j = 0; j < TOPN_UPW; ++j) acc[j] = __dadd_rn(acc[j], __dmul_rn(q, prow[j * k + f]));
        }
        const double ibias = (biased && item < I) ? bi[item] : 0.0;

#pragma unroll
        for (int j = 0; j < TOPN_UPW; ++j) {
            if (uu[j] < 0) continue;   // warp-uniform
            double score = acc[j];
            if (biased) score = __dadd_rn(__dadd_rn(__dadd_rn(score, ubias[j]), ibias), mu);
            // train mask for [base, base+32): MatrixRecommender.java:170-174
            const bool in_win = tc[j] < base + 32;
            const uint32_t mybit = in_win ? (1u << (tc[j] - base)) : 0u;
            const uint32_t tmask = __reduce_or_sync(0xffffffffu, mybit);
            tp[j] += __popc(__ballot_sync(0xffffffffu, in_win));
            const bool valid = item < I && !((tmask >> lane) & 1u) && !(score != score);
            HeapRef h{hv_all + (size_t)(warp * TOPN_UPW + j) * topn, hk_all + (size_t)(warp * TOPN_UPW + j) * topn};
            uint32_t pend = __ballot_sync(0xffffffffu, valid);
            // Lists.java:431-433 : the first k entries are added unconditionally
            while (pend != 0u && hsize[j] < topn) {
                const int b = __ffs(pend) - 1;
                pend &= pend - 1;
                const double xv = __shfl_sync(0xffffffffu, score, b);
                if (lane == 0) heap_sift_up(h, hsize[j], xv, base + b);
                hsize[j]++;
                __syncwarp();
            }
            if (pend != 0u) {
                // Lists.java:434-441 : strictly greater than the current minimum replaces it
                const double hmin = h.v[0];
                pend &= __ballot_sync(0xffffffffu, valid && jcompare(score, hmin) > 0);
                while (pend != 0u) {
                    const int b = __ffs(pend) - 1;
                    pend &= pend - 1;
                    const double xv = __shfl_sync(0xffffffffu, score, b);
                    if (lane == 0 && jcompare(xv, h.v[0]) > 0) heap_replace_min(h, topn, xv, base + b);
                    __syncwarp();
                }
            }
        }
    }

    // new ArrayList<>(heap) then Collections.sort descending, stable (Lists.java:442-443,458-467)
    __syncwarp();
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < TOPN_UPW; ++j) {
            if (uu[j] < 0) continue;
            const int32_t c = c0 + warp * TOPN_UPW + j;
            double* hv = hv_all + (size_t)(warp * TOPN_UPW + j) * topn;
            int32_t* hk = hk_all + (size_t)(warp * TOPN_UPW + j) * topn;
            const int n = hsize[j];
            for (int a = 1; a < n; ++a) {
                const double xv = hv[a]; const int32_t xk = hk[a];
                int b = a - 1;
                while (b >= 0 && jcompare(hv[b], xv) < 0) { hv[b + 1] = hv[b]; hk[b + 1] = hk[b]; --b; }
                hv[b + 1] = xv; hk[b + 1] = xk;
            }
            for (int t = 0; t < topn; ++t) {
                out_items[(int64_t)c * topn + t] = t < n ? hk[t] : -1;
                out_scores[(int64_t)c * topn + t] = t < n ? hv[t] : 0.0;
            }
            out_counts[c] = n;
        }
    }
}

// exact fp64 top-N for `nq` query slots whose user ids are in d_users (device) or NULL (= 0..nq-1);
// results to device buffers
static int topn_exact_launch(lrk_handle_s* h, const int32_t* d_users, int32_t nq, int topn, int exclude_train,
                             int32_t* d_items, double* d_scores, int32_t* d_counts) {
    const size_t smem = topn_exact_smem(h->k, topn);
    LRK_CUDA(h, cudaFuncSetAttribute(topn_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = lrk_ceil_div(nq, TOPN_UPB);
    topn_exact_kernel<<<grid, TOPN_WARPS * 32, smem, h->stream>>>(
        h->P64, h->Q64, h->bu64, h->bi64, h->mu, lrk_has_bias(h), h->k, h->I,
        h->d_rowptr, h->d_col, exclude_train, d_users, nq, topn, d_items, d_scores, d_counts);
    LRK_LAUNCH_CHECK(h);
    return LRK_OK;
}


// ---------------------------------------------------------------------------------------------
// Item-parallel exact top-N for FEW users over a LARGE catalogue (the fallback of the tensor-core
// path and small query batches).  The Java heap replay above is sequential per user; but when the
// best N+1 exact scores of a user are pairwise different under Double.compareTo, the reference's
// result is simply those N items in descending order (ties are the only place where heap order
// matters).  So: (1) score item parts in parallel in fp64 with the reference's summation order and
// keep each part's best T=N+1, (2) merge per user and test for ties; users with a tie among the
// first N+1 (rare) are replayed by topn_exact_kernel.
// ---------------------------------------------------------------------------------------------
#define TOPN_PAR_THREADS 256
__global__ void __launch_bounds__(TOPN_PAR_THREADS) topn_exact_parts_kernel(
    const double* __restrict__ P, const double* __restrict__ Q, const double* __restrict__ bu, const double* __restrict__ bi,
    double mu, int biased, int k, int32_t I, const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
    int exclude_train, const int32_t* __restrict__ users, int n_parts, int32_t part_items, int T,
    int32_t* __restrict__ part_item_out, double* __restrict__ part_score_out, int32_t* __restrict__ part_cnt_out) {
    extern __shared__ __align__(16) unsigned char par_smem[];
    double* ps = reinterpret_cast<double*>(par_smem);                         // [k] user row
    double* lv = ps + k;                                                      // [T][256] per-thread sorted lists (slot-major)
    int32_t* li = reinterpret_cast<int32_t*>(lv + (size_t)T * TOPN_PAR_THREADS);
    double* red_v = reinterpret_cast<double*>(li + (size_t)T * TOPN_PAR_THREADS);   // [8]
    int32_t* red_i = reinterpret_cast<int32_t*>(red_v + 8);                   // [8] item
    int32_t* red_t = red_i + 8;                                               // [8] owner thread
    const int slot = blockIdx.x / n_parts, part = blockIdx.x - slot * n_parts;
    const int32_t u = users[slot];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int f = tid; f < k; f += blockDim.x) ps[f] = P[(int64_t)u * k + f];
    __syncthreads();
    const int64_t tb = (exclude_train && rowptr) ? rowptr[u] : 0, te = (exclude_train && rowptr) ? rowptr[u + 1] : 0;
    const double ub = biased ? bu[u] : 0.0;
    const int32_t i0 = part * part_items, i1 = min(I, i0 + part_items);
    int cnt = 0;
    for (int32_t it = i0 + tid; it < i1; it += blockDim.x) {
        bool skip = false;
        if (te > tb) {
            int64_t lo = tb, hi = te;
            while (lo < hi) { const int64_t m = (lo + hi) >> 1; if (__ldg(col + m) < it) lo = m + 1; else hi = m; }
            skip = lo < te && __ldg(col + lo) == it;
        }
        if (skip) continue;
        double s = dot_lr_f64(ps, Q + (int64_t)it * k, k);
        if (biased) s = __dadd_rn(__dadd_rn(__dadd_rn(s, ub), bi[it]), mu);
        if (s != s) continue;                                                  // NaN dropped (MatrixRecommender.java:186)
        // sorted insertion (descending by Double.compareTo, earlier item first among equals)
        if (cnt == T && jcompare(s, lv[(size_t)(T - 1) * TOPN_PAR_THREADS + tid]) <= 0) continue;
        int pos = cnt < T ? cnt : T - 1;
        while (pos > 0 && jcompare(lv[(size_t)(pos - 1) * TOPN_PAR_THREADS + tid], s) < 0) {
            lv[(size_t)pos * TOPN_PAR_THREADS + tid] = lv[(size_t)(pos - 1) * TOPN_PAR_THREADS + tid];
            li[(size_t)pos * TOPN_PAR_THREADS + tid] = li[(size_t)(pos - 1) * TOPN_PAR_THREADS + tid];
            --pos;
        }
        lv[(size_t)pos * TOPN_PAR_THREADS + tid] = s; li[(size_t)pos * TOPN_PAR_THREADS + tid] = it;
        if (cnt < T) ++cnt;
    }
    // merge the 256 sorted lists: T rounds of block-wide argmax over the list heads
    int head = 0, out_n = 0;
    const int64_t obase = ((int64_t)slot * n_parts + part) * T;
    for (int r = 0; r < T; ++r) {
        double bv = 0.0; int32_t bi_ = -1; int bt = -1;
        if (head < cnt) { bv = lv[(size_t)head * TOPN_PAR_THREADS + tid]; bi_ = li[(size_t)head * TOPN_PAR_THREADS + tid]; bt = tid; }
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, m);
            const int32_t oi = __shfl_xor_sync(0xffffffffu, bi_, m);
            const int ot = __shfl_xor_sync(0xffffffffu, bt, m);
            if (oi >= 0 && (bi_ < 0 || jcompare(ov, bv) > 0 || (jcompare(ov, bv) == 0 && oi < bi_))) { bv = ov; bi_ = oi; bt = ot; }
        }
        if (lane == 0) { red_v[warp] = bv; red_i[warp] = bi_; red_t[warp] = bt; }
        __syncthreads();
        bv = red_v[0]; bi_ = red_i[0]; bt = red_t[0];
        for (int w = 1; w < TOPN_PAR_THREADS / 32; ++w) {
            const double ov = red_v[w]; const int32_t oi = red_i[w];
            if (oi >= 0 && (bi_ < 0 || jcompare(ov, bv) > 0 || (jcompare(ov, bv) == 0 && oi < bi_))) { bv = ov; bi_ = oi; bt = red_t[w]; }
        }
        __syncthreads();
        if (bi_ < 0) break;
        if (tid == bt) ++head;
        if (tid == 0) { part_item_out[obase + r] = bi_; part_score_out[obase + r] = bv; }
        ++out_n;
    }
    if (tid == 0) part_cnt_out[(int64_t)slot * n_parts + part] = out_n;
}

// one warp per user: merge the parts, tie test, write the list (or flag the user for the heap replay)
__global__ void topn_exact_merge_kernel(int nq, int n_parts, int T, int topn, const int32_t* __restrict__ part_item,
                                        const double* __restrict__ part_score, const int32_t* __restrict__ part_cnt,
                                        int32_t* __restrict__ out_items, double* __restrict__ out_scores, int32_t* __restrict__ out_counts,
                                        int32_t* __restrict__ tie_flags) {
    const int slot = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (slot >= nq) return;
    int heads = 0;                       // lane p < n_parts walks part p (n_parts <= 32)
    const int mycnt = lane < n_parts ? part_cnt[(int64_t)slot * n_parts + lane] : 0;
    double prev = 0.0;
    bool tie = false;
    int n = 0;
    for (int r = 0; r < topn + 1; ++r) {
        double bv = 0.0; int32_t bi_ = -1; int bl = -1;
        if (heads < mycnt) {
            const int64_t o = ((int64_t)slot * n_parts + lane) * T + heads;
            bv = part_score[o]; bi_ = part_item[o]; bl = lane;
        }
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, m);
            const int32_t oi = __shfl_xor_sync(0xffffffffu, bi_, m);
            const int ol = __shfl_xor_sync(0xffffffffu, bl, m);
            if (oi >= 0 && (bi_ < 0 || jcompare(ov, bv) > 0 || (jcompare(ov, bv) == 0 && oi < bi_))) { bv = ov; bi_ = oi; bl = ol; }
        }
        if (bi_ < 0) break;
        if (r > 0 && jcompare(bv, prev) == 0) { tie = true; break; }
        if (r < topn) {
            if (lane == 0) { out_items[(int64_t)slot * topn + r] = bi_; out_scores[(int64_t)slot * topn + r] = bv; }
            ++n;
        }
        if (lane == bl) ++heads;
        prev = bv;
    }
    if (lane == 0) {
        for (int t = n; t < topn; ++t) { out_items[(int64_t)slot * topn + t] = -1; out_scores[(int64_t)slot * topn + t] = 0.0; }
        out_counts[slot] = n;
        tie_flags[slot] = tie ? 1 : 0;
    }
}

__global__ void topn_collect_ties_kernel(const int32_t* __restrict__ tie_flags, const int32_t* __restrict__ users, int nq,
                                         int32_t* __restrict__ tie_slots, int32_t* __restrict__ tie_users, int* __restrict__ tie_count) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nq && tie_flags[t]) { const int pos = atomicAdd(tie_count, 1); tie_slots[pos] = t; tie_users[pos] = users[t]; }
}
__global__ void topn_scatter_kernel(const int32_t* __restrict__ slots, int n, int topn, const int32_t* __restrict__ fi,
                                    const double* __restrict__ fs, const int32_t* __restrict__ fc,
                                    int32_t* __restrict__ out_items, double* __restrict__ out_scores, int32_t* __restrict__ out_counts) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * topn) return;
    const int f = t / topn, r = t - f * topn;
    const int32_t c = slots[f];
    out_items[(int64_t)c * topn + r] = fi[t];
    out_scores[(int64_t)c * topn + r] = fs[t];
    if (r == 0) out_counts[c] = fc[f];
}

// d_users: device array of nq user ids (required).  Results to device buffers [nq x topn].  Takes the staging arena: the
// callers (topn_to_device, topn_tc_run) hold none of it.
static int topn_exact_parallel_launch(lrk_handle_s* h, const int32_t* d_users, int32_t nq, int topn, int exclude_train,
                                      int32_t* d_items, double* d_scores, int32_t* d_counts) {
    cudaStream_t st = h->stream;
    const int T = topn + 1;
    int n_parts = lrk_ceil_div(2 * h->sm_count, nq);
    n_parts = n_parts < 1 ? 1 : (n_parts > 32 ? 32 : n_parts);
    int32_t part_items = lrk_ceil_div(h->I, n_parts);
    part_items = ((part_items + TOPN_PAR_THREADS - 1) / TOPN_PAR_THREADS) * TOPN_PAR_THREADS;
    n_parts = lrk_ceil_div(h->I, part_items);
    // partial lists, tie flags and the tie replay (at most nq rows) in the staging arena
    const size_t np = (size_t)nq * n_parts;
    LrkScratch sc;
    int rc = lrk_scratch_begin(h, np * T * 12 + np * 4 + (size_t)nq * 16 + (size_t)nq * topn * 12 + 9 * 256, &sc);
    if (rc) return rc;
    int32_t* pi = sc.take<int32_t>(np * T);
    double* psc = sc.take<double>(np * T);
    int32_t* pc = sc.take<int32_t>(np);
    int32_t* tie = sc.take<int32_t>((size_t)nq * 3);
    int* tcount = sc.take<int>(1);
    int32_t* fi = sc.take<int32_t>((size_t)nq * topn);
    double* fs = sc.take<double>((size_t)nq * topn);
    int32_t* fc = sc.take<int32_t>((size_t)nq);
    if (!pi || !psc || !pc || !tie || !tcount || !fi || !fs || !fc)
        return lrk_fail(h, LRK_ERR_NOMEM, "topn_exact_parallel_launch", "scratch arena too small", __FILE__, __LINE__);
    int32_t *tslots = tie + nq, *tusers = tie + 2 * (size_t)nq;
    LRK_CUDA(h, cudaMemsetAsync(tcount, 0, sizeof(int), st));
    const size_t smem = sizeof(double) * ((size_t)h->k + (size_t)T * TOPN_PAR_THREADS + 8) + sizeof(int32_t) * ((size_t)T * TOPN_PAR_THREADS + 16);
    LRK_CUDA(h, cudaFuncSetAttribute(topn_exact_parts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    topn_exact_parts_kernel<<<nq * n_parts, TOPN_PAR_THREADS, smem, st>>>(
        h->P64, h->Q64, h->bu64, h->bi64, h->mu, lrk_has_bias(h), h->k, h->I, h->d_rowptr, h->d_col,
        exclude_train, d_users, n_parts, part_items, T, pi, psc, pc);
    LRK_LAUNCH_CHECK(h);
    topn_exact_merge_kernel<<<lrk_ceil_div(nq, 4), 128, 0, st>>>(nq, n_parts, T, topn, pi, psc, pc, d_items, d_scores, d_counts, tie);
    topn_collect_ties_kernel<<<lrk_ceil_div(nq, 256), 256, 0, st>>>(tie, d_users, nq, tslots, tusers, tcount);
    h->launches += 2;
    LRK_CUDA(h, cudaGetLastError());
    int ntie = 0;
    LRK_CUDA(h, cudaMemcpyAsync(&ntie, tcount, sizeof(int), cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    if (ntie > 0) {
        if ((rc = topn_exact_launch(h, tusers, ntie, topn, exclude_train, fi, fs, fc))) return rc;
        topn_scatter_kernel<<<lrk_ceil_div((int64_t)ntie * topn, 256), 256, 0, st>>>(tslots, ntie, topn, fi, fs, fc, d_items, d_scores, d_counts);
        LRK_LAUNCH_CHECK(h);
        LRK_CUDA(h, cudaStreamSynchronize(st));
    }
    return LRK_OK;
}


// ---------------------------------------------------------------------------------------------
// Ranking evaluators over the top-N lists while they are still on the device (SURVEY.md 8f, N1):
// eval/ranking/{AUC,AveragePrecision,NormalizedDCG,Precision,Recall,ReciprocalRank}Evaluator.java.
// One thread per user; per-user terms to part[7][U] (6 measures + "user counts" flags: bit0 test row not empty,
// bit1 AP's extra condition topK != 0), reduced in a fixed order by eval_ranking_final_kernel.
// Java behaviour kept: Precision / topN; AP / min(|test|, topK);
// "NDCG" with the ideal DCG of the hit entries only; AUC's pair count in java.util.HashSet<Integer> iteration
// order of the test items (bucket (h ^ h>>>16) & (cap-1) ascending, insertion order inside a bucket).
// ---------------------------------------------------------------------------------------------
#define LRK_EVAL_MAX_TOPN 64
__device__ __forceinline__ int64_t er_find(const int32_t* __restrict__ col, int64_t b, int64_t e, int32_t key) {
    int64_t lo = b, hi = e;
    while (lo < hi) { const int64_t m = (lo + hi) >> 1; if (col[m] < key) lo = m + 1; else hi = m; }
    return (lo < e && col[lo] == key) ? lo : -1;
}
__global__ void eval_ranking_kernel(int32_t U, int32_t I, int topn, const int32_t* __restrict__ rec_items, const int32_t* __restrict__ rec_counts,
                                    const int64_t* __restrict__ t_rowptr, const int32_t* __restrict__ t_col, const double* __restrict__ t_val,
                                    const int64_t* __restrict__ train_rowptr, const int32_t* __restrict__ purchased,
                                    int32_t* __restrict__ reco_cnt, double* __restrict__ part) {
    const int32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    double auc = 0, ap = 0, ndcg = 0, prec = 0, rec = 0, rr = 0, flags = 0, info = 0;
    {   // Novelty / Entropy terms: every user's list counts (NoveltyEvaluator.java:70-82, EntropyEvaluator.java:68-76)
        const int topk_all = topn <= rec_counts[u] ? topn : rec_counts[u];
        for (int i = 0; i < topk_all; ++i) {
            const int32_t it = rec_items[(int64_t)u * topn + i];
            atomicAdd(reco_cnt + it, 1);
            const int32_t c = purchased[it];
            if (c > 0) info += -log(((double)c) / U);
        }
    }
    const int64_t tb = t_rowptr[u], te = t_rowptr[u + 1], nt = te - tb;
    if (nt > 0) {
        flags = 1;
        const int32_t* r = rec_items + (int64_t)u * topn;
        const int topk = topn <= rec_counts[u] ? topn : rec_counts[u];
        int hits = 0, miss = 0; double tmp = 0.0, dcg = 0.0; bool first = true;
        double hv[LRK_EVAL_MAX_TOPN];                      // ratings of the hit entries, kept in descending order
        for (int i = 0; i < topk; ++i) {
            const int64_t pos = er_find(t_col, tb, te, r[i]);
            if (pos >= 0) {
                const double v = t_val[pos];
                int j = hits;
                while (j > 0 && hv[j - 1] < v) { hv[j] = hv[j - 1]; --j; }
                hv[j] = v;
                ++hits;
                tmp += 1.0 * hits / (i + 1);
                if (first) { rr = 1.0 / (i + 1.0); first = false; }
                dcg += v / (log((double)(i + 2)) / log(2.0));
            } else ++miss;
        }
        prec = hits / (topn + 0.0);
        rec = hits / (nt + 0.0);
        if (topk != 0) { ap = tmp / (double)(nt < topk ? nt : topk); flags = 3; }
        if (hits > 0 && dcg != 0.0) {
            double idcg = 0.0;
            for (int j = 0; j < hits; ++j) idcg += hv[j] / (log((double)(j + 2)) / log(2.0));
            if (idcg != 0.0) ndcg = dcg / idcg;
        }
        // AUC
        const int num_dropped = (int)(I - (train_rowptr[u + 1] - train_rowptr[u])) - topk;
        const long long n_pairs = ((long long)num_dropped + topk - hits) * hits;
        if (n_pairs == 0) auc = 0.5;
        else {
            uint32_t cap = 16;
            while ((double)nt > 0.75 * (double)cap) cap <<= 1;
            long long correct = 0;
            for (int64_t e = tb; e < te; ++e) {
                const int32_t b = t_col[e];
                bool in_rec = false;
                for (int i = 0; i < topk; ++i) if (r[i] == b) { in_rec = true; break; }
                if (in_rec) continue;
                const uint32_t hb = (((uint32_t)b) ^ (((uint32_t)b) >> 16)) & (cap - 1);
                // hits that the HashSet iteration meets before b
                for (int i = 0; i < topk; ++i) {
                    const int64_t pos = er_find(t_col, tb, te, r[i]);
                    if (pos < 0) continue;
                    const uint32_t ha = (((uint32_t)r[i]) ^ (((uint32_t)r[i]) >> 16)) & (cap - 1);
                    if (ha < hb || (ha == hb && pos < e)) ++correct;
                }
            }
            correct += (long long)hits * (num_dropped - miss);
            auc = (correct + 0.0) / (double)n_pairs;
        }
    }
    part[0 * (size_t)U + u] = auc; part[1 * (size_t)U + u] = ap; part[2 * (size_t)U + u] = ndcg;
    part[3 * (size_t)U + u] = prec; part[4 * (size_t)U + u] = rec; part[5 * (size_t)U + u] = rr; part[6 * (size_t)U + u] = flags;
    part[7 * (size_t)U + u] = info;
}
__global__ void item_count_add_kernel(const int32_t* __restrict__ col, int64_t n, int32_t* __restrict__ cnt) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) atomicAdd(cnt + col[t], 1);
}
// block m sums measure m over the users (fixed order); the mean is over the users that count.
// m = 6: Novelty = sum of self-information / (U ln 2); m = 7: Entropy over the items' list frequencies.
__global__ void eval_ranking_final_kernel(const double* __restrict__ part, int32_t U, const int32_t* __restrict__ reco_cnt, int32_t I,
                                          double* __restrict__ out) {
    __shared__ double s_sum[256], s_cnt[256];
    const int m = blockIdx.x;
    double sum = 0.0, cnt = 0.0;
    if (m == 7) {
        for (int32_t i = threadIdx.x; i < I; i += blockDim.x) {
            const int32_t c = reco_cnt[i];
            if (c > 0) { const double p = ((double)c) / U; sum += p * (-log(p)); }
        }
    } else for (int32_t u = threadIdx.x; u < U; u += blockDim.x) {
        const int f = (int)part[6 * (size_t)U + u];
        if (m < 6) { sum += part[(size_t)m * U + u]; cnt += (m == 1) ? ((f & 2) ? 1.0 : 0.0) : ((f & 1) ? 1.0 : 0.0); }
        else sum += part[7 * (size_t)U + u];
    }
    s_sum[threadIdx.x] = sum; s_cnt[threadIdx.x] = cnt;
    __syncthreads();
    for (int st = 128; st >= 1; st >>= 1) {
        if ((int)threadIdx.x < st) { s_sum[threadIdx.x] += s_sum[threadIdx.x + st]; s_cnt[threadIdx.x] += s_cnt[threadIdx.x + st]; }
        __syncthreads();
    }
    if (threadIdx.x == 0)
        out[m] = m < 6 ? (s_cnt[0] > 0.0 ? s_sum[0] / s_cnt[0] : 0.0) : (m == 6 ? s_sum[0] / (U * log(2.0)) : s_sum[0] / log(2.0));
}
