// SGD epoch kernels (sm_100a): BiasedMF / PMF over a shuffled COO stream, BPR over device-drawn
// (user, positive, negative) samples.
//
// Reference semantics restated per rating (paths relative to core/src/main/java/net/librec/):
//   BiasedMF  recommender/cf/rating/BiasedMFRecommender.java:72-98
//   PMF       recommender/cf/rating/PMFSimilarityRecommender.java:64-82
//   BPR       recommender/cf/ranking/BPRRecommender.java:54-93
// The reference walks the ratings sequentially (one thread, CSR order, fp64, Gauss-Seidel).
// Here G lanes cooperate on one rating, 32/G ratings per warp step, thousands of ratings in
// flight; every update is applied with a vectorised L2 reduction (REDG.E.ADD.F32x4) so that no
// update is lost -- plain racy stores (LRK_UPDATE_HOGWILD) drift RMSE by >1e-3 on ml-100k,
// the atomic mode stays within 2e-4 of the sequential reference (DESIGN.md, "SGD update mode").
//
// Memory behaviour: triples are streamed once (ld.global.cs, 3 coalesced 128 B lines per 32
// ratings); factor rows are gathered as one float4 per lane through L2 (ld.global.cg -- L1 is
// not coherent with the REDs of other SMs), next step's rows are prefetched while the current
// step is reduced with warp shuffles.
//
// Item-run tiles: popular items receive most of the updates (Zipf), and the L2 atomic units serialise
// REDs to one address, so hot item rows bound the epoch long before HBM does -- and the more so under
// DSGD, where a sub-epoch concentrates every SM on 1/G of the catalogue (measured: 5.8 G -> 3.3 G
// updates/s per GPU at 4 strata).  Staging therefore groups the ratings of items with >= LRK_RUN_MIN_DEGREE
// ratings into runs of 32 (staging.cuh); a warp that finds all 32 items of its tile equal reads the item row once
// per flush period, accumulates the item-side deltas in registers and issues ONE vector RED for them (a
// mini-batch for that item; the user side is untouched).  The period is 8 ratings, 16 from hot_flush_deg
// ratings per item and the whole tile from twice that (default 512 / 1024: <= 1/32 of the item's ratings).
// Every flush of a hot item is 16 REDs to the same two lines, and same-line REDs serialise in L2: on one of 8
// DSGD item blocks of the ML-20M shape the epoch kernel took 0.32 ms with 8-rating flushes, 0.24 ms with these
// (tools/probe_block_shape.py); the whole matrix 1.74 -> 1.64 ms.
//
// Stability: B ratings of one item in flight at once act like ONE step of size lr*B on its bias
// (e' = (1 - lr*B) e; unstable from lr*B = 2), whereas the reference's sequential walk over the same B ratings
// contracts the error by (1 - lr)^B ~ exp(-lr*B) and never overshoots.  With x = lr * B_i,
// B_i = deg_i * (ratings in flight) / n, the item-side delta of a run tile is therefore scaled by
// (1 - exp(-x)) / x: identical to plain SGD for x -> 0, the sequential limit for popular items, stable at any
// concurrency.  The item row has curvature |p_u|^2 along p_u (PMF on un-centred ratings aligns all user vectors,
// |p|^2 grows to ~8 at k=128), so x is multiplied by max(1, mean |p_u|^2): the value at the start of the epoch
// (user_norm2_kernel, read from device memory) for a warp's first run tile, then the mean over the 32 users of
// the warp's previous run tile (the factors grow fast in the first epochs; 5 shuffles per tile).  Config C4 (PMF k=128, lr 0.01, Netflix
// shape) ran at 1.2 G updates/s behind the rollback safeguard (grid / 8) before this, at 6.6 G without a rollback after.  (Without it the grid had to be capped at lr * s * in-flight <= 1, s = share of the hottest item,
// which left 142 of 592 CTAs at 8 DSGD strata; that cap is gone.)
#pragma once
#include "lrk_common.cuh"

struct SgdParams {
    const int32_t* __restrict__ su;
    const int32_t* __restrict__ si;
    const float* __restrict__ sr;
    int64_t n;
    int64_t n_entries;      // AoBPR: entries of the staged stream (su / si), the population of its (u, i) draw
    float* P;
    float* Q;
    float* bu;
    float* bi;
    float mu, lr, reg_u, reg_i, reg_b;
    double* loss;
    int ld;
    // tile t of the epoch is read from stream position (t * tile_mul) % ntiles: the staged stream is
    // [item-run tiles | shuffled remainder], the multiplicative walk interleaves the two evenly in time
    int64_t tile_mul;
    int conc_div;           // >= 1: divisor of the grid (rollback safeguard, lrk_epoch.cuh), filled in by sgd_grid
    // staleness-aware step of item-run tiles: item_deg[i] = ratings of item i in this launch (NULL = off),
    // inflight_frac = (ratings in flight) / n, filled in by sgd_grid
    const uint32_t* item_deg;
    float inflight_frac;
    // run tiles of items with at least this many ratings flush every 16 ratings, from twice this on once per tile
    uint32_t hot_flush_deg;
    const float* pnorm2;    // device scalar: mean |p_u|^2 of the rank's user factors at the start of the epoch (NULL = 1)
    // RankSGD only: inclusive prefix sums of the item degrees (item_cum[I-1] == n); a uniform t in [0, n) picks the first
    // item with item_cum[item] > t, i.e. an item with probability users(j) / numRates
    const uint32_t* item_cum;
    // BPR only
    const int64_t* __restrict__ rowptr;
    const int32_t* __restrict__ col;
    int32_t U, I;
    uint32_t seed_lo, seed_hi, epoch;
    int64_t sample_base;    // first Philox sample counter of this launch (the windows of one epoch draw from disjoint ranges)
    // AoBPR only (adaptive oversampling, AoBPRRecommender.java:100-138): per-factor item rankings, factor variances and the
    // cumulative rank distribution, refreshed by the host every |I| ln |I| samples (sgd_aobpr.cuh)
    const int32_t* __restrict__ ao_rank;   // [k][I]: ao_rank[f * I + r] = item of rank r in factor f (descending value)
    const float* __restrict__ ao_var;      // [k]
    const float* __restrict__ ao_cum;      // [I] inclusive cumulative of exp(-((r + 1) / lambda)) / sum
};

__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }

template <bool ATOMIC>
__device__ __forceinline__ void apply4(float* addr, const float4& old, const float4& d) {
    if (ATOMIC) {
        asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(addr), "f"(d.x), "f"(d.y), "f"(d.z), "f"(d.w)
                     : "memory");
    } else {
        float4 nv = make_float4(old.x + d.x, old.y + d.y, old.z + d.z, old.w + d.w);
        __stcg(reinterpret_cast<float4*>(addr), nv);
    }
}
template <bool ATOMIC>
__device__ __forceinline__ void apply1(float* addr, float old, float d) {
    if (ATOMIC) {
        asm volatile("red.global.add.f32 [%0], %1;" ::"l"(addr), "f"(d) : "memory");
    } else {
        __stcg(addr, old + d);
    }
}

template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int m = G / 2; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    return v;
}

__device__ __forceinline__ float dot4(const float4& a, const float4& b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }

__device__ __forceinline__ void block_loss_commit(double v, double* out) {
    __shared__ double s_part[32];
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) s_part[w] = v;
    __syncthreads();
    if (w == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        double t = l < nw ? s_part[l] : 0.0;
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) t += __shfl_xor_sync(0xffffffffu, t, m);
        if (l == 0) atomicAdd(out, t);
    }
}

// ---------------------------------------------------------------------------------------------
// BiasedMF / PMF.  G lanes per rating, V float4 per lane (row length ld = 4*G*V floats).
// ---------------------------------------------------------------------------------------------
// TRACK: refresh the curvature estimate max(1, mean |p_u|^2) from every run tile (a few registers and 5 shuffles per
// tile; chosen by the launcher when the user factors are no longer small, see sgd_want_track)
template <int G, int V, bool BIASED, bool ATOMIC, bool TRACK = false>
__global__ void __launch_bounds__(256, (G * V <= 16 && !TRACK) ? 4 : ((G * V <= 32) ? 3 : 1)) sgd_rating_epoch_kernel(SgdParams p) {
#include "sgd_rating_body.inc"
    block_loss_commit(loss_d, p.loss);
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11) -- counter-based, so a sample's draws depend only on
// (seed, epoch, sample index, attempt) and lrk_bpr_peek_samples can replay them.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += 0x9E3779B9u; key.y += 0xBB67AE85u;
    }
    return ctr;
}

__device__ __forceinline__ bool row_contains(const int32_t* __restrict__ col, int64_t b, int64_t e, int32_t x) {
    while (b < e) {
        const int64_t m = (b + e) >> 1;
        const int32_t c = __ldg(col + m);
        if (c == x) return true;
        if (c < x) b = m + 1; else e = m;
    }
    return false;
}

// BPRRecommender.java:54-67 restated with a counter-based generator: user uniform over users that
// have at least one and fewer than numItems train items; positive uniform over the user's row;
// negative uniform over items NOT in the row (rejection).  uniform(n) = mulhi(r32, n).
// Both loops are bounded (LRK_BPR_MAX_ATTEMPTS Philox blocks each): the reference spins for ever when no user qualifies or a
// user has rated (practically) everything; here such a sample is skipped (u = -1) instead of hanging the GPU.
#define LRK_BPR_MAX_ATTEMPTS 256u
__device__ __forceinline__ void bpr_draw(const SgdParams& p, int64_t s_in, int32_t& u, int32_t& pi, int32_t& nj) {
    const uint2 key = make_uint2(p.seed_lo, p.seed_hi);
    const int64_t s = s_in + p.sample_base;        // multi-GPU: the windows of one epoch draw from disjoint counter ranges
    uint32_t attempt = 0;
    while (attempt < LRK_BPR_MAX_ATTEMPTS) {
        uint4 x = philox4x32_10(make_uint4((uint32_t)s, (uint32_t)(s >> 32), p.epoch, attempt++), key);
        u = (int32_t)__umulhi(x.x, (uint32_t)p.U);
        const int64_t b = __ldg(p.rowptr + u), e = __ldg(p.rowptr + u + 1);
        const int64_t len = e - b;
        if (len == 0 || len == p.I) continue;
        pi = __ldg(p.col + b + (int64_t)__umulhi(x.y, (uint32_t)len));
        nj = (int32_t)__umulhi(x.z, (uint32_t)p.I);
        if (!row_contains(p.col, b, e, nj)) return;
        nj = (int32_t)__umulhi(x.w, (uint32_t)p.I);
        if (!row_contains(p.col, b, e, nj)) return;
        for (const uint32_t stop = attempt + LRK_BPR_MAX_ATTEMPTS; attempt < stop;) {
            x = philox4x32_10(make_uint4((uint32_t)s, (uint32_t)(s >> 32), p.epoch, attempt++), key);
            nj = (int32_t)__umulhi(x.x, (uint32_t)p.I); if (!row_contains(p.col, b, e, nj)) return;
            nj = (int32_t)__umulhi(x.y, (uint32_t)p.I); if (!row_contains(p.col, b, e, nj)) return;
            nj = (int32_t)__umulhi(x.z, (uint32_t)p.I); if (!row_contains(p.col, b, e, nj)) return;
            nj = (int32_t)__umulhi(x.w, (uint32_t)p.I); if (!row_contains(p.col, b, e, nj)) return;
        }
        break;
    }
    u = -1; pi = 0; nj = 0;
}

// AoBPR draw (AoBPRRecommender.java:100-138): a train ENTRY uniformly (u, i) -- the staged stream is a permutation of the entries, so
// a uniform stream position is a uniform entry --, then the negative by adaptive oversampling: rank r from the geometric-like step
// distribution exp(-((r + 1) / lambda)), factor f with probability |p_uf| var_f / sum, item = the r-th item of factor f's ranking
// from the top if p_uf > 0, from the bottom otherwise; redrawn while the user has rated it.
__device__ __forceinline__ void aobpr_draw(const SgdParams& p, int64_t s_in, int32_t& u, int32_t& pi, int32_t& nj) {
    const uint2 key = make_uint2(p.seed_lo, p.seed_hi);
    const int64_t s = s_in + p.sample_base;
    const int k = p.ld;                                    // padded columns are zero: they never win a draw
    uint32_t attempt = 0;
    while (attempt < LRK_BPR_MAX_ATTEMPTS) {
        uint4 x = philox4x32_10(make_uint4((uint32_t)s, (uint32_t)(s >> 32), p.epoch, attempt++), key);
        const int64_t d = (int64_t)(((unsigned long long)x.x * (unsigned long long)p.n_entries) >> 32);
        u = __ldg(p.su + d);
        const int64_t b = __ldg(p.rowptr + u), e = __ldg(p.rowptr + u + 1);
        if (e - b == 0 || e - b == p.I) continue;
        pi = __ldg(p.si + d);
        const float* pu = p.P + (int64_t)u * p.ld;
        float tot = 0.f;
        for (int f = 0; f < k; ++f) tot += fabsf(__ldcg(pu + f)) * __ldg(p.ao_var + f);
        uint32_t w[3] = {x.y, x.z, x.w};
        int have = 3;
        for (const uint32_t stop = attempt + LRK_BPR_MAX_ATTEMPTS; attempt < stop;) {
            if (have < 2) {
                x = philox4x32_10(make_uint4((uint32_t)s, (uint32_t)(s >> 32), p.epoch, attempt++), key);
                w[0] = x.x; w[1] = x.y; w[2] = x.z; have = 3;
            }
            // rank: first r with cum[r] > t
            const float t = (float)w[--have] * 2.3283064e-10f;
            int lo = 0, hi = p.I - 1;
            while (lo < hi) { const int m = (lo + hi) >> 1; if (__ldg(p.ao_cum + m) > t) hi = m; else lo = m + 1; }
            const int r = lo;
            // factor: first f whose cumulative |p_uf| var_f exceeds t2 * total
            const float t2 = (float)w[--have] * 2.3283064e-10f * tot;
            float acc = 0.f;
            int fsel = k - 1;
            for (int f = 0; f < k; ++f) { acc += fabsf(__ldcg(pu + f)) * __ldg(p.ao_var + f); if (acc > t2) { fsel = f; break; } }
            nj = __ldcg(pu + fsel) > 0.f ? __ldg(p.ao_rank + (int64_t)fsel * p.I + r) : __ldg(p.ao_rank + (int64_t)fsel * p.I + (p.I - r - 1));
            if (!row_contains(p.col, b, e, nj)) return;
        }
        break;
    }
    u = -1; pi = 0; nj = 0;
}

__global__ void bpr_peek_kernel(SgdParams p, int64_t first, int64_t n, int32_t* out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int32_t u, pi, nj;
    if (p.ao_rank) aobpr_draw(p, first + t, u, pi, nj); else bpr_draw(p, first + t, u, pi, nj);
    out[3 * t] = u; out[3 * t + 1] = pi; out[3 * t + 2] = nj;
}

template <int G, int V, bool ATOMIC, bool AOBPR = false>
__global__ void __launch_bounds__(256) sgd_bpr_epoch_kernel(SgdParams p) {
    constexpr int RPS = 32 / G;
    constexpr int STEPS = G;
    const int lane = threadIdx.x & 31;
    const int sub = lane % G;
    const int grp = lane / G;
    const int64_t gwarp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t ntiles = (p.n + 31) >> 5;
    const float lr = p.lr, reg_u = p.reg_u, reg_i = p.reg_i;
    double loss_d = 0.0;

    for (int64_t tile = gwarp; tile < ntiles; tile += nwarps) {
        int32_t u_l = -1, i_l = 0, j_l = 0;
        {
            const int64_t s = (tile << 5) + lane;
            if (s < p.n) {
                if (AOBPR) aobpr_draw(p, s, u_l, i_l, j_l);
                else bpr_draw(p, s, u_l, i_l, j_l);
            }
        }
        float loss_f = 0.f;
        float4 pn[V], qin[V], qjn[V];
        int32_t un, in_, jn;
        un = __shfl_sync(0xffffffffu, u_l, grp);
        in_ = __shfl_sync(0xffffffffu, i_l, grp);
        jn = __shfl_sync(0xffffffffu, j_l, grp);
#pragma unroll
        for (int v = 0; v < V; ++v) {
            pn[v] = make_float4(0.f, 0.f, 0.f, 0.f); qin[v] = pn[v]; qjn[v] = pn[v];
            if (un >= 0) {
                pn[v] = ldcg4(p.P + (int64_t)un * p.ld + (v * G + sub) * 4);
                qin[v] = ldcg4(p.Q + (int64_t)in_ * p.ld + (v * G + sub) * 4);
                qjn[v] = ldcg4(p.Q + (int64_t)jn * p.ld + (v * G + sub) * 4);
            }
        }
#pragma unroll
        for (int s = 0; s < STEPS; ++s) {
            float4 pc[V], qic[V], qjc[V];
#pragma unroll
            for (int v = 0; v < V; ++v) { pc[v] = pn[v]; qic[v] = qin[v]; qjc[v] = qjn[v]; }
            const int32_t uc = un, ic = in_, jc = jn;
            if (s + 1 < STEPS) {
                const int src = (s + 1) * RPS + grp;
                un = __shfl_sync(0xffffffffu, u_l, src);
                in_ = __shfl_sync(0xffffffffu, i_l, src);
                jn = __shfl_sync(0xffffffffu, j_l, src);
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    pn[v] = make_float4(0.f, 0.f, 0.f, 0.f); qin[v] = pn[v]; qjn[v] = pn[v];
                    if (un >= 0) {
                        pn[v] = ldcg4(p.P + (int64_t)un * p.ld + (v * G + sub) * 4);
                        qin[v] = ldcg4(p.Q + (int64_t)in_ * p.ld + (v * G + sub) * 4);
                        qjn[v] = ldcg4(p.Q + (int64_t)jn * p.ld + (v * G + sub) * 4);
                    }
                }
            }
            float part = 0.f;
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const float4 a = pc[v], b = qic[v], c = qjc[v];
                part += a.x * (b.x - c.x) + a.y * (b.y - c.y) + a.z * (b.z - c.z) + a.w * (b.w - c.w);
            }
            const float x = group_sum<G>(part);             // posPredict - negPredict
            // deri = logistic(-x) = 1/(1+e^x); lossValue = -ln(logistic(x)) = ln(1+e^-x)
            const float deri = 1.f / (1.f + expf(x));
            if (uc >= 0) {
                float reg_acc = 0.f;
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const float4 a = pc[v], b = qic[v], c = qjc[v];
                    float4 dp, di, dj;
                    dp.x = lr * (deri * (b.x - c.x) - reg_u * a.x); di.x = lr * (deri * a.x - reg_i * b.x); dj.x = lr * (-deri * a.x - reg_i * c.x);
                    dp.y = lr * (deri * (b.y - c.y) - reg_u * a.y); di.y = lr * (deri * a.y - reg_i * b.y); dj.y = lr * (-deri * a.y - reg_i * c.y);
                    dp.z = lr * (deri * (b.z - c.z) - reg_u * a.z); di.z = lr * (deri * a.z - reg_i * b.z); dj.z = lr * (-deri * a.z - reg_i * c.z);
                    dp.w = lr * (deri * (b.w - c.w) - reg_u * a.w); di.w = lr * (deri * a.w - reg_i * b.w); dj.w = lr * (-deri * a.w - reg_i * c.w);
                    apply4<ATOMIC>(p.P + (int64_t)uc * p.ld + (v * G + sub) * 4, a, dp);
                    apply4<ATOMIC>(p.Q + (int64_t)ic * p.ld + (v * G + sub) * 4, b, di);
                    apply4<ATOMIC>(p.Q + (int64_t)jc * p.ld + (v * G + sub) * 4, c, dj);
                    reg_acc += reg_u * dot4(a, a) + reg_i * dot4(b, b) + reg_i * dot4(c, c);
                }
                if (sub == 0) reg_acc += (x > 0.f) ? log1pf(expf(-x)) : (-x + log1pf(expf(x)));
                loss_f += reg_acc;
            }
        }
        loss_d += (double)loss_f;
    }
    block_loss_commit(loss_d, p.loss);
}

// ---------------------------------------------------------------------------------------------
// RankSGD (SURVEY.md 8f, row N3): recommender/cf/ranking/RankSGDRecommender.java:62-108.  One update per TRAIN ENTRY
// (u, i, r) -- the staged COO stream, position s = sample s -- against a negative item j drawn with probability
// users(j) / numRates and redrawn while the user has rated it (:73-89): uniform t in [0, nnz) -> first item whose
// inclusive degree prefix exceeds t (exact integer arithmetic; the reference walks an ascending probability list with
// a double).  error = (p_u.q_i - p_u.q_j) - r (:94); p_u -= lr e (q_i - q_j), q_i -= lr e p_u, q_j += lr e p_u with the
// OLD p_u (:99-105); no regularisation; loss = 0.5 * sum e^2.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int32_t ranksgd_pick(const uint32_t* __restrict__ cum, int32_t I, uint32_t t) {
    int32_t lo = 0, hi = I;
    while (lo < hi) {
        const int32_t m = (lo + hi) >> 1;
        if (__ldg(cum + m) > t) hi = m; else lo = m + 1;
    }
    return lo < I ? lo : I - 1;
}
// false: 256 draws all hit items of the row (the user has rated practically everything that has ratings; the reference
// would spin) -- the entry is skipped
__device__ __forceinline__ bool ranksgd_draw_neg(const SgdParams& p, int64_t s, int32_t u, int32_t& nj) {
    const uint2 key = make_uint2(p.seed_lo, p.seed_hi);
    const int64_t b = __ldg(p.rowptr + u), e = __ldg(p.rowptr + u + 1);
    for (uint32_t attempt = 0; attempt < 64u; ++attempt) {
        const uint4 x = philox4x32_10(make_uint4((uint32_t)s, (uint32_t)(s >> 32), p.epoch, attempt), key);
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const uint32_t r = w == 0 ? x.x : (w == 1 ? x.y : (w == 2 ? x.z : x.w));
            nj = ranksgd_pick(p.item_cum, p.I, __umulhi(r, (uint32_t)p.n));
            if (!row_contains(p.col, b, e, nj)) return true;
        }
    }
    return false;
}

__global__ void ranksgd_peek_kernel(SgdParams p, int64_t first, int64_t n, int32_t* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int64_t s = first + t;
    const int32_t u = p.su[s];
    int32_t nj = -1;
    if (!ranksgd_draw_neg(p, s, u, nj)) nj = -1;
    out[3 * t] = u; out[3 * t + 1] = p.si[s]; out[3 * t + 2] = nj;
}

template <int G, int V, bool ATOMIC>
__global__ void __launch_bounds__(256) sgd_ranksgd_epoch_kernel(SgdParams p) {
    constexpr int RPS = 32 / G;
    constexpr int STEPS = G;
    const int lane = threadIdx.x & 31;
    const int sub = lane % G;
    const int grp = lane / G;
    const int64_t gwarp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t ntiles = (p.n + 31) >> 5;
    const float lr = p.lr;
    double loss_d = 0.0;

    for (int64_t tile = gwarp; tile < ntiles; tile += nwarps) {
        int32_t u_l = -1, i_l = 0, j_l = 0;
        float r_l = 0.f;
        {
            // same multiplicative tile walk as the rating kernel: the staged stream is [item-run tiles | rest], and walking it
            // front to back would end every epoch on the unpopular items (measured on C1 with the oracle's arithmetic:
            // Precision@10 0.136 in that order, 0.209 in a shuffled one).  Sample index = stream position either way.
            const int64_t s = ((int64_t)(((unsigned long long)tile * (unsigned long long)p.tile_mul) % (unsigned long long)ntiles) << 5) + lane;
            if (s < p.n) {
                u_l = __ldcs(p.su + s); i_l = __ldcs(p.si + s); r_l = __ldcs(p.sr + s);
                if (!ranksgd_draw_neg(p, s, u_l, j_l)) { u_l = -1; j_l = 0; }
            }
        }
        float loss_f = 0.f;
#pragma unroll 2
        for (int s = 0; s < STEPS; ++s) {
            const int src = s * RPS + grp;
            const int32_t uc = __shfl_sync(0xffffffffu, u_l, src);
            const int32_t ic = __shfl_sync(0xffffffffu, i_l, src);
            const int32_t jc = __shfl_sync(0xffffffffu, j_l, src);
            const float rc = __shfl_sync(0xffffffffu, r_l, src);
            float4 pc[V], qic[V], qjc[V], df[V];
            float part = 0.f;
#pragma unroll
            for (int v = 0; v < V; ++v) {
                pc[v] = make_float4(0.f, 0.f, 0.f, 0.f); qic[v] = pc[v]; qjc[v] = pc[v];
                if (uc >= 0) {
                    pc[v] = ldcg4(p.P + (int64_t)uc * p.ld + (v * G + sub) * 4);
                    qic[v] = ldcg4(p.Q + (int64_t)ic * p.ld + (v * G + sub) * 4);
                    qjc[v] = ldcg4(p.Q + (int64_t)jc * p.ld + (v * G + sub) * 4);
                }
                df[v] = make_float4(qic[v].x - qjc[v].x, qic[v].y - qjc[v].y, qic[v].z - qjc[v].z, qic[v].w - qjc[v].w);
                part += dot4(pc[v], df[v]);
            }
            const float err = group_sum<G>(part) - rc;      // (posPredict - negPredict) - (posRating - 0)
            // staleness-aware step of the item side (r02; as in the rating kernel): about 2 * deg * inflight_frac samples touching the
            // same item row are in flight at once (an item is drawn as positive and, by popularity, as negative equally often), the
            // squared loss has curvature |p_u|^2 along p_u, and B concurrent steps act like one step of size lr * B * |p_u|^2 where the
            // reference's sequential walk contracts by exp(-lr * B * |p_u|^2): scale the item deltas by (1 - exp(-x)) / x
            float damp_i = 1.f, damp_j = 1.f;
            if (p.item_deg) {
                float pp = 0.f;
#pragma unroll
                for (int v = 0; v < V; ++v) pp += dot4(pc[v], pc[v]);
                pp = group_sum<G>(pp);
                if (uc >= 0) {
                    const float c = 2.f * lr * pp * p.inflight_frac;
                    const float xi = c * (float)__ldg(p.item_deg + ic), xj = c * (float)__ldg(p.item_deg + jc);
                    if (xi > 1e-3f) damp_i = (1.f - __expf(-xi)) / xi;
                    if (xj > 1e-3f) damp_j = (1.f - __expf(-xj)) / xj;
                }
            }
            if (uc >= 0) {
                const float sgd = lr * err;
                const float si_ = sgd * damp_i, sj_ = sgd * damp_j;
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const float4 a = pc[v], d = df[v];
                    const float4 dp = make_float4(-sgd * d.x, -sgd * d.y, -sgd * d.z, -sgd * d.w);
                    const float4 di = make_float4(-si_ * a.x, -si_ * a.y, -si_ * a.z, -si_ * a.w);
                    const float4 dj = make_float4(sj_ * a.x, sj_ * a.y, sj_ * a.z, sj_ * a.w);
                    apply4<ATOMIC>(p.P + (int64_t)uc * p.ld + (v * G + sub) * 4, a, dp);
                    apply4<ATOMIC>(p.Q + (int64_t)ic * p.ld + (v * G + sub) * 4, qic[v], di);
                    apply4<ATOMIC>(p.Q + (int64_t)jc * p.ld + (v * G + sub) * 4, qjc[v], dj);
                }
                if (sub == 0) loss_f += err * err;
            }
        }
        loss_d += (double)loss_f;
    }
    block_loss_commit(loss_d, p.loss);
}

// mean |p_u|^2 over the rank's users -> out[0] (float); out must be zeroed before
__global__ void user_norm2_kernel(const float* __restrict__ P, int64_t U, int ld, float* __restrict__ out) {
    float acc = 0.f;
    const int64_t n = U * ld;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) { const float v = __ldg(P + t); acc += v * v; }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, m);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc / (float)U);
}

// mean |p_u|^2 of the working user factors -> d_pnorm2 (device, read by the SGD kernel) and pnorm2_host (after the next
// stream synchronisation; pinned)
static int refresh_user_norm2(lrk_handle_s* h, bool sync) {
    cudaStream_t st = h->stream;
    int rc;
    if ((rc = lrk_dev_alloc(h, &h->d_pnorm2, 1))) return rc;
    if (!h->h_pnorm2) LRK_CUDA(h, cudaMallocHost((void**)&h->h_pnorm2, sizeof(float)));
    LRK_CUDA(h, cudaMemsetAsync(h->d_pnorm2, 0, sizeof(float), st));
    user_norm2_kernel<<<2 * h->sm_count, 256, 0, st>>>(h->P32, h->U, h->ld, h->d_pnorm2);
    LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaMemcpyAsync(h->h_pnorm2, h->d_pnorm2, sizeof(float), cudaMemcpyDeviceToHost, st));
    if (sync) LRK_CUDA(h, cudaStreamSynchronize(st));
    return LRK_OK;
}

// ---------------------------------------------------------------------------------------------
// Launch plan of the stream kernels: every launcher (one GPU, the DSGD sub-epoch loop, the fused DSGD epoch, the sample
// windows of BPR / AoBPR) takes its parameters, kernel variant, grid and in-flight share from the functions below.
// ---------------------------------------------------------------------------------------------
// A/B probes of the plan, read once per process (DESIGN.md §6.1)
struct SgdProbes {
    uint32_t hot_flush_deg = 512u;  // LRK_SGD_HOT_FLUSH: degree from which run tiles flush every 16 ratings (0 = always every 8)
    int track = -1;                 // LRK_SGD_TRACK=0/1: forces the TRACK variant of the damped atomic launches off / on
    bool trace = false;             // LRK_SGD_TRACE=1: one line per launched segment on stderr (sgd_trace)
};
static const SgdProbes& sgd_probes() {
    static const SgdProbes probes = [] {
        SgdProbes p;
        if (const char* e = getenv("LRK_SGD_HOT_FLUSH")) p.hot_flush_deg = atoi(e) > 0 ? (uint32_t)atoi(e) : 0xffffffffu;
        if (const char* e = getenv("LRK_SGD_TRACK")) p.track = atoi(e) != 0;
        if (const char* e = getenv("LRK_SGD_TRACE")) p.trace = atoi(e) != 0;
        return p;
    }();
    return probes;
}

// The handle's whole stream and model; read-only with respect to the handle (lrk_bpr_peek_samples uses it too).  DSGD ranks
// draw their samples from seeds of their own.
static SgdParams sgd_params(const lrk_handle_s* h, float lr, float reg_u, float reg_i, double reg_b, int32_t epoch_idx) {
    SgdParams sp;
    memset(&sp, 0, sizeof sp);
    sp.su = h->d_su; sp.si = h->d_si; sp.sr = h->d_sr; sp.n = h->nnz;
    sp.P = h->P32; sp.Q = h->Q32; sp.bu = h->bu32; sp.bi = h->bi32;
    sp.mu = (float)h->mu; sp.lr = lr; sp.reg_u = reg_u; sp.reg_i = reg_i; sp.reg_b = (float)reg_b;
    sp.loss = h->d_loss; sp.ld = h->ld;
    sp.item_deg = k_lrk_models[h->cfg.model].damped ? h->d_item_deg.ptr : nullptr;
    sp.hot_flush_deg = sgd_probes().hot_flush_deg;
    sp.item_cum = h->cfg.model == LRK_MODEL_RANKSGD ? h->d_item_cum.ptr : nullptr;
    sp.rowptr = h->d_rowptr; sp.col = h->d_col; sp.U = h->U; sp.I = h->I;
    const uint64_t seed = h->cfg.seed + 977u * (uint64_t)h->rank;
    sp.seed_lo = (uint32_t)seed; sp.seed_hi = (uint32_t)(seed >> 32); sp.epoch = (uint32_t)epoch_idx;
    return sp;
}

// multiplier of the tile walk: close to the golden-ratio fraction of the tile count and coprime with it
static int64_t sgd_tile_mul(int64_t n) {
    const int64_t T = (n + 31) / 32;
    if (T < 3) return 1;
    int64_t a = (int64_t)((double)T * 0.6180339887498949);
    if (a < 1) a = 1;
    auto gcd = [](int64_t x, int64_t y) { while (y) { const int64_t t = x % y; x = y; y = t; } return x; };
    while (gcd(a, T) != 1) ++a;
    return a % T ? a % T : 1;
}

// base narrowed to ratings [off, off + n) of the staged stream, trained against the item rows Q / bi of the item block that
// starts at item0 (the stream's item ids are block-local): one GPU passes the whole stream, DSGD one stratum, the sample
// windows of BPR / AoBPR their length (with sample_base set by the caller)
static SgdParams sgd_segment(const lrk_handle_s* h, const SgdParams& base, int64_t off, int64_t n, float* Q, float* bi, int32_t item0) {
    SgdParams sp = base;
    sp.su = base.su + off; sp.si = base.si + off; sp.sr = base.sr + off; sp.n = n;
    sp.tile_mul = sgd_tile_mul(n);
    sp.Q = Q; sp.bi = bi;
    sp.item_deg = base.item_deg ? base.item_deg + item0 : nullptr;
    sp.pnorm2 = sp.item_deg ? h->d_pnorm2.ptr : nullptr;
    return sp;
}

// LRK_SGD_TRACE=1: the plan of one segment (the prefix up to `track` is what tests parse)
static void sgd_trace(const lrk_handle_s* h, const SgdParams& sp, bool track, int grid, float inflight_frac) {
    if (!sgd_probes().trace) return;
    fprintf(stderr, "[sgd] epoch %u n %lld mean|p|^2 %.5f (prev %.5f) track %d conc_div %d grid %d inflight_frac %.9g tile_mul %lld hot_flush_deg %u\n",
            sp.epoch, (long long)sp.n, h->pnorm2_host, h->pnorm2_prev, (int)track, h->conc_div, grid, inflight_frac, (long long)sp.tile_mul,
            sp.hot_flush_deg);
}

// Grid of one launch over the segments seg[0..nseg) -- one, or the strata of a fused DSGD epoch -- for a kernel with rps
// ratings per warp step: whole multiples of the SM count for big inputs, no more blocks than the tiles need (8 warps per
// block, one tile per warp), and at most nnz/16 ratings in flight (8 warps x ratings-per-step x 2 pipeline stages per block)
// for the smallest segment: with the whole matrix in flight at once the epoch degenerates into one full-batch gradient
// step, which is unstable at SGD learning rates (observed: PMF on ml-100k diverges) -- DESIGN.md "staleness cap".  The
// rollback safeguard divides the result.  Writes each segment's conc_div and inflight_frac = (ratings in flight) / n.
static int sgd_grid(lrk_handle_s* h, const void* kernel, int rps, bool track, SgdParams* seg, int nseg, int* grid_out) {
    int per_sm = 0;
    LRK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0));
    int64_t grid = (int64_t)h->sm_count * std::max(per_sm, 1);
    for (int t = 0; t < nseg; ++t) {
        const int64_t n = seg[t].n;
        if (n <= 0) continue;
        grid = std::min(grid, ((n + 31) / 32 + 7) / 8);
        grid = std::min(grid, (n / 16) / (8 * (int64_t)rps * 2));
    }
    if (h->conc_div > 1) grid /= h->conc_div;
    if (grid < 1) grid = 1;
    for (int t = 0; t < nseg; ++t) {
        seg[t].conc_div = h->conc_div;
        seg[t].inflight_frac = (float)((double)grid * 8.0 * (double)std::max(rps, 8) / (double)std::max<int64_t>(seg[t].n, 1));
        sgd_trace(h, seg[t], track, (int)grid, seg[t].inflight_frac);
    }
    *grid_out = (int)grid;
    return LRK_OK;
}

// Which epoch kernel variant: TRACK follows mean |p_u|^2 of the rows in flight (curvature of the item-side step) instead of taking the
// epoch-start value.  It is needed as soon as the user factors are no longer small, and whenever they may grow within the epoch:
// PMF on un-centred ratings takes mean |p_u|^2 from 1e-4 to ~2 inside the FIRST epoch, so an epoch that starts far below any
// threshold ends far above it (r01: config C4 under 2-GPU DSGD rolled back for exactly that reason).  Hence: always for the k > 64
// layouts (3 CTAs/SM either way, the variant costs five shuffles per run tile), for the first two epochs after lrk_set_factors,
// and from mean |p_u|^2 > 0.02 on.
static bool sgd_want_track(const lrk_handle_s* h, int gv) {
    return gv >= 32 || h->epochs_done < 2 || h->pnorm2_host > 0.02f;
}
// the variant of a launch: only the damped atomic launches have a TRACK variant; LRK_SGD_TRACK overrides the rule above
static bool sgd_track(const lrk_handle_s* h, const SgdParams& sp) {
    if (h->cfg.update_mode != LRK_UPDATE_ATOMIC || !sp.item_deg) return false;
    return sgd_probes().track >= 0 ? sgd_probes().track != 0 : sgd_want_track(h, h->G * h->V);
}

// the stream kernel for (model, update mode, variant)
template <int G, int V>
static const void* sgd_kernel(const lrk_handle_s* h, const SgdParams& sp, bool track) {
    const bool atomic = h->cfg.update_mode == LRK_UPDATE_ATOMIC;
    switch (h->cfg.model) {
        case LRK_MODEL_BIASEDMF:
            return track ? (const void*)sgd_rating_epoch_kernel<G, V, true, true, true>
                         : atomic ? (const void*)sgd_rating_epoch_kernel<G, V, true, true> : (const void*)sgd_rating_epoch_kernel<G, V, true, false>;
        case LRK_MODEL_PMF:
            return track ? (const void*)sgd_rating_epoch_kernel<G, V, false, true, true>
                         : atomic ? (const void*)sgd_rating_epoch_kernel<G, V, false, true> : (const void*)sgd_rating_epoch_kernel<G, V, false, false>;
        case LRK_MODEL_RANKSGD:
            return atomic ? (const void*)sgd_ranksgd_epoch_kernel<G, V, true> : (const void*)sgd_ranksgd_epoch_kernel<G, V, false>;
        default:    // BPR, AoBPR
            if (sp.ao_rank) return atomic ? (const void*)sgd_bpr_epoch_kernel<G, V, true, true> : (const void*)sgd_bpr_epoch_kernel<G, V, false, true>;
            return atomic ? (const void*)sgd_bpr_epoch_kernel<G, V, true> : (const void*)sgd_bpr_epoch_kernel<G, V, false>;
    }
}

template <int G, int V>
static int sgd_launch_gv(lrk_handle_s* h, const SgdParams& seg) {
    SgdParams sp = seg;
    const bool track = sgd_track(h, sp);
    const void* kernel = sgd_kernel<G, V>(h, sp, track);
    int grid = 1, rc;
    if ((rc = sgd_grid(h, kernel, 32 / G, track, &sp, 1, &grid))) return rc;
    void* args[] = {(void*)&sp};
    LRK_CUDA(h, cudaLaunchKernel(kernel, dim3((unsigned)grid), dim3(256), args, 0, h->stream));
    h->launches++;
    return LRK_OK;
}

static int sgd_launch(lrk_handle_s* h, const SgdParams& seg) {
    return lrk_with_layout(h, [&](auto G, auto V) { return sgd_launch_gv<decltype(G)::value, decltype(V)::value>(h, seg); });
}
