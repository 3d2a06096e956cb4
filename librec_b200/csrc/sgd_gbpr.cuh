// GBPR (group preference BPR; SURVEY.md 8f row N3): recommender/cf/ranking/GBPRRecommender.java:82-172 on the device.
//
// A sample is (u, i, G, j): u uniform over the users with ratings (:91-98), i uniform in u's row (:101), G a group of gLen users who
// rated i -- all of them when at most gLen did, otherwise u plus uniform draws from the item's column until gLen distinct users are
// found (:104-116) --, j uniform over the items u has not rated (:121-123).  Prediction of (u, i, G) =
// rho * (mean_{g in G} p_g.q_i + b_i) + (1 - rho) * (b_i + p_u.q_i) (:185-192), of (u, j) = b_j + p_u.q_j; loss and derivative as
// BPR (:127-131).  The item BIASES move immediately (:134-140); the FACTOR updates are accumulated in temporaries and added at the
// END of the epoch (:85-86,167-168), so inside an epoch every sample sees the epoch-start factors: on the device the factor side
// is an embarrassingly parallel pass (vector REDs into zeroed accumulators, one add kernel at the end of the epoch -- no staleness
// question at all), only the biases are Hogwild.  Draws are Philox4x32-10 keyed by (seed, epoch, sample, attempt) like bpr_draw.
#pragma once
#include "lrk_common.cuh"
#include "sgd.cuh"

#define LRK_GBPR_MAX_GROUP 8

struct GbprParams {
    int64_t n;                      // samples of the epoch (numRates)
    const float* P; const float* Q; // epoch-start factors (read only)
    float* tP; float* tQ;           // accumulators (zeroed before the launch)
    float* bi;
    float lr, reg_u, reg_i, reg_b, rho;
    int glen;
    double* loss;
    int ld;
    const int64_t* __restrict__ rowptr; const int32_t* __restrict__ col;     // train CSR
    const int64_t* __restrict__ colptr; const int32_t* __restrict__ cusers;   // train CSC: users of every item, ascending
    int32_t U, I;
    uint32_t seed_lo, seed_hi, epoch;
};

// one thread draws a whole sample; returns false when the sample has to be skipped (no user with ratings found / the user rated
// practically everything: bounded like bpr_draw)
__device__ __forceinline__ bool gbpr_draw(const GbprParams& p, int64_t s, int32_t& u, int32_t& pi, int32_t& nj, int32_t* grp, int& gn) {
    const uint2 key = make_uint2(p.seed_lo, p.seed_hi);
    uint32_t attempt = 0;
    uint4 x;
    int64_t b = 0, e = 0;
    for (;;) {
        if (attempt >= LRK_BPR_MAX_ATTEMPTS) return false;
        x = philox4x32_10(make_uint4((uint32_t)s, (uint32_t)(s >> 32), p.epoch, attempt++), key);
        u = (int32_t)__umulhi(x.x, (uint32_t)p.U);
        b = __ldg(p.rowptr + u); e = __ldg(p.rowptr + u + 1);
        if (e - b > 0 && e - b < p.I) break;
    }
    pi = __ldg(p.col + b + (int64_t)__umulhi(x.y, (uint32_t)(e - b)));
    // group
    const int64_t cb = __ldg(p.colptr + pi), ce = __ldg(p.colptr + pi + 1);
    const uint32_t clen = (uint32_t)(ce - cb);
    if ((int)clen <= p.glen) {
        gn = (int)clen;
        for (int t = 0; t < gn; ++t) grp[t] = __ldg(p.cusers + cb + t);
    } else {
        grp[0] = u; gn = 1;                                   // u in G, then uniform draws from the item's column until gLen distinct
        uint32_t r[4] = {x.z, x.w, 0u, 0u};
        int have = 2;
        for (int tries = 0; gn < p.glen; ++tries) {
            if (tries >= 64 * LRK_GBPR_MAX_GROUP) return false;
            if (have == 0) {
                const uint4 y = philox4x32_10(make_uint4((uint32_t)s, (uint32_t)(s >> 32), p.epoch, attempt++), key);
                r[0] = y.x; r[1] = y.y; r[2] = y.z; r[3] = y.w; have = 4;
            }
            const int32_t t1 = __ldg(p.cusers + cb + (int64_t)__umulhi(r[--have], clen));
            bool dup = false;
            for (int t = 0; t < gn; ++t) dup |= grp[t] == t1;
            if (!dup) grp[gn++] = t1;
        }
    }
    // negative item: not in u's row
    for (const uint32_t stop = attempt + LRK_BPR_MAX_ATTEMPTS; attempt < stop;) {
        const uint4 y = philox4x32_10(make_uint4((uint32_t)s, (uint32_t)(s >> 32), p.epoch, attempt++), key);
        nj = (int32_t)__umulhi(y.x, (uint32_t)p.I); if (!row_contains(p.col, b, e, nj)) return true;
        nj = (int32_t)__umulhi(y.y, (uint32_t)p.I); if (!row_contains(p.col, b, e, nj)) return true;
        nj = (int32_t)__umulhi(y.z, (uint32_t)p.I); if (!row_contains(p.col, b, e, nj)) return true;
        nj = (int32_t)__umulhi(y.w, (uint32_t)p.I); if (!row_contains(p.col, b, e, nj)) return true;
    }
    return false;
}

// debug / test aid: out[(3 + LRK_GBPR_MAX_GROUP) * t] = {u, i, j, group (padded with -1)}
__global__ void gbpr_peek_kernel(GbprParams p, int64_t first, int64_t n, int32_t* __restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int32_t u = -1, pi = -1, nj = -1, grp[LRK_GBPR_MAX_GROUP];
    int gn = 0;
    const bool ok = gbpr_draw(p, first + t, u, pi, nj, grp, gn);
    int32_t* o = out + (3 + LRK_GBPR_MAX_GROUP) * t;
    o[0] = ok ? u : -1; o[1] = pi; o[2] = nj;
    for (int g = 0; g < LRK_GBPR_MAX_GROUP; ++g) o[3 + g] = (ok && g < gn) ? grp[g] : -1;
}

// G lanes per sample (one float4 of a row per lane), 32/G samples per warp step; lane `lane` of a tile draws sample tile*32+lane
template <int G, int V>
__global__ void __launch_bounds__(256) sgd_gbpr_epoch_kernel(GbprParams p) {
    constexpr int RPS = 32 / G;
    const int lane = threadIdx.x & 31;
    const int sub = lane % G;
    const int grp_id = lane / G;
    const int64_t gwarp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t ntiles = (p.n + 31) >> 5;
    const float lr = p.lr, reg_u = p.reg_u, reg_i = p.reg_i, reg_b = p.reg_b, rho = p.rho, omr = 1.f - p.rho;
    double loss_d = 0.0;
    for (int64_t tile = gwarp; tile < ntiles; tile += nwarps) {
        int32_t u_l = -1, i_l = 0, j_l = 0, g_l[LRK_GBPR_MAX_GROUP];
        int gn_l = 0;
#pragma unroll
        for (int g = 0; g < LRK_GBPR_MAX_GROUP; ++g) g_l[g] = -1;
        {
            const int64_t s = (tile << 5) + lane;
            if (s < p.n && !gbpr_draw(p, s, u_l, i_l, j_l, g_l, gn_l)) u_l = -1;
        }
        float loss_f = 0.f;
#pragma unroll 1
        for (int st = 0; st < G; ++st) {
            const int src = st * RPS + grp_id;
            const int32_t uc = __shfl_sync(0xffffffffu, u_l, src);
            const int32_t ic = __shfl_sync(0xffffffffu, i_l, src);
            const int32_t jc = __shfl_sync(0xffffffffu, j_l, src);
            const int gn = __shfl_sync(0xffffffffu, gn_l, src);
            int32_t gu[LRK_GBPR_MAX_GROUP];
#pragma unroll
            for (int g = 0; g < LRK_GBPR_MAX_GROUP; ++g) gu[g] = __shfl_sync(0xffffffffu, g_l[g], src);
            const bool act = uc >= 0;
            float4 pu[V], qi[V], qj[V], sumg[V];
            float part_ui = 0.f, part_uj = 0.f, part_g = 0.f;
#pragma unroll
            for (int v = 0; v < V; ++v) {
                pu[v] = make_float4(0.f, 0.f, 0.f, 0.f); qi[v] = pu[v]; qj[v] = pu[v]; sumg[v] = pu[v];
                if (act) {
                    pu[v] = ldcg4(p.P + (int64_t)uc * p.ld + (v * G + sub) * 4);
                    qi[v] = ldcg4(p.Q + (int64_t)ic * p.ld + (v * G + sub) * 4);
                    qj[v] = ldcg4(p.Q + (int64_t)jc * p.ld + (v * G + sub) * 4);
                }
                part_ui += dot4(pu[v], qi[v]);
                part_uj += dot4(pu[v], qj[v]);
            }
            // group rows: sum over g of p_g (for the item update) and of p_g.q_i (for the prediction)
#pragma unroll
            for (int g = 0; g < LRK_GBPR_MAX_GROUP; ++g) {
                if (act && g < gn) {
#pragma unroll
                    for (int v = 0; v < V; ++v) {
                        const float4 pg = gu[g] == uc ? pu[v] : ldcg4(p.P + (int64_t)gu[g] * p.ld + (v * G + sub) * 4);
                        sumg[v].x += pg.x; sumg[v].y += pg.y; sumg[v].z += pg.z; sumg[v].w += pg.w;
                    }
                }
            }
#pragma unroll
            for (int v = 0; v < V; ++v) part_g += dot4(sumg[v], qi[v]);
            const float d_ui = group_sum<G>(part_ui), d_uj = group_sum<G>(part_uj), d_g = group_sum<G>(part_g);
            if (act) {
                const float avgw = 1.f / (float)gn;
                const float b_i = __ldcg(p.bi + ic), b_j = __ldcg(p.bi + jc);
                const float pos = rho * (d_g * avgw + b_i) + omr * (b_i + d_ui);
                const float neg = b_j + d_uj;
                const float x = pos - neg;
                const float deri = 1.f / (1.f + expf(x));
                float reg_acc = 0.f;
                // factor accumulators: every group member, then the two item rows
#pragma unroll
                for (int g = 0; g < LRK_GBPR_MAX_GROUP; ++g) {
                    if (g < gn) {
                        const float delta = gu[g] == uc ? 1.f : 0.f;
#pragma unroll
                        for (int v = 0; v < V; ++v) {
                            const float4 pg = gu[g] == uc ? pu[v] : ldcg4(p.P + (int64_t)gu[g] * p.ld + (v * G + sub) * 4);
                            const float4 a = qi[v], c = qj[v];
                            float4 d;
                            d.x = lr * (deri * (rho * avgw * a.x + omr * delta * a.x - delta * c.x) - reg_u * pg.x);
                            d.y = lr * (deri * (rho * avgw * a.y + omr * delta * a.y - delta * c.y) - reg_u * pg.y);
                            d.z = lr * (deri * (rho * avgw * a.z + omr * delta * a.z - delta * c.z) - reg_u * pg.z);
                            d.w = lr * (deri * (rho * avgw * a.w + omr * delta * a.w - delta * c.w) - reg_u * pg.w);
                            apply4<true>(p.tP + (int64_t)gu[g] * p.ld + (v * G + sub) * 4, d, d);
                            reg_acc += reg_u * dot4(pg, pg);
                        }
                    }
                }
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const float4 a = qi[v], c = qj[v], pu_ = pu[v], sg = sumg[v];
                    float4 di, dj;
                    di.x = lr * (deri * (rho * avgw * sg.x + omr * pu_.x) - reg_i * a.x); dj.x = lr * (-deri * pu_.x - reg_i * c.x);
                    di.y = lr * (deri * (rho * avgw * sg.y + omr * pu_.y) - reg_i * a.y); dj.y = lr * (-deri * pu_.y - reg_i * c.y);
                    di.z = lr * (deri * (rho * avgw * sg.z + omr * pu_.z) - reg_i * a.z); dj.z = lr * (-deri * pu_.z - reg_i * c.z);
                    di.w = lr * (deri * (rho * avgw * sg.w + omr * pu_.w) - reg_i * a.w); dj.w = lr * (-deri * pu_.w - reg_i * c.w);
                    apply4<true>(p.tQ + (int64_t)ic * p.ld + (v * G + sub) * 4, di, di);
                    apply4<true>(p.tQ + (int64_t)jc * p.ld + (v * G + sub) * 4, dj, dj);
                    reg_acc += reg_i * dot4(a, a) + reg_i * dot4(c, c);
                }
                if (sub == 0) {
                    reg_acc += (x > 0.f) ? log1pf(expf(-x)) : (-x + log1pf(expf(x)));
                    apply1<true>(p.bi + ic, 0.f, lr * (deri - reg_b * b_i));
                    apply1<true>(p.bi + jc, 0.f, lr * (-deri - reg_b * b_j));
                    reg_acc += reg_b * (b_i * b_i + b_j * b_j);
                }
                loss_f += reg_acc;
            }
        }
        loss_d += (double)loss_f;
    }
    block_loss_commit(loss_d, p.loss);
}

// factors += accumulators (end of the epoch, GBPRRecommender.java:167-168)
__global__ void gbpr_apply_kernel(float* __restrict__ dst, const float* __restrict__ acc, int64_t n) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) dst[t] += acc[t];
}
// train CSC from the CSR: (item, user) pairs sorted by item (stable: users ascending inside an item)
__global__ void gbpr_colptr_kernel(const uint32_t* __restrict__ deg_excl, const uint32_t* __restrict__ deg, int32_t I, int64_t* __restrict__ colptr) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < I) colptr[i] = (int64_t)deg_excl[i];
    if (i == I - 1) colptr[I] = (int64_t)deg_excl[i] + (int64_t)deg[i];
}

struct GbprState {
    LrkBuf<int64_t> d_colptr;
    LrkBuf<int32_t> d_cusers;
    LrkBuf<float> tP, tQ;
    float rho = 1.5f;            // rec.gpbr.rho   (GBPRRecommender.java:71)
    int glen = 2;                // rec.gpbr.gsize (GBPRRecommender.java:72)
};
