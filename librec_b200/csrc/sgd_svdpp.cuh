// SVD++ on the device (SURVEY.md 8f row N3): recommender/cf/rating/SVDPlusPlusRecommender.java:62-123 (extends BiasedMF).
//
// The fork's trainModel is user-major: per user with a non-empty row (:65-69)
//   1. fv = |N(u)|^-1/2 * sum_{j in N(u)} y_j over the user's row (:70-75), FIXED while the row is walked;
//   2. per rating in item order (:77-98): e = r - ((b_u + b_i + mu) + sum_f (fv_f + p_uf) q_if); the bias and factor updates of
//      BiasedMF except that the item gradient uses (p_uf + fv_f); steps_f += e * q_if(old) * scale;
//   3. every y_j of the row moves by lr * (steps_f - regImp * y_jf * n), the loss takes regImp * y_jf^2 * n (:99-107).
// On the device a WORKER (G lanes, one float4 of a row per lane) owns a user for all three passes: p_u, b_u, fv and steps stay in
// registers (the user side is exact and needs no atomics: read once, stored once), pass 2 is the reference's sequential walk
// (every rating sees the previous one's update of p_u), and only the item-side rows (q_i, b_i in pass 2, y_j in pass 3) are shared
// between users: vector REDs (red.global.add.v4.f32), one per rating and row.  Users are handed out heaviest first (degree-sorted
// order, dynamic fetch), so the two workers of a warp get rows of almost equal length and the heavy tail starts first.
// Per rating: 3 row gathers (y_j, q_i, y_j) + 2 row REDs (q_i, y_j).
#pragma once
#include "lrk_common.cuh"
#include "sgd.cuh"

struct SvdppParams {
    const int64_t* __restrict__ rowptr; const int32_t* __restrict__ col; const float* __restrict__ cval;   // train CSR (values in CSR order)
    const int32_t* __restrict__ uorder;      // users by descending degree
    int32_t U;
    unsigned int* counter;                   // dynamic user fetch (zeroed before the launch)
    float* P; float* Q; float* Y; float* bu; float* bi;
    float mu, lr, reg_u, reg_i, reg_b, reg_imp;
    double* loss;
    int ld;
};

template <int G, int V>
__global__ void __launch_bounds__(256) sgd_svdpp_epoch_kernel(SvdppParams p) {
    constexpr int NWW = 32 / G;
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int sub = lane % G;
    const int grp = lane / G;
    const float lr = p.lr, reg_u = p.reg_u, reg_i = p.reg_i, reg_b = p.reg_b, reg_imp = p.reg_imp, mu = p.mu;
    double loss_d = 0.0;
    for (;;) {
        // one fetch per warp: NWW consecutive positions of the degree-sorted order (rows of almost equal length)
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(p.counter, (unsigned)NWW);
        base = __shfl_sync(FULL, base, 0);
        if (base >= (unsigned)p.U) break;
        const unsigned pos = base + (unsigned)grp;
        const bool on = pos < (unsigned)p.U;
        const int32_t u = on ? __ldg(p.uorder + pos) : 0;
        const int64_t rb = on ? __ldg(p.rowptr + u) : 0, re = on ? __ldg(p.rowptr + u + 1) : 0;
        const int n = (int)(re - rb);
        int nmax = n;
#pragma unroll
        for (int m = G; m < 32; m <<= 1) nmax = max(nmax, __shfl_xor_sync(FULL, nmax, m));
        if (nmax == 0) break;                         // the order is descending: everything that follows is empty too
        const float scale = n > 0 ? rsqrtf((float)n) : 0.f;
        // ---- pass 1: fv = scale * sum of the row's y_j
        float4 fv[V];
#pragma unroll
        for (int v = 0; v < V; ++v) fv[v] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int c = 0; c < nmax; c += G) {
            int32_t j_l = -1;
            if (c + sub < n) j_l = __ldg(p.col + rb + c + sub);
#pragma unroll 4
            for (int s = 0; s < G; ++s) {
                const int32_t j = __shfl_sync(FULL, j_l, s, G);
                if (j >= 0) {
#pragma unroll
                    for (int v = 0; v < V; ++v) {
                        const float4 y = ldcg4(p.Y + (int64_t)j * p.ld + (v * G + sub) * 4);
                        fv[v].x += y.x; fv[v].y += y.y; fv[v].z += y.z; fv[v].w += y.w;
                    }
                }
            }
        }
#pragma unroll
        for (int v = 0; v < V; ++v) { fv[v].x *= scale; fv[v].y *= scale; fv[v].z *= scale; fv[v].w *= scale; }
        // ---- pass 2: the row's ratings in item order against p_u (registers); q_i / b_i by RED
        float4 pu[V], steps[V];
#pragma unroll
        for (int v = 0; v < V; ++v) {
            pu[v] = n > 0 ? ldcg4(p.P + (int64_t)u * p.ld + (v * G + sub) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            steps[v] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float ub = (n > 0 && sub == 0) ? __ldcg(p.bu + u) : 0.f;
        float loss_f = 0.f;
        for (int c = 0; c < nmax; c += G) {
            int32_t i_l = -1;
            float r_l = 0.f;
            if (c + sub < n) { i_l = __ldg(p.col + rb + c + sub); r_l = __ldg(p.cval + rb + c + sub); }
            // rows of the chunk's first rating, then one rating of look-ahead
            int32_t in_ = __shfl_sync(FULL, i_l, 0, G);
            float4 qn[V];
            float bin = 0.f;
#pragma unroll
            for (int v = 0; v < V; ++v) qn[v] = in_ >= 0 ? ldcg4(p.Q + (int64_t)in_ * p.ld + (v * G + sub) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (in_ >= 0 && sub == 0) bin = __ldcg(p.bi + in_);
#pragma unroll 2
            for (int s = 0; s < G; ++s) {
                const int32_t ic = in_;
                const float rc = __shfl_sync(FULL, r_l, s, G);
                float4 q[V];
#pragma unroll
                for (int v = 0; v < V; ++v) q[v] = qn[v];
                const float ib = bin;
                if (s + 1 < G) {
                    in_ = __shfl_sync(FULL, i_l, s + 1, G);
#pragma unroll
                    for (int v = 0; v < V; ++v) qn[v] = in_ >= 0 ? ldcg4(p.Q + (int64_t)in_ * p.ld + (v * G + sub) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                    bin = (in_ >= 0 && sub == 0) ? __ldcg(p.bi + in_) : 0.f;
                }
                float part = 0.f;
#pragma unroll
                for (int v = 0; v < V; ++v)
                    part += (fv[v].x + pu[v].x) * q[v].x + (fv[v].y + pu[v].y) * q[v].y + (fv[v].z + pu[v].z) * q[v].z + (fv[v].w + pu[v].w) * q[v].w;
                if (sub == 0) part += ub + ib + mu;
                const float err = rc - group_sum<G>(part);
                if (ic >= 0) {
                    float reg_acc = 0.f;
                    const float es = err * scale;
#pragma unroll
                    for (int v = 0; v < V; ++v) {
                        const float4 a = pu[v], b = q[v], z = fv[v];
                        float4 dq;
                        dq.x = lr * (err * (a.x + z.x) - reg_i * b.x); dq.y = lr * (err * (a.y + z.y) - reg_i * b.y);
                        dq.z = lr * (err * (a.z + z.z) - reg_i * b.z); dq.w = lr * (err * (a.w + z.w) - reg_i * b.w);
                        apply4<true>(p.Q + (int64_t)ic * p.ld + (v * G + sub) * 4, dq, dq);
                        pu[v].x = a.x + lr * (err * b.x - reg_u * a.x); pu[v].y = a.y + lr * (err * b.y - reg_u * a.y);
                        pu[v].z = a.z + lr * (err * b.z - reg_u * a.z); pu[v].w = a.w + lr * (err * b.w - reg_u * a.w);
                        steps[v].x += es * b.x; steps[v].y += es * b.y; steps[v].z += es * b.z; steps[v].w += es * b.w;
                        reg_acc += reg_u * dot4(a, a) + reg_i * dot4(b, b);
                    }
                    if (sub == 0) {
                        reg_acc += err * err + reg_b * (ub * ub + ib * ib);
                        apply1<true>(p.bi + ic, 0.f, lr * (err - reg_b * ib));
                        ub += lr * (err - reg_b * ub);
                    }
                    loss_f += reg_acc;
                }
            }
        }
        if (n > 0) {                                   // the user side: exclusive owner, plain stores
#pragma unroll
            for (int v = 0; v < V; ++v) __stcg(reinterpret_cast<float4*>(p.P + (int64_t)u * p.ld + (v * G + sub) * 4), pu[v]);
            if (sub == 0) __stcg(p.bu + u, ub);
        }
        // ---- pass 3: y_j += lr * (steps - regImp * y_j * n) for every item of the row
        const float fn = (float)n;
        for (int c = 0; c < nmax; c += G) {
            int32_t j_l = -1;
            if (c + sub < n) j_l = __ldg(p.col + rb + c + sub);
#pragma unroll 4
            for (int s = 0; s < G; ++s) {
                const int32_t j = __shfl_sync(FULL, j_l, s, G);
                if (j >= 0) {
#pragma unroll
                    for (int v = 0; v < V; ++v) {
                        float* a = p.Y + (int64_t)j * p.ld + (v * G + sub) * 4;
                        const float4 y = ldcg4(a);
                        const float4 d = make_float4(lr * (steps[v].x - reg_imp * y.x * fn), lr * (steps[v].y - reg_imp * y.y * fn),
                                                     lr * (steps[v].z - reg_imp * y.z * fn), lr * (steps[v].w - reg_imp * y.w * fn));
                        apply4<true>(a, d, d);
                        loss_f += reg_imp * dot4(y, y) * fn;
                    }
                }
            }
        }
        loss_d += (double)loss_f;
    }
    block_loss_commit(loss_d, p.loss);
}

struct SvdppState {
    LrkBuf<float> d_cval;          // train values in CSR order
    LrkBuf<int32_t> d_uorder;      // users by descending degree
    LrkBuf<unsigned int> d_counter;
    LrkBuf<float> Y32;             // impItemFactors, padded rows like Q32
    LrkBuf<double> Y64;
    bool has_y = false;
    double reg_imp = 0.015;        // rec.impItem.regularization (SVDPlusPlusRecommender.java:52)
};
__global__ void svdpp_deg_kernel(const int64_t* __restrict__ rowptr, int32_t U, uint32_t* __restrict__ deg, int32_t* __restrict__ ids) {
    const int32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u < U) { deg[u] = (uint32_t)(rowptr[u + 1] - rowptr[u]); ids[u] = u; }
}
__global__ void f64_to_f32_kernel(const double* __restrict__ src, float* __restrict__ dst, int64_t n) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) dst[t] = (float)src[t];
}
