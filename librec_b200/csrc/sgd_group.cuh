// BiasedMF / PMF epoch over a unit-ordered stream (staging_group.cuh) -- the order-faithful fast kernel of the rating models
// (LRK_SGD_GROUP=1; the default is the item-run-tile kernel of sgd.cuh, see the measurement at lrk_use_group_kernel).
//
// Reference loop restated per rating (core/src/main/java/net/librec/): recommender/cf/rating/BiasedMFRecommender.java:72-98,
// recommender/cf/rating/PMFSimilarityRecommender.java:64-82.  The reference walks users in CSR order, items ascending, one rating
// at a time.  Here a WORKER (G lanes, one float4 of a row per lane) owns a unit: up to 16 consecutive users whose factor rows (and
// biases) it keeps in shared memory for the whole unit -- read once, written once, exclusively, with plain loads / stores -- and
// walks the unit's ratings item by item (rotated ascending order).  For every (unit, item) pair it reads the item row once, applies
// the pair's ratings SEQUENTIALLY (every rating sees the previous one's update of the item row and of its own user row: exact
// Gauss-Seidel inside the unit, as in the reference) and adds the accumulated change of the item row to global memory with one
// vector reduction (red.global.add.v4.f32).  What is concurrent is only the item side ACROSS units.
//
// Why: the item-run-tile kernel (sgd.cuh) pays one row gather + one row RED per rating for the user side; lrk_probe_l2 shows the L2
// serves such REDs at ~6.3 TB/s against ~19.6 TB/s for gathers, and that kernel sits at ~0.87 of the 1:1 mix rate.  Units cut the
// gathers + REDs per rating to the number of distinct (unit, item) pairs per rating: 0.60-0.69 on the ML-20M shape, 0.53-0.64 on the
// Netflix shape, with the user side down to two row transfers per user and unit.
//
// Concurrency of the item side: W workers hold an item row for the length of a pair (+ one rating of prefetch), so about
// deg_i * (W * hold) / n ratings of item i are in flight at once.  As in sgd.cuh the RED of a pair is scaled by (1 - exp(-x)) / x,
// x = lr * max(1, mean |p_u|^2 of the unit) * (deg_i - pair) * (W / n) * (pair + 1): plain SGD for x -> 0, the sequential
// limit for the items everybody rates.  The curvature term comes from the unit's own rows (computed while they are loaded).
//
// Heavy users (more ratings in the block than a unit holds) are single-user units per slice; their slices run concurrently, each on a
// private copy of the user's row, so such a unit merges every 16 / 32 ratings: it adds its change of the row with a RED (scaled for
// the ratings the other slices have in flight, like an item row) and continues from the row as it then stands in global memory.
#pragma once
#include "lrk_common.cuh"
#include "sgd.cuh"
#include "staging_group.cuh"

struct SgdGroupParams {
    const int32_t* __restrict__ su;
    const int32_t* __restrict__ si;
    const float* __restrict__ sr;
    const int4* __restrict__ units;     // first unit of this launch
    int32_t n_units;
    unsigned int* counter;              // dynamic unit fetch (zeroed before the launch)
    float* P; float* Q; float* bu; float* bi;
    float mu, lr, reg_u, reg_i, reg_b;
    double* loss;
    int ld;
    const uint32_t* __restrict__ item_deg;   // ratings per item in this launch's shard (block-local ids); NULL: no damping
    float inflight_frac;                // resident workers / ratings of the launch: share of the stream one rating-time covers
};

#define LRK_GROUP_RING 8          // item rows a worker keeps in flight (cp.async ring in shared memory)
#define LRK_GROUP_AHEAD 8         // entries of look-ahead: the row of entry s + 8 is requested while entry s is processed

// per worker: LRK_GS user rows + LRK_GS user biases | ring of item rows | ring metadata (16 B chunk of item biases + 16 B chunk of degrees)
template <int G, int V>
__host__ __device__ constexpr int sgd_group_smem_floats_per_worker() {
    return LRK_GS * (4 * G * V) + LRK_GS + LRK_GROUP_RING * (4 * G * V) + LRK_GROUP_RING * 8;
}

template <int G>
__device__ __forceinline__ float group_sum_masked(unsigned mask, float v) {
#pragma unroll
    for (int m = G / 2; m >= 1; m >>= 1) v += __shfl_xor_sync(mask, v, m);
    return v;
}
__device__ __forceinline__ void lrk_cp_async16(void* smem_dst, const void* gmem_src) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void lrk_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void lrk_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// One worker = G lanes; the 32/G workers of a warp share its instruction stream.  The chunk loop is warp-uniform (G ratings per
// worker and iteration, everything that depends on a worker's own data predicated); taking the next unit is a divergent block of
// its own, entered by a worker whenever ITS unit is used up, so workers never wait for each other's units.  A lane only ever touches
// its own four columns of the rows in shared memory and only sub-lane 0 touches the user biases: no __syncwarp inside a unit.
//
// Latency: a worker is a sequential chain (that is the point: Gauss-Seidel inside the unit), so the item rows must be there when
// their pair starts.  The row (+ the 16 B chunks holding the item's bias and degree) of the pair that starts at entry s + 8 is
// requested with cp.async.cg (L2 -> shared memory, no register staging, L1 bypassed: the rows are RED targets of other SMs) while
// entry s is processed; one commit group per step, so `wait_group 7` at step s guarantees the row of entry s.  The next chunk's
// triples are loaded one chunk ahead.
template <int G, int V, bool BIASED>
__device__ __forceinline__ void sgd_group_segment(const SgdGroupParams& p, float* smem_cta, double& loss_d) {
    constexpr int NWW = 32 / G;                    // workers per warp
    constexpr int LDS = 4 * G * V;                 // floats per row
    constexpr int D = LRK_GROUP_AHEAD, R = LRK_GROUP_RING;
    static_assert(G >= 8 && D <= G && D <= R, "look-ahead must fit the chunk and the ring");
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int sub = lane % G;
    const int grp = lane / G;
    const unsigned wmask = G == 32 ? FULL : (((1u << (G & 31)) - 1u) << (grp * G));   // the lanes of this worker
    const int wk = (threadIdx.x >> 5) * NWW + grp;
    float* Ps = smem_cta + (size_t)wk * sgd_group_smem_floats_per_worker<G, V>();
    float* bus = Ps + LRK_GS * LDS;
    float* Rq = bus + LRK_GS;                      // ring of item rows
    float* Rm = Rq + R * LDS;                      // ring metadata: [slot][0..3] bias chunk, [slot][4..7] degree chunk
    const float lr = p.lr, reg_u = p.reg_u, reg_i = p.reg_i, reg_b = p.reg_b, mu = p.mu;

    bool alive = true, have = false;
    int64_t start = 0;
    int count = 0, first = 0, nus = 0, c = 0, slices = 1;
    bool shared = false;
    float curv = 1.f, bu0 = 0.f;
    float4 p0[V], q[V], dq[V];
    int32_t cur = -1;                              // item whose row is in q (block-local id)
    float bic = 0.f, dbi = 0.f, degc = 0.f;
    int pair_len = 0;
    unsigned issued = 0, consumed = 0;             // pair heads requested / taken (ring slots are used in this order)
    int32_t u_l = -1, i_l = -1, u_x = -1, i_x = -1;   // current / next chunk: entry `sub` of each
    float r_l = 0.f, r_x = 0.f;
#pragma unroll
    for (int v = 0; v < V; ++v) { p0[v] = make_float4(0.f, 0.f, 0.f, 0.f); q[v] = p0[v]; dq[v] = p0[v]; }

    // request the item row (and bias / degree chunks) of a pair head into the next ring slot
    auto request = [&](int32_t item) {
        const unsigned slot = issued % R;
#pragma unroll
        for (int v = 0; v < V; ++v) lrk_cp_async16(Rq + slot * LDS + (v * G + sub) * 4, p.Q + (int64_t)item * p.ld + (v * G + sub) * 4);
        if (BIASED && sub == 0) lrk_cp_async16(Rm + slot * 8, (const void*)((uintptr_t)(p.bi + item) & ~(uintptr_t)15));
        if (sub == 0 && p.item_deg) lrk_cp_async16(Rm + slot * 8 + 4, (const void*)((uintptr_t)(p.item_deg + item) & ~(uintptr_t)15));
        ++issued;
    };
    // the change of the current item row -> global memory, scaled for the ratings of that item other workers have in flight:
    // while this worker held the row for pair_len ratings (+ the look-ahead), the others applied about deg_i * (W / n) * that many
    auto flush = [&]() {
        if (cur >= 0) {
            float damp = 1.f;
            if (p.item_deg) {
                const float others = fmaxf(degc - (float)pair_len, 0.f);
                const float x = lr * curv * others * p.inflight_frac * (float)(pair_len + D);
                if (x > 1e-3f) damp = (1.f - __expf(-x)) / x;
            }
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const float4 t = make_float4(dq[v].x * damp, dq[v].y * damp, dq[v].z * damp, dq[v].w * damp);
                apply4<true>(p.Q + (int64_t)cur * p.ld + (v * G + sub) * 4, t, t);
            }
            if (BIASED && sub == 0) apply1<true>(p.bi + cur, 0.f, dbi * damp);
        }
        cur = -1; pair_len = 0;
    };
    // slice of a heavy user: its other slices run concurrently on other workers, each on a private copy of the user's row.  Merge:
    // add this slice's change since the last merge (scaled like an item row: the other slices have (slices - 1) * ratings-per-merge
    // ratings in flight) and continue from the row as it now stands in global memory
    auto merge_shared_row = [&](int since) {
        const float x = lr * curv * (float)((slices - 1) * since);
        const float damp = x > 1e-3f ? (1.f - __expf(-x)) / x : 1.f;
#pragma unroll
        for (int v = 0; v < V; ++v) {
            float* g = p.P + (int64_t)first * p.ld + (v * G + sub) * 4;
            const float4 x4 = *reinterpret_cast<const float4*>(Ps + (v * G + sub) * 4);
            const float4 t = make_float4((x4.x - p0[v].x) * damp, (x4.y - p0[v].y) * damp, (x4.z - p0[v].z) * damp, (x4.w - p0[v].w) * damp);
            apply4<true>(g, t, t);
            p0[v] = ldcg4(g);                     // same thread, same address: ordered after its own RED
            *reinterpret_cast<float4*>(Ps + (v * G + sub) * 4) = p0[v];
        }
        if (BIASED && sub == 0) {
            apply1<true>(p.bu + first, 0.f, (bus[0] - bu0) * damp);
            bu0 = __ldcg(p.bu + first);
            bus[0] = bu0;
        }
    };
    auto load_chunk = [&](int at, int32_t& u, int32_t& i, float& r) {
        u = -1; i = -1; r = 0.f;
        if (at + sub < count) {
            const int64_t e = start + at + sub;
            u = __ldcs(p.su + e) - first; i = __ldcs(p.si + e); r = __ldcs(p.sr + e);
        }
    };

    for (;;) {
        if (alive && (!have || c >= count)) {
            // ---- this worker's unit is used up: finish it, take the next one (divergent between the workers of a warp)
            if (have) {
                flush();
                if (shared) merge_shared_row(count % G == 0 ? G : count % G);
                else {
                    for (int j = 0; j < nus; ++j) {
#pragma unroll
                        for (int v = 0; v < V; ++v)
                            __stcg(reinterpret_cast<float4*>(p.P + (int64_t)(first + j) * p.ld + (v * G + sub) * 4),
                                   *reinterpret_cast<const float4*>(Ps + j * LDS + (v * G + sub) * 4));
                        if (BIASED && sub == 0) __stcg(p.bu + first + j, bus[j]);
                    }
                }
                have = false;
            }
            int unit = -1;
            if (sub == 0) unit = (int)atomicAdd(p.counter, 1u);
            unit = __shfl_sync(wmask, unit, grp * G);
            if (unit >= p.n_units) { alive = false; u_l = -1; u_x = -1; i_l = -1; i_x = -1; count = 0; }
            else {
                const int4 d = __ldg(p.units + unit);
                start = (int64_t)(uint32_t)d.x; count = d.y; first = d.z; nus = d.w & 0xffff; shared = (d.w >> 16) != 0;
                slices = shared ? (d.w >> 16) : 1;
                c = 0; have = true; cur = -1; pair_len = 0;
                load_chunk(0, u_l, i_l, r_l);
                load_chunk(G, u_x, i_x, r_x);
                // the unit's user rows -> shared memory, four rows in flight at a time
                float pn2 = 0.f;
                for (int j0 = 0; j0 < nus; j0 += 4) {
                    float4 x[4][V];
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj)
#pragma unroll
                        for (int v = 0; v < V; ++v)
                            x[jj][v] = j0 + jj < nus ? ldcg4(p.P + (int64_t)(first + j0 + jj) * p.ld + (v * G + sub) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj)
                        if (j0 + jj < nus) {
#pragma unroll
                            for (int v = 0; v < V; ++v) {
                                *reinterpret_cast<float4*>(Ps + (j0 + jj) * LDS + (v * G + sub) * 4) = x[jj][v];
                                pn2 += dot4(x[jj][v], x[jj][v]);
                                if (j0 + jj == 0) p0[v] = x[jj][v];
                            }
                        }
                }
                if (BIASED && sub == 0) for (int j = 0; j < nus; ++j) bus[j] = __ldcg(p.bu + first + j);
                pn2 = group_sum_masked<G>(wmask, pn2);
                curv = fmaxf(1.f, nus > 0 ? pn2 / (float)nus : 0.f);     // curvature of the item-side step: mean |p_u|^2 of the rows held
                bu0 = (BIASED && sub == 0 && nus > 0) ? bus[0] : 0.f;
                // prologue of the look-ahead: the pair heads among the first D entries (one commit group per entry, like a step)
                int32_t prev = -1;
#pragma unroll
                for (int t = 0; t < D; ++t) {
                    const int32_t it = __shfl_sync(wmask, i_l, grp * G + t);
                    if (it >= 0 && it != prev) request(it);
                    lrk_cp_async_commit();
                    prev = it;
                }
            }
        }
        if (!__any_sync(FULL, alive)) break;
        const bool on = alive && have;

        // ---- one chunk: G steps of one rating per worker; entry s + D (this chunk or the next) is looked ahead at step s
        float loss_f = 0.f;
        int32_t un = __shfl_sync(FULL, u_l, 0, G), in_ = __shfl_sync(FULL, i_l, 0, G);
        float rn = __shfl_sync(FULL, r_l, 0, G);
        int32_t la_prev = __shfl_sync(FULL, i_l, D - 1, G);          // item of entry D - 1 (the last one already looked at)
#pragma unroll
        for (int s = 0; s < G; ++s) {
            const int32_t uc = un, ic = in_;
            const float rc = rn;
            if (s + 1 < G) {
                un = __shfl_sync(FULL, u_l, s + 1, G); in_ = __shfl_sync(FULL, i_l, s + 1, G); rn = __shfl_sync(FULL, r_l, s + 1, G);
            }
            // look-ahead: entry s + D
            const int32_t la = (s + D < G) ? __shfl_sync(FULL, i_l, s + D, G) : __shfl_sync(FULL, i_x, s + D - G, G);
            lrk_cp_async_wait<D - 1>();
            const bool act = uc >= 0;
            if (act && ic != cur) {          // new pair: flush the old one, take the row from the ring
                flush();
                const unsigned slot = consumed % R;
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    q[v] = *reinterpret_cast<const float4*>(Rq + slot * LDS + (v * G + sub) * 4);
                    dq[v] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
                // sub-lane 0 requested the two metadata chunks, so it is the lane that may read them
                if (BIASED && sub == 0) bic = Rm[slot * 8 + (int)(((uintptr_t)(p.bi + ic) & 15) >> 2)];
                degc = (p.item_deg && sub == 0) ? (float)reinterpret_cast<const uint32_t*>(Rm)[slot * 8 + 4 + (int)(((uintptr_t)(p.item_deg + ic) & 15) >> 2)] : 0.f;
                degc = __shfl_sync(wmask, degc, grp * G);
                dbi = 0.f; cur = ic;
                ++consumed;
            }
            if (on && la >= 0 && la != la_prev) request(la);
            lrk_cp_async_commit();
            la_prev = la;
            float4 pc[V];
            float part = 0.f, buc = 0.f;
            const int urow = act ? uc : 0;
#pragma unroll
            for (int v = 0; v < V; ++v) {
                pc[v] = act ? *reinterpret_cast<const float4*>(Ps + urow * LDS + (v * G + sub) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                part += dot4(pc[v], q[v]);
            }
            if (BIASED && sub == 0 && act) { buc = bus[urow]; part += buc + bic + mu; }
            const float pred = group_sum<G>(part);
            const float err = rc - pred;
            if (act) {
                float reg_acc = 0.f;
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const float4 a = pc[v], b = q[v];
                    float4 np, dqs;
                    np.x = a.x + lr * (err * b.x - reg_u * a.x); dqs.x = lr * (err * a.x - reg_i * b.x);
                    np.y = a.y + lr * (err * b.y - reg_u * a.y); dqs.y = lr * (err * a.y - reg_i * b.y);
                    np.z = a.z + lr * (err * b.z - reg_u * a.z); dqs.z = lr * (err * a.z - reg_i * b.z);
                    np.w = a.w + lr * (err * b.w - reg_u * a.w); dqs.w = lr * (err * a.w - reg_i * b.w);
                    *reinterpret_cast<float4*>(Ps + urow * LDS + (v * G + sub) * 4) = np;
                    q[v].x += dqs.x; q[v].y += dqs.y; q[v].z += dqs.z; q[v].w += dqs.w;
                    dq[v].x += dqs.x; dq[v].y += dqs.y; dq[v].z += dqs.z; dq[v].w += dqs.w;
                    reg_acc += reg_u * dot4(a, a) + reg_i * dot4(b, b);
                }
                if (sub == 0) {
                    reg_acc += err * err;
                    if (BIASED) {
                        bus[urow] = buc + lr * (err - reg_b * buc);
                        const float dbs = lr * (err - reg_b * bic);
                        reg_acc += reg_b * (buc * buc + bic * bic);
                        bic += dbs; dbi += dbs;
                    }
                }
                loss_f += reg_acc;
                ++pair_len;
            }
        }
        loss_d += (double)loss_f;
        c += G;
        u_l = u_x; i_l = i_x; r_l = r_x;
        if (on) load_chunk(c + G, u_x, i_x, r_x);
        if (on && shared && c < count) merge_shared_row(G);
    }
    lrk_cp_async_wait<0>();
}

template <int G, int V, bool BIASED>
__global__ void __launch_bounds__(256, 2) sgd_group_epoch_kernel(SgdGroupParams p) {
    extern __shared__ float4 lrk_group_smem4[];
    double loss_d = 0.0;
    sgd_group_segment<G, V, BIASED>(p, reinterpret_cast<float*>(lrk_group_smem4), loss_d);
    block_loss_commit(loss_d, p.loss);
}

template <int G, int V>
static size_t sgd_group_smem_bytes() { return sizeof(float) * (size_t)(8 * (32 / G)) * sgd_group_smem_floats_per_worker<G, V>(); }

static bool sgd_group_layout_supported(const lrk_handle_s* h) { return h->V == 1 && (h->G == 8 || h->G == 16 || h->G == 32); }
// f(G, V) for the layouts the user-group kernels are built for (sgd_group_layout_supported)
template <class F>
static int sgd_with_group_layout(lrk_handle_s* h, F&& f) {
    return lrk_with_layout(h, [&](auto G, auto V) -> int {
        if constexpr (decltype(G)::value >= 8 && decltype(V)::value == 1) return f(G, V);
        else return lrk_fail(h, LRK_ERR_INVALID, "sgd_with_group_layout", "unsupported factor layout", __FILE__, __LINE__);
    });
}

// CTAs of the group kernel resident at once (sets the unit size at staging and bounds the grid at launch)
template <int G, int V>
static int sgd_group_ctas(lrk_handle_s* h) {
    const size_t smem = sgd_group_smem_bytes<G, V>();
    cudaFuncSetAttribute(sgd_group_epoch_kernel<G, V, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaFuncSetAttribute(sgd_group_epoch_kernel<G, V, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sgd_group_epoch_kernel<G, V, true>, 256, smem) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        per_sm = 1;
    }
    return per_sm * h->sm_count;
}
static int sgd_group_resident_workers(lrk_handle_s* h) {
    return sgd_with_group_layout(h, [&](auto G, auto V) { return sgd_group_ctas<decltype(G)::value, decltype(V)::value>(h) * 8 * (32 / decltype(G)::value); });
}
// Selected with LRK_SGD_GROUP=1 (read at lrk_create).  r02 measurement on one B200 (ML-20M shape, BiasedMF k=64): this
// kernel is bit-for-bit the closer one to the reference (held-out RMSE within 1.3e-5 of the sequential oracle, first-epoch loss of
// config C4 92.9 M vs the oracle's 94.6 M against 134 M for the item-run-tile kernel), but it is INSTRUCTION bound, not L2 bound:
// 140 warp-instructions per rating (ncu, profiles/r02_group_kernel_ncu_summary.md) against 53 for the item-run-tile kernel -- the
// sequential chain needs per-rating control flow (pair heads, look-ahead, ring slots) and the two workers of a warp diverge on it --
// 4.0-4.8 ms per epoch against 1.5 ms.  So the item-run-tile kernel stays the default and this one is the order-faithful option.
static bool lrk_use_group_kernel(const lrk_handle_s* h) { return h->sgd_group && sgd_group_layout_supported(h); }

// The group kernel's parameters for item block b (0 on one GPU): those of the block's stream segment (sgd_segment), with the
// block's units in place of its ratings (unit starts index the whole stream).  A block without ratings gets no units.
static SgdGroupParams sgd_group_params(const lrk_handle_s* h, const SgdParams& seg, int b) {
    const GroupUnits* gu = h->group.get();
    SgdGroupParams gp;
    memset(&gp, 0, sizeof gp);
    gp.su = h->d_su; gp.si = h->d_si; gp.sr = h->d_sr;
    gp.units = gu->d_units + gu->unit_base[(size_t)b];
    gp.n_units = seg.n > 0 ? (int32_t)(gu->unit_base[(size_t)b + 1] - gu->unit_base[(size_t)b]) : 0;
    gp.counter = gu->d_counter + b;
    gp.P = seg.P; gp.Q = seg.Q; gp.bu = seg.bu; gp.bi = seg.bi;
    gp.mu = seg.mu; gp.lr = seg.lr; gp.reg_u = seg.reg_u; gp.reg_i = seg.reg_i; gp.reg_b = seg.reg_b;
    gp.loss = seg.loss; gp.ld = seg.ld; gp.item_deg = seg.item_deg;
    return gp;
}

// Grid of one group-kernel launch over the blocks gseg[0..nseg) (one, or the strata of a fused DSGD epoch; seg: their stream
// segments): at most `ctas`, no more CTAs than the block with the most units can keep busy, divided by the rollback safeguard.
// Per block the workers in flight are min(grid * WPC, units) and inflight_frac = those workers / the block's ratings.
static int sgd_group_grid(lrk_handle_s* h, int64_t ctas, int wpc, const SgdParams* seg, SgdGroupParams* gseg, int nseg) {
    int64_t most = 1;
    for (int t = 0; t < nseg; ++t) most = std::max<int64_t>(most, (gseg[t].n_units + wpc - 1) / wpc);
    int64_t grid = std::min(ctas, most);
    if (h->conc_div > 1) grid /= h->conc_div;
    if (grid < 1) grid = 1;
    for (int t = 0; t < nseg; ++t) {
        const double workers = (double)std::min<int64_t>(grid * wpc, gseg[t].n_units);
        gseg[t].inflight_frac = (float)(workers / (double)std::max<int64_t>(seg[t].n, 1));
        sgd_trace(h, seg[t], false, (int)grid, gseg[t].inflight_frac);
    }
    return (int)grid;
}

template <int G, int V>
static int sgd_group_launch_gv(lrk_handle_s* h, const SgdParams& seg, int b) {
    SgdGroupParams gp = sgd_group_params(h, seg, b);
    const int grid = sgd_group_grid(h, sgd_group_ctas<G, V>(h), 8 * (32 / G), &seg, &gp, 1);
    const size_t smem = sgd_group_smem_bytes<G, V>();
    if (h->cfg.model == LRK_MODEL_BIASEDMF) sgd_group_epoch_kernel<G, V, true><<<(unsigned)grid, 256, smem, h->stream>>>(gp);
    else sgd_group_epoch_kernel<G, V, false><<<(unsigned)grid, 256, smem, h->stream>>>(gp);
    LRK_LAUNCH_CHECK(h);
    return LRK_OK;
}
// the epoch (one GPU) or one sub-epoch (DSGD) of item block b over the stream segment seg of that block
static int sgd_group_launch(lrk_handle_s* h, const SgdParams& seg, int b) {
    return sgd_with_group_layout(h, [&](auto G, auto V) { return sgd_group_launch_gv<decltype(G)::value, decltype(V)::value>(h, seg, b); });
}
