// Tensor-core top-N (sm_100a): recommendRank()'s user x item score sweep
// (recommender/MatrixRecommender.java:153-201) as a tcgen05 / TMA fp16 GEMM with the selection fused
// into the epilogue, followed by an exact fp64 re-score -- so the lists that leave the library are
// still bit-identical to the reference (util/Lists.java:416-468 semantics).
//
//   1. operands: A = queried user factors, B = item factors, both K-major fp16 after an exact power-of-two
//      scaling (per user row / per item matrix), K padded to 64; BiasedMF folds the item bias into two extra
//      K columns (hi/lo fp16 split against the row's scale in A).
//   2. topn_tc_kernel (persistent, warp-specialised, 1 CTA/SM, 320 threads):
//        warp 0  TMA producer   item tiles, cp.async.bulk.tensor.2d, SWIZZLE_128B, mbarrier ring (3 stages at k=128)
//        warp 1  MMA issuer     tcgen05.mma.cta_group::1.kind::f16 with the A operand in TENSOR MEMORY (.ts form),
//                               M=128 N=128 K=16; two user sub-tiles (256 users) share every item tile; the loop is
//                               warp-uniform with elect.sync around the issue (8 back-to-back UTCHMMA per sub-tile);
//                               accumulators in a ring of three 128-column TMEM slots
//        warps 2-9 epilogue     stage their user rows into TMEM (tcgen05.st), then per tile tcgen05.ld 32x32b.x32:
//                               one thread owns one user row; a score is appended to the row's candidate list
//                               (shared memory, 64 slots) only if it beats the row's running threshold tau --
//                               common case 15 FMNMX3/FMNMX + 1 compare + 1 warp vote per 32 scores; full lists are
//                               compacted warp-cooperatively to the best K' (train items masked there, tau rises).
//      Invariant: every item that is NOT in a row's candidate list has sweep score <= tau_row
//      (or is a train item / NaN / out of range).
//   3. topn_tc_rescore_kernel: exact fp64 scores of the candidates in Java's summation order, top-N,
//      and an exactness certificate: N-th exact score > tau + error bound of the fp16 sweep, and no
//      exact ties among the first N+1.  Rows whose margin is too thin are swept a second time from the
//      threshold their first result implies (K' = 32); what still fails (exact ties, fewer than N
//      candidates) is re-done by the exact kernel (topn_exact.cuh).
#pragma once
#include "lrk_common.cuh"
#include "topn_exact.cuh"
#include <cuda.h>
#include <cuda_fp16.h>
#include <cudaTypedefs.h>
#include <cmath>
#include <cstdlib>
#include <algorithm>

#define TC_TILE_M 128          // users per accumulator
#define TC_UT 2                // user sub-tiles per CTA
#define TC_TILE_N 128          // items per MMA tile
#define TC_KB 64               // bf16 elements per 128-byte swizzle row
#define TC_KEEP_MAX 32         // largest K' (candidates a compaction keeps per (row, chunk))
#define TC_MAX_TOPN 26         // the first pass keeps K' = max(16, N + 6) <= TC_KEEP_MAX candidates: N up to 26 (r01: 16)
#define TC_CAP 64              // candidate slots per (row, chunk) in global memory (append buffer, compacted to K')
#define TC_ROWS (TC_TILE_M * TC_UT)   // user rows per CTA
#define TC_THREADS 320
#define TC_MAX_CHUNKS 16

struct TcState {
    LrkBuf<__half> Bq;                // [I x Kp] item operand: fp16(2^eQ * q), BiasedMF: + {hi, lo} split of 2^eQ * b_i
    int Kp = 0;
    bool valid = false;
    bool finite = true;               // false: some item factor / bias is NaN or Inf -> exact path only
    int eQ = 0;                       // power-of-two scale of the item operand
    double qnorm_max = 0.0, bi_max = 0.0, qabs_max = 0.0;
    LrkBuf<unsigned long long> d_stats;      // [0] max ||q||^2 bits, [1] max |bi| bits, [2] max |q_f| bits, [3] max err/bound (float bits)
    PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
    LrkBuf<char> work;                       // per-pass scratch (user operand, candidate lists, ...)
    LrkBuf<char> lists;                      // per-call lists of rows without a certificate
    LrkBuf<int32_t> fail_items, fail_counts; // exact results of the rows without a certificate
    LrkBuf<double> fail_scores;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // phase boundaries of the last call
    ~TcState() { for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e); }
};

static inline TcState* tc_state(lrk_handle_s* h) {
    if (!h->tc) h->tc.reset(new TcState());
    return h->tc.get();
}
static inline void topn_tc_invalidate(lrk_handle_s* h) {
    if (h->tc) h->tc->valid = false;
}
static inline int tc_kp(lrk_handle_s* h) {
    const int kaug = h->k + (lrk_has_bias(h) ? 2 : 0);
    return ((kaug + TC_KB - 1) / TC_KB) * TC_KB;
}
static inline bool topn_tc_profitable(lrk_handle_s* h, int32_t nq, int topn) {
    return topn <= TC_MAX_TOPN && tc_kp(h) <= 128 && h->I >= 8192 && nq >= 512;
}

// ------------------------------------------------------------------------------------------------
// operand builders.  Operands are fp16 (11 significant bits; the products are exact in the fp32 accumulator)
// after an exact power-of-two scaling that puts the largest magnitude of the item matrix / of each user
// row into [2^9, 2^10): |fp16(s x) - s x| <= max(2^-11 |s x|, 2^-25).
// ------------------------------------------------------------------------------------------------
#define TC_EXP_TARGET 9
__host__ __device__ inline int tc_scale_exp(double maxabs, int lo, int hi) {
    if (!(maxabs > 0.0) || !(maxabs < 1e300)) return 0;
    int e;
    frexp(maxabs, &e);                       // maxabs = m * 2^e, m in [0.5, 1)
    const int s = TC_EXP_TARGET + 1 - e;     // maxabs * 2^s in [2^9, 2^10)
    return s < lo ? lo : (s > hi ? hi : s);
}
// user rows: 2^e must itself be an fp16 number (BiasedMF keeps it in the two bias columns)
#define TC_USER_EXP_LO (-24)
#define TC_USER_EXP_HI 14

__global__ void tc_item_stats_kernel(const double* __restrict__ Q, const double* __restrict__ bi, int biased, int k, int32_t I,
                                     unsigned long long* __restrict__ stats) {
    const int32_t i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= I) return;
    double n2 = 0.0, ma = 0.0;
    bool bad = false;
    for (int f = lane; f < k; f += 32) { const double q = Q[(int64_t)i * k + f]; n2 += q * q; ma = fmax(ma, fabs(q)); bad |= !(fabs(q) <= 1.7e308); }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) { n2 += __shfl_xor_sync(0xffffffffu, n2, m); ma = fmax(ma, __shfl_xor_sync(0xffffffffu, ma, m)); }
    bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) {
        if (bad) n2 = INFINITY;                                    // NaN / Inf anywhere -> the host disables the fp16 path
        atomicMax(stats, (unsigned long long)__double_as_longlong(n2));
        atomicMax(stats + 2, (unsigned long long)__double_as_longlong(ma));
        if (biased) { const double b = fabs(bi[i]); atomicMax(stats + 1, (unsigned long long)__double_as_longlong(b <= 1.7e308 ? b : INFINITY)); }
    }
}
__global__ void tc_build_items_kernel(const double* __restrict__ Q, const double* __restrict__ bi, int biased, int k, int Kp,
                                      int32_t I, int eQ, __half* __restrict__ out) {
    const int32_t i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= I) return;
    for (int f = lane; f < Kp; f += 32) {
        double v = 0.0;
        if (f < k) v = ldexp(Q[(int64_t)i * k + f], eQ);
        else if (biased && f == k) v = ldexp(bi[i], eQ);
        else if (biased && f == k + 1) { const double b = ldexp(bi[i], eQ); v = b - (double)__half2float(__double2half(b)); }
        out[(int64_t)i * Kp + f] = __double2half(v);
    }
}
// pstat[c] = {||p_u||_2, max_f |p_uf|}
__global__ void tc_build_users_kernel(const double* __restrict__ P, int biased, int k, int Kp, const int32_t* __restrict__ users,
                                      int32_t nq, __half* __restrict__ out, double2* __restrict__ pstat) {
    const int32_t c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= nq) return;
    const int32_t u = users ? users[c] : c;
    double n2 = 0.0, ma = 0.0;
    for (int f = lane; f < k; f += 32) { const double p = P[(int64_t)u * k + f]; n2 += p * p; ma = fmax(ma, fabs(p)); }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) { n2 += __shfl_xor_sync(0xffffffffu, n2, m); ma = fmax(ma, __shfl_xor_sync(0xffffffffu, ma, m)); }
    const int e = tc_scale_exp(ma, TC_USER_EXP_LO, TC_USER_EXP_HI);
    for (int f = lane; f < Kp; f += 32) {
        double v = 0.0;
        if (f < k) v = ldexp(P[(int64_t)u * k + f], e);
        else if (biased && (f == k || f == k + 1)) v = ldexp(1.0, e);
        out[(int64_t)c * Kp + f] = __double2half(v);
    }
    if (lane == 0) pstat[c] = make_double2(sqrt(n2), ma);
}

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ bool tc_elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// K-major, SWIZZLE_128B operand tile: rows of 128 bytes, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t addr) {
    uint64_t d = 0;
    d |= (uint64_t)((addr & 0x3FFFFu) >> 4);      // start address, 16-byte units
    d |= (uint64_t)1 << 16;                       // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;             // stride byte offset
    d |= (uint64_t)1 << 46;                       // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                       // SWIZZLE_128B
    return d;
}
// kind::f16 instruction descriptor: D=f32 (bit 4), A=B=f16 (format fields 0), K-major both, N=128, M=128
#define TC_IDESC ((1u << 4) | ((uint32_t)(TC_TILE_N >> 3) << 17) | ((uint32_t)(TC_TILE_M >> 4) << 24))

struct TcParams {
    int32_t nq, I;
    int n_chunks, tiles_per_chunk, total_tiles, num_kb, stages;
    int exclude_train;
    int keep;               // K': candidates a compaction keeps per (row, chunk), <= TC_KEEP_MAX
    int debug;              // LRK_TC_DEBUG (profiling probes only): bit0 = drain TMEM but skip the selection, bit1 = do not even read TMEM, bit2 = issue no MMA
    const int64_t* __restrict__ rowptr;
    const int32_t* __restrict__ col;
    const int32_t* __restrict__ users;
    const float* init_tau;  // per query slot: threshold the row starts from (second pass), or NULL = -inf
    uint2* cand;            // [nq_pad][n_chunks][TC_CAP] {approximate score bits, item}
    int32_t* cand_cnt;      // [nq_pad][n_chunks]
    float* cand_tau;
};

__device__ __forceinline__ float tc_max3(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));      // FMNMX3
    return r;
}
template <typename T>
__device__ __forceinline__ T* tc_shfl_ptr(T* ptr, int src) {
    const unsigned long long v = (unsigned long long)ptr;
    const uint32_t lo = __shfl_sync(0xffffffffu, (uint32_t)v, src), hi = __shfl_sync(0xffffffffu, (uint32_t)(v >> 32), src);
    return (T*)(((unsigned long long)hi << 32) | lo);
}

// Warp-cooperative compaction of the candidate lists of every row (lane) whose list holds more than `trig`
// entries.  A list is {entries [0,kept): survivors of earlier compactions, train items already removed;
// entries [kept,cnt): appended since, in ascending item order}.  One row at a time, all 32 lanes:
//   1. load the <= TC_CAP entries (two per lane);
//   2. drop train items among the new entries (MatrixRecommender.java:170-174): the sorted CSR row is walked
//      32 items per load from a per-row cursor, membership by a 5-step binary search across lanes;
//   3. rank by (score desc, slot asc), keep the best K', tau := score of rank K'-1.
// Everything dropped here has approximate score <= the new tau (or is a train item), which is the invariant the
// exactness certificate of topn_tc_rescore_kernel rests on.
// Candidate lists live in shared memory: TC_ROWS rows x TC_CAP slots of {score bits, item}; entry e of row r sits in
// slot (e & 32) | ((e ^ r) & 31) of the row's 512-byte line, which keeps both access patterns conflict-free: the lanes
// of a warp (32 consecutive rows) appending at equal counts, and the 32 lanes of a compaction reading one row.
__device__ __forceinline__ uint32_t tc_slot(uint32_t row_base, int sw, int e) { return row_base + (uint32_t)(((e & 32) | ((e ^ sw) & 31)) << 3); }
__device__ __forceinline__ void tc_sts2(uint32_t addr, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ uint2 tc_lds2(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __noinline__ int4 tc_compact(uint32_t lp, int sw, int cnt, int kept, float tau, const int32_t* col_row, int tlen, int tp, int32_t nt,
                                        int trig, int keep, int32_t n_items) {
    const int lane = threadIdx.x & 31;
    unsigned flagged = __ballot_sync(0xffffffffu, cnt > trig);
    while (flagged) {
        const int r = __ffs(flagged) - 1;
        flagged &= flagged - 1;
        const uint32_t L = __shfl_sync(0xffffffffu, lp, r);
        const int rsw = __shfl_sync(0xffffffffu, sw, r);
        const int32_t* cr = tc_shfl_ptr(col_row, r);
        const int n = __shfl_sync(0xffffffffu, cnt, r), kp = __shfl_sync(0xffffffffu, kept, r);
        const int tl = __shfl_sync(0xffffffffu, tlen, r);
        int cur = __shfl_sync(0xffffffffu, tp, r);
        float new_tau = __shfl_sync(0xffffffffu, tau, r);
        const int32_t nt_r = __shfl_sync(0xffffffffu, nt, r);          // next train item at / after the row's cursor
        __syncwarp();
        bool al0 = lane < n, al1 = lane + 32 < n;
        uint2 e0 = make_uint2(0u, 0u), e1 = make_uint2(0u, 0u);
        if (al0) e0 = tc_lds2(tc_slot(L, rsw, lane));
        if (al1) e1 = tc_lds2(tc_slot(L, rsw, lane + 32));
        // columns past the catalogue end (zero-filled by TMA) are appended unchecked by the sweep; drop them here
        if ((int32_t)e0.y >= n_items) al0 = false;
        if ((int32_t)e1.y >= n_items) al1 = false;
        if (tl > cur && n > kp) {
            // item range of the new entries (ascending by construction); nothing to mask if the next train item lies beyond
            const int32_t lo_a = (int32_t)__shfl_sync(0xffffffffu, e0.y, kp & 31), lo_b = (int32_t)__shfl_sync(0xffffffffu, e1.y, kp & 31);
            const int32_t hi_a = (int32_t)__shfl_sync(0xffffffffu, e0.y, (n - 1) & 31), hi_b = (int32_t)__shfl_sync(0xffffffffu, e1.y, (n - 1) & 31);
            const int32_t i_lo = kp < 32 ? lo_a : lo_b, i_hi = (n - 1) < 32 ? hi_a : hi_b;
            if (nt_r <= i_hi) for (;;) {
                const int32_t tv = (cur + lane < tl) ? __ldg(cr + cur + lane) : 0x7fffffff;
                const int32_t last = __shfl_sync(0xffffffffu, tv, 31);
                if (last < i_lo) { cur += 32; continue; }
                int p0 = 0, p1 = 0;
#pragma unroll
                for (int s = 16; s >= 1; s >>= 1) {
                    const int32_t v0 = __shfl_sync(0xffffffffu, tv, p0 + s - 1), v1 = __shfl_sync(0xffffffffu, tv, p1 + s - 1);
                    if (v0 < (int32_t)e0.y) p0 += s;
                    if (v1 < (int32_t)e1.y) p1 += s;
                }
                const int32_t m0 = __shfl_sync(0xffffffffu, tv, p0), m1 = __shfl_sync(0xffffffffu, tv, p1);
                if (lane >= kp && m0 == (int32_t)e0.y) al0 = false;
                if (lane + 32 >= kp && m1 == (int32_t)e1.y) al1 = false;
                if (last >= i_hi) { cur += __popc(__ballot_sync(0xffffffffu, tv <= i_hi)); break; }
                cur += 32;
            }
        }
        const float s0 = al0 ? __uint_as_float(e0.x) : -INFINITY, s1 = al1 ? __uint_as_float(e1.x) : -INFINITY;
        int rk0 = 0, rk1 = 0;
#pragma unroll 4
        for (int j = 0; j < 32; ++j) {
            const float a = __shfl_sync(0xffffffffu, s0, j), b = __shfl_sync(0xffffffffu, s1, j);
            rk0 += (a > s0 || (a == s0 && j < lane)) ? 1 : 0;
            rk0 += (b > s0) ? 1 : 0;
            rk1 += (a >= s1) ? 1 : 0;
            rk1 += (b > s1 || (b == s1 && j < lane)) ? 1 : 0;
        }
        const int alive = __popc(__ballot_sync(0xffffffffu, al0)) + __popc(__ballot_sync(0xffffffffu, al1));
        const int keep_n = min(alive, keep);
        __syncwarp();
        if (al0 && rk0 < keep_n) tc_sts2(tc_slot(L, rsw, rk0), e0.x, e0.y);
        if (al1 && rk1 < keep_n) tc_sts2(tc_slot(L, rsw, rk1), e1.x, e1.y);
        if (alive >= keep) {
            const unsigned b0 = __ballot_sync(0xffffffffu, al0 && rk0 == keep - 1);
            const unsigned b1 = __ballot_sync(0xffffffffu, al1 && rk1 == keep - 1);
            const float t0 = __shfl_sync(0xffffffffu, s0, b0 ? __ffs(b0) - 1 : 0), t1 = __shfl_sync(0xffffffffu, s1, b1 ? __ffs(b1) - 1 : 0);
            new_tau = b0 ? t0 : t1;
        }
        if (lane == r) { cnt = keep_n; kept = keep_n; tau = new_tau; tp = cur; }
        __syncwarp();
    }
    return make_int4(cnt, kept, __float_as_int(tau), tp);
}
#define TC_COMPACT(TRIG)                                                                  \
    do {                                                                                  \
        const int4 r_ = tc_compact(lp, sw, cnt, kept, tau, col_row, tlen, tp, nt, (TRIG), p.keep, p.I); \
        cnt = r_.x; kept = r_.y; tau = __int_as_float(r_.z);                              \
        if (r_.w != tp) { tp = r_.w; nt = tp < tlen ? __ldg(col_row + tp) : 0x7fffffff; }  \
    } while (0)

// raw TMEM load of 32 accumulator columns of this thread's row (no wait)
__device__ __forceinline__ void tc_ld32_nowait(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tc_st32(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
          "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
          "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
          "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: the user operand is read from tensor memory, so shared-memory operand
// bandwidth is spent on the item tile alone (an M=128 N=128 SS-mode MMA measured 113 cycles instead of 64)
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// Stages one thread's operand row (fp16 pairs, Kp/2 words) into its TMEM lane once the MMAs of the previous unit
// have retired, then tells the MMA warp (one arrival per warp).
__device__ __noinline__ void tc_stage_user_row(const __half* row, int num_kb, uint32_t taddr, uint32_t bar_free, uint32_t parity,
                                               uint32_t bar_ready) {
    const uint4* src = reinterpret_cast<const uint4*>(row);
    mbar_wait(bar_free, parity);
    tc_fence_after();
    for (int kb = 0; kb < num_kb; ++kb) {
        uint32_t w[32];
#pragma unroll
        for (int v = 0; v < 8; ++v) {
            const uint4 x = __ldg(src + kb * 8 + v);
            w[v * 4] = x.x; w[v * 4 + 1] = x.y; w[v * 4 + 2] = x.z; w[v * 4 + 3] = x.w;
        }
        tc_st32(taddr + (uint32_t)(kb * 32), w);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    tc_fence_before();
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(bar_ready);
}

// barrier map (S = B stages): [0,S) b_full, [S,2S) b_empty, 2S a_full (8 epilogue warps), 2S+1 a_empty,
// 2S+2+slot acc_full, 2S+5+slot acc_empty (4 epilogue warps).
// TMEM: columns [0,128) user operand (sub-tile a at a*64: fp16 pairs, row == lane), then a ring of three
// 128-column accumulator slots; accumulator n = 2*tile + sub-tile lives in slot n % 3.
#define TC_NBARS(S) (2 * (S) + 8)
#define TC_ACC_BASE 128
#define TC_ACC_SLOTS 3

__global__ void __launch_bounds__(TC_THREADS, 1)
topn_tc_kernel(const __grid_constant__ CUtensorMap tmB, const __half* __restrict__ Aq, TcParams p) {
    extern __shared__ __align__(1024) unsigned char tc_smem_raw[];
    // carve: 1024-aligned item tiles, then barriers
    unsigned char* base = (unsigned char*)(((uintptr_t)tc_smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t tile_bytes = TC_TILE_N * TC_KB * 2;               // 16 KB: 128 rows x 128 B
    unsigned char* smB = base;                                       // [stages][num_kb] tiles
    unsigned char* lists = smB + (size_t)p.stages * p.num_kb * tile_bytes;            // [TC_ROWS][TC_CAP] {score bits, item}
    uint64_t* bars = (uint64_t*)(lists + (size_t)TC_ROWS * TC_CAP * 8);
    const int S = p.stages;
    uint32_t* tmem_slot = (uint32_t*)(bars + TC_NBARS(S));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    auto BAR = [&](int i) { return smem_u32(bars + i); };

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) { mbar_init(BAR(s), 1); mbar_init(BAR(S + s), 1); }
        mbar_init(BAR(2 * S), 8); mbar_init(BAR(2 * S + 1), 1);
        for (int s = 0; s < TC_ACC_SLOTS; ++s) { mbar_init(BAR(2 * S + 2 + s), 1); mbar_init(BAR(2 * S + 5 + s), 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int m_tiles = (p.nq + TC_ROWS - 1) / TC_ROWS;
    const int num_units = m_tiles * p.n_chunks;

    // The producer and the MMA issuer run their loops warp-uniformly (all 32 lanes wait on the barriers) and
    // elect one lane only around the asynchronous instructions: inside a lane-divergent branch the compiler wraps
    // every UTCHMMA in an election loop, and the issue rate of that single thread capped the tensor pipe.
    if (warp == 0) {
        // ================= TMA producer (item tiles) =================
        int st = 0; uint32_t ph = 0;
        for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
            const int ch = unit % p.n_chunks;
            const int t0 = ch * p.tiles_per_chunk;
            const int t1 = min(p.total_tiles, t0 + p.tiles_per_chunk);
            for (int t = t0; t < t1; ++t) {
                mbar_wait(BAR(S + st), ph ^ 1);                            // B slot free
                if (tc_elect_one()) {
                    mbar_expect_tx(BAR(st), p.num_kb * tile_bytes);
                    for (int kb = 0; kb < p.num_kb; ++kb)
                        tma_load_2d(smem_u32(smB + (size_t)(st * p.num_kb + kb) * tile_bytes), &tmB, kb * TC_KB, t * TC_TILE_N, BAR(st));
                }
                __syncwarp();
                if (++st == S) { st = 0; ph ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        int st = 0; uint32_t ph = 0, a_ph = 0; int slot = 0; uint32_t slot_ph = 0;
        const uint64_t desc0 = tc_smem_desc(smem_u32(smB));
        const uint32_t stage_units = (uint32_t)(p.num_kb * tile_bytes) >> 4;   // descriptor address units (16 B) per B stage
        const int nkb = (p.debug & 4) ? 0 : p.num_kb;
        for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
            const int ch = unit % p.n_chunks;
            mbar_wait(BAR(2 * S), a_ph);                                   // user operand of this unit is in TMEM
            a_ph ^= 1;
            tc_fence_after();
            const int t0 = ch * p.tiles_per_chunk;
            const int t1 = min(p.total_tiles, t0 + p.tiles_per_chunk);
            for (int t = t0; t < t1; ++t) {
                mbar_wait(BAR(st), ph);                                    // B landed
                const uint64_t bdesc = desc0 + (uint64_t)((uint32_t)st * stage_units);
#pragma unroll
                for (int a = 0; a < TC_UT; ++a) {
                    mbar_wait(BAR(2 * S + 5 + slot), slot_ph ^ 1);         // accumulator slot drained by its 4 epilogue warps
                    tc_fence_after();
                    if (tc_elect_one()) {
                        const uint32_t d = tmem_base + (uint32_t)(TC_ACC_BASE + slot * TC_TILE_N);
                        const uint32_t at = tmem_base + (uint32_t)(a * 64);
#pragma unroll
                        for (int kb = 0; kb < 2; ++kb) {
                            if (kb < nkb) {
#pragma unroll
                                for (int k4 = 0; k4 < TC_KB / 16; ++k4)
                                    tc_mma_f16_ts(d, at + (uint32_t)(kb * 32 + k4 * 8), bdesc + (uint64_t)(kb * (tile_bytes >> 4) + k4 * 2),
                                                  TC_IDESC, (kb | k4) != 0 ? 1u : 0u);
                            }
                        }
                        tc_commit(BAR(2 * S + 2 + slot));                  // this sub-tile's scores are ready
                        if (a == TC_UT - 1) tc_commit(BAR(S + st));        // B slot reusable once these MMAs retire
                    }
                    __syncwarp();
                    if (++slot == TC_ACC_SLOTS) { slot = 0; slot_ph ^= 1; }
                }
                if (++st == S) { st = 0; ph ^= 1; }
            }
            if (tc_elect_one()) tc_commit(BAR(2 * S + 1));                 // user operand may be overwritten
            __syncwarp();
        }
    } else {
        // ================= epilogue: one thread == one user row =================
        const int ew = warp - 2;
        const int a = ew >> 2;                 // user sub-tile
        const int q = warp & 3;                // TMEM lane quarter this warp may access
        const int row_in_cta = a * TC_TILE_M + q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        // accumulator sequence of this sub-tile: n = a, a+2, a+4, ... ; slot = n % 3, parity = (n / 3) & 1
        int slot = a; uint32_t slot_ph = 0;
        uint32_t a_ph = 0;
        auto stage_user_rows = [&](int unit) {
            const int mt = unit / p.n_chunks;
            tc_stage_user_row(Aq + ((size_t)mt * TC_ROWS + row_in_cta) * (size_t)(p.num_kb * TC_KB), p.num_kb,
                              tlane + (uint32_t)(a * 64), BAR(2 * S + 1), a_ph ^ 1, BAR(2 * S));
            a_ph ^= 1;
        };
        if ((int)blockIdx.x < num_units) stage_user_rows(blockIdx.x);
        for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
            const int mt = unit / p.n_chunks, ch = unit - mt * p.n_chunks;
            const int32_t c = mt * TC_ROWS + row_in_cta;
            const bool valid = c < p.nq;
            const int t0 = ch * p.tiles_per_chunk;
            const int t1 = min(p.total_tiles, t0 + p.tiles_per_chunk);
            const uint32_t lp = smem_u32(lists) + (uint32_t)row_in_cta * (TC_CAP * 8);     // this row's candidate list (shared memory)
            const int sw = row_in_cta & 31;
            const int32_t* col_row = p.col;
            int tlen = 0, tp = 0;
            int32_t nt = 0x7fffffff;               // next train item at / after the cursor (lets a compaction skip the mask)
            if (valid && p.exclude_train) {
                const int32_t u = p.users ? p.users[c] : c;
                const int64_t rb = p.rowptr[u], re = p.rowptr[u + 1];
                col_row = p.col + rb; tlen = (int)(re - rb);
                const int32_t i0 = t0 * TC_TILE_N;
                int lo = 0, hi_ = tlen;
                while (lo < hi_) { const int m = (lo + hi_) >> 1; if (__ldg(col_row + m) < i0) lo = m + 1; else hi_ = m; }
                tp = lo;
                nt = tp < tlen ? __ldg(col_row + tp) : 0x7fffffff;
            }
            // Rows past nq carry tau = +inf so that nothing ever passes.  Common path per 32-column slab: 15
            // FMNMX3/FMNMX, one compare and one warp vote, no divergence.  A slab is looked into only if SOME lane of
            // the warp has a score above its row's threshold there: by groups of 8, then 4 columns, 4 predicated appends.
            // The two 64-column halves of a tile run through ONE copy of this code (rolled loop): the tile loop has to
            // stay well inside the instruction cache (at ~36 KB it stalled 3.6 cycles per issue on instruction fetch).
            float tau = valid ? (p.init_tau ? p.init_tau[c] : -INFINITY) : INFINITY;
            int cnt = 0, kept = 0;
#define TC_APPEND(R, J)                                                                                            \
            do {                                                                                                   \
                if (__uint_as_float(R[J]) > tau) {                                                                 \
                    tc_sts2(tc_slot(lp, sw, cnt), R[J], (uint32_t)(item0 + (J)));                                  \
                    ++cnt;                                                                                         \
                }                                                                                                  \
            } while (0)
#define TC_MAX8(R, O) tc_max3(tc_max3(__uint_as_float(R[O]), __uint_as_float(R[O + 1]), __uint_as_float(R[O + 2])),     \
                              tc_max3(__uint_as_float(R[O + 3]), __uint_as_float(R[O + 4]), __uint_as_float(R[O + 5])), \
                              fmaxf(__uint_as_float(R[O + 6]), __uint_as_float(R[O + 7])))
#define TC_MAX4(R, O) fmaxf(tc_max3(__uint_as_float(R[O]), __uint_as_float(R[O + 1]), __uint_as_float(R[O + 2])), __uint_as_float(R[O + 3]))
#define TC_HALF(R, O)                                                                                              \
            do {                                                                                                   \
                if (__any_sync(0xffffffffu, TC_MAX4(R, O) > tau)) {                                                \
                    if (__any_sync(0xffffffffu, cnt > TC_CAP - 4)) TC_COMPACT(TC_CAP - 4);                         \
                    TC_APPEND(R, O); TC_APPEND(R, O + 1); TC_APPEND(R, O + 2); TC_APPEND(R, O + 3);                \
                }                                                                                                  \
            } while (0)
#define TC_GROUP(R, O, MG)                                                                                         \
            do {                                                                                                   \
                if (__any_sync(0xffffffffu, (MG) > tau)) { TC_HALF(R, O); TC_HALF(R, O + 4); }                     \
            } while (0)
#define TC_PROCESS(R, ITEM0)                                                                                       \
            do {                                                                                                   \
                const float g0_ = TC_MAX8(R, 0), g1_ = TC_MAX8(R, 8), g2_ = TC_MAX8(R, 16), g3_ = TC_MAX8(R, 24);  \
                if (__any_sync(0xffffffffu, fmaxf(tc_max3(g0_, g1_, g2_), g3_) > tau)) {                           \
                    const int32_t item0 = (ITEM0);                                                                 \
                    TC_GROUP(R, 0, g0_); TC_GROUP(R, 8, g1_); TC_GROUP(R, 16, g2_); TC_GROUP(R, 24, g3_);          \
                }                                                                                                  \
            } while (0)
            for (int t = t0; t < t1; ++t) {
                mbar_wait(BAR(2 * S + 2 + slot), slot_ph);
                tc_fence_after();
                const int32_t n0 = t * TC_TILE_N;
                const uint32_t tcol = tlane + (uint32_t)(TC_ACC_BASE + slot * TC_TILE_N);
#pragma unroll 1
                for (int hf = 0; hf < 2; ++hf) {
                    // 64 columns at a time (the register file holds 170 registers per thread at 10 warps per SM); the
                    // accumulator slot goes back to the MMA warp as soon as the second half sits in registers
                    uint32_t r0[32], r1[32];
                    if (!(p.debug & 2)) {
                        tc_ld32_nowait(tcol + (uint32_t)(hf * 64), r0);
                        tc_ld32_nowait(tcol + (uint32_t)(hf * 64 + 32), r1);
                        tc_ld_wait();
                    }
                    if (hf == 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(BAR(2 * S + 5 + slot));    // this warp has drained the slot
                    }
                    if (!(p.debug & 3)) {
                        TC_PROCESS(r0, n0 + hf * 64);
                        TC_PROCESS(r1, n0 + hf * 64 + 32);
                    } else if (!(p.debug & 2) && r0[0] == 0x7fc00001u && r1[1] == 1u) {
                        tau = 0.f;      // keeps the loads alive
                    }
                }
                // this sub-tile's next accumulator is two further down the ring of three
                slot += 2;
                if (slot >= TC_ACC_SLOTS) { slot -= TC_ACC_SLOTS; slot_ph ^= 1; }
            }
#undef TC_PROCESS
#undef TC_GROUP
#undef TC_HALF
#undef TC_MAX4
#undef TC_MAX8
#undef TC_APPEND
            // hand the next unit's user rows to the MMA warp before the final compaction of this one
            if (unit + (int)gridDim.x < num_units) stage_user_rows(unit + gridDim.x);
            // final pass: masks over the entries appended since the last compaction, trim to K'
            TC_COMPACT(kept);
            if (valid) {
                uint2* out = p.cand + ((size_t)c * p.n_chunks + ch) * TC_CAP;
                for (int e = 0; e < cnt; ++e) out[e] = tc_lds2(tc_slot(lp, sw, e));
                p.cand_cnt[(size_t)c * p.n_chunks + ch] = cnt;
                p.cand_tau[(size_t)c * p.n_chunks + ch] = tau;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------
// exact re-score + certificate, one warp per query slot
// ------------------------------------------------------------------------------------------------
#define TC_RS_WARPS 4
__global__ void __launch_bounds__(TC_RS_WARPS * 32) topn_tc_rescore_kernel(
    const double* __restrict__ P, const double* __restrict__ Q, const double* __restrict__ bu, const double* __restrict__ bi,
    double mu, int biased, int k, const int32_t* __restrict__ users, int32_t nq, int n_chunks, int topn,
    const uint2* __restrict__ cand, const int32_t* __restrict__ cand_cnt,
    const float* __restrict__ cand_tau, const double2* __restrict__ pstat, int eQ, double qnorm_max, double bi_max,
    double qabs_scaled_max, double c_err, int Kp, unsigned int* __restrict__ err_ratio_bits,
    const int32_t* __restrict__ slot_map,      // output slot of query slot c (second pass), or NULL = c
    int32_t* __restrict__ out_items, double* __restrict__ out_scores, int32_t* __restrict__ out_counts,
    // rows without a certificate: {output slot, user}; margin failures also get the threshold a second sweep
    // should start from (rs_*, only if rs_count != NULL), everything else goes to the exact kernel (ex_*)
    int32_t* __restrict__ rs_slots, int32_t* __restrict__ rs_users, float* __restrict__ rs_tau0, int* __restrict__ rs_count,
    int32_t* __restrict__ ex_slots, int32_t* __restrict__ ex_users, int* __restrict__ ex_count) {
    extern __shared__ __align__(16) unsigned char rs_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int max_cand = n_chunks * TC_CAP;
    double* sv = reinterpret_cast<double*>(rs_smem) + (size_t)warp * max_cand;
    int32_t* si = reinterpret_cast<int32_t*>(reinterpret_cast<double*>(rs_smem) + (size_t)TC_RS_WARPS * max_cand) + (size_t)warp * max_cand;
    float* sa = reinterpret_cast<float*>(reinterpret_cast<int32_t*>(reinterpret_cast<double*>(rs_smem) + (size_t)TC_RS_WARPS * max_cand) +
                                         (size_t)TC_RS_WARPS * max_cand) + (size_t)warp * max_cand;
    const int32_t c = blockIdx.x * TC_RS_WARPS + warp;
    if (c >= nq) return;
    const int32_t u = users ? users[c] : c;
    const int64_t oslot = slot_map ? slot_map[c] : c;
    // error bound of the fp16 sweep for this row, in the units of the exact scores.  With a = fp16(2^eu p),
    // b = fp16(2^eQ q): |a.b - 2^(eu+eQ) p.q| <= (2^-10 + 2^-22) sum|a_f b_f| + 2^-25 (sum|a_f| + sum|b_f|) + fp32
    // accumulation slop (Kp+8) 2^-22 sum|a_f b_f|; sum|a_f b_f| <= ||a|| ||b||.  c_err carries the relative part.
    const double2 ps = pstat[c];
    const int eu = tc_scale_exp(ps.y, TC_USER_EXP_LO, TC_USER_EXP_HI);
    const double ub = biased ? bu[u] : 0.0;
    const double scale = ps.x * qnorm_max + bi_max;
    const double eta = ldexp((double)Kp * (ldexp(ps.y, eu) + qabs_scaled_max) * 1.001, -25 - eu - eQ);
    const double bound0 = c_err * scale + eta;
    // gather candidates of all chunks
    int M = 0;
    float tau_max = -INFINITY;
    for (int ch = 0; ch < n_chunks; ++ch) {
        const int cnt = cand_cnt[(size_t)c * n_chunks + ch];
        tau_max = fmaxf(tau_max, cand_tau[(size_t)c * n_chunks + ch]);
        for (int e = lane; e < cnt; e += 32) {
            const uint2 ce = cand[((size_t)c * n_chunks + ch) * TC_CAP + e];
            si[M + e] = (int32_t)ce.y; sa[M + e] = __uint_as_float(ce.x);
        }
        M += cnt;
    }
    __syncwarp();
    const double tau_d = ldexp((double)tau_max, -eu - eQ);       // threshold in exact-score units (power-of-two scaling is exact)
    float worst = 0.f;
    // exact scores in Java's order (DenseVector.java:104-111; BiasedMFRecommender.java:119)
    const double* pu = P + (int64_t)u * k;
    for (int e = lane; e < M; e += 32) {
        const int32_t it = si[e];
        double d = dot_lr_f64(pu, Q + (int64_t)it * k, k);
        const double core = biased ? d + bi[it] : d;
        if (biased) d = __dadd_rn(__dadd_rn(__dadd_rn(d, bu[u]), bi[it]), mu);
        sv[e] = d;
        // observed sweep error over the bound (diagnostic: must stay below 1)
        const double err = fabs(ldexp((double)sa[e], -eu - eQ) - core);
        if (bound0 > 0.0 && err == err) worst = fmaxf(worst, (float)(err / bound0));
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) worst = fmaxf(worst, __shfl_xor_sync(0xffffffffu, worst, m));
    if (lane == 0 && worst > 0.f) atomicMax(err_ratio_bits, __float_as_uint(worst));
    __syncwarp();
    bool ok = M >= topn;
    float tau0 = 0.f;
    bool margin_fail = false;
    // selection of the best topn+1 by (Double.compareTo desc); a tie anywhere in that prefix fails the row
    double prev = 0.0;
    const int want = min(M, topn + 1);
    for (int r = 0; ok && r < want; ++r) {
        double bv = -INFINITY; int be = -1;
        for (int e = lane; e < M; e += 32) {
            const double x = sv[e];
            if (si[e] >= 0 && (be < 0 || jcompare(x, bv) > 0)) { bv = x; be = e; }
        }
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, m);
            const int oe = __shfl_xor_sync(0xffffffffu, be, m);
            if (oe >= 0 && (be < 0 || jcompare(ov, bv) > 0 || (jcompare(ov, bv) == 0 && oe < be))) { bv = ov; be = oe; }
        }
        if (be < 0 || bv != bv) { ok = false; break; }
        if (r > 0 && jcompare(bv, prev) == 0) { ok = false; break; }      // exact tie: heap-order semantics needed
        if (r < topn && lane == 0) { out_items[oslot * topn + r] = si[be]; out_scores[oslot * topn + r] = bv; }
        if (r == topn - 1) {
            // certificate: nothing outside the candidate lists can reach the N-th exact score
            const double bound = bound0 + 1e-12 * (scale + fabs(ub) + fabs(mu) + fabs(tau_d));
            const double reach = tau_d + bound + (biased ? (ub + mu) : 0.0);
            if (!(bv > reach)) {
                // A second sweep that starts from tau0 collects every item whose exact score can reach bv, and its
                // certificate then holds with room to spare (unless more than K' items crowd that band).
                const double core_n = bv - (biased ? (ub + mu) : 0.0);
                tau0 = __double2float_rd(ldexp(core_n - 2.5 * bound, eu + eQ));
                margin_fail = tau0 == tau0 && fabsf(tau0) < INFINITY;
                ok = false; break;
            }
        }
        prev = bv;
        __syncwarp();
        if (lane == 0) si[be] = -1 - si[be];     // taken
        __syncwarp();
    }
    if (lane == 0) {
        if (ok) out_counts[oslot] = topn;
        else if (margin_fail && rs_count) {
            const int pos = atomicAdd(rs_count, 1);
            rs_slots[pos] = (int32_t)oslot; rs_users[pos] = u; rs_tau0[pos] = tau0;
        } else {
            const int pos = atomicAdd(ex_count, 1);
            ex_slots[pos] = (int32_t)oslot; ex_users[pos] = u;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// host driver
// ------------------------------------------------------------------------------------------------
static int tc_make_map(lrk_handle_s* h, TcState* s, CUtensorMap* map, const void* gptr, int Kp, int64_t rows) {
    if (!s->encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        LRK_CUDA(h, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess)
            return lrk_fail(h, LRK_ERR_CUDA, "cuTensorMapEncodeTiled", "driver entry point not available", __FILE__, __LINE__);
        s->encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
    }
    cuuint64_t dims[2] = {(cuuint64_t)Kp, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)Kp * 2};
    cuuint32_t box[2] = {TC_KB, TC_TILE_M};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = s->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(gptr), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return lrk_fail(h, LRK_ERR_CUDA, "cuTensorMapEncodeTiled", "encode failed", __FILE__, __LINE__);
    return LRK_OK;
}

#define TC_KEEP_DEFAULT(topn) std::min(TC_KEEP_MAX, std::max(16, (topn) + 6))

// One pass: operand rows of the queried users -> tcgen05 sweep with fused selection -> exact fp64 re-score with
// certificate.  Results go to out_*[slot_map ? slot_map[c] : c]; rows without a certificate are appended to the
// rs_* (second sweep, only for the first pass) / ex_* (exact kernel) lists.
static int tc_pass(lrk_handle_s* h, TcState* s, const int32_t* d_users, int32_t nq, const float* init_tau, const int32_t* slot_map,
                   int topn, int exclude_train, int keep, int32_t* d_items, double* d_scores, int32_t* d_counts,
                   int32_t* rs_slots, int32_t* rs_users, float* rs_tau0, int* rs_count,
                   int32_t* ex_slots, int32_t* ex_users, int* ex_count, bool first_pass) {
    cudaStream_t st = h->stream;
    const bool biased = lrk_has_bias(h);
    const int Kp = s->Kp;
    const int num_kb = Kp / TC_KB;
    // ---- work decomposition
    const int total_tiles = lrk_ceil_div(h->I, TC_TILE_N);
    const int m_tiles = lrk_ceil_div(nq, TC_ROWS);
    int n_chunks = lrk_ceil_div(h->sm_count, m_tiles);
    n_chunks = std::max(1, std::min(n_chunks, std::min(TC_MAX_CHUNKS, std::max(1, total_tiles / 16))));
    const int tiles_per_chunk = lrk_ceil_div(total_tiles, n_chunks);
    n_chunks = lrk_ceil_div(total_tiles, tiles_per_chunk);
    const int64_t nq_pad = (int64_t)m_tiles * TC_ROWS;
    const size_t tile_bytes = (size_t)TC_TILE_N * TC_KB * 2;
    const size_t b_stage = (size_t)num_kb * tile_bytes;
    const size_t list_bytes = (size_t)TC_ROWS * TC_CAP * 8;
    int stages = (int)((227 * 1024 - 1024 - 256 - list_bytes) / b_stage);
    stages = std::max(2, std::min(stages, 8));
    { const char* es = getenv("LRK_TC_STAGES"); if (es && atoi(es) >= 2) stages = std::min(stages, atoi(es)); }   // profiling probe
    const size_t smem = 1024 + (size_t)stages * b_stage + list_bytes + TC_NBARS(stages) * 8 + 16;
    // ---- scratch
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t b_aq = up(sizeof(__half) * (size_t)nq_pad * Kp), b_pn = up(sizeof(double2) * (size_t)nq_pad);
    const size_t b_cs = up(sizeof(uint2) * (size_t)nq_pad * n_chunks * TC_CAP);
    const size_t b_cc = up(sizeof(int32_t) * (size_t)nq_pad * n_chunks), b_ct = up(sizeof(float) * (size_t)nq_pad * n_chunks);
    int rc = lrk_dev_alloc(h, &s->work, b_aq + b_pn + b_cs + b_cc + b_ct + 256);
    if (rc) return rc;
    char* w = s->work;
    __half* Aq = (__half*)w; w += b_aq;
    double2* pstat = (double2*)w; w += b_pn;
    uint2* cand = (uint2*)w; w += b_cs;
    int32_t* ccnt = (int32_t*)w; w += b_cc;
    float* ctau = (float*)w; w += b_ct;
    if (nq_pad > nq) LRK_CUDA(h, cudaMemsetAsync(Aq + (size_t)nq * Kp, 0, sizeof(__half) * (size_t)(nq_pad - nq) * Kp, st));
    LRK_CUDA(h, cudaMemsetAsync(ccnt, 0, sizeof(int32_t) * (size_t)nq_pad * n_chunks, st));
    tc_build_users_kernel<<<lrk_ceil_div(nq, 8), 256, 0, st>>>(h->P64, biased, h->k, Kp, d_users, nq, Aq, pstat);
    LRK_LAUNCH_CHECK(h);
    CUtensorMap tmB;
    rc = tc_make_map(h, s, &tmB, s->Bq, Kp, h->I);
    if (rc) return rc;
    TcParams p;
    memset(&p, 0, sizeof p);
    p.nq = nq; p.I = h->I; p.n_chunks = n_chunks; p.tiles_per_chunk = tiles_per_chunk; p.total_tiles = total_tiles;
    p.num_kb = num_kb; p.stages = stages; p.exclude_train = exclude_train ? 1 : 0;
    p.keep = keep;
    { const char* ek = getenv("LRK_TC_KEEP"); if (first_pass && ek && atoi(ek) >= topn + 1 && atoi(ek) <= TC_KEEP_MAX) p.keep = atoi(ek); }   // tuning probe
    { const char* dbg = getenv("LRK_TC_DEBUG"); p.debug = dbg ? atoi(dbg) : 0; }
    p.rowptr = h->d_rowptr; p.col = h->d_col; p.users = d_users; p.init_tau = init_tau;
    p.cand = cand; p.cand_cnt = ccnt; p.cand_tau = ctau;
    LRK_CUDA(h, cudaFuncSetAttribute(topn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = std::min(h->sm_count, m_tiles * n_chunks);
    if (first_pass) LRK_CUDA(h, cudaEventRecord(s->ev[1], st));
    topn_tc_kernel<<<grid, TC_THREADS, smem, st>>>(tmB, Aq, p);
    LRK_LAUNCH_CHECK(h);
    if (first_pass) LRK_CUDA(h, cudaEventRecord(s->ev[2], st));
    // ---- exact re-score + certificate
    const double c_err = ldexp(1.0, -10) * (1.0 + ldexp(1.0, -11)) + (double)(Kp + 8) * ldexp(1.0, -22);
    const double qabs_scaled_max = ldexp(std::max(s->qabs_max, s->bi_max), s->eQ);
    const size_t rs_smem_bytes = (size_t)TC_RS_WARPS * n_chunks * TC_CAP * (sizeof(double) + sizeof(int32_t) + sizeof(float));
    LRK_CUDA(h, cudaFuncSetAttribute(topn_tc_rescore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs_smem_bytes));
    topn_tc_rescore_kernel<<<lrk_ceil_div(nq, TC_RS_WARPS), TC_RS_WARPS * 32, rs_smem_bytes, st>>>(
        h->P64, h->Q64, h->bu64, h->bi64, h->mu, biased, h->k, d_users, nq, n_chunks, topn, cand, ccnt, ctau, pstat,
        s->eQ, s->qnorm_max, s->bi_max, qabs_scaled_max, c_err, Kp, (unsigned int*)(s->d_stats + 3), slot_map, d_items, d_scores, d_counts,
        rs_slots, rs_users, rs_tau0, rs_count, ex_slots, ex_users, ex_count);
    LRK_LAUNCH_CHECK(h);
    return LRK_OK;
}

static int topn_tc_run(lrk_handle_s* h, const int32_t* d_users, int32_t nq, int topn, int exclude_train,
                       int32_t* d_items, double* d_scores, int32_t* d_counts) {
    TcState* s = tc_state(h);
    cudaStream_t st = h->stream;
    const bool biased = lrk_has_bias(h);
    const int Kp = tc_kp(h);
    const int num_kb = Kp / TC_KB;
    if (num_kb > 2 || topn > TC_MAX_TOPN)
        return lrk_fail(h, LRK_ERR_INVALID, "lrk_topn", "tensor-core path supports k (+2 for BiasedMF) <= 128 and topn <= 26", __FILE__, __LINE__);
    for (cudaEvent_t& ev : s->ev) if (!ev) LRK_CUDA(h, cudaEventCreate(&ev));
    LRK_CUDA(h, cudaEventRecord(s->ev[0], st));
    int rc;
    // ---- item operand (cached until the factors change)
    if (!s->valid || s->Kp != Kp) {
        if ((rc = lrk_dev_alloc(h, &s->Bq, (size_t)h->I * Kp))) return rc;
        if ((rc = lrk_dev_alloc(h, &s->d_stats, 4))) return rc;
        LRK_CUDA(h, cudaMemsetAsync(s->d_stats, 0, 32, st));
        tc_item_stats_kernel<<<lrk_ceil_div(h->I, 8), 256, 0, st>>>(h->Q64, h->bi64, biased, h->k, h->I, s->d_stats);
        LRK_LAUNCH_CHECK(h);
        unsigned long long stats[3];
        LRK_CUDA(h, cudaMemcpyAsync(stats, s->d_stats, 24, cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
        double n2, bm, qa;
        memcpy(&n2, &stats[0], 8); memcpy(&bm, &stats[1], 8); memcpy(&qa, &stats[2], 8);
        s->finite = std::isfinite(n2) && std::isfinite(bm) && std::isfinite(qa);
        s->qnorm_max = sqrt(n2); s->bi_max = biased ? bm : 0.0; s->qabs_max = qa;
        s->eQ = tc_scale_exp(std::max(qa, s->bi_max), -60, 60);
        if (s->finite) {
            tc_build_items_kernel<<<lrk_ceil_div(h->I, 8), 256, 0, st>>>(h->Q64, h->bi64, biased, h->k, Kp, h->I, s->eQ, s->Bq);
            LRK_LAUNCH_CHECK(h);
        }
        s->Kp = Kp; s->valid = true;
    }
    if (!s->finite) {
        // NaN / Inf among the item factors: Double.compareTo semantics for those need the exact kernel
        if ((rc = topn_exact_launch(h, d_users, nq, topn, exclude_train, d_items, d_scores, d_counts))) return rc;
        LRK_CUDA(h, cudaStreamSynchronize(st));
        h->topn_fast_users = 0; h->topn_fallback_users = nq;
        return LRK_OK;
    }
    // ---- fail lists of the call (outside the per-pass scratch, which a second pass may regrow)
    if ((rc = lrk_dev_alloc(h, &s->lists, sizeof(int32_t) * 5 * (size_t)nq + 64))) return rc;
    int* counters = (int*)s->lists.ptr;                               // [0] second-sweep rows, [1] exact-kernel rows
    int32_t* rs_slots = (int32_t*)(s->lists + 64);
    int32_t* rs_users = rs_slots + nq;
    float* rs_tau0 = (float*)(rs_users + nq);
    int32_t* ex_slots = (int32_t*)(rs_tau0 + nq);
    int32_t* ex_users = ex_slots + nq;
    LRK_CUDA(h, cudaMemsetAsync(counters, 0, 64, st));
    LRK_CUDA(h, cudaMemsetAsync(s->d_stats + 3, 0, 8, st));
    int cnts[2] = {0, 0};
    // pass 1: every queried row from tau = -inf
    rc = tc_pass(h, s, d_users, nq, nullptr, nullptr, topn, exclude_train, TC_KEEP_DEFAULT(topn), d_items, d_scores, d_counts,
                     rs_slots, rs_users, rs_tau0, counters, ex_slots, ex_users, counters + 1, true);
    if (rc) return rc;
    LRK_CUDA(h, cudaMemcpyAsync(cnts, counters, sizeof cnts, cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    const int n_resweep = cnts[0];
    if (n_resweep > 0) {
        // pass 2: rows whose margin was too thin, from the threshold their first result implies, widest K'
        rc = tc_pass(h, s, rs_users, n_resweep, rs_tau0, rs_slots, topn, exclude_train, TC_KEEP_MAX, d_items, d_scores, d_counts,
                     nullptr, nullptr, nullptr, nullptr, ex_slots, ex_users, counters + 1, false);
        if (rc) return rc;
        LRK_CUDA(h, cudaMemcpyAsync(cnts, counters, sizeof cnts, cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
    }
    LRK_CUDA(h, cudaEventRecord(s->ev[3], st));
    LRK_CUDA(h, cudaMemcpyAsync(&h->topn_err_ratio, s->d_stats + 3, sizeof(float), cudaMemcpyDeviceToHost, st));
    const int nfail = cnts[1];
    if (nfail > 0) {
        // rows still without a certificate (exact ties, fewer than N candidates, crowded bands): exact fp64 path
        if ((rc = lrk_dev_alloc(h, &s->fail_items, (size_t)nfail * topn))) return rc;
        if ((rc = lrk_dev_alloc(h, &s->fail_scores, (size_t)nfail * topn))) return rc;
        if ((rc = lrk_dev_alloc(h, &s->fail_counts, (size_t)nfail))) return rc;
        rc = topn_parts_fit(h, topn) ? topn_exact_parallel_launch(h, ex_users, nfail, topn, exclude_train, s->fail_items, s->fail_scores, s->fail_counts)
                                     : topn_exact_launch(h, ex_users, nfail, topn, exclude_train, s->fail_items, s->fail_scores, s->fail_counts);
        if (rc) return rc;
        topn_scatter_kernel<<<lrk_ceil_div((int64_t)nfail * topn, 256), 256, 0, st>>>(ex_slots, nfail, topn, s->fail_items, s->fail_scores,
                                                                                   s->fail_counts, d_items, d_scores, d_counts);
        LRK_LAUNCH_CHECK(h);
        LRK_CUDA(h, cudaStreamSynchronize(st));
    }
    LRK_CUDA(h, cudaEventRecord(s->ev[4], st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    for (int i = 0; i < 4; ++i) cudaEventElapsedTime(&h->topn_phase_ms[i], s->ev[i], s->ev[i + 1]);
    h->topn_resweep_users = n_resweep;
    h->topn_fast_users = nq - nfail;
    h->topn_fallback_users = nfail;
    return LRK_OK;
}
