// Reference-order BPR (LRK_UPDATE_REFERENCE_ORDER with LRK_MODEL_BPR): one epoch of BPRRecommender.java:48-93 as the reference
// runs it -- numRates samples drawn from the one global java.util.Random (Randoms.r), each update applied in sample order in fp64
// with Java's operation order -- so that the learned factors and the generator state after the epoch are bit-identical to the
// sequential loop (with StrictMath.exp, i.e. fdlibm's __ieee754_exp, in Maths.logistic).
//
// Which samples an epoch draws never depends on the factors, only on the train matrix and the generator state, so the epoch
// runs in two stages.
//
// Draw stage (bpr_ref_draw): the triples (u, i, j) of samples [0, n) and the number of draws they consume.
//   1. stream: next(31) for positions [0, L) of the generator, every position's state by LCG jump-ahead from the epoch's state.
//   2. speculative parse: at EVERY position, parse a sample as if one started there (nextInt with its power-of-two branch and
//      rejection loop, the user redraw while the row is empty or full, the positive, the negative redrawn while it is in the row,
//      a binary search like the oracle's) and record the triple and the draws consumed, cons(t).  W = max cons(t).
//   3. resolve: the true sample starts are the orbit of 0 under t -> t + cons(t).  Parses that start off the orbit do not
//      rejoin it quickly (almost every sample takes exactly 3 draws), so the orbit is found exactly: the stream is cut into chunks
//      of C >= W positions; the first orbit position of a chunk lies within W of its start, so every chunk is walked from each of
//      its first W positions, giving per entry offset the exit offset into the next chunk and the samples on the way.  These
//      maps compose; one thread chains them over the chunks (about a thousand for the ML-20M shape), and a last pass walks every
//      chunk from its true entry and writes the samples in order.  A parse that needs positions past L, or an orbit that does
//      not reach n samples inside L, doubles L and repeats.
//
// Update stage (bpr_ref_update_kernel): a persistent dataflow kernel.  A stable radix sort of the 3n (row, sample) keys -- users
// and items in one key space -- gives every sample its sequence number on each of its three rows.  Warps claim samples in
// increasing order from a counter, wait until each row's completion counter equals the sample's sequence number, update the
// three rows and release the counters.  Progress: the smallest claimed sample that is not finished has all its predecessors
// finished (they are smaller, so they were claimed, by warps that are running), so its warp can always proceed; no level
// barrier is needed, and the chain of the epoch (about 223 k samples for the ML-20M shape, set by the most drawn positive item)
// is walked at the latency of one update per hop.  Spins are bounded: a wait that exceeds spin_limit cycles raises `abort`, every
// warp leaves, and the epoch fails with LRK_ERR_CUDA instead of hanging.
//
// Arithmetic: only + - * / in _rn form and bit manipulation (no FMA contraction), the dots as one sequential __dadd_rn chain
// from 0.0 over products the lanes leave in shared memory (DenseVector.dot, DenseVector.java:104-111), exp and log as fdlibm.
// Only the reported loss is summed in another order (it agrees to ~1e-15 relative).
#pragma once
#include "lrk_common.cuh"
#include <cub/cub.cuh>
#include <vector>

#define LRK_JR_MULT 0x5DEECE66DULL
#define LRK_JR_ADD 0xBULL
#define LRK_JR_MASK ((1ULL << 48) - 1)

// (A, C) of the LCG advanced `steps` times: S -> A * S + C (mod 2^48), by doubling (A, C) o (A, C) = (A^2, A * C + C)
__host__ __device__ __forceinline__ uint64_t jr_jump(uint64_t s, uint64_t steps) {
    uint64_t a = LRK_JR_MULT, c = LRK_JR_ADD, ar = 1, cr = 0;
    while (steps) {
        if (steps & 1) { ar = (a * ar) & LRK_JR_MASK; cr = (a * cr + c) & LRK_JR_MASK; }
        c = (a * c + c) & LRK_JR_MASK;
        a = (a * a) & LRK_JR_MASK;
        steps >>= 1;
    }
    return (ar * s + cr) & LRK_JR_MASK;
}

struct BprRefState {
    uint64_t jstate = 0;          // Randoms.r's 48-bit state ("jdk.random.state"): the next epoch starts from it
    int64_t drawable = 0;         // users with 0 < |row| < numItems
    double draws_per_sample = 3.2;
    int64_t L = 0;                // stream length that sufficed last
    LrkBuf<int32_t> d_v, d_cons, d_trip;          // per stream position: next(31), draws consumed (-1: ran past L), triple
    LrkBuf<int2> d_map;                           // per (chunk, entry offset): {exit offset or -1, samples}
    LrkBuf<long long> d_chunk;                    // per chunk: {entry offset, first sample}
    LrkBuf<long long> d_res;                      // {W, overflow, chunks used, end position}
    LrkBuf<int32_t> d_samp;                       // the epoch's triples in sample order, 3 n
    LrkBuf<int32_t> d_seq;                        // sequence number of each sample on its rows u, U + i, U + j, 3 n
    LrkBuf<uint32_t> d_keys, d_keys2, d_vals, d_vals2;
    LrkBuf<int32_t> d_row_start;
    LrkBuf<char> d_sort_tmp;
    LrkBuf<unsigned int> d_done;                  // per row (users, then items): samples of this epoch finished on it
    LrkBuf<unsigned long long> d_claim;
    LrkBuf<int> d_abort;
};

// ---- draw stage ---------------------------------------------------------------------------------------------------------
#define LRK_BPR_STREAM_PER_THREAD 16

__global__ void bpr_ref_stream_kernel(uint64_t s0, int64_t L, int32_t* __restrict__ v) {
    const int64_t t0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * LRK_BPR_STREAM_PER_THREAD;
    if (t0 >= L) return;
    uint64_t s = jr_jump(s0, (uint64_t)t0);
    for (int r = 0; r < LRK_BPR_STREAM_PER_THREAD && t0 + r < L; ++r) {
        s = (s * LRK_JR_MULT + LRK_JR_ADD) & LRK_JR_MASK;
        v[t0 + r] = (int32_t)(uint32_t)(s >> 17);      // next(31)
    }
}

// java.util.Random.nextInt(bound) over the stream from position *p; false when it needs a position >= L
__device__ __forceinline__ bool jr_next_int(const int32_t* __restrict__ v, int64_t L, int64_t* p, int32_t bound, int32_t* out) {
    if (*p >= L) return false;
    int32_t x = v[(*p)++];
    const int32_t m = bound - 1;
    if ((bound & m) == 0) { *out = (int32_t)(((int64_t)bound * (int64_t)x) >> 31); return true; }
    for (;;) {
        const int32_t r = x % bound;
        if ((int32_t)((uint32_t)x - (uint32_t)r + (uint32_t)m) >= 0) { *out = r; return true; }
        if (*p >= L) return false;
        x = v[(*p)++];
    }
}

__global__ void bpr_ref_parse_kernel(const int32_t* __restrict__ v, int64_t L, const int64_t* __restrict__ rowptr,
                                     const int32_t* __restrict__ col, int32_t U, int32_t I, int32_t* __restrict__ cons,
                                     int32_t* __restrict__ trip, long long* __restrict__ res) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int32_t used = 0;
    if (t < L) {
        int64_t p = t;
        int32_t u = 0, i = 0, j = 0;
        bool ok;
        for (;;) {                                                   // BPRRecommender.java:54-67
            if (!(ok = jr_next_int(v, L, &p, U, &u))) break;
            const int64_t b = rowptr[u], len = rowptr[u + 1] - b;
            if (len == 0 || len == I) continue;
            int32_t r;
            if (!(ok = jr_next_int(v, L, &p, (int32_t)len, &r))) break;
            i = col[b + r];
            for (;;) {
                if (!(ok = jr_next_int(v, L, &p, I, &j))) break;
                int64_t lo = 0, hi = len;                            // is j in the (ascending) row?
                while (lo < hi) {
                    const int64_t mid = (lo + hi) >> 1;
                    if (col[b + mid] < j) lo = mid + 1; else hi = mid;
                }
                if (lo == len || col[b + lo] != j) break;
            }
            break;
        }
        if (ok) {
            used = (int32_t)(p - t);
            trip[3 * t] = u; trip[3 * t + 1] = i; trip[3 * t + 2] = j;
        }
        cons[t] = ok ? used : -1;
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) used = max(used, __shfl_xor_sync(0xffffffffu, used, m));
    if ((threadIdx.x & 31) == 0 && used > 0) atomicMax(res, (long long)used);
}

// one thread per (chunk, entry offset < W): walk the chunk, record the exit offset past its end (-1: a parse ran past L) and the
// samples started inside it
__global__ void bpr_ref_walk_kernel(const int32_t* __restrict__ cons, int64_t L, int64_t C, int64_t K, int W, int2* __restrict__ map) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= K * W) return;
    const int64_t c = g / W, cend = min((c + 1) * C, L);
    int64_t t = c * C + g % W;
    int cnt = 0, exit_off = 0;
    while (t < cend) {
        const int32_t d = cons[t];
        if (d < 0) { exit_off = -1; break; }
        t += d; ++cnt;
    }
    if (exit_off == 0) exit_off = (int)(t - cend);
    map[g] = make_int2(exit_off, cnt);
}

// one thread: chain the chunk maps from position 0 until n samples have started; res = {W, overflow, chunks used, -}
__global__ void bpr_ref_resolve_kernel(const int2* __restrict__ map, int64_t K, int W, int64_t n, long long* __restrict__ chunk,
                                       long long* __restrict__ res) {
    long long s = 0;
    int e = 0;
    for (int64_t c = 0; c < K; ++c) {
        chunk[2 * c] = e; chunk[2 * c + 1] = s;
        const int2 m = map[c * W + e];
        if (s + m.y >= n) { res[1] = 0; res[2] = c + 1; return; }
        if (m.x < 0 || c + 1 == K) break;
        s += m.y; e = m.x;
    }
    res[1] = 1;                                                      // the stream is too short
}

// one thread per chunk in use: walk from the true entry, write samples [first, n) to out (3 ints each) and the end position
__global__ void bpr_ref_emit_kernel(const int32_t* __restrict__ cons, const int32_t* __restrict__ trip, int64_t L, int64_t C,
                                    const long long* __restrict__ chunk, long long* __restrict__ res, int64_t first, int64_t n,
                                    int32_t* __restrict__ out) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= res[2]) return;
    const int64_t cend = min((c + 1) * C, L);
    int64_t t = c * C + chunk[2 * c], s = chunk[2 * c + 1];
    while (t < cend && s < n) {
        if (s >= first) {
            out[3 * (s - first)] = trip[3 * t]; out[3 * (s - first) + 1] = trip[3 * t + 1]; out[3 * (s - first) + 2] = trip[3 * t + 2];
        }
        t += cons[t]; ++s;
        if (s == n) res[3] = t;
    }
}

// samples [first, n) of the epoch that starts from b->jstate into out (device, 3 * (n - first) ints); *end_out = draws consumed
static int bpr_ref_draw(lrk_handle_s* h, BprRefState* b, int64_t first, int64_t n, int32_t* out, int64_t* end_out) {
    cudaStream_t st = h->stream;
    *end_out = 0;
    if (n == 0) return LRK_OK;
    LRK_REQUIRE(h, b->drawable > 0, "BPR reference order: no user has 0 < |row| < numItems, so the reference would draw users forever");
    int64_t L = std::max<int64_t>(b->L, (int64_t)((double)n * b->draws_per_sample) + 4096);
    int rc;
    for (;;) {
        if ((rc = lrk_dev_alloc(h, &b->d_v, (size_t)L))) return rc;
        if ((rc = lrk_dev_alloc(h, &b->d_cons, (size_t)L))) return rc;
        if ((rc = lrk_dev_alloc(h, &b->d_trip, 3 * (size_t)L))) return rc;
        if ((rc = lrk_dev_alloc(h, &b->d_res, 4))) return rc;
        LRK_CUDA(h, cudaMemsetAsync(b->d_res, 0, 4 * sizeof(long long), st));
        const int64_t nthr = (L + LRK_BPR_STREAM_PER_THREAD - 1) / LRK_BPR_STREAM_PER_THREAD;
        bpr_ref_stream_kernel<<<lrk_ceil_div(nthr, 256), 256, 0, st>>>(b->jstate, L, b->d_v); LRK_LAUNCH_CHECK(h);
        bpr_ref_parse_kernel<<<lrk_ceil_div(L, 256), 256, 0, st>>>(b->d_v, L, h->d_rowptr, h->d_col, h->U, h->I, b->d_cons, b->d_trip,
                                                                    b->d_res);
        LRK_LAUNCH_CHECK(h);
        long long res[4];
        LRK_CUDA(h, cudaMemcpyAsync(res, b->d_res, sizeof res, cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
        const int W = (int)std::max<long long>(res[0], 1);
        const int64_t C = std::max<int64_t>(65536, W);
        const int64_t K = (L + C - 1) / C;
        if ((rc = lrk_dev_alloc(h, &b->d_map, (size_t)(K * W)))) return rc;
        if ((rc = lrk_dev_alloc(h, &b->d_chunk, 2 * (size_t)K))) return rc;
        bpr_ref_walk_kernel<<<lrk_ceil_div(K * W, 128), 128, 0, st>>>(b->d_cons, L, C, K, W, b->d_map); LRK_LAUNCH_CHECK(h);
        bpr_ref_resolve_kernel<<<1, 1, 0, st>>>(b->d_map, K, W, n, b->d_chunk, b->d_res); LRK_LAUNCH_CHECK(h);
        LRK_CUDA(h, cudaMemcpyAsync(res, b->d_res, sizeof res, cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
        if (res[1]) {                                               // the orbit ran past the stream: twice as long
            L *= 2;
            continue;
        }
        bpr_ref_emit_kernel<<<lrk_ceil_div(res[2], 128), 128, 0, st>>>(b->d_cons, b->d_trip, L, C, b->d_chunk, b->d_res, first, n, out);
        LRK_LAUNCH_CHECK(h);
        LRK_CUDA(h, cudaMemcpyAsync(res, b->d_res, sizeof res, cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
        b->L = L;
        *end_out = res[3];
        return LRK_OK;
    }
}

// ---- update stage -------------------------------------------------------------------------------------------------------
// fdlibm 5.3 e_exp.c (__ieee754_exp == StrictMath.exp) in _rn operations
__device__ __forceinline__ double bx_with_hi(double y, uint32_t hi) { return __hiloint2double((int)hi, __double2loint(y)); }
__device__ double bx_exp(double x) {
    const double huge = 1.0e+300, twom1000 = 9.33263618503218878990e-302, o_threshold = 7.09782712893383973096e+02,
                 u_threshold = -7.45133219101941108420e+02, ln2HI = 6.93147180369123816490e-01, ln2LO = 1.90821492927058770002e-10,
                 invln2 = 1.44269504088896338700e+00, P1 = 1.66666666666666019037e-01, P2 = -2.77777777770155933842e-03,
                 P3 = 6.61375632143793436117e-05, P4 = -1.65339022054652515390e-06, P5 = 4.13813679705723846039e-08;
    uint32_t hx = (uint32_t)__double2hiint(x);
    const int xsb = (int)(hx >> 31);
    hx &= 0x7fffffffu;
    double hi = 0.0, lo = 0.0;
    int k = 0;
    if (hx >= 0x40862E42u) {
        if (hx >= 0x7ff00000u) {
            if (((hx & 0xfffffu) | (uint32_t)__double2loint(x)) != 0) return __dadd_rn(x, x);
            return xsb == 0 ? x : 0.0;
        }
        if (x > o_threshold) return __dmul_rn(huge, huge);
        if (x < u_threshold) return __dmul_rn(twom1000, twom1000);
    }
    if (hx > 0x3fd62e42u) {
        if (hx < 0x3FF0A2B2u) {
            hi = __dsub_rn(x, xsb ? -ln2HI : ln2HI); lo = xsb ? -ln2LO : ln2LO; k = 1 - xsb - xsb;
        } else {
            k = __double2int_rz(__dadd_rn(__dmul_rn(invln2, x), xsb ? -0.5 : 0.5));
            const double t = (double)k;
            hi = __dsub_rn(x, __dmul_rn(t, ln2HI));
            lo = __dmul_rn(t, ln2LO);
        }
        x = __dsub_rn(hi, lo);
    } else if (hx < 0x3e300000u) {
        if (__dadd_rn(huge, x) > 1.0) return __dadd_rn(1.0, x);
    }
    const double t = __dmul_rn(x, x);
    const double c = __dsub_rn(x, __dmul_rn(t, __dadd_rn(P1, __dmul_rn(t, __dadd_rn(P2, __dmul_rn(t, __dadd_rn(P3,
                                   __dmul_rn(t, __dadd_rn(P4, __dmul_rn(t, P5))))))))));
    if (k == 0) return __dsub_rn(1.0, __dsub_rn(__ddiv_rn(__dmul_rn(x, c), __dsub_rn(c, 2.0)), x));
    const double y = __dsub_rn(1.0, __dsub_rn(__dsub_rn(lo, __ddiv_rn(__dmul_rn(x, c), __dsub_rn(2.0, c))), hi));
    if (k >= -1021) return bx_with_hi(y, (uint32_t)__double2hiint(y) + ((uint32_t)k << 20));
    return __dmul_rn(bx_with_hi(y, (uint32_t)__double2hiint(y) + ((uint32_t)(k + 1000) << 20)), twom1000);
}

// fdlibm 5.3 e_log.c (== StrictMath.log) in _rn operations, for the loss term
__device__ double bx_log(double x) {
    const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10, two54 = 1.80143985094819840000e+16,
                 Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01, Lg3 = 2.857142874366239149e-01,
                 Lg4 = 2.222219843214978396e-01, Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
                 Lg7 = 1.479819860511658591e-01;
    int hx = __double2hiint(x);
    const uint32_t lx = (uint32_t)__double2loint(x);
    int k = 0;
    if (hx < 0x00100000) {
        if (((hx & 0x7fffffff) | (int)lx) == 0) return __longlong_as_double((long long)0xfff0000000000000ULL);   // -inf
        if (hx < 0) return __longlong_as_double((long long)0x7ff8000000000000ULL);                              // NaN
        k -= 54; x = __dmul_rn(x, two54); hx = __double2hiint(x);
    }
    if (hx >= 0x7ff00000) return __dadd_rn(x, x);
    k += (hx >> 20) - 1023;
    hx &= 0x000fffff;
    int i = (hx + 0x95f64) & 0x100000;
    x = __hiloint2double(hx | (i ^ 0x3ff00000), __double2loint(x));
    k += (i >> 20);
    const double f = __dsub_rn(x, 1.0);
    double dk;
    if ((0x000fffff & (2 + hx)) < 3) {
        if (f == 0.0) { if (k == 0) return 0.0; dk = (double)k; return __dadd_rn(__dmul_rn(dk, ln2_hi), __dmul_rn(dk, ln2_lo)); }
        const double R = __dmul_rn(__dmul_rn(f, f), __dsub_rn(0.5, __dmul_rn(0.33333333333333333, f)));
        if (k == 0) return __dsub_rn(f, R);
        dk = (double)k;
        return __dsub_rn(__dmul_rn(dk, ln2_hi), __dsub_rn(__dsub_rn(R, __dmul_rn(dk, ln2_lo)), f));
    }
    const double s = __ddiv_rn(f, __dadd_rn(2.0, f));
    dk = (double)k;
    const double z = __dmul_rn(s, s);
    i = hx - 0x6147a;
    const double w = __dmul_rn(z, z);
    const int j = 0x6b851 - hx;
    const double t1 = __dmul_rn(w, __dadd_rn(Lg2, __dmul_rn(w, __dadd_rn(Lg4, __dmul_rn(w, Lg6)))));
    const double t2 = __dmul_rn(z, __dadd_rn(Lg1, __dmul_rn(w, __dadd_rn(Lg3, __dmul_rn(w, __dadd_rn(Lg5, __dmul_rn(w, Lg7)))))));
    i |= j;
    const double R = __dadd_rn(t2, t1);
    if (i > 0) {
        const double hfsq = __dmul_rn(__dmul_rn(0.5, f), f);
        if (k == 0) return __dsub_rn(f, __dsub_rn(hfsq, __dmul_rn(s, __dadd_rn(hfsq, R))));
        return __dsub_rn(__dmul_rn(dk, ln2_hi), __dsub_rn(__dsub_rn(hfsq, __dadd_rn(__dmul_rn(s, __dadd_rn(hfsq, R)), __dmul_rn(dk, ln2_lo))), f));
    }
    if (k == 0) return __dsub_rn(f, __dmul_rn(s, __dsub_rn(f, R)));
    return __dsub_rn(__dmul_rn(dk, ln2_hi), __dsub_rn(__dsub_rn(__dmul_rn(s, __dsub_rn(f, R)), __dmul_rn(dk, ln2_lo)), f));
}

// Maths.logistic (Maths.java:127-129) with StrictMath.exp
__device__ __forceinline__ double bx_logistic(double x) { return __ddiv_rn(1.0, __dadd_rn(1.0, bx_exp(-x))); }

__device__ __forceinline__ unsigned int bx_ld_acquire(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void bx_red_release(unsigned int* p) {
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(p) : "memory");
}

#define LRK_BPR_REF_WARPS 8
#define LRK_BPR_REF_ROWS (LRK_MAX_FACTORS / 32)     // factors per lane

struct BprRefParams {
    const int32_t* __restrict__ samp;     // 3 n: u, i, j in sample order
    const int32_t* __restrict__ seq;      // 3 n: the sample's sequence number on rows u, U + i, U + j
    int64_t n;
    double* P; double* Q;
    int k; int32_t U;
    double lr, reg_u, reg_i;
    unsigned int* done;
    unsigned long long* claim;
    int* abort;
    long long spin_limit;
    double* loss;
};

__global__ void __launch_bounds__(32 * LRK_BPR_REF_WARPS) bpr_ref_update_kernel(BprRefParams p) {
    extern __shared__ double bx_smem[];
    const int lane = threadIdx.x & 31;
    double* prod = bx_smem + (size_t)(threadIdx.x >> 5) * 2 * p.k;     // this warp's q_i.p_u and q_j.p_u products
    const int k = p.k;
    double loss_acc = 0.0;
    for (;;) {
        unsigned long long s = 0;
        if (lane == 0) s = *(volatile int*)p.abort ? (unsigned long long)p.n : atomicAdd(p.claim, 1ULL);
        s = __shfl_sync(0xffffffffu, s, 0);
        if (s >= (unsigned long long)p.n) break;
        const int32_t u = p.samp[3 * s], i = p.samp[3 * s + 1], j = p.samp[3 * s + 2];
        // lanes 0..2 wait for rows u, U + i, U + j: every earlier sample on the row has released it
        bool failed = false;
        if (lane < 3) {
            const unsigned int* c = p.done + (lane == 0 ? (int64_t)u : (int64_t)p.U + (lane == 1 ? i : j));
            const unsigned int want = (unsigned int)p.seq[3 * s + lane];
            const long long t0 = clock64();
            while (bx_ld_acquire(c) < want) {
                if (*(volatile int*)p.abort) { failed = true; break; }
                if (clock64() - t0 > p.spin_limit) { atomicExch(p.abort, 1); failed = true; break; }
            }
        }
        if (__any_sync(0xffffffffu, failed)) break;
        double* pu = p.P + (int64_t)u * k;
        double* qi = p.Q + (int64_t)i * k;
        double* qj = p.Q + (int64_t)j * k;
        double uf[LRK_BPR_REF_ROWS], pf[LRK_BPR_REF_ROWS], nf[LRK_BPR_REF_ROWS];
#pragma unroll
        for (int r = 0; r < LRK_BPR_REF_ROWS; ++r) {
            const int f = lane + 32 * r;
            if (f < k) {
                uf[r] = __ldcg(pu + f); pf[r] = __ldcg(qi + f); nf[r] = __ldcg(qj + f);
                prod[f] = __dmul_rn(pf[r], uf[r]);
                prod[k + f] = __dmul_rn(nf[r], uf[r]);
            }
        }
        __syncwarp();
        // DenseVector.dot: one left-to-right chain from 0.0 each (every lane computes it, so no broadcast follows)
        double dp = 0.0, dn = 0.0;
        for (int f = 0; f < k; ++f) { dp = __dadd_rn(dp, prod[f]); dn = __dadd_rn(dn, prod[k + f]); }
        __syncwarp();                                                      // prod is rewritten by the next sample
        const double diff = __dsub_rn(dp, dn);
        const double deri = bx_logistic(-diff);                            // BPRRecommender.java:77-78
        if (lane == 0) loss_acc = __dadd_rn(loss_acc, -bx_log(bx_logistic(diff)));
#pragma unroll
        for (int r = 0; r < LRK_BPR_REF_ROWS; ++r) {
            const int f = lane + 32 * r;
            if (f < k) {
                // :80-88  p_u += lr * (deri * (q_i - q_j) - regU * p_u) ; q_i += lr * (deri * p_u - regI * q_i) ;
                //         q_j += lr * (deri * (-p_u) - regI * q_j) ; loss += regU p_u^2 + regI q_i^2 + regI q_j^2
                __stcg(pu + f, __dadd_rn(uf[r], __dmul_rn(p.lr, __dsub_rn(__dmul_rn(deri, __dsub_rn(pf[r], nf[r])), __dmul_rn(p.reg_u, uf[r])))));
                __stcg(qi + f, __dadd_rn(pf[r], __dmul_rn(p.lr, __dsub_rn(__dmul_rn(deri, uf[r]), __dmul_rn(p.reg_i, pf[r])))));
                __stcg(qj + f, __dadd_rn(nf[r], __dmul_rn(p.lr, __dsub_rn(__dmul_rn(deri, -uf[r]), __dmul_rn(p.reg_i, nf[r])))));
                loss_acc = __dadd_rn(loss_acc, __dadd_rn(__dadd_rn(__dmul_rn(__dmul_rn(p.reg_u, uf[r]), uf[r]),
                                                                   __dmul_rn(__dmul_rn(p.reg_i, pf[r]), pf[r])),
                                                         __dmul_rn(__dmul_rn(p.reg_i, nf[r]), nf[r])));
            }
        }
        __threadfence();
        __syncwarp();
        if (lane < 3) bx_red_release(p.done + (lane == 0 ? (int64_t)u : (int64_t)p.U + (lane == 1 ? i : j)));
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) loss_acc = __dadd_rn(loss_acc, __shfl_xor_sync(0xffffffffu, loss_acc, m));
    if (lane == 0) atomicAdd(p.loss, loss_acc);
}

// sequence numbers: the stable sort of the keys (row, sample) puts the samples of a row in sample order
__global__ void bpr_ref_keys_kernel(const int32_t* __restrict__ samp, int64_t n3, int32_t U, uint32_t* __restrict__ keys,
                                    uint32_t* __restrict__ vals) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n3) return;
    keys[t] = (uint32_t)samp[t] + (t % 3 == 0 ? 0u : (uint32_t)U);
    vals[t] = (uint32_t)t;
}
__global__ void bpr_ref_row_start_kernel(const uint32_t* __restrict__ keys, int64_t n3, int32_t* __restrict__ row_start) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n3 && (t == 0 || keys[t] != keys[t - 1])) row_start[keys[t]] = (int32_t)t;
}
__global__ void bpr_ref_seq_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, int64_t n3,
                                   const int32_t* __restrict__ row_start, int32_t* __restrict__ seq) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n3) seq[vals[t]] = (int32_t)t - row_start[keys[t]];
}

// set_train_csr: which users can be drawn, and the draws a sample takes on average (sizes the first stream)
static void bpr_ref_stage(BprRefState* b, int32_t U, int32_t I, const int64_t* rowptr) {
    int64_t drawable = 0;
    double neg = 0.0;
    for (int32_t u = 0; u < U; ++u) {
        const int64_t len = rowptr[u + 1] - rowptr[u];
        if (len > 0 && len < I) { ++drawable; neg += (double)I / (double)(I - len); }
    }
    b->drawable = drawable;
    b->L = 0;
    b->draws_per_sample = drawable ? (double)U / (double)drawable + 1.0 + neg / (double)drawable + 0.1 : 3.2;
}

// one epoch: the draw stage, the sequence numbers, the update kernel.  *end_out = draws consumed (the caller advances the state)
static int bpr_ref_epoch(lrk_handle_s* h, BprRefState* b, float lr, float reg_u, float reg_i, int64_t* end_out) {
    cudaStream_t st = h->stream;
    const int64_t n = h->nnz, n3 = 3 * n;
    *end_out = 0;
    if (n == 0) return LRK_OK;
    LRK_REQUIRE(h, n3 < (int64_t)0x7fffffffLL, "BPR reference order: 3 * numRates must stay below 2^31 (the sequence sort takes an int count)");
    int rc;
    if ((rc = lrk_dev_alloc(h, &b->d_samp, (size_t)n3))) return rc;
    if ((rc = bpr_ref_draw(h, b, 0, n, b->d_samp, end_out))) return rc;
    const int64_t rows = (int64_t)h->U + h->I;
    int bits = 1;
    while (bits < 32 && (1LL << bits) < rows) ++bits;
    size_t tb = 0;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, tb, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr,
                                                (int)n3, 0, bits, st));
    if ((rc = lrk_dev_alloc(h, &b->d_keys, (size_t)n3)) || (rc = lrk_dev_alloc(h, &b->d_keys2, (size_t)n3)) ||
        (rc = lrk_dev_alloc(h, &b->d_vals, (size_t)n3)) || (rc = lrk_dev_alloc(h, &b->d_vals2, (size_t)n3)) ||
        (rc = lrk_dev_alloc(h, &b->d_seq, (size_t)n3)) || (rc = lrk_dev_alloc(h, &b->d_row_start, (size_t)rows)) ||
        (rc = lrk_dev_alloc(h, &b->d_sort_tmp, tb)) || (rc = lrk_dev_alloc(h, &b->d_done, (size_t)rows)) ||
        (rc = lrk_dev_alloc(h, &b->d_claim, 1)) || (rc = lrk_dev_alloc(h, &b->d_abort, 1)))
        return rc;
    const int nb = lrk_ceil_div(n3, 256);
    bpr_ref_keys_kernel<<<nb, 256, 0, st>>>(b->d_samp, n3, h->U, b->d_keys, b->d_vals); LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(b->d_sort_tmp.ptr, tb, b->d_keys.ptr, b->d_keys2.ptr, b->d_vals.ptr, b->d_vals2.ptr,
                                                (int)n3, 0, bits, st));
    h->launches++;
    bpr_ref_row_start_kernel<<<nb, 256, 0, st>>>(b->d_keys2, n3, b->d_row_start); LRK_LAUNCH_CHECK(h);
    bpr_ref_seq_kernel<<<nb, 256, 0, st>>>(b->d_keys2, b->d_vals2, n3, b->d_row_start, b->d_seq); LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaMemsetAsync(b->d_done, 0, sizeof(unsigned int) * (size_t)rows, st));
    LRK_CUDA(h, cudaMemsetAsync(b->d_claim, 0, sizeof(unsigned long long), st));
    LRK_CUDA(h, cudaMemsetAsync(b->d_abort, 0, sizeof(int), st));
    BprRefParams p;
    memset(&p, 0, sizeof p);
    p.samp = b->d_samp; p.seq = b->d_seq; p.n = n; p.P = h->P64; p.Q = h->Q64; p.k = h->k; p.U = h->U;
    p.lr = (double)lr; p.reg_u = (double)reg_u; p.reg_i = (double)reg_i;
    p.done = b->d_done; p.claim = b->d_claim; p.abort = b->d_abort; p.loss = h->d_loss;
    p.spin_limit = 4000000000LL;                          // ~2 s at 2 GHz: far above any wait of a correct epoch
    const size_t smem = sizeof(double) * 2 * (size_t)h->k * LRK_BPR_REF_WARPS;
    // one CTA per SM: ~1200 warps look ahead ~1200 samples, far more than the ~90 that are ready at a time on the ML-20M shape
    bpr_ref_update_kernel<<<(unsigned)h->sm_count, 32 * LRK_BPR_REF_WARPS, smem, st>>>(p);
    LRK_LAUNCH_CHECK(h);
    return LRK_OK;
}

// after the epoch has completed: a raised abort flag is an error, otherwise the generator moves past the epoch's draws
static int bpr_ref_finish(lrk_handle_s* h, BprRefState* b, int64_t end) {
    int abort_flag = 0;
    if (h->nnz > 0) LRK_CUDA(h, cudaMemcpy(&abort_flag, b->d_abort, sizeof(int), cudaMemcpyDeviceToHost));
    if (abort_flag)
        return lrk_fail(h, LRK_ERR_CUDA, "lrk_sgd_epoch", "BPR reference order: a wait for a factor row timed out; the factors are incomplete", __FILE__, __LINE__);
    b->jstate = jr_jump(b->jstate, (uint64_t)end);
    return LRK_OK;
}
