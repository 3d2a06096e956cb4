// ALS siblings of the MF path on the device (SURVEY.md 8f row N3): WRMF and eALS.
//   recommender/cf/ranking/WRMFRecommender.java:74-166  -- per row: (F^T F + reg + sum_e w_e f_e f_e^T)^-1 . sum_e (w_e + 1) f_e
//   recommender/cf/ranking/EALSRecommender.java:114-214 -- element-wise coordinate descent with the k x k caches Sq / Sp
//   math/structure/DenseMatrix.java:229-249,362-437     -- times() and the Gauss-Jordan inverse() they call
//
// Both models are deterministic: no RNG inside trainModel, and a row's update reads only the OTHER side's matrix, so the order of
// the reference's parallelStream does not matter.  That allows the strongest parity bar of the whole path: the kernels below work
// on the fp64 masters and perform every floating-point operation of the reference in the reference's order (explicit
// __dmul_rn / __dadd_rn / __dsub_rn, never an FMA; IEEE double division), so the factors are BIT-identical to the oracle's
// (tests/test_gpu_als.py).  Parallelism comes from what the reference leaves independent:
//   * Gram matrices (Y^T Y, X^T X, Sq): k^2 independent accumulation chains over the rows, one thread per entry, an 8 x 8 tile of
//     entries per CTA, the tile's columns of the rows staged through shared memory;
//   * WRMF: one CTA per row.  Thread (tr, tc) of a 16 x 16 grid keeps a TILE x TILE block of A in registers while the row's entries
//     stream through shared memory in order (each entry of A has its own chain), then the CTA runs the reference's Gauss-Jordan
//     on [A | I] in shared memory (k pivot steps, every step parallel over rows x columns) and the final W . b;
//   * eALS: one warp per row.  The sums over a row's entries are sequential in the reference, so the lanes compute the 32 terms of a
//     batch in parallel and then fold them in entry order through shuffles; the per-entry predictions live in a global scratch
//     array in CSR / CSC order.
// The rounding-order fidelity costs throughput (fp64, no FMA, sequential chains); these models are HBM/L2-light and the point here
// is the drop-in result, not a roofline -- DESIGN.md 4.4b6 has the measured epoch times next to the oracle's.
#pragma once
#include "lrk_common.cuh"
#include "staging.cuh"
#include "lrk_epoch.cuh"

struct AlsState {
    LrkBuf<double> d_val;           // weighted train values, CSR order (fp64: the weights are log / affine functions of the rating)
    LrkBuf<int64_t> d_colptr;       // the same matrix by columns: users ascending (SequentialAccessSparseMatrix.viewColumn)
    LrkBuf<int32_t> d_cusers;
    LrkBuf<double> d_cval;
    LrkBuf<double> d_gram;          // k x k
    LrkBuf<double> d_conf;          // eALS: confidences[numItems] (lrk_set_matrix "eals.confidences")
    LrkBuf<double> d_pred;          // eALS: per-entry predictions
    LrkBuf<double> d_tn, d_td;      // eALS heavy rows: per-entry terms
    LrkBuf<unsigned int> d_counter;
    bool has_conf = false;
};

#define ALS_MAX_K 112          // [A | I] of the Gauss-Jordan step must fit the 227 KB of shared memory: k (2k + 2) doubles

__global__ void als_csc_gather_kernel(const int32_t* __restrict__ perm, const int32_t* __restrict__ rows, const double* __restrict__ val, int64_t nnz,
                                      int32_t* __restrict__ cusers, double* __restrict__ cval) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nnz) return;
    const int32_t e = perm[t];
    cusers[t] = rows[e];
    cval[t] = val[e];
}
__global__ void als_iota_kernel(int32_t* __restrict__ out, int64_t n) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) out[t] = (int32_t)t;
}

// out[r][c] = sum_i M[i][c] * M[i][r] (w == nullptr; DenseMatrix.times over the transpose) or, with weights, the eALS cache
// sum_i (w[i] * M[i][max(r,c)]) * M[i][min(r,c)] (EALSRecommender.java:128-137 computes the lower triangle and mirrors it).
// One thread per entry, rows i in order: every entry is one chain of n dependent adds, so the kernel's time is that chain as long
// as the rows arrive fast enough.  A CTA owns an 8 x 8 tile of `out` and stages only the 16 columns the tile reads (columns
// r0.. and c0..), so the ceil(k/8)^2 tiles spread over the SMs and no SM has to stream whole rows; the next stage's rows travel
// in registers while the current one is consumed.
#define ALS_GRAM_TILE 8
#define ALS_GRAM_STAGE 128
__global__ void __launch_bounds__(ALS_GRAM_TILE * ALS_GRAM_TILE) als_gram_kernel(const double* __restrict__ M, int64_t n, int k, const double* __restrict__ w, double* __restrict__ out) {
    constexpr int T = ALS_GRAM_TILE, S = ALS_GRAM_STAGE, NT = T * T, W = 2 * T, NPT = S * W / NT, NPW = S / NT;
    __shared__ double rs[S * W];       // stage rows x {columns r0 .. r0+T-1, columns c0 .. c0+T-1}
    __shared__ double ws[S];
    const int tiles = (k + T - 1) / T;
    const int r0 = (blockIdx.x / tiles) * T, c0 = (blockIdx.x % tiles) * T;
    const int tid = threadIdx.x, tr = tid / T, tc = tid % T;
    const int r = r0 + tr, c = c0 + tc;
    const bool live = r < k && c < k;
    // slots of M[i][a] and M[i][b] in a staged row: a = c, b = r without weights; a = max(r, c), b = min(r, c) with them
    const int sa = (w && r > c) ? tr : T + tc, sb = (w && r > c) ? T + tc : tr;
    double pre[NPT], prew[NPW];
    auto fetch = [&](int64_t base) {
#pragma unroll
        for (int j = 0; j < NPT; ++j) {
            const int t = tid + NT * j, e = t / W, f = t % W, col = f < T ? r0 + f : c0 + f - T;
            pre[j] = (base + e < n && col < k) ? M[(base + e) * k + col] : 0.0;
        }
#pragma unroll
        for (int j = 0; j < NPW; ++j) { const int e = tid + NT * j; prew[j] = (w && base + e < n) ? w[base + e] : 0.0; }
    };
    double v = 0.0;
    if (n > 0) fetch(0);
    for (int64_t base = 0; base < n; base += S) {
        const int cnt = (int)((n - base) < S ? (n - base) : S);
        __syncthreads();
#pragma unroll
        for (int j = 0; j < NPT; ++j) rs[tid + NT * j] = pre[j];
#pragma unroll
        for (int j = 0; j < NPW; ++j) ws[tid + NT * j] = prew[j];
        __syncthreads();
        if (base + S < n) fetch(base + S);
        if (live) {
            if (w) {
#pragma unroll 8
                for (int j = 0; j < cnt; ++j) v = __dadd_rn(v, __dmul_rn(__dmul_rn(ws[j], rs[j * W + sa]), rs[j * W + sb]));
            } else {
#pragma unroll 8
                for (int j = 0; j < cnt; ++j) v = __dadd_rn(v, __dmul_rn(rs[j * W + sa], rs[j * W + sb]));
            }
        }
    }
    if (live) out[r * k + c] = v;
}

struct AlsSolveParams {
    const int64_t* ptr;       // rows of the weighted matrix (CSR for the user step, CSC for the item step)
    const int32_t* idx;
    const double* w;
    const double* F;          // the other side's factors (fixed during the step)
    const double* G;          // F^T F
    double* OUT;              // this side's factors
    double reg;
    int32_t row0;             // the rows [row0, row0 + n_rows) are solved (a device's range on a multi-device handle)
    int32_t n_rows;
    int k;
};

// entries of a row staged per step of the WRMF accumulation (shared memory next to the k x (2k + 2) Gauss-Jordan tableau)
__host__ __device__ constexpr int als_chunk(int tile) { return tile <= 4 ? 32 : (tile <= 6 ? 16 : 8); }

// WRMFRecommender.java:93-126 (users) / :129-163 (items), one CTA per row
template <int TILE>
__global__ void __launch_bounds__(256) als_wrmf_solve_kernel(AlsSolveParams p) {
    extern __shared__ double sm[];
    constexpr int KP = 16 * TILE, CH = als_chunk(TILE), NPT = (CH * KP + 255) / 256;
    const int k = p.k, S = 2 * k + 2;
    double* Mx = sm;                               // k x S: A in columns [0, k), the inverse in [k, 2k)
    double* ys = Mx + (size_t)k * S;               // CH x KP, zero padded
    double* wsh = ys + CH * KP;                    // CH
    double* bs = wsh + CH;                         // k
    double* colp = bs + k;                         // k
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tr = tid >> 4, tc = tid & 15;
    for (int32_t row = p.row0 + blockIdx.x; row < p.row0 + p.n_rows; row += gridDim.x) {
        const int64_t b0 = p.ptr[row], e0 = p.ptr[row + 1];
        double acc[TILE][TILE];
#pragma unroll
        for (int a = 0; a < TILE; ++a)
#pragma unroll
            for (int c = 0; c < TILE; ++c) {
                const int rr = tr * TILE + a, cc = tc * TILE + c;
                acc[a][c] = (rr < k && cc < k) ? __dadd_rn(p.G[rr * k + cc], p.reg) : 0.0;         // :110, the regulariser lands on EVERY entry
            }
        double bacc = 0.0;
        // the next chunk's factor rows travel in registers while the current one is consumed (a long row is a chain of dependent
        // gathers otherwise: 2 us per 8 entries)
        double pre[NPT], prew = 0.0;
        auto fetch = [&](int64_t base) {
            const int cnt = (int)((e0 - base) < CH ? (e0 - base) : CH);
#pragma unroll
            for (int j = 0; j < NPT; ++j) {
                const int t = tid + 256 * j, e = t / KP, f = t - e * KP;
                pre[j] = (t < CH * KP && e < cnt && f < k) ? p.F[(int64_t)p.idx[base + e] * k + f] : 0.0;
            }
            prew = tid < cnt ? p.w[base + tid] : 0.0;
        };
        if (b0 < e0) fetch(b0);
        for (int64_t base = b0; base < e0; base += CH) {
            const int cnt = (int)((e0 - base) < CH ? (e0 - base) : CH);
            __syncthreads();
#pragma unroll
            for (int j = 0; j < NPT; ++j) { const int t = tid + 256 * j; if (t < CH * KP) ys[t] = pre[j]; }
            if (tid < CH) wsh[tid] = prew;
            __syncthreads();
            if (base + CH < e0) fetch(base + CH);
            for (int e = 0; e < cnt; ++e) {
                const double wv = wsh[e];
                const double* y = ys + e * KP;
                double yc[TILE];
#pragma unroll
                for (int c = 0; c < TILE; ++c) yc[c] = y[tc * TILE + c];
#pragma unroll
                for (int a = 0; a < TILE; ++a) {
                    const double temp = __dmul_rn(y[tr * TILE + a], wv);                           // :118
#pragma unroll
                    for (int c = 0; c < TILE; ++c) acc[a][c] = __dadd_rn(acc[a][c], __dmul_rn(temp, yc[c]));
                }
                if (tid < k) bacc = __dadd_rn(bacc, __dmul_rn(y[tid], __dadd_rn(wv, 1.0)));         // :103-107
            }
        }
        __syncthreads();
#pragma unroll
        for (int a = 0; a < TILE; ++a)
#pragma unroll
            for (int c = 0; c < TILE; ++c) {
                const int rr = tr * TILE + a, cc = tc * TILE + c;
                if (rr < k && cc < k) Mx[rr * S + cc] = acc[a][c];
            }
        for (int t = tid; t < k * k; t += 256) { const int rr = t / k, cc = t - rr * k; Mx[rr * S + k + cc] = rr == cc ? 1.0 : 0.0; }
        if (tid < k) bs[tid] = bacc;
        __syncthreads();
        // DenseMatrix.inverse(): :362-437.  Three barriers per pivot: every warp runs the pivot search itself (same tableau, same
        // answer), the row swap and the division of the pivot row are one pass over the columns, the elimination another.
        if (k == 1) {
            if (tid == 0) Mx[k] = 1.0 / Mx[0];
        } else {
            for (int pv = 0; pv < k; ++pv) {
                double mag = 0.0;
                int best = -1;
                for (int j = pv + lane; j < k; j += 32) {
                    const double m2 = fabs(Mx[j * S + pv]);
                    if (m2 > mag) { mag = m2; best = j; }
                }
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    const double om = __shfl_xor_sync(0xffffffffu, mag, off);
                    const int oj = __shfl_xor_sync(0xffffffffu, best, off);
                    if (om > mag || (om == mag && om > 0.0 && oj < best)) { mag = om; best = oj; }       // first strictly-largest in row order
                }
                if (best == -1 || mag == 0.0) break;                                               // :393-394: the inverse as it stands
                const int piv = best;
                const double pm = Mx[piv * S + pv];                                                // :412, read after the swap in the reference
                // elimination factors of the rows as they stand AFTER the swap (:421); colp[pv] is not used
                for (int r2 = tid; r2 < k; r2 += 256) colp[r2] = Mx[(r2 == piv ? pv : r2) * S + pv];
                __syncthreads();
                for (int c = pv + tid; c < 2 * k; c += 256) {                                       // :397-410 swap, :412-417 normalise
                    const double a = Mx[piv * S + c];
                    if (piv != pv) Mx[piv * S + c] = Mx[pv * S + c];
                    Mx[pv * S + c] = a / pm;
                }
                __syncthreads();
                double prow[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) { const int c = pv + lane + 32 * j; prow[j] = c < 2 * k ? Mx[pv * S + c] : 0.0; }
                for (int r2 = warp; r2 < k; r2 += 8) {
                    if (r2 == pv) continue;
                    const double m2 = colp[r2];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int c = pv + lane + 32 * j;
                        if (c < 2 * k) Mx[r2 * S + c] = __dsub_rn(Mx[r2 * S + c], __dmul_rn(m2, prow[j]));
                    }
                }
                __syncthreads();
            }
        }
        __syncthreads();
        if (tid < k) {                                                                              // Wu.times(YtCuPu): row(a).dot(b)
            double v = 0.0;
            for (int c = 0; c < k; ++c) v = __dadd_rn(v, __dmul_rn(bs[c], Mx[tid * S + k + c]));
            p.OUT[(int64_t)row * k + tid] = v;
        }
        __syncthreads();
    }
}

struct AlsEalsParams {
    const int64_t* ptr;
    const int32_t* idx;
    const double* w;
    double* Fself;            // the side being updated, in place
    const double* Fother;
    const double* S;          // Sq (user step) or Sp (item step), k x k
    const double* conf;       // confidences[numItems]
    double* pred;             // per-entry scratch in the order of ptr / idx
    double* tn;               // heavy rows: the per-entry terms of numer / denom (same order)
    double* td;
    unsigned int* counter;    // heavy rows: dynamic row scheduler
    double reg;
    int32_t n_rows;
    int k;
    int heavy;                // rows with more entries take the CTA-per-row kernel
};

// EALSRecommender.java:139-171 (ITEM_STEP false) / :175-209 (true), one warp per row; rows with more than p.heavy entries are
// left to als_eals_heavy_kernel (a lone warp walking 10^5 entries k times is latency bound: 112 cycles per entry and factor)
template <bool ITEM_STEP>
__global__ void __launch_bounds__(256) als_eals_side_kernel(AlsEalsParams p) {
    extern __shared__ double sm[];
    const int k = p.k, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* own = sm + warp * k;
    double* f1 = sm + 8 * k + warp * 64;           // the 32 numer / denom terms of a batch
    double* f2s = f1 + 32;
    const int64_t stride = (int64_t)gridDim.x * 8;
    for (int64_t row = (int64_t)blockIdx.x * 8 + warp; row < p.n_rows; row += stride) {
        const int64_t b = p.ptr[row], e = p.ptr[row + 1];
        if (e - b > p.heavy) continue;
        __syncwarp();
        for (int f = lane; f < k; f += 32) own[f] = p.Fself[row * k + f];
        __syncwarp();
        for (int64_t x = b + lane; x < e; x += 32) {
            const double* o = p.Fother + (int64_t)p.idx[x] * k;
            double d = 0.0;
            for (int f = 0; f < k; ++f) d = __dadd_rn(d, __dmul_rn(o[f], own[f]));
            p.pred[x] = d;
        }
        const double c_row = ITEM_STEP ? p.conf[row] : 0.0;
        for (int f = 0; f < k; ++f) {
            double numer = 0.0;
            for (int f2 = 0; f2 < k; ++f2)
                if (f2 != f) numer = __dsub_rn(numer, __dmul_rn(own[f2], ITEM_STEP ? p.S[f2 * k + f] : p.S[f * k + f2]));
            double denom;
            if (ITEM_STEP) { numer = __dmul_rn(numer, c_row); denom = __dadd_rn(__dmul_rn(c_row, p.S[f * k + f]), p.reg); }
            else denom = __dadd_rn(p.reg, p.S[f * k + f]);
            const double of = own[f];
            for (int64_t base = b; base < e; base += 32) {
                const int64_t x = base + lane;
                double tn = 0.0, td = 0.0;
                if (x < e) {
                    const int32_t o = p.idx[x];
                    const double wv = p.w[x], qf = p.Fother[(int64_t)o * k + f];
                    const double c = ITEM_STEP ? c_row : p.conf[o];
                    const double pm = __dsub_rn(p.pred[x], __dmul_rn(of, qf));
                    p.pred[x] = pm;
                    const double wc = __dsub_rn(wv, c);
                    tn = __dmul_rn(__dsub_rn(wv, __dmul_rn(wc, pm)), qf);
                    td = __dmul_rn(__dmul_rn(wc, qf), qf);
                }
                const int cnt = (int)((e - base) < 32 ? (e - base) : 32);
                __syncwarp();
                f1[lane] = tn; f2s[lane] = td;                     // fold in entry order: broadcast reads, the adds are the only chain
                __syncwarp();
                for (int l = 0; l < cnt; ++l) {
                    numer = __dadd_rn(numer, f1[l]);
                    denom = __dadd_rn(denom, f2s[l]);
                }
            }
            const double nf = numer / denom;
            __syncwarp();
            if (lane == 0) own[f] = nf;
            __syncwarp();
            for (int64_t x = b + lane; x < e; x += 32) p.pred[x] = __dadd_rn(p.pred[x], __dmul_rn(nf, p.Fother[(int64_t)p.idx[x] * k + f]));
        }
        __syncwarp();
        for (int f = lane; f < k; f += 32) p.Fself[row * k + f] = own[f];
    }
}

// the same update for one HEAVY row per CTA.  Per factor: all 256 threads compute the entries' terms in parallel (together with the
// prediction update the previous factor left open), then warp 0 folds them in entry order -- the only sequential part, ~8 cycles per
// entry and factor.  Rows are handed out by an atomic counter so that the few very long rows do not queue behind each other.
template <bool ITEM_STEP>
__global__ void __launch_bounds__(256) als_eals_heavy_kernel(AlsEalsParams p) {
    __shared__ double own[LRK_MAX_FACTORS];
    __shared__ double s_t1[128], s_t2[128];
    __shared__ double s_nf;
    __shared__ unsigned int s_row;
    const int k = p.k, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_row = atomicAdd(p.counter, 1u);
        __syncthreads();
        const int64_t row = s_row;
        if (row >= p.n_rows) break;
        const int64_t b = p.ptr[row], e = p.ptr[row + 1];
        if (e - b <= p.heavy) continue;
        for (int f = tid; f < k; f += 256) own[f] = p.Fself[row * k + f];
        __syncthreads();
        for (int64_t x = b + tid; x < e; x += 256) {
            const double* o = p.Fother + (int64_t)p.idx[x] * k;
            double d = 0.0;
            for (int f = 0; f < k; ++f) d = __dadd_rn(d, __dmul_rn(o[f], own[f]));
            p.pred[x] = d;
        }
        const double c_row = ITEM_STEP ? p.conf[row] : 0.0;
        double nf_prev = 0.0;
        for (int f = 0; f < k; ++f) {
            __syncthreads();
            const double of = own[f];
            for (int64_t x = b + tid; x < e; x += 256) {
                const int32_t o = p.idx[x];
                const double* orow = p.Fother + (int64_t)o * k;
                const double qf = orow[f];
                double pr = p.pred[x];
                if (f > 0) pr = __dadd_rn(pr, __dmul_rn(nf_prev, orow[f - 1]));        // the previous factor's "+= new * q" (:165-168)
                const double pm = __dsub_rn(pr, __dmul_rn(of, qf));
                p.pred[x] = pm;
                const double wv = p.w[x];
                const double c = ITEM_STEP ? c_row : p.conf[o];
                const double wc = __dsub_rn(wv, c);
                p.tn[x] = __dmul_rn(__dsub_rn(wv, __dmul_rn(wc, pm)), qf);
                p.td[x] = __dmul_rn(__dmul_rn(wc, qf), qf);
            }
            __syncthreads();
            if (warp == 0) {
                double numer = 0.0;
                for (int f2 = 0; f2 < k; ++f2)
                    if (f2 != f) numer = __dsub_rn(numer, __dmul_rn(own[f2], ITEM_STEP ? p.S[f2 * k + f] : p.S[f * k + f2]));
                double denom;
                if (ITEM_STEP) { numer = __dmul_rn(numer, c_row); denom = __dadd_rn(__dmul_rn(c_row, p.S[f * k + f]), p.reg); }
                else denom = __dadd_rn(p.reg, p.S[f * k + f]);
                // ordered fold: 128 terms at a time go through shared memory (broadcast reads; the two add chains are the only
                // dependency), the next 128 are already in flight in registers
                double t1[4], t2[4];
                auto fetch = [&](int64_t base) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int64_t x = base + 32 * j + lane;
                        t1[j] = x < e ? p.tn[x] : 0.0;
                        t2[j] = x < e ? p.td[x] : 0.0;
                    }
                };
                fetch(b);
                for (int64_t base = b; base < e; base += 128) {
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 4; ++j) { s_t1[32 * j + lane] = t1[j]; s_t2[32 * j + lane] = t2[j]; }
                    __syncwarp();
                    if (base + 128 < e) fetch(base + 128);
                    const int cnt = (int)((e - base) < 128 ? (e - base) : 128);
                    if (cnt == 128) {
#pragma unroll 16
                        for (int j = 0; j < 128; ++j) { numer = __dadd_rn(numer, s_t1[j]); denom = __dadd_rn(denom, s_t2[j]); }
                    } else {
                        for (int j = 0; j < cnt; ++j) { numer = __dadd_rn(numer, s_t1[j]); denom = __dadd_rn(denom, s_t2[j]); }
                    }
                }
                const double nf = numer / denom;
                if (lane == 0) { own[f] = nf; s_nf = nf; }
            }
            __syncthreads();
            nf_prev = s_nf;
        }
        // (the last factor's prediction update is not needed: predictions are re-initialised per row, :141-145)
        __syncthreads();
        for (int f = tid; f < k; f += 256) p.Fself[row * k + f] = own[f];
    }
}

// the train matrix by columns + the fp64 values (lrk_set_train_csr tail for WRMF / eALS)
static int als_stage(lrk_handle_s* h, const double* h_val) {
    cudaStream_t st = h->stream;
    if (!h->als) h->als.reset(new AlsState());
    AlsState* a = h->als.get();
    a->has_conf = false;               // confidences belong to a train matrix (EALSRecommender.java:65-83)
    const int64_t nnz = h->nnz;
    const int32_t U = h->U, I = h->I;
    int rc;
    if ((rc = lrk_dev_alloc(h, &a->d_val, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &a->d_colptr, (size_t)I + 1))) return rc;
    if ((rc = lrk_dev_alloc(h, &a->d_cusers, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &a->d_cval, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &a->d_gram, (size_t)h->k * h->k))) return rc;
    if (h->cfg.model == LRK_MODEL_EALS) {
        if ((rc = lrk_dev_alloc(h, &a->d_pred, (size_t)nnz))) return rc;
        if ((rc = lrk_dev_alloc(h, &a->d_tn, (size_t)nnz))) return rc;
        if ((rc = lrk_dev_alloc(h, &a->d_td, (size_t)nnz))) return rc;
        if ((rc = lrk_dev_alloc(h, &a->d_counter, 1))) return rc;
    }
    if (nnz == 0) { LRK_CUDA(h, cudaMemsetAsync(a->d_colptr, 0, sizeof(int64_t) * ((size_t)I + 1), st)); return LRK_OK; }
    LRK_CUDA(h, cudaMemcpyAsync(a->d_val, h_val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, st));
    size_t tb_sort = 0, tb_scan = 0;
    int end_bit = 1;
    while (end_bit < 32 && ((int64_t)1 << end_bit) < (int64_t)I) ++end_bit;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, tb_sort, (uint32_t*)nullptr, (uint32_t*)nullptr, (int32_t*)nullptr, (int32_t*)nullptr, (int)nnz, 0, end_bit, st));
    LRK_CUDA(h, cub::DeviceScan::ExclusiveSum(nullptr, tb_scan, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)I, st));
    const size_t tb = std::max(tb_sort, tb_scan) + 256;
    LrkScratch sc;
    if ((rc = lrk_scratch_begin(h, (size_t)nnz * 20 + (size_t)I * 8 + tb + 16 * 256, &sc))) return rc;
    uint32_t *k_in = sc.take<uint32_t>((size_t)nnz), *k_out = sc.take<uint32_t>((size_t)nnz);
    int32_t *rows = sc.take<int32_t>((size_t)nnz), *iota = sc.take<int32_t>((size_t)nnz), *perm = sc.take<int32_t>((size_t)nnz);
    uint32_t *deg = sc.take<uint32_t>((size_t)I), *deg_ex = sc.take<uint32_t>((size_t)I);
    void* tmp = sc.take<char>(tb);
    if (!k_in || !k_out || !rows || !iota || !perm || !deg || !deg_ex || !tmp) return lrk_fail(h, LRK_ERR_NOMEM, "als_stage", "scratch arena too small", __FILE__, __LINE__);
    const int nb = lrk_ceil_div(nnz, 256);
    coo_rows_kernel<<<nb, 256, 0, st>>>(h->d_rowptr, U, nnz, rows); LRK_LAUNCH_CHECK(h);
    als_iota_kernel<<<nb, 256, 0, st>>>(iota, nnz); LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaMemcpyAsync(k_in, h->d_col, sizeof(uint32_t) * (size_t)nnz, cudaMemcpyDeviceToDevice, st));
    LRK_CUDA(h, cudaMemsetAsync(deg, 0, sizeof(uint32_t) * (size_t)I, st));
    item_degree_kernel<<<nb, 256, 0, st>>>(h->d_col, nnz, deg); LRK_LAUNCH_CHECK(h);
    size_t t1 = tb;
    LRK_CUDA(h, cub::DeviceScan::ExclusiveSum(tmp, t1, deg, deg_ex, (int)I, st));
    gbpr_colptr_kernel<<<lrk_ceil_div(I, 256), 256, 0, st>>>(deg_ex, deg, I, a->d_colptr); LRK_LAUNCH_CHECK(h);
    t1 = tb;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(tmp, t1, k_in, k_out, iota, perm, (int)nnz, 0, end_bit, st));   // stable: users ascending within an item
    als_csc_gather_kernel<<<nb, 256, 0, st>>>(perm, rows, a->d_val, nnz, a->d_cusers, a->d_cval); LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaStreamSynchronize(st));
    h->launches += 6;
    return LRK_OK;
}

static int als_gram(lrk_handle_s* h, const double* M, int64_t n, const double* w, double* out) {
    const int tiles = lrk_ceil_div(h->k, ALS_GRAM_TILE);
    als_gram_kernel<<<tiles * tiles, ALS_GRAM_TILE * ALS_GRAM_TILE, 0, h->stream>>>(M, n, h->k, w, out);
    LRK_LAUNCH_CHECK(h);
    h->launches++;
    return LRK_OK;
}

template <int TILE>
static int als_wrmf_launch(lrk_handle_s* h, const AlsSolveParams& p) {
    const int k = p.k;
    const size_t smem = sizeof(double) * ((size_t)k * (2 * k + 2) + (size_t)als_chunk(TILE) * 16 * TILE + als_chunk(TILE) + 2 * (size_t)k);
    LRK_CUDA(h, cudaFuncSetAttribute(als_wrmf_solve_kernel<TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    LRK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, als_wrmf_solve_kernel<TILE>, 256, smem));
    LRK_REQUIRE(h, per_sm >= 1, "WRMF solve kernel does not fit the SM");
    int64_t grid = (int64_t)h->sm_count * per_sm;
    if (grid > p.n_rows) grid = p.n_rows;
    if (grid < 1) return LRK_OK;
    als_wrmf_solve_kernel<TILE><<<(unsigned)grid, 256, smem, h->stream>>>(p);
    LRK_LAUNCH_CHECK(h);
    h->launches++;
    return LRK_OK;
}

static int als_wrmf_side(lrk_handle_s* h, const AlsSolveParams& p) {
    switch ((p.k + 15) / 16) {
        case 1: return als_wrmf_launch<1>(h, p);
        case 2: return als_wrmf_launch<2>(h, p);
        case 3: return als_wrmf_launch<3>(h, p);
        case 4: return als_wrmf_launch<4>(h, p);
        case 5: return als_wrmf_launch<5>(h, p);
        case 6: return als_wrmf_launch<6>(h, p);
        case 7: return als_wrmf_launch<7>(h, p);
        default: return lrk_fail(h, LRK_ERR_INVALID, "lrk_sgd_epoch", "WRMF on the device needs rec.factor.number <= 112", __FILE__, __LINE__);
    }
}

template <bool ITEM_STEP>
static int als_eals_side(lrk_handle_s* h, const AlsEalsParams& p) {
    const size_t smem = sizeof(double) * (8 * (size_t)p.k + 8 * 64);
    int per_sm = 0;
    LRK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, als_eals_side_kernel<ITEM_STEP>, 256, smem));
    int64_t grid = (int64_t)h->sm_count * (per_sm < 1 ? 1 : per_sm);
    const int64_t need = ((int64_t)p.n_rows + 7) / 8;
    if (need < grid) grid = need;
    if (grid < 1) return LRK_OK;
    als_eals_side_kernel<ITEM_STEP><<<(unsigned)grid, 256, smem, h->stream>>>(p);
    LRK_LAUNCH_CHECK(h);
    h->launches++;
    // rows above the threshold: one CTA each
    LRK_CUDA(h, cudaMemsetAsync(p.counter, 0, sizeof(unsigned int), h->stream));
    LRK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, als_eals_heavy_kernel<ITEM_STEP>, 256, 0));
    grid = (int64_t)h->sm_count * (per_sm < 1 ? 1 : per_sm);
    if (grid > p.n_rows) grid = p.n_rows;
    als_eals_heavy_kernel<ITEM_STEP><<<(unsigned)grid, 256, 0, h->stream>>>(p);
    LRK_LAUNCH_CHECK(h);
    h->launches++;
    return LRK_OK;
}

// the Gram matrix a WRMF half-iteration reads: Q^T Q before the user side, P^T P before the item side
static int als_wrmf_gram(lrk_handle_s* h, bool item_side) {
    return item_side ? als_gram(h, h->P64, h->U, nullptr, h->als->d_gram) : als_gram(h, h->Q64, h->I, nullptr, h->als->d_gram);
}

// the user side (rows of the CSR, solved against Q) or the item side (rows of the CSC, solved against P), rows [row0, row0 + n_rows)
static AlsSolveParams als_wrmf_params(lrk_handle_s* h, bool item_side, float reg, int32_t row0, int32_t n_rows) {
    AlsState* a = h->als.get();
    AlsSolveParams p;
    memset(&p, 0, sizeof p);
    p.k = h->k; p.G = a->d_gram; p.reg = (double)reg; p.row0 = row0; p.n_rows = n_rows;
    if (item_side) { p.ptr = a->d_colptr; p.idx = a->d_cusers; p.w = a->d_cval; p.F = h->P64; p.OUT = h->Q64; }
    else { p.ptr = h->d_rowptr; p.idx = h->d_col; p.w = a->d_val; p.F = h->Q64; p.OUT = h->P64; }
    return p;
}

// keep the fp32 working copies in step (nothing on the ALS path reads them, the scoring entry points use the masters)
static int als_refresh_f32(lrk_handle_s* h) {
    cudaStream_t st = h->stream;
    f64_to_f32_rows_kernel<<<lrk_ceil_div((int64_t)h->U * h->ld, 256), 256, 0, st>>>(h->P64, h->P32, h->U, h->k, h->ld); LRK_LAUNCH_CHECK(h);
    f64_to_f32_rows_kernel<<<lrk_ceil_div((int64_t)h->I * h->ld, 256), 256, 0, st>>>(h->Q64, h->Q32, h->I, h->k, h->ld); LRK_LAUNCH_CHECK(h);
    return LRK_OK;
}

// one iteration of WRMFRecommender.trainModel / EALSRecommender.trainModel on the fp64 masters; the models have no loss (0 is returned)
static int als_epoch(lrk_handle_s* h, float reg_u, float reg_i, double* loss_out) {
    AlsState* a = h->als.get();
    LRK_REQUIRE(h, a != nullptr, "ALS state missing: call lrk_set_train_csr first");
    const bool eals = h->cfg.model == LRK_MODEL_EALS;
    LRK_REQUIRE(h, !eals || a->has_conf, "eALS needs the item confidences: lrk_set_matrix(h, \"eals.confidences\", c)");
    LRK_REQUIRE(h, h->f64_valid, "internal: fp64 masters out of date");
    LrkEpoch e;
    e.enqueue = [&](int) -> int {
        const int k = h->k;
        int rc;
        if (!eals) {
            if ((rc = als_wrmf_gram(h, false)) || (rc = als_wrmf_side(h, als_wrmf_params(h, false, reg_u, 0, h->U)))) return rc;
            if ((rc = als_wrmf_gram(h, true)) || (rc = als_wrmf_side(h, als_wrmf_params(h, true, reg_i, 0, h->I)))) return rc;
        } else {
            AlsEalsParams p;
            memset(&p, 0, sizeof p);
            p.k = k; p.S = a->d_gram; p.conf = a->d_conf; p.pred = a->d_pred; p.tn = a->d_tn; p.td = a->d_td; p.counter = a->d_counter;
            {
                const char* env = getenv("LRK_EALS_HEAVY");          // test hook: a small value sends the rows of small matrices down the CTA-per-row path
                p.heavy = env && atoi(env) > 0 ? atoi(env) : 512;
            }
            if ((rc = als_gram(h, h->Q64, h->I, a->d_conf, a->d_gram))) return rc;
            p.ptr = h->d_rowptr; p.idx = h->d_col; p.w = a->d_val; p.Fself = h->P64; p.Fother = h->Q64; p.reg = (double)reg_u; p.n_rows = h->U;
            if ((rc = als_eals_side<false>(h, p))) return rc;
            if ((rc = als_gram(h, h->P64, h->U, nullptr, a->d_gram))) return rc;
            p.ptr = a->d_colptr; p.idx = a->d_cusers; p.w = a->d_cval; p.Fself = h->Q64; p.Fother = h->P64; p.reg = (double)reg_i; p.n_rows = h->I;
            if ((rc = als_eals_side<true>(h, p))) return rc;
        }
        return als_refresh_f32(h);
    };
    return lrk_epoch(h, e, loss_out);             // loss 0: trainModel never assigns `loss` in either class
}
