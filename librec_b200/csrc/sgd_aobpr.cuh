// AoBPR host side (SURVEY.md 8f row N3): recommender/cf/ranking/AoBPRRecommender.java:60-200 -- BPR with adaptive oversampling of
// the negative item (Rendle & Freudenthaler, WSDM'14).  The update is BPR's (sgd_bpr_epoch_kernel, sampler aobpr_draw in sgd.cuh);
// what this file adds is the state the sampler reads and its refresh:
//   * rankingPro (:70-78): p(r) = exp(-((r + 1) / lambda)) / sum with INTEGER division (lambda = (int)(rec.item.distribution.parameter *
//     numItems)), kept as an inclusive cumulative array;
//   * updateRankingInFactor (:186-200) every loopNumber = (int)(numItems * ln numItems) samples, counted ACROSS iterations (:92-97):
//     per factor the items sorted by descending factor value (stable: ties keep ascending item id) and the population variance of
//     the column.  On the device: one stable radix sort of (factor : value-descending) keys over k * I elements + one variance
//     kernel, between WINDOWS of the epoch -- an epoch of n samples is ceil(n / loopNumber) launches of the BPR kernel.
#pragma once
#include "lrk_common.cuh"
#include "sgd.cuh"
#include <cub/cub.cuh>
#include <cmath>
#include <vector>

struct AobprState {
    LrkBuf<int32_t> d_rank;        // [ld][I]
    LrkBuf<float> d_var;           // [ld] (padded factors: 0)
    LrkBuf<float> d_cum;           // [I]
    LrkBuf<uint64_t> d_keys, d_keys2;
    LrkBuf<int32_t> d_vals;
    LrkBuf<char> d_tmp; size_t tmp_bytes = 0;
    int32_t I = 0; int ld = 0;
    float dist_param = 0.f;        // rec.item.distribution.parameter (no default in the reference: setup() throws without it)
    int32_t lambda = 0, loop = 0;
    int64_t count = 0;             // countIter (:92-97)
};
// key of (item i, factor f): f in the high word, the factor value mapped to an unsigned that sorts DESCENDING in the low word
__global__ void aobpr_keys_kernel(const float* __restrict__ Q, int32_t I, int ld, int k, uint64_t* __restrict__ keys, int32_t* __restrict__ vals) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)I * k) return;
    const int f = (int)(t / I);
    const int32_t i = (int32_t)(t - (int64_t)f * I);
    const uint32_t b = __float_as_uint(Q[(int64_t)i * ld + f]);
    const uint32_t asc = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
    keys[t] = ((uint64_t)f << 32) | (uint64_t)(~asc);
    vals[t] = i;
}
// population variance of column f of Q (Stats.variance as used at :198): one block per factor
__global__ void aobpr_var_kernel(const float* __restrict__ Q, int32_t I, int ld, float* __restrict__ var) {
    __shared__ double s_sum[32], s_sq[32];
    const int f = blockIdx.x;
    double a = 0.0, b = 0.0;
    for (int32_t i = threadIdx.x; i < I; i += blockDim.x) { const double v = (double)Q[(int64_t)i * ld + f]; a += v; b += v * v; }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, m); b += __shfl_xor_sync(0xffffffffu, b, m); }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { s_sum[w] = a; s_sq[w] = b; }
    __syncthreads();
    if (w == 0) {
        a = l < (int)(blockDim.x >> 5) ? s_sum[l] : 0.0; b = l < (int)(blockDim.x >> 5) ? s_sq[l] : 0.0;
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, m); b += __shfl_xor_sync(0xffffffffu, b, m); }
        if (l == 0) { const double mean = a / I; var[f] = (float)fmax(b / I - mean * mean, 0.0); }
    }
}

static int aobpr_prepare(lrk_handle_s* h, AobprState* a) {
    cudaStream_t st = h->stream;
    const int32_t I = h->I;
    LRK_REQUIRE(h, a->dist_param > 0.f, "AoBPR needs rec.item.distribution.parameter: lrk_set_param(h, \"aobpr.lambda\", value)");
    a->lambda = (int32_t)(a->dist_param * (float)I);                            // AoBPRRecommender.java:63
    a->loop = (int32_t)((double)I * log((double)I));                            // :65
    LRK_REQUIRE(h, a->lambda > 0 && a->loop > 0, "rec.item.distribution.parameter * numItems must be at least 1");
    if (a->I == I && a->ld == h->ld && a->d_rank) return LRK_OK;
    const size_t n = (size_t)I * h->k;
    int rc;
    if ((rc = lrk_dev_alloc(h, &a->d_rank, (size_t)I * h->ld))) return rc;
    if ((rc = lrk_dev_alloc(h, &a->d_var, (size_t)h->ld))) return rc;
    if ((rc = lrk_dev_alloc(h, &a->d_cum, (size_t)I))) return rc;
    if ((rc = lrk_dev_alloc(h, &a->d_keys, n))) return rc;
    if ((rc = lrk_dev_alloc(h, &a->d_keys2, n))) return rc;
    if ((rc = lrk_dev_alloc(h, &a->d_vals, n))) return rc;
    a->tmp_bytes = 0;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, a->tmp_bytes, a->d_keys.ptr, a->d_keys2.ptr, a->d_vals.ptr, a->d_rank.ptr, (int)n, 0, 40, st));
    if ((rc = lrk_dev_alloc(h, &a->d_tmp, a->tmp_bytes + 16))) return rc;
    LRK_CUDA(h, cudaMemsetAsync(a->d_var, 0, sizeof(float) * (size_t)h->ld, st));
    LRK_CUDA(h, cudaMemsetAsync(a->d_rank, 0, sizeof(int32_t) * (size_t)I * h->ld, st));   // padded factors (never drawn unless p_u is all zero) rank item 0
    // cumulative rank distribution in double on the host (I values), float on the device
    std::vector<double> pro((size_t)I);
    double sum = 0.0;
    for (int32_t i = 0; i < I; ++i) { pro[(size_t)i] = exp((double)(-((i + 1) / a->lambda))); sum += pro[(size_t)i]; }
    std::vector<float> cum((size_t)I);
    double acc = 0.0;
    for (int32_t i = 0; i < I; ++i) { acc += pro[(size_t)i] / sum; cum[(size_t)i] = (float)acc; }
    cum[(size_t)I - 1] = 2.f;                                                    // the search always terminates inside the array
    LRK_CUDA(h, cudaMemcpyAsync(a->d_cum, cum.data(), sizeof(float) * (size_t)I, cudaMemcpyHostToDevice, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    a->I = I; a->ld = h->ld; a->count = 0;
    return LRK_OK;
}

// updateRankingInFactor (:186-200) on the current item factors
static int aobpr_refresh(lrk_handle_s* h, AobprState* a) {
    cudaStream_t st = h->stream;
    const int64_t n = (int64_t)h->I * h->k;
    aobpr_keys_kernel<<<lrk_ceil_div(n, 256), 256, 0, st>>>(h->Q32, h->I, h->ld, h->k, a->d_keys, a->d_vals); LRK_LAUNCH_CHECK(h);
    size_t tb = a->tmp_bytes;
    int hi_bits = 1;
    while ((1 << hi_bits) < h->k) ++hi_bits;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(a->d_tmp, tb, a->d_keys.ptr, a->d_keys2.ptr, a->d_vals.ptr, a->d_rank.ptr, (int)n, 0, 32 + hi_bits, st));
    h->launches++;
    aobpr_var_kernel<<<h->k, 256, 0, st>>>(h->Q32, h->I, h->ld, a->d_var); LRK_LAUNCH_CHECK(h);
    return LRK_OK;
}
