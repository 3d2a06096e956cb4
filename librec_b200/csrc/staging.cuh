// Staging kernels: flat CSR (what the Java shim flattens SequentialAccessSparseMatrix into,
// math/structure/SequentialAccessSparseMatrix.java:23, RowSequentialAccessSparseMatrix.java:19)
// -> device CSR + shuffled COO stream; DenseMatrix double[][] <-> padded fp32 working rows.
#pragma once
#include "lrk_common.cuh"
#include <cub/cub.cuh>

__device__ __forceinline__ uint32_t lrk_hash32(uint64_t x) {   // splitmix64 finaliser, high word
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    x ^= x >> 31;
    return (uint32_t)(x >> 32);
}

// entry e -> (row, shuffle key).  Row found by binary search in rowptr (robust to skewed rows).
__global__ void coo_expand_kernel(const int64_t* __restrict__ rowptr, int32_t U, int64_t nnz, uint64_t seed,
                                  int32_t* __restrict__ row_of, uint32_t* __restrict__ keys, uint32_t* __restrict__ idx) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    int32_t lo = 0, hi = U;
    while (hi - lo > 1) { const int32_t m = (lo + hi) >> 1; if (rowptr[m] <= e) lo = m; else hi = m; }
    row_of[e] = lo;
    keys[e] = lrk_hash32((uint64_t)e ^ (seed * 0xD6E8FEB86659FD93ull));
    idx[e] = (uint32_t)e;
}

__global__ void coo_gather_kernel(const uint32_t* __restrict__ perm, const int32_t* __restrict__ row_of,
                                  const int32_t* __restrict__ col, const double* __restrict__ val, int64_t nnz,
                                  int32_t* __restrict__ su, int32_t* __restrict__ si, float* __restrict__ sr) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nnz) return;
    const uint32_t e = perm[t];
    su[t] = row_of[e]; si[t] = col[e]; sr[t] = (float)val[e];
}

// 0 = ok; bit0: rowptr not monotone / bad ends, bit1: column out of range, bit2: row not strictly ascending
__global__ void csr_validate_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, int32_t U,
                                    int32_t I, int64_t nnz, int* __restrict__ flags) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < U) { if (rowptr[t + 1] < rowptr[t]) atomicOr(flags, 1); }
    if (t == 0) { if (rowptr[0] != 0 || rowptr[U] != nnz) atomicOr(flags, 1); }
    if (t < nnz) {
        const int32_t c = col[t];
        if (c < 0 || c >= I) atomicOr(flags, 2);
    }
}
__global__ void csr_validate_rows_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                         const int32_t* __restrict__ row_of, int64_t nnz, int* __restrict__ flags) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t + 1 < nnz && row_of[t] == row_of[t + 1] && col[t] >= col[t + 1]) atomicOr(flags, 4);
}

// double[rows][k] -> float[rows][ld] (zero padded), and back
__global__ void f64_to_f32_rows_kernel(const double* __restrict__ src, float* __restrict__ dst, int64_t rows, int k, int ld) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= rows * ld) return;
    const int64_t r = t / ld; const int f = (int)(t - r * ld);
    dst[t] = f < k ? (float)src[r * k + f] : 0.f;
}
__global__ void f32_to_f64_rows_kernel(const float* __restrict__ src, double* __restrict__ dst, int64_t rows, int k, int ld) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= rows * k) return;
    const int64_t r = t / k; const int f = (int)(t - r * k);
    dst[t] = (double)src[r * ld + f];
}

// ---------------------------------------------------------------------------------------------
// Stream order.  The COO stream of an epoch is, per item block (one block on a single GPU, `world`
// blocks under DSGD): [item-run tiles] [everything else, shuffled].  An item-run tile is 32 ratings
// of ONE item (items with >= LRK_RUN_MIN_DEGREE ratings in the block's shard give floor(deg/32) of
// them, the CSR-order remainder joins the shuffled part); tiles are shuffled among themselves.  The
// kernel flushes the item-side delta of a run every 8 ratings (16 / 32 for hot items, sgd.cuh), so a flush of
// a 128-rating item is a mini-batch of 1/16 of its ratings -- the share the staleness cap of sgd_grid
// allows in flight -- and its step is damped by the staleness-aware factor.  (Before that factor existed,
// runs from 64 ratings up made PMF at lr 0.01 diverge on ml-100k and the threshold was 512; 512 -> 128 moves
// half of the remaining ratings into run tiles: C2 epoch 1.65 -> 1.50 ms.)  The
// SGD kernel turns a run tile into a single update of the item row (sgd.cuh) and walks the tiles with
// a multiplicative stride so that the two parts interleave in time.  All of it is one radix sort on
//   key = block : 6 | is_rest : 1 | hash : 32 | tile or entry id : 25
// ---------------------------------------------------------------------------------------------
#ifndef LRK_RUN_MIN_DEGREE
#define LRK_RUN_MIN_DEGREE 128
#endif

__global__ void item_degree_kernel(const int32_t* __restrict__ col, int64_t nnz, uint32_t* __restrict__ deg) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nnz) atomicAdd(deg + col[t], 1u);
}
// runs per item; max_deg[b] = largest item degree of block b (lrk_stage_stats)
__global__ void item_runs_kernel(const uint32_t* __restrict__ deg, int32_t I, uint32_t* __restrict__ runs,
                                 const int32_t* __restrict__ bounds, int world, uint32_t* __restrict__ max_deg) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= I) return;
    runs[i] = deg[i] >= LRK_RUN_MIN_DEGREE ? deg[i] / 32u : 0u;
    int b = 0;
    if (bounds) while (b + 1 < world && i >= bounds[b + 1]) ++b;
    if (deg[i]) atomicMax(max_deg + b, deg[i]);
}
__global__ void col_keys_kernel(const int32_t* __restrict__ col, int64_t nnz, uint32_t* __restrict__ k, uint32_t* __restrict__ v) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < nnz) { k[e] = (uint32_t)col[e]; v[e] = (uint32_t)e; }
}
// pos = position of entry e in the by-item order (stable: CSR order inside an item)
__global__ void tile_keys_kernel(const uint32_t* __restrict__ sorted_e, const int32_t* __restrict__ col, int64_t nnz,
                                 const uint32_t* __restrict__ item_start, const uint32_t* __restrict__ runs,
                                 const uint32_t* __restrict__ run_base, const int32_t* __restrict__ bounds, int world,
                                 uint64_t seed, uint64_t* __restrict__ keys, uint32_t* __restrict__ idx) {
    const int64_t pos = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= nnz) return;
    const uint32_t e = sorted_e[pos];
    const int32_t i = col[e];
    const uint32_t rank = (uint32_t)pos - item_start[i];
    int b = 0;
    if (bounds) while (b + 1 < world && i >= bounds[b + 1]) ++b;
    uint64_t key = (uint64_t)b << 58;
    if (rank < 32u * runs[i]) {
        const uint32_t tile = run_base[i] + rank / 32u;
        key |= ((uint64_t)lrk_hash32((uint64_t)tile ^ (seed * 0xA24BAED4963EE407ull)) << 25) | (uint64_t)(tile & 0x1ffffffu);
    } else {
        key |= (1ull << 57) | ((uint64_t)lrk_hash32((uint64_t)e ^ (seed * 0xD6E8FEB86659FD93ull)) << 25) | (uint64_t)(e & 0x1ffffffu);
    }
    keys[e] = key;
    idx[e] = e;
}

struct TileKeyWork {          // device scratch of stage_tile_keys
    uint32_t *deg, *item_start, *runs, *run_base;       // [I]
    uint32_t* max_deg;                                  // [64] out: largest item degree per block
    uint32_t *k32, *v32, *k32_out, *sorted_e;           // [nnz]
    void* tmp; size_t tmp_bytes;                        // cub temp (see stage_tile_keys_tmp_bytes)
};
static size_t stage_tile_keys_tmp_bytes(int32_t I, int64_t nnz) {
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)nnz, 0, 32);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)I);
    return std::max(a, b) + 256;
}
// keys[e], idx[e] = e for every entry; sorting the pairs by key gives the stream order described above
static int stage_tile_keys(lrk_handle_s* h, const int32_t* d_col, int32_t I, int64_t nnz, const int32_t* d_bounds, int world,
                           uint64_t seed, const TileKeyWork& w, uint64_t* keys, uint32_t* idx) {
    cudaStream_t st = h->stream;
    LRK_REQUIRE(h, world <= 64 && nnz < (int64_t)32 * 0x2000000, "stream too large for the tile key layout");
    const int nb = lrk_ceil_div(nnz, 256), ib = lrk_ceil_div(I, 256);
    int end_bit = 1;
    while (end_bit < 32 && ((int64_t)1 << end_bit) < (int64_t)I) ++end_bit;
    LRK_CUDA(h, cudaMemsetAsync(w.deg, 0, sizeof(uint32_t) * (size_t)I, st));
    item_degree_kernel<<<nb, 256, 0, st>>>(d_col, nnz, w.deg); LRK_LAUNCH_CHECK(h);
    LRK_CUDA(h, cudaMemsetAsync(w.max_deg, 0, sizeof(uint32_t) * 64, st));
    item_runs_kernel<<<ib, 256, 0, st>>>(w.deg, I, w.runs, d_bounds, world, w.max_deg); LRK_LAUNCH_CHECK(h);
    size_t tb = w.tmp_bytes;
    LRK_CUDA(h, cub::DeviceScan::ExclusiveSum(w.tmp, tb, w.deg, w.item_start, (int)I, st));
    tb = w.tmp_bytes;
    LRK_CUDA(h, cub::DeviceScan::ExclusiveSum(w.tmp, tb, w.runs, w.run_base, (int)I, st));
    col_keys_kernel<<<nb, 256, 0, st>>>(d_col, nnz, w.k32, w.v32); LRK_LAUNCH_CHECK(h);
    tb = w.tmp_bytes;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(w.tmp, tb, w.k32, w.k32_out, w.v32, w.sorted_e, (int)nnz, 0, end_bit, st));
    tile_keys_kernel<<<nb, 256, 0, st>>>(w.sorted_e, d_col, nnz, w.item_start, w.runs, w.run_base, d_bounds, world, seed, keys, idx);
    LRK_LAUNCH_CHECK(h);
    return LRK_OK;
}

// Host driver: device CSR (already resident: d_rowptr, d_col) + host values -> shuffled COO stream.
// Stream order: see stage_tile_keys.
__global__ void coo_rows_kernel(const int64_t* __restrict__ rowptr, int32_t U, int64_t nnz, int32_t* __restrict__ row_of) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    int32_t lo = 0, hi = U;
    while (hi - lo > 1) { const int32_t m = (lo + hi) >> 1; if (rowptr[m] <= e) lo = m; else hi = m; }
    row_of[e] = lo;
}
struct GroupUnits;
static int stage_group_stream(lrk_handle_s* h, const int64_t* d_rowptr, const int32_t* d_col, const int32_t* row_of, const double* d_val,
                              int32_t U, int32_t I, int64_t nnz, const int32_t* d_bounds, int world, int workers, uint64_t seed,
                              LrkScratch& sc, void* tmp, size_t tmp_bytes, uint64_t* keys, uint64_t* keys2, uint32_t* idx, uint32_t* perm,
                              int32_t* su, int32_t* si, float* sr, std::unique_ptr<GroupUnits>* out);
// group_workers > 0: stage the unit-ordered stream of the user-group kernel (staging_group.cuh) for that many resident workers
static int stage_coo_from_csr(lrk_handle_s* h, const int64_t* d_rowptr, const int32_t* d_col, const double* h_val,
                              int32_t U, int32_t I, int64_t nnz, int32_t* su, int32_t* si, float* sr, bool validate,
                              int group_workers = 0, std::unique_ptr<GroupUnits>* group_out = nullptr) {
    cudaStream_t st = h->stream;
    if (nnz == 0) { LRK_CUDA(h, cudaStreamSynchronize(st)); return LRK_OK; }
    size_t tmp64 = 0;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, tmp64, (uint64_t*)nullptr, (uint64_t*)nullptr, (uint32_t*)nullptr,
                                                (uint32_t*)nullptr, (int)nnz, 0, 64, st));
    const size_t tmp_bytes = std::max(tmp64, stage_tile_keys_tmp_bytes(I, nnz));
    const size_t n = (size_t)nnz;
    LrkScratch sc;
    int rc = lrk_scratch_begin(h, n * (8 + 4 + 8 + 8 + 4 * 6) + (size_t)I * 16 + (size_t)U * 20 + tmp_bytes + 48 * 256, &sc);
    if (rc) return rc;
    double* d_val = sc.take<double>(n);
    int32_t* row_of = sc.take<int32_t>(n);
    uint64_t *keys = sc.take<uint64_t>(n), *keys2 = sc.take<uint64_t>(n);
    uint32_t *idx = sc.take<uint32_t>(n), *perm = sc.take<uint32_t>(n);
    TileKeyWork w;
    w.k32 = sc.take<uint32_t>(n); w.v32 = sc.take<uint32_t>(n); w.k32_out = sc.take<uint32_t>(n); w.sorted_e = sc.take<uint32_t>(n);
    w.deg = sc.take<uint32_t>((size_t)I); w.item_start = sc.take<uint32_t>((size_t)I);
    w.runs = sc.take<uint32_t>((size_t)I); w.run_base = sc.take<uint32_t>((size_t)I);
    w.max_deg = sc.take<uint32_t>(64);
    w.tmp = sc.take<char>(tmp_bytes); w.tmp_bytes = tmp_bytes;
    int* d_flags = sc.take<int>(1);
    if (!d_val || !row_of || !keys || !idx || !keys2 || !perm || !w.k32 || !w.v32 || !w.k32_out || !w.sorted_e || !w.deg ||
        !w.item_start || !w.runs || !w.run_base || !w.max_deg || !w.tmp || !d_flags)
        return lrk_fail(h, LRK_ERR_NOMEM, "stage_coo_from_csr", "scratch arena too small", __FILE__, __LINE__);
    int flags = 0;
    // the values (8 B per rating, two thirds of the H2D bytes) are needed only by the final gather: copy them on a second stream
    // while the keys are built and sorted
    if (!h->copy_stream) {
        LRK_CUDA(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        LRK_CUDA(h, cudaEventCreateWithFlags(&h->ev_copy0, cudaEventDisableTiming));
        LRK_CUDA(h, cudaEventCreateWithFlags(&h->ev_copy1, cudaEventDisableTiming));
    }
    LRK_CUDA(h, cudaEventRecord(h->ev_copy0, st));                       // earlier users of the scratch arena are done
    LRK_CUDA(h, cudaStreamWaitEvent(h->copy_stream, h->ev_copy0, 0));
    LRK_CUDA(h, cudaMemcpyAsync(d_val, h_val, sizeof(double) * n, cudaMemcpyHostToDevice, h->copy_stream));
    LRK_CUDA(h, cudaEventRecord(h->ev_copy1, h->copy_stream));
    LRK_CUDA(h, cudaMemsetAsync(d_flags, 0, sizeof(int), st));
    const int nb = lrk_ceil_div(nnz, 256);
    coo_rows_kernel<<<nb, 256, 0, st>>>(d_rowptr, U, nnz, row_of);
    LRK_LAUNCH_CHECK(h);
    {   // validate BEFORE anything indexes by column
        const int64_t m = nnz > U ? nnz : U;
        csr_validate_kernel<<<lrk_ceil_div(m, 256), 256, 0, st>>>(d_rowptr, d_col, U, I, nnz, d_flags);
        LRK_LAUNCH_CHECK(h);
        csr_validate_rows_kernel<<<nb, 256, 0, st>>>(d_rowptr, d_col, row_of, nnz, d_flags);
        LRK_LAUNCH_CHECK(h);
        LRK_CUDA(h, cudaMemcpyAsync(&flags, d_flags, sizeof(int), cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
    }
    (void)validate;
    if (!flags && group_workers > 0) {
        // item degrees (staleness-aware step), then the unit-ordered stream
        LRK_CUDA(h, cudaMemsetAsync(w.deg, 0, sizeof(uint32_t) * (size_t)I, st));
        item_degree_kernel<<<nb, 256, 0, st>>>(d_col, nnz, w.deg); LRK_LAUNCH_CHECK(h);
        if ((rc = lrk_dev_alloc(h, &h->d_item_deg, (size_t)I + 4))) return rc;
        LRK_CUDA(h, cudaMemcpyAsync(h->d_item_deg, w.deg, sizeof(uint32_t) * (size_t)I, cudaMemcpyDeviceToDevice, st));
        LRK_CUDA(h, cudaStreamWaitEvent(st, h->ev_copy1, 0));
        if ((rc = stage_group_stream(h, d_rowptr, d_col, row_of, d_val, U, I, nnz, nullptr, 1, group_workers, h->cfg.seed, sc, w.tmp, tmp_bytes,
                                     keys, keys2, idx, perm, su, si, sr, group_out))) return rc;
        LRK_CUDA(h, cudaStreamSynchronize(st));
        h->run_tiles = 0; h->max_item_deg = 0;
    } else if (!flags) {
        if ((rc = stage_tile_keys(h, d_col, I, nnz, nullptr, 1, h->cfg.seed, w, keys, idx))) return rc;
        size_t tb = tmp_bytes;
        LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(w.tmp, tb, keys, keys2, idx, perm, (int)nnz, 0, 58, st));
        LRK_CUDA(h, cudaStreamWaitEvent(st, h->ev_copy1, 0));
        coo_gather_kernel<<<nb, 256, 0, st>>>(perm, row_of, d_col, d_val, nnz, su, si, sr);
        LRK_LAUNCH_CHECK(h);
        uint32_t max_deg = 0, last_base = 0, last_runs = 0;
        LRK_CUDA(h, cudaMemcpyAsync(&last_base, w.run_base + (I - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaMemcpyAsync(&last_runs, w.runs + (I - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        if ((rc = lrk_dev_alloc(h, &h->d_item_deg, (size_t)I + 4))) return rc;
        LRK_CUDA(h, cudaMemcpyAsync(h->d_item_deg, w.deg, sizeof(uint32_t) * (size_t)I, cudaMemcpyDeviceToDevice, st));
        LRK_CUDA(h, cudaMemcpyAsync(&max_deg, w.max_deg, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
        h->run_tiles = (int64_t)last_base + (int64_t)last_runs;
        h->max_item_deg = max_deg;
    }
    if (flags) LRK_CUDA(h, cudaStreamSynchronize(h->copy_stream));      // the caller may reuse its buffers on return
    if (flags & 1) return lrk_fail(h, LRK_ERR_INVALID, "lrk_set_train_csr", "rowptr is not a monotone prefix sum ending at nnz", __FILE__, __LINE__);
    if (flags & 2) return lrk_fail(h, LRK_ERR_INVALID, "lrk_set_train_csr", "column index out of range", __FILE__, __LINE__);
    if (flags & 4) return lrk_fail(h, LRK_ERR_INVALID, "lrk_set_train_csr", "columns must be strictly ascending inside a row", __FILE__, __LINE__);
    return LRK_OK;
}
