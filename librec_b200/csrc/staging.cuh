// Staging kernels: flat CSR (what the Java shim flattens SequentialAccessSparseMatrix into,
// math/structure/SequentialAccessSparseMatrix.java:23, RowSequentialAccessSparseMatrix.java:19)
// -> device CSR + shuffled COO stream; DenseMatrix double[][] <-> padded fp32 working rows.
#pragma once
#include "lrk_common.cuh"
#include "lrk_nccl.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <vector>

__device__ __forceinline__ uint32_t lrk_hash32(uint64_t x) {   // splitmix64 finaliser, high word
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    x ^= x >> 31;
    return (uint32_t)(x >> 32);
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

// the stream at sorted position t.  With item blocks (DSGD) the item id is local to its block (key bits 58..63), so that Q can
// address a rotating block buffer; without them it is the column itself and the sorted keys are not read
__global__ void stage_gather_kernel(const uint32_t* __restrict__ perm, const uint64_t* __restrict__ keys_sorted,
                                    const int32_t* __restrict__ row_of, const int32_t* __restrict__ col,
                                    const double* __restrict__ val, const int32_t* __restrict__ bounds, int64_t nnz,
                                    int32_t* __restrict__ su, int32_t* __restrict__ si, float* __restrict__ sr) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nnz) return;
    const uint32_t e = perm[t];
    su[t] = row_of[e]; si[t] = bounds ? col[e] - bounds[keys_sorted[t] >> 58] : col[e]; sr[t] = (float)val[e];
}

// ---- the by-item (CSC) order of the train matrix: the run tiles of the stream, the GBPR group draws and the ALS item solves
// colptr[i] = first entry of item i in the by-item order, colptr[I] = nnz
__global__ void csc_colptr_kernel(const uint32_t* __restrict__ deg_excl, const uint32_t* __restrict__ deg, int32_t I, int64_t* __restrict__ colptr) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < I) colptr[i] = (int64_t)deg_excl[i];
    if (i == I - 1) colptr[I] = (int64_t)deg_excl[i] + (int64_t)deg[i];
}
// cusers[t] = user of the t-th entry in the by-item order
__global__ void csc_rows_kernel(const uint32_t* __restrict__ perm, const int32_t* __restrict__ row_of, int64_t nnz, int32_t* __restrict__ cusers) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nnz) cusers[t] = row_of[perm[t]];
}
static size_t by_item_order_tmp_bytes(int32_t I, int64_t nnz) {
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)nnz, 0, 32);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)I);
    return std::max(a, b) + 256;
}
// deg[i] = entries of item i, start = the exclusive prefix sums of deg, perm = the entry ids sorted by column, stable (CSR order,
// i.e. ascending users, inside an item).  keys, keys_out, ids: [nnz] scratch; tmp: by_item_order_tmp_bytes
static int by_item_order(lrk_handle_s* h, const int32_t* d_col, int32_t I, int64_t nnz, uint32_t* deg, uint32_t* start, uint32_t* perm,
                         uint32_t* keys, uint32_t* keys_out, uint32_t* ids, void* tmp, size_t tmp_bytes) {
    cudaStream_t st = h->stream;
    const int nb = lrk_ceil_div(nnz, 256);
    int end_bit = 1;
    while (end_bit < 32 && ((int64_t)1 << end_bit) < (int64_t)I) ++end_bit;
    LRK_CUDA(h, cudaMemsetAsync(deg, 0, sizeof(uint32_t) * (size_t)I, st));
    if (nnz == 0) return LRK_OK;
    item_degree_kernel<<<nb, 256, 0, st>>>(d_col, nnz, deg); LRK_LAUNCH_CHECK(h);
    size_t tb = tmp_bytes;
    LRK_CUDA(h, cub::DeviceScan::ExclusiveSum(tmp, tb, deg, start, (int)I, st));
    col_keys_kernel<<<nb, 256, 0, st>>>(d_col, nnz, keys, ids); LRK_LAUNCH_CHECK(h);
    tb = tmp_bytes;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(tmp, tb, keys, keys_out, ids, perm, (int)nnz, 0, end_bit, st));
    return LRK_OK;
}

struct TileKeyWork {          // device arrays of stage_tile_keys
    const uint32_t *deg, *item_start, *sorted_e;        // in: the by-item order (by_item_order)
    uint32_t *runs, *run_base;                          // [I]
    uint32_t* max_deg;                                  // [64] out: largest item degree per block
    void* tmp; size_t tmp_bytes;                        // cub temp (by_item_order_tmp_bytes)
};
// keys[e], idx[e] = e for every entry; sorting the pairs by key gives the stream order described above
static int stage_tile_keys(lrk_handle_s* h, const int32_t* d_col, int32_t I, int64_t nnz, const int32_t* d_bounds, int world,
                           uint64_t seed, const TileKeyWork& w, uint64_t* keys, uint32_t* idx) {
    cudaStream_t st = h->stream;
    LRK_REQUIRE(h, world <= 64 && nnz < (int64_t)32 * 0x2000000, "stream too large for the tile key layout");
    const int nb = lrk_ceil_div(nnz, 256), ib = lrk_ceil_div(I, 256);
    LRK_CUDA(h, cudaMemsetAsync(w.max_deg, 0, sizeof(uint32_t) * 64, st));
    item_runs_kernel<<<ib, 256, 0, st>>>(w.deg, I, w.runs, d_bounds, world, w.max_deg); LRK_LAUNCH_CHECK(h);
    size_t tb = w.tmp_bytes;
    LRK_CUDA(h, cub::DeviceScan::ExclusiveSum(w.tmp, tb, w.runs, w.run_base, (int)I, st));
    tile_keys_kernel<<<nb, 256, 0, st>>>(w.sorted_e, d_col, nnz, w.item_start, w.runs, w.run_base, d_bounds, world, seed, keys, idx);
    LRK_LAUNCH_CHECK(h);
    return LRK_OK;
}

__global__ void coo_rows_kernel(const int64_t* __restrict__ rowptr, int32_t U, int64_t nnz, int32_t* __restrict__ row_of) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    int32_t lo = 0, hi = U;
    while (hi - lo > 1) { const int32_t m = (lo + hi) >> 1; if (rowptr[m] <= e) lo = m; else hi = m; }
    row_of[e] = lo;
}

// ---- item blocks of a DSGD rank: every rank cuts the catalogue at the same bounds, from the all-reduced item degrees
// contiguous item blocks balanced by rating count: block b = [bounds[b], bounds[b+1]); mirrored by librec_b200/dsgd_plan.py
static inline void dsgd_item_bounds(const int64_t* item_count, int32_t I, int world, std::vector<int32_t>& bounds) {
    int64_t total = 0;
    for (int32_t i = 0; i < I; ++i) total += item_count[i];
    bounds.assign(world + 1, I);
    bounds[0] = 0;
    int64_t acc = 0;
    int b = 1;
    for (int32_t i = 0; i < I && b < world; ++i) {
        acc += item_count[i];
        // close block b-1 after item i once it holds its share; keep at least one item per remaining block
        while (b < world && (acc * world >= total * b || I - (i + 1) <= world - b)) { bounds[b] = i + 1; ++b; }
    }
    for (int j = 1; j <= world; ++j) if (bounds[j] < bounds[j - 1]) bounds[j] = bounds[j - 1];
    bounds[world] = I;
}
struct ItemBlocks {                     // the staged layout of a DSGD rank's stream (DsgdState)
    std::vector<int32_t> bounds;        // world+1 item block bounds
    std::vector<int64_t> seg_off;       // world+1 offsets of the COO segments, one per item block
    int32_t max_blk = 0;                // rows of the largest item block
    LrkBuf<int32_t> d_bounds;
};
__global__ void flag_bits_kernel(const int* __restrict__ flags, int* __restrict__ bits) {
    if (threadIdx.x < 3) bits[threadIdx.x] = (flags[0] >> threadIdx.x) & 1;
}
// local ratings per item block from the local item degrees (one thread per item)
__global__ void dsgd_block_counts_kernel(const uint32_t* __restrict__ deg, int32_t I, const int32_t* __restrict__ bounds, int world,
                                         unsigned long long* __restrict__ cnt) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= I || deg[i] == 0) return;
    int b = 0;
    while (b + 1 < world && i >= bounds[b + 1]) ++b;
    atomicAdd(cnt + b, (unsigned long long)deg[i]);
}
__global__ void u32_to_u64_kernel(const uint32_t* __restrict__ in, int32_t n, unsigned long long* __restrict__ out) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}

struct GroupUnits;
static int stage_group_stream(lrk_handle_s* h, const int64_t* d_rowptr, const int32_t* d_col, const int32_t* row_of, const double* d_val,
                              int32_t U, int32_t I, int64_t nnz, const int32_t* d_bounds, int world, int workers, uint64_t seed,
                              LrkScratch& sc, void* tmp, size_t tmp_bytes, uint64_t* keys, uint64_t* keys2, uint32_t* idx, uint32_t* perm,
                              int32_t* su, int32_t* si, float* sr, std::unique_ptr<GroupUnits>* out);

// Host driver of lrk_set_train_csr, on one GPU and on a DSGD rank (blocks != nullptr: the rank's user block with GLOBAL item
// ids, h->world > 1): uploads the CSR, validates it, counts the item degrees into h->d_item_deg and stages the COO stream in
// d_su / d_si / d_sr -- the order of stage_tile_keys, or with group_workers > 0 the unit-ordered stream of the user-group kernel
// (staging_group.cuh) for that many resident workers.  Everything that walks the entries runs on the device and takes its
// temporaries from the staging arena (the host only sees O(numItems) and O(world) arrays).
static int stage_train_csr(lrk_handle_s* h, int32_t U, int32_t I, const int64_t* rowptr, const int32_t* col, const double* val,
                           int group_workers, ItemBlocks* blocks) {
    cudaStream_t st = h->stream;
    const int world = h->world;
    const int64_t nnz = rowptr[U];
    h->has_train = false;
    int rc;
    if ((rc = lrk_dev_alloc(h, &h->d_rowptr, (size_t)U + 1))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->d_col, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->d_su, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->d_si, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->d_sr, (size_t)nnz))) return rc;
    if ((rc = lrk_dev_alloc(h, &h->d_item_deg, (size_t)I + 4))) return rc;
    if (blocks && (rc = lrk_dev_alloc(h, &blocks->d_bounds, (size_t)world + 1))) return rc;
    LRK_CUDA(h, cudaMemcpyAsync(h->d_rowptr, rowptr, sizeof(int64_t) * ((size_t)U + 1), cudaMemcpyHostToDevice, st));
    if (nnz > 0) LRK_CUDA(h, cudaMemcpyAsync(h->d_col, col, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, st));
    h->U = U; h->I = I; h->nnz = nnz;

    const size_t n = (size_t)std::max<int64_t>(nnz, 1);
    size_t tmp64 = 0;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, tmp64, (uint64_t*)nullptr, (uint64_t*)nullptr, (uint32_t*)nullptr,
                                                (uint32_t*)nullptr, (int)n, 0, 64, st));
    const size_t tmp_bytes = std::max(tmp64, by_item_order_tmp_bytes(I, n));
    LrkScratch sc;
    if ((rc = lrk_scratch_begin(h, n * (8 + 4 + 8 + 8 + 4 * 6) + (size_t)I * (12 + 8) + (size_t)U * world * 20 + tmp_bytes + 80 * 256, &sc)))
        return rc;
    double* d_val = sc.take<double>(n);
    int32_t* row_of = sc.take<int32_t>(n);
    uint64_t *keys = sc.take<uint64_t>(n), *keys2 = sc.take<uint64_t>(n);
    uint32_t *idx = sc.take<uint32_t>(n), *perm = sc.take<uint32_t>(n);
    uint32_t *k32 = sc.take<uint32_t>(n), *v32 = sc.take<uint32_t>(n), *k32_out = sc.take<uint32_t>(n), *sorted_e = sc.take<uint32_t>(n);
    uint32_t *item_start = sc.take<uint32_t>((size_t)I), *runs = sc.take<uint32_t>((size_t)I), *run_base = sc.take<uint32_t>((size_t)I);
    uint32_t* max_deg = sc.take<uint32_t>(64);
    void* tmp = sc.take<char>(tmp_bytes);
    unsigned long long* d_cnt = sc.take<unsigned long long>((size_t)I);
    unsigned long long* d_small = sc.take<unsigned long long>(128);        // [0,64) block counts, [64] flags
    if (!d_val || !row_of || !keys || !keys2 || !idx || !perm || !k32 || !v32 || !k32_out || !sorted_e || !item_start || !runs ||
        !run_base || !max_deg || !tmp || !d_cnt || !d_small)
        return lrk_fail(h, LRK_ERR_NOMEM, "stage_train_csr", "scratch arena too small", __FILE__, __LINE__);
    int* d_flags = reinterpret_cast<int*>(d_small + 64);
    const int nb = lrk_ceil_div(n, 256), ib = lrk_ceil_div(I, 256);

    // the values (8 B per rating, two thirds of the H2D bytes) are needed only by the final gather: copy them on a second stream
    // while the keys are built and sorted
    if (!h->copy_stream) {
        LRK_CUDA(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        LRK_CUDA(h, cudaEventCreateWithFlags(&h->ev_copy0, cudaEventDisableTiming));
        LRK_CUDA(h, cudaEventCreateWithFlags(&h->ev_copy1, cudaEventDisableTiming));
    }
    LRK_CUDA(h, cudaEventRecord(h->ev_copy0, st));                       // earlier users of the scratch arena are done
    LRK_CUDA(h, cudaStreamWaitEvent(h->copy_stream, h->ev_copy0, 0));
    if (nnz > 0) LRK_CUDA(h, cudaMemcpyAsync(d_val, val, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, h->copy_stream));
    LRK_CUDA(h, cudaEventRecord(h->ev_copy1, h->copy_stream));

    // validate BEFORE anything indexes by column.  A DSGD rank all-reduces the verdict, so that every rank fails together and
    // nobody is left waiting in a collective
    LRK_CUDA(h, cudaMemsetAsync(d_small, 0, sizeof(unsigned long long) * 128, st));
    if (nnz > 0) { coo_rows_kernel<<<nb, 256, 0, st>>>(h->d_rowptr, U, nnz, row_of); LRK_LAUNCH_CHECK(h); }
    csr_validate_kernel<<<lrk_ceil_div(std::max<int64_t>(nnz, U), 256), 256, 0, st>>>(h->d_rowptr, h->d_col, U, I, nnz, d_flags);
    LRK_LAUNCH_CHECK(h);
    if (nnz > 0) { csr_validate_rows_kernel<<<nb, 256, 0, st>>>(h->d_rowptr, h->d_col, row_of, nnz, d_flags); LRK_LAUNCH_CHECK(h); }
    int flags = 0;
    if (blocks) {   // bit-wise OR across ranks: three counters (one per bit) summed
        int* d_bits = d_flags + 4;
        int bits[3];
        flag_bits_kernel<<<1, 32, 0, st>>>(d_flags, d_bits); LRK_LAUNCH_CHECK(h);
        LRK_NCCL(h, nccl_api()->AllReduce(d_bits, d_bits, 3, ncclInt32, ncclSum, (ncclComm_t)h->comm, st));
        LRK_CUDA(h, cudaMemcpyAsync(bits, d_bits, sizeof bits, cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
        for (int j = 0; j < 3; ++j) if (bits[j]) flags |= 1 << j;
    } else {
        LRK_CUDA(h, cudaMemcpyAsync(&flags, d_flags, sizeof(int), cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
    }
    if (flags) LRK_CUDA(h, cudaStreamSynchronize(h->copy_stream));      // the caller may reuse its buffers on return
    if (flags & 1) return lrk_fail(h, LRK_ERR_INVALID, "lrk_set_train_csr", "rowptr is not a monotone prefix sum ending at nnz", __FILE__, __LINE__);
    if (flags & 2) return lrk_fail(h, LRK_ERR_INVALID, "lrk_set_train_csr", "column index out of range", __FILE__, __LINE__);
    if (flags & 4) return lrk_fail(h, LRK_ERR_INVALID, "lrk_set_train_csr", "columns must be strictly ascending inside a row", __FILE__, __LINE__);

    // item degrees (the staleness-aware step of the SGD kernels reads them); the run tiles also need the by-item order.
    // group_workers > 0 implies nnz > 0 (group_order_supported)
    if (group_workers > 0) {
        LRK_CUDA(h, cudaMemsetAsync(h->d_item_deg, 0, sizeof(uint32_t) * (size_t)I, st));
        item_degree_kernel<<<nb, 256, 0, st>>>(h->d_col, nnz, h->d_item_deg); LRK_LAUNCH_CHECK(h);
    } else if ((rc = by_item_order(h, h->d_col, I, nnz, h->d_item_deg, item_start, sorted_e, k32, k32_out, v32, tmp, tmp_bytes))) {
        return rc;
    }
    if (blocks) {   // global item popularity -> identical block bounds on every rank (host work is O(numItems))
        u32_to_u64_kernel<<<ib, 256, 0, st>>>(h->d_item_deg, I, d_cnt); LRK_LAUNCH_CHECK(h);
        LRK_NCCL(h, nccl_api()->AllReduce(d_cnt, d_cnt, (size_t)I, ncclUint64, ncclSum, (ncclComm_t)h->comm, st));
        std::vector<int64_t> cnt((size_t)I);
        LRK_CUDA(h, cudaMemcpyAsync(cnt.data(), d_cnt, sizeof(int64_t) * (size_t)I, cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
        dsgd_item_bounds(cnt.data(), I, world, blocks->bounds);
        blocks->max_blk = 0;
        for (int b = 0; b < world; ++b) blocks->max_blk = std::max(blocks->max_blk, blocks->bounds[b + 1] - blocks->bounds[b]);
        LRK_CUDA(h, cudaMemcpyAsync(blocks->d_bounds, blocks->bounds.data(), sizeof(int32_t) * ((size_t)world + 1), cudaMemcpyHostToDevice, st));
        dsgd_block_counts_kernel<<<ib, 256, 0, st>>>(h->d_item_deg, I, blocks->d_bounds, world, d_small); LRK_LAUNCH_CHECK(h);
    }

    // bucket by item block; inside a block: item-run tiles, then the shuffled rest.  One GPU sorts 58 key bits: the block bits are 0
    const int32_t* d_bounds = blocks ? blocks->d_bounds.ptr : nullptr;
    const uint64_t seed = h->cfg.seed + 977u * h->rank;
    uint32_t md[64] = {0}, last_base = 0, last_runs = 0;
    if (group_workers > 0) {
        LRK_CUDA(h, cudaStreamWaitEvent(st, h->ev_copy1, 0));
        if ((rc = stage_group_stream(h, h->d_rowptr, h->d_col, row_of, d_val, U, I, nnz, d_bounds, world, group_workers, seed, sc, tmp,
                                     tmp_bytes, keys, keys2, idx, perm, h->d_su, h->d_si, h->d_sr, &h->group))) return rc;
    } else if (nnz > 0) {
        const TileKeyWork w{h->d_item_deg, item_start, sorted_e, runs, run_base, max_deg, tmp, tmp_bytes};
        if ((rc = stage_tile_keys(h, h->d_col, I, nnz, d_bounds, world, seed, w, keys, idx))) return rc;
        size_t tb = tmp_bytes;
        LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(tmp, tb, keys, keys2, idx, perm, (int)nnz, 0, blocks ? 64 : 58, st));
        LRK_CUDA(h, cudaStreamWaitEvent(st, h->ev_copy1, 0));
        stage_gather_kernel<<<nb, 256, 0, st>>>(perm, keys2, row_of, h->d_col, d_val, d_bounds, nnz, h->d_su, h->d_si, h->d_sr);
        LRK_LAUNCH_CHECK(h);
        LRK_CUDA(h, cudaMemcpyAsync(&last_base, run_base + (I - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaMemcpyAsync(&last_runs, runs + (I - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaMemcpyAsync(md, max_deg, sizeof md, cudaMemcpyDeviceToHost, st));
    }
    unsigned long long seg_cnt[64];
    if (blocks) LRK_CUDA(h, cudaMemcpyAsync(seg_cnt, d_small, sizeof seg_cnt, cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    h->run_tiles = (int64_t)last_base + (int64_t)last_runs;
    h->max_item_deg = 0;
    for (int b = 0; b < world; ++b) h->max_item_deg = std::max(h->max_item_deg, md[b]);
    if (blocks) {
        blocks->seg_off.assign((size_t)world + 1, 0);
        for (int b = 0; b < world; ++b) blocks->seg_off[(size_t)b + 1] = blocks->seg_off[(size_t)b] + (int64_t)seg_cnt[b];
    }
    return LRK_OK;
}
