// Staging for the user-group SGD epoch (sgd_group.cuh): the COO stream is ordered by UNIT, inside a unit by (rotated) item, inside an
// item by user.  A unit is the work one worker (G lanes) owns exclusively:
//   * a normal unit  = up to LRK_GS consecutive users (never across an aligned block of LRK_GS users) with ALL their ratings inside one
//     item block (the whole catalogue on one GPU, one DSGD stratum otherwise), cut so that a unit holds about `target` ratings;
//   * a heavy user (more than `target` ratings in the block) is a unit of its own per slice of `target` ratings -- those slices
//     run concurrently, so they merge their user-row deltas with a RED instead of a plain store (flag `shared`).
// Because every rating of a (unit, item) pair is adjacent, the kernel reads the item row ONCE per pair, walks the pair sequentially
// against the unit's user rows in shared memory (exact Gauss-Seidel inside the pair, like the reference's loop), and issues ONE
// vector RED for the item row; user rows are read once and written once per unit with plain loads / stores.  Per rating that is
// ~0.6-0.7 row gathers + REDs (measured on the ML-20M / Netflix shapes, 16 users per unit) against 1.05 for the item-run-tile stream,
// and the RED rate of the L2 is what bounds the epoch (lrk_probe_l2).
// The item order inside a unit is a rotation of the ascending order by a per-unit offset: same-item ratings stay adjacent, the walk
// stays close to the reference's CSR order (users in blocks, items ascending), and concurrently running units are spread over the
// catalogue instead of all hitting the low item ids at once.
#pragma once
#include "lrk_common.cuh"
#include "staging.cuh"
#include <vector>

#define LRK_GS 16                 // users per unit (4 bits of the sort key)
#define LRK_GROUP_MAX_ITEMS (1 << 21)
#define LRK_GROUP_MAX_UNITS (1 << 27)

struct GroupUnits {               // device unit table of a staged stream + host-side block ranges
    LrkBuf<int4> d_units;         // {stream start, ratings, first user, users | slices << 16 (0: the unit owns its users exclusively)}
    LrkBuf<unsigned int> d_counter;      // one work counter per item block (dynamic unit fetch)
    int64_t n_units = 0;
    uint32_t target = 0;
    std::vector<int64_t> unit_base;      // world + 1: units of block b are [unit_base[b], unit_base[b+1])
};

__device__ __forceinline__ int64_t lrk_lower_bound_col(const int32_t* __restrict__ col, int64_t b, int64_t e, int32_t x) {
    while (b < e) { const int64_t m = (b + e) >> 1; if (__ldg(col + m) < x) b = m + 1; else e = m; }
    return b;
}
// v = block * U + user: ratings of the user inside the block, and where they start in its CSR row
__global__ void group_block_deg_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, int32_t U, int32_t I,
                                       const int32_t* __restrict__ bounds, int world, uint32_t* __restrict__ degv, uint32_t* __restrict__ rowlo) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= (int64_t)U * world) return;
    const int b = (int)(v / U);
    const int32_t u = (int32_t)(v - (int64_t)b * U);
    const int64_t rb = rowptr[u], re = rowptr[u + 1];
    const int32_t lo_i = bounds ? bounds[b] : 0, hi_i = bounds ? bounds[b + 1] : I;
    const int64_t lo = lrk_lower_bound_col(col, rb, re, lo_i), hi = lrk_lower_bound_col(col, lo, re, hi_i);
    degv[v] = (uint32_t)(hi - lo);
    rowlo[v] = (uint32_t)lo;
}
// started[v] = units that start at v (0: v continues the previous user's unit)
__global__ void group_unit_flags_kernel(const uint32_t* __restrict__ degv, const uint32_t* __restrict__ S, int32_t U, int world,
                                        uint32_t target, uint32_t* __restrict__ started) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= (int64_t)U * world) return;
    const int32_t u = (int32_t)(v % U);
    const uint32_t deg = degv[v];
    const bool heavy = deg > target;
    bool flag = (u % LRK_GS) == 0 || heavy;
    if (!flag) {
        const bool heavy_prev = degv[v - 1] > target;
        flag = heavy_prev || (S[v] / target) != (S[v - 1] / target);
    }
    started[v] = flag ? (heavy ? (deg + target - 1) / target : 1u) : 0u;
}
// unit id of v's (first) unit = incl[v] - started[v] if it starts one, else incl[v] - 1; fills first_user / users / shared
__global__ void group_unit_desc_kernel(const uint32_t* __restrict__ started, const uint32_t* __restrict__ incl, int32_t U, int world,
                                       int4* __restrict__ units) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= (int64_t)U * world) return;
    const int32_t u = (int32_t)(v % U);
    const uint32_t st = started[v];
    if (st) {
        const uint32_t first = incl[v] - st;
        for (uint32_t s = 0; s < st; ++s) { units[first + s].z = u; if (st > 1) atomicAdd(&units[first + s].w, (int)(st << 16)); }
        for (uint32_t s = 0; s < st; ++s) atomicAdd(&units[first + s].w, 1);
    } else {
        atomicAdd(&units[incl[v] - 1].w, 1);
    }
}
// sort key of entry e: unit : 27 | rotated item : 21 | user inside the unit : 4  (52 bits); counts the unit's ratings
__global__ void group_keys_kernel(const int32_t* __restrict__ row_of, const int32_t* __restrict__ col, int64_t nnz, int32_t U, int32_t I,
                                  const int32_t* __restrict__ bounds, int world, const uint32_t* __restrict__ degv,
                                  const uint32_t* __restrict__ rowlo, const uint32_t* __restrict__ started, const uint32_t* __restrict__ incl,
                                  uint32_t target, uint64_t seed, int rotate, int4* __restrict__ units, uint64_t* __restrict__ keys, uint32_t* __restrict__ idx) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    const int32_t u = row_of[e], i = col[e];
    int b = 0;
    if (bounds) while (b + 1 < world && i >= bounds[b + 1]) ++b;
    const int64_t v = (int64_t)b * U + u;
    const uint32_t st = started[v];
    uint32_t unit = st ? incl[v] - st : incl[v] - 1;
    if (st > 1) unit += ((uint32_t)e - rowlo[v]) / target;           // heavy user: slice by position in its (block) row
    const int32_t lo_i = bounds ? bounds[b] : 0, hi_i = bounds ? bounds[b + 1] : I;
    const uint32_t width = (uint32_t)(hi_i - lo_i);
    const uint32_t rot = rotate ? lrk_hash32((uint64_t)unit ^ (seed * 0xA24BAED4963EE407ull)) % width : 0u;
    uint32_t ritem = (uint32_t)(i - lo_i) + width - rot;
    if (ritem >= width) ritem -= width;
    const uint32_t first_user = (uint32_t)units[unit].z;
    keys[e] = ((uint64_t)unit << 25) | ((uint64_t)ritem << 4) | (uint64_t)((uint32_t)u - first_user);
    idx[e] = (uint32_t)e;
    atomicAdd(&units[unit].y, 1);
}
__global__ void group_unit_counts_kernel(const int4* __restrict__ units, int64_t n, uint32_t* __restrict__ cnt) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) cnt[t] = (uint32_t)units[t].y;
}
__global__ void group_unit_starts_kernel(int4* __restrict__ units, int64_t n, const uint32_t* __restrict__ start) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) units[t].x = (int32_t)start[t];
}
// item ids of the stream are block-local (bounds) so that Q can address a rotating block buffer
__global__ void group_gather_kernel(const uint32_t* __restrict__ perm, const int32_t* __restrict__ row_of, const int32_t* __restrict__ col,
                                    const double* __restrict__ val, const int32_t* __restrict__ bounds, int world, int64_t nnz,
                                    int32_t* __restrict__ su, int32_t* __restrict__ si, float* __restrict__ sr) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nnz) return;
    const uint32_t e = perm[t];
    const int32_t i = col[e];
    int b = 0;
    if (bounds) while (b + 1 < world && i >= bounds[b + 1]) ++b;
    su[t] = row_of[e]; si[t] = i - (bounds ? bounds[b] : 0); sr[t] = (float)val[e];
}

static bool group_order_supported(int32_t U, int32_t I, int64_t nnz, int world) {
    return I <= LRK_GROUP_MAX_ITEMS && (int64_t)U * world < (int64_t)0x7fffffff && nnz < (int64_t)0xffffffffLL && nnz > 0;
}

// d_rowptr / d_col: the (rank-local) CSR on the device; row_of / d_val: per-entry row and value (device scratch of the caller).
// workers = resident workers of the epoch kernel (sets the unit size).  Leaves the stream in su / si / sr and the unit table in *out.
static int stage_group_stream(lrk_handle_s* h, const int64_t* d_rowptr, const int32_t* d_col, const int32_t* row_of, const double* d_val,
                              int32_t U, int32_t I, int64_t nnz, const int32_t* d_bounds, int world, int workers, uint64_t seed,
                              LrkScratch& sc, void* tmp, size_t tmp_bytes, uint64_t* keys, uint64_t* keys2, uint32_t* idx, uint32_t* perm,
                              int32_t* su, int32_t* si, float* sr, std::unique_ptr<GroupUnits>* out) {
    cudaStream_t st = h->stream;
    const int64_t nv = (int64_t)U * world;
    uint32_t *degv = sc.take<uint32_t>((size_t)nv), *rowlo = sc.take<uint32_t>((size_t)nv), *S = sc.take<uint32_t>((size_t)nv);
    uint32_t *started = sc.take<uint32_t>((size_t)nv), *incl = sc.take<uint32_t>((size_t)nv);
    if (!degv || !rowlo || !S || !started || !incl) return lrk_fail(h, LRK_ERR_NOMEM, "stage_group_stream", "scratch arena too small", __FILE__, __LINE__);
    std::unique_ptr<GroupUnits> g(new GroupUnits());
    // unit size: >= 4 units per worker and stratum so that the dynamic fetch balances the tail; 384 .. 2048 ratings
    int64_t target = (nnz / world) / (4 * (int64_t)(workers > 0 ? workers : 1));
    if (target < 384) target = 384;
    if (target > 2048) target = 2048;
    g->target = (uint32_t)target;
    const int vb = lrk_ceil_div(nv, 256), nb = lrk_ceil_div(nnz, 256);
    group_block_deg_kernel<<<vb, 256, 0, st>>>(d_rowptr, d_col, U, I, d_bounds, world, degv, rowlo); LRK_LAUNCH_CHECK(h);
    size_t tb = tmp_bytes;
    LRK_CUDA(h, cub::DeviceScan::ExclusiveSum(tmp, tb, degv, S, (int)nv, st));
    group_unit_flags_kernel<<<vb, 256, 0, st>>>(degv, S, U, world, g->target, started); LRK_LAUNCH_CHECK(h);
    tb = tmp_bytes;
    LRK_CUDA(h, cub::DeviceScan::InclusiveSum(tmp, tb, started, incl, (int)nv, st));
    uint32_t n_units = 0;
    std::vector<uint32_t> first_incl((size_t)world), first_started((size_t)world);
    LRK_CUDA(h, cudaMemcpyAsync(&n_units, incl + (nv - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    for (int b = 0; b < world; ++b) {
        LRK_CUDA(h, cudaMemcpyAsync(&first_incl[(size_t)b], incl + (int64_t)b * U, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaMemcpyAsync(&first_started[(size_t)b], started + (int64_t)b * U, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    }
    LRK_CUDA(h, cudaStreamSynchronize(st));
    if (n_units == 0 || n_units >= LRK_GROUP_MAX_UNITS)
        return lrk_fail(h, LRK_ERR_INVALID, "stage_group_stream", "unit count out of range", __FILE__, __LINE__);
    g->n_units = n_units;
    g->unit_base.assign((size_t)world + 1, (int64_t)n_units);
    for (int b = 0; b < world; ++b) g->unit_base[(size_t)b] = (int64_t)first_incl[(size_t)b] - (int64_t)first_started[(size_t)b];
    int rc;
    if ((rc = lrk_dev_alloc(h, &g->d_units, (size_t)n_units))) return rc;
    if ((rc = lrk_dev_alloc(h, &g->d_counter, 64))) return rc;
    LRK_CUDA(h, cudaMemsetAsync(g->d_units, 0, sizeof(int4) * (size_t)n_units, st));
    LRK_CUDA(h, cudaMemsetAsync(g->d_counter, 0, sizeof(unsigned int) * 64, st));
    group_unit_desc_kernel<<<vb, 256, 0, st>>>(started, incl, U, world, g->d_units); h->launches++;
    // LRK_SGD_GROUP_ROTATE=0: every unit walks its items in plain ascending order, exactly like a row of the reference's CSR walk
    // (all concurrently running units then start on the low item ids together; a probe for small matrices)
    const char* rot_env = getenv("LRK_SGD_GROUP_ROTATE");
    const int rotate = (rot_env && atoi(rot_env) == 0) ? 0 : 1;
    group_keys_kernel<<<nb, 256, 0, st>>>(row_of, d_col, nnz, U, I, d_bounds, world, degv, rowlo, started, incl, g->target, seed, rotate, g->d_units, keys, idx);
    LRK_LAUNCH_CHECK(h);
    tb = tmp_bytes;
    LRK_CUDA(h, cub::DeviceRadixSort::SortPairs(tmp, tb, keys, keys2, idx, perm, (int)nnz, 0, 52, st));
    group_gather_kernel<<<nb, 256, 0, st>>>(perm, row_of, d_col, d_val, d_bounds, world, nnz, su, si, sr); h->launches++;
    // unit starts = exclusive prefix sums of the unit sizes (keys2 is free again: reuse it as two uint32 arrays)
    uint32_t* cnt = reinterpret_cast<uint32_t*>(keys);
    uint32_t* start = cnt + n_units;
    if ((size_t)n_units * 2 * sizeof(uint32_t) > (size_t)nnz * sizeof(uint64_t)) LRK_CUDA(h, cudaErrorInvalidValue);
    group_unit_counts_kernel<<<lrk_ceil_div(n_units, 256), 256, 0, st>>>(g->d_units, n_units, cnt); h->launches++;
    tb = tmp_bytes;
    LRK_CUDA(h, cub::DeviceScan::ExclusiveSum(tmp, tb, cnt, start, (int)n_units, st));
    group_unit_starts_kernel<<<lrk_ceil_div(n_units, 256), 256, 0, st>>>(g->d_units, n_units, start); LRK_LAUNCH_CHECK(h);
    *out = std::move(g);
    return LRK_OK;
}
