// DSGD (Gemulla et al., KDD'11 -- the paper the reference cites at
// recommender/MatrixFactorizationRecommender.java:111-112) across the GPUs of one box, one process
// per GPU.  SURVEY.md 8(e).
//
//   * users are sharded: rank g owns its user block (P rows, user biases) for the whole run;
//   * items are cut into G contiguous blocks balanced by global rating count; the rank's ratings
//     are bucketed by item block into G independently shuffled COO segments;
//   * sub-epoch s in [0,G): rank g runs the SGD kernel on segment b = (g+s) mod G against the item
//     block it currently holds, then the ring rotates: send block b to rank g-1, receive block
//     (g+s+1) mod G from rank g+1 (grouped ncclSend/ncclRecv on the handle's stream, NVLink 5);
//   * strata of one sub-epoch touch disjoint users AND items, so there is no cross-GPU race;
//   * one fp64 ncclAllReduce of the loss per epoch.
// NCCL is dlopen'ed lazily so that the single-GPU path has no NCCL dependency (lrk_nccl.cuh).
#pragma once
#include "lrk_common.cuh"
#include "staging.cuh"
#include "sgd.cuh"
#include "sgd_group.cuh"
#include "dsgd_fused.cuh"
#include "lrk_epoch.cuh"
#include "lrk_nccl.cuh"
#include <vector>
#include <algorithm>

// ---- the DSGD plan: pure functions of (rank, world, sub-epoch); mirrored by librec_b200/dsgd_plan.py
static inline int dsgd_block_at(int rank, int world, int sub) { return (rank + sub) % world; }
static inline int dsgd_send_peer(int rank, int world) { return (rank - 1 + world) % world; }
static inline int dsgd_recv_peer(int rank, int world) { return (rank + 1) % world; }
struct DsgdState : ItemBlocks {          // the item blocks and segments of the stream: staging.cuh
    size_t buf_floats = 0;              // floats per rotating buffer: max_blk*ld + max_blk
    LrkBuf<float> qbuf[2];
    int cur = 0;                        // which buffer holds the current block
    int cur_block = 0;                  // item block id currently held
    // LRK_DSGD_TRACE=1: events around every sub-epoch kernel / ring exchange of the last epoch
    std::vector<cudaEvent_t> trace_ev;
    int trace = -1;
    LrkBuf<float> gather_buf;           // lrk_get_factors: all ranks' ring buffers (world * buf_floats)
    LrkBuf<float> q_ref;                // BPR: the item factors at the start of the current window (delta all-reduce)
    LrkBuf<float> q_delta;
    int64_t bpr_samples = 0;            // BPR: samples this rank draws per epoch = numRates * (its users / all users)
    DsgdFused fused;                    // the in-kernel ring of the rating models (dsgd_fused.cuh); LRK_DSGD_FUSED=0 turns it off
    ~DsgdState() {
        dsgd_fused_unmap(&fused);       // the IPC mappings go before the ring buffers
        for (cudaEvent_t ev : trace_ev) if (ev) cudaEventDestroy(ev);
    }
};

// BPR windows: delta = Q - Qref ; after the all-reduce Q = Qref + sum of all ranks' deltas
__global__ void dsgd_delta_kernel(const float* __restrict__ q, const float* __restrict__ ref, float* __restrict__ delta, int64_t n) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) delta[t] = q[t] - ref[t];
}
__global__ void dsgd_apply_delta_kernel(float* __restrict__ q, float* __restrict__ ref, const float* __restrict__ delta, int64_t n) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) { const float v = ref[t] + delta[t]; q[t] = v; ref[t] = v; }
}
__global__ void dsgd_pack_block_kernel(const float* __restrict__ Q, const float* __restrict__ bi, int32_t first, int32_t rows,
                                       int ld, int32_t max_blk, float* __restrict__ buf) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nq = (int64_t)rows * ld;
    if (t < nq) buf[t] = Q[(int64_t)first * ld + t];
    else if (t < nq + rows) buf[(int64_t)max_blk * ld + (t - nq)] = bi ? bi[first + (t - nq)] : 0.f;
}
__global__ void dsgd_unpack_block_kernel(float* __restrict__ Q, float* __restrict__ bi, int32_t first, int32_t rows, int ld,
                                         int32_t max_blk, const float* __restrict__ buf) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nq = (int64_t)rows * ld;
    if (t < nq) Q[(int64_t)first * ld + t] = buf[t];
    else if (t < nq + rows && bi) bi[first + (t - nq)] = buf[(int64_t)max_blk * ld + (t - nq)];
}

static int dsgd_unique_id(uint8_t* out) {
    NcclApi* n = nccl_api();
    if (!n) return lrk_fail(nullptr, LRK_ERR_NCCL, "lrk_comm_unique_id", "libnccl.so.2 could not be loaded", __FILE__, __LINE__);
    if (!out) return lrk_fail(nullptr, LRK_ERR_INVALID, "lrk_comm_unique_id", "out is NULL", __FILE__, __LINE__);
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    LRK_NCCL(nullptr, n->GetUniqueId(&id));
    memcpy(out, &id, 128);
    return LRK_OK;
}

static int dsgd_comm_init(lrk_handle_s* h, int rank, int world, const uint8_t* uid) {
    NcclApi* n = nccl_api();
    if (!n) return lrk_fail(h, LRK_ERR_NCCL, "lrk_comm_init", "libnccl.so.2 could not be loaded", __FILE__, __LINE__);
    LRK_REQUIRE(h, uid != nullptr && world >= 1 && rank >= 0 && rank < world, "bad rank/world");
    LRK_REQUIRE(h, h->comm == nullptr, "communicator already initialised");
    LRK_REQUIRE(h, !h->has_train && !h->has_factors, "lrk_comm_init must precede staging");
    LRK_CUDA(h, cudaSetDevice(h->cfg.device));
    ncclUniqueId id;
    memcpy(&id, uid, 128);
    ncclComm_t comm;
    LRK_NCCL(h, n->CommInitRank(&comm, world, id, rank));
    h->comm = comm; h->rank = rank; h->world = world;
    return LRK_OK;
}

// the rest of lrk_set_train_csr on a rank (stage_train_csr staged the stream and the item blocks)
static int dsgd_set_train_csr(lrk_handle_s* h) {
    DsgdState* s = h->dsgd.get();
    cudaStream_t st = h->stream;
    int rc;
    if (h->cfg.model == LRK_MODEL_BPR) {
        // BPRRecommender.java:48-58 draws numRates samples per iteration, the user uniformly over ALL users: this rank's share is
        // numRates * (its users / all users)
        LrkScratch sc;
        if ((rc = lrk_scratch_begin(h, 256, &sc))) return rc;
        double tot[2] = {(double)h->nnz, (double)h->U};
        double* d_tot = sc.take<double>(2);
        LRK_CUDA(h, cudaMemcpyAsync(d_tot, tot, sizeof tot, cudaMemcpyHostToDevice, st));
        LRK_NCCL(h, nccl_api()->AllReduce(d_tot, d_tot, 2, ncclFloat64, ncclSum, (ncclComm_t)h->comm, st));
        LRK_CUDA(h, cudaMemcpyAsync(tot, d_tot, sizeof tot, cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
        s->bpr_samples = tot[1] > 0.0 ? (int64_t)(tot[0] * ((double)h->U / tot[1]) + 0.5) : 0;
    }
    s->buf_floats = (size_t)s->max_blk * h->ld + (size_t)s->max_blk;
    s->buf_floats = (s->buf_floats + 3) & ~(size_t)3;                       // float4-copyable
    for (int j = 0; j < 2; ++j) if ((rc = lrk_dev_alloc(h, &s->qbuf[j], s->buf_floats))) return rc;
    return LRK_OK;
}

// the rest of lrk_set_factors on a rank (P/bu: the rank's user block; Q/bi: the FULL item factors, identical on every rank):
// the rank starts the epoch holding item block `rank`
static int dsgd_load_ring(lrk_handle_s* h) {
    DsgdState* s = h->dsgd.get();
    cudaStream_t st = h->stream;
    const int b = dsgd_block_at(h->rank, h->world, 0);
    const int32_t first = s->bounds[b], rows = s->bounds[b + 1] - first;
    LRK_CUDA(h, cudaMemsetAsync(s->qbuf[0], 0, sizeof(float) * s->buf_floats, st));
    LRK_CUDA(h, cudaMemsetAsync(s->qbuf[1], 0, sizeof(float) * s->buf_floats, st));
    if (rows > 0) {
        dsgd_pack_block_kernel<<<lrk_ceil_div((int64_t)rows * h->ld + rows, 256), 256, 0, st>>>(h->Q32, h->bi32, first, rows, h->ld, s->max_blk, s->qbuf[0]);
        LRK_LAUNCH_CHECK(h);
    }
    s->cur = 0; s->cur_block = b;
    s->fused.needs_reset = s->fused.mapped;
    return LRK_OK;
}

// ---- fused epoch (dsgd_fused.cuh, the default; LRK_DSGD_FUSED=0 turns it off): IPC mapping of the ring neighbours, then one
// cooperative launch per epoch
static int dsgd_fused_map(lrk_handle_s* h, DsgdState* s) {
    NcclApi* n = nccl_api();
    DsgdFused* f = &s->fused;
    cudaStream_t st = h->stream;
    const int world = h->world, rank = h->rank;
    if (f->mapped && f->my_qbuf[0] == s->qbuf[0] && f->my_qbuf[1] == s->qbuf[1]) return LRK_OK;
    dsgd_fused_unmap(f);
    int rc;
    if ((rc = lrk_dev_alloc(h, &f->d_flags, 4))) return rc;
    if ((rc = lrk_dev_alloc(h, &f->d_abort, 1))) return rc;
    LRK_CUDA(h, cudaMemsetAsync(f->d_flags, 0, sizeof(unsigned long long) * 4, st));
    LRK_CUDA(h, cudaMemsetAsync(f->d_abort, 0, sizeof(int), st));
    // handles of (qbuf[0], qbuf[1], flags) of every rank.  A rank on which CUDA IPC does not work (other container, allocator without
    // IPC support) still takes part in every collective below, and the verdict is all-reduced: either every rank maps its neighbours
    // or all of them keep the ncclSend / ncclRecv ring -- a split decision would leave a kernel spinning on a flag nobody writes.
    cudaIpcMemHandle_t mine[3];
    memset(mine, 0, sizeof mine);
    const bool local = h->same_process && h->siblings != nullptr;      // ranks of one process (multi handle): peer pointers, no IPC
    bool ok = local || (cudaIpcGetMemHandle(&mine[0], s->qbuf[0]) == cudaSuccess && cudaIpcGetMemHandle(&mine[1], s->qbuf[1]) == cudaSuccess &&
                        cudaIpcGetMemHandle(&mine[2], f->d_flags) == cudaSuccess);
    cudaGetLastError();
    const size_t hb = sizeof(cudaIpcMemHandle_t) * 3;
    LrkBuf<uint8_t> d_mine, d_all;
    if ((rc = lrk_dev_alloc(h, &d_mine, hb))) return rc;
    if ((rc = lrk_dev_alloc(h, &d_all, hb * (size_t)world))) return rc;
    std::vector<uint8_t> all(hb * (size_t)world);
    cudaError_t e = cudaMemcpyAsync(d_mine, mine, hb, cudaMemcpyHostToDevice, st);
    ncclResult_t nr = ncclSuccess;
    if (e == cudaSuccess) nr = n->AllGather(d_mine, d_all, hb, ncclUint8, (ncclComm_t)h->comm, st);
    if (e == cudaSuccess && nr == ncclSuccess) e = cudaMemcpyAsync(all.data(), d_all, all.size(), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && nr == ncclSuccess) e = cudaStreamSynchronize(st);
    LRK_NCCL(h, nr);
    LRK_CUDA(h, e);
    auto handle_of = [&](int r, int which) {
        cudaIpcMemHandle_t v;
        memcpy(&v, all.data() + hb * (size_t)r + sizeof(cudaIpcMemHandle_t) * (size_t)which, sizeof v);
        return v;
    };
    auto open = [&](int r, int which, void** out) -> bool {
        if (cudaIpcOpenMemHandle(out, handle_of(r, which), cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); *out = nullptr; return false; }
        f->opened[f->n_opened++] = *out;
        return true;
    };
    const int prev = dsgd_send_peer(rank, world), next = dsgd_recv_peer(rank, world);
    void *q0 = nullptr, *q1 = nullptr, *pf = nullptr, *nf = nullptr;
    if (local) {
        // the all-gather above completed, so every rank of this process has allocated its flags (it enqueues after allocating)
        auto peer = [&](int r) -> bool {
            const int dev = h->siblings[r]->cfg.device;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, h->cfg.device, dev) != cudaSuccess || !can) { cudaGetLastError(); return false; }
            const cudaError_t pe = cudaDeviceEnablePeerAccess(dev, 0);
            if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return false; }
            cudaGetLastError();
            return true;
        };
        DsgdState* ps = h->siblings[prev]->dsgd.get();
        DsgdState* ns = h->siblings[next]->dsgd.get();
        ok = ps && ns && ps->fused.d_flags && ns->fused.d_flags && peer(prev) && peer(next);
        if (ok) { q0 = ps->qbuf[0]; q1 = ps->qbuf[1]; pf = ps->fused.d_flags; nf = ns->fused.d_flags; }
    } else {
        ok = ok && open(prev, 0, &q0) && open(prev, 1, &q1) && open(prev, 2, &pf);
        if (ok) { if (next == prev) nf = pf; else ok = open(next, 2, &nf); }
    }
    // all-reduce the verdict (min); it doubles as the barrier after which every rank's flags are zeroed
    int verdict = ok ? 1 : 0;
    LRK_CUDA(h, cudaMemcpyAsync(f->d_abort, &verdict, sizeof(int), cudaMemcpyHostToDevice, st));
    LRK_NCCL(h, n->AllReduce(f->d_abort, f->d_abort, 1, ncclInt32, ncclMin, (ncclComm_t)h->comm, st));
    LRK_CUDA(h, cudaMemcpyAsync(&verdict, f->d_abort, sizeof(int), cudaMemcpyDeviceToHost, st));
    LRK_CUDA(h, cudaMemsetAsync(f->d_abort, 0, sizeof(int), st));
    LRK_CUDA(h, cudaStreamSynchronize(st));
    if (!verdict) {
        dsgd_fused_unmap(f);
        f->enabled = 0;                  // this communicator keeps the NCCL ring
        return LRK_OK;
    }
    f->peer_qbuf[0] = (float*)q0; f->peer_qbuf[1] = (float*)q1;
    f->prev_flags = (unsigned long long*)pf; f->next_flags = (unsigned long long*)nf;
    f->my_qbuf[0] = s->qbuf[0]; f->my_qbuf[1] = s->qbuf[1];
    f->seq = 0;
    f->mapped = true;
    return LRK_OK;
}

// the fused epoch kernel for (model, variant)
template <int G, int V>
static const void* dsgd_fused_kernel(const lrk_handle_s* h, bool track) {
    if (h->cfg.model == LRK_MODEL_BIASEDMF)
        return track ? (const void*)dsgd_fused_epoch_kernel<G, V, true, true> : (const void*)dsgd_fused_epoch_kernel<G, V, true, false>;
    return track ? (const void*)dsgd_fused_epoch_kernel<G, V, false, true> : (const void*)dsgd_fused_epoch_kernel<G, V, false, false>;
}

template <int G, int V>
static int dsgd_fused_launch_gv(lrk_handle_s* h, DsgdFusedParams& fp) {
    const bool track = sgd_track(h, fp.seg[0]);
    const void* kern = dsgd_fused_kernel<G, V>(h, track);
    int grid = 1, rc;
    if ((rc = sgd_grid(h, kern, 32 / G, track, fp.seg, h->world, &grid))) return rc;
    void* args[] = {(void*)&fp};
    LRK_CUDA(h, cudaLaunchCooperativeKernel(kern, dim3((unsigned)grid), dim3(256), args, 0, h->stream));
    h->launches++;
    return LRK_OK;
}

template <int G, int V>
static int dsgd_fused_group_launch_gv(lrk_handle_s* h, const SgdParams* seg, DsgdFusedGroupParams& fp) {
    const bool biased = h->cfg.model == LRK_MODEL_BIASEDMF;
    void* kern = biased ? (void*)dsgd_fused_group_epoch_kernel<G, V, true> : (void*)dsgd_fused_group_epoch_kernel<G, V, false>;
    const size_t smem = sgd_group_smem_bytes<G, V>();
    LRK_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    LRK_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem));
    const int grid = sgd_group_grid(h, (int64_t)h->sm_count * std::max(per_sm, 1), 8 * (32 / G), seg, fp.seg, h->world);
    void* args[] = {(void*)&fp};
    LRK_CUDA(h, cudaLaunchCooperativeKernel(kern, dim3((unsigned)grid), dim3(256), args, smem, h->stream));
    h->launches++;
    return LRK_OK;
}

// true: the epoch's strata were run by the fused kernel (s->cur advanced like the loop would have); false: not applicable here
static int dsgd_fused_epoch(lrk_handle_s* h, DsgdState* s, const SgdParams& base, bool* done) {
    *done = false;
    DsgdFused* f = &s->fused;
    if (f->enabled < 0) { const char* e = getenv("LRK_DSGD_FUSED"); f->enabled = (e && atoi(e) == 0) ? 0 : 1; }     // default on
    const int world = h->world;
    if (!f->enabled || world < 2 || world > LRK_FUSED_MAX_WORLD || h->cfg.model == LRK_MODEL_BPR ||
        h->cfg.update_mode != LRK_UPDATE_ATOMIC || h->V != 1 || (h->G < 16 && !h->group))
        return LRK_OK;
    int coop = 0;
    LRK_CUDA(h, cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, h->cfg.device));
    if (!coop) return LRK_OK;
    int rc = dsgd_fused_map(h, s);
    if (rc) return rc;
    if (!f->enabled || !f->mapped) return LRK_OK;      // the ranks agreed to keep the ncclSend / ncclRecv ring
    if (f->needs_reset) {
        // every rank re-packed its ring buffers in lrk_set_factors: zero the flags, restart the sequence, and let nobody push before
        // all ranks have done so
        LRK_CUDA(h, cudaMemsetAsync(f->d_flags, 0, sizeof(unsigned long long) * 4, h->stream));
        LRK_NCCL(h, nccl_api()->AllReduce(f->d_abort, f->d_abort, 1, ncclInt32, ncclMin, (ncclComm_t)h->comm, h->stream));
        LRK_CUDA(h, cudaMemsetAsync(f->d_abort, 0, sizeof(int), h->stream));
        LRK_CUDA(h, cudaStreamSynchronize(h->stream));
        f->seq = 0;
        f->needs_reset = false;
    }
    SgdParams seg[LRK_FUSED_MAX_WORLD];
    for (int t = 0; t < world; ++t) {
        const int b = dsgd_block_at(h->rank, world, t);
        const int64_t off = s->seg_off[(size_t)b];
        seg[t] = sgd_segment(h, base, off, s->seg_off[(size_t)b + 1] - off, nullptr, nullptr, s->bounds[(size_t)b]);   // Q / bi: in-kernel
    }
    auto ring = [&](auto& p) {
        p.qbuf[0] = s->qbuf[0]; p.qbuf[1] = s->qbuf[1];
        p.peer_qbuf[0] = f->peer_qbuf[0]; p.peer_qbuf[1] = f->peer_qbuf[1];
        p.ready = f->d_flags; p.peer_free = f->d_flags + 2;
        p.prev_ready = f->prev_flags; p.next_peer_free = f->next_flags + 2;
        p.seq0 = f->seq; p.cur0 = s->cur; p.world = world;
        p.buf_floats = (long long)s->buf_floats; p.bi_off = (long long)s->max_blk * h->ld;
        p.abort = f->d_abort;
        p.spin_limit = 4000000000LL;                            // ~2 s at 2 GHz
    };
    LRK_CUDA(h, cudaMemsetAsync(f->d_abort, 0, sizeof(int), h->stream));      // a timeout of an earlier epoch must not silence this one
    if (h->group) {
        DsgdFusedGroupParams gp{};
        ring(gp);
        for (int t = 0; t < world; ++t) gp.seg[t] = sgd_group_params(h, seg[t], dsgd_block_at(h->rank, world, t));
        rc = sgd_with_group_layout(h, [&](auto G, auto V) { return dsgd_fused_group_launch_gv<decltype(G)::value, decltype(V)::value>(h, seg, gp); });
    } else {
        DsgdFusedParams fp{};
        ring(fp);
        for (int t = 0; t < world; ++t) fp.seg[t] = seg[t];
        rc = lrk_with_layout(h, [&](auto G, auto V) -> int {
            // k in 33..64 and 65..128: the benchmark shapes; smaller k stays on the sub-epoch loop (checked above)
            if constexpr (decltype(G)::value >= 16 && decltype(V)::value == 1) return dsgd_fused_launch_gv<decltype(G)::value, decltype(V)::value>(h, fp);
            else return lrk_fail(h, LRK_ERR_INVALID, "dsgd_fused_epoch", "unsupported factor layout", __FILE__, __LINE__);
        });
    }
    if (rc) return rc;
    f->seq += (unsigned long long)world;
    s->cur = (s->cur + world) & 1;
    s->cur_block = dsgd_block_at(h->rank, world, world);
    *done = true;
    return LRK_OK;
}

// BPR across GPUs.  r01 sampled positives AND negatives inside the item block a rank holds (DSGD strata): items of different blocks
// are then never compared and Precision@10 fell from 0.325 (one GPU) to 0.225 (2 GPUs) / 0.142 (8 GPUs).  The reference's sampler
// (BPRRecommender.java:54-67) compares a positive with a negative from the WHOLE catalogue, so every rank keeps the full item
// matrix (27 k x 128 floats = 14 MB on the ML-20M shape) and trains on its own users with exactly the reference's sampling
// distribution; the epoch is cut into windows, and after each window the ranks all-reduce the CHANGE of the item matrix and
// apply the sum -- the one real exchange step of this path.  Within a window a rank does not see the other ranks' item updates
// (the same kind of staleness as ratings in flight on one GPU, one window long).
#define LRK_BPR_WINDOWS 8
static int dsgd_bpr_epoch(lrk_handle_s* h, DsgdState* s, const SgdParams& base) {
    NcclApi* n = nccl_api();
    cudaStream_t st = h->stream;
    const int64_t nq = (int64_t)h->I * h->ld;
    int rc;
    if ((rc = lrk_dev_alloc(h, &s->q_ref, (size_t)nq))) return rc;
    if ((rc = lrk_dev_alloc(h, &s->q_delta, (size_t)nq))) return rc;
    LRK_CUDA(h, cudaMemcpyAsync(s->q_ref, h->Q32, sizeof(float) * (size_t)nq, cudaMemcpyDeviceToDevice, st));
    int64_t done = 0;
    for (int w = 0; w < LRK_BPR_WINDOWS; ++w) {
        const int64_t cnt = s->bpr_samples * (w + 1) / LRK_BPR_WINDOWS - done;
        if (cnt > 0 && h->U > 0 && h->nnz > 0) {
            SgdParams sp = sgd_segment(h, base, 0, cnt, h->Q32, h->bi32, 0);
            sp.sample_base = done;
            if ((rc = sgd_launch(h, sp))) return rc;
        }
        done += cnt;
        dsgd_delta_kernel<<<lrk_ceil_div(nq, 256), 256, 0, st>>>(h->Q32, s->q_ref, s->q_delta, nq); LRK_LAUNCH_CHECK(h);
        LRK_NCCL(h, n->AllReduce(s->q_delta, s->q_delta, (size_t)nq, ncclFloat32, ncclSum, (ncclComm_t)h->comm, st));
        dsgd_apply_delta_kernel<<<lrk_ceil_div(nq, 256), 256, 0, st>>>(h->Q32, s->q_ref, s->q_delta, nq); LRK_LAUNCH_CHECK(h);
    }
    return LRK_OK;
}

static int dsgd_epoch(lrk_handle_s* h, float lr, float reg_u, float reg_i, double reg_b, int32_t epoch_idx, double* loss_out) {
    NcclApi* n = nccl_api();
    DsgdState* s = h->dsgd.get();
    cudaStream_t st = h->stream;
    const int world = h->world, rank = h->rank;
    const bool bpr_ = h->cfg.model == LRK_MODEL_BPR;
    LrkEpoch e;
    // safeguard: what this rank owns at the epoch boundary -- its user block and the item block it holds (BPR: the full item
    // matrix); the loss is all-reduced, so every rank takes the same rollback decision
    e.saved = [&] {
        std::vector<LrkSaved> v{{h->P32, &h->bk_P, (size_t)h->U * h->ld}};
        if (bpr_) v.push_back({h->Q32, &h->bk_Q, (size_t)h->I * h->ld});
        else v.push_back({s->qbuf[s->cur], &h->bk_Q, s->buf_floats});
        if (lrk_has_bias(h)) v.push_back({h->bu32, &h->bk_bu, (size_t)h->U});
        return v;
    };
    if (h->h_pnorm2) { h->pnorm2_prev = h->pnorm2_host; h->pnorm2_host = *h->h_pnorm2; }
    const SgdParams base = sgd_params(h, lr, reg_u, reg_i, reg_b, epoch_idx);
    bool fused_done = false;
    e.enqueue = [&](int) -> int {
        if (h->group) LRK_CUDA(h, cudaMemsetAsync(h->group->d_counter, 0, sizeof(unsigned int) * 64, st));
        if (s->trace < 0) { const char* t = getenv("LRK_DSGD_TRACE"); s->trace = t && atoi(t) ? 1 : 0; }
        if (s->trace && s->trace_ev.empty()) {
            s->trace_ev.resize((size_t)2 * world + 1);
            for (auto& ev : s->trace_ev) LRK_CUDA(h, cudaEventCreate(&ev));
        }
        if (s->trace) LRK_CUDA(h, cudaEventRecord(s->trace_ev[0], st));
        fused_done = false;
        int rc;
        if (bpr_) { if ((rc = dsgd_bpr_epoch(h, s, base))) return rc; }
        else if ((rc = dsgd_fused_epoch(h, s, base, &fused_done))) return rc;
        for (int sub = 0; !bpr_ && !fused_done && sub < world; ++sub) {
            const int b = dsgd_block_at(rank, world, sub);
            float* buf = s->qbuf[s->cur];
            const int64_t off = s->seg_off[(size_t)b], cnt = s->seg_off[(size_t)b + 1] - off;
            if (cnt > 0) {
                const SgdParams sp = sgd_segment(h, base, off, cnt, buf, buf + (size_t)s->max_blk * h->ld, s->bounds[(size_t)b]);
                if ((rc = h->group ? sgd_group_launch(h, sp, b) : sgd_launch(h, sp))) return rc;
            }
            if (s->trace) LRK_CUDA(h, cudaEventRecord(s->trace_ev[(size_t)2 * sub + 1], st));
            if (world > 1) {
                float* nxt = s->qbuf[s->cur ^ 1];
                LRK_NCCL(h, n->GroupStart());
                LRK_NCCL(h, n->Send(buf, s->buf_floats, ncclFloat32, dsgd_send_peer(rank, world), (ncclComm_t)h->comm, st));
                LRK_NCCL(h, n->Recv(nxt, s->buf_floats, ncclFloat32, dsgd_recv_peer(rank, world), (ncclComm_t)h->comm, st));
                LRK_NCCL(h, n->GroupEnd());
                s->cur ^= 1;
            }
            if (s->trace) LRK_CUDA(h, cudaEventRecord(s->trace_ev[(size_t)2 * sub + 2], st));
            s->cur_block = dsgd_block_at(rank, world, sub + 1);
        }
        LRK_NCCL(h, n->AllReduce(h->d_loss, h->d_loss, 1, ncclFloat64, ncclSum, (ncclComm_t)h->comm, st));
        return LRK_OK;
    };
    e.refresh_norm = k_lrk_models[h->cfg.model].damped && h->d_item_deg && !h->group;
    e.after_sync = [&]() -> int {
        if (!fused_done) return LRK_OK;
        int aborted = 0;
        LRK_CUDA(h, cudaMemcpy(&aborted, s->fused.d_abort, sizeof(int), cudaMemcpyDeviceToHost));
        if (aborted) return lrk_fail(h, LRK_ERR_NCCL, "lrk_sgd_epoch", "fused DSGD epoch: a ring neighbour did not answer within the spin limit", __FILE__, __LINE__);
        return LRK_OK;
    };
    // unlike the single-device path, the restored norm is not read back: the retry keeps the epoch's kernel variant
    e.rolled_back = [&]() { return e.refresh_norm ? refresh_user_norm2(h, false) : (int)LRK_OK; };
    const int rc = lrk_epoch(h, e, loss_out);
    if (s->trace && !fused_done && !bpr_ && (rc == LRK_OK || rc == LRK_ERR_DIVERGED)) {
        std::string line = "[dsgd rank " + std::to_string(rank) + " epoch " + std::to_string(epoch_idx) + "]";
        for (int sub = 0; sub < world; ++sub) {
            float k_ms = 0.f, x_ms = 0.f;
            cudaEventElapsedTime(&k_ms, s->trace_ev[(size_t)2 * sub], s->trace_ev[(size_t)2 * sub + 1]);
            cudaEventElapsedTime(&x_ms, s->trace_ev[(size_t)2 * sub + 1], s->trace_ev[(size_t)2 * sub + 2]);
            char buf[96];
            snprintf(buf, sizeof buf, " sub%d: kernel %.3f ms (%lld ratings) exchange %.3f ms;", sub, k_ms,
                     (long long)(s->seg_off[(size_t)dsgd_block_at(rank, world, sub) + 1] - s->seg_off[(size_t)dsgd_block_at(rank, world, sub)]), x_ms);
            line += buf;
        }
        fprintf(stderr, "%s total %.3f ms\n", line.c_str(), h->last_epoch_ms);
    }
    return rc;
}

// the full item factors into Q32 / bi32 (lrk_get_factors then refreshes the masters and copies them out); the masters are stale after it
static int dsgd_gather_items(lrk_handle_s* h) {
    NcclApi* n = nccl_api();
    DsgdState* s = h->dsgd.get();
    cudaStream_t st = h->stream;
    const int world = h->world;
    const bool biased = h->cfg.model == LRK_MODEL_BIASEDMF;
    // all-gather the rotating buffers (every rank holds block `cur_block`), then unpack into Q32 / bi32
    // (BPR keeps the full item matrix on every rank: nothing to gather)
    // (the gather buffer stays with the handle: cudaMalloc / cudaFree per call synchronise the device, and with the ring buffers
    // exported over CUDA IPC a cudaFree was seen to take 60-100 ms now and then at 8 ranks)
    const bool gather = h->cfg.model != LRK_MODEL_BPR;
    if (gather) { int rc_g = lrk_dev_alloc(h, &s->gather_buf, s->buf_floats * (size_t)world); if (rc_g) return rc_g; }
    float* all = s->gather_buf;
    ncclResult_t nr = gather ? n->AllGather(s->qbuf[s->cur], all, s->buf_floats, ncclFloat32, (ncclComm_t)h->comm, st) : ncclSuccess;
    cudaError_t e = cudaSuccess;
    if (nr == ncclSuccess && gather) {
        for (int r = 0; r < world && e == cudaSuccess; ++r) {
            const int b = dsgd_block_at(r, world, 0);     // between epochs rank r holds block r
            const int32_t first = s->bounds[b], rows = s->bounds[b + 1] - first;
            if (rows > 0) {
                dsgd_unpack_block_kernel<<<lrk_ceil_div((int64_t)rows * h->ld + rows, 256), 256, 0, st>>>(
                    h->Q32, biased ? h->bi32.ptr : nullptr, first, rows, h->ld, s->max_blk, all + s->buf_floats * (size_t)r);
                h->launches++;
                e = cudaGetLastError();
            }
        }
    }
    if (nr == ncclSuccess && e == cudaSuccess) e = cudaStreamSynchronize(st);
    LRK_NCCL(h, nr);
    LRK_CUDA(h, e);
    h->f64_valid = false;
    return LRK_OK;
}
