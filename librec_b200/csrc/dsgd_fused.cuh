// One persistent kernel per DSGD epoch with the ring exchange inside it -- the default of the rating models between processes
// (LRK_DSGD_FUSED=0 selects the sub-epoch loop of dsgd.cuh: SGD kernel + grouped ncclSend/ncclRecv per stratum; that loop is also
// what BPR and communicators without working CUDA IPC / peer access use).  r02, 8 x B200, config C4 (PMF k=128,
// Netflix shape, strong scaling): 2.04 ms per epoch = 49.3 G updates/s against 2.17 ms = 46.4 G with the NCCL ring, parity checks
// (conflict-free epoch = oracle to 2e-8, C1 within 1e-3) green at 2 and 8 ranks (profiles/r02_*).
//
// Why: after r01 a DSGD stratum runs at the whole-matrix rate, so what separates N GPUs from N x one GPU is per sub-epoch the
// NCCL send/recv pair (0.026-0.03 ms when both ranks are in step), launch gaps and the wait for the slower neighbour.  NCCL's
// copy kernels cannot overlap with the epoch kernel (it occupies every SM), so a second stream does not help.
//
// How: every rank maps its ring neighbours' block buffers and flag words with CUDA IPC (handles exchanged once through the NCCL
// communicator; the ranks of a single-process multi handle take them as plain peer pointers, csrc/multi.cuh).  The epoch kernel is launched cooperatively and loops over the G strata:
//   wait   until the block for this stratum has arrived in my buffer b        (ready[b]     >= seq, written by rank+1)
//   train  the stratum's COO segment against buffer b                          (sgd_rating_body.inc, the same tile code)
//   grid.sync
//   wait   until rank-1 no longer needs its buffer 1-b                         (peer_free[1-b] >= seq, written by rank-1)
//   push   buffer b into rank-1's buffer 1-b with coalesced peer stores over NVLink; __threadfence_system; grid.sync
//   signal rank-1: ready[1-b] = seq + 1 (st.release.sys);  rank+1: its buffer b here is free again (peer_free[b] = seq + 1)
// and finally waits for the block of the NEXT epoch's first stratum, so that the buffer is complete when the kernel ends
// (snapshot, all-gather in lrk_get_factors and the next launch read it).  seq = seq0 + stratum increases monotonically over the
// epochs, so no flag is ever reset.  A spin that exceeds spin_limit cycles raises `abort` in every rank's own memory and the
// remaining strata fall through (all grid.sync calls are still executed), the host then reports LRK_ERR_NCCL.
#pragma once
#include "lrk_common.cuh"
#include "sgd.cuh"
#include "sgd_group.cuh"
#include <cooperative_groups.h>

#define LRK_FUSED_MAX_WORLD 8

struct DsgdFusedParams {
    SgdParams seg[LRK_FUSED_MAX_WORLD];     // per stratum: COO segment, n, tile_mul, degrees, in-flight share; Q / bi filled in-kernel
    float* qbuf[2];                         // my rotating block buffers
    float* peer_qbuf[2];                    // rank-1's buffers (push target)
    unsigned long long* ready;              // mine [2]: written by rank+1
    unsigned long long* peer_free;          // mine [2]: written by rank-1
    unsigned long long* prev_ready;         // rank-1's ready[2]
    unsigned long long* next_peer_free;     // rank+1's peer_free[2]
    unsigned long long seq0;
    int cur0, world;
    long long buf_floats, bi_off;           // floats per buffer; offset of the bias slice (max_blk * ld)
    int* abort;
    long long spin_limit;                   // clock64 cycles
};

__device__ __forceinline__ unsigned long long lrk_ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void lrk_st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// thread 0 of every CTA spins; returns false once any wait of this rank has timed out.  The verdict is CTA-uniform (it gates
// code that contains __syncthreads): thread 0 samples the abort flag once and hands it to the others through shared memory.
__device__ __forceinline__ bool lrk_fused_wait(const unsigned long long* flag, unsigned long long want, int* abort_flag, long long spin_limit) {
    __shared__ int s_ok;
    if (threadIdx.x == 0) {
        const long long t0 = clock64();
        while (lrk_ld_acquire_sys(flag) < want) {
            if (*(volatile int*)abort_flag) break;
            if (clock64() - t0 > spin_limit) { atomicExch(abort_flag, 1); break; }
            __nanosleep(100);
        }
        s_ok = *(volatile int*)abort_flag == 0;
    }
    __syncthreads();
    const bool ok = s_ok != 0;
    __syncthreads();                       // s_ok is reused by the next wait
    return ok;
}

template <int G, int V, bool BIASED, bool TRACK>
__global__ void __launch_bounds__(256, (G * V <= 16 && !TRACK) ? 4 : ((G * V <= 32) ? 3 : 1)) dsgd_fused_epoch_kernel(DsgdFusedParams fp) {
    constexpr bool ATOMIC = true;
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long gthreads = (long long)gridDim.x * blockDim.x;
    for (int t = 0; t < fp.world; ++t) {
        const int b = (fp.cur0 + t) & 1;
        const unsigned long long seq = fp.seq0 + (unsigned long long)t;
        bool ok = lrk_fused_wait(fp.ready + b, seq, fp.abort, fp.spin_limit);
        if (ok) {
            SgdParams p = fp.seg[t];
            p.Q = fp.qbuf[b];
            p.bi = fp.qbuf[b] + fp.bi_off;
#include "sgd_rating_body.inc"
            block_loss_commit(loss_d, p.loss);
        }
        __threadfence();
        grid.sync();
        ok = lrk_fused_wait(fp.peer_free + (b ^ 1), seq, fp.abort, fp.spin_limit);
        if (ok) {
            const float4* src = reinterpret_cast<const float4*>(fp.qbuf[b]);
            float4* dst = reinterpret_cast<float4*>(fp.peer_qbuf[b ^ 1]);
            const long long n4 = fp.buf_floats >> 2;
            for (long long i = gtid; i < n4; i += gthreads) dst[i] = __ldcg(src + i);
            for (long long i = (n4 << 2) + gtid; i < fp.buf_floats; i += gthreads) fp.peer_qbuf[b ^ 1][i] = __ldcg(fp.qbuf[b] + i);
        }
        __threadfence_system();
        grid.sync();
        if (gtid == 0 && *(volatile int*)fp.abort == 0) {
            lrk_st_release_sys(fp.prev_ready + (b ^ 1), seq + 1ull);
            lrk_st_release_sys(fp.next_peer_free + b, seq + 1ull);
        }
    }
    // the block of the next epoch's first stratum must be complete before the kernel ends
    lrk_fused_wait(fp.ready + ((fp.cur0 + fp.world) & 1), fp.seq0 + (unsigned long long)fp.world, fp.abort, fp.spin_limit);
}

// the same epoch over the unit-ordered stream of the user-group kernel (sgd_group.cuh): per stratum the CTAs pull units from the
// stratum's work counter (zeroed by the host before the launch), then the ring step as above
struct DsgdFusedGroupParams {
    SgdGroupParams seg[LRK_FUSED_MAX_WORLD];   // per stratum: units, counter, degrees, in-flight share; Q / bi filled in-kernel
    float* qbuf[2];
    float* peer_qbuf[2];
    unsigned long long* ready;
    unsigned long long* peer_free;
    unsigned long long* prev_ready;
    unsigned long long* next_peer_free;
    unsigned long long seq0;
    int cur0, world;
    long long buf_floats, bi_off;
    int* abort;
    long long spin_limit;
};

template <int G, int V, bool BIASED>
__global__ void __launch_bounds__(256, 2) dsgd_fused_group_epoch_kernel(DsgdFusedGroupParams fp) {
    extern __shared__ float4 lrk_fused_group_smem4[];
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long gthreads = (long long)gridDim.x * blockDim.x;
    double loss_d = 0.0;
    for (int t = 0; t < fp.world; ++t) {
        const int b = (fp.cur0 + t) & 1;
        const unsigned long long seq = fp.seq0 + (unsigned long long)t;
        bool ok = lrk_fused_wait(fp.ready + b, seq, fp.abort, fp.spin_limit);
        if (ok && fp.seg[t].n_units > 0) {
            SgdGroupParams p = fp.seg[t];
            p.Q = fp.qbuf[b];
            p.bi = fp.qbuf[b] + fp.bi_off;
            sgd_group_segment<G, V, BIASED>(p, reinterpret_cast<float*>(lrk_fused_group_smem4), loss_d);
        }
        __threadfence();
        grid.sync();
        ok = lrk_fused_wait(fp.peer_free + (b ^ 1), seq, fp.abort, fp.spin_limit);
        if (ok) {
            const float4* src = reinterpret_cast<const float4*>(fp.qbuf[b]);
            float4* dst = reinterpret_cast<float4*>(fp.peer_qbuf[b ^ 1]);
            const long long n4 = fp.buf_floats >> 2;
            for (long long i = gtid; i < n4; i += gthreads) dst[i] = __ldcg(src + i);
        }
        __threadfence_system();
        grid.sync();
        if (gtid == 0 && *(volatile int*)fp.abort == 0) {
            lrk_st_release_sys(fp.prev_ready + (b ^ 1), seq + 1ull);
            lrk_st_release_sys(fp.next_peer_free + b, seq + 1ull);
        }
    }
    lrk_fused_wait(fp.ready + ((fp.cur0 + fp.world) & 1), fp.seq0 + (unsigned long long)fp.world, fp.abort, fp.spin_limit);
    block_loss_commit(loss_d, fp.seg[0].loss);
}

struct DsgdFused {
    int enabled = -1;                        // -1: environment not read yet
    bool mapped = false;
    float* my_qbuf[2] = {nullptr, nullptr};  // the buffers the mappings were made for
    LrkBuf<unsigned long long> d_flags;      // [0,1] ready, [2,3] peer_free
    LrkBuf<int> d_abort;
    float* peer_qbuf[2] = {nullptr, nullptr};
    unsigned long long* prev_flags = nullptr;
    unsigned long long* next_flags = nullptr;
    void* opened[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int n_opened = 0;
    unsigned long long seq = 0;
    bool needs_reset = false;                // lrk_set_factors re-packed the ring (buffer 0 holds the block again): restart the flag sequence
};

static void dsgd_fused_unmap(DsgdFused* f) {
    for (int i = 0; i < f->n_opened; ++i) if (f->opened[i]) cudaIpcCloseMemHandle(f->opened[i]);
    f->n_opened = 0;
    f->d_flags.reset(); f->d_abort.reset(); f->mapped = false;
}
