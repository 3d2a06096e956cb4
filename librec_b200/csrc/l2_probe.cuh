// L2 roofline probe for the SGD epoch kernels (VERDICT r01, "give SGD a roofline that can read below 1").
// The epoch kernels do not stream: per rating they gather two factor rows through L2 (ld.global.cg, one float4 per lane) and
// apply two vector reductions (red.global.add.v4.f32) to the same rows, on a factor set that is resident in the 126 MB L2
// (ML-20M shape: 42 MB).  Their bound is therefore the rate at which the L2 serves random row gathers and row REDs, not HBM.
// This kernel issues exactly those two instructions, with the same widths and the same row length, against uniformly random rows
// of a working set of the given size, and nothing else (no dot product, no dependent shuffles): its throughput is the peak the
// epoch kernel's L2 traffic is measured against in bench.py (roofline.bound = "l2").
//   mode 0: gathers only   mode 1: REDs only   mode 2: one RED per gather (the epoch kernel's mix)
#pragma once
#include "lrk_common.cuh"

template <int G, int MODE>
__global__ void __launch_bounds__(256) l2_probe_kernel(float* __restrict__ base, uint32_t rows, int ld, int steps, uint32_t seed, float* sink) {
    const int lane = threadIdx.x & 31;
    const int sub = lane % G, grp = lane / G;
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t s = (gwarp * (32u / G) + (uint32_t)grp) * 2654435761u + seed;      // one stream of row numbers per lane group
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    constexpr int UNROLL = 8;                                                   // independent rows in flight per lane group
    for (int it = 0; it < steps; it += UNROLL) {
        float4 v[UNROLL];
        uint32_t r[UNROLL];
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) {
            s = s * 1664525u + 1013904223u;
            r[j] = __umulhi(s, rows);
            if (MODE != 1) v[j] = __ldcg(reinterpret_cast<const float4*>(base + (size_t)r[j] * ld + sub * 4));
            else v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < UNROLL; ++j) {
            acc.x += v[j].x; acc.y += v[j].y; acc.z += v[j].z; acc.w += v[j].w;
            if (MODE != 0) {
                float* a = base + (size_t)r[j] * ld + sub * 4;
                asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(a), "f"(0.f), "f"(0.f), "f"(0.f), "f"(0.f) : "memory");
            }
        }
    }
    if (acc.x + acc.y + acc.z + acc.w == 123456.789f) *sink = acc.x;             // keeps the loads alive
}

// out[0..2] = GB/s of row bytes moved through L2 (gathered bytes + reduced bytes) for modes 0, 1, 2
static int l2_probe_run(lrk_handle_s* h, size_t working_set_bytes, int row_floats, double out[3]) {
    cudaStream_t st = h->stream;
    LRK_REQUIRE(h, row_floats == 64 || row_floats == 128, "row length must be 64 or 128 floats (the k=64 / k=128 layouts)");
    const int G = row_floats / 4;
    const uint32_t rows = (uint32_t)(working_set_bytes / (sizeof(float) * (size_t)row_floats));
    LRK_REQUIRE(h, rows >= 1024, "working set too small");
    LrkBuf<float> buf, sink;
    int rc;
    if ((rc = lrk_dev_alloc(h, &buf, (size_t)rows * row_floats))) return rc;
    if ((rc = lrk_dev_alloc(h, &sink, 1))) return rc;
    cudaError_t e = cudaMemsetAsync(buf, 0, sizeof(float) * (size_t)rows * row_floats, st);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (e == cudaSuccess) e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    const int grid = h->sm_count * 4, steps = 4096;
    for (int mode = 0; mode < 3 && e == cudaSuccess; ++mode) {
        float best = 1e30f;
        for (int rep = 0; rep < 4 && e == cudaSuccess; ++rep) {          // first repetition warms the L2
            cudaEventRecord(e0, st);
            if (G == 16) {
                if (mode == 0) l2_probe_kernel<16, 0><<<grid, 256, 0, st>>>(buf, rows, row_floats, steps, 17u + rep, sink);
                else if (mode == 1) l2_probe_kernel<16, 1><<<grid, 256, 0, st>>>(buf, rows, row_floats, steps, 17u + rep, sink);
                else l2_probe_kernel<16, 2><<<grid, 256, 0, st>>>(buf, rows, row_floats, steps, 17u + rep, sink);
            } else {
                if (mode == 0) l2_probe_kernel<32, 0><<<grid, 256, 0, st>>>(buf, rows, row_floats, steps, 17u + rep, sink);
                else if (mode == 1) l2_probe_kernel<32, 1><<<grid, 256, 0, st>>>(buf, rows, row_floats, steps, 17u + rep, sink);
                else l2_probe_kernel<32, 2><<<grid, 256, 0, st>>>(buf, rows, row_floats, steps, 17u + rep, sink);
            }
            h->launches++;
            e = cudaGetLastError();
            cudaEventRecord(e1, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            float ms = 0.f;
            if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
            if (rep > 0 && ms < best) best = ms;
        }
        const double row_ops = (double)grid * 8.0 * (32.0 / G) * steps;    // rows touched per launch
        const double bytes = row_ops * row_floats * 4.0 * (mode == 2 ? 2.0 : 1.0);
        out[mode] = bytes / ((double)best * 1e-3) / 1e9;
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    LRK_CUDA(h, e);
    return LRK_OK;
}
