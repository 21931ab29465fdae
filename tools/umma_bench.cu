// Microbenchmark: cycles per tcgen05.mma (kind::f16, cta_group::1, M=128) as a
// function of N, smem layout / alignment of the A operand, and the number of
// TMEM accumulators the MMAs rotate over; and per cta_group::2 MMA (clusters of
// two CTAs, M=256, each CTA holding its 128 rows of A and half of B's N
// columns).  Timing only; operands are zeros.  Also prints how many clusters of
// two a conv-stack-sized CTA (one per SM) can keep resident.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/umma_bench tools/umma_bench.cu
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

struct Params {
    int n;           // UMMA N
    int a_off;       // byte offset added to the A start address (tap shift)
    int n_acc;       // accumulators rotated over
    int layout;      // 0 = no swizzle (LBO/SBO given), 2 = SWIZZLE_128B
    int a_lbo, a_sbo, b_lbo, b_sbo;
    int mmas;        // MMAs per timed batch
    int a_stride;    // bytes added to A start per MMA (k advance), wraps at 64 KB
    int b_stride;
    int ts;          // 1: A operand from TMEM
};

__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo, uint32_t sbo, int layout) {
    return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}

__global__ void __launch_bounds__(128, 1) bench(Params p, long long* cycles) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_base_s;
    for (int i = threadIdx.x; i < 200 * 1024 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base_s)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;
    if (threadIdx.x < 32) {
        // warp-uniform issue loop: every lane runs it, one elected lane issues
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.n >> 3) << 17) | (8u << 24);
        const uint64_t da0 = make_desc(smem_u32(smem) + p.a_off, p.a_lbo, p.a_sbo, p.layout);
        const uint64_t db0 = make_desc(smem_u32(smem) + 96 * 1024, p.b_lbo, p.b_sbo, p.layout);
        const uint32_t acc_stride = 512 / p.n_acc;
        const uint32_t a_step = p.a_stride >> 4, b_step = p.b_stride >> 4;
        uint32_t parity = 0;
        long long best = 1ll << 60;
        for (int rep = 0; rep < 5; ++rep) {
            long long t0 = clock64();
            for (int i = 0; i < p.mmas; i += 8) {
                uint32_t elected;
                asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}" : "=r"(elected));
                if (elected) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint32_t d = tmem + ((j) % p.n_acc) * acc_stride;
                        const uint64_t db = db0 + (uint64_t)((j & 3) * b_step);
                        if (p.ts) {
                            asm volatile(
                                "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %4, 0;\n\t"
                                "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, q;\n\t}"
                                ::"r"(d), "r"(tmem + 256), "l"(db), "r"(idesc), "r"(1u) : "memory");
                        } else {
                            const uint64_t da = da0 + (uint64_t)((j & 3) * a_step);
                            asm volatile(
                                "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %4, 0;\n\t"
                                "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, q;\n\t}"
                                ::"r"(d), "l"(da), "l"(db), "r"(idesc), "r"(1u) : "memory");
                        }
                    }
                }
                __syncwarp();
            }
            uint32_t elected;
            asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}" : "=r"(elected));
            if (elected)
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&bar)) : "memory");
            __syncwarp();
            uint32_t done;
            do {
                asm volatile("{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}"
                             : "=r"(done) : "r"(smem_u32(&bar)), "r"(parity) : "memory");
            } while (!done);
            parity ^= 1;
            long long t1 = clock64();
            if (t1 - t0 < best) best = t1 - t0;
        }
        if (threadIdx.x == 0) cycles[blockIdx.x] = best;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x < 32)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// cta_group::2: rank 0 of each cluster issues M=256 MMAs; A is the 128 rows of
// each CTA's own smem, B the N/2 columns each CTA holds at the same address.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1) bench_pair(Params p, long long* cycles) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_base_s;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    for (int i = threadIdx.x; i < 200 * 1024 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base_s)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;
    if (rank == 0 && threadIdx.x < 32) {
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.n >> 3) << 17) | (16u << 24);
        const uint64_t da0 = make_desc(smem_u32(smem) + p.a_off, p.a_lbo, p.a_sbo, p.layout);
        const uint64_t db0 = make_desc(smem_u32(smem) + 96 * 1024, p.b_lbo, p.b_sbo, p.layout);
        const uint32_t acc_stride = 512 / p.n_acc;
        const uint32_t a_step = p.a_stride >> 4, b_step = p.b_stride >> 4;
        uint32_t parity = 0;
        long long best = 1ll << 60;
        for (int rep = 0; rep < 5; ++rep) {
            long long t0 = clock64();
            for (int i = 0; i < p.mmas; i += 8) {
                uint32_t elected;
                asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}" : "=r"(elected));
                if (elected) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const uint32_t d = tmem + ((j) % p.n_acc) * acc_stride;
                        const uint64_t da = da0 + (uint64_t)((j & 3) * a_step);
                        const uint64_t db = db0 + (uint64_t)((j & 3) * b_step);
                        asm volatile(
                            "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %4, 0;\n\t"
                            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, q;\n\t}"
                            ::"r"(d), "l"(da), "l"(db), "r"(idesc), "r"(1u) : "memory");
                    }
                }
                __syncwarp();
            }
            uint32_t elected;
            asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}" : "=r"(elected));
            if (elected)
                asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                             ::"r"(smem_u32(&bar)), "h"((uint16_t)1) : "memory");
            __syncwarp();
            uint32_t done;
            do {
                asm volatile("{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}"
                             : "=r"(done) : "r"(smem_u32(&bar)), "r"(parity) : "memory");
            } while (!done);
            parity ^= 1;
            long long t1 = clock64();
            if (t1 - t0 < best) best = t1 - t0;
        }
        if (threadIdx.x == 0) cycles[blockIdx.x / 2] = best;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (threadIdx.x < 32)
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// stands in for the conv-stack kernel in the cluster-occupancy query
__global__ void __launch_bounds__(576, 1) occupancy_probe() {}

static void run_pair(const char* name, Params p, int clusters) {
    long long* d;
    cudaMalloc(&d, clusters * sizeof(long long));
    cudaFuncSetAttribute(bench_pair, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    bench_pair<<<2 * clusters, 128, 200 * 1024>>>(p, d);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("%-44s ERROR %s\n", name, cudaGetErrorString(e)); exit(1); }
    long long* h = (long long*)malloc(clusters * sizeof(long long));
    cudaMemcpy(h, d, clusters * sizeof(long long), cudaMemcpyDeviceToHost);
    long long worst = 0, sum = 0;
    for (int i = 0; i < clusters; ++i) { sum += h[i]; if (h[i] > worst) worst = h[i]; }
    printf("%-44s N=%3d clusters=%3d  cycles/MMA avg %.1f max %.1f\n", name, p.n, clusters,
           (double)sum / clusters / p.mmas, (double)worst / p.mmas);
    cudaFree(d); free(h);
}

static void max_clusters(int threads, int smem) {
    cudaFuncSetAttribute(occupancy_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(occupancy_probe, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * 148);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    int n = -1;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&n, (void*)occupancy_probe, &cfg);
    printf("max active clusters of 2: threads=%d smem=%d B -> %d (%s)\n", threads, smem, n,
           cudaGetErrorString(e));
}

static void run(const char* name, Params p, int grid) {
    long long* d;
    cudaMalloc(&d, grid * sizeof(long long));
    cudaFuncSetAttribute(bench, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    bench<<<grid, 128, 200 * 1024>>>(p, d);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("%-44s ERROR %s\n", name, cudaGetErrorString(e)); exit(1); }
    long long* h = (long long*)malloc(grid * sizeof(long long));
    cudaMemcpy(h, d, grid * sizeof(long long), cudaMemcpyDeviceToHost);
    long long worst = 0, sum = 0;
    for (int i = 0; i < grid; ++i) { sum += h[i]; if (h[i] > worst) worst = h[i]; }
    printf("%-44s N=%3d grid=%3d  cycles/MMA avg %.1f max %.1f\n", name, p.n, grid,
           (double)sum / grid / p.mmas, (double)worst / p.mmas);
    cudaFree(d); free(h);
}

int main() {
    const int RB = 130;
    for (int grid : {1, 148}) {
        Params base{80, 0, 1, 0, RB * 16, 128, 80 * 16, 128, 256, 0, 0, 0};
        run("none  N=80 aligned 1acc static", base, grid);
        Params q = base; q.a_off = 16; run("none  N=80 +16B 1acc", q, grid);
        q = base; q.n_acc = 4; run("none  N=80 aligned 4acc", q, grid);
        q = base; q.a_stride = 2 * RB * 16; q.b_stride = 2 * 80 * 16; run("none  N=80 aligned 1acc k-advance", q, grid);
        q = base; q.n = 256; q.b_lbo = 256 * 16; run("none  N=256 aligned 1acc", q, grid);
        q = base; q.n = 128; q.b_lbo = 128 * 16; run("none  N=128 aligned 1acc", q, grid);
        q = base; q.n = 160; q.b_lbo = 160 * 16; run("none  N=160 aligned 1acc", q, grid);
        q = base; q.n = 16; run("none  N=16 aligned 1acc", q, grid);
        q = base; q.n = 240; q.b_lbo = 240 * 16; q.n_acc = 2; run("none  N=240 2acc", q, grid);
        q = base; q.n = 240; q.b_lbo = 240 * 16; q.n_acc = 2; q.a_lbo = 128 * 16; q.a_stride = 2 * 128 * 16; q.b_stride = 2 * 240 * 16; run("none  N=240 2acc k-advance", q, grid);
        q = base; q.layout = 2; q.a_lbo = 16; q.a_sbo = 1024; q.b_lbo = 16; q.b_sbo = 1024; run("sw128 N=80 1acc", q, grid);
        q.n = 256; run("sw128 N=256 1acc", q, grid);
        q = base; q.layout = 6; q.a_lbo = 16; q.a_sbo = 256; q.b_lbo = 16; q.b_sbo = 256; run("sw32  N=80 1acc", q, grid);
        q = base; q.ts = 1; run("TS    N=80 A in TMEM", q, grid);
        q = base; q.ts = 1; q.n = 256; q.b_lbo = 256 * 16; run("TS    N=256 A in TMEM", q, grid);
    }
    for (int clusters : {1, 74}) {
        // B half per CTA: [k-group][N/2 rows][8] (LBO = N/2 * 16)
        Params base{80, 0, 1, 0, RB * 16, 128, 40 * 16, 128, 256, 0, 0, 0};
        run_pair("2cta none N=80 aligned 1acc", base, clusters);
        Params q = base; q.a_off = 16; run_pair("2cta none N=80 +16B 1acc", q, clusters);
        q = base; q.n_acc = 4; run_pair("2cta none N=80 aligned 4acc", q, clusters);
        q = base; q.a_stride = 2 * RB * 16; q.b_stride = 2 * 40 * 16; run_pair("2cta none N=80 aligned 1acc k-advance", q, clusters);
        q = base; q.n = 128; q.b_lbo = 64 * 16; run_pair("2cta none N=128 aligned 1acc", q, clusters);
        q = base; q.n = 256; q.b_lbo = 128 * 16; run_pair("2cta none N=256 aligned 1acc", q, clusters);
        q = base; q.n = 16; q.b_lbo = 8 * 16; run_pair("2cta none N=16 aligned 1acc", q, clusters);
    }
    for (int smem : {150 * 1024, 180 * 1024, 200 * 1024, 227 * 1024}) {
        max_clusters(576, smem);
        max_clusters(320, smem);
    }
    return 0;
}
