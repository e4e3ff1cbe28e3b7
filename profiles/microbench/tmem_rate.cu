// profiles/microbench/tmem_rate.cu -- measured rate of tensor-memory loads (tcgen05.ld -> LDTM) next to shared-memory loads
// (LDS.128) on B200 (sm_100a), in thread-instructions and bytes per clock per SM, and the LDTM -> use latency.  It answers
// whether profile lookups moved from shared memory into tensor memory add bandwidth to the LSU pipe or share it.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tmem_rate tmem_rate.cu && ./tmem_rate
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>

constexpr int ITERS = 2048;
constexpr int TCOLS = 512;  // the whole tensor memory of an SM: one CTA per SM

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                   "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
}
// wait::ld with the loaded registers as operands, so that no use of them is scheduled above the wait
__device__ __forceinline__ void tmem_wait16(uint32_t (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                   "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])::"memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
                 "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
                 "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
                 : "memory");
}

// Allocates all 512 columns (warp 0), fills them with a per-lane pattern (warps 0..3, one per lane quadrant) and returns the
// base address with this warp's lane quadrant in bits 31:16.
__device__ uint32_t tmem_setup(uint32_t *slot, uint32_t seed) {
    const int warp = threadIdx.x >> 5;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(TCOLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t base = *slot;
    const uint32_t lane_base = (uint32_t) (32 * (warp & 3)) << 16;
    if (warp < 4) {
        uint32_t v[16];
        for (int c = 0; c < TCOLS; c += 16) {
#pragma unroll
            for (int i = 0; i < 16; i++) v[i] = seed * (threadIdx.x + 1) + (uint32_t) (c + i);
            tmem_st16(base + lane_base + c, v);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    return base + lane_base;
}

__device__ void tmem_teardown(uint32_t base) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if ((threadIdx.x >> 5) == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base & 0xffffu), "r"(TCOLS) : "memory");
}

// NLDS LDS.128 and NLDTM tcgen05.ld.32x32b.x16 per loop iteration and thread; the LDTMs of one iteration share one wait.
template <int NLDS, int NLDTM>
__global__ void __launch_bounds__(1024) mix_kernel(uint32_t *out, long long *cycles, uint32_t seed) {
    __shared__ uint4 buf[2048];
    __shared__ uint32_t slot;
    for (int i = threadIdx.x; i < 2048; i += blockDim.x) buf[i] = make_uint4(i, seed, i ^ seed, 1);
    const uint32_t taddr = tmem_setup(&slot, seed);
    uint32_t acc0 = 0, acc1 = 0, acc2 = 0, acc3 = 0;
    int idx = threadIdx.x;
    const uint32_t wcol = (uint32_t) (threadIdx.x >> 5) * 16u;
    const long long t0 = clock64();
#pragma unroll 1
    for (int it = 0; it < ITERS; it++) {
        uint32_t v[NLDTM > 0 ? NLDTM : 1][16];
#pragma unroll
        for (int j = 0; j < NLDTM; j++) tmem_ld16(taddr + ((wcol + (uint32_t) (it * NLDTM + j) * 16u) & (TCOLS - 1)), v[j]);
#pragma unroll
        for (int r = 0; r < NLDS; r++) {
            const uint4 s = buf[(idx + r * 32) & 2047];
            acc0 ^= s.x; acc1 ^= s.y; acc2 ^= s.z; acc3 ^= s.w;
        }
        idx += 32 * NLDS;
#pragma unroll
        for (int j = 0; j < NLDTM; j++) {
            tmem_wait16(v[j]);
#pragma unroll
            for (int i = 0; i < 16; i += 4) { acc0 ^= v[j][i]; acc1 ^= v[j][i + 1]; acc2 ^= v[j][i + 2]; acc3 ^= v[j][i + 3]; }
        }
    }
    const long long t1 = clock64();
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc0 ^ acc1 ^ acc2 ^ acc3;
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
    tmem_teardown(taddr);
}

// Dependent chain in one warp: each load's first word (zero at run time) feeds the next address.
template <bool TMEM>
__global__ void __launch_bounds__(32) latency_kernel(uint32_t *out, long long *cycles, uint32_t seed) {
    __shared__ uint32_t sbuf[4096];
    __shared__ uint32_t slot;
    for (int i = threadIdx.x; i < 4096; i += 32) sbuf[i] = 0;
    const uint32_t taddr = tmem_setup(&slot, 0u);
    // zero column block 0 so that the chain reads 0 and stays put without the compiler knowing it
    uint32_t z[16];
#pragma unroll
    for (int i = 0; i < 16; i++) z[i] = 0;
    tmem_st16(taddr, z);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    __syncwarp();
    uint32_t col = 0, acc = 0;
    const int n = 1024;
    const long long t0 = clock64();
#pragma unroll 1
    for (int it = 0; it < n; it++) {
        if (TMEM) {
            uint32_t v[16];
            tmem_ld16(taddr + col, v);
            tmem_wait16(v);
            col = __shfl_sync(0xffffffffu, v[0], 0);   // uniform by construction, as the column of the scan kernel is
            acc ^= v[5];
        } else {
            col = sbuf[(col + threadIdx.x) & 4095];
            col = __shfl_sync(0xffffffffu, col, 0);
        }
    }
    const long long t1 = clock64();
    out[threadIdx.x] = col ^ acc ^ seed;
    if (threadIdx.x == 0) cycles[0] = t1 - t0;
    tmem_teardown(taddr);
}

struct Timer {
    cudaEvent_t e0, e1;
    Timer() { cudaEventCreate(&e0); cudaEventCreate(&e1); }
};

template <typename F>
static bool run(const char *name, F launch, int threads, double lds_per_thread, double ldtm_per_thread, long long *d_cyc, int blocks) {
    launch(); launch();
    cudaError_t err = cudaDeviceSynchronize();
    if (err != cudaSuccess) { printf("%s: %s\n", name, cudaGetErrorString(err)); return false; }
    Timer t;
    cudaEventRecord(t.e0);
    launch();
    cudaEventRecord(t.e1);
    cudaEventSynchronize(t.e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, t.e0, t.e1);
    long long cyc[1024];
    cudaMemcpy(cyc, d_cyc, sizeof(long long) * blocks, cudaMemcpyDeviceToHost);
    double mean = 0;
    for (int i = 0; i < blocks; i++) mean += (double) cyc[i];
    mean /= blocks;
    const double lds = lds_per_thread * threads / mean, ldtm = ldtm_per_thread * threads / mean;
    printf("%-34s %4d thr  LDS.128 %6.2f  LDTM.x16 %6.2f thread-instr/clk/SM   bytes %7.1f + %7.1f = %7.1f B/clk/SM   (%.0f cycles, %.0f MHz)\n",
           name, threads, lds, ldtm, 16 * lds, 64 * ldtm, 16 * lds + 64 * ldtm, mean, mean / (ms * 1e3));
    return true;
}

int main() {
    cudaDeviceProp p;
    cudaGetDeviceProperties(&p, 0);
    const int blocks = p.multiProcessorCount;  // one CTA per SM: it holds all 512 TMEM columns
    printf("device %s, %d SMs\n", p.name, blocks);
    uint32_t *d_out; long long *d_cyc;
    cudaMalloc(&d_out, sizeof(uint32_t) * 1024 * blocks);
    cudaMalloc(&d_cyc, sizeof(long long) * blocks);
    bool ok = true;
    for (int threads : {512, 1024}) {
#define MIX(A, B, NAME) \
        ok = ok && run(NAME, [&] { mix_kernel<A, B><<<blocks, threads>>>(d_out, d_cyc, 12345u); }, threads, (double) ITERS * A, (double) ITERS * B, d_cyc, blocks)
        MIX(8, 0, "LDS.128 alone");
        MIX(0, 2, "LDTM.x16 alone (2 per wait)");
        MIX(0, 4, "LDTM.x16 alone (4 per wait)");
        MIX(4, 1, "LDS:LDTM 1:1 bytes");
        MIX(8, 1, "LDS:LDTM 2:1 bytes");
        MIX(8, 2, "LDS:LDTM 1:1 bytes (2 LDTM/wait)");
#undef MIX
    }
    for (int t = 0; t < 2 && ok; t++) {
        long long cyc = 0;
        if (t) latency_kernel<true><<<1, 32>>>(d_out, d_cyc, 1u); else latency_kernel<false><<<1, 32>>>(d_out, d_cyc, 1u);
        cudaError_t err = cudaDeviceSynchronize();
        if (err != cudaSuccess) { printf("latency: %s\n", cudaGetErrorString(err)); ok = false; break; }
        cudaMemcpy(&cyc, d_cyc, sizeof(long long), cudaMemcpyDeviceToHost);
        printf("%-34s %.1f cycles per dependent load (incl. one SHFL)\n", t ? "LDTM.x16 -> use latency" : "LDS.32 -> use latency", cyc / 1024.0);
    }
    return ok ? 0 : 1;
}
