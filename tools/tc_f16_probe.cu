// Probe for the fp16-split conditioner path (flow_tc_h.cu, round 2):
//   (1) layout check: tcgen05.mma.kind::f16 with the A operand in TENSOR MEMORY as packed half2 (column c of lane m
//       holds K elements 2c (low half) and 2c+1 (high half)), B in shared memory K-major / 128-byte swizzle,
//       fp32 accumulator — compared with a host product;
//   (2) issue-rate measurement: cycles per instruction and TFLOP/s per SM of kind::tf32 (K=8) and kind::f16 (K=16)
//       at N = 64 / 128 / 256, TS mode, back-to-back accumulating MMAs from one thread (what the flow kernels do).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O2 -std=c++17 -I nf_b200/csrc tools/tc_f16_probe.cu -o oracle/_ref/tc_f16_probe
#include <cstdio>
#include <cmath>
#include <vector>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include "tc_common.cuh"

__device__ __forceinline__ void mma_f16_ts(uint32_t d, uint32_t a, uint64_t db, uint32_t idesc, uint32_t acc) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(d), "r"(a), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
// instruction descriptor for kind::f16: c_format F32 (1) at [4,6), a/b format F16 (0) at [7,10)/[10,13)
__host__ __device__ constexpr uint32_t idesc_f16(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// byte offset of (row, k) in a [rows x 64] fp16 K-major operand: 128 B per row, 8-row groups of 1024 B, 16-byte chunks
// XOR-swizzled with row % 8
__host__ __device__ static inline int off16(int row, int k) {
    return (row >> 3) * 1024 + (row & 7) * 128 + ((((k >> 3) ^ (row & 7)) << 4) | ((k & 7) << 1));
}

// ---- (1) layout ------------------------------------------------------------------------------------------------
__global__ void layout_probe(const __half* Ag /*[128][64]*/, const __half* Bg /*[64][64] (n,k)*/, float* Dg /*[128][64]*/) {
    extern __shared__ char smraw[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tb_s;
    char* sm = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(smraw) + 1023) & ~(uintptr_t)1023);
    for (int i = threadIdx.x; i < 64 * 64; i += blockDim.x) {
        const int n = i / 64, k = i % 64;
        *reinterpret_cast<__half*>(sm + off16(n, k)) = Bg[i];
    }
    if (threadIdx.x == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tb_s)), "r"(128));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tb = tb_s;
    const uint32_t lane_base = ((uint32_t)((threadIdx.x >> 5) * 32) << 16);
    {   // thread m writes row m of A as 32 packed columns at TMEM columns [64, 96)
        float packed[32];
        for (int c = 0; c < 32; ++c) {
            const __half2 h = __halves2half2(Ag[threadIdx.x * 64 + 2 * c], Ag[threadIdx.x * 64 + 2 * c + 1]);   // .x = low half
            packed[c] = __uint_as_float(*reinterpret_cast<const uint32_t*>(&h));
        }
        tc_st32(tb + 64 + lane_base, packed);
        tc_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (threadIdx.x == 0) {
        const uint32_t idesc = idesc_f16(128, 64);
        for (int ks = 0; ks < 4; ++ks)       // K = 16 per instruction: 8 TMEM columns of A, 32 bytes of a B row
            mma_f16_ts(tb, tb + 64 + ks * 8, tc_desc(smem_u32(sm) + ks * 32), idesc, ks > 0);
        tc_commit(&bar);
    }
    mbar_wait(&bar, 0);
    tc_fence_after();
    float v[64];
    tc_ld32(tb + lane_base, v);
    tc_ld32(tb + 32 + lane_base, v + 32);
    tc_ld_wait();
    for (int j = 0; j < 64; ++j) Dg[threadIdx.x * 64 + j] = v[j];
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(128));
}

// ---- (2) rates ---------------------------------------------------------------------------------------------------
template <int KIND /*0 tf32, 1 f16*/>
__global__ void rate_probe(int N, int iters, long long* cycles) {
    extern __shared__ char smraw[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tb_s;
    char* sm = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(smraw) + 1023) & ~(uintptr_t)1023);
    for (int i = threadIdx.x; i < 256 * 128 / 4; i += blockDim.x) reinterpret_cast<float*>(sm)[i] = 0.f;
    if (threadIdx.x == 0) { mbar_init(&bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tb_s)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tb = tb_s;
    {
        float z[32];
        for (int c = 0; c < 32; ++c) z[c] = 0.f;
        const uint32_t lane_base = ((uint32_t)((threadIdx.x >> 5) * 32) << 16);
        tc_st32(tb + 256 + lane_base, z);
        tc_st32(tb + 288 + lane_base, z);
        tc_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (threadIdx.x == 0) {
        const uint32_t idesc = KIND == 0 ? tc_idesc(128, N) : idesc_f16(128, N);
        const long long t0 = clock64();
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
                const uint64_t db = tc_desc(smem_u32(sm) + (ks & 3) * 32);
                if (KIND == 0) tc_mma_tf32_ts(tb, tb + 256 + ks * 8, db, idesc, 1);
                else mma_f16_ts(tb, tb + 256 + ks * 8, db, idesc, 1);
            }
        }
        tc_commit(&bar);
        mbar_wait(&bar, 0);
        cycles[blockIdx.x] = clock64() - t0;
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(512));
}

int main() {
    // (1)
    std::vector<__half> A(128 * 64), B(64 * 64);
    std::vector<float> Af(128 * 64), Bf(64 * 64), D(128 * 64);
    unsigned s = 12345u;
    auto rnd = [&]() { s = s * 1664525u + 1013904223u; return ((s >> 8) & 0xFFFF) / 65536.0f - 0.5f; };
    for (int i = 0; i < 128 * 64; ++i) { A[i] = __float2half(rnd()); Af[i] = __half2float(A[i]); }
    for (int i = 0; i < 64 * 64; ++i) { B[i] = __float2half(rnd()); Bf[i] = __half2float(B[i]); }
    __half *dA, *dB; float* dD;
    cudaMalloc(&dA, A.size() * 2); cudaMalloc(&dB, B.size() * 2); cudaMalloc(&dD, D.size() * 4);
    cudaMemcpy(dA, A.data(), A.size() * 2, cudaMemcpyHostToDevice);
    cudaMemcpy(dB, B.data(), B.size() * 2, cudaMemcpyHostToDevice);
    cudaFuncSetAttribute(layout_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 + 1024);
    layout_probe<<<1, 128, 16384 + 1024>>>(dA, dB, dD);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("layout probe failed: %s\n", cudaGetErrorString(e)); return 1; }
    cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost);
    double maxerr = 0.0, maxerr_swapped = 0.0;
    for (int m = 0; m < 128; ++m)
        for (int n = 0; n < 64; ++n) {
            double ref = 0.0, sw = 0.0;
            for (int k = 0; k < 64; ++k) { ref += (double)Af[m * 64 + k] * Bf[n * 64 + k]; sw += (double)Af[m * 64 + (k ^ 1)] * Bf[n * 64 + k]; }
            maxerr = fmax(maxerr, fabs(ref - D[m * 64 + n]));
            maxerr_swapped = fmax(maxerr_swapped, fabs(sw - D[m * 64 + n]));
        }
    printf("{\"probe\": \"f16_ts_layout\", \"max_abs_err_low_half_is_even_k\": %.3e, \"max_abs_err_if_swapped\": %.3e, \"ok\": %s}\n",
           maxerr, maxerr_swapped, maxerr < 1e-4 ? "true" : "false");
    // (2)
    int dev = 0, sms = 0, khz = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, dev);
    long long* dcyc;
    cudaMalloc(&dcyc, sizeof(long long) * sms);
    std::vector<long long> cyc(sms);
    const int smem = 256 * 128 + 1024;
    cudaFuncSetAttribute(rate_probe<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(rate_probe<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    for (int kind = 0; kind < 2; ++kind)
        for (int N : {64, 128, 256}) {
            const int iters = 4096;
            float best_ms = 1e30f;
            for (int rep = 0; rep < 4; ++rep) {
                cudaEvent_t e0, e1;
                cudaEventCreate(&e0); cudaEventCreate(&e1);
                cudaEventRecord(e0);
                if (kind == 0) rate_probe<0><<<sms, 128, smem>>>(N, iters, dcyc);
                else rate_probe<1><<<sms, 128, smem>>>(N, iters, dcyc);
                cudaEventRecord(e1);
                e = cudaDeviceSynchronize();
                if (e != cudaSuccess) { printf("rate probe failed: %s\n", cudaGetErrorString(e)); return 1; }
                float ms;
                cudaEventElapsedTime(&ms, e0, e1);
                if (rep && ms < best_ms) best_ms = ms;
            }
            cudaMemcpy(cyc.data(), dcyc, sizeof(long long) * sms, cudaMemcpyDeviceToHost);
            const double n_mma = 8.0 * iters, K = kind == 0 ? 8 : 16;
            const double flop = n_mma * 2.0 * 128 * N * K;
            printf("{\"probe\": \"mma_rate\", \"kind\": \"%s\", \"M\": 128, \"N\": %d, \"K\": %d, \"cycles_per_mma\": %.2f, "
                   "\"tflops_all_sms\": %.1f, \"sms\": %d, \"ms\": %.3f}\n",
                   kind == 0 ? "tf32" : "f16", N, (int)K, cyc[0] / n_mma, flop * sms / (best_ms * 1e-3) / 1e12, sms, best_ms);
        }
    return 0;
}
