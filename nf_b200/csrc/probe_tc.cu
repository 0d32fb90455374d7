// Measurement aid for bench.py: the tensor-pipe roofline denominators, measured with the instruction shapes the flow
// kernels use (tcgen05.mma.cta_group::1, M = 128, A operand in tensor memory, B in shared memory, fp32 accumulate,
// issued back to back by one thread per SM): kind::tf32 (K = 8, the 3xTF32 kernels) and kind::f16 (K = 16, the fp16-
// split kernel).  Round 1 quoted "bf16 cuBLAS peak / 2" for TF32; this is the measured number (VERDICT r1 item 4).
#include "common.cuh"
#include "tc_common.cuh"

template <int KIND>
__global__ void __launch_bounds__(128, 1) mma_rate_kernel(int N, int iters) {
    extern __shared__ char smraw[];
    __shared__ uint64_t bar;
    __shared__ uint32_t tb_s;
    char* sm = smem_align1024(smraw);
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
#pragma unroll
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
        // instruction descriptors: c_format F32; a/b TF32 (2) for kind::tf32, F16 (0) for kind::f16
        const uint32_t idesc = KIND == 0 ? tc_idesc(128, N) : ((1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24));
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
                const uint64_t db = tc_desc(smem_u32(sm) + (ks & 3) * 32);
                if (KIND == 0) tc_mma_tf32_ts(tb, tb + 256 + ks * 8, db, idesc, 1);
                else asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
                                  ::"r"(tb), "r"(tb + 256 + ks * 8), "l"(db), "r"(idesc), "r"(1u) : "memory");
            }
        }
        tc_commit(&bar);
        mbar_wait(&bar, 0);
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tb), "r"(512));
}

extern "C" int64_t nis_probe_tensor(int32_t kind, int32_t n, int32_t iters, void* stream) {
    if ((kind != 0 && kind != 1) || (n != 64 && n != 128 && n != 256) || iters <= 0 || iters > (1 << 16)) return NIS_EINVAL;
    const int sms = nis_sm_count();
    const int smem = 256 * 128 + 1024;
    cudaStream_t s = (cudaStream_t)stream;
    if (kind == 0) {
        cudaFuncSetAttribute(mma_rate_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        mma_rate_kernel<0><<<sms, 128, smem, s>>>(n, iters);
    } else {
        cudaFuncSetAttribute(mma_rate_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        mma_rate_kernel<1><<<sms, 128, smem, s>>>(n, iters);
    }
    NIS_CUDA_CHECK_LAUNCH();
    return (int64_t)sms * iters * 8 * 2 * 128 * n * (kind == 0 ? 8 : 16);
}
