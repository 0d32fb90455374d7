// tcgen05 / TMEM / bulk-copy building blocks shared by the tensor-core flow kernels (flow_tc_h.cu, flow_wide.cu
// forward; flow_bwd_tc.cu, flow_bwd_wide.cu backward): PTX wrappers, the K-major 128-byte-swizzled operand layout,
// TMEM <-> register moves, the 3xTF32 split.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

#define TCM 128              // points per CTA tile (= MMA M)
#define TCH 64               // hidden width
#define TC_KT 32             // tf32 elements per 128-byte swizzle row
#define TC_NOUT 128          // widest output-layer MMA block

// ---- tiny PTX wrappers ------------------------------------------------------------------------------
// TF32 split with round-to-nearest on both parts: hi = rn_tf32(a), lo = rn_tf32(a - hi).  (Masking the
// low mantissa bits instead — truncation — leaves a one-sided 2^-20 relative bias in every product,
// measured as a 5x loss of accuracy on log J; rounding makes the residual ~2^-22 and unbiased.)
// (integer add + mask on the ALU pipe = cvt.rna.tf32.f32, which would run on the quarter-rate XU pipe)
__device__ __forceinline__ float tf32_rn(float a) {
    return __uint_as_float((__float_as_uint(a) + 0x1000u) & 0xFFFFE000u);
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 1024-byte aligned start inside the dynamic shared-memory window, formed as base + offset: a pointer rebuilt from an
// integer loses its address space and every access through it becomes a generic LD / ST instead of LDS / STS
__device__ __forceinline__ char* smem_align1024(char* smraw) { return smraw + ((1024u - (smem_u32(smraw) & 1023u)) & 1023u); }
// (Until the last session of round 2 the wide weight-gradient kernel rebuilt its base through an integer on purpose: generic
// stores measured faster there, 283 against 380 us -- they only kept the compiler from reordering the kernel's load batches.
// With the loads issued explicitly ahead of the stores it runs LDS / STS like every other kernel: 127 us.)

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// bounded wait: a broken pipeline traps instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t a = smem_u32(bar);
    for (int it = 0; it < (1 << 22); ++it) {
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
        if (ok) return;
    }
    __trap();
}
// non-blocking probe of a barrier phase (the MMA issuer polls its groups round-robin)
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// pull a contiguous global range into L2 ahead of its use (TMA engine, no completion to wait for)
__device__ __forceinline__ void bulk_prefetch_l2(const void* gmem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gmem_src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem desc]^T, kind::tf32, cta_group::1 (A from tensor memory)
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, kind::tf32, cta_group::1 (both operands from shared memory)
__device__ __forceinline__ void tc_mma_tf32_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// 1-D bulk copy global -> shared (TMA engine), completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// 1-D bulk copy shared -> global; the shared source may be reused once wait_group.read has returned
__device__ __forceinline__ void bulk_store(void* gmem_dst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void group_sync(int g) { asm volatile("bar.sync %0, %1;" ::"r"(1 + g), "r"(TCM) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 in
// bits [0,14), leading byte offset >> 4 in [16,30) (unused for swizzled K-major: 1), stride byte offset
// >> 4 in [32,46) (= 1024 B between 8-row groups), version 1 in [46,48), layout type 2 (128B swizzle) in [61,64).
__device__ __forceinline__ uint64_t tc_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 (1) at [4,6), a/b format TF32 (2) at
// [7,10)/[10,13), both K-major, N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t tc_idesc(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// byte offset of element (row, k) of a [rows x 64] tf32 operand stored as two K-tiles of [rows x 32]
// (128 B per row, 8-row groups of 1024 B, 16-byte chunks XOR-swizzled with row % 8)
__host__ __device__ static inline int tc_off(int rows, int row, int k) {
    const int kt = k >> 5, kk = k & 31;
    return kt * rows * 128 + (row >> 3) * 1024 + (row & 7) * 128 + ((((kk >> 2) ^ (row & 7)) << 4) | ((kk & 3) << 2));
}

// byte offset of (row, point) in a [rows x 128 points] K-major operand whose K dimension is the tile's points
// (weight-gradient MMAs): four K-tiles of 32 points, same 128-byte swizzle
__host__ __device__ static inline int tc_slab_off(int rows, int row, int p) {
    return (p >> 5) * rows * 128 + (row >> 3) * 1024 + (row & 7) * 128 + (((((p & 31) >> 2) ^ (row & 7)) << 4) | ((p & 3) << 2));
}

// Output layer as a sequence of MMA blocks: PWLin with 32 bins -> ONE block of N=128 covering four
// transformed dimensions; otherwise (PWQuad with 32 bins: 65 logits per dimension) one block of N=80 per
// transformed dimension, issued one after the other into the same accumulator columns.
__host__ __device__ static inline int tc_out_n(const DevFlow& F) { return F.K == 32 ? 128 : 80; }
__host__ __device__ static inline int tc_out_tper(const DevFlow& F) { return F.K == 32 ? 4 : 1; }
__host__ __device__ static inline int tc_out_slot(const DevFlow& F) { return F.K == 32 ? 32 : 80; }
__host__ __device__ static inline int tc_out_blocks(const DevFlow& F, int T) { return (T + tc_out_tper(F) - 1) / tc_out_tper(F); }
__host__ __device__ static inline int tc_max_blocks(const DevFlow& F) {
    int m = 1;
    for (int c = 0; c < F.n_cells; ++c) { const int b = tc_out_blocks(F, F.cells[c].T); m = b > m ? b : m; }
    return m;
}
// floats in one cell's tensor-core weight pack: hidden layers 1..depth-1 (hi, lo), then the output blocks (hi, lo)
__host__ __device__ static inline int tc_cell_floats(const DevFlow& F) {
    return (F.depth - 1) * 2 * TCH * TCH + tc_max_blocks(F) * 2 * tc_out_n(F) * TCH;
}

#define TC_THREADS 288       // 2 groups x 4 warps + 1 MMA warp
#define TC_COLS_PER_GROUP 256
#define TC_COL_AHI 128
#define TC_COL_ALO 192

struct TcSmem {      // byte offsets from the 1024-aligned base
    int w, w0, aff, bias, st, sst, red, zb, total;
    int wl[NIS_MAX_HIDDEN + 1];     // per MMA layer l (1..depth): offset of (hi, lo) inside w, or -1
};
// MMA layers [l_begin, l_end] are staged (hidden: 2 x 16 KB, output: 2 x 32 KB)
__host__ __device__ static inline TcSmem tc_layout(const DevFlow& F, int P, int l_begin, int l_end, bool zstage = false) {
    TcSmem s;
    int o = 0;
    s.w = o;
    for (int l = 0; l <= F.depth; ++l) {
        s.wl[l] = -1;
        if (l >= 1 && l >= l_begin && l <= l_end) {
            s.wl[l] = o;
            o += l == F.depth ? tc_max_blocks(F) * 2 * tc_out_n(F) * TCH * 4 : 2 * TCH * TCH * 4;
        }
    }
    s.w0 = o; o += pad8(P) * TCH * 4;
    s.aff = o; o += (F.depth + 1) * 2 * TCH * 4;
    s.bias = o; o += tc_max_blocks(F) * tc_out_n(F) * 4;
    s.st = o; o += 2 * (F.d + 1) * TCM * 4;
    o = (o + 15) & ~15;
    s.sst = o; o += 2 * (F.d + 1) * TCM * 4;     // landing zone of the next tile's state rows (bulk copy), per group
    o = (o + 7) & ~7;
    s.red = o; o += (8 * 2 * TCH + 2 * F.maxW) * 8;
    o = (o + 127) & ~127;
    s.zb = o;                                  // [2 groups][2 buffers][64][128] floats, bulk-copy landing zone
    if (zstage) o += 2 * 2 * TCH * TCM * 4;
    s.total = o;
    return s;
}

#define TC_R32(v, b) "=r"(v[b+0]), "=r"(v[b+1]), "=r"(v[b+2]), "=r"(v[b+3]), "=r"(v[b+4]), "=r"(v[b+5]), "=r"(v[b+6]), "=r"(v[b+7])
#define TC_W32(v, b) "r"(v[b+0]), "r"(v[b+1]), "r"(v[b+2]), "r"(v[b+3]), "r"(v[b+4]), "r"(v[b+5]), "r"(v[b+6]), "r"(v[b+7])

// 32 consecutive columns of this thread's TMEM lane <-> registers
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float* vf) {
    uint32_t* v = reinterpret_cast<uint32_t*>(vf);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : TC_R32(v, 0), TC_R32(v, 8), TC_R32(v, 16), TC_R32(v, 24)
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float* vf) {
    uint32_t* v = reinterpret_cast<uint32_t*>(vf);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : TC_R32(v, 0), TC_R32(v, 8)
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_st32(uint32_t taddr, const float* vf) {
    const uint32_t* v = reinterpret_cast<const uint32_t*>(vf);
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%32], "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31};"
        :: TC_W32(v, 0), TC_W32(v, 8), TC_W32(v, 16), TC_W32(v, 24), "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_st16(uint32_t taddr, const uint32_t* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%16], "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15};"
        :: TC_W32(v, 0), TC_W32(v, 8), "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_st8(uint32_t taddr, const uint32_t* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x8.b32 [%8], {%0, %1, %2, %3, %4, %5, %6, %7};"
        :: TC_W32(v, 0), "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// BN scale/shift + ReLU of this thread's 64 pre-activations, split into TF32 hi / residual lo, written to
// the group's A-operand columns of tensor memory
__device__ __forceinline__ void tc_store_act(const float* v, const float* sc, const float* sh, uint32_t t_hi, uint32_t t_lo) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        float hi[32], lo[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const float a = fmaxf(fmaf(v[32 * h + j], sc[32 * h + j], sh[32 * h + j]), 0.f);
            hi[j] = tf32_rn(a);
            lo[j] = a - hi[j];            // exact; the MMA reads its top 19 bits (truncation of a value of random sign: unbiased)
        }
        tc_st32(t_hi + 32 * h, hi);
        tc_st32(t_lo + 32 * h, lo);
    }
    tc_st_wait();
}

// 3xTF32 product of the group's [128 x 64] activations (TMEM) with a [N x 64] weight matrix (smem): 8 K-steps x 3.
// tcgen05.mma truncates when it adds a K=8 step into the fp32 accumulator (tools/tc_accum_probe.cu), losing about
// one ulp OF THE ACCUMULATOR per instruction.  The sixteen cross-term steps (a_hi w_lo, a_lo w_hi: 2^-11 of the
// result) are therefore issued first, while the accumulator is still tiny, and the eight a_hi w_hi steps last:
// the truncation of 8 instead of 24 steps is felt.
__device__ __forceinline__ void tc_issue_layer(uint32_t tmem_d, uint32_t t_hi, uint32_t t_lo, uint32_t w_hi, uint32_t w_lo,
                                               int n_rows, uint32_t idesc) {
    uint32_t acc = 0;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
        const uint32_t wo = (ks >> 2) * n_rows * 128 + (ks & 3) * 32;
        tc_mma_tf32_ts(tmem_d, t_hi + ks * 8, tc_desc(w_lo + wo), idesc, acc);
        acc = 1;
        tc_mma_tf32_ts(tmem_d, t_lo + ks * 8, tc_desc(w_hi + wo), idesc, 1);
    }
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
        const uint32_t wo = (ks >> 2) * n_rows * 128 + (ks & 3) * 32;
        tc_mma_tf32_ts(tmem_d, t_hi + ks * 8, tc_desc(w_hi + wo), idesc, 1);
    }
}

// per-feature sums over the 32 lanes of a warp by recursive halving: afterwards lane i holds the sums of
// features 2i and 2i+1.  62 shuffles instead of 64 x 5.
__device__ __forceinline__ void tc_warp_feature_sums(const float* v, int lane, float& s0, float& s1) {
    float a[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        const bool up = lane & 16;
        const float keep = up ? v[i + 32] : v[i], send = up ? v[i] : v[i + 32];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const bool up = lane & 8;
        const float keep = up ? a[i + 16] : a[i], send = up ? a[i] : a[i + 16];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const bool up = lane & 4;
        const float keep = up ? a[i + 8] : a[i], send = up ? a[i] : a[i + 8];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const bool up = lane & 2;
        const float keep = up ? a[i + 4] : a[i], send = up ? a[i] : a[i + 4];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const bool up = lane & 1;
        const float keep = up ? a[i + 2] : a[i], send = up ? a[i] : a[i + 2];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
    }
    s0 = a[0]; s1 = a[1];
}

