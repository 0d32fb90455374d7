// Train-mode backward of width-64 PWLin cells (32 bins) on the 5th-generation tensor cores.
//
// What torch.autograd does for the reference's loss.backward() (manager.py:278) through one coupling cell
// (coupling_cells.py:107-142, 230-254) is, per cell and in reverse order, a chain of small GEMMs with a
// batch-wide BatchNorm reduction between every two of them.  The chain is cut at those reductions:
//
//   head   : recompute the conditioner (3xTF32 tcgen05 pipeline, that of the round-1 forward), store the pre-BN
//            activations z_1..z_depth, run the spline forward + hand-derived spline backward on the logits
//            in registers -> dL/dlogits (stored), dL/dx of the transformed columns, dL/dJ
//   layer  : one launch per linear layer lam = depth (output layer) .. 0.  Upstream gradient dz (logits
//            gradient, or BN backward of the stored dL/dh with the batch means the previous launch left)
//              dgrad  dL/dh_lam = dz W_lam        A = dz in TENSOR MEMORY (lane = point), B = W_lam^T in smem
//              wgrad  dL/dW_lam += dz^T h_lam     both operands in shared memory, K = the 128 points of the
//                                                 tile, accumulated in tensor memory over the tiles of the
//                                                 CTA and added to its slice every 16 tiles (tcgen05
//                                                 accumulation truncates); fixed-order reduce, no atomics
//            then ReLU mask, store dL/dh_lam, per-feature sums of dL/dh and dL/dh * xhat (recursive-halving
//            warp shuffles, float64 across tiles, last CTA finalises = dL/dbeta, dL/dgamma and the means the
//            next launch needs)
//   tail   : BatchNorm backward of the input normalisation -> dL/dx of the pass-through columns (flow_bwd_tail_kernel,
//            which the wide backward of flow_bwd_wide.cu launches with its own tile stride)
//
// 3xTF32 everywhere (hi rounded to nearest, exact residual).  For the wgrad the hi and lo parts of dz are STACKED
// along M ([dz_hi ; dz_lo], 128 rows) so that two M=128 MMAs (against h_hi and h_lo) give all four partial
// products; rows o and 64+o of the accumulator are added on read-out.
//
// CTA of 8 point warps (two 128-point groups) + one MMA-issuing warp; in the layer launches the 8 warps work
// on ONE tile, two threads per point (see flow_bwd_tc_layer_kernel).
#include <stdlib.h>
#include "common.cuh"
#include "tc_common.cuh"
#include "flow_host.cuh"

#define BT_GROUP_COLS 192     // per point group: dz hi [0,64), dz lo [64,128), dgrad accumulator [128,192)
#define BT_COL_LO 64
#define BT_COL_D 128
#define BT_COL_ACC 384        // weight-gradient accumulators [384,448) and (output layer) [448,512)
#define BT_TILE (TCH * TCM)   // floats in one stored [64][128] activation tile

struct BtArgs {
    const float* saved;                    // [C+1][B][d+1]
    const void* grad_out; int grad_dtype;
    float* gstate;                         // [B][d+1]
    const float* params; const float* wpack; const float* bn_saved;
    const float* tcpack;                   // forward operands (flow_tc_pack_kernel)
    const float* bdpack;                   // dgrad operands (W^T hi/lo)
    float* zbuf;                           // [depth][tiles][64][128] pre-BN activations z_1..z_depth
    float* dl;                             // [tiles][128][128] dL/dlogits
    const float* dh_in; float* dh_out;     // [tiles][64][128] dL/dh between the layer launches
    float* bnb;                            // [depth+1][2][maxW] batch means of dL/dh and dL/dh*xhat
    float* slices;                         // [depth+1][grid][2][128][64] per-CTA wgrad accumulators
    float* grad_params;
    double* partials; unsigned* counter;
    long long B, ntiles;
    int c, lam, first, grid;
};

// Operands of the head's conditioner recompute: hidden layers 1..depth-1 and the output blocks, each as TF32 hi / lo
// splits in the K-major 128-byte-swizzled layout, tc_cell_floats(F) per cell (tc_common.cuh)
__global__ void flow_tc_pack_kernel(DevFlow F, const float* __restrict__ params, float* __restrict__ tcpack) {
    const int c = blockIdx.y;
    const DevCell& q = F.cells[c];
    const float* p = params + q.param_off;
    char* dst = reinterpret_cast<char*>(tcpack + (size_t)c * tc_cell_floats(F));
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (int l = 1; l < F.depth; ++l) {
        const float* w = p + F.p_lin(c, l);                     // [64][64] torch layout (out, in)
        char* hi = dst + (size_t)(l - 1) * 2 * TCH * TCH * 4;
        char* lo = hi + (size_t)TCH * TCH * 4;
        for (int i = tid; i < TCH * TCH; i += nth) {
            const int n = i / TCH, k = i - n * TCH;
            const float v = w[(size_t)n * TCH + k];
            const float h = tf32_rn(v);
            const int o = tc_off(TCH, n, k);
            *reinterpret_cast<float*>(hi + o) = h;
            *reinterpret_cast<float*>(lo + o) = tf32_rn(v - h);
        }
    }
    const float* wo = p + F.p_lin(c, F.depth);                  // [T*K][64]
    const int Nb = tc_out_n(F), tper = tc_out_tper(F), slot = tc_out_slot(F);
    for (int b = 0; b < tc_out_blocks(F, q.T); ++b) {
        char* hi = dst + (size_t)(F.depth - 1) * 2 * TCH * TCH * 4 + (size_t)b * 2 * Nb * TCH * 4;
        char* lo = hi + (size_t)Nb * TCH * 4;
        for (int i = tid; i < Nb * TCH; i += nth) {
            const int n = i / TCH, k = i - n * TCH;
            const int t = b * tper + n / slot, jj = n % slot;
            const float v = (t < q.T && jj < F.K) ? wo[((size_t)t * F.K + jj) * TCH + k] : 0.f;
            const float h = tf32_rn(v);
            const int o = tc_off(Nb, n, k);
            *reinterpret_cast<float*>(hi + o) = h;
            *reinterpret_cast<float*>(lo + o) = tf32_rn(v - h);
        }
    }
}

__host__ __device__ static inline int bd_layer_off(const DevFlow& F, int lam) {      // floats, inside a cell's block
    return lam == 0 ? 0 : 2 * 16 * TCH + (lam - 1) * 2 * TCH * TCH;
}
__host__ __device__ static inline int bd_cell_floats(const DevFlow& F) { return bd_layer_off(F, F.depth) + 2 * 2 * TCH * TCH; }

// dgrad operands.  B operand of "dL/dh = dz W": rows n = input feature i, K = output feature o, i.e. W^T, K-major swizzled;
// the output layer has K = 128 as two blocks of 64.
__global__ void flow_bwd_tc_pack_kernel(DevFlow F, const float* __restrict__ params, float* __restrict__ bdpack) {
    const int c = blockIdx.y;
    const DevCell& q = F.cells[c];
    const float* p = params + q.param_off;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    char* dst = reinterpret_cast<char*>(bdpack + (size_t)c * bd_cell_floats(F));
    for (int lam = 0; lam <= F.depth; ++lam) {
        const int rows = lam == 0 ? 16 : TCH, in = lam == 0 ? q.P : TCH;
        const int nblk = lam == F.depth ? 2 : 1;
        const int nout = lam == F.depth ? q.T * F.K : TCH;
        const float* w = p + F.p_lin(c, lam);                      // [nout][in]
        for (int b = 0; b < nblk; ++b) {
            char* hi = dst + (size_t)bd_layer_off(F, lam) * 4 + (size_t)b * 2 * rows * TCH * 4;
            char* lo = hi + (size_t)rows * TCH * 4;
            for (int i = tid; i < rows * TCH; i += nth) {
                const int n = i / TCH, k = i - n * TCH, o = b * TCH + k;
                const float v = (n < in && o < nout) ? w[(size_t)o * in + n] : 0.f;
                const float h = tf32_rn(v);
                const int off = tc_off(rows, n, k);
                *reinterpret_cast<float*>(hi + off) = h;
                *reinterpret_cast<float*>(lo + off) = tf32_rn(v - h);
            }
        }
    }
}

// ===================================================================================================
// head: conditioner recompute + spline backward
// ===================================================================================================
__global__ void __launch_bounds__(TC_THREADS, 1) flow_bwd_tc_head_kernel(const __grid_constant__ DevFlow F, const BtArgs A) {
    extern __shared__ char smraw[];
    __shared__ uint64_t a_ready[2], d_ready[2];
    __shared__ uint32_t tmem_base_s;
    char* sm = smem_align1024(smraw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c = A.c;
    const DevCell& q = F.cells[c];
    const int d = F.d, depth = F.depth;
    const TcSmem L = tc_layout(F, q.P, 1, depth, false);
    float* w0s = reinterpret_cast<float*>(sm + L.w0);
    float* affs = reinterpret_cast<float*>(sm + L.aff);
    float* biass = reinterpret_cast<float*>(sm + L.bias);
    float* gsm = reinterpret_cast<float*>(sm + L.total);            // gradient rows [2][(d+1)][128]
    const float* pk = A.wpack + q.pk_off;

    for (int l = 1; l <= depth; ++l) {
        const int fl = l == depth ? 2 * TC_NOUT * TCH : 2 * TCH * TCH;
        const float4* src = reinterpret_cast<const float4*>(A.tcpack + (size_t)c * tc_cell_floats(F) + (size_t)(l - 1) * 2 * TCH * TCH);
        float4* dst = reinterpret_cast<float4*>(sm + L.wl[l]);
        for (int i = tid; i < fl / 4; i += TC_THREADS) dst[i] = src[i];
    }
    {
        const float* s0 = pk + q.wt_off[0];
        for (int i = tid; i < q.P * TCH; i += TC_THREADS) w0s[i] = s0[i];
    }
    for (int l = 0; l <= depth; ++l) {
        const int W = l == 0 ? q.P : TCH, Wp = pad8(W);
        const float* s = pk + q.aff_off[l];
        for (int i = tid; i < W; i += TC_THREADS) { affs[l * 2 * TCH + i] = s[i]; affs[l * 2 * TCH + TCH + i] = s[Wp + i]; }
    }
    for (int i = tid; i < TC_NOUT; i += TC_THREADS) {
        const int t = i >> 5, jj = i & 31;
        biass[i] = t < q.T ? pk[q.bo_off + t * F.Kpad + jj] : 0.f;
    }
    if (tid == 0) {
        mbar_init(&a_ready[0], TCM); mbar_init(&a_ready[1], TCM);
        mbar_init(&d_ready[0], 1); mbar_init(&d_ready[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const long long ntiles = A.ntiles;
    const long long rowlen = d + 1;

    if (warp == 8) {
        if (lane == 0) {
            uint32_t pa[2] = {0, 0};
            const uint32_t idesc64 = tc_idesc(TCM, TCH), idescO = tc_idesc(TCM, TC_NOUT);
            for (long long it = 0;; ++it) {
                const long long t0 = ((long long)blockIdx.x + it * gridDim.x) * 2;
                if (t0 >= ntiles) break;
                for (int l = 1; l <= depth; ++l) {
                    const bool outl = l == depth;
                    const int rows = outl ? TC_NOUT : TCH;
                    const uint32_t whi = smem_u32(sm + L.wl[l]);
                    for (int g = 0; g < 2; ++g) {
                        if (t0 + g >= ntiles) continue;
                        mbar_wait(&a_ready[g], pa[g]);
                        pa[g] ^= 1;
                        tc_fence_after();
                        const uint32_t tb = tmem_base + g * TC_COLS_PER_GROUP;
                        tc_issue_layer(tb, tb + TC_COL_AHI, tb + TC_COL_ALO, whi, whi + rows * TCH * 4, rows, outl ? idescO : idesc64);
                        tc_commit(&d_ready[g]);
                    }
                }
            }
        }
    } else {
        const int g = warp >> 2, gt = tid & (TCM - 1);
        float* st = reinterpret_cast<float*>(sm + L.st) + g * (d + 1) * TCM + gt;
        float* gr = gsm + g * (d + 1) * TCM + gt;
        const uint32_t tg = tmem_base + g * TC_COLS_PER_GROUP + ((uint32_t)((warp & 3) * 32) << 16);
        uint32_t pd = 0;
        for (long long it = 0;; ++it) {
            const long long tile = ((long long)blockIdx.x + it * gridDim.x) * 2 + g;
            if (tile >= ntiles) break;
            const long long pt = tile * TCM + gt;
            const bool valid = pt < A.B;
            float Jout = 1.f;
            if (valid) {
                const float* sv = A.saved + ((long long)c * A.B + pt) * rowlen;
                for (int i = 0; i <= d; ++i) st[i * TCM] = sv[i];
                Jout = A.saved[((long long)(c + 1) * A.B + pt) * rowlen + d];
                if (A.first) {
                    for (int i = 0; i < d; ++i) gr[F.out_perm[i] * TCM] = load_io(A.grad_out, A.grad_dtype, pt * rowlen + i);
                    gr[d * TCM] = load_io(A.grad_out, A.grad_dtype, pt * rowlen + d);
                } else {
                    for (int i = 0; i <= d; ++i) gr[i * TCM] = A.gstate[pt * rowlen + i];
                }
            } else {
                for (int i = 0; i < d; ++i) { st[i * TCM] = 0.5f; gr[i * TCM] = 0.f; }
                st[d * TCM] = 1.f; gr[d * TCM] = 0.f;
            }
            // layer 0 on the FP32 pipe -> z_1
            float v[TCH];
#pragma unroll
            for (int j = 0; j < TCH; ++j) v[j] = 0.f;
            for (int k = 0; k < q.P; ++k) {
                const float a = fmaf(st[q.feed[k] * TCM], affs[k], affs[TCH + k]);
                const float4* wr = reinterpret_cast<const float4*>(w0s + k * TCH);
#pragma unroll
                for (int j4 = 0; j4 < TCH / 4; ++j4) {
                    const float4 w = wr[j4];
                    v[4 * j4] = fmaf(a, w.x, v[4 * j4]); v[4 * j4 + 1] = fmaf(a, w.y, v[4 * j4 + 1]);
                    v[4 * j4 + 2] = fmaf(a, w.z, v[4 * j4 + 2]); v[4 * j4 + 3] = fmaf(a, w.w, v[4 * j4 + 3]);
                }
            }
            for (int l = 1; l <= depth; ++l) {
                float* zo = A.zbuf + ((size_t)(l - 1) * ntiles + tile) * BT_TILE + gt;       // z_l, read back by the layer launches
#pragma unroll
                for (int j = 0; j < TCH; ++j) zo[(size_t)j * TCM] = v[j];
                tc_store_act(v, affs + l * 2 * TCH, affs + l * 2 * TCH + TCH, tg + TC_COL_AHI, tg + TC_COL_ALO);
                tc_fence_before();
                mbar_arrive(&a_ready[g]);
                mbar_wait(&d_ready[g], pd);
                pd ^= 1;
                tc_fence_after();
                if (l < depth) {
                    tc_ld32(tg, v);
                    tc_ld32(tg + 32, v + 32);
                    tc_ld_wait();
                }
            }
            // splines: forward + backward on the 32 logits of each transformed dimension (coupling_cells.py:114-141)
            const float gJ = gr[d * TCM];
            const float gJJ = gJ * Jout;
            float Fprod = 1.f;
            float* dlo = A.dl + (size_t)tile * 2 * BT_TILE + gt;
            for (int t = 0; t < 4; ++t) {
                float z[32];
                if (t < q.T) {
                    tc_ld32(tg + t * 32, z);
                    tc_ld_wait();
                    const int col = q.trafo[t];
                    const float xv = st[col * TCM], gy = gr[col * TCM];
                    const float a = xv * 32.f;
                    int kb = (int)floorf(a);
                    kb = kb < 0 ? 0 : (kb > 31 ? 31 : kb);
                    const float alpha = a - (float)kb;
                    float m = -3.0e38f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) { z[j] += biass[t * 32 + j]; m = fmaxf(m, z[j]); }
                    float S = 0.f, C = 0.f, ek = 0.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float e = __expf(z[j] - m);          // ex2.approx, like the forward (flow_tc_h.cu); the accurate expf was 16 % of this kernel
                        z[j] = e;
                        S += e;
                        C += j < kb ? e : 0.f;
                        ek = j == kb ? e : ek;
                    }
                    const float inv = 1.f / S;
                    const float y = (ek * alpha + C) * inv;
                    const float f = ek * inv * 32.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float p = z[j] * inv;
                        const float ind = j < kb ? 1.f : (j == kb ? alpha : 0.f);
                        z[j] = gy * p * (ind - y) + gJJ * ((j == kb ? 1.f : 0.f) - p);
                    }
                    gr[col * TCM] = gy * f;
                    Fprod *= f;
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) z[j] = 0.f;
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) dlo[(size_t)(t * 32 + j) * TCM] = z[j];
            }
            if (valid) {
                float* so = A.gstate + pt * rowlen;
                for (int i = 0; i < d; ++i) so[i] = gr[i * TCM];
                so[d] = gJ * Fprod;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

// ===================================================================================================
// layer: dgrad + wgrad of linear layer lam, ReLU/BN bookkeeping for BN layer lam
// ===================================================================================================
__device__ __forceinline__ void bt_prefetch_l2(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
// per-feature sums of 32 values over the 32 lanes of a warp (recursive halving): lane i returns the sum of feature i
__device__ __forceinline__ float bt_warp_feature_sums32(const float* v, int lane) {
    float a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const bool up = lane & 16;
        const float keep = up ? v[i + 16] : v[i], send = up ? v[i] : v[i + 16];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const bool up = lane & 8;
        const float keep = up ? a[i + 8] : a[i], send = up ? a[i] : a[i + 8];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const bool up = lane & 4;
        const float keep = up ? a[i + 4] : a[i], send = up ? a[i] : a[i + 4];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const bool up = lane & 2;
        const float keep = up ? a[i + 2] : a[i], send = up ? a[i] : a[i + 2];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    {
        const bool up = lane & 1;
        const float keep = up ? a[1] : a[0], send = up ? a[0] : a[1];
        a[0] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
    }
    return a[0];
}

// tcgen05.mma adds each K=8 step into the fp32 accumulator with TRUNCATION (tools/tc_accum_probe.cu: about
// one ulp lost per instruction, always toward zero), so an accumulator that lives across all tiles of a CTA
// would drift by ~1e-4 relative after a few thousand instructions.  The wgrad accumulators are therefore
// added to the CTA's slice in global memory (fp32, round-to-nearest) every 2 BT_FLUSH tiles (512 instructions) and restarted.
#define BT_FLUSH 8
template <int NH>
__device__ __noinline__ void bt_flush_acc(uint32_t tl, float* sl, int lam, int nin, bool add) {
    for (int h = 0; h < NH; ++h) {
        for (int j0 = 0; j0 < nin; j0 += 16) {
            float r[16];
            tc_ld16(tl + h * TCH + j0, r);
            tc_ld_wait();
            float4* o4 = reinterpret_cast<float4*>(sl + (size_t)h * 128 * TCH + j0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float4 v = make_float4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                if (add) { const float4 o = o4[j]; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
                o4[j] = v;
            }
        }
    }
}

struct BtSmem { int slabA, slabBh, slabBl, bd, coef, total; };
__host__ __device__ static inline BtSmem bt_layout(int KW) {
    BtSmem s;
    s.slabA = 0;                         // [128 rows: dz hi (64) ; dz lo (64)][128 points]
    s.slabBh = 65536;                    // [nin rows][128 points] h hi
    s.slabBl = 98304;                    //                         h lo
    s.bd = 131072;                       // dgrad operand: KW/64 blocks of (hi, lo) [nin][64]
    s.coef = s.bd + (KW / 64) * 2 * TCH * TCH * 4;
    s.total = s.coef + 8 * TCH * 4;
    return s;
}

// ---------------------------------------------------------------------------------------------------
// ONE tile in flight per CTA, TWO threads per point.  (The first version gave each of two point groups its own
// tile and made them take turns on the operand slab; with a thread carrying all 64 features the loads of a
// tile could not be issued together and half of the stall samples sat on the slab hand-over: 22.8 ms per
// 2^20-point training step against 18.9 ms now.)
// Warps 0-3 own features 0..31 of a point's 64-feature blocks and warps 4-7 features 32..63 (a warp may touch
// the 32 TMEM lanes 32 (warp % 4).., any column), so a thread carries half the loads and half the operand
// preparation and nobody queues for the operand slab.  The tensor-memory columns of the A operand and of the
// dgrad accumulator are double-buffered by tile parity: while the MMAs of tile i run, every thread already
// loads and prepares tile i+1 (its dz goes to the other A buffer, its h_lam waits in registers), then runs
// the epilogue of tile i and only then fills the slab for tile i+1 (the wgrad MMAs of tile i are done by then).
// ---------------------------------------------------------------------------------------------------
template <int KW>
__global__ void __launch_bounds__(TC_THREADS, 1) flow_bwd_tc_layer_kernel(const __grid_constant__ DevFlow F, const BtArgs A) {
    constexpr int NH = KW / 64;
    extern __shared__ char smraw[];
    __shared__ uint64_t a_ready, done[2], hdone, acc_ready, acc_free;
    __shared__ uint32_t tmem_base_s;
    __shared__ bool s_last;
    char* sm = smem_align1024(smraw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c = A.c, lam = A.lam;
    const DevCell& q = F.cells[c];
    const int d = F.d, maxW = F.maxW;
    const int nin = lam == 0 ? 16 : TCH;
    const int win = lam == 0 ? q.P : TCH;
    const BtSmem L = bt_layout(KW);
    char* slabA = sm + L.slabA;
    char* slabBh = sm + L.slabBh;
    char* slabBl = sm + L.slabBl;
    float* coef = reinterpret_cast<float*>(sm + L.coef);
    float* cA1 = coef, *cA2 = coef + TCH, *cA3 = coef + 2 * TCH;
    float* scp = coef + 3 * TCH, *shp = coef + 4 * TCH, *mup = coef + 5 * TCH, *rsp = coef + 6 * TCH;
    const float* pk = A.wpack + q.pk_off;
    {
        const int fl = NH * 2 * nin * TCH;
        const float4* src = reinterpret_cast<const float4*>(A.bdpack + (size_t)c * bd_cell_floats(F) + bd_layer_off(F, lam));
        float4* dst = reinterpret_cast<float4*>(sm + L.bd);
        for (int i = tid; i < fl / 4; i += TC_THREADS) dst[i] = src[i];
    }
    for (int j = tid; j < TCH; j += TC_THREADS) {
        if (KW == 64) {
            const int lu = lam + 1;
            const float* sv = A.bn_saved + q.sv_off + lu * 2 * maxW;
            const float sc = pk[q.aff_off[lu] + j];
            const float m1 = A.bnb[lu * 2 * maxW + j], m2 = A.bnb[lu * 2 * maxW + maxW + j];
            const float mu = sv[j], rs = sv[maxW + j];
            cA1[j] = sc; cA2[j] = -sc * m2 * rs; cA3[j] = -sc * m1 + sc * m2 * rs * mu;
        }
        if (j < win) {
            const float* sv = A.bn_saved + q.sv_off + lam * 2 * maxW;
            scp[j] = pk[q.aff_off[lam] + j];
            shp[j] = pk[q.aff_off[lam] + pad8(win) + j];
            mup[j] = sv[j]; rsp[j] = sv[maxW + j];
        } else { scp[j] = 0.f; shp[j] = 0.f; mup[j] = 0.f; rsp[j] = 0.f; }
    }
    if (tid == 0) {
        mbar_init(&a_ready, 2 * TCM);
        mbar_init(&done[0], 1); mbar_init(&done[1], 1); mbar_init(&hdone, 1);
        mbar_init(&acc_ready, 1); mbar_init(&acc_free, TCM);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const long long ntiles = A.ntiles, rowlen = d + 1;
    constexpr int fevery = 2 * BT_FLUSH;                   // in tiles
    int nflush = 0;
    double acc1 = 0.0, acc2 = 0.0, accb[NH];
#pragma unroll
    for (int h = 0; h < NH; ++h) accb[h] = 0.0;

    if (warp == 8) {
        // ===================== MMA issuer ======================================================
        if (lane == 0) {
            uint32_t pa = 0, pf = 0;
            bool fresh = true;
            const uint32_t idesc = tc_idesc(TCM, nin);
            const uint32_t sA = smem_u32(slabA), sBh = smem_u32(slabBh), sBl = smem_u32(slabBl), sBd = smem_u32(sm + L.bd);
            long long it = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
                const int b = (int)(it & 1);
                const uint32_t tb = tmem_base + b * BT_GROUP_COLS;
                for (int h = 0; h < NH; ++h) {
                    mbar_wait(&a_ready, pa);
                    pa ^= 1;
                    tc_fence_after();
                    const uint32_t bh = sBd + h * 2 * nin * TCH * 4, bl = bh + nin * TCH * 4;
                    uint32_t acc = h > 0;
                    // cross terms first, hi*hi last (the accumulate truncation is relative to the accumulator, tc_common.cuh)
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks) {
                        const uint32_t wo = (ks >> 2) * nin * 128 + (ks & 3) * 32;
                        tc_mma_tf32_ts(tb + BT_COL_D, tb + ks * 8, tc_desc(bl + wo), idesc, acc);
                        acc = 1;
                        tc_mma_tf32_ts(tb + BT_COL_D, tb + BT_COL_LO + ks * 8, tc_desc(bh + wo), idesc, 1);
                    }
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks) {
                        const uint32_t wo = (ks >> 2) * nin * 128 + (ks & 3) * 32;
                        tc_mma_tf32_ts(tb + BT_COL_D, tb + ks * 8, tc_desc(bh + wo), idesc, 1);
                    }
                    const uint32_t ta = tmem_base + BT_COL_ACC + h * TCH;
                    uint32_t accw = !fresh;
#pragma unroll
                    for (int ks = 0; ks < 16; ++ks) {
                        const uint32_t ao = (ks >> 2) * 128 * 128 + (ks & 3) * 32;
                        const uint32_t bo = (ks >> 2) * nin * 128 + (ks & 3) * 32;
                        tc_mma_tf32_ss(ta, tc_desc(sA + ao), tc_desc(sBh + bo), idesc, accw);
                        accw = 1;
                        tc_mma_tf32_ss(ta, tc_desc(sA + ao), tc_desc(sBl + bo), idesc, 1);
                    }
                    if (h < NH - 1) tc_commit(&hdone); else tc_commit(&done[b]);
                }
                fresh = false;
                if (((it + 1) % fevery) == 0 && tile + gridDim.x < ntiles) {
                    tc_commit(&acc_ready);
                    mbar_wait(&acc_free, pf);
                    pf ^= 1;
                    tc_fence_after();
                    fresh = true;
                }
            }
        }
    } else {
        // ===================== point threads: (point gt, feature half sub) ===================================
        const int sub = warp >> 2, gt = tid & (TCM - 1), f0 = 32 * sub;
        const uint32_t tl = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
        uint32_t pdn[2] = {0, 0}, phd = 0, pfr = 0;
        uint32_t mask = 0, maskn = 0;
        float hv[32];
        for (long long it = -1;; ++it) {
            const long long tile = (long long)blockIdx.x + it * (long long)gridDim.x;            // current (epilogue)
            const long long tn = tile + gridDim.x;                                               // next (operands)
            const bool have_n = tn < ntiles;
            const int bn = (int)((it + 1) & 1);
            const uint32_t tgn = tl + bn * BT_GROUP_COLS;
            const long long ptn = tn * TCM + gt;
            const bool validn = have_n && ptn < A.B;
            if (have_n) {
                if (gt == 0 && sub == 0) {                       // the tile after the next one -> L2
                    const long long t2 = tn + gridDim.x;
                    if (t2 < ntiles) {
                        if (lam > 0) bt_prefetch_l2(A.zbuf + ((size_t)(lam - 1) * ntiles + t2) * BT_TILE, BT_TILE * 4);
                        if (KW == 128) bt_prefetch_l2(A.dl + (size_t)t2 * 2 * BT_TILE, 2 * BT_TILE * 4);
                        else {
                            bt_prefetch_l2(A.dh_in + (size_t)t2 * BT_TILE, BT_TILE * 4);
                            bt_prefetch_l2(A.zbuf + ((size_t)lam * ntiles + t2) * BT_TILE, BT_TILE * 4);
                        }
                    }
                }
                // ---- stage 1: this thread's 32 features of dz (first 64-block) -> the other A buffer of tensor memory
                {
                    float dz[32], lo[32];
                    if (KW == 128) {
                        const float* up = A.dl + (size_t)tn * 2 * BT_TILE + (size_t)f0 * TCM + gt;
#pragma unroll
                        for (int j = 0; j < 32; ++j) dz[j] = up[(size_t)j * TCM];
                    } else {
                        const float* up = A.dh_in + (size_t)tn * BT_TILE + (size_t)f0 * TCM + gt;
                        const float* zu = A.zbuf + ((size_t)lam * ntiles + tn) * BT_TILE + (size_t)f0 * TCM + gt;
#pragma unroll
                        for (int j = 0; j < 32; ++j) { dz[j] = up[(size_t)j * TCM]; lo[j] = zu[(size_t)j * TCM]; }
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            dz[j] = validn ? fmaf(cA1[f0 + j], dz[j], fmaf(cA2[f0 + j], lo[j], cA3[f0 + j])) : 0.f;
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float a = dz[j];
                        dz[j] = tf32_rn(a);
                        lo[j] = a - dz[j];
                    }
                    tc_st32(tgn + f0, dz);
                    tc_st32(tgn + BT_COL_LO + f0, lo);
                    if (KW == 128) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) dz[j] += lo[j];
                        accb[0] += (double)bt_warp_feature_sums32(dz, lane);
                    }
                    tc_st_wait();
                }
                // ---- h_lam of the next tile, in registers until the slab is free
                maskn = 0;
                if (lam > 0) {
                    const float* zpn = A.zbuf + ((size_t)(lam - 1) * ntiles + tn) * BT_TILE + (size_t)f0 * TCM + gt;
#pragma unroll
                    for (int j = 0; j < 32; ++j) hv[j] = zpn[(size_t)j * TCM];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float a = fmaf(hv[j], scp[f0 + j], shp[f0 + j]);
                        maskn |= (uint32_t)(a > 0.f) << j;
                        hv[j] = fmaxf(a, 0.f);
                    }
                } else if (sub == 0) {
                    const float* xs = A.saved + ((long long)c * A.B + (validn ? ptn : 0)) * rowlen;
#pragma unroll
                    for (int k = 0; k < 16; ++k) hv[k] = k < q.P ? fmaf(xs[q.feed[k]], scp[k], shp[k]) : 0.f;
                }
            }
            // ---- wait for the current tile --------------------------------------------------------------------------
            const int b = (int)(it & 1);
            if (it >= 0) {                                     // the MMAs of the current tile are complete: its dgrad
                mbar_wait(&done[b], pdn[b]);                   // accumulator is valid and the operand slab is free
                pdn[b] ^= 1;
                tc_fence_after();
            }
            if (have_n) {
                // ---- stage 2: operands of the next tile into the slab; its MMAs then overlap the epilogue below ----------
                if (lam > 0) {
    #pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float hi = tf32_rn(hv[j]);
                        const int off = tc_slab_off(TCH, f0 + j, gt);
                        *reinterpret_cast<float*>(slabBh + off) = hi;
                        *reinterpret_cast<float*>(slabBl + off) = hv[j] - hi;
                    }
                } else if (sub == 0) {
    #pragma unroll
                    for (int k = 0; k < 16; ++k) {
                        const float hi = tf32_rn(hv[k]);
                        const int off = tc_slab_off(16, k, gt);
                        *reinterpret_cast<float*>(slabBh + off) = hi;
                        *reinterpret_cast<float*>(slabBl + off) = hv[k] - hi;
                    }
                }
                {
                    float hi[32], lo[32];
                    tc_ld32(tgn + f0, hi);
                    tc_ld32(tgn + BT_COL_LO + f0, lo);
                    tc_ld_wait();
    #pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        *reinterpret_cast<float*>(slabA + tc_slab_off(128, f0 + j, gt)) = hi[j];
                        *reinterpret_cast<float*>(slabA + tc_slab_off(128, TCH + f0 + j, gt)) = lo[j];
                    }
                }
                proxy_fence();
                tc_fence_before();
                mbar_arrive(&a_ready);
            }
            // ---- stage 3: epilogue of the current tile ---------------------------------------------------------------
            if (it >= 0) {
                const uint32_t tg = tl + b * BT_GROUP_COLS;
                const long long pt = tile * TCM + gt;
                const bool valid = pt < A.B;
                float* out = A.dh_out + (size_t)tile * BT_TILE + gt;
                if (lam > 0) {
                    const float* zp = A.zbuf + ((size_t)(lam - 1) * ntiles + tile) * BT_TILE + (size_t)f0 * TCM + gt;
                    float dv[32], pr[32];
                    // z_lam from global memory, all 32 loads ahead of the stores below (interleaved, every load has to stay
                    // behind the previous store - the pointers may alias - and the loop runs at one memory latency per feature)
#pragma unroll
                    for (int j = 0; j < 32; ++j) pr[j] = __ldg(zp + (size_t)j * TCM);
                    tc_ld32(tg + BT_COL_D + f0, dv);
                    tc_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        dv[j] = ((mask >> j) & 1u) ? dv[j] : 0.f;
                        pr[j] = dv[j] * (pr[j] - mup[f0 + j]) * rsp[f0 + j];
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) out[(size_t)(f0 + j) * TCM] = dv[j];
                    acc1 += (double)bt_warp_feature_sums32(dv, lane);
                    acc2 += (double)bt_warp_feature_sums32(pr, lane);
                } else if (sub == 0) {
                    const float* xs = A.saved + ((long long)c * A.B + (valid ? pt : 0)) * rowlen;
                    float dv[32], pr[32];
                    tc_ld16(tg + BT_COL_D, dv);
                    tc_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        dv[j] = j < q.P ? dv[j] : 0.f;
                        out[(size_t)j * TCM] = dv[j];
                        pr[j] = j < q.P ? dv[j] * (xs[q.feed[j]] - mup[j]) * rsp[j] : 0.f;
                    }
#pragma unroll
                    for (int j = 16; j < 32; ++j) { dv[j] = 0.f; pr[j] = 0.f; }
                    acc1 += (double)bt_warp_feature_sums32(dv, lane);
                    acc2 += (double)bt_warp_feature_sums32(pr, lane);
                }
                if (sub == 0 && ((it + 1) % fevery) == 0 && have_n) {
                    mbar_wait(&acc_ready, pfr);
                    pfr ^= 1;
                    tc_fence_after();
                    bt_flush_acc<NH>(tl + BT_COL_ACC, A.slices + (((size_t)lam * A.grid + blockIdx.x) * 2) * 128 * TCH + (size_t)gt * TCH,
                                     lam, nin, nflush > 0);
                    ++nflush;
                    tc_fence_before();
                    mbar_arrive(&acc_free);
                }
            }
            if (!have_n) break;
            if (KW == 128) {
                // second 64 logits: loaded while the MMAs of the first block run
                float dz[32], lo[32];
                const float* up = A.dl + (size_t)tn * 2 * BT_TILE + BT_TILE + (size_t)f0 * TCM + gt;
#pragma unroll
                for (int j = 0; j < 32; ++j) dz[j] = up[(size_t)j * TCM];
                mbar_wait(&hdone, phd);
                phd ^= 1;
                tc_fence_after();
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float a = dz[j];
                    const float hi = tf32_rn(a);
                    lo[j] = a - hi;
                    *reinterpret_cast<float*>(slabA + tc_slab_off(128, f0 + j, gt)) = hi;
                    *reinterpret_cast<float*>(slabA + tc_slab_off(128, TCH + f0 + j, gt)) = lo[j];
                    dz[j] = hi;
                }
                tc_st32(tgn + f0, dz);
                tc_st32(tgn + BT_COL_LO + f0, lo);
                tc_st_wait();
                proxy_fence();
                tc_fence_before();
                mbar_arrive(&a_ready);
#pragma unroll
                for (int j = 0; j < 32; ++j) dz[j] += lo[j];
                accb[NH - 1] += (double)bt_warp_feature_sums32(dz, lane);
            }
            mask = maskn;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp < 4)
        bt_flush_acc<NH>(tmem_base + ((uint32_t)(warp * 32) << 16) + BT_COL_ACC,
                         A.slices + (((size_t)lam * A.grid + blockIdx.x) * 2) * 128 * TCH + (size_t)tid * TCH, lam, nin, nflush > 0);
    tc_fence_before();
    __syncthreads();
    if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    // ---- per-feature sums: lane l of a warp holds feature 32 sub + l ----------------------------------------------------
    double* red = reinterpret_cast<double*>(sm);            // [8 warps][32 lanes][4]
    if (warp < 8) {
        double* r = red + ((size_t)warp * 32 + lane) * 4;
        r[0] = acc1; r[1] = acc2; r[2] = accb[0]; r[3] = NH > 1 ? accb[NH - 1] : 0.0;
    }
    __syncthreads();
    double* mine = A.partials + (size_t)blockIdx.x * 256;
    for (int i = tid; i < 256; i += TC_THREADS) {
        const int f = i & 63, kind = i >> 6;                // kind 0: s1, 1: s2, 2: bias block 0, 3: bias block 1
        const int sb = f >> 5, ln = f & 31;
        double s = 0.0;
        for (int w = 0; w < 4; ++w) s += red[((size_t)(sb * 4 + w) * 32 + ln) * 4 + kind];
        mine[i] = s;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(A.counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    float* gp = A.grad_params + q.param_off;
    for (int i = tid; i < 256; i += TC_THREADS) {
        const int f = i & 63, kind = i >> 6;
        double s = 0.0;
        for (unsigned bb = 0; bb < gridDim.x; ++bb) s += __ldcg(A.partials + (size_t)bb * 256 + i);
        if (kind == 0 && f < win) {
            A.bnb[lam * 2 * maxW + f] = (float)(s / (double)A.B);
            gp[F.p_bn_gamma(c, lam) + win + f] += (float)s;
        } else if (kind == 1 && f < win) {
            A.bnb[lam * 2 * maxW + maxW + f] = (float)(s / (double)A.B);
            gp[F.p_bn_gamma(c, lam) + f] += (float)s;
        } else if (kind >= 2 && KW == 128) {
            const int n = (kind - 2) * TCH + f;
            if (n < q.T * F.K) gp[F.p_out_b(c) + n] += (float)s;
        }
    }
    if (tid == 0) *A.counter = 0u;
}

// ===================================================================================================
// tail: BatchNorm backward of the input normalisation, dL/dx of the pass-through columns (both tensor-core backwards)
// ===================================================================================================
__global__ void __launch_bounds__(256) flow_bwd_tail_kernel(const __grid_constant__ DevFlow F, const BwdTailArgs A) {
    const int c = A.c;
    const DevCell& q = F.cells[c];
    const int d = F.d, maxW = F.maxW;
    const long long rowlen = d + 1;
    const float* pk = A.wpack + q.pk_off;
    const float* sv = A.bn_saved + q.sv_off;
    for (long long pt = (long long)blockIdx.x * blockDim.x + threadIdx.x; pt < A.B; pt += (long long)gridDim.x * blockDim.x) {
        const float* xs = A.saved + ((long long)c * A.B + pt) * rowlen;
        float* gs = A.gstate + pt * rowlen;
        const float* da = A.dh_in + (size_t)(pt >> 7) * A.tile_floats + (pt & 127);
        float g[NIS_MAX_DIM + 1];
        for (int i = 0; i <= d; ++i) g[i] = gs[i];
        for (int k = 0; k < q.P; ++k) {
            const int col = q.feed[k];
            const float xh = (xs[col] - sv[k]) * sv[maxW + k];
            g[col] += pk[q.aff_off[0] + k] * (da[(size_t)k * TCM] - A.bnb[k] - xh * A.bnb[maxW + k]);
        }
        for (int i = 0; i <= d; ++i) gs[i] = g[i];
        if (A.grad_in)
            for (int i = 0; i <= d; ++i) store_io(A.grad_in, A.grad_dtype, pt * rowlen + i, g[i]);
    }
}

int launch_flow_bwd_tail(const DevFlow& F, const BwdTailArgs& A, cudaStream_t s) {
    const long long blocks = (A.B + 255) / 256;
    flow_bwd_tail_kernel<<<(int)(blocks < NIS_MAX_GRID ? blocks : NIS_MAX_GRID), 256, 0, s>>>(F, A);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

// grad_params[cell] += per-CTA slices (fixed order).  blockIdx.y = linear layer.
__global__ void flow_bwd_tc_reduce_kernel(DevFlow F, const float* __restrict__ slices, int grid, int c, float* __restrict__ grad_params) {
    // four lanes per weight: lane g adds the slices of CTAs [g * chunk, (g + 1) * chunk) in CTA order (eight loads in flight),
    // the four partial sums are combined as (s0 + s1) + (s2 + s3): fixed order, no atomics
    const int lam = blockIdx.y;
    const DevCell& q = F.cells[c];
    const int in = lam == 0 ? q.P : TCH;
    const int nout = lam == F.depth ? q.T * F.K : TCH;
    float* gw = grad_params + q.param_off + F.p_lin(c, lam);
    const int lane = threadIdx.x & 31, g = lane >> 3;
    const int chunk = (grid + 3) >> 2;
    const int b0 = g * chunk, b1 = b0 + chunk < grid ? b0 + chunk : grid;
    const int total = nout * in, per_block = blockDim.x >> 2;
    for (int base = blockIdx.x * per_block; base < ((total + per_block - 1) / per_block) * per_block; base += gridDim.x * per_block) {
        const int i = base + (threadIdx.x >> 5) * 8 + (lane & 7);
        float s = 0.f;
        if (i < total) {
            const int o = i / in, k = i - o * in;
            const int h = o >> 6, r = o & 63;
            const float* sl0 = slices + ((((size_t)lam * grid) * 2 + h) * 128) * TCH + (size_t)r * TCH + k;
            const size_t step = (size_t)2 * 128 * TCH;
            int b = b0;
            for (; b + 8 <= b1; b += 8) {
                float t[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float* sl = sl0 + (size_t)(b + u) * step;
                    t[u] = __ldcg(sl) + __ldcg(sl + TCH * TCH);
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) s += t[u];
            }
            for (; b < b1; ++b) {
                const float* sl = sl0 + (size_t)b * step;
                s += __ldcg(sl) + __ldcg(sl + TCH * TCH);
            }
        }
        s += __shfl_xor_sync(0xffffffffu, s, 8);
        s += __shfl_xor_sync(0xffffffffu, s, 16);
        if (i < total && g == 0) gw[i] += s;
    }
}

// ---------------------------------------------------------------------------------------------------
size_t nis_tc_pack_floats(const DevFlow& F) {
    if (F.depth < 1) return 0;
    return (size_t)F.n_cells * tc_cell_floats(F);
}

int nis_tc_pack(const DevFlow& F, const float* params, float* tcpack, cudaStream_t s) {
    flow_tc_pack_kernel<<<dim3(16, F.n_cells), 256, 0, s>>>(F, params, tcpack);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

// Width-64 cells with 32 bins (PWLin or PWQuad) whose operands in the 3xTF32 layout (tc_layout) fit an SM's shared memory
// in each launch shape of the round-1 forward: fused eval cell, layer pass, final pass.  The tensor-core backward below
// takes the PWLin ones; the fp16-split forward and inverse take all of them (nis_flow_plan).
bool nis_tc_supported(const DevFlow& F) {
    if (F.depth < 1 || F.maxW != TCH || F.nb != 32) return false;
    for (int l = 0; l < F.depth; ++l) if (F.widths[l] != TCH) return false;
    if (F.kind == NIS_KIND_PWLIN ? F.K != 32 : F.K != 65) return false;
    for (int c = 0; c < F.n_cells; ++c) {
        const int P = F.cells[c].P, T = F.cells[c].T;
        if (P > 16) return false;
        if (F.K == 32 && T * 32 > TC_NOUT) return false;
        const size_t lim = 226 * 1024;
        if ((size_t)tc_layout(F, P, 1, F.depth, false).total + 1024 > lim && F.K == 32) return false;      // fused eval cell
        if ((size_t)tc_layout(F, P, 1, F.depth - 1, true).total + 1024 > lim) return false;               // hidden pass(es)
        if ((size_t)tc_layout(F, P, F.depth, F.depth, F.K == 32).total + 1024 > lim) return false;        // final pass
    }
    return true;
}

bool nis_bwd_tc_supported(const DevFlow& F) { return F.kind == NIS_KIND_PWLIN && nis_tc_supported(F); }

// CTAs of the head and layer launches at most (a B200's SM count): bt_carve reserves one wgrad slice per layer CTA
#define BT_MAX_CTAS 148

struct BtScratch { float *gstate, *zbuf, *dl, *dh[2], *bnb, *slices, *bdpack; size_t floats; };
static void bt_carve(const DevFlow& F, int64_t B, float* base, BtScratch* s) {
    auto up = [](size_t x) { return (x + 63) & ~(size_t)63; };
    const size_t tiles = (size_t)((B + TCM - 1) / TCM);
    size_t off = 0;
    s->gstate = base + off; off = up(off + (size_t)B * (F.d + 1));
    s->zbuf = base + off; off = up(off + (size_t)F.depth * tiles * BT_TILE);
    s->dl = base + off; off = up(off + tiles * 2 * BT_TILE);
    s->dh[0] = base + off; off = up(off + tiles * BT_TILE);
    s->dh[1] = base + off; off = up(off + tiles * BT_TILE);
    s->bnb = base + off; off = up(off + (size_t)(F.depth + 1) * 2 * F.maxW);
    s->slices = base + off; off = up(off + (size_t)(F.depth + 1) * BT_MAX_CTAS * 2 * 128 * TCH);
    s->bdpack = base + off; off = up(off + (size_t)F.n_cells * bd_cell_floats(F));
    s->floats = off;
}

size_t nis_bwd_tc_scratch_floats(const DevFlow& F, int64_t B) {
    BtScratch s;
    bt_carve(F, B, nullptr, &s);
    return s.floats;
}

int nis_flow_backward_tc(const DevFlow& F, const FlowWorkspace& ws, const float* params, const float* saved,
                         const float* bn_saved, const void* grad_out, int grad_dtype, float* grad_params, void* grad_in,
                         int64_t B, cudaStream_t s) {
    BtScratch sc;
    bt_carve(F, B, ws.bwd, &sc);
    const long long ntiles = (B + TCM - 1) / TCM;
    const int sms = nis_sm_count(), ctas = sms < BT_MAX_CTAS ? sms : BT_MAX_CTAS;
    const int grid = (int)((ntiles + 1) / 2 < ctas ? (ntiles + 1) / 2 : ctas);    // head: two tiles at a time per CTA
    const int lgrid = (int)(ntiles < ctas ? ntiles : ctas);                       // layers: one tile at a time, one slice each
    flow_bwd_tc_pack_kernel<<<dim3(16, F.n_cells), 256, 0, s>>>(F, params, sc.bdpack);
    NIS_CUDA_CHECK_LAUNCH();
    int rc = nis_tc_pack(F, params, ws.tcpack, s);
    if (rc) return rc;
    BtArgs A;
    A.saved = saved; A.grad_out = grad_out; A.grad_dtype = grad_dtype;
    A.gstate = sc.gstate; A.params = params; A.wpack = ws.wpack; A.bn_saved = bn_saved;
    A.tcpack = ws.tcpack; A.bdpack = sc.bdpack; A.zbuf = sc.zbuf; A.dl = sc.dl;
    A.bnb = sc.bnb; A.slices = sc.slices; A.grad_params = grad_params;
    A.partials = ws.partials; A.counter = ws.counter; A.B = B; A.ntiles = ntiles; A.grid = lgrid;
    A.dh_in = nullptr; A.dh_out = nullptr; A.lam = 0;
    BwdTailArgs Ta;
    Ta.saved = saved; Ta.gstate = sc.gstate; Ta.wpack = ws.wpack; Ta.bn_saved = bn_saved; Ta.bnb = sc.bnb;
    Ta.grad_dtype = grad_dtype; Ta.B = B; Ta.tile_floats = BT_TILE;
    const size_t smem64 = (size_t)bt_layout(64).total + 1024, smem128 = (size_t)bt_layout(128).total + 1024;
    NIS_ENSURE_SMEM((flow_bwd_tc_layer_kernel<64>), (int)smem64);
    NIS_ENSURE_SMEM((flow_bwd_tc_layer_kernel<128>), (int)smem128);
    for (int c = F.n_cells - 1; c >= 0; --c) {
        A.c = c; A.first = c == F.n_cells - 1;
        const size_t smem_head = (size_t)tc_layout(F, F.cells[c].P, 1, F.depth, false).total + 2 * (F.d + 1) * TCM * 4 + 1024;
        NIS_ENSURE_SMEM((flow_bwd_tc_head_kernel), (int)smem_head);
        flow_bwd_tc_head_kernel<<<grid, TC_THREADS, smem_head, s>>>(F, A);
        NIS_CUDA_CHECK_LAUNCH();
        int pp = 0;
        for (int lam = F.depth; lam >= 0; --lam) {
            A.lam = lam;
            A.dh_in = sc.dh[pp]; A.dh_out = sc.dh[pp ^ 1];
            if (lam == F.depth) flow_bwd_tc_layer_kernel<128><<<lgrid, TC_THREADS, smem128, s>>>(F, A);
            else flow_bwd_tc_layer_kernel<64><<<lgrid, TC_THREADS, smem64, s>>>(F, A);
            NIS_CUDA_CHECK_LAUNCH();
            pp ^= 1;
        }
        Ta.c = c; Ta.dh_in = sc.dh[pp]; Ta.grad_in = c == 0 ? grad_in : nullptr;
        rc = launch_flow_bwd_tail(F, Ta, s);
        if (rc) return rc;
        flow_bwd_tc_reduce_kernel<<<dim3(128, F.depth + 1), 256, 0, s>>>(F, sc.slices, lgrid, c, grad_params);
        NIS_CUDA_CHECK_LAUNCH();
    }
    return NIS_OK;
}
