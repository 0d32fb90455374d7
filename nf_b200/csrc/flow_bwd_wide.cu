// Train-mode backward for WIDE conditioners (hidden width 128..256) on tcgen05 — BASELINE configs[4].
//
// Same cut of the autograd chain as flow_bwd_tc.cu (one launch per BatchNorm reduction), with the GEMMs in the
// streamed-weights form of flow_wide.cu because neither the weights nor the gradient accumulators of a
// 256-wide layer fit an SM:
//   z_1..z_depth : kept by the forward (nis_flow_forward_cached: the activation cache), or recomputed by the forward's
//               wide layer passes (flow_wide_tc_kernel, no statistics) when the caller passed no cache
//   head      : output layer per transformed dimension (streamed panels, A chunks in tensor memory), logits
//               staged in shared memory, spline forward + hand-derived backward of spline.cuh in place ->
//               dL/dlogits tile, dL/dx of the transformed columns, dL/dJ, output-layer bias gradient
//   dgrad     : dL/dh_lam = dz W_lam.  dz (the logits gradient, or the BN backward of the stored dL/dh) is
//               formed 32 features at a time by the point threads, split hi/lo into tensor memory (A operand);
//               W_lam^T streams through the TMA ring as K-panels; epilogue = ReLU mask, store, float64 sums
//               of dL/dh and dL/dh * xhat (last CTA finalises: dL/dbeta, dL/dgamma, means for the next launch)
//   wgrad     : dL/dW_lam = dz^T h_lam as SS-mode MMAs with K = the tile's 128 points.  One CTA owns a
//               64-row block of dz (hi and lo stacked to M = 128) x a 128-column block of h_lam and a slice of
//               the tiles; eight point warps (two threads per point, half of the operand rows each) write both operands
//               into a K-major swizzled slab from values loaded while the previous tile's MMAs ran, thread 0 issues the
//               MMAs; the accumulator lives in tensor memory and is flushed to the CTA's slice every 8 tiles (tcgen05
//               accumulation truncates; the first flush stores, the later ones are vector reductions); a fixed-order
//               reduce adds the slices.
//   tail      : BatchNorm backward of the input normalisation (flow_bwd_tail_kernel of flow_bwd_tc.cu, with this file's
//               tile stride).
#include <stdlib.h>
#include "common.cuh"
#include "spline.cuh"
#include "tc_common.cuh"
#include "wide_common.cuh"
#include "flow_fwd_common.cuh"
#include "flow_host.cuh"

struct BwArgs {
    const float* saved; const void* grad_out; int grad_dtype;
    float* gstate;
    const float* params; const float* wpack; const float* bn_saved;
    const float* widepack;                 // forward operand pack (the head uses the output-layer panels)
    const float* dgpack;                   // dgrad operand pack (W^T panels)
    const float* zbuf;                     // [depth][tiles][W][128] pre-BN activations z_1..z_depth
    float* dl;                             // [tiles][T*Kp][128] dL/dlogits
    const float* dh_in; float* dh_out;     // [tiles][W][128]
    float* dz;                             // [tiles][W][128] BN-backward result of the current hidden layer (wgrad operand)
    float* bnb;                            // [depth+1][2][maxW]
    float* slices; float* grad_params;
    double* partials; unsigned* counter;
    long long B, ntiles;
    int c, lam, first, nparts;
};

__host__ __device__ static inline int bw_tmax(const DevFlow& F) {
    int T = 0;
    for (int c = 0; c < F.n_cells; ++c) T = F.cells[c].T > T ? F.cells[c].T : T;
    return T;
}
__host__ __device__ static inline int bw_kout(const DevFlow& F, int T) { return (T * wd_kp16(F) + 31) & ~31; }   // padded logit count
// dgrad pack of a cell (floats): layer 0 [16 x W], hidden 1..depth-1 [W x W], output [W x Kout], each x 2 (hi, lo)
__host__ __device__ static inline size_t bw_dg_off(const DevFlow& F, int lam) {
    const int W = F.widths[0];
    return lam == 0 ? 0 : (size_t)16 * W * 2 + (size_t)(lam - 1) * W * W * 2;
}
__host__ __device__ static inline size_t bw_dg_cell_floats(const DevFlow& F) {
    return bw_dg_off(F, F.depth) + (size_t)F.widths[0] * bw_kout(F, bw_tmax(F)) * 2;
}

// W^T as K-panels of 32 upstream features: [N rows = input feature][32] hi then lo
__global__ void flow_bwd_wide_pack_kernel(DevFlow F, const float* __restrict__ params, float* __restrict__ dgpack) {
    const int c = blockIdx.y;
    const DevCell& q = F.cells[c];
    const float* p = params + q.param_off;
    const int W = F.widths[0], Kp = wd_kp16(F);
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nth = (long long)gridDim.x * blockDim.x;
    float* cell = dgpack + (size_t)c * bw_dg_cell_floats(F);
    for (int lam = 0; lam <= F.depth; ++lam) {
        const int N = lam == 0 ? 16 : W;                    // rows of the operand = width of h_lam
        const int in = lam == 0 ? q.P : W;
        const int Kin = lam == F.depth ? bw_kout(F, q.T) : W;
        const float* w = p + F.p_lin(c, lam);               // [out][in]
        char* base = reinterpret_cast<char*>(cell + bw_dg_off(F, lam));
        for (long long i = tid; i < (long long)N * Kin; i += nth) {
            const int n = (int)(i / Kin), k = (int)(i - (long long)n * Kin);
            float v = 0.f;
            if (n < in) {
                if (lam == F.depth) {
                    const int t = k / Kp, j = k - t * Kp;
                    if (t < q.T && j < F.K) v = w[((size_t)t * F.K + j) * in + n];
                } else {
                    v = w[(size_t)k * in + n];
                }
            }
            const float h = tf32_rn(v);
            const int kt = k >> 5, kk = k & 31;
            char* panel = base + (size_t)kt * N * 64 * 4;
            const int off = (n >> 3) * 1024 + (n & 7) * 128 + ((((kk >> 2) ^ (n & 7)) << 4) | ((kk & 3) << 2));
            *reinterpret_cast<float*>(panel + off) = h;
            *reinterpret_cast<float*>(panel + (size_t)N * 128 + off) = tf32_rn(v - h);
        }
    }
}

// ===================================================================================================
// head: output layer + spline backward
// ===================================================================================================
struct BwHeadSmem { int ring, slots, slot_bytes, w0, aff, bias, st, gs, stg, bacc, total; };
__host__ __device__ static inline BwHeadSmem bw_head_layout(const DevFlow& F, int P, bool from_state) {
    BwHeadSmem s;
    const int W = F.widths[0], Kp = wd_kp16(F), T = bw_tmax(F);
    s.slot_bytes = Kp * 256;
    const int w0b = from_state ? pad8(P) * W * 4 : 0;
    const int affb = (2 * 16 + 2 * W) * 4, biasb = T * Kp * 4, stb = (F.d + 1) * TCM * 4, stgb = Kp * TCM * 4;
    const int baccb = T * Kp * 8;
    const int other = w0b + affb + biasb + 2 * stb + stgb + baccb + 256;
    int slots = (226 * 1024 - other) / s.slot_bytes;
    s.slots = slots > WD_MAX_SLOTS ? WD_MAX_SLOTS : slots;
    int o = 0;
    s.ring = o; o += s.slots * s.slot_bytes;
    s.w0 = o; o += w0b;
    s.aff = o; o += affb;
    s.bias = o; o += biasb;
    s.st = o; o += stb;
    s.gs = o; o += stb;
    s.stg = o; o += stgb;
    o = (o + 7) & ~7;
    s.bacc = o; o += baccb;
    s.total = o;
    return s;
}

template <int KIND>
__global__ void __launch_bounds__(WD_THREADS, 1) flow_bwd_wide_head_kernel(const __grid_constant__ DevFlow F, const BwArgs A) {
    extern __shared__ char smraw[];
    __shared__ uint64_t full[WD_MAX_SLOTS], empty[WD_MAX_SLOTS], a_ready[2], a_free[2], d_ready, d_free;
    __shared__ uint32_t tmem_base_s;
    __shared__ bool s_last;
    char* sm = smem_align1024(smraw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c = A.c;
    const DevCell& q = F.cells[c];
    const int d = F.d, depth = F.depth, W = F.widths[0], kc = W >> 5, Kp = wd_kp16(F);
    const bool from_z = depth >= 2;                        // z_depth from the recompute passes; depth 1: from the state
    const BwHeadSmem L = bw_head_layout(F, q.P, !from_z);
    const int RS = L.slots;
    float* w0s = reinterpret_cast<float*>(sm + L.w0);
    float* affs = reinterpret_cast<float*>(sm + L.aff);
    float* biass = reinterpret_cast<float*>(sm + L.bias);
    double* bacc = reinterpret_cast<double*>(sm + L.bacc);
    const float* pk = A.wpack + q.pk_off;
    const float* cellpack = A.widepack + (size_t)c * wd_cell_floats(F) + (size_t)(depth - 1) * W * W * 2;
    const float* zin = A.zbuf + (size_t)(depth - 1) * A.ntiles * W * TCM;

    if (!from_z) {
        const float* s0 = pk + q.wt_off[0];
        for (int i = tid; i < q.P * W; i += WD_THREADS) w0s[i] = s0[i];
    }
    for (int i = tid; i < 16; i += WD_THREADS) {
        affs[i] = i < q.P ? pk[q.aff_off[0] + i] : 0.f;
        affs[16 + i] = i < q.P ? pk[q.aff_off[0] + pad8(q.P) + i] : 0.f;
    }
    for (int i = tid; i < W; i += WD_THREADS) {
        affs[32 + i] = pk[q.aff_off[depth] + i];
        affs[32 + W + i] = pk[q.aff_off[depth] + W + i];
    }
    for (int i = tid; i < q.T * Kp; i += WD_THREADS) {
        const int t = i / Kp, n = i - t * Kp;
        biass[i] = n < F.K ? pk[q.bo_off + t * F.Kpad + n] : 0.f;
        bacc[i] = 0.0;
    }
    if (tid == 0) {
        for (int s = 0; s < WD_MAX_SLOTS; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(&a_ready[0], TCM); mbar_init(&a_ready[1], TCM);
        mbar_init(&a_free[0], 1); mbar_init(&a_free[1], 1);
        mbar_init(&d_ready, 1); mbar_init(&d_free, TCM);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const long long ntiles = A.ntiles, rowlen = d + 1;
    const size_t panel_floats = (size_t)Kp * 64;

    if (warp == 5) {
        if (lane == 0) {
            unsigned pc = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
                for (int r = 0; r < q.T; ++r) {
                    const float* src = cellpack + (size_t)r * Kp * W * 2;
                    for (int p = 0; p < kc; ++p, ++pc) {
                        const unsigned slot = pc % RS;
                        mbar_wait(&empty[slot], ((pc / RS) & 1) ^ 1);
                        bulk_load(sm + L.ring + slot * L.slot_bytes, src + p * panel_floats, (uint32_t)L.slot_bytes, &full[slot]);
                    }
                }
        }
    } else if (warp == 4) {
        if (lane == 0) {
            unsigned pc = 0, cc = 0, rr = 0;
            const uint32_t idesc = tc_idesc(TCM, Kp);
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
                for (int r = 0; r < q.T; ++r, ++rr) {
                    mbar_wait(&d_free, (rr & 1) ^ 1);
                    tc_fence_after();
                    uint32_t acc = 0;
                    for (int i = 0; i < kc; ++i, ++cc, ++pc) {
                        const unsigned buf = cc & 1;
                        mbar_wait(&a_ready[buf], (cc >> 1) & 1);
                        const unsigned slot = pc % RS;
                        mbar_wait(&full[slot], (pc / RS) & 1);
                        tc_fence_after();
                        const uint32_t ta = tmem_base + WD_COL_A + buf * 64;
                        const uint32_t bh = smem_u32(sm + L.ring + slot * L.slot_bytes), bl = bh + Kp * 128;
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            const uint32_t ah = ta + ks * 8;
                            tc_mma_tf32_ts(tmem_base, ah, tc_desc(bh + ks * 32), idesc, acc);
                            tc_mma_tf32_ts(tmem_base + WD_COL_X, ah, tc_desc(bl + ks * 32), idesc, acc);
                            acc = 1;
                            tc_mma_tf32_ts(tmem_base + WD_COL_X, ah + 32, tc_desc(bh + ks * 32), idesc, 1);
                        }
                        tc_commit(&empty[slot]);
                        tc_commit(&a_free[buf]);
                    }
                    tc_commit(&d_ready);
                }
        }
    } else {
        const int gt = tid;
        float* st = reinterpret_cast<float*>(sm + L.st) + gt;
        float* gr = reinterpret_cast<float*>(sm + L.gs) + gt;
        float* stg0 = reinterpret_cast<float*>(sm + L.stg);
        float* stg = stg0 + gt;
        const uint32_t tg = tmem_base + ((uint32_t)(warp * 32) << 16);
        unsigned cc = 0, rr = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
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
            float a0[16];
            if (!from_z) {
#pragma unroll
                for (int k = 0; k < 16; ++k) a0[k] = k < q.P ? fmaf(st[q.feed[k] * TCM], affs[k], affs[16 + k]) : 0.f;
            }
            const float gJ = gr[d * TCM], gJJ = gJ * Jout;
            float Fprod = 1.f;
            for (int r = 0; r < q.T; ++r, ++rr) {
                for (int i = 0; i < kc; ++i, ++cc) {
                    const unsigned buf = cc & 1;
                    float v[32];
                    if (from_z) {
                        const float* zr = zin + ((size_t)tile * W + 32 * i) * TCM + gt;
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = zr[(size_t)j * TCM];
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = 0.f;
#pragma unroll
                        for (int k = 0; k < 16; ++k) {
                            if (k < q.P) {
                                const float4* wr = reinterpret_cast<const float4*>(w0s + k * W + 32 * i);
#pragma unroll
                                for (int j4 = 0; j4 < 8; ++j4) {
                                    const float4 w = wr[j4];
                                    v[4 * j4] = fmaf(a0[k], w.x, v[4 * j4]); v[4 * j4 + 1] = fmaf(a0[k], w.y, v[4 * j4 + 1]);
                                    v[4 * j4 + 2] = fmaf(a0[k], w.z, v[4 * j4 + 2]); v[4 * j4 + 3] = fmaf(a0[k], w.w, v[4 * j4 + 3]);
                                }
                            }
                        }
                        if (r == 0) {                                  // depth 1: this IS z_1, the layer launches need it
                            float* z1 = const_cast<float*>(A.zbuf) + ((size_t)tile * W + 32 * i) * TCM + gt;
#pragma unroll
                            for (int j = 0; j < 32; ++j) z1[(size_t)j * TCM] = v[j];
                        }
                    }
                    float lo[32];
                    const float* sc = affs + 32 + 32 * i, *sh = affs + 32 + W + 32 * i;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float a = fmaxf(fmaf(v[j], sc[j], sh[j]), 0.f);
                        v[j] = tf32_rn(a);
                        lo[j] = tf32_rn(a - v[j]);
                    }
                    mbar_wait(&a_free[buf], ((cc >> 1) & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t ta = tg + WD_COL_A + buf * 64;
                    tc_st32(ta, v);
                    tc_st32(ta + 32, lo);
                    tc_st_wait();
                    tc_fence_before();
                    mbar_arrive(&a_ready[buf]);
                }
                mbar_wait(&d_ready, rr & 1);
                tc_fence_after();
                const int t = r;
                for (int j0 = 0; j0 < Kp; j0 += 16) {
                    float v[16], xx[16];
                    tc_ld16(tg + j0, v);
                    tc_ld16(tg + WD_COL_X + j0, xx);
                    tc_ld_wait();
#pragma unroll
                    for (int x = 0; x < 16; ++x) stg[(j0 + x) * TCM] = (v[x] + xx[x]) + biass[t * Kp + j0 + x];
                }
                tc_fence_before();
                mbar_arrive(&d_free);
                // spline forward + backward in place: stg[j] becomes dL/dlogit_j
                const int col = q.trafo[t];
                const float xv = st[col * TCM], gy = gr[col * TCM];
                float dx, f;
                if (KIND == NIS_KIND_PWLIN) {
                    float S, al;
                    int kbin;
                    const float y = pwlin_fwd(stg, TCM, F.nb, xv, f, kbin, S, al);
                    dx = pwlin_bwd(stg, TCM, F.nb, kbin, S, al, y, f, gy, gJJ);
                } else {
                    QuadCtx qc;
                    pwquad_fwd<true>(stg, TCM, F.nb, xv, qc);
                    f = qc.f;
                    dx = pwquad_bwd<true>(stg, TCM, F.nb, qc, gy, gJJ / qc.f);
                }
                gr[col * TCM] = dx;
                Fprod *= f;
                float* dlo = A.dl + ((size_t)tile * q.T * Kp + (size_t)t * Kp) * TCM + gt;
                for (int j = 0; j < Kp; ++j) {
                    const float g = (valid && j < F.K) ? stg[j * TCM] : 0.f;
                    stg[j * TCM] = g;
                    dlo[(size_t)j * TCM] = g;
                }
                // output-layer bias gradient: row sums of the staged tile (thread j owns logits j, j + 128)
                group_sync(0);
                for (int j = gt; j < F.K; j += TCM) {
                    const float4* row = reinterpret_cast<const float4*>(stg0 + j * TCM);     // rotated 16-byte loads: conflict-free
                    float s0 = 0.f, s1 = 0.f;
#pragma unroll 8
                    for (int i = 0; i < TCM / 4; ++i) {
                        const float4 x = row[(i + gt) & (TCM / 4 - 1)];
                        s0 += x.x + x.y;
                        s1 += x.z + x.w;
                    }
                    bacc[t * Kp + j] += (double)(s0 + s1);
                }
                group_sync(0);
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
    if (warp == 4) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    // bias gradient: CTA partials -> last CTA adds them to the parameter gradient
    const int nb_ = q.T * Kp;
    double* mine = A.partials + (size_t)blockIdx.x * nb_;
    for (int i = tid; i < nb_; i += WD_THREADS) mine[i] = bacc[i];
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(A.counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    float* gb = A.grad_params + q.param_off + F.p_out_b(c);
    for (int i = tid; i < nb_; i += WD_THREADS) {
        const int t = i / Kp, j = i - t * Kp;
        if (j >= F.K) continue;
        double s = 0.0;
        for (unsigned b = 0; b < gridDim.x; ++b) s += __ldcg(A.partials + (size_t)b * nb_ + i);
        gb[t * F.K + j] += (float)s;
    }
    if (tid == 0) *A.counter = 0u;
}

// ===================================================================================================
// dgrad of linear layer lam
// ===================================================================================================
struct BwDgSmem { int ring, slots, slot_bytes, coef, red, total; };
__host__ __device__ static inline BwDgSmem bw_dg_layout(const DevFlow& F, int lam) {
    BwDgSmem s;
    const int W = F.widths[0], N = lam == 0 ? 16 : W;
    s.slot_bytes = N * 256;
    const int coefb = 7 * W * 4, redb = 2 * W * 8;
    int slots = (226 * 1024 - coefb - redb - 4 * 32 * 16 * 8 - 256) / s.slot_bytes;
    s.slots = slots > WD_MAX_SLOTS ? WD_MAX_SLOTS : slots;
    int o = 0;
    s.ring = o; o += s.slots * s.slot_bytes;
    s.coef = o; o += coefb;
    o = (o + 7) & ~7;
    s.red = o; o += 4 * 32 * 16 * 8;                         // [4 warps][32 lanes][16] doubles
    s.total = o;
    return s;
}

// OUTL: upstream gradient = dL/dlogits (lam == depth); else BN backward of dL/dh_{lam+1}
template <bool OUTL>
__global__ void __launch_bounds__(WD_THREADS, 1) flow_bwd_wide_dgrad_kernel(const __grid_constant__ DevFlow F, const BwArgs A) {
    extern __shared__ char smraw[];
    __shared__ uint64_t full[WD_MAX_SLOTS], empty[WD_MAX_SLOTS], a_ready[2], a_free[2], d_ready, d_free;
    __shared__ uint32_t tmem_base_s;
    __shared__ bool s_last;
    char* sm = smem_align1024(smraw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c = A.c, lam = A.lam;
    const DevCell& q = F.cells[c];
    const int d = F.d, maxW = F.maxW, W = F.widths[0], Kp = wd_kp16(F);
    const int N = lam == 0 ? 16 : W;                        // width of h_lam (MMA N)
    const int win = lam == 0 ? q.P : W;
    const int nlog = q.T * Kp;                              // real rows of the logits-gradient tile
    const int Kin = OUTL ? bw_kout(F, q.T) : W;
    const int kc = Kin >> 5;
    const BwDgSmem L = bw_dg_layout(F, lam);
    const int RS = L.slots;
    float* coef = reinterpret_cast<float*>(sm + L.coef);
    float* cA1 = coef, *cA2 = coef + W, *cA3 = coef + 2 * W;
    float* scp = coef + 3 * W, *shp = coef + 4 * W, *mup = coef + 5 * W, *rsp = coef + 6 * W;
    const float* pk = A.wpack + q.pk_off;
    const float* src = A.dgpack + (size_t)c * bw_dg_cell_floats(F) + bw_dg_off(F, lam);
    for (int j = tid; j < W; j += WD_THREADS) {
        if (!OUTL) {
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
        for (int s = 0; s < WD_MAX_SLOTS; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(&a_ready[0], TCM); mbar_init(&a_ready[1], TCM);
        mbar_init(&a_free[0], 1); mbar_init(&a_free[1], 1);
        mbar_init(&d_ready, 1); mbar_init(&d_free, TCM);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const long long ntiles = A.ntiles, rowlen = d + 1;
    const size_t panel_floats = (size_t)N * 64;
    double s1[4][2], s2[4][2];
#pragma unroll
    for (int j = 0; j < 4; ++j) { s1[j][0] = s1[j][1] = s2[j][0] = s2[j][1] = 0.0; }

    if (warp == 5) {
        if (lane == 0) {
            unsigned pc = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
                for (int p = 0; p < kc; ++p, ++pc) {
                    const unsigned slot = pc % RS;
                    mbar_wait(&empty[slot], ((pc / RS) & 1) ^ 1);
                    bulk_load(sm + L.ring + slot * L.slot_bytes, src + p * panel_floats, (uint32_t)L.slot_bytes, &full[slot]);
                }
        }
    } else if (warp == 4) {
        if (lane == 0) {
            unsigned pc = 0, cc = 0, rr = 0;
            const uint32_t idesc = tc_idesc(TCM, N);
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++rr) {
                mbar_wait(&d_free, (rr & 1) ^ 1);
                tc_fence_after();
                uint32_t acc = 0;
                for (int i = 0; i < kc; ++i, ++cc, ++pc) {
                    const unsigned buf = cc & 1;
                    mbar_wait(&a_ready[buf], (cc >> 1) & 1);
                    const unsigned slot = pc % RS;
                    mbar_wait(&full[slot], (pc / RS) & 1);
                    tc_fence_after();
                    const uint32_t ta = tmem_base + WD_COL_A + buf * 64;
                    const uint32_t bh = smem_u32(sm + L.ring + slot * L.slot_bytes), bl = bh + N * 128;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint32_t ah = ta + ks * 8;
                        tc_mma_tf32_ts(tmem_base, ah, tc_desc(bh + ks * 32), idesc, acc);
                        acc = 1;
                        tc_mma_tf32_ts(tmem_base, ah, tc_desc(bl + ks * 32), idesc, 1);
                        tc_mma_tf32_ts(tmem_base, ah + 32, tc_desc(bh + ks * 32), idesc, 1);
                    }
                    tc_commit(&empty[slot]);
                    tc_commit(&a_free[buf]);
                }
                tc_commit(&d_ready);
            }
        }
    } else {
        const int gt = tid;
        const uint32_t tg = tmem_base + ((uint32_t)(warp * 32) << 16);
        unsigned cc = 0, rr = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++rr) {
            const long long pt = tile * TCM + gt;
            const bool valid = pt < A.B;
            // ---- A operand: upstream gradient dz, 32 features per chunk ---------------------------------------------
            for (int i = 0; i < kc; ++i, ++cc) {
                const unsigned buf = cc & 1;
                float v[32], lo[32];
                if (OUTL) {
                    const float* up = A.dl + ((size_t)tile * nlog + 32 * i) * TCM + gt;
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = 32 * i + j < nlog ? up[(size_t)j * TCM] : 0.f;
                } else {
                    const float* up = A.dh_in + ((size_t)tile * W + 32 * i) * TCM + gt;
                    const float* zu = A.zbuf + (((size_t)lam * ntiles + tile) * W + 32 * i) * TCM + gt;     // z_{lam+1}
                    float* dzo = A.dz + ((size_t)tile * W + 32 * i) * TCM + gt;
#pragma unroll
                    for (int j = 0; j < 32; ++j) { v[j] = up[(size_t)j * TCM]; lo[j] = zu[(size_t)j * TCM]; }
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int r = 32 * i + j;
                        v[j] = valid ? fmaf(cA1[r], v[j], fmaf(cA2[r], lo[j], cA3[r])) : 0.f;
                        dzo[(size_t)j * TCM] = v[j];
                    }
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float a = v[j];
                    v[j] = tf32_rn(a);
                    lo[j] = tf32_rn(a - v[j]);
                }
                mbar_wait(&a_free[buf], ((cc >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t ta = tg + WD_COL_A + buf * 64;
                tc_st32(ta, v);
                tc_st32(ta + 32, lo);
                tc_st_wait();
                tc_fence_before();
                mbar_arrive(&a_ready[buf]);
            }
            mbar_wait(&d_ready, rr & 1);
            tc_fence_after();
            // ---- epilogue: ReLU mask, store dL/dh_lam, sums for BN layer lam -------------------------------------------
            float* out = A.dh_out + (size_t)tile * W * TCM + gt;
            if (lam > 0) {
                const float* zp = A.zbuf + ((size_t)(lam - 1) * ntiles + tile) * W * TCM + gt;               // z_lam
#pragma unroll
                for (int jb = 0; jb < 4; ++jb) {
                    if (64 * jb >= W) break;
                    float dv[TCH];
                    tc_ld32(tg + 64 * jb, dv);
                    tc_ld32(tg + 64 * jb + 32, dv + 32);
                    tc_ld_wait();
                    // z_lam comes from global memory: 32 loads are issued before the first use (interleaved with the stores
                    // of dL/dh the compiler has to keep every load behind the previous store - the two pointers may alias for
                    // all it knows - and the loop ran at one DRAM latency per feature: 53 % of this kernel's stall samples)
                    float zn[32];
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
#pragma unroll
                        for (int x = 0; x < 32; ++x) zn[x] = __ldg(zp + (size_t)(64 * jb + 32 * hh + x) * TCM);
#pragma unroll
                        for (int x = 0; x < 32; ++x) {
                            const int r = 64 * jb + 32 * hh + x;
                            const bool on = fmaf(zn[x], scp[r], shp[r]) > 0.f;
                            dv[32 * hh + x] = on ? dv[32 * hh + x] : 0.f;
                        }
#pragma unroll
                        for (int x = 0; x < 32; ++x) out[(size_t)(64 * jb + 32 * hh + x) * TCM] = dv[32 * hh + x];
                    }
                    // per-warp sums in float32 (32 addends), float64 across tiles: ample for gradients
                    float a[2], b[2];
                    tc_warp_feature_sums(dv, lane, a[0], a[1]);
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
#pragma unroll
                        for (int x = 0; x < 32; ++x) zn[x] = __ldg(zp + (size_t)(64 * jb + 32 * hh + x) * TCM);
#pragma unroll
                        for (int x = 0; x < 32; ++x) {
                            const int r = 64 * jb + 32 * hh + x;
                            dv[32 * hh + x] *= (zn[x] - mup[r]) * rsp[r];
                        }
                    }
                    tc_warp_feature_sums(dv, lane, b[0], b[1]);
#pragma unroll
                    for (int y = 0; y < 4; ++y)
                        if (y == jb) { s1[y][0] += (double)a[0]; s1[y][1] += (double)a[1]; s2[y][0] += (double)b[0]; s2[y][1] += (double)b[1]; }
                }
            } else {
                const float* xs = A.saved + ((long long)c * A.B + (valid ? pt : 0)) * rowlen;
                float dv[TCH];
                tc_ld16(tg, dv);
                tc_ld_wait();
#pragma unroll
                for (int x = 0; x < 16; ++x) {
                    dv[x] = x < q.P ? dv[x] : 0.f;
                    out[(size_t)x * TCM] = dv[x];
                }
#pragma unroll
                for (int x = 16; x < TCH; ++x) dv[x] = 0.f;
                float a[2], b[2];
                tc_warp_feature_sums(dv, lane, a[0], a[1]);
#pragma unroll
                for (int x = 0; x < 16; ++x) dv[x] = x < q.P ? dv[x] * (xs[q.feed[x]] - mup[x]) * rsp[x] : 0.f;
                tc_warp_feature_sums(dv, lane, b[0], b[1]);
                s1[0][0] += (double)a[0]; s1[0][1] += (double)a[1]; s2[0][0] += (double)b[0]; s2[0][1] += (double)b[1];
            }
            tc_fence_before();
            mbar_arrive(&d_free);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    // ---- fold: lane i of a warp holds features 64 jb + 2 i, 64 jb + 2 i + 1 -----------------------------------------
    double* red = reinterpret_cast<double*>(sm + L.red);
    if (warp < 4) {
        double* r = red + ((size_t)warp * 32 + lane) * 16;
#pragma unroll
        for (int j = 0; j < 4; ++j) { r[4 * j] = s1[j][0]; r[4 * j + 1] = s1[j][1]; r[4 * j + 2] = s2[j][0]; r[4 * j + 3] = s2[j][1]; }
    }
    __syncthreads();
    double* mine = A.partials + (size_t)blockIdx.x * 2 * maxW;
    for (int f = tid; f < maxW; f += WD_THREADS) {
        double a = 0.0, b = 0.0;
        if (f < win) {
            const int j = f >> 6, ln = (f & 63) >> 1, ix = f & 1;
            for (int w = 0; w < 4; ++w) {
                a += red[((size_t)w * 32 + ln) * 16 + 4 * j + ix];
                b += red[((size_t)w * 32 + ln) * 16 + 4 * j + 2 + ix];
            }
        }
        mine[f] = a; mine[maxW + f] = b;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(A.counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    float* gp = A.grad_params + q.param_off + F.p_bn_gamma(c, lam);
    for (int f = tid; f < win; f += WD_THREADS) {
        double a = 0.0, b = 0.0;
        for (unsigned k = 0; k < gridDim.x; ++k) {
            a += __ldcg(A.partials + (size_t)k * 2 * maxW + f);
            b += __ldcg(A.partials + (size_t)k * 2 * maxW + maxW + f);
        }
        A.bnb[lam * 2 * maxW + f] = (float)(a / (double)A.B);
        A.bnb[lam * 2 * maxW + maxW + f] = (float)(b / (double)A.B);
        gp[f] += (float)b;              // dL/dgamma
        gp[win + f] += (float)a;        // dL/dbeta
    }
    if (tid == 0) *A.counter = 0u;
}

// ===================================================================================================
// wgrad of linear layer lam
// ===================================================================================================
#define BWW_THREADS 256       // 8 point warps, two threads per point (each fills half of the operand rows); thread 0 issues the MMAs
                              // (a ninth warp would put three warps on one scheduler: 168 registers per thread instead of 255)
#define BWW_FLUSH 8

// grid = (row blocks of 64 upstream features) x (column blocks of 128 features of h_lam) x nparts
template <bool OUTL>
__global__ void __launch_bounds__(BWW_THREADS, 1) flow_bwd_wide_wgrad_kernel(const __grid_constant__ DevFlow F, const BwArgs A) {
    extern __shared__ char smraw[];
    __shared__ uint64_t a_ready, done;
    __shared__ uint32_t tmem_base_s;
    __shared__ float coef[256];                             // sc[128] sh[128] of this column block
    char* sm = smem_align1024(smraw);
    const int tid = threadIdx.x, warp = tid >> 5;
    const int c = A.c, lam = A.lam;
    const DevCell& q = F.cells[c];
    const int d = F.d, W = F.widths[0], Kp = wd_kp16(F);
    const int N = lam == 0 ? 16 : (W < 128 ? W : 128);      // columns of this CTA's block
    const int nlog = q.T * Kp;
    const int nrows = OUTL ? nlog : W;                      // real upstream features
    const int rb = blockIdx.x, nh = blockIdx.y, part = blockIdx.z;
    char* slabA = sm;                                       // [128: dz hi (64) ; dz lo (64)][128 points]
    char* slabBh = sm + 65536;                              // [N][128 points]
    char* slabBl = sm + 65536 + 65536;
    const float* pk = A.wpack + q.pk_off;
    for (int j = tid; j < 128; j += BWW_THREADS) {
        const int f = 128 * nh + j;
        const bool ok = lam == 0 ? j < q.P : (f < W && j < N);
        coef[j] = ok ? pk[q.aff_off[lam] + f] : 0.f;
        coef[128 + j] = ok ? pk[q.aff_off[lam] + pad8(lam == 0 ? q.P : W) + f] : 0.f;
    }
    if (tid == 0) {
        mbar_init(&a_ready, 2 * TCM); mbar_init(&done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(128));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    const long long ntiles = A.ntiles, rowlen = d + 1;
    float* slice = A.slices + ((((size_t)rb * gridDim.y + nh) * gridDim.z + part) * 128) * 128;

    {
        // two threads per point: `half` 0 / 1 fills rows [0,32) / [32,64) of the upstream block and the lower / upper half of
        // the h block, all of a thread's loads of a round issued before the first shared-memory store (the stores are
        // generic, so the compiler keeps later global loads behind them)
        const int gt = tid & 127, half = tid >> 7;
        const uint32_t idesc = tc_idesc(TCM, N);
        const uint32_t sA = smem_u32(slabA), sBh = smem_u32(slabBh), sBl = smem_u32(slabBl);
        const uint32_t tg = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
        unsigned n = 0;
        int nflush = 0;
        // A: 64 upstream features [64 rb, 64 rb + 64), 32 per thread; B: h_lam features [128 nh, 128 nh + N), nb = N / 2 per
        // thread (lam = 0: the normalised pass-through columns, 16 rows, by half 0).  The operand values of the NEXT tile
        // are loaded into registers before the wait for this tile's MMAs, so their latency hides behind the tensor work.
        const int nb = N >> 1;
        const bool two = lam > 0 && nb > 32;
        // K-major 128B-swizzled slab address of (row, point gt) = base[row & 7] + (row >> 3) * 1024: eight bases per operand,
        // this thread's first row folded in, so that every store is base + immediate
        char* pA[8];
        char* pB[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int sw = i * 128 + (((((gt & 31) >> 2) ^ i) << 4) | ((gt & 3) << 2));
            pA[i] = slabA + (gt >> 5) * 128 * 128 + (32 * half >> 3) * 1024 + sw;
            pB[i] = slabBh + (gt >> 5) * N * 128 + (lam > 0 ? (nb * half >> 3) * 1024 : 0) + sw;
        }
        const float* cf = coef + nb * half;
        float v[32], w[32], w2[32];
        auto load_tile = [&](long long tile) {
            const float* up = (OUTL ? A.dl + (size_t)tile * nlog * TCM : A.dz + (size_t)tile * W * TCM) + (size_t)(64 * rb + 32 * half) * TCM + gt;
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = 64 * rb + 32 * half + j < nrows ? up[(size_t)j * TCM] : 0.f;
            if (lam > 0) {
                const float* zp = A.zbuf + (((size_t)(lam - 1) * ntiles + tile) * W + 128 * nh + nb * half) * TCM + gt;
#pragma unroll
                for (int j = 0; j < 32; ++j) w[j] = zp[(size_t)j * TCM];
                if (two) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) w2[j] = zp[(size_t)(32 + j) * TCM];
                }
            }
        };
        if (part < ntiles) load_tile(part);
        for (long long tile = part; tile < ntiles; tile += gridDim.z, ++n) {
            const long long pt = tile * TCM + gt;
            const bool valid = pt < A.B;
            // pull the tile after the next one into L2 (its operand blocks are contiguous in the tile-blocked buffers)
            if (tid == 0 && tile + 2 * gridDim.z < ntiles) {
                const long long tn = tile + 2 * gridDim.z;
                const int rows_here = nrows - 64 * rb < 64 ? nrows - 64 * rb : 64;
                if (rows_here > 0)
                    bulk_prefetch_l2((OUTL ? A.dl + (size_t)tn * nlog * TCM : A.dz + (size_t)tn * W * TCM) + (size_t)(64 * rb) * TCM,
                                     (uint32_t)rows_here * TCM * 4);
                if (lam > 0) bulk_prefetch_l2(A.zbuf + (((size_t)(lam - 1) * ntiles + tn) * W + 128 * nh) * TCM, (uint32_t)N * TCM * 4);
            }
            // hi rounded to nearest; the residual is exact in float32 and left as it is (the MMA truncates it: 2^-22 of the value)
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const float hi = tf32_rn(v[j]);
                *reinterpret_cast<float*>(pA[j & 7] + (j >> 3) * 1024) = hi;
                *reinterpret_cast<float*>(pA[j & 7] + (8 + (j >> 3)) * 1024) = v[j] - hi;
            }
            if (lam > 0) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float h = fmaxf(fmaf(w[j], cf[j], cf[128 + j]), 0.f);
                    const float hi = tf32_rn(h);
                    *reinterpret_cast<float*>(pB[j & 7] + (j >> 3) * 1024) = hi;
                    *reinterpret_cast<float*>(pB[j & 7] + (j >> 3) * 1024 + 65536) = h - hi;
                }
                if (two) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float h = fmaxf(fmaf(w2[j], cf[32 + j], cf[160 + j]), 0.f);
                        const float hi = tf32_rn(h);
                        *reinterpret_cast<float*>(pB[j & 7] + (4 + (j >> 3)) * 1024) = hi;
                        *reinterpret_cast<float*>(pB[j & 7] + (4 + (j >> 3)) * 1024 + 65536) = h - hi;
                    }
                }
            }
            if (lam == 0 && half == 0) {
                const float* xs = A.saved + ((long long)c * A.B + (valid ? pt : 0)) * rowlen;
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const float a = k < q.P ? fmaf(xs[q.feed[k]], coef[k], coef[128 + k]) : 0.f;
                    const float hi = tf32_rn(a);
                    *reinterpret_cast<float*>(pB[k & 7] + (k >> 3) * 1024) = hi;
                    *reinterpret_cast<float*>(pB[k & 7] + (k >> 3) * 1024 + 65536) = a - hi;
                }
            }
            proxy_fence();
            tc_fence_before();
            mbar_arrive(&a_ready);
            const bool lastt = tile + gridDim.z >= ntiles;
            if (!lastt) load_tile(tile + gridDim.z);
            if (tid == 0) {
                mbar_wait(&a_ready, n & 1);
                tc_fence_after();
                uint32_t acc = (n % BWW_FLUSH) != 0;
#pragma unroll
                for (int ks = 0; ks < 16; ++ks) {
                    const uint32_t ao = (ks >> 2) * 128 * 128 + (ks & 3) * 32;
                    const uint32_t bo = (ks >> 2) * N * 128 + (ks & 3) * 32;
                    tc_mma_tf32_ss(tmem_base, tc_desc(sA + ao), tc_desc(sBh + bo), idesc, acc);
                    acc = 1;
                    tc_mma_tf32_ss(tmem_base, tc_desc(sA + ao), tc_desc(sBl + bo), idesc, 1);
                }
                tc_commit(&done);
            }
            __syncwarp();
            mbar_wait(&done, n & 1);
            tc_fence_after();
            if ((n % BWW_FLUSH) == BWW_FLUSH - 1 || lastt) {
                // accumulator -> slice (fp32, round to nearest); the next tile starts a new accumulation
                float* sl = slice + (size_t)gt * 128;
                const int jb = N >= 32 ? (N >> 1) * half : 0, je = N >= 32 ? jb + (N >> 1) : (half == 0 ? N : 0);
                for (int j0 = jb; j0 < je; j0 += 16) {
                    float r[16];
                    tc_ld16(tg + j0, r);
                    tc_ld_wait();
                    // the first flush stores, the later ones add with vector reductions (no round trip to wait for; every
                    // element belongs to this thread alone, so the order of the additions is fixed)
                    float4* o4 = reinterpret_cast<float4*>(sl + j0);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (nflush)
                            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o4 + j), "f"(r[4 * j]), "f"(r[4 * j + 1]),
                                         "f"(r[4 * j + 2]), "f"(r[4 * j + 3]) : "memory");
                        else
                            o4[j] = make_float4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                    }
                }
                ++nflush;
                tc_fence_before();
            }
        }
        if (nflush == 0 && half == 0) {                      // a CTA without tiles still owns a slice
            float* sl = slice + (size_t)gt * 128;
            for (int j = 0; j < N; ++j) sl[j] = 0.f;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(128));
}

// grad_params[layer lam of cell c] += slices (fixed order)
__global__ void flow_bwd_wide_reduce_kernel(DevFlow F, const float* __restrict__ slices, int c, int lam, int nrb, int nnh, int nparts,
                                            float* __restrict__ grad_params) {
    const DevCell& q = F.cells[c];
    const int W = F.widths[0], Kp = wd_kp16(F);
    const int in = lam == 0 ? q.P : W;
    const int nout = lam == F.depth ? q.T * F.K : W;
    float* gw = grad_params + q.param_off + F.p_lin(c, lam);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)nout * in; i += (long long)gridDim.x * blockDim.x) {
        const int o = (int)(i / in), k = (int)(i - (long long)o * in);
        int row = o;                                         // row of the upstream tile
        if (lam == F.depth) { const int t = o / F.K, j = o - t * F.K; row = t * Kp + j; }
        const int rb = row >> 6, r = row & 63, nh = lam == 0 ? 0 : k >> 7, col = lam == 0 ? k : k & 127;
        // eight slices' loads in flight at a time, added in slice order (the sum is the same as one slice after the other)
        const float* sl0 = slices + (((size_t)rb * nnh + nh) * nparts * 128) * 128 + (size_t)r * 128 + col;
        float s = 0.f;
        int p = 0;
        for (; p + 8 <= nparts; p += 8) {
            float t[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const float* sl = sl0 + (size_t)(p + u) * 128 * 128;
                t[u] = __ldcg(sl) + __ldcg(sl + 64 * 128);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) s += t[u];
        }
        for (; p < nparts; ++p) {
            const float* sl = sl0 + (size_t)p * 128 * 128;
            s += __ldcg(sl) + __ldcg(sl + 64 * 128);
        }
        gw[i] += s;
    }
}

// ---------------------------------------------------------------------------------------------------
bool nis_bwd_wide_supported(const DevFlow& F) {
    if (!nis_wide_supported(F, NIS_BN_TRAIN)) return false;
    const int W = F.widths[0];
    if (W != 64 && W != 128 && W != 256) return false;      // wgrad column blocks of min(W, 128)
    for (int c = 0; c < F.n_cells; ++c) {
        if (bw_head_layout(F, F.cells[c].P, F.depth == 1).slots < 2) return false;
        if (bw_kout(F, F.cells[c].T) > 4096) return false;
    }
    if (bw_dg_layout(F, 1).slots < 2) return false;
    return true;
}

// wgrad slices: one [128][128] accumulator per CTA of a wgrad launch (row block x column block x part of the tiles)
#define BW_SLICES 320

struct BwScratch { float *gstate, *zbuf, *dl, *dh[2], *dz, *bnb, *slices, *dgpack; size_t floats; };
static void bw_carve(const DevFlow& F, int64_t B, float* base, BwScratch* s) {
    auto up = [](size_t x) { return (x + 63) & ~(size_t)63; };
    const size_t tiles = (size_t)((B + TCM - 1) / TCM), W = F.widths[0];
    const int T = bw_tmax(F);
    size_t off = 0;
    s->gstate = base + off; off = up(off + (size_t)B * (F.d + 1));
    s->zbuf = base + off; off = up(off + (size_t)F.depth * tiles * W * TCM);
    s->dl = base + off; off = up(off + tiles * (size_t)bw_kout(F, T) * TCM);
    s->dh[0] = base + off; off = up(off + tiles * W * TCM);
    s->dh[1] = base + off; off = up(off + tiles * W * TCM);
    s->dz = base + off; off = up(off + tiles * W * TCM);
    s->bnb = base + off; off = up(off + (size_t)(F.depth + 1) * 2 * F.maxW);
    s->slices = base + off; off = up(off + (size_t)BW_SLICES * 128 * 128);
    s->dgpack = base + off; off = up(off + (size_t)F.n_cells * bw_dg_cell_floats(F));
    s->floats = off;
}
size_t nis_bwd_wide_scratch_floats(const DevFlow& F, int64_t B) {
    BwScratch s;
    bw_carve(F, B, nullptr, &s);
    return s.floats;
}

int nis_flow_backward_wide(const DevFlow& F, const FlowWorkspace& ws, const float* params, const float* saved,
                           const float* bn_saved, const float* act_saved, const void* grad_out, int grad_dtype,
                           float* grad_params, void* grad_in, int64_t B, cudaStream_t s) {
    BwScratch sc;
    bw_carve(F, B, ws.bwd, &sc);
    const int sms = nis_sm_count();
    const long long ntiles = (B + TCM - 1) / TCM;
    const int grid = (int)(ntiles < sms ? ntiles : sms);
    const int W = F.widths[0], Kp = wd_kp16(F), depth = F.depth;
    flow_bwd_wide_pack_kernel<<<dim3(128, F.n_cells), 256, 0, s>>>(F, params, sc.dgpack);
    NIS_CUDA_CHECK_LAUNCH();
    int rc = nis_wide_pack(F, params, ws.tcpack, s);
    if (rc) return rc;
    BwArgs A;
    A.saved = saved; A.grad_out = grad_out; A.grad_dtype = grad_dtype; A.gstate = sc.gstate;
    A.params = params; A.wpack = ws.wpack; A.bn_saved = bn_saved; A.widepack = ws.tcpack; A.dgpack = sc.dgpack;
    A.zbuf = sc.zbuf; A.dl = sc.dl; A.dz = sc.dz; A.bnb = sc.bnb; A.slices = sc.slices; A.grad_params = grad_params;
    A.partials = ws.partials; A.counter = ws.counter; A.B = B; A.ntiles = ntiles;
    A.dh_in = nullptr; A.dh_out = nullptr; A.lam = 0; A.nparts = 1;
    const size_t tile_fl = (size_t)W * TCM;
    BwdTailArgs Ta;
    Ta.saved = saved; Ta.gstate = sc.gstate; Ta.wpack = ws.wpack; Ta.bn_saved = bn_saved; Ta.bnb = sc.bnb;
    Ta.grad_dtype = grad_dtype; Ta.B = B; Ta.tile_floats = (int)tile_fl;
    const long long rows = (long long)B * (F.d + 1);
    auto headk = F.kind == NIS_KIND_PWLIN ? flow_bwd_wide_head_kernel<NIS_KIND_PWLIN> : flow_bwd_wide_head_kernel<NIS_KIND_PWQUAD>;
    NIS_ENSURE_SMEM((flow_bwd_wide_wgrad_kernel<true>), 196608 + 1024);
    NIS_ENSURE_SMEM((flow_bwd_wide_wgrad_kernel<false>), 196608 + 1024);
    for (int c = F.n_cells - 1; c >= 0; --c) {
        const DevCell& q = F.cells[c];
        A.c = c; A.first = c == F.n_cells - 1;
        // ---- z_1 .. z_depth: kept by nis_flow_forward_cached, or recomputed with the forward's layer passes (BN from the
        //      saved batch statistics) ------------------------------------------------------------------------------------
        if (act_saved) {
            A.zbuf = act_saved + (size_t)c * depth * ntiles * tile_fl;
        } else {
            FwdArgs Fa;
            Fa.in_cols = F.d + 1;
            Fa.state_in = saved + (long long)c * rows; Fa.from_state = 1;
            Fa.params = params; Fa.wpack = ws.wpack; Fa.partials = ws.partials; Fa.counter = ws.counter;
            Fa.B = B; Fa.c_begin = c; Fa.c_end = c + 1;
            Fa.no_stats = 1;
            for (int l = 2; l <= depth; ++l) {
                Fa.stats_layer = l;
                Fa.zin = l > 2 ? sc.zbuf + (size_t)(l - 2) * ntiles * tile_fl : nullptr;
                Fa.zout = sc.zbuf + (size_t)(l - 1) * ntiles * tile_fl;
                Fa.z1out = l == 2 ? sc.zbuf : nullptr;
                rc = nis_launch_wide(F, Fa, ws.tcpack, s);
                if (rc) return rc;
            }
        }
        // ---- head ----------------------------------------------------------------------------------------------------
        {
            const size_t smem = (size_t)bw_head_layout(F, q.P, depth == 1).total + 1024;
            if (F.kind == NIS_KIND_PWLIN) NIS_ENSURE_SMEM((flow_bwd_wide_head_kernel<NIS_KIND_PWLIN>), (int)smem);
            else NIS_ENSURE_SMEM((flow_bwd_wide_head_kernel<NIS_KIND_PWQUAD>), (int)smem);
            headk<<<grid, WD_THREADS, smem, s>>>(F, A);
            NIS_CUDA_CHECK_LAUNCH();
        }
        // ---- linear layers depth .. 0: dgrad then wgrad ---------------------------------------------------------------
        int pp = 0;
        for (int lam = depth; lam >= 0; --lam) {
            A.lam = lam;
            A.dh_in = sc.dh[pp]; A.dh_out = sc.dh[pp ^ 1];
            const size_t smem = (size_t)bw_dg_layout(F, lam).total + 1024;
            if (lam == depth) {
                NIS_ENSURE_SMEM((flow_bwd_wide_dgrad_kernel<true>), (int)smem);
                flow_bwd_wide_dgrad_kernel<true><<<grid, WD_THREADS, smem, s>>>(F, A);
            } else {
                NIS_ENSURE_SMEM((flow_bwd_wide_dgrad_kernel<false>), (int)smem);
                flow_bwd_wide_dgrad_kernel<false><<<grid, WD_THREADS, smem, s>>>(F, A);
            }
            NIS_CUDA_CHECK_LAUNCH();
            pp ^= 1;
            const int nrows = lam == depth ? q.T * Kp : W;
            const int nrb = (nrows + 63) / 64, nnh = lam == 0 ? 1 : (W + 127) / 128;
            int nparts = (2 * sms) / (nrb * nnh);
            if (nparts < 1) nparts = 1;
            if (nparts > BW_SLICES / (nrb * nnh)) nparts = BW_SLICES / (nrb * nnh);
            if (nparts > ntiles) nparts = (int)ntiles;
            if (nparts < 1) return NIS_EUNSUPPORTED;
            A.nparts = nparts;
            const size_t wsm = 196608 + 1024;
            if (lam == depth) flow_bwd_wide_wgrad_kernel<true><<<dim3(nrb, nnh, nparts), BWW_THREADS, wsm, s>>>(F, A);
            else flow_bwd_wide_wgrad_kernel<false><<<dim3(nrb, nnh, nparts), BWW_THREADS, wsm, s>>>(F, A);
            NIS_CUDA_CHECK_LAUNCH();
            flow_bwd_wide_reduce_kernel<<<148, 256, 0, s>>>(F, sc.slices, c, lam, nrb, nnh, nparts, grad_params);
            NIS_CUDA_CHECK_LAUNCH();
        }
        // ---- tail ------------------------------------------------------------------------------------------------------
        Ta.c = c; Ta.dh_in = sc.dh[pp]; Ta.grad_in = c == 0 ? grad_in : nullptr;
        rc = launch_flow_bwd_tail(F, Ta, s);
        if (rc) return rc;
    }
    return NIS_OK;
}
