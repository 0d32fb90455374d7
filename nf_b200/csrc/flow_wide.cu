// Coupling-cell forward for WIDE conditioners (hidden width 128..256, any bin count) on tcgen05 / TMEM —
// BASELINE configs[4]: 16-D PWQuad, 64 bins, MLP [256]*4, where the conditioner is a real dense contraction
// (7.4 MFLOP per point).
//
// A 256-wide layer does not fit the resident-weights scheme of flow_tc_h.cu (one layer's hi/lo operand is
// 512 KB), so the layer runs as a streamed GEMM per 128-point tile:
//   * weights are packed once per forward as K-panels of 32 input features, [N rows][32] hi then lo in the
//     K-major 128B-swizzled UMMA layout, and STREAMED from L2 through a ring of shared-memory slots by
//     cp.async.bulk (TMA) from a dedicated producer warp (full/empty mbarriers per slot);
//   * the activations enter as the A operand from TENSOR MEMORY, 32 input features at a time (two ping-pong
//     chunks of 32 hi + 32 lo columns): the point threads load the stored pre-BN activations of the previous
//     layer, apply BN scale/shift + ReLU, split hi/lo and tcgen05.st them while the MMAs of the previous
//     chunk run;
//   * 3xTF32 as everywhere (hi*hi + hi*lo + lo*hi), but into TWO accumulators: tcgen05.mma truncates when it
//     adds a K=8 step into the fp32 accumulator (tools/tc_accum_probe.cu: ~1 ulp per instruction, toward
//     zero), and with K = 256 one accumulator would take 96 such steps (measured: log J twice as far from
//     the float64 oracle as torch-fp32).  The hi*hi products (32 steps) go to D_hi, the two cross products
//     (2^-11 smaller, so their truncation does not matter) to D_x, and the epilogue adds the two in fp32.
//     N <= 192 per round (2 x 192 accumulator columns); a 256-wide layer is two rounds of 128 outputs.
// One launch = one layer of one cell (the train-mode layer-pass scheme of flow_tiled.cu / flow_tc_h.cu, which
// also serves eval mode here: activations round-trip through HBM tile-blocked [tile][W][128], 1 KB/point/layer,
// far below the tensor time).  The final pass runs the output layer one transformed dimension at a time
// (N = K logits padded to 16), stages the logits in shared memory and runs the spline of spline.cuh on them.
#include <stdlib.h>
#include "common.cuh"
#include "spline.cuh"
#include "tc_common.cuh"
#include "flow_fwd_common.cuh"
#include "flow_host.cuh"

#include "wide_common.cuh"

__global__ void flow_wide_pack_kernel(DevFlow F, const float* __restrict__ params, float* __restrict__ widepack) {
    const int c = blockIdx.y;
    const DevCell& q = F.cells[c];
    const float* p = params + q.param_off;
    const int W = F.widths[0], Kp = wd_kp16(F);
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nth = (long long)gridDim.x * blockDim.x;
    char* dst = reinterpret_cast<char*>(widepack + (size_t)c * wd_cell_floats(F));
    for (int l = 1; l < F.depth; ++l) {
        const float* w = p + F.p_lin(c, l);                 // [W][W]
        char* base = dst + (size_t)(l - 1) * W * W * 2 * 4;
        for (long long i = tid; i < (long long)W * W; i += nth) {
            const int no = (int)(i / W), k = (int)(i - (long long)no * W);
            const int Nr = wd_hid_n(W), r = no / Nr, n = no - r * Nr;      // round r holds outputs [r Nr, r Nr + Nr)
            const int kt = k >> 5, kk = k & 31;
            const float v = w[i];
            const float h = tf32_rn(v);
            char* panel = base + ((size_t)r * Nr * W * 2 + (size_t)kt * Nr * 64) * 4;
            const int off = (n >> 3) * 1024 + (n & 7) * 128 + ((((kk >> 2) ^ (n & 7)) << 4) | ((kk & 3) << 2));
            *reinterpret_cast<float*>(panel + off) = h;
            *reinterpret_cast<float*>(panel + (size_t)Nr * 128 + off) = tf32_rn(v - h);
        }
    }
    const float* wo = p + F.p_out_w(c);                     // [T*K][W]
    char* obase = dst + (size_t)(F.depth - 1) * W * W * 2 * 4;
    for (long long i = tid; i < (long long)q.T * Kp * W; i += nth) {
        const int t = (int)(i / ((long long)Kp * W));
        const int r = (int)(i - (long long)t * Kp * W);
        const int n = r / W, k = r - n * W;
        const int kt = k >> 5, kk = k & 31;
        const float v = n < F.K ? wo[((size_t)t * F.K + n) * W + k] : 0.f;
        const float h = tf32_rn(v);
        char* panel = obase + ((size_t)t * Kp * W * 2 + (size_t)kt * Kp * 64) * 4;
        const int off = (n >> 3) * 1024 + (n & 7) * 128 + ((((kk >> 2) ^ (n & 7)) << 4) | ((kk & 3) << 2));
        *reinterpret_cast<float*>(panel + off) = h;
        *reinterpret_cast<float*>(panel + (size_t)Kp * 128 + off) = tf32_rn(v - h);
    }
}

template <int KIND>
__global__ void __launch_bounds__(WD_THREADS, 1) flow_wide_tc_kernel(const __grid_constant__ DevFlow F, const FwdArgs A,
                                                                      const float* __restrict__ widepack) {
    extern __shared__ char smraw[];
    __shared__ uint64_t full[WD_MAX_SLOTS], empty[WD_MAX_SLOTS], a_ready[2], a_free[2], d_ready, d_free;
    __shared__ uint32_t tmem_base_s;
    char* sm = smem_align1024(smraw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c = A.c_begin;
    const DevCell& q = F.cells[c];
    const int d = F.d, depth = F.depth, W = F.widths[0], kc = W >> 5, Kp = wd_kp16(F);     // kc: chunks of 32 features
    const bool stats = A.stats_layer >= 1;                 // hidden pass producing z_{stats_layer}
    const bool final_pass = !stats;
    const int lam = stats ? A.stats_layer - 1 : depth;     // the linear layer this launch multiplies by (1..depth)
    const bool from_z = A.zin != nullptr;                  // else lam == 1 and z_1 is computed from the state
    const WdSmem L = wd_layout(F, q.P, final_pass, !from_z);
    const int RS = L.slots;
    const int npanel = final_pass ? Kp : wd_hid_n(W);      // N of the MMAs
    const int rounds = final_pass ? q.T : wd_hid_rounds(W);
    float* w0s = reinterpret_cast<float*>(sm + L.w0);
    float* affs = reinterpret_cast<float*>(sm + L.aff);    // sc0[16] sh0[16] sc_lam[W] sh_lam[W]
    float* biass = reinterpret_cast<float*>(sm + L.bias);
    const float* pk = A.wpack + q.pk_off;
    const float* cellpack = widepack + (size_t)c * wd_cell_floats(F);

    if (!from_z) {
        const float* s0 = pk + q.wt_off[0];                // layer 0, [P][W] k-major
        for (int i = tid; i < q.P * W; i += WD_THREADS) w0s[i] = s0[i];
    }
    for (int i = tid; i < 16; i += WD_THREADS) {
        affs[i] = i < q.P ? pk[q.aff_off[0] + i] : 0.f;
        affs[16 + i] = i < q.P ? pk[q.aff_off[0] + pad8(q.P) + i] : 0.f;
    }
    for (int i = tid; i < W; i += WD_THREADS) {
        affs[32 + i] = pk[q.aff_off[lam] + i];
        affs[32 + W + i] = pk[q.aff_off[lam] + W + i];
    }
    if (final_pass)
        for (int i = tid; i < q.T * Kp; i += WD_THREADS) {
            const int t = i / Kp, n = i - t * Kp;
            biass[i] = n < F.K ? pk[q.bo_off + t * F.Kpad + n] : 0.f;
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
    const long long ntiles = (A.B + TCM - 1) / TCM;
    const long long rowlen = d + 1;
    const int kpanels = kc;                                 // K-panels of 32 per round (one per A chunk)
    const size_t panel_floats = (size_t)npanel * 64;
    // BatchNorm statistics of a hidden pass: thread t of the point warps owns feature 64 j + (t >> 1) of every 64-feature block j
    // (both threads of a pair hold the same sums)
    double dsum[4], dsq[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { dsum[j] = dsq[j] = 0.0; }

    if (warp == 5) {
        // ===================== weight producer: panels in consumption order through the ring ===============
        if (lane == 0) {
            unsigned pc = 0;
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                for (int r = 0; r < rounds; ++r) {
                    const float* src = cellpack + (final_pass ? (size_t)(depth - 1) * W * W * 2 + (size_t)r * Kp * W * 2
                                                              : (size_t)(lam - 1) * W * W * 2 + (size_t)r * npanel * W * 2);
                    for (int p = 0; p < kpanels; ++p, ++pc) {
                        const unsigned slot = pc % RS;
                        mbar_wait(&empty[slot], ((pc / RS) & 1) ^ 1);
                        bulk_load(sm + L.ring + slot * L.slot_bytes, src + p * panel_floats, (uint32_t)L.slot_bytes, &full[slot]);
                    }
                }
            }
        }
    } else if (warp == 4) {
        // ===================== MMA issuer ======================================================
        if (lane == 0) {
            unsigned pc = 0, cc = 0, rr = 0;
            const uint32_t idesc = tc_idesc(TCM, npanel);
            for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                for (int r = 0; r < rounds; ++r, ++rr) {
                    mbar_wait(&d_free, (rr & 1) ^ 1);               // the previous accumulator has been read out
                    tc_fence_after();
                    uint32_t acc = 0;
                    for (int i = 0; i < kc; ++i, ++cc, ++pc) {
                        const unsigned buf = cc & 1;
                        mbar_wait(&a_ready[buf], (cc >> 1) & 1);
                        const unsigned slot = pc % RS;
                        mbar_wait(&full[slot], (pc / RS) & 1);
                        tc_fence_after();
                        const uint32_t ta = tmem_base + WD_COL_A + buf * 64;
                        const uint32_t bh = smem_u32(sm + L.ring + slot * L.slot_bytes), bl = bh + npanel * 128;
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            const uint32_t ah = ta + ks * 8;
                            tc_mma_tf32_ts(tmem_base, ah, tc_desc(bh + ks * 32), idesc, acc);                 // D_hi += a_hi w_hi
                            tc_mma_tf32_ts(tmem_base + WD_COL_X, ah, tc_desc(bl + ks * 32), idesc, acc);      // D_x  += a_hi w_lo
                            acc = 1;
                            tc_mma_tf32_ts(tmem_base + WD_COL_X, ah + 32, tc_desc(bh + ks * 32), idesc, 1);   // D_x  += a_lo w_hi
                        }
                        tc_commit(&empty[slot]);
                        tc_commit(&a_free[buf]);
                    }
                    tc_commit(&d_ready);
                }
            }
        }
    } else {
        // ===================== point threads ====================================================
        const int gt = tid;
        float* st = reinterpret_cast<float*>(sm + L.st) + gt;
        float* stg = reinterpret_cast<float*>(sm + L.stg) + gt;
        const uint32_t tg = tmem_base + ((uint32_t)(warp * 32) << 16);
        unsigned cc = 0, rr = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const long long pt = tile * TCM + gt;
            const bool valid = pt < A.B;
            if (valid) {
                if (A.from_state) {
                    for (int i = 0; i <= d; ++i) st[i * TCM] = A.state_in[pt * rowlen + i];
                } else {
                    for (int i = 0; i < d; ++i) st[i * TCM] = load_io(A.in, A.in_dtype, pt * A.in_cols + i);
                    st[d * TCM] = A.in_cols > d ? load_io(A.in, A.in_dtype, pt * A.in_cols + d) : 1.f;
                }
                if (final_pass && A.saved && !A.from_state) {
                    float* sv = A.saved + ((long long)c * A.B + pt) * rowlen;
                    for (int i = 0; i <= d; ++i) sv[i] = st[i * TCM];
                }
            } else {
                for (int i = 0; i < d; ++i) st[i * TCM] = 0.5f;
                st[d * TCM] = 1.f;
            }
            float a0[16];
            if (!from_z) {
#pragma unroll
                for (int k = 0; k < 16; ++k) a0[k] = k < q.P ? fmaf(st[q.feed[k] * TCM], affs[k], affs[16 + k]) : 0.f;
            }
            float jfac = 1.f;
            // A operand of round r: h_lam = ReLU(BN_lam(z_lam)), 32 features per chunk, handed to the MMA warp chunk by chunk
            auto feed = [&](int r) {
                for (int i = 0; i < kc; ++i, ++cc) {
                    const unsigned buf = cc & 1;
                    float v[32];
                    if (from_z) {
                        const float* zr = A.zin + ((size_t)tile * W + 32 * i) * TCM + gt;
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
                    }
                    if (!from_z && A.z1out && r == 0) {                // backward recompute: keep z_1
                        float* z1 = A.z1out + ((size_t)tile * W + 32 * i) * TCM + gt;
#pragma unroll
                        for (int j = 0; j < 32; ++j) z1[(size_t)j * TCM] = v[j];
                    }
                    float lo[32];
                    const float* sc = affs + 32 + 32 * i, *sh = affs + 32 + W + 32 * i;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float a = fmaxf(fmaf(v[j], sc[j], sh[j]), 0.f);
                        v[j] = tf32_rn(a);
                        lo[j] = tf32_rn(a - v[j]);
                    }
                    mbar_wait(&a_free[buf], ((cc >> 1) & 1) ^ 1);      // the MMAs that read this chunk buffer are done
                    tc_fence_after();
                    const uint32_t ta = tg + WD_COL_A + buf * 64;
                    tc_st32(ta, v);
                    tc_st32(ta + 32, lo);
                    tc_st_wait();
                    tc_fence_before();
                    mbar_arrive(&a_ready[buf]);
                }
            };
            feed(0);
            for (int r = 0; r < rounds; ++r, ++rr) {
                mbar_wait(&d_ready, rr & 1);
                tc_fence_after();
                if (stats) {
                    // ---- hidden pass: z_{lam+1} to HBM (tile-blocked) and its per-feature sums ----------------------
                    float* zo = A.zout + ((size_t)tile * W + (size_t)r * npanel) * TCM + gt;
#pragma unroll
                    for (int j = 0; j < 3; ++j) {
                        if (64 * j >= npanel) break;
                        float v[TCH], xx[TCH];
                        tc_ld32(tg + 64 * j, v);
                        tc_ld32(tg + 64 * j + 32, v + 32);
                        tc_ld32(tg + WD_COL_X + 64 * j, xx);
                        tc_ld32(tg + WD_COL_X + 64 * j + 32, xx + 32);
                        tc_ld_wait();
#pragma unroll
                        for (int x = 0; x < TCH; ++x) {
                            v[x] = valid ? v[x] + xx[x] : 0.f;
                            zo[(size_t)(64 * j + x) * TCM] = v[x];
                        }
                        if (!A.no_stats) {
                            // per-feature sums over the tile: the 64 x 128 block goes through shared memory (conflict-free
                            // column writes), then two threads per feature add half a row each with rotated 16-byte loads
                            // (float32 over the 128 points of the tile, float64 across tiles -- as flow_tc_h.cu does); the
                            // float64 shuffle tree this replaces was a third of the pass
#pragma unroll
                            for (int x = 0; x < TCH; ++x) stg[x * TCM] = v[x];
                            asm volatile("bar.sync 1, 128;" ::: "memory");
                            const float4* row = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(sm + L.stg) + (gt >> 1) * TCM + (gt & 1) * 64);
                            float s_ = 0.f, q_ = 0.f, q1 = 0.f;
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                const float4 x = row[(i + lane) & 15];
                                s_ += (x.x + x.y) + (x.z + x.w);
                                q_ = fmaf(x.x, x.x, fmaf(x.y, x.y, q_));
                                q1 = fmaf(x.z, x.z, fmaf(x.w, x.w, q1));
                            }
                            q_ += q1;
                            s_ += __shfl_xor_sync(0xffffffffu, s_, 1);
                            q_ += __shfl_xor_sync(0xffffffffu, q_, 1);
                            const int fb = (r * npanel >> 6) + j;          // 64-feature block of the layer
#pragma unroll
                            for (int y = 0; y < 4; ++y)
                                if (y == fb) { dsum[y] += (double)s_; dsq[y] += (double)q_; }
                            asm volatile("bar.sync 1, 128;" ::: "memory");
                        }
                    }
                    tc_fence_before();
                    mbar_arrive(&d_free);
                    if (r + 1 < rounds) feed(r + 1);
                } else {
                    // ---- final pass, transformed dimension t = r: logits -> shared memory -> spline ----------------
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
                    if (r + 1 < rounds) feed(r + 1);           // the next dimension's MMAs run while this one's spline does
                    const int col = q.trafo[t];
                    const float xv = st[col * TCM];
                    float y, f;
                    int kbin;
                    if (KIND == NIS_KIND_PWLIN) {
                        float S, al;
                        y = pwlin_fwd(stg, TCM, F.nb, xv, f, kbin, S, al);
                    } else {
                        QuadCtx qc;
                        pwquad_fwd<true>(stg, TCM, F.nb, xv, qc);
                        y = qc.y; f = qc.f; kbin = qc.k;
                    }
                    st[col * TCM] = y;
                    jfac *= f;
                    if (A.bins && valid) A.bins[((long long)c * A.B + pt) * d + t] = kbin;
                }
            }
            if (final_pass) {
                st[d * TCM] *= jfac;
                if (valid) {
                    if (A.state_out) {
                        float* so = A.state_out + pt * rowlen;
                        for (int i = 0; i <= d; ++i) so[i] = st[i * TCM];
                    }
                    if (A.to_out) {
                        for (int i = 0; i < d; ++i) store_io(A.out, A.out_dtype, pt * rowlen + i, st[F.out_perm[i] * TCM]);
                        store_io(A.out, A.out_dtype, pt * rowlen + d, st[d * TCM]);
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    if (!stats || A.no_stats) return;
    // ---- this CTA's sums: the even thread of a pair publishes feature 64 j + (tid >> 1) -------------------------------
    double* sacc = reinterpret_cast<double*>(sm + L.red);            // [2 * maxW]
    for (int f = W + tid; f < F.maxW; f += WD_THREADS) { sacc[f] = 0.0; sacc[F.maxW + f] = 0.0; }
    if (warp < 4 && !(tid & 1)) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int f = 64 * j + (tid >> 1);
            if (f < W) { sacc[f] = dsum[j]; sacc[F.maxW + f] = dsq[j]; }
        }
    }
    bn_stats_finalize(F, A, sacc, WD_THREADS);
}

// ---------------------------------------------------------------------------------------------------
// first hidden width of the streamed-weights kernels: 64, 128, 192 or 256
static bool wide_width(const DevFlow& F) { return F.depth >= 1 && F.widths[0] >= 64 && F.widths[0] <= 256 && !(F.widths[0] & 63); }

bool nis_wide_supported(const DevFlow& F, int bn_mode) {
    if (F.kind == NIS_KIND_AFFINE || !wide_width(F)) return false;  // (width 64 with 32 bins is taken by flow_tc_h.cu first where it applies)
    const int W = F.widths[0];
    for (int l = 0; l < F.depth; ++l) if (F.widths[l] != W) return false;
    if (F.maxW != W) return false;
    if (wd_kp16(F) > WD_NMAX) return false;
    for (int c = 0; c < F.n_cells; ++c) {
        if (F.cells[c].P > 16) return false;
        if (bn_mode == NIS_BN_TRAIN && !nis_moments_supported(F, c)) return false;
        if (wd_layout(F, F.cells[c].P, true, F.depth == 1).slots < 2) return false;
        if (wd_layout(F, F.cells[c].P, false, true).slots < 2) return false;
    }
    return true;
}

size_t nis_wide_pack_floats(const DevFlow& F) { return wide_width(F) ? (size_t)F.n_cells * wd_cell_floats(F) : 0; }

int nis_wide_pack(const DevFlow& F, const float* params, float* widepack, cudaStream_t s) {
    flow_wide_pack_kernel<<<dim3(128, F.n_cells), 256, 0, s>>>(F, params, widepack);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

int nis_launch_wide(const DevFlow& F, const FwdArgs& A, const float* widepack, cudaStream_t s) {
    const int sms = nis_sm_count();
    const bool final_pass = A.stats_layer < 1;
    const WdSmem L = wd_layout(F, F.cells[A.c_begin].P, final_pass, A.zin == nullptr);
    const size_t smem = (size_t)L.total + 1024;
    auto kern = F.kind == NIS_KIND_PWLIN ? flow_wide_tc_kernel<NIS_KIND_PWLIN> : flow_wide_tc_kernel<NIS_KIND_PWQUAD>;
    if (F.kind == NIS_KIND_PWLIN) NIS_ENSURE_SMEM((flow_wide_tc_kernel<NIS_KIND_PWLIN>), (int)smem);
    else NIS_ENSURE_SMEM((flow_wide_tc_kernel<NIS_KIND_PWQUAD>), (int)smem);
    const long long ntiles = (A.B + TCM - 1) / TCM;
    const int grid = (int)(ntiles < sms ? ntiles : sms);
    kern<<<grid, WD_THREADS, smem, s>>>(F, A, widepack);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}
