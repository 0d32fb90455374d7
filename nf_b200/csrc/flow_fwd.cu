// Fused coupling-cell flow, forward — shape-generic kernel (any n_flow / widths / bins).
//
// One thread owns one point for the whole flow: its state row, every conditioner activation and the
// per-dimension logits live in a private shared-memory column (stride NT, conflict-free), the weights
// are read as warp-uniform 128-bit loads from the repacked, transposed, zero-padded arena `wpack`
// (L1-resident), and the bin search / CDF / Jacobian product run in registers.  Eval-mode BN is one
// launch for all cells.  Train-mode BN (batch statistics, which is what the reference runs both in
// training and in integrate(): manager.py:225,397) needs one grid-wide reduction per BN layer; each
// is a "statistics pass" of the same kernel that stops at that layer, accumulates sum / sum-of-squares
// per feature in float64 and lets the last CTA to finish fold them into the layer's scale/shift.
//
// Reference semantics: coupling_cells.py:107-142 (PWLin), :159-228 (PWQuad), :230-254 (RectNN),
// layers.py:27-32,43-51,75-77,90-91 (Mask/DeMask/AddJacobian/Roll, folded into column tables).
#include <stdlib.h>
#include "common.cuh"
#include "spline.cuh"
#include <cooperative_groups.h>
#include "flow_fwd_common.cuh"
#include "flow_host.cuh"

// ---------------------------------------------------------------------------------------------------
// repack: torch-layout params -> transposed zero-padded weights (+ BN scale/shift: eval mode from the running statistics;
// train mode from bn_saved, the batch statistics a forward saved, for its backward; none in a train-mode forward, whose
// statistics passes write them)
// grid = (blocks, n_cells)
// ---------------------------------------------------------------------------------------------------
__global__ void flow_pack_kernel(DevFlow F, const float* __restrict__ params, const float* __restrict__ bn_running,
                                 const float* __restrict__ bn_saved, float* __restrict__ wpack, int bn_mode) {
    const int c = blockIdx.y;
    const DevCell& q = F.cells[c];
    const float* p = params + q.param_off;
    float* pk = wpack + q.pk_off;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    if (bn_mode == NIS_BN_EVAL || bn_saved) {
        for (int l = 0; l <= F.depth; ++l) {
            const int W = F.W(c, l), Wp = F.Wp(c, l);
            const long long g = F.p_bn_gamma(c, l), r = F.r_mean(c, l);
            for (int j = tid; j < Wp; j += nth) {
                float sc = 0.f, sh = 0.f;
                if (j < W && bn_mode == NIS_BN_EVAL) {
                    const float* rs = bn_running + q.bn_off;
                    sc = p[g + j] / sqrtf(rs[r + W + j] + F.eps);
                    sh = p[g + W + j] - rs[r + j] * sc;
                } else if (j < W) {
                    const float* sv = bn_saved + q.sv_off + l * 2 * F.maxW;
                    sc = p[g + j] * sv[F.maxW + j];
                    sh = p[g + W + j] - sv[j] * sc;
                }
                pk[q.aff_off[l] + j] = sc;
                pk[q.aff_off[l] + Wp + j] = sh;
            }
        }
    }
    int in = q.P;
    for (int l = 0; l < F.depth; ++l) {
        const int H = F.widths[l], Hp = pad8(H);
        const float* w = p + F.p_lin(c, l);
        float* wt = pk + q.wt_off[l];
        for (int i = tid; i < in * Hp; i += nth) {
            const int k = i / Hp, j = i - k * Hp;
            wt[i] = j < H ? w[(long long)j * in + k] : 0.f;
        }
        in = H;
    }
    const float* wo = p + F.p_out_w(c);
    const float* bo = p + F.p_out_b(c);
    const int K = F.K, Kp = F.Kpad;
    for (int i = tid; i < q.T * in * Kp; i += nth) {
        const int t = i / (in * Kp), r = i - t * in * Kp, k = r / Kp, j = r - k * Kp;
        pk[q.wo_off + i] = j < K ? wo[(long long)F.out_row(c, t, j) * in + k] : 0.f;
    }
    for (int i = tid; i < q.T * Kp; i += nth) {
        const int t = i / Kp, j = i - t * Kp;
        pk[q.bo_off + i] = j < K ? bo[F.out_row(c, t, j)] : 0.f;
    }
}

// one block per 256 floats of the largest cell, at most 64
int nis_pack_blocks(const DevFlow& F) {
    int mx = 0;
    for (int c = 0; c < F.n_cells; ++c) {
        int sz = (c + 1 < F.n_cells ? F.cells[c + 1].pk_off : F.pack_total) - F.cells[c].pk_off;
        if (sz > mx) mx = sz;
    }
    int bx = (mx + 255) / 256;
    return bx > 64 ? 64 : bx;
}

int launch_flow_pack(const DevFlow& F, const float* params, const float* bn_running, const float* bn_saved, float* wpack,
                     int bn_mode, cudaStream_t s) {
    flow_pack_kernel<<<dim3(nis_pack_blocks(F), F.n_cells), 256, 0, s>>>(F, params, bn_running, bn_saved, wpack, bn_mode);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

// ---------------------------------------------------------------------------------------------------
// dense layer for one point: out[j] = sum_k a[k] * Wt[k][j], 8 outputs per sweep
// ---------------------------------------------------------------------------------------------------
template <int NT, typename Epi>
__device__ __forceinline__ void dense8(const float* __restrict__ Wt, int in, int outp, const float* a_col, Epi epi) {
    for (int jb = 0; jb < outp; jb += 8) {
        float acc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = 0.f;
        const float* wrow = Wt + jb;
#pragma unroll 4
        for (int k = 0; k < in; ++k) {
            const float a = a_col[k * NT];
            const float4 w0 = __ldg(reinterpret_cast<const float4*>(wrow + (size_t)k * outp));
            const float4 w1 = __ldg(reinterpret_cast<const float4*>(wrow + (size_t)k * outp + 4));
            acc[0] = fmaf(a, w0.x, acc[0]); acc[1] = fmaf(a, w0.y, acc[1]);
            acc[2] = fmaf(a, w0.z, acc[2]); acc[3] = fmaf(a, w0.w, acc[3]);
            acc[4] = fmaf(a, w1.x, acc[4]); acc[5] = fmaf(a, w1.y, acc[5]);
            acc[6] = fmaf(a, w1.z, acc[6]); acc[7] = fmaf(a, w1.w, acc[7]);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) epi(jb + i, acc[i]);
    }
}

// per-feature sum / sum of squares of a [W][NT] tile into the CTA's float64 accumulators
template <int NT>
__device__ __forceinline__ void reduce_rows(const float* buf, int W, double* sacc, int maxW) {
    __syncthreads();
    for (int j = threadIdx.x; j < W; j += NT) {
        double s = 0.0, q = 0.0;
        for (int i = 0; i < NT; ++i) {
            const double v = (double)buf[j * NT + ((i + threadIdx.x) & (NT - 1))];
            s += v; q += v * v;
        }
        sacc[j] += s; sacc[maxW + j] += q;
    }
    __syncthreads();
}

template <int NT>
__device__ __forceinline__ void fwd_generic_body(const DevFlow& F, const FwdArgs& A, float* sm) {
    const int tid = threadIdx.x;
    const int d = F.d, maxW = F.maxW;
    const int bw = maxW > F.Kpad ? maxW : F.Kpad;
    float* st = sm + tid;                         // [(d+1)][NT]
    float* bufA = sm + (d + 1) * NT + tid;        // [bw][NT]  (either buffer may receive the logits)
    float* bufB = bufA + bw * NT;                 // [bw][NT]
    double* sacc = reinterpret_cast<double*>(sm + ((d + 1) + 2 * bw) * NT + (((d + 1) + 2 * bw) * NT & 1));
    const bool stats = A.stats_layer >= 0;
    if (stats) {
        for (int i = tid; i < 2 * maxW; i += NT) sacc[i] = 0.0;
        __syncthreads();
    }
    const long long ntiles = (A.B + NT - 1) / NT;
    const long long rowlen = d + 1;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long pt = tile * NT + tid;
        const bool valid = pt < A.B;
        // ---- load the state row -------------------------------------------------------------
        if (valid) {
            if (A.from_state) {
                for (int i = 0; i <= d; ++i) st[i * NT] = A.state_in[pt * rowlen + i];
            } else {
                // (inverse: the input is in the reference's OUTPUT column order, out_perm scatters it back)
                for (int i = 0; i < d; ++i) st[(A.inverse ? F.out_perm[i] : i) * NT] = load_io(A.in, A.in_dtype, pt * A.in_cols + i);
                st[d * NT] = A.in_cols > d ? load_io(A.in, A.in_dtype, pt * A.in_cols + d) : 1.f;
            }
        } else {
            for (int i = 0; i < d; ++i) st[i * NT] = 0.5f;
            st[d * NT] = 1.f;
        }
        bool tile_done = false;
        for (int ci = A.c_begin; ci < A.c_end && !tile_done; ++ci) {
            const int c = A.inverse ? A.c_end - 1 - (ci - A.c_begin) : ci;
            const DevCell& q = F.cells[c];
            const float* pk = A.wpack + q.pk_off;
            if (!stats && A.saved && valid && (!A.from_state || c > A.c_begin)) {
                float* sv = A.saved + ((long long)c * A.B + pt) * rowlen;
                for (int i = 0; i <= d; ++i) sv[i] = st[i * NT];
            }
            // ---- BN0 on the pass-through columns ----------------------------------------------
            if (A.stats_layer == 0) {
                for (int k = 0; k < q.P; ++k) bufA[k * NT] = valid ? st[q.feed[k] * NT] : 0.f;
                reduce_rows<NT>(bufA - tid, q.P, sacc, maxW);
                tile_done = true;
                break;
            }
            {
                const float* sc = pk + q.aff_off[0];
                const float* sh = sc + pad8(q.P);
                for (int k = 0; k < q.P; ++k) bufA[k * NT] = fmaf(st[q.feed[k] * NT], sc[k], sh[k]);
            }
            float* cur = bufA;
            float* nxt = bufB;
            int in = q.P;
            // ---- hidden layers: Linear(no bias) -> BN -> ReLU ----------------------------------
            for (int l = 0; l < F.depth; ++l) {
                const int H = F.widths[l], Hp = pad8(H);
                const float* Wt = pk + q.wt_off[l];
                if (A.stats_layer == l + 1) {
                    dense8<NT>(Wt, in, Hp, cur, [&](int j, float z) { nxt[j * NT] = valid ? z : 0.f; });
                    reduce_rows<NT>(nxt - tid, H, sacc, maxW);
                    tile_done = true;
                    break;
                }
                const float* sc = pk + q.aff_off[l + 1];
                const float* sh = sc + Hp;
                dense8<NT>(Wt, in, Hp, cur, [&](int j, float z) { nxt[j * NT] = fmaxf(fmaf(z, sc[j], sh[j]), 0.f); });
                float* t_ = cur; cur = nxt; nxt = t_;
                in = H;
            }
            if (tile_done) break;
            // ---- output layer + spline, one transformed dimension at a time --------------------
            float jfac = 1.f;
            for (int t = 0; t < q.T; ++t) {
                const float* Wt = pk + q.wo_off + (size_t)t * in * F.Kpad;
                const float* bo = pk + q.bo_off + t * F.Kpad;
                dense8<NT>(Wt, in, F.Kpad, cur, [&](int j, float z) { nxt[j * NT] = z + bo[j]; });
                const int col = q.trafo[t];
                const float x = st[col * NT];
                float y, f;
                int k;
                if (F.kind == NIS_KIND_AFFINE) {
                    // AffineCoupling (coupling_cells.py:49-68): y = atan(20 e^{Z0} x + relu(Z1)) / (pi/2); the Jacobian takes
                    // 20 e^{Z0} / (v^2 + 1) per dimension and 1/(pi/2) ONCE per cell (as the reference writes it)
                    const float s0 = 20.f * expf(nxt[0]), s1 = fmaxf(nxt[NT], 0.f);
                    k = 0;
                    if (A.inverse) {
                        const float v = tanf(x * 1.5707963267948966f);
                        y = (v - s1) / s0;
                        f = (v * v + 1.f) / s0;
                    } else {
                        const float v = fmaf(s0, x, s1);
                        y = atanf(v) * 0.6366197723675814f;
                        f = s0 / (v * v + 1.f);
                    }
                } else if (A.inverse) {
                    y = F.kind == NIS_KIND_PWLIN ? pwlin_inv(nxt, NT, F.nb, x, f, k) : pwquad_inv(nxt, NT, F.nb, x, f, k);
                    f = 1.f / f;
                } else if (F.kind == NIS_KIND_PWLIN) {
                    float S, al;
                    y = pwlin_fwd(nxt, NT, F.nb, x, f, k, S, al);
                } else {
                    QuadCtx qc;
                    pwquad_fwd(nxt, NT, F.nb, x, qc);
                    y = qc.y; f = qc.f; k = qc.k;
                }
                st[col * NT] = y;
                jfac *= f;
                if (A.bins && valid) A.bins[((long long)c * A.B + pt) * d + t] = k;
            }
            if (F.kind == NIS_KIND_AFFINE) jfac *= A.inverse ? 1.5707963267948966f : 0.6366197723675814f;
            st[d * NT] *= jfac;
        }
        if (stats || !valid) continue;
        // ---- store ------------------------------------------------------------------------------
        if (A.saved && A.c_end == F.n_cells) {
            float* sv = A.saved + ((long long)F.n_cells * A.B + pt) * rowlen;
            for (int i = 0; i <= d; ++i) sv[i] = st[i * NT];
        }
        if (A.state_out) {
            float* so = A.state_out + pt * rowlen;
            for (int i = 0; i <= d; ++i) so[i] = st[i * NT];
        }
        if (A.to_out) {
            for (int i = 0; i < d; ++i) store_io(A.out, A.out_dtype, pt * rowlen + i, st[(A.inverse ? i : F.out_perm[i]) * NT]);
            store_io(A.out, A.out_dtype, pt * rowlen + d, st[d * NT]);
        }
    }
    if (!stats) return;
    bn_stats_finalize(F, A, sacc, NT);
}

template <int NT>
__global__ void __launch_bounds__(NT) flow_fwd_generic_kernel(const __grid_constant__ DevFlow F, const FwdArgs A) {
    extern __shared__ __align__(16) float sm[];
    fwd_generic_body<NT>(F, A, sm);
}

// Small batches in train mode (the README example: 2000-point minibatches, 2 cells x 5 BatchNorm layers): the launch
// sequence above is one statistics pass per BN layer plus a final pass per cell - 11 launches of ~9 us each for a few
// microseconds of arithmetic.  When the whole batch is co-resident (one tile per CTA slot) the same passes run inside ONE
// cooperative launch with a grid-wide barrier where the next pass needs the folded statistics (VERDICT r1 item 8).
template <int NT>
__global__ void __launch_bounds__(NT) flow_fwd_coop_kernel(const __grid_constant__ DevFlow F, const FwdArgs A0) {
    extern __shared__ __align__(16) float sm[];
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    const long long rows = A0.B * (F.d + 1);
    FwdArgs A = A0;
    for (int c = 0; c < F.n_cells; ++c) {
        A.c_begin = c; A.c_end = c + 1;
        A.from_state = c > 0;
        A.state_in = c > 0 ? (A0.saved ? A0.saved + (long long)c * rows : A0.scratch_state) : nullptr;
        A.state_out = nullptr; A.to_out = 0;
        for (int l = 0; l <= F.depth; ++l) {
            A.stats_layer = l;
            fwd_generic_body<NT>(F, A, sm);
            grid.sync();                               // the folded scale / shift of layer l (its own 128-byte lines in wpack,
                                                       // not read before in this launch) is visible to every CTA
        }
        const bool last = c == F.n_cells - 1;
        A.stats_layer = -1;
        A.to_out = last;
        A.state_out = A0.saved ? A0.saved + (long long)(c + 1) * rows : (last ? nullptr : A0.scratch_state);
        fwd_generic_body<NT>(F, A, sm);
        // (the next cell's passes read the rows this CTA's threads have just written: no barrier needed)
    }
}

// ---------------------------------------------------------------------------------------------------
// launcher
// ---------------------------------------------------------------------------------------------------
// ---- measurement aid: per-launch device times of nis_flow_forward and nis_flow_inverse (bench.py's roofline object) -----
// nis_flow_timing_begin() arms a per-thread sink; every kernel launch of the following nis_flow_forward / nis_flow_inverse
// calls is then bracketed by CUDA events recorded on the launch stream; nis_flow_timing_end() synchronises those events and
// returns the elapsed time and a tag per launch (0 pack, 1 column moments, 10 + mode for the tensor-core cell kernel: 10
// fused cell, 11 layer pass from the state, 12 final pass from stored activations, 13 layer pass from stored activations;
// 2 other, including the shape-generic kernel and the inverse's input gather).
#define NIS_TIMING_MAX 512
struct TimingSink { bool on; int n; cudaEvent_t ev[NIS_TIMING_MAX + 1]; int tag[NIS_TIMING_MAX]; bool made; };
static thread_local TimingSink g_timing = {false, 0, {}, {}, false};
static inline void timing_mark(cudaStream_t s, int tag) {
    TimingSink& T = g_timing;
    if (!T.on || T.n >= NIS_TIMING_MAX) return;
    if (tag >= 0) T.tag[T.n++] = tag;
    cudaEventRecord(T.ev[T.n], s);         // ev[n] closes launch n-1 and opens launch n
}
extern "C" int nis_flow_timing_begin(void* stream) {
    TimingSink& T = g_timing;
    if (!T.made) {
        for (int i = 0; i <= NIS_TIMING_MAX; ++i) if (cudaEventCreate(&T.ev[i]) != cudaSuccess) return NIS_ECUDA;
        T.made = true;
    }
    T.on = true; T.n = 0;
    cudaEventRecord(T.ev[0], (cudaStream_t)stream);
    return NIS_OK;
}
extern "C" int nis_flow_timing_end(float* ms, int32_t* tags, int32_t max_n) {
    TimingSink& T = g_timing;
    if (!T.on) return NIS_EINVAL;
    T.on = false;
    if (cudaEventSynchronize(T.ev[T.n]) != cudaSuccess) return NIS_ECUDA;
    const int n = T.n < max_n ? T.n : max_n;
    for (int i = 0; i < n; ++i) {
        if (cudaEventElapsedTime(&ms[i], T.ev[i], T.ev[i + 1]) != cudaSuccess) return NIS_ECUDA;
        tags[i] = T.tag[i];
    }
    return n;
}

static size_t fwd_smem_bytes(const DevFlow& F, int NT) {
    const int bw = F.maxW > F.Kpad ? F.maxW : F.Kpad;
    size_t fl = (size_t)((F.d + 1) + 2 * bw) * NT;
    fl += fl & 1;
    return fl * sizeof(float) + sizeof(double) * 2 * F.maxW;
}

// floats of one stored-activation buffer ([tile][width][128], tiles padded to pairs)
static size_t zbuf_floats(const DevFlow& F, int64_t B) { return nis_tiled_zbuf_floats(B) / 64 * (size_t)(F.maxW > 64 ? F.maxW : 64); }

extern "C" size_t nis_flow_workspace_bytes(const NisFlowDesc* desc, int64_t B) {
    DevFlow F;
    if (nis_build_dev_flow(desc, &F) != NIS_OK || B < 0) return 0;
    FlowWorkspace ws;
    size_t fwd = nis_flow_carve(F, B, nullptr, &ws);
    // one workspace serves both BN modes: what the train-mode and the eval-mode plan need.  The backward scratch and the
    // forward's activation buffers are never live together.
    const FlowPlan train = nis_flow_plan(F, B, NIS_BN_TRAIN), eval = nis_flow_plan(F, B, NIS_BN_EVAL);
    size_t tail = nis_flow_bwd_scratch_floats(F, B);
    const size_t zfl = (train.fwd != FWD_GENERIC || eval.fwd != FWD_GENERIC) ? 2 * zbuf_floats(F, B) : 0;
    if (zfl > tail) tail = zfl;
    const size_t tcb = train.bwd == BWD_TC ? nis_bwd_tc_scratch_floats(F, B) : 0;
    if (tcb > tail) tail = tcb;
    // (the wide backward's scratch is also reserved where the tensor-core backward takes the shape first)
    const size_t wdb = (train.bwd != BWD_GENERIC && nis_bwd_wide_supported(F)) ? nis_bwd_wide_scratch_floats(F, B) : 0;
    if (wdb > tail) tail = wdb;
    return fwd + sizeof(float) * tail + 256;
}

template <int NT>
static int launch_fwd(const DevFlow& F, const FwdArgs& A, cudaStream_t s) {
    const size_t smem = fwd_smem_bytes(F, NT);
    NIS_ENSURE_SMEM((flow_fwd_generic_kernel<NT>), (int)smem);
    long long ntiles = (A.B + NT - 1) / NT;
    int grid = (int)(ntiles < NIS_MAX_GRID ? ntiles : NIS_MAX_GRID);
    flow_fwd_generic_kernel<NT><<<grid, NT, smem, s>>>(F, A);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

// Co-residency: every CTA of a cooperative launch must be resident at once.
template <int NT>
static int coop_max_grid(size_t smem) {
    static int cached[16] = {0};
    static size_t cached_smem[16] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 15;
    if (cached[dev] == 0 || cached_smem[dev] != smem) {
        int per_sm = 0;
        NIS_ENSURE_SMEM((flow_fwd_coop_kernel<NT>), (int)smem);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, flow_fwd_coop_kernel<NT>, NT, smem);
        cached[dev] = per_sm > 0 ? per_sm * nis_sm_count() : -1;
        cached_smem[dev] = smem;
    }
    return cached[dev];
}

// the whole train-mode forward in one cooperative launch, or NIS_EUNSUPPORTED when the batch is not co-resident
static int launch_fwd_coop(const DevFlow& F, FwdArgs A, cudaStream_t s) {
    constexpr int NT = 128;
    const size_t smem = fwd_smem_bytes(F, NT);
    if (smem > 200 * 1024) return NIS_EUNSUPPORTED;
    const long long ntiles = (A.B + NT - 1) / NT;
    const int maxg = coop_max_grid<NT>(smem);
    if (maxg <= 0 || ntiles > maxg) return NIS_EUNSUPPORTED;
    void* args[] = {(void*)&F, (void*)&A};
    if (cudaLaunchCooperativeKernel((const void*)flow_fwd_coop_kernel<NT>, dim3((unsigned)ntiles), dim3(NT), args, smem, s) != cudaSuccess) {
        cudaGetLastError();
        return NIS_EUNSUPPORTED;
    }
    return NIS_OK;
}

static int launch_fwd_any(const DevFlow& F, const FwdArgs& A, cudaStream_t s) {
    const size_t lim = 200 * 1024;
    if (fwd_smem_bytes(F, 128) <= lim / 2) return launch_fwd<128>(F, A, s);   // >= 2 CTAs per SM
    if (fwd_smem_bytes(F, 64) <= lim) return launch_fwd<64>(F, A, s);
    if (fwd_smem_bytes(F, 32) <= lim) return launch_fwd<32>(F, A, s);
    return NIS_EUNSUPPORTED;
}

// Activation cache of the streamed-weights path (cfg5-like shapes): a train-mode forward that a backward will follow can
// keep z_1..z_depth of every cell ([cell][layer][tile][W][128] float32) so that the backward does not run the layer passes
// again.  Nonzero only where both the forward and the backward take the wide kernels.
extern "C" int64_t nis_flow_act_saved_count(const NisFlowDesc* desc, int64_t B) {
    DevFlow F;
    if (nis_build_dev_flow(desc, &F) != NIS_OK || B < 0 || !nis_flow_plan(F, B, NIS_BN_TRAIN).act_cache) return 0;
    const size_t tiles = (size_t)((B + 127) / 128);
    return (int64_t)((size_t)F.n_cells * F.depth * tiles * F.widths[0] * 128);
}

// One cell on the fp16-split kernel, forward or inverse (A.inverse).  Train mode: BN_0 and BN_1 from the column moments
// unless the previous cell's final pass has taken them (moments_ready), then a layer pass per remaining BN layer.  With
// depth >= 3 PWLin cells the last layer pass only takes the statistics of z_depth (no 256 B/point store) and the final pass
// starts from z_{depth-1} and runs the last hidden layer again: 7.74 -> 7.29 ms on cfg2 (the PWQuad final pass is bound by
// its spline and loses 1 %).  The final pass reads the state rows from state_in (nullptr: the input rows A.in) and writes
// them to state_out and, with to_out, to A.out; it also takes the column moments of cell `next` (-1: none) when that cell
// has P <= 4, and moments_ready tells the next call whether it did.
static int h_cell(const DevFlow& F, FwdArgs& A, const FlowWorkspace& ws, int bn_mode, int c, int next, const float* state_in,
                  float* state_out, bool to_out, bool& moments_ready, cudaStream_t s) {
    const bool train = bn_mode == NIS_BN_TRAIN;
    const bool moments = train && nis_moments_supported(F, c);
    const bool skip_last = moments && F.depth >= 3 && F.kind == NIS_KIND_PWLIN;
    float* zb[2] = {ws.bwd, ws.bwd + zbuf_floats(F, A.B)};
    A.c_begin = c; A.c_end = c + 1;
    A.from_state = state_in != nullptr; A.state_in = state_in;
    A.state_out = nullptr; A.to_out = 0;
    A.zin_layer = 0; A.next_moments = 0;
    int rc;
    if (train) {
        int l0 = 0;
        if (moments) {
            if (!moments_ready) {
                A.stats_layer = 0;
                rc = nis_launch_col_moments(F, A, s);
                if (rc) return rc;
                timing_mark(s, 1);
            }
            l0 = 2;
        }
        for (int l = l0; l <= F.depth; ++l) {
            A.stats_layer = l;
            if (l >= 1) {
                // layer pass: reads the pre-BN activations of layer l-1, writes those of layer l
                A.zin = (l >= 2 && !(moments && l == 2)) ? zb[(l - 1) & 1] : nullptr;
                A.zout = (skip_last && l == F.depth) ? nullptr : zb[l & 1];
                rc = nis_launch_h(F, A, ws.tcpack, s);
            } else {
                rc = nis_launch_col_stats(F, A, s);
            }
            if (rc) return rc;
            timing_mark(s, l >= 1 ? 10 + 1 + (A.zin ? 2 : 0) : 2);
        }
    }
    A.stats_layer = -1;
    A.zin = (train && !(moments && F.depth == 1)) ? zb[F.depth & 1] : nullptr;
    A.zout = nullptr;
    if (skip_last) { A.zin = zb[(F.depth - 1) & 1]; A.zin_layer = F.depth - 1; }
    A.next_moments = train && next >= 0 && A.zin != nullptr && nis_moments_supported(F, next) && F.cells[next].P <= 4;
    A.next_cell = next;
    moments_ready = A.next_moments != 0;
    A.state_out = state_out; A.to_out = to_out;
    rc = nis_launch_h(F, A, ws.tcpack, s);
    if (rc) return rc;
    timing_mark(s, 10 + (A.zin ? 2 : 0));
    return NIS_OK;
}

// One train-mode cell on the shape-generic kernel, forward or inverse (A.inverse): a statistics pass per BN layer, then the
// final pass.  It reads the state rows from state_in (nullptr: the input rows A.in) and writes them to state_out and, with
// to_out, to A.out.
static int generic_cell(const DevFlow& F, FwdArgs& A, int c, const float* state_in, float* state_out, bool to_out,
                        cudaStream_t s) {
    A.c_begin = c; A.c_end = c + 1;
    A.from_state = state_in != nullptr; A.state_in = state_in;
    A.state_out = nullptr; A.to_out = 0;
    int rc;
    for (int l = 0; l <= F.depth; ++l) {
        A.stats_layer = l;
        rc = launch_fwd_any(F, A, s);
        if (rc) return rc;
        timing_mark(s, 2);
    }
    A.stats_layer = -1;
    A.state_out = state_out; A.to_out = to_out;
    rc = launch_fwd_any(F, A, s);
    if (rc) return rc;
    timing_mark(s, 2);
    return NIS_OK;
}

// Start of nis_flow_forward and nis_flow_inverse: checks the arguments, carves the workspace, zeroes the last-block ticket,
// packs the weights (wpack) and fills the fields of A that both calls set alike.  B == 0 returns NIS_OK with nothing launched.
static int fwd_prologue(const NisFlowDesc* desc, const float* params, const float* bn_running, const void* in, int in_dtype,
                        int in_cols, void* out, int out_dtype, int bn_mode, void* workspace, size_t workspace_bytes, int64_t B,
                        cudaStream_t s, DevFlow& F, FlowWorkspace& ws, FwdArgs& A) {
    int rc = nis_build_dev_flow(desc, &F);
    if (rc) return rc;
    if (!params || !workspace || B < 0 || (B > 0 && (!in || !out))) return NIS_EINVAL;
    if (in_cols != F.d && in_cols != F.d + 1) return NIS_EINVAL;
    if ((in_dtype != NIS_F32 && in_dtype != NIS_F64) || (out_dtype != NIS_F32 && out_dtype != NIS_F64)) return NIS_EINVAL;
    if (bn_mode == NIS_BN_EVAL && !bn_running) return NIS_EINVAL;
    if (workspace_bytes < nis_flow_workspace_bytes(desc, B)) return NIS_EWORKSPACE;
    if (B == 0) return NIS_OK;
    nis_flow_carve(F, B, workspace, &ws);
    cudaMemsetAsync(ws.counter, 0, 256, s);
    timing_mark(s, -1);                     // open the first interval on this stream (after the counter memset)
    rc = launch_flow_pack(F, params, bn_running, nullptr, ws.wpack, bn_mode, s);   // bn_saved: filled by this forward
    if (rc) return rc;
    timing_mark(s, 0);
    A.in = in; A.in_dtype = in_dtype; A.in_cols = in_cols;
    A.out = out; A.out_dtype = out_dtype;
    A.params = params; A.wpack = ws.wpack;
    A.partials = ws.partials; A.counter = ws.counter; A.B = B;
    return NIS_OK;
}

extern "C" int nis_flow_forward(const NisFlowDesc* desc, const float* params, float* bn_running,
                                const void* xj_in, int32_t in_dtype, int32_t in_cols,
                                void* xj_out, int32_t out_dtype, int32_t* bins_out,
                                float* saved, float* bn_saved, int32_t bn_mode,
                                void* workspace, size_t workspace_bytes, int64_t B, void* stream) {
    return nis_flow_forward_cached(desc, params, bn_running, xj_in, in_dtype, in_cols, xj_out, out_dtype, bins_out, saved,
                                   bn_saved, nullptr, bn_mode, workspace, workspace_bytes, B, stream);
}

extern "C" int nis_flow_forward_cached(const NisFlowDesc* desc, const float* params, float* bn_running,
                                       const void* xj_in, int32_t in_dtype, int32_t in_cols,
                                       void* xj_out, int32_t out_dtype, int32_t* bins_out,
                                       float* saved, float* bn_saved, float* act_saved, int32_t bn_mode,
                                       void* workspace, size_t workspace_bytes, int64_t B, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    DevFlow F;
    FlowWorkspace ws;
    FwdArgs A;
    int rc = fwd_prologue(desc, params, bn_running, xj_in, in_dtype, in_cols, xj_out, out_dtype, bn_mode, workspace,
                          workspace_bytes, B, s, F, ws, A);
    if (rc || B == 0) return rc;
    A.saved = saved; A.bins = bins_out; A.bn_running = bn_running; A.bn_saved = bn_saved;
    const long long rows = (long long)B * (F.d + 1);
    const bool train = bn_mode == NIS_BN_TRAIN;
    const FlowPlan plan = nis_flow_plan(F, B, bn_mode);
    if (plan.fwd == FWD_H) {
        rc = nis_h_pack(F, params, ws.tcpack, s);
        if (rc) return rc;
        timing_mark(s, 0);
        bool moments_ready = false;
        for (int c = 0; c < F.n_cells; ++c) {
            const bool last = c == F.n_cells - 1;
            rc = h_cell(F, A, ws, bn_mode, c, last ? -1 : c + 1, c > 0 ? (saved ? saved + c * rows : ws.state) : nullptr,
                        saved ? saved + (c + 1) * rows : (last ? nullptr : ws.state), last, moments_ready, s);
            if (rc) return rc;
        }
        return NIS_OK;
    }
    if (plan.fwd == FWD_GENERIC) {
        if (!train) {
            A.to_out = 1; A.c_begin = 0; A.c_end = F.n_cells; A.stats_layer = -1;
            return launch_fwd_any(F, A, s);
        }
        // small batch: every pass of every cell inside one cooperative launch, else one launch sequence per cell
        A.scratch_state = ws.state;
        A.c_begin = 0; A.c_end = 1; A.stats_layer = 0;
        rc = launch_fwd_coop(F, A, s);
        if (rc == NIS_OK) { timing_mark(s, 2); return NIS_OK; }
        for (int c = 0; c < F.n_cells; ++c) {
            const bool last = c == F.n_cells - 1;
            rc = generic_cell(F, A, c, c > 0 ? (saved ? saved + c * rows : ws.state) : nullptr,
                              saved ? saved + (c + 1) * rows : (last ? nullptr : ws.state), last, s);
            if (rc) return rc;
        }
        return NIS_OK;
    }
    // streamed-weights tcgen05 kernel (flow_wide.cu) or FP32 register-tiled kernel (flow_tiled.cu)
    const bool wide = plan.fwd == FWD_WIDE;
    if (wide) { rc = nis_wide_pack(F, params, ws.tcpack, s); if (rc) return rc; }
    // activation cache (nis_flow_forward_cached): the wide layer passes write z_1..z_depth of every cell there instead of the
    // two rotating workspace buffers
    float* acts = (plan.act_cache && act_saved && saved) ? act_saved : nullptr;
    const size_t act_layer = (size_t)((B + 127) / 128) * (size_t)F.widths[0] * 128;
    // One launch sequence per cell.  TRAIN: the statistics of BN_0 (and BN_1), a layer pass per remaining BN layer, then
    // the final pass.  EVAL: on the wide kernel a layer pass per hidden layer after the first, then the final pass.
    for (int c = 0; c < F.n_cells; ++c) {
        A.c_begin = c; A.c_end = c + 1;
        A.from_state = c > 0;
        A.state_in = c > 0 ? (saved ? saved + (long long)c * rows : ws.state) : nullptr;
        A.state_out = nullptr; A.to_out = 0;
        float* zb[2] = {ws.bwd, ws.bwd + zbuf_floats(F, B)};
        float* const acell = acts ? acts + (size_t)c * F.depth * act_layer : nullptr;
        // BN0 + BN1 from one streaming pass over the pass-through columns (flow_col_moments_kernel), then
        // the layer passes start at layer 2 (recomputing the K=P layer 0 on the way)
        const bool moments = train && nis_moments_supported(F, c);
        if (train) {
            int l0 = 0;
            if (moments) {
                A.stats_layer = 0;
                rc = nis_launch_col_moments(F, A, s);
                if (rc) return rc;
                timing_mark(s, 1);
                l0 = 2;
            }
            for (int l = l0; l <= F.depth; ++l) {
                A.stats_layer = l;
                if (l >= 1) {
                    // layer pass: reads the pre-BN activations of layer l-1, writes those of layer l
                    A.zin = (l >= 2 && !(moments && l == 2)) ? zb[(l - 1) & 1] : nullptr;
                    A.zout = zb[l & 1];
                    if (acell) {
                        if (A.zin) A.zin = acell + (size_t)(l - 2) * act_layer;
                        A.zout = acell + (size_t)(l - 1) * act_layer;
                        A.z1out = (!A.zin && l == 2) ? acell : nullptr;
                    }
                    rc = wide ? nis_launch_wide(F, A, ws.tcpack, s) : nis_launch_tiled(F, A, s);
                } else {
                    rc = nis_launch_col_stats(F, A, s);
                }
                if (rc) return rc;
                timing_mark(s, wide && l >= 1 ? 10 + 1 + (A.zin ? 2 : 0) : 2);
            }
        }
        A.stats_layer = -1;
        A.zin = (train && !(moments && F.depth == 1)) ? zb[F.depth & 1] : nullptr;
        A.zout = nullptr;
        if (acell) { A.zin = acell + (size_t)(F.depth - 1) * act_layer; A.z1out = nullptr; }
        if (wide && !train) {
            // eval, wide conditioner: one launch per hidden layer (no statistics), then the final pass
            A.no_stats = 1;
            for (int l = 2; l <= F.depth; ++l) {
                A.stats_layer = l;
                A.zin = l > 2 ? zb[(l - 1) & 1] : nullptr;
                A.zout = zb[l & 1];
                rc = nis_launch_wide(F, A, ws.tcpack, s);
                if (rc) return rc;
            }
            A.stats_layer = -1; A.no_stats = 0; A.zin = F.depth >= 2 ? zb[F.depth & 1] : nullptr; A.zout = nullptr;
        }
        const bool last = c == F.n_cells - 1;
        A.to_out = last;
        A.state_out = saved ? saved + (long long)(c + 1) * rows : (last ? nullptr : ws.state);
        rc = wide ? nis_launch_wide(F, A, ws.tcpack, s) : nis_launch_tiled(F, A, s);
        if (rc) return rc;
        timing_mark(s, wide ? 10 + (A.zin ? 2 : 0) : 2);
    }
    return NIS_OK;
}

// ---------------------------------------------------------------------------------------------------
// Inverse flow (SURVEY 8 f4): y -> x with the Jacobian column divided by the product of the densities, so that
// nis_flow_inverse(nis_flow_forward(x)) = x with Jacobian 1.  Eval-mode BN uses the running statistics, train-mode BN the
// batch statistics of the pass-through columns each cell sees on the way back (the same values as in the forward pass of
// the same batch); running statistics are not updated.  Width-64 PWLin / PWQuad cells with 32 bins run on the fp16-split
// tensor-core kernel (flow_tc_h.cu, inverse mode bit), every other shape on the shape-generic kernel.
// ---------------------------------------------------------------------------------------------------

// input rows [B][in_cols] in the flow's output column order -> float32 state rows [B][d+1] in the physical order (out_perm
// scatters them back; J = 1 when in_cols = d), so that every inverse cell of the tensor-core path starts from the state
__global__ void __launch_bounds__(256) flow_inverse_gather_kernel(const __grid_constant__ DevFlow F, const void* __restrict__ in,
                                                                  int in_dtype, int in_cols, long long B, float* __restrict__ state) {
    const int d = F.d;
    const long long n = B * (d + 1);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long pt = i / (d + 1);
        const int r = (int)(i - pt * (d + 1));
        const float v = (r < d || in_cols > d) ? load_io(in, in_dtype, pt * in_cols + r) : 1.f;
        state[pt * (d + 1) + (r < d ? F.out_perm[r] : d)] = v;
    }
}

extern "C" int nis_flow_inverse(const NisFlowDesc* desc, const float* params, const float* bn_running,
                                const void* yj_in, int32_t in_dtype, int32_t in_cols,
                                void* xj_out, int32_t out_dtype, int32_t* bins_out, int32_t bn_mode,
                                void* workspace, size_t workspace_bytes, int64_t B, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    DevFlow F;
    FlowWorkspace ws;
    FwdArgs A;
    int rc = fwd_prologue(desc, params, bn_running, yj_in, in_dtype, in_cols, xj_out, out_dtype, bn_mode, workspace,
                          workspace_bytes, B, s, F, ws, A);
    if (rc || B == 0) return rc;
    A.bins = bins_out; A.inverse = 1;
    if (nis_flow_plan(F, B, bn_mode).fwd == FWD_H) {
        // the forward's launch sequence with the cells in reverse order, from float32 state rows in the physical column
        // order.  The statistics and layer passes are the forward's (they read only the pass-through columns); the fused
        // cell and the final pass run the inverse splines; the fused column moments of a final pass are those of cell c - 1.
        rc = nis_h_pack(F, params, ws.tcpack, s);
        if (rc) return rc;
        timing_mark(s, 0);
        const long long nb = (B * (F.d + 1) + 255) / 256;
        flow_inverse_gather_kernel<<<(unsigned)(nb < 4096 ? nb : 4096), 256, 0, s>>>(F, yj_in, in_dtype, in_cols, B, ws.state);
        NIS_CUDA_CHECK_LAUNCH();
        timing_mark(s, 2);
        bool moments_ready = false;
        for (int c = F.n_cells - 1; c >= 0; --c) {
            rc = h_cell(F, A, ws, bn_mode, c, c - 1, ws.state, c == 0 ? nullptr : ws.state, c == 0, moments_ready, s);
            if (rc) return rc;
        }
        return NIS_OK;
    }
    if (bn_mode == NIS_BN_EVAL) {
        A.to_out = 1; A.c_begin = 0; A.c_end = F.n_cells; A.stats_layer = -1;
        rc = launch_fwd_any(F, A, s);
        if (rc == NIS_OK) timing_mark(s, 2);
        return rc;
    }
    for (int c = F.n_cells - 1; c >= 0; --c) {
        rc = generic_cell(F, A, c, c < F.n_cells - 1 ? ws.state : nullptr, c == 0 ? nullptr : ws.state, c == 0, s);
        if (rc) return rc;
    }
    return NIS_OK;
}
