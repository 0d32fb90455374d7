// Fused coupling-cell flow, backward — shape-generic kernel matching flow_fwd.cu.
//
// Reverse sweep over the cells.  For one cell the chain is split into steps
//     OUT   : recompute the conditioner, spline forward + hand-derived spline backward per transformed
//             dimension -> dL/dlogits; dW_out, db_out; dL/da_depth; dL/dx for the transformed columns
//     l>=1  : ReLU + BatchNorm backward of hidden layer l, dW_{l-1}, dL/da_{l-1}
//     0     : BatchNorm backward of the input normalisation -> dL/dx for the pass-through columns
// One thread owns one point (private shared-memory columns, as in the forward); parameter gradients
// are reductions over points and are formed cooperatively per 128/64/32-point tile as small outer
// products accumulated in a per-CTA slice (no atomics, fixed order => deterministic), then summed over
// CTAs.  Eval-mode BN runs all steps in one launch.  Train-mode BN needs the batch means of dL/dy and
// dL/dy * xhat of every BN layer before it can propagate through that layer, so each step is its own
// launch: it leaves dL/da for the next step in a tile-blocked global buffer and accumulates the two
// sums in float64, the last CTA finalising them (and, since they ARE dL/dbeta and dL/dgamma, adding
// them to the parameter gradient).
//
// Autograd semantics reproduced: torch.autograd through coupling_cells.py:107-142,159-228,230-254 as
// the reference's loss.backward() does (manager.py:278); bin indices carry no gradient, the PWQuad
// clamp (:167) passes gradient only to unclamped points.
#include <stdlib.h>
#include <cooperative_groups.h>
#include "common.cuh"
#include "spline.cuh"
#include "flow_host.cuh"

// floats between the BN-backward means of consecutive layers: whole 128-byte lines per layer (a layer's block is rewritten by
// one CTA of the cooperative kernel while the others may hold its neighbours in L1)
__host__ __device__ static inline int bnb_stride(int maxW) { return (2 * maxW + 31) & ~31; }

struct BwdArgs {
    const float* saved;                    // [C+1][B][d+1]
    const void* grad_out; int grad_dtype;  // external upstream gradient (first launch of the last cell)
    void* grad_in;                         // external downstream gradient (last launch of cell 0) or null
    float* gstate;                         // [B][d+1] gradient state, physical column order
    float* dact;                           // [tiles][maxW][NT] dL/da between train-mode launches
    const float* params; const float* wpack; const float* wb;
    float* bnb;                            // [depth+1][bnb_stride]: mean(dh)[maxW], mean(dh*xhat)[maxW] of the current cell
    float* gpart;                          // [grid][cell_params]
    float* grad_params;
    double* partials; unsigned* counter;
    long long B; int c, step_begin, step_end, train, first, cell_params;
    int rotate;                            // activations in three rotating buffers (single-step launches of wide conditioners)
};

// backward weight pack: torch rows padded to 8 so that W^T dz is a dense8 sweep
//   per cell: for l<depth: Wb_l[H_l][pad8(in_l)] ; Wb_o[T][K][pad8(in_last)]
__host__ __device__ static inline int wb_cell_floats(const DevFlow& F, int c) {
    int n = 0, in = F.cells[c].P;
    for (int l = 0; l < F.depth; ++l) { n += F.widths[l] * pad8(in); in = F.widths[l]; }
    return n + F.cells[c].T * F.K * pad8(in);
}
__host__ __device__ static inline int wb_cell_off(const DevFlow& F, int c) {
    int o = 0;
    for (int i = 0; i < c; ++i) o += wb_cell_floats(F, i);
    return o;
}
__host__ __device__ static inline int wb_layer_off(const DevFlow& F, int c, int l) {   // l == depth: output layer
    int n = 0, in = F.cells[c].P;
    for (int i = 0; i < l; ++i) { n += F.widths[i] * pad8(in); in = F.widths[i]; }
    return n;
}

__global__ void flow_bwd_pack_kernel(DevFlow F, const float* __restrict__ params, float* __restrict__ wb) {
    const int c = blockIdx.y;
    const DevCell& q = F.cells[c];
    const float* p = params + q.param_off;
    float* o = wb + wb_cell_off(F, c);
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    int in = q.P;
    for (int l = 0; l <= F.depth; ++l) {
        const int rows = l < F.depth ? F.widths[l] : q.T * F.K;
        const int inp = pad8(in);
        const float* w = p + F.p_lin(c, l);
        float* dst = o + wb_layer_off(F, c, l);
        for (int i = tid; i < rows * inp; i += nth) {
            const int j = i / inp, k = i - j * inp;
            // (output layer: staged per transformed dimension, [t][K][inp], whatever the torch row order is)
            const int src = l < F.depth ? j : F.out_row(c, j / F.K, j % F.K);
            dst[i] = k < in ? w[(long long)src * in + k] : 0.f;
        }
        if (l < F.depth) in = F.widths[l];
    }
}

// out[j] = sum_k act(a[k]) * Wt[k][j], 8 outputs per sweep; RELU applies max(.,0) to the input on read
// (hidden activations are stored as the signed BN output so that xhat stays recoverable for dead units)
template <int NT, bool RELU, typename Epi>
__device__ __forceinline__ void dense8b(const float* __restrict__ Wt, int in, int outp, const float* a_col, Epi epi) {
    for (int jb = 0; jb < outp; jb += 8) {
        float acc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = 0.f;
        const float* wrow = Wt + jb;
#pragma unroll 4
        for (int k = 0; k < in; ++k) {
            const float a = RELU ? fmaxf(a_col[k * NT], 0.f) : a_col[k * NT];
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

// gw[j][k] += sum_i dz[j][i] * a[k][i] over the NT points of the tile (rows complete: caller synced)
template <int NT>
__device__ __forceinline__ void outer_accum(const float* dz, int J, const float* a, int Kn, float* gw, bool relu_a) {
    const int tj = (J + 3) >> 2, tk = (Kn + 3) >> 2;
    for (int tix = threadIdx.x; tix < tj * tk; tix += NT) {
        const int jb = (tix / tk) << 2, kb = (tix % tk) << 2;
        int rj[4], rk[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) { rj[r] = min(jb + r, J - 1) * NT; rk[r] = min(kb + r, Kn - 1) * NT; }
        float acc[4][4];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int s = 0; s < 4; ++s) acc[r][s] = 0.f;
        for (int i = 0; i < NT; ++i) {
            const int col = (i + threadIdx.x) & (NT - 1);
            float dv[4], av[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) { dv[r] = dz[rj[r] + col]; av[r] = a[rk[r] + col]; if (relu_a) av[r] = fmaxf(av[r], 0.f); }
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int s = 0; s < 4; ++s) acc[r][s] = fmaf(dv[r], av[s], acc[r][s]);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int s = 0; s < 4; ++s)
                if (jb + r < J && kb + s < Kn) gw[(size_t)(jb + r) * Kn + kb + s] += acc[r][s];
    }
}

// gv[j] += sum_i buf[j][i]
template <int NT>
__device__ __forceinline__ void rowsum_accum(const float* buf, int J, float* gv) {
    for (int j = threadIdx.x; j < J; j += NT) {
        float s = 0.f;
        for (int i = 0; i < NT; ++i) s += buf[j * NT + ((i + threadIdx.x) & (NT - 1))];
        gv[j] += s;
    }
}

template <int NT>
__device__ __forceinline__ void bwd_generic_body(const DevFlow& F, const BwdArgs& A, float* sm) {
    const int tid = threadIdx.x;
    const int d = F.d, maxW = F.maxW, depth = F.depth, OUT = depth + 1;
    const int c = A.c;
    const DevCell& q = F.cells[c];
    // shared-memory columns (all [rows][NT]); bases without the tid offset are kept for the tile-wide ops
    int rows = 0;
    float* st0 = sm + rows * NT; rows += d + 1;
    float* g0 = sm + rows * NT; rows += d + 1;
    int acto[NIS_MAX_HIDDEN + 1];      // offsets, not pointers: a pointer read back from a local array is generic (LD instead of LDS)
    if (A.rotate) {
        // a launch that runs ONE step touches a_l and a_{l-1} only: layer l lives in buffer l % 3, so the
        // recompute never overwrites the two it still needs
        for (int l = 0; l <= depth; ++l) acto[l] = (rows + (l % 3) * maxW) * NT;
        rows += 3 * maxW;
    } else {
        acto[0] = rows * NT; rows += maxW;                // a_0 (BN0 output), P <= maxW rows used
        for (int l = 1; l <= depth; ++l) { acto[l] = rows * NT; rows += pad8(F.widths[l - 1]); }
    }
    float* lg0 = sm + rows * NT; rows += F.Kpad;
    float* GA0 = sm + rows * NT; rows += maxW;
    float* GB0 = sm + rows * NT; rows += maxW;
    double* sacc = reinterpret_cast<double*>(sm + rows * NT + ((rows * NT) & 1));
    float* st = st0 + tid;
    float* g = g0 + tid;
    float* lg = lg0 + tid;

    const float* pk = A.wpack + q.pk_off;
    const float* prm = A.params + q.param_off;
    const float* wbc = A.wb + wb_cell_off(F, c);
    float* gp = A.gpart + (size_t)blockIdx.x * A.cell_params;
    const bool do_stats = A.train && A.step_end > 0;
    const int stat_l = A.step_end - 1;                     // BN layer whose sums this launch accumulates
    if (do_stats) {
        for (int i = tid; i < 2 * maxW; i += NT) sacc[i] = 0.0;
    }
    __syncthreads();
    const long long ntiles = (A.B + NT - 1) / NT;
    const long long rowlen = d + 1;
    const int fwd_upto = A.step_begin < depth ? A.step_begin : depth;   // activations a_0..a_fwd_upto needed
    const int in_last = F.in_last(c);

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long pt = tile * NT + tid;
        const bool valid = pt < A.B;
        // ---- load state (cell input), gradient state ---------------------------------------------
        float Jout = 1.f;
        if (valid) {
            const float* sv = A.saved + ((long long)c * A.B + pt) * rowlen;
            for (int i = 0; i <= d; ++i) st[i * NT] = sv[i];
            Jout = A.saved[((long long)(c + 1) * A.B + pt) * rowlen + d];
            if (A.step_begin == OUT && A.first) {
                for (int i = 0; i < d; ++i) g[F.out_perm[i] * NT] = load_io(A.grad_out, A.grad_dtype, pt * rowlen + i);
                g[d * NT] = load_io(A.grad_out, A.grad_dtype, pt * rowlen + d);
            } else {
                for (int i = 0; i <= d; ++i) g[i * NT] = A.gstate[pt * rowlen + i];
            }
        } else {
            for (int i = 0; i < d; ++i) { st[i * NT] = 0.5f; g[i * NT] = 0.f; }
            st[d * NT] = 1.f; g[d * NT] = 0.f;
        }
        // ---- recompute the conditioner activations a_0 .. a_fwd_upto -----------------------------
        {
            const float* sc = pk + q.aff_off[0];
            const float* sh = sc + pad8(q.P);
            float* a0 = (sm + acto[0]) + tid;
            for (int k = 0; k < q.P; ++k) a0[k * NT] = fmaf(st[q.feed[k] * NT], sc[k], sh[k]);
            int in = q.P;
            for (int l = 0; l < fwd_upto; ++l) {
                const int H = F.widths[l], Hp = pad8(H);
                const float* scl = pk + q.aff_off[l + 1];
                const float* shl = scl + Hp;
                float* an = (sm + acto[l + 1]) + tid;
                auto epi = [&](int j, float z) { an[j * NT] = fmaf(z, scl[j], shl[j]); };   // signed: ReLU on read
                if (l == 0) dense8b<NT, false>(pk + q.wt_off[l], in, Hp, (sm + acto[l]) + tid, epi);
                else dense8b<NT, true>(pk + q.wt_off[l], in, Hp, (sm + acto[l]) + tid, epi);
                in = H;
            }
        }
        float* GA = GA0 + tid;
        float* GB = GB0 + tid;
        float* GAb = GA0;
        float* GBb = GB0;
        // dL/da entering this launch
        if (A.step_begin != OUT) {
            const int W = F.W(c, A.step_begin);
            const float* src = A.dact + (size_t)tile * maxW * NT + tid;
            for (int j = 0; j < W; ++j) GA[j * NT] = src[(size_t)j * NT];
        }
        for (int step = A.step_begin; step >= A.step_end; --step) {
            if (step == OUT) {
                // ================= output layer + splines =====================================
                const float* ad = (sm + acto[depth]) + tid;
                const int inp = pad8(in_last);
                for (int k = 0; k < in_last; ++k) GA[k * NT] = 0.f;
                const float gJ = g[d * NT];
                const float gJJ = gJ * Jout;
                float Fprod = 1.f;
                for (int t = 0; t < q.T; ++t) {
                    const float* Wt = pk + q.wo_off + (size_t)t * in_last * F.Kpad;
                    const float* bo = pk + q.bo_off + t * F.Kpad;
                    auto epi = [&](int j, float z) { lg[j * NT] = z + bo[j]; };
                    if (depth == 0) dense8b<NT, false>(Wt, in_last, F.Kpad, ad, epi);
                    else dense8b<NT, true>(Wt, in_last, F.Kpad, ad, epi);
                    const int col = q.trafo[t];
                    const float x = st[col * NT];
                    const float gy = g[col * NT];
                    float dx;
                    if (F.kind == NIS_KIND_AFFINE) {
                        // v = s0 x + s1, s0 = 20 e^{Z0}, s1 = relu(Z1); y = (2/pi) atan v; log f = log s0 - log(1 + v^2)
                        const float z1 = lg[NT];
                        const float s0 = 20.f * expf(lg[0]), s1 = fmaxf(z1, 0.f);
                        const float v = fmaf(s0, x, s1);
                        const float iv = 1.f / (v * v + 1.f);
                        const float dv = gy * 0.6366197723675814f * iv - gJJ * 2.f * v * iv;
                        lg[0] = dv * s0 * x + gJJ;
                        lg[NT] = z1 > 0.f ? dv : 0.f;
                        dx = dv * s0;
                        Fprod *= s0 * iv;
                    } else if (F.kind == NIS_KIND_PWLIN) {
                        float f, S, al;
                        int k;
                        const float y = pwlin_fwd(lg, NT, F.nb, x, f, k, S, al);
                        dx = pwlin_bwd(lg, NT, F.nb, k, S, al, y, f, gy, gJJ);
                        Fprod *= f;
                    } else {
                        QuadCtx qc;
                        pwquad_fwd(lg, NT, F.nb, x, qc);
                        dx = pwquad_bwd(lg, NT, F.nb, qc, gy, gJJ / qc.f);
                        Fprod *= qc.f;
                    }
                    g[col * NT] = dx;
                    if (!valid) for (int j = 0; j < F.K; ++j) lg[j * NT] = 0.f;
                    for (int j = F.K; j < F.Kpad; ++j) lg[j * NT] = 0.f;
                    // dL/da_depth += W_o[t]^T dz_t   (Wb_o[t]: [K][inp])
                    dense8b<NT, false>(wbc + wb_layer_off(F, c, depth) + (size_t)t * F.K * inp, F.K, inp, lg,
                                [&](int k, float v) { if (k < in_last) GA[k * NT] += v; });
                    __syncthreads();
                    if (F.kind == NIS_KIND_AFFINE) {           // rows j T + t of the torch weight (Reshape(2, T))
                        for (int j = 0; j < 2; ++j) {
                            outer_accum<NT>(lg0 + j * NT, 1, (sm + acto[depth]), in_last,
                                            gp + F.p_out_w(c) + (size_t)F.out_row(c, t, j) * in_last, depth > 0);
                            rowsum_accum<NT>(lg0 + j * NT, 1, gp + F.p_out_b(c) + F.out_row(c, t, j));
                        }
                    } else {
                        outer_accum<NT>(lg0, F.K, (sm + acto[depth]), in_last, gp + F.p_out_w(c) + (size_t)t * F.K * in_last, depth > 0);
                        rowsum_accum<NT>(lg0, F.K, gp + F.p_out_b(c) + t * F.K);
                    }
                    __syncthreads();
                }
                if (F.kind == NIS_KIND_AFFINE) Fprod *= 0.6366197723675814f;    // 1 / (pi/2), once per cell
                g[d * NT] = gJ * Fprod;
            } else {
                // ================= BatchNorm (+ReLU) backward of layer `step` =================
                const int l = step;
                const int W = F.W(c, l), Wp = F.Wp(c, l);
                const float* sc = pk + q.aff_off[l];
                const float* gam = prm + F.p_bn_gamma(c, l);
                const float* bet = gam + W;
                const float* al = (sm + acto[l]) + tid;
                const float* m1 = A.bnb + l * bnb_stride(maxW);
                const float* m2 = m1 + maxW;
                if (!A.train) {    // eval: dgamma / dbeta are plain sums over points
                    for (int j = 0; j < W; ++j) {
                        const float a = al[j * NT];
                        const bool on = l == 0 || a > 0.f;
                        const float dh = (on && valid) ? GA[j * NT] : 0.f;
                        const float xh = gam[j] != 0.f ? (a - bet[j]) / gam[j] : 0.f;
                        GA[j * NT] = dh;
                        GB[j * NT] = dh * xh;
                    }
                    __syncthreads();
                    rowsum_accum<NT>(GBb, W, gp + F.p_bn_gamma(c, l));
                    rowsum_accum<NT>(GAb, W, gp + F.p_bn_gamma(c, l) + W);
                    __syncthreads();
                    for (int j = 0; j < W; ++j) GA[j * NT] *= sc[j];
                } else {
                    for (int j = 0; j < W; ++j) {
                        const float a = al[j * NT];
                        const bool on = l == 0 || a > 0.f;
                        const float dh = on ? GA[j * NT] : 0.f;
                        const float xh = gam[j] != 0.f ? (a - bet[j]) / gam[j] : 0.f;
                        GA[j * NT] = valid ? sc[j] * (dh - m1[j] - xh * m2[j]) : 0.f;
                    }
                }
                if (l == 0) {
                    for (int k = 0; k < q.P; ++k) g[q.feed[k] * NT] += GA[k * NT];
                } else {
                    // dW_{l-1} += dz_l (x) a_{l-1};  dL/da_{l-1} = W_{l-1}^T dz_l
                    const int in = F.W(c, l - 1), inp = pad8(in);
                    for (int j = W; j < Wp; ++j) GA[j * NT] = 0.f;
                    dense8b<NT, false>(wbc + wb_layer_off(F, c, l - 1), W, inp, GA, [&](int k, float v) { if (k < in) GB[k * NT] = v; });
                    __syncthreads();
                    outer_accum<NT>(GAb, W, (sm + acto[l - 1]), in, gp + F.p_lin(c, l - 1), l - 1 > 0);
                    __syncthreads();
                    float* t_ = GA; GA = GB; GB = t_;
                    t_ = GAb; GAb = GBb; GBb = t_;
                }
            }
        }
        // ---- leave dL/da for the next launch and accumulate its BN sums (train) -------------------
        if (do_stats) {
            const int l = stat_l;
            const int W = F.W(c, l);
            const float* gam = prm + F.p_bn_gamma(c, l);
            const float* bet = gam + W;
            const float* al = (sm + acto[l]) + tid;
            float* dst = A.dact + (size_t)tile * maxW * NT + tid;
            for (int j = 0; j < W; ++j) {
                const float a = al[j * NT];
                const bool on = l == 0 || a > 0.f;
                const float dh = (on && valid) ? GA[j * NT] : 0.f;
                const float xh = gam[j] != 0.f ? (a - bet[j]) / gam[j] : 0.f;
                dst[(size_t)j * NT] = dh;
                GA[j * NT] = dh;
                GB[j * NT] = dh * xh;
            }
            __syncthreads();
            for (int j = tid; j < W; j += NT) {
                double s1 = 0.0, s2 = 0.0;
                for (int i = 0; i < NT; ++i) {
                    const int col = (i + tid) & (NT - 1);
                    s1 += (double)GAb[j * NT + col];
                    s2 += (double)GBb[j * NT + col];
                }
                sacc[j] += s1; sacc[maxW + j] += s2;
            }
            __syncthreads();
        }
        // ---- store the gradient state ------------------------------------------------------------
        if (valid && (A.step_begin == OUT || A.step_end == 0)) {
            if (A.grad_in && A.step_end == 0)
                for (int i = 0; i <= d; ++i) store_io(A.grad_in, A.grad_dtype, pt * rowlen + i, g[i * NT]);
            for (int i = 0; i <= d; ++i) A.gstate[pt * rowlen + i] = g[i * NT];
        }
    }
    if (!do_stats) return;
    // ---- finalise the BN sums of layer stat_l (last CTA) ---------------------------------------------
    __syncthreads();
    double* mine = A.partials + (size_t)blockIdx.x * 2 * maxW;
    for (int i = tid; i < 2 * maxW; i += NT) mine[i] = sacc[i];
    __threadfence();
    __syncthreads();
    __shared__ bool s_last;
    if (tid == 0) s_last = atomicAdd(A.counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int l = stat_l;
    const int W = F.W(c, l);
    float* gg = A.grad_params + q.param_off + F.p_bn_gamma(c, l);
    for (int j = tid; j < W; j += NT) {
        double s1 = 0.0, s2 = 0.0;
        for (unsigned b = 0; b < gridDim.x; ++b) {
            s1 += __ldcg(A.partials + (size_t)b * 2 * maxW + j);
            s2 += __ldcg(A.partials + (size_t)b * 2 * maxW + maxW + j);
        }
        A.bnb[l * bnb_stride(maxW) + j] = (float)(s1 / (double)A.B);
        A.bnb[l * bnb_stride(maxW) + maxW + j] = (float)(s2 / (double)A.B);
        // (read through L2: in the cooperative kernel another CTA may have updated a neighbouring cell's gradients on the
        //  same 128-byte line earlier in the launch)
        gg[j] = __ldcg(gg + j) + (float)s2;          // dL/dgamma
        gg[W + j] = __ldcg(gg + W + j) + (float)s1;  // dL/dbeta
    }
    if (tid == 0) *A.counter = 0u;
}

template <int NT>
__global__ void __launch_bounds__(NT) flow_bwd_generic_kernel(const __grid_constant__ DevFlow F, const BwdArgs A) {
    extern __shared__ __align__(16) float sm[];
    bwd_generic_body<NT>(F, A, sm);
}

// Small batches in train mode: the per-step launches of every cell (output layer, each BatchNorm layer: the next step needs
// the batch means the previous one folds), the zeroing of the per-CTA gradient slices and their reduction run inside ONE
// cooperative launch with grid-wide barriers (README example: 16 launches of ~20 us -> one; VERDICT r1 item 8).
template <int NT>
__global__ void __launch_bounds__(NT) flow_bwd_coop_kernel(const __grid_constant__ DevFlow F, const BwdArgs A0) {
    extern __shared__ __align__(16) float sm[];
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    const int tid = threadIdx.x, OUT = F.depth + 1;
    BwdArgs A = A0;
    for (int c = F.n_cells - 1; c >= 0; --c) {
        const int np = (int)(F.p_out_b(c) + (long long)F.cells[c].T * F.K);
        float* gp = A0.gpart + (size_t)blockIdx.x * np;
        for (int i = tid; i < np; i += NT) gp[i] = 0.f;
        __syncthreads();
        A.c = c; A.cell_params = np; A.first = c == F.n_cells - 1;
        for (int L = OUT; L >= 0; --L) {
            A.step_begin = A.step_end = L;
            A.grad_in = (c == 0 && L == 0) ? A0.grad_in : nullptr;
            bwd_generic_body<NT>(F, A, sm);
            grid.sync();
        }
        // grad_params[cell block] += sum over CTAs of their slices, in CTA order (deterministic)
        float* out = A0.grad_params + F.cells[c].param_off;
        for (int i = blockIdx.x * NT + tid; i < np; i += gridDim.x * NT) {
            float s_ = 0.f;
            for (unsigned b = 0; b < gridDim.x; ++b) s_ += __ldcg(A0.gpart + (size_t)b * np + i);
            out[i] = __ldcg(out + i) + s_;
        }
        grid.sync();                                   // the slices are free for the next cell
    }
}

// grad_params[cell block] += sum over CTAs of their slices (fixed order)
__global__ void bwd_reduce_gpart_kernel(const float* __restrict__ gpart, int grid, int n, float* __restrict__ out) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int b = 0; b < grid; ++b) s += gpart[(size_t)b * n + i];
        out[i] += s;
    }
}

// ---------------------------------------------------------------------------------------------------
static int max_cell_params(const DevFlow& F) {
    int m = 0;
    for (int c = 0; c < F.n_cells; ++c) {
        long long n = F.p_out_b(c) + (long long)F.cells[c].T * F.K;
        if (n > m) m = (int)n;
    }
    return m;
}
static int wb_total(const DevFlow& F) { return wb_cell_off(F, F.n_cells); }

static size_t bwd_smem_bytes(const DevFlow& F, int NT, bool rotate = false) {
    int rows = 2 * (F.d + 1);
    if (rotate) rows += 3 * F.maxW;
    else {
        rows += F.maxW;
        for (int l = 1; l <= F.depth; ++l) rows += pad8(F.widths[l - 1]);
    }
    rows += F.Kpad + 2 * F.maxW;
    size_t fl = (size_t)rows * NT;
    fl += fl & 1;
    return fl * sizeof(float) + sizeof(double) * 2 * F.maxW;
}
// Points per CTA.  Train-mode launches run one step each and may keep the activations in three rotating
// buffers (`rotate`), which is what lets deep/wide conditioners (cfg5: [256]*4, 64 bins) fit.
static int bwd_pick_nt(const DevFlow& F, bool train = false, bool* rotate = nullptr) {
    const size_t lim = 227 * 1024 - 1024;
    if (rotate) *rotate = false;
    if (bwd_smem_bytes(F, 128) <= lim / 2) return 128;
    if (bwd_smem_bytes(F, 64) <= lim) return 64;
    if (bwd_smem_bytes(F, 32) <= lim) return 32;
    if (train && rotate && bwd_smem_bytes(F, 32, true) <= lim) { *rotate = true; return 32; }
    return 0;
}
static int bwd_grid(const DevFlow& F, int64_t B, int NT) {
    long long ntiles = (B + NT - 1) / NT;
    long long cap = (48ll << 20) / (max_cell_params(F) > 0 ? max_cell_params(F) : 1);   // <= 192 MiB of slices
    if (cap > 296) cap = 296;
    if (cap < 16) cap = 16;
    return (int)(ntiles < cap ? (ntiles > 0 ? ntiles : 1) : cap);
}

struct BwdScratch { float *wb, *gstate, *dact, *bnb, *gpart; size_t floats; };
static void bwd_carve(const DevFlow& F, int64_t B, float* base, BwdScratch* s) {
    auto up = [](size_t x) { return (x + 63) & ~(size_t)63; };
    size_t off = 0;
    s->wb = base + off; off = up(off + wb_total(F));
    s->gstate = base + off; off = up(off + (size_t)B * (F.d + 1));
    s->dact = base + off; off = up(off + (size_t)((B + 127) / 128) * 128 * F.maxW);
    s->bnb = base + off; off = up(off + (size_t)(F.depth + 1) * bnb_stride(F.maxW));
    s->gpart = base + off;
    bool rot = false;
    int NT = bwd_pick_nt(F, true, &rot);
    off = up(off + (size_t)(NT ? bwd_grid(F, B, NT) : 0) * max_cell_params(F));
    s->floats = off;
}

size_t nis_flow_bwd_scratch_floats(const DevFlow& F, int64_t B) {
    BwdScratch s;
    bwd_carve(F, B, nullptr, &s);
    return s.floats;
}

template <int NT>
static int launch_bwd(const DevFlow& F, const BwdArgs& A, int grid, cudaStream_t s) {
    const size_t smem = bwd_smem_bytes(F, NT, A.rotate != 0);
    NIS_ENSURE_SMEM((flow_bwd_generic_kernel<NT>), (int)smem);
    flow_bwd_generic_kernel<NT><<<grid, NT, smem, s>>>(F, A);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

static int launch_bwd_any(const DevFlow& F, const BwdArgs& A, int NT, int grid, cudaStream_t s) {
    switch (NT) {
        case 128: return launch_bwd<128>(F, A, grid, s);
        case 64: return launch_bwd<64>(F, A, grid, s);
        case 32: return launch_bwd<32>(F, A, grid, s);
    }
    return NIS_EUNSUPPORTED;
}

// Shape-generic backward, train or eval mode: one launch per step of each cell (train), one per cell (eval), or the whole
// backward in one cooperative launch.
static int nis_flow_backward_generic(const DevFlow& F, const FlowWorkspace& ws, const float* params, const float* saved,
                                     int bn_mode, const void* grad_out, int grad_dtype, float* grad_params, void* grad_in,
                                     int64_t B, cudaStream_t s) {
    const int train = bn_mode == NIS_BN_TRAIN;
    bool rotate = false;
    const int NT = bwd_pick_nt(F, train != 0, &rotate);
    BwdScratch sc;
    bwd_carve(F, B, ws.bwd, &sc);
    const int grid = bwd_grid(F, B, NT);
    flow_bwd_pack_kernel<<<dim3(nis_pack_blocks(F), F.n_cells), 256, 0, s>>>(F, params, sc.wb);
    NIS_CUDA_CHECK_LAUNCH();
    BwdArgs A;
    A.saved = saved; A.grad_out = grad_out; A.grad_dtype = grad_dtype;
    A.gstate = sc.gstate; A.dact = sc.dact; A.params = params; A.wpack = ws.wpack; A.wb = sc.wb;
    A.bnb = sc.bnb; A.gpart = sc.gpart; A.grad_params = grad_params;
    A.partials = ws.partials; A.counter = ws.counter; A.B = B; A.train = train; A.rotate = rotate;
    const int OUT = F.depth + 1;
    int rc;
    if (train && NT == 128 && !rotate) {
        // small batch: the whole backward in one cooperative launch when every tile has its own resident CTA
        const long long ntiles = (B + NT - 1) / NT;
        const size_t smem = bwd_smem_bytes(F, 128, false);
        static int maxg[16] = {0};
        int dev = 0;
        cudaGetDevice(&dev);
        dev &= 15;
        if (maxg[dev] == 0) {
            int per_sm = 0;
            NIS_ENSURE_SMEM((flow_bwd_coop_kernel<128>), (int)smem);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, flow_bwd_coop_kernel<128>, 128, smem);
            maxg[dev] = per_sm > 0 ? per_sm * nis_sm_count() : -1;
        }
        if (ntiles == grid && ntiles <= maxg[dev]) {
            NIS_ENSURE_SMEM((flow_bwd_coop_kernel<128>), (int)smem);
            A.grad_in = grad_in; A.c = 0; A.cell_params = 0; A.first = 1; A.step_begin = A.step_end = OUT;
            void* args[] = {(void*)&F, (void*)&A};
            if (cudaLaunchCooperativeKernel((const void*)flow_bwd_coop_kernel<128>, dim3((unsigned)grid), dim3(128), args, smem, s) == cudaSuccess)
                return NIS_OK;
            cudaGetLastError();
        }
    }
    for (int c = F.n_cells - 1; c >= 0; --c) {
        const int np = (int)(F.p_out_b(c) + (long long)F.cells[c].T * F.K);
        cudaMemsetAsync(sc.gpart, 0, sizeof(float) * (size_t)grid * np, s);
        A.c = c; A.cell_params = np; A.first = c == F.n_cells - 1;
        if (!train) {
            A.step_begin = OUT; A.step_end = 0; A.grad_in = c == 0 ? grad_in : nullptr;
            rc = launch_bwd_any(F, A, NT, grid, s);
            if (rc) return rc;
        } else {
            for (int L = OUT; L >= 0; --L) {
                A.step_begin = A.step_end = L;
                A.grad_in = (c == 0 && L == 0) ? grad_in : nullptr;
                rc = launch_bwd_any(F, A, NT, grid, s);
                if (rc) return rc;
            }
        }
        int rb = (np + 255) / 256;
        if (rb > 592) rb = 592;
        bwd_reduce_gpart_kernel<<<rb, 256, 0, s>>>(sc.gpart, grid, np, grad_params + F.cells[c].param_off);
        NIS_CUDA_CHECK_LAUNCH();
    }
    return NIS_OK;
}

extern "C" int nis_flow_backward(const NisFlowDesc* desc, const float* params, const float* bn_running,
                                 const float* saved, const float* bn_saved, const void* grad_out,
                                 int32_t grad_dtype, float* grad_params, void* grad_in, int32_t bn_mode,
                                 void* workspace, size_t workspace_bytes, int64_t B, void* stream) {
    return nis_flow_backward_cached(desc, params, bn_running, saved, bn_saved, nullptr, grad_out, grad_dtype, grad_params,
                                    grad_in, bn_mode, workspace, workspace_bytes, B, stream);
}

// Checks the arguments and everything that can refuse the call before any launch, then zeroes the last-block ticket and packs
// the weights and this batch's BN scale/shift (wpack) for whichever backward nis_flow_plan picks.
extern "C" int nis_flow_backward_cached(const NisFlowDesc* desc, const float* params, const float* bn_running,
                                        const float* saved, const float* bn_saved, const float* act_saved,
                                        const void* grad_out, int32_t grad_dtype, float* grad_params, void* grad_in,
                                        int32_t bn_mode, void* workspace, size_t workspace_bytes, int64_t B, void* stream) {
    DevFlow F;
    int rc = nis_build_dev_flow(desc, &F);
    if (rc) return rc;
    if (!params || !saved || !grad_out || !grad_params || !workspace || B < 0) return NIS_EINVAL;
    if (grad_dtype != NIS_F32 && grad_dtype != NIS_F64) return NIS_EINVAL;
    const int train = bn_mode == NIS_BN_TRAIN;
    if (train && !bn_saved) return NIS_EINVAL;
    if (!train && !bn_running) return NIS_EINVAL;
    if (workspace_bytes < nis_flow_workspace_bytes(desc, B)) return NIS_EWORKSPACE;
    if (B == 0) return NIS_OK;
    cudaStream_t s = (cudaStream_t)stream;
    FlowWorkspace ws;
    nis_flow_carve(F, B, workspace, &ws);
    const FlowPlan plan = nis_flow_plan(F, B, bn_mode);
    bool rotate;
    if (plan.bwd == BWD_GENERIC && !bwd_pick_nt(F, train != 0, &rotate)) return NIS_EUNSUPPORTED;
    cudaMemsetAsync(ws.counter, 0, 256, s);
    rc = launch_flow_pack(F, params, bn_running, bn_saved, ws.wpack, bn_mode, s);
    if (rc) return rc;
    if (plan.bwd == BWD_TC)
        return nis_flow_backward_tc(F, ws, params, saved, bn_saved, grad_out, grad_dtype, grad_params, grad_in, B, s);
    if (plan.bwd == BWD_WIDE)
        return nis_flow_backward_wide(F, ws, params, saved, bn_saved, plan.act_cache ? act_saved : nullptr, grad_out,
                                      grad_dtype, grad_params, grad_in, B, s);
    return nis_flow_backward_generic(F, ws, params, saved, bn_mode, grad_out, grad_dtype, grad_params, grad_in, B, s);
}
