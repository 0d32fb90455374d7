// Fused coupling-cell forward, register-tiled FP32 path for width-64 conditioners (BASELINE cfg2).
//
// One launch = one coupling cell over the whole batch (or one train-mode statistics pass of it).
// Persistent CTAs (one per SM) loop over tiles of M points.  The cell's weights are staged ONCE per CTA
// into shared memory (k-major, 64-wide rows); a tile's activations live in shared memory as [feature][M]
// so that every conditioner layer is an (M x in) x (in x 64) product computed with a 4x8 (points x
// outputs) register tile per thread: per k-step one 128-bit LDS of activations + two 128-bit LDS of
// weights feed 32 FFMA (the FP32 pipe is the roofline of this path, SURVEY.md §8d).  The output layer is
// produced 64 logits at a time (two transformed dimensions of 32 bins), each followed in place by the
// per-bin softmax, CDF, bin lookup and Jacobian factor, so logits never leave shared memory.
//
// Reference semantics: coupling_cells.py:107-142 (PWLin) with the conditioner of :84-104.
#include <stdlib.h>
#include "common.cuh"
#include "spline.cuh"
#include "flow_fwd_common.cuh"
#include "flow_host.cuh"

#define TH 64            // hidden width handled by this path
#define TCH 64           // logits per output-layer chunk

struct TiledSmem {
    int st, A0, A1, W, aff, bias, fbuf, total;   // float offsets
    int wl[NIS_MAX_HIDDEN + 1];                  // per-layer weight offsets inside W (last = output layer)
};

// Shared-memory plan of one launch: hidden layers [first, last) are computed, plus the output layer
// when with_out.  Layer passes of the train path need one activation buffer and one layer of weights
// (~50 KB at M=128), which lets two CTAs share an SM and overlap one's global traffic with the other's FMAs.
__host__ __device__ static inline TiledSmem tiled_layout(const DevFlow& F, int c, int M, int first, int last, bool with_out) {
    TiledSmem s;
    const DevCell& q = F.cells[c];
    int o = 0;
    s.st = o; o += (F.d + 1) * M;
    s.A0 = o; o += TH * M;
    s.A1 = o;
    if (with_out || last - first >= 2) o += TH * M;
    s.W = o;
    int w = 0, in = q.P;
    for (int l = 0; l < F.depth; ++l) {
        s.wl[l] = w;
        if (l >= first && l < last) w += in * TH;
        in = TH;
    }
    const int nch = (q.T * F.K + TCH - 1) / TCH;
    s.wl[F.depth] = w;
    if (with_out) w += nch * TH * TCH;
    o += w;
    s.aff = o; o += (F.depth + 1) * 2 * TH;
    s.bias = o; o += nch * TCH;
    s.fbuf = o; o += (TCH / F.K) * M;
    if (o < s.A0 + 2 * (M / 4) * TH * 2 + 4 * F.maxW + 2) o = s.A0 + 2 * (M / 4) * TH * 2 + 4 * F.maxW + 2;   // statistics fold scratch
    s.total = o;
    return s;
}

// Activation rows are XOR-swizzled at 4-float granularity so that both the k-major GEMM reads and the
// epilogue's 128-bit stores of one output row per lane are bank-conflict free.
template <int M>
__device__ __forceinline__ int swz(int row, int pt) { return row * M + ((((pt >> 2) ^ ((row >> 2) & 7)) << 2) | (pt & 3)); }

// 4x8 register tiles (16 warps/SM) measured faster than 8x8 (8 warps/SM) on B200: 26.0 vs 29.0 ms for cfg2 eval at 2^22 points
constexpr int TM = 4;

template <int M>
__global__ void __launch_bounds__(M * 8 / TM, M == 128 ? 2 : 1) flow_cell_tiled_kernel(const __grid_constant__ DevFlow F, const FwdArgs A) {
    constexpr int NT = M * 8 / TM;
    constexpr int NV = TM / 4;            // float4 per thread row
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x;
    const int c = A.c_begin;
    const DevCell& q = F.cells[c];
    const int d = F.d, depth = F.depth, K = F.K, nb = F.nb;
    const float* pk = A.wpack + q.pk_off;
    const int tpc = TCH / K;                                  // transformed dims per chunk
    const int nch = (q.T * K + TCH - 1) / TCH;
    const bool stats = A.stats_layer >= 1;
    const int last_layer = stats ? A.stats_layer : depth;     // hidden layers to run (1-based count)
    // Train-mode layer passes: with A.zin the activations below `first_layer` are not recomputed; the
    // pre-BN output of hidden layer first_layer-1 is read back (tile-blocked [tile][64][M]) and BN+ReLU
    // of that layer is applied while it is staged into shared memory.
    const int first_layer = A.zin ? last_layer - (stats ? 1 : 0) : 0;
    const TiledSmem L = tiled_layout(F, c, M, first_layer, last_layer, !stats);
    float* st = sm + L.st;
    float* Ws = sm + L.W;
    float* affs = sm + L.aff;
    float* biass = sm + L.bias;
    float* fbuf = sm + L.fbuf;

    // ---- stage the cell's weights / BN scale+shift / bias once ---------------------------------------
    {
        int in = q.P;
        for (int l = 0; l < last_layer; ++l) {
            const float* src = pk + q.wt_off[l];               // [in][64]
            if (l >= first_layer)
                for (int i = tid; i < in * TH; i += NT) Ws[L.wl[l] + i] = src[i];
            in = TH;
        }
        for (int l = 0; l <= depth; ++l) {
            const int W = l == 0 ? q.P : TH, Wp = pad8(W);
            const float* src = pk + q.aff_off[l];
            for (int i = tid; i < W; i += NT) { affs[l * 2 * TH + i] = src[i]; affs[l * 2 * TH + TH + i] = src[Wp + i]; }
        }
        if (!stats) {
            // output layer: per-t [in][Kpad] in wpack -> chunked [chunk][k][64]
            for (int i = tid; i < nch * TH * TCH; i += NT) {
                const int ch = i / (TH * TCH), r = i - ch * TH * TCH, k = r / TCH, j = r - k * TCH;
                const int t = ch * tpc + j / K, jj = j % K;
                Ws[L.wl[depth] + i] = t < q.T ? pk[q.wo_off + ((size_t)t * TH + k) * F.Kpad + jj] : 0.f;
            }
            for (int i = tid; i < nch * TCH; i += NT) {
                const int t = i / K, jj = i % K;
                biass[i] = t < q.T ? pk[q.bo_off + t * F.Kpad + jj] : 0.f;
            }
        }
    }
    const int tc = tid & 7, tr = tid >> 3;                     // thread column (outputs), row (points)
    double dsum[8], dsq[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { dsum[j] = 0.0; dsq[j] = 0.0; }
    __syncthreads();

    const long long ntiles = (A.B + M - 1) / M;
    const long long rowlen = d + 1;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long base = tile * M;
        const int cnt = (int)((A.B - base) < M ? (A.B - base) : M);
        // ---- state tile -> shared memory, transposed to [col][M] ------------------------------------
        if (A.from_state) {
            const float* src = A.state_in + base * rowlen;
            for (int i = tid; i < M * (d + 1); i += NT) {
                const int pt = i / (d + 1), col = i - pt * (d + 1);
                st[col * M + pt] = pt < cnt ? src[i] : (col == d ? 1.f : 0.5f);
            }
        } else {
            for (int i = tid; i < M * (d + 1); i += NT) {
                const int pt = i / (d + 1), col = i - pt * (d + 1);
                float v = col == d ? 1.f : 0.5f;
                if (pt < cnt && col < A.in_cols) v = load_io(A.in, A.in_dtype, (base + pt) * A.in_cols + col);
                st[col * M + pt] = v;
            }
        }
        __syncthreads();
        if (!stats && A.saved && !A.from_state) {
            float* sv = A.saved + ((long long)c * A.B + base) * rowlen;
            for (int i = tid; i < cnt * (d + 1); i += NT) { const int pt = i / (d + 1), col = i - pt * (d + 1); sv[i] = st[col * M + pt]; }
        }
        // ---- input activations: BN0 of the pass-through columns, or BN+ReLU of the stored layer ------
        float* cur = sm + L.A0;
        float* nxt = sm + L.A1;
        if (first_layer == 0) {
            for (int i = tid; i < q.P * M; i += NT) {
                const int k = i / M, pt = i - k * M;
                cur[swz<M>(k, pt)] = fmaf(st[q.feed[k] * M + pt], affs[k], affs[TH + k]);
            }
        } else {
            const float4* src = reinterpret_cast<const float4*>(A.zin + (size_t)tile * TH * M);
            const float* sc = affs + first_layer * 2 * TH;
            const float* sh = sc + TH;
            for (int i = tid; i < TH * M / 4; i += NT) {
                const int k = i / (M / 4), pt = (i - k * (M / 4)) * 4;
                float4 v = src[i];
                v.x = fmaxf(fmaf(v.x, sc[k], sh[k]), 0.f); v.y = fmaxf(fmaf(v.y, sc[k], sh[k]), 0.f);
                v.z = fmaxf(fmaf(v.z, sc[k], sh[k]), 0.f); v.w = fmaxf(fmaf(v.w, sc[k], sh[k]), 0.f);
                *reinterpret_cast<float4*>(cur + swz<M>(k, pt)) = v;
            }
        }
        __syncthreads();
        // ---- hidden layers ---------------------------------------------------------------------------
        int in = first_layer == 0 ? q.P : TH;
        for (int l = first_layer; l < last_layer; ++l) {
            float acc[TM][8];
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
            const float* wp = Ws + L.wl[l] + tc * 4;
#pragma unroll 4
            for (int k = 0; k < in; ++k) {
                float av[TM];
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    const float4 a = *reinterpret_cast<const float4*>(cur + swz<M>(k, tr * TM + 4 * v));
                    av[4 * v] = a.x; av[4 * v + 1] = a.y; av[4 * v + 2] = a.z; av[4 * v + 3] = a.w;
                }
                const float4 w0 = *reinterpret_cast<const float4*>(wp + k * TH);
                const float4 w1 = *reinterpret_cast<const float4*>(wp + k * TH + 32);
                const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                for (int i = 0; i < TM; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
            }
            if (stats && l + 1 == A.stats_layer) {
                // per-feature sums of the pre-BN activations of this tile (points beyond the batch masked)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float s = 0.f, s2 = 0.f;
#pragma unroll
                    for (int i = 0; i < TM; ++i) {
                        const float v = (tr * TM + i) < cnt ? acc[i][j] : 0.f;
                        s += v; s2 = fmaf(v, v, s2);
                    }
                    dsum[j] += (double)s; dsq[j] += (double)s2;
                }
                if (A.zout) {      // leave the pre-BN activations for the next layer pass (whole tile, valid or not)
                    float* dst = A.zout + (size_t)tile * TH * M;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int o = (j < 4 ? 0 : 28) + tc * 4 + j;
#pragma unroll
                        for (int v4 = 0; v4 < NV; ++v4)
                            *reinterpret_cast<float4*>(dst + o * M + tr * TM + 4 * v4) =
                                make_float4(acc[4 * v4][j], acc[4 * v4 + 1][j], acc[4 * v4 + 2][j], acc[4 * v4 + 3][j]);
                    }
                }
                break;
            }
            const float* sc = affs + (l + 1) * 2 * TH;
            const float* sh = sc + TH;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int o = (j < 4 ? 0 : 28) + tc * 4 + j;
#pragma unroll
                for (int v4 = 0; v4 < NV; ++v4) {
                    float4 v;
                    v.x = fmaxf(fmaf(acc[4 * v4][j], sc[o], sh[o]), 0.f);
                    v.y = fmaxf(fmaf(acc[4 * v4 + 1][j], sc[o], sh[o]), 0.f);
                    v.z = fmaxf(fmaf(acc[4 * v4 + 2][j], sc[o], sh[o]), 0.f);
                    v.w = fmaxf(fmaf(acc[4 * v4 + 3][j], sc[o], sh[o]), 0.f);
                    *reinterpret_cast<float4*>(nxt + swz<M>(o, tr * TM + 4 * v4)) = v;
                }
            }
            __syncthreads();
            float* t_ = cur; cur = nxt; nxt = t_;
            in = TH;
        }
        if (stats) { __syncthreads(); continue; }
        // ---- output layer in chunks of 64 logits, spline in place ------------------------------------
        for (int ch = 0; ch < nch; ++ch) {
            float acc[TM][8];
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
            const float* wp = Ws + L.wl[depth] + ch * TH * TCH + tc * 4;
#pragma unroll 4
            for (int k = 0; k < TH; ++k) {
                float av[TM];
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    const float4 a = *reinterpret_cast<const float4*>(cur + swz<M>(k, tr * TM + 4 * v));
                    av[4 * v] = a.x; av[4 * v + 1] = a.y; av[4 * v + 2] = a.z; av[4 * v + 3] = a.w;
                }
                const float4 w0 = *reinterpret_cast<const float4*>(wp + k * TCH);
                const float4 w1 = *reinterpret_cast<const float4*>(wp + k * TCH + 32);
                const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                for (int i = 0; i < TM; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int o = (j < 4 ? 0 : 28) + tc * 4 + j;
                const float b = biass[ch * TCH + o];
#pragma unroll
                for (int v4 = 0; v4 < NV; ++v4) {
                    float4 v;
                    v.x = acc[4 * v4][j] + b; v.y = acc[4 * v4 + 1][j] + b; v.z = acc[4 * v4 + 2][j] + b; v.w = acc[4 * v4 + 3][j] + b;
                    *reinterpret_cast<float4*>(nxt + swz<M>(o, tr * TM + 4 * v4)) = v;
                }
            }
            __syncthreads();
            for (int pair = tid; pair < tpc * M; pair += NT) {
                const int tt = pair / M, pt = pair - tt * M;
                const int t = ch * tpc + tt;
                if (t < q.T) {
                    const int col = q.trafo[t];
                    const float x = st[col * M + pt];
                    float f, S, al;
                    int k;
                    const int r0 = tt * K;
                    auto zacc = [&](int j) -> float& { return nxt[swz<M>(r0 + j, pt)]; };
                    const float y = pwlin_fwd_z(zacc, nb, x, f, k, S, al);
                    st[col * M + pt] = y;
                    fbuf[tt * M + pt] = f;
                    if (A.bins && pt < cnt) A.bins[((long long)c * A.B + base + pt) * d + t] = k;
                } else {
                    fbuf[tt * M + pt] = 1.f;
                }
            }
            __syncthreads();
            for (int pt = tid; pt < M; pt += NT) {
                float f = 1.f;
                for (int tt = 0; tt < tpc; ++tt) f *= fbuf[tt * M + pt];
                st[d * M + pt] *= f;
            }
        }
        __syncthreads();
        // ---- store the tile ---------------------------------------------------------------------------
        if (A.state_out) {
            float* dst = A.state_out + base * rowlen;
            for (int i = tid; i < cnt * (d + 1); i += NT) { const int pt = i / (d + 1), col = i - pt * (d + 1); dst[i] = st[col * M + pt]; }
        }
        if (A.to_out) {
            for (int i = tid; i < cnt * (d + 1); i += NT) {
                const int pt = i / (d + 1), col = i - pt * (d + 1);
                const int src = col == d ? d : F.out_perm[col];
                store_io(A.out, A.out_dtype, base * rowlen + i, st[src * M + pt]);
            }
        }
        __syncthreads();
    }
    if (!stats) return;
    // ---- statistics pass: fold rows -> per-feature sums, then the shared finalisation -----------------
    double* red = reinterpret_cast<double*>(sm + L.A0 + (L.A0 & 1));   // [2][M/TM rows][64]  (A0/A1 are free now)
    double* sacc = red + 2 * (M / TM) * TH;                    // [2*maxW]
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int o = (j < 4 ? 0 : 28) + tc * 4 + j;
        red[tr * TH + o] = dsum[j];
        red[(M / TM) * TH + tr * TH + o] = dsq[j];
    }
    __syncthreads();
    for (int o = tid; o < 2 * F.maxW; o += NT) sacc[o] = 0.0;
    __syncthreads();
    if (tid < TH) {
        double s = 0.0, s2 = 0.0;
        for (int r = 0; r < M / TM; ++r) { s += red[r * TH + tid]; s2 += red[(M / TM) * TH + r * TH + tid]; }
        sacc[tid] = s; sacc[F.maxW + tid] = s2;
    }
    bn_stats_finalize(F, A, sacc, NT);
}

// ---------------------------------------------------------------------------------------------------
// Batch statistics of the pass-through columns (BN layer 0 of a cell) straight from the state rows: a
// streaming reduction (the shape-generic statistics pass stages whole tiles through shared memory and
// costs 10x the HBM time of this read).
__global__ void __launch_bounds__(256) flow_col_stats_kernel(const __grid_constant__ DevFlow F, const FwdArgs A) {
    __shared__ double red[8][2][NIS_MAX_DIM];
    __shared__ double sacc_s[2 * NIS_MAX_WIDTH];
    const int c = A.c_begin;
    const DevCell& q = F.cells[c];
    const int d = F.d, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double s[NIS_MAX_DIM], s2[NIS_MAX_DIM];
#pragma unroll
    for (int k = 0; k < NIS_MAX_DIM; ++k) { s[k] = 0.0; s2[k] = 0.0; }
    for (long long pt = (long long)blockIdx.x * 256 + tid; pt < A.B; pt += (long long)gridDim.x * 256) {
#pragma unroll
        for (int k = 0; k < NIS_MAX_DIM; ++k) {
            if (k < q.P) {
                const int col = q.feed[k];
                const float x = A.from_state ? A.state_in[pt * (d + 1) + col] : load_io(A.in, A.in_dtype, pt * A.in_cols + col);
                s[k] += (double)x; s2[k] += (double)x * (double)x;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < NIS_MAX_DIM; ++k) {
        if (k < q.P) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { s[k] += __shfl_xor_sync(0xffffffffu, s[k], o); s2[k] += __shfl_xor_sync(0xffffffffu, s2[k], o); }
            if (lane == 0) { red[warp][0][k] = s[k]; red[warp][1][k] = s2[k]; }
        }
    }
    for (int i = tid; i < 2 * F.maxW; i += 256) sacc_s[i] = 0.0;
    __syncthreads();
    if (tid < q.P) {
        double a = 0.0, b = 0.0;
        for (int w = 0; w < 8; ++w) { a += red[w][0][tid]; b += red[w][1][tid]; }
        sacc_s[tid] = a; sacc_s[F.maxW + tid] = b;
    }
    bn_stats_finalize(F, A, sacc_s, 256);
}

// ---------------------------------------------------------------------------------------------------
// BN layers 0 AND 1 of a cell from the first and second moments of its pass-through columns.
// z1 = W0 * a0 with a0 = BN0(x) is linear in x, so its batch mean and variance follow from mean(x) and
// Cov(x):  mean(z1_j) = sum_k W0[j][k] beta0_k ,  var(z1_j) = w~_j^T Cov(x) w~_j  with
// w~_jk = W0[j][k] gamma0_k / sqrt(var_k + eps)  — evaluated in float64.  This replaces two passes over
// the batch (the BN0 statistics pass and the layer-1 statistics pass with its 256 B/point store) by one
// streaming read of P columns.  Used when P <= 8.
// ---------------------------------------------------------------------------------------------------
#define MOM_PMAX 8
// PM = compile-time bound on the pass-through width (4: 14 sums, the bench shapes; 8: 44 sums)
template <int MOM_P>
__global__ void __launch_bounds__(256, MOM_P <= 4 ? 4 : 2) flow_col_moments_kernel(const __grid_constant__ DevFlow F, const FwdArgs A) {
    constexpr int MOM_N = MOM_P + MOM_P * (MOM_P + 1) / 2;
    __shared__ double red[8][MOM_N];
    __shared__ double tot[MOM_N];
    __shared__ double fold_s[(256 / (MOM_N <= 16 ? 16 : 64)) * MOM_N];
    __shared__ double sc0s[MOM_P + MOM_P * MOM_P];
    __shared__ bool s_last;
    const int c = A.c_begin;
    const DevCell& q = F.cells[c];
    const int d = F.d, P = q.P, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // Per-thread partial sums in float32 (a thread sees B / (grid * 256) ~ 30 points of magnitude <= 1: 3e-7 relative, averaged
    // down over the ~150 000 threads), everything across threads in float64.  (Round 1 kept 44 float64 accumulators per
    // thread: 88 registers, two blocks per SM, 1.7 TB/s.)
    float acc[MOM_N];
#pragma unroll
    for (int i = 0; i < MOM_N; ++i) acc[i] = 0.f;
    constexpr int MOM_U = 4;
    const long long stride = (long long)gridDim.x * 256;
    for (long long pt0 = (long long)blockIdx.x * 256 + tid; pt0 < A.B; pt0 += MOM_U * stride) {
        float x[MOM_U][MOM_P];
#pragma unroll
        for (int u = 0; u < MOM_U; ++u) {
            const long long pt = pt0 + u * stride;
#pragma unroll
            for (int k = 0; k < MOM_P; ++k)
                x[u][k] = (k < P && pt < A.B) ? (A.from_state ? A.state_in[pt * (d + 1) + q.feed[k]]
                                                              : load_io(A.in, A.in_dtype, pt * A.in_cols + q.feed[k])) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < MOM_U; ++u) {
            int o = MOM_P;
#pragma unroll
            for (int k = 0; k < MOM_P; ++k) {
                acc[k] += x[u][k];
#pragma unroll
                for (int k2 = k; k2 < MOM_P; ++k2) { acc[o] = fmaf(x[u][k], x[u][k2], acc[o]); ++o; }
            }
        }
    }
#pragma unroll
    for (int i = 0; i < MOM_N; ++i) {
        double a = (double)acc[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if (lane == 0) red[warp][i] = a;
    }
    __syncthreads();
    double* mine = A.partials + (size_t)blockIdx.x * MOM_N;
    if (tid < MOM_N) {
        double s_ = 0.0;
        for (int w = 0; w < 8; ++w) s_ += red[w][tid];
        mine[tid] = s_;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(A.counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    fold_partials<MOM_N>(A.partials, gridDim.x, fold_s, tot, tid, 256);
    moments_finalize<MOM_P>(F, A, c, tot, sc0s, tid, 256);
    if (tid == 0) *A.counter = 0u;
}

bool nis_moments_supported(const DevFlow& F, int c) { return F.depth >= 1 && F.cells[c].P <= MOM_PMAX; }

int nis_launch_col_moments(const DevFlow& F, const FwdArgs& A, cudaStream_t s) {
    long long blocks = (A.B + 255) / 256;
    int grid = (int)(blocks < 592 ? blocks : 592);
    if (F.cells[A.c_begin].P <= 4) flow_col_moments_kernel<4><<<grid, 256, 0, s>>>(F, A);
    else flow_col_moments_kernel<8><<<grid, 256, 0, s>>>(F, A);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

int nis_launch_col_stats(const DevFlow& F, const FwdArgs& A, cudaStream_t s) {
    long long blocks = (A.B + 255) / 256;
    int grid = (int)(blocks < 592 ? blocks : 592);
    flow_col_stats_kernel<<<grid, 256, 0, s>>>(F, A);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

size_t nis_tiled_zbuf_floats(int64_t B) { return (size_t)((B + 255) / 256) * 256 * TH; }

bool nis_tiled_supported(const DevFlow& F) {
    if (F.kind != NIS_KIND_PWLIN || F.depth < 1) return false;
    for (int l = 0; l < F.depth; ++l) if (F.widths[l] != TH) return false;
    if (F.K != 8 && F.K != 16 && F.K != 32 && F.K != 64) return false;
    if (F.maxW != TH) return false;
    for (int c = 0; c < F.n_cells; ++c) {
        TiledSmem s = tiled_layout(F, c, 128, 0, F.depth, true);
        if ((size_t)s.total * 4 > 220 * 1024) return false;
    }
    return true;
}

template <int M>
static int launch_tiled_m(const DevFlow& F, const FwdArgs& A, int sms, cudaStream_t s) {
    const bool stats = A.stats_layer >= 1;
    const int last = stats ? A.stats_layer : F.depth;
    const int first = A.zin ? last - (stats ? 1 : 0) : 0;
    TiledSmem L = tiled_layout(F, A.c_begin, M, first, last, !stats);
    const size_t smem = (size_t)L.total * sizeof(float);
    NIS_ENSURE_SMEM((flow_cell_tiled_kernel<M>), (int)smem);
    long long ntiles = (A.B + M - 1) / M;
    const int per_sm = (M == 128 && smem <= 110 * 1024) ? 2 : 1;
    int grid = (int)(ntiles < (long long)sms * per_sm ? ntiles : (long long)sms * per_sm);
    flow_cell_tiled_kernel<M><<<grid, M * 8 / TM, smem, s>>>(F, A);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

int nis_launch_tiled(const DevFlow& F, const FwdArgs& A, cudaStream_t s) {
    const int sms = nis_sm_count();
    // train-mode layer passes exchange tile-blocked activations: every launch of a forward must use the
    // same M; they run at M=128 with two CTAs per SM.  The fused eval cell runs at M=256.
    const bool layer_pass = A.zin || A.zout;
    TiledSmem L256 = tiled_layout(F, A.c_begin, 256, 0, F.depth, true);
    if (!layer_pass && (size_t)L256.total * 4 <= 225 * 1024 && A.B >= (long long)sms * 256) return launch_tiled_m<256>(F, A, sms, s);
    return launch_tiled_m<128>(F, A, sms, s);
}
