// Pieces shared by the forward kernels (flow_fwd.cu: shape-generic; flow_tiled.cu: register-tiled).
#pragma once
#include "common.cuh"

struct FwdArgs {
    const void* in; int in_dtype; int in_cols;   // external input rows (first cell, !from_state)
    const float* state_in;                       // fp32 [B][d+1] (from_state)
    float* state_out;                            // fp32 [B][d+1] or null
    void* out; int out_dtype;                    // external output (to_out)
    int from_state, to_out;
    float* saved;                                // [n_cells+1][B][d+1] or null
    int32_t* bins;
    const float* params; float* wpack; float* bn_running; float* bn_saved;
    double* partials; unsigned* counter;
    long long B; int c_begin, c_end, stats_layer;
    const float* zin;                            // tiled train path: pre-BN activations of the layer below,
    float* zout;                                 // tile-blocked [tile][64][M] (written by a statistics pass)
    int no_stats;                                // layer pass that only stores its activations (eval-mode split cell)
    float* z1out;                          // wide kernel, pass from the state: also store z_1 (backward recompute) or null
    float* scratch_state;                  // cooperative small-batch kernel: fp32 [B][d+1] state between cells when `saved` is null
    int zin_layer;                         // fp16-split kernel: which layer's pre-activations `zin` holds (0: the default,
                                           // stats_layer - 1 for a layer pass, depth for the final pass)
    int next_moments;                      // fp16-split final pass: also accumulate the column moments of cell next_cell (its
                                           // BN_0 / BN_1 statistics) from the state this pass writes - no pass of their own
    int next_cell;                         // the cell that runs after c_begin: c_begin + 1, or c_begin - 1 in the inverse
    int inverse;                           // nis_flow_inverse: cells backwards, inverse splines, J divided (shape-generic
                                           // kernel; fp16-split fused cell and final pass)
};


__device__ __forceinline__ float load_io(const void* p, int dtype, long long idx) {
    return dtype == NIS_F64 ? (float)reinterpret_cast<const double*>(p)[idx] : reinterpret_cast<const float*>(p)[idx];
}
__device__ __forceinline__ void store_io(void* p, int dtype, long long idx, float v) {
    if (dtype == NIS_F64) reinterpret_cast<double*>(p)[idx] = (double)v; else reinterpret_cast<float*>(p)[idx] = v;
}


// Train-mode BN statistics: every CTA of a statistics pass hands in its float64 per-feature sums
// (sacc[0..maxW) = sum z, sacc[maxW..2maxW) = sum z^2, in shared memory); the last CTA to arrive adds
// the per-CTA partials in index order (deterministic) and folds them into the layer's scale/shift
// (wpack), the saved batch statistics (backward) and the running statistics (torch BatchNorm1d
// semantics: biased variance for normalisation, unbiased for the running estimate, momentum 0.1).
// `scratch` (optional, 2 * NT doubles of shared memory): the last CTA then adds the per-CTA partials with all its threads
// (NT / Wp slices per feature, combined in slice order - still a fixed order) instead of one thread per feature walking
// all gridDim.x partials: 148 x 2 dependent-latency loads per feature were ~25 us at the tail of every statistics pass.
__device__ __forceinline__ void bn_stats_finalize(const DevFlow& F, const FwdArgs& A, const double* sacc, int NT,
                                                  double* scratch = nullptr) {
    const int tid = threadIdx.x;
    const int maxW = F.maxW;
    __syncthreads();
    const int c = A.c_begin, l = A.stats_layer;
    const DevCell& q = F.cells[c];
    const int W = F.W(c, l), Wp = F.Wp(c, l);
    double* mine = A.partials + (size_t)blockIdx.x * 2 * maxW;
    for (int i = tid; i < 2 * maxW; i += NT) mine[i] = sacc[i];
    __threadfence();
    __syncthreads();
    __shared__ bool s_last;
    if (tid == 0) s_last = atomicAdd(A.counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const float* p = A.params + q.param_off + F.p_bn_gamma(c, l);
    float* aff = A.wpack + q.pk_off + q.aff_off[l];
    const int slices = scratch ? NT / Wp : 0;
    if (slices > 1) {
        const int sl = tid / Wp, j = tid - sl * Wp;
        if (sl < slices) {
            double s = 0.0, s2 = 0.0;
            for (unsigned b = sl; b < gridDim.x; b += slices) {
                s += __ldcg(A.partials + (size_t)b * 2 * maxW + j);
                s2 += __ldcg(A.partials + (size_t)b * 2 * maxW + maxW + j);
            }
            scratch[sl * Wp + j] = s;
            scratch[NT + sl * Wp + j] = s2;
        }
        __syncthreads();
    }
    for (int j = tid; j < Wp; j += NT) {
        float sc = 0.f, sh = 0.f;
        if (j < W) {
            double s = 0.0, s2 = 0.0;
            if (slices > 1) {
                for (int sl = 0; sl < slices; ++sl) { s += scratch[sl * Wp + j]; s2 += scratch[NT + sl * Wp + j]; }
            } else {
                for (unsigned b = 0; b < gridDim.x; ++b) {
                    s += __ldcg(A.partials + (size_t)b * 2 * maxW + j);
                    s2 += __ldcg(A.partials + (size_t)b * 2 * maxW + maxW + j);
                }
            }
            const double n = (double)A.B;
            const double mean = s / n;
            double var = s2 / n - mean * mean;
            var = var > 0.0 ? var : 0.0;
            const double invstd = 1.0 / sqrt(var + (double)F.eps);
            sc = (float)((double)p[j] * invstd);
            sh = (float)((double)p[W + j] - mean * (double)p[j] * invstd);
            if (A.bn_saved) {
                A.bn_saved[q.sv_off + l * 2 * maxW + j] = (float)mean;
                A.bn_saved[q.sv_off + l * 2 * maxW + maxW + j] = (float)invstd;
            }
            if (A.bn_running) {
                float* rs = A.bn_running + q.bn_off + F.r_mean(c, l);
                const double m = (double)F.momentum;
                const double unb = A.B > 1 ? var * n / (n - 1.0) : var;
                rs[j] = (float)((1.0 - m) * (double)rs[j] + m * mean);
                rs[W + j] = (float)((1.0 - m) * (double)rs[W + j] + m * unb);
            }
        }
        aff[j] = sc;
        aff[Wp + j] = sh;
    }
    if (tid == 0) *A.counter = 0u;
}


// Sum of per-CTA partials [nblk][N] (global memory, written by the other CTAs before their counter arrival) into tot[N]
// (shared), by all NT threads of the last CTA in a fixed order: slices of the CTA list are summed side by side and then
// combined in slice order.  (N threads walking all nblk partials one dependent L2 latency after the other was a 20-40 us
// tail on every launch.)  scratch: (NT / W) * N doubles of shared memory, W = 16 for N <= 16, else 64.
template <int N>
__device__ __forceinline__ void fold_partials(const double* partials, unsigned nblk, double* scratch, double* tot, int tid, int NT) {
    constexpr int W = N <= 16 ? 16 : 64;
    const int slices = NT / W, sl = tid / W, i = tid - sl * W;
    if (i < N && sl < slices) {
        double s_ = 0.0;
        for (unsigned b = sl; b < nblk; b += slices) s_ += __ldcg(partials + (size_t)b * N + i);
        scratch[sl * N + i] = s_;
    }
    __syncthreads();
    if (tid < N) {
        double s_ = 0.0;
        for (int k = 0; k < slices; ++k) s_ += scratch[k * N + tid];
        tot[tid] = s_;
    }
    __syncthreads();
}

// BN_0 and BN_1 of cell c from the first and second moments of its pass-through columns (tot[0..P) = sum x_k,
// tot[s2i(k, k2)] = sum x_k x_k2 over the batch, in shared memory): BN_0 is per column; layer 0 is linear in BN_0's
// output, so the batch mean and variance of each of its outputs follow from the covariance matrix - no pass over z_1.
// Writes scale / shift (wpack), the saved batch statistics (backward) and the running statistics.  Called by every
// thread of the last CTA (NT threads) after a __syncthreads(); sc0s: MOM_P + MOM_P^2 doubles of shared scratch.
template <int MOM_P>
__device__ __forceinline__ void moments_finalize(const DevFlow& F, const FwdArgs& A, int c, const double* tot, double* sc0s,
                                                 int tid, int NT) {
    const DevCell& q = F.cells[c];
    const int P = q.P;
    const double n = (double)A.B, mom = (double)F.momentum, unb = A.B > 1 ? n / (n - 1.0) : 1.0;
    const float* prm = A.params + q.param_off;
    float* pk = A.wpack + q.pk_off;
    const int maxW = F.maxW;
    // index of S2[k][k2], k <= k2, in the packed upper triangle
    auto s2i = [](int k, int k2) { return MOM_P + k * MOM_P - k * (k - 1) / 2 + (k2 - k); };
    // ---- BN0 -------------------------------------------------------------------------------------------
    if (tid < pad8(P)) {
        float sc = 0.f, sh = 0.f;
        if (tid < P) {
            const double mean = tot[tid] / n;
            double var = tot[s2i(tid, tid)] / n - mean * mean;
            var = var > 0.0 ? var : 0.0;
            const double invstd = 1.0 / sqrt(var + (double)F.eps);
            const double g = (double)prm[tid], b = (double)prm[P + tid];
            sc = (float)(g * invstd);
            sh = (float)(b - mean * g * invstd);
            sc0s[tid] = g * invstd;
            if (A.bn_saved) { A.bn_saved[q.sv_off + tid] = (float)mean; A.bn_saved[q.sv_off + maxW + tid] = (float)invstd; }
            if (A.bn_running) {
                float* rs = A.bn_running + q.bn_off + F.r_mean(c, 0);
                rs[tid] = (float)((1.0 - mom) * (double)rs[tid] + mom * mean);
                rs[P + tid] = (float)((1.0 - mom) * (double)rs[P + tid] + mom * var * unb);
            }
        }
        pk[q.aff_off[0] + tid] = sc;
        pk[q.aff_off[0] + pad8(P) + tid] = sh;
    }
    __syncthreads();
    // covariance of BN_0's outputs (without the shift), once: sc_k sc_k2 (E[x_k x_k2] - E[x_k] E[x_k2])
    double* covs = sc0s + MOM_P;                                    // [P][P]
    for (int i = tid; i < P * P; i += NT) {
        const int k = i / P, k2 = i - k * P;
        covs[i] = sc0s[k] * sc0s[k2] * (tot[k <= k2 ? s2i(k, k2) : s2i(k2, k)] / n - (tot[k] / n) * (tot[k2] / n));
    }
    __syncthreads();
    // ---- BN1 from the moments ------------------------------------------------------------------------------
    const int H = F.widths[0], Hp = pad8(H);
    const float* W0 = prm + F.p_lin(c, 0);                 // [H][P]
    const float* g1 = prm + F.p_bn_gamma(c, 1);
    for (int j = tid; j < Hp; j += NT) {
        float sc = 0.f, sh = 0.f;
        if (j < H) {
            double mean1 = 0.0, var1 = 0.0;
            for (int k = 0; k < P; ++k) {
                const double wk = (double)W0[j * P + k];
                mean1 += wk * (double)prm[P + k];
                for (int k2 = 0; k2 < P; ++k2) var1 += wk * (double)W0[j * P + k2] * covs[k * P + k2];
            }
            var1 = var1 > 0.0 ? var1 : 0.0;
            const double invstd = 1.0 / sqrt(var1 + (double)F.eps);
            sc = (float)((double)g1[j] * invstd);
            sh = (float)((double)g1[H + j] - mean1 * (double)g1[j] * invstd);
            if (A.bn_saved) {
                A.bn_saved[q.sv_off + 2 * maxW + j] = (float)mean1;
                A.bn_saved[q.sv_off + 2 * maxW + maxW + j] = (float)invstd;
            }
            if (A.bn_running) {
                float* rs = A.bn_running + q.bn_off + F.r_mean(c, 1);
                rs[j] = (float)((1.0 - mom) * (double)rs[j] + mom * mean1);
                rs[H + j] = (float)((1.0 - mom) * (double)rs[H + j] + mom * var1 * unb);
            }
        }
        pk[q.aff_off[1] + j] = sc;
        pk[q.aff_off[1] + Hp + j] = sh;
    }
}
