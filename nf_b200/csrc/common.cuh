// Shared device/host definitions for libnisb200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/nis_b200.h"

#define NIS_CUDA_CHECK_LAUNCH()                          \
    do {                                                 \
        cudaError_t e__ = cudaGetLastError();            \
        if (e__ != cudaSuccess) return NIS_ECUDA;        \
    } while (0)

// Opt a kernel in to `bytes` of dynamic shared memory: cudaFuncSetAttribute once per device and per growth of the
// requirement instead of on every launch (a driver call of a few microseconds each: the latency-bound small-batch
// steps launch ~20 kernels per forward/backward pair, VERDICT r1 item 11).
#define NIS_ENSURE_SMEM(kernel, bytes)                                                                    \
    do {                                                                                                  \
        static int have__[16] = {0};                                                                      \
        int dev__ = 0;                                                                                    \
        cudaGetDevice(&dev__);                                                                            \
        dev__ &= 15;                                                                                      \
        if ((int)(bytes) > have__[dev__]) {                                                               \
            cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes));      \
            have__[dev__] = (int)(bytes);                                                                 \
        }                                                                                                 \
    } while (0)

// Streaming multiprocessors of the current device, queried once per device (148, a B200's count, if the query fails).
static inline int nis_sm_count() {
    static int sms[16] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 15;
    if (sms[dev] <= 0 && (cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms[dev] <= 0))
        sms[dev] = 148;
    return sms[dev];
}

static inline __host__ __device__ int pad8(int x) { return (x + 7) & ~7; }
static inline __host__ __device__ int pad4(int x) { return (x + 3) & ~3; }

// element idx of an external f32 / f64 array (NIS_F32 / NIS_F64): the flow's input and output rows, grad_out and grad_in
__device__ __forceinline__ float load_io(const void* p, int dtype, long long idx) {
    return dtype == NIS_F64 ? (float)reinterpret_cast<const double*>(p)[idx] : reinterpret_cast<const float*>(p)[idx];
}
__device__ __forceinline__ void store_io(void* p, int dtype, long long idx, float v) {
    if (dtype == NIS_F64) reinterpret_cast<double*>(p)[idx] = (double)v; else reinterpret_cast<float*>(p)[idx] = v;
}

// Device-side view of one coupling cell: column tables + offsets into the three float arenas
//   params      (torch layout, read-only)
//   bn_running  (running mean/var)
//   wpack       (per-forward repack: BN scale/shift per layer, transposed zero-padded weights)
struct DevCell {
    int P, T;
    uint8_t feed[NIS_MAX_DIM];
    uint8_t trafo[NIS_MAX_DIM];
    long long param_off, bn_off;
    int pk_off;                         // base of this cell in wpack
    int aff_off[NIS_MAX_HIDDEN + 1];    // scale[Wpad_l] then shift[Wpad_l], relative to pk_off
    int wt_off[NIS_MAX_HIDDEN];         // Wt_l[in_l][Hpad_l]
    int wo_off, bo_off;                 // Wt_o[T][in][Kpad], bias_o[T][Kpad]
    int sv_off;                         // base of this cell in bn_saved
};

struct DevFlow {
    int d, n_cells, kind, nb, depth;
    int K, Kpad;                        // conditioner outputs per transformed dim
    int maxW;                           // max over cells/layers of the padded BN width
    int widths[NIS_MAX_HIDDEN];
    uint8_t out_perm[NIS_MAX_DIM];
    float eps, momentum;
    int pack_total;                     // floats in wpack
    int saved_total;                    // floats in bn_saved
    DevCell cells[NIS_MAX_CELLS];

    __host__ __device__ int W(int c, int l) const { return l == 0 ? cells[c].P : widths[l - 1]; }
    // row of output j of transformed dimension t in the output layer's torch weight: Reshape(T, K) for the spline cells,
    // Reshape(2, T) for the affine cell (coupling_cells.py:46)
    __host__ __device__ int out_row(int c, int t, int j) const { return kind == NIS_KIND_AFFINE ? j * cells[c].T + t : t * K + j; }
    __host__ __device__ int Wp(int c, int l) const { return pad8(W(c, l)); }
    // offsets inside a cell's torch-layout parameter block
    __host__ __device__ long long p_bn_gamma(int c, int l) const {
        long long o = 0;
        int in = cells[c].P;
        if (l == 0) return o;
        o += 2 * in;
        for (int i = 0; i < depth; ++i) {
            o += (long long)widths[i] * in;
            if (i + 1 == l) return o;
            o += 2 * widths[i];
            in = widths[i];
        }
        return -1;
    }
    __host__ __device__ long long p_lin(int c, int l) const {   // hidden layer l weight [H_l][in_l]
        long long o = 2 * cells[c].P;
        int in = cells[c].P;
        for (int i = 0; i < l; ++i) { o += (long long)widths[i] * in + 2 * widths[i]; in = widths[i]; }
        return o;
    }
    __host__ __device__ int in_last(int c) const { return depth == 0 ? cells[c].P : widths[depth - 1]; }
    __host__ __device__ long long p_out_w(int c) const { return p_lin(c, depth); }
    __host__ __device__ long long p_out_b(int c) const {
        return p_out_w(c) + (long long)cells[c].T * K * in_last(c);
    }
    __host__ __device__ long long r_mean(int c, int l) const {  // running mean offset in the cell's bn block
        long long o = 0;
        for (int i = 0; i < l; ++i) o += 2 * W(c, i);
        return o;
    }
};

// Fills a DevFlow from the public descriptor; returns NIS_OK or NIS_EINVAL.
int nis_build_dev_flow(const NisFlowDesc* desc, DevFlow* out);

// workspace carve-up (all offsets 256-byte aligned)
struct FlowWorkspace {
    float* wpack;        // [pack_total]
    float* tcpack;       // tensor-core weight pack (hi/lo splits in UMMA layout): flow_tc_h.cu, flow_wide.cu, flow_bwd_tc.cu
    float* state;        // [B][d+1] scratch state (train mode without `saved`)
    double* partials;    // [max_grid][2][maxW]
    unsigned* counter;   // last-block ticket
    float* bwd;          // backward scratch
    size_t total;
};
size_t nis_flow_carve(const DevFlow& F, int64_t B, void* base, FlowWorkspace* ws);

#define NIS_MAX_GRID 1184   // 148 SMs x 8
