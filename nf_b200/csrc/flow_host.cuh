// Host functions that one flow source file calls in another, and the per-call kernel plan (flow_desc.cu).
#pragma once
#include "common.cuh"

struct FwdArgs;

// ---- which kernel family runs a call: nis_flow_plan (flow_desc.cu) is the only place that decides --------------------
enum FwdPath { FWD_H, FWD_WIDE, FWD_TILED, FWD_GENERIC };   // fp16-split, streamed-weights, register-tiled, shape-generic
enum BwdPath { BWD_TC, BWD_WIDE, BWD_GENERIC };             // tensor-core, wide-conditioner, shape-generic
struct FlowPlan {
    FwdPath fwd;
    BwdPath bwd;           // train mode; eval mode always runs the shape-generic backward
    bool act_cache;        // a train-mode forward keeps z_1 .. z_depth for the wide backward (nis_act_cache_floats)
};
FlowPlan nis_flow_plan(const DevFlow& F, int64_t B, int bn_mode);

// ---- shape predicates of the kernel families (no batch size, no knobs) -------------------------------------------------
bool nis_tc_supported(const DevFlow& F);                  // flow_bwd_tc.cu: fp16-split forward / inverse, tensor-core backward
bool nis_bwd_tc_supported(const DevFlow& F);              // flow_bwd_tc.cu
bool nis_wide_supported(const DevFlow& F, int bn_mode);   // flow_wide.cu
bool nis_bwd_wide_supported(const DevFlow& F);            // flow_bwd_wide.cu
bool nis_tiled_supported(const DevFlow& F);               // flow_tiled.cu
bool nis_moments_supported(const DevFlow& F, int c);      // flow_tiled.cu

// ---- flow_fwd.cu -------------------------------------------------------------------------------------------------------
// torch-layout parameters -> wpack (flow_pack_kernel), and the x-extent of its grid (y: one row of blocks per cell).
// BN scale/shift: eval mode from bn_running; train mode from bn_saved, or none when bn_saved is null.
int nis_pack_blocks(const DevFlow& F);
int launch_flow_pack(const DevFlow& F, const float* params, const float* bn_running, const float* bn_saved, float* wpack,
                     int bn_mode, cudaStream_t s);

// ---- workspace: pack and scratch sizes ---------------------------------------------------------------------------------
size_t nis_tc_pack_floats(const DevFlow& F);              // flow_bwd_tc.cu
size_t nis_wide_pack_floats(const DevFlow& F);            // flow_wide.cu
size_t nis_tiled_zbuf_floats(int64_t B);                  // flow_tiled.cu
size_t nis_flow_bwd_scratch_floats(const DevFlow& F, int64_t B);    // flow_bwd.cu
size_t nis_bwd_tc_scratch_floats(const DevFlow& F, int64_t B);      // flow_bwd_tc.cu
size_t nis_bwd_wide_scratch_floats(const DevFlow& F, int64_t B);    // flow_bwd_wide.cu

// ---- forward launches --------------------------------------------------------------------------------------------------
int nis_h_pack(const DevFlow& F, const float* params, float* tcpack, cudaStream_t s);              // flow_tc_h.cu
int nis_launch_h(const DevFlow& F, const FwdArgs& A, const float* tcpack, cudaStream_t s);
int nis_wide_pack(const DevFlow& F, const float* params, float* widepack, cudaStream_t s);         // flow_wide.cu
int nis_launch_wide(const DevFlow& F, const FwdArgs& A, const float* widepack, cudaStream_t s);
int nis_launch_tiled(const DevFlow& F, const FwdArgs& A, cudaStream_t s);                           // flow_tiled.cu
int nis_launch_col_stats(const DevFlow& F, const FwdArgs& A, cudaStream_t s);
int nis_launch_col_moments(const DevFlow& F, const FwdArgs& A, cudaStream_t s);

// ---- train-mode backwards: launches after nis_flow_backward_cached's counter memset and flow_pack_kernel ---------------
int nis_flow_backward_tc(const DevFlow& F, const FlowWorkspace& ws, const float* params, const float* saved,
                         const float* bn_saved, const void* grad_out, int grad_dtype, float* grad_params, void* grad_in,
                         int64_t B, cudaStream_t s);                                                       // flow_bwd_tc.cu
int nis_flow_backward_wide(const DevFlow& F, const FlowWorkspace& ws, const float* params, const float* saved,
                           const float* bn_saved, const float* act_saved, const void* grad_out, int grad_dtype,
                           float* grad_params, void* grad_in, int64_t B, cudaStream_t s);                  // flow_bwd_wide.cu

// BatchNorm backward of a cell's input normalisation, dL/dx of its pass-through columns (flow_bwd_tc.cu): the last launch of
// a cell in both tensor-core backwards.  dh_in holds dL/dh_0 in 128-point tiles of tile_floats floats.
struct BwdTailArgs {
    const float* saved; float* gstate; const float* dh_in; const float* wpack; const float* bn_saved; const float* bnb;
    void* grad_in; int grad_dtype; long long B; int c, tile_floats;
};
int launch_flow_bwd_tail(const DevFlow& F, const BwdTailArgs& A, cudaStream_t s);
