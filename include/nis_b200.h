/*
 * nis_b200.h — C ABI of libnisb200.so: the B200 (sm_100a) kernels under the NIS hot path of NGoetz/NF.
 *
 * The reference (`nisrep`, pure Python/PyTorch) has no FFI; its boundary is the Python class surface
 * (SURVEY.md §8b).  Each entry point below replaces the body of one reference method and is what a
 * binding from that method would call (see INTEGRATION.md for the ctypes stub):
 *
 *   nis_flow_forward      <- torch.nn.Sequential.__call__ over AddJacobian/PWLin/PWQuad/RectNN/
 *                            RollLayer/MaskLayer/DeMaskLayer
 *                            (nisrep/normalizing_flows/layers/coupling_cells.py:107-142,159-228,230-254;
 *                             layers/layers.py:27-32,43-51,75-77,90-91; called at manager.py:174,225,341,397)
 *   nis_flow_backward     <- loss.backward() through the same modules (manager.py:278)
 *   nis_reduce_moments    <- torch.var / torch.mean of f*J (manager.py:255,399-400)
 *   nis_reduce_stats      <- the same plus torch.max / torch.min and a non-finite count
 *                            (nisrep/utils/experiment_mg.py:73-76,101)
 *   nis_rambo_generate    <- FlatInvertiblePhasespace.generateKinematics_batch, pdf inactive and pdf active
 *                            (nisrep/PhaseSpace/flat_phase_space_generator.py:81-137, 139-308, 313-441;
 *                             PhaseSpace/utils.py:5-146, 151-187)
 *   nis_rambo_invert      <- (no reference body: README.md:68-69 "inverse phase space" to do) the inverse of the map above
 *   nis_uniform_fill      <- torch.nn.init.uniform_(w) (manager.py:222,395)
 *
 * Conventions: plain pointers and sizes only; every pointer is DEVICE memory owned by the caller
 * unless marked host; work is enqueued on `stream` and the call returns without synchronising; no
 * allocation; re-entrant.  Process-wide state is limited to caches of launch attributes (the dynamic
 * shared-memory opt-in per kernel and device, the SM count) and to environment variables that select a
 * kernel family for tests and A/B measurements (NIS_TC, NIS_DISABLE_TILED, NIS_BWD_TC - INTEGRATION.md section 7;
 * read on every call, unset in production); the measurement aid nis_flow_timing_* keeps a per-thread
 * event list.  Return value: 0 on success, a negative NIS_E* code otherwise (nis_strerror() gives
 * text).  `stream` is a cudaStream_t passed as void*.
 */
#ifndef NIS_B200_H
#define NIS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NIS_MAX_DIM 32     /* max n_flow */
#define NIS_MAX_CELLS 32   /* max coupling cells */
#define NIS_MAX_HIDDEN 8   /* max hidden layers of the conditioner */
#define NIS_MAX_WIDTH 512  /* max hidden width */
#define NIS_MAX_FINAL 8    /* max final-state particles of the phase-space generator */

enum { NIS_KIND_PWLIN = 0, NIS_KIND_PWQUAD = 1,
       NIS_KIND_AFFINE = 2 /* AffineCoupling (layers/coupling_cells.py:6-70): two conditioner outputs per transformed
                              dimension in Reshape(2, T) row order; n_bins is ignored; shape-generic kernels only */ };
enum { NIS_F32 = 0, NIS_F64 = 1 };
enum { NIS_BN_EVAL = 0, NIS_BN_TRAIN = 1 };

enum {
    NIS_OK = 0,
    NIS_EINVAL = -1,     /* bad descriptor / argument */
    NIS_EWORKSPACE = -2, /* workspace too small */
    NIS_ECUDA = -3,      /* CUDA launch error (cudaGetLastError) */
    NIS_EUNSUPPORTED = -4
};

/* One coupling cell.  Roll / Mask / DeMask layers are folded into column tables over a state whose
 * columns never move (layers.py:27-32,43-51,90-91): the cell conditions on physical columns
 * feed_idx[0..n_pass) and transforms physical columns trafo_idx[0..n_flow-n_pass), in the order the
 * reference cell sees them. */
typedef struct NisCellDesc {
    int32_t n_pass;
    int32_t feed_idx[NIS_MAX_DIM];
    int32_t trafo_idx[NIS_MAX_DIM];
    int64_t param_off; /* float offset of this cell's parameter block in `params` */
    int64_t bn_off;    /* float offset of this cell's running-statistics block in `bn_running` */
} NisCellDesc;

/* Parameter block of a cell (float32, torch-native layouts, same order as the reference state_dict
 * "{cell}.NN.{idx}.*", SURVEY.md §5):
 *   bn0.weight[P] bn0.bias[P]
 *   for l in 0..depth-1:  lin_l.weight[H_l][in_l]  bn_{l+1}.weight[H_l]  bn_{l+1}.bias[H_l]
 *   out.weight[OUT][H_last]  out.bias[OUT]            OUT = T*n_bins (PWLIN) or T*(2*n_bins+1) (PWQUAD)
 * Running-statistics block: for l in 0..depth: running_mean[W_l] running_var[W_l], W_0=P, W_l=H_{l-1}. */
typedef struct NisFlowDesc {
    int32_t n_flow;
    int32_t n_cells;
    int32_t kind;   /* NIS_KIND_* */
    int32_t n_bins;
    int32_t depth;  /* hidden layers */
    int32_t widths[NIS_MAX_HIDDEN];
    int32_t out_perm[NIS_MAX_DIM]; /* reference's final column i = physical column out_perm[i] */
    float bn_eps;
    float bn_momentum;
    NisCellDesc cells[NIS_MAX_CELLS];
} NisFlowDesc;

/* floats in one cell's parameter / running-stat block (host helpers, no CUDA) */
int64_t nis_flow_cell_param_count(const NisFlowDesc* desc, int32_t cell);
int64_t nis_flow_cell_bn_count(const NisFlowDesc* desc, int32_t cell);
/* floats in the saved-batch-statistics buffer written by a TRAIN forward and read by backward */
int64_t nis_flow_bn_saved_count(const NisFlowDesc* desc);
/* bytes of scratch needed by forward / backward for a batch of B points */
size_t nis_flow_workspace_bytes(const NisFlowDesc* desc, int64_t B);

/* Forward of the whole flow: xj_out[B, n_flow+1] = flow(xj_in), last column = accumulated Jacobian.
 *   params      float32 parameter pack (see above)
 *   bn_running  float32 running statistics; read in EVAL mode, updated in TRAIN mode (may be NULL in
 *               TRAIN mode to skip the update)
 *   xj_in       [B, in_cols] row-major, in_cols = n_flow (J=1 implied) or n_flow+1; dtype in_dtype
 *   xj_out      [B, n_flow+1] row-major, dtype out_dtype, reference column order
 *   bins_out    optional int32 [n_cells, B, n_flow]: bin index of transformed dim t of cell c at
 *               [c, i, t] (entries t >= T_c are left untouched)
 *   saved       optional float32 [n_cells+1, B, n_flow+1]: state before each cell and after the last
 *               (physical column order); required by nis_flow_backward
 *   bn_saved    optional float32 [nis_flow_bn_saved_count]: batch mean / inverse std of every BN layer
 *               (TRAIN mode); required by nis_flow_backward in TRAIN mode
 */
int nis_flow_forward(const NisFlowDesc* desc, const float* params, float* bn_running,
                     const void* xj_in, int32_t in_dtype, int32_t in_cols,
                     void* xj_out, int32_t out_dtype, int32_t* bins_out,
                     float* saved, float* bn_saved, int32_t bn_mode,
                     void* workspace, size_t workspace_bytes, int64_t B, void* stream);

/* Activation cache for training (round 2).  Where both the forward and the backward of a shape run the streamed-weights
 * tcgen05 kernels (wide conditioners such as BASELINE configs[4]: [256]*4), the backward needs the pre-BatchNorm
 * activations z_1..z_depth of every cell.  nis_flow_forward_cached writes them to act_saved
 * (float32 [nis_flow_act_saved_count(desc, B)], layout [cell][layer][tile][width][128]) and nis_flow_backward_cached reads
 * them instead of running the layer passes again (what torch.autograd does for the reference's loss.backward(),
 * manager.py:278: it keeps every intermediate of the forward).  nis_flow_act_saved_count returns 0 for shapes / batch sizes
 * that have no use for the cache; act_saved == NULL (or the plain entry points) keeps the recomputing backward (its z is
 * rebuilt from the saved float32 batch statistics: the two gradients agree to float32 rounding, tested at 1e-5 of the
 * gradient scale). */
int64_t nis_flow_act_saved_count(const NisFlowDesc* desc, int64_t B);
int nis_flow_forward_cached(const NisFlowDesc* desc, const float* params, float* bn_running,
                            const void* xj_in, int32_t in_dtype, int32_t in_cols,
                            void* xj_out, int32_t out_dtype, int32_t* bins_out,
                            float* saved, float* bn_saved, float* act_saved, int32_t bn_mode,
                            void* workspace, size_t workspace_bytes, int64_t B, void* stream);
int nis_flow_backward_cached(const NisFlowDesc* desc, const float* params, const float* bn_running,
                             const float* saved, const float* bn_saved, const float* act_saved,
                             const void* grad_out, int32_t grad_dtype,
                             float* grad_params, void* grad_in, int32_t bn_mode,
                             void* workspace, size_t workspace_bytes, int64_t B, void* stream);

/* Inverse flow (SURVEY 8 f4; the reference lists it as to do, README.md:68-69): yj_in [B, n_flow(+1)] in the flow's OUTPUT
 * column order -> xj_out [B, n_flow+1] with column n_flow = J_in / prod of the densities, so that
 * nis_flow_inverse(nis_flow_forward(x)) == x with Jacobian 1 (away from PWQuad's clamp at 1 - 1e-6).  EVAL: running
 * statistics; TRAIN: batch statistics of what each cell sees on the way back (running statistics are not updated).
 * Width-64 PWLin / PWQuad flows with 32 bins (the shapes the fp16-split forward serves) run on the tensor-core kernel, every
 * other shape on the shape-generic FP32 kernels; bins_out as in nis_flow_forward. */
int nis_flow_inverse(const NisFlowDesc* desc, const float* params, const float* bn_running,
                     const void* yj_in, int32_t in_dtype, int32_t in_cols,
                     void* xj_out, int32_t out_dtype, int32_t* bins_out, int32_t bn_mode,
                     void* workspace, size_t workspace_bytes, int64_t B, void* stream);

/* Backward: given dL/d(xj_out) computes dL/d(params) (accumulated into grad_params, which the caller
 * zeroes when it wants a fresh gradient) and optionally dL/d(xj_in).
 *   bn_running  running statistics (EVAL mode; may be NULL in TRAIN mode)
 *   saved / bn_saved  as written by the matching nis_flow_forward
 *   grad_out    [B, n_flow+1] dtype grad_dtype, reference column order
 *   grad_in     optional [B, n_flow+1] same dtype (column n_flow = dL/dJ_in)
 */
int nis_flow_backward(const NisFlowDesc* desc, const float* params, const float* bn_running,
                      const float* saved, const float* bn_saved, const void* grad_out, int32_t grad_dtype,
                      float* grad_params, void* grad_in, int32_t bn_mode,
                      void* workspace, size_t workspace_bytes, int64_t B, void* stream);

/* out[0..3) = { sum v, sum v^2, n } in float64 over v[0..n) (dtype NIS_F32/NIS_F64), accumulated onto
 * the existing contents of `out` when accumulate != 0.  Deterministic (fixed reduction order).
 * workspace: at least nis_reduce_workspace_bytes(). */
size_t nis_reduce_workspace_bytes(void);
int nis_reduce_moments(const void* v, int32_t dtype, int64_t n, double* out, int32_t accumulate,
                       void* workspace, size_t workspace_bytes, void* stream);

/* The same plus what the unweighting step needs and a non-finite guard (experiment_mg.py:73-76,101 take
 * torch.max / torch.mean / torch.var of f*J):  out[0..6) = { sum v, sum v^2, n, max v, min v, number of non-finite
 * entries }.  Sums, max and min follow torch semantics (a NaN propagates); out[5] lets the caller say how many
 * entries were inf / NaN instead of returning a silent NaN estimate. */
int nis_reduce_stats(const void* v, int32_t dtype, int64_t n, double* out, int32_t accumulate,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Phase-space generator descriptor (flat_phase_space_generator.py:25-39). */
typedef struct NisRamboDesc {
    int32_t n_final;
    double initial_masses[2];
    double final_masses[NIS_MAX_FINAL];
    double E_cm;        /* collider energy; the partonic energy is sqrt(x1 x2) E_cm when pdf_active */
    double pT_mincut;   /* event weight -> 0 if min_j pT_j < pT_mincut      (:285-288) */
    double delR_mincut; /* ... if any pair |deltaR| < delR_mincut           (:290-296) */
    double rap_maxcut;  /* ... if rap_maxcut > 0 and rap_maxcut < |max eta| (:298-301) */
    /* ---- parton-density mode (:157-187, 213-219, 283; utils.py:83-146) -------------------------------------------
     * pdf_active != 0: r has two more columns (3n-2 in all) that sample the Bjorken x of the beams; the event is
     * generated at E = sqrt(x1 x2) E_cm, the weight carries the sampling Jacobian, the two parton densities
     * f(x) = xf(x, Q2) / x, the x cut and 1 / (2 x1 x2 E_cm^2), and the cuts act on the momenta boosted to the lab
     * frame (the momenta returned stay in the partonic CM frame, like the reference's).
     *   tau_mode != 0: column 3n-4 samples tau in [tau_min, 1], column 3n-3 samples y_cm in [ln(tau)/2, -ln(tau)/2],
     *                  x1,2 = sqrt(tau) exp(+-y_cm);   tau_mode == 0: x2 = column 3n-4, x1 = column 3n-3.
     *   pdf_grid[i]: DEVICE pointer to pdf_nodes float64 values of x f_i(x, Q2 = 91.188^2) on nodes uniform in ln x
     *                over [pdf_lnx_lo, 0] (4-point Lagrange interpolation in ln x), or NULL for density 1
     *                (what get_pdfQ2 returns without a PDF set or for a non-parton pdg code, :124-128). */
    int32_t pdf_active;
    int32_t tau_mode;
    double tau_min;     /* (max(sum of final masses, absolute_Ecm_min) / E_cm)^2  (:163-164) */
    double x_cut;       /* weight -> 0 if x1 or x2 < x_cut; the reference uses 1e-4 (:185-186) */
    const double* pdf_grid[2];
    int32_t pdf_nodes;
    double pdf_lnx_lo;
} NisRamboDesc;

/* r[B, 3n-4 (+2 when pdf_active)] (dtype r_dtype) -> momenta[B, 2+n, 4] float64 (E,px,py,pz; CM frame; optional),
 * weight[B] float64 (cuts applied, divided by 2 s), cutmask[B] uint8 (1 = passed; optional).
 * r must be 16-byte and momenta 32-byte aligned (rows are moved as 16- / 32-byte vectors). */
int nis_rambo_generate(const NisRamboDesc* desc, const void* r, int32_t r_dtype, double* momenta,
                       double* weight, uint8_t* cutmask, int64_t B, void* stream);

/* Inverse of the pdf-inactive map (SURVEY 8 f4; the reference lists it as to do, README.md:68-69): momenta[B, 2+n, 4]
 * float64 as nis_rambo_generate writes them (CM frame; the two beam rows are skipped) -> r[B, 3n-4] float64, the uniforms
 * generateKinematics_batch maps to these momenta, and weight[B] float64 = the weight of that point WITHOUT cuts (optional).
 * desc->pdf_active must be 0 (NIS_EUNSUPPORTED otherwise). */
int nis_rambo_invert(const NisRamboDesc* desc, const double* momenta, double* r, double* weight, int64_t B, void* stream);

/* Philox4x32-10 uniforms in [0,1): out[n] of dtype; element i is a pure function of (seed, offset+i),
 * so ranks draw disjoint streams by offsetting. */
int nis_uniform_fill(void* out, int32_t dtype, int64_t n, uint64_t seed, uint64_t offset, void* stream);

/* Measurement aid for bench.py: launches a kernel of pure FP32 FMA chains on `stream` and returns the
 * number of floating-point operations it performs (or a negative error).  Timing it with CUDA events
 * gives the measured FP32-pipe peak the compute-bound flow kernels are quoted against. */
int64_t nis_probe_fp32_fma(float* out, int32_t iters, void* stream);

/* Measurement aid for bench.py: launches `iters` x 8 back-to-back tcgen05.mma (cta_group::1, M = 128, N = n in
 * {64, 128, 256}, A in tensor memory, fp32 accumulate) per SM on `stream` and returns the floating-point operations
 * performed (or a negative error).  kind 0 = kind::tf32 (K = 8), 1 = kind::f16 (K = 16).  Timing it with CUDA events
 * gives the MEASURED tensor-pipe peak the tcgen05 flow kernels are quoted against. */
int64_t nis_probe_tensor(int32_t kind, int32_t n, int32_t iters, void* stream);

/* Measurement aid for bench.py: per-launch device times of nis_flow_forward and nis_flow_inverse.  After
 * nis_flow_timing_begin(stream) every kernel launch of the nis_flow_forward / nis_flow_inverse calls made by THIS thread
 * is bracketed by CUDA events recorded on the launch
 * stream; nis_flow_timing_end synchronises them and returns the number of launches written to ms[] / tags[] (tags: 0 weight
 * packs, 1 column moments, 10 fused eval cell, 11 layer pass from the state, 13 layer pass from stored activations, 12
 * final pass from stored activations, 2 other), or a negative error. */
int nis_flow_timing_begin(void* stream);
int nis_flow_timing_end(float* ms, int32_t* tags, int32_t max_n);

/* sizeof(NisFlowDesc) / sizeof(NisRamboDesc) as compiled, so a foreign-language binding can verify its
 * struct layout at load time. */
size_t nis_sizeof_flow_desc(void);
size_t nis_sizeof_rambo_desc(void);

const char* nis_strerror(int code);
const char* nis_version(void);

#ifdef __cplusplus
}
#endif
#endif /* NIS_B200_H */
