// Fused coupling-cell forward, width-64 PWLin cells, on tcgen05 with a HALF-PRECISION SPLIT of the operands —
// the round-2 successor of flow_tc.cu's 3xTF32 kernel (which stays for PWQuad cells and as the A/B reference).
//
// Why: ncu on the 3xTF32 kernel (profiles/r01_ncu_tc.md) showed a latency-bound chain epilogue -> MMA -> epilogue
// with only TWO 128-point groups per SM to overlap (warp slots 14 % occupied, 52 % of the stall samples on the
// mbarrier / tcgen05.ld hand-over): TF32 operands in tensor memory take 64 + 64 columns per group next to a 128-
// column accumulator, i.e. all 512 columns for two groups.  Here
//   * activations and weights are split as x = x_hi + x_lo with BOTH parts in fp16 (11-bit significands: the same
//     22 bits as the TF32 split) after an exact power-of-two scaling that keeps x_lo out of fp16's subnormal range
//     (activations x 2^3, saturating at 65504 / 8 = 8188 — a BatchNorm output that large does not occur; weights by a
//     per-layer 2^k chosen at pack time so that max |w| lands in [2^13, 2^14)); D += a_hi w_lo + a_lo w_hi + a_hi w_hi
//     as tcgen05.mma.kind::f16 with fp32 accumulation, K = 16 per instruction: 12 instructions per 64x64 layer
//     instead of 24 (tools/tc_f16_probe.cu: same 44.7 cycles per M128 N64 instruction as kind::tf32);
//   * the packed A operand takes 32 + 32 columns and every MMA block is N = 64 (the 128 logits of the output layer
//     are two blocks into the same accumulator columns, the splines of the first pair run while the second block's
//     MMAs execute), so a group needs 128 columns and FOUR groups (16 warps) share an SM;
//   * there is no issuer warp: thread 0 of a group issues the group's own MMAs once the group's 128 "my operand row
//     is in tensor memory" arrivals are in (a 17th warp would cap the kernel at 96 registers per thread, and a
//     group never queues behind a slower one).
// The layer-pass scheme for train-mode BatchNorm, the tile-blocked activation buffers and the statistics fold are
// those of flow_tc.cu / flow_tiled.cu (DESIGN.md 4.2b).  Reference: coupling_cells.py:84-142 (PWLin + conditioner).
#include <stdlib.h>
#include <cuda_fp16.h>
#include "common.cuh"
#include "spline.cuh"
#include "flow_fwd_common.cuh"
#include "tc_common.cuh"
#include "tc_spline.cuh"

#define H_SA 8.0f                                  // activation scale before the split (exact power of two)
#define H_AMAX 65504.0f                            // largest finite fp16
#define H_HID_BYTES (2 * TCH * TCH * 2)            // hi + lo of a 64x64 layer in fp16: 16 KB
#define H_MAXG 4
// Output layer as N-wide MMA blocks into the same accumulator columns.  PWLin, 32 bins: N = 64 = two transformed
// dimensions per block, 128 rows in all; tensor-memory columns per group: D 64 | A_hi 32 | A_lo 32 = 128 -> four groups.
// PWQuad, 32 bins (65 logits per dimension): N = 80 = one dimension per block (rows 65..79 zero); D 80 | pad 16 |
// A_hi 32 | A_lo 32 = 160 -> three groups.
template <int KIND> struct HK {
    static constexpr int OUT_N = KIND == NIS_KIND_PWLIN ? 64 : 80;          // MMA N of an output block
    static constexpr int TPER = KIND == NIS_KIND_PWLIN ? 2 : 1;             // transformed dimensions per block
    static constexpr int SLOT = KIND == NIS_KIND_PWLIN ? 32 : 80;           // rows per dimension
    static constexpr int COLS = KIND == NIS_KIND_PWLIN ? 128 : 160;
    static constexpr int COL_AHI = KIND == NIS_KIND_PWLIN ? 64 : 96;
    static constexpr int COL_ALO = COL_AHI + 32;
    static constexpr int MAXG = KIND == NIS_KIND_PWLIN ? 4 : 3;
};
__host__ __device__ static inline int h_slot(const DevFlow& F) { return F.kind == NIS_KIND_PWLIN ? 32 : 80; }
__host__ __device__ static inline int h_out_rows(const DevFlow& F) {      // rows of the staged output-layer operand
    int mt = 1;
    for (int c = 0; c < F.n_cells; ++c) mt = F.cells[c].T > mt ? F.cells[c].T : mt;
    const int r = mt * h_slot(F);
    return F.kind == NIS_KIND_PWLIN ? (r < 128 ? 128 : r) : r;
}
__host__ __device__ static inline int h_out_bytes(const DevFlow& F) { return 2 * h_out_rows(F) * TCH * 2; }

// byte offset of (row, k) in a [rows x 64] fp16 K-major operand: 128 B per row, 8-row groups of 1024 B, 16-byte
// chunks XOR-swizzled with row % 8 (the canonical SWIZZLE_128B layout; one 128-byte row holds all of K = 64)
__host__ __device__ static inline int h_off(int row, int k) {
    return (row >> 3) * 1024 + (row & 7) * 128 + ((((k >> 3) ^ (row & 7)) << 4) | ((k & 7) << 1));
}
// instruction descriptor for kind::f16: c_format F32 (1) at [4,6), a/b format F16 (0) at [7,10)/[10,13), K-major,
// N >> 3 at [17,23), M >> 4 at [24,29)
__host__ __device__ constexpr uint32_t h_idesc(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// a cell's pack: hidden layers 1 .. depth-1 | output layer | layer 0 (K = P <= 16, zero-padded to a 64x64 block: the
// swizzled rows are 128 bytes whatever K is) | the per-layer 1 / (SA * SW) factors
__host__ __device__ static inline size_t h_l0_off(const DevFlow& F) { return (size_t)(F.depth - 1) * H_HID_BYTES + h_out_bytes(F); }
__host__ __device__ static inline size_t h_cell_bytes(const DevFlow& F) { return h_l0_off(F) + H_HID_BYTES + 64; }

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// two floats -> packed fp16 pair (x in the low half), round to nearest, saturating to +-65504 instead of infinity
__device__ __forceinline__ uint32_t h_pack_sat(float x, float y) {
    uint32_t d;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(y), "f"(x));
    return d;
}

__device__ __forceinline__ void h_mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}

// ---- weight pack: one CTA per (MMA layer, cell): max |w| -> power-of-two scale -> fp16 hi / lo in UMMA layout -------
__global__ void __launch_bounds__(256) flow_h_pack_kernel(DevFlow F, const float* __restrict__ params, char* __restrict__ hpack) {
    __shared__ float red[8];
    __shared__ float sw_s;
    const int c = blockIdx.y, li = blockIdx.x, tid = threadIdx.x;
    const DevCell& q = F.cells[c];
    const bool outl = li == F.depth - 1, first = li == F.depth;      // (the block of layer 0 comes last in the pack)
    const int l = first ? 0 : li + 1;                                // MMA layer 0..depth (depth = output layer)
    const float* w = params + q.param_off + F.p_lin(c, l);           // layer 0: [64][P]; hidden: [64][64]; output: [T*K][64] (out, in)
    const int kin = first ? q.P : TCH;
    const int rows_src = outl ? q.T * F.K : TCH, rows = outl ? h_out_rows(F) : TCH, slot = h_slot(F);
    float m = 0.f;
    for (int i = tid; i < rows_src * kin; i += 256) m = fmaxf(m, fabsf(w[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((tid & 31) == 0) red[tid >> 5] = m;
    __syncthreads();
    if (tid == 0) {
        for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]);
        int e = 14;
        if (m > 0.f && m < 3.0e38f) frexpf(m, &e);                   // m = f * 2^e, f in [0.5, 1)
        e = e < -100 ? -100 : (e > 100 ? 100 : e);
        sw_s = ldexpf(1.f, 14 - e);                                  // max |w| * SW in [2^13, 2^14)
    }
    __syncthreads();
    const float SW = sw_s;
    char* dst = hpack + (size_t)c * h_cell_bytes(F);
    char* hi = dst + (first ? h_l0_off(F) : (size_t)li * H_HID_BYTES);   // (the output layer follows the depth-1 hidden ones)
    char* lo = hi + (size_t)rows * TCH * 2;
    for (int i = tid; i < rows * TCH; i += 256) {
        const int n = i / TCH, k = i - n * TCH;
        // staged row n = dimension n / slot, logit n % slot (PWLin: slot = K = 32, the torch row order itself)
        const int t = outl ? n / slot : 0, jj = outl ? n - t * slot : n;
        const bool live = outl ? (t < q.T && jj < F.K) : k < kin;
        const float v = live ? w[(size_t)(outl ? t * F.K + jj : n) * kin + k] * SW : 0.f;
        const __half h = __float2half_rn(v);
        const int o = h_off(n, k);
        *reinterpret_cast<__half*>(hi + o) = h;
        *reinterpret_cast<__half*>(lo + o) = __float2half_rn(v - __half2float(h));
    }
    if (tid == 0) reinterpret_cast<float*>(dst + h_cell_bytes(F) - 64)[l] = 1.f / (H_SA * SW);
}

struct HSmem {      // byte offsets from the 1024-aligned base
    int w0, aff, bias, st, sst, red, zb, total;
    int wfirst;     // the staged MMA layers wfirst .. l_end (hi, lo) start at offset 0, hidden ones 16 KB apart, the
                    // output layer (l = depth) last
    // offset of staged layer l: a closed form, so that the kernel indexes no array (which would live in local memory:
    // a 136-byte stack frame, reloaded in the tile loop)
    __host__ __device__ int wl(int l) const { return (l - wfirst) * H_HID_BYTES; }
};
__host__ __device__ static inline HSmem h_layout(const DevFlow& F, int P, int l_begin, int l_end, bool zstage, int NG,
                                                 bool layer0 = true, bool stats = true) {
    HSmem s;
    int o = 0;
    s.wfirst = l_begin > 1 ? l_begin : 1;
    for (int l = s.wfirst; l <= l_end; ++l) o += l == F.depth ? h_out_bytes(F) : H_HID_BYTES;
    (void)P;
    s.w0 = o; o += layer0 ? H_HID_BYTES : 0;                  // layer-0 operand (hi, lo): only when the pass starts from the state
    s.aff = o; o += (F.depth + 1) * 2 * TCH * 4;
    s.bias = o; o += h_out_rows(F) * 4;
    s.st = o; o += NG * (F.d + 1) * TCM * 4;
    o = (o + 15) & ~15;
    s.sst = o; o += NG * (F.d + 1) * TCM * 4;          // landing zone of the next tile's state rows (bulk copy), per group
    o = (o + 7) & ~7;
    s.red = o; o += stats ? (NG * TCM * 2 + 2 * F.maxW) * 8 : 0;   // statistics fold: only in statistics passes
    o = (o + 127) & ~127;
    s.zb = o;                                          // [NG][64][128] floats: stored-activation tile in, then out
    if (zstage) o += NG * TCH * TCM * 4;
    s.total = o;
    return s;
}

// 32 activations: a = min(max(v * sc + sh, 0), 65504) with sc / sh pre-multiplied by SA, split a = hi + lo (both fp16),
// packed two per 32-bit column (even feature in the low half) into the group's A operand.
__device__ __forceinline__ void h_store_act32(const float* v, const float* sc, const float* sh, uint32_t t_hi, uint32_t t_lo) {
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int j4 = 0; j4 < 8; ++j4) {
        const float4 s4 = reinterpret_cast<const float4*>(sc)[j4], h4 = reinterpret_cast<const float4*>(sh)[j4];
        const float a0 = fmaxf(fmaf(v[4 * j4], s4.x, h4.x), 0.f), a1 = fmaxf(fmaf(v[4 * j4 + 1], s4.y, h4.y), 0.f);
        const float a2 = fmaxf(fmaf(v[4 * j4 + 2], s4.z, h4.z), 0.f), a3 = fmaxf(fmaf(v[4 * j4 + 3], s4.w, h4.w), 0.f);
        // hi = fp16(a) (round to nearest, saturating at 65504: one packed conversion per pair), lo = fp16(a - hi) with
        // the subtraction exact in float32; even feature in the low half
        const uint32_t p01 = h_pack_sat(a0, a1), p23 = h_pack_sat(a2, a3);
        const float2 f01 = __half22float2(*reinterpret_cast<const __half2*>(&p01));
        const float2 f23 = __half22float2(*reinterpret_cast<const __half2*>(&p23));
        hi[2 * j4] = p01;
        hi[2 * j4 + 1] = p23;
        lo[2 * j4] = h_pack_sat(a0 - f01.x, a1 - f01.y);
        lo[2 * j4 + 1] = h_pack_sat(a2 - f23.x, a3 - f23.y);
    }
    tc_st16(t_hi, hi);
    tc_st16(t_lo, lo);
}

// one N = 64 block of a layer: D (+)= a_hi w_lo + a_lo w_hi (cross terms first: the tensor core truncates when it adds
// into the accumulator, so the small terms go in while it is small, DESIGN.md 4.3c), then a_hi w_hi; K = 16 per step
__device__ __forceinline__ void h_issue_block(uint32_t tmem_d, uint32_t t_hi, uint32_t t_lo, uint32_t w_hi, uint32_t w_lo, uint32_t idesc) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        h_mma_ts(tmem_d, t_hi + ks * 8, tc_desc(w_lo + ks * 32), idesc, ks > 0);
        h_mma_ts(tmem_d, t_lo + ks * 8, tc_desc(w_hi + ks * 32), idesc, 1);
    }
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) h_mma_ts(tmem_d, t_hi + ks * 8, tc_desc(w_hi + ks * 32), idesc, 1);
}

// MODE: bit 0 = statistics (layer) pass, bit 1 = the first operand comes from stored activations, bit 2 (final pass of a
// train-mode cell) = the column moments of the NEXT cell's pass-through columns are accumulated from the state this pass
// writes (14 sums for P <= 4) and folded into that cell's BN_0 / BN_1 by the last CTA, bit 3 (fused cell or final pass)
// = the inverse cell (nis_flow_inverse): inverse splines, Jacobian divided by the densities, and the last inverse cell
// (c = 0) stores the physical column order.  Statistics and layer passes have no inverse bit: they read only the
// pass-through columns, which a cell conditions on in either direction.  Compile-time, so that
// every instantiation carries only its own path: the all-in-one kernel was 64 KB of SASS and its four groups, each in
// another phase, missed the instruction cache (ncu: `no_instruction` 0.8 stalled warps per issue).
template <int NG, int KIND, int MODE>
__global__ void __launch_bounds__(NG * TCM, 1) flow_cell_h_kernel(const __grid_constant__ DevFlow F, const FwdArgs A,
                                                                        const char* __restrict__ hpack) {
    constexpr int NT = NG * TCM;
    typedef HK<KIND> K_;
    constexpr int H_COLS = K_::COLS, H_COL_AHI = K_::COL_AHI, H_COL_ALO = K_::COL_ALO;
    extern __shared__ char smraw[];
    __shared__ uint64_t a_ready[NG], d_ready[NG], z_full[NG], s_full[NG];
    __shared__ uint32_t tmem_base_s;
    char* sm = smem_align1024(smraw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int c = A.c_begin;
    const DevCell& q = F.cells[c];
    const int d = F.d, depth = F.depth;
    // which slice of the cell this launch computes (same table as flow_tc.cu)
    constexpr bool stats = (MODE & 1) != 0;
    constexpr bool from_z = (MODE & 2) != 0;
    constexpr bool nextmom = (MODE & 4) != 0;
    constexpr bool inverse = (MODE & 8) != 0;
    // the state feeds layer 0, the splines and the stores: a statistics pass from stored activations has none of them
    constexpr bool needs_state = !(from_z && stats);
    constexpr int MOM_N = 4 + 4 * 5 / 2;                                    // sum x_k, sum x_k x_k2 (k <= k2), P <= 4
    float macc[nextmom ? MOM_N : 1];
#pragma unroll
    for (int i = 0; i < (nextmom ? MOM_N : 1); ++i) macc[i] = 0.f;
    const int lz = from_z ? (A.zin_layer > 0 ? A.zin_layer : (stats ? A.stats_layer - 1 : depth)) : 1;   // first A operand: z_{lz}
    const int l_end = stats ? A.stats_layer - 1 : depth;                   // MMA layers lz .. l_end
    const bool zst = from_z || stats;
    const HSmem L = h_layout(F, q.P, lz, l_end, zst, NG, !from_z, stats);
    float* affs = reinterpret_cast<float*>(sm + L.aff);
    float* biass = reinterpret_cast<float*>(sm + L.bias);
    const float* pk = A.wpack + q.pk_off;
    const char* cellpack = hpack + (size_t)c * h_cell_bytes(F);
    const float* inv_scale = reinterpret_cast<const float*>(cellpack + h_cell_bytes(F) - 64);    // [l] = 1 / (SA * SW_l)

    // ---- one-time setup: weights, barriers, tensor memory ---------------------------------------------
    for (int l = L.wfirst; l <= l_end; ++l) {
        const int n16 = (l == depth ? h_out_bytes(F) : H_HID_BYTES) / 16;
        const uint4* src = reinterpret_cast<const uint4*>(cellpack + (size_t)(l - 1) * H_HID_BYTES);
        uint4* dst = reinterpret_cast<uint4*>(sm + L.wl(l));
        for (int i = tid; i < n16; i += NT) dst[i] = src[i];
    }
    if (!from_z) {                                                // layer 0 (hi, lo): one K = 16 step of a 64x64 block
        const uint4* src = reinterpret_cast<const uint4*>(cellpack + h_l0_off(F));
        uint4* dst = reinterpret_cast<uint4*>(sm + L.w0);
        for (int i = tid; i < H_HID_BYTES / 16; i += NT) dst[i] = src[i];
    }
    for (int l = 0; l <= depth; ++l) {                            // BN scale / shift; layers feeding an MMA carry the SA factor
        const int W = l == 0 ? q.P : TCH, Wp = pad8(W);
        const float* s = pk + q.aff_off[l];
        const float f = H_SA;
        // a layer fed by the accumulator of the layer below (D = z * SA * SW: chained in this launch, or stored as it is
        // by the statistics pass of that layer) takes that factor into its scale
        const float fs = (l >= 1 && l >= lz && l <= l_end) ? f * inv_scale[l - 1] : f;
        for (int i = tid; i < W; i += NT) { affs[l * 2 * TCH + i] = fs * s[i]; affs[l * 2 * TCH + TCH + i] = f * s[Wp + i]; }
    }
    const int out_rows = h_out_rows(F);
    // the splines only need exp(logit - max): the logits are kept in units of log 2 (scale and bias carry log2(e)) so
    // that the exponential is a bare ex2
    constexpr float LOGIT_UNIT = 1.4426950408889634f;
    for (int i = tid; i < out_rows; i += NT) {
        const int t = i / K_::SLOT, jj = i - t * K_::SLOT;
        biass[i] = (t < q.T && jj < F.K) ? LOGIT_UNIT * pk[q.bo_off + t * F.Kpad + jj] : 0.f;
    }
    if (tid == 0) {
        for (int g = 0; g < NG; ++g) {
            mbar_init(&a_ready[g], TCM); mbar_init(&d_ready[g], 1); mbar_init(&z_full[g], 1); mbar_init(&s_full[g], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
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
    const int nblk = (q.T + K_::TPER - 1) / K_::TPER;            // output layer: MMA blocks of TPER transformed dimensions
    const bool has_out = l_end == depth;
    double dsum = 0.0, dsq = 0.0;

    const uint32_t idesc = h_idesc(TCM, TCH), idesc_out = h_idesc(TCM, K_::OUT_N);
    {
        // ===================== point groups ====================================================
        const int g = warp >> 2, gt = tid & (TCM - 1);
        float* st = reinterpret_cast<float*>(sm + L.st) + g * (d + 1) * TCM + gt;   // this thread's state column
        const uint32_t tg = tmem_base + g * H_COLS + ((uint32_t)((warp & 3) * 32) << 16);
        uint32_t pd = 0, pa = 0, zph = 0, sph = 0;
        float* zs = reinterpret_cast<float*>(sm + L.zb) + g * TCH * TCM;
        constexpr uint32_t ZBYTES = TCH * TCM * 4;
        // the state rows of a full tile are one contiguous block: they arrive by bulk copy, issued one tile ahead
        // (the landing zone is free as soon as every thread has moved its row into its state column)
        float* sst = reinterpret_cast<float*>(sm + L.sst) + g * (d + 1) * TCM;
        const uint32_t SBYTES = (uint32_t)((d + 1) * TCM * 4);
        const bool st_bulk = needs_state && A.from_state && (reinterpret_cast<uintptr_t>(A.state_in) & 15) == 0 && (SBYTES & 15) == 0;
        if (st_bulk && gt == 0) {
            const long long t0 = (long long)blockIdx.x * NG + g;
            if ((t0 + 1) * TCM <= A.B) bulk_load(sst, A.state_in + t0 * TCM * rowlen, SBYTES, &s_full[g]);
        }
        const float inv_out = has_out ? LOGIT_UNIT * inv_scale[depth] : 0.f;
        for (long long it = 0;; ++it) {
            const long long tile = ((long long)blockIdx.x + it * gridDim.x) * NG + g;
            if (tile >= ntiles) break;
            const long long tn = tile + (long long)gridDim.x * NG;
            if (from_z && gt == 0) {
                // single staging buffer per group: the previous tile's output (if any) must have left it
                if (A.zout) bulk_store_wait_read();
                bulk_load(zs, A.zin + (size_t)tile * TCH * TCM, ZBYTES, &z_full[g]);
                if (tn < ntiles) bulk_prefetch_l2(A.zin + (size_t)tn * TCH * TCM, ZBYTES);
            }
            const long long pt = tile * TCM + gt;
            const bool valid = pt < A.B;
            // ---- this thread's point --------------------------------------------------------------
            if (!needs_state) {
            } else if (st_bulk && (tile + 1) * TCM <= A.B) {
                mbar_wait(&s_full[g], sph);
                sph ^= 1;
                for (int i = 0; i <= d; ++i) st[i * TCM] = sst[gt * rowlen + i];
                proxy_fence();                       // our reads of the landing zone precede the next bulk write into it
                group_sync(g);
                if (gt == 0 && (tn + 1) * TCM <= A.B) bulk_load(sst, A.state_in + tn * TCM * rowlen, SBYTES, &s_full[g]);
            } else if (valid) {
                if (A.from_state) {
                    for (int i = 0; i <= d; ++i) st[i * TCM] = A.state_in[pt * rowlen + i];
                } else {
                    for (int i = 0; i < d; ++i) st[i * TCM] = load_io(A.in, A.in_dtype, pt * A.in_cols + i);
                    st[d * TCM] = A.in_cols > d ? load_io(A.in, A.in_dtype, pt * A.in_cols + d) : 1.f;
                }
                if (!stats && A.saved && !A.from_state) {
                    float* sv = A.saved + ((long long)c * A.B + pt) * rowlen;
                    for (int i = 0; i <= d; ++i) sv[i] = st[i * TCM];
                }
            } else {
                for (int i = 0; i < d; ++i) st[i * TCM] = 0.5f;
                st[d * TCM] = 1.f;
            }
            if (from_z) { mbar_wait(&z_full[g], zph); zph ^= 1; }
            if (!from_z) {
                // ---- layer 0 (K = P <= 16): BN_0 of the pass-through columns, split like every other operand, one K = 16
                //      step (3 instructions) - 4 x 64 multiply-adds per point on the FP32 pipe were 13 % of the fused cell's
                //      instructions.  Columns beyond P are zero (and so are the weight's).
                uint32_t hi[8], lo[8];
#pragma unroll
                for (int j2 = 0; j2 < 8; ++j2) {
                    float a0 = 0.f, a1 = 0.f;
                    if (2 * j2 < q.P) a0 = fmaf(st[q.feed[2 * j2] * TCM], affs[2 * j2], affs[TCH + 2 * j2]);
                    if (2 * j2 + 1 < q.P) a1 = fmaf(st[q.feed[2 * j2 + 1] * TCM], affs[2 * j2 + 1], affs[TCH + 2 * j2 + 1]);
                    const uint32_t p01 = h_pack_sat(a0, a1);
                    const float2 f01 = __half22float2(*reinterpret_cast<const __half2*>(&p01));
                    hi[j2] = p01;
                    lo[j2] = h_pack_sat(a0 - f01.x, a1 - f01.y);
                }
                tc_st8(tg + H_COL_AHI, hi);
                tc_st8(tg + H_COL_ALO, lo);
                tc_st_wait();
                tc_fence_before();
                mbar_arrive(&a_ready[g]);
                if (gt == 0) {
                    mbar_wait(&a_ready[g], pa);
                    tc_fence_after();
                    const uint32_t whi = smem_u32(sm + L.w0), wlo = whi + TCH * TCH * 2;
                    const uint32_t tb = tmem_base + g * H_COLS;
                    h_mma_ts(tb, tb + H_COL_AHI, tc_desc(wlo), idesc, 0);
                    h_mma_ts(tb, tb + H_COL_ALO, tc_desc(whi), idesc, 1);
                    h_mma_ts(tb, tb + H_COL_AHI, tc_desc(whi), idesc, 1);
                    tc_commit(&d_ready[g]);
                }
                pa ^= 1;
                mbar_wait(&d_ready[g], pd);
                pd ^= 1;
                tc_fence_after();
            }
            // ---- MMA layers lz .. l_end: build the A operand of layer l from z_l, 32 features at a time -----------
            for (int l = lz; l <= l_end; ++l) {
                const float* sc = affs + l * 2 * TCH;
#pragma unroll 1
                for (int h = 0; h < 2; ++h) {
                    float v[32];
                    if (l > lz || !from_z) {                      // chained: the accumulator of layer l-1
                        tc_ld32(tg + 32 * h, v);
                        tc_ld_wait();
                    } else {                                      // stored pre-BN activations
                        const float* zr = zs + (32 * h) * TCM + gt;
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = zr[j * TCM];
                    }
                    h_store_act32(v, sc + 32 * h, sc + TCH + 32 * h, tg + H_COL_AHI + 16 * h, tg + H_COL_ALO + 16 * h);
                }
                if (l == lz && from_z) proxy_fence();             // our reads of the staging tile precede the next bulk write into it
                tc_st_wait();
                tc_fence_before();
                mbar_arrive(&a_ready[g]);
                if (gt == 0) {                                    // the group's issuer: all 128 operand rows are in place
                    mbar_wait(&a_ready[g], pa);
                    tc_fence_after();
                    const uint32_t whi = smem_u32(sm + L.wl(l));
                    const uint32_t tb = tmem_base + g * H_COLS;
                    h_issue_block(tb, tb + H_COL_AHI, tb + H_COL_ALO, whi, whi + (l == depth ? out_rows : TCH) * TCH * 2,
                                  l == depth ? idesc_out : idesc);
                    tc_commit(&d_ready[g]);
                }
                pa ^= 1;
                if (l < depth) {
                    mbar_wait(&d_ready[g], pd);
                    pd ^= 1;
                    tc_fence_after();
                }
            }
            if (stats) {
                // ---- statistics pass: z_L goes to the staging tile [64][128] (over the input tile), from there to HBM by
                //      ONE bulk store, and its per-feature sums are row sums of the tile
                if (!from_z) {
                    if (gt == 0) bulk_store_wait_read();          // the previous tile's store has read the buffer
                    group_sync(g);
                }
                // the accumulator is stored as it is (z * SA * SW: the next pass and the statistics fold carry the factor);
                // rows beyond the batch (ragged last tile only) are stored as zeros
                const bool full = (tile + 1) * TCM <= A.B;
#pragma unroll 1
                for (int h = 0; h < 2; ++h) {
                    float v[32];
                    tc_ld32(tg + 32 * h, v);
                    tc_ld_wait();
                    if (full) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) zs[(32 * h + j) * TCM + gt] = v[j];
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) zs[(32 * h + j) * TCM + gt] = valid ? v[j] : 0.f;
                    }
                }
                proxy_fence();
                group_sync(g);
                if (gt == 0 && A.zout) bulk_store(A.zout + (size_t)tile * TCH * TCM, zs, ZBYTES);
                if (!A.no_stats) {
                    // thread gt sums half a row (64 points) of feature gt & 63, 16 bytes at a time; the start is
                    // rotated by the lane so that a warp's 32 rows do not hit the same banks
                    const float4* row = reinterpret_cast<const float4*>(zs + (gt & 63) * TCM + (gt >> 6) * 64);
                    float s_ = 0.f, q_ = 0.f;
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const float4 x = row[(i + lane) & 15];
                        s_ += (x.x + x.y) + (x.z + x.w);
                        q_ = fmaf(x.x, x.x, fmaf(x.y, x.y, fmaf(x.z, x.z, fmaf(x.w, x.w, q_))));
                    }
                    dsum += (double)s_; dsq += (double)q_;
                }
                proxy_fence();
                group_sync(g);
                continue;
            }
            // ---- output layer, one MMA block at a time; the splines run on the thread's logits in registers while the
            //      next block's MMAs execute (the accumulator is released as soon as tcgen05.ld has returned)
            float jfac = 1.f;
            for (int b = 0; b < nblk; ++b) {
                mbar_wait(&d_ready[g], pd);
                pd ^= 1;
                tc_fence_after();
                float z[K_::OUT_N];
                tc_ld32(tg, z);
                tc_ld32(tg + 32, z + 32);
                if (KIND != NIS_KIND_PWLIN) tc_ld16(tg + 64, z + 64);
                tc_ld_wait();
                if (b + 1 < nblk) {                  // accumulator consumed: the next block's MMAs may overwrite it
                    tc_fence_before();
                    mbar_arrive(&a_ready[g]);
                    if (gt == 0) {
                        mbar_wait(&a_ready[g], pa);
                        tc_fence_after();
                        const uint32_t whi = smem_u32(sm + L.wl(depth)) + (uint32_t)(b + 1) * (K_::OUT_N * 128);
                        const uint32_t tb = tmem_base + g * H_COLS;
                        h_issue_block(tb, tb + H_COL_AHI, tb + H_COL_ALO, whi, whi + out_rows * TCH * 2, idesc_out);
                        tc_commit(&d_ready[g]);
                    }
                    pa ^= 1;
                }
                if (KIND == NIS_KIND_PWLIN) {
                    // PWLin, 32 bins (coupling_cells.py:114-141): two transformed dimensions per block
#pragma unroll
                    for (int tt = 0; tt < 2; ++tt) {
                        const int t = 2 * b + tt;
                        if (t >= q.T) break;
                        const float xv = st[q.trafo[t] * TCM];
                        const float a = xv * 32.f;
                        int kb = (int)floorf(a);
                        kb = kb < 0 ? 0 : (kb > 31 ? 31 : kb);
                        const float alpha = a - (float)kb;
                        const float* bs = biass + t * 32;
                        float m = -3.0e38f;
#pragma unroll
                        for (int j = 0; j < 32; ++j) { z[32 * tt + j] = fmaf(z[32 * tt + j], inv_out, bs[j]); m = fmaxf(m, z[32 * tt + j]); }
                        if (inverse) {
                            float xo, jinv;
                            int ki;
                            pwlin32_tree_inv(z + 32 * tt, m, xv, xo, jinv, ki);
                            st[q.trafo[t] * TCM] = xo;
                            jfac *= jinv;
                            if (A.bins && valid) A.bins[((long long)c * A.B + pt) * d + t] = ki;
                        } else {
                            // S = sum of the 32 exponentials, C = the kb below the bin, ek = the bin's own: a pairwise sum tree, then
                            // a descent along the bits of kb that keeps the half / quarter / ... holding the bin (53 selects + 36
                            // adds; the predicated running sums `C += j < kb ? e : 0`, `ek = j == kb ? e : ek` were 128 + 32)
                            float e[32], s1[16], s2[8], s4[4];
#pragma unroll
                            for (int j = 0; j < 32; ++j) e[j] = ex2_approx(z[32 * tt + j] - m);
#pragma unroll
                            for (int j = 0; j < 16; ++j) s1[j] = e[2 * j] + e[2 * j + 1];
#pragma unroll
                            for (int j = 0; j < 8; ++j) s2[j] = s1[2 * j] + s1[2 * j + 1];
#pragma unroll
                            for (int j = 0; j < 4; ++j) s4[j] = s2[2 * j] + s2[2 * j + 1];
                            const float s8a = s4[0] + s4[1], s8b = s4[2] + s4[3];
                            const float S = s8a + s8b;
                            const bool b4 = kb & 16, b3 = kb & 8, b2 = kb & 4, b1 = kb & 2, b0 = kb & 1;
                            float C = b4 ? s8a : 0.f;
#pragma unroll
                            for (int j = 0; j < 16; ++j) e[j] = b4 ? e[16 + j] : e[j];
#pragma unroll
                            for (int j = 0; j < 8; ++j) s1[j] = b4 ? s1[8 + j] : s1[j];
#pragma unroll
                            for (int j = 0; j < 4; ++j) s2[j] = b4 ? s2[4 + j] : s2[j];
#pragma unroll
                            for (int j = 0; j < 2; ++j) s4[j] = b4 ? s4[2 + j] : s4[j];
                            C += b3 ? s4[0] : 0.f;
#pragma unroll
                            for (int j = 0; j < 8; ++j) e[j] = b3 ? e[8 + j] : e[j];
#pragma unroll
                            for (int j = 0; j < 4; ++j) s1[j] = b3 ? s1[4 + j] : s1[j];
#pragma unroll
                            for (int j = 0; j < 2; ++j) s2[j] = b3 ? s2[2 + j] : s2[j];
                            C += b2 ? s2[0] : 0.f;
#pragma unroll
                            for (int j = 0; j < 4; ++j) e[j] = b2 ? e[4 + j] : e[j];
#pragma unroll
                            for (int j = 0; j < 2; ++j) s1[j] = b2 ? s1[2 + j] : s1[j];
                            C += b1 ? s1[0] : 0.f;
                            const float e0 = b1 ? e[2] : e[0], e1 = b1 ? e[3] : e[1];
                            C += b0 ? e0 : 0.f;
                            const float ek = b0 ? e1 : e0;
                            const float inv = 1.f / S;
                            st[q.trafo[t] * TCM] = (ek * alpha + C) * inv;
                            jfac *= ek * inv * 32.f;
                            if (A.bins && valid) A.bins[((long long)c * A.B + pt) * d + t] = kb;
                        }
                    }
                } else {
                    // PWQuad, 32 bins (coupling_cells.py:159-228): one transformed dimension per block, 65 logits
                    const float xv = st[q.trafo[b] * TCM];
                    const float* bs = biass + b * K_::SLOT;
#pragma unroll
                    for (int j = 0; j < 65; ++j) z[j] = fmaf(z[j], inv_out, bs[j]);
                    float y, f;
                    int kb;
                    if (inverse) pwquad32_tree_inv<true>(z, xv, y, f, kb);      // (f = 1 / density)
                    else pwquad32_tree<true>(z, xv, y, f, kb);
                    st[q.trafo[b] * TCM] = y;
                    jfac *= f;
                    if (A.bins && valid) A.bins[((long long)c * A.B + pt) * d + b] = kb;
                }
            }
            st[d * TCM] *= jfac;
            if (nextmom && valid) {
                // per-thread float32 partials, like flow_col_moments_kernel (a thread sees ~B / (SMs * 512) points <= 1)
                const DevCell& qn = F.cells[A.next_cell];
                float x[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) x[k] = k < qn.P ? st[qn.feed[k] * TCM] : 0.f;
                int o = 4;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    macc[k] += x[k];
#pragma unroll
                    for (int k2 = k; k2 < 4; ++k2) { macc[o] = fmaf(x[k], x[k2], macc[o]); ++o; }
                }
            }
            // ---- store ----------------------------------------------------------------------------------
            if (valid) {
                if (A.state_out) {
                    float* so = A.state_out + pt * rowlen;
                    for (int i = 0; i <= d; ++i) so[i] = st[i * TCM];
                }
                if (A.to_out) {
                    for (int i = 0; i < d; ++i) store_io(A.out, A.out_dtype, pt * rowlen + i, st[(inverse ? i : F.out_perm[i]) * TCM]);
                    store_io(A.out, A.out_dtype, pt * rowlen + d, st[d * TCM]);
                }
            }
        }
    }
    bulk_store_wait_read();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    if (nextmom) {
        // ---- fold the next cell's column moments: warps -> CTA -> (last CTA) grid, in float64 and fixed order ------
        __shared__ bool s_last_m;
        __shared__ double sc0s_m[4 + 16];
        double* redm = reinterpret_cast<double*>(sm + L.zb);           // the staging tiles are free now: [NT / 32][MOM_N], then tot
        double* totm = redm + (NT / 32) * MOM_N;
#pragma unroll
        for (int i = 0; i < MOM_N; ++i) {
            double a = (double)macc[i];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == 0) redm[warp * MOM_N + i] = a;
        }
        __syncthreads();
        if (tid < MOM_N) {
            double s_ = 0.0;
            for (int w = 0; w < NT / 32; ++w) s_ += redm[w * MOM_N + tid];
            A.partials[(size_t)blockIdx.x * MOM_N + tid] = s_;
        }
        __threadfence();
        __syncthreads();
        if (tid == 0) s_last_m = atomicAdd(A.counter, 1u) == gridDim.x - 1;
        __syncthreads();
        if (!s_last_m) return;
        __threadfence();
        fold_partials<MOM_N>(A.partials, gridDim.x, totm + MOM_N, totm, tid, NT);
        moments_finalize<4>(F, A, A.next_cell, totm, sc0s_m, tid, NT);
        if (tid == 0) *A.counter = 0u;
        return;
    }
    if (!stats || A.no_stats) return;
    // ---- fold: thread gt of a group holds the sums of feature gt & 63 over half of each of its tiles -----------
    double* red = reinterpret_cast<double*>(sm + L.red);          // [2][NG * 128]: sum / sum of squares per group thread
    double* sacc = red + NG * TCM * 2;                            // [2 * maxW]
    red[tid] = dsum; red[NG * TCM + tid] = dsq;
    for (int i = tid; i < 2 * F.maxW; i += NT) sacc[i] = 0.0;
    __syncthreads();
    if (tid < TCH) {
        double s = 0.0, s2 = 0.0;
        for (int k = 0; k < 2 * NG; ++k) { s += red[tid + 64 * k]; s2 += red[NG * TCM + tid + 64 * k]; }
        const double k1 = (double)inv_scale[l_end];               // the sums are of z * SA * SW (a power of two: exact)
        sacc[tid] = s * k1; sacc[F.maxW + tid] = s2 * k1 * k1;
    }
    bn_stats_finalize(F, A, sacc, NT, red);           // (red: 2 * NT doubles, free again once sacc is formed)
}

// ---------------------------------------------------------------------------------------------------
size_t nis_h_pack_floats(const DevFlow& F) {
    if (F.depth < 1) return 0;
    return (size_t)F.n_cells * (h_cell_bytes(F) / 4);
}

int64_t nis_tc_min_batch(int64_t dflt);

static int h_groups(const DevFlow& F) {
    // the largest group count whose three launch shapes fit the shared memory of an SM
    const size_t lim = 226 * 1024;
    for (int ng = F.kind == NIS_KIND_PWLIN ? HK<NIS_KIND_PWLIN>::MAXG : HK<NIS_KIND_PWQUAD>::MAXG; ng >= 2; --ng) {
        bool ok = true;
        for (int c = 0; c < F.n_cells && ok; ++c) {
            const int P = F.cells[c].P;
            ok = (size_t)h_layout(F, P, 1, F.depth, false, ng).total + 1024 <= lim               // fused eval cell
                 && (size_t)h_layout(F, P, F.depth - 1, F.depth - 1, true, ng).total + 1024 <= lim   // a layer pass
                 && (size_t)h_layout(F, P, F.depth, F.depth, true, ng, false, false).total + 1024 <= lim      // final pass
                 && (F.depth < 3 || (size_t)h_layout(F, P, F.depth - 1, F.depth, true, ng, false, false).total + 1024 <= lim);   // final pass from z_{depth-1}
        }
        if (ok) return ng;
    }
    return 0;
}

// Width-64 cells with 32 bins: PWLin (BASELINE configs[1]) and PWQuad (configs[3]); NIS_TC_H=0 keeps the 3xTF32 kernel
// (A/B test knob)
bool nis_h_supported(const DevFlow& F, int64_t B, int bn_mode) {
    (void)bn_mode;
    const char* off = getenv("NIS_TC_H");
    if (off && off[0] == '0') return false;
    const char* tcoff = getenv("NIS_TC");
    if (tcoff && tcoff[0] == '0') return false;
    if (F.nb != 32 || F.depth < 1 || F.maxW != TCH) return false;
    if (F.kind == NIS_KIND_PWLIN ? F.K != 32 : F.K != 65) return false;
    if (B < nis_tc_min_batch(256)) return false;
    for (int l = 0; l < F.depth; ++l) if (F.widths[l] != TCH) return false;
    for (int c = 0; c < F.n_cells; ++c)
        if (F.cells[c].P > 16 || (F.kind == NIS_KIND_PWLIN && F.cells[c].T * 32 > 128)) return false;
    return h_groups(F) >= 2;
}

int nis_h_pack(const DevFlow& F, const float* params, float* tcpack, cudaStream_t s) {
    flow_h_pack_kernel<<<dim3(F.depth + 1, F.n_cells), 256, 0, s>>>(F, params, reinterpret_cast<char*>(tcpack));
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

template <int NG, int KIND, int MODE>
static int h_launch_mode(const DevFlow& F, const FwdArgs& A, const char* hpack, size_t smem, int sms, cudaStream_t s) {
    static int attr_smem = 0;                            // cudaFuncSetAttribute only when the requirement grows
    if ((int)smem > attr_smem) {
        if (cudaFuncSetAttribute(flow_cell_h_kernel<NG, KIND, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return NIS_ECUDA;
        attr_smem = (int)smem;
    }
    const long long nsets = ((A.B + TCM - 1) / TCM + NG - 1) / NG;
    const int grid = (int)(nsets < sms ? nsets : sms);
    flow_cell_h_kernel<NG, KIND, MODE><<<grid, NG * TCM, smem, s>>>(F, A, hpack);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

template <int NG, int KIND>
static int h_launch(const DevFlow& F, const FwdArgs& A, const char* hpack, size_t smem, int sms, cudaStream_t s) {
    const int mode = (A.stats_layer >= 1 ? 1 : 0) | (A.zin != nullptr ? 2 : 0);
    if (A.inverse && mode == 0) return h_launch_mode<NG, KIND, 8>(F, A, hpack, smem, sms, s);
    if (A.inverse && mode == 2) return A.next_moments ? h_launch_mode<NG, KIND, 14>(F, A, hpack, smem, sms, s)
                                                      : h_launch_mode<NG, KIND, 10>(F, A, hpack, smem, sms, s);
    switch (mode) {
        case 0: return h_launch_mode<NG, KIND, 0>(F, A, hpack, smem, sms, s);
        case 1: return h_launch_mode<NG, KIND, 1>(F, A, hpack, smem, sms, s);
        case 2: return A.next_moments ? h_launch_mode<NG, KIND, 6>(F, A, hpack, smem, sms, s)
                                      : h_launch_mode<NG, KIND, 2>(F, A, hpack, smem, sms, s);
    }
    return h_launch_mode<NG, KIND, 3>(F, A, hpack, smem, sms, s);
}

int nis_launch_h(const DevFlow& F, const FwdArgs& A, const float* tcpack, cudaStream_t s) {
    static int sms = 0;
    if (sms <= 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    const bool stats = A.stats_layer >= 1;
    const int lz = A.zin ? (A.zin_layer > 0 ? A.zin_layer : (stats ? A.stats_layer - 1 : F.depth)) : 1;
    const int l_end = stats ? A.stats_layer - 1 : F.depth;
    const int ng = h_groups(F);
    const size_t smem = (size_t)h_layout(F, F.cells[A.c_begin].P, lz, l_end, A.zin != nullptr || stats, ng, A.zin == nullptr, stats).total + 1024;
    const char* hp = reinterpret_cast<const char*>(tcpack);
    if (F.kind == NIS_KIND_PWLIN) {
        switch (ng) {
            case 4: return h_launch<4, NIS_KIND_PWLIN>(F, A, hp, smem, sms, s);
            case 3: return h_launch<3, NIS_KIND_PWLIN>(F, A, hp, smem, sms, s);
            case 2: return h_launch<2, NIS_KIND_PWLIN>(F, A, hp, smem, sms, s);
        }
    } else {
        switch (ng) {
            case 3: return h_launch<3, NIS_KIND_PWQUAD>(F, A, hp, smem, sms, s);
            case 2: return h_launch<2, NIS_KIND_PWQUAD>(F, A, hp, smem, sms, s);
        }
    }
    return NIS_EUNSUPPORTED;
}
