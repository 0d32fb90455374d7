// Host-side descriptor handling for the flow kernels: validation, arena layouts, workspace carve-up, kernel plan.
#include <stdlib.h>
#include <string.h>
#include "common.cuh"
#include "flow_host.cuh"

static int cond_out(const NisFlowDesc* d) {
    return d->kind == NIS_KIND_PWLIN ? d->n_bins : (d->kind == NIS_KIND_AFFINE ? 2 : 2 * d->n_bins + 1);
}

extern "C" int64_t nis_flow_cell_param_count(const NisFlowDesc* d, int32_t c) {
    if (!d || c < 0 || c >= d->n_cells) return NIS_EINVAL;
    int P = d->cells[c].n_pass, T = d->n_flow - P, in = P;
    int64_t n = 2 * P;
    for (int l = 0; l < d->depth; ++l) { n += (int64_t)d->widths[l] * in + 2 * d->widths[l]; in = d->widths[l]; }
    n += (int64_t)T * cond_out(d) * in + (int64_t)T * cond_out(d);
    return n;
}

extern "C" int64_t nis_flow_cell_bn_count(const NisFlowDesc* d, int32_t c) {
    if (!d || c < 0 || c >= d->n_cells) return NIS_EINVAL;
    int64_t n = 2 * d->cells[c].n_pass;
    for (int l = 0; l < d->depth; ++l) n += 2 * d->widths[l];
    return n;
}

int nis_build_dev_flow(const NisFlowDesc* d, DevFlow* F) {
    if (!d || !F) return NIS_EINVAL;
    if (d->n_flow < 2 || d->n_flow > NIS_MAX_DIM) return NIS_EINVAL;
    if (d->n_cells < 1 || d->n_cells > NIS_MAX_CELLS) return NIS_EINVAL;
    if (d->kind != NIS_KIND_PWLIN && d->kind != NIS_KIND_PWQUAD && d->kind != NIS_KIND_AFFINE) return NIS_EINVAL;
    if (d->n_bins < 1 || d->n_bins > 512) return NIS_EINVAL;
    if (d->depth < 0 || d->depth > NIS_MAX_HIDDEN) return NIS_EINVAL;
    memset(F, 0, sizeof(*F));
    F->d = d->n_flow; F->n_cells = d->n_cells; F->kind = d->kind; F->nb = d->n_bins; F->depth = d->depth;
    F->K = cond_out(d); F->Kpad = pad8(F->K);
    F->eps = d->bn_eps; F->momentum = d->bn_momentum;
    int maxW = 8;
    for (int l = 0; l < d->depth; ++l) {
        if (d->widths[l] < 1 || d->widths[l] > NIS_MAX_WIDTH) return NIS_EINVAL;
        F->widths[l] = d->widths[l];
        if (pad8(d->widths[l]) > maxW) maxW = pad8(d->widths[l]);
    }
    bool seen[NIS_MAX_DIM];
    memset(seen, 0, sizeof(seen));
    for (int i = 0; i < d->n_flow; ++i) {
        int p = d->out_perm[i];
        if (p < 0 || p >= d->n_flow || seen[p]) return NIS_EINVAL;
        seen[p] = true;
        F->out_perm[i] = (uint8_t)p;
    }
    for (int c = 0; c < d->n_cells; ++c)
        if (pad8(d->cells[c].n_pass) > maxW) maxW = pad8(d->cells[c].n_pass);
    F->maxW = maxW;
    int pk = 0;
    for (int c = 0; c < d->n_cells; ++c) {
        const NisCellDesc& s = d->cells[c];
        DevCell& q = F->cells[c];
        if (s.n_pass < 1 || s.n_pass >= d->n_flow) return NIS_EINVAL;
        q.P = s.n_pass; q.T = d->n_flow - s.n_pass;
        memset(seen, 0, sizeof(seen));
        for (int i = 0; i < d->n_flow; ++i) {
            int col = i < q.P ? s.feed_idx[i] : s.trafo_idx[i - q.P];
            if (col < 0 || col >= d->n_flow || seen[col]) return NIS_EINVAL;
            seen[col] = true;
            if (i < q.P) q.feed[i] = (uint8_t)col; else q.trafo[i - q.P] = (uint8_t)col;
        }
        if (s.param_off < 0 || s.bn_off < 0) return NIS_EINVAL;
        q.param_off = s.param_off; q.bn_off = s.bn_off;
        q.pk_off = pk;
        int o = 0;
        // each layer's scale / shift block starts on its own 128-byte line: the cooperative small-batch kernels let one CTA
        // rewrite a block while the others still hold its neighbours in L1 (no stale line may be shared)
        for (int l = 0; l <= d->depth; ++l) { q.aff_off[l] = o; o += 2 * F->Wp(c, l); o = (o + 31) & ~31; }
        int in = q.P;
        for (int l = 0; l < d->depth; ++l) { q.wt_off[l] = o; o += in * pad8(d->widths[l]); in = d->widths[l]; }
        q.wo_off = o; o += q.T * in * F->Kpad;
        q.bo_off = o; o += q.T * F->Kpad;
        pk += (o + 31) & ~31;
        q.sv_off = c * (d->depth + 1) * 2 * maxW;
    }
    F->pack_total = pk;
    F->saved_total = d->n_cells * (d->depth + 1) * 2 * maxW;
    return NIS_OK;
}

extern "C" int64_t nis_flow_bn_saved_count(const NisFlowDesc* d) {
    DevFlow F;
    int rc = nis_build_dev_flow(d, &F);
    return rc ? rc : F.saved_total;
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// Smallest batches the tensor-core kernels (fp16-split, streamed-weights, both tensor-core backwards) and the register-
// tiled kernel take; smaller ones run on the kernels of the next family down.
static const int64_t TC_MIN_BATCH = 256;
static const int64_t TILED_MIN_BATCH = 2048;

// Which kernel family runs one call.  Knobs, read on every call so that a process can switch between them (the tests
// compare each family against the reference kernels this way): NIS_TC=0 disables the tensor-core forwards and backwards,
// NIS_DISABLE_TILED=1 the register-tiled forward, NIS_BWD_TC=0 both tensor-core backwards.
// The fp16-split forward and inverse take the shapes nis_tc_supported accepts.  Its own shared-memory limit (at least two
// point groups per CTA) is met by each of them: a sweep of the 6256 width-64, 32-bin PWLin and PWQuad shapes with n_flow
// 2-32, P 1-17 and depth 1-8 found none it rejects.  It would accept about five times as many shapes (for example every
// n_flow >= 10 at depth 1), which run on the streamed-weights kernel; giving them to the fp16-split kernel needs parity
// tests and B200 timings against that kernel of their own.
FlowPlan nis_flow_plan(const DevFlow& F, int64_t B, int bn_mode) {
    auto knob = [](const char* name, char value) { const char* e = getenv(name); return e && e[0] == value; };
    const bool tc = B >= TC_MIN_BATCH && !knob("NIS_TC", '0');
    const bool train = bn_mode == NIS_BN_TRAIN;
    FlowPlan p;
    if (tc && nis_tc_supported(F)) p.fwd = FWD_H;
    else if (tc && nis_wide_supported(F, bn_mode)) p.fwd = FWD_WIDE;
    else if (B >= TILED_MIN_BATCH && !knob("NIS_DISABLE_TILED", '1') && nis_tiled_supported(F)) p.fwd = FWD_TILED;
    else p.fwd = FWD_GENERIC;
    const bool bwd_tc = train && tc && !knob("NIS_BWD_TC", '0');
    if (bwd_tc && nis_bwd_tc_supported(F)) p.bwd = BWD_TC;
    else if (bwd_tc && nis_bwd_wide_supported(F)) p.bwd = BWD_WIDE;
    else p.bwd = BWD_GENERIC;
    // both sides on the wide kernels: the backward can skip the layer passes
    p.act_cache = p.fwd == FWD_WIDE && p.bwd == BWD_WIDE && F.depth >= 2;
    return p;
}

// Backward scratch (floats), see flow_bwd.cu: gradient state [B][d+1], per-CTA parameter-gradient
// partials [NIS_BWD_GRID][max cell params], BN backward sums [n_cells][depth+1][2][maxW].

size_t nis_flow_carve(const DevFlow& F, int64_t B, void* base, FlowWorkspace* ws) {
    size_t off = 0;
    char* b = (char*)base;
    ws->wpack = (float*)(b + off); off = align256(off + sizeof(float) * (size_t)F.pack_total);
    {   // tensor-core operand pack: 3xTF32 resident-weights layout (flow_bwd_tc.cu), which also holds the fp16-split one
        // (flow_tc_h.cu), or K-panels (flow_wide.cu)
        size_t fl = nis_tc_pack_floats(F), wf = nis_wide_pack_floats(F);
        ws->tcpack = (float*)(b + off); off = align256(off + sizeof(float) * (fl > wf ? fl : wf));
    }
    ws->state = (float*)(b + off); off = align256(off + sizeof(float) * (size_t)B * (F.d + 1));
    ws->partials = (double*)(b + off); off = align256(off + sizeof(double) * (size_t)NIS_MAX_GRID * 2 * F.maxW);
    ws->counter = (unsigned*)(b + off); off = align256(off + 256);
    ws->bwd = (float*)(b + off);
    ws->total = off;
    return off;
}
