// Register-resident splines shared by the tensor-core forward kernels (flow_tc.cu, flow_tc_h.cu).
#pragma once
#include "spline.cuh"

// PWQuad with 32 bins on a register-resident logit vector z[0..64] (33 vertex heights, 32 widths): the
// reference's map (coupling_cells.py:167-225, see spline.cuh::pwquad_fwd) with static indexing only — the bin
// is found by counting edges, the per-bin quantities by predicated accumulation.
__device__ __forceinline__ void pwquad32_regs(const float* z, float x, float& y, float& f, int& kbin) {
    float mv = z[0], mw = z[33];
#pragma unroll
    for (int j = 1; j <= 32; ++j) mv = fmaxf(mv, z[j]);
#pragma unroll
    for (int j = 1; j < 32; ++j) mw = fmaxf(mw, z[33 + j]);
    float w[32], v[33];
    double Sw = 0.0;
#pragma unroll
    for (int j = 0; j < 32; ++j) { w[j] = expf(z[33 + j] - mw); Sw += (double)w[j]; }
#pragma unroll
    for (int j = 0; j <= 32; ++j) v[j] = expf(z[j] - mv);
    double Araw = 0.0;
#pragma unroll
    for (int j = 0; j < 32; ++j) Araw += 0.5 * ((double)v[j] + (double)v[j + 1]) * (double)w[j];
    const float xb = x > NIS_QUAD_CLAMP ? NIS_QUAD_CLAMP : x;
    const double target = (double)xb * Sw;
    int k = 0;
    double cum = 0.0;
#pragma unroll
    for (int j = 0; j < 31; ++j) { cum += (double)w[j]; k += cum <= target ? 1 : 0; }
    double cw = 0.0, ca = 0.0;
    float wk = 0.f, vk = 0.f, vk1 = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const bool below = j < k;
        cw += below ? (double)w[j] : 0.0;
        ca += below ? 0.5 * ((double)v[j] + (double)v[j + 1]) * (double)w[j] : 0.0;
        wk = j == k ? w[j] : wk;
        vk = j == k ? v[j] : vk;
        vk1 = j == k ? v[j + 1] : vk1;
    }
    const float invA = (float)(Sw / Araw);
    const float alpha = (float)((target - cw) / (double)wk);
    const float Vk = vk * invA, Vk1 = vk1 * invA;
    const float Wk = (float)((double)wk / Sw);
    y = alpha * alpha * 0.5f * (Vk1 - Vk) * Wk + alpha * Vk * Wk + (float)(ca / Araw);
    f = Vk + alpha * (Vk1 - Vk);
    kbin = k;
}


// ---- round 2: the same map with pairwise trees and a binary descent -----------------------------------------------------
// pwquad32_regs above spends ~920 instructions per transformed dimension, ~400 of them float64 (running sums of the widths
// and of the trapezoids, 31 float64 compares, two predicated float64 accumulations per bin, four float64 divisions): the
// PWQuad final pass was 2.0 ms per cell against 0.41 ms for PWLin.  Here only what 1/W_k amplifies stays float64 - the sum
// of the widths below the bin, from a pairwise tree of float64 partial sums - and the bin is found by descending that tree
// (5 compares).  The trapezoid sums (no amplification: they enter y and the normalisation directly) are a float32 tree; the
// per-bin quantities are picked by select trees along the bits of the bin index; the divisions are float32.
// LOG2: the logits are in units of log 2 (bare ex2).
__device__ __forceinline__ float tcs_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// element `i` (bits b3 b2 b1 b0, b0 the least significant) of 16 values at stride `st` of a register array
template <typename T>
__device__ __forceinline__ T tcs_sel16(const T* a, int st, bool b3, bool b2, bool b1, bool b0) {
    T s8[8], s4[4], s2[2];
#pragma unroll
    for (int i = 0; i < 8; ++i) s8[i] = b0 ? a[(2 * i + 1) * st] : a[2 * i * st];
#pragma unroll
    for (int i = 0; i < 4; ++i) s4[i] = b1 ? s8[2 * i + 1] : s8[2 * i];
#pragma unroll
    for (int i = 0; i < 2; ++i) s2[i] = b2 ? s4[2 * i + 1] : s4[2 * i];
    return b3 ? s2[1] : s2[0];
}
template <typename T>
__device__ __forceinline__ T tcs_sel8(const T* a, int st, bool b2, bool b1, bool b0) {
    T s4[4], s2[2];
#pragma unroll
    for (int i = 0; i < 4; ++i) s4[i] = b0 ? a[(2 * i + 1) * st] : a[2 * i * st];
#pragma unroll
    for (int i = 0; i < 2; ++i) s2[i] = b1 ? s4[2 * i + 1] : s4[2 * i];
    return b2 ? s2[1] : s2[0];
}
template <typename T>
__device__ __forceinline__ T tcs_sel4(const T* a, int st, bool b1, bool b0) {
    const T lo = b0 ? a[st] : a[0], hi = b0 ? a[3 * st] : a[2 * st];
    return b1 ? hi : lo;
}

template <bool LOG2>
__device__ __forceinline__ void pwquad32_tree(const float* z, float x, float& y, float& f, int& kbin) {
    float mv = z[0], mw = z[33];
#pragma unroll
    for (int j = 1; j <= 32; ++j) mv = fmaxf(mv, z[j]);
#pragma unroll
    for (int j = 1; j < 32; ++j) mw = fmaxf(mw, z[33 + j]);
    float w[32], v[33], a[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) w[j] = LOG2 ? tcs_ex2(z[33 + j] - mw) : __expf(z[33 + j] - mw);
#pragma unroll
    for (int j = 0; j <= 32; ++j) v[j] = LOG2 ? tcs_ex2(z[j] - mv) : __expf(z[j] - mv);
#pragma unroll
    for (int j = 0; j < 32; ++j) a[j] = (v[j] + v[j + 1]) * (0.5f * w[j]);              // trapezoid j (raw widths)
    double W1[16], W2[8], W4[4];
    float A1[16], A2[8], A4[4];
#pragma unroll
    for (int j = 0; j < 16; ++j) { W1[j] = (double)w[2 * j] + (double)w[2 * j + 1]; A1[j] = a[2 * j] + a[2 * j + 1]; }
#pragma unroll
    for (int j = 0; j < 8; ++j) { W2[j] = W1[2 * j] + W1[2 * j + 1]; A2[j] = A1[2 * j] + A1[2 * j + 1]; }
#pragma unroll
    for (int j = 0; j < 4; ++j) { W4[j] = W2[2 * j] + W2[2 * j + 1]; A4[j] = A2[2 * j] + A2[2 * j + 1]; }
    const double W8a = W4[0] + W4[1], W8b = W4[2] + W4[3];
    const float A8a = A4[0] + A4[1], A8b = A4[2] + A4[3];
    const double Sw = W8a + W8b;
    const float Araw = A8a + A8b;
    const float xb = x > NIS_QUAD_CLAMP ? NIS_QUAD_CLAMP : x;
    const double target = (double)xb * Sw;
    // bin = number of right edges E_1..E_32 <= xb (coupling_cells.py:199-202) = the leaf the descent ends on: at a node
    // whose left half sums to L, go right iff base + L <= target
    const bool b4 = W8a <= target;
    double base = b4 ? W8a : 0.0;
    float abase = b4 ? A8a : 0.f;
    {
        const double L = b4 ? W4[2] : W4[0];
        const float La = b4 ? A4[2] : A4[0];
        const bool g = base + L <= target;
        base = g ? base + L : base;
        abase = g ? abase + La : abase;
        kbin = g ? 8 : 0;
    }
    const bool b3 = kbin != 0;
    {
        const double L = tcs_sel4(W2, 2, b4, b3);                       // W2[2 * (2 b4 + b3)]
        const float La = tcs_sel4(A2, 2, b4, b3);
        const bool g = base + L <= target;
        base = g ? base + L : base;
        abase = g ? abase + La : abase;
        kbin += g ? 4 : 0;
    }
    const bool b2 = (kbin & 4) != 0;
    {
        const double L = tcs_sel8(W1, 2, b4, b3, b2);                   // W1[2 * (4 b4 + 2 b3 + b2)]
        const float La = tcs_sel8(A1, 2, b4, b3, b2);
        const bool g = base + L <= target;
        base = g ? base + L : base;
        abase = g ? abase + La : abase;
        kbin += g ? 2 : 0;
    }
    const bool b1 = (kbin & 2) != 0;
    // pair i = 8 b4 + 4 b3 + 2 b2 + b1: widths w[2i], w[2i+1], trapezoid a[2i], heights v[2i], v[2i+1], v[2i+2]
    const float w0 = tcs_sel16(w, 2, b4, b3, b2, b1), w1 = tcs_sel16(w + 1, 2, b4, b3, b2, b1);
    const float a0 = tcs_sel16(a, 2, b4, b3, b2, b1);
    const float v0 = tcs_sel16(v, 2, b4, b3, b2, b1), v1 = tcs_sel16(v + 1, 2, b4, b3, b2, b1), v2 = tcs_sel16(v + 2, 2, b4, b3, b2, b1);
    const bool b0 = base + (double)w0 <= target;
    base = b0 ? base + (double)w0 : base;
    abase = b0 ? abase + a0 : abase;
    kbin = (b4 ? 16 : 0) + kbin + (b0 ? 1 : 0);
    const float wk = b0 ? w1 : w0, vk = b0 ? v1 : v0, vk1 = b0 ? v2 : v1;
    const float Swf = (float)Sw;
    const float invA = Swf / Araw;                                        // 1/A, A = Araw / Sw
    const float alpha = (float)(target - base) / wk;                      // (x Sw - sum_{j<k} w_j) / w_k: float64 difference
    const float Vk = vk * invA, Vk1 = vk1 * invA;
    const float Wk = wk / Swf;
    y = alpha * alpha * 0.5f * (Vk1 - Vk) * Wk + alpha * Vk * Wk + abase / Araw;
    f = Vk + alpha * (Vk1 - Vk);
}

// ---- inverse maps (nis_flow_inverse on the fp16-split kernel) -----------------------------------------------------------
// PWLin with 32 bins: y -> x on the logits z[0..31] (units of log 2, m = their maximum).  The exponentials and the pairwise
// sum tree are the forward's (flow_tc_h.cu); descending the tree with target = y S (at a node whose left half sums to L, go
// right iff base + L <= target) gives the largest k with C_k <= target and adds the same nodes in the same order as the
// forward's descent along the bits of k, so C_k is bit-identical to the forward's and a round trip lands in the forward's
// bin except right at an edge.  x = (k + (target - C_k) / e_k) / 32; jinv = S / (32 e_k) = 1 / (the bin's density).
__device__ __forceinline__ void pwlin32_tree_inv(const float* z, float m, float y, float& x, float& jinv, int& kbin) {
    float e[32], s1[16], s2[8], s4[4];
#pragma unroll
    for (int j = 0; j < 32; ++j) e[j] = tcs_ex2(z[j] - m);
#pragma unroll
    for (int j = 0; j < 16; ++j) s1[j] = e[2 * j] + e[2 * j + 1];
#pragma unroll
    for (int j = 0; j < 8; ++j) s2[j] = s1[2 * j] + s1[2 * j + 1];
#pragma unroll
    for (int j = 0; j < 4; ++j) s4[j] = s2[2 * j] + s2[2 * j + 1];
    const float s8a = s4[0] + s4[1], s8b = s4[2] + s4[3];
    const float S = s8a + s8b;
    const float target = y * S;
    const bool b4 = s8a <= target;
    float C = b4 ? s8a : 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) e[j] = b4 ? e[16 + j] : e[j];
#pragma unroll
    for (int j = 0; j < 8; ++j) s1[j] = b4 ? s1[8 + j] : s1[j];
#pragma unroll
    for (int j = 0; j < 4; ++j) s2[j] = b4 ? s2[4 + j] : s2[j];
#pragma unroll
    for (int j = 0; j < 2; ++j) s4[j] = b4 ? s4[2 + j] : s4[j];
    const bool b3 = C + s4[0] <= target;
    C = b3 ? C + s4[0] : C;
#pragma unroll
    for (int j = 0; j < 8; ++j) e[j] = b3 ? e[8 + j] : e[j];
#pragma unroll
    for (int j = 0; j < 4; ++j) s1[j] = b3 ? s1[4 + j] : s1[j];
#pragma unroll
    for (int j = 0; j < 2; ++j) s2[j] = b3 ? s2[2 + j] : s2[j];
    const bool b2 = C + s2[0] <= target;
    C = b2 ? C + s2[0] : C;
#pragma unroll
    for (int j = 0; j < 4; ++j) e[j] = b2 ? e[4 + j] : e[j];
#pragma unroll
    for (int j = 0; j < 2; ++j) s1[j] = b2 ? s1[2 + j] : s1[j];
    const bool b1 = C + s1[0] <= target;
    C = b1 ? C + s1[0] : C;
    const float e0 = b1 ? e[2] : e[0], e1 = b1 ? e[3] : e[1];
    const bool b0 = C + e0 <= target;
    C = b0 ? C + e0 : C;
    const float ek = b0 ? e1 : e0;
    kbin = (b4 ? 16 : 0) + (b3 ? 8 : 0) + (b2 ? 4 : 0) + (b1 ? 2 : 0) + (b0 ? 1 : 0);
    // (fmaxf first: a NaN from e_k = 0 becomes 0)
    x = fminf(fmaxf(((float)kbin + (target - C) / ek) * (1.f / 32.f), 0.f), 1.f);
    jinv = S / (32.f * ek);
}

// PWQuad with 32 bins: y -> x on z[0..64] (33 heights, 32 widths; units of log 2 when LOG2), the inverse of pwquad32_tree.
// The bin is found by descending the float32 trapezoid-area tree with target y A_raw (the largest k with S_k <= y, as
// spline.cuh::pwquad_inv); E_k Sw is picked from the float64 width tree along the same bits.  Inside the bin
// y - S_k = alpha V_k W_k + alpha^2 (V_{k+1} - V_k) W_k / 2, scaled by A_raw: c = target - A_k, b = v_k w_k,
// a = (v_{k+1} - v_k) w_k / 2, alpha = 2c / (b + sqrt(b^2 + 4ac)) (no cancellation for a < 0).  x = (E_k Sw + alpha w_k) / Sw,
// jinv = 1 / f with f = V_k + alpha (V_{k+1} - V_k).  The forward reads x only up to NIS_QUAD_CLAMP, so x is clamped there.
template <bool LOG2>
__device__ __forceinline__ void pwquad32_tree_inv(const float* z, float y, float& x, float& jinv, int& kbin) {
    float mv = z[0], mw = z[33];
#pragma unroll
    for (int j = 1; j <= 32; ++j) mv = fmaxf(mv, z[j]);
#pragma unroll
    for (int j = 1; j < 32; ++j) mw = fmaxf(mw, z[33 + j]);
    float w[32], v[33], a[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) w[j] = LOG2 ? tcs_ex2(z[33 + j] - mw) : __expf(z[33 + j] - mw);
#pragma unroll
    for (int j = 0; j <= 32; ++j) v[j] = LOG2 ? tcs_ex2(z[j] - mv) : __expf(z[j] - mv);
#pragma unroll
    for (int j = 0; j < 32; ++j) a[j] = (v[j] + v[j + 1]) * (0.5f * w[j]);
    double W1[16], W2[8], W4[4];
    float A1[16], A2[8], A4[4];
#pragma unroll
    for (int j = 0; j < 16; ++j) { W1[j] = (double)w[2 * j] + (double)w[2 * j + 1]; A1[j] = a[2 * j] + a[2 * j + 1]; }
#pragma unroll
    for (int j = 0; j < 8; ++j) { W2[j] = W1[2 * j] + W1[2 * j + 1]; A2[j] = A1[2 * j] + A1[2 * j + 1]; }
#pragma unroll
    for (int j = 0; j < 4; ++j) { W4[j] = W2[2 * j] + W2[2 * j + 1]; A4[j] = A2[2 * j] + A2[2 * j + 1]; }
    const double W8a = W4[0] + W4[1], W8b = W4[2] + W4[3];
    const float A8a = A4[0] + A4[1], A8b = A4[2] + A4[3];
    const double Sw = W8a + W8b;
    const float Araw = A8a + A8b;
    const float target = y * Araw;
    const bool b4 = A8a <= target;
    double base = b4 ? W8a : 0.0;
    float abase = b4 ? A8a : 0.f;
    {
        const double L = b4 ? W4[2] : W4[0];
        const float La = b4 ? A4[2] : A4[0];
        const bool g = abase + La <= target;
        base = g ? base + L : base;
        abase = g ? abase + La : abase;
        kbin = g ? 8 : 0;
    }
    const bool b3 = kbin != 0;
    {
        const double L = tcs_sel4(W2, 2, b4, b3);
        const float La = tcs_sel4(A2, 2, b4, b3);
        const bool g = abase + La <= target;
        base = g ? base + L : base;
        abase = g ? abase + La : abase;
        kbin += g ? 4 : 0;
    }
    const bool b2 = (kbin & 4) != 0;
    {
        const double L = tcs_sel8(W1, 2, b4, b3, b2);
        const float La = tcs_sel8(A1, 2, b4, b3, b2);
        const bool g = abase + La <= target;
        base = g ? base + L : base;
        abase = g ? abase + La : abase;
        kbin += g ? 2 : 0;
    }
    const bool b1 = (kbin & 2) != 0;
    const float w0 = tcs_sel16(w, 2, b4, b3, b2, b1), w1 = tcs_sel16(w + 1, 2, b4, b3, b2, b1);
    const float a0 = tcs_sel16(a, 2, b4, b3, b2, b1);
    const float v0 = tcs_sel16(v, 2, b4, b3, b2, b1), v1 = tcs_sel16(v + 1, 2, b4, b3, b2, b1), v2 = tcs_sel16(v + 2, 2, b4, b3, b2, b1);
    const bool b0 = abase + a0 <= target;
    base = b0 ? base + (double)w0 : base;
    abase = b0 ? abase + a0 : abase;
    kbin = (b4 ? 16 : 0) + kbin + (b0 ? 1 : 0);
    const float wk = b0 ? w1 : w0, vk = b0 ? v1 : v0, vk1 = b0 ? v2 : v1;
    const float c = fmaxf(target - abase, 0.f);
    const float qa = 0.5f * (vk1 - vk) * wk, qb = vk * wk;
    const float disc = fmaxf(fmaf(qb, qb, 4.f * qa * c), 0.f);
    // (fmaxf first: a NaN from 0 / 0 becomes 0)
    const float alpha = fminf(fmaxf(2.f * c / (qb + sqrtf(disc)), 0.f), 1.f);
    const float Swf = (float)Sw;
    x = fminf(fmaxf((float)(base + (double)(alpha * wk)) / Swf, 0.f), NIS_QUAD_CLAMP);
    jinv = Araw / ((vk + alpha * (vk1 - vk)) * Swf);
}
