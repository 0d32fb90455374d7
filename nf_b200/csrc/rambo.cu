// RAMBO-on-diet 2 -> n: momenta + Jacobian weight + pT / deltaR / rapidity cuts in one pass.
// One thread per event, float64.  The uniforms of a 128-event tile are staged through shared memory
// with coalesced 16-byte loads and the momenta tile is written back the same way; rows are padded to
// an odd number of doubles so the per-thread row accesses are bank-conflict free.
// Reference: nisrep/PhaseSpace/flat_phase_space_generator.py:139-308 (see rambo_core.cuh).
#include <math.h>
#include <stdlib.h>
#include "common.cuh"
#include "rambo_core.cuh"

#define RAMBO_NT 128
#ifndef RAMBO_CTAS
#define RAMBO_CTAS 7
#endif

// doubles of a thread's momenta row: with PDFs the whole event (beams + final state, the beam slots double as the cut
// scratch); without, the beams are constants the kernel stores itself and the row is [n scratch | 4n final state]
__host__ __device__ static inline int rambo_row_doubles(int n, bool pdf) { return pdf ? (n + 2) * 4 : 5 * n; }

// seven CTAs per SM (what the shared-memory rows of a 2 -> 4 event allow: 9 + 21 doubles per thread): without the bound
// ptxas takes 255 registers for the inlined event variants and the kernel runs at half speed
template <typename RT>
__global__ void __launch_bounds__(RAMBO_NT, RAMBO_CTAS) rambo_kernel(const __grid_constant__ RamboConst C, const RT* __restrict__ r,
                                                         double* __restrict__ momenta, double* __restrict__ weight,
                                                         uint8_t* __restrict__ cutmask, long long B) {
    const int ND = 3 * C.n - 4 + (C.pdf_active ? 2 : 0);    // uniforms per event
    const int NDP = ND | 1;                 // odd row stride (doubles): conflict-free per-thread rows
    const int NM = (C.n + 2) * 4;           // momentum components per event
    const int NMP = rambo_row_doubles(C.n, C.pdf_active != 0) | 1;
    extern __shared__ __align__(16) double smd[];
    double* rs = smd;                       // [NT][NDP]
    double* mo = smd + RAMBO_NT * NDP;      // [NT][NMP]  (scratch even when momenta are not requested)
    const int tid = threadIdx.x;
    // the kinematics are needed for the momenta and for the cuts; a weight-only call without cuts stops after the masses
    const bool kin = momenta != nullptr || C.pT_min > 0.0 || C.dR_min > 0.0 || C.rap_max > 0.0;
    const long long ntiles = (B + RAMBO_NT - 1) / RAMBO_NT;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long base = tile * RAMBO_NT;
        const int cnt = (int)((B - base) < RAMBO_NT ? (B - base) : RAMBO_NT);
        if (tid < cnt) {
            // this thread's uniforms: one contiguous row, loaded 16 bytes at a time where the row allows it; it is
            // staged in the thread's own (odd-stride) shared-memory row only because rambo_event indexes it at run time
            const RT* src = r + (base + tid) * ND;
            double* row = rs + tid * NDP;
            if (sizeof(RT) == 8 && (ND & 1) == 0) {
                for (int i = 0; i < ND; i += 2) {
                    const double2 v = *reinterpret_cast<const double2*>(reinterpret_cast<const double*>(src) + i);
                    row[i] = v.x; row[i + 1] = v.y;
                }
            } else if (sizeof(RT) == 4 && (ND & 3) == 0) {
                for (int i = 0; i < ND; i += 4) {
                    const float4 v = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(src) + i);
                    row[i] = (double)v.x; row[i + 1] = (double)v.y; row[i + 2] = (double)v.z; row[i + 3] = (double)v.w;
                }
            } else {
                for (int i = 0; i < ND; ++i) row[i] = (double)src[i];
            }
            double w;
            uint8_t pass;
            if (C.pdf_active) {
                if (kin) rambo_event<true, true>(C, row, 1, mo + tid * NMP, 1, w, pass);
                else rambo_event<false, true>(C, row, 1, mo + tid * NMP, 1, w, pass);
            } else if (kin) rambo_event<true, false, false>(C, row, 1, mo + tid * NMP, 1, w, pass);
            else rambo_event<false, false, false>(C, row, 1, mo + tid * NMP, 1, w, pass);
            weight[base + tid] = w;
            if (cutmask) cutmask[base + tid] = pass;
        }
        if (momenta && tid < cnt) {
            // every thread writes its own event: (n+2)*4 doubles = a whole number of 32-byte sectors, one 256-bit store
            // each (st.global.v4.f64), read back from the thread's own odd-stride shared-memory row - no staging pass,
            // no barrier (the cooperative 16-byte copy-out was ~10 % of the kernel's instructions)
            const double* srow = mo + tid * NMP;
            double* dst = momenta + (base + tid) * NM;
            int c0 = 0;
            if (!C.pdf_active) {                                   // the beams straight from the launch constants
                asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};"
                             :: "l"(dst), "d"(C.beam[0][0]), "d"(C.beam[0][1]), "d"(C.beam[0][2]), "d"(C.beam[0][3]) : "memory");
                asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};"
                             :: "l"(dst + 4), "d"(C.beam[1][0]), "d"(C.beam[1][1]), "d"(C.beam[1][2]), "d"(C.beam[1][3]) : "memory");
                srow += C.n - 8;                                   // final state at srow[n ..): component c of the event at srow[c - 8 + n]
                c0 = 8;
            }
            for (int c = c0; c < NM; c += 4)
                asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};"
                             :: "l"(dst + c), "d"(srow[c]), "d"(srow[c + 1]), "d"(srow[c + 2]), "d"(srow[c + 3]) : "memory");
        }
    }
}

template <typename RT>
static int rambo_launch(const RamboConst& C, const void* r, double* momenta, double* weight, uint8_t* cutmask,
                        long long B, cudaStream_t s) {
    const int NDP = (3 * C.n - 4 + (C.pdf_active ? 2 : 0)) | 1, NMP = rambo_row_doubles(C.n, C.pdf_active != 0) | 1;
    const size_t smem = sizeof(double) * RAMBO_NT * (NDP + NMP);
    NIS_ENSURE_SMEM((rambo_kernel<RT>), (int)smem);
    long long ntiles = (B + RAMBO_NT - 1) / RAMBO_NT;
    // one resident wave: every CTA strides over the same number of tiles (+-1), no partial last wave
    const int sms = nis_sm_count();
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rambo_kernel<RT>, RAMBO_NT, smem) != cudaSuccess || per_sm < 1)
        per_sm = 4;
    const long long wave = (long long)sms * per_sm;
    int grid = (int)(ntiles < wave ? ntiles : wave);
    rambo_kernel<RT><<<grid, RAMBO_NT, smem, s>>>(C, (const RT*)r, momenta, weight, cutmask, B);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}

extern "C" int nis_rambo_generate(const NisRamboDesc* desc, const void* r, int32_t r_dtype, double* momenta,
                                  double* weight, uint8_t* cutmask, int64_t B, void* stream) {
    if (!desc || B < 0 || (B > 0 && (!r || !weight))) return NIS_EINVAL;
    if (r_dtype != NIS_F32 && r_dtype != NIS_F64) return NIS_EINVAL;
    // rows of uniforms are read 16 bytes at a time, events are written 32 bytes at a time
    if ((reinterpret_cast<uintptr_t>(r) & 15) || (reinterpret_cast<uintptr_t>(momenta) & 31)) return NIS_EINVAL;
    RamboConst C;
    int rc = rambo_fill_const(desc, &C);
    if (rc) return rc;
    if (B == 0) return NIS_OK;
    cudaStream_t s = (cudaStream_t)stream;
    return r_dtype == NIS_F64 ? rambo_launch<double>(C, r, momenta, weight, cutmask, B, s)
                              : rambo_launch<float>(C, r, momenta, weight, cutmask, B, s);
}


// ---- inverse map: one thread per event, momenta read straight from global memory (32-byte vectors), the recovered
//      uniforms kept in a local row until the weight is evaluated on them ---------------------------------------------
__global__ void __launch_bounds__(128) rambo_invert_kernel(const __grid_constant__ RamboConst C, const double* __restrict__ momenta,
                                                           double* __restrict__ r, double* __restrict__ weight, long long B) {
    const int n = C.n, ND = 3 * n - 4, NM = (n + 2) * 4;
    for (long long ev = (long long)blockIdx.x * blockDim.x + threadIdx.x; ev < B; ev += (long long)gridDim.x * blockDim.x) {
        double fin[NIS_MAX_FINAL * 4], row[3 * NIS_MAX_FINAL - 4];
        const double* src = momenta + ev * NM + 8;                 // final state after the two beams
        for (int i = 0; i < 4 * n; i += 4) {
            double a, b, c, d;
            asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(src + i));
            fin[i] = a; fin[i + 1] = b; fin[i + 2] = c; fin[i + 3] = d;
        }
        double w;
        rambo_invert_event(C, fin, 1, row, 1, w);
        for (int i = 0; i < ND; ++i) r[ev * ND + i] = row[i];
        if (weight) weight[ev] = w;
    }
}

extern "C" int nis_rambo_invert(const NisRamboDesc* desc, const double* momenta, double* r, double* weight, int64_t B, void* stream) {
    if (!desc || B < 0 || (B > 0 && (!momenta || !r))) return NIS_EINVAL;
    if (desc->pdf_active) return NIS_EUNSUPPORTED;
    if (reinterpret_cast<uintptr_t>(momenta) & 31) return NIS_EINVAL;      // events are read 32 bytes at a time
    RamboConst C;
    int rc = rambo_fill_const(desc, &C);
    if (rc) return rc;
    if (B == 0) return NIS_OK;
    const long long blocks = (B + 127) / 128;
    const int grid = (int)(blocks < 148 * 16 ? blocks : 148 * 16);
    rambo_invert_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(C, momenta, r, weight, B);
    NIS_CUDA_CHECK_LAUNCH();
    return NIS_OK;
}
