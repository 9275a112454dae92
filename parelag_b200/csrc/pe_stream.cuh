// pe_stream.cuh -- device helpers shared by the streaming kernels (pe_sell.cu) and the
// persistent program kernel (pe_prog.cu).
#pragma once
#include <stdint.h>
#include "../../include/parelag_b200.h"

// Matrix streams are read once per pass: no L1 allocation, and an L2 evict-first policy so
// that the vectors (u, f, l1 -- re-read by every colour) are what stays resident in L2.
__device__ __forceinline__ uint64_t l2_evict_first_policy()
{
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ double ld_stream_f64(const double *p, uint64_t pol)
{
    double v;
    asm("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ int ld_stream_s32(const int *p, uint64_t pol)
{
    int v;
    asm("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}

// "Prologue" variants: volatile, so the compiler keeps them ahead of griddepcontrol.wait (pdl_wait)
// -- they fetch immutable matrix data while the preceding kernel is still draining.
__device__ __forceinline__ double ld_stream_f64_pro(const double *p, uint64_t pol)
{
    double v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ int ld_stream_s32_pro(const int *p, uint64_t pol)
{
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
// sign-encoded SELL values (-1, 0, +1 stored as int8): decoded to the same double
__device__ __forceinline__ double ld_stream_s8(const int8_t *p, uint64_t pol)
{
    int v;
    asm("ld.global.nc.L1::no_allocate.L2::cache_hint.s8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return (double)v;
}
__device__ __forceinline__ double ld_stream_s8_pro(const int8_t *p, uint64_t pol)
{
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return (double)v;
}
__device__ __forceinline__ int ld_nc_s32_pro(const int *p)
{
    int v;
    asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double ld_nc_f64_pro(const double *p)
{
    double v;
    asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

// scalar recurrences of mfem::CGSolver::Mult, one phase per call (single thread)
//  phase 0: DOT = (d, r) before the loop        phase 1: DOT = (z, d) before the loop
//  phase 2: DOT = (r, z) in iteration `iter`    phase 3: DOT = (d, z) in iteration `iter`
// As in mfem (and KrylovSolver::Mult on the host): a negative initial (B r, r) stops at once (FetchStats
// reports it as the final norm, unsquared); a negative (Ad, d) continues with a negative step; only an
// exact zero (Ad, d) stops, unconverged, with final_iter the iteration that computed it.
__device__ __forceinline__ void pe_pcg_scalar_step_dev(double *s, int phase, int iter, int max_iter, double rel, double abs_tol)
{
    const double dot = s[PE_PCG_DOT];
    bool done = s[PE_PCG_DONE] != 0.0;
    if (phase == 0)
    {
        s[PE_PCG_NOM] = s[PE_PCG_NOM0] = s[PE_PCG_BETANOM] = dot;
        s[PE_PCG_HIST] = dot; s[PE_PCG_NHIST] = 1.0;
        s[PE_PCG_CONVERGED] = 0.0; s[PE_PCG_FINAL_ITER] = 0.0; s[PE_PCG_ALPHA] = 0.0; s[PE_PCG_BETA] = 0.0;
        const double r0 = fmax(dot * rel * rel, abs_tol * abs_tol);
        s[PE_PCG_R0] = r0;
        done = false;
        if (dot < 0.0) done = true;
        else if (dot <= r0) { done = true; s[PE_PCG_CONVERGED] = 1.0; }
    }
    else if (phase == 1)
    {
        if (!done)
        {
            s[PE_PCG_DEN] = dot;
            if (dot == 0.0) done = true;
            else s[PE_PCG_ALPHA] = s[PE_PCG_NOM] / dot;
        }
    }
    else if (phase == 2)
    {
        if (!done)
        {
            s[PE_PCG_BETANOM] = dot;
            s[PE_PCG_HIST + iter] = dot; s[PE_PCG_NHIST] = (double)(iter + 1);
            if (dot < s[PE_PCG_R0]) { done = true; s[PE_PCG_CONVERGED] = 1.0; s[PE_PCG_FINAL_ITER] = (double)iter; }
            else if (iter + 1 > max_iter) { done = true; s[PE_PCG_FINAL_ITER] = (double)max_iter; }
            else s[PE_PCG_BETA] = dot / s[PE_PCG_NOM];
        }
    }
    else
    {
        if (!done)
        {
            s[PE_PCG_DEN] = dot;
            if (dot == 0.0) { done = true; s[PE_PCG_FINAL_ITER] = (double)(iter + 1); }
            else { s[PE_PCG_NOM] = s[PE_PCG_BETANOM]; s[PE_PCG_ALPHA] = s[PE_PCG_BETANOM] / dot; }
        }
    }
    if (done) { s[PE_PCG_ALPHA] = 0.0; s[PE_PCG_BETA] = 0.0; }
    s[PE_PCG_DONE] = done ? 1.0 : 0.0;
}
