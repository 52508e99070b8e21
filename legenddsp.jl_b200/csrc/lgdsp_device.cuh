// Device-side parameter blocks and small helpers shared by the kernels.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "../../include/lgdsp_b200.h"

namespace lgdsp {

// TrapezoidalChargeFilter in samples, with derived constants
struct TrapDev {
    int a, g, a2, L, nout, pad_;
    double inv1, inv2;
};

// SG kernel folded onto the inclusive prefix sum TT of the PZ waveform (summation by parts):
// s[j] = sum_k h[k] (TT[j+k+1]-TT[j+k]) = sum_{k=0}^{n_taps} gg[k] TT[j+k]
struct SgDev {
    int n_taps, offset, nout, pad_;
    double gg[LGDSP_MAX_SG + 1];
};

struct DniDev {
    int n_w, m;  // window, degree+1
};

// Structured evaluation of a CUSP/ZAC filter (see lgdsp_icpc.cu, "CUSP/ZAC through their analytic structure").
// One descriptor = one (sigma, flat, tau, L); it can emit the CUSP output (B = 0) and/or the ZAC output.
constexpr int CZ_CH = 33;  // samples per thread chunk (odd: conflict-free linear SMEM layout)
struct CzDev {
    int L, F, lt, Rn;
    int oc[4], oa[4];          // in-chunk offsets of the decimated prefix-table positions (logical order)
    // capture events of the single forward scan, sorted by sample index: after sample ev_k (-1: before the first)
    // the running causal values (kind 0: P-, D1, D2 -> tables 3*ev_tab..) or the running anti-causal partial sum
    // (kind 1 -> table 12+ev_tab) are stored
    int n_ev, ev_k[8], ev_kind[8], ev_tab[8];
    double ev_pw[8];           // carry multiplier: rho^(oc+1) (causal) / rho^(CH-oa) (anti-causal)
    double ev_rinv[8];         // anti-causal: rho^(-oa)
    double r, rho, rho_inv, inv_sigma;
    double cA, cA_rho_lt, cA_rhoinv_lt, cA_rhoinv_Rn, cA_rho_Rn;   // recurrence input gains (cA = a/2)
    double rho_lt, rho_Rn, cA_rhoinv_ltm1, cA_rho;                 // closed-form initial states
    double rho_ch_pow[5];      // rho^(CH*2^s)
    double rho_lane[32];       // rho^(CH*(lane+1))
    double rho_warp;           // rho^(CH*32)
    double h2, B, lt_d, lt2_d, Rn_d, Rn2_d;
    double g, gclast_cusp, gclast_zac;  // output gain, g*r*c[L-1] of the cusp / zac shape
    double lip_cusp, lip_zac;           // sum_k |h[k]-h[k-1]| of the zero-extended FIR taps: |out[j+1]-out[j]| <= lip * max|y|
};

// kernel-argument block of the fused dsp_icpc kernel (lives in the constant bank, ~2 KB)
struct IcpcDev {
    int n;
    unsigned groups;
    double t_first, dt;
    int sat_low, sat_high;  // -1: can never match a uint16 sample
    int bl_from, bl_until, tail_from, tail_until;
    double km1;
    double bl_inv_n;        // 1/(number of baseline-window samples), as the reference's inv_n
    double tail_inv_n;      // same for the tail window
    double bl_sX, bl_sXX, tail_sX, tail_sXX;   // sum of X and X^2 (X = time of the sample) over the two windows
    TrapDev t0, t0inv, e10410, e535, e313, etrap;
    int t0inv_same, t0_min_n, tx_min_n, direct;
    double t0_thr;
    double tx_frac[5];
    double qd_first, qd_last, lq_first, lq_last;
    DniDev int_dni, sig_dni;
    double trap_pick, cusp_pick, zac_pick;
    SgDev sg[3];
    int cur_from[4], cur_until[4];
    int sg_alias[4];           // sg_alias[f] >= 0: filter f (taps and window) is identical to that earlier filter
    double nsigma;
    double intr_inv_n;      // 1/(samples of the in-trace sigma window)
    int intr_min_n, intr_from, intr_until, pad0;
    int cusp_L, zac_L;
    int cz_shared, pad1;   // 1: cusp and zac share (sigma, flat, tau, L) -> one structured pass emits both
    CzDev cz[2];           // [0]: cusp (or shared), [1]: zac
    // global-memory tables (owned by the handle):
    const double* dni_A;    // [2][LGDSP_MAX_DNI*4]: int_dni, sig_dni fit matrices
    const double* cusp_g;   // differenced CUSP taps on TT, cusp_L+1 values
    const double* zac_g;    // differenced ZAC taps on TT, zac_L+1 values
};


// ---- TMA 1-D bulk copy + mbarrier (sm_90+/sm_100a): SASS UBLKCP / SYNCS ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// hint: bring `bytes` (multiple of 16, 16-byte aligned source) into L2 ahead of a later bulk copy
__device__ __forceinline__ void tma_prefetch_l2(const void* src_gmem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t phase)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(phase)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase)
{
    while (!mbar_try_wait(bar, phase)) {}
}

// ---- cp.async (LDGSTS): 8-byte copies global -> shared, completed by commit / wait groups of the issuing thread ----
__device__ __forceinline__ void cp_async_8(void* dst_smem, const void* src_gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- warp / block reductions (results broadcast to all threads) ----
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const double w = __shfl_xor_sync(FULL, v, o); v = w > v ? w : v; }   // (fmax() costs 2x: NaN handling)
    return v;
}
__device__ __forceinline__ double warp_min(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const double w = __shfl_xor_sync(FULL, v, o); v = w < v ? w : v; }
    return v;
}
// (value, index) maximum with FIRST index on ties
__device__ __forceinline__ void warp_argmax(double& v, int& i)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ov = __shfl_xor_sync(FULL, v, o);
        int oi = __shfl_xor_sync(FULL, i, o);
        if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
    }
}

// explicit round-to-nearest ops that the compiler never contracts into FMAs (scalar statistics formulas follow
// the reference's operation order: src/tailstats.jl:54-70)
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }

}  // namespace lgdsp
