// Trapezoid sweeps, ONE WARP per waveform: dsp_trap_rt_optimization / dsp_trap_ft_optimization and the (rt, ft) grid
// (/root/reference/src/dsp_filter_optimization.jl:102-133, 241-274).  Included by lgdsp_icpc.cu.
//
// sweep_kernel (one CTA per waveform) spends a quarter of its time in block barriers between phases that are too short
// to amortise them, and builds the prefix sums of the WHOLE pole-zero waveform although a trapezoid sweep only reads
// them in a window of ~2 200 samples around t50.  Here a warp owns a waveform from the first load to the last store:
//
//   pass 1     whole waveform, INTEGERS only, 16 consecutive samples per lane and step (two 128-bit streaming loads, three steps ahead):
//              exact prefix sums P (warp scan); per 16-sample group P at its start and its largest / smallest sample -> SMEM;
//              P and PP = cumsum(P) at every 512-sample boundary -> SMEM
//   baseline   sum x, sum i*x over bl_window as differences of P / PP (two or three look-ups)                      [:250-253]
//   pass 1a    y = w + km1*cumsum(w) [:255-256] is NOT evaluated everywhere: from a group's extreme samples and P follow rigorous
//              bounds of y over the group (float, rounded outwards -> SMEM); every lane evaluates its most promising group in
//              float64, and only groups whose upper bound reaches the best value found are evaluated too (a few per cent of
//              a flat top) -> max(y), exactly the float64 value a full evaluation gives
//   pass 1b    threshold 0.5*max(y) [:260]: a group whose bounds lie below / above the threshold gives 16 mask bits 0x0000 / 0xffff,
//              the others (the rising edge; every group of a noise-only event) are evaluated sample by sample;
//              bit-parallel Intersect run detection (resolve_runs) -> first crossing sample
//   pass 2     prefix sums TT of the pole-zero waveform ONLY in a window [lo, lo + W) around the crossing (W from the host:
//              what the variant set can reach), 9 consecutive samples per lane and step (odd stride: conflict-free 64-bit
//              shared-memory stores), closed form from P / PP exactly as sweep_kernel -> identical TT values
//   t50        linear interpolation of the crossing [:260]
//   variants   warp-uniform rounds of 32 variants, one LANE per (rt, ft) point, which walks the n_w outputs of its PolynomialDNI
//              pick-off window [:262-268] (4 look-ups in TT per output; fit matrix from the constant bank through the uniform
//              datapath, blocks of 11 outputs: a complete unroll ran instruction-fetch bound); results straight to global memory.
//              A variant whose window leaves [lo, lo + W) -- clamped pick-offs of events with t50 at the trace ends -- waits
//              for a second window built where it needs it (rare; the loop ends because every variant fits W on its own).
//
// No block barrier, no atomics: one warp is one CTA.  Residency is limited by the float64 window in shared memory, not by the
// thread count.  A team of two warps per waveform (every phase split, ~8 barriers of 64 threads per waveform, twice the resident
// warps) was measured slower, 37.0 vs 40.4 M wf/s (instruction fetch: 16 % more instructions for the redundant scalar work), and
// was removed.  Outputs are bit-identical to sweep_kernel's (same arithmetic on the same exact integers), which stays the path of
// FIR / Savitzky-Golay variants, 32-bit samples and variant sets whose reach exceeds the window capacity.

constexpr int SWW_STEP = 288;        // samples per window-build step (9 per lane)
constexpr int SWW_MIN_STEPS = 4;     // the window area also holds pass 1's group table (8 KB)
constexpr int SWW_MAX_STEPS = 10;
constexpr int SWW_EXT_BYTES = 4096;  // float2 per 16-sample group
__host__ __device__ constexpr int sww_win_bytes(int steps) { return (steps * SWW_STEP + 8) * 8; }
// per waveform: window | mask | cP[20] | cPP[18] | 272 spare bytes   (11 CTAs per SM at 8 window steps).  The spare bytes keep
// the CTAs per SM that every window size was measured with: without them a 9-step window would fit 10 CTAs per SM instead of 9.
__host__ __device__ constexpr int sww_warp_bytes(int steps)
{
    return sww_win_bytes(steps) + NWORDS * 4 + 20 * 4 + 18 * 8 + 272;
}

struct SweepDni {
    double A[LGDSP_MAX_DNI * (LGDSP_MAX_DNI_DEG + 1)];
};

__device__ __forceinline__ uint4 sww_ld8(const uint16_t* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
// the same for the single pass over the whole waveform: no L1 allocation (the small L1 left beside 220 KB of shared memory keeps
// the variant table and the window's samples instead)
__device__ __forceinline__ uint4 sww_ld8_stream(const uint16_t* p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// closed-form pole-zero sample (the arithmetic of sweep_kernel's P2 body)
__device__ __forceinline__ double sww_y(uint32_t x, uint32_t Pincl, double ip1, double m, double km1)
{
    const double Sd = fma(-ip1, m, u2d(Pincl));
    const double w = u2d(x) - m;
    return fma(km1, Sd, w);
}

// the 16 consecutive samples of lane-group i0 (multiple of 16; the trace length is a multiple of 8: the second half may lie
// beyond the trace and reads as zeros)
__device__ __forceinline__ void sww_unpack16(const uint4& r0, const uint4& r1, uint32_t (&v)[16])
{
    v[0] = r0.x & 0xffffu; v[1] = r0.x >> 16; v[2] = r0.y & 0xffffu; v[3] = r0.y >> 16;
    v[4] = r0.z & 0xffffu; v[5] = r0.z >> 16; v[6] = r0.w & 0xffffu; v[7] = r0.w >> 16;
    v[8] = r1.x & 0xffffu; v[9] = r1.x >> 16; v[10] = r1.y & 0xffffu; v[11] = r1.y >> 16;
    v[12] = r1.z & 0xffffu; v[13] = r1.z >> 16; v[14] = r1.w & 0xffffu; v[15] = r1.w >> 16;
}
// streaming load of a lane group, left packed (the stream pass keeps three steps in flight)
__device__ __forceinline__ void sww_ld16_raw(const uint16_t* __restrict__ x, int i0, int n, uint4& r0, uint4& r1)
{
    r0 = make_uint4(0u, 0u, 0u, 0u);
    r1 = r0;
    if (i0 < n) r0 = sww_ld8_stream(x + i0);
    if (i0 + 8 < n) r1 = sww_ld8_stream(x + i0 + 8);
}
template <bool STREAM = false>
__device__ __forceinline__ void sww_ld16(const uint16_t* __restrict__ x, int i0, int n, uint32_t (&v)[16])
{
    uint4 r0 = make_uint4(0u, 0u, 0u, 0u), r1 = r0;
    if (i0 < n) r0 = STREAM ? sww_ld8_stream(x + i0) : sww_ld8(x + i0);
    if (i0 + 8 < n) r1 = STREAM ? sww_ld8_stream(x + i0 + 8) : sww_ld8(x + i0 + 8);
    v[0] = r0.x & 0xffffu; v[1] = r0.x >> 16; v[2] = r0.y & 0xffffu; v[3] = r0.y >> 16;
    v[4] = r0.z & 0xffffu; v[5] = r0.z >> 16; v[6] = r0.w & 0xffffu; v[7] = r0.w >> 16;
    v[8] = r1.x & 0xffffu; v[9] = r1.x >> 16; v[10] = r1.y & 0xffffu; v[11] = r1.y >> 16;
    v[12] = r1.z & 0xffffu; v[13] = r1.z >> 16; v[14] = r1.w & 0xffffu; v[15] = r1.w >> 16;
}

// P_excl(i) = sum_{j<i} x_j and PP_excl(i) = sum_{j<i} P_incl(j) for 0 <= i <= n from the 512-sample boundary carries plus the
// partial step before i (warp-cooperative, i warp-uniform; every lane gets the result)
__device__ __noinline__ void sww_prefix_at(const uint16_t* __restrict__ x, int n, const uint32_t* cP, const double* cPP, int i,
                                              int lane, uint32_t& Pq, double& PPq)
{
    const int bq = i >> 9, rem = i & 511;
    Pq = cP[bq];
    PPq = cPP[bq];
    if (rem) {
        const int j0 = 16 * lane;
        uint32_t v[16];
        sww_ld16(x, bq * 512 + j0, n, v);
        uint32_t dP = 0, dPP = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const int j = j0 + k;
            dP += (j < rem) ? v[k] : 0u;
            dPP += (j < rem) ? v[k] * (uint32_t)(rem - j) : 0u;
        }
        PPq += (double)rem * u2d(Pq) + warp_sum((double)dPP);
        Pq += __reduce_add_sync(FULL, dP);
    }
}

// exact maximum of y over the 16-sample group that starts at sample i0 (P_excl(i0) = Pst); samples beyond the trace excluded
__device__ __noinline__ double sww_group_max(const uint16_t* __restrict__ x, int i0, int n, uint32_t Pst, double m, double km1)
{
    uint32_t v[16];
    sww_ld16(x, i0, n, v);
    const double ib = (double)(i0 + 1);
    double gmax = -CUDART_INF;
    uint32_t Pr = Pst;
    const int kn = (i0 + 8 < n) ? 16 : 8;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        Pr += v[k];
        const double y = sww_y(v[k], Pr, ib + (double)k, m, km1);
        gmax = (y > gmax && k < kn) ? y : gmax;
    }
    return gmax;
}
// bit k: y(i0 + k) >= thr
__device__ __noinline__ uint32_t sww_group_bits(const uint16_t* __restrict__ x, int i0, int n, uint32_t Pst, double m, double km1,
                                                   double thr)
{
    uint32_t v[16];
    sww_ld16(x, i0, n, v);
    const double ib = (double)(i0 + 1);
    uint32_t Pr = Pst, b = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        Pr += v[k];
        b |= (sww_y(v[k], Pr, ib + (double)k, m, km1) >= thr) ? (1u << k) : 0u;
    }
    return (i0 + 8 < n) ? b : (b & 0xffu);
}

// sum_i A[i][j] * trap(from + i), j < mdeg: the PolynomialDNI coefficient sums of one variant.  NW/MD > 0: the window length and
// degree+1 are compile-time constants, the loop is unrolled completely and the fit matrix enters the FMAs as constant-bank
// operands (no load instruction, no index arithmetic); NW = 0: run-time sizes
template <int NW, int MD>
__device__ __forceinline__ void sww_dni_sums(const SweepDni& D, const double* p0, const TrapDev& t, int n_w, int mdeg, double& c0,
                                             double& c1, double& c2, double& c3)
{
    const double* p1 = p0 + t.a;
    const double* p2 = p1 + t.g;
    const double* p3 = p0 + t.L;
    c0 = 0; c1 = 0; c2 = 0; c3 = 0;
    if (NW > 0) {
        // blocks of 11 outputs: the loop body stays inside the instruction cache of a scheduler; a complete unroll (44 x 12
        // instructions) ran fetch-bound (measured: blocks of 2 / 4 / 11 / 44 -> 37.3 / 38.9 / 39.9 / 33.6 M wf/s)
        constexpr int UNR = 11;
        static_assert(NW % UNR == 0, "window length must be a multiple of the unroll factor");
#pragma unroll 1
        for (int ib = 0; ib < NW; ib += UNR) {
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                const int i = ib + u;
                const double val = __fma_rn(p3[i] - p2[i], t.inv2, -__dmul_rn(p1[i] - p0[i], t.inv1));
                c0 = fma(D.A[i * MD], val, c0);
                if (MD > 1) c1 = fma(D.A[i * MD + 1], val, c1);
                if (MD > 2) c2 = fma(D.A[i * MD + 2], val, c2);
                if (MD > 3) c3 = fma(D.A[i * MD + 3], val, c3);
            }
        }
    } else {
#pragma unroll 4
        for (int i = 0; i < n_w; ++i) {
            const double val = __fma_rn(p3[i] - p2[i], t.inv2, -__dmul_rn(p1[i] - p0[i], t.inv1));
            const double* a = D.A + i * mdeg;
            c0 = fma(a[0], val, c0);
            if (mdeg > 1) c1 = fma(a[1], val, c1);
            if (mdeg > 2) c2 = fma(a[2], val, c2);
            if (mdeg > 3) c3 = fma(a[3], val, c3);
        }
    }
}

__global__ void __launch_bounds__(32, 11)
sweep_warp_kernel(const __grid_constant__ SweepDev P, const __grid_constant__ SweepDni D, const uint16_t* __restrict__ wf,
                  long long n_events, long long ld, const double* __restrict__ bl_ext, void* __restrict__ out,
                  double* __restrict__ aux)
{
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31;
    const int steps = P.win_steps;
    const int W = steps * SWW_STEP;
    unsigned char* base = smem;
    double* win = reinterpret_cast<double*>(base);
    float2* ext = reinterpret_cast<float2*>(base);
    uint32_t* pst = reinterpret_cast<uint32_t*>(base + SWW_EXT_BYTES);
    uint32_t* xmm = pst + MAXN / 16;
    uint32_t* mask = reinterpret_cast<uint32_t*>(base + sww_win_bytes(steps));
    uint32_t* cP = mask + NWORDS;
    double* cPP = reinterpret_cast<double*>(cP + 20);

    const int n = P.n;
    const double t_first = P.t_first, dt = P.dt, km1 = P.km1;
    const int n_w = P.sig_dni.n_w, mdeg = P.sig_dni.m;

    for (long long e = blockIdx.x; e < n_events; e += gridDim.x) {
        const uint16_t* __restrict__ x = wf + e * ld;
        // Fixed pick-offs (win_mode 0) without the aux outputs read nothing that depends on t50: max(y), the threshold mask and the
        // crossing are skipped (dsp_trap_rt_optimization, src/dsp_filter_optimization.jl:102-133), and no sample behind the last
        // look-up of the set (stream_n, exact on the host: the windows do not depend on the event) is read at all
        const bool need_t50 = P.win_mode == 1 || aux != nullptr;
        const int n_s = need_t50 ? n : min(n, (P.stream_n + 15) & ~15);   // samples of the integer pass (multiple of 8: n is)
        const int n_it_s = (n_s + 511) >> 9;
        if (threadIdx.x == 0 && e + gridDim.x < n_events) tma_prefetch_l2(wf + (e + gridDim.x) * ld, (uint32_t)n_s * 2u);
        // ---- pass 1 (integers only): steps of 512 samples; prefix sums, group table, P and PP at the step boundaries ----
        {
            uint32_t carryP = 0;
            unsigned long long carryPP = 0;
            uint4 ra[3], rb[3];   // raw samples of the next three steps
#pragma unroll
            for (int q = 0; q < 3; ++q) sww_ld16_raw(x, q * 512 + 16 * lane, n_s, ra[q], rb[q]);
#pragma unroll 1
            for (int it = 0; it < n_it_s; ++it) {
                uint32_t v[16];
                sww_unpack16(ra[0], rb[0], v);
                ra[0] = ra[1]; rb[0] = rb[1]; ra[1] = ra[2]; rb[1] = rb[2];
                sww_ld16_raw(x, (it + 3) * 512 + 16 * lane, n_s, ra[2], rb[2]);    // three steps ahead
                uint32_t s[16];
                s[0] = v[0];
#pragma unroll
                for (int k = 1; k < 16; ++k) s[k] = s[k - 1] + v[k];
                const int i0 = it * 512 + 16 * lane;
                uint32_t xmax = 0, xmin = 0;
                if (need_t50) {
                    xmax = __vimax3_u32(__vimax3_u32(v[0], v[1], v[2]), __vimax3_u32(v[3], v[4], v[5]), __vimax3_u32(v[6], v[7], v[7]));
                    xmin = __vimin3_u32(__vimin3_u32(v[0], v[1], v[2]), __vimin3_u32(v[3], v[4], v[5]), __vimin3_u32(v[6], v[7], v[7]));
                }
                if (need_t50 && i0 + 8 < n) {
                    xmax = __vimax3_u32(__vimax3_u32(v[8], v[9], v[10]), __vimax3_u32(v[11], v[12], v[13]), __vimax3_u32(v[14], v[15], xmax));
                    xmin = __vimin3_u32(__vimin3_u32(v[8], v[9], v[10]), __vimin3_u32(v[11], v[12], v[13]), __vimin3_u32(v[14], v[15], xmin));
                }
                uint32_t incl = s[15];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(FULL, incl, o);
                    if (lane >= o) incl += t;
                }
                // sum over the 512 samples of the step of (P(i) - P(step start)): 16*sum_l excl_l + sum_l sum_k s_l[k]
                uint32_t tl = 0;
#pragma unroll
                for (int k = 0; k < 16; k += 4) tl += (s[k] + s[k + 1]) + (s[k + 2] + s[k + 3]);
                const uint32_t sum_t = __reduce_add_sync(FULL, tl);
                const uint32_t sum_ex = __reduce_add_sync(FULL, (uint32_t)(31 - lane) * s[15]);
                // P and PP = cumsum(P) at every 512-sample boundary (exact integers; PP < 2^43 in float64)
                if (lane == 0) { cP[it] = carryP; cPP[it] = (double)carryPP; }
                if (need_t50 && i0 < n) pst[it * 32 + lane] = carryP + incl - s[15];
                carryPP += 512ull * carryP + 16ull * sum_ex + sum_t;
                carryP += __shfl_sync(FULL, incl, 31);
                if (need_t50 && i0 < n) xmm[it * 32 + lane] = (xmax << 16) | xmin;
            }
            if (lane == 0) { cP[n_it_s] = carryP; cPP[n_it_s] = (double)carryPP; }
        }
        __syncwarp();

        // ---- baseline window from the prefix sums: sum x = P(b+1) - P(a), sum i*x = b*P(b+1) - a*P(a) - (PP(b) - PP(a)) ----
        double blSd, blSXd = 0.0;
        {
            uint32_t Qa, Qb1;
            double PPa, PPb, PPb1;
            sww_prefix_at(x, n, cP, cPP, P.bl_from, lane, Qa, PPa);
            sww_prefix_at(x, n, cP, cPP, P.bl_until + 1, lane, Qb1, PPb1);
            blSd = u2d(Qb1 - Qa);
            if (aux) {
                uint32_t Qb;
                sww_prefix_at(x, n, cP, cPP, P.bl_until, lane, Qb, PPb);
                blSXd = ((double)P.bl_until * u2d(Qb1) - (double)P.bl_from * u2d(Qa)) - (PPb - PPa);
            }
        }
        const double m_own = mul_rn(blSd, P.bl_inv_n);
        const double m = bl_ext ? bl_ext[e] : m_own;

        int pos = -1;
        double thr = 0.0;
        if (need_t50) {
            // ---- pass 1a: rigorous bounds of y over every group -> table; max(y) from the few groups that can hold it ----
            // y_k = d_k + km1*Sd_k, d_k = x_k - m, Sd_k = Sd_0 + sum_{j<=k} d_j with Sd_0 = P(group start) - i0*m, so within a group
            //   Sd_0 + 16*min(0, d_min) <= Sd_k <= Sd_0 + 16*max(0, d_max);  the sample that attains d_max has y >= d_max + km1*Sd_lo.
            // G covers the rounding of the float64 evaluation (|terms| < 2^17 + |km1| n 2^16, one ulp each).
            const double G = 1e-9 * (65536.0 + fabs(m) + fabs(km1) * (double)n * 65536.0);
            double lbmax = -CUDART_INF;
            float best_ub = -CUDART_INF_F;
            int best_it = -1;
            const int my_groups = (n - 16 * lane + 511) >> 9;   // groups of this lane's column (<= 0: none)
            // (the group loops of pass 1a / 1b unrolled by 2 or 4: 38.0-38.4 M wf/s, code size)
#pragma unroll 1
            for (int it = 0; it < my_groups; ++it) {
                const int i0 = it * 512 + 16 * lane;
                const uint32_t xm = xmm[it * 32 + lane];
                const double dmax = u2d(xm >> 16) - m, dmin = u2d(xm & 0xffffu) - m;
                const double Sd0 = fma(-(double)i0, m, u2d(pst[it * 32 + lane]));
                const double Sd_hi = fma(16.0, dmax > 0.0 ? dmax : 0.0, Sd0), Sd_lo = fma(16.0, dmin < 0.0 ? dmin : 0.0, Sd0);
                const double k_hi = km1 >= 0.0 ? Sd_hi : Sd_lo, k_lo = km1 >= 0.0 ? Sd_lo : Sd_hi;
                const double ub = fma(km1, k_hi, dmax) + G;
                const double lb_all = fma(km1, k_lo, dmin) - G;
                const double lb_top = fma(km1, k_lo, dmax) - G;
                lbmax = lb_top > lbmax ? lb_top : lbmax;
                const float ubf = __double2float_ru(ub);
                ext[it * 32 + lane] = make_float2(ubf, __double2float_rd(lb_all));
                if (ubf > best_ub) { best_ub = ubf; best_it = it; }
            }
            // every lane evaluates the group with its largest upper bound exactly: a lower bound close to the maximum ...
            double ymax = -CUDART_INF;
            if (best_it >= 0) ymax = sww_group_max(x, best_it * 512 + 16 * lane, n, pst[best_it * 32 + lane], m, km1);
            const double LB = fmax(warp_max(ymax), warp_max(lbmax));
            // ... and only groups whose upper bound reaches it can hold a larger sample
#pragma unroll 1
            for (int it = 0; it < my_groups; ++it) {
                const int i0 = it * 512 + 16 * lane;
                if ((double)ext[it * 32 + lane].x >= LB && it != best_it) {
                    const double gm = sww_group_max(x, i0, n, pst[it * 32 + lane], m, km1);
                    ymax = gm > ymax ? gm : ymax;
                }
            }
            ymax = warp_max(ymax);
            thr = ymax * 0.5;

            // ---- pass 1b: threshold mask of y >= thr, first run of >= tx_min_n samples ----
#pragma unroll 1
            for (int it = 0; it < NWORDS / 16; ++it) {
                uint32_t b = 0;
                const int i0 = it * 512 + 16 * lane;
                if (i0 < n) {
                    const float2 ex = ext[it * 32 + lane];
                    if ((double)ex.x >= thr) {
                        if ((double)ex.y >= thr) b = (i0 + 8 < n) ? 0xffffu : 0xffu;
                        else b = sww_group_bits(x, i0, n, pst[it * 32 + lane], m, km1, thr);
                    }
                }
                b <<= 16 * (lane & 1);
                b |= __shfl_xor_sync(FULL, b, 1);
                if ((lane & 1) == 0) mask[it * 16 + (lane >> 1)] = b;
            }
            __syncwarp();
            int mult;
            resolve_runs(mask, P.tx_min_n, lane, pos, mult);

        }
        // ---- pass 2 + variants ----
        const int lo_max = n > W ? n - W : 0;
        int lo = (pos >= 1 && P.win_mode == 1) ? pos + P.win_rel_lo : P.win_abs_lo;
        lo = max(0, min(lo, lo_max));
        // the crossing samples pos-1 .. pos+1 are always inside the first window (t50 is read from it)
        if (pos >= 1 && (lo > pos - 1 || pos + 1 > lo + W)) lo = max(0, min(pos - (W >> 1), lo_max));
        unsigned done = 0;
        double t50_us = 0.0;
        bool first = true;
        // (the first round's variant parameters travel while the window is built)
        const TrapDev t_first_round = P.vars[min(lane, P.nvar - 1)].t;
        const double pick_first_round = P.vars[min(lane, P.nvar - 1)].pick_ns;
        const int mode_first_round = P.vars[min(lane, P.nvar - 1)].mode;
        int rounds = 0;
#pragma unroll 1
        while (true) {
            __syncwarp();   // every read of the group table / the previous window is over
            if (steps > 0) {   // (always true: the launch needs SWW_MIN_STEPS; the guard keeps the measured code generation)
                // prefix sums at the window's first sample
                uint32_t cp;
                double cpp;
                sww_prefix_at(x, n, cP, cPP, min(lo, n), lane, cp, cpp);
                if (lane == 0) {
                    const double lod = (double)lo;
                    const double tri = 0.5 * lod * (lod + 1.0);
                    win[0] = fma(km1, fma(-tri, m, cpp), fma(-lod, m, u2d(cp)));
                }
                uint32_t q[9];
                {
                    const int i0 = lo + 9 * lane;
#pragma unroll
                    for (int k = 0; k < 9; ++k) q[k] = (i0 + k < n) ? (uint32_t)__ldg(x + i0 + k) : 0u;
                }
#pragma unroll 1
                for (int j = 0; j < steps; ++j) {
                    uint32_t v[9];
#pragma unroll
                    for (int k = 0; k < 9; ++k) v[k] = q[k];
                    const int i0 = lo + SWW_STEP * j + 9 * lane;
                    if (j + 1 < steps) {
#pragma unroll
                        for (int k = 0; k < 9; ++k) q[k] = (i0 + SWW_STEP + k < n) ? (uint32_t)__ldg(x + i0 + SWW_STEP + k) : 0u;
                    }
                    uint32_t s[9];
                    s[0] = v[0];
#pragma unroll
                    for (int k = 1; k < 9; ++k) s[k] = s[k - 1] + v[k];
                    uint32_t incl = s[8];
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t t = __shfl_up_sync(FULL, incl, o);
                        if (lane >= o) incl += t;
                    }
                    const uint32_t Pst = cp + incl - s[8];
                    uint32_t tl = s[0];
#pragma unroll
                    for (int k = 1; k < 9; ++k) tl += s[k];
                    const double qd = fma(9.0, u2d(incl - s[8]), u2d(tl));   // lane sum of (P(i) - cp): exact (< 2^37)
                    double inclq = qd;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const double t = __shfl_up_sync(FULL, inclq, o);
                        if (lane >= o) inclq += t;
                    }
                    // PP before this lane's first sample: cpp + 9*lane*cp + (scan of the lane sums)
                    double PPr = cpp + (double)(9 * lane) * u2d(cp) + (inclq - qd);
                    uint32_t Pr = Pst;
                    double ip1 = (double)i0;
                    double tri = 0.5 * ip1 * (ip1 + 1.0);
                    double* tp = win + SWW_STEP * j + 9 * lane + 1;
#pragma unroll
                    for (int k = 0; k < 9; ++k) {
                        Pr += v[k];
                        const double Pd = u2d(Pr);
                        PPr += Pd;
                        ip1 += 1.0;
                        tri += ip1;
                        const double Sd = fma(-ip1, m, Pd);
                        const double SS = fma(-tri, m, PPr);
                        tp[k] = (i0 + k < n) ? fma(km1, SS, Sd) : 0.0;
                    }
                    cpp += (double)SWW_STEP * u2d(cp) + __shfl_sync(FULL, inclq, 31);
                    cp += __shfl_sync(FULL, incl, 31);
                }
            }
            __syncwarp();
            const double* TTw = win - lo;   // TTw[i] = TT[i] for lo <= i <= lo + W
            if (first) {
                first = false;
                if (pos >= 1) {
                    t50_us = cross_x(thr, y_at(TTw, pos - 1), y_at(TTw, pos), t_first + (double)(pos - 1) * dt, dt) * 0.001;
                    if (t50_us != t50_us) t50_us = 0.0;
                }
                if (aux && threadIdx.x == 0) {
                    const Stats st = stats_finalize(P.bl_inv_n, P.bl_sX, P.bl_sXX, blSd, 0.0, t_first * blSd + dt * blSXd);
                    double* a = aux + e * 4;
                    a[0] = m_own; a[1] = st.slope; a[2] = t50_us; a[3] = 0.0;
                }
            }
            int minfrom = 0x7fffffff;
            // Warp-uniform loop over rounds of 32 variants: every lane runs the arithmetic (a lane without work reads the start of
            // the window), so the inner loop sits in convergent code and the fit matrix is read through the uniform datapath
            const int n_rounds = (P.nvar + 31) / 32;
            int rnd;
            // this lane's variant of the next round is loaded one round ahead (the table comes from L2 / L1)
            TrapDev tn = t_first_round;
            double pickn = pick_first_round;
            int moden = mode_first_round;
#pragma unroll 1
            for (rnd = 0; rnd < n_rounds; ++rnd) {
                const int v = rnd * 32 + lane;
                const TrapDev tv = tn;
                const double pick = pickn;
                const int mode = moden;
                {
                    const SweepVar& nx = P.vars[min(v + 32, P.nvar - 1)];
                    tn = nx.t; pickn = nx.pick_ns; moden = nx.mode;
                }
                bool eval = false;
                TrapDev t;
                t.a = 0; t.g = 0; t.L = 0; t.inv1 = 0.0; t.inv2 = 0.0;
                double pc = 0.0;
                int from = lo, nout = 0;
                if (v < P.nvar && !((done >> rnd) & 1u)) {
                    nout = n - tv.L + 1;
                    const double tf = __fma_rn((double)(tv.L - 1), dt, t_first);
                    const double t_ns = mode ? __fma_rn(t50_us, 1000.0, pick) : pick;
                    int fr;
                    dni_window(n_w, nout, P.dt_pow2 ? (t_ns - tf) * P.rdt : (t_ns - tf) / dt, pc, fr);
                    if (fr < lo || fr + tv.L + n_w - 1 > lo + W) {   // look-ups TT[from .. from + L + n_w - 1]
                        minfrom = min(minfrom, fr);
                    } else {
                        eval = true;
                        done |= 1u << rnd;
                        from = fr;
                        t = tv;
                    }
                }
                if (__ballot_sync(FULL, eval) == 0u) continue;
                double c0, c1, c2, c3;
                if (n_w == 44 && mdeg == 4) sww_dni_sums<44, 4>(D, TTw + from, t, n_w, mdeg, c0, c1, c2, c3);
                else sww_dni_sums<0, 0>(D, TTw + from, t, n_w, mdeg, c0, c1, c2, c3);
                if (eval) {
                    const double u = pc - (double)from;
                    const double res = (nout >= n_w) ? fma(fma(fma(c3, u, c2), u, c1), u, c0) : CUDART_NAN;
                    if (P.out_f64) reinterpret_cast<double*>(out)[e * (long long)P.nvar + v] = res;
                    else reinterpret_cast<float*>(out)[e * (long long)P.nvar + v] = (float)res;
                }
            }
            minfrom = __reduce_min_sync(FULL, minfrom);
            if (minfrom == 0x7fffffff) break;
            if (++rounds > 2 * 1024 / 32 + 2) {
                // cannot happen (every variant fits a window that starts at its own `from`); never spin on the device
                rnd = 0;
                for (int v = lane; v < P.nvar; v += 32, ++rnd) {
                    if ((done >> rnd) & 1u) continue;
                    if (P.out_f64) reinterpret_cast<double*>(out)[e * (long long)P.nvar + v] = CUDART_NAN;
                    else reinterpret_cast<float*>(out)[e * (long long)P.nvar + v] = CUDART_NAN_F;
                }
                break;
            }
            lo = max(0, min(minfrom, lo_max));
        }
        __syncwarp();   // the window area becomes the next event's group table
    }
}

// launch geometry for a window of `steps` steps: CTAs (one waveform each) per SM, 0 if the kernel cannot run
inline int sww_geometry(int steps)
{
    static int cache[SWW_MAX_STEPS + 1];
    static bool attr_set = false;
    if (steps < SWW_MIN_STEPS || steps > SWW_MAX_STEPS) return 0;
    if (cache[steps]) return cache[steps];
    if (!attr_set) {
        int dev = 0, optin = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (cudaFuncSetAttribute(sweep_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin) != cudaSuccess) return 0;
        attr_set = true;
    }
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, sweep_warp_kernel, 32, (size_t)sww_warp_bytes(steps)) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    cache[steps] = nb;
    return nb;
}
