// Split dsp_icpc pipeline for sm_100a (included by lgdsp_icpc.cu, inside namespace lgdsp).
//
// The fused icpc_kernel keeps 115 KB of shared memory and 128 registers per waveform (16 resident warps per SM, one
// instruction stream of ~150 KB).  This path runs the same arithmetic as three kernels, each with its own shared-memory /
// register budget, coupled through a ring of float64 prefix sums that stays in L2:
//
//   icpc_prefix_kernel   raw samples (TMA, double-buffered) -> saturation [:93-95], baseline stats [:102], min/max
//                        [:111-112], tailstats [:115], closed-form pole-zero prefix sums TT [:105,:119-120] -> global ring,
//                        t10..t99 threshold masks [:132-136] and their crossings; 39 KB SMEM, 4 CTAs/SM
//   icpc_extract_kernel  TT (TMA bulk load) -> everything that is a window on TT: PZ tail stats [:123], trapezoids
//                        [:126,:147-164,:202-207], currents [:181-195], in-trace pile-up [:189], Q-drift [:141-144];
//                        74 KB SMEM, 3 CTAs/SM
//   icpc_cuspzac_kernel  TT -> CUSP / ZAC through their analytic structure [:167-178]; 106 KB SMEM, 2 CTAs/SM
//
// (reference lines: /root/reference/src/dsp_icpc.jl).  The three kernels of one event batch run back to back on a stream;
// the batch is sized so that its prefix sums (65.6 KB per event) are still in L2 when the consumers read them.
// Every value is produced by the same expressions as in icpc_kernel (same helpers, same operation order).

constexpr int TTG_LEN = TT_LEN;     // doubles per event slot of the global prefix-sum ring
constexpr int AUX_LEN = 16;         // doubles per event: values handed from the prefix kernel to the consumers
enum { AX_M = 0, AX_EMAX = 1, AX_YMAX = 2, AX_THR = 3 /* 5 */, AX_POS = 8 /* 5 */, AX_BAD = 13 /* 1: sample sum beyond 32 bits */ };

// ---- prefix kernel: shared memory ----
enum { K1R_BLS = 0, K1R_BLSS, K1R_BLSX, K1R_MX /* + K1R_MN: 4 x NWARP uint32 */, K1R_MN, K1R_SLEN, K1R_SS, K1R_SQ,
       K1R_TLS, K1R_TLSS, K1R_TLSX, K1R_TLBAD, K1R_YMAX, K1R_N };

constexpr int K1_XS = 0;                                   // 2 x (MAXN * 2) bytes: double-buffered raw samples
constexpr int K1_MASK = K1_XS + 2 * MAXN * 2;              // uint32 masks[5][NWORDS]: t10..t99
constexpr int K1_RED = K1_MASK + 5 * NWORDS * 4;
constexpr int K1_IRED = K1_MASK;                           // int[64]: saturation run partials (before the masks are written)
constexpr int K1_BAR = K1_RED + K1R_N * NWARP * 8;         // 2 mbarriers
constexpr int TILE_LD = 9;                                 // row stride of the staging tile (odd: 2-way = optimal for 64-bit words)
constexpr int K1_TILE = K1_BAR + 16;                       // double tile[NWARP][32][TILE_LD]: transposition of the prefix-sum stores
constexpr int K1_TOTAL = K1_TILE + NWARP * 32 * TILE_LD * 8;
static_assert(4 * (K1_TOTAL + 1024) <= 233472, "four CTAs per SM");

// GMASK: compile-time column-group mask (0: from the parameter block), see icpc_extract_kernel
template <typename SAMPLE, unsigned GMASK>
__global__ void __launch_bounds__(NT, 4)
icpc_prefix_kernel(const __grid_constant__ IcpcDev P, const SAMPLE* __restrict__ wf, long long n_events, long long ld,
                   const double* __restrict__ bl_ext, long long bl_stride, double bl_div, double* __restrict__ ttg,
                   double* __restrict__ auxg, double* __restrict__ rows)
{
    extern __shared__ __align__(128) unsigned char smem[];
    uint32_t* masks = reinterpret_cast<uint32_t*>(smem + K1_MASK);
    double* red = reinterpret_cast<double*>(smem + K1_RED);
    int* ired = reinterpret_cast<int*>(smem + K1_IRED);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + K1_BAR);

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n = P.n;
    const uint32_t wf_bytes = (uint32_t)n * (uint32_t)sizeof(SAMPLE);
    const double t_first = P.t_first, dt = P.dt;
    const unsigned G = GMASK ? GMASK : P.groups;
    const bool lean = (G & LGDSP_GROUP_LEAN) != 0;   // only {blmean, t0, t50, e_trap, e_10410} are wanted (+ e_max / e_min / saturation counts)

    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (tid == 0 && (long long)blockIdx.x < n_events) {
        mbar_expect_tx(&bar[0], wf_bytes);
        tma_load_1d(smem + K1_XS, wf + (long long)blockIdx.x * ld, wf_bytes, &bar[0]);
    }
    const int i0 = tid * CH;
    const int cvalid = max(0, min(CH, n - i0));
    const unsigned long long chunk_all = (1ull << cvalid) - 1ull;

    uint32_t it = 0;
    for (long long e = blockIdx.x; e < n_events; e += gridDim.x, ++it) {
        const int b = (int)(it & 1u);
        SAMPLE* xs = reinterpret_cast<SAMPLE*>(smem + K1_XS + b * (MAXN * 2));
        // the other buffer was last read before the barrier that ended the previous event: prefetch the next event into it
        if (tid == 0) {
            const long long en = e + gridDim.x;
            if (en < n_events) {
                fence_proxy_async();
                mbar_expect_tx(&bar[b ^ 1], wf_bytes);
                tma_load_1d(smem + K1_XS + (b ^ 1) * (MAXN * 2), wf + en * ld, wf_bytes, &bar[b ^ 1]);
            }
        }
        mbar_wait(&bar[b], (it >> 1) & 1u);

        // ==========================================================================================
        // raw samples (same as P1 of icpc_kernel)
        // ==========================================================================================
        const SAMPLE* xp = xs + i0;
        uint32_t csum = 0, cq = 0, cmn = 0xFFFFFFFFu, cmx = 0;
#pragma unroll 3
        for (int k = 0; k < cvalid; ++k) {
            const uint32_t x = xp[k];
            csum += x;
            cq += csum;
            cmn = min(cmn, x);
            cmx = max(cmx, x);
        }
        {
            unsigned long long blSS = 0, blSX = 0;
            uint32_t blS = 0;
#pragma unroll 2
            for (int idx = P.bl_from + tid; idx <= P.bl_until; idx += NT) {
                const uint32_t x = xs[idx];
                blS += x;
                if (!lean) {   // (slope / sigma of the baseline are not among the lean columns)
                    blSX += (unsigned long long)x * (unsigned long long)idx;
                    blSS += (unsigned long long)x * (unsigned long long)x;
                }
            }
            const double a = wsum_d((double)blS), bq = wsum_d((double)blSS), c = wsum_d((double)blSX);
            if (lane == 0) { red[K1R_BLS * NWARP + wid] = a; red[K1R_BLSS * NWARP + wid] = bq; red[K1R_BLSX * NWARP + wid] = c; }
        }
        int nlow = 0, nhigh = 0;
        if ((int)cmn == P.sat_low || (int)cmx == P.sat_high) {
            for (int k = 0; k < cvalid; ++k) {
                const int x = xp[k];
                nlow += (x == P.sat_low);
                nhigh += (x == P.sat_high);
            }
        }
        {
            const uint32_t wmn = __reduce_min_sync(FULL, cmn), wmx = __reduce_max_sync(FULL, cmx);
            const uint32_t wl = __reduce_add_sync(FULL, (uint32_t)nlow), wh = __reduce_add_sync(FULL, (uint32_t)nhigh);
            if (lane == 0) {
                uint32_t* ured = reinterpret_cast<uint32_t*>(red + K1R_MX * NWARP);
                ured[wid] = wmx; ured[NWARP + wid] = wmn; ured[2 * NWARP + wid] = wl; ured[3 * NWARP + wid] = wh;
            }
        }
        int sl = cvalid;
        uint32_t ss = csum;
        double sq = (double)cq;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int l2 = __shfl_up_sync(FULL, sl, o);
            const uint32_t s2 = __shfl_up_sync(FULL, ss, o);
            const double q2 = __shfl_up_sync(FULL, sq, o);
            if (lane >= o) {
                sq = q2 + sq + (double)sl * (double)s2;
                ss += s2;
                sl += l2;
            }
        }
        if (lane == 31) {
            red[K1R_SLEN * NWARP + wid] = (double)sl;
            red[K1R_SS * NWARP + wid] = (double)ss;
            red[K1R_SQ * NWARP + wid] = sq;
        }
        int el = __shfl_up_sync(FULL, sl, 1);
        uint32_t es = __shfl_up_sync(FULL, ss, 1);
        double eq = __shfl_up_sync(FULL, sq, 1);
        if (lane == 0) { el = 0; es = 0; eq = 0.0; }
        __syncthreads();   // ---- B1 ----

        uint32_t P_excl;
        double PP_excl;
        {
            double cs = 0.0, cqd = 0.0;
#pragma unroll 1
            for (int w = 0; w < wid; ++w) {
                const double lw = red[K1R_SLEN * NWARP + w], sw = red[K1R_SS * NWARP + w], qw = red[K1R_SQ * NWARP + w];
                cqd = cqd + qw + lw * cs;
                cs += sw;
            }
            P_excl = (uint32_t)cs + es;
            PP_excl = cqd + eq + (double)el * cs;
        }
        uint32_t mx, mn;
        {
            const uint32_t* ured = reinterpret_cast<const uint32_t*>(red + K1R_MX * NWARP);
            const int l8 = lane & 7;
            mx = __reduce_max_sync(FULL, ured[l8]);
            mn = __reduce_min_sync(FULL, ured[NWARP + l8]);
            nlow = (int)__reduce_add_sync(FULL, lane < 8 ? ured[2 * NWARP + l8] : 0u);
            nhigh = (int)__reduce_add_sync(FULL, lane < 8 ? ured[3 * NWARP + l8] : 0u);
        }
        int cons_low = 0, cons_high = 0;
        if (nlow + nhigh > 0) {
            Run rl = {0, 0, 0, cvalid}, rh = {0, 0, 0, cvalid};
            {
                int cl = 0, chh = 0;
                bool pl = true, ph = true;
                for (int k = 0; k < cvalid; ++k) {
                    const int x = xp[k];
                    const bool il = (x == P.sat_low), ih = (x == P.sat_high);
                    cl = il ? cl + 1 : 0;
                    chh = ih ? chh + 1 : 0;
                    rl.best = max(rl.best, cl);
                    rh.best = max(rh.best, chh);
                    if (pl && il) rl.pre = cl; else pl = false;
                    if (ph && ih) rh.pre = chh; else ph = false;
                }
                rl.suf = cl; rh.suf = chh;
            }
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                Run bl_ = run_shfl_down(rl, o), bh_ = run_shfl_down(rh, o);
                if ((lane & (2 * o - 1)) == 0) { rl = run_merge(rl, bl_); rh = run_merge(rh, bh_); }
            }
            if (lane == 0) {
                ired[wid * 8 + 0] = rl.pre; ired[wid * 8 + 1] = rl.suf; ired[wid * 8 + 2] = rl.best; ired[wid * 8 + 3] = rl.len;
                ired[wid * 8 + 4] = rh.pre; ired[wid * 8 + 5] = rh.suf; ired[wid * 8 + 6] = rh.best; ired[wid * 8 + 7] = rh.len;
            }
            __syncthreads();
            Run al = {ired[0], ired[1], ired[2], ired[3]}, ah = {ired[4], ired[5], ired[6], ired[7]};
            for (int w = 1; w < NWARP; ++w) {
                Run bl_ = {ired[w * 8], ired[w * 8 + 1], ired[w * 8 + 2], ired[w * 8 + 3]};
                Run bh_ = {ired[w * 8 + 4], ired[w * 8 + 5], ired[w * 8 + 6], ired[w * 8 + 7]};
                al = run_merge(al, bl_);
                ah = run_merge(ah, bh_);
            }
            cons_low = al.best; cons_high = ah.best;
            __syncthreads();   // the partials share their storage with the threshold masks written below
        }

        // 32-bit samples: the prefix sums are exact uint32 only while the waveform sums to < 2^32 (any 16-bit trace does; a
        // presummed trace does up to a mean of 2^20).  Beyond that the event's row is NaN instead of silently wrong.
        const bool wrapped = sum_exceeds_u32<SAMPLE>(xp, cvalid, mx, n, red + K1R_TLS * NWARP);
        const double m = bl_ext ? div_rn(bl_ext[e * bl_stride], bl_div) : mul_rn(red_sum(red, K1R_BLS), P.bl_inv_n);
        const double e_max = (double)mx - m, e_min = (double)mn - m;
        double thr[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) thr[k] = e_max * P.tx_frac[k];
        if (lean) { thr[0] = CUDART_INF; thr[2] = CUDART_INF; thr[3] = CUDART_INF; thr[4] = CUDART_INF; }   // only t50

        // ==========================================================================================
        // prefix sums of the pole-zero waveform -> global ring; t10..t99 masks from the values in flight
        // ==========================================================================================
        double* tg = ttg + e * TTG_LEN;
        {
            const double km1 = P.km1;
            const double Sd0 = fma(-(double)i0, m, u2d(P_excl));
            const double tri0 = 0.5 * (double)i0 * ((double)i0 + 1.0);
            const double TT0 = fma(km1, fma(-tri0, m, PP_excl), Sd0);
            const double wmin = (double)cmn - m, wmax = (double)cmx - m;
            const double ak = fabs(km1);
            const double srange = (double)CH * fmax(fabs(wmin), fabs(wmax));
            const double ylo = wmin + km1 * Sd0 - ak * srange, yhi = wmax + km1 * Sd0 + ak * srange;
            const double guard = 1e-9 * (fabs(ylo) + fabs(yhi)) + 1e-6;
            bool straddle = false;
            if (G & LGDSP_GROUP_TIMING) {
#pragma unroll
                for (int t = 0; t < 5; ++t)
                    if (!(lean && t != 1)) straddle |= !(ylo - guard >= thr[t]) && !(yhi + guard < thr[t]);
                straddle = straddle && cvalid > 0;
            }
            const bool wstr = __any_sync(FULL, straddle);   // warp-uniform: compare inside the loop or not
            uint32_t lo[5] = {0, 0, 0, 0, 0}, hi = 0;
            {
                uint32_t Pr = P_excl;
                double PPr = PP_excl;
                double ip1 = (double)i0;
                double tri = tri0;
                auto body = [&](int k) -> double {
                    Pr += xp[k];
                    const double Pd = u2d(Pr);
                    PPr += Pd;
                    ip1 += 1.0;
                    tri += ip1;
                    const double Sd = fma(-ip1, m, Pd);
                    const double SS = fma(-tri, m, PPr);
                    return fma(km1, SS, Sd);
                };
                // The chunk values go to HBM through a per-warp staging tile, eight samples of every chunk at a time: the warp then
                // stores runs of eight consecutive doubles (whole 32-byte sectors) instead of 32 scattered 8-byte words per
                // instruction, which quartered the L2 write traffic of this kernel.
                double* tile = reinterpret_cast<double*>(smem + K1_TILE) + wid * (32 * TILE_LD);
                double tprev = TT0;
                const int cbase = wid * 32;   // first chunk of this warp
                // store pass: lane -> (chunk 4r + lane/8, sample kb + lane%8); everything but r and kb is loop invariant.
                // (tile rows 1 apart share one bank pair per half warp: 17 % of this kernel's SMEM wavefronts are that 2-way
                //  conflict.  Pairing chunks 8 apart removes it -- rows 72 = 8 mod 16 doubles apart -- but spreads each store
                //  instruction over 2 KB instead of 1 KB of the ring and was 2.3 % SLOWER, 0.7375 vs 0.7210 ms per 16 384 events)
                const double* trd = tile + (lane >> 3) * TILE_LD + (lane & 7);
                double* gwr = tg + (cbase + (lane >> 3)) * CH + (lane & 7) + 1;
                const int glim = n - ((cbase + (lane >> 3)) * CH + (lane & 7));   // sample kb of chunk 4r is valid iff kb + 4r*CH < glim
                const bool wfull = (cbase + 32) * CH <= n;                        // every chunk of this warp is complete
                // sample k of the chunk: prefix sum, threshold bits, scan step
                auto sample = [&](int k, bool with_thr) -> double {
                    const double tn = body(k);
                    if (with_thr) {
                        const double y = tn - tprev;     // = TT[i+1] - TT[i] as every consumer forms it
                        if (k < 32) {
                            const uint32_t bit = 1u << k;
#pragma unroll
                            for (int t = 0; t < 5; ++t)
                                if (!(lean && t != 1)) lo[t] |= (y >= thr[t]) ? bit : 0u;
                        } else {
#pragma unroll
                            for (int t = 0; t < 5; ++t)
                                if (!(lean && t != 1)) hi |= (y >= thr[t]) ? (1u << t) : 0u;
                        }
                    }
                    tprev = tn;
                    return tn;
                };
#pragma unroll 1
                for (int kb = 0; kb < 32; kb += 8) {
                    if (wfull && !wstr) {
                        // common case: complete chunks, no threshold inside this warp's samples
#pragma unroll
                        for (int kk = 0; kk < 8; ++kk) tile[lane * TILE_LD + kk] = sample(kb + kk, false);
                    } else {
#pragma unroll
                        for (int kk = 0; kk < 8; ++kk) {
                            const int k = kb + kk;
                            if (k < cvalid) tile[lane * TILE_LD + kk] = sample(k, wstr);
                        }
                    }
                    __syncwarp();
                    if (wfull) {
#pragma unroll
                        for (int r = 0; r < 8; ++r) gwr[kb + r * (4 * CH)] = trd[r * (4 * TILE_LD)];
                    } else {
#pragma unroll
                        for (int r = 0; r < 8; ++r)
                            if (kb + r * (4 * CH) < glim) gwr[kb + r * (4 * CH)] = trd[r * (4 * TILE_LD)];
                    }
                    __syncwarp();
                }
                if (cvalid > 32) tg[i0 + 33] = sample(32, wstr);
                if (tid == 0) tg[0] = 0.0;
                if (i0 <= n && n < i0 + CH) tg[n + 1] = 0.0;   // the consumers load (n + 2) doubles (16-byte granularity)
            }
            if (G & LGDSP_GROUP_TIMING) {
#pragma unroll
                for (int t = 0; t < 5; ++t) {
                    if (lean && t != 1) continue;
                    unsigned long long mbt = (unsigned long long)lo[t] | ((unsigned long long)((hi >> t) & 1u) << 32);
                    if (cvalid <= 0) mbt = 0ull;
                    else if (ylo - guard >= thr[t]) mbt = chunk_all;
                    else if (yhi + guard < thr[t]) mbt = 0ull;
                    const unsigned long long up = __shfl_up_sync(FULL, mbt, 1);
                    uint32_t word = (uint32_t)(mbt << lane);
                    if (lane > 0) word |= (uint32_t)(up >> (33 - lane));
                    uint32_t* M = masks + t * NWORDS;
                    const int w = (CH * wid) + lane;
                    if (w < NWORDS) M[w] = word;
                    if (lane == 31 && w + 1 < NWORDS) M[w + 1] = (uint32_t)(mbt >> 1);
                }
            }
            const double ya = wmax_d(cvalid > 0 ? fmax(fabs(ylo), fabs(yhi)) : 0.0);
            red_put(red, K1R_YMAX, wid, lane, ya);
        }
        // tailstats: log-regression on the PRE-PZ waveform (src/tailstats.jl:22-72).  Every thread takes a run of CONSECUTIVE
        // tail samples: log(w) = log(c) + log1p((w - c)/c) around the thread's first sample c, and inside such a run (w - c)/c
        // is noise over amplitude, so a short Taylor polynomial reaches 1e-16 (the warp picks the degree its largest |u| needs;
        // a sample further than 1/8 away takes the full logarithm and becomes the new reference).
        {
            double tl_S = 0, tl_SS = 0, tl_SX = 0;
            bool bad = lean;
            double cref = 0.0, cinv = 0.0, clog = 0.0;
            const int ntail = P.tail_until - P.tail_from + 1;
            const int q = lean ? 0 : (ntail + NT - 1) / NT;
            const int ia = P.tail_from + tid * q, ib = min(ia + q - 1, P.tail_until);
            // Integer pre-pass over the thread's run: the samples are integers, so w - c is the exact integer x - x_ref and the
            // largest |u| = |x - x_ref| / c of the run is known before any logarithm; the warp picks ONE series for the whole run
            // (no per-sample category, vote or branch on data), and a non-positive sample is an integer compare with floor(m).
            int wcat = 3;
            double c_run = 0.0, cinv_run = 0.0;
            int xref = 0;
            if (q > 0) {
                const int mfl = (int)floor(fmin(fmax(m, -2.0e9), 2.0e9));   // x <= m  <=>  x <= floor(m) for integer x
                int dmx = 0;
                bool nonpos = false;
                xref = ia <= ib ? (int)xs[ia] : 0;
#pragma unroll 2
                for (int idx = ia; idx <= ib; ++idx) {
                    const int xv = (int)xs[idx];
                    nonpos |= xv <= mfl;
                    dmx = max(dmx, abs(xv - xref));
                }
                int cat = 0;
                if (ia <= ib) {
                    c_run = u2d((uint32_t)xref) - m;
                    cinv_run = 1.0 / c_run;
                    const double au = (double)dmx * cinv_run;
                    cat = (nonpos || !(c_run > 0.0) || au > 0.125) ? 3 : (au > 0.015625 ? 2 : (au > 0.0009765625 ? 1 : 0));
                }
                wcat = __reduce_max_sync(FULL, cat);
            }
            if (wcat < 3) {
                const double clog_run = ia <= ib ? log_d(c_run) : 0.0;
#pragma unroll 1
                for (int idx = ia; idx <= ib; ++idx) {
                    const double u = (double)((int)xs[idx] - xref) * cinv_run;
                    double lg;
                    if (wcat == 0) {
                        double pl = fma(u, 1.0 / 5.0, -1.0 / 4.0);
                        pl = fma(u, pl, 1.0 / 3.0); pl = fma(u, pl, -1.0 / 2.0); pl = fma(u, pl, 1.0);
                        lg = fma(u, pl, clog_run);
                    } else if (wcat == 1) {
                        const double u2 = u * u, u4 = u2 * u2;
                        const double a0 = fma(-1.0 / 2.0, u, 1.0), a1 = fma(-1.0 / 4.0, u, 1.0 / 3.0), a2 = fma(-1.0 / 6.0, u, 1.0 / 5.0),
                                     a3 = fma(-1.0 / 8.0, u, 1.0 / 7.0);
                        const double b0 = fma(a1, u2, a0), b1 = fma(a3, u2, a2);
                        const double c0 = fma(b1, u4, b0);
                        lg = fma(u, fma(u4 * u4, 1.0 / 9.0, c0), clog_run);
                    } else {
                        lg = clog_run + log1p_small(u);
                    }
                    const double X = t_first + (double)idx * dt;
                    tl_S += lg;
                    tl_SS = fma(lg, lg, tl_SS);
                    tl_SX = fma(X, lg, tl_SX);
                }
            } else {
                // a run with a sample more than 1/8 away from its first one (small or noisy tails), or with a non-positive sample:
                // the sample-by-sample form with re-referencing
#pragma unroll 1
                for (int i = 0; i < q; ++i) {
                    const int idx = ia + i;
                    const bool act = idx <= ib;
                    const double w = act ? u2d(xs[idx]) - m : cref;
                    const bool pos = w > 0.0;
                    if (act && !pos) bad = true;
                    const double u = (w - cref) * cinv, au = fabs(u);
                    const bool use = act && pos;
                    int cat = 0;
                    if (use) cat = !(cref > 0.0) || au > 0.125 ? 3 : (au > 0.015625 ? 2 : (au > 0.0009765625 ? 1 : 0));
                    const int wcat = __reduce_max_sync(FULL, cat);
                    double lg;
                    if (wcat == 0) {
                        // |u| <= 2^-10: terms to u^5 (truncation u^5/6 < 2e-16 relative)
                        double pl = fma(u, 1.0 / 5.0, -1.0 / 4.0);
                        pl = fma(u, pl, 1.0 / 3.0); pl = fma(u, pl, -1.0 / 2.0); pl = fma(u, pl, 1.0);
                        lg = fma(u, pl, clog);
                    } else if (wcat == 1) {
                        // |u| <= 2^-6: terms to u^9
                        const double u2 = u * u, u4 = u2 * u2;
                        const double a0 = fma(-1.0 / 2.0, u, 1.0), a1 = fma(-1.0 / 4.0, u, 1.0 / 3.0), a2 = fma(-1.0 / 6.0, u, 1.0 / 5.0),
                                     a3 = fma(-1.0 / 8.0, u, 1.0 / 7.0);
                        const double b0 = fma(a1, u2, a0), b1 = fma(a3, u2, a2);
                        const double c0 = fma(b1, u4, b0);
                        lg = fma(u, fma(u4 * u4, 1.0 / 9.0, c0), clog);
                    } else {
                        lg = clog + log1p_small(u);
                        if (cat == 3) {
                            lg = log_d(w);
                            cref = w; cinv = 1.0 / w; clog = lg;
                        }
                    }
                    if (use) {
                        const double X = t_first + (double)idx * dt;
                        tl_S += lg;
                        tl_SS = fma(lg, lg, tl_SS);
                        tl_SX = fma(X, lg, tl_SX);
                    }
                }
            }
            tl_S = wsum_d(tl_S); tl_SS = wsum_d(tl_SS); tl_SX = wsum_d(tl_SX);
            const bool anybad = __any_sync(FULL, bad);
            if (lane == 0) {
                red[K1R_TLS * NWARP + wid] = tl_S; red[K1R_TLSS * NWARP + wid] = tl_SS;
                red[K1R_TLSX * NWARP + wid] = tl_SX; red[K1R_TLBAD * NWARP + wid] = anybad ? 1.0 : 0.0;
            }
        }
        __syncthreads();   // ---- B2: masks and reduction slots complete; this event's samples are dead ----

        double* ax = auxg + e * AUX_LEN;
        double* ro = rows + e * LGDSP_NCOL;
        if (wid < 5) {
            // crossing resolution of t10..t99 (positions; the consumers interpolate on TT)
            int pos = -1, mult = 0;
            if ((G & LGDSP_GROUP_TIMING) && !(lean && wid != 1)) resolve_runs(masks + wid * NWORDS, P.tx_min_n, lane, pos, mult);
            if (lane == 0) { ax[AX_POS + wid] = (double)pos; ax[AX_THR + wid] = thr[wid == 0 ? 0 : wid == 1 ? 1 : wid == 2 ? 2 : wid == 3 ? 3 : 4]; }
        } else if (wid == 5) {
            // baseline [:102] and tailstats [:115] (lane 0 / lane 1, same code path)
            const double blS = red_sum(red, K1R_BLS), blSS = red_sum(red, K1R_BLSS), blSX = red_sum(red, K1R_BLSX);
            const double tlS = red_sum(red, K1R_TLS), tlSS = red_sum(red, K1R_TLSS), tlSX = red_sum(red, K1R_TLSX);
            const double tlbad = red_sum(red, K1R_TLBAD);
            if (lane < 2) {
                const double sY = lane == 0 ? blS : tlS;
                const double sYY = lane == 0 ? blSS : tlSS;
                const double sXY = lane == 0 ? t_first * blS + dt * blSX : tlSX;
                const Stats st = stats_finalize(lane == 0 ? P.bl_inv_n : P.tail_inv_n, lane == 0 ? P.bl_sX : P.tail_sX,
                                                lane == 0 ? P.bl_sXX : P.tail_sXX, sY, sYY, sXY);
                const double bad = wrapped ? CUDART_NAN : 0.0;   // (x + NaN = NaN)
                if (lane == 0) {
                    ro[LGDSP_COL_blmean] = st.mean + bad; ro[LGDSP_COL_blsigma] = st.sigma + bad;
                    ro[LGDSP_COL_blslope] = st.slope + bad; ro[LGDSP_COL_bloffset] = st.offset + bad;
                    ro[LGDSP_COL_qc_label] = -1.0 + bad;
                    ro[LGDSP_COL_e_max] = e_max + bad; ro[LGDSP_COL_e_min] = e_min + bad;
                    ro[LGDSP_COL_n_sat_low] = (double)nlow + bad; ro[LGDSP_COL_n_sat_high] = (double)nhigh + bad;
                    ro[LGDSP_COL_n_sat_low_cons] = (double)cons_low + bad; ro[LGDSP_COL_n_sat_high_cons] = (double)cons_high + bad;
                } else {
                    const bool ok = tlbad == 0.0;
                    ro[LGDSP_COL_tail_mean] = (ok ? st.mean : 0.0) + bad; ro[LGDSP_COL_tail_sigma] = (ok ? st.sigma : 0.0) + bad;
                    ro[LGDSP_COL_tail_tau] = (ok ? div_rn(-1.0, st.slope) : 0.0) + bad;
                }
            }
        } else if (wid == 6) {
            const double Ymax = red_max(red, K1R_YMAX);
            if (lane == 0) { ax[AX_M] = m; ax[AX_EMAX] = e_max; ax[AX_YMAX] = Ymax; ax[AX_BAD] = wrapped ? 1.0 : 0.0; }
        }
        __syncthreads();   // ---- B3: reduction slots / masks may be reused ----
    }
}

// ==================================================================================================
// extract kernel
// ==================================================================================================
constexpr int NT2 = 256;
constexpr int NW2 = NT2 / 32;
static_assert(NT2 == NT && NW2 == NWARP, "the extract kernel shares the block-reduction helpers and the 33-sample chunking");
enum { MK_T0 = 0, MK_T0INV, MK_CUR, MK_PILE, MK_N };
enum { K2R_PZS = 0, K2R_PZSS, K2R_PZSX, K2R_E104, K2R_E104N, K2R_E313, K2R_E313N, K2R_C535, K2R_CET, K2R_SGMAX, K2R_SGS, K2R_SGSS,
       K2R_CMAX0, K2R_CMAX1, K2R_CMAX2, K2R_CMAX3, K2R_CARG0, K2R_CARG1, K2R_CARG2, K2R_CARG3, K2R_E535, K2R_ETMAX, K2R_ETARG, K2R_N };
constexpr int K2_NTYPE = 5;                                 // flagged-interval types
constexpr int K2_TT = 0;                                    // double TT[TT_LEN]
constexpr int K2_MASK = K2_TT + TT_LEN * 8;                 // uint32 masks[MK_N][NWORDS]
constexpr int K2_RED = K2_MASK + MK_N * NWORDS * 4;         // double red[K2R_N][NW2]
constexpr int K2_STASH = K2_RED + K2R_N * NW2 * 8;          // double stash[LGDSP_MAX_DNI]: trap(rt,ft) outputs of the pick-off window
constexpr int K2_ROW = K2_STASH + LGDSP_MAX_DNI * 8;        // double row[64]
constexpr int K2_AUX = K2_ROW + 64 * 8;                     // double aux[AUX_LEN]
constexpr int K2_SGG = K2_AUX + AUX_LEN * 8;                // double sgg[3][8]
constexpr int K2_FLAG = K2_SGG + 24 * 8;                    // uint8 flagb[NT2]: flagged-interval types of every coarse interval
constexpr int K2_BAR = K2_FLAG + NT2;
constexpr int K2_TOTAL = K2_BAR + 16;
static_assert(3 * (K2_TOTAL + 1024) <= 233472, "three CTAs per SM");

// GMASK != 0: the column-group mask is a compile-time constant (the full chain and the lean configs[1] group get their own
// instantiation without the other's branches: smaller hot code for the instruction cache); 0: mask from the parameter block
template <unsigned GMASK>
__global__ void __launch_bounds__(NT2, 3)
icpc_extract_kernel(const __grid_constant__ IcpcDev P, const double* __restrict__ ttg, const double* __restrict__ auxg,
                    long long n_events, int write_cz_zeros, double* __restrict__ rows)
{
    extern __shared__ __align__(128) unsigned char smem[];
    double* TT = reinterpret_cast<double*>(smem + K2_TT);
    uint32_t* masks = reinterpret_cast<uint32_t*>(smem + K2_MASK);
    double* red = reinterpret_cast<double*>(smem + K2_RED);
    double* stash = reinterpret_cast<double*>(smem + K2_STASH);
    double* row = reinterpret_cast<double*>(smem + K2_ROW);
    double* aux = reinterpret_cast<double*>(smem + K2_AUX);
    double (*sgg)[8] = reinterpret_cast<double (*)[8]>(smem + K2_SGG);
    unsigned char* flagb = smem + K2_FLAG;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + K2_BAR);

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n = P.n;
    const uint32_t tt_bytes = (uint32_t)(n + 2) * 8u;
    const double t_first = P.t_first, dt = P.dt;
    const unsigned G = GMASK ? GMASK : P.groups;
    const double* A_int = P.dni_A;
    const double* A_sig = P.dni_A + LGDSP_MAX_DNI * 4;

    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    if (tid < TT_LEN - 2 - n) TT[n + 2 + tid] = 0.0;   // finite padding behind the loaded part (zero-padded SG kernels read it)
    if (tid < 24) sgg[tid >> 3][tid & 7] = P.sg[tid >> 3].gg[tid & 7];
    __syncthreads();
    auto sg_at = [&](int f, int j) -> double {
        return (P.sg[f].n_taps + 1 <= 8) ? sg_eval8(TT, sgg[f], j) : sg_eval(TT, P.sg[f].gg, P.sg[f].n_taps, j);
    };
    const int i0 = tid * CH;
    const int nsg = P.sg[0].nout;
    const bool want_cur = (G & LGDSP_GROUP_CURRENT) != 0, want_intr = (G & LGDSP_GROUP_INTRACE) != 0;

    uint32_t it = 0;
    for (long long e = blockIdx.x; e < n_events; e += gridDim.x, ++it) {
        // (the barrier that ended the previous event ordered every read of TT / masks / aux before this point)
        if (tid == 0) {
            fence_proxy_async();
            mbar_expect_tx(bar, tt_bytes);
            tma_load_1d(TT, ttg + e * TTG_LEN, tt_bytes, bar);
            // the next event of this CTA into L2 while this one computes: its bulk copy then runs at L2 speed (+2 %)
            if (e + gridDim.x < n_events) tma_prefetch_l2(ttg + (e + gridDim.x) * TTG_LEN, tt_bytes);
        }
#pragma unroll
        for (int q = 0; q < MK_N; ++q) masks[q * NWORDS + tid] = 0u;
        if (tid < AUX_LEN) aux[tid] = auxg[e * AUX_LEN + tid];
        mbar_wait(bar, it & 1u);

        // ==========================================================================================
        // phase A: window passes over TT that depend on nothing else
        // ==========================================================================================
        const bool lean = (G & LGDSP_GROUP_LEAN) != 0;   // BASELINE configs[1]: only {blmean, t0, t50, e_trap, e_10410}
        const TrapDev& T5 = lean ? P.e10410 : P.e535;    // the trapezoid whose maximum alone is wanted (coarse-to-fine)
        if (!lean) {
            double pz_S = 0, pz_SS = 0, pz_SX = 0;
#pragma unroll 2
            for (int idx = P.tail_from + tid; idx <= P.tail_until; idx += NT2) {
                const double y = TT[idx + 1] - TT[idx];
                const double X = t_first + (double)idx * dt;
                pz_S += y;
                pz_SS = fma(y, y, pz_SS);
                pz_SX = fma(X, y, pz_SX);
            }
            pz_S = wsum_d(pz_S); pz_SS = wsum_d(pz_SS); pz_SX = wsum_d(pz_SX);
            if (lane == 0) {
                red[K2R_PZS * NW2 + wid] = pz_S; red[K2R_PZSS * NW2 + wid] = pz_SS; red[K2R_PZSX * NW2 + wid] = pz_SX;
            }
        }
        // (lean: only the MAXIMUM of the (10 us, 4 us) trapezoid is wanted, so it is pruned coarse-to-fine like e_535 below -- T5)
        if (!lean && (G & LGDSP_GROUP_TRAPS)) {
            double o4[4];
            trap_full2_minmax(TT, P.e10410, P.e313, tid, o4);
            const double a = wmax_d(o4[0]), b = wmax_d(o4[1]), c = wmax_d(o4[2]), d = wmax_d(o4[3]);
            if (lane == 0) {
                red[K2R_E104 * NW2 + wid] = a; red[K2R_E104N * NW2 + wid] = b;
                red[K2R_E313 * NW2 + wid] = c; red[K2R_E313N * NW2 + wid] = d;
            }
        }
        // coarse grid (outputs 33*tid and 33*(tid+1)) of the pruned trapezoids
        double c0a = 0, c0b = 0, cia = 0, cib = 0, c5a = -CUDART_INF, c5b = -CUDART_INF, cea = -CUDART_INF, ceb = -CUDART_INF;
        {
            const int ja = i0, jb = i0 + CH;
            if (G & LGDSP_GROUP_TIMING) {
                if (ja < P.t0.nout) c0a = trap_at_i(TT, P.t0, ja);
                if (jb < P.t0.nout) c0b = trap_at_i(TT, P.t0, jb);
                if (!P.t0inv_same && !lean) {
                    if (ja < P.t0inv.nout) cia = trap_at_i(TT, P.t0inv, ja);
                    if (jb < P.t0inv.nout) cib = trap_at_i(TT, P.t0inv, jb);
                }
            }
            if (G & LGDSP_GROUP_TRAPS) {
                if (ja < T5.nout) c5a = trap_at_i(TT, T5, ja);
                if (jb < T5.nout) c5b = trap_at_i(TT, T5, jb);
                const double w5 = wmax_d(c5a);
                red_put(red, K2R_C535, wid, lane, w5);
                if (!lean) {
                    if (ja < P.etrap.nout) cea = trap_at_i(TT, P.etrap, ja);
                    if (jb < P.etrap.nout) ceb = trap_at_i(TT, P.etrap, jb);
                    const double we = wmax_d(cea);
                    red_put(red, K2R_CET, wid, lane, we);
                }
            }
        }
        double sgcmax = -CUDART_INF;
        if (want_cur || want_intr) {
            double cmax[4] = {-CUDART_INF, -CUDART_INF, -CUDART_INF, -CUDART_INF};
            int carg[4] = {0x7fffffff, 0x7fffffff, 0x7fffffff, 0x7fffffff};
            double sg_S = 0, sg_SS = 0;
            if (want_intr) sg_chunk(TT, P.sg[0], i0, min(CH, nsg - i0), [&](int k, double s) { sgcmax = s > sgcmax ? s : sgcmax; });
#pragma unroll 1
            for (int f = 0; f < 3; ++f) {
                if (f > 0 && P.sg_alias[f] >= 0) continue;
                if (f > 0 && !want_cur) continue;
                double bm = -CUDART_INF;
                int ba = 0x7fffffff;
                if (P.sg[f].n_taps + 1 <= 8) {
                    double g[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) g[q] = sgg[f][q];
                    auto ev = [&](int j) -> double {
                        const double* p = TT + j;
                        double a0 = g[0] * p[0], a1 = g[1] * p[1];
                        a0 = fma(g[2], p[2], a0); a1 = fma(g[3], p[3], a1);
                        a0 = fma(g[4], p[4], a0); a1 = fma(g[5], p[5], a1);
                        a0 = fma(g[6], p[6], a0); a1 = fma(g[7], p[7], a1);
                        return a0 + a1;
                    };
                    if (want_cur) {
#pragma unroll 2
                        for (int j = P.cur_from[f] + tid; j <= P.cur_until[f]; j += NT2) {
                            const double v = ev(j);
                            if (v > bm) { bm = v; ba = j; }
                        }
                    }
                    if (f == 0 && want_intr) {
#pragma unroll 2
                        for (int j = P.intr_from + tid; j <= P.intr_until; j += NT2) {
                            const double v = ev(j);
                            sg_S += v;
                            sg_SS = fma(v, v, sg_SS);
                        }
                    }
                } else {
                    if (want_cur) {
#pragma unroll 1
                        for (int j = P.cur_from[f] + tid; j <= P.cur_until[f]; j += NT2) {
                            const double v = sg_at(f, j);
                            if (v > bm) { bm = v; ba = j; }
                        }
                    }
                    if (f == 0 && want_intr) {
#pragma unroll 1
                        for (int j = P.intr_from + tid; j <= P.intr_until; j += NT2) {
                            const double v = sg_at(0, j);
                            sg_S += v;
                            sg_SS = fma(v, v, sg_SS);
                        }
                    }
                }
                if (f == 0) { cmax[0] = bm; carg[0] = ba; } else if (f == 1) { cmax[1] = bm; carg[1] = ba; } else { cmax[2] = bm; carg[2] = ba; }
            }
            if (want_cur) {
#pragma unroll 2
                for (int j = P.cur_from[3] + tid; j <= P.cur_until[3]; j += NT2) {
                    const double d = deriv_at(TT, j);
                    if (d > cmax[3]) { cmax[3] = d; carg[3] = j; }
                }
            }
            const double wsm = wmax_d(sgcmax);
            sg_S = wsum_d(sg_S); sg_SS = wsum_d(sg_SS);
#pragma unroll
            for (int f = 0; f < 4; ++f) cmax[f] = wargmax_d(cmax[f], carg[f]);
            if (lane == 0) {
                red[K2R_SGMAX * NW2 + wid] = wsm; red[K2R_SGS * NW2 + wid] = sg_S; red[K2R_SGSS * NW2 + wid] = sg_SS;
#pragma unroll
                for (int f = 0; f < 4; ++f) {
                    red[(K2R_CMAX0 + f) * NW2 + wid] = cmax[f];
                    red[(K2R_CARG0 + f) * NW2 + wid] = (double)carg[f];
                }
            }
        }
        __syncthreads();   // ---- BA ----

        // ==========================================================================================
        // phase B: decisions that need block-wide values; flagged intervals
        // ==========================================================================================
        if (tid < 64) row[tid] = 0.0;
        const double thr50 = aux[AX_THR + 1];
        const double Ymax = aux[AX_YMAX];
        const double kslack = 1e-7 * Ymax;
        // t10..t99 [us] from the positions the prefix kernel resolved; NaN -> 0
        auto tx_us = [&](int k) -> double {
            const int pos = (int)aux[AX_POS + k];
            const double th = aux[AX_THR + k];
            double t = 0.0;
            if (pos >= 1) t = cross_x(th, y_at(TT, pos - 1), y_at(TT, pos), t_first + (double)(pos - 1) * dt, dt) * 0.001;
            return t != t ? 0.0 : t;
        };
        // DNI window of the trap(rt,ft) energy pick-off at t50 + pick (every thread: uniform values)
        double pk_p;
        int pk_from;
        {
            double t50_us = 0.0;
            const int pos = (int)aux[AX_POS + 1];
            if (pos >= 1) {
                const double x = cross_x(thr50, y_at(TT, pos - 1), y_at(TT, pos), t_first + (double)(pos - 1) * dt, dt);
                t50_us = x * 0.001;
            }
            const double tf = t_first + (double)(P.etrap.L - 1) * dt;
            dni_window(P.sig_dni.n_w, n - P.etrap.L + 1, (t50_us * 1000.0 + P.trap_pick - tf) / dt, pk_p, pk_from);
        }
        if ((G & LGDSP_GROUP_TRAPS) && tid < P.sig_dni.n_w) stash[tid] = trap_at_i(TT, P.etrap, pk_from + tid);

        double pile_thr = 0.0, cur_thr = 0.0;
        if (G & LGDSP_GROUP_INTRACE) {
            cur_thr = red_max(red, K2R_SGMAX) * 0.5;
            const double sS = red_sum(red, K2R_SGS), sSS = red_sum(red, K2R_SGSS);
            const double mean_Y = mul_rn(sS, P.intr_inv_n);
            double var_Y = sub_rn(mul_rn(sSS, P.intr_inv_n), mul_rn(mean_Y, mean_Y));
            if (var_Y < 0) var_Y = 0;
            pile_thr = sqrt(var_Y) * P.nsigma;
            if (pile_thr == 0.0) pile_thr = 1.0;  // src/dsp_routines.jl:77
        }
        double e535 = c5a, etmax = cea;
        int etarg = (cea > -CUDART_INF) ? i0 : 0x7fffffff;
        // one flagged interval / chunk q, evaluated by a whole warp (one output per lane); types as in icpc_kernel
        auto do_item = [&](int type, int q) {
            if (type <= 1) {
                const TrapDev& tr = type == 0 ? P.t0 : P.t0inv;
                const double th = P.t0_thr;
                const int j = q * CH + 1 + lane;
                const bool v = j < tr.nout;
                const double o = v ? trap_at_i(TT, tr, j) : 0.0;
                const unsigned mp = __ballot_sync(FULL, v && (o >= th));
                const unsigned mn_ = __ballot_sync(FULL, v && (-o >= th));
                commit_pair(type == 0 ? masks + MK_T0 * NWORDS : nullptr, (unsigned long long)mp << 1,
                            ((type == 1 || P.t0inv_same) && !lean) ? masks + MK_T0INV * NWORDS : nullptr, (unsigned long long)mn_ << 1,
                            false, 0, q, lane);
            } else if (type == 2) {
                const int j = q * CH + 1 + lane;
                if (j < T5.nout) {
                    const double o = trap_at_i(TT, T5, j);
                    e535 = o > e535 ? o : e535;
                }
            } else if (type == 3) {
                const int j = q * CH + 1 + lane;
                if (j < P.etrap.nout) {
                    const double o = trap_at_i(TT, P.etrap, j);
                    if (o > etmax || (o == etmax && j < etarg)) { etmax = o; etarg = j; }
                }
            } else {
                const int j = q * CH + lane;
                const bool v = j < nsg;
                const double sv = v ? sg_at(0, j) : 0.0;
                const int j2 = q * CH + 32;
                const double s2 = (j2 < nsg) ? sg_at(0, j2) : -CUDART_INF;
                const unsigned long long bc = (unsigned long long)__ballot_sync(FULL, v && (sv >= cur_thr)) |
                                              ((s2 >= cur_thr) ? (1ull << 32) : 0ull);
                const unsigned long long bp = (unsigned long long)__ballot_sync(FULL, v && (sv >= pile_thr)) |
                                              ((s2 >= pile_thr) ? (1ull << 32) : 0ull);
                commit_pair(masks + MK_CUR * NWORDS, bc, masks + MK_PILE * NWORDS, bp, true, nsg, q, lane);
            }
        };
        unsigned flags = 0;
        {
            bool f0 = false, fi = false, f5 = false, fe = false;
            if (G & LGDSP_GROUP_TIMING) {
                const double th = P.t0_thr;
                const int rule = P.t0_min_n >= 2 * CH ? 2 : (P.t0_min_n > CH ? 1 : 0);
                auto need = [&](bool a, bool b, bool valid) -> bool {
                    bool prev = __shfl_up_sync(FULL, a, 1), next = __shfl_down_sync(FULL, b, 1);
                    if (lane == 0) prev = true;
                    if (lane == 31) next = true;
                    if (!valid) return false;
                    return rule == 2 ? ((a && b) || (a && prev) || (b && next)) : (rule == 1 ? (a || b) : true);
                };
                {
                    const bool va = i0 < P.t0.nout, vb = i0 + CH < P.t0.nout;
                    const bool pa = va && (c0a >= th), pb = vb && (c0b >= th);
                    const bool na = va && (-c0a >= th), nb = vb && (-c0b >= th);
                    const bool fp = need(pa, pb, va), fn = need(na, nb, va);
                    f0 = (P.t0inv_same && !lean) ? (fp || fn) : fp;
                    if (pa) mask_commit(masks + MK_T0 * NWORDS, tid, 1ull);
                    if (P.t0inv_same && na && !lean) mask_commit(masks + MK_T0INV * NWORDS, tid, 1ull);
                }
                if (!P.t0inv_same && !lean) {
                    const bool wa = i0 < P.t0inv.nout, wb = i0 + CH < P.t0inv.nout;
                    const bool na = wa && (-cia >= th), nb = wb && (-cib >= th);
                    fi = need(na, nb, wa);
                    if (na) mask_commit(masks + MK_T0INV * NWORDS, tid, 1ull);
                }
            }
            if (G & LGDSP_GROUP_TRAPS) {
                const double M5 = red_max(red, K2R_C535);
                const double k5 = Ymax * 2.0 * (T5.inv1 + T5.inv2) * 1.000001;
                if (i0 + 1 < T5.nout) f5 = interval_bound(c5a, c5b, i0 + CH < T5.nout, k5) + kslack >= M5;
                if (!lean) {
                    const double Me = red_max(red, K2R_CET);
                    const double ke = Ymax * 2.0 * (P.etrap.inv1 + P.etrap.inv2) * 1.000001;
                    if (i0 + 1 < P.etrap.nout) fe = interval_bound(cea, ceb, i0 + CH < P.etrap.nout, ke) + kslack >= Me;
                }
            }
            flags = (f0 ? 1u : 0u) | (fi ? 2u : 0u) | (f5 ? 4u : 0u) | (fe ? 8u : 0u);
        }
        if (G & LGDSP_GROUP_INTRACE) {
            const bool flag = sgcmax >= fmin(cur_thr, pile_thr);
            const unsigned bf = __ballot_sync(FULL, flag);
            if (__popc(bf) > 10) {
                if (flag) {
                    unsigned long long bc = 0, bp = 0;
                    sg_chunk(TT, P.sg[0], i0, min(CH, nsg - i0), [&](int k, double s) {
                        bc |= (s >= cur_thr) ? (1ull << k) : 0ull;
                        bp |= (s >= pile_thr) ? (1ull << k) : 0ull;
                    });
                    mask_commit(masks + MK_CUR * NWORDS, tid, bc);
                    mask_commit_reversed(masks + MK_PILE * NWORDS, tid, bp, nsg);
                }
            } else if (flag) {
                flags |= 16u;
            }
        }
        // The flagged intervals are re-dealt through shared memory: after the barrier warp w evaluates the intervals
        // q = NW2 * lane + w, so the few neighbouring intervals of the pulse region go to different warps instead of all to the
        // warp that owns them (no queue, no atomics, deterministic order).
        flagb[tid] = (unsigned char)flags;
        __syncthreads();   // ---- BB1 ----
        {
            const unsigned myf = flagb[NW2 * lane + wid];
#pragma unroll 1
            for (int type = 0; type < K2_NTYPE; ++type) {
                unsigned word = __ballot_sync(FULL, (myf >> type) & 1u);
                while (word) {
                    const int bq = __ffs(word) - 1;
                    word &= word - 1;
                    do_item(type, NW2 * bq + wid);
                }
            }
            e535 = wmax_d(e535);
            etmax = wargmax_d(etmax, etarg);
            if (lane == 0) {
                red[K2R_E535 * NW2 + wid] = e535;
                red[K2R_ETMAX * NW2 + wid] = etmax; red[K2R_ETARG * NW2 + wid] = (double)etarg;
            }
        }
        __syncthreads();   // ---- BB2: masks and trapezoid partials complete ----

        // ==========================================================================================
        // phase C: scalar results, one self-contained job per warp
        // ==========================================================================================
        auto t0_us = [&](bool inv, int pos) -> double {
            const TrapDev& tr = inv ? P.t0inv : P.t0;
            double t = 0.0;
            if (pos >= 1) {
                const double tl = t_first + (double)(pos - 1 + tr.L - 1) * dt;
                const double sgn = inv ? -1.0 : 1.0;
                t = cross_x(P.t0_thr, sgn * trap_at_i(TT, tr, pos - 1), sgn * trap_at_i(TT, tr, pos), tl, dt) * 0.001;
            }
            return t != t ? 0.0 : t;
        };
        auto qdrift_warp = [&](double t_us, double first, double last) -> double {
            const double tns = t_us * 1000.0;
            if (P.int_dni.n_w <= 8) {
                const int g = lane >> 3;
                const double ts = g == 0 ? tns : (g == 1 ? tns + first : tns + last);
                double pc;
                int from;
                dni_window(P.int_dni.n_w, n, (ts - t_first) / dt, pc, from);
                const double r = dni3_warp(A_int, P.int_dni.n_w, P.int_dni.m, TT + 1, from, pc - (double)from, lane);
                const double a0 = __shfl_sync(FULL, r, 0), a1 = __shfl_sync(FULL, r, 8), a2 = __shfl_sync(FULL, r, 16);
                return (a2 - a1) - (a1 - a0);
            }
            double a[3];
#pragma unroll 1
            for (int q = 0; q < 3; ++q) {
                const double ts = q == 0 ? tns : (q == 1 ? tns + first : tns + last);
                double pc;
                int from;
                dni_window(P.int_dni.n_w, n, (ts - t_first) / dt, pc, from);
                a[q] = dni_eval_warp(A_int, P.int_dni.n_w, P.int_dni.m, TT + from + 1, pc - (double)from, lane);
            }
            const double area1 = a[1] - a[0], area2 = a[2] - a[1];
            return area2 - area1;
        };
        if (wid == 0 && !lean) {
            // PZ tail statistics (signalstats on the tail window, src/dsp_icpc.jl:123)
            const double pzS = red_sum(red, K2R_PZS), pzSS = red_sum(red, K2R_PZSS), pzSX = red_sum(red, K2R_PZSX);
            if (lane == 0) {
                const Stats st = stats_finalize(P.tail_inv_n, P.tail_sX, P.tail_sXX, pzS, pzSS, pzSX);
                row[LGDSP_COL_tailmean] = st.mean; row[LGDSP_COL_tailsigma] = st.sigma;
                row[LGDSP_COL_tailslope] = st.slope; row[LGDSP_COL_tailoffset] = st.offset;
            }
            // t0 of the inverted waveform (src/dsp_icpc.jl:207) here: warp 1 then resolves one mask, not two (the two long-run
            // resolutions in a row made it the slowest job of the phase)
            if (G & LGDSP_GROUP_TIMING) {
                int pos0i, mult_;
                resolve_runs(masks + MK_T0INV * NWORDS, P.t0_min_n, lane, pos0i, mult_);
                if (lane == 0) row[LGDSP_COL_t0_inv] = t0_us(true, pos0i);
            }
        } else if (wid == 1) {
            int pos0, mult_;
            resolve_runs(masks + MK_T0 * NWORDS, P.t0_min_n, lane, pos0, mult_);
            double t = 0.0;
            if (lane < 5) {
                t = tx_us(lane);
                if (G & LGDSP_GROUP_TIMING) row[LGDSP_COL_t10 + lane] = t;
            } else if (lane == 5) {
                t = t0_us(false, pos0);
                if (G & LGDSP_GROUP_TIMING) row[LGDSP_COL_t0] = t;
            }
            const double t90 = __shfl_sync(FULL, t, 3), t0v = __shfl_sync(FULL, t, 5);
            if (lane == 0 && (G & LGDSP_GROUP_TIMING)) row[LGDSP_COL_drift_time] = (t90 - t0v) * 1000.0;
        } else if (wid == 2) {
            if (G & LGDSP_GROUP_TRAPS) {
                const double v = dni_eval_warp(A_sig, P.sig_dni.n_w, P.sig_dni.m, stash, pk_p - (double)pk_from, lane);
                if (lean) {
                    const double a = red_max(red, K2R_E535);   // (the pruned maximum of T5 = e_10410)
                    if (lane == 0) { row[LGDSP_COL_e_10410] = a; row[LGDSP_COL_e_trap] = v; }
                }
                double em = 0;
                int ea = 0;
                if (!lean) red_argmax(red, K2R_ETMAX, K2R_ETARG, em, ea);
                const double a = lean ? 0.0 : red_max(red, K2R_E104), b = lean ? 0.0 : red_max(red, K2R_E535), c = lean ? 0.0 : red_max(red, K2R_E313);
                const double d = lean ? 0.0 : red_max(red, K2R_E104N), f = lean ? 0.0 : red_max(red, K2R_E313N);
                if (lane == 0 && !lean) {
                    row[LGDSP_COL_e_10410] = a; row[LGDSP_COL_e_535] = b; row[LGDSP_COL_e_313] = c;
                    row[LGDSP_COL_e_10410_inv] = d; row[LGDSP_COL_e_313_inv] = f;
                    row[LGDSP_COL_e_trap_max] = em;
                    row[LGDSP_COL_t_trap_max] = t_first + (double)(ea + P.etrap.L - 1) * dt;
                    row[LGDSP_COL_e_trap] = v;
                }
            }
        } else if (wid == 3) {
            if (G & LGDSP_GROUP_CURRENT) {
                // get_wvf_maximum  src/interpolation.jl:30-46: parabola only if strictly inside the window
                double vv[4];
                int aa[4];
#pragma unroll
                for (int f = 0; f < 4; ++f) {
                    const int fs = (f < 3 && P.sg_alias[f] >= 0) ? P.sg_alias[f] : f;
                    red_argmax(red, K2R_CMAX0 + fs, K2R_CARG0 + fs, vv[f], aa[f]);
                }
                if (lane < 4) {
                    const int f = lane;
                    double v = f == 0 ? vv[0] : f == 1 ? vv[1] : f == 2 ? vv[2] : vv[3];
                    const int a = f == 0 ? aa[0] : f == 1 ? aa[1] : f == 2 ? aa[2] : aa[3];
                    if (a > P.cur_from[f] && a < P.cur_until[f]) {
                        const double y1 = (f < 3) ? sg_at(f, a - 1) : deriv_at(TT, a - 1);
                        const double y3 = (f < 3) ? sg_at(f, a + 1) : deriv_at(TT, a + 1);
                        v = extrema3(y1, v, y3);
                    }
                    row[LGDSP_COL_a_sg + f] = v;
                }
            }
        } else if (wid == 4) {
            if (G & LGDSP_GROUP_INTRACE) {
                int posc, multc;
                resolve_runs(masks + MK_CUR * NWORDS, P.tx_min_n, lane, posc, multc);
                if (lane == 0) {
                    // t50_current  src/dsp_icpc.jl:192-195
                    const double tf = t_first + (double)P.sg[0].offset * dt;
                    double t = 0.0;
                    if (posc >= 1) {
                        t = cross_x(cur_thr, sg_at(0, posc - 1), sg_at(0, posc), tf + (double)(posc - 1) * dt, dt) * 0.001;
                        if (t != t) t = 0.0;
                    }
                    row[LGDSP_COL_t50_current] = t;
                }
            }
        } else if (wid == 5) {
            if (G & LGDSP_GROUP_INTRACE) {
                // in-trace pile-up  src/dsp_routines.jl:72-82 (reversed trace r[j] = s[nsg-1-j], same time axis)
                int posp, multp;
                resolve_runs(masks + MK_PILE * NWORDS, P.intr_min_n, lane, posp, multp);
                if (lane == 0) {
                    const double tf = t_first + (double)P.sg[0].offset * dt;
                    double xi = CUDART_NAN;
                    if (posp >= 1) {
                        const double yl = sg_at(0, nsg - 1 - (posp - 1)), yr = sg_at(0, nsg - 1 - posp);
                        xi = cross_x(pile_thr, yl, yr, tf + (double)(posp - 1) * dt, dt);
                    }
                    const double last_t = tf + (double)(nsg - 1) * dt;
                    row[LGDSP_COL_inTrace_intersect] = last_t - xi;
                    row[LGDSP_COL_inTrace_n] = (double)multp;
                }
            }
        } else if (wid == 7) {
            if (G & LGDSP_GROUP_QDRIFT) {
                int pos0, mult_;
                resolve_runs(masks + MK_T0 * NWORDS, P.t0_min_n, lane, pos0, mult_);
                const double v = qdrift_warp(t0_us(false, pos0), P.qd_first, P.qd_last);   // qdrift @ t0
                if (lane == 0) row[LGDSP_COL_qdrift] = v;
            }
        } else if (wid == 6) {
            if (G & LGDSP_GROUP_QDRIFT) {
                const double v = qdrift_warp(tx_us(2), P.lq_first, P.lq_last);       // lq @ t80
                if (lane == 0) row[LGDSP_COL_lq] = v;
            }
        }
        __syncthreads();   // ---- BC ----
        // this kernel's columns (the prefix kernel wrote the raw-sample statistics, the CUSP/ZAC kernel writes its six)
        if (tid < LGDSP_NCOL) {
            const bool k1col = tid <= LGDSP_COL_bloffset || tid == LGDSP_COL_qc_label ||
                               (tid >= LGDSP_COL_tail_tau && tid <= LGDSP_COL_e_min) || tid >= LGDSP_COL_n_sat_low;
            const bool k3col = tid == LGDSP_COL_e_cusp || tid == LGDSP_COL_e_zac || tid == LGDSP_COL_e_cusp_max ||
                               tid == LGDSP_COL_e_zac_max || tid == LGDSP_COL_t_cusp_max || tid == LGDSP_COL_t_zac_max;
            if (!k1col && (!k3col || write_cz_zeros)) rows[e * LGDSP_NCOL + tid] = aux[AX_BAD] != 0.0 ? CUDART_NAN : row[tid];
        }
        // (phase B of the next event zeroes `row` behind its first barrier: every thread has stored its column by then)
    }
}

// ==================================================================================================
// CUSP / ZAC: select kernel (prefix tables, coarse grid, candidate chunks) + finish kernel (recurrences, one lane per
// candidate chunk, one warp per event)
// ==================================================================================================
// In icpc_kernel the 33-step recurrences of the ~25 candidate chunks of an event run in the two or three warps that own
// them while the rest of the block waits at a barrier (a fifth of the samples of that kernel).  Here the block only selects
// the candidates and hands their closed-form window states over; a second kernel steps the recurrences with one LANE per
// candidate chunk and one warp per event, so the serial part is 33 full-width steps per event and nobody waits for it.
constexpr int CZ_REC = 12;                    // doubles per candidate record: the 11 window states + the chunk index
constexpr int CZ_MAXC = NT;                   // candidate capacity per (event, pass): every chunk
constexpr int CZ_HDR = 16;                    // doubles per (event, pass) header
enum { CZH_N = 0, CZH_MAXC, CZH_ARGC, CZH_MAXZ, CZH_ARGZ, CZH_PKP0, CZH_PKF0, CZH_PKP1, CZH_PKF1,
       CZH_CNT };                                    // (pass 0 only) arrival counter of the finish kernel's warps, zeroed here
constexpr int CZP_LEN = CZ_HDR + CZ_MAXC * CZ_REC;   // doubles per (event, pass)
constexpr int K4_NBLK = 4;                           // warps of the finish kernel that may share one event
constexpr int CZ_SCR = K4_NBLK * 4 + 2 * LGDSP_MAX_DNI;   // their exchange area: partial (max, argmax) x 2 + the two pick-off windows
constexpr int CZG_LEN = 2 * CZP_LEN + CZ_SCR;        // doubles per event slot

enum { K3R_CZC0 = 0, K3R_CZC1, K3R_CZMAX0, K3R_CZARG0, K3R_CZMAX1, K3R_CZARG1, K3R_CZSCR, K3R_CZSCR1, K3R_CZSCR2, K3R_CZSCR3, K3R_N };
enum { K3I_CZN = 0, K3I_PKFROM = 1 /* 2 */, K3I_N = 4 };
constexpr int K3_TT = 0;
constexpr int K3_TABA = K3_TT + TT_LEN * 8;                 // double tabA[8][NT]
constexpr int K3_TABB = K3_TABA + 8 * NT * 8;               // double tabB[8][NT]: tables 8..15 (contiguous with tabA: cz_scan<.., true>)
constexpr int K3_CZCO = K3_TABB + 8 * NT * 8;               // double czco[2][NT]: coarse CUSP / ZAC values
constexpr int K3_RED = K3_CZCO + 2 * NT * 8;
constexpr int K3_STASH = K3_RED + K3R_N * NWARP * 8;        // double stash[2][LGDSP_MAX_DNI] (direct mode)
constexpr int K3_SCR = K3_STASH + 2 * LGDSP_MAX_DNI * 8;    // double scr[8]: pk_p[2], pp0, Ymax
constexpr int K3_IBUF = K3_SCR + 8 * 8;                     // int ibuf[K3I_N]
constexpr int K3_BAR = K3_IBUF + K3I_N * 4;
constexpr int K3_PAR = K3_BAR + 16;                         // SmemPar (CzDev copies for cz_scan)
constexpr int K3_TOTAL = K3_PAR + (int)sizeof(SmemPar);
static_assert(2 * (K3_TOTAL + 1024) <= 233472, "two CTAs per SM");
enum { K3S_PKP = 0 /* 2 */, K3S_PP0 = 2, K3S_YMAX = 3 };

// Candidate selection of one structured pass: closed-form window states at every chunk
// start (tab_c / tab_a read the prefix tables), coarse CUSP / ZAC values, Lipschitz bound against the best coarse value,
// candidate records + header -> cg.  Contains two block barriers; every thread of the block must call it.  tt_dead() runs in
// every thread right behind the first of them, from where on nothing here reads TT.
template <typename TC, typename TA, typename TD>
__device__ __forceinline__ void cz_select(const CzDev& Z, const double* TT, int n, int nw, double pp0, double Ymax, const int* pk_from,
                                          const double* pk_p, bool want_cusp, bool want_zac, double* czco, double* red, int* czn,
                                          double* cg, TC&& tab_c, TA&& tab_a, TD&& tt_dead)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int i0 = tid * CH;
    CzState st;
    st.active = false;
    double oc = -CUDART_INF, oz = -CUDART_INF;
    cz_init_with(Z, TT, n, tid, pp0, st, tab_c, tab_a);
    cz_coarse(Z, TT, n, tid, st, oc, oz);
    if (!want_cusp) oc = -CUDART_INF;
    if (!want_zac) oz = -CUDART_INF;
    // the coarse points are outputs themselves
    const int j0 = i0 - Z.L + 1;
    czco[tid] = oc;
    czco[NT + tid] = oz;
    {
        int ac = oc > -CUDART_INF ? j0 : 0x7fffffff, az = oz > -CUDART_INF ? j0 : 0x7fffffff;
        const double wc = wargmax_d(oc, ac), wz = wargmax_d(oz, az);
        if (lane == 0) {
            red[K3R_CZMAX0 * NWARP + wid] = wc; red[K3R_CZARG0 * NWARP + wid] = (double)ac;
            red[K3R_CZMAX1 * NWARP + wid] = wz; red[K3R_CZARG1 * NWARP + wid] = (double)az;
        }
    }
    __syncthreads();   // tables are dead, coarse values complete
    tt_dead();
    double Mc, Mz;
    int Ac, Az;
    red_argmax(red, K3R_CZMAX0, K3R_CZARG0, Mc, Ac);
    red_argmax(red, K3R_CZMAX1, K3R_CZARG1, Mz, Az);
    // candidate chunks: Lipschitz bound on (33 tid, 33 tid + 33) against the best coarse value; chunks that
    // hold part of a pick-off window are always evaluated
    bool cand = false;
    if (st.active) {
        const int t1 = min(tid + 1, NT - 1);
        const double kap = Ymax * 1.000001;
        const int jlo = i0 - Z.L + 1, jhi = jlo + CH - 1;
        if (want_cusp) {
            const double a = oc, b = (tid + 1 < NT) ? czco[t1] : -CUDART_INF;
            const double kc = kap * Z.lip_cusp;
            double bound;
            if (a > -CUDART_INF) bound = interval_bound(a, b, b > -CUDART_INF, kc);
            else if (b > -CUDART_INF) bound = fma((double)CH, kc, b);
            else bound = CUDART_INF;
            cand |= bound + 1e-6 * (fabs(Mc) + Ymax * fabs(Z.g)) >= Mc;
            cand |= (jhi >= pk_from[0] && jlo < pk_from[0] + nw);
        }
        if (want_zac) {
            const double a = oz, b = (tid + 1 < NT) ? czco[NT + t1] : -CUDART_INF;
            const double kz = kap * Z.lip_zac;
            double bound;
            if (a > -CUDART_INF) bound = interval_bound(a, b, b > -CUDART_INF, kz);
            else if (b > -CUDART_INF) bound = fma((double)CH, kz, b);
            else bound = CUDART_INF;
            cand |= bound + 1e-6 * (fabs(Mz) + Ymax * fabs(Z.g)) >= Mz;
            cand |= (jhi >= pk_from[1] && jlo < pk_from[1] + nw);
        }
    }
    // candidate records: the window states at the chunk start + the chunk index
    {
        const unsigned bc = __ballot_sync(FULL, cand);
        int base = 0;
        if (lane == 0 && bc) base = atomicAdd(czn, __popc(bc));
        base = __shfl_sync(FULL, base, 0);
        if (cand) {
            double* r = cg + CZ_HDR + (size_t)(base + __popc(bc & ((1u << lane) - 1u))) * CZ_REC;
            r[0] = st.EmL; r[1] = st.EpL; r[2] = st.W0L; r[3] = st.W1L; r[4] = st.W2L; r[5] = st.W0F;
            r[6] = st.V0; r[7] = st.V1; r[8] = st.V2; r[9] = st.EpR; r[10] = st.EmR; r[11] = (double)tid;
        }
    }
    __syncthreads();   // candidate count complete
    if (tid == 0) {
        cg[CZH_N] = (double)*czn;
        cg[CZH_MAXC] = Mc; cg[CZH_ARGC] = (double)Ac; cg[CZH_MAXZ] = Mz; cg[CZH_ARGZ] = (double)Az;
        cg[CZH_PKP0] = pk_p[0]; cg[CZH_PKF0] = (double)pk_from[0];
        cg[CZH_PKP1] = pk_p[1]; cg[CZH_PKF1] = (double)pk_from[1];
        cg[CZH_CNT] = 0.0;
    }
}

__global__ void __launch_bounds__(NT, 2)
icpc_cuspzac_kernel(const __grid_constant__ IcpcDev P, const double* __restrict__ ttg, const double* __restrict__ auxg,
                    long long n_events, double* __restrict__ czg, double* __restrict__ rows)
{
    extern __shared__ __align__(128) unsigned char smem[];
    double* TT = reinterpret_cast<double*>(smem + K3_TT);
    double* tabA = reinterpret_cast<double*>(smem + K3_TABA);
    double* tabB = reinterpret_cast<double*>(smem + K3_TABB);
    double* czco = reinterpret_cast<double*>(smem + K3_CZCO);
    double* red = reinterpret_cast<double*>(smem + K3_RED);
    double* stash = reinterpret_cast<double*>(smem + K3_STASH);
    double* scr = reinterpret_cast<double*>(smem + K3_SCR);
    int* ibuf = reinterpret_cast<int*>(smem + K3_IBUF);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + K3_BAR);
    SmemPar* spar = reinterpret_cast<SmemPar*>(smem + K3_PAR);

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n = P.n;
    const uint32_t tt_bytes = (uint32_t)(n + 2) * 8u;
    const double t_first = P.t_first, dt = P.dt;
    const double* A_sig = P.dni_A + LGDSP_MAX_DNI * 4;
    const int npass = P.direct ? 0 : (P.cz_shared ? 1 : 2);
    const int nw = P.sig_dni.n_w;

    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    if (tid < TT_LEN - 2 - n) TT[n + 2 + tid] = 0.0;
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&P.cz[0]);
        uint32_t* dst = reinterpret_cast<uint32_t*>(&spar->cz[0]);
        for (int i = tid; i < (int)(2 * sizeof(CzDev) / 4); i += NT) dst[i] = src[i];
    }
    __syncthreads();

    // one bulk copy of TT per event, one expect_tx per mbarrier phase (it & 1); the issuing thread orders the generic-proxy
    // reads of the previous event (made visible to it by a block barrier) before the copy with fence_proxy_async
    auto load_tt = [&](long long ee) {
        fence_proxy_async();
        mbar_expect_tx(bar, tt_bytes);
        tma_load_1d(TT, ttg + ee * TTG_LEN, tt_bytes, bar);
        // the event after it into L2 while this one computes: its bulk copy then runs at L2 speed (+2 %)
        if (ee + gridDim.x < n_events) tma_prefetch_l2(ttg + (ee + gridDim.x) * TTG_LEN, tt_bytes);
    };
    // structured passes: the first event's copy is issued here and every further one as soon as the last pass of the event
    // before has stopped reading TT (cz_select's tt_dead), so that it lands while that event's candidates are selected
    if (npass != 0 && tid == 0 && blockIdx.x < n_events) load_tt(blockIdx.x);

    uint32_t it = 0;
    for (long long e = blockIdx.x; e < n_events; e += gridDim.x, ++it) {
        if (tid == 0) {
            if (npass == 0) load_tt(e);
            ibuf[K3I_CZN] = 0;
        }
        mbar_wait(bar, it & 1u);
        // DNI windows of the two pick-offs (t50 + L/2) from the t50 position of the prefix kernel; Ymax
        if (wid == 0 && lane < 2) {
            const double* ax = auxg + e * AUX_LEN;
            const int pos = (int)ax[AX_POS + 1];
            double t50_us = 0.0;
            if (pos >= 1) {
                const double x = cross_x(ax[AX_THR + 1], y_at(TT, pos - 1), y_at(TT, pos), t_first + (double)(pos - 1) * dt, dt);
                t50_us = x * 0.001;
            }
            const int Lf = lane == 0 ? P.cusp_L : P.zac_L;
            const double pick = lane == 0 ? P.cusp_pick : P.zac_pick;
            const double tf = t_first + (double)(Lf - 1) * dt;
            double pp;
            int pf;
            dni_window(nw, n - Lf + 1, (t50_us * 1000.0 + pick - tf) / dt, pp, pf);
            scr[K3S_PKP + lane] = pp;
            ibuf[K3I_PKFROM + lane] = pf;
            if (lane == 0) scr[K3S_YMAX] = ax[AX_YMAX];
        }
        if (npass == 0) {
            // direct form (validation mode only): the whole evaluation in this kernel
            double czmax[2] = {-CUDART_INF, -CUDART_INF};
            int czarg[2] = {0x7fffffff, 0x7fffffff};
            __syncthreads();
            const int pk_from[2] = {ibuf[K3I_PKFROM], ibuf[K3I_PKFROM + 1]};
#pragma unroll 1
            for (int f = 0; f < 2; ++f) {
                const int L = f ? P.zac_L : P.cusp_L;
                const double* g = f ? P.zac_g : P.cusp_g;
                const int nout = n - L + 1;
                double bm = -CUDART_INF;
                int ba = 0x7fffffff;
#pragma unroll 1
                for (int j = tid; j < nout; j += NT) {
                    const double o = fir_at(TT, g, L, j);
                    if (o > bm) { bm = o; ba = j; }
                    const int r = j - pk_from[f];
                    if (r >= 0 && r < nw) stash[f * LGDSP_MAX_DNI + r] = o;
                }
                if (f == 0) { czmax[0] = bm; czarg[0] = ba; } else { czmax[1] = bm; czarg[1] = ba; }
            }
            czmax[0] = wargmax_d(czmax[0], czarg[0]);
            czmax[1] = wargmax_d(czmax[1], czarg[1]);
            if (lane == 0) {
                red[K3R_CZMAX0 * NWARP + wid] = czmax[0]; red[K3R_CZARG0 * NWARP + wid] = (double)czarg[0];
                red[K3R_CZMAX1 * NWARP + wid] = czmax[1]; red[K3R_CZARG1 * NWARP + wid] = (double)czarg[1];
            }
            __syncthreads();
            if (wid < 2) {
                const int f = wid;
                const double v = dni_eval_warp(A_sig, nw, P.sig_dni.m, stash + f * LGDSP_MAX_DNI,
                                               scr[K3S_PKP + f] - (double)ibuf[K3I_PKFROM + f], lane);
                double cm;
                int ca;
                red_argmax(red, f ? K3R_CZMAX1 : K3R_CZMAX0, f ? K3R_CZARG1 : K3R_CZARG0, cm, ca);
                if (lane == 0) {
                    const int L = f ? P.zac_L : P.cusp_L;
                    const double bad = auxg[e * AUX_LEN + AX_BAD] != 0.0 ? CUDART_NAN : 0.0;
                    double* ro = rows + e * LGDSP_NCOL;
                    ro[f ? LGDSP_COL_e_zac_max : LGDSP_COL_e_cusp_max] = cm + bad;
                    ro[f ? LGDSP_COL_t_zac_max : LGDSP_COL_t_cusp_max] = t_first + (double)(ca + L - 1) * dt + bad;
                    ro[f ? LGDSP_COL_e_zac : LGDSP_COL_e_cusp] = v + bad;
                }
            }
            __syncthreads();
            continue;
        }
        // One pass of the structured evaluation up to the candidate selection.  The descriptor index is a compile-time
        // constant so that its fields are immediate constant-bank operands.
        auto cz_pass = [&](auto psc, const bool want_cusp, const bool want_zac, const bool rescan, const bool last) {
            constexpr int ps = decltype(psc)::value;
            const CzDev& Z = P.cz[ps];
            double* cg = czg + e * CZG_LEN + ps * CZP_LEN;
            if (rescan) {
                __syncthreads();   // the previous pass is done with the tables, the coarse values and the counters
                if (tid == 0) ibuf[K3I_CZN] = 0;
            }
            cz_scan<K3_PAR, true>(ps, TT, n, tid, tabA, tabB, red + K3R_CZSCR * NWARP, scr + K3S_PP0);
            __syncthreads();   // tables (and the pick-off windows) are complete
            const int pk_from[2] = {ibuf[K3I_PKFROM], ibuf[K3I_PKFROM + 1]};
            cz_select(Z, TT, n, nw, scr[K3S_PP0], scr[K3S_YMAX], pk_from, scr + K3S_PKP, want_cusp, want_zac, czco, red,
                      &ibuf[K3I_CZN], cg,
                      [&](int q, int kind, int c) -> double { return tabA[(q * 3 + kind) * NT + c]; },
                      [&](int q, int c) -> double { return tabA[(12 + q) * NT + c]; },
                      [&]() {
                          // Past this barrier of the last pass nothing of this event reads TT again: the pick-off windows,
                          // the scan (cz_scan), the window states (cz_init_with) and the coarse grid (cz_coarse) are all
                          // behind it, and the rest of cz_select works on registers, czco, red, scr and the header.
                          if (last && tid == 0 && e + gridDim.x < n_events) load_tt(e + gridDim.x);
                      });
        };
        if (npass == 2) {
            cz_pass(std::integral_constant<int, 1>{}, false, true, false, false);
            cz_pass(std::integral_constant<int, 0>{}, true, false, true, true);
        } else {
            cz_pass(std::integral_constant<int, 0>{}, true, true, false, true);
        }
        __syncthreads();   // scr, ibuf may be overwritten by the next event
    }
}

// finish: one lane per candidate chunk, one warp per event -- and up to K4_NBLK warps for an event with more than 32
// candidates.  The kernel is bound by the latency of a round (33 dependent recurrence steps; cz_out_staged feeds them from shared memory), and
// 93 % of the events need one round (median 11 candidates) while the 3 % noise-only events, where all 248 chunks are
// candidates, needed eight rounds on one warp: they set the duration of every launch.  Warp w < n_events takes the first 32
// candidates of event w; the warps behind take the further blocks of the few events that have them (and exit at once
// otherwise).  Warps that share an event leave their partial maxima and pick-off windows in the event's slot of the ring;
// the last one to arrive (counter in the header) combines them.  Maxima / first indices do not depend on the order and the
// pick-off estimate is dni_eval_warp on the same values: bit-identical to one warp per event.
constexpr int K4_WARPS = 4;
__global__ void __launch_bounds__(K4_WARPS * 32, 5)
icpc_cuspzac_finish_kernel(const __grid_constant__ IcpcDev P, const double* __restrict__ ttg, const double* __restrict__ auxg,
                           double* __restrict__ czg, long long n_events, double* __restrict__ rows)
{
    __shared__ double stash_s[K4_WARPS][2][LGDSP_MAX_DNI];
    __shared__ __align__(16) double slab_s[K4_WARPS][CZ_SLAB];   // cz_out_staged
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int n = P.n;
    const int nw = P.sig_dni.n_w;
    const double* A_sig = P.dni_A + LGDSP_MAX_DNI * 4;
    const int npass = P.cz_shared ? 1 : 2;
    const long long w = (long long)blockIdx.x * K4_WARPS + wid;
    long long e;
    int kb;
    if (w < n_events) { e = w; kb = 0; }
    else { e = (w - n_events) / (K4_NBLK - 1); kb = 1 + (int)((w - n_events) % (K4_NBLK - 1)); }
    if (e >= n_events) return;
    double* ce = czg + e * CZG_LEN;
    int nwork = 1;
    {
        const int n0 = (int)ce[CZH_N], n1 = npass == 2 ? (int)ce[CZP_LEN + CZH_N] : 0;
        nwork = min(K4_NBLK, max(1, (max(n0, n1) + 31) >> 5));
    }
    if (kb >= nwork) return;
    const bool shared_event = nwork > 1;
    double* scr = ce + 2 * CZP_LEN;                       // [K4_NBLK][4] partials, then the two pick-off windows
    double* stash = shared_event ? scr + K4_NBLK * 4 : &stash_s[wid][0][0];
    {
        const double* TT = ttg + e * TTG_LEN;
        double czmax[2] = {-CUDART_INF, -CUDART_INF};
        int czarg[2] = {0x7fffffff, 0x7fffffff};
        int pk_from[2] = {0, 0};
        auto pass = [&](auto psc, const bool want_cusp, const bool want_zac) {
            constexpr int ps = decltype(psc)::value;
            const CzDev& Z = P.cz[ps];
            const double* cg = ce + ps * CZP_LEN;
            const int ncand = (int)cg[CZH_N];
            pk_from[0] = (int)cg[CZH_PKF0]; pk_from[1] = (int)cg[CZH_PKF1];
            if (lane == 0 && kb == 0) {
                // the coarse points are outputs themselves
                if (want_cusp) { czmax[0] = cg[CZH_MAXC]; czarg[0] = (int)cg[CZH_ARGC]; }
                if (want_zac) { czmax[1] = cg[CZH_MAXZ]; czarg[1] = (int)cg[CZH_ARGZ]; }
            }
#pragma unroll 1
            for (int c0 = 32 * kb; c0 < ncand; c0 += 32 * nwork) {
                const bool has = c0 + lane < ncand;
                CzState st;
                int chunk = 0;
                if (has) {
                    const double* r = cg + CZ_HDR + (size_t)(c0 + lane) * CZ_REC;
                    st.EmL = r[0]; st.EpL = r[1]; st.W0L = r[2]; st.W1L = r[3]; st.W2L = r[4]; st.W0F = r[5];
                    st.V0 = r[6]; st.V1 = r[7]; st.V2 = r[8]; st.EpR = r[9]; st.EmR = r[10];
                    chunk = (int)r[11];
                } else {
                    st.EmL = st.EpL = st.W0L = st.W1L = st.W2L = st.W0F = st.V0 = st.V1 = st.V2 = st.EpR = st.EmR = 0.0;
                }
                st.active = has;
                {
                    const int jb = chunk * CH - Z.L + 1;
                    cz_out_staged(Z, TT, n, chunk, has, min(32, ncand - c0), st, slab_s[wid], lane, [&](int k, double o_c, double o_z) {
                        const int j = jb + k;
                        if (want_cusp) {
                            if (o_c > czmax[0] || (o_c == czmax[0] && j < czarg[0])) { czmax[0] = o_c; czarg[0] = j; }
                            const int q = j - pk_from[0];
                            if (q >= 0 && q < nw && o_c > -CUDART_INF) stash[q] = o_c;
                        }
                        if (want_zac) {
                            if (o_z > czmax[1] || (o_z == czmax[1] && j < czarg[1])) { czmax[1] = o_z; czarg[1] = j; }
                            const int q = j - pk_from[1];
                            if (q >= 0 && q < nw && o_z > -CUDART_INF) stash[LGDSP_MAX_DNI + q] = o_z;
                        }
                    });
                }
            }
        };
        if (npass == 2) {
            pass(std::integral_constant<int, 1>{}, false, true);
            pass(std::integral_constant<int, 0>{}, true, false);
        } else {
            pass(std::integral_constant<int, 0>{}, true, true);
        }
        __syncwarp();
        czmax[0] = wargmax_d(czmax[0], czarg[0]);
        czmax[1] = wargmax_d(czmax[1], czarg[1]);
        const double* win = stash;
        if (shared_event) {
            if (lane == 0) {
                double* pr = scr + kb * 4;
                pr[0] = czmax[0]; pr[1] = (double)czarg[0]; pr[2] = czmax[1]; pr[3] = (double)czarg[1];
            }
            __threadfence();    // this warp's partials and pick-off samples are visible before it counts itself in
            __syncwarp();
            unsigned prev = 0;
            if (lane == 0) prev = atomicAdd(reinterpret_cast<unsigned*>(ce + CZH_CNT), 1u);
            prev = __shfl_sync(FULL, prev, 0);
            if (prev != (unsigned)(nwork - 1)) return;   // a later warp finishes the event
            __threadfence();
            double pm0 = -CUDART_INF, pm1 = -CUDART_INF;
            int pa0 = 0x7fffffff, pa1 = 0x7fffffff;
            if (lane < nwork) {
                const double* pr = scr + lane * 4;
                pm0 = __ldcg(pr); pa0 = (int)__ldcg(pr + 1); pm1 = __ldcg(pr + 2); pa1 = (int)__ldcg(pr + 3);
            }
            czmax[0] = wargmax_d(pm0, pa0); czarg[0] = pa0;
            czmax[1] = wargmax_d(pm1, pa1); czarg[1] = pa1;
            double* sm = &stash_s[wid][0][0];
            for (int i = lane; i < 2 * LGDSP_MAX_DNI; i += 32) sm[i] = __ldcg(stash + i);
            __syncwarp();
            win = sm;
        }
        // (the pick-off positions of the last pass, pass 0, read only here: they would hold four registers in the recurrence)
        const double vc = dni_eval_warp(A_sig, nw, P.sig_dni.m, win, ce[CZH_PKP0] - (double)pk_from[0], lane);
        const double vz = dni_eval_warp(A_sig, nw, P.sig_dni.m, win + LGDSP_MAX_DNI, ce[CZH_PKP1] - (double)pk_from[1], lane);
        if (lane == 0 && auxg[e * AUX_LEN + AX_BAD] != 0.0) {
            double* ro = rows + e * LGDSP_NCOL;
            ro[LGDSP_COL_e_cusp_max] = ro[LGDSP_COL_t_cusp_max] = ro[LGDSP_COL_e_cusp] = CUDART_NAN;
            ro[LGDSP_COL_e_zac_max] = ro[LGDSP_COL_t_zac_max] = ro[LGDSP_COL_e_zac] = CUDART_NAN;
        } else if (lane == 0) {
            double* ro = rows + e * LGDSP_NCOL;
            ro[LGDSP_COL_e_cusp_max] = czmax[0];
            ro[LGDSP_COL_t_cusp_max] = P.t_first + (double)(czarg[0] + P.cusp_L - 1) * P.dt;
            ro[LGDSP_COL_e_cusp] = vc;
            ro[LGDSP_COL_e_zac_max] = czmax[1];
            ro[LGDSP_COL_t_zac_max] = P.t_first + (double)(czarg[1] + P.zac_L - 1) * P.dt;
            ro[LGDSP_COL_e_zac] = vz;
        }
    }
}
