// Fused dsp_icpc kernel for sm_100a: one CTA (256 threads) per waveform, persistent over the event slice.
//
// Data flow per waveform (reference steps in brackets, /root/reference/src/dsp_icpc.jl):
//   TMA bulk copy (cp.async.bulk, 16 KB UInt16) HBM -> SMEM, prefetched one event ahead
//   P1  raw samples: saturation [:93-95], baseline regression sums [:102], min/max [:111-112], block scan of the
//       chunk sums (exact integers) -> P = cumsum(x), PP = cumsum(P) at every chunk start
//   P2  pole-zero in closed form y = w + km1*cumsum(w), w = x - blmean [:105,:119-120]; writes
//       TT[i+1] = cumsum(y)[i] (float64, SMEM); t10..t99 threshold masks [:132-136] only for chunks whose
//       [ymin, ymax] straddles a threshold; tail log-regression [:115] spread evenly over all threads
//   P3  everything that only needs TT: PZ tail stats [:123]; the two trapezoids whose minimum is needed
//       (e_10410, e_313 and their *_inv, [:147-154,:202-204]) in full; the other trapezoids [:126,:150,:160,:207]
//       on a COARSE grid (every 33rd output); Savitzky-Golay / derivative currents [:181-186]; prefix tables of the
//       CUSP/ZAC evaluation
//   P4  coarse-to-fine: an interval between two coarse points is only evaluated when it can matter --
//         maxima (e_535, e_trap_max, e_cusp_max, e_zac_max): |out[j+1]-out[j]| <= max|y| * sum_k |h[k]-h[k-1]| for any FIR
//           h (Lipschitz bound), so an interval whose bound stays below the best coarse value is skipped;
//         t0 / t0_inv (Intersect with mintot >= 34 samples): a qualifying run overlapping an interval must contain
//           one of its end points, so intervals whose end points are both below threshold are skipped;
//         t50_current / in-trace pile-up masks: only chunks whose maximum reaches the smaller threshold.
//       Both rules are exact (never change a result); how much they save is data dependent.
//       CUSP/ZAC [:167-178] through their analytic structure (sliding exponential/polynomial windows): closed-form
//       states at every chunk start give the coarse values; the 33-step recurrences run on candidate chunks only.
//   P5  crossing resolution with bit-parallel run detection (Intersect state machine, SURVEY.md App. B),
//       interpolated pick-offs (PolynomialDNI), qdrift/lq [:141-144], output row (49 doubles)
//
// Work mapping: scans use chunks of CH = 33 consecutive samples per thread (33 is odd: with the plain linear layout
// of TT the 32 lanes of a warp hit different banks for every window offset); all other passes are strided over the
// threads (consecutive lanes <-> consecutive samples), so windowed work is spread evenly.
// The waveform is read from HBM exactly once (16 KB) and 392 B are written.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include "lgdsp_device.cuh"
#include "lgdsp_kernels.h"

namespace lgdsp {

constexpr int NT = 256;          // threads per CTA
constexpr int NWARP = NT / 32;
constexpr int CH = CZ_CH;        // samples per thread in the scan passes (33)
constexpr int MAXN = LGDSP_MAX_SAMPLES;
constexpr int NWORDS = MAXN / 32;  // mask words
static_assert(NT * CH >= MAXN + 1, "chunks must cover the waveform");
static_assert(NWORDS == NT, "one mask word per thread");

// T10..T99 last: their 5 KB are reused for the coarse CUSP/ZAC values once they are resolved
enum { M_T0 = 0, M_T0INV, M_CUR, M_PILE, M_T10, M_T50, M_T80, M_T90, M_T99, NMASK };

// reduction slots: red[slot][warp].  The slots of the raw-sample pass (raw_pass) come first in icpc_kernel and in
// icpc_prefix_kernel alike.
enum { R_BLS = 0, R_BLSS, R_BLSX, R_MX /* + R_MN: 4 x NWARP uint32 */, R_MN, R_SLEN, R_SS, R_SQ, R_RAW_N };
enum {
    // stage C (after P2/P3)
    R_TLS = R_RAW_N, R_TLSS, R_TLSX, R_TLBAD, R_PZS, R_PZSS, R_PZSX, R_YMIN, R_YMAX,
    R_E104, R_E104N, R_E313, R_E313N, R_C535, R_CET, R_SGMAX, R_SGS, R_SGSS,
    R_CMAX0, R_CMAX1, R_CMAX2, R_CMAX3, R_CARG0, R_CARG1, R_CARG2, R_CARG3,
    // stage D
    R_CZC0, R_CZC1,
    // stage E
    R_E535, R_ETMAX, R_ETARG, R_CZMAX0, R_CZARG0, R_CZMAX1, R_CZARG1,
    // scratch of cz_scan (4 slots = 32 doubles)
    R_CZSCR, R_CZSCR1, R_CZSCR2, R_CZSCR3,
    NSLOT
};

// ---- shared memory carve-up (bytes) ----
constexpr int SM_XS = 0;                                   // uint16 xs[8192]  (aliased by CUSP/ZAC tables 0..7)
constexpr int TT_LEN = MAXN + 8;
constexpr int SM_TT = SM_XS + MAXN * 2;                    // double TT[8193+]
constexpr int SM_MASK = SM_TT + TT_LEN * 8;                // uint32 masks[NMASK][NWORDS]
constexpr int SM_RED = SM_MASK + NMASK * NWORDS * 4;       // double red[NSLOT][NWARP]
constexpr int SM_STASH = SM_RED + NSLOT * NWARP * 8;       // double stash[3][LGDSP_MAX_DNI]
constexpr int SM_TAB = SM_STASH + 3 * LGDSP_MAX_DNI * 8;   // double tabB[8][256]: CUSP/ZAC prefix tables 8..15
constexpr int SM_ROW = SM_TAB + 8 * NT * 8;                // double row[64]
constexpr int SM_SCR = SM_ROW + 64 * 8;                    // double scr[32]: scalars passed between warps
constexpr int SM_IBUF = SM_SCR + 32 * 8;                   // int ibuf[64]
constexpr int SM_BAR = SM_IBUF + 64 * 4;                   // uint64 mbarrier
constexpr int SM_PAR = SM_BAR + 16;                        // SmemPar: parameter tables read by the noinline helpers
struct SmemPar {
    CzDev cz[2];
    double sgg[3][8];      // zero-padded SG taps folded on TT (filters with <= 7 taps)
};
constexpr int SM_TOTAL = SM_PAR + (int)sizeof(SmemPar);
static_assert(2 * (SM_TOTAL + 1024) <= 233472, "two CTAs per SM");
static_assert(2 * NT * 8 <= 5 * NWORDS * 4, "coarse CUSP/ZAC values fit into the T10..T99 mask area");

int icpc_smem_bytes() { return SM_TOTAL; }
int icpc_threads() { return NT; }

enum { IB_POS0 = 0 /* NMASK positions */, IB_MULT = 16, IB_PKFROM = 20 /* 3 */, IB_QN = 24, IB_CZN = 25, IB_CZT = 32 /* 31 chunk ids */ };
constexpr int QCAP = 480;    // work queue of flagged intervals (uint16 codes behind the coarse CUSP/ZAC values)
constexpr int CZCAP = 31;    // candidate chunks per round of the CUSP/ZAC output buffer (31 * 33 * 2 doubles <= 16 KB)
static_assert(2 * NT * 8 + QCAP * 2 <= 5 * NWORDS * 4, "coarse values + queue fit into the T10..T99 mask area");
static_assert(CZCAP * CH * 2 * 8 <= 8 * NT * 8, "output buffer fits into the tables 8..15 area");
enum { SC_TX = 0 /* 5 */, SC_T0 = 5, SC_T0INV = 6, SC_PKP = 8 /* 3 */, SC_PP0 = 16 };

// ---------------------------------------------------------------------------------------------------
// reductions.  Maxima/minima of doubles go through an order-preserving 64-bit integer key and two 32-bit
// REDUX instructions instead of 5 shuffle rounds; every warp publishes its partial in red[slot][warp]; after the
// next barrier a warp combines the 8 partials with its lanes (lane l reads partial l & 7).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ long long d2key(double v)
{
    const long long b = __double_as_longlong(v);
    return b ^ ((b >> 63) & 0x7fffffffffffffffLL);
}
__device__ __forceinline__ double key2d(long long k) { return __longlong_as_double(k ^ ((k >> 63) & 0x7fffffffffffffffLL)); }
// maximum over the warp (no NaNs), result in every lane
__device__ __noinline__ double wmax_d(double v)
{
    const long long k = d2key(v);
    const int hi = (int)(k >> 32);
    const unsigned lo = (unsigned)k;
    const int mh = __reduce_max_sync(FULL, hi);
    const unsigned ml = __reduce_max_sync(FULL, hi == mh ? lo : 0u);
    return key2d(((long long)mh << 32) | (long long)ml);
}
__device__ __forceinline__ double wmin_d(double v) { return -wmax_d(-v); }
// (maximum, FIRST index) over the warp
__device__ __forceinline__ double wargmax_d(double v, int& ix)
{
    const double m = wmax_d(v);
    ix = __reduce_min_sync(FULL, v == m ? ix : 0x7fffffff);
    return m;
}
__device__ __noinline__ double wsum_d(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ void red_put(double* red, int slot, int wid, int lane, double v)
{
    if (lane == 0) red[slot * NWARP + wid] = v;
}
__device__ __noinline__ double red_sum(const double* red, int slot)
{
    double v = red[slot * NWARP + (threadIdx.x & 7)];
    v += __shfl_xor_sync(FULL, v, 4);
    v += __shfl_xor_sync(FULL, v, 2);
    v += __shfl_xor_sync(FULL, v, 1);
    return v;
}
__device__ __noinline__ double red_max(const double* red, int slot) { return wmax_d(red[slot * NWARP + (threadIdx.x & 7)]); }
__device__ __forceinline__ double red_min(const double* red, int slot) { return -wmax_d(-red[slot * NWARP + (threadIdx.x & 7)]); }
// (max value, FIRST index)
__device__ __forceinline__ void red_argmax(const double* red, int slot_v, int slot_i, double& v, int& ix)
{
    const double pv = red[slot_v * NWARP + (threadIdx.x & 7)];
    int pi = (int)red[slot_i * NWARP + (threadIdx.x & 7)];
    v = wargmax_d(pv, pi);
    ix = pi;
}

// exact uint32 -> double without the conversion pipe: 2^52 + v has v in its low mantissa word
__device__ __forceinline__ double u2d(uint32_t v) { return __hiloint2double(0x43300000, (int)v) - 4503599627370496.0; }

// run-length monoid for the saturation counters (src/saturation.jl:28-65)
struct Run {
    int pre, suf, best, len;
};
__device__ __forceinline__ Run run_merge(const Run& A, const Run& B)
{
    Run r;
    r.pre = (A.pre == A.len) ? A.len + B.pre : A.pre;
    r.suf = (B.suf == B.len) ? B.len + A.suf : B.suf;
    r.best = max(max(A.best, B.best), A.suf + B.pre);
    r.len = A.len + B.len;
    return r;
}
__device__ __forceinline__ Run run_shfl_down(const Run& a, int o)
{
    Run r;
    r.pre = __shfl_down_sync(FULL, a.pre, o);
    r.suf = __shfl_down_sync(FULL, a.suf, o);
    r.best = __shfl_down_sync(FULL, a.best, o);
    r.len = __shfl_down_sync(FULL, a.len, o);
    return r;
}

// regression statistics from accumulated sums, operation order of the reference (src/tailstats.jl:54-70 and
// its RDDSP original signalstats); never contracted
struct Stats {
    double mean, sigma, slope, offset;
};
__device__ __noinline__ Stats stats_finalize(double inv_n, double sX, double sXX, double sY, double sYY, double sXY)
{
    const double mean_X = mul_rn(sX, inv_n);
    const double mean_Y = mul_rn(sY, inv_n);
    const double var_X = sub_rn(mul_rn(sXX, inv_n), mul_rn(mean_X, mean_X));
    double var_Y = sub_rn(mul_rn(sYY, inv_n), mul_rn(mean_Y, mean_Y));
    const double cov = sub_rn(mul_rn(sXY, inv_n), mul_rn(mean_X, mean_Y));
    Stats s;
    s.slope = div_rn(cov, var_X);
    s.offset = sub_rn(mean_Y, mul_rn(s.slope, mean_X));
    if (var_Y < 0) var_Y = 0;
    s.mean = mean_Y;
    s.sigma = sqrt(var_Y);
    return s;
}

// extrema3points  src/interpolation.jl:8-10
__device__ __forceinline__ double extrema3(double y1, double y2, double y3)
{
    const double a = y3 - 4.0 * y2 + 3.0 * y1;
    return y1 - a * a / (8.0 * (y3 - 2.0 * y2 + y1));
}

// ---- single-sample evaluations on the prefix sums TT (TT[i] = sum_{k<i} y[k]) ----
// trapezoid output j, inlined at every call site (no call frame; the trapezoid's constants stay in uniform registers)
__device__ __forceinline__ double trap_at_i(const double* TT, const TrapDev& t, int j)
{
    const double* p = TT + j;
    const double s1 = p[t.a] - p[0];
    const double s2 = p[t.L] - p[t.a + t.g];
    return __fma_rn(s2, t.inv2, -__dmul_rn(s1, t.inv1));
}
__device__ __forceinline__ double y_at(const double* TT, int i) { return TT[i + 1] - TT[i]; }
__device__ __noinline__ double sg_eval(const double* TT, const double* gg, int n_taps, int j)
{
    double a0 = 0, a1 = 0;   // same association as sg_chunk_t
#pragma unroll 1
    for (int k = 0; k <= n_taps; k += 2) {
        a0 = fma(gg[k], TT[j + k], a0);
        if (k + 1 <= n_taps) a1 = fma(gg[k + 1], TT[j + k + 1], a1);
    }
    return a0 + a1;
}
// 8-tap version for the zero-padded SMEM copy of a short kernel (bit-identical to sg_eval / sg_chunk_t<8>)
__device__ __noinline__ double sg_eval8(const double* TT, const double* gg, int j)
{
    const double* p = TT + j;
    double a0 = gg[0] * p[0], a1 = gg[1] * p[1];
    a0 = fma(gg[2], p[2], a0); a1 = fma(gg[3], p[3], a1);
    a0 = fma(gg[4], p[4], a0); a1 = fma(gg[5], p[5], a1);
    a0 = fma(gg[6], p[6], a0); a1 = fma(gg[7], p[7], a1);
    return a0 + a1;
}
// DerivativeFilter sample i  (src/derivative.jl:47-55)
__device__ __forceinline__ double deriv_at(const double* TT, int i)
{
    const int ii = i < 1 ? 1 : i;
    return (TT[ii + 1] - TT[ii]) - (TT[ii] - TT[ii - 1]);
}
// direct FIR output j of a CUSP/ZAC filter with differenced taps g[0..L] on TT: out[j] = sum_k g[k] TT[j+L-k]
__device__ __forceinline__ double fir_at(const double* TT, const double* __restrict__ g, int L, int j)
{
    double acc = 0;
    for (int k = 0; k <= L; ++k) acc = fma(__ldg(g + k), TT[j + L - k], acc);
    return acc;
}

// thread-local 33-bit mask -> block mask (bit position 33*tid + k)
__device__ __noinline__ void mask_commit(uint32_t* M, int tid, unsigned long long bits)
{
    if (bits == 0ull) return;
    const int p0 = tid * CH, w0 = p0 >> 5, s0 = p0 & 31;
    const unsigned long long sh = bits << s0;   // 33 bits shifted by <= 31: fits in 64
    const uint32_t lo = (uint32_t)sh, mid = (uint32_t)(sh >> 32);
    if (lo) atomicOr(&M[w0], lo);
    if (mid && w0 + 1 < NWORDS) atomicOr(&M[w0 + 1], mid);
}
// same for the time-reversed trace of length nlen: forward bit i <-> reversed bit nlen-1-i
__device__ __noinline__ void mask_commit_reversed(uint32_t* M, int tid, unsigned long long bits, int nlen)
{
    if (bits == 0ull) return;
    // reversed positions of the chunk: base = nlen-1-(33*tid+32) holds forward bit 32, base+32 holds forward bit 0
    unsigned long long rev = __brevll(bits) >> (64 - CH);   // rev bit (32-k) = bits bit k
    int base = nlen - 1 - (tid * CH + CH - 1);
    if (base < 0) { rev >>= (-base); base = 0; }
    const int w0 = base >> 5, s0 = base & 31;
    const unsigned long long sh = rev << s0;
    const uint32_t lo = (uint32_t)sh, mid = (uint32_t)(sh >> 32);
    if (lo) atomicOr(&M[w0], lo);
    if (mid && w0 + 1 < NWORDS) atomicOr(&M[w0 + 1], mid);
}

// Warp-cooperative commit of two 33-bit chunk masks of chunk q (bit k <-> position 33q + k): lanes 0,1 write the two words
// of mask A, lanes 2,3 those of mask B (B optionally on the time-reversed trace of length nlen) -- one atomic instruction
// for the warp instead of four sequential ones.  Every lane passes the same arguments.
__device__ __forceinline__ void commit_pair(uint32_t* MA, unsigned long long bits_a, uint32_t* MB, unsigned long long bits_b,
                                            bool b_reversed, int nlen, int q, int lane)
{
    if (lane >= 4) return;
    const bool isb = lane >= 2;
    unsigned long long bits = isb ? bits_b : bits_a;
    uint32_t* M = isb ? MB : MA;
    if (M == nullptr || bits == 0ull) return;
    int base = q * CH;
    if (isb && b_reversed) {
        bits = __brevll(bits) >> (64 - CH);            // reversed bit (32-k) = forward bit k
        base = nlen - 1 - (q * CH + CH - 1);
        if (base < 0) { bits >>= (-base); base = 0; }
    }
    const int w = (base >> 5) + (lane & 1), s0 = base & 31;
    const unsigned long long sh = bits << s0;          // 33 bits shifted by <= 31: fits in 64
    const uint32_t word = (lane & 1) ? (uint32_t)(sh >> 32) : (uint32_t)sh;
    if (word && w < NWORDS) atomicOr(&M[w], word);
}

// One warp: find runs of >= k consecutive set bits in the NWORDS-word mask M (bits beyond the trace are zero)
// that do not start at bit 0 -- the Intersect state machine (SURVEY.md App. B): `pos` = start of the first such
// run (-1 if none), `mult` = number of such runs.  Every lane looks for run STARTS (set bit after a clear bit) in its
// 8 words and measures each run forward, word by word; M is left intact.  Words are dealt round-robin (word w -> lane
// w % 32): the noisy stretch around a crossing spans a few neighbouring words, which then go to different lanes.
__device__ __noinline__ int resolve_runs_packed(const uint32_t* M, int k, int lane)
{
    constexpr int Q = NWORDS / 32;
    int p = 0x7fffffff, cnt = 0;
#pragma unroll 1
    for (int q = 0; q < Q; ++q) {
        const int w0 = q * 32 + lane;
        const uint32_t mq = M[w0];
        const uint32_t prev = w0 ? M[w0 - 1] : 0u;
        uint32_t starts = mq & ~((mq << 1) | (prev >> 31));
        if (w0 == 0) starts &= ~1u;  // a run that starts at the first sample never fires
        if (k <= 32) {
            // short runs (t10..t99, current and pile-up masks): bit-parallel test "k set bits from here on" on the 64-bit window
            // of this word and the next (AND-doubling) -- no loop over the starts, whose number explodes on noise-only events
            unsigned long long r = (unsigned long long)mq | ((unsigned long long)(w0 + 1 < NWORDS ? M[w0 + 1] : 0u) << 32);
            for (int len = 1; len < k;) {
                const int sft = min(len, k - len);
                r &= r >> sft;
                len += sft;
            }
            starts &= (uint32_t)r;
            cnt += __popc(starts);
            if (starts) p = min(p, w0 * 32 + __ffs(starts) - 1);
            continue;
        }
        while (starts) {
            const int b = __ffs(starts) - 1;
            starts &= starts - 1;
            const uint32_t rest = ~(mq >> b);            // first clear bit above b (the shifted-in zeros stop it at the word end)
            int len = rest ? __ffs(rest) - 1 : 32;
            if (len == 32 - b) {
                // the run reaches the top of its word: follow it through the next words
                for (int w = w0 + 1; w < NWORDS && len < k; ++w) {
                    const uint32_t x = M[w];
                    if (x == 0xffffffffu) { len += 32; continue; }
                    len += __ffs(~x) - 1;
                    break;
                }
            }
            if (len >= k) {
                ++cnt;
                p = min(p, w0 * 32 + b);
            }
        }
    }
    p = __reduce_min_sync(FULL, p);
    cnt = __reduce_add_sync(FULL, cnt);
    return ((p == 0x7fffffff) ? 0 : p + 1) | (cnt << 16);   // (pos + 1) in the low half, multiplicity in the high half
}
__device__ __forceinline__ void resolve_runs(const uint32_t* M, int k, int lane, int& pos, int& mult)
{
    const int r = resolve_runs_packed(M, k, lane);
    pos = (r & 0xffff) - 1;
    mult = r >> 16;
}

// linear interpolation of Intersect: x = (thr - y_l)*(x_r - x_l)/(y_r - y_l) + x_l
__device__ __noinline__ double cross_x(double thr, double yl, double yr, double tl, double dt)
{
    return (thr - yl) * dt / (yr - yl) + tl;
}

// window placement policy (include/lgdsp_b200.h, lgdsp_dni)
__device__ __noinline__ void dni_window(int n_w, int n_trace, double p, double& pc, int& from)
{
    if (!(p >= 0)) p = 0;
    if (p > n_trace - 1) p = n_trace - 1;
    long long f = (long long)rint(p) - n_w / 2;
    if (f < 0) f = 0;
    if (f > n_trace - n_w) f = n_trace - n_w;
    pc = p;
    from = (int)f;
}
// PolynomialDNI estimate, one warp: window values win[0..n_w) (SMEM/any), fit matrix A (global); result in every lane.
// (coefficients beyond the degree are zero, so the fixed-length Horner scheme gives the same value as a shorter one)
__device__ __noinline__ double dni_eval_warp(const double* __restrict__ A, int n_w, int m, const double* win, double u,
                                                int lane)
{
    double c0 = 0, c1 = 0, c2 = 0, c3 = 0;
#pragma unroll 1
    for (int i = lane; i < n_w; i += 32) {
        const double v = win[i];
        const double* a = A + i * m;
        c0 = fma(__ldg(a), v, c0);
        if (m > 1) c1 = fma(__ldg(a + 1), v, c1);
        if (m > 2) c2 = fma(__ldg(a + 2), v, c2);
        if (m > 3) c3 = fma(__ldg(a + 3), v, c3);
    }
    c0 = wsum_d(c0); c1 = wsum_d(c1); c2 = wsum_d(c2); c3 = wsum_d(c3);
    return fma(fma(fma(c3, u, c2), u, c1), u, c0);
}

// Three PolynomialDNI estimates at once for windows of <= 8 samples: lanes [8g, 8g+8) work on estimate g (its window
// start `from` and evaluation point `u` are per lane, equal inside a group); every lane of group g gets estimate g.
// Same products and the same xor-4,2,1 reduction order as dni_eval_warp: bit-identical results.
__device__ __noinline__ double dni3_warp(const double* __restrict__ A, int n_w, int m, const double* trace, int from, double u,
                                         int lane)
{
    const int i = lane & 7;
    const bool on = i < n_w && lane < 24;
    const double v = on ? trace[from + i] : 0.0;
    double c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    if (on) {
        const double* a = A + i * m;
        c0 = __ldg(a) * v;
        if (m > 1) c1 = __ldg(a + 1) * v;
        if (m > 2) c2 = __ldg(a + 2) * v;
        if (m > 3) c3 = __ldg(a + 3) * v;
    }
#pragma unroll 1
    for (int o = 4; o > 0; o >>= 1) {
        c0 += __shfl_xor_sync(FULL, c0, o);
        c1 += __shfl_xor_sync(FULL, c1, o);
        c2 += __shfl_xor_sync(FULL, c2, o);
        c3 += __shfl_xor_sync(FULL, c3, o);
    }
    return fma(fma(fma(c3, u, c2), u, c1), u, c0);
}

// ---------------------------------------------------------------------------------------------------
// chunk passes over the prefix sums
// ---------------------------------------------------------------------------------------------------
// sliding-window FIR on TT (the SG kernels folded onto the prefix sums): s[j] = sum_{q<NW} gg[q]*TT[j+q].
// f(k, s) is called for every output j0+k of the chunk, k < cnt.
template <int NW, typename F>
__device__ __forceinline__ void sg_chunk_t(const double* TT, const SgDev& S, int j0, int cnt, F&& f)
{
    double g[NW], w[NW];
#pragma unroll
    for (int q = 0; q < NW; ++q) g[q] = S.gg[q];
    const double* p = TT + j0;
#pragma unroll
    for (int q = 0; q < NW - 1; ++q) w[q] = p[q];
    int k = 0;
    // groups of NW outputs: the window rotates through the NW registers with compile-time indices (no moves)
#pragma unroll 1
    for (; k + NW <= cnt; k += NW) {
#pragma unroll
        for (int u = 0; u < NW; ++u) {
            w[(u + NW - 1) % NW] = p[k + u + NW - 1];
            double a0 = 0, a1 = 0;   // two accumulators: halves the dependent FMA chain
#pragma unroll
            for (int q = 0; q < NW; q += 2) {
                a0 = fma(g[q], w[(u + q) % NW], a0);
                if (q + 1 < NW) a1 = fma(g[q + 1], w[(u + q + 1) % NW], a1);
            }
            f(k + u, a0 + a1);
        }
    }
#pragma unroll 1
    for (; k < cnt; ++k) {
        double a0 = 0, a1 = 0;
#pragma unroll
        for (int q = 0; q < NW; q += 2) {
            a0 = fma(g[q], p[k + q], a0);
            if (q + 1 < NW) a1 = fma(g[q + 1], p[k + q + 1], a1);
        }
        f(k, a0 + a1);
    }
}
template <typename F>
__device__ __forceinline__ void sg_chunk(const double* TT, const SgDev& S, int j0, int cnt, F&& f)
{
    if (cnt <= 0) return;
    if (S.n_taps + 1 <= 8) {
        // one 8-wide instantiation for every short kernel: gg is zero-padded and TT is finite (zero) beyond the trace
        sg_chunk_t<8>(TT, S, j0, cnt, f);
    } else {
        for (int k = 0; k < cnt; ++k) f(k, sg_eval(TT, S.gg, S.n_taps, j0 + k));
    }
}

// ==================================================================================================
// CUSP/ZAC through their analytic structure (replaces two 2375-tap FIRs = 27.6 M MAC per waveform by O(n) work).
//
//   coeffs[k] = g*(c[k] - r*c[k-1])  =>  out[j] = g*( sum_k c[k]*d[m-k] + r*c[L-1]*y[m-L] ),  m = j+L-1,
//   d[i] = y[i] - r*y[i-1]  (the "current"),   c = sinh flank | flat top | mirrored sinh flank (+ parabolas for ZAC).
//
// Every piece of c is an exponential or a polynomial in k, so sum_k c[k]*d[m-k] splits into sliding windows
//   E-(m) = sum rho^k d, E+(m) = sum rho^-k d, W0/W1/W2 = sum {1,k,k^2} d      (rho = exp(-1/sigma))
// over the left flank, the flat top and the right flank.  Each window obeys a 1-step linear recurrence in m.
// Thread t owns outputs m in [33t, 33t+33): it gets the window states at m = 33t in closed form from
// block-wide prefix scans of d (decayed prefix P-, anti-causal decayed prefix P+, moments D1 = sum i*d,
// D2 = sum i^2*d; D0 = sum d comes from TT directly), which are only ever needed at 4 positions per chunk
// (fixed in-chunk offsets) -> 16 tables x 256 entries instead of 4 full-resolution arrays; then it steps the
// recurrences 33 times.  The growing exponentials are only propagated over 33 samples, so nothing blows up.
// (validated against the direct FIR in tools/proto_cuspzac.py and tests/test_gpu_*.py)
// ==================================================================================================
__device__ __noinline__ double exp_d(double x) { return exp(x); }

struct CzState {
    double EmL, EpL, W0L, W1L, W2L, W0F, V0, V1, V2, EpR, EmR;
    bool active;
};

__device__ __forceinline__ double* cz_tab(double* tabA, double* tabB, int idx)
{
    return idx < 8 ? tabA + idx * NT : tabB + (idx - 8) * NT;
}

// block-wide scans of d over the whole waveform; fills the 16 decimated tables and *pp0 = P+[0].
// One forward loop per chunk: P- (decayed prefix), D1, D2 (moments) and the partial sums acc = sum_{k'<=k} rho^k' d
// of the anti-causal prefix (P+ at in-chunk offset o is (total - acc[o-1]) * rho^-o; the weights only span one
// chunk, so nothing cancels).  The running values are stored at the capture events the host sorted by sample index.
// CONTIG: tables 8..15 follow tables 0..7 in memory (the split pipeline's layout): no per-access choice of the half
template <int PAR_OFF, bool CONTIG = false>
__device__ __noinline__ void cz_scan(int ps, const double* TT, int n, int tid, double* tabA, double* tabB, double* red,
                        double* pp0)
{
    // SMEM copy of the descriptor, addressed through the dynamic shared memory base so that the loads are LDS
    // (a reference to the kernel parameter or a generic pointer would force generic loads)
    extern __shared__ __align__(128) unsigned char smem_dyn[];
    const CzDev& Z = reinterpret_cast<const SmemPar*>(smem_dyn + PAR_OFF)->cz[ps];
    auto tabp = [&](int idx) -> double* { return CONTIG ? tabA + idx * NT : cz_tab(tabA, tabB, idx); };
    const int lane = tid & 31, wid = tid >> 5;
    const int i0 = tid * CH;
    const double r = Z.r, rho = Z.rho;
    double pm = 0, d1 = 0, d2 = 0, acc = 0;
    const bool live = i0 < n;
    if (live) {
        const int cnt = min(CH, n - i0);
        const double* p = TT + i0 + 1;
        double tcur = p[-1];
        double yprev = (i0 >= 1) ? tcur - p[-2] : 0.0;
        double di = (double)i0, w = 1.0;
        double tpre = p[0];   // software prefetch of the next prefix sum
        auto step = [&](double d) {
            pm = fma(rho, pm, d);
            const double kd = di * d;
            d1 += kd;
            d2 = fma(di, kd, d2);
            di += 1.0;
            acc = fma(w, d, acc);
            w *= rho;
        };
        int k = 0;
        auto run_to = [&](int kend) {
            if (cnt == CH) {
#pragma unroll 1
                for (; k <= kend; ++k) {
                    const double tnext = tpre;
                    tpre = p[k + 1];                    // (<= TT[i0+34]: exists for every full chunk)
                    const double y = tnext - tcur;      // exact difference of neighbouring prefix sums
                    const double d = fma(-r, yprev, y);
                    yprev = y;
                    tcur = tnext;
                    step(d);
                }
            } else {
                // last chunk of the trace: samples beyond the trace contribute d = 0
#pragma unroll 1
                for (; k <= kend; ++k) {
                    double d = 0.0;
                    if (k < cnt) {
                        const double tnext = p[k];
                        const double y = tnext - tcur;
                        d = fma(-r, yprev, y);
                        yprev = y;
                        tcur = tnext;
                    }
                    step(d);
                }
            }
        };
#pragma unroll 1
        for (int ev = 0; ev <= Z.n_ev; ++ev) {
            const bool last = ev == Z.n_ev;            // pseudo event: the rest of the chunk, nothing to capture
            run_to(last ? CH - 1 : Z.ev_k[ev]);
            if (last) break;
            const int tb = Z.ev_tab[ev];
            if (Z.ev_kind[ev] == 0) {
                tabp(tb * 3 + 0)[tid] = pm;
                tabp(tb * 3 + 1)[tid] = d1;
                tabp(tb * 3 + 2)[tid] = d2;
            } else {
                tabp(12 + tb)[tid] = acc;
            }
        }
    }
    const double pp = acc;   // P+ of the chunk alone at its first sample
    // warp-level scans (linear recurrences with constant multiplier rho^CH; plain sums for the moments)
    double vpm = pm, vd1 = d1, vd2 = d2, vpp = pp;
#pragma unroll 1
    for (int s = 0; s < 5; ++s) {
        const int o = 1 << s;
        const double upm = __shfl_up_sync(FULL, vpm, o), ud1 = __shfl_up_sync(FULL, vd1, o), ud2 = __shfl_up_sync(FULL, vd2, o);
        const double upp = __shfl_down_sync(FULL, vpp, o);
        if (lane >= o) { vpm = fma(Z.rho_ch_pow[s], upm, vpm); vd1 += ud1; vd2 += ud2; }
        if (lane + o < 32) vpp = fma(Z.rho_ch_pow[s], upp, vpp);
    }
    if (lane == 31) { red[wid] = vpm; red[8 + wid] = vd1; red[16 + wid] = vd2; }
    if (lane == 0) red[24 + wid] = vpp;
    __syncthreads();
    double gpm = 0, gd1 = 0, gd2 = 0, gpp = 0;   // carries of the neighbouring warps
    for (int w = 0; w < wid; ++w) { gpm = fma(Z.rho_warp, gpm, red[w]); gd1 += red[8 + w]; gd2 += red[16 + w]; }
    for (int w = NWARP - 1; w > wid; --w) gpp = fma(Z.rho_warp, gpp, red[24 + w]);
    // global inclusive values of this thread, then the carry-in = inclusive value of the neighbour thread
    const double ipm = fma(Z.rho_lane[lane], gpm, vpm);
    const double ipp = fma(Z.rho_lane[31 - lane], gpp, vpp);
    double c_pm = __shfl_up_sync(FULL, ipm, 1), c_pp = __shfl_down_sync(FULL, ipp, 1);
    if (lane == 0) c_pm = gpm;
    if (lane == 31) c_pp = gpp;
    const double c_d1 = gd1 + (vd1 - d1), c_d2 = gd2 + (vd2 - d2);
    // fix-up of this thread's own table entries: add the carried-in prefixes
    if (live) {
#pragma unroll 1
        for (int ev = 0; ev < Z.n_ev; ++ev) {
            const int tb = Z.ev_tab[ev];
            const double pw = Z.ev_pw[ev];
            if (Z.ev_kind[ev] == 0) {
                double* t0 = tabp(tb * 3 + 0) + tid;
                double* t1 = tabp(tb * 3 + 1) + tid;
                double* t2 = tabp(tb * 3 + 2) + tid;
                *t0 = fma(pw, c_pm, *t0);
                *t1 += c_d1;
                *t2 += c_d2;
            } else {
                double* t = tabp(12 + tb) + tid;
                *t = fma(pw, c_pp, (pp - *t) * Z.ev_rinv[ev]);
            }
        }
    }
    if (tid == 0) *pp0 = ipp;
}

// window states at m = CH*tid in closed form from the tables
// tab_c(q, kind, chunk) / tab_a(q, chunk): the decimated prefix tables (causal P-, D1, D2 / anti-causal P+) at a chunk
template <typename TC, typename TA>
__device__ __forceinline__ void cz_init_with(const CzDev& Z, const double* TT, int n, int tid, double pp0, CzState& S, TC&& tab_c,
                                             TA&& tab_a)
{
    const int m = tid * CH;
    S.active = (m < n) && (m + CH - 1 >= Z.L - 1);
    if (!S.active) return;
    auto lc = [&](int q, int kind, int pos) -> double {   // causal prefixes (P-, D1, D2): zero before the trace
        return pos < 0 ? 0.0 : tab_c(q, kind, pos / CH);
    };
    auto la = [&](int q, int pos) -> double {             // anti-causal prefix P+
        if (pos >= n) return 0.0;
        if (pos < 0) return exp_d((double)pos * Z.inv_sigma) * pp0;   // rho^(-pos) * P+[0]
        return tab_a(q, pos / CH);
    };
    auto d0 = [&](int j) -> double {                      // D0[j] = sum_{i<=j} d[i] = TT[j+1] - r*TT[j]
        return j < 0 ? 0.0 : fma(-Z.r, TT[j], TT[j + 1]);
    };
    const int lt = Z.lt, L = Z.L, Rn = Z.Rn, F = Z.F;
    const double dm = (double)m;
    S.EmL = Z.cA * (lc(0, 0, m) - Z.rho_lt * lc(1, 0, m - lt));
    S.EpL = Z.cA_rhoinv_ltm1 * (la(0, m - lt + 1) - Z.rho_lt * la(1, m + 1));
    S.EpR = Z.cA_rhoinv_Rn * (lc(2, 0, m - L + Rn) - Z.rho_Rn * lc(3, 0, m - L));
    S.EmR = Z.cA_rho * (la(2, m - L + 1) - Z.rho_Rn * la(3, m - L + Rn + 1));
    const double a0 = d0(m) - d0(m - lt), a1 = lc(0, 1, m) - lc(1, 1, m - lt), a2 = lc(0, 2, m) - lc(1, 2, m - lt);
    S.W0L = a0;
    S.W1L = dm * a0 - a1;
    S.W2L = dm * dm * a0 - 2.0 * dm * a1 + a2;
    S.W0F = d0(m - lt) - d0(m - lt - F - 1);
    const double b0 = d0(m - L + Rn) - d0(m - L);
    const double b1 = lc(2, 1, m - L + Rn) - lc(3, 1, m - L), b2 = lc(2, 2, m - L + Rn) - lc(3, 2, m - L);
    const double qq = (double)(m - L);
    S.V0 = b0;
    S.V1 = b1 - qq * b0;
    S.V2 = b2 - 2.0 * qq * b1 + qq * qq * b0;
}
__device__ __forceinline__ void cz_init(const CzDev& Z, const double* TT, int n, int tid, double* tabA, double* tabB, double pp0,
                        CzState& S)
{
    cz_init_with(Z, TT, n, tid, pp0, S,
                 [&](int q, int kind, int c) -> double { return cz_tab(tabA, tabB, q * 3 + kind)[c]; },
                 [&](int q, int c) -> double { return cz_tab(tabA, tabB, 12 + q)[c]; });
}

// one input stream d[j], j advancing by one per step
struct CzStream {
    const double* p;   // &TT[j+1] of the NEXT d to produce (fast path) / TT base (safe path)
    double t, yprev;
    int j;
    __device__ __forceinline__ void init(const double* TT, int j0)
    {
        j = j0;
        t = TT[max(j0, 0)];
        yprev = (j0 >= 1) ? t - TT[j0 - 1] : 0.0;
        p = TT + j0 + 1;
    }
    // all indices known to be inside [1, n]: no clamping
    __device__ __forceinline__ double next_fast(double r, int k)
    {
        const double tn = p[k];
        const double y = tn - t;
        const double d = fma(-r, yprev, y);
        yprev = y;
        t = tn;
        return d;
    }
    // the same from a prefix sum TT[j + 1] read elsewhere (the finish kernel's shared-memory slab); j is not advanced
    __device__ __forceinline__ double next_from(double r, double tn)
    {
        const double y = tn - t;
        const double d = fma(-r, yprev, y);
        yprev = y;
        t = tn;
        return d;
    }
    // indices before the trace read as zero, beyond the end clamp
    __device__ __forceinline__ double next_safe(const double* TT, double r, int n)
    {
        const int jj = min(max(j + 1, 0), n);
        const double tn = TT[jj];
        const double y = tn - t;
        const double d = fma(-r, yprev, y);
        yprev = y;
        t = tn;
        ++j;
        return d;
    }
};

// the CUSP and ZAC outputs of the current window state (s3 = the y[m-L] stream) and the state update by one step from the
// four stream inputs a..d; shared by cz_out_each and cz_out_staged
template <typename F>
__device__ __forceinline__ void cz_emit(const CzDev& Z, const CzState& S, const CzStream& s3, int k, F&& f)
{
    const double ylast = s3.yprev;   // y[m-L]
    const double Dc = (S.EpL - S.EmL + S.EpR - S.EmR) + S.W0F;
    const double poly = (S.W2L - Z.h2 * S.W1L) + (S.V2 - Z.h2 * S.V1);
    f(k, fma(Z.g, Dc, Z.gclast_cusp * ylast), fma(Z.g, fma(Z.B, poly, Dc), Z.gclast_zac * ylast));
}
__device__ __forceinline__ void cz_update(const CzDev& Z, CzState& S, double a, double b, double c, double d)
{
    S.EmL = fma(Z.rho, S.EmL, fma(Z.cA, a, -Z.cA_rho_lt * b));
    S.EpL = fma(Z.rho_inv, S.EpL, fma(Z.cA, a, -Z.cA_rhoinv_lt * b));
    S.W2L = S.W2L + 2.0 * S.W1L + S.W0L - Z.lt2_d * b;
    S.W1L = S.W1L + S.W0L - Z.lt_d * b;
    S.W0L = S.W0L + a - b;
    S.W0F = S.W0F + b - c;
    S.V2 = S.V2 - 2.0 * S.V1 + S.V0 + Z.Rn2_d * c;
    S.V1 = S.V1 - S.V0 + Z.Rn_d * c;
    S.V0 = S.V0 + c - d;
    S.EpR = fma(Z.rho, S.EpR, fma(Z.cA_rhoinv_Rn, c, -Z.cA * d));
    S.EmR = fma(Z.rho_inv, S.EmR, fma(Z.cA_rho_Rn, c, -Z.cA * d));
}

// CH recurrence steps of one candidate chunk: the CUSP and ZAC outputs go to obuf[k][0..1] (-inf where m0+k is not a
// valid output); maxima, argmaxima and the pick-off windows are taken from there by a block-parallel pass.  No
// compares or branches in the loop: the only loop-carried dependency is the state update.
template <typename F>
__device__ __forceinline__ void cz_out_each(const CzDev& Z, const double* TT, int n, int tid, CzState& S, F&& f)
{
    const int m0 = tid * CH;
    const int L = Z.L, lt = Z.lt, F_ = Z.F;
    const double r = Z.r;
    CzStream s0, s1, s2, s3;
    s0.init(TT, m0 + 1);
    s1.init(TT, m0 + 1 - lt);
    s2.init(TT, m0 - lt - F_);
    s3.init(TT, m0 + 1 - L);
    const bool interior = (m0 - L >= 1) && (m0 + CH + 1 <= n);
    if (interior) {
#pragma unroll 1
        for (int k = 0; k < CH; ++k) {
            cz_emit(Z, S, s3, k, f);
            const double a = s0.next_fast(r, k), b = s1.next_fast(r, k), c = s2.next_fast(r, k), d = s3.next_fast(r, k);
            cz_update(Z, S, a, b, c, d);
        }
    } else {
#pragma unroll 1
        for (int k = 0; k < CH; ++k) {
            const int m = m0 + k;
            if (m >= L - 1 && m < n) cz_emit(Z, S, s3, k, f);
            else f(k, -CUDART_INF, -CUDART_INF);
            const double a = s0.next_safe(TT, r, n), b = s1.next_safe(TT, r, n), c = s2.next_safe(TT, r, n),
                         d = s3.next_safe(TT, r, n);
            cz_update(Z, S, a, b, c, d);
        }
    }
}

// The same CH steps for the candidate chunks of a whole warp, one lane each, with TT in global memory (the finish kernel of
// the split pipeline).  Lane-private loads there would make every load instruction touch 32 unrelated sectors and leave the
// recurrence waiting on L2 each step; instead the warp stages steps 1..CH-1 in pieces of CZ_STAGE steps into a
// double-buffered slab in shared memory, cooperatively: one cp.async instruction fetches CZ_STAGE consecutive prefix sums
// of 32 / CZ_STAGE candidates, and the next piece is in flight while the current one is stepped.  Slab layout
// [buffer][stream][step][lane ^ swizzle(step)]: a step of all 32 lanes is one conflict-free LDS.64 row, and the swizzle
// makes the cooperative stores conflict-free too.  Every lane reads TT[clamp(j + 1, 0, n)] as next_safe does, so chunks at
// the trace ends take the same values as in cz_out_each (for interior chunks the clamp is void), and every float64
// operation keeps its operands and order.  All 32 lanes must call it (warp-synchronous); lanes without a candidate
// (has == false, chunk 0) help to stage and never call f.  nact: candidates of the warp (lanes 0..nact-1).
constexpr int CZ_STAGE = 4;   // steps per staged piece (a power of two dividing CH - 1 = 32)
static_assert(CZ_STAGE >= 1 && CZ_STAGE <= 32 && (CZ_STAGE & (CZ_STAGE - 1)) == 0 && (CH - 1) % CZ_STAGE == 0, "stage piece");
constexpr int CZ_SLAB = 2 * 4 * CZ_STAGE * 32;   // doubles of one warp's slab
template <typename F>
__device__ __forceinline__ void cz_out_staged(const CzDev& Z, const double* TT, int n, int chunk, bool has, int nact, CzState& S,
                                              double* slab, int lane, F&& f)
{
    constexpr int G = 32 / CZ_STAGE;   // candidates per cp.async instruction
    const int m0 = chunk * CH;
    const int L = Z.L, lt = Z.lt, F_ = Z.F;
    const double r = Z.r;
    const int jofs[4] = {1, 1 - lt, -lt - F_, 1 - L};   // stream starts j0 - m0 (CzStream::init)
    // staging piece p = steps 1 + p * CZ_STAGE + i, i < CZ_STAGE; this lane copies step i = lane % CZ_STAGE of candidates
    // g * G + lane / CZ_STAGE
    const int si = lane % CZ_STAGE;
    auto stage = [&](int p) {
        double* b = slab + (p & 1) * (4 * CZ_STAGE * 32) + si * 32;
        const int kk = 2 + p * CZ_STAGE + si;   // TT index of this step's input = j0 + 1 + k
#pragma unroll
        for (int g = 0; g < CZ_STAGE; ++g) {
            const int c = g * G + lane / CZ_STAGE;
            const int mc = __shfl_sync(FULL, m0, c);
            if (c < nact) {
#pragma unroll
                for (int s = 0; s < 4; ++s)
                    cp_async_8(b + s * (CZ_STAGE * 32) + (c ^ (si * G)), TT + min(max(mc + jofs[s] + kk, 0), n));
            }
        }
        cp_async_commit();
    };
    stage(0);
    CzStream s0, s1, s2, s3;
    s0.init(TT, m0 + jofs[0]);
    s1.init(TT, m0 + jofs[1]);
    s2.init(TT, m0 + jofs[2]);
    s3.init(TT, m0 + jofs[3]);
    auto out = [&](int k) {
        const int m = m0 + k;
        if (m >= L - 1 && m < n) cz_emit(Z, S, s3, k, f);   // always so for interior chunks
        else f(k, -CUDART_INF, -CUDART_INF);
    };
    if (has) out(0);
    {
        const double a = s0.next_safe(TT, r, n), b = s1.next_safe(TT, r, n), c = s2.next_safe(TT, r, n), d = s3.next_safe(TT, r, n);
        cz_update(Z, S, a, b, c, d);
    }
    constexpr int NP = (CH - 1) / CZ_STAGE;
#pragma unroll 1
    for (int p = 0; p < NP; ++p) {
        if (p + 1 < NP) {
            __syncwarp();   // every lane is done with the buffer of piece p - 1
            stage(p + 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncwarp();       // piece p of every lane has landed
        const double* b = slab + (p & 1) * (4 * CZ_STAGE * 32);
#pragma unroll 1
        for (int i = 0; i < CZ_STAGE; ++i) {
            const int k = 1 + p * CZ_STAGE + i;
            if (has) out(k);
            const int col = i * 32 + (lane ^ (i * G));
            const double a = s0.next_from(r, b[col]), bb = s1.next_from(r, b[CZ_STAGE * 32 + col]),
                         c = s2.next_from(r, b[2 * CZ_STAGE * 32 + col]), d = s3.next_from(r, b[3 * CZ_STAGE * 32 + col]);
            cz_update(Z, S, a, bb, c, d);
        }
    }
}
__device__ __forceinline__ void cz_out(const CzDev& Z, const double* TT, int n, int tid, CzState& S, double* obuf)
{
    cz_out_each(Z, TT, n, tid, S, [&](int k, double oc, double oz) { obuf[2 * k] = oc; obuf[2 * k + 1] = oz; });
}

// CUSP / ZAC outputs at the chunk start m0 = CH*tid from the closed-form state (the coarse grid of the pruning);
// -inf where m0 is not a valid output
__device__ __forceinline__ void cz_coarse(const CzDev& Z, const double* TT, int n, int tid, const CzState& S, double& oc, double& oz)
{
    const int m0 = tid * CH;
    oc = -CUDART_INF;
    oz = -CUDART_INF;
    if (!S.active || m0 < Z.L - 1 || m0 >= n) return;
    const double ylast = (m0 - Z.L >= 0) ? TT[m0 - Z.L + 1] - TT[m0 - Z.L] : 0.0;   // y[m0-L]
    const double Dc = (S.EpL - S.EmL + S.EpR - S.EmR) + S.W0F;
    oc = fma(Z.g, Dc, Z.gclast_cusp * ylast);
    const double poly = (S.W2L - Z.h2 * S.W1L) + (S.V2 - Z.h2 * S.V1);
    oz = fma(Z.g, fma(Z.B, poly, Dc), Z.gclast_zac * ylast);
}

// ==================================================================================================
// the fused kernel
// ==================================================================================================
// the two full trapezoid traces (e_10410-like A, e_313-like B), outputs strided over the block: maximum and maximum
// of the negated trace of each; the TT[j] stream is shared
__device__ __forceinline__ void trap_full2_minmax(const double* TT, const TrapDev& A, const TrapDev& B, int tid, double (&out)[4])
{
    double mxa = -CUDART_INF, mna = CUDART_INF, mxb = -CUDART_INF, mnb = CUDART_INF;
    const double* p0 = TT + tid;
    const double* a1 = p0 + A.a; const double* a2 = a1 + A.g; const double* a3 = p0 + A.L;
    const double* b1 = p0 + B.a; const double* b2 = b1 + B.g; const double* b3 = p0 + B.L;
    const double ai1 = A.inv1, ai2 = A.inv2, bi1 = B.inv1, bi2 = B.inv2;
    const int cnt = min(A.nout, B.nout) - tid;
    int off = 0;
    // (ternaries, not fmax/fmin: the NaN handling of those doubles the instruction count; an LDS-bound loop -- scaling
    //  the extrema once instead of every output was measured and changes nothing)
#pragma unroll 1
    for (; off < cnt; off += NT) {
        const double t0 = p0[off];
        const double oa = __fma_rn(a3[off] - a2[off], ai2, -__dmul_rn(a1[off] - t0, ai1));
        const double ob = __fma_rn(b3[off] - b2[off], bi2, -__dmul_rn(b1[off] - t0, bi1));
        mxa = oa > mxa ? oa : mxa; mna = oa < mna ? oa : mna;
        mxb = ob > mxb ? ob : mxb; mnb = ob < mnb ? ob : mnb;
    }
    // remainder of the longer trace
    const bool a_longer = A.nout > B.nout;
    const TrapDev& R = a_longer ? A : B;
    const double* r1 = p0 + R.a; const double* r2 = r1 + R.g; const double* r3 = p0 + R.L;
    const double ri1 = R.inv1, ri2 = R.inv2;
    double mx = -CUDART_INF, mn = CUDART_INF;
    const int cntr = R.nout - tid;
#pragma unroll 1
    for (; off < cntr; off += NT) {
        const double o = __fma_rn(r3[off] - r2[off], ri2, -__dmul_rn(r1[off] - p0[off], ri1));
        mx = o > mx ? o : mx; mn = o < mn ? o : mn;
    }
    if (a_longer) { mxa = mx > mxa ? mx : mxa; mna = mn < mna ? mn : mna; }
    else { mxb = mx > mxb ? mx : mxb; mnb = mn < mnb ? mn : mnb; }
    out[0] = mxa; out[1] = -mna; out[2] = mxb; out[3] = -mnb;
}

// upper bound of a trace on the open interval between two coarse points 33 samples apart, from the Lipschitz
// constant kap of the trace: a = value at the left point (always valid), b = value at the right point
__device__ __forceinline__ double interval_bound(double a, double b, bool b_valid, double kap)
{
    return b_valid ? fma(0.5 * (double)CH, kap, 0.5 * (a + b)) : fma((double)(CH - 1), kap, a);
}

__device__ __noinline__ double log_d(double x) { return log(x); }
// log1p(u) for |u| <= 1/8: Taylor series to u^18 (truncation < 1e-17 relative), Estrin scheme (dependency depth 6)
__device__ __forceinline__ double log1p_small(double u)
{
    const double u2 = u * u, u4 = u2 * u2, u8 = u4 * u4, u16 = u8 * u8;
    // c_k = (-1)^k / (k+1):  log1p(u) = u * sum_{k=0}^{17} c_k u^k
    const double a0 = fma(-1.0 / 2.0, u, 1.0), a1 = fma(-1.0 / 4.0, u, 1.0 / 3.0), a2 = fma(-1.0 / 6.0, u, 1.0 / 5.0),
                 a3 = fma(-1.0 / 8.0, u, 1.0 / 7.0), a4 = fma(-1.0 / 10.0, u, 1.0 / 9.0), a5 = fma(-1.0 / 12.0, u, 1.0 / 11.0),
                 a6 = fma(-1.0 / 14.0, u, 1.0 / 13.0), a7 = fma(-1.0 / 16.0, u, 1.0 / 15.0), a8 = fma(-1.0 / 18.0, u, 1.0 / 17.0);
    const double b0 = fma(a1, u2, a0), b1 = fma(a3, u2, a2), b2 = fma(a5, u2, a4), b3 = fma(a7, u2, a6);
    const double c0 = fma(b1, u4, b0), c1 = fma(b3, u4, b2);
    const double d0 = fma(c1, u8, c0);
    return u * fma(a8, u16, d0);
}
// threshold mask of one chunk of the PZ waveform: bit k = (y[i0+k] >= th), y from the prefix sums (tt0 = TT[i0])
__device__ __noinline__ unsigned long long mask_chunk(const double* tp, double tt0, int cvalid, double th)
{
    uint32_t lo = 0;
    double tprev = tt0;
    const int c32 = min(cvalid, 32);
#pragma unroll 1
    for (int k = 0; k < c32; ++k) {
        const double tn = tp[k + 1];
        lo |= ((tn - tprev) >= th) ? (1u << k) : 0u;
        tprev = tn;
    }
    unsigned long long m = lo;
    if (cvalid > 32 && (tp[33] - tprev) >= th) m |= 1ull << 32;
    return m;
}

// 32-bit samples: does the waveform sum to more than 32 bits (the uint32 prefix sums P would wrap)?  Block-uniform result.
// mx = block-wide maximum sample: the exact 64-bit sum is only formed when mx * n could reach 2^32; scratch = NWARP doubles
// (the sums are integers < 2^53: exact in double, in any order).  Contains two barriers on the slow path.
template <typename SAMPLE>
__device__ __forceinline__ bool sum_exceeds_u32(const SAMPLE* xp, int cvalid, uint32_t mx, int n, double* scratch)
{
    if (sizeof(SAMPLE) != 4 || (unsigned long long)mx * (unsigned long long)n <= 0xFFFFFFFFull) return false;
    unsigned long long c64 = 0;
    for (int k = 0; k < cvalid; ++k) c64 += (unsigned long long)xp[k];
    const double w = wsum_d((double)c64);
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = w;
    __syncthreads();
    const double total = red_sum(scratch, 0);
    __syncthreads();
    return total > 4294967295.0;
}

// ---------------------------------------------------------------------------------------------------
// Per-event arithmetic of both dsp_icpc paths: icpc_kernel and the split pipeline (lgdsp_icpc_split.cuh) call these
// functions, so both compute each of these values with the same expressions in the same order.
// ---------------------------------------------------------------------------------------------------
// SG trace sample j of filter f; sgg: shared-memory copy of the zero-padded taps of the short filters
__device__ __forceinline__ double sg_sample(const SgDev* sg, const double* TT, const double (*sgg)[8], int f, int j)
{
    return (sg[f].n_taps + 1 <= 8) ? sg_eval8(TT, sgg[f], j) : sg_eval(TT, sg[f].gg, sg[f].n_taps, j);
}
// t10..t99 [us] from the resolved position pos of threshold th on the PZ waveform; NaN -> 0
__device__ __forceinline__ double tx_us_at(const double* TT, int pos, double th, double t_first, double dt)
{
    double t = 0.0;
    if (pos >= 1) t = cross_x(th, y_at(TT, pos - 1), y_at(TT, pos), t_first + (double)(pos - 1) * dt, dt) * 0.001;
    return t != t ? 0.0 : t;
}
// t0 / t0_inv [us] from the resolved position of the t0 (inv: t0_inv) mask; NaN -> 0
__device__ __forceinline__ double t0_us_at(const IcpcDev& P, const double* TT, bool inv, int pos, double t_first, double dt)
{
    const TrapDev& tr = inv ? P.t0inv : P.t0;
    double t = 0.0;
    if (pos >= 1) {
        const double tl = t_first + (double)(pos - 1 + tr.L - 1) * dt;
        const double sgn = inv ? -1.0 : 1.0;
        t = cross_x(P.t0_thr, sgn * trap_at_i(TT, tr, pos - 1), sgn * trap_at_i(TT, tr, pos), tl, dt) * 0.001;
    }
    return t != t ? 0.0 : t;
}
// get_qdrift  src/dsp_routines.jl:51-64 on the integrator trace I[i] = TT[i+1] at t_us, one warp
__device__ __forceinline__ double qdrift_at(const IcpcDev& P, const double* TT, const double* A_int, int n, double t_first, double dt,
                                            double t_us, double first, double last, int lane)
{
    const double tns = t_us * 1000.0;
    if (P.int_dni.n_w <= 8) {
        // the three estimates in parallel, 8 lanes each
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
}

// CUSP/ZAC candidate chunk: Lipschitz bound on (33 tid, 33 tid + 33) against the best coarse values Mc / Mz; chunks that
// hold part of a pick-off window (pk_from[ic] for CUSP, pk_from[iz] for ZAC, nw samples each) are always evaluated.
// czco: the coarse values [2][NT]
__device__ __forceinline__ bool cz_candidate(const CzDev& Z, const CzState& st, double oc, double oz, const double* czco, int tid, int i0,
                                             double Ymax, double Mc, double Mz, bool want_cusp, bool want_zac, const int* pk_from,
                                             int ic, int iz, int nw)
{
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
            cand |= (jhi >= pk_from[ic] && jlo < pk_from[ic] + nw);
        }
        if (want_zac) {
            const double a = oz, b = (tid + 1 < NT) ? czco[NT + t1] : -CUDART_INF;
            const double kz = kap * Z.lip_zac;
            double bound;
            if (a > -CUDART_INF) bound = interval_bound(a, b, b > -CUDART_INF, kz);
            else if (b > -CUDART_INF) bound = fma((double)CH, kz, b);
            else bound = CUDART_INF;
            cand |= bound + 1e-6 * (fabs(Mz) + Ymax * fabs(Z.g)) >= Mz;
            cand |= (jhi >= pk_from[iz] && jlo < pk_from[iz] + nw);
        }
    }
    return cand;
}

// Raw-sample pass of one event: this thread's chunk of cvalid samples at xs + i0 and block-wide results.  Writes the
// R_BLS .. R_SQ slots of red, ends behind one block barrier.  lean: the baseline slope / sigma sums are not wanted.
struct RawPass {
    uint32_t cmn, cmx;      // chunk min / max
    uint32_t mn, mx;        // block min / max
    int nlow, nhigh;        // block-wide saturation counts
    uint32_t P_excl;        // exclusive prefixes of the chunk: cumsum(x) and cumsum(cumsum(x)) before sample i0
    double PP_excl;
};
template <typename SAMPLE>
__device__ __forceinline__ RawPass raw_pass(const SAMPLE* xs, int i0, int cvalid, int bl_from, int bl_until, int sat_low, int sat_high,
                                            bool lean, double* red, int tid, int lane, int wid)
{
    RawPass r;
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
    r.cmn = cmn; r.cmx = cmx;
    // baseline regression sums (exact integers), samples of the window strided over ALL threads (the window covers the
    // first chunks only: summed chunk-wise, three warps would do the whole job while the others wait at the barrier)
    {
        unsigned long long blSS = 0, blSX = 0;
        uint32_t blS = 0;
#pragma unroll 2
        for (int idx = bl_from + tid; idx <= bl_until; idx += NT) {
            const uint32_t x = xs[idx];
            blS += x;
            if (!lean) {
                blSX += (unsigned long long)x * (unsigned long long)idx;
                blSS += (unsigned long long)x * (unsigned long long)x;
            }
        }
        // (all sums < 2^53: exact in double, in any order)
        const double a = wsum_d((double)blS), bq = wsum_d((double)blSS), c = wsum_d((double)blSX);
        if (lane == 0) { red[R_BLS * NWARP + wid] = a; red[R_BLSS * NWARP + wid] = bq; red[R_BLSX * NWARP + wid] = c; }
    }
    // saturation counts: a sample can only equal low/high if the chunk's min/max says so
    int nlow = 0, nhigh = 0;
    if ((int)cmn == sat_low || (int)cmx == sat_high) {
        for (int k = 0; k < cvalid; ++k) {
            const int x = xp[k];
            nlow += (x == sat_low);
            nhigh += (x == sat_high);
        }
    }
    {
        const uint32_t wmn = __reduce_min_sync(FULL, cmn), wmx = __reduce_max_sync(FULL, cmx);
        const uint32_t wl = __reduce_add_sync(FULL, (uint32_t)nlow), wh = __reduce_add_sync(FULL, (uint32_t)nhigh);
        if (lane == 0) {
            uint32_t* ured = reinterpret_cast<uint32_t*>(red + R_MX * NWARP);
            ured[wid] = wmx; ured[NWARP + wid] = wmn; ured[2 * NWARP + wid] = wl; ured[3 * NWARP + wid] = wh;
        }
    }
    // one scan for P = cumsum(x) and PP = cumsum(P): segments (len, s = sum x, q = sum of the inclusive
    // prefix sums inside the segment) combine as (lenA+lenB, sA+sB, qA+qB+lenB*sA); all values exact
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
        red[R_SLEN * NWARP + wid] = (double)sl;
        red[R_SS * NWARP + wid] = (double)ss;
        red[R_SQ * NWARP + wid] = sq;
    }
    int el = __shfl_up_sync(FULL, sl, 1);
    uint32_t es = __shfl_up_sync(FULL, ss, 1);
    double eq = __shfl_up_sync(FULL, sq, 1);
    if (lane == 0) { el = 0; es = 0; eq = 0.0; }
    __syncthreads();

    {
        double cs = 0.0, cqd = 0.0;
#pragma unroll 1
        for (int w = 0; w < wid; ++w) {
            const double lw = red[R_SLEN * NWARP + w], sw = red[R_SS * NWARP + w], qw = red[R_SQ * NWARP + w];
            cqd = cqd + qw + lw * cs;
            cs += sw;
        }
        r.P_excl = (uint32_t)cs + es;
        r.PP_excl = cqd + eq + (double)el * cs;
    }
    {
        const uint32_t* ured = reinterpret_cast<const uint32_t*>(red + R_MX * NWARP);
        const int l8 = lane & 7;
        r.mx = __reduce_max_sync(FULL, ured[l8]);
        r.mn = __reduce_min_sync(FULL, ured[NWARP + l8]);
        r.nlow = (int)__reduce_add_sync(FULL, lane < 8 ? ured[2 * NWARP + l8] : 0u);
        r.nhigh = (int)__reduce_add_sync(FULL, lane < 8 ? ured[3 * NWARP + l8] : 0u);
    }
    return r;
}

// Closed-form prefix sums of the pole-zero waveform y = w + km1 * cumsum(w), w = x - m, along one chunk:
// next(x) turns the following raw sample into TT[i + 1] = cumsum(y)[i]
struct PzScan {
    uint32_t Pr;     // cumsum(x)[i]
    double PPr;      // cumsum(cumsum(x))[i]
    double ip1;      // i + 1 after the update
    double tri;      // (i + 1)(i + 2) / 2 after the update
    __device__ __forceinline__ double next(uint32_t x, double m, double km1)
    {
        Pr += x;
        const double Pd = u2d(Pr);
        PPr += Pd;
        ip1 += 1.0;
        tri += ip1;
        const double Sd = fma(-ip1, m, Pd);    // cumsum(w)[i]
        const double SS = fma(-tri, m, PPr);   // cumsum(cumsum(w))[i]
        return fma(km1, SS, Sd);
    }
};
// Start of the chunk at i0 from its exclusive prefixes, and conservative bounds ylo / yhi (+- guard) of y on the chunk from
// the integer min / max of its raw samples: cumsum(w)[i0+k] lies between S0 + (k+1)*wmin and S0 + (k+1)*wmax.
struct PzChunk {
    PzScan scan;
    double TT0;                // TT[i0] (bit-identical to the neighbour's)
    double ylo, yhi, guard;
};
__device__ __forceinline__ PzChunk pz_chunk(int i0, double m, double km1, uint32_t P_excl, double PP_excl, uint32_t cmn, uint32_t cmx)
{
    PzChunk c;
    const double Sd0 = fma(-(double)i0, m, u2d(P_excl));   // cumsum(w)[i0-1]
    const double tri0 = 0.5 * (double)i0 * ((double)i0 + 1.0);
    c.TT0 = fma(km1, fma(-tri0, m, PP_excl), Sd0);
    c.scan = {P_excl, PP_excl, (double)i0, tri0};
    const double wmin = (double)cmn - m, wmax = (double)cmx - m;
    const double ak = fabs(km1);
    const double srange = (double)CH * fmax(fabs(wmin), fabs(wmax));
    c.ylo = wmin + km1 * Sd0 - ak * srange;
    c.yhi = wmax + km1 * Sd0 + ak * srange;
    c.guard = 1e-9 * (fabs(c.ylo) + fabs(c.yhi)) + 1e-6;   // >> rounding of the TT differences
    return c;
}

// Saturation run lengths (n_sat_low_cons, n_sat_high_cons) of an event with a saturated sample; block-wide, two barriers.
// ired: int[8 * NWARP] of scratch.
template <typename SAMPLE>
__device__ __forceinline__ int2 sat_runs(int sat_low, int sat_high, const SAMPLE* xp, int cvalid, int lane, int wid, int* ired)
{
    Run rl = {0, 0, 0, cvalid}, rh = {0, 0, 0, cvalid};
    {
        int cl = 0, chh = 0;
        bool pl = true, ph = true;
        for (int k = 0; k < cvalid; ++k) {
            const int x = xp[k];
            const bool il = (x == sat_low), ih = (x == sat_high);
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
    __syncthreads();   // the scratch may be reused behind this barrier
    return make_int2(al.best, ah.best);
}

// get_wvf_maximum  src/interpolation.jl:30-46 of current trace f = lane (0..2: sg[f], 3: the derivative), lanes 0..3,
// from the block-wide first argmax in the slots cmax0 + f / carg0 + f of red: parabola only if strictly inside the window
__device__ __forceinline__ void currents_job(const double* TT, const SgDev* sg, const double (*sgg)[8], const int* sg_alias,
                                             const int* cur_from, const int* cur_until, const double* red, int cmax0, int carg0,
                                             double* row, int lane)
{
    double vv[4];
    int aa[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        const int fs = (f < 3 && sg_alias[f] >= 0) ? sg_alias[f] : f;   // aliased filter: same trace and window
        red_argmax(red, cmax0 + fs, carg0 + fs, vv[f], aa[f]);
    }
    if (lane < 4) {
        const int f = lane;
        double v = f == 0 ? vv[0] : f == 1 ? vv[1] : f == 2 ? vv[2] : vv[3];
        const int a = f == 0 ? aa[0] : f == 1 ? aa[1] : f == 2 ? aa[2] : aa[3];
        if (a > cur_from[f] && a < cur_until[f]) {
            const double y1 = (f < 3) ? sg_sample(sg, TT, sgg, f, a - 1) : deriv_at(TT, a - 1);
            const double y3 = (f < 3) ? sg_sample(sg, TT, sgg, f, a + 1) : deriv_at(TT, a + 1);
            v = extrema3(y1, v, y3);
        }
        row[LGDSP_COL_a_sg + f] = v;
    }
}

// Levels of an event from its baseline mean m and its sample min / max: e_max, e_min and the t10..t99 thresholds
// (lean: only t50)
struct Levels { double e_max, e_min, thr[5]; };
__device__ __forceinline__ Levels event_levels(double m, uint32_t mx, uint32_t mn, const double* tx_frac, bool lean)
{
    Levels v;
    v.e_max = (double)mx - m;
    v.e_min = (double)mn - m;
#pragma unroll
    for (int k = 0; k < 5; ++k) v.thr[k] = v.e_max * tx_frac[k];
    if (lean) { v.thr[0] = CUDART_INF; v.thr[2] = CUDART_INF; v.thr[3] = CUDART_INF; v.thr[4] = CUDART_INF; }
    return v;
}

// SAMPLE = uint16_t (raw FADC samples) or uint32_t (presummed waveforms of dsp_icpc_compressed, n <= 4096).
// bl_ext != NULL: the baseline mean of event e is bl_ext[e] instead of the bl_window mean (windowed waveforms of
// dsp_icpc_compressed are shifted by blmean_presummed / presum_rate, src/dsp_icpc.jl:350).
template <typename SAMPLE>
__global__ void __launch_bounds__(NT, 2)
icpc_kernel(const __grid_constant__ IcpcDev P, const SAMPLE* __restrict__ wf, long long n_events, long long ld,
            const double* __restrict__ bl_ext, long long bl_stride, double bl_div, double* __restrict__ rows)
{
    extern __shared__ __align__(128) unsigned char smem[];
    SAMPLE* xs = reinterpret_cast<SAMPLE*>(smem + SM_XS);
    double* TT = reinterpret_cast<double*>(smem + SM_TT);
    uint32_t* masks = reinterpret_cast<uint32_t*>(smem + SM_MASK);
    double* red = reinterpret_cast<double*>(smem + SM_RED);
    double* stash = reinterpret_cast<double*>(smem + SM_STASH);
    double* row = reinterpret_cast<double*>(smem + SM_ROW);
    double* scr = reinterpret_cast<double*>(smem + SM_SCR);
    int* ibuf = reinterpret_cast<int*>(smem + SM_IBUF);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + SM_BAR);
    double* czco = reinterpret_cast<double*>(masks + M_T10 * NWORDS);   // coarse CUSP/ZAC values [2][NT]
    double* tabA = reinterpret_cast<double*>(smem + SM_XS);
    double* tabB = reinterpret_cast<double*>(smem + SM_TAB);

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n = P.n;
    const uint32_t wf_bytes = (uint32_t)n * (uint32_t)sizeof(SAMPLE);
    const double t_first = P.t_first, dt = P.dt;
    const unsigned G = P.groups;
    const double* A_int = P.dni_A;                       // global, L1/L2 resident (4 KB)
    const double* A_sig = P.dni_A + LGDSP_MAX_DNI * 4;

    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    if (tid < TT_LEN - 1 - n) TT[n + 1 + tid] = 0.0;   // finite padding behind the trace (zero-padded SG kernels read it)
    SmemPar* spar = reinterpret_cast<SmemPar*>(smem + SM_PAR);
    {
        // parameter tables used by noinline helpers: SMEM copies (once per CTA; the kernel is persistent)
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&P.cz[0]);
        uint32_t* dst = reinterpret_cast<uint32_t*>(&spar->cz[0]);
        for (int i = tid; i < (int)(2 * sizeof(CzDev) / 4); i += NT) dst[i] = src[i];
        if (tid < 24) spar->sgg[tid >> 3][tid & 7] = P.sg[tid >> 3].gg[tid & 7];
    }
    __syncthreads();
    // SG trace sample j of filter f
    auto sg_at = [&](int f, int j) -> double { return sg_sample(P.sg, TT, spar->sgg, f, j); };
    long long e = blockIdx.x;
    if (tid == 0 && e < n_events) {
        mbar_expect_tx(bar, wf_bytes);
        tma_load_1d(xs, wf + e * ld, wf_bytes, bar);
    }
    uint32_t phase = 0;
    const int i0 = tid * CH;
    const int cvalid = max(0, min(CH, n - i0));
    const unsigned long long chunk_all = (1ull << cvalid) - 1ull;   // cvalid <= 33
    const bool cz_on = (G & LGDSP_GROUP_CUSPZAC) != 0;
    const bool cz_structured = cz_on && !P.direct;
    const int npass = cz_structured ? (P.cz_shared ? 1 : 2) : 0;

    for (; e < n_events; e += gridDim.x) {
        // ==========================================================================================
        // P1: raw samples
        // ==========================================================================================
        mbar_wait(bar, phase);
        phase ^= 1;
        // zero the masks and the queue counters of this event (committed with atomics later)
#pragma unroll
        for (int q = 0; q < NMASK; ++q) masks[q * NWORDS + tid] = 0u;
        if (tid == 0) { ibuf[IB_QN] = 0; ibuf[IB_CZN] = 0; }
        const SAMPLE* xp = xs + i0;
        const RawPass rp = raw_pass<SAMPLE>(xs, i0, cvalid, P.bl_from, P.bl_until, P.sat_low, P.sat_high, (G & LGDSP_GROUP_LEAN) != 0,
                                            red, tid, lane, wid);   // ---- B1 ----
        const uint32_t mx = rp.mx, mn = rp.mn;
        const int nlow = rp.nlow, nhigh = rp.nhigh;
        // saturation run lengths (only when a saturated sample exists; block-uniform branch)
        int cons_low = 0, cons_high = 0;
        if (nlow + nhigh > 0) {
            const int2 c = sat_runs<SAMPLE>(P.sat_low, P.sat_high, xp, cvalid, lane, wid, reinterpret_cast<int*>(stash));   // stash is idle here
            cons_low = c.x; cons_high = c.y;
        }

        // (32-bit samples whose sum leaves 32 bits: the row is NaN instead of silently wrong)
        const bool wrapped = sum_exceeds_u32<SAMPLE>(xp, cvalid, mx, n, red + R_TLS * NWARP);
        // blmean = mean_Y = sum_Y * inv_n exactly as signalstats computes it (the other baseline statistics: P5)
        const double m = bl_ext ? div_rn(bl_ext[e * bl_stride], bl_div) : mul_rn(red_sum(red, R_BLS), P.bl_inv_n);
        const Levels lv = event_levels(m, mx, mn, P.tx_frac, (G & LGDSP_GROUP_LEAN) != 0);
        const double e_max = lv.e_max, e_min = lv.e_min;
        double thr[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) thr[k] = lv.thr[k];

        // ==========================================================================================
        // P2: prefix sums of the pole-zero waveform; t10..t99 masks; tail log-regression
        // ==========================================================================================
        {
            const double km1 = P.km1;
            PzChunk pz = pz_chunk(i0, m, km1, rp.P_excl, rp.PP_excl, rp.cmn, rp.cmx);
            const double TT0 = pz.TT0, ylo = pz.ylo, yhi = pz.yhi, guard = pz.guard;
            {
                double* tp = TT + i0 + 1;
                auto body = [&](int k) { tp[k] = pz.scan.next(xp[k], m, km1); };
                int k = 0;
#pragma unroll 1
                for (; k + 3 <= cvalid; k += 3) { body(k); body(k + 1); body(k + 2); }
#pragma unroll 1
                for (; k < cvalid; ++k) body(k);
                if (tid == 0) TT[0] = 0.0;
            }
            // t10..t99: a chunk entirely below (above) a threshold contributes zeros (ones) without a compare
            if (G & LGDSP_GROUP_TIMING) {
                uint32_t lo[5] = {0, 0, 0, 0, 0}, hi = 0;   // bits 0..31 of every threshold; bit t of hi = sample 32
                bool straddle = false;
#pragma unroll
                for (int t = 0; t < 5; ++t) straddle |= !(ylo - guard >= thr[t]) && !(yhi + guard < thr[t]);
                if (straddle && cvalid > 0) {
                    // one pass over the chunk, the five compares are independent (y from the prefix sums)
                    const double* tp = TT + i0;
                    double tprev = TT0;
                    const int c32 = min(cvalid, 32);
                    double tnx = tp[1];                       // software prefetch: the load of sample k+1 overlaps sample k
#pragma unroll 1
                    for (int k = 0; k < c32; ++k) {
                        const double tn = tnx;
                        tnx = tp[k + 2];                      // (<= TT[i0+34]: inside the zero padding for the last chunk)
                        const double y = tn - tprev;
                        tprev = tn;
                        const uint32_t bit = 1u << k;
#pragma unroll
                        for (int t = 0; t < 5; ++t) lo[t] |= (y >= thr[t]) ? bit : 0u;
                    }
                    if (cvalid > 32) {
                        const double y = tnx - tprev;
#pragma unroll
                        for (int t = 0; t < 5; ++t) hi |= (y >= thr[t]) ? (1u << t) : 0u;
                    }
                }
                // The 32 chunks of a warp cover the 33 mask words [33*wid, 33*wid + 32] exactly (chunk of lane l starts at bit l
                // of word 33*wid + l): every word is assembled from this lane's chunk and its neighbour's top bits and written
                // with a plain store -- no atomics, no dependence on the zero fill.
#pragma unroll
                for (int t = 0; t < 5; ++t) {
                    unsigned long long mbt = (unsigned long long)lo[t] | ((unsigned long long)((hi >> t) & 1u) << 32);
                    if (cvalid <= 0) mbt = 0ull;
                    else if (ylo - guard >= thr[t]) mbt = chunk_all;
                    else if (yhi + guard < thr[t]) mbt = 0ull;
                    const unsigned long long up = __shfl_up_sync(FULL, mbt, 1);
                    uint32_t word = (uint32_t)(mbt << lane);
                    if (lane > 0) word |= (uint32_t)(up >> (33 - lane));
                    uint32_t* M = masks + (M_T10 + t) * NWORDS;
                    const int w = (CH * wid) + lane;
                    if (w < NWORDS) M[w] = word;
                    if (lane == 31 && w + 1 < NWORDS) M[w + 1] = (uint32_t)(mbt >> 1);
                }
            }
            // bound of max |y| over the block (Lipschitz constants of the pruning)
            const double ya = wmax_d(cvalid > 0 ? fmax(fabs(ylo), fabs(yhi)) : 0.0);
            red_put(red, R_YMAX, wid, lane, ya);
        }
        // tailstats: log-regression on the PRE-PZ waveform (src/tailstats.jl:22-72), samples strided over the block
        {
            double tl_S = 0, tl_SS = 0, tl_SX = 0;
            bool bad = false;
            // log(w) = log(c) + log1p((w - c)/c) around a per-thread reference sample c: one full log per thread, the
            // others are short polynomials unless the tail moves by more than 1/8 (then the full log again);
            // two samples per iteration so that their polynomial chains overlap
            double cref = 0.0, cinv = 0.0, clog = 0.0;
            auto one = [&](int idx, double w, double u) {
                if (w <= 0.0) { bad = true; return; }
                double lg;
                if (cref > 0.0 && fabs(u) <= 0.125) {
                    lg = clog + log1p_small(u);
                } else {
                    lg = log_d(w);
                    cref = w; cinv = 1.0 / w; clog = lg;
                }
                const double X = t_first + (double)idx * dt;
                tl_S += lg;
                tl_SS = fma(lg, lg, tl_SS);
                tl_SX = fma(X, lg, tl_SX);
            };
#pragma unroll 1
            for (int idx = P.tail_from + tid; idx <= P.tail_until; idx += 2 * NT) {
                const bool two = idx + NT <= P.tail_until;
                const double w0 = u2d(xs[idx]) - m, w1 = two ? u2d(xs[idx + NT]) - m : cref;
                const double u0 = (w0 - cref) * cinv, u1 = (w1 - cref) * cinv;
                if (two && cref > 0.0 && w0 > 0.0 && w1 > 0.0 && fabs(u0) <= 0.125 && fabs(u1) <= 0.125) {
                    // common case: both through the polynomial, interleaved
                    const double l0 = clog + log1p_small(u0), l1 = clog + log1p_small(u1);
                    const double X0 = t_first + (double)idx * dt, X1 = t_first + (double)(idx + NT) * dt;
                    tl_S += l0; tl_SS = fma(l0, l0, tl_SS); tl_SX = fma(X0, l0, tl_SX);
                    tl_S += l1; tl_SS = fma(l1, l1, tl_SS); tl_SX = fma(X1, l1, tl_SX);
                } else {
#pragma unroll 1
                    for (int q = 0; q < (two ? 2 : 1); ++q) {
                        const double w = q ? w1 : w0;
                        one(idx + q * NT, w, (w - cref) * cinv);
                    }
                }
            }
            tl_S = wsum_d(tl_S); tl_SS = wsum_d(tl_SS); tl_SX = wsum_d(tl_SX);
            const bool anybad = __any_sync(FULL, bad);
            if (lane == 0) {
                red[R_TLS * NWARP + wid] = tl_S; red[R_TLSS * NWARP + wid] = tl_SS;
                red[R_TLSX * NWARP + wid] = tl_SX; red[R_TLBAD * NWARP + wid] = anybad ? 1.0 : 0.0;
            }
        }
        __syncthreads();   // ---- B2: TT and the t10..t99 masks are complete; xs is dead ----

        // xs is free now: prefetch the next event (TMA, async proxy) -- unless the structured CUSP/ZAC pass borrows
        // xs for its prefix tables; then the prefetch is issued when the tables are dead
        auto prefetch_next = [&]() {
            if (tid == 0) {
                const long long en = e + gridDim.x;
                if (en < n_events) {
                    fence_proxy_async();
                    mbar_expect_tx(bar, wf_bytes);
                    tma_load_1d(xs, wf + en * ld, wf_bytes, bar);
                }
            }
        };
        if (!cz_structured) prefetch_next();

        // ==========================================================================================
        // P3: work that only needs TT
        // ==========================================================================================
        // resolve t10..t99 (t50 positions the energy pick-off windows)
        if (wid < 5) {
            int pos, mult;
            resolve_runs(masks + (M_T10 + wid) * NWORDS, P.tx_min_n, lane, pos, mult);
            if (lane == 0) ibuf[IB_POS0 + M_T10 + wid] = pos;
            if (wid == M_T50 - M_T10 && lane < 3) {
                // t50 [us] and the DNI window of energy pick-off `lane` (0 trap, 1 cusp, 2 zac): published for everyone
                double t50_us = 0.0;
                if (pos >= 1) {
                    const double x = cross_x(thr[1], y_at(TT, pos - 1), y_at(TT, pos), t_first + (double)(pos - 1) * dt, dt);
                    t50_us = x * 0.001;
                }
                const int Lf = lane == 0 ? P.etrap.L : lane == 1 ? P.cusp_L : P.zac_L;
                const double pick = lane == 0 ? P.trap_pick : lane == 1 ? P.cusp_pick : P.zac_pick;
                const double tf = t_first + (double)(Lf - 1) * dt;
                double pp;
                int pf;
                dni_window(P.sig_dni.n_w, n - Lf + 1, (t50_us * 1000.0 + pick - tf) / dt, pp, pf);
                scr[SC_PKP + lane] = pp;
                ibuf[IB_PKFROM + lane] = pf;
            }
        }
        // PZ tail statistics (signalstats on the tail window, src/dsp_icpc.jl:123)
        {
            double pz_S = 0, pz_SS = 0, pz_SX = 0;
#pragma unroll 1
            for (int idx = P.tail_from + tid; idx <= P.tail_until; idx += NT) {
                const double y = TT[idx + 1] - TT[idx];
                const double X = t_first + (double)idx * dt;
                pz_S += y;
                pz_SS = fma(y, y, pz_SS);
                pz_SX = fma(X, y, pz_SX);
            }
            pz_S = wsum_d(pz_S); pz_SS = wsum_d(pz_SS); pz_SX = wsum_d(pz_SX);
            if (lane == 0) {
                red[R_PZS * NWARP + wid] = pz_S; red[R_PZSS * NWARP + wid] = pz_SS; red[R_PZSX * NWARP + wid] = pz_SX;
            }
        }
        // trapezoids whose minimum is needed as well: full traces
        if (G & LGDSP_GROUP_TRAPS) {
            double o4[4];
            trap_full2_minmax(TT, P.e10410, P.e313, tid, o4);
            const double a = wmax_d(o4[0]), b = wmax_d(o4[1]), c = wmax_d(o4[2]), d = wmax_d(o4[3]);
            if (lane == 0) {
                red[R_E104 * NWARP + wid] = a; red[R_E104N * NWARP + wid] = b;
                red[R_E313 * NWARP + wid] = c; red[R_E313N * NWARP + wid] = d;
            }
        }
        // coarse grid (outputs 33*tid and 33*(tid+1)) of the other trapezoids
        double c0a = 0, c0b = 0, cia = 0, cib = 0, c5a = -CUDART_INF, c5b = -CUDART_INF, cea = -CUDART_INF, ceb = -CUDART_INF;
        {
            const int ja = i0, jb = i0 + CH;
            if (G & LGDSP_GROUP_TIMING) {
                if (ja < P.t0.nout) c0a = trap_at_i(TT, P.t0, ja);
                if (jb < P.t0.nout) c0b = trap_at_i(TT, P.t0, jb);
                if (!P.t0inv_same) {
                    if (ja < P.t0inv.nout) cia = trap_at_i(TT, P.t0inv, ja);
                    if (jb < P.t0inv.nout) cib = trap_at_i(TT, P.t0inv, jb);
                }
            }
            if (G & LGDSP_GROUP_TRAPS) {
                if (ja < P.e535.nout) c5a = trap_at_i(TT, P.e535, ja);
                if (jb < P.e535.nout) c5b = trap_at_i(TT, P.e535, jb);
                if (ja < P.etrap.nout) cea = trap_at_i(TT, P.etrap, ja);
                if (jb < P.etrap.nout) ceb = trap_at_i(TT, P.etrap, jb);
                const double w5 = wmax_d(c5a), we = wmax_d(cea);
                red_put(red, R_C535, wid, lane, w5);
                red_put(red, R_CET, wid, lane, we);
            }
        }
        // currents: sg[0] over the whole trace (chunked, sliding window in registers): trace maximum, windowed first
        // argmax, baseline-window sums; the chunk maximum is kept for the mask pass
        double sgcmax = -CUDART_INF;
        const int nsg = P.sg[0].nout;
        const bool want_cur = (G & LGDSP_GROUP_CURRENT) != 0, want_intr = (G & LGDSP_GROUP_INTRACE) != 0;
        if (want_cur || want_intr) {
            double cmax[4] = {-CUDART_INF, -CUDART_INF, -CUDART_INF, -CUDART_INF};
            int carg[4] = {0x7fffffff, 0x7fffffff, 0x7fffffff, 0x7fffffff};
            double sg_S = 0, sg_SS = 0;
            // (a) whole trace, one chunk per thread: only the chunk maximum (uniform cost for every thread)
            if (want_intr) sg_chunk(TT, P.sg[0], i0, min(CH, nsg - i0), [&](int k, double s) { sgcmax = s > sgcmax ? s : sgcmax; });
            // (b) windowed quantities, strided over the block (same operation order as the chunk pass: identical values):
            //     first argmax of sg[0..2] and of the plain derivative inside the current window, baseline-window sums of sg[0]
#pragma unroll 1
            for (int f = 0; f < 3; ++f) {
                if (f > 0 && P.sg_alias[f] >= 0) continue;   // identical to an earlier filter: copied after the reduction
                if (f > 0 && !want_cur) continue;            // only the in-trace statistics of sg[0] are wanted
                double bm = -CUDART_INF;
                int ba = 0x7fffffff;
                if (P.sg[f].n_taps + 1 <= 8) {
                    double g[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) g[q] = spar->sgg[f][q];
                    auto ev = [&](int j) -> double {
                        const double* p = TT + j;
                        double a0 = g[0] * p[0], a1 = g[1] * p[1];
                        a0 = fma(g[2], p[2], a0); a1 = fma(g[3], p[3], a1);
                        a0 = fma(g[4], p[4], a0); a1 = fma(g[5], p[5], a1);
                        a0 = fma(g[6], p[6], a0); a1 = fma(g[7], p[7], a1);
                        return a0 + a1;
                    };
                    if (want_cur) {
#pragma unroll 1
                        for (int j = P.cur_from[f] + tid; j <= P.cur_until[f]; j += NT) {
                            const double v = ev(j);
                            if (v > bm) { bm = v; ba = j; }
                        }
                    }
                    if (f == 0 && want_intr) {
#pragma unroll 1
                        for (int j = P.intr_from + tid; j <= P.intr_until; j += NT) {
                            const double v = ev(j);
                            sg_S += v;
                            sg_SS = fma(v, v, sg_SS);
                        }
                    }
                } else {
                    if (want_cur) {
#pragma unroll 1
                        for (int j = P.cur_from[f] + tid; j <= P.cur_until[f]; j += NT) {
                            const double v = sg_at(f, j);
                            if (v > bm) { bm = v; ba = j; }
                        }
                    }
                    if (f == 0 && want_intr) {
#pragma unroll 1
                        for (int j = P.intr_from + tid; j <= P.intr_until; j += NT) {
                            const double v = sg_at(0, j);
                            sg_S += v;
                            sg_SS = fma(v, v, sg_SS);
                        }
                    }
                }
                if (f == 0) { cmax[0] = bm; carg[0] = ba; } else if (f == 1) { cmax[1] = bm; carg[1] = ba; } else { cmax[2] = bm; carg[2] = ba; }
            }
            if (want_cur) {
#pragma unroll 1
                for (int j = P.cur_from[3] + tid; j <= P.cur_until[3]; j += NT) {
                    const double d = deriv_at(TT, j);
                    if (d > cmax[3]) { cmax[3] = d; carg[3] = j; }
                }
            }
            const double wsm = wmax_d(sgcmax);
            sg_S = wsum_d(sg_S); sg_SS = wsum_d(sg_SS);
#pragma unroll
            for (int f = 0; f < 4; ++f) cmax[f] = wargmax_d(cmax[f], carg[f]);
            if (lane == 0) {
                red[R_SGMAX * NWARP + wid] = wsm; red[R_SGS * NWARP + wid] = sg_S; red[R_SGSS * NWARP + wid] = sg_SS;
#pragma unroll
                for (int f = 0; f < 4; ++f) {
                    red[(R_CMAX0 + f) * NWARP + wid] = cmax[f];
                    red[(R_CARG0 + f) * NWARP + wid] = (double)carg[f];
                }
            }
        }
        // CUSP/ZAC prefix tables (first descriptor)
        if (cz_structured) cz_scan<SM_PAR>(npass == 2 ? 1 : 0, TT, n, tid, tabA, tabB, red + R_CZSCR * NWARP, scr + SC_PP0);
        __syncthreads();   // ---- B3 ----

        // ==========================================================================================
        // P4a: decisions that need block-wide values; fine evaluation of the flagged intervals
        // ==========================================================================================
        if (tid < 64) row[tid] = 0.0;
        // DNI windows of the three energy pick-offs (computed by the t50 warp in P3)
        double pk_p[3];
        int pk_from[3];
#pragma unroll
        for (int f = 0; f < 3; ++f) { pk_p[f] = scr[SC_PKP + f]; pk_from[f] = ibuf[IB_PKFROM + f]; }
        const double Ymax = red_max(red, R_YMAX);     // bound of max |y| of the PZ waveform
        const double kslack = 1e-7 * Ymax;            // >> float64 rounding of any trace
        // the 44 trap(rt,ft) outputs of the e_trap pick-off window
        if ((G & LGDSP_GROUP_TRAPS) && tid < P.sig_dni.n_w) stash[tid] = trap_at_i(TT, P.etrap, pk_from[0] + tid);

        // ---- thresholds of the sg[0] masks (t50_current at half the trace maximum; pile-up at n sigma of the baseline
        //      window, sigma exactly as signalstats computes it) ----
        double pile_thr = 0.0, cur_thr = 0.0;
        if (G & LGDSP_GROUP_INTRACE) {
            cur_thr = red_max(red, R_SGMAX) * 0.5;
            const double sS = red_sum(red, R_SGS), sSS = red_sum(red, R_SGSS);
            const double mean_Y = mul_rn(sS, P.intr_inv_n);
            double var_Y = sub_rn(mul_rn(sSS, P.intr_inv_n), mul_rn(mean_Y, mean_Y));
            if (var_Y < 0) var_Y = 0;
            pile_thr = sqrt(var_Y) * P.nsigma;
            if (pile_thr == 0.0) pile_thr = 1.0;  // src/dsp_routines.jl:77
        }
        uint16_t* qitems = reinterpret_cast<uint16_t*>(czco + 2 * NT);   // work queue behind the coarse CUSP/ZAC values
        double e535 = c5a, etmax = cea;
        int etarg = (cea > -CUDART_INF) ? i0 : 0x7fffffff;
        // one flagged interval / chunk q, evaluated by a whole warp (one output per lane):
        //   type 0: trap(t0) on (33q, 33q+33) -> t0 mask (and t0_inv mask when both use the same filter); 1: t0_inv filter;
        //   2: trap(5,3) maximum; 3: trap(rt,ft) maximum + first argmax; 4: sg[0] chunk q -> t50_current / pile-up masks
        auto do_item = [&](int type, int q) {
            if (type <= 1) {
                const TrapDev& tr = type == 0 ? P.t0 : P.t0inv;
                const double th = P.t0_thr;
                const int j = q * CH + 1 + lane;
                const bool v = j < tr.nout;
                const double o = v ? trap_at_i(TT, tr, j) : 0.0;
                const unsigned mp = __ballot_sync(FULL, v && (o >= th));
                const unsigned mn_ = __ballot_sync(FULL, v && (-o >= th));
                commit_pair(type == 0 ? masks + M_T0 * NWORDS : nullptr, (unsigned long long)mp << 1,
                            (type == 1 || P.t0inv_same) ? masks + M_T0INV * NWORDS : nullptr, (unsigned long long)mn_ << 1,
                            false, 0, q, lane);
            } else if (type == 2) {
                const int j = q * CH + 1 + lane;
                if (j < P.e535.nout) {
                    const double o = trap_at_i(TT, P.e535, j);
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
                // the 33rd output of the chunk: evaluated by every lane (same value), no divergence
                const int j2 = q * CH + 32;
                const double s2 = (j2 < nsg) ? sg_at(0, j2) : -CUDART_INF;
                const unsigned long long bc = (unsigned long long)__ballot_sync(FULL, v && (sv >= cur_thr)) |
                                              ((s2 >= cur_thr) ? (1ull << 32) : 0ull);
                const unsigned long long bp = (unsigned long long)__ballot_sync(FULL, v && (sv >= pile_thr)) |
                                              ((s2 >= pile_thr) ? (1ull << 32) : 0ull);
                commit_pair(masks + M_CUR * NWORDS, bc, masks + M_PILE * NWORDS, bp, true, nsg, q, lane);
            }
        };
        // ---- coarse-to-fine trapezoids: lane i of warp w owns the interval (33q, 33q+33), q = 32w + i ----
        unsigned flags = 0;
        {
            bool f0 = false, fi = false, f5 = false, fe = false;
            if (G & LGDSP_GROUP_TIMING) {
                // Which intervals can hold part of a qualifying run (>= min_n consecutive samples above threshold)?
                //   min_n >= 2*33: such a run contains two CONSECUTIVE coarse points, and one of them is an end point of
                //                  every interval it overlaps -> need (a && b) || (a && prev) || (b && next);
                //   min_n  >  33 : it contains an end point of every interval it overlaps -> need a || b;
                //   otherwise every interval is evaluated.
                // (prev/next = coarse points q-1 / q+2; unknown across a warp boundary -> assumed above threshold)
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
                    f0 = P.t0inv_same ? (fp || fn) : fp;
                    if (pa) mask_commit(masks + M_T0 * NWORDS, tid, 1ull);
                    if (P.t0inv_same && na) mask_commit(masks + M_T0INV * NWORDS, tid, 1ull);
                }
                if (!P.t0inv_same) {
                    const bool wa = i0 < P.t0inv.nout, wb = i0 + CH < P.t0inv.nout;
                    const bool na = wa && (-cia >= th), nb = wb && (-cib >= th);
                    fi = need(na, nb, wa);
                    if (na) mask_commit(masks + M_T0INV * NWORDS, tid, 1ull);
                }
            }
            if (G & LGDSP_GROUP_TRAPS) {
                const double M5 = red_max(red, R_C535), Me = red_max(red, R_CET);
                const double k5 = Ymax * 2.0 * (P.e535.inv1 + P.e535.inv2) * 1.000001;
                const double ke = Ymax * 2.0 * (P.etrap.inv1 + P.etrap.inv2) * 1.000001;
                if (i0 + 1 < P.e535.nout) f5 = interval_bound(c5a, c5b, i0 + CH < P.e535.nout, k5) + kslack >= M5;
                if (i0 + 1 < P.etrap.nout) fe = interval_bound(cea, ceb, i0 + CH < P.etrap.nout, ke) + kslack >= Me;
            }
            flags = (f0 ? 1u : 0u) | (fi ? 2u : 0u) | (f5 ? 4u : 0u) | (fe ? 8u : 0u);
        }

        // ---- masks on the sg[0] trace (t50_current, in-trace pile-up on the REVERSED trace): only chunks whose
        //      maximum reaches the smaller threshold can contribute a bit ----
        if (G & LGDSP_GROUP_INTRACE) {
            const bool flag = sgcmax >= fmin(cur_thr, pile_thr);
            const unsigned bf = __ballot_sync(FULL, flag);
            if (__popc(bf) > 10) {
                // many flagged chunks in this warp (low threshold): every flagged lane redoes its own chunk
                if (flag) {
                    unsigned long long bc = 0, bp = 0;
                    sg_chunk(TT, P.sg[0], i0, min(CH, nsg - i0), [&](int k, double s) {
                        bc |= (s >= cur_thr) ? (1ull << k) : 0ull;
                        bp |= (s >= pile_thr) ? (1ull << k) : 0ull;
                    });
                    mask_commit(masks + M_CUR * NWORDS, tid, bc);
                    mask_commit_reversed(masks + M_PILE * NWORDS, tid, bp, nsg);
                }
            } else if (flag) {
                flags |= 16u;   // few: queued, a warp evaluates one chunk with one output per lane (identical values)
            }
        }
        // flagged intervals / chunks go to a block-wide work queue (processed by all warps after B4, so the pulse-region
        // warp does not evaluate all of them alone); what does not fit stays with the owning warp (ovf bits)
        unsigned ovf = 0;
#pragma unroll 1
        for (int type = 0; type < 5; ++type) {
            const bool flag = (flags >> type) & 1u;
            const unsigned b = __ballot_sync(FULL, flag);
            if (b == 0u) continue;
            int base = 0;
            if (lane == 0) base = atomicAdd(&ibuf[IB_QN], __popc(b));
            base = __shfl_sync(FULL, base, 0);
            const int idx = base + __popc(b & ((1u << lane) - 1u));
            if (flag) {
                if (idx < QCAP) qitems[idx] = (uint16_t)((type << 8) | tid);
                else ovf |= 1u << type;
            }
        }

        // ---- CUSP / ZAC ----
        double czmax[2] = {-CUDART_INF, -CUDART_INF};
        int czarg[2] = {0x7fffffff, 0x7fffffff};
        if (cz_on && P.direct) {
            // direct form (validation mode only)
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
                    const int r = j - pk_from[1 + f];
                    if (r >= 0 && r < P.sig_dni.n_w) stash[(1 + f) * LGDSP_MAX_DNI + r] = o;
                }
                if (f == 0) { czmax[0] = bm; czarg[0] = ba; } else { czmax[1] = bm; czarg[1] = ba; }
            }
        }
        // ---- scalar results, one self-contained job per warp.  Everything that does not need the CUSP/ZAC outputs runs
        //      while the candidate warps step their recurrences (scalar_jobs), the two CUSP/ZAC jobs after B6 ----
        // t10..t99 [us] (k = 0..4) and t0 / t0_inv [us] from the resolved positions; NaN -> 0
        auto tx_us = [&](int k) -> double {
            const double th = k == 0 ? thr[0] : k == 1 ? thr[1] : k == 2 ? thr[2] : k == 3 ? thr[3] : thr[4];
            return tx_us_at(TT, ibuf[IB_POS0 + M_T10 + k], th, t_first, dt);
        };
        auto t0_us = [&](bool inv, int pos) -> double { return t0_us_at(P, TT, inv, pos, t_first, dt); };
        auto qdrift_warp = [&](double t_us, double first, double last) -> double {
            return qdrift_at(P, TT, A_int, n, t_first, dt, t_us, first, last, lane);
        };
        auto scalar_jobs = [&]() {
        if (wid == 0) {
            // block-wide sums first (warp-collective), then lanes 0..2 finish one statistics block each (same code path):
            // lane 0 baseline [:102], lane 1 tailstats [:115, src/tailstats.jl:22-72], lane 2 PZ tail stats [:123]
            const double blS = red_sum(red, R_BLS), blSS = red_sum(red, R_BLSS), blSX = red_sum(red, R_BLSX);
            const double tlS = red_sum(red, R_TLS), tlSS = red_sum(red, R_TLSS), tlSX = red_sum(red, R_TLSX);
            const double tlbad = red_sum(red, R_TLBAD);
            const double pzS = red_sum(red, R_PZS), pzSS = red_sum(red, R_PZSS), pzSX = red_sum(red, R_PZSX);
            if (lane < 3) {
                const double sY = lane == 0 ? blS : lane == 1 ? tlS : pzS;
                const double sYY = lane == 0 ? blSS : lane == 1 ? tlSS : pzSS;
                const double sXY = lane == 0 ? t_first * blS + dt * blSX : lane == 1 ? tlSX : pzSX;
                const Stats st = stats_finalize(lane == 0 ? P.bl_inv_n : P.tail_inv_n, lane == 0 ? P.bl_sX : P.tail_sX,
                                                lane == 0 ? P.bl_sXX : P.tail_sXX, sY, sYY, sXY);
                if (lane == 0) {
                    row[LGDSP_COL_blmean] = st.mean; row[LGDSP_COL_blsigma] = st.sigma;
                    row[LGDSP_COL_blslope] = st.slope; row[LGDSP_COL_bloffset] = st.offset;
                    row[LGDSP_COL_qc_label] = -1.0;
                    row[LGDSP_COL_e_max] = e_max; row[LGDSP_COL_e_min] = e_min;
                    row[LGDSP_COL_n_sat_low] = (double)nlow; row[LGDSP_COL_n_sat_high] = (double)nhigh;
                    row[LGDSP_COL_n_sat_low_cons] = (double)cons_low; row[LGDSP_COL_n_sat_high_cons] = (double)cons_high;
                } else if (lane == 1) {
                    if (tlbad == 0.0) {
                        row[LGDSP_COL_tail_mean] = st.mean; row[LGDSP_COL_tail_sigma] = st.sigma;
                        row[LGDSP_COL_tail_tau] = div_rn(-1.0, st.slope);
                    }
                } else {
                    row[LGDSP_COL_tailmean] = st.mean; row[LGDSP_COL_tailsigma] = st.sigma;
                    row[LGDSP_COL_tailslope] = st.slope; row[LGDSP_COL_tailoffset] = st.offset;
                }
            }
        } else if (wid == 1) {
            // interpolated crossings: lanes 0..4 t10..t99, lane 5 t0, lane 6 t0_inv; then drift_time = t90 - t0
            // crossing resolution of the t0 / t0_inv masks (complete since B6) by this warp
            int pos0, pos0i, mult_;
            resolve_runs(masks + M_T0 * NWORDS, P.t0_min_n, lane, pos0, mult_);
            resolve_runs(masks + M_T0INV * NWORDS, P.t0_min_n, lane, pos0i, mult_);
            double t = 0.0;
            if (lane < 5) {
                t = tx_us(lane);
                if (G & LGDSP_GROUP_TIMING) row[LGDSP_COL_t10 + lane] = t;
            } else if (lane == 5 || lane == 6) {
                t = t0_us(lane == 6, lane == 6 ? pos0i : pos0);
                if (G & LGDSP_GROUP_TIMING) row[lane == 6 ? LGDSP_COL_t0_inv : LGDSP_COL_t0] = t;
            }
            const double t90 = __shfl_sync(FULL, t, 3), t0v = __shfl_sync(FULL, t, 5);
            if (lane == 0 && (G & LGDSP_GROUP_TIMING)) row[LGDSP_COL_drift_time] = (t90 - t0v) * 1000.0;
        } else if (wid == 2) {
            if (G & LGDSP_GROUP_TRAPS) {
                const double v = dni_eval_warp(A_sig, P.sig_dni.n_w, P.sig_dni.m, stash, pk_p[0] - (double)pk_from[0], lane);
                double em;
                int ea;
                red_argmax(red, R_ETMAX, R_ETARG, em, ea);
                const double a = red_max(red, R_E104), b = red_max(red, R_E535), c = red_max(red, R_E313);
                const double d = red_max(red, R_E104N), f = red_max(red, R_E313N);
                if (lane == 0) {
                    row[LGDSP_COL_e_10410] = a; row[LGDSP_COL_e_535] = b; row[LGDSP_COL_e_313] = c;
                    row[LGDSP_COL_e_10410_inv] = d; row[LGDSP_COL_e_313_inv] = f;
                    row[LGDSP_COL_e_trap_max] = em;
                    row[LGDSP_COL_t_trap_max] = t_first + (double)(ea + P.etrap.L - 1) * dt;
                    row[LGDSP_COL_e_trap] = v;
                }
            }
        } else if (wid == 5) {
            if (G & LGDSP_GROUP_CURRENT) {
                currents_job(TT, P.sg, spar->sgg, P.sg_alias, P.cur_from, P.cur_until, red, R_CMAX0, R_CARG0, row, lane);
            }
            if (G & LGDSP_GROUP_INTRACE) {
                // crossing resolution of the sg[0] masks (complete since Bq), then t50_current and the in-trace pile-up
                int posc, posp, multc, multp;
                resolve_runs(masks + M_CUR * NWORDS, P.tx_min_n, lane, posc, multc);
                resolve_runs(masks + M_PILE * NWORDS, P.intr_min_n, lane, posp, multp);
                if (lane >= 4 && lane < 6) {
                    const double tf = t_first + (double)P.sg[0].offset * dt;
                    if (lane == 4) {
                        // t50_current  src/dsp_icpc.jl:192-195
                        double t = 0.0;
                        if (posc >= 1) {
                            t = cross_x(cur_thr, sg_at(0, posc - 1), sg_at(0, posc), tf + (double)(posc - 1) * dt, dt) * 0.001;
                            if (t != t) t = 0.0;
                        }
                        row[LGDSP_COL_t50_current] = t;
                    } else {
                        // in-trace pile-up  src/dsp_routines.jl:72-82 (reversed trace r[j] = s[nsg-1-j], same time axis)
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
            }
        } else if (wid == 7) {
            if (G & LGDSP_GROUP_QDRIFT) {
                int pos0, mult_;
                resolve_runs(masks + M_T0 * NWORDS, P.t0_min_n, lane, pos0, mult_);
                const double v = qdrift_warp(t0_us(false, pos0), P.qd_first, P.qd_last);   // qdrift @ t0
                if (lane == 0) row[LGDSP_COL_qdrift] = v;
            }
        } else if (wid == 6) {
            if (G & LGDSP_GROUP_QDRIFT) {
                const double v = qdrift_warp(tx_us(2), P.lq_first, P.lq_last);       // lq @ t80
                if (lane == 0) row[LGDSP_COL_lq] = v;
            }
        }
        };
        // the queued intervals, spread over all warps; then the trapezoid partials of the block-wide maxima
        auto run_queue = [&]() {
            const int nq = min(ibuf[IB_QN], QCAP);
            int it = wid, otype = 0;
            unsigned ob = __ballot_sync(FULL, ovf & 1u);
#pragma unroll 1
            for (;;) {
                int type, q;
                if (it < nq) {
                    const int code = qitems[it];
                    it += NWARP;
                    type = code >> 8;
                    q = code & 255;
                } else {
                    while (ob == 0u && otype < 4) {
                        ++otype;
                        ob = __ballot_sync(FULL, (ovf >> otype) & 1u);
                    }
                    if (ob == 0u) break;
                    const int i = __ffs(ob) - 1;
                    ob &= ob - 1;
                    type = otype;
                    q = wid * 32 + i;
                }
                do_item(type, q);
            }
            e535 = wmax_d(e535);
            etmax = wargmax_d(etmax, etarg);
            if (lane == 0) {
                red[R_E535 * NWARP + wid] = e535;
                red[R_ETMAX * NWARP + wid] = etmax; red[R_ETARG * NWARP + wid] = (double)etarg;
            }
        };
        bool queue_done = false;
        // One pass of the structured CUSP/ZAC evaluation.  The descriptor index is a compile-time constant so that its
        // fields are immediate constant-bank operands inside the recurrences (a run-time index costs an indexed constant
        // load per use).  The LAST pass always uses descriptor 0 (CUSP, or both filters when they share their parameters)
        // and carries the work queue's scalar jobs; a separate ZAC descriptor (index 1) is evaluated in a pass before it.
        auto cz_pass = [&](auto psc, const bool czp, const bool want_cusp, const bool want_zac, const bool rescan,
                           const bool last_pass) {
            constexpr int ps = decltype(psc)::value;
            const CzDev& Z = P.cz[ps];
            if (rescan) {
                __syncthreads();   // the previous pass is done with the tables, the coarse values and the output buffer
                if (tid == 0) ibuf[IB_CZN] = 0;
                cz_scan<SM_PAR>(ps, TT, n, tid, tabA, tabB, red + R_CZSCR * NWARP, scr + SC_PP0);
                __syncthreads();
            }
            CzState st;
            st.active = false;
            double oc = -CUDART_INF, oz = -CUDART_INF;
            if (czp) {
                cz_init(Z, TT, n, tid, tabA, tabB, scr[SC_PP0], st);
                cz_coarse(Z, TT, n, tid, st, oc, oz);
                if (!want_cusp) oc = -CUDART_INF;
                if (!want_zac) oz = -CUDART_INF;
                // the coarse points are outputs themselves
                const int j0 = i0 - Z.L + 1;
                if (oc > czmax[0]) { czmax[0] = oc; czarg[0] = j0; }
                if (oz > czmax[1]) { czmax[1] = oz; czarg[1] = j0; }
                czco[tid] = oc;
                czco[NT + tid] = oz;
                const double wc = wmax_d(oc), wz = wmax_d(oz);
                red_put(red, R_CZC0, wid, lane, wc);
                red_put(red, R_CZC1, wid, lane, wz);
            }
            __syncthreads();   // ---- B4: tables are dead, coarse values and the work queue are complete ----
            if (czp && last_pass) prefetch_next();   // every thread has read its table entries: xs may be overwritten
            // candidate chunks: Lipschitz bound on (33 tid, 33 tid + 33) against the best coarse value; chunks that
            // hold part of a pick-off window are always evaluated
            double Mc = 0.0, Mz = 0.0;
            if (czp) { Mc = red_max(red, R_CZC0); Mz = red_max(red, R_CZC1); }
            const bool cand = czp && cz_candidate(Z, st, oc, oz, czco, tid, i0, Ymax, Mc, Mz, want_cusp, want_zac, pk_from, 1, 2,
                                                  P.sig_dni.n_w);
            // slot of every candidate chunk in the output buffer (rounds of CZCAP chunks)
            int slot = -1;
            {
                const unsigned bc = __ballot_sync(FULL, cand);
                int base = 0;
                if (lane == 0 && bc) base = atomicAdd(&ibuf[IB_CZN], __popc(bc));
                base = __shfl_sync(FULL, base, 0);
                if (cand) slot = base + __popc(bc & ((1u << lane) - 1u));
            }
            // the queued intervals, spread over all warps (before the long recurrences of the candidate warps)
            if (!queue_done) {
                run_queue();
                queue_done = true;
            }
            if (last_pass) __syncthreads();   // ---- Bq: masks and trapezoid partials are complete ----
            // rounds: recurrences of up to CZCAP candidate chunks write their outputs to SMEM, then the whole block
            // takes maxima / first argmaxima / pick-off windows from there
            double* czbuf = tabB;
#pragma unroll 1
            for (int r0 = 0;; r0 += CZCAP) {
                if (cand && slot >= r0 && slot < r0 + CZCAP) {
                    ibuf[IB_CZT + slot - r0] = tid;
                    cz_out(Z, TT, n, tid, st, czbuf + (size_t)(slot - r0) * (CH * 2));
                }
                if (last_pass && r0 == 0) scalar_jobs();   // overlaps the recurrences of the candidate warps
                __syncthreads();   // ---- B5 ----
                const int ncz = czp ? ibuf[IB_CZN] : 0;
                const int nslot = min(ncz - r0, CZCAP);
                const int nw = P.sig_dni.n_w;
#pragma unroll 1
                for (int i = tid; i < nslot * CH; i += NT) {
                    const int sl = i / CH, k = i - sl * CH;
                    const int j = ibuf[IB_CZT + sl] * CH + k - Z.L + 1;
                    const double o_c = czbuf[2 * i], o_z = czbuf[2 * i + 1];
                    if (want_cusp) {
                        if (o_c > czmax[0] || (o_c == czmax[0] && j < czarg[0])) { czmax[0] = o_c; czarg[0] = j; }
                        const int q = j - pk_from[1];
                        if (q >= 0 && q < nw && o_c > -CUDART_INF) stash[LGDSP_MAX_DNI + q] = o_c;
                    }
                    if (want_zac) {
                        if (o_z > czmax[1] || (o_z == czmax[1] && j < czarg[1])) { czmax[1] = o_z; czarg[1] = j; }
                        const int q = j - pk_from[2];
                        if (q >= 0 && q < nw && o_z > -CUDART_INF) stash[2 * LGDSP_MAX_DNI + q] = o_z;
                    }
                }
                if (r0 + CZCAP >= ncz) break;
                __syncthreads();   // the buffer is reused by the next round
            }
        };
        if (npass == 2) cz_pass(std::integral_constant<int, 1>{}, true, false, true, false, false);
        cz_pass(std::integral_constant<int, 0>{}, npass >= 1, npass >= 1, npass == 1, npass == 2, true);
        // CUSP/ZAC partials
        {
            czmax[0] = wargmax_d(czmax[0], czarg[0]);
            czmax[1] = wargmax_d(czmax[1], czarg[1]);
            if (lane == 0) {
                red[R_CZMAX0 * NWARP + wid] = czmax[0]; red[R_CZARG0 * NWARP + wid] = (double)czarg[0];
                red[R_CZMAX1 * NWARP + wid] = czmax[1]; red[R_CZARG1 * NWARP + wid] = (double)czarg[1];
            }
        }
        __syncthreads();   // ---- B6 ----

        if (wid == 3 || wid == 4) {
            if (cz_on) {
                const int f = wid - 3;
                const double v = dni_eval_warp(A_sig, P.sig_dni.n_w, P.sig_dni.m, stash + (1 + f) * LGDSP_MAX_DNI,
                                               pk_p[1 + f] - (double)pk_from[1 + f], lane);
                double cm;
                int ca;
                red_argmax(red, f ? R_CZMAX1 : R_CZMAX0, f ? R_CZARG1 : R_CZARG0, cm, ca);
                if (lane == 0) {
                    const int L = f ? P.zac_L : P.cusp_L;
                    row[f ? LGDSP_COL_e_zac_max : LGDSP_COL_e_cusp_max] = cm;
                    row[f ? LGDSP_COL_t_zac_max : LGDSP_COL_t_cusp_max] = t_first + (double)(ca + L - 1) * dt;
                    row[f ? LGDSP_COL_e_zac : LGDSP_COL_e_cusp] = v;
                }
            }
        }
        __syncthreads();   // ---- B8 ----
        if (tid < LGDSP_NCOL) rows[e * LGDSP_NCOL + tid] = wrapped ? CUDART_NAN : row[tid];
        // (the next iteration's first barrier orders the reuse of row/stash/masks/scr/red)
    }
}

// ==================================================================================================
// Trapezoid sweep kernel: dsp_trap_rt_optimization / dsp_trap_ft_optimization
// (/root/reference/src/dsp_filter_optimization.jl:102-133, 241-274).  The reference re-filters every waveform
// once per grid point and reads ONE interpolated sample of each filtered trace; here the waveform's prefix sums
// stay resident in SMEM and every (rt, ft) variant only evaluates the n_w trapezoid outputs of its
// PolynomialDNI window (4 look-ups each).  One warp per variant.
// ==================================================================================================
constexpr int RED_W = 24;
// block-wide sum / max of one double (two barriers); every thread gets the result
__device__ __forceinline__ double block_sum1(double v, double* red, int tid)
{
    const int lane = tid & 31, wid = tid >> 5;
    v = warp_sum(v);
    if (lane == 0) red[wid] = v;
    __syncthreads();
    double s = 0;
#pragma unroll
    for (int w = 0; w < NWARP; ++w) s += red[w];
    __syncthreads();
    return s;
}
__device__ __forceinline__ double block_max1(double v, double* red, int tid)
{
    const int lane = tid & 31, wid = tid >> 5;
    v = warp_max(v);
    if (lane == 0) red[wid] = v;
    __syncthreads();
    double s = red[0];
#pragma unroll
    for (int w = 1; w < NWARP; ++w) s = red[w] > s ? red[w] : s;
    __syncthreads();
    return s;
}
constexpr int SW_XS = 0;
constexpr int SW_TT = SW_XS + MAXN * 2;
constexpr int SW_MASK = SW_TT + TT_LEN * 8;
constexpr int SW_RED = SW_MASK + NWORDS * 4;
constexpr int SW_DNI = SW_RED + NWARP * RED_W * 8;
constexpr int SW_OUT = SW_DNI + LGDSP_MAX_DNI * 4 * 8;
constexpr int SW_MAXVAR = 1024;
constexpr int SW_IBUF = SW_OUT + SW_MAXVAR * 8;
constexpr int SW_DSCAN = SW_IBUF + 64 * 4;
constexpr int SW_BAR = SW_DSCAN + 8 * 8;
constexpr int SW_TOTAL = SW_BAR + 16;

// SAMPLE = uint16_t, or uint32_t for presummed waveforms (n <= 4096); bl_ext != NULL: event e is shifted by bl_ext[e] instead
// of its own bl_window mean (dsp_sg_optimization_compressed shifts the windowed waveform by the presummed baseline /
// presum_rate, /root/reference/src/dsp_filter_optimization.jl:477); the aux outputs keep the waveform's own statistics
template <typename SAMPLE>
__global__ void __launch_bounds__(NT, 2)
sweep_kernel(const __grid_constant__ SweepDev P, const SAMPLE* __restrict__ wf, long long n_events, long long ld,
             const double* __restrict__ bl_ext, void* __restrict__ out, double* __restrict__ aux)
{
    extern __shared__ __align__(128) unsigned char smem[];
    SAMPLE* xs = reinterpret_cast<SAMPLE*>(smem + SW_XS);
    double* TT = reinterpret_cast<double*>(smem + SW_TT);
    uint32_t* mask = reinterpret_cast<uint32_t*>(smem + SW_MASK);
    double* red = reinterpret_cast<double*>(smem + SW_RED);
    double* dniA = reinterpret_cast<double*>(smem + SW_DNI);
    double* obuf = reinterpret_cast<double*>(smem + SW_OUT);
    int* ibuf = reinterpret_cast<int*>(smem + SW_IBUF);
    double* dscan = reinterpret_cast<double*>(smem + SW_DSCAN);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + SW_BAR);

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n = P.n;
    const uint32_t wf_bytes = (uint32_t)n * (uint32_t)sizeof(SAMPLE);
    const double t_first = P.t_first, dt = P.dt;
    for (int i = tid; i < LGDSP_MAX_DNI * 4; i += NT) dniA[i] = P.dni_A[i];
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
    }
    if (tid < TT_LEN - 1 - n) TT[n + 1 + tid] = 0.0;
    __syncthreads();
    long long e = blockIdx.x;
    if (tid == 0 && e < n_events) {
        mbar_expect_tx(bar, wf_bytes);
        tma_load_1d(xs, wf + e * ld, wf_bytes, bar);
    }
    uint32_t phase = 0;
    const int i0 = tid * CH;
    const int cvalid = max(0, min(CH, n - i0));
    for (; e < n_events; e += gridDim.x) {
        mbar_wait(bar, phase);
        phase ^= 1;
        const SAMPLE* xp = xs + i0;
        uint32_t csum = 0, cq = 0, blS = 0, blSK = 0;
        {
            const int ka = P.bl_from - i0, kb = P.bl_until - i0;
            for (int k = 0; k < cvalid; ++k) {
                const uint32_t x = xp[k];
                csum += x;
                cq += csum;
                const bool in = (k >= ka && k <= kb);
                blS += in ? x : 0u;
                blSK += in ? x * (uint32_t)k : 0u;
            }
        }
        uint32_t incl = csum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += t;
        }
        uint32_t* ured = reinterpret_cast<uint32_t*>(ibuf + 32);
        if (lane == 31) ured[wid] = incl;
        mask[tid] = 0u;
        // 32-bit samples: the uint32 prefix sums are exact only while the waveform sums to < 2^32; beyond that the event's
        // outputs are NaN (the sum of the chunk sums is exact in double)
        bool wrapped = false;
        if (sizeof(SAMPLE) == 4) {
            unsigned long long c64 = 0;
            for (int k = 0; k < cvalid; ++k) c64 += (unsigned long long)xp[k];
            wrapped = block_sum1((double)c64, red, tid) > 4294967295.0;
        }
        const double blSd = block_sum1((double)blS, red, tid);
        // sum_i i*x over the baseline window (for blslope of the aux outputs; exact in double)
        const double blSXd = aux ? block_sum1((double)i0 * (double)blS + (double)blSK, red, tid) : 0.0;
        uint32_t woff = 0;
#pragma unroll
        for (int w = 0; w < NWARP; ++w) woff += (w < wid) ? ured[w] : 0u;
        const uint32_t P_excl = woff + incl - csum;
        const double v2 = (double)cvalid * (double)P_excl + (double)cq;
        double incl2 = v2;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            double t = __shfl_up_sync(FULL, incl2, o);
            if (lane >= o) incl2 += t;
        }
        if (lane == 31) dscan[wid] = incl2;
        __syncthreads();
        double woff2 = 0;
#pragma unroll
        for (int w = 0; w < NWARP; ++w) woff2 += (w < wid) ? dscan[w] : 0.0;
        const double PP_excl = woff2 + incl2 - v2;
        // blmean exactly as signalstats: mean_Y = sum_Y * inv_n
        const double m_own = mul_rn(blSd, P.bl_inv_n);
        const double m = bl_ext ? bl_ext[e] : m_own;
        double ymax = -CUDART_INF, ymin = CUDART_INF;   // of this thread's chunk
        {
            uint32_t Pr = P_excl;
            double PPr = PP_excl;
            const double km1 = P.km1;
            double ip1 = (double)i0;
            double tri = 0.5 * (double)i0 * ((double)i0 + 1.0);
            double* tp = TT + i0 + 1;
            auto body = [&](int k) {
                const uint32_t x = xp[k];
                Pr += x;
                const double Pd = u2d(Pr);
                PPr += Pd;
                ip1 += 1.0;
                tri += ip1;
                const double Sd = fma(-ip1, m, Pd);
                const double w = u2d(x) - m;
                const double y = fma(km1, Sd, w);
                const double SS = fma(-tri, m, PPr);
                tp[k] = fma(km1, SS, Sd);
                ymax = y > ymax ? y : ymax;
                ymin = y < ymin ? y : ymin;
            };
            {
                int k = 0;
#pragma unroll 1
                for (; k + 3 <= cvalid; k += 3) { body(k); body(k + 1); body(k + 2); }
#pragma unroll 1
                for (; k < cvalid; ++k) body(k);
            }
        }
        if (tid == 0) TT[0] = 0.0;
        const double cmax = ymax, cmin = ymin;
        ymax = block_max1(ymax, red, tid);
        if (tid == 0) {
            const long long en = e + gridDim.x;
            if (en < n_events) {
                fence_proxy_async();
                mbar_expect_tx(bar, wf_bytes);
                tma_load_1d(xs, wf + en * ld, wf_bytes, bar);
            }
        }
        // t50 on the PZ waveform at 0.5*maximum  (src/dsp_filter_optimization.jl:260)
        const double thr = ymax * 0.5;
        {
            // the chunk's own extrema decide most chunks: below the threshold everywhere (baseline) or above it everywhere
            // (flat top after the pole-zero correction).  y from the closed form and y = TT[k+1] - TT[k] differ by
            // rounding (< 3e-7: |TT| < 2^29, one ulp = 6e-8): chunks within that guard of the threshold are evaluated sample by sample.
            unsigned long long b = 0;
            const double guard = 1e-5 * fmax(1.0, fabs(thr));
            if (cvalid > 0 && cmax >= thr - guard) {
                if (cmin >= thr + guard) {
                    b = (1ull << cvalid) - 1ull;
                } else {
                    const double* p = TT + i0;
                    for (int k = 0; k < cvalid; ++k) b |= ((p[k + 1] - p[k]) >= thr) ? (1ull << k) : 0ull;
                }
            }
            mask_commit(mask, tid, b);
        }
        __syncthreads();
        if (wid == 0) {
            int pos, mult;
            resolve_runs(mask, P.tx_min_n, lane, pos, mult);
            if (lane == 0) ibuf[0] = pos;
        }
        __syncthreads();
        double t50_us = 0.0;
        {
            const int pos = ibuf[0];
            if (pos >= 1) {
                t50_us = cross_x(thr, y_at(TT, pos - 1), y_at(TT, pos), t_first + (double)(pos - 1) * dt, dt) * 0.001;
                if (t50_us != t50_us) t50_us = 0.0;
            }
        }
        if (aux && tid == 0) {
            const Stats st = stats_finalize(P.bl_inv_n, P.bl_sX, P.bl_sXX, blSd, 0.0, t_first * blSd + dt * blSXd);
            double* a = aux + e * 4;
            a[0] = m_own; a[1] = st.slope; a[2] = t50_us; a[3] = 0.0;
        }
        const int n_w = P.sig_dni.n_w, mdeg = P.sig_dni.m;
        // trapezoid variants: ONE THREAD per variant walks its pick-off window (4 look-ups in TT per output; the DNI
        // matrix row is a broadcast read) -- a 200-variant grid is one window per thread instead of 25 per warp
#pragma unroll 1
        for (int v = tid; v < P.nvar; v += NT) {
            if (P.vars[v].kind != 0) continue;
            const TrapDev t = P.vars[v].t;
            const double pick = P.vars[v].pick_ns;
            const int mode = P.vars[v].mode;
            const int nout = n - t.L + 1;
            const double tf = __fma_rn((double)(t.L - 1), dt, t_first);
            const double t_ns = mode ? __fma_rn(t50_us, 1000.0, pick) : pick;
            double pc;
            int from;
            dni_window(n_w, nout, (t_ns - tf) / dt, pc, from);
            const double* p0 = TT + from;
            const double* p1 = p0 + t.a;
            const double* p2 = p1 + t.g;
            const double* p3 = p0 + t.L;
            double c0 = 0, c1 = 0, c2 = 0, c3 = 0;
#pragma unroll 2
            for (int i = 0; i < n_w; ++i) {
                const double val = __fma_rn(p3[i] - p2[i], t.inv2, -__dmul_rn(p1[i] - p0[i], t.inv1));
                const double* a = dniA + i * mdeg;
                c0 = fma(a[0], val, c0);
                if (mdeg > 1) c1 = fma(a[1], val, c1);
                if (mdeg > 2) c2 = fma(a[2], val, c2);
                if (mdeg > 3) c3 = fma(a[3], val, c3);
            }
            const double u = pc - (double)from;
            obuf[v] = (nout >= n_w) ? fma(fma(fma(c3, u, c2), u, c1), u, c0) : CUDART_NAN;
        }
        // FIR and Savitzky-Golay variants: one warp per variant
#pragma unroll 1
        for (int v = wid; v < (P.n_other ? P.nvar : 0); v += NWARP) {
            if (P.vars[v].kind == 0) continue;
            const SweepVar sv = P.vars[v];
            if (sv.kind == 2) {
                // SavitzkyGolay derivative trace s[j] = sum_k g[k] TT[j+k] (taps folded on the prefix sums); first argmax
                // inside the window, parabola through its neighbours when strictly inside  (src/interpolation.jl:30-46)
                auto sgv = [&](int j) -> double {
                    double a0 = 0, a1 = 0;
                    for (int k = 0; k <= sv.L; k += 2) {
                        a0 = fma(__ldg(sv.g + k), TT[j + k], a0);
                        if (k + 1 <= sv.L) a1 = fma(__ldg(sv.g + k + 1), TT[j + k + 1], a1);
                    }
                    return a0 + a1;
                };
                double bm = -CUDART_INF;
                int ba = 0x7fffffff;
                for (int j = sv.win_from + lane; j <= sv.win_until; j += 32) {
                    const double s = sgv(j);
                    if (s > bm) { bm = s; ba = j; }
                }
                bm = wargmax_d(bm, ba);
                if (lane == 0) {
                    double val = bm;
                    if (ba > sv.win_from && ba < sv.win_until) val = extrema3(sgv(ba - 1), bm, sgv(ba + 1));
                    obuf[v] = val;
                }
                continue;
            }
            const int Lf = sv.L;
            const int nout = n - Lf + 1;
            const double tf = t_first + (double)(Lf - 1) * dt;
            const double t_ns = sv.mode ? t50_us * 1000.0 + sv.pick_ns : sv.pick_ns;
            double pc;
            int from;
            dni_window(n_w, nout, (t_ns - tf) / dt, pc, from);
            double c[LGDSP_MAX_DNI_DEG + 1] = {0, 0, 0, 0};
            for (int i = lane; i < n_w; i += 32) {
                const double val = fir_at(TT, sv.g, Lf, from + i);
#pragma unroll
                for (int j = 0; j <= LGDSP_MAX_DNI_DEG; ++j)
                    if (j < mdeg) c[j] = fma(dniA[i * mdeg + j], val, c[j]);
            }
#pragma unroll
            for (int j = 0; j <= LGDSP_MAX_DNI_DEG; ++j) c[j] = warp_sum(c[j]);
            if (lane == 0) {
                const double u = pc - (double)from;
                double r = c[mdeg - 1];
                for (int j = mdeg - 2; j >= 0; --j) r = r * u + c[j];
                obuf[v] = (nout >= n_w) ? r : CUDART_NAN;
            }
        }
        __syncthreads();
        if (P.out_f64) {
            double* o = reinterpret_cast<double*>(out);
            for (int v = tid; v < P.nvar; v += NT) o[e * (long long)P.nvar + v] = wrapped ? CUDART_NAN : obuf[v];
        } else {
            float* o = reinterpret_cast<float*>(out);
            for (int v = tid; v < P.nvar; v += NT) o[e * (long long)P.nvar + v] = wrapped ? CUDART_NAN_F : (float)obuf[v];
        }
        __syncthreads();
    }
}

cudaError_t sweep_configure(int* max_blocks_per_sm)
{
    cudaError_t err = cudaFuncSetAttribute(sweep_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, SW_TOTAL);
    if (err != cudaSuccess) return err;
    err = cudaFuncSetAttribute(sweep_kernel<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, SW_TOTAL);
    if (err != cudaSuccess) return err;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(max_blocks_per_sm, sweep_kernel<uint16_t>, NT, SW_TOTAL);
}

#include "lgdsp_sweep_warp.cuh"

int sweep_warp_max_window() { return SWW_MAX_STEPS * SWW_STEP; }

int sweep_launch(const SweepDev& P, const double* dni_A_host, const void* d_wf, int sample_bytes, long long n_events, long long ld,
                 const double* d_bl_ext, void* d_out, double* d_aux, int grid, int sm_count, cudaStream_t stream)
{
    // LGDSP_SWEEP_PATH=cta forces the one-CTA-per-waveform kernel (A/B tests)
    const char* env = getenv("LGDSP_SWEEP_PATH");
    if (P.warp_ok && sample_bytes == 2 && dni_A_host && !(env && strcmp(env, "cta") == 0)) {
        const int ctas_per_sm = sww_geometry(P.win_steps);
        if (ctas_per_sm > 0) {
            SweepDni D;
            memcpy(D.A, dni_A_host, sizeof(D.A));
            const long long cap = (long long)sm_count * ctas_per_sm;
            const int wgrid = (int)(n_events < cap ? n_events : cap);
            const size_t smem = (size_t)sww_warp_bytes(P.win_steps);
            sweep_warp_kernel<<<wgrid, 32, smem, stream>>>(P, D, static_cast<const uint16_t*>(d_wf), n_events, ld, d_bl_ext, d_out, d_aux);
            return 1;
        }
    }
    if (env && strcmp(env, "warp") == 0) return -1;   // the test suite demands the warp path
    if (sample_bytes == 4)
        sweep_kernel<uint32_t><<<grid, NT, SW_TOTAL, stream>>>(P, static_cast<const uint32_t*>(d_wf), n_events, ld, d_bl_ext, d_out, d_aux);
    else
        sweep_kernel<uint16_t><<<grid, NT, SW_TOTAL, stream>>>(P, static_cast<const uint16_t*>(d_wf), n_events, ld, d_bl_ext, d_out, d_aux);
    return 0;
}

void icpc_launch(const IcpcDev& P, const void* d_wf, int sample_bytes, long long n_events, long long ld, const double* d_bl_ext,
                 long long bl_stride, double bl_div,
                 double* d_rows, int grid, cudaStream_t stream)
{
    if (sample_bytes == 4)
        icpc_kernel<uint32_t><<<grid, NT, SM_TOTAL, stream>>>(P, static_cast<const uint32_t*>(d_wf), n_events, ld, d_bl_ext, bl_stride, bl_div, d_rows);
    else
        icpc_kernel<uint16_t><<<grid, NT, SM_TOTAL, stream>>>(P, static_cast<const uint16_t*>(d_wf), n_events, ld, d_bl_ext, bl_stride, bl_div, d_rows);
}

// ==================================================================================================
// signalstats on arbitrary windows of raw (optionally shifted) waveforms: the auxiliary baseline / pole-zero windows
// of dsp_icpc_compressed (/root/reference/src/dsp_icpc.jl:338-339, 365-366).  One warp per (event, window); the sums
// over the integer samples are exact (int64), the shift enters in closed form.
// out[(e * n_windows + w) * 5 + {0..4}] = mean, sigma, slope, offset, slope_residual_sigma
// ==================================================================================================
template <typename SAMPLE>
__global__ void window_stats_kernel(const SAMPLE* __restrict__ wf, long long n_events, long long ld, double t_first, double dt,
                                    const double* __restrict__ shift, long long shift_stride, unsigned shift_mask,
                                    const int* __restrict__ win /* [n_windows][2] */, int n_windows, double* __restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const long long item = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= n_events * n_windows) return;
    const long long e = item / n_windows;
    const int w = (int)(item - e * n_windows);
    const int from = win[2 * w], until = win[2 * w + 1];
    const SAMPLE* x = wf + e * ld;
    // integer part of the shift is taken out exactly (int64 sums of x - c0), the fractional rest in closed form
    const bool shifted = shift != nullptr && ((shift_mask >> w) & 1u);
    const double c = shifted ? shift[e * shift_stride] : 0.0;
    const long long c0 = shifted ? __double2ll_rn(c) : 0ll;
    // exact in int64: samples are < 2^20 after presumming (16-bit ADC x presum rate <= 16) and a window holds < 2^13
    // samples, so sum v < 2^33, sum v^2 < 2^53, sum k v < 2^46
    long long sY = 0, sYY = 0, sKY = 0;
    for (int i = from + lane; i <= until; i += 32) {
        const long long v = (long long)x[i] - c0;
        sY += v;
        sYY += v * v;
        sKY += v * (long long)(i - from);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sY += __shfl_xor_sync(FULL, sY, o);
        sYY += __shfl_xor_sync(FULL, sYY, o);
        sKY += __shfl_xor_sync(FULL, sKY, o);
    }
    if (lane == 0) {
        // statistics of y = v - d (d = c - c0, |d| <= 1/2): sum y = sY - n d, sum y^2 = sYY - 2 d sY + n d^2,
        // sum X y with X_i = t_first + i dt
        const double d = c - (double)c0;
        const double nn = (double)(until - from + 1);
        const double Sy = (double)sY - nn * d;
        const double Syy = (double)sYY - 2.0 * d * (double)sY + nn * d * d;
        const double Sk = 0.5 * nn * (nn - 1.0);                       // sum of (i - from)
        const double Skk = (nn - 1.0) * nn * (2.0 * nn - 1.0) / 6.0;   // sum of (i - from)^2
        const double Sky = (double)sKY - d * Sk;
        const double x0 = t_first + (double)from * dt;
        const double sX = nn * x0 + dt * Sk;
        const double sXX = nn * x0 * x0 + 2.0 * x0 * dt * Sk + dt * dt * Skk;
        const double sXY = x0 * Sy + dt * Sky;
        const double inv_n = 1.0 / nn;
        const Stats st = stats_finalize(inv_n, sX, sXX, Sy, Syy, sXY);
        // residual sigma of the straight-line fit (population): var_res = var_Y - slope * cov_XY, clamped at 0
        const double mX = sX * inv_n, mY = Sy * inv_n;
        const double var_Y = Syy * inv_n - mY * mY, cov = sXY * inv_n - mX * mY;
        const double var_r = fmax(var_Y - st.slope * cov, 0.0);
        double* o = out + item * 5;
        o[0] = st.mean; o[1] = st.sigma; o[2] = st.slope; o[3] = st.offset; o[4] = sqrt(var_r);
    }
}

void window_stats_launch(const void* d_wf, int sample_bytes, long long n_events, long long ld, double t_first, double dt,
                         const double* d_shift, long long shift_stride, unsigned shift_mask, const int* d_win, int n_windows,
                         double* d_out, cudaStream_t stream)
{
    const long long items = n_events * n_windows;
    const int wpb = 8;
    const unsigned grid = (unsigned)((items + wpb - 1) / wpb);
    if (grid == 0) return;
    if (sample_bytes == 4)
        window_stats_kernel<uint32_t><<<grid, wpb * 32, 0, stream>>>(static_cast<const uint32_t*>(d_wf), n_events, ld, t_first, dt,
                                                                      d_shift, shift_stride, shift_mask, d_win, n_windows, d_out);
    else
        window_stats_kernel<uint16_t><<<grid, wpb * 32, 0, stream>>>(static_cast<const uint16_t*>(d_wf), n_events, ld, t_first, dt,
                                                                      d_shift, shift_stride, shift_mask, d_win, n_windows, d_out);
}

#include "lgdsp_icpc_split.cuh"

// ---- split pipeline: host side ----
cudaError_t icpc_split_configure(int* bps3)
{
    cudaError_t err;
    if ((err = cudaFuncSetAttribute(icpc_prefix_kernel<uint16_t, 0u>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1_TOTAL)) != cudaSuccess) return err;
    if ((err = cudaFuncSetAttribute(icpc_prefix_kernel<uint32_t, 0u>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1_TOTAL)) != cudaSuccess) return err;
    if ((err = cudaFuncSetAttribute(icpc_prefix_kernel<uint16_t, LGDSP_GROUP_ALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1_TOTAL)) != cudaSuccess) return err;
    if ((err = cudaFuncSetAttribute(icpc_prefix_kernel<uint16_t, LGDSP_GROUP_PZTRAP_LEAN>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1_TOTAL)) != cudaSuccess) return err;
    if ((err = cudaFuncSetAttribute(icpc_extract_kernel<0u>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_TOTAL)) != cudaSuccess) return err;
    if ((err = cudaFuncSetAttribute(icpc_extract_kernel<LGDSP_GROUP_ALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_TOTAL)) != cudaSuccess) return err;
    if ((err = cudaFuncSetAttribute(icpc_extract_kernel<LGDSP_GROUP_PZTRAP_LEAN>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_TOTAL)) != cudaSuccess) return err;
    if ((err = cudaFuncSetAttribute(icpc_cuspzac_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, K3_TOTAL)) != cudaSuccess) return err;
    if ((err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps3[0], icpc_prefix_kernel<uint16_t, 0u>, NT, K1_TOTAL)) != cudaSuccess) return err;
    if ((err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps3[1], icpc_extract_kernel<0u>, NT2, K2_TOTAL)) != cudaSuccess) return err;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps3[2], icpc_cuspzac_kernel, NT, K3_TOTAL);
}
long long icpc_split_tt_doubles() { return TTG_LEN; }
long long icpc_split_aux_doubles() { return AUX_LEN; }
long long icpc_split_cz_doubles() { return CZG_LEN; }

// one event batch: prefix -> extract || CUSP/ZAC (select + finish) on `stream` (and `stream_cz`); the d_* scratch buffers hold
// n_events slots.  bps3: resident blocks per SM of {prefix, extract, CUSP/ZAC select}
void icpc_split_launch_batch(const IcpcDev& P, const void* d_wf, int sample_bytes, long long n_events, long long ld,
                             const double* d_bl_ext, long long bl_stride, double bl_div, double* d_rows, double* d_tt, double* d_aux,
                             double* d_cz, const int* bps3, int sm_count, cudaStream_t stream, cudaStream_t stream_cz,
                             cudaEvent_t ev_prefix, cudaEvent_t ev_cz, cudaEvent_t* marks)
{
    // marks != NULL (profiling): everything on `stream`, an event after every kernel (marks[0] in front of the first)
    if (marks) { stream_cz = nullptr; cudaEventRecord(marks[0], stream); }
    const bool cz = (P.groups & LGDSP_GROUP_CUSPZAC) != 0;
    auto grid = [&](int k) { const long long cap = (long long)sm_count * bps3[k]; return (int)(n_events < cap ? n_events : cap); };
    // (16-bit samples with the full chain or the lean configs[1] group run instantiations with a compile-time group mask)
#define LGDSP_PREFIX_ARGS P, static_cast<const uint16_t*>(d_wf), n_events, ld, d_bl_ext, bl_stride, bl_div, d_tt, d_aux, d_rows
    if (sample_bytes == 4)
        icpc_prefix_kernel<uint32_t, 0u><<<grid(0), NT, K1_TOTAL, stream>>>(P, static_cast<const uint32_t*>(d_wf), n_events, ld, d_bl_ext,
                                                                            bl_stride, bl_div, d_tt, d_aux, d_rows);
    else if (P.groups == LGDSP_GROUP_ALL)
        icpc_prefix_kernel<uint16_t, LGDSP_GROUP_ALL><<<grid(0), NT, K1_TOTAL, stream>>>(LGDSP_PREFIX_ARGS);
    else if (P.groups == LGDSP_GROUP_PZTRAP_LEAN)
        icpc_prefix_kernel<uint16_t, LGDSP_GROUP_PZTRAP_LEAN><<<grid(0), NT, K1_TOTAL, stream>>>(LGDSP_PREFIX_ARGS);
    else
        icpc_prefix_kernel<uint16_t, 0u><<<grid(0), NT, K1_TOTAL, stream>>>(LGDSP_PREFIX_ARGS);
#undef LGDSP_PREFIX_ARGS
    if (marks) cudaEventRecord(marks[1], stream);
    const int fin_grid = (int)((n_events * K4_NBLK + K4_WARPS - 1) / K4_WARPS);   // warps: one per event + K4_NBLK - 1 helpers
    auto launch_cz = [&](cudaStream_t st) {
        icpc_cuspzac_kernel<<<grid(2), NT, K3_TOTAL, st>>>(P, d_tt, d_aux, n_events, d_cz, d_rows);
        if (marks) cudaEventRecord(marks[3], st);
        if (!P.direct) icpc_cuspzac_finish_kernel<<<fin_grid, K4_WARPS * 32, 0, st>>>(P, d_tt, d_aux, d_cz, n_events, d_rows);
        if (marks) cudaEventRecord(marks[4], st);
    };
    // the two consumers only depend on the prefix kernel: with a second stream their tails overlap
    const bool par = cz && stream_cz != nullptr && stream_cz != stream;
    if (par) {
        cudaEventRecord(ev_prefix, stream);
        cudaStreamWaitEvent(stream_cz, ev_prefix, 0);
        launch_cz(stream_cz);
        cudaEventRecord(ev_cz, stream_cz);
    }
    if (P.groups == LGDSP_GROUP_ALL)
        icpc_extract_kernel<LGDSP_GROUP_ALL><<<grid(1), NT2, K2_TOTAL, stream>>>(P, d_tt, d_aux, n_events, cz ? 0 : 1, d_rows);
    else if (P.groups == LGDSP_GROUP_PZTRAP_LEAN)
        icpc_extract_kernel<LGDSP_GROUP_PZTRAP_LEAN><<<grid(1), NT2, K2_TOTAL, stream>>>(P, d_tt, d_aux, n_events, cz ? 0 : 1, d_rows);
    else
        icpc_extract_kernel<0u><<<grid(1), NT2, K2_TOTAL, stream>>>(P, d_tt, d_aux, n_events, cz ? 0 : 1, d_rows);
    if (marks) cudaEventRecord(marks[2], stream);
    if (cz && !par) launch_cz(stream);
    if (par) cudaStreamWaitEvent(stream, ev_cz, 0);   // the ring slot is reused behind both consumers
}

cudaError_t icpc_configure(int* max_blocks_per_sm)
{
    cudaError_t err = cudaFuncSetAttribute(icpc_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL);
    if (err != cudaSuccess) return err;
    err = cudaFuncSetAttribute(icpc_kernel<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL);
    if (err != cudaSuccess) return err;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(max_blocks_per_sm, icpc_kernel<uint16_t>, NT, SM_TOTAL);
}

}  // namespace lgdsp
