// SiPM / PMT trigger chain on sm_100a: dsp_sipm (/root/reference/src/dsp_sipm.jl:47-158) as ONE kernel, one CTA per
// waveform, every intermediate trace resident in shared memory, plus the in-tree primitives it is built from as block-wide
// device routines:
//   thresholdstats / thresholdstats_mad   /root/reference/src/thresholdstats.jl:19-41, 61-71
//   IntersectMaximum                      /root/reference/src/intersect_maximum.jl:24-119
// The same routines, together with saturation, extremestats, tailstats and get_wvf_maximum, serve wfstats_kernel: the
// per-waveform primitives on whole waveform arrays (lgdsp_wfstats_run).
//
// Medians (thresholdstats_mad needs two per call, the chain eight per waveform) are exact order statistics found by
// value-range refinement: a 2048-bin LINEAR histogram between the current minimum and maximum (bin index is a monotone
// function of the value, so ranks are preserved), descend into the bin that holds the wanted rank, and as soon as that
// bin holds <= 256 elements rank them by brute force.  Noise-like traces need one histogram pass; degenerate ones
// (constant, quantised) terminate through the min == max test.
//
// IntersectMaximum: one ballot pass turns the trace into a bit mask (y >= threshold), every thread owns consecutive mask
// words, finds the run starts in them, keeps the runs of >= min_n samples (the up-crossing state machine of :41-56 in closed
// form), and an exclusive block scan of the per-thread counts gives every trigger its position in the ordered output list.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <cstdint>
#include <type_traits>

#include "../../include/lgdsp_b200.h"
#include "lgdsp_kernels.h"

namespace lgdsp {
namespace {

constexpr int SNT = 256;           // threads per CTA
constexpr int SNW = SNT / 32;      // warps per CTA
constexpr unsigned FULLM = 0xffffffffu;
constexpr int NBIN = 2048;         // histogram bins of one refinement level
constexpr int BPT = NBIN / SNT;    // bins per thread in the rank search
constexpr int CANDCAP = 256;       // candidates ranked by brute force

struct Scratch {
    unsigned hist[NBIN];
    double cand[CANDCAP];
    double red[4][SNW];
    int ired[SNW + 1];
    int ibuf[8];
    double dbuf[8];
};

__device__ __forceinline__ double mulrn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double addrn(double a, double b) { return __dadd_rn(a, b); }
// X[i] = t0 + i*dt with separately rounded product and sum (a time axis is a range: first + i*step)
__device__ __forceinline__ double time_at(int i, double t0, double dt) { return __dadd_rn(t0, __dmul_rn((double)i, dt)); }

__device__ __forceinline__ double wsum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULLM, v, o);
    return v;
}
__device__ __forceinline__ double wmin(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULLM, v, o));
    return v;
}
__device__ __forceinline__ double wmax(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULLM, v, o));
    return v;
}

// block-wide sum / min / max of up to 4 values at once (fixed combination order: deterministic); two barriers
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], Scratch& S)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < K; ++q) {
        const double w = wsum(v[q]);
        if (lane == 0) S.red[q][wid] = w;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < K; ++q) {
        double r = 0.0;
#pragma unroll
        for (int w = 0; w < SNW; ++w) r += S.red[q][w];
        v[q] = r;
    }
    __syncthreads();
}
// (count, min, max) of a per-thread partial
__device__ __forceinline__ void block_cnt_min_max(long long& cnt, double& mn, double& mx, Scratch& S)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const double c = wsum((double)cnt), a = wmin(mn), b = wmax(mx);
    if (lane == 0) { S.red[0][wid] = c; S.red[1][wid] = a; S.red[2][wid] = b; }
    __syncthreads();
    double rc = 0.0, ra = CUDART_INF, rb = -CUDART_INF;
#pragma unroll
    for (int w = 0; w < SNW; ++w) { rc += S.red[0][w]; ra = fmin(ra, S.red[1][w]); rb = fmax(rb, S.red[2][w]); }
    __syncthreads();
    cnt = (long long)rc; mn = ra; mx = rb;
}
// exclusive block scan of one int per thread; returns the thread's offset, total in `total`; two barriers
__device__ __forceinline__ int block_exscan(int v, int& total, Scratch& S)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(FULLM, inc, o);
        if (lane >= o) inc += u;
    }
    if (lane == 31) S.ired[wid] = inc;
    __syncthreads();
    int base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < SNW; ++w) {
        const int c = S.ired[w];
        if (w < wid) base += c;
        tot += c;
    }
    __syncthreads();
    total = tot;
    return base + inc - v;
}

// ---------------------------------------------------------------------------------------------------
// exact order statistics.  The population is described by data, not by a functor, so that ONE copy of the selection code
// serves all eight medians of the chain (instruction-cache footprint): sample i has the raw value y = sgn * tr[i], takes
// part if mn <= y <= mx, and enters with the value y (mode 0) or |y - med| (mode 1).
// SH: the trace lives in shared memory (LDS) or in global memory (lgdsp_wfstats_run on traces longer than LGDSP_MAX_SAMPLES).
// ---------------------------------------------------------------------------------------------------
struct Sel {
    const double* tr;
    double sgn, mn, mx, med;
    int mode;
};
template <bool SH>
__device__ __forceinline__ bool sel_elem(const Sel& s, int i, double& v)
{
    double raw;
    if (SH) {
        const unsigned a = (unsigned)__cvta_generic_to_shared(s.tr + i);
        asm volatile("ld.shared.f64 %0, [%1];" : "=d"(raw) : "r"(a));
    } else {
        raw = s.tr[i];
    }
    const double y = raw * s.sgn;
    v = s.mode ? fabs(y - s.med) : y;
    return s.mn <= y && y <= s.mx;
}

// Statistics.median of the population (middle element, or x/2 + y/2 of the two middle ones).
// [lo, hi]: bounds of the population (every value lies inside; the tighter, the fewer refinement levels).
// m: size of the population if known, else -1 (taken from the first histogram).  binbuf (optional, n entries of shared
// memory): the histogram pass leaves every sample's bin there, so that the gather pass is a 16-bit compare per sample.
// Returns the median; m_out = size of the population (0: empty, the return value is 0).
template <bool SH>
__device__ __noinline__ double block_median(const Sel sel, int n, double lo, double hi, long long m, unsigned short* binbuf, Scratch& S,
                                            long long& m_out)
{
    const int tid = threadIdx.x;
    long long k = m >= 0 ? (m - 1) / 2 : 0;
    bool want2 = m >= 0 ? ((m & 1) == 0) : false;
    bool need_next = false;    // v2 is the smallest element above `above`
    double above = 0.0, v1 = 0.0, v2 = 0.0;
    for (;;) {
        if (lo == hi) {
            // every remaining candidate has the same value; count them (population size / second rank)
            long long c = 0;
            double dmn = 0, dmx = 0;
            for (int i = tid; i < n; i += SNT) {
                double v;
                if (sel_elem<SH>(sel, i, v) && v == lo) ++c;
            }
            block_cnt_min_max(c, dmn, dmx, S);
            if (m < 0) { m = c; k = (m - 1) / 2; want2 = (m & 1) == 0; }
            if (m == 0) { m_out = 0; return 0.0; }
            v1 = lo;
            if (!want2 || k + 1 < c) v2 = lo;
            else { need_next = true; above = lo; }
            break;
        }
        for (int b = tid; b < NBIN; b += SNT) S.hist[b] = 0u;
        __syncthreads();
        const double width = hi - lo;
        const double scale = (double)NBIN / width;
        const bool usediv = !(scale < 1e300);            // denormal width: scale overflows
        auto bin_of = [&](double v) -> int {
            const double r = usediv ? (v - lo) / width * (double)NBIN : (v - lo) * scale;
            const int b = (int)r;
            return b < NBIN - 1 ? b : NBIN - 1;
        };
        for (int i = tid; i < n; i += SNT) {
            double v;
            int b = 0xFFFF;
            if (sel_elem<SH>(sel, i, v) && v >= lo && v <= hi) { b = bin_of(v); atomicAdd(&S.hist[b], 1u); }
            if (binbuf) binbuf[i] = (unsigned short)b;
        }
        __syncthreads();
        // the bin that holds rank k
        unsigned local[BPT];
        int mine = 0;
#pragma unroll
        for (int q = 0; q < BPT; ++q) { local[q] = S.hist[tid * BPT + q]; mine += (int)local[q]; }
        int total;
        const int before = block_exscan(mine, total, S);
        if (m < 0) { m = total; k = (m - 1) / 2; want2 = (m & 1) == 0; }
        if (m == 0) { m_out = 0; return 0.0; }
        if ((long long)before <= k && k < (long long)before + mine) {
            int cum = before;
#pragma unroll
            for (int q = 0; q < BPT; ++q) {
                if (k >= cum && k < cum + (int)local[q]) { S.ibuf[0] = tid * BPT + q; S.ibuf[1] = cum; S.ibuf[2] = (int)local[q]; }
                cum += (int)local[q];
            }
        }
        if (tid == 0) S.ibuf[3] = 0;
        __syncthreads();
        const int bsel = S.ibuf[0], cum_before = S.ibuf[1], cnt_b = S.ibuf[2];
        k -= cum_before;
        auto in_bin = [&](int i, double& v) -> bool {
            if (binbuf) return binbuf[i] == (unsigned short)bsel && (sel_elem<SH>(sel, i, v), true);
            return sel_elem<SH>(sel, i, v) && v >= lo && v <= hi && bin_of(v) == bsel;
        };
        if (cnt_b <= CANDCAP) {
            // gather the bin and rank its elements (ties broken by slot: equal values get consecutive ranks)
            for (int i = tid; i < n; i += SNT) {
                double v;
                if (in_bin(i, v)) S.cand[atomicAdd(&S.ibuf[3], 1)] = v;
            }
            __syncthreads();
            if (tid < cnt_b) {
                const double c = S.cand[tid];
                int rank = 0;
                for (int j = 0; j < cnt_b; ++j) {
                    const double o = S.cand[j];
                    rank += (o < c || (o == c && j < tid)) ? 1 : 0;
                }
                if (rank == (int)k) S.dbuf[0] = c;
                if (rank == (int)k + 1) S.dbuf[1] = c;
                if (rank == cnt_b - 1) S.dbuf[2] = c;   // maximum of the bin
            }
            __syncthreads();
            v1 = S.dbuf[0];
            if (!want2) v2 = v1;
            else if (k + 1 < cnt_b) v2 = S.dbuf[1];
            else { need_next = true; above = S.dbuf[2]; }
            __syncthreads();
            break;
        }
        // too many: new range = actual minimum / maximum inside the bin
        long long c = 0;
        double mn = CUDART_INF, mx = -CUDART_INF;
        for (int i = tid; i < n; i += SNT) {
            double v;
            if (in_bin(i, v)) { mn = fmin(mn, v); mx = fmax(mx, v); ++c; }
        }
        block_cnt_min_max(c, mn, mx, S);
        lo = mn; hi = mx;
    }
    if (need_next) {
        long long c = 0;
        double mn = CUDART_INF, mx = 0;
        for (int i = tid; i < n; i += SNT) {
            double v;
            if (sel_elem<SH>(sel, i, v) && v > above) mn = fmin(mn, v);
        }
        block_cnt_min_max(c, mn, mx, S);
        v2 = mn;
    }
    m_out = m;
    return want2 ? v1 / 2 + v2 / 2 : v1;
}

// _thresholdstats_mad_impl  src/thresholdstats.jl:61-71 on the trace y_i = sgn * tr[i], i < n
template <bool SH>
__device__ __noinline__ double block_thresholdstats_mad(const double* tr, double sgn, int n, double mn, double mx, unsigned short* binbuf,
                                                        Scratch& S)
{
    Sel sel{tr, sgn, mn, mx, 0.0, 0};
    double lo = mn, hi = mx;
    long long m = -1;
    if (!(fabs(mn) < CUDART_INF && fabs(mx) < CUDART_INF)) {
        // open bounds: one pass for the size, minimum and maximum of the population
        m = 0;
        lo = CUDART_INF; hi = -CUDART_INF;
        for (int i = threadIdx.x; i < n; i += SNT) {
            double v;
            if (sel_elem<SH>(sel, i, v)) { ++m; lo = fmin(lo, v); hi = fmax(hi, v); }
        }
        block_cnt_min_max(m, lo, hi, S);
        if (m == 0) return 0.0;
    } else if (mn > mx) {
        return 0.0;
    }
    long long m1, m2;
    const double med = block_median<SH>(sel, n, lo, hi, m, binbuf, S, m1);
    if (m1 == 0) return 0.0;                                                                      // :63
    // the absolute deviations lie in [0, max(med - lo, hi - med)]: no min/max pass
    sel.med = med;
    sel.mode = 1;
    const double mad = block_median<SH>(sel, n, 0.0, fmax(med - lo, hi - med), m1, binbuf, S, m2);
    return 1.4826 * mad;                                                                          // :70
}

// _thresholdstats_impl  src/thresholdstats.jl:19-41
template <class Val>
__device__ double block_thresholdstats(Val val, int n, double mn, double mx, Scratch& S)
{
    double s[3] = {0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < n; i += SNT) {
        const double y = val(i);
        if (mn <= y && y <= mx) { s[0] += y; s[1] = fma(y, y, s[1]); s[2] += 1.0; }
    }
    block_sum<3>(s, S);
    const double inv_n = 1.0 / s[2];
    const double mean = s[0] * inv_n;
    const double var = s[1] * inv_n - mean * mean;
    return sqrt(var > 0.0 ? var : (var != var ? var : 0.0));
}

// ---------------------------------------------------------------------------------------------------
// IntersectMaximum  src/intersect_maximum.jl:24-119 on the trace val(i), i < n, X[i] = t0 + i*dt.
// out: [4][cap] = x, x_high, x_tot, max (global memory), zero-filled behind the last trigger.  Returns the multiplicity;
// *first_x (shared memory, optional) receives x of the first trigger.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ int next_zero(const unsigned* mask, int from)
{
    // first index >= from whose bit is 0 (the mask is followed by a zero word and bits >= n are 0)
    int w = from >> 5;
    unsigned inv = ~mask[w] & (FULLM << (from & 31));
    while (inv == 0u) inv = ~mask[++w];
    return (w << 5) + __ffs(inv) - 1;
}

template <class Val>
__device__ int block_intersect_maximum(Val val, int n, double t0, double dt, double thr, int min_n, int max_n, int cap, double* out,
                                       unsigned* mask, Scratch& S, double* first_x)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int nwords = (n + 31) >> 5;
    for (int w = wid; w <= nwords; w += SNW) {
        const int i = (w << 5) + lane;
        const unsigned m = __ballot_sync(FULLM, i < n && val(i) >= thr);
        if (lane == 0) mask[w] = m;                      // word nwords: all zero (terminator)
    }
    __syncthreads();
    const int wpt = (nwords + SNT - 1) / SNT;            // consecutive words per thread: the output order is the thread order
    const int w0 = tid * wpt, w1 = min(nwords, w0 + wpt);
    auto starts_of = [&](int w) -> unsigned {
        const unsigned m = mask[w];
        const unsigned prev = w > 0 ? (mask[w - 1] >> 31) : 1u;   // sample 0 never starts a trigger (cand_pos > firstindex, :53)
        return m & ~((m << 1) | prev);
    };
    int mine = 0;
    for (int w = w0; w < w1; ++w) {
        unsigned st = starts_of(w);
        while (st) {
            const int s = (w << 5) + __ffs(st) - 1;
            st &= st - 1;
            mine += (next_zero(mask, s) - s >= min_n) ? 1 : 0;    // y_high_counter reaches min_n (:50-51)
        }
    }
    int total;
    int slot = block_exscan(mine, total, S);
    for (int w = w0; w < w1 && slot < cap; ++w) {
        unsigned st = starts_of(w);
        while (st && slot < cap) {
            const int up = (w << 5) + __ffs(st) - 1;
            st &= st - 1;
            const int run_end = next_zero(mask, up);
            if (run_end - up < min_n) continue;
            const double x_l = time_at(up - 1, t0, dt), x_r = time_at(up, t0, dt);
            const double y_l = val(up - 1), y_r = val(up);
            const double x = (thr - y_l) * (x_r - x_l) / (y_r - y_l) + x_l;                            // :73
            const int from = max(up - 2, 0), until = min(up + max_n, n - 1);                            // :77-78
            int ind = from;
            double best = val(from);
            for (int i = from + 1; i <= until; ++i) {
                const double v = val(i);
                if (v > best) { best = v; ind = i; }
            }
            double mxv = best;
            if (ind > from && ind < until) {                                                          // :82-83
                const double y1 = val(ind - 1), y3 = val(ind + 1);
                const double a = y3 - 4.0 * best + 3.0 * y1;
                mxv = y1 - a * a / (8.0 * (y3 - 2.0 * best + y1));
            }
            double xh;
            if (run_end < n) {                                                                        // :90-104
                const double xl = time_at(run_end - 1, t0, dt), xr = time_at(run_end, t0, dt);
                const double yl = val(run_end - 1), yr = val(run_end);
                xh = (thr - yl) * (xr - xl) / (yr - yl) + xl;
            } else {
                xh = time_at(n - 1, t0, dt);                                                    // :107
            }
            out[slot] = x;
            out[cap + slot] = xh;
            out[2 * cap + slot] = xh - x;
            out[3 * cap + slot] = mxv;
            if (slot == 0 && first_x) *first_x = x;
            ++slot;
        }
    }
    for (int i = min(total, cap) + tid; i < cap; i += SNT) { out[i] = 0.0; out[cap + i] = 0.0; out[2 * cap + i] = 0.0; out[3 * cap + i] = 0.0; }
    __syncthreads();
    return total;
}

// inclusive cumulative sum dst[i] = sum_{j<=i} src(j), i < n: thread-contiguous chunks of `chs` samples + block scan
template <class Src>
__device__ void block_cumsum(Src src, double* dst, int n, int chs, Scratch& S)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int i0 = tid * chs, i1 = min(n, i0 + chs);
    double acc = 0.0;
    for (int i = i0; i < i1; ++i) { acc += src(i); dst[i] = acc; }
    double inc = acc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double u = __shfl_up_sync(FULLM, inc, o);
        if (lane >= o) inc += u;
    }
    if (lane == 31) S.red[0][wid] = inc;
    __syncthreads();
    double base = 0.0;
    for (int w = 0; w < wid; ++w) base += S.red[0][w];
    const double off = base + (inc - acc);
    for (int i = i0; i < i1; ++i) dst[i] += off;
    __syncthreads();
}

// signalstats [RDDSP] on src(i), i in [from, until], X_i = t0 + i*dt: mean, sigma, slope, offset
template <class Src>
__device__ void block_signalstats(Src src, int from, int until, double t0, double dt, Scratch& S, double out[4])
{
    double s[4] = {0.0, 0.0, 0.0, 0.0};   // sum Y, sum Y^2, sum X Y, (unused)
    double sx = 0.0, sxx = 0.0;
    for (int i = from + threadIdx.x; i <= until; i += SNT) {
        const double x = time_at(i, t0, dt), y = src(i);
        s[0] += y; s[1] = fma(y, y, s[1]); s[2] = fma(x, y, s[2]);
        sx += x; sxx = fma(x, x, sxx);
    }
    s[3] = sx;
    block_sum<4>(s, S);
    double t[1] = {sxx};
    block_sum<1>(t, S);
    const double inv_n = 1.0 / (double)(until - from + 1);
    const double mean_X = s[3] * inv_n, mean_Y = s[0] * inv_n;
    const double var_X = t[0] * inv_n - mean_X * mean_X;
    double var_Y = s[1] * inv_n - mean_Y * mean_Y;
    const double cov = s[2] * inv_n - mean_X * mean_Y;
    const double slope = cov / var_X;
    if (var_Y < 0) var_Y = 0;
    out[0] = mean_Y; out[1] = sqrt(var_Y); out[2] = slope; out[3] = mean_Y - slope * mean_X;
}

// extremestats  src/extremestats.jl:25-40 on src(i), i in [from, until]: min, max and the FIRST indices
template <class Src>
__device__ void block_extremestats(Src src, int from, int until, Scratch& S, double& vmin, int& imin, double& vmax, int& imax)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double mn = CUDART_INF, mx = -CUDART_INF;
    int an = 0x7fffffff, ax = 0x7fffffff;
    for (int i = from + threadIdx.x; i <= until; i += SNT) {
        const double v = src(i);
        if (v < mn) { mn = v; an = i; }
        if (v > mx) { mx = v; ax = i; }
    }
    const double wmn = wmin(mn), wmx = wmax(mx);
    an = __reduce_min_sync(FULLM, mn == wmn ? an : 0x7fffffff);
    ax = __reduce_min_sync(FULLM, mx == wmx ? ax : 0x7fffffff);
    if (lane == 0) { S.red[0][wid] = wmn; S.red[1][wid] = wmx; S.red[2][wid] = (double)an; S.red[3][wid] = (double)ax; }
    __syncthreads();
    vmin = S.red[0][0]; imin = (int)S.red[2][0]; vmax = S.red[1][0]; imax = (int)S.red[3][0];
    for (int w = 1; w < SNW; ++w) {
        const double a = S.red[0][w], b = S.red[1][w];
        const int ia = (int)S.red[2][w], ib = (int)S.red[3][w];
        if (a < vmin || (a == vmin && ia < imin)) { vmin = a; imin = ia; }
        if (b > vmax || (b == vmax && ib < imax)) { vmax = b; imax = ib; }
    }
    __syncthreads();
}

// Runs of a predicate over a range of samples: count, length of the leading / trailing run, longest run, whole range set.
// Ranges are joined in order (a then b), the empty range (full, all 0) is the identity.
struct Runs {
    int cnt, pre, suf, best, full;
};
__device__ __forceinline__ void runs_cat(Runs& a, const Runs& b)
{
    a.best = max(max(a.best, b.best), a.suf + b.pre);
    a.pre = a.full ? a.pre + b.pre : a.pre;
    a.suf = b.full ? a.suf + b.suf : b.suf;
    a.full &= b.full;
    a.cnt += b.cnt;
}
__device__ __forceinline__ void runs_step(Runs& r, bool on)
{
    r.cnt += on;
    if (on) { ++r.suf; return; }
    if (r.full) { r.pre = r.suf; r.full = 0; }
    r.best = max(r.best, r.suf);
    r.suf = 0;
}
__device__ __forceinline__ Runs runs_shfl_down(const Runs& r, int o)
{
    return Runs{__shfl_down_sync(FULLM, r.cnt, o), __shfl_down_sync(FULLM, r.pre, o), __shfl_down_sync(FULLM, r.suf, o),
                __shfl_down_sync(FULLM, r.best, o), __shfl_down_sync(FULLM, r.full, o)};
}

// _saturation_impl  src/saturation.jl:28-65 on src(i), i in [from, until]: the number of samples == low / == high and the
// longest runs of them (a sample equal to low ends a high run and vice versa; trailing runs count).  Every thread walks a
// contiguous chunk (odd length: conflict-free on a staged trace), the chunk summaries are joined in thread order.
// out: n_low, n_high, max_cons_low, max_cons_high (valid in thread 0)
template <class Src>
__device__ void block_saturation(Src src, int from, int until, double low, double high, Scratch& S, double out[4])
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int chs = ((until - from + SNT) / SNT) | 1;
    const int i0 = from + tid * chs, i1 = min(until + 1, i0 + chs);
    Runs rl{0, 0, 0, 0, 1}, rh{0, 0, 0, 0, 1};
    for (int i = i0; i < i1; ++i) {
        const double v = src(i);
        const bool is_low = v == low;
        runs_step(rl, is_low);
        runs_step(rh, !is_low && v == high);
    }
    if (rl.full) rl.pre = rl.suf;
    if (rh.full) rh.pre = rh.suf;
    rl.best = max(rl.best, rl.suf);
    rh.best = max(rh.best, rh.suf);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const Runs bl = runs_shfl_down(rl, o), bh = runs_shfl_down(rh, o);
        if ((lane & (2 * o - 1)) == 0) { runs_cat(rl, bl); runs_cat(rh, bh); }
    }
    Runs* wr = reinterpret_cast<Runs*>(S.hist);   // [2][SNW]
    if (lane == 0) { wr[wid] = rl; wr[SNW + wid] = rh; }
    __syncthreads();
    if (tid == 0) {
        Runs a = wr[0], b = wr[SNW];
        for (int w = 1; w < SNW; ++w) { runs_cat(a, wr[w]); runs_cat(b, wr[SNW + w]); }
        out[0] = a.cnt; out[1] = b.cnt; out[2] = a.best; out[3] = b.best;
    }
    __syncthreads();
}

// _tailstats_impl  src/tailstats.jl:22-72 on src(i), i in [from, until]: any sample <= 0 gives (0, 0, 0) (:27-33), else the
// straight-line fit of log(y) over the sample time; out: mean, sigma, tau = -1/slope (unguarded, as the reference)
template <class Src>
__device__ void block_tailstats(Src src, int from, int until, double t0, double dt, Scratch& S, double out[3])
{
    bool nonpos = false;
    for (int i = from + threadIdx.x; i <= until; i += SNT) nonpos |= src(i) <= 0.0;
    if (__syncthreads_or(nonpos)) { out[0] = 0.0; out[1] = 0.0; out[2] = 0.0; return; }
    double st[4];
    block_signalstats([&](int i) { return log(src(i)); }, from, until, t0, dt, S, st);
    out[0] = st[0]; out[1] = st[1]; out[2] = -1.0 / st[2];
}

// extrema3points  src/interpolation.jl:8-10, rounded operation by operation (no contraction): the oracle's result bit for bit
__device__ __forceinline__ double extrema3points_rn(double y1, double y2, double y3)
{
    const double a = __dadd_rn(__dsub_rn(y3, __dmul_rn(4.0, y2)), __dmul_rn(3.0, y1));
    const double d = __dmul_rn(8.0, __dadd_rn(__dsub_rn(y3, __dmul_rn(2.0, y2)), y1));
    return __dsub_rn(y1, __ddiv_rn(__dmul_rn(a, a), d));
}

// _get_wvf_maximum_impl  src/interpolation.jl:30-46 on src(i), i in [from, until]: the first maximum, refined by the parabola
// through its neighbours only when it lies strictly inside the WINDOW
template <class Src>
__device__ double block_wvf_maximum(Src src, int from, int until, Scratch& S)
{
    double vmin, vmax;
    int imin, imax;
    block_extremestats(src, from, until, S, vmin, imin, vmax, imax);
    if (imax > from && imax < until) return extrema3points_rn(src(imax - 1), vmax, src(imax + 1));
    return vmax;
}

// ==================================================================================================
// dsp_sipm  src/dsp_sipm.jl:47-158, one CTA per waveform
// ==================================================================================================
template <typename SAMPLE>
__global__ void __launch_bounds__(SNT, 2) sipm_kernel(const __grid_constant__ SipmDev P, const SAMPLE* __restrict__ wf, long long n_events,
                                                   long long ld, double* __restrict__ rows, double* __restrict__ trig)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Scratch& S = *reinterpret_cast<Scratch*>(smem_raw);
    const int n = P.n, npad = (n + 2 + 1) & ~1;
    double* bufA = reinterpret_cast<double*>(smem_raw + ((sizeof(Scratch) + 15) & ~size_t(15)));
    double* bufB = bufA + npad;
    unsigned* mask = reinterpret_cast<unsigned*>(bufB + npad);
    const int tid = threadIdx.x;
    const int n_sg = n - P.sg_taps + 1, n_tr = n_sg - P.tL + 1;
    const double t_sg = time_at(P.sg_off, P.t_first, P.dt), t_tr = time_at(P.tL - 1, t_sg, P.dt);
    const int cap = P.cap;
    const int chs = ((n + SNT - 1) / SNT) | 1;        // odd chunk length: conflict-free chunked access

    for (long long e = blockIdx.x; e < n_events; e += gridDim.x) {
        const SAMPLE* x = wf + e * ld;
        double* row = rows + e * LGDSP_SIPM_NCOL;
        double* tg = trig + (size_t)e * LGDSP_SIPM_NLIST * LGDSP_SIPM_NFIELD * cap;
        // :88 Float64 conversion
        for (int i = tid; i < n; i += SNT) bufB[i] = (double)x[i];
        __syncthreads();
        // :91, :94-95 extremestats on the waveform and on the t0_hpge_window slice
        {
            double vmin, vmax;
            int imin, imax;
            block_extremestats([&](int i) { return bufB[i]; }, 0, n - 1, S, vmin, imin, vmax, imax);
            if (tid == 0) {
                row[LGDSP_SIPM_e_min] = vmin; row[LGDSP_SIPM_e_max] = vmax;
                row[LGDSP_SIPM_t_min] = time_at(imin, P.t_first, P.dt) * 0.001;
                row[LGDSP_SIPM_t_max] = time_at(imax, P.t_first, P.dt) * 0.001;
            }
            block_extremestats([&](int i) { return bufB[i]; }, P.trunc_from, P.trunc_until, S, vmin, imin, vmax, imax);
            if (tid == 0) {
                row[LGDSP_SIPM_e_min_lar] = vmin; row[LGDSP_SIPM_e_max_lar] = vmax;
                row[LGDSP_SIPM_t_min_lar] = time_at(imin, P.t_first, P.dt) * 0.001;
                row[LGDSP_SIPM_t_max_lar] = time_at(imax, P.t_first, P.dt) * 0.001;
            }
        }
        // :99-100 Savitzky-Golay derivative, same operation order as a sequential correlation (bit-identical trace)
        for (int j = tid; j < n_sg; j += SNT) {
            double acc = 0.0;
            for (int k = 0; k < P.sg_taps; ++k) acc = addrn(acc, mulrn(P.sgh[k], bufB[j + k]));
            bufA[j] = acc;
        }
        __syncthreads();
        // :103-105
        const double thr = block_thresholdstats_mad<true>(bufA, 1.0, n_sg, P.sg_min_thr, P.sg_max_thr, reinterpret_cast<unsigned short*>(bufB), S);
        if (tid == 0) S.dbuf[4] = 0.0;
        __syncthreads();
        const int nt0 = block_intersect_maximum([&](int i) { return bufA[i]; }, n_sg, t_sg, P.dt, P.sg_nsigma * thr, P.sg_min_n, P.sg_max_n,
                                                cap, tg, mask, S, &S.dbuf[4]);
        // :108-109 integrate the derivative
        block_cumsum([&](int i) { return bufA[i]; }, bufB, n_sg, chs, S);
        // :112-115 statistics of the integrated waveform; minimum(inters.x; init = 0) is min(0, x...)
        {
            const double first_x = nt0 > 0 ? S.dbuf[4] : 0.0;
            const double m = fmin(0.0, first_x), d3 = 3.0 * P.dt;
            const double stop = (m < t_sg + d3) ? t_sg + d3 : m;
            int until = (int)rint((stop - t_sg) / P.dt);
            until = min(until, n_sg - 1);
            double st[4];
            block_signalstats([&](int i) { return bufB[i]; }, 0, until, t_sg, P.dt, S, st);
            if (tid == 0) { row[LGDSP_SIPM_blmean] = st[0]; row[LGDSP_SIPM_blsigma] = st[1]; row[LGDSP_SIPM_blslope] = st[2]; row[LGDSP_SIPM_bloffset] = st[3]; }
            block_signalstats([&](int i) { return bufB[i]; }, 0, n_sg - 1, t_sg, P.dt, S, st);
            if (tid == 0) { row[LGDSP_SIPM_wfmean] = st[0]; row[LGDSP_SIPM_wfsigma] = st[1]; row[LGDSP_SIPM_wfslope] = st[2]; row[LGDSP_SIPM_wfoffset] = st[3]; }
        }
        // :118-121 discharges: flipped integrated waveform
        auto flip = [&](int i) { return bufB[i] * -1.0; };
        const double thr_dc = block_thresholdstats_mad<true>(bufB, -1.0, n_sg, P.sg_min_dc, P.sg_max_dc, reinterpret_cast<unsigned short*>(bufA), S);
        const int nt1 = block_intersect_maximum(flip, n_sg, t_sg, P.dt, P.sg_nsigma_dc * thr_dc, P.sg_min_n, P.sg_max_n, cap,
                                                tg + (size_t)1 * LGDSP_SIPM_NFIELD * cap, mask, S, nullptr);
        // :138-139 (the SG pipeline's IntersectMaximum with the trap pipeline's discharge bounds)
        const double thr_dct = block_thresholdstats_mad<true>(bufB, -1.0, n_sg, P.trap_min_dc, P.trap_max_dc, reinterpret_cast<unsigned short*>(bufA), S);
        const int nt3 = block_intersect_maximum(flip, n_sg, t_sg, P.dt, P.trap_nsigma_dc * thr_dct, P.sg_min_n, P.sg_max_n, cap,
                                                tg + (size_t)3 * LGDSP_SIPM_NFIELD * cap, mask, S, nullptr);
        // :125-126 pole-zero: y[i] = x[i] + km1 * cumsum(x)[i]
        block_cumsum([&](int i) { return bufB[i]; }, bufA, n_sg, chs, S);
        for (int i = tid; i < n_sg; i += SNT) bufA[i] = fma(P.km1, bufA[i], bufB[i]);
        __syncthreads();
        // :129-130 trapezoid through the prefix sums of the pole-zero corrected trace: T[0] = 0, T[i+1] = sum_{j<=i} pz[j]
        if (tid == 0) bufB[0] = 0.0;
        block_cumsum([&](int i) { return bufA[i]; }, bufB + 1, n_sg, chs, S);
        for (int j = tid; j < n_tr; j += SNT) {
            const double s1 = bufB[j + P.ta] - bufB[j];
            const double s2 = bufB[j + P.tL] - bufB[j + P.ta + P.tg];
            bufA[j] = s2 * P.inv2 - s1 * P.inv1;
        }
        __syncthreads();
        // :133-135
        const double thr_tr = block_thresholdstats_mad<true>(bufA, 1.0, n_tr, P.trap_min_thr, P.trap_max_thr, reinterpret_cast<unsigned short*>(bufB), S);
        const int nt2 = block_intersect_maximum([&](int i) { return bufA[i]; }, n_tr, t_tr, P.dt, P.trap_nsigma * thr_tr, P.trap_min_n,
                                                P.trap_max_n, cap, tg + (size_t)2 * LGDSP_SIPM_NFIELD * cap, mask, S, nullptr);
        if (tid == 0) {
            row[LGDSP_SIPM_threshold] = thr; row[LGDSP_SIPM_threshold_DC] = thr_dc;
            row[LGDSP_SIPM_threshold_trap] = thr_tr; row[LGDSP_SIPM_threshold_DC_trap] = thr_dct;
            row[LGDSP_SIPM_n_trig] = (double)nt0; row[LGDSP_SIPM_n_trig_DC] = (double)nt1;
            row[LGDSP_SIPM_n_trig_trap] = (double)nt2; row[LGDSP_SIPM_n_trig_DC_trap] = (double)nt3;
        }
        __syncthreads();
    }
}

// ==================================================================================================
// The per-waveform primitives on a batch (lgdsp_wfstats_run): one CTA per waveform, persistent grid; every primitive selected
// in P.what runs on the same copy of the trace.  SH: the trace is staged once as doubles in shared memory (n <=
// LGDSP_MAX_SAMPLES); otherwise every primitive reads the samples from global memory, and thresholdstats_mad on non-double
// samples first converts the trace into the CTA's slice of `work`.
// Dynamic shared memory: Scratch | double trace[n, even] (SH) | uint16 bin of every sample (SH, MAD) | mask words (IM).
// ==================================================================================================
__host__ __device__ constexpr size_t up16(size_t v) { return (v + 15) & ~size_t(15); }

__host__ __device__ inline size_t wfstats_smem_bytes(int n, unsigned what, bool sh)
{
    size_t b = up16(sizeof(Scratch));
    if (sh) {
        b += up16((size_t)n * sizeof(double));
        if (what & LGDSP_WFSTAT_THRESHOLDSTATS_MAD) b += up16((size_t)n * sizeof(unsigned short));
    }
    if (what & LGDSP_WFSTAT_INTERSECT_MAXIMUM) b += (size_t)(((n + 31) >> 5) + 1) * sizeof(unsigned);
    return b;
}

template <typename SAMPLE, bool SH>
__global__ void __launch_bounds__(SNT) wfstats_kernel(const __grid_constant__ WfstatsDev P, const SAMPLE* __restrict__ wf,
                                                      const double* __restrict__ thr, long long n_events, long long ld,
                                                      double* __restrict__ rows, double* __restrict__ lists, double* __restrict__ work)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Scratch& S = *reinterpret_cast<Scratch*>(smem_raw);
    const int n = P.n, tid = threadIdx.x;
    const unsigned what = P.what;
    unsigned char* p = smem_raw + up16(sizeof(Scratch));
    double* buf = reinterpret_cast<double*>(p);
    unsigned short* binbuf = nullptr;
    if (SH) {
        p += up16((size_t)n * sizeof(double));
        if (what & LGDSP_WFSTAT_THRESHOLDSTATS_MAD) { binbuf = reinterpret_cast<unsigned short*>(p); p += up16((size_t)n * sizeof(unsigned short)); }
    }
    unsigned* mask = reinterpret_cast<unsigned*>(p);

    for (long long e = blockIdx.x; e < n_events; e += gridDim.x) {
        const SAMPLE* x = wf + e * ld;
        double* row = rows + e * LGDSP_WFSTAT_NCOL;
        if (SH) {
            for (int i = tid; i < n; i += SNT) buf[i] = (double)x[i];
            __syncthreads();
        }
        auto val = [&](int i) -> double { return SH ? buf[i] : (double)x[i]; };
        if (what & LGDSP_WFSTAT_SATURATION) {
            double o[4];
            block_saturation(val, P.sat_from, P.sat_until, (double)P.sat_low, (double)P.sat_high, S, o);
            if (tid == 0) {
                row[LGDSP_WFSTAT_sat_low] = o[0]; row[LGDSP_WFSTAT_sat_high] = o[1];
                row[LGDSP_WFSTAT_sat_max_cons_low] = o[2]; row[LGDSP_WFSTAT_sat_max_cons_high] = o[3];
            }
        } else if (tid == 0) {
            row[LGDSP_WFSTAT_sat_low] = 0.0; row[LGDSP_WFSTAT_sat_high] = 0.0;
            row[LGDSP_WFSTAT_sat_max_cons_low] = 0.0; row[LGDSP_WFSTAT_sat_max_cons_high] = 0.0;
        }
        if (what & LGDSP_WFSTAT_EXTREMESTATS) {
            double vmin, vmax;
            int imin, imax;
            block_extremestats(val, P.ext_from, P.ext_until, S, vmin, imin, vmax, imax);
            if (tid == 0) {
                row[LGDSP_WFSTAT_min] = vmin; row[LGDSP_WFSTAT_max] = vmax;
                row[LGDSP_WFSTAT_tmin] = time_at(imin, P.t0, P.dt); row[LGDSP_WFSTAT_tmax] = time_at(imax, P.t0, P.dt);
            }
        } else if (tid == 0) {
            row[LGDSP_WFSTAT_min] = 0.0; row[LGDSP_WFSTAT_max] = 0.0; row[LGDSP_WFSTAT_tmin] = 0.0; row[LGDSP_WFSTAT_tmax] = 0.0;
        }
        {
            double o[3] = {0.0, 0.0, 0.0};
            if (what & LGDSP_WFSTAT_TAILSTATS) block_tailstats(val, P.tail_from, P.tail_until, P.t0, P.dt, S, o);
            if (tid == 0) { row[LGDSP_WFSTAT_tail_mean] = o[0]; row[LGDSP_WFSTAT_tail_sigma] = o[1]; row[LGDSP_WFSTAT_tail_tau] = o[2]; }
        }
        {
            const double m = (what & LGDSP_WFSTAT_WVF_MAXIMUM) ? block_wvf_maximum(val, P.max_from, P.max_until, S) : 0.0;
            if (tid == 0) row[LGDSP_WFSTAT_wvf_max] = m;
        }
        {
            const double s = (what & LGDSP_WFSTAT_THRESHOLDSTATS) ? block_thresholdstats(val, n, P.thr_min, P.thr_max, S) : 0.0;
            if (tid == 0) row[LGDSP_WFSTAT_thr_sigma] = s;
        }
        {
            double mad = 0.0;
            if (what & LGDSP_WFSTAT_THRESHOLDSTATS_MAD) {
                if (SH) {
                    mad = block_thresholdstats_mad<true>(buf, 1.0, n, P.thr_min, P.thr_max, binbuf, S);
                } else if constexpr (std::is_same<SAMPLE, double>::value) {
                    mad = block_thresholdstats_mad<false>(x, 1.0, n, P.thr_min, P.thr_max, nullptr, S);
                } else {
                    double* w = work + (size_t)blockIdx.x * n;
                    for (int i = tid; i < n; i += SNT) w[i] = (double)x[i];
                    __syncthreads();
                    mad = block_thresholdstats_mad<false>(w, 1.0, n, P.thr_min, P.thr_max, nullptr, S);
                }
            }
            if (tid == 0) row[LGDSP_WFSTAT_thr_mad] = mad;
        }
        {
            int mult = 0;
            if (what & LGDSP_WFSTAT_INTERSECT_MAXIMUM)
                mult = block_intersect_maximum(val, n, P.t0, P.dt, thr[e], P.im_min_n, P.im_max_n, P.cap,
                                               lists + (size_t)e * 4 * P.cap, mask, S, nullptr);
            if (tid == 0) row[LGDSP_WFSTAT_multiplicity] = (double)mult;
        }
        __syncthreads();
    }
}

template <typename SAMPLE, bool SH>
cudaError_t wfstats_configure_one(size_t bytes, int* bps)
{
    cudaError_t err = cudaFuncSetAttribute(wfstats_kernel<SAMPLE, SH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (err != cudaSuccess) return err;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(bps, wfstats_kernel<SAMPLE, SH>, SNT, bytes);
}

template <typename SAMPLE>
cudaError_t wfstats_configure_kind(const WfstatsDev& P, int* bps)
{
    const bool sh = P.n <= LGDSP_MAX_SAMPLES;
    const size_t bytes = wfstats_smem_bytes(P.n, P.what, sh);
    return sh ? wfstats_configure_one<SAMPLE, true>(bytes, bps) : wfstats_configure_one<SAMPLE, false>(bytes, bps);
}

template <typename SAMPLE>
void wfstats_launch_kind(const WfstatsDev& P, const void* d_wf, const double* d_thr, long long n_events, long long ld, double* d_rows,
                         double* d_lists, double* d_work, int grid, cudaStream_t stream)
{
    const bool sh = P.n <= LGDSP_MAX_SAMPLES;
    const size_t bytes = wfstats_smem_bytes(P.n, P.what, sh);
    const SAMPLE* wf = static_cast<const SAMPLE*>(d_wf);
    if (sh)
        wfstats_kernel<SAMPLE, true><<<grid, SNT, bytes, stream>>>(P, wf, d_thr, n_events, ld, d_rows, d_lists, d_work);
    else
        wfstats_kernel<SAMPLE, false><<<grid, SNT, bytes, stream>>>(P, wf, d_thr, n_events, ld, d_rows, d_lists, d_work);
}

// ==================================================================================================
// MultiIntersect  src/multi_intersect.jl:36-104, one WARP per trace (global memory, coalesced 32-sample steps).
// The sequential search (:59-73) advances 32 samples per ballot; blocks without a sample above the current threshold are
// skipped in one step, the others are walked bit by bit in registers (same state machine, no memory traffic).
// ==================================================================================================
constexpr int MI_WARPS = 8;
#ifndef MI_MAXU
#define MI_MAXU 8
#endif
constexpr int MI_SB = 8;      // 32-sample blocks per fetch while looking for the first crossing

// The state machine of :59-73 on one block of `steps` <= 32 samples, bit-parallel: bit l of m <=> sample i+l is high (bits
// beyond `steps` are clear).  counter = length of the run of high samples that ends just before the block (a value above
// k marks a run that may not fire any more, :56), cand = its first sample.  Returns true when a run reaches exactly k
// samples inside the block (cand = its start); otherwise counter / cand describe the run that touches the block end.
__device__ __forceinline__ bool mi_block(unsigned m, int steps, int i, int k, int& counter, int& cand)
{
    unsigned rest = m;
    if (counter > 0) {
        const int t = (m == 0xffffffffu) ? 32 : __ffs(~m) - 1;     // high samples at the start of the block (<= steps)
        if (counter < k && counter + t >= k) return true;           // the carried run fires here
        if (t == steps) { counter += t; return false; }             // the whole block is high
        counter = 0;                                                // the carried run ends at bit t
        rest = (t >= 31) ? 0u : (m >> (t + 1)) << (t + 1);
    }
    if (rest == 0u) { counter = 0; return false; }
    unsigned r = (k > 32) ? 0u : rest;                              // bit p <=> bits p .. p+k-1 of rest are all set
    for (int have = 1; have < k && r != 0u;) {
        const int sh = min(have, k - have);
        r &= r >> sh;
        have += sh;
    }
    if (r != 0u) {
        cand = i + __ffs(r) - 1;
        counter = k;
        return true;
    }
    const unsigned top = rest << (32 - steps);
    const int tl = (top == 0xffffffffu) ? 32 : __clz(~top);          // high samples at the end of the block
    counter = tl;
    if (tl > 0) cand = i + steps - tl;
    return false;
}

__global__ void __launch_bounds__(MI_WARPS * 32) multi_intersect_kernel(const __grid_constant__ MiDev P, const double* __restrict__ y,
                                                                        long long n_events, long long ld, double* __restrict__ x_out,
                                                                        int* __restrict__ flags)
{
    __shared__ int pos_s[MI_WARPS][LGDSP_MI_MAX_THR];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int len = P.len, n_thr = P.n_thr, min_n = P.min_n;
    int* pos = pos_s[wid];
    for (long long e = (long long)blockIdx.x * MI_WARPS + wid; e < n_events; e += (long long)gridDim.x * MI_WARPS) {
        const double* Y = y + e * ld;
        // maximum(Y) :31 -- MI_MAXU independent loads per lane in flight (the pass is latency bound otherwise)
        double ymax = -CUDART_INF;
        {
            double m0 = -CUDART_INF, m1 = -CUDART_INF, m2 = -CUDART_INF, m3 = -CUDART_INF;
            // from the END of the trace towards its start: the crossing search below begins at sample 0, so the part it
            // re-reads is the part that was fetched last (L2 / L1 hits instead of a second trip to HBM)
            const int nfull = len / (MI_MAXU * 32);
            for (int i = nfull * MI_MAXU * 32 + lane; i < len; i += 32) m0 = fmax(m0, Y[i]);
            for (int g = nfull - 1; g >= 0; --g) {
                const double* q = Y + g * (MI_MAXU * 32) + lane;
                double a[MI_MAXU];
#pragma unroll
                for (int u = 0; u < MI_MAXU; ++u) a[u] = q[(MI_MAXU - 1 - u) * 32];
#pragma unroll
                for (int u = 0; u < MI_MAXU; u += 4) {
                    m0 = fmax(m0, a[u]); m1 = fmax(m1, a[u + 1]); m2 = fmax(m2, a[u + 2]); m3 = fmax(m3, a[u + 3]);
                }
            }
            ymax = fmax(fmax(m0, m1), fmax(m2, m3));
        }
        ymax = wmax(ymax);
        for (int j = lane; j < n_thr; j += 32) pos[j] = 1;                            // :55
        __syncwarp();
        int cand = 1, ic = 0, i = 0;
        int counter = (Y[0] >= P.ratios[0] * ymax) ? min_n + 1 : 0;                   // :56
        while (i < len && ic < n_thr) {                                               // :59-73
            if (ic == 0 && i + MI_SB * 32 <= len) {
                // the search for the FIRST crossing runs through the whole baseline: fetch MI_SB blocks with independent
                // loads and examine them in order (one block per step would pay the memory latency for every block)
                const double thr0 = P.ratios[0] * ymax;
                double v[MI_SB];
#pragma unroll
                for (int u = 0; u < MI_SB; ++u) v[u] = Y[i + u * 32 + lane];
#pragma unroll
                for (int u = 0; u < MI_SB; ++u) {
                    if (ic != 0) continue;
                    const unsigned m = __ballot_sync(FULLM, v[u] >= thr0);
                    if (mi_block(m, 32, i, min_n, counter, cand)) {
                        if (lane == 0) pos[0] = cand;
                        i = cand;
                        ic = 1;
                        counter = 0;
                    } else {
                        i += 32;
                    }
                }
                continue;
            }
            const double thr = P.ratios[ic] * ymax;
            const int idx = i + lane;
            const unsigned m = __ballot_sync(FULLM, idx < len && Y[idx] >= thr);
            const int steps = min(32, len - i);
            if (mi_block(m, steps, i, min_n, counter, cand)) {
                if (lane == 0) pos[ic] = cand;
                i = cand;                                                             // :69 restart at the crossing
                ++ic;
                counter = 0;
            } else {
                i += steps;
            }
        }
        __syncwarp();
        // :76-79 boundary assertion on the first and the last crossing
        const int n = P.n;
        const bool bad = !(pos[0] - n >= 0) || !(pos[n_thr - 1] + n - 1 <= len - 1);
        if (lane == 0) flags[e] = bad ? 1 : 0;
        const int nw = 2 * n, m_up = 2 * n * P.rate, md = P.degree + 1;
        for (int j = lane; j < n_thr; j += 32) {
            double res = CUDART_NAN;
            const int from = pos[j] - n, to = pos[j] + n - 1;
            if (!bad && from >= 0 && to <= len - 1) {
                const double thr = P.ratios[j] * ymax;
                double c[LGDSP_MAX_DNI_DEG + 1];
#pragma unroll
                for (int q = 0; q <= LGDSP_MAX_DNI_DEG; ++q) {
                    double a = 0.0;
                    if (q < md)
                        for (int r = 0; r < nw; ++r) a = fma(P.A[r * md + q], Y[from + r], a);   // :113-116
                    c[q] = a;
                }
                const double xa = time_at(from, P.t0, P.dt), xb = time_at(to, P.t0, P.dt);
                const double st = (xb - xa) / (double)(m_up - 1);
                // _find_intersect_impl(axis, y_up, thr, 1): first k with y_up[k] >= thr after a sample below it
                double prev = 0.0;
                bool armed = false;
                for (int k = 0; k < m_up; ++k) {
                    const double xu = (double)(2 * n - 1) * (double)k / (double)(m_up - 1);        // range(0, 2n-1, m) :83
                    double v = 0.0, pw = 1.0;
#pragma unroll
                    for (int q = 0; q <= LGDSP_MAX_DNI_DEG; ++q) {
                        if (q < md) { v = fma(c[q], pw, v); pw *= xu; }                           // :117-119
                    }
                    const bool high = v >= thr;
                    if (high && armed) {
                        const double tl = time_at(k - 1, xa, st), tr = time_at(k, xa, st);
                        res = (thr - prev) * (tr - tl) / (v - prev) + tl;
                        break;
                    }
                    armed = !high;
                    prev = v;
                }
            }
            x_out[e * n_thr + j] = res;
        }
        __syncwarp();
    }
}

// ==================================================================================================
// trigger lists -> VectorOfVectors form on the device (flat data + element pointers, the reference's
// VectorOfVectors(inters.x) etc., src/dsp_sipm.jl:150-157).  Step 1: one block scans the per-event counts of one list
// (min(count, cap)) into elem_ptr[n_events + 1] with a running carry over tiles of 1024 events; step 2: one warp per
// event copies its entries of the four fields to flat[field][elem_ptr[e] + k].
// ==================================================================================================
__global__ void __launch_bounds__(1024) sipm_count_scan_kernel(const double* __restrict__ rows, long long n_events, int list, int cap,
                                                               long long* __restrict__ elem_ptr)
{
    __shared__ long long wsum[32];
    __shared__ long long carry_s;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (long long base = 0; base < n_events; base += 1024) {
        const long long e = base + tid;
        long long c = 0;
        if (e < n_events) {
            const double cnt = rows[e * LGDSP_SIPM_NCOL + LGDSP_SIPM_n_trig + list];
            c = (long long)(cnt < (double)cap ? cnt : (double)cap);
        }
        long long inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long u = __shfl_up_sync(FULLM, inc, o);
            if (lane >= o) inc += u;
        }
        if (lane == 31) wsum[wid] = inc;
        __syncthreads();
        long long before = carry_s;
        for (int w = 0; w < wid; ++w) before += wsum[w];
        if (e < n_events) elem_ptr[e] = before + inc - c;
        __syncthreads();
        if (tid == 1023) carry_s = before + inc;
        __syncthreads();
    }
    if (tid == 0) elem_ptr[n_events] = carry_s;
}

__global__ void sipm_compact_kernel(const double* __restrict__ trig, long long n_events, int list, int cap,
                                    const long long* __restrict__ elem_ptr, double* __restrict__ flat, long long flat_stride)
{
    const int lane = threadIdx.x & 31;
    const long long e = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (e >= n_events) return;
    const long long p0 = elem_ptr[e];
    const int cnt = (int)(elem_ptr[e + 1] - p0);
    const double* src = trig + ((size_t)e * LGDSP_SIPM_NLIST + list) * LGDSP_SIPM_NFIELD * cap;
    for (int f = 0; f < LGDSP_SIPM_NFIELD; ++f)
        for (int k = lane; k < cnt; k += 32) flat[(size_t)f * flat_stride + p0 + k] = src[(size_t)f * cap + k];
}

size_t sipm_smem_bytes(int n)
{
    const int npad = (n + 2 + 1) & ~1;
    const int nwords = ((n + 31) >> 5) + 1;
    return ((sizeof(Scratch) + 15) & ~size_t(15)) + (size_t)2 * npad * sizeof(double) + (size_t)nwords * sizeof(unsigned) + 16;
}

}  // namespace

cudaError_t sipm_configure(int n, int sample_kind, int* max_blocks_per_sm)
{
    const size_t bytes = sipm_smem_bytes(n);
    cudaError_t err;
    if (sample_kind == LGDSP_SAMPLE_F32) {
        err = cudaFuncSetAttribute(sipm_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (err != cudaSuccess) return err;
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(max_blocks_per_sm, sipm_kernel<float>, SNT, bytes);
    }
    err = cudaFuncSetAttribute(sipm_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (err != cudaSuccess) return err;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(max_blocks_per_sm, sipm_kernel<uint16_t>, SNT, bytes);
}

void sipm_launch(const SipmDev& P, const void* d_wf, long long n_events, long long ld, double* d_rows, double* d_trig, int grid,
                 cudaStream_t stream)
{
    const size_t bytes = sipm_smem_bytes(P.n);
    if (P.kind == LGDSP_SAMPLE_F32)
        sipm_kernel<float><<<grid, SNT, bytes, stream>>>(P, static_cast<const float*>(d_wf), n_events, ld, d_rows, d_trig);
    else
        sipm_kernel<uint16_t><<<grid, SNT, bytes, stream>>>(P, static_cast<const uint16_t*>(d_wf), n_events, ld, d_rows, d_trig);
}

cudaError_t wfstats_configure(const WfstatsDev& P, int* max_blocks_per_sm)
{
    if (P.kind == LGDSP_SAMPLE_F64) return wfstats_configure_kind<double>(P, max_blocks_per_sm);
    if (P.kind == LGDSP_SAMPLE_F32) return wfstats_configure_kind<float>(P, max_blocks_per_sm);
    return wfstats_configure_kind<uint16_t>(P, max_blocks_per_sm);
}

long long wfstats_work_doubles(const WfstatsDev& P)
{
    const bool sh = P.n <= LGDSP_MAX_SAMPLES;
    return (!sh && (P.what & LGDSP_WFSTAT_THRESHOLDSTATS_MAD) && P.kind != LGDSP_SAMPLE_F64) ? P.n : 0;
}

void wfstats_launch(const WfstatsDev& P, const void* d_wf, const double* d_thr, long long n_events, long long ld, double* d_rows,
                    double* d_lists, double* d_work, int grid, cudaStream_t stream)
{
    if (P.kind == LGDSP_SAMPLE_F64) wfstats_launch_kind<double>(P, d_wf, d_thr, n_events, ld, d_rows, d_lists, d_work, grid, stream);
    else if (P.kind == LGDSP_SAMPLE_F32) wfstats_launch_kind<float>(P, d_wf, d_thr, n_events, ld, d_rows, d_lists, d_work, grid, stream);
    else wfstats_launch_kind<uint16_t>(P, d_wf, d_thr, n_events, ld, d_rows, d_lists, d_work, grid, stream);
}

void sipm_count_scan_launch(const double* d_rows, long long n_events, int list, int cap, long long* d_elem_ptr, cudaStream_t stream)
{
    sipm_count_scan_kernel<<<1, 1024, 0, stream>>>(d_rows, n_events, list, cap, d_elem_ptr);
}

void sipm_compact_launch(const double* d_trig, long long n_events, int list, int cap, const long long* d_elem_ptr, double* d_flat,
                         long long flat_stride, cudaStream_t stream)
{
    if (n_events <= 0) return;
    const unsigned grid = (unsigned)((n_events + 7) / 8);
    sipm_compact_kernel<<<grid, 256, 0, stream>>>(d_trig, n_events, list, cap, d_elem_ptr, d_flat, flat_stride);
}

void multi_intersect_launch(const MiDev& P, const double* d_y, long long n_events, long long ld, double* d_x, int* d_flags,
                            cudaStream_t stream)
{
    const long long blocks = (n_events + MI_WARPS - 1) / MI_WARPS;
    const unsigned grid = (unsigned)(blocks < 148 * 8 ? blocks : 148 * 8);
    if (grid == 0) return;
    multi_intersect_kernel<<<grid, MI_WARPS * 32, 0, stream>>>(P, d_y, n_events, ld, d_x, d_flags);
}

}  // namespace lgdsp
