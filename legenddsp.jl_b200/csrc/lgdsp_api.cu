// C ABI of liblgdsp_b200 (include/lgdsp_b200.h): handle management, parameter validation/upload, launches.
// No CPU fallback: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>
#include "lgdsp_kernels.h"

using namespace lgdsp;

#define LGDSP_SPLIT_MAX_STREAMS 6
#define LGDSP_HOST_ARRAYS 5   // per-event arrays one host entry point moves (dsp_icpc_compressed: 2 in, 3 out)

struct lgdsp_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0;
    int icpc_bps = 0, sweep_bps = 0;
    std::string err;
    // device tables
    double* d_dniA = nullptr;      // [2][LGDSP_MAX_DNI*4]
    double* d_cusp_g = nullptr;    // [LGDSP_MAX_FIR+1]
    double* d_zac_g = nullptr;     // [LGDSP_MAX_FIR+1]
    double* d_sweep_dniA = nullptr;
    SweepVar* d_vars = nullptr;
    size_t vars_cap = 0;
    double* d_taps = nullptr;      // differenced FIR / SG taps of the sweep variants
    size_t taps_cap = 0;
    IcpcDev icpc{};
    bool have_icpc = false;
    // second parameter slot: the windowed-waveform pass of dsp_icpc_compressed
    IcpcDev icpc_w{};
    bool have_icpc_w = false;
    double* d_dniA_w = nullptr;
    double* d_cusp_g_w = nullptr;
    double* d_zac_g_w = nullptr;
    int* d_win = nullptr;      // window list of the window statistics: [LGDSP_MAX_STAT_WINDOWS][2]
    // device slots of the chunked host paths (run_chunked): [buffer][array], the dense rows of one chunk
    void* d_slot[2][LGDSP_HOST_ARRAYS] = {};
    size_t slot_cap[2][LGDSP_HOST_ARRAYS] = {};
    double* d_work = nullptr;  // converted traces of lgdsp_wfstats_run when they are not staged in shared memory
    size_t work_cap = 0;
    cudaStream_t s_copy = nullptr;
    cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    // pinned staging of the host paths (HostIO below): pageable caller memory goes through these double buffers
    void* h_pin[2] = {nullptr, nullptr};
    size_t pin_cap = 0;
    void* h_out[2] = {nullptr, nullptr};
    size_t out_cap = 0;
    cudaEvent_t ev_pin[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    int copy_threads = 4;
    int64_t host_chunk_direct = 8192;   // the same for raw samples copied directly from page-locked caller memory
    int64_t host_chunk = 16384;    // events per chunk of the host paths (4096 / 8192 / 16384 / 32768 measured: 16384 is the best of the four for pageable, pinned and encoded input)
    // encoded-waveform staging (decode_data on the device)
    uint8_t* d_enc[2][2] = {};     // [buffer][input]
    size_t enc_cap[2][2] = {};
    long long* d_off[2][2] = {};
    size_t off_cap[2][2] = {};
    void* d_dec[2] = {};           // [input] decoded waveforms of the current chunk
    size_t dec_cap[2] = {};
    int* d_dstat = nullptr;
    size_t dstat_cap = 0;
    // timing
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    int64_t launches = 0;
    // split dsp_icpc pipeline (lgdsp_icpc_split.cuh): ring of prefix sums + per-event hand-over values, side streams
    int icpc_path = 1;             // 0: fused icpc_kernel, 1: split pipeline
    int split_bps[3] = {0, 0, 0};
    int64_t split_batch = 0;       // events per batch (0: default)
    int split_streams = 4;         // stream pairs the sub-batches go round (2 / 3 / 4: 6.35 / 6.56 / 6.67 M wf/s)
    double* d_tt = nullptr;
    double* d_saux = nullptr;
    double* d_scz = nullptr;       // candidate records of the CUSP/ZAC kernels
    int64_t split_cap = 0;         // allocated slots
    cudaStream_t s_split[LGDSP_SPLIT_MAX_STREAMS] = {};
    cudaStream_t s_cz[LGDSP_SPLIT_MAX_STREAMS] = {};   // CUSP/ZAC kernel next to the extract kernel
    cudaEvent_t ev_pre[LGDSP_SPLIT_MAX_STREAMS] = {}, ev_cz[LGDSP_SPLIT_MAX_STREAMS] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[LGDSP_SPLIT_MAX_STREAMS] = {nullptr, nullptr, nullptr, nullptr};
};

static thread_local std::string g_create_err;

static int fail(lgdsp_handle* h, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_err = buf;
    return code;
}

#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess)                                                                         \
            return fail(h, e_ == cudaErrorMemoryAllocation ? LGDSP_ERR_OOM : LGDSP_ERR_CUDA, "%s: %s", \
                        #call, cudaGetErrorString(e_));                                                \
    } while (0)

extern "C" {

const char* lgdsp_version(void) { return "lgdsp_b200 0.1 (sm_100a)"; }

const char* lgdsp_last_error(const lgdsp_handle* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int lgdsp_create(int device, void* stream, lgdsp_handle** out)
{
    lgdsp_handle* h = nullptr;
    if (!out) return fail(nullptr, LGDSP_ERR_INVALID_ARG, "lgdsp_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0)
        return fail(nullptr, LGDSP_ERR_NO_DEVICE, "lgdsp_create: no CUDA device (%s); this library has no CPU path",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= ndev) return fail(nullptr, LGDSP_ERR_INVALID_ARG, "lgdsp_create: device %d of %d", device, ndev);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
        return fail(nullptr, LGDSP_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major < 10)
        return fail(nullptr, LGDSP_ERR_UNSUPPORTED, "lgdsp_create: device %d is sm_%d%d; this library is built for sm_100a only",
                    device, prop.major, prop.minor);
    h = new lgdsp_handle();
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    auto bail = [&](int code) { lgdsp_destroy(h); return code; };
    if ((e = cudaSetDevice(device)) != cudaSuccess) { fail(nullptr, LGDSP_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e)); return bail(LGDSP_ERR_CUDA); }
    if (stream) {
        h->stream = (cudaStream_t)stream;
    } else {
        if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) {
            fail(nullptr, LGDSP_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
            return bail(LGDSP_ERR_CUDA);
        }
        h->own_stream = true;
    }
    bool ok = cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < 2 && ok; ++i) {
        ok = ok && cudaEventCreateWithFlags(&h->ev_ready[i], cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&h->ev_free[i], cudaEventDisableTiming) == cudaSuccess;
    }
    for (int i = 0; i < 2 && ok; ++i) {
        ok = ok && cudaEventCreateWithFlags(&h->ev_pin[i], cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&h->ev_out[i], cudaEventDisableTiming) == cudaSuccess;
    }
    {
        unsigned hw = std::thread::hardware_concurrency();
        h->copy_threads = hw >= 16 ? 8 : (hw >= 4 ? (int)hw / 2 : 1);
        if (const char* env = getenv("LGDSP_COPY_THREADS")) h->copy_threads = atoi(env) > 0 ? atoi(env) : 1;
        if (const char* env = getenv("LGDSP_HOST_CHUNK")) h->host_chunk = atoll(env) > 0 ? atoll(env) : 16384;
        if (const char* env = getenv("LGDSP_HOST_CHUNK_DIRECT")) h->host_chunk_direct = atoll(env) > 0 ? atoll(env) : 8192;
    }
    ok = ok && cudaEventCreate(&h->ev0) == cudaSuccess && cudaEventCreate(&h->ev1) == cudaSuccess;
    ok = ok && cudaMalloc(&h->d_dniA, sizeof(double) * 2 * LGDSP_MAX_DNI * 4) == cudaSuccess;
    ok = ok && cudaMalloc(&h->d_cusp_g, sizeof(double) * (LGDSP_MAX_FIR + 1)) == cudaSuccess;
    ok = ok && cudaMalloc(&h->d_zac_g, sizeof(double) * (LGDSP_MAX_FIR + 1)) == cudaSuccess;
    ok = ok && cudaMalloc(&h->d_sweep_dniA, sizeof(double) * LGDSP_MAX_DNI * 4) == cudaSuccess;
    ok = ok && cudaMalloc(&h->d_win, sizeof(int) * 2 * LGDSP_MAX_STAT_WINDOWS) == cudaSuccess;
    if (!ok) { fail(nullptr, LGDSP_ERR_CUDA, "lgdsp_create: resource allocation failed: %s", cudaGetErrorString(cudaGetLastError())); return bail(LGDSP_ERR_CUDA); }
    if ((e = icpc_configure(&h->icpc_bps)) != cudaSuccess || (e = sweep_configure(&h->sweep_bps)) != cudaSuccess) {
        fail(nullptr, LGDSP_ERR_CUDA, "kernel configuration failed: %s (is the library built for this GPU?)", cudaGetErrorString(e));
        return bail(LGDSP_ERR_CUDA);
    }
    if (h->icpc_bps < 1 || h->sweep_bps < 1) { fail(nullptr, LGDSP_ERR_CUDA, "kernels do not fit on an SM"); return bail(LGDSP_ERR_CUDA); }
    if ((e = icpc_split_configure(h->split_bps)) != cudaSuccess || h->split_bps[0] < 1 || h->split_bps[1] < 1 || h->split_bps[2] < 1) {
        fail(nullptr, LGDSP_ERR_CUDA, "split pipeline configuration failed: %s", cudaGetErrorString(e));
        return bail(LGDSP_ERR_CUDA);
    }
    for (int i = 0; i < LGDSP_SPLIT_MAX_STREAMS && ok; ++i) {
        ok = ok && cudaStreamCreateWithFlags(&h->s_split[i], cudaStreamNonBlocking) == cudaSuccess;
        ok = ok && cudaStreamCreateWithFlags(&h->s_cz[i], cudaStreamNonBlocking) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&h->ev_pre[i], cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&h->ev_cz[i], cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&h->ev_join[i], cudaEventDisableTiming) == cudaSuccess;
    }
    ok = ok && cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) { fail(nullptr, LGDSP_ERR_CUDA, "lgdsp_create: stream allocation failed: %s", cudaGetErrorString(cudaGetLastError())); return bail(LGDSP_ERR_CUDA); }
    if (const char* env = getenv("LGDSP_ICPC_PATH")) h->icpc_path = (strcmp(env, "fused") == 0) ? 0 : 1;
    if (const char* env = getenv("LGDSP_SPLIT_BATCH")) h->split_batch = atoll(env);
    if (const char* env = getenv("LGDSP_SPLIT_STREAMS")) h->split_streams = atoi(env);
    if (h->split_streams < 1) h->split_streams = 1;
    if (h->split_streams > LGDSP_SPLIT_MAX_STREAMS) h->split_streams = LGDSP_SPLIT_MAX_STREAMS;
    *out = h;
    return LGDSP_OK;
}

void lgdsp_destroy(lgdsp_handle* h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (int i = 0; i < LGDSP_SPLIT_MAX_STREAMS; ++i) {
        if (h->s_split[i]) { cudaStreamSynchronize(h->s_split[i]); cudaStreamDestroy(h->s_split[i]); }
        if (h->s_cz[i]) { cudaStreamSynchronize(h->s_cz[i]); cudaStreamDestroy(h->s_cz[i]); }
        if (h->ev_pre[i]) cudaEventDestroy(h->ev_pre[i]);
        if (h->ev_cz[i]) cudaEventDestroy(h->ev_cz[i]);
        if (h->ev_join[i]) cudaEventDestroy(h->ev_join[i]);
    }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    cudaFree(h->d_tt); cudaFree(h->d_saux); cudaFree(h->d_scz);
    cudaFree(h->d_dniA); cudaFree(h->d_cusp_g); cudaFree(h->d_zac_g); cudaFree(h->d_sweep_dniA); cudaFree(h->d_vars); cudaFree(h->d_taps);
    cudaFree(h->d_win); cudaFree(h->d_work);
    cudaFree(h->d_dniA_w); cudaFree(h->d_cusp_g_w); cudaFree(h->d_zac_g_w);
    for (int i = 0; i < 2; ++i) {
        for (int k = 0; k < LGDSP_HOST_ARRAYS; ++k) cudaFree(h->d_slot[i][k]);
        if (h->ev_ready[i]) cudaEventDestroy(h->ev_ready[i]);
        if (h->ev_free[i]) cudaEventDestroy(h->ev_free[i]);
        if (h->ev_pin[i]) cudaEventDestroy(h->ev_pin[i]);
        if (h->ev_out[i]) cudaEventDestroy(h->ev_out[i]);
        if (h->h_pin[i]) cudaFreeHost(h->h_pin[i]);
        if (h->h_out[i]) cudaFreeHost(h->h_out[i]);
        for (int k = 0; k < 2; ++k) { cudaFree(h->d_enc[i][k]); cudaFree(h->d_off[i][k]); }
        cudaFree(h->d_dec[i]);
    }
    cudaFree(h->d_dstat);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->s_copy) cudaStreamDestroy(h->s_copy);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int64_t lgdsp_launch_count(const lgdsp_handle* h) { return h ? h->launches : 0; }

int lgdsp_synchronize(lgdsp_handle* h)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return LGDSP_OK;
}

double lgdsp_last_kernel_ms(const lgdsp_handle* h)
{
    if (!h || !h->timed) return -1.0;
    float ms = 0;
    if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) != cudaSuccess) return -1.0;
    return (double)ms;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// parameter validation and conversion
// ---------------------------------------------------------------------------------------------------
static bool make_trap(const lgdsp_trap& t, int n, int min_out, TrapDev& d)
{
    if (t.navg < 1 || t.navg2 < 1 || t.ngap < 0) return false;
    d.a = t.navg; d.g = t.ngap; d.a2 = t.navg2;
    d.L = t.navg + t.ngap + t.navg2;
    d.nout = n - d.L + 1;
    d.pad_ = 0;
    d.inv1 = 1.0 / t.navg;
    d.inv2 = 1.0 / t.navg2;
    return d.nout >= min_out;
}


// analytic descriptor of a CUSP/ZAC filter for the structured device evaluation (lgdsp_icpc.cu)
static bool make_czdev(const lgdsp_cuspzac& z, const double* cusp_coeffs, const double* zac_coeffs, CzDev& D, std::string& why)
{
    typedef long double ld;
    const int L = z.n_taps, F = z.flat;
    const int lt = (L - F) / 2, Rn = L - lt - F - 1;
    if (lt < 2 || Rn < 1 || !(z.sigma > 0) || !(z.tau > 0)) { why = "flank too short for the structured evaluation"; return false; }
    const ld sg = z.sigma, x = (ld)lt / sg;
    if (x > 700.0L) { why = "lt/sigma too large"; return false; }
    const ld a = 1.0L / sinhl(x), cA = 0.5L * a, h = lt / 2.0L;
    const ld r = expl(-1.0L / (ld)z.tau), rho = expl(-1.0L / sg);
    memset(&D, 0, sizeof(D));
    D.L = L; D.F = F; D.lt = lt; D.Rn = Rn;
    auto mod = [](int v) { return ((v % CZ_CH) + CZ_CH) % CZ_CH; };
    D.oc[0] = 0; D.oc[1] = mod(-lt); D.oc[2] = mod(-lt - F - 1); D.oc[3] = mod(-L);
    D.oa[0] = mod(1 - lt); D.oa[1] = mod(1); D.oa[2] = mod(1 - L); D.oa[3] = mod(-lt - F);
    D.r = (double)r; D.rho = (double)rho; D.rho_inv = (double)(1.0L / rho); D.inv_sigma = (double)(1.0L / sg);
    D.cA = (double)cA;
    D.cA_rho_lt = (double)(cA * expl(-(ld)lt / sg));
    D.cA_rhoinv_lt = (double)(cA * expl((ld)lt / sg));
    D.cA_rhoinv_Rn = (double)(cA * expl((ld)Rn / sg));
    D.cA_rho_Rn = (double)(cA * expl(-(ld)Rn / sg));
    D.rho_lt = (double)expl(-(ld)lt / sg);
    D.rho_Rn = (double)expl(-(ld)Rn / sg);
    D.cA_rhoinv_ltm1 = (double)(cA * expl((ld)(lt - 1) / sg));
    D.cA_rho = (double)(cA * rho);
    {
        // capture events: causal table q after sample oc[q]; anti-causal table q after sample oa[q]-1
        struct Ev { int k, kind, tab; };
        Ev ev[8];
        for (int q = 0; q < 4; ++q) { ev[q] = {D.oc[q], 0, q}; ev[4 + q] = {D.oa[q] - 1, 1, q}; }
        for (int a_ = 0; a_ < 8; ++a_)
            for (int b_ = a_ + 1; b_ < 8; ++b_)
                if (ev[b_].k < ev[a_].k) { Ev t_ = ev[a_]; ev[a_] = ev[b_]; ev[b_] = t_; }
        D.n_ev = 8;
        for (int i = 0; i < 8; ++i) {
            D.ev_k[i] = ev[i].k; D.ev_kind[i] = ev[i].kind; D.ev_tab[i] = ev[i].tab;
            if (ev[i].kind == 0) {
                D.ev_pw[i] = (double)expl(-(ld)(ev[i].k + 1) / sg);
                D.ev_rinv[i] = 0.0;
            } else {
                const int o = ev[i].k + 1;
                D.ev_pw[i] = (double)expl(-(ld)(CZ_CH - o) / sg);
                D.ev_rinv[i] = (double)expl((ld)o / sg);
            }
        }
    }
    for (int s2 = 0; s2 < 5; ++s2) D.rho_ch_pow[s2] = (double)expl(-(ld)(CZ_CH << s2) / sg);
    for (int l = 0; l < 32; ++l) D.rho_lane[l] = (double)expl(-(ld)(CZ_CH * (l + 1)) / sg);
    D.rho_warp = (double)expl(-(ld)(CZ_CH * 32) / sg);
    D.h2 = (double)(2.0L * h);
    D.lt_d = lt; D.lt2_d = (double)lt * lt; D.Rn_d = Rn; D.Rn2_d = (double)Rn * Rn;
    // shape sums -> parabola amplitude of the ZAC
    ld acusp = 0, apar = 0;
    auto cusp_at = [&](int k) -> ld { return k < lt ? sinhl(k / sg) * a : (k <= lt + F ? 1.0L : sinhl((L - k) / sg) * a); };
    auto par_at = [&](int k) -> ld { return k < lt ? (k - h) * (k - h) - h * h : (k <= lt + F ? 0.0L : (L - k - h) * (L - k - h) - h * h); };
    for (int k = 0; k < L; ++k) { acusp += cusp_at(k); apar += par_at(k); }
    const ld B = apar != 0.0L ? -(acusp / apar) : 0.0L;
    D.B = (double)B;
    const ld g = (ld)z.beta / L;
    D.g = (double)g;
    D.gclast_cusp = (double)(g * r * cusp_at(L - 1));
    D.gclast_zac = (double)(g * r * (cusp_at(L - 1) + B * par_at(L - 1)));
    // Lipschitz constants of the two output traces (coarse-to-fine pruning in the kernel): total variation of the
    // zero-extended taps h[k] = g*(c[k] - r*c[k-1])
    for (int which = 0; which < 2; ++which) {
        const ld bb = which ? B : 0.0L;
        ld prev_c = 0.0L, prev_h = 0.0L, tv = 0.0L;
        for (int k = 0; k < L; ++k) {
            const ld ck = cusp_at(k) + bb * par_at(k);
            const ld hk = g * (ck - r * prev_c);
            tv += fabsl(hk - prev_h);
            prev_c = ck;
            prev_h = hk;
        }
        tv += fabsl(prev_h);
        (which ? D.lip_zac : D.lip_cusp) = (double)(tv * (1.0L + 1e-9L));
    }
    // the coefficient arrays passed through the ABI must be the ones this structure reproduces
    for (int which = 0; which < 2; ++which) {
        const double* co = which ? zac_coeffs : cusp_coeffs;
        if (!co) continue;
        double scale = 0;
        for (int k = 0; k < L; ++k) scale = fmax(scale, fabs(co[k]));
        const ld bb = which ? B : 0.0L;
        ld prev = 0.0L;
        for (int k = 0; k < L; ++k) {
            const ld ck = cusp_at(k) + bb * par_at(k);
            const double expect = (double)(g * (ck - r * prev));
            prev = ck;
            if (!(fabs(expect - co[k]) <= 1e-9 * scale)) {
                why = which ? "zac.coeffs do not match (sigma, flat, tau, n_taps, beta)" : "cusp.coeffs do not match (sigma, flat, tau, n_taps, beta)";
                return false;
            }
        }
    }
    return true;
}

static int icpc_prepare(lgdsp_handle* h, const lgdsp_icpc_params* p, int slot = 0)
{
    if (!p) return fail(h, LGDSP_ERR_INVALID_ARG, "params is NULL");
    if (slot && !h->d_dniA_w) {
        CK(cudaMalloc(&h->d_dniA_w, sizeof(double) * 2 * LGDSP_MAX_DNI * 4));
        CK(cudaMalloc(&h->d_cusp_g_w, sizeof(double) * (LGDSP_MAX_FIR + 1)));
        CK(cudaMalloc(&h->d_zac_g_w, sizeof(double) * (LGDSP_MAX_FIR + 1)));
    }
    double* const t_dniA = slot ? h->d_dniA_w : h->d_dniA;
    double* const t_cusp = slot ? h->d_cusp_g_w : h->d_cusp_g;
    double* const t_zac = slot ? h->d_zac_g_w : h->d_zac_g;
    if (p->struct_size != sizeof(lgdsp_icpc_params) || p->version != LGDSP_PARAMS_VERSION)
        return fail(h, LGDSP_ERR_INVALID_ARG, "lgdsp_icpc_params: size/version mismatch (got %u/%u, want %zu/%u)",
                    p->struct_size, p->version, sizeof(lgdsp_icpc_params), LGDSP_PARAMS_VERSION);
    const int n = p->n_samples;
    if (n < 64 || n > LGDSP_MAX_SAMPLES || n % 8 != 0)
        return fail(h, LGDSP_ERR_UNSUPPORTED, "n_samples = %d: need a multiple of 8 in [64, %d]", n, LGDSP_MAX_SAMPLES);
    if (!(p->dt_ns > 0) || !std::isfinite(p->t_first_ns)) return fail(h, LGDSP_ERR_INVALID_ARG, "bad time axis");
    auto win_ok = [&](int a, int b, int len) { return 0 <= a && a <= b && b <= len - 1; };
    // @assert firstindex(X) <= first(idxs) <= last(idxs) <= lastindex(X)   /root/reference/src/tailstats.jl:23-25
    if (!win_ok(p->bl_from, p->bl_until, n)) return fail(h, LGDSP_ERR_INVALID_ARG, "bl_window %d:%d outside the waveform", p->bl_from, p->bl_until);
    if (!win_ok(p->tail_from, p->tail_until, n)) return fail(h, LGDSP_ERR_INVALID_ARG, "tail_window %d:%d outside the waveform", p->tail_from, p->tail_until);
    IcpcDev D{};
    D.n = n;
    D.groups = p->groups | LGDSP_GROUP_BASE;
    D.t_first = p->t_first_ns;
    D.dt = p->dt_ns;
    D.sat_low = (p->sat_low >= 0 && p->sat_low <= 0x7fffffffLL) ? (int)p->sat_low : -1;
    D.sat_high = (p->sat_high >= 0 && p->sat_high <= 0x7fffffffLL) ? (int)p->sat_high : -1;
    D.bl_from = p->bl_from; D.bl_until = p->bl_until; D.tail_from = p->tail_from; D.tail_until = p->tail_until;
    D.km1 = p->pz_km1;
    D.bl_inv_n = 1.0 / (double)(p->bl_until - p->bl_from + 1);
    D.tail_inv_n = 1.0 / (double)(p->tail_until - p->tail_from + 1);
    {
        // sum_{i=a}^{b} X_i and X_i^2 with X_i = t_first + i*dt (configuration constants of the two regressions)
        auto xs = [&](int a, int b, double& sX, double& sXX) {
            typedef long double ld;
            const ld t0 = p->t_first_ns, dt = p->dt_ns, cnt = (ld)(b - a + 1);
            auto s2 = [](ld k) { return k * (k + 1.0L) * (2.0L * k + 1.0L) / 6.0L; };
            const ld si = 0.5L * (ld)(a + b) * cnt, sii = s2((ld)b) - s2((ld)a - 1.0L);
            sX = (double)(cnt * t0 + dt * si);
            sXX = (double)(cnt * t0 * t0 + 2.0L * t0 * dt * si + dt * dt * sii);
        };
        xs(p->bl_from, p->bl_until, D.bl_sX, D.bl_sXX);
        xs(p->tail_from, p->tail_until, D.tail_sX, D.tail_sXX);
    }
    const int nw_sig = p->sig_dni.n_w, nw_int = p->int_dni.n_w;
    auto dni_ok = [](const lgdsp_dni& d) { return d.degree >= 0 && d.degree <= LGDSP_MAX_DNI_DEG && d.n_w > d.degree && d.n_w <= LGDSP_MAX_DNI; };
    if (!dni_ok(p->sig_dni) || !dni_ok(p->int_dni)) return fail(h, LGDSP_ERR_UNSUPPORTED, "PolynomialDNI window/degree outside the supported range");
    if (nw_int > n) return fail(h, LGDSP_ERR_INVALID_ARG, "int_dni window longer than the waveform");
    D.int_dni.n_w = nw_int; D.int_dni.m = p->int_dni.degree + 1;
    D.sig_dni.n_w = nw_sig; D.sig_dni.m = p->sig_dni.degree + 1;
    if (!make_trap(p->t0_trap, n, 2, D.t0) || !make_trap(p->t0inv_trap, n, 2, D.t0inv))
        return fail(h, LGDSP_ERR_INVALID_ARG, "t0 trapezoid does not fit the waveform");
    if (!make_trap(p->trap_10410, n, 1, D.e10410) || !make_trap(p->trap_535, n, 1, D.e535) || !make_trap(p->trap_313, n, 1, D.e313))
        return fail(h, LGDSP_ERR_INVALID_ARG, "fixed trapezoid does not fit the waveform");
    if (!make_trap(p->trap_e, n, nw_sig, D.etrap)) return fail(h, LGDSP_ERR_INVALID_ARG, "trap(rt,ft) leaves fewer outputs than the DNI window");
    D.t0inv_same = (D.t0.a == D.t0inv.a && D.t0.g == D.t0inv.g && D.t0.a2 == D.t0inv.a2) ? 1 : 0;
    if (p->t0_min_n < 1 || p->tx_min_n < 1 || p->intrace_min_n < 1) return fail(h, LGDSP_ERR_INVALID_ARG, "min_n must be >= 1");
    D.t0_min_n = p->t0_min_n; D.tx_min_n = p->tx_min_n; D.direct = p->cuspzac_direct;
    D.t0_thr = p->t0_threshold;
    for (int i = 0; i < 5; ++i) D.tx_frac[i] = p->tx_frac[i];
    D.qd_first = p->qdrift_first_ns; D.qd_last = p->qdrift_last_ns; D.lq_first = p->lq_first_ns; D.lq_last = p->lq_last_ns;
    D.trap_pick = p->trap_pickoff_ns; D.cusp_pick = p->cusp_pickoff_ns; D.zac_pick = p->zac_pickoff_ns;
    for (int k = 0; k < 3; ++k) {
        const lgdsp_sg& s = p->sg[k];
        if (s.n_taps < 1 || s.n_taps > LGDSP_MAX_SG || s.n_taps > n || s.offset < 0 || s.offset >= s.n_taps)
            return fail(h, LGDSP_ERR_INVALID_ARG, "sg[%d]: bad tap count/offset", k);
        SgDev& d = D.sg[k];
        d.n_taps = s.n_taps; d.offset = s.offset; d.nout = n - s.n_taps + 1; d.pad_ = 0;
        d.gg[0] = -s.h[0];
        for (int i = 1; i < s.n_taps; ++i) d.gg[i] = s.h[i - 1] - s.h[i];
        d.gg[s.n_taps] = s.h[s.n_taps - 1];
        if (!win_ok(p->cur_from[k], p->cur_until[k], d.nout))
            return fail(h, LGDSP_ERR_INVALID_ARG, "current_window %d:%d outside sg[%d] trace", p->cur_from[k], p->cur_until[k], k);
    }
    if (!win_ok(p->cur_from[3], p->cur_until[3], n)) return fail(h, LGDSP_ERR_INVALID_ARG, "current_window outside the waveform");
    for (int k = 0; k < 4; ++k) { D.cur_from[k] = p->cur_from[k]; D.cur_until[k] = p->cur_until[k]; D.sg_alias[k] = -1; }
    for (int k = 1; k < 3; ++k)
        for (int q = 0; q < k && D.sg_alias[k] < 0; ++q)
            if (p->sg[k].n_taps == p->sg[q].n_taps && p->cur_from[k] == p->cur_from[q] && p->cur_until[k] == p->cur_until[q] &&
                memcmp(p->sg[k].h, p->sg[q].h, sizeof(double) * p->sg[k].n_taps) == 0)
                D.sg_alias[k] = q;
    D.nsigma = p->intrace_nsigma;
    D.intr_min_n = p->intrace_min_n;
    if (!win_ok(p->intrace_bl_from, p->intrace_bl_until, D.sg[0].nout)) return fail(h, LGDSP_ERR_INVALID_ARG, "in-trace sigma window outside the sg trace");
    D.intr_from = p->intrace_bl_from; D.intr_until = p->intrace_bl_until;
    D.intr_inv_n = 1.0 / (double)(p->intrace_bl_until - p->intrace_bl_from + 1);
    // CUSP / ZAC
    // (all validation first: the device tables of the handle are only touched once the whole parameter set is accepted, so
    // a rejected set leaves the previous one -- descriptors AND tables -- intact)
    const lgdsp_cuspzac* cz[2] = {&p->cusp, &p->zac};
    double* dst[2] = {t_cusp, t_zac};
    std::vector<double> g[2];
    for (int f = 0; f < 2; ++f) {
        const int L = cz[f]->n_taps;
        if (L < 4 || L > LGDSP_MAX_FIR || n - L + 1 < nw_sig)
            return fail(h, LGDSP_ERR_INVALID_ARG, "%s: %d taps do not fit (need >= %d outputs)", f ? "zac" : "cusp", L, nw_sig);
        // differenced taps on the prefix sum TT: out[j] = sum_{k=0}^{L} g[k] TT[j+L-k]
        const double* c = cz[f]->coeffs;
        g[f].resize(L + 1);
        g[f][0] = c[0];
        for (int k = 1; k < L; ++k) g[f][k] = c[k] - c[k - 1];
        g[f][L] = -c[L - 1];
    }
    D.cusp_L = p->cusp.n_taps; D.zac_L = p->zac.n_taps;
    if (!D.direct && (D.groups & LGDSP_GROUP_CUSPZAC)) {
        const lgdsp_cuspzac &c = p->cusp, &z = p->zac;
        D.cz_shared = (c.n_taps == z.n_taps && c.flat == z.flat && c.sigma == z.sigma && c.tau == z.tau && c.beta == z.beta) ? 1 : 0;
        std::string why;
        bool ok;
        if (D.cz_shared) {
            ok = make_czdev(c, c.coeffs, z.coeffs, D.cz[0], why);
            D.cz[1] = D.cz[0];
        } else {
            ok = make_czdev(c, c.coeffs, nullptr, D.cz[0], why) && make_czdev(z, nullptr, z.coeffs, D.cz[1], why);
        }
        if (!ok) return fail(h, LGDSP_ERR_UNSUPPORTED, "CUSP/ZAC structured evaluation: %s (set cuspzac_direct = 1)", why.c_str());
    }
    for (int f = 0; f < 2; ++f) CK(cudaMemcpyAsync(dst[f], g[f].data(), sizeof(double) * g[f].size(), cudaMemcpyHostToDevice, h->stream));
    std::vector<double> A(2 * LGDSP_MAX_DNI * 4, 0.0);
    memcpy(A.data(), p->int_dni.A, sizeof(double) * LGDSP_MAX_DNI * 4);
    memcpy(A.data() + LGDSP_MAX_DNI * 4, p->sig_dni.A, sizeof(double) * LGDSP_MAX_DNI * 4);
    CK(cudaMemcpyAsync(t_dniA, A.data(), sizeof(double) * A.size(), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    D.dni_A = t_dniA; D.cusp_g = t_cusp; D.zac_g = t_zac;
    if (slot) { h->icpc_w = D; h->have_icpc_w = true; }
    else { h->icpc = D; h->have_icpc = true; }
    return LGDSP_OK;
}

static int check_wf(lgdsp_handle* h, const void* wf, int64_t n_events, int64_t ld, int n, bool device, int sample_bytes = 2)
{
    if (sample_bytes != 2 && sample_bytes != 4) return fail(h, LGDSP_ERR_UNSUPPORTED, "sample_bytes = %d: uint16 (2) or uint32 (4) samples", sample_bytes);
    if (sample_bytes == 4 && n > LGDSP_MAX_SAMPLES / 2)
        return fail(h, LGDSP_ERR_UNSUPPORTED, "32-bit samples: n_samples = %d > %d", n, LGDSP_MAX_SAMPLES / 2);
    if (n_events < 0) return fail(h, LGDSP_ERR_INVALID_ARG, "n_events < 0");
    if (n_events == 0) return LGDSP_OK;  // empty table in, empty table out
    if (n_events > 0 && !wf) return fail(h, LGDSP_ERR_INVALID_ARG, "waveform pointer is NULL");
    if (ld < n) return fail(h, LGDSP_ERR_INVALID_ARG, "ld_samples (%lld) < n_samples (%d)", (long long)ld, n);
    if (device && (((uintptr_t)wf & 15u) != 0 || (ld * sample_bytes) % 16 != 0))
        return fail(h, LGDSP_ERR_INVALID_ARG, "device waveforms must be 16-byte aligned with rows of a multiple of 16 bytes (TMA bulk copy)");
    return LGDSP_OK;
}

// Grows a device buffer of the handle to at least `bytes`; the contents are not kept.  Work on either stream may still use
// the old buffer, so both are synchronised before it is freed.
template <class T>
static int grow(lgdsp_handle* h, T** p, size_t* cap, size_t bytes)
{
    if (bytes <= *cap) return LGDSP_OK;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaStreamSynchronize(h->s_copy));
    cudaFree(*p); *p = nullptr; *cap = 0;
    CK(cudaMalloc(p, bytes));
    *cap = bytes;
    return LGDSP_OK;
}

// One dsp_icpc pass over a device batch, in stream order behind h->stream.  Fused path: one launch of icpc_kernel.  Split
// path: the batch is cut into sub-batches whose prefix sums (65.6 KB per event) fit the L2; sub-batches alternate between
// side streams (forked from / joined to h->stream with events) so that the tail of one kernel overlaps the next sub-batch.
static int icpc_dispatch(lgdsp_handle* h, const IcpcDev& D, const void* d_wf, int sample_bytes, int64_t ne, int64_t ld,
                         const double* d_bl, int64_t bl_stride, double bl_div, double* d_rows)
{
    if (h->icpc_path == 0) {
        const long long cap = (long long)h->sm_count * h->icpc_bps;
        const int grid = (int)(ne < cap ? ne : cap);
        icpc_launch(D, d_wf, sample_bytes, ne, ld, d_bl, bl_stride, bl_div, d_rows, grid, h->stream);
        CK(cudaGetLastError());
        h->launches += 1;
        return LGDSP_OK;
    }
    const int S = h->split_streams;
    const int64_t B = h->split_batch > 0 ? h->split_batch : 4096;
    const int64_t need = B * S;
    if (need > h->split_cap) {
        CK(cudaStreamSynchronize(h->stream));
        for (int i = 0; i < LGDSP_SPLIT_MAX_STREAMS; ++i) CK(cudaStreamSynchronize(h->s_split[i]));
        cudaFree(h->d_tt); cudaFree(h->d_saux); cudaFree(h->d_scz);
        h->d_tt = nullptr; h->d_saux = nullptr; h->d_scz = nullptr; h->split_cap = 0;
        CK(cudaMalloc(&h->d_tt, sizeof(double) * (size_t)need * (size_t)icpc_split_tt_doubles()));
        CK(cudaMalloc(&h->d_saux, sizeof(double) * (size_t)need * (size_t)icpc_split_aux_doubles()));
        CK(cudaMalloc(&h->d_scz, sizeof(double) * (size_t)need * (size_t)icpc_split_cz_doubles()));
        h->split_cap = need;
    }
    const bool fork = S > 1 && ne > B;
    if (fork) {
        CK(cudaEventRecord(h->ev_fork, h->stream));
        for (int i = 0; i < S; ++i) CK(cudaStreamWaitEvent(h->s_split[i], h->ev_fork, 0));
    }
    const unsigned char* wf = static_cast<const unsigned char*>(d_wf);
    const bool cz = (D.groups & LGDSP_GROUP_CUSPZAC) != 0;
    int64_t b = 0;
    for (int64_t e0 = 0; e0 < ne; e0 += B, ++b) {
        const int64_t nb = (ne - e0) < B ? (ne - e0) : B;
        const int si = fork ? (int)(b % S) : 0;
        cudaStream_t st = fork ? h->s_split[si] : h->stream;
        icpc_split_launch_batch(D, wf + (size_t)e0 * (size_t)ld * (size_t)sample_bytes, sample_bytes, nb, ld,
                                d_bl ? d_bl + e0 * bl_stride : nullptr, bl_stride, bl_div, d_rows + e0 * LGDSP_NCOL,
                                h->d_tt + (size_t)si * (size_t)B * (size_t)icpc_split_tt_doubles(),
                                h->d_saux + (size_t)si * (size_t)B * (size_t)icpc_split_aux_doubles(),
                                h->d_scz + (size_t)si * (size_t)B * (size_t)icpc_split_cz_doubles(),
                                h->split_bps, h->sm_count, st,
                                h->s_cz[si], h->ev_pre[si], h->ev_cz[si], nullptr);
        CK(cudaGetLastError());
        h->launches += cz ? (D.direct ? 3 : 4) : 2;
    }
    if (fork) {
        for (int i = 0; i < S; ++i) {
            CK(cudaEventRecord(h->ev_join[i], h->s_split[i]));
            CK(cudaStreamWaitEvent(h->stream, h->ev_join[i], 0));
        }
    }
    return LGDSP_OK;
}

extern "C" {

/* path: 0 = fused icpc_kernel, 1 = split pipeline (default); batch <= 0 / streams <= 0: keep the defaults */
int lgdsp_icpc_set_path(lgdsp_handle* h, int32_t path, int64_t batch, int32_t streams)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    if (path != 0 && path != 1) return fail(h, LGDSP_ERR_INVALID_ARG, "lgdsp_icpc_set_path: path %d (0 fused, 1 split)", path);
    h->icpc_path = path;
    if (batch > 0) h->split_batch = batch;
    if (streams > 0) h->split_streams = streams > LGDSP_SPLIT_MAX_STREAMS ? LGDSP_SPLIT_MAX_STREAMS : streams;
    return LGDSP_OK;
}

int lgdsp_icpc_set_params(lgdsp_handle* h, const lgdsp_icpc_params* p)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    return icpc_prepare(h, p);
}

static int icpc_run_device_impl(lgdsp_handle* h, const lgdsp_icpc_params* p, const void* d_wf, int sample_bytes,
                                const double* d_baseline, int64_t n_events, int64_t ld_samples, double* d_out_rows)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (p) { int rc = icpc_prepare(h, p); if (rc) return rc; }
    if (!h->have_icpc) return fail(h, LGDSP_ERR_INVALID_ARG, "no parameters set (pass params or call lgdsp_icpc_set_params)");
    int rc = check_wf(h, d_wf, n_events, ld_samples, h->icpc.n, true, sample_bytes);
    if (rc) return rc;
    if (n_events == 0) return LGDSP_OK;  // empty input -> empty table
    if (!d_out_rows) return fail(h, LGDSP_ERR_INVALID_ARG, "output pointer is NULL");
    CK(cudaEventRecord(h->ev0, h->stream));
    rc = icpc_dispatch(h, h->icpc, d_wf, sample_bytes, n_events, ld_samples, d_baseline, 1, 1.0, d_out_rows);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev1, h->stream));
    h->timed = true;
    return LGDSP_OK;
}

// per-kernel device times of the split pipeline on ONE batch run serially (prefix, extract, CUSP/ZAC select, CUSP/ZAC finish)
int lgdsp_icpc_profile_device(lgdsp_handle* h, const uint16_t* d_wf, int64_t n_events, int64_t ld_samples, double* d_out_rows,
                              double* ms4)
{
    if (!h || !ms4) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (!h->have_icpc) return fail(h, LGDSP_ERR_INVALID_ARG, "no parameters set");
    int rc = check_wf(h, d_wf, n_events, ld_samples, h->icpc.n, true, 2);
    if (rc) return rc;
    if (n_events <= 0 || !d_out_rows) return fail(h, LGDSP_ERR_INVALID_ARG, "nothing to profile");
    // scratch for the whole batch in one piece
    const int64_t keepB = h->split_batch;
    const int keepS = h->split_streams;
    h->split_batch = n_events; h->split_streams = 1;
    const IcpcDev& D = h->icpc;
    rc = icpc_dispatch(h, D, d_wf, 2, n_events, ld_samples, nullptr, 1, 1.0, d_out_rows);   // sizes the scratch, warms up
    h->split_batch = keepB; h->split_streams = keepS;
    if (rc) return rc;
    cudaEvent_t marks[5];
    for (int i = 0; i < 5; ++i) CK(cudaEventCreate(&marks[i]));
    icpc_split_launch_batch(D, d_wf, 2, n_events, ld_samples, nullptr, 1, 1.0, d_out_rows, h->d_tt, h->d_saux, h->d_scz, h->split_bps,
                            h->sm_count, h->stream, nullptr, h->ev_pre[0], h->ev_cz[0], marks);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    const bool cz = (D.groups & LGDSP_GROUP_CUSPZAC) != 0;
    float t;
    CK(cudaEventElapsedTime(&t, marks[0], marks[1])); ms4[0] = t;
    CK(cudaEventElapsedTime(&t, marks[1], marks[2])); ms4[1] = t;
    ms4[2] = ms4[3] = 0.0;
    if (cz) {
        CK(cudaEventElapsedTime(&t, marks[2], marks[3])); ms4[2] = t;
        if (!D.direct) { CK(cudaEventElapsedTime(&t, marks[3], marks[4])); ms4[3] = t; }
    }
    for (int i = 0; i < 5; ++i) cudaEventDestroy(marks[i]);
    h->launches += cz ? 4 : 2;
    return LGDSP_OK;
}

/* pinned host memory for callers that want the direct (unstaged) copy path of the host entry points */
int lgdsp_host_alloc(void** p, int64_t bytes)
{
    if (!p || bytes < 0) return LGDSP_ERR_INVALID_ARG;
    return cudaHostAlloc(p, (size_t)bytes, cudaHostAllocDefault) == cudaSuccess ? LGDSP_OK : LGDSP_ERR_OOM;
}
int lgdsp_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? LGDSP_OK : LGDSP_ERR_CUDA; }
int lgdsp_host_register(void* p, int64_t bytes)
{
    if (!p || bytes <= 0) return LGDSP_ERR_INVALID_ARG;
    return cudaHostRegister(p, (size_t)bytes, cudaHostRegisterDefault) == cudaSuccess ? LGDSP_OK : LGDSP_ERR_CUDA;
}
int lgdsp_host_unregister(void* p) { return cudaHostUnregister(p) == cudaSuccess ? LGDSP_OK : LGDSP_ERR_CUDA; }

int lgdsp_icpc_run_device(lgdsp_handle* h, const lgdsp_icpc_params* p, const uint16_t* d_wf, int64_t n_events,
                          int64_t ld_samples, double* d_out_rows)
{
    return icpc_run_device_impl(h, p, d_wf, 2, nullptr, n_events, ld_samples, d_out_rows);
}

int lgdsp_icpc_run_ext_device(lgdsp_handle* h, const lgdsp_icpc_params* p, const void* d_wf, int32_t sample_bytes,
                              const double* d_baseline, int64_t n_events, int64_t ld_samples, double* d_out_rows)
{
    return icpc_run_device_impl(h, p, d_wf, sample_bytes, d_baseline, n_events, ld_samples, d_out_rows);
}

// ---------------------------------------------------------------------------------------------------
// Host <-> device traffic of the chunked host paths.  Caller memory that is already page-locked (cudaHostAlloc /
// cudaHostRegister / torch pin_memory) is copied directly; PAGEABLE caller memory (a Julia `flatview(wvfs.signal)`, a numpy
// array) is first packed into the handle's pinned double buffers by a few threads, so that the H2D copy of chunk k+1 and the
// D2H copy of chunk k-1 still run asynchronously beside the kernels of chunk k.  (A cudaMemcpyAsync straight from pageable
// memory is a blocking staged copy: the overlap the pipeline depends on would be gone.)
// ---------------------------------------------------------------------------------------------------
static bool is_pinned(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// dst[r*dpitch .. +width) = src[r*spitch .. +width), rows split over a few threads
static void pack_rows(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t rows, int threads)
{
    const size_t total = width * rows;
    if (threads > 1 && total < ((size_t)4 << 20)) threads = 1;
    if (rows < (size_t)threads && !(dpitch == width && spitch == width)) threads = rows ? (int)rows : 1;
    auto work = [=](int t) {
        if (dpitch == width && spitch == width) {   // dense: split the bytes
            const size_t a0 = total * t / threads, a1 = total * (t + 1) / threads;
            memcpy(static_cast<char*>(dst) + a0, static_cast<const char*>(src) + a0, a1 - a0);
        } else {
            const size_t r0 = rows * t / threads, r1 = rows * (t + 1) / threads;
            for (size_t r = r0; r < r1; ++r)
                memcpy(static_cast<char*>(dst) + r * dpitch, static_cast<const char*>(src) + r * spitch, width);
        }
    };
    if (threads <= 1) { work(0); return; }
    std::vector<std::thread> th;
    th.reserve(threads - 1);
    for (int t = 1; t < threads; ++t) th.emplace_back(work, t);
    work(0);
    for (auto& x : th) x.join();
}

struct HostIO {
    lgdsp_handle* h;
    int b = 0;                 // double-buffer index of the current chunk
    size_t in_used = 0, out_used = 0;
    struct Pending { void* dst; size_t dpitch; const void* src; size_t width, rows; };
    std::vector<Pending> pending[2];   // pinned -> caller copies that wait for ev_out[b]
    bool used_pin[2] = {false, false}, used_out[2] = {false, false};

    explicit HostIO(lgdsp_handle* hh) : h(hh) {}

    // capacity of the two pinned staging areas per chunk (grown on demand; growing synchronises)
    int reserve(size_t in_bytes, size_t out_bytes)
    {
        if (in_bytes > h->pin_cap) {
            CK(cudaStreamSynchronize(h->s_copy));
            for (int i = 0; i < 2; ++i) { if (h->h_pin[i]) cudaFreeHost(h->h_pin[i]); h->h_pin[i] = nullptr; }
            h->pin_cap = 0;
            for (int i = 0; i < 2; ++i) CK(cudaHostAlloc(&h->h_pin[i], in_bytes, cudaHostAllocDefault));
            h->pin_cap = in_bytes;
        }
        if (out_bytes > h->out_cap) {
            CK(cudaStreamSynchronize(h->stream));
            for (int i = 0; i < 2; ++i) { if (h->h_out[i]) cudaFreeHost(h->h_out[i]); h->h_out[i] = nullptr; }
            h->out_cap = 0;
            for (int i = 0; i < 2; ++i) CK(cudaHostAlloc(&h->h_out[i], out_bytes, cudaHostAllocDefault));
            h->out_cap = out_bytes;
        }
        return LGDSP_OK;
    }
    int flush(int bb)
    {
        if (used_out[bb]) { CK(cudaEventSynchronize(h->ev_out[bb])); used_out[bb] = false; }
        for (const Pending& q : pending[bb]) pack_rows(q.dst, q.dpitch, q.src, q.width, q.width, q.rows, h->copy_threads);
        pending[bb].clear();
        return LGDSP_OK;
    }
    // chunk c starts: its staging buffers must be free again (the copies of chunk c-2 that used them are done)
    int begin_chunk(int c)
    {
        b = c & 1;
        in_used = out_used = 0;
        if (used_pin[b]) { CK(cudaEventSynchronize(h->ev_pin[b])); used_pin[b] = false; }
        return flush(b);
    }
    static size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }
    // rows of `width` bytes (source pitch `spitch`) -> dense device rows, on the copy stream
    int h2d(void* d_dst, const void* src, size_t spitch, size_t width, size_t rows, bool src_pinned)
    {
        if (width == 0 || rows == 0) return LGDSP_OK;
        if (src_pinned) {
            if (spitch == width) CK(cudaMemcpyAsync(d_dst, src, width * rows, cudaMemcpyHostToDevice, h->s_copy));
            else CK(cudaMemcpy2DAsync(d_dst, width, src, spitch, width, rows, cudaMemcpyHostToDevice, h->s_copy));
            return LGDSP_OK;
        }
        const size_t bytes = width * rows;
        if (in_used + bytes > h->pin_cap) return fail(h, LGDSP_ERR_CUDA, "internal: pinned input staging too small");
        char* stage = static_cast<char*>(h->h_pin[b]) + in_used;
        pack_rows(stage, width, src, spitch, width, rows, h->copy_threads);
        in_used = up256(in_used + bytes);
        CK(cudaMemcpyAsync(d_dst, stage, bytes, cudaMemcpyHostToDevice, h->s_copy));
        used_pin[b] = true;
        return LGDSP_OK;
    }
    // every H2D copy of the chunk is issued: the compute stream waits for them
    int inputs_ready()
    {
        CK(cudaEventRecord(h->ev_ready[b], h->s_copy));
        if (used_pin[b]) CK(cudaEventRecord(h->ev_pin[b], h->s_copy));
        CK(cudaStreamWaitEvent(h->stream, h->ev_ready[b], 0));
        return LGDSP_OK;
    }
    // dense device rows of `width` bytes -> caller rows `dpitch` bytes apart, in stream order behind the kernels of this chunk
    int d2h(void* dst, size_t dpitch, const void* d_src, size_t width, size_t rows, bool dst_pinned)
    {
        if (width == 0 || rows == 0) return LGDSP_OK;
        if (dst_pinned) {
            if (dpitch == width) CK(cudaMemcpyAsync(dst, d_src, width * rows, cudaMemcpyDeviceToHost, h->stream));
            else CK(cudaMemcpy2DAsync(dst, dpitch, d_src, width, width, rows, cudaMemcpyDeviceToHost, h->stream));
            return LGDSP_OK;
        }
        const size_t bytes = width * rows;
        if (out_used + bytes > h->out_cap) return fail(h, LGDSP_ERR_CUDA, "internal: pinned output staging too small");
        char* stage = static_cast<char*>(h->h_out[b]) + out_used;
        out_used = up256(out_used + bytes);
        CK(cudaMemcpyAsync(stage, d_src, bytes, cudaMemcpyDeviceToHost, h->stream));
        pending[b].push_back({dst, dpitch, stage, width, rows});
        used_out[b] = true;
        return LGDSP_OK;
    }
    int end_chunk()
    {
        if (used_out[b]) CK(cudaEventRecord(h->ev_out[b], h->stream));
        return LGDSP_OK;
    }
    int finish()
    {
        CK(cudaStreamSynchronize(h->s_copy));
        CK(cudaStreamSynchronize(h->stream));
        used_pin[0] = used_pin[1] = false;
        int rc = flush(0);
        return rc ? rc : flush(1);
    }
};

// One encoded stream set of a chunk -> decoded device rows: upload of the byte range and of the offsets slice (copy stream),
// decode kernel (compute stream, behind inputs_ready).  `slot` = 0 / 1: the input index (dsp_icpc_compressed has two).
struct EncodedInput {
    int codec, sample_bytes, n_samples, shift;
    const uint8_t* enc;
    const int64_t* offsets;
    bool enc_pinned, off_pinned;
};
// device buffers of one encoded input; adds what its uploads take of the pinned input staging to *stage_in
static int encoded_reserve(lgdsp_handle* h, const EncodedInput& in, int slot, int64_t chunk, int64_t n_events, size_t* stage_in)
{
    size_t max_bytes = 0;   // the longest byte range of one chunk
    for (int64_t e0 = 0; e0 < n_events; e0 += chunk)
        max_bytes = std::max(max_bytes, (size_t)(in.offsets[std::min(e0 + chunk, n_events)] - in.offsets[e0]));
    if (!in.enc_pinned || !in.off_pinned) *stage_in += max_bytes + (size_t)(chunk + 1) * sizeof(int64_t) + 512;
    int rc = LGDSP_OK;
    for (int b = 0; b < 2 && !rc; ++b) {
        rc = grow(h, &h->d_enc[b][slot], &h->enc_cap[b][slot], max_bytes + 16);
        if (!rc) rc = grow(h, &h->d_off[b][slot], &h->off_cap[b][slot], (size_t)(chunk + 1) * sizeof(long long));
    }
    if (!rc) rc = grow(h, &h->d_dec[slot], &h->dec_cap[slot], (size_t)chunk * in.n_samples * in.sample_bytes);
    return rc ? rc : grow(h, &h->d_dstat, &h->dstat_cap, 2 * sizeof(int));
}
// d_dstat = {number of malformed streams, smallest event index among them} of the running call
static int decode_err_reset(lgdsp_handle* h)
{
    const int init[2] = {0, 0x7fffffff};
    CK(cudaMemcpyAsync(h->d_dstat, init, sizeof(init), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return LGDSP_OK;
}
static int decode_err_check(lgdsp_handle* h)
{
    int st[2] = {0, 0};
    CK(cudaMemcpy(st, h->d_dstat, sizeof(st), cudaMemcpyDeviceToHost));
    if (st[0]) return fail(h, LGDSP_ERR_INVALID_ARG, "%d malformed encoded waveform(s), first at event %d", st[0], st[1]);
    return LGDSP_OK;
}
static int encoded_upload(lgdsp_handle* h, HostIO& io, const EncodedInput& in, int slot, int64_t e0, int64_t ne)
{
    const size_t nb = (size_t)(in.offsets[e0 + ne] - in.offsets[e0]);
    int rc = io.h2d(h->d_enc[io.b][slot], in.enc + in.offsets[e0], nb, nb, nb ? 1 : 0, in.enc_pinned);
    if (rc) return rc;
    return io.h2d(h->d_off[io.b][slot], in.offsets + e0, (size_t)(ne + 1) * sizeof(int64_t), (size_t)(ne + 1) * sizeof(int64_t), 1,
                  in.off_pinned);
}
static int encoded_decode(lgdsp_handle* h, HostIO& io, const EncodedInput& in, int slot, int64_t e0, int64_t ne)
{
    long long longest = 0;   // sizes the decoder's per-warp stream buffers
    for (int64_t k = e0; k < e0 + ne; ++k) {
        const long long nb = (long long)(in.offsets[k + 1] - in.offsets[k]);
        longest = nb > longest ? nb : longest;
    }
    cudaError_t e = codec_decode_launch(in.codec, h->d_enc[io.b][slot], h->d_off[io.b][slot], (long long)in.offsets[e0], ne, in.n_samples,
                                        in.shift, h->d_dec[slot], in.sample_bytes, in.n_samples, nullptr, h->d_dstat, (int)e0, longest,
                                        h->sm_count, h->stream);
    if (e != cudaSuccess) return fail(h, LGDSP_ERR_CUDA, "decode kernel: %s", cudaGetErrorString(e));
    h->launches += 1;
    return LGDSP_OK;
}
static int check_encoded(lgdsp_handle* h, int codec, const void* enc, const int64_t* offsets, int64_t n_events, int sample_bytes)
{
    if (codec != LGDSP_CODEC_RADWARE && codec != LGDSP_CODEC_ULEB128ZZD) return fail(h, LGDSP_ERR_UNSUPPORTED, "unknown codec %d", codec);
    if (codec == LGDSP_CODEC_RADWARE && sample_bytes != 2) return fail(h, LGDSP_ERR_UNSUPPORTED, "RadwareSigcompress holds 16-bit samples");
    if (sample_bytes != 2 && sample_bytes != 4) return fail(h, LGDSP_ERR_UNSUPPORTED, "sample_bytes = %d", sample_bytes);
    if (n_events > 0 && (!enc || !offsets)) return fail(h, LGDSP_ERR_INVALID_ARG, "encoded data / offsets pointer is NULL");
    for (int64_t e = 0; e < n_events; ++e)
        if (offsets[e + 1] < offsets[e]) return fail(h, LGDSP_ERR_INVALID_ARG, "offsets must be non-decreasing (event %lld)", (long long)e);
    return LGDSP_OK;
}
// One per-event array of caller memory that a host entry point moves: `width` bytes per event, `pitch` bytes from one event to
// the next in caller memory, dense rows on the device (the TMA and the 128-bit loads of the kernels rely on that).
// host == NULL: an optional array that is not given; its device pointer is NULL.
struct HostArray {
    const void* host;
    size_t pitch, width;
    bool pinned;
    const EncodedInput* enc;   // input given as encoded streams (decode_data on the device in front of the launch)
    int from_input;            // output whose device rows are those of this input (no device buffer of its own), else -1
};
static HostArray host_array(const void* p, size_t pitch, size_t width)
{
    return HostArray{p, pitch, width, p && is_pinned(p), nullptr, -1};
}
static HostArray wf_array(const void* wf, size_t pitch, size_t width, const EncodedInput* enc)
{
    return enc ? HostArray{nullptr, 0, 0, false, enc, -1} : host_array(wf, pitch, width);
}

// The chunk loop of every host entry point.  The inputs of chunk c go up on the copy stream while the compute stream runs
// chunk c-1; the compute stream waits for them, decodes encoded inputs, runs launch(ne, d) and copies the outputs back.
// d[k] holds the device rows of input k, then of output k - in.size(), in double-buffered slots of the handle.
typedef std::function<int(int64_t ne, void* const* d)> ChunkLaunch;
static int run_chunked(lgdsp_handle* h, int64_t n_events, int64_t chunk, const std::vector<HostArray>& in,
                       const std::vector<HostArray>& out, const ChunkLaunch& launch)
{
    chunk = std::min(chunk, n_events);
    const size_t ni = in.size(), na = ni + out.size();
    if (na > LGDSP_HOST_ARRAYS) return fail(h, LGDSP_ERR_CUDA, "internal: %zu host arrays", na);
    HostIO io(h);
    size_t stage_in = 0, stage_out = 0;
    bool encoded = false;
    int rc = LGDSP_OK;
    for (size_t k = 0; k < na && !rc; ++k) {
        const HostArray& a = k < ni ? in[k] : out[k - ni];
        if (a.enc) {
            encoded = true;
            rc = encoded_reserve(h, *a.enc, (int)k, chunk, n_events, &stage_in);
        } else if (a.host) {
            if (!a.pinned) (k < ni ? stage_in : stage_out) += (size_t)chunk * a.width + 256;
            for (int b = 0; b < 2 && !rc && a.from_input < 0; ++b) rc = grow(h, &h->d_slot[b][k], &h->slot_cap[b][k], (size_t)chunk * a.width);
        }
    }
    if (!rc) rc = io.reserve(stage_in, stage_out);
    if (!rc && encoded) rc = decode_err_reset(h);
    if (rc) return rc;
    void* d[LGDSP_HOST_ARRAYS];
    int c = 0;
    for (int64_t e0 = 0; e0 < n_events; e0 += chunk, ++c) {
        const int64_t ne = std::min(chunk, n_events - e0);
        rc = io.begin_chunk(c);
        if (rc) return rc;
        const int b = io.b;
        if (c >= 2) CK(cudaStreamWaitEvent(h->s_copy, h->ev_free[b], 0));   // the device buffers of chunk c-2 are consumed
        for (size_t k = 0; k < na; ++k) {
            const HostArray& a = k < ni ? in[k] : out[k - ni];
            d[k] = a.enc ? h->d_dec[k] : a.from_input >= 0 ? d[a.from_input] : a.host ? h->d_slot[b][k] : nullptr;
            if (k >= ni) continue;
            if (a.enc) rc = encoded_upload(h, io, *a.enc, (int)k, e0, ne);
            else if (a.host) rc = io.h2d(d[k], static_cast<const char*>(a.host) + (size_t)e0 * a.pitch, a.pitch, a.width, (size_t)ne, a.pinned);
            if (rc) return rc;
        }
        rc = io.inputs_ready();
        if (rc) return rc;
        // (d_dec is single-buffered: what reads it -- the launch, or the D2H of decode_data -- is in stream order in front of
        // the next chunk's decode kernel)
        for (size_t k = 0; k < ni && !rc; ++k)
            if (in[k].enc) rc = encoded_decode(h, io, *in[k].enc, (int)k, e0, ne);
        if (!rc) rc = launch(ne, d);
        if (rc) return rc;
        CK(cudaEventRecord(h->ev_free[b], h->stream));
        for (size_t k = ni; k < na && !rc; ++k) {
            const HostArray& a = out[k - ni];
            if (a.host) rc = io.d2h(const_cast<char*>(static_cast<const char*>(a.host)) + (size_t)e0 * a.pitch, a.pitch, d[k], a.width,
                                    (size_t)ne, a.pinned);
        }
        if (!rc) rc = io.end_chunk();
        if (rc) return rc;
    }
    rc = io.finish();
    if (rc) return rc;
    return encoded ? decode_err_check(h) : LGDSP_OK;
}

// host buffers in, host rows out.  `encin` != NULL: the input is an encoded waveform set (decode_data on the device), else
// raw samples `wf`.
static int icpc_run_host_impl(lgdsp_handle* h, const lgdsp_icpc_params* p, const void* wf, int sample_bytes,
                              const double* baseline, int64_t n_events, int64_t ld_samples, double* out_rows,
                              EncodedInput* encin = nullptr)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (p) { int rc = icpc_prepare(h, p); if (rc) return rc; }
    if (!h->have_icpc) return fail(h, LGDSP_ERR_INVALID_ARG, "no parameters set");
    const int n = h->icpc.n;
    int rc;
    if (encin) {
        encin->n_samples = n;
        if (n_events < 0) return fail(h, LGDSP_ERR_INVALID_ARG, "n_events < 0");
        if (sample_bytes == 4 && n > LGDSP_MAX_SAMPLES / 2) return fail(h, LGDSP_ERR_UNSUPPORTED, "32-bit samples: n_samples = %d > %d", n, LGDSP_MAX_SAMPLES / 2);
        rc = check_encoded(h, encin->codec, encin->enc, encin->offsets, n_events, sample_bytes);
    } else {
        rc = check_wf(h, wf, n_events, ld_samples, n, false, sample_bytes);
    }
    if (rc) return rc;
    if (n_events == 0) return LGDSP_OK;
    if (!out_rows) return fail(h, LGDSP_ERR_INVALID_ARG, "output pointer is NULL");
    const HostArray wf_in = wf_array(wf, (size_t)ld_samples * sample_bytes, (size_t)n * sample_bytes, encin);
    // raw samples straight from page-locked memory are bound by the host link: smaller chunks shorten the un-overlapped first
    // copy / last kernel (3.25 vs 3.13 M wf/s); staged and encoded input prefers the larger chunk (2.27 vs 1.76 M wf/s pageable)
    const int64_t chunk = (wf_in.pinned && h->host_chunk_direct < h->host_chunk) ? h->host_chunk_direct : h->host_chunk;
    const size_t row = LGDSP_NCOL * sizeof(double);
    return run_chunked(h, n_events, chunk, {wf_in, host_array(baseline, sizeof(double), sizeof(double))}, {host_array(out_rows, row, row)},
                       [&](int64_t ne, void* const* d) {
                           return icpc_dispatch(h, h->icpc, d[0], sample_bytes, ne, n, static_cast<const double*>(d[1]), 1, 1.0,
                                                static_cast<double*>(d[2]));
                       });
}

int lgdsp_icpc_run(lgdsp_handle* h, const lgdsp_icpc_params* p, const uint16_t* wf, int64_t n_events,
                   int64_t ld_samples, double* out_rows)
{
    return icpc_run_host_impl(h, p, wf, 2, nullptr, n_events, ld_samples, out_rows);
}

int lgdsp_icpc_run_ext(lgdsp_handle* h, const lgdsp_icpc_params* p, const void* wf, int32_t sample_bytes,
                       const double* baseline, int64_t n_events, int64_t ld_samples, double* out_rows)
{
    return icpc_run_host_impl(h, p, wf, sample_bytes, baseline, n_events, ld_samples, out_rows);
}

// ---- decode_data (LegendDataTypes.jl codecs; /root/reference/src/dsp_icpc.jl:313-314) ----
int64_t lgdsp_codec_max_encoded_bytes(int32_t codec, int32_t n_samples, int32_t sample_bytes)
{
    if ((codec != LGDSP_CODEC_RADWARE && codec != LGDSP_CODEC_ULEB128ZZD) || n_samples < 0) return -1;
    return codec_max_encoded_bytes(codec, n_samples, sample_bytes);
}

int lgdsp_codec_encode_host(int32_t codec, const void* wf, int32_t sample_bytes, int64_t n_events, int32_t n_samples, int64_t ld_samples,
                            int32_t shift, uint8_t* enc, int64_t enc_capacity, int64_t* offsets)
{
    if ((codec != LGDSP_CODEC_RADWARE && codec != LGDSP_CODEC_ULEB128ZZD) || !offsets || n_events < 0 || n_samples < 0 ||
        (n_events > 0 && (!wf || !enc)) || ld_samples < n_samples || (sample_bytes != 2 && sample_bytes != 4) ||
        (codec == LGDSP_CODEC_RADWARE && (sample_bytes != 2 || n_samples > 65535)))
        return LGDSP_ERR_INVALID_ARG;
    static_assert(sizeof(long long) == sizeof(int64_t), "offset type");
    const int rc = codec_encode_host(codec, wf, sample_bytes, n_events, n_samples, ld_samples, shift, enc, enc_capacity,
                                     reinterpret_cast<long long*>(offsets));
    return rc == 0 ? LGDSP_OK : (rc == -1 ? LGDSP_ERR_OOM : LGDSP_ERR_INVALID_ARG);
}

int lgdsp_decode_data_device(lgdsp_handle* h, int32_t codec, const uint8_t* d_enc, const int64_t* d_offsets, int64_t n_events,
                             int32_t n_samples, int32_t shift, void* d_wf, int32_t sample_bytes, int64_t ld_samples, int32_t* d_status)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (codec != LGDSP_CODEC_RADWARE && codec != LGDSP_CODEC_ULEB128ZZD) return fail(h, LGDSP_ERR_UNSUPPORTED, "unknown codec %d", codec);
    if ((codec == LGDSP_CODEC_RADWARE && sample_bytes != 2) || (sample_bytes != 2 && sample_bytes != 4))
        return fail(h, LGDSP_ERR_UNSUPPORTED, "codec %d with %d-byte samples", codec, sample_bytes);
    if (n_events < 0 || n_samples < 1 || n_samples > LGDSP_MAX_SAMPLES || ld_samples < n_samples) return fail(h, LGDSP_ERR_INVALID_ARG, "bad sizes");
    if (n_events == 0) return LGDSP_OK;
    if (!d_enc || !d_offsets || !d_wf) return fail(h, LGDSP_ERR_INVALID_ARG, "NULL pointer");
    CK(cudaEventRecord(h->ev0, h->stream));
    cudaError_t e = codec_decode_launch(codec, d_enc, reinterpret_cast<const long long*>(d_offsets), 0, n_events, n_samples, shift, d_wf,
                                        sample_bytes, ld_samples, d_status, nullptr, 0, 0 /* offsets live on the device */, h->sm_count,
                                        h->stream);
    if (e != cudaSuccess) return fail(h, LGDSP_ERR_CUDA, "decode kernel: %s", cudaGetErrorString(e));
    CK(cudaEventRecord(h->ev1, h->stream));
    h->timed = true;
    h->launches += 1;
    return LGDSP_OK;
}

int lgdsp_decode_data(lgdsp_handle* h, int32_t codec, const uint8_t* enc, const int64_t* offsets, int64_t n_events, int32_t n_samples,
                      int32_t shift, void* wf, int32_t sample_bytes, int64_t ld_samples)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    int rc = check_encoded(h, codec, enc, offsets, n_events, sample_bytes);
    if (rc) return rc;
    if (n_events < 0 || n_samples < 1 || n_samples > LGDSP_MAX_SAMPLES || ld_samples < n_samples) return fail(h, LGDSP_ERR_INVALID_ARG, "bad sizes");
    if (n_events == 0) return LGDSP_OK;
    if (!wf) return fail(h, LGDSP_ERR_INVALID_ARG, "output pointer is NULL");
    EncodedInput in{codec, sample_bytes, n_samples, shift, enc, offsets, is_pinned(enc), is_pinned(offsets)};
    // the output is the decoded rows themselves: nothing to launch
    HostArray rows = host_array(wf, (size_t)ld_samples * sample_bytes, (size_t)n_samples * sample_bytes);
    rows.from_input = 0;
    return run_chunked(h, n_events, 8192, {wf_array(nullptr, 0, 0, &in)}, {rows}, [](int64_t, void* const*) { return (int)LGDSP_OK; });
}

// dsp_icpc on ENCODED waveforms: the host link carries the codec's bytes, decode_data runs on the device in front of the chain
int lgdsp_icpc_run_encoded(lgdsp_handle* h, const lgdsp_icpc_params* p, int32_t codec, const uint8_t* enc, const int64_t* offsets,
                           int32_t shift, int32_t sample_bytes, const double* baseline, int64_t n_events, double* out_rows)
{
    EncodedInput in{codec, sample_bytes, 0, shift, enc, offsets, enc ? is_pinned(enc) : false, offsets ? is_pinned(offsets) : false};
    return icpc_run_host_impl(h, p, nullptr, sample_bytes, baseline, n_events, 0, out_rows, &in);
}

// the checks lgdsp_window_stats_run and _run_device share (nothing to do when n_events or n_windows is 0)
static int window_stats_check(lgdsp_handle* h, const void* wf, int sample_bytes, int64_t n_events, int n_samples, int64_t ld_samples,
                              double t_first_ns, double dt_ns, const int32_t* windows, int n_windows, const double* out)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (sample_bytes != 2 && sample_bytes != 4) return fail(h, LGDSP_ERR_UNSUPPORTED, "sample_bytes = %d", sample_bytes);
    if (n_events < 0 || n_windows < 0 || n_windows > LGDSP_MAX_STAT_WINDOWS) return fail(h, LGDSP_ERR_INVALID_ARG, "bad n_events / n_windows");
    if (n_events == 0 || n_windows == 0) return LGDSP_OK;
    if (!wf || !windows || !out) return fail(h, LGDSP_ERR_INVALID_ARG, "NULL pointer");
    if (n_samples < 1 || ld_samples < n_samples) return fail(h, LGDSP_ERR_INVALID_ARG, "bad n_samples / ld_samples");
    if (!(dt_ns > 0) || !std::isfinite(t_first_ns)) return fail(h, LGDSP_ERR_INVALID_ARG, "bad time axis");
    for (int w = 0; w < n_windows; ++w) {
        const int a = windows[2 * w], b = windows[2 * w + 1];
        // @assert firstindex(X) <= first(idxs) <= last(idxs) <= lastindex(X)   /root/reference/src/tailstats.jl:23-25
        if (!(0 <= a && a <= b && b <= n_samples - 1)) return fail(h, LGDSP_ERR_INVALID_ARG, "window %d (%d:%d) outside the waveform", w, a, b);
    }
    return LGDSP_OK;
}

// signalstats on n_windows windows of every waveform (optionally shifted by -shift[e]): out double[n_events][n_windows][5]
int lgdsp_window_stats_run_device(lgdsp_handle* h, const void* d_wf, int32_t sample_bytes, int64_t n_events, int32_t n_samples,
                                  int64_t ld_samples, double t_first_ns, double dt_ns, const double* d_shift,
                                  const int32_t* windows, int32_t n_windows, double* d_out)
{
    int rc = window_stats_check(h, d_wf, sample_bytes, n_events, n_samples, ld_samples, t_first_ns, dt_ns, windows, n_windows, d_out);
    if (rc || n_events == 0 || n_windows == 0) return rc;
    CK(cudaMemcpyAsync(h->d_win, windows, sizeof(int) * 2 * (size_t)n_windows, cudaMemcpyHostToDevice, h->stream));
    CK(cudaEventRecord(h->ev0, h->stream));
    window_stats_launch(d_wf, sample_bytes, n_events, ld_samples, t_first_ns, dt_ns, d_shift, 1, 0xFFFFFFFFu, h->d_win, n_windows, d_out, h->stream);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev1, h->stream));
    h->timed = true;
    h->launches += 1;
    // the window list is read from pageable host memory by the async copy: make sure it is consumed before returning
    CK(cudaStreamSynchronize(h->stream));
    return LGDSP_OK;
}

int lgdsp_window_stats_run(lgdsp_handle* h, const void* wf, int32_t sample_bytes, int64_t n_events, int32_t n_samples,
                           int64_t ld_samples, double t_first_ns, double dt_ns, const double* shift,
                           const int32_t* windows, int32_t n_windows, double* out)
{
    int rc = window_stats_check(h, wf, sample_bytes, n_events, n_samples, ld_samples, t_first_ns, dt_ns, windows, n_windows, out);
    if (rc || n_events == 0 || n_windows == 0) return rc;
    // (run_chunked synchronises the stream before it returns: the window list is consumed by then)
    CK(cudaMemcpyAsync(h->d_win, windows, sizeof(int) * 2 * (size_t)n_windows, cudaMemcpyHostToDevice, h->stream));
    const size_t sb = (size_t)sample_bytes, out_per = (size_t)n_windows * 5 * sizeof(double);
    return run_chunked(h, n_events, 8192, {host_array(wf, (size_t)ld_samples * sb, (size_t)n_samples * sb), host_array(shift, sizeof(double), sizeof(double))},
                       {host_array(out, out_per, out_per)}, [&](int64_t ne, void* const* d) {
                           window_stats_launch(d[0], sample_bytes, ne, n_samples, t_first_ns, dt_ns, static_cast<const double*>(d[1]), 1,
                                               0xFFFFFFFFu, h->d_win, n_windows, static_cast<double*>(d[2]), h->stream);
                           CK(cudaGetLastError());
                           h->launches += 1;
                           return (int)LGDSP_OK;
                       });
}

// ---- dsp_icpc_compressed: presummed + windowed waveform per event (/root/reference/src/dsp_icpc.jl:293-499) ----
static int compressed_prepare(lgdsp_handle* h, const lgdsp_icpc_params* p_pre, const lgdsp_icpc_params* p_wdw, int pre_bytes,
                              int wdw_bytes, double presum_rate, const int32_t* aux)
{
    if (p_pre) { int rc = icpc_prepare(h, p_pre, 0); if (rc) return rc; }
    if (p_wdw) { int rc = icpc_prepare(h, p_wdw, 1); if (rc) return rc; }
    if (!h->have_icpc || !h->have_icpc_w) return fail(h, LGDSP_ERR_INVALID_ARG, "dsp_icpc_compressed: parameters of both waveforms are needed");
    if (!(presum_rate >= 1.0)) return fail(h, LGDSP_ERR_INVALID_ARG, "presum_rate must be >= 1");
    if ((pre_bytes != 2 && pre_bytes != 4) || (wdw_bytes != 2 && wdw_bytes != 4))
        return fail(h, LGDSP_ERR_UNSUPPORTED, "sample_bytes: uint16 (2) or uint32 (4) samples");
    if (!aux) return fail(h, LGDSP_ERR_INVALID_ARG, "aux_windows is NULL");
    const int n = h->icpc.n;
    for (int w = 0; w < 4; ++w) {
        const int a = aux[2 * w], b = aux[2 * w + 1];
        if (!(0 <= a && a <= b && b <= n - 1)) return fail(h, LGDSP_ERR_INVALID_ARG, "auxiliary window %d (%d:%d) outside the presummed waveform", w, a, b);
    }
    // window order of the statistics output: auxbl1, auxbl2, bl_window (raw), auxpz1, auxpz2 (baseline-subtracted)
    const int win[10] = {aux[0], aux[1], aux[2], aux[3], h->icpc.bl_from, h->icpc.bl_until, aux[4], aux[5], aux[6], aux[7]};
    CK(cudaMemcpyAsync(h->d_win, win, sizeof(win), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return LGDSP_OK;
}

// the three launches of one batch, in stream order
static int compressed_launch(lgdsp_handle* h, const void* d_pre, int pre_bytes, int64_t ld_pre, const void* d_wdw, int wdw_bytes,
                              int64_t ld_wdw, double presum_rate, int64_t ne, double* d_rows_pre, double* d_rows_wdw, double* d_stats)
{
    // :332-346, :356-375, :383, :397-428, :439-455 on the presummed waveform
    int rc = icpc_dispatch(h, h->icpc, d_pre, pre_bytes, ne, ld_pre, nullptr, 1, 1.0, d_rows_pre);
    if (rc) return rc;
    // :338-339, :346 (slope_residual_sigma), :365-366: windows 3, 4 are shifted by the baseline mean of the first launch
    window_stats_launch(d_pre, pre_bytes, ne, ld_pre, h->icpc.t_first, h->icpc.dt, d_rows_pre + LGDSP_COL_blmean, LGDSP_NCOL, 0x18u,
                        h->d_win, 5, d_stats, h->stream);
    // :350 the windowed waveform is shifted by -blmean / presum_rate; :378-394, :431-435, :458
    rc = icpc_dispatch(h, h->icpc_w, d_wdw, wdw_bytes, ne, ld_wdw, d_rows_pre + LGDSP_COL_blmean, LGDSP_NCOL, presum_rate, d_rows_wdw);
    if (rc) return rc;
    h->launches += 1;
    return LGDSP_OK;
}

int lgdsp_icpc_compressed_run_device(lgdsp_handle* h, const lgdsp_icpc_params* p_pre, const lgdsp_icpc_params* p_wdw,
                                     const void* d_wf_pre, int32_t pre_sample_bytes, int64_t ld_pre, const void* d_wf_wdw,
                                     int32_t wdw_sample_bytes, int64_t ld_wdw, double presum_rate, const int32_t* aux_windows,
                                     int64_t n_events, double* d_rows_pre, double* d_rows_wdw, double* d_stats)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    int rc = compressed_prepare(h, p_pre, p_wdw, pre_sample_bytes, wdw_sample_bytes, presum_rate, aux_windows);
    if (rc) return rc;
    rc = check_wf(h, d_wf_pre, n_events, ld_pre, h->icpc.n, true, pre_sample_bytes);
    if (rc) return rc;
    rc = check_wf(h, d_wf_wdw, n_events, ld_wdw, h->icpc_w.n, true, wdw_sample_bytes);
    if (rc) return rc;
    if (n_events == 0) return LGDSP_OK;
    if (!d_rows_pre || !d_rows_wdw || !d_stats) return fail(h, LGDSP_ERR_INVALID_ARG, "output pointer is NULL");
    CK(cudaEventRecord(h->ev0, h->stream));
    rc = compressed_launch(h, d_wf_pre, pre_sample_bytes, ld_pre, d_wf_wdw, wdw_sample_bytes, ld_wdw, presum_rate, n_events, d_rows_pre,
                           d_rows_wdw, d_stats);
    if (rc) return rc;
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev1, h->stream));
    h->timed = true;
    return LGDSP_OK;
}

// host buffers: raw samples (wf_* != NULL) or encoded waveform sets (enc_* != NULL) per waveform kind
static int compressed_run_host_impl(lgdsp_handle* h, const lgdsp_icpc_params* p_pre, const lgdsp_icpc_params* p_wdw, const void* wf_pre,
                                    int pre_sample_bytes, int64_t ld_pre, const void* wf_wdw, int wdw_sample_bytes, int64_t ld_wdw,
                                    EncodedInput* enc_pre, EncodedInput* enc_wdw, double presum_rate,
                                    const int32_t* aux_windows, int64_t n_events, double* rows_pre, double* rows_wdw, double* stats)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    int rc = compressed_prepare(h, p_pre, p_wdw, pre_sample_bytes, wdw_sample_bytes, presum_rate, aux_windows);
    if (rc) return rc;
    const int np = h->icpc.n, nw = h->icpc_w.n;
    if (enc_pre) { enc_pre->n_samples = np; rc = check_encoded(h, enc_pre->codec, enc_pre->enc, enc_pre->offsets, n_events, pre_sample_bytes); }
    else rc = check_wf(h, wf_pre, n_events, ld_pre, np, false, pre_sample_bytes);
    if (rc) return rc;
    if (enc_wdw) { enc_wdw->n_samples = nw; rc = check_encoded(h, enc_wdw->codec, enc_wdw->enc, enc_wdw->offsets, n_events, wdw_sample_bytes); }
    else rc = check_wf(h, wf_wdw, n_events, ld_wdw, nw, false, wdw_sample_bytes);
    if (rc) return rc;
    if (n_events < 0) return fail(h, LGDSP_ERR_INVALID_ARG, "n_events < 0");
    if (n_events == 0) return LGDSP_OK;
    if (!rows_pre || !rows_wdw || !stats) return fail(h, LGDSP_ERR_INVALID_ARG, "output pointer is NULL");
    const size_t sbp = (size_t)pre_sample_bytes, sbw = (size_t)wdw_sample_bytes;
    const size_t row = LGDSP_NCOL * sizeof(double), st = 5 * LGDSP_NSTAT * sizeof(double);
    return run_chunked(h, n_events, h->host_chunk,
                       {wf_array(wf_pre, (size_t)ld_pre * sbp, (size_t)np * sbp, enc_pre), wf_array(wf_wdw, (size_t)ld_wdw * sbw, (size_t)nw * sbw, enc_wdw)},
                       {host_array(rows_pre, row, row), host_array(rows_wdw, row, row), host_array(stats, st, st)},
                       [&](int64_t ne, void* const* d) {
                           int rc = compressed_launch(h, d[0], pre_sample_bytes, np, d[1], wdw_sample_bytes, nw, presum_rate, ne,
                                                      static_cast<double*>(d[2]), static_cast<double*>(d[3]), static_cast<double*>(d[4]));
                           if (rc) return rc;
                           CK(cudaGetLastError());
                           return (int)LGDSP_OK;
                       });
}

int lgdsp_icpc_compressed_run(lgdsp_handle* h, const lgdsp_icpc_params* p_pre, const lgdsp_icpc_params* p_wdw, const void* wf_pre,
                              int32_t pre_sample_bytes, int64_t ld_pre, const void* wf_wdw, int32_t wdw_sample_bytes,
                              int64_t ld_wdw, double presum_rate, const int32_t* aux_windows, int64_t n_events, double* rows_pre,
                              double* rows_wdw, double* stats)
{
    return compressed_run_host_impl(h, p_pre, p_wdw, wf_pre, pre_sample_bytes, ld_pre, wf_wdw, wdw_sample_bytes, ld_wdw, nullptr, nullptr,
                                    presum_rate, aux_windows, n_events, rows_pre, rows_wdw, stats);
}

// dsp_icpc_compressed with decode_data on the device (/root/reference/src/dsp_icpc.jl:313-314): both waveform kinds arrive
// as encoded byte streams in host memory
int lgdsp_icpc_compressed_run_encoded(lgdsp_handle* h, const lgdsp_icpc_params* p_pre, const lgdsp_icpc_params* p_wdw,
                                      int32_t pre_codec, const uint8_t* enc_pre, const int64_t* off_pre, int32_t pre_shift,
                                      int32_t pre_sample_bytes, int32_t wdw_codec, const uint8_t* enc_wdw, const int64_t* off_wdw,
                                      int32_t wdw_shift, int32_t wdw_sample_bytes, double presum_rate, const int32_t* aux_windows,
                                      int64_t n_events, double* rows_pre, double* rows_wdw, double* stats)
{
    EncodedInput ep{pre_codec, pre_sample_bytes, 0, pre_shift, enc_pre, off_pre, enc_pre ? is_pinned(enc_pre) : false,
                    off_pre ? is_pinned(off_pre) : false};
    EncodedInput ew{wdw_codec, wdw_sample_bytes, 0, wdw_shift, enc_wdw, off_wdw, enc_wdw ? is_pinned(enc_wdw) : false,
                    off_wdw ? is_pinned(off_wdw) : false};
    return compressed_run_host_impl(h, p_pre, p_wdw, nullptr, pre_sample_bytes, 0, nullptr, wdw_sample_bytes, 0, &ep, &ew, presum_rate,
                                    aux_windows, n_events, rows_pre, rows_wdw, stats);
}

// ---------------------------------------------------------------------------------------------------
// trapezoid sweeps
// ---------------------------------------------------------------------------------------------------
// variants -> device table (filter taps are differenced onto the prefix sums TT and uploaded)
static int sweep_prepare(lgdsp_handle* h, const lgdsp_sweep_params* p, const lgdsp_sweep_variant* variants, int32_t nvar,
                         SweepDev& D)
{
    if (!p || !variants) return fail(h, LGDSP_ERR_INVALID_ARG, "sweep params/variants NULL");
    if (p->struct_size != sizeof(lgdsp_sweep_params) || p->version != LGDSP_PARAMS_VERSION)
        return fail(h, LGDSP_ERR_INVALID_ARG, "lgdsp_sweep_params: size/version mismatch");
    const int n = p->n_samples;
    if (n < 64 || n > LGDSP_MAX_SAMPLES || n % 8 != 0) return fail(h, LGDSP_ERR_UNSUPPORTED, "n_samples = %d unsupported", n);
    if (nvar < 1 || nvar > 1024) return fail(h, LGDSP_ERR_UNSUPPORTED, "n_variants = %d: need 1..1024", nvar);
    if (!(0 <= p->bl_from && p->bl_from <= p->bl_until && p->bl_until < n)) return fail(h, LGDSP_ERR_INVALID_ARG, "bl_window outside the waveform");
    const lgdsp_dni& d = p->sig_dni;
    if (!(d.degree >= 0 && d.degree <= LGDSP_MAX_DNI_DEG && d.n_w > d.degree && d.n_w <= LGDSP_MAX_DNI))
        return fail(h, LGDSP_ERR_UNSUPPORTED, "PolynomialDNI outside the supported range");
    if (p->tx_min_n < 1) return fail(h, LGDSP_ERR_INVALID_ARG, "tx_min_n < 1");
    std::vector<SweepVar> sv(nvar);
    std::vector<double> taps;            // all differenced tap arrays, back to back
    std::vector<size_t> tap_off(nvar, 0);
    for (int v = 0; v < nvar; ++v) {
        const lgdsp_sweep_variant& in = variants[v];
        SweepVar& o = sv[v];
        memset(&o, 0, sizeof(o));
        o.kind = in.kind;
        o.pick_ns = in.pickoff_ns;
        o.mode = in.pickoff_mode;
        if (in.kind == 0) {
            if (!make_trap(in.trap, n, d.n_w, o.t))
                return fail(h, LGDSP_ERR_INVALID_ARG, "variant %d: trapezoid (%d,%d,%d) leaves fewer outputs than the DNI window", v,
                            in.trap.navg, in.trap.ngap, in.trap.navg2);
            o.L = o.t.L;
        } else if (in.kind == 1) {
            const int L = in.n_taps;
            if (!in.coeffs || L < 2 || L > LGDSP_MAX_FIR || n - L + 1 < d.n_w)
                return fail(h, LGDSP_ERR_INVALID_ARG, "variant %d: FIR with %d taps does not fit (need >= %d outputs)", v, L, d.n_w);
            o.L = L;
            tap_off[v] = taps.size();
            // out[j] = sum_k c[k] y[j+L-1-k] = sum_{k=0}^{L} g[k] TT[j+L-k],  g = first difference of c
            taps.push_back(in.coeffs[0]);
            for (int k = 1; k < L; ++k) taps.push_back(in.coeffs[k] - in.coeffs[k - 1]);
            taps.push_back(-in.coeffs[L - 1]);
        } else if (in.kind == 2) {
            const int T = in.n_taps;
            if (!in.coeffs || T < 1 || T > LGDSP_MAX_SG || T > n || in.sg_offset < 0 || in.sg_offset >= T)
                return fail(h, LGDSP_ERR_INVALID_ARG, "variant %d: bad Savitzky-Golay tap count/offset", v);
            if (!(0 <= in.win_from && in.win_from <= in.win_until && in.win_until <= n - T))
                return fail(h, LGDSP_ERR_INVALID_ARG, "variant %d: current_window %d:%d outside the SG trace", v, in.win_from, in.win_until);
            o.L = T; o.sg_off = in.sg_offset; o.win_from = in.win_from; o.win_until = in.win_until;
            tap_off[v] = taps.size();
            // s[j] = sum_k h[k] y[j+k] = sum_{k=0}^{T} gg[k] TT[j+k]
            taps.push_back(-in.coeffs[0]);
            for (int k = 1; k < T; ++k) taps.push_back(in.coeffs[k - 1] - in.coeffs[k]);
            taps.push_back(in.coeffs[T - 1]);
        } else {
            return fail(h, LGDSP_ERR_INVALID_ARG, "variant %d: unknown kind %d", v, in.kind);
        }
    }
    int rc = grow(h, &h->d_vars, &h->vars_cap, sizeof(SweepVar) * nvar);
    if (!rc) rc = grow(h, &h->d_taps, &h->taps_cap, sizeof(double) * taps.size());
    if (rc) return rc;
    for (int v = 0; v < nvar; ++v)
        if (sv[v].kind != 0) sv[v].g = h->d_taps + tap_off[v];
    if (!taps.empty()) CK(cudaMemcpyAsync(h->d_taps, taps.data(), sizeof(double) * taps.size(), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_vars, sv.data(), sizeof(SweepVar) * nvar, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_sweep_dniA, d.A, sizeof(double) * LGDSP_MAX_DNI * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    D.n = n; D.tx_min_n = p->tx_min_n; D.t_first = p->t_first_ns; D.dt = p->dt_ns;
    D.bl_from = p->bl_from; D.bl_until = p->bl_until; D.km1 = p->pz_km1;
    D.sig_dni.n_w = d.n_w; D.sig_dni.m = d.degree + 1;
    D.dni_A = h->d_sweep_dniA; D.vars = h->d_vars; D.nvar = nvar; D.out_f64 = p->out_f64 ? 1 : 0;
    D.n_other = 0;
    for (int v = 0; v < nvar; ++v) D.n_other += (sv[v].kind != 0);
    // Reach of the variant set around the crossing sample `pos` of t50 (t50 lies in [pos-1, pos]):
    // from = rint(pc) - n_w/2, pc = (t50 - t_first)/dt + pick/dt - (L-1)  (dni_window), look-ups in [from, from + L + n_w)
    D.warp_ok = 0;
    {
        int ex = 0;
        D.dt_pow2 = (p->dt_ns > 0 && std::frexp(p->dt_ns, &ex) == 0.5) ? 1 : 0;
        D.rdt = 1.0 / p->dt_ns;
    }
    if (D.n_other == 0) {
        bool all1 = true, all0 = true;
        double lo = 1e300, hi = -1e300;
        for (int v = 0; v < nvar; ++v) {
            all1 = all1 && sv[v].mode != 0;
            all0 = all0 && sv[v].mode == 0;
            const double rel = sv[v].pick_ns / p->dt_ns - (double)(sv[v].L - 1) - (double)(d.n_w / 2);
            const double base = sv[v].mode ? rel : rel - p->t_first_ns / p->dt_ns;
            lo = std::min(lo, std::floor(base - 1.5) - 2.0);
            hi = std::max(hi, std::ceil(base + 0.5) + (double)(sv[v].L + d.n_w) + 2.0);
        }
        if (all1) { lo = std::min(lo, -3.0); hi = std::max(hi, 3.0); }
        const int wmax = sweep_warp_max_window();
        int longest = 0;
        for (int v = 0; v < nvar; ++v) longest = std::max(longest, sv[v].L + d.n_w + 2);
        if ((all1 || all0) && wmax > 0 && hi - lo <= (double)wmax && longest <= wmax && std::fabs(lo) < 1e9) {
            const int need = std::max((int)(hi - lo), longest);
            D.win_steps = std::max(4, (need + 287) / 288);   // (>= 4: the window area also holds pass 1's group table)
            D.win_mode = all1 ? 1 : 0;
            D.win_rel_lo = all1 ? (int)lo : 0;
            D.win_abs_lo = all1 ? 0 : std::max(0, (int)lo);
            D.warp_ok = D.win_steps * 288 <= wmax ? 1 : 0;
        }
        // fixed pick-offs: the windows are the same for every event -- the exact last look-up of the set (dni_window's arithmetic)
        D.stream_n = n;
        if (all0) {
            long long last = p->bl_until + 1;
            for (int v = 0; v < nvar; ++v) {
                const int Lf = sv[v].L, nout = n - Lf + 1;
                const double tf = std::fma((double)(Lf - 1), p->dt_ns, p->t_first_ns);
                double pc = (sv[v].pick_ns - tf) / p->dt_ns;
                if (!(pc >= 0)) pc = 0;
                if (pc > nout - 1) pc = nout - 1;
                long long f = (long long)std::nearbyint(pc) - d.n_w / 2;
                if (f < 0) f = 0;
                if (f > nout - d.n_w) f = nout - d.n_w;
                last = std::max(last, f + Lf + d.n_w);
            }
            D.stream_n = (int)std::min<long long>(n, last + 8);
        }
    }
    D.bl_inv_n = 1.0 / (double)(p->bl_until - p->bl_from + 1);
    {
        typedef long double ld;
        const int a = p->bl_from, b = p->bl_until;
        const ld t0 = p->t_first_ns, dt = p->dt_ns, cnt = (ld)(b - a + 1);
        auto s2 = [](ld k) { return k * (k + 1.0L) * (2.0L * k + 1.0L) / 6.0L; };
        const ld si = 0.5L * (ld)(a + b) * cnt, sii = s2((ld)b) - s2((ld)a - 1.0L);
        D.bl_sX = (double)(cnt * t0 + dt * si);
        D.bl_sXX = (double)(cnt * t0 * t0 + 2.0L * t0 * dt * si + dt * dt * sii);
    }
    return LGDSP_OK;
}

static int sweep_run_device_impl(lgdsp_handle* h, const lgdsp_sweep_params* p, const void* d_wf, int sample_bytes,
                                 const double* d_baseline, int64_t n_events, int64_t ld_samples,
                                 const lgdsp_sweep_variant* variants, int32_t n_variants, void* d_out, double* d_aux)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    SweepDev D{};
    int rc = sweep_prepare(h, p, variants, n_variants, D);
    if (rc) return rc;
    rc = check_wf(h, d_wf, n_events, ld_samples, D.n, true, sample_bytes);
    if (rc) return rc;
    if (n_events == 0) return LGDSP_OK;
    if (!d_out) return fail(h, LGDSP_ERR_INVALID_ARG, "output pointer is NULL");
    const long long cap = (long long)h->sm_count * h->sweep_bps;
    const int grid = (int)(n_events < cap ? n_events : cap);
    CK(cudaEventRecord(h->ev0, h->stream));
    if (sweep_launch(D, p->sig_dni.A, d_wf, sample_bytes, n_events, ld_samples, d_baseline, d_out, d_aux, grid, h->sm_count, h->stream) < 0)
        return fail(h, LGDSP_ERR_UNSUPPORTED, "LGDSP_SWEEP_PATH=warp: this variant set / sample type runs on the one-CTA-per-waveform kernel");
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev1, h->stream));
    h->timed = true;
    h->launches += 1;
    return LGDSP_OK;
}

static int sweep_run_host_impl(lgdsp_handle* h, const lgdsp_sweep_params* p, const void* wf, int sample_bytes,
                               const double* baseline, int64_t n_events, int64_t ld_samples,
                               const lgdsp_sweep_variant* variants, int32_t n_variants, void* out, double* aux)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    SweepDev D{};
    int rc = sweep_prepare(h, p, variants, n_variants, D);
    if (rc) return rc;
    const int n = D.n;
    rc = check_wf(h, wf, n_events, ld_samples, n, false, sample_bytes);
    if (rc) return rc;
    if (n_events == 0) return LGDSP_OK;
    if (!out) return fail(h, LGDSP_ERR_INVALID_ARG, "output pointer is NULL");
    const size_t sb = (size_t)sample_bytes;
    const size_t ow = (size_t)n_variants * (D.out_f64 ? sizeof(double) : sizeof(float)), aw = 4 * sizeof(double);
    const long long cap = (long long)h->sm_count * h->sweep_bps;
    return run_chunked(h, n_events, 8192, {host_array(wf, (size_t)ld_samples * sb, (size_t)n * sb), host_array(baseline, sizeof(double), sizeof(double))},
                       {host_array(out, ow, ow), host_array(aux, aw, aw)}, [&](int64_t ne, void* const* d) {
                           const int grid = (int)(ne < cap ? ne : cap);
                           if (sweep_launch(D, p->sig_dni.A, d[0], sample_bytes, ne, n, static_cast<const double*>(d[1]), d[2],
                                            static_cast<double*>(d[3]), grid, h->sm_count, h->stream) < 0)
                               return fail(h, LGDSP_ERR_UNSUPPORTED, "LGDSP_SWEEP_PATH=warp: this variant set / sample type runs on the one-CTA-per-waveform kernel");
                           CK(cudaGetLastError());
                           h->launches += 1;
                           return (int)LGDSP_OK;
                       });
}

int lgdsp_sweep_run_device(lgdsp_handle* h, const lgdsp_sweep_params* p, const uint16_t* d_wf, int64_t n_events,
                           int64_t ld_samples, const lgdsp_sweep_variant* variants, int32_t n_variants, void* d_out,
                           double* d_aux)
{
    return sweep_run_device_impl(h, p, d_wf, 2, nullptr, n_events, ld_samples, variants, n_variants, d_out, d_aux);
}

int lgdsp_sweep_run(lgdsp_handle* h, const lgdsp_sweep_params* p, const uint16_t* wf, int64_t n_events, int64_t ld_samples,
                    const lgdsp_sweep_variant* variants, int32_t n_variants, void* out, double* aux)
{
    return sweep_run_host_impl(h, p, wf, 2, nullptr, n_events, ld_samples, variants, n_variants, out, aux);
}

int lgdsp_sweep_run_ext_device(lgdsp_handle* h, const lgdsp_sweep_params* p, const void* d_wf, int32_t sample_bytes,
                               const double* d_baseline, int64_t n_events, int64_t ld_samples,
                               const lgdsp_sweep_variant* variants, int32_t n_variants, void* d_out, double* d_aux)
{
    return sweep_run_device_impl(h, p, d_wf, sample_bytes, d_baseline, n_events, ld_samples, variants, n_variants, d_out, d_aux);
}

int lgdsp_sweep_run_ext(lgdsp_handle* h, const lgdsp_sweep_params* p, const void* wf, int32_t sample_bytes, const double* baseline,
                        int64_t n_events, int64_t ld_samples, const lgdsp_sweep_variant* variants, int32_t n_variants, void* out,
                        double* aux)
{
    return sweep_run_host_impl(h, p, wf, sample_bytes, baseline, n_events, ld_samples, variants, n_variants, out, aux);
}

// the trapezoid-only entry points (kept for callers of the first ABI revision): thin wrappers
static std::vector<lgdsp_sweep_variant> trap_to_general(const lgdsp_trap_variant* variants, int32_t n)
{
    std::vector<lgdsp_sweep_variant> v((size_t)(n > 0 ? n : 0));
    for (int i = 0; i < n; ++i) {
        memset(&v[i], 0, sizeof(v[i]));
        v[i].kind = 0;
        v[i].pickoff_mode = variants[i].pickoff_mode;
        v[i].pickoff_ns = variants[i].pickoff_ns;
        v[i].trap = variants[i].trap;
    }
    return v;
}

int lgdsp_trap_sweep_run_device(lgdsp_handle* h, const lgdsp_sweep_params* p, const uint16_t* d_wf, int64_t n_events,
                                int64_t ld_samples, const lgdsp_trap_variant* variants, int32_t n_variants, float* d_out)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    if (!variants) return fail(h, LGDSP_ERR_INVALID_ARG, "sweep params/variants NULL");
    if (p && p->out_f64) return fail(h, LGDSP_ERR_INVALID_ARG, "lgdsp_trap_sweep_run_device writes float: out_f64 must be 0");
    std::vector<lgdsp_sweep_variant> v = trap_to_general(variants, n_variants);
    return lgdsp_sweep_run_device(h, p, d_wf, n_events, ld_samples, v.data(), n_variants, d_out, nullptr);
}

int lgdsp_trap_sweep_run(lgdsp_handle* h, const lgdsp_sweep_params* p, const uint16_t* wf, int64_t n_events,
                         int64_t ld_samples, const lgdsp_trap_variant* variants, int32_t n_variants, float* out)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    if (!variants) return fail(h, LGDSP_ERR_INVALID_ARG, "sweep params/variants NULL");
    if (p && p->out_f64) return fail(h, LGDSP_ERR_INVALID_ARG, "lgdsp_trap_sweep_run writes float: out_f64 must be 0");
    std::vector<lgdsp_sweep_variant> v = trap_to_general(variants, n_variants);
    return lgdsp_sweep_run(h, p, wf, n_events, ld_samples, v.data(), n_variants, out, nullptr);
}

// ---------------------------------------------------------------------------------------------------
// dsp_sipm  (/root/reference/src/dsp_sipm.jl:47-158)
// ---------------------------------------------------------------------------------------------------
static int sipm_prepare(lgdsp_handle* h, const lgdsp_sipm_params* p, SipmDev& D, int& bps)
{
    if (!p) return fail(h, LGDSP_ERR_INVALID_ARG, "params is NULL");
    if (p->struct_size != sizeof(lgdsp_sipm_params) || p->version != LGDSP_PARAMS_VERSION)
        return fail(h, LGDSP_ERR_INVALID_ARG, "lgdsp_sipm_params: size/version mismatch (got %u/%u, want %zu/%u)", p->struct_size,
                    p->version, sizeof(lgdsp_sipm_params), LGDSP_PARAMS_VERSION);
    const int n = p->n_samples;
    if (n < 16 || n > LGDSP_MAX_SAMPLES) return fail(h, LGDSP_ERR_UNSUPPORTED, "n_samples = %d: need 16 .. %d", n, LGDSP_MAX_SAMPLES);
    if (p->sample_kind != LGDSP_SAMPLE_U16 && p->sample_kind != LGDSP_SAMPLE_F32)
        return fail(h, LGDSP_ERR_UNSUPPORTED, "sample_kind = %d: LGDSP_SAMPLE_U16 or LGDSP_SAMPLE_F32", p->sample_kind);
    if (!(p->dt_ns > 0) || !std::isfinite(p->t_first_ns)) return fail(h, LGDSP_ERR_INVALID_ARG, "bad time axis");
    if (!(0 <= p->trunc_from && p->trunc_from <= p->trunc_until && p->trunc_until <= n - 1))
        return fail(h, LGDSP_ERR_INVALID_ARG, "t0_hpge_window %d:%d outside the waveform", p->trunc_from, p->trunc_until);
    const lgdsp_sg& sg = p->sg;
    if (sg.n_taps < 1 || sg.n_taps > LGDSP_MAX_SG || sg.n_taps > n || sg.offset < 0 || sg.offset >= sg.n_taps)
        return fail(h, LGDSP_ERR_INVALID_ARG, "sg: bad tap count/offset");
    const int n_sg = n - sg.n_taps + 1;
    const lgdsp_trap& t = p->trap;
    if (t.navg < 1 || t.navg2 < 1 || t.ngap < 0 || t.navg + t.ngap + t.navg2 > n_sg)
        return fail(h, LGDSP_ERR_INVALID_ARG, "trapezoidal filter does not fit the Savitzky-Golay trace");
    if (p->sg_min_n < 1 || p->sg_max_n < 1 || p->trap_min_n < 1 || p->trap_max_n < 1) return fail(h, LGDSP_ERR_INVALID_ARG, "min_n / max_n must be >= 1");
    if (p->max_triggers < 1 || p->max_triggers > LGDSP_SIPM_MAX_TRIGGERS) return fail(h, LGDSP_ERR_INVALID_ARG, "max_triggers outside 1..%d", LGDSP_SIPM_MAX_TRIGGERS);
    D = SipmDev{};
    D.n = n; D.kind = p->sample_kind; D.t_first = p->t_first_ns; D.dt = p->dt_ns;
    D.trunc_from = p->trunc_from; D.trunc_until = p->trunc_until;
    D.sg_taps = sg.n_taps; D.sg_off = sg.offset;
    for (int k = 0; k < sg.n_taps; ++k) D.sgh[k] = sg.h[k];
    D.sg_min_n = p->sg_min_n; D.sg_max_n = p->sg_max_n;
    D.sg_min_thr = p->sg_min_thr; D.sg_max_thr = p->sg_max_thr; D.sg_nsigma = p->sg_nsigma;
    D.sg_min_dc = p->sg_min_dc; D.sg_max_dc = p->sg_max_dc; D.sg_nsigma_dc = p->sg_nsigma_dc;
    D.ta = t.navg; D.tg = t.ngap; D.ta2 = t.navg2; D.tL = t.navg + t.ngap + t.navg2;
    D.inv1 = 1.0 / t.navg; D.inv2 = 1.0 / t.navg2; D.km1 = p->pz_km1;
    D.trap_min_n = p->trap_min_n; D.trap_max_n = p->trap_max_n;
    D.trap_min_thr = p->trap_min_thr; D.trap_max_thr = p->trap_max_thr; D.trap_nsigma = p->trap_nsigma;
    D.trap_min_dc = p->trap_min_dc; D.trap_max_dc = p->trap_max_dc; D.trap_nsigma_dc = p->trap_nsigma_dc;
    D.cap = p->max_triggers;
    CK(sipm_configure(n, p->sample_kind, &bps));
    if (bps < 1) return fail(h, LGDSP_ERR_CUDA, "sipm kernel does not fit on an SM");
    return LGDSP_OK;
}

// sipm_prepare plus the checks lgdsp_sipm_run and _run_device share (nothing to do when n_events is 0)
static int sipm_check(lgdsp_handle* h, const lgdsp_sipm_params* p, const void* wf, int64_t n_events, int64_t ld_samples,
                      const double* rows, const double* trig, SipmDev& D, int& bps)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    int rc = sipm_prepare(h, p, D, bps);
    if (rc) return rc;
    if (n_events < 0) return fail(h, LGDSP_ERR_INVALID_ARG, "n_events < 0");
    if (n_events == 0) return LGDSP_OK;
    if (!wf || !rows || !trig) return fail(h, LGDSP_ERR_INVALID_ARG, "NULL pointer");
    if (ld_samples < D.n) return fail(h, LGDSP_ERR_INVALID_ARG, "ld_samples (%lld) < n_samples (%d)", (long long)ld_samples, D.n);
    return LGDSP_OK;
}

int lgdsp_sipm_run_device(lgdsp_handle* h, const lgdsp_sipm_params* p, const void* d_wf, int64_t n_events, int64_t ld_samples,
                          double* d_rows, double* d_trig)
{
    SipmDev D;
    int bps = 0;
    int rc = sipm_check(h, p, d_wf, n_events, ld_samples, d_rows, d_trig, D, bps);
    if (rc || n_events == 0) return rc;
    const long long cap = (long long)h->sm_count * bps;
    const int grid = (int)(n_events < cap ? n_events : cap);
    CK(cudaEventRecord(h->ev0, h->stream));
    sipm_launch(D, d_wf, n_events, ld_samples, d_rows, d_trig, grid, h->stream);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev1, h->stream));
    h->timed = true;
    h->launches += 1;
    return LGDSP_OK;
}

int lgdsp_sipm_run(lgdsp_handle* h, const lgdsp_sipm_params* p, const void* wf, int64_t n_events, int64_t ld_samples, double* rows,
                   double* trig)
{
    SipmDev D;
    int bps = 0;
    int rc = sipm_check(h, p, wf, n_events, ld_samples, rows, trig, D, bps);
    if (rc || n_events == 0) return rc;
    const size_t sb = (size_t)D.kind;   // bytes per sample
    const size_t rw = LGDSP_SIPM_NCOL * sizeof(double), tw = (size_t)LGDSP_SIPM_NLIST * LGDSP_SIPM_NFIELD * D.cap * sizeof(double);
    const long long gcap = (long long)h->sm_count * bps;
    return run_chunked(h, n_events, 8192, {host_array(wf, (size_t)ld_samples * sb, (size_t)D.n * sb)}, {host_array(rows, rw, rw), host_array(trig, tw, tw)},
                       [&](int64_t ne, void* const* d) {
                           const int grid = (int)(ne < gcap ? ne : gcap);
                           sipm_launch(D, d[0], ne, D.n, static_cast<double*>(d[1]), static_cast<double*>(d[2]), grid, h->stream);
                           CK(cudaGetLastError());
                           h->launches += 1;
                           return (int)LGDSP_OK;
                       });
}

int lgdsp_sipm_list_pointers_device(lgdsp_handle* h, const double* d_rows, int64_t n_events, int32_t list, int32_t max_triggers,
                                    int64_t* d_elem_ptr, int64_t* total)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (n_events < 0 || list < 0 || list >= LGDSP_SIPM_NLIST || max_triggers < 1) return fail(h, LGDSP_ERR_INVALID_ARG, "bad n_events / list / max_triggers");
    if (!d_elem_ptr || (n_events > 0 && !d_rows)) return fail(h, LGDSP_ERR_INVALID_ARG, "NULL pointer");
    static_assert(sizeof(long long) == sizeof(int64_t), "int64");
    sipm_count_scan_launch(d_rows, n_events, list, max_triggers, reinterpret_cast<long long*>(d_elem_ptr), h->stream);
    CK(cudaGetLastError());
    h->launches += 1;
    long long tot = 0;
    CK(cudaMemcpyAsync(&tot, d_elem_ptr + n_events, sizeof(long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (total) *total = tot;
    return LGDSP_OK;
}

int lgdsp_sipm_list_gather_device(lgdsp_handle* h, const double* d_trig, int64_t n_events, int32_t list, int32_t max_triggers,
                                  const int64_t* d_elem_ptr, double* d_flat, int64_t flat_stride)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (n_events < 0 || list < 0 || list >= LGDSP_SIPM_NLIST || max_triggers < 1 || flat_stride < 0) return fail(h, LGDSP_ERR_INVALID_ARG, "bad argument");
    if (n_events == 0) return LGDSP_OK;
    if (!d_trig || !d_elem_ptr || !d_flat) return fail(h, LGDSP_ERR_INVALID_ARG, "NULL pointer");
    sipm_compact_launch(d_trig, n_events, list, max_triggers, reinterpret_cast<const long long*>(d_elem_ptr), d_flat, flat_stride, h->stream);
    CK(cudaGetLastError());
    h->launches += 1;
    return LGDSP_OK;
}

// ---------------------------------------------------------------------------------------------------
// per-waveform primitives on waveform arrays (lgdsp_wfstats_run)
// ---------------------------------------------------------------------------------------------------
static int wfstats_prepare(lgdsp_handle* h, const lgdsp_wfstats_params* p, WfstatsDev& D, int& bps)
{
    if (!p) return fail(h, LGDSP_ERR_INVALID_ARG, "params is NULL");
    if (p->struct_size != sizeof(lgdsp_wfstats_params) || p->version != LGDSP_PARAMS_VERSION)
        return fail(h, LGDSP_ERR_INVALID_ARG, "lgdsp_wfstats_params: size/version mismatch (got %u/%u, want %zu/%u)", p->struct_size,
                    p->version, sizeof(lgdsp_wfstats_params), LGDSP_PARAMS_VERSION);
    const unsigned what = p->what;
    if (what == 0 || (what & ~LGDSP_WFSTAT_ALL)) return fail(h, LGDSP_ERR_INVALID_ARG, "what = 0x%x: a non-empty LGDSP_WFSTAT_* mask", what);
    const int n = p->n_samples;
    if (n < 0 || n > LGDSP_WFSTAT_MAX_SAMPLES) return fail(h, LGDSP_ERR_UNSUPPORTED, "n_samples = %d: need 0 .. %d", n, LGDSP_WFSTAT_MAX_SAMPLES);
    const int kind = p->sample_kind;
    if (kind != LGDSP_SAMPLE_U16 && kind != LGDSP_SAMPLE_F32 && kind != LGDSP_SAMPLE_F64)
        return fail(h, LGDSP_ERR_UNSUPPORTED, "sample_kind = %d: LGDSP_SAMPLE_U16, _F32 or _F64", kind);
    // saturation compares raw ADC samples with integer levels (src/saturation.jl; SURVEY.md App. F)
    if ((what & LGDSP_WFSTAT_SATURATION) && kind != LGDSP_SAMPLE_U16)
        return fail(h, LGDSP_ERR_UNSUPPORTED, "saturation takes raw UInt16 samples (LGDSP_SAMPLE_U16)");
    if (!std::isfinite(p->dt_ns) || !std::isfinite(p->t_first_ns)) return fail(h, LGDSP_ERR_INVALID_ARG, "bad time axis");
    // @assert firstindex(X) <= first(idxs) <= last(idxs) <= lastindex(X)   src/tailstats.jl:23-25
    const struct { unsigned bit; int from, until; const char* name; } win[4] = {
        {LGDSP_WFSTAT_SATURATION, p->sat_from, p->sat_until, "saturation"},
        {LGDSP_WFSTAT_EXTREMESTATS, p->ext_from, p->ext_until, "extremestats"},
        {LGDSP_WFSTAT_TAILSTATS, p->tail_from, p->tail_until, "tailstats"},
        {LGDSP_WFSTAT_WVF_MAXIMUM, p->max_from, p->max_until, "get_wvf_maximum"}};
    for (const auto& w : win)
        if ((what & w.bit) && !(0 <= w.from && w.from <= w.until && w.until <= n - 1))
            return fail(h, LGDSP_ERR_INVALID_ARG, "%s window %d:%d outside the waveform (0:%d)", w.name, w.from, w.until, n - 1);
    const bool im = (what & LGDSP_WFSTAT_INTERSECT_MAXIMUM) != 0;
    if (im && (p->im_min_n < 1 || p->im_max_n < 1)) return fail(h, LGDSP_ERR_INVALID_ARG, "im_min_n / im_max_n must be >= 1");
    if (im && (p->max_triggers < 1 || p->max_triggers > LGDSP_WFSTAT_MAX_TRIGGERS))
        return fail(h, LGDSP_ERR_INVALID_ARG, "max_triggers outside 1..%d", LGDSP_WFSTAT_MAX_TRIGGERS);
    D = WfstatsDev{};
    D.n = n; D.kind = kind; D.what = what; D.cap = im ? p->max_triggers : 0;
    D.t0 = p->t_first_ns; D.dt = p->dt_ns;
    D.sat_from = p->sat_from; D.sat_until = p->sat_until; D.ext_from = p->ext_from; D.ext_until = p->ext_until;
    D.tail_from = p->tail_from; D.tail_until = p->tail_until; D.max_from = p->max_from; D.max_until = p->max_until;
    D.sat_low = p->sat_low; D.sat_high = p->sat_high;
    D.thr_min = p->thr_min; D.thr_max = p->thr_max;
    D.im_min_n = p->im_min_n; D.im_max_n = p->im_max_n;
    CK(wfstats_configure(D, &bps));
    if (bps < 1) return fail(h, LGDSP_ERR_CUDA, "wfstats kernel does not fit on an SM");
    return LGDSP_OK;
}

// wfstats_prepare plus the checks lgdsp_wfstats_run and _run_device share (nothing to do when n_events is 0)
static int wfstats_check(lgdsp_handle* h, const lgdsp_wfstats_params* p, const void* wf, const double* thresholds, int64_t n_events,
                         int64_t ld_samples, const double* rows, const double* lists, WfstatsDev& D, int& bps)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    int rc = wfstats_prepare(h, p, D, bps);
    if (rc) return rc;
    const bool im = (D.what & LGDSP_WFSTAT_INTERSECT_MAXIMUM) != 0;
    if (n_events < 0) return fail(h, LGDSP_ERR_INVALID_ARG, "n_events < 0");
    if (n_events == 0) return LGDSP_OK;
    if (ld_samples < D.n) return fail(h, LGDSP_ERR_INVALID_ARG, "ld_samples (%lld) < n_samples (%d)", (long long)ld_samples, D.n);
    if (im && !thresholds) return fail(h, LGDSP_ERR_INVALID_ARG, "IntersectMaximum needs the per-event thresholds (NULL pointer)");
    if ((D.n > 0 && !wf) || !rows || (im && !lists)) return fail(h, LGDSP_ERR_INVALID_ARG, "NULL pointer");
    return LGDSP_OK;
}

// persistent grid; when thresholdstats_mad needs the converted trace in global memory (long non-double traces) the grid is also
// limited so that those per-CTA copies take at most 256 MiB (at least one CTA per SM)
static int wfstats_grid(lgdsp_handle* h, const WfstatsDev& D, int bps, int64_t n_events, int& grid)
{
    long long g = (long long)h->sm_count * bps;
    const long long per_cta = wfstats_work_doubles(D);
    if (per_cta > 0) {
        g = std::min(g, std::max((long long)h->sm_count, (256ll << 20) / (per_cta * (long long)sizeof(double))));
        const int rc = grow(h, &h->d_work, &h->work_cap, (size_t)g * per_cta * sizeof(double));
        if (rc) return rc;
    }
    grid = (int)std::min<long long>(g, n_events);
    return LGDSP_OK;
}

int lgdsp_wfstats_run_device(lgdsp_handle* h, const lgdsp_wfstats_params* p, const void* d_wf, const double* d_thresholds,
                             int64_t n_events, int64_t ld_samples, double* d_rows, double* d_lists)
{
    WfstatsDev D;
    int bps = 0, grid = 0;
    int rc = wfstats_check(h, p, d_wf, d_thresholds, n_events, ld_samples, d_rows, d_lists, D, bps);
    if (rc || n_events == 0) return rc;
    rc = wfstats_grid(h, D, bps, n_events, grid);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev0, h->stream));
    wfstats_launch(D, d_wf, d_thresholds, n_events, ld_samples, d_rows, d_lists, h->d_work, grid, h->stream);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev1, h->stream));
    h->timed = true;
    h->launches += 1;
    return LGDSP_OK;
}

int lgdsp_wfstats_run(lgdsp_handle* h, const lgdsp_wfstats_params* p, const void* wf, const double* thresholds, int64_t n_events,
                      int64_t ld_samples, double* rows, double* lists)
{
    WfstatsDev D;
    int bps = 0, grid = 0;
    int rc = wfstats_check(h, p, wf, thresholds, n_events, ld_samples, rows, lists, D, bps);
    if (rc || n_events == 0) return rc;
    rc = wfstats_grid(h, D, bps, n_events, grid);
    if (rc) return rc;
    const bool im = (D.what & LGDSP_WFSTAT_INTERSECT_MAXIMUM) != 0;
    const size_t sb = (size_t)D.kind;   // bytes per sample
    const size_t rw = LGDSP_WFSTAT_NCOL * sizeof(double), lw = (size_t)4 * D.cap * sizeof(double);
    // events per chunk: at most 8192, and few enough that one chunk's device rows (samples, threshold, row, lists) take at most
    // 64 MiB -- the lists alone are 2 MiB per event at max_triggers = 65536; the double-buffered slots and the pinned staging
    // of pageable memory stay bounded the same way
    const size_t per_event = (size_t)D.n * sb + rw + (im ? sizeof(double) + lw : 0);
    const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(8192, (int64_t)((64ull << 20) / per_event)));
    return run_chunked(h, n_events, chunk,
                       {host_array(D.n > 0 ? wf : nullptr, (size_t)ld_samples * sb, (size_t)D.n * sb),
                        host_array(im ? thresholds : nullptr, sizeof(double), sizeof(double))},
                       {host_array(rows, rw, rw), host_array(im ? lists : nullptr, lw, lw)}, [&](int64_t ne, void* const* d) {
                           wfstats_launch(D, d[0], static_cast<const double*>(d[1]), ne, D.n, static_cast<double*>(d[2]),
                                          static_cast<double*>(d[3]), h->d_work, (int)std::min<int64_t>(grid, ne), h->stream);
                           CK(cudaGetLastError());
                           h->launches += 1;
                           return (int)LGDSP_OK;
                       });
}

// the single-trace primitives: n_events = 1 calls of lgdsp_wfstats_run on a trace of doubles
static lgdsp_wfstats_params single_trace_params(int32_t n, unsigned what)
{
    lgdsp_wfstats_params p;
    memset(&p, 0, sizeof(p));
    p.struct_size = sizeof(p);
    p.version = LGDSP_PARAMS_VERSION;
    p.n_samples = n;
    p.sample_kind = LGDSP_SAMPLE_F64;
    p.what = what;
    p.dt_ns = 1.0;
    return p;
}

int lgdsp_thresholdstats(lgdsp_handle* h, const double* y, int32_t n, double min, double max, int32_t mad, double* out)
{
    if (!out) return h ? fail(h, LGDSP_ERR_INVALID_ARG, "output pointer is NULL") : LGDSP_ERR_INVALID_ARG;
    lgdsp_wfstats_params p = single_trace_params(n, mad ? LGDSP_WFSTAT_THRESHOLDSTATS_MAD : LGDSP_WFSTAT_THRESHOLDSTATS);
    p.thr_min = min;
    p.thr_max = max;
    double row[LGDSP_WFSTAT_NCOL];
    const int rc = lgdsp_wfstats_run(h, &p, y, nullptr, 1, n, row, nullptr);
    if (rc) return rc;
    *out = row[mad ? LGDSP_WFSTAT_thr_mad : LGDSP_WFSTAT_thr_sigma];
    return LGDSP_OK;
}

int lgdsp_intersect_maximum(lgdsp_handle* h, const double* y, int32_t n, double t_first_ns, double dt_ns, double threshold,
                            int32_t min_n, int32_t max_n, int32_t max_triggers, double* x, double* x_high, double* x_tot,
                            double* max, int32_t* n_found)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    if (!x || !x_high || !x_tot || !max || !n_found) return fail(h, LGDSP_ERR_INVALID_ARG, "output pointer is NULL");
    lgdsp_wfstats_params p = single_trace_params(n, LGDSP_WFSTAT_INTERSECT_MAXIMUM);
    p.t_first_ns = t_first_ns;
    p.dt_ns = dt_ns;
    p.im_min_n = min_n;
    p.im_max_n = max_n;
    p.max_triggers = max_triggers;
    if (max_triggers < 1 || max_triggers > LGDSP_WFSTAT_MAX_TRIGGERS)
        return fail(h, LGDSP_ERR_INVALID_ARG, "max_triggers outside 1..%d", LGDSP_WFSTAT_MAX_TRIGGERS);
    std::vector<double> buf((size_t)4 * max_triggers);
    double row[LGDSP_WFSTAT_NCOL];
    const int rc = lgdsp_wfstats_run(h, &p, y, &threshold, 1, n, row, buf.data());
    if (rc) return rc;
    const size_t c = (size_t)max_triggers;
    memcpy(x, buf.data(), c * sizeof(double));
    memcpy(x_high, buf.data() + c, c * sizeof(double));
    memcpy(x_tot, buf.data() + 2 * c, c * sizeof(double));
    memcpy(max, buf.data() + 3 * c, c * sizeof(double));
    *n_found = (int32_t)row[LGDSP_WFSTAT_multiplicity];
    return LGDSP_OK;
}

// ---------------------------------------------------------------------------------------------------
// MultiIntersect  (/root/reference/src/multi_intersect.jl:10-121)
// ---------------------------------------------------------------------------------------------------
static int mi_prepare(lgdsp_handle* h, const lgdsp_multi_intersect_params* p, MiDev& D)
{
    if (!p) return fail(h, LGDSP_ERR_INVALID_ARG, "params is NULL");
    if (p->struct_size != sizeof(lgdsp_multi_intersect_params) || p->version != LGDSP_PARAMS_VERSION)
        return fail(h, LGDSP_ERR_INVALID_ARG, "lgdsp_multi_intersect_params: size/version mismatch");
    if (p->n_samples < 2) return fail(h, LGDSP_ERR_INVALID_ARG, "n_samples < 2");
    if (p->n_thresholds < 1 || p->n_thresholds > LGDSP_MI_MAX_THR) return fail(h, LGDSP_ERR_UNSUPPORTED, "n_thresholds outside 1..%d", LGDSP_MI_MAX_THR);
    if (!(p->dt_ns > 0) || !std::isfinite(p->t_first_ns)) return fail(h, LGDSP_ERR_INVALID_ARG, "bad time axis");
    if (p->min_n < 1) return fail(h, LGDSP_ERR_INVALID_ARG, "min_n must be >= 1");
    if (p->half_window < 1 || p->half_window > LGDSP_MI_MAX_HALF || p->degree < 0 || p->degree > LGDSP_MAX_DNI_DEG ||
        p->degree >= 2 * p->half_window || p->rate < 1 || 2 * p->half_window * p->rate > 256)
        return fail(h, LGDSP_ERR_UNSUPPORTED, "polynomial window / degree / sampling rate outside the supported range");
    D = MiDev{};
    D.len = p->n_samples; D.n_thr = p->n_thresholds; D.t0 = p->t_first_ns; D.dt = p->dt_ns;
    D.min_n = p->min_n; D.n = p->half_window; D.degree = p->degree; D.rate = p->rate;
    for (int j = 0; j < p->n_thresholds; ++j) D.ratios[j] = p->ratios[j];
    for (int i = 0; i < 2 * p->half_window * (p->degree + 1); ++i) D.A[i] = p->A[i];
    return LGDSP_OK;
}

// mi_prepare plus the checks lgdsp_multi_intersect_run and _run_device share (nothing to do when n_events is 0)
static int mi_check(lgdsp_handle* h, const lgdsp_multi_intersect_params* p, const double* y, int64_t n_events, int64_t ld_samples,
                    const double* x, const int32_t* flags, MiDev& D)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    int rc = mi_prepare(h, p, D);
    if (rc) return rc;
    if (n_events < 0) return fail(h, LGDSP_ERR_INVALID_ARG, "n_events < 0");
    if (n_events == 0) return LGDSP_OK;
    if (!y || !x || !flags) return fail(h, LGDSP_ERR_INVALID_ARG, "NULL pointer");
    if (ld_samples < D.len) return fail(h, LGDSP_ERR_INVALID_ARG, "ld_samples < n_samples");
    return LGDSP_OK;
}

int lgdsp_multi_intersect_run_device(lgdsp_handle* h, const lgdsp_multi_intersect_params* p, const double* d_y, int64_t n_events,
                                     int64_t ld_samples, double* d_x, int32_t* d_flags)
{
    MiDev D;
    int rc = mi_check(h, p, d_y, n_events, ld_samples, d_x, d_flags, D);
    if (rc || n_events == 0) return rc;
    CK(cudaEventRecord(h->ev0, h->stream));
    multi_intersect_launch(D, d_y, n_events, ld_samples, d_x, d_flags, h->stream);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev1, h->stream));
    h->timed = true;
    h->launches += 1;
    return LGDSP_OK;
}

int lgdsp_multi_intersect_run(lgdsp_handle* h, const lgdsp_multi_intersect_params* p, const double* y, int64_t n_events,
                              int64_t ld_samples, double* x, int32_t* flags)
{
    MiDev D;
    int rc = mi_check(h, p, y, n_events, ld_samples, x, flags, D);
    if (rc || n_events == 0) return rc;
    const size_t xw = (size_t)D.n_thr * sizeof(double);
    return run_chunked(h, n_events, 4096, {host_array(y, (size_t)ld_samples * sizeof(double), (size_t)D.len * sizeof(double))},
                       {host_array(x, xw, xw), host_array(flags, sizeof(int32_t), sizeof(int32_t))}, [&](int64_t ne, void* const* d) {
                           multi_intersect_launch(D, static_cast<const double*>(d[0]), ne, D.len, static_cast<double*>(d[1]),
                                                  static_cast<int*>(d[2]), h->stream);
                           CK(cudaGetLastError());
                           h->launches += 1;
                           return (int)LGDSP_OK;
                       });
}

// ---------------------------------------------------------------------------------------------------
// synthetic input
// ---------------------------------------------------------------------------------------------------
int lgdsp_synth_generate_device(lgdsp_handle* h, const lgdsp_synth_params* sp, int64_t first_event, int64_t n_events,
                                int64_t ld_samples, uint16_t* d_wf)
{
    if (!h) return LGDSP_ERR_INVALID_ARG;
    CK(cudaSetDevice(h->device));
    if (!sp || sp->n_samples < 8 || sp->n_samples % 8 != 0 || sp->n_samples > LGDSP_MAX_SAMPLES || !(sp->tau_samples > 0))
        return fail(h, LGDSP_ERR_INVALID_ARG, "bad synth params");
    int rc = check_wf(h, d_wf, n_events, ld_samples, sp->n_samples, true);
    if (rc) return rc;
    if (n_events == 0) return LGDSP_OK;
    synth_launch(*sp, first_event, n_events, ld_samples, d_wf, h->stream);
    CK(cudaGetLastError());
    h->launches += 1;
    return LGDSP_OK;
}

}  // extern "C"
