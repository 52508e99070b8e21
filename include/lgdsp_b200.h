/*
 * lgdsp_b200.h -- C ABI of the B200-native (sm_100a) implementation of the LegendDSP.jl
 * `dsp_icpc` hot path and of the trapezoidal filter-optimisation sweeps.
 *
 * Every entry point replaces one reference interface; citations are relative to the
 * reference tree (legend-exp/LegendDSP.jl v0.3.0):
 *
 *   lgdsp_icpc_run / lgdsp_icpc_run_device   <- dsp_icpc(data, config, tau, pars_filter)
 *                                               src/dsp_icpc.jl:62-230
 *   lgdsp_trap_sweep_run / _device           <- dsp_trap_rt_optimization  src/dsp_filter_optimization.jl:102-133
 *                                               dsp_trap_ft_optimization  src/dsp_filter_optimization.jl:241-274
 *   lgdsp_sweep_run / _device                <- the same two plus dsp_cusp_rt/zac_rt_optimization :145-231,
 *                                               dsp_cusp_ft/zac_ft_optimization :286-375, dsp_sg_optimization :393-441
 *                                               (every sweep of the file except the _compressed / qc variants)
 *   lgdsp_sg_coeffs / lgdsp_lsq_fit_matrix /
 *   lgdsp_cusp_coeffs / lgdsp_zac_coeffs     <- filter-instance construction that the reference delegates to
 *                                               RadiationDetectorDSP.jl (fltinstance(...), src/dsp_icpc.jl:157-181)
 *   lgdsp_synth_generate_device/_host        <- make_fake_waveform  test/test_dsp_icpc.jl:11-32 (generalised,
 *                                               SURVEY.md section 8d)
 *
 * The boundary is the whole chain, not the per-filter `rdfilt!` plugin API (src/derivative.jl:37-55):
 * a per-filter boundary would force one HBM round trip per step.
 *
 * All time quantities are resolved by the host language into SAMPLE units (integers) or nanoseconds
 * (doubles) with the reference's own expressions before they cross this ABI: Julia's round() is
 * ties-to-even and several windows of the reference's example config are exact ties (SURVEY.md App. A).
 *
 * Conventions: plain pointers and sizes, no C++/torch types; every function returning int returns
 * LGDSP_OK (0) or a negative status, with a message available from lgdsp_last_error(). The library never
 * keeps or frees caller memory. A handle is bound to one CUDA device and is not thread-safe.
 * There is NO CPU fallback: without a usable CUDA device lgdsp_create() fails.
 */
#ifndef LGDSP_B200_H
#define LGDSP_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LGDSP_VERSION_MAJOR 0
#define LGDSP_VERSION_MINOR 1
#define LGDSP_PARAMS_VERSION 4u

/* status codes */
#define LGDSP_OK 0
#define LGDSP_ERR_INVALID_ARG (-1)
#define LGDSP_ERR_CUDA (-2)
#define LGDSP_ERR_UNSUPPORTED (-3)
#define LGDSP_ERR_NO_DEVICE (-4)
#define LGDSP_ERR_OOM (-5)

/* limits of this implementation */
#define LGDSP_MAX_SAMPLES 8192   /* samples per waveform (multiple of 8) */
#define LGDSP_MAX_DNI 64         /* PolynomialDNI window length */
#define LGDSP_MAX_DNI_DEG 3
#define LGDSP_MAX_SG 33          /* Savitzky-Golay taps */
#define LGDSP_MAX_FIR 4096       /* CUSP/ZAC taps */

/* waveform codecs of `decode_data` (LegendDataTypes.jl; call sites /root/reference/src/dsp_icpc.jl:313-314) */
#define LGDSP_CODEC_RADWARE 1     /* RadwareSigcompress(shift): radware-sigcompress v1.0, 16-bit samples, big-endian words */
#define LGDSP_CODEC_ULEB128ZZD 2  /* ULEB128 zig-zag difference codec (VarlenDiffArrayCodec): 16- or 32-bit samples */

/* ---- output schema: computed columns of dsp_icpc, order of src/dsp_icpc.jl:210-229.
 * The four pass-through columns (blfc, timestamp, eventID_fadc, e_fc) never touch the GPU.
 * Device rows are double[LGDSP_NCOL]; integer columns (qc_label, inTrace_n, n_sat_*) hold exact small
 * integers. Times t0..t50_current, t0_inv are in microseconds; drift_time, tail_tau, t_*_max and
 * inTrace_intersect are in the unit of the time axis (nanoseconds); blslope/tailslope are per ns. */
enum lgdsp_col {
    LGDSP_COL_blmean = 0, LGDSP_COL_blsigma, LGDSP_COL_blslope, LGDSP_COL_bloffset,
    LGDSP_COL_tailmean, LGDSP_COL_tailsigma, LGDSP_COL_tailslope, LGDSP_COL_tailoffset,
    LGDSP_COL_qc_label,
    LGDSP_COL_t0, LGDSP_COL_t10, LGDSP_COL_t50, LGDSP_COL_t80, LGDSP_COL_t90, LGDSP_COL_t99,
    LGDSP_COL_t50_current,
    LGDSP_COL_drift_time,
    LGDSP_COL_tail_tau, LGDSP_COL_tail_mean, LGDSP_COL_tail_sigma,
    LGDSP_COL_e_max, LGDSP_COL_e_min,
    LGDSP_COL_e_10410, LGDSP_COL_e_535, LGDSP_COL_e_313,
    LGDSP_COL_e_10410_inv, LGDSP_COL_e_313_inv,
    LGDSP_COL_t0_inv,
    LGDSP_COL_e_trap, LGDSP_COL_e_cusp, LGDSP_COL_e_zac,
    LGDSP_COL_e_trap_max, LGDSP_COL_e_cusp_max, LGDSP_COL_e_zac_max,
    LGDSP_COL_t_trap_max, LGDSP_COL_t_cusp_max, LGDSP_COL_t_zac_max,
    LGDSP_COL_qdrift, LGDSP_COL_lq,
    LGDSP_COL_a_sg, LGDSP_COL_a_60, LGDSP_COL_a_100, LGDSP_COL_a_raw,
    LGDSP_COL_inTrace_intersect, LGDSP_COL_inTrace_n,
    LGDSP_COL_n_sat_low, LGDSP_COL_n_sat_high, LGDSP_COL_n_sat_low_cons, LGDSP_COL_n_sat_high_cons,
    LGDSP_NCOL /* = 49 */
};

/* which groups of columns to compute (bit mask). Columns of groups that are switched off are written as 0.
 * LGDSP_GROUP_ALL is the full dsp_icpc; LGDSP_GROUP_PZTRAP is BASELINE.json config 2
 * (blmean, t0, t50, e_trap, e_10410 and what they depend on). */
#define LGDSP_GROUP_BASE   0x01u  /* saturation, baseline stats, e_max/e_min, tailstats, PZ, pz_stats */
#define LGDSP_GROUP_TIMING 0x02u  /* t0, t10..t99, drift_time, t0_inv */
#define LGDSP_GROUP_TRAPS  0x04u  /* e_10410, e_535, e_313, *_inv, e_trap, e_trap_max, t_trap_max */
#define LGDSP_GROUP_QDRIFT 0x08u  /* qdrift, lq */
#define LGDSP_GROUP_CUSPZAC 0x10u /* e_cusp, e_zac, e_*_max, t_*_max */
#define LGDSP_GROUP_CURRENT 0x20u /* a_sg, a_60, a_100, a_raw */
#define LGDSP_GROUP_INTRACE 0x40u /* inTrace_intersect, inTrace_n, t50_current (masks on the sg[0] trace) */
#define LGDSP_GROUP_ALL    0x7Fu
#define LGDSP_GROUP_PZTRAP (LGDSP_GROUP_BASE | LGDSP_GROUP_TIMING | LGDSP_GROUP_TRAPS)
/* modifier of LGDSP_GROUP_PZTRAP (split pipeline only): compute nothing but {blmean, t0, t50, e_trap, e_10410} -- no tail
 * statistics, no t10/t80/t90/t99, no e_535/e_313/inverted traces, no trapezoid maxima; every other column is 0 or unspecified
 * (BASELINE.json configs[1]: "pole-zero + trapezoidal energy/t0 only") */
#define LGDSP_GROUP_LEAN   0x80u
#define LGDSP_GROUP_PZTRAP_LEAN (LGDSP_GROUP_PZTRAP | LGDSP_GROUP_LEAN)

/* TrapezoidalChargeFilter(avgtime, gaptime, avgtime2) in samples [RDDSP]:
 * out[j] = mean(y[j+navg+ngap .. j+navg+ngap+navg2-1]) - mean(y[j .. j+navg-1]), j = 0 .. n-L, L = navg+ngap+navg2;
 * trace index j carries the time of sample j+L-1 (trailing edge). */
typedef struct lgdsp_trap {
    int32_t navg, ngap, navg2, reserved;
} lgdsp_trap;

/* SignalEstimator(PolynomialDNI(degree, length)) [RDDSP]; A is the least-squares fit matrix
 * (n_w x (degree+1), row-major): coef_j = sum_i A[i*(degree+1)+j] * y[from+i], value = sum_j coef_j u^j with
 * u = p - from, p the fractional trace index, from = clamp(round_half_even(p) - n_w/2, 0, n_trace-n_w). */
typedef struct lgdsp_dni {
    int32_t n_w, degree;
    double A[LGDSP_MAX_DNI * (LGDSP_MAX_DNI_DEG + 1)];
} lgdsp_dni;

/* SavitzkyGolayFilter(length, degree, 1) [RDDSP] as a valid-mode correlation:
 * s[j] = sum_k h[k] * y[j+k], j = 0 .. n-n_taps; trace index j carries the time of sample j+offset. */
typedef struct lgdsp_sg {
    int32_t n_taps, offset;
    double h[LGDSP_MAX_SG];
} lgdsp_sg;

/* CUSPChargeFilter / ZACChargeFilter(sigma, toplen, tau, length, beta) [RDDSP], in samples.
 * The FIR is  out[j] = sum_k coeffs[k] * y[j+L-1-k]  (valid convolution), trace index j <-> sample j+L-1.
 * `coeffs` must be what lgdsp_cusp_coeffs / lgdsp_zac_coeffs produce for the same (sigma, flat, tau, L,
 * beta): the device path evaluates the filter through its analytic structure (sliding exponential and
 * polynomial windows), the coefficient array is used for the pick-off window and by the direct mode. */
typedef struct lgdsp_cuspzac {
    int32_t n_taps;  /* L = round(length/dt) */
    int32_t flat;    /* round(toplen/dt) */
    double sigma;    /* sigma/dt */
    double tau;      /* tau/dt */
    double beta;     /* scaling factor as passed by the reference (length/dt, src/dsp_icpc.jl:88,90) */
    double coeffs[LGDSP_MAX_FIR];
} lgdsp_cuspzac;

typedef struct lgdsp_icpc_params {
    uint32_t struct_size;      /* sizeof(lgdsp_icpc_params), checked */
    uint32_t version;          /* LGDSP_PARAMS_VERSION */
    int32_t n_samples;         /* samples per waveform, <= LGDSP_MAX_SAMPLES, multiple of 8 */
    uint32_t groups;           /* LGDSP_GROUP_* mask */
    double t_first_ns;         /* time of sample 0 (first(wvfs[1].time)) */
    double dt_ns;              /* step(wvfs[1].time) */

    /* saturation(wvf, low, high): src/dsp_icpc.jl:93-95; compared with the raw integer samples */
    int64_t sat_low, sat_high;

    /* windows as 0-based inclusive sample index ranges (reference: 1-based, src/tailstats.jl:16-18) */
    int32_t bl_from, bl_until;       /* config.bl_window */
    int32_t tail_from, tail_until;   /* config.tail_window */

    /* InvCRFilter(tau): y[i] = y[i-1] + x[i]/alpha - x[i-1], alpha = RC/(RC+1), RC = tau/dt;
     * closed form y[i] = x[i] + pz_km1 * sum_{j<=i} x[j]  with pz_km1 = 1/alpha - 1 */
    double pz_km1;

    /* get_t0: src/dsp_routines.jl:9-25, called at src/dsp_icpc.jl:126 and :207 (inverted, default flt_pars) */
    lgdsp_trap t0_trap;
    lgdsp_trap t0inv_trap;
    double t0_threshold;
    int32_t t0_min_n;          /* max(1, round(t0_mintot/dt)) */
    int32_t tx_min_n;          /* max(1, round(tx_mintot/dt)) */
    double tx_frac[5];         /* 0.1, 0.5, 0.8, 0.9, 0.99  (src/dsp_icpc.jl:132-136) */

    /* get_qdrift: src/dsp_routines.jl:51-64; first/last of the integration-length range in ns */
    double qdrift_first_ns, qdrift_last_ns;
    double lq_first_ns, lq_last_ns;
    lgdsp_dni int_dni;         /* PolynomialDNI(int_interpolation_order, int_interpolation_length) */
    lgdsp_dni sig_dni;         /* PolynomialDNI(sig_interpolation_order, sig_interpolation_length) */

    /* energy filters: src/dsp_icpc.jl:147-178 */
    lgdsp_trap trap_10410, trap_535, trap_313, trap_e;
    double trap_pickoff_ns;    /* trap_rt + trap_ft/2 */
    double cusp_pickoff_ns;    /* flt_length_cusp/2 */
    double zac_pickoff_ns;     /* flt_length_zac/2 */

    /* currents: src/dsp_icpc.jl:181-195; index 0: sg_wl, 1: 60 ns, 2: 100 ns */
    lgdsp_sg sg[3];
    /* current_window as 0-based inclusive index ranges in the index space of each trace:
     * 0..2: the three SG traces, 3: DerivativeFilter trace (same axis as the waveform) */
    int32_t cur_from[4], cur_until[4];

    /* get_intracePileUp: src/dsp_routines.jl:72-82, on the sg[0] trace */
    double intrace_nsigma;
    int32_t intrace_min_n;
    int32_t intrace_bl_from, intrace_bl_until;  /* sigma window in sg[0]-trace index space */

    /* 0: evaluate CUSP/ZAC through their analytic structure (default); 1: direct FIR with `coeffs` */
    int32_t cuspzac_direct;
    int32_t reserved0;

    lgdsp_cuspzac cusp, zac;
} lgdsp_icpc_params;

/* ---- SiPM / PMT trigger chain: dsp_sipm(data, config, pars_optimization)  /root/reference/src/dsp_sipm.jl:47-158 ----
 * scalar output columns (double rows[n_events][LGDSP_SIPM_NCOL]); t_* in microseconds (:145), the rest in ADC units /
 * per ns; the four n_trig_* columns are the lengths of the event's trigger lists (exact small integers) */
enum lgdsp_sipm_col {
    LGDSP_SIPM_t_max = 0, LGDSP_SIPM_t_min, LGDSP_SIPM_t_max_lar, LGDSP_SIPM_t_min_lar,
    LGDSP_SIPM_e_max, LGDSP_SIPM_e_min, LGDSP_SIPM_e_max_lar, LGDSP_SIPM_e_min_lar,
    LGDSP_SIPM_blmean, LGDSP_SIPM_blsigma, LGDSP_SIPM_blslope, LGDSP_SIPM_bloffset,
    LGDSP_SIPM_wfmean, LGDSP_SIPM_wfsigma, LGDSP_SIPM_wfslope, LGDSP_SIPM_wfoffset,
    LGDSP_SIPM_threshold, LGDSP_SIPM_threshold_DC, LGDSP_SIPM_threshold_trap, LGDSP_SIPM_threshold_DC_trap,
    LGDSP_SIPM_n_trig, LGDSP_SIPM_n_trig_DC, LGDSP_SIPM_n_trig_trap, LGDSP_SIPM_n_trig_DC_trap,
    LGDSP_SIPM_NCOL /* = 24 */
};
/* trigger lists (variable length per event, VectorOfVectors in the reference :150-157): list 0 = SG triggers
 * (trig_pos, trig_max), 1 = SG discharge triggers, 2 = trap triggers (pos, pos_high, pos_tot, max), 3 = trap discharge
 * triggers; every list entry has the four fields of IntersectMaximum's result (x, x_high, x_tot, max;
 * src/intersect_maximum.jl:112-118), times in ns.  Padded layout: double trig[n_events][4 lists][4 fields][max_triggers];
 * entries beyond the event's count are 0.  The count columns hold the TRUE counts: a count > max_triggers means the
 * lists were cut and the call should be repeated with a larger capacity. */
#define LGDSP_SIPM_NLIST 4
#define LGDSP_SIPM_NFIELD 4
#define LGDSP_SAMPLE_U16 2
#define LGDSP_SAMPLE_F32 4
#define LGDSP_SAMPLE_F64 8

typedef struct lgdsp_sipm_params {
    uint32_t struct_size;      /* sizeof(lgdsp_sipm_params), checked */
    uint32_t version;          /* LGDSP_PARAMS_VERSION */
    int32_t n_samples;         /* samples per waveform, <= LGDSP_MAX_SAMPLES (any count, no alignment rule) */
    int32_t sample_kind;       /* LGDSP_SAMPLE_U16 (raw ADC) or LGDSP_SAMPLE_F32 */
    double t_first_ns, dt_ns;
    /* TruncateFilter(t0_hpge_window) [RDDSP] as 0-based inclusive sample range (:94-95) */
    int32_t trunc_from, trunc_until;
    /* SavitzkyGolayFilter(pars_optimization.sg.wl, sg_flt_degree, 1)  (:99) */
    lgdsp_sg sg;
    /* SG pipeline (:103-105, :120-121): IntersectMaximum(min_tot_intersect, max_tot_intersect) in samples,
     * thresholdstats_mad bounds and n_sigma factors */
    int32_t sg_min_n, sg_max_n;
    double sg_min_thr, sg_max_thr, sg_nsigma;
    double sg_min_dc, sg_max_dc, sg_nsigma_dc;
    /* trap pipeline (:125-139): InvCRFilter(pz_tau) as pz_km1 (see lgdsp_icpc_params), TrapezoidalChargeFilter(rt, ft) */
    lgdsp_trap trap;
    double pz_km1;
    int32_t trap_min_n, trap_max_n;
    double trap_min_thr, trap_max_thr, trap_nsigma;
    double trap_min_dc, trap_max_dc, trap_nsigma_dc;
    int32_t max_triggers;      /* capacity of every trigger list, 1 .. LGDSP_SIPM_MAX_TRIGGERS */
    int32_t reserved0;
} lgdsp_sipm_params;
#define LGDSP_SIPM_MAX_TRIGGERS 1024

/* ---- MultiIntersect(threshold_ratios, mintot, n, d, sampling_rate)(wvf)  /root/reference/src/multi_intersect.jl:10-121 ----
 * first crossings of the thresholds ratios[j] * maximum(Y) (sequential search: threshold j+1 is looked for from the crossing
 * of threshold j on, :59-73), each refined by a least-squares polynomial of `degree` over the 2*half_window samples around the
 * crossing, up-sampled by `rate` (:81-101) */
#define LGDSP_MI_MAX_THR 128
#define LGDSP_MI_MAX_HALF 8
typedef struct lgdsp_multi_intersect_params {
    uint32_t struct_size;      /* sizeof(lgdsp_multi_intersect_params), checked */
    uint32_t version;          /* LGDSP_PARAMS_VERSION */
    int32_t n_samples;         /* samples per trace (doubles), any count >= 2 */
    int32_t n_thresholds;      /* 1 .. LGDSP_MI_MAX_THR */
    double t_first_ns, dt_ns;
    int32_t min_n;             /* max(1, round(mintot/dt)) */
    int32_t half_window;       /* n: the fit window is pos-n .. pos+n-1; 1 .. LGDSP_MI_MAX_HALF */
    int32_t degree;            /* d <= LGDSP_MAX_DNI_DEG, d < 2n */
    int32_t rate;              /* sampling_rate >= 1, 2n*rate <= 256 */
    double ratios[LGDSP_MI_MAX_THR];
    double A[2 * LGDSP_MI_MAX_HALF * (LGDSP_MAX_DNI_DEG + 1)];   /* lgdsp_lsq_fit_matrix(2n, degree), row-major */
} lgdsp_multi_intersect_params;

/* one point of a trapezoidal sweep: filter + pick-off.
 * pickoff_mode 0: fixed time pickoff_ns (dsp_trap_rt_optimization: enc_pickoff_trap);
 * pickoff_mode 1: t50 + pickoff_ns (dsp_trap_ft_optimization: t50 + rt + ft/2), t50 found on the PZ
 * waveform at 0.5*maximum(PZ waveform) with tx_min_n (src/dsp_filter_optimization.jl:260). */
typedef struct lgdsp_trap_variant {
    lgdsp_trap trap;
    double pickoff_ns;
    int32_t pickoff_mode;
    int32_t reserved;
} lgdsp_trap_variant;

typedef struct lgdsp_sweep_params {
    uint32_t struct_size;
    uint32_t version;
    int32_t n_samples;
    int32_t tx_min_n;
    double t_first_ns, dt_ns;
    int32_t bl_from, bl_until;
    double pz_km1;
    lgdsp_dni sig_dni;
    int32_t out_f64;       /* 0: float output (the ft sweeps' Union{Missing,Float32} matrices, :263); 1: double output
                              (the rt sweeps' zeros(Float64, ...), :122, and dsp_sg_optimization) */
    int32_t reserved0;
} lgdsp_sweep_params;

/* one point of a general filter sweep:
 * kind 0  TrapezoidalChargeFilter(`trap`), value = SignalEstimator at the pick-off            (:109-127, :264-270)
 * kind 1  FIR `coeffs[n_taps]` as produced by lgdsp_cusp_coeffs / lgdsp_zac_coeffs (valid convolution, trailing-edge
 *         time axis), value = SignalEstimator at the pick-off                                  (:173-176, :316-318)
 * kind 2  SavitzkyGolayFilter taps `coeffs[n_taps]` (valid correlation, trace index j <-> sample j + sg_offset),
 *         value = get_wvf_maximum of the trace inside [win_from, win_until] (trace indices)      (:432-433)
 * pick-off (kinds 0/1): pickoff_mode 0: fixed time pickoff_ns; 1: t50 + pickoff_ns, t50 on the PZ waveform at half its
 * maximum with tx_min_n (:260). */
typedef struct lgdsp_sweep_variant {
    int32_t kind;
    int32_t pickoff_mode;
    double pickoff_ns;
    lgdsp_trap trap;
    int32_t n_taps;
    int32_t sg_offset;
    int32_t win_from, win_until;
    const double* coeffs;      /* host pointer, read during the call only */
} lgdsp_sweep_variant;

/* synthetic ICPC waveform generator (SURVEY.md 8d): counter-based Philox4x32-10, identical on host and device */
typedef struct lgdsp_synth_params {
    uint64_t seed;
    int32_t n_samples;
    int32_t mode;          /* 0: mixed population (SURVEY 8d); 1: the reference's noise-free fixture
                              (test/test_dsp_icpc.jl:11-32) for every event */
    double noise_sigma;    /* ADC, default 3.0 */
    double tau_samples;    /* decay constant in samples, default 31250 */
} lgdsp_synth_params;

typedef struct lgdsp_handle lgdsp_handle;

/* ---- library / handle ---- */
const char* lgdsp_version(void);
/* last error message of the handle (or of the last failed lgdsp_create when handle == NULL) */
const char* lgdsp_last_error(const lgdsp_handle* h);
/* create a handle on CUDA device `device`; stream = 0 creates an own NON-BLOCKING stream (it does not synchronise with
 * the legacy default stream: work the caller enqueued elsewhere on the buffers of a *_device call must be complete, and the
 * caller reads results after lgdsp_synchronize), otherwise a cudaStream_t to launch on (e.g. torch's current stream) */
int lgdsp_create(int device, void* stream, lgdsp_handle** out);
void lgdsp_destroy(lgdsp_handle* h);
/* number of kernels this handle has launched so far (for bench bookkeeping) */
int64_t lgdsp_launch_count(const lgdsp_handle* h);
/* block until all work submitted by the handle has finished */
int lgdsp_synchronize(lgdsp_handle* h);

/* ---- host-side filter construction (pure CPU, no handle) ---- */
int lgdsp_lsq_fit_matrix(int32_t n, int32_t degree, double* A /* n*(degree+1) */);
int lgdsp_sg_coeffs(int32_t n_taps, int32_t degree, int32_t derivative, double* h /* n_taps */);
int lgdsp_cusp_coeffs(double sigma, int32_t flat, double tau, int32_t n_taps, double beta, double* c);
int lgdsp_zac_coeffs(double sigma, int32_t flat, double tau, int32_t n_taps, double beta, double* c);

/* ---- dsp_icpc ---- */
/* waveforms on the HOST: wf[e*ld_samples + i], i < n_samples; out_rows: host double[n_events][LGDSP_NCOL].
 * Copies in chunks overlapped with compute and blocks until the result is in out_rows.  Page-locked caller memory
 * (cudaHostAlloc / cudaHostRegister) is copied directly; pageable memory is packed into the handle's pinned double buffers by
 * LGDSP_COPY_THREADS host threads (default: half the cores, at most 8) so that the copies stay asynchronous. */
int lgdsp_icpc_run(lgdsp_handle* h, const lgdsp_icpc_params* p, const uint16_t* wf, int64_t n_events,
                   int64_t ld_samples, double* out_rows);
/* waveforms and output rows in DEVICE memory (wf 16-byte aligned, ld_samples multiple of 8); asynchronous
 * on the handle's stream */
int lgdsp_icpc_run_device(lgdsp_handle* h, const lgdsp_icpc_params* p, const uint16_t* d_wf, int64_t n_events,
                          int64_t ld_samples, double* d_out_rows);
/* ---- decode_data: LegendDataTypes.jl `decode_data(encoded_waveforms)`, called at /root/reference/src/dsp_icpc.jl:313-314,
 * src/dsp_puls.jl:103, src/dsp_sipm.jl:241 ----
 * Encoded waveform sets are a byte buffer `enc` plus `offsets[n_events + 1]` (the element pointers of the reference's
 * VectorOfEncodedArrays): event e occupies enc[offsets[e] .. offsets[e+1]).  codec = LGDSP_CODEC_RADWARE (RadwareSigcompress(shift),
 * 16-bit samples; the reference uses shift = -32768 for UInt16 waveforms) or LGDSP_CODEC_ULEB128ZZD (16- / 32-bit samples).
 * A malformed stream makes the call return LGDSP_ERR_INVALID_ARG (device entry: status[e] = 1, zero-filled waveform). */
int64_t lgdsp_codec_max_encoded_bytes(int32_t codec, int32_t n_samples, int32_t sample_bytes);
/* host-side encoder (tests, benchmarks, round trips): fills enc and offsets; LGDSP_ERR_OOM when enc_capacity is too small */
int lgdsp_codec_encode_host(int32_t codec, const void* wf, int32_t sample_bytes, int64_t n_events, int32_t n_samples, int64_t ld_samples,
                            int32_t shift, uint8_t* enc, int64_t enc_capacity, int64_t* offsets);
/* device buffers, asynchronous on the handle's stream; d_status (int32[n_events], may be NULL) */
int lgdsp_decode_data_device(lgdsp_handle* h, int32_t codec, const uint8_t* d_enc, const int64_t* d_offsets, int64_t n_events,
                             int32_t n_samples, int32_t shift, void* d_wf, int32_t sample_bytes, int64_t ld_samples, int32_t* d_status);
/* host buffers: encoded bytes in, decoded samples out (chunked; blocks until wf is filled) */
int lgdsp_decode_data(lgdsp_handle* h, int32_t codec, const uint8_t* enc, const int64_t* offsets, int64_t n_events, int32_t n_samples,
                      int32_t shift, void* wf, int32_t sample_bytes, int64_t ld_samples);
/* dsp_icpc on encoded waveforms in HOST memory: only the codec's bytes cross the host link, decode_data runs on the device in front
 * of the chain (n_samples from the parameters; baseline as lgdsp_icpc_run_ext, may be NULL) */
int lgdsp_icpc_run_encoded(lgdsp_handle* h, const lgdsp_icpc_params* p, int32_t codec, const uint8_t* enc, const int64_t* offsets,
                           int32_t shift, int32_t sample_bytes, const double* baseline, int64_t n_events, double* out_rows);

/* dsp_icpc_compressed with both `decode_data` calls of /root/reference/src/dsp_icpc.jl:313-314 on the device: the presummed
 * and the windowed waveforms arrive as encoded streams in host memory (in LEGEND data: ULEB128ZZD for the 32-bit presummed
 * samples, RadwareSigcompress(-32768) for the windowed UInt16 samples); everything else as lgdsp_icpc_compressed_run */
int lgdsp_icpc_compressed_run_encoded(lgdsp_handle* h, const lgdsp_icpc_params* p_pre, const lgdsp_icpc_params* p_wdw,
                                      int32_t pre_codec, const uint8_t* enc_pre, const int64_t* off_pre, int32_t pre_shift,
                                      int32_t pre_sample_bytes, int32_t wdw_codec, const uint8_t* enc_wdw, const int64_t* off_wdw,
                                      int32_t wdw_shift, int32_t wdw_sample_bytes, double presum_rate, const int32_t* aux_windows,
                                      int64_t n_events, double* rows_pre, double* rows_wdw, double* stats);

/* dsp_icpc_compressed building block (/root/reference/src/dsp_icpc.jl:293-499): the same chain on waveforms of
 * 16-bit (sample_bytes = 2) or 32-bit unsigned samples (sample_bytes = 4: presummed traces, n_samples <=
 * LGDSP_MAX_SAMPLES/2), with an optional per-event EXTERNAL baseline: when baseline != NULL the waveform is shifted by
 * -baseline[e] instead of by its own bl_window mean -- the windowed waveform of the compressed format is shifted by the
 * presummed waveform's baseline / presum_rate (:349-350).  blmean..bloffset still report the statistics of the
 * waveform's own bl_window.
 * Range of 32-bit samples: the prefix sums are exact uint32 arithmetic, so a waveform must sum to < 2^32 (presummed 16-bit
 * traces of <= 4096 samples do up to a mean of 2^20, i.e. any presum rate <= 16).  An event beyond that gets a row of NaN
 * (all 49 columns; sweep outputs likewise) instead of wrapped sums. */
int lgdsp_icpc_run_ext(lgdsp_handle* h, const lgdsp_icpc_params* p, const void* wf, int32_t sample_bytes,
                       const double* baseline, int64_t n_events, int64_t ld_samples, double* out_rows);
int lgdsp_icpc_run_ext_device(lgdsp_handle* h, const lgdsp_icpc_params* p, const void* d_wf, int32_t sample_bytes,
                              const double* d_baseline, int64_t n_events, int64_t ld_samples, double* d_out_rows);

/* signalstats.(wvfs, from, until) on several windows of every waveform: the auxiliary baseline / pole-zero windows of
 * dsp_icpc_compressed (:338-339 on the raw waveform, :365-366 on the baseline-subtracted one: pass shift = blmean).
 * windows: HOST int32[n_windows][2], 0-based inclusive sample ranges; shift: NULL or double[n_events], subtracted from
 * the samples; out: double[n_events][n_windows][LGDSP_NSTAT] = (mean, sigma, slope [1/ns], offset,
 * slope_residual_sigma).  slope_residual_sigma = population sigma of the residuals of the straight-line fit
 * (RadiationDetectorDSP's definition is not in the reference tree: parity unpinned). */
#define LGDSP_NSTAT 5
#define LGDSP_MAX_STAT_WINDOWS 16
int lgdsp_window_stats_run(lgdsp_handle* h, const void* wf, int32_t sample_bytes, int64_t n_events, int32_t n_samples,
                           int64_t ld_samples, double t_first_ns, double dt_ns, const double* shift,
                           const int32_t* windows, int32_t n_windows, double* out);
int lgdsp_window_stats_run_device(lgdsp_handle* h, const void* d_wf, int32_t sample_bytes, int64_t n_events,
                                  int32_t n_samples, int64_t ld_samples, double t_first_ns, double dt_ns,
                                  const double* d_shift, const int32_t* windows, int32_t n_windows, double* d_out);

/* ---- dsp_icpc_compressed(data, config, tau, pars_filter)  /root/reference/src/dsp_icpc.jl:293-499 ----
 * Every event has a presummed waveform (energies, tail, saturation, in-trace pile-up; step = presum_rate x ADC step)
 * and a windowed waveform (t0, t10..t99, Q-drift, currents).  p_pre / p_wdw: the constants of the two time axes (NULL
 * reuses the previous call's).  The library runs the fused chain on the presummed batch, signalstats on the five
 * windows (auxbl1, auxbl2, bl_window on the raw trace; auxpz1, auxpz2 on the baseline-subtracted trace, :338-339, :346,
 * :365-366) and the fused chain on the windowed batch shifted by -blmean_pre / presum_rate (:350).
 * aux_windows: HOST int32[4][2] = auxbl1, auxbl2, auxpz1, auxpz2 as 0-based inclusive sample ranges of the presummed
 * axis.  Outputs: rows_pre, rows_wdw: double[n_events][LGDSP_NCOL] (the caller picks the columns the reference takes
 * from each waveform, :463-499); stats: double[n_events][5][LGDSP_NSTAT] in the window order auxbl1, auxbl2, bl,
 * auxpz1, auxpz2. */
int lgdsp_icpc_compressed_run(lgdsp_handle* h, const lgdsp_icpc_params* p_pre, const lgdsp_icpc_params* p_wdw,
                              const void* wf_pre, int32_t pre_sample_bytes, int64_t ld_pre, const void* wf_wdw,
                              int32_t wdw_sample_bytes, int64_t ld_wdw, double presum_rate, const int32_t* aux_windows,
                              int64_t n_events, double* rows_pre, double* rows_wdw, double* stats);
int lgdsp_icpc_compressed_run_device(lgdsp_handle* h, const lgdsp_icpc_params* p_pre, const lgdsp_icpc_params* p_wdw,
                                     const void* d_wf_pre, int32_t pre_sample_bytes, int64_t ld_pre, const void* d_wf_wdw,
                                     int32_t wdw_sample_bytes, int64_t ld_wdw, double presum_rate,
                                     const int32_t* aux_windows, int64_t n_events, double* d_rows_pre, double* d_rows_wdw,
                                     double* d_stats);

/* upload/validate params once and reuse them for many _device calls (avoids the per-call upload);
 * pass p == NULL to lgdsp_icpc_run_device afterwards */
int lgdsp_icpc_set_params(lgdsp_handle* h, const lgdsp_icpc_params* p);
/* execution path of every dsp_icpc pass of this handle (results are the same values):
 *   1 (default) split pipeline: prefix / extract / CUSP-ZAC kernels coupled through a ring of float64 prefix sums that stays in
 *     L2; `batch` = events per sub-batch (<= 0: default, 6 per SM), `streams` = side streams the sub-batches alternate on
 *     (<= 0: default 2, at most 4);
 *   0 fused: one launch of the single-kernel chain (round-1 path, kept for cross-checks).
 * Environment overrides at lgdsp_create: LGDSP_ICPC_PATH=fused|split, LGDSP_SPLIT_BATCH, LGDSP_SPLIT_STREAMS. */
int lgdsp_icpc_set_path(lgdsp_handle* h, int32_t path, int64_t batch, int32_t streams);

/* ---- trapezoidal sweeps ---- */
/* out: float[n_events][n_variants], i.e. the memory layout of the reference's column-major Julia matrix
 * (n_variants x n_events), Float32 as src/dsp_filter_optimization.jl:263 */
int lgdsp_trap_sweep_run(lgdsp_handle* h, const lgdsp_sweep_params* p, const uint16_t* wf, int64_t n_events,
                         int64_t ld_samples, const lgdsp_trap_variant* variants, int32_t n_variants, float* out);
int lgdsp_trap_sweep_run_device(lgdsp_handle* h, const lgdsp_sweep_params* p, const uint16_t* d_wf,
                                int64_t n_events, int64_t ld_samples, const lgdsp_trap_variant* variants,
                                int32_t n_variants, float* d_out);

/* general sweep: out is float or double [n_events][n_variants] (lgdsp_sweep_params.out_f64); aux, when not NULL,
 * receives double[n_events][4] = (blmean, blslope [1/ns], t50 [us], 0) -- the extra columns of dsp_sg_optimization's
 * result table (:435-439) */
int lgdsp_sweep_run(lgdsp_handle* h, const lgdsp_sweep_params* p, const uint16_t* wf, int64_t n_events, int64_t ld_samples,
                    const lgdsp_sweep_variant* variants, int32_t n_variants, void* out, double* aux);
int lgdsp_sweep_run_device(lgdsp_handle* h, const lgdsp_sweep_params* p, const uint16_t* d_wf, int64_t n_events,
                           int64_t ld_samples, const lgdsp_sweep_variant* variants, int32_t n_variants, void* d_out,
                           double* d_aux);
/* dsp_sg_optimization_compressed building block (/root/reference/src/dsp_filter_optimization.jl:460-511): the same sweep on
 * waveforms of 16-bit (sample_bytes = 2) or 32-bit unsigned samples (4: presummed traces, n_samples <= LGDSP_MAX_SAMPLES/2)
 * with an optional per-event EXTERNAL baseline: when baseline != NULL the waveform is shifted by -baseline[e] instead of
 * by its own bl_window mean (:476-477: the windowed waveform is shifted by the presummed baseline / presum_rate).  The aux
 * outputs keep the statistics of the waveform's own bl_window. */
int lgdsp_sweep_run_ext(lgdsp_handle* h, const lgdsp_sweep_params* p, const void* wf, int32_t sample_bytes, const double* baseline,
                        int64_t n_events, int64_t ld_samples, const lgdsp_sweep_variant* variants, int32_t n_variants, void* out,
                        double* aux);
int lgdsp_sweep_run_ext_device(lgdsp_handle* h, const lgdsp_sweep_params* p, const void* d_wf, int32_t sample_bytes,
                               const double* d_baseline, int64_t n_events, int64_t ld_samples,
                               const lgdsp_sweep_variant* variants, int32_t n_variants, void* d_out, double* d_aux);

/* ---- dsp_sipm ---- */
/* wf: n_events waveforms of `sample_kind` samples, row stride ld_samples (in samples); rows: double[n_events][
 * LGDSP_SIPM_NCOL]; trig: double[n_events][4][4][max_triggers] (see above).  Host buffers / device buffers. */
int lgdsp_sipm_run(lgdsp_handle* h, const lgdsp_sipm_params* p, const void* wf, int64_t n_events, int64_t ld_samples,
                   double* rows, double* trig);
int lgdsp_sipm_run_device(lgdsp_handle* h, const lgdsp_sipm_params* p, const void* d_wf, int64_t n_events,
                          int64_t ld_samples, double* d_rows, double* d_trig);
/* trigger list `list` (0..3) of a finished lgdsp_sipm_run_device call in the reference's VectorOfVectors form, on the
 * device: d_elem_ptr: int64[n_events + 1] (element pointers, 0-based; d_elem_ptr[n_events] = total number of triggers),
 * d_flat: double[4 fields][flat_stride] with the entries of event e at [d_elem_ptr[e], d_elem_ptr[e+1]).  Two calls:
 * lgdsp_sipm_list_pointers_device fills d_elem_ptr and returns the total in *total (synchronises), then the caller
 * provides d_flat with flat_stride >= total and calls lgdsp_sipm_list_gather_device.  Lists cut at max_triggers stay cut. */
int lgdsp_sipm_list_pointers_device(lgdsp_handle* h, const double* d_rows, int64_t n_events, int32_t list, int32_t max_triggers,
                                    int64_t* d_elem_ptr, int64_t* total);
int lgdsp_sipm_list_gather_device(lgdsp_handle* h, const double* d_trig, int64_t n_events, int32_t list, int32_t max_triggers,
                                  const int64_t* d_elem_ptr, double* d_flat, int64_t flat_stride);
/* the in-tree primitives of the chain on single traces of doubles (host buffers; one trace per call, for tests and
 * small jobs; n = 0 .. 65536): thresholdstats / thresholdstats_mad (src/thresholdstats.jl:19-41, 61-71) and IntersectMaximum
 * (src/intersect_maximum.jl:24-119; x/x_high/x_tot/max: double[max_triggers], returns the count in *n_found).  Both are
 * n_events = 1 calls of lgdsp_wfstats_run. */
int lgdsp_thresholdstats(lgdsp_handle* h, const double* y, int32_t n, double min, double max, int32_t mad, double* out);
int lgdsp_intersect_maximum(lgdsp_handle* h, const double* y, int32_t n, double t_first_ns, double dt_ns, double threshold,
                            int32_t min_n, int32_t max_n, int32_t max_triggers, double* x, double* x_high, double* x_tot,
                            double* max, int32_t* n_found);

/* ---- per-waveform primitives on whole waveform arrays: the broadcasts f.(wvfs, ...) of the in-tree primitives ----
 * One pass over each waveform computes every primitive selected in `what`; every window is a 0-based inclusive sample range
 * and must lie inside [0, n_samples-1] for a selected primitive (the reference's @assert, src/tailstats.jl:23-25).
 * Times (tmin, tmax, tail_tau, the IntersectMaximum x / x_high / x_tot) are in ns on the axis X[i] = t_first + i*dt. */
#define LGDSP_WFSTAT_SATURATION         0x01u   /* saturation(wvf, low, high[, start, stop])   src/saturation.jl:12-65; U16 only */
#define LGDSP_WFSTAT_EXTREMESTATS       0x02u   /* extremestats(wvf[, start, stop])           src/extremestats.jl:14-40 */
#define LGDSP_WFSTAT_TAILSTATS          0x04u   /* tailstats(wvf, start, stop)                src/tailstats.jl:13-72 */
#define LGDSP_WFSTAT_WVF_MAXIMUM        0x08u   /* get_wvf_maximum(wvf, start, stop)          src/interpolation.jl:21-46 */
#define LGDSP_WFSTAT_THRESHOLDSTATS     0x10u   /* thresholdstats(wvf, min, max)              src/thresholdstats.jl:19-41 */
#define LGDSP_WFSTAT_THRESHOLDSTATS_MAD 0x20u   /* thresholdstats_mad(wvf, min, max)          src/thresholdstats.jl:61-71 */
#define LGDSP_WFSTAT_INTERSECT_MAXIMUM  0x40u   /* IntersectMaximum(mintot, maxtot)(wvf, thr) src/intersect_maximum.jl:24-119 */
#define LGDSP_WFSTAT_ALL                0x7Fu
/* output rows: double rows[n_events][LGDSP_WFSTAT_NCOL]; columns of unselected primitives are 0.  The saturation counts and
 * the multiplicity are exact small integers; the multiplicity is the TRUE number of triggers (a value > max_triggers means
 * the lists were cut and the call should be repeated with a larger capacity). */
enum lgdsp_wfstat_col {
    LGDSP_WFSTAT_sat_low = 0, LGDSP_WFSTAT_sat_high, LGDSP_WFSTAT_sat_max_cons_low, LGDSP_WFSTAT_sat_max_cons_high,
    LGDSP_WFSTAT_min, LGDSP_WFSTAT_max, LGDSP_WFSTAT_tmin, LGDSP_WFSTAT_tmax,
    LGDSP_WFSTAT_tail_mean, LGDSP_WFSTAT_tail_sigma, LGDSP_WFSTAT_tail_tau,
    LGDSP_WFSTAT_wvf_max, LGDSP_WFSTAT_thr_sigma, LGDSP_WFSTAT_thr_mad, LGDSP_WFSTAT_multiplicity,
    LGDSP_WFSTAT_NCOL /* = 15 */
};
#define LGDSP_WFSTAT_MAX_SAMPLES 65536
#define LGDSP_WFSTAT_MAX_TRIGGERS 65536

typedef struct lgdsp_wfstats_params {
    uint32_t struct_size;      /* sizeof(lgdsp_wfstats_params), checked */
    uint32_t version;          /* LGDSP_PARAMS_VERSION */
    int32_t n_samples;         /* 0 .. LGDSP_WFSTAT_MAX_SAMPLES */
    int32_t sample_kind;       /* LGDSP_SAMPLE_U16 / _F32 / _F64, converted exactly to double */
    uint32_t what;             /* LGDSP_WFSTAT_* mask, at least one bit */
    int32_t reserved0;
    double t_first_ns, dt_ns;
    int32_t sat_from, sat_until;     /* saturation window */
    int32_t ext_from, ext_until;     /* extremestats window */
    int32_t tail_from, tail_until;   /* tailstats window */
    int32_t max_from, max_until;     /* get_wvf_maximum window */
    int64_t sat_low, sat_high;       /* saturation levels, compared with the raw integer samples */
    double thr_min, thr_max;         /* bounds of thresholdstats / thresholdstats_mad (+-Inf: open) */
    int32_t im_min_n, im_max_n;      /* IntersectMaximum: max(1, round(mintot/dt)), max(1, round(maxtot/dt)) */
    int32_t max_triggers;            /* capacity of every trigger list, 1 .. LGDSP_WFSTAT_MAX_TRIGGERS */
    int32_t reserved1;
} lgdsp_wfstats_params;
/* wf: n_events waveforms of `sample_kind` samples, row stride ld_samples (in samples); thresholds: double[n_events], the
 * IntersectMaximum threshold of every event (read only when it is selected, may be NULL otherwise); rows: see above;
 * lists: double[n_events][4][max_triggers] = x, x_high, x_tot, max of the triggers, zero-filled behind the last one (written
 * only when IntersectMaximum is selected, may be NULL otherwise).  Host buffers (chunked copies, blocks until the results are
 * in rows / lists) / device buffers (asynchronous on the handle's stream). */
int lgdsp_wfstats_run(lgdsp_handle* h, const lgdsp_wfstats_params* p, const void* wf, const double* thresholds, int64_t n_events,
                      int64_t ld_samples, double* rows, double* lists);
int lgdsp_wfstats_run_device(lgdsp_handle* h, const lgdsp_wfstats_params* p, const void* d_wf, const double* d_thresholds,
                             int64_t n_events, int64_t ld_samples, double* d_rows, double* d_lists);

/* MultiIntersect on a batch of traces of doubles: y[e*ld_samples + i]; x: double[n_events][n_thresholds] (ns);
 * flags: int32[n_events], 1 where the reference's boundary assertion (:85-88) fails (that event's x are NaN) */
int lgdsp_multi_intersect_run(lgdsp_handle* h, const lgdsp_multi_intersect_params* p, const double* y, int64_t n_events,
                              int64_t ld_samples, double* x, int32_t* flags);
int lgdsp_multi_intersect_run_device(lgdsp_handle* h, const lgdsp_multi_intersect_params* p, const double* d_y,
                                     int64_t n_events, int64_t ld_samples, double* d_x, int32_t* d_flags);

/* ---- synthetic input ---- */
/* events [first_event, first_event + n_events) of the stream defined by (seed, mode) */
int lgdsp_synth_generate_device(lgdsp_handle* h, const lgdsp_synth_params* sp, int64_t first_event,
                                int64_t n_events, int64_t ld_samples, uint16_t* d_wf);
int lgdsp_synth_generate_host(const lgdsp_synth_params* sp, int64_t first_event, int64_t n_events,
                              int64_t ld_samples, uint16_t* wf);

/* ---- page-locked host memory: buffers allocated / registered here take the direct copy path of the host entry points (no
 * staging through the handle's pinned ring); register once, reuse across calls, unregister before the memory is freed ---- */
int lgdsp_host_alloc(void** p, int64_t bytes);
int lgdsp_host_free(void* p);
int lgdsp_host_register(void* p, int64_t bytes);
int lgdsp_host_unregister(void* p);

/* ---- measurement: device times [ms] of the four kernels of the split dsp_icpc pipeline on one batch run serially on the
 * handle's stream: ms4 = prefix, extract, CUSP/ZAC select, CUSP/ZAC finish (bench.py's roofline shares) ---- */
int lgdsp_icpc_profile_device(lgdsp_handle* h, const uint16_t* d_wf, int64_t n_events, int64_t ld_samples, double* d_out_rows,
                              double* ms4);

/* ---- timing helper: elapsed milliseconds of the last *_device call measured with CUDA events on the
 * handle's stream (valid after lgdsp_synchronize) ---- */
double lgdsp_last_kernel_ms(const lgdsp_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* LGDSP_B200_H */
