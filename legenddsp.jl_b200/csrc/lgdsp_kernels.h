// Host-callable launchers of the CUDA kernels (internal to the library).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "lgdsp_device.cuh"

namespace lgdsp {

// fused dsp_icpc kernel
int icpc_smem_bytes();
int icpc_threads();
cudaError_t icpc_configure(int* max_blocks_per_sm);
// d_bl_ext != NULL: event e is shifted by -(d_bl_ext[e * bl_stride] / bl_div) instead of by its own baseline mean
void icpc_launch(const IcpcDev& P, const void* d_wf, int sample_bytes, long long n_events, long long ld, const double* d_bl_ext,
                 long long bl_stride, double bl_div, double* d_rows, int grid, cudaStream_t stream);
// split pipeline (lgdsp_icpc_split.cuh): resident blocks per SM of {prefix, extract, CUSP/ZAC select}; scratch sizes per event
cudaError_t icpc_split_configure(int* bps3);
long long icpc_split_tt_doubles();
long long icpc_split_aux_doubles();
long long icpc_split_cz_doubles();
void icpc_split_launch_batch(const IcpcDev& P, const void* d_wf, int sample_bytes, long long n_events, long long ld,
                             const double* d_bl_ext, long long bl_stride, double bl_div, double* d_rows, double* d_tt, double* d_aux,
                             double* d_cz, const int* bps3, int sm_count, cudaStream_t stream, cudaStream_t stream_cz,
                             cudaEvent_t ev_prefix, cudaEvent_t ev_cz, cudaEvent_t* marks);
// window w is shifted by -d_shift[e * shift_stride] when d_shift != NULL and bit w of shift_mask is set
void window_stats_launch(const void* d_wf, int sample_bytes, long long n_events, long long ld, double t_first, double dt,
                         const double* d_shift, long long shift_stride, unsigned shift_mask, const int* d_win, int n_windows,
                         double* d_out, cudaStream_t stream);

// trapezoid sweep kernel
struct SweepVar {
    TrapDev t;             // kind 0
    double pick_ns;
    int mode, kind;        // kind 0 trapezoid, 1 FIR on TT (differenced taps), 2 Savitzky-Golay + windowed maximum
    int L;                 // filter length (trap L / FIR taps / SG taps)
    int sg_off, win_from, win_until;
    const double* g;       // device: kind 1: L+1 differenced FIR taps on TT; kind 2: L+1 differenced SG taps on TT
};
struct SweepDev {
    int n, tx_min_n;
    double t_first, dt;
    int bl_from, bl_until;
    double km1;
    DniDev sig_dni;
    const double* dni_A;     // [LGDSP_MAX_DNI*4]
    const SweepVar* vars;    // device array
    int nvar, out_f64;
    int n_other, reserved;   // variants of kind != 0 (0: the per-warp FIR / SG pass is skipped)
    double bl_inv_n, bl_sX, bl_sXX;   // baseline regression constants (aux outputs)
    // one-warp-per-waveform path (lgdsp_sweep_warp.cuh): warp_ok = 1 when every variant is a trapezoid of one pick-off mode
    // and the prefix-sum window the set can reach fits win_steps * 288 samples.  win_mode 1: the first window starts at
    // (crossing sample + win_rel_lo); 0: at win_abs_lo
    int warp_ok, win_steps, win_mode, win_rel_lo, win_abs_lo;
    int dt_pow2;             // dt is a power of two: x / dt == x * rdt bit for bit
    int stream_n, reserved3; // win_mode 0: samples [0, stream_n) cover the baseline window and every look-up of the set
    double rdt;
};
cudaError_t sweep_configure(int* max_blocks_per_sm);
// dni_A_host: the fit matrix on the host (the warp path passes it in the constant bank); sm_count sizes the warp path's grid.
// Returns 1: one-warp-per-waveform kernel launched, 0: one-CTA-per-waveform kernel launched, -1: nothing launched
// (LGDSP_SWEEP_PATH=warp demands the warp path and the variant set is not eligible)
int sweep_launch(const SweepDev& P, const double* dni_A_host, const void* d_wf, int sample_bytes, long long n_events, long long ld,
                 const double* d_bl_ext, void* d_out, double* d_aux, int grid, int sm_count, cudaStream_t stream);
// window capacity of the warp path in samples (0: path unavailable on this device)
int sweep_warp_max_window();

// ---- waveform codecs of decode_data (lgdsp_codec.cu) ----
long long codec_max_encoded_bytes(int codec, int n_samples, int sample_bytes);
int codec_encode_host(int codec, const void* wf, int sample_bytes, long long n_events, int n_samples, long long ld, int shift,
                      uint8_t* enc, long long cap, long long* offsets);
cudaError_t codec_decode_launch(int codec, const uint8_t* d_enc, const long long* d_off, long long off_base, long long n_events,
                                int n_samples, int shift, void* d_out, int sample_bytes, long long ld, int* d_status, int* d_err,
                                int err_base, long long max_stream_bytes, int sm_count, cudaStream_t stream);

// synthetic generator
void synth_launch(const lgdsp_synth_params& sp, long long first_event, long long n_events, long long ld, uint16_t* d_wf,
                  cudaStream_t stream);

// ---- dsp_sipm (lgdsp_sipm.cu) ----
struct SipmDev {
    int n, kind;
    double t_first, dt;
    int trunc_from, trunc_until;
    int sg_taps, sg_off;
    double sgh[LGDSP_MAX_SG];
    int sg_min_n, sg_max_n;
    double sg_min_thr, sg_max_thr, sg_nsigma, sg_min_dc, sg_max_dc, sg_nsigma_dc;
    int ta, tg, ta2, tL;
    double inv1, inv2, km1;
    int trap_min_n, trap_max_n;
    double trap_min_thr, trap_max_thr, trap_nsigma, trap_min_dc, trap_max_dc, trap_nsigma_dc;
    int cap, pad_;
};
cudaError_t sipm_configure(int n, int sample_kind, int* max_blocks_per_sm);
void sipm_launch(const SipmDev& P, const void* d_wf, long long n_events, long long ld, double* d_rows, double* d_trig, int grid,
                 cudaStream_t stream);

// ---- per-waveform primitives on waveform arrays (lgdsp_sipm.cu, lgdsp_wfstats_run) ----
struct WfstatsDev {
    int n, kind;
    unsigned what;
    int cap;
    double t0, dt;
    int sat_from, sat_until, ext_from, ext_until, tail_from, tail_until, max_from, max_until;
    long long sat_low, sat_high;
    double thr_min, thr_max;
    int im_min_n, im_max_n;
};
// shared memory per CTA, whether the trace is staged there, and CTAs per SM of the kernel for (n, kind, what)
cudaError_t wfstats_configure(const WfstatsDev& P, int* max_blocks_per_sm);
// d_work: grid * n doubles, the converted trace of every CTA when it is not staged in shared memory and thresholdstats_mad is
// selected on non-double samples (wfstats_work_doubles(P) > 0), else unused
long long wfstats_work_doubles(const WfstatsDev& P);
void wfstats_launch(const WfstatsDev& P, const void* d_wf, const double* d_thr, long long n_events, long long ld, double* d_rows,
                    double* d_lists, double* d_work, int grid, cudaStream_t stream);

// trigger lists -> flat data + element pointers on the device
void sipm_count_scan_launch(const double* d_rows, long long n_events, int list, int cap, long long* d_elem_ptr, cudaStream_t stream);
void sipm_compact_launch(const double* d_trig, long long n_events, int list, int cap, const long long* d_elem_ptr, double* d_flat,
                         long long flat_stride, cudaStream_t stream);

// ---- MultiIntersect (lgdsp_sipm.cu): one warp per trace ----
struct MiDev {
    int len, n_thr;
    double t0, dt;
    int min_n, n, degree, rate;
    double ratios[LGDSP_MI_MAX_THR];
    double A[2 * LGDSP_MI_MAX_HALF * (LGDSP_MAX_DNI_DEG + 1)];
};
void multi_intersect_launch(const MiDev& P, const double* d_y, long long n_events, long long ld, double* d_x, int* d_flags,
                            cudaStream_t stream);

}  // namespace lgdsp
