"""Loader of the in-tree CUDA library liblgdsp_b200.so (built by build.py / __graft_entry__.build()).

There is NO fallback: if the library is missing this raises; if no CUDA device is usable `Handle()` raises.
"""
import ctypes as C
import os

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LGDSP_B200_LIB") or os.path.join(_HERE, "liblgdsp_b200.so")   # (override: A/B builds of tools/)

_dp = C.POINTER(C.c_double)
_lib = None


class LgdspError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"lgdsp error {code}: {msg}")
        self.code = code


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
            "legenddsp.jl_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.lgdsp_version.restype = C.c_char_p
    L.lgdsp_last_error.restype = C.c_char_p
    L.lgdsp_last_error.argtypes = [vp]
    L.lgdsp_create.argtypes = [C.c_int, vp, C.POINTER(vp)]
    L.lgdsp_destroy.argtypes = [vp]
    L.lgdsp_destroy.restype = None
    L.lgdsp_launch_count.argtypes = [vp]
    L.lgdsp_launch_count.restype = i64
    L.lgdsp_synchronize.argtypes = [vp]
    L.lgdsp_last_kernel_ms.argtypes = [vp]
    L.lgdsp_last_kernel_ms.restype = C.c_double
    L.lgdsp_lsq_fit_matrix.argtypes = [i32, i32, _dp]
    L.lgdsp_sg_coeffs.argtypes = [i32, i32, i32, _dp]
    L.lgdsp_cusp_coeffs.argtypes = [C.c_double, i32, C.c_double, i32, C.c_double, _dp]
    L.lgdsp_zac_coeffs.argtypes = [C.c_double, i32, C.c_double, i32, C.c_double, _dp]
    L.lgdsp_icpc_set_params.argtypes = [vp, C.POINTER(_abi.IcpcParams)]
    L.lgdsp_icpc_set_path.argtypes = [vp, i32, i64, i32]
    L.lgdsp_icpc_profile_device.argtypes = [vp, vp, i64, i64, vp, _dp]
    L.lgdsp_host_alloc.argtypes = [C.POINTER(vp), i64]
    L.lgdsp_host_free.argtypes = [vp]
    L.lgdsp_host_register.argtypes = [vp, i64]
    L.lgdsp_host_unregister.argtypes = [vp]
    L.lgdsp_icpc_run.argtypes = [vp, C.POINTER(_abi.IcpcParams), vp, i64, i64, vp]
    L.lgdsp_icpc_run_device.argtypes = [vp, C.POINTER(_abi.IcpcParams), vp, i64, i64, vp]
    L.lgdsp_icpc_run_ext.argtypes = [vp, C.POINTER(_abi.IcpcParams), vp, i32, vp, i64, i64, vp]
    L.lgdsp_icpc_run_ext_device.argtypes = [vp, C.POINTER(_abi.IcpcParams), vp, i32, vp, i64, i64, vp]
    L.lgdsp_codec_max_encoded_bytes.argtypes = [i32, i32, i32]
    L.lgdsp_codec_max_encoded_bytes.restype = i64
    L.lgdsp_codec_encode_host.argtypes = [i32, vp, i32, i64, i32, i64, i32, vp, i64, vp]
    L.lgdsp_decode_data_device.argtypes = [vp, i32, vp, vp, i64, i32, i32, vp, i32, i64, vp]
    L.lgdsp_decode_data.argtypes = [vp, i32, vp, vp, i64, i32, i32, vp, i32, i64]
    L.lgdsp_icpc_run_encoded.argtypes = [vp, C.POINTER(_abi.IcpcParams), i32, vp, vp, i32, i32, vp, i64, vp]
    L.lgdsp_icpc_compressed_run_encoded.argtypes = [vp, C.POINTER(_abi.IcpcParams), C.POINTER(_abi.IcpcParams), i32, vp, vp, i32, i32,
                                                    i32, vp, vp, i32, i32, C.c_double, vp, i64, vp, vp, vp]
    L.lgdsp_window_stats_run.argtypes = [vp, vp, i32, i64, i32, i64, C.c_double, C.c_double, vp, vp, i32, vp]
    L.lgdsp_window_stats_run_device.argtypes = [vp, vp, i32, i64, i32, i64, C.c_double, C.c_double, vp, vp, i32, vp]
    _comp = [vp, C.POINTER(_abi.IcpcParams), C.POINTER(_abi.IcpcParams), vp, i32, i64, vp, i32, i64, C.c_double, vp, i64,
             vp, vp, vp]
    L.lgdsp_icpc_compressed_run.argtypes = _comp
    L.lgdsp_icpc_compressed_run_device.argtypes = _comp
    L.lgdsp_sipm_run.argtypes = [vp, C.POINTER(_abi.SipmParams), vp, i64, i64, vp, vp]
    L.lgdsp_sipm_run_device.argtypes = [vp, C.POINTER(_abi.SipmParams), vp, i64, i64, vp, vp]
    L.lgdsp_sipm_list_pointers_device.argtypes = [vp, vp, i64, i32, i32, vp, C.POINTER(i64)]
    L.lgdsp_sipm_list_gather_device.argtypes = [vp, vp, i64, i32, i32, vp, vp, i64]
    L.lgdsp_thresholdstats.argtypes = [vp, vp, i32, C.c_double, C.c_double, i32, _dp]
    L.lgdsp_intersect_maximum.argtypes = [vp, vp, i32, C.c_double, C.c_double, C.c_double, i32, i32, i32, vp, vp, vp, vp,
                                          C.POINTER(i32)]
    L.lgdsp_wfstats_run.argtypes = [vp, C.POINTER(_abi.WfstatsParams), vp, vp, i64, i64, vp, vp]
    L.lgdsp_wfstats_run_device.argtypes = [vp, C.POINTER(_abi.WfstatsParams), vp, vp, i64, i64, vp, vp]
    L.lgdsp_multi_intersect_run.argtypes = [vp, C.POINTER(_abi.MultiIntersectParams), vp, i64, i64, vp, vp]
    L.lgdsp_multi_intersect_run_device.argtypes = [vp, C.POINTER(_abi.MultiIntersectParams), vp, i64, i64, vp, vp]
    L.lgdsp_trap_sweep_run.argtypes = [vp, C.POINTER(_abi.SweepParams), vp, i64, i64, C.POINTER(_abi.TrapVariant), i32, vp]
    L.lgdsp_trap_sweep_run_device.argtypes = [vp, C.POINTER(_abi.SweepParams), vp, i64, i64,
                                              C.POINTER(_abi.TrapVariant), i32, vp]
    L.lgdsp_sweep_run.argtypes = [vp, C.POINTER(_abi.SweepParams), vp, i64, i64, C.POINTER(_abi.SweepVariant), i32, vp, vp]
    L.lgdsp_sweep_run_device.argtypes = [vp, C.POINTER(_abi.SweepParams), vp, i64, i64, C.POINTER(_abi.SweepVariant), i32, vp, vp]
    L.lgdsp_sweep_run_ext.argtypes = [vp, C.POINTER(_abi.SweepParams), vp, i32, vp, i64, i64, C.POINTER(_abi.SweepVariant), i32, vp, vp]
    L.lgdsp_sweep_run_ext_device.argtypes = [vp, C.POINTER(_abi.SweepParams), vp, i32, vp, i64, i64, C.POINTER(_abi.SweepVariant), i32,
                                             vp, vp]
    L.lgdsp_synth_generate_device.argtypes = [vp, C.POINTER(_abi.SynthParams), i64, i64, i64, vp]
    L.lgdsp_synth_generate_host.argtypes = [C.POINTER(_abi.SynthParams), i64, i64, i64, vp]
    _lib = L
    return L


# every symbol include/lgdsp_b200.h declares (tests/test_abi.py checks the library exports them all)
EXPORTED_SYMBOLS = (
    "lgdsp_version", "lgdsp_last_error", "lgdsp_create", "lgdsp_destroy", "lgdsp_launch_count", "lgdsp_synchronize",
    "lgdsp_lsq_fit_matrix", "lgdsp_sg_coeffs", "lgdsp_cusp_coeffs", "lgdsp_zac_coeffs",
    "lgdsp_icpc_run", "lgdsp_icpc_run_device", "lgdsp_icpc_set_params", "lgdsp_icpc_set_path", "lgdsp_icpc_profile_device", "lgdsp_host_alloc", "lgdsp_host_free", "lgdsp_host_register",
    "lgdsp_host_unregister", "lgdsp_icpc_run_ext", "lgdsp_icpc_run_ext_device",
    "lgdsp_codec_max_encoded_bytes", "lgdsp_codec_encode_host", "lgdsp_decode_data", "lgdsp_decode_data_device", "lgdsp_icpc_run_encoded", "lgdsp_icpc_compressed_run_encoded",
    "lgdsp_window_stats_run", "lgdsp_window_stats_run_device", "lgdsp_sipm_run", "lgdsp_sipm_run_device",
    "lgdsp_sipm_list_pointers_device", "lgdsp_sipm_list_gather_device", "lgdsp_thresholdstats", "lgdsp_intersect_maximum", "lgdsp_wfstats_run", "lgdsp_wfstats_run_device", "lgdsp_multi_intersect_run", "lgdsp_multi_intersect_run_device", "lgdsp_icpc_compressed_run", "lgdsp_icpc_compressed_run_device",
    "lgdsp_trap_sweep_run", "lgdsp_trap_sweep_run_device", "lgdsp_sweep_run", "lgdsp_sweep_run_device",
    "lgdsp_sweep_run_ext", "lgdsp_sweep_run_ext_device",
    "lgdsp_synth_generate_device", "lgdsp_synth_generate_host", "lgdsp_last_kernel_ms",
)


class Handle:
    """RAII wrapper of lgdsp_handle: one per (thread, GPU)."""

    def __init__(self, device=0, stream=None):
        self._lib = load_library()
        self._h = C.c_void_p()
        rc = self._lib.lgdsp_create(int(device), C.c_void_p(stream) if stream else None, C.byref(self._h))
        if rc != 0:
            msg = self._lib.lgdsp_last_error(None).decode()
            self._h = None
            raise LgdspError(rc, msg)
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.lgdsp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise LgdspError(rc, self._lib.lgdsp_last_error(self._h).decode())

    @property
    def launch_count(self):
        return int(self._lib.lgdsp_launch_count(self._h))

    def synchronize(self):
        self._check(self._lib.lgdsp_synchronize(self._h))

    def icpc_profile_device(self, d_wf_ptr, n_events, ld, d_out_ptr):
        """device ms of (prefix, extract, CUSP/ZAC select, CUSP/ZAC finish) on one batch run serially"""
        ms = (C.c_double * 4)()
        self._check(self._lib.lgdsp_icpc_profile_device(self._h, C.c_void_p(d_wf_ptr), int(n_events), int(ld), C.c_void_p(d_out_ptr), ms))
        return list(ms)

    def set_icpc_path(self, path, batch=0, streams=0):
        """'split' (default: prefix / extract / CUSP-ZAC kernels coupled through an L2-resident ring) or 'fused' (icpc_kernel)"""
        code = {"fused": 0, "split": 1}[path] if isinstance(path, str) else int(path)
        self._check(self._lib.lgdsp_icpc_set_path(self._h, code, int(batch), int(streams)))

    def last_kernel_ms(self):
        return float(self._lib.lgdsp_last_kernel_ms(self._h))

    # ---- dsp_icpc ----
    def icpc_set_params(self, params):
        self._check(self._lib.lgdsp_icpc_set_params(self._h, C.byref(params)))

    def icpc_run_host(self, params, wf_ptr, n_events, ld, out_ptr):
        self._check(self._lib.lgdsp_icpc_run(self._h, C.byref(params) if params is not None else None,
                                             C.c_void_p(wf_ptr), int(n_events), int(ld), C.c_void_p(out_ptr)))

    def icpc_run_device(self, params, d_wf_ptr, n_events, ld, d_out_ptr):
        self._check(self._lib.lgdsp_icpc_run_device(self._h, C.byref(params) if params is not None else None,
                                                    C.c_void_p(d_wf_ptr), int(n_events), int(ld), C.c_void_p(d_out_ptr)))

    def icpc_run_ext_host(self, params, wf_ptr, sample_bytes, baseline_ptr, n_events, ld, out_ptr):
        """dsp_icpc chain on uint16 / uint32 samples with an optional external per-event baseline (host buffers)"""
        self._check(self._lib.lgdsp_icpc_run_ext(self._h, C.byref(params) if params is not None else None, C.c_void_p(wf_ptr),
                                                 int(sample_bytes), C.c_void_p(baseline_ptr) if baseline_ptr else None,
                                                 int(n_events), int(ld), C.c_void_p(out_ptr)))

    def icpc_run_ext_device(self, params, d_wf_ptr, sample_bytes, d_baseline_ptr, n_events, ld, d_out_ptr):
        self._check(self._lib.lgdsp_icpc_run_ext_device(self._h, C.byref(params) if params is not None else None,
                                                        C.c_void_p(d_wf_ptr), int(sample_bytes),
                                                        C.c_void_p(d_baseline_ptr) if d_baseline_ptr else None,
                                                        int(n_events), int(ld), C.c_void_p(d_out_ptr)))

    # ---- decode_data ----
    def decode_data_host(self, codec, enc_ptr, offsets_ptr, n_events, n_samples, shift, wf_ptr, sample_bytes, ld):
        self._check(self._lib.lgdsp_decode_data(self._h, int(codec), C.c_void_p(enc_ptr), C.c_void_p(offsets_ptr), int(n_events),
                                                int(n_samples), int(shift), C.c_void_p(wf_ptr), int(sample_bytes), int(ld)))

    def decode_data_device(self, codec, d_enc_ptr, d_offsets_ptr, n_events, n_samples, shift, d_wf_ptr, sample_bytes, ld,
                           d_status_ptr=None):
        self._check(self._lib.lgdsp_decode_data_device(self._h, int(codec), C.c_void_p(d_enc_ptr), C.c_void_p(d_offsets_ptr),
                                                       int(n_events), int(n_samples), int(shift), C.c_void_p(d_wf_ptr),
                                                       int(sample_bytes), int(ld),
                                                       C.c_void_p(d_status_ptr) if d_status_ptr else None))

    def icpc_run_encoded_host(self, params, codec, enc_ptr, offsets_ptr, shift, sample_bytes, baseline_ptr, n_events, out_ptr):
        """dsp_icpc on encoded waveforms in host memory (decode_data on the device)"""
        self._check(self._lib.lgdsp_icpc_run_encoded(self._h, C.byref(params) if params is not None else None, int(codec),
                                                     C.c_void_p(enc_ptr), C.c_void_p(offsets_ptr), int(shift), int(sample_bytes),
                                                     C.c_void_p(baseline_ptr) if baseline_ptr else None, int(n_events),
                                                     C.c_void_p(out_ptr)))

    def icpc_compressed_run_encoded_host(self, p_pre, p_wdw, enc_pre, enc_wdw, presum_rate, aux_windows, rows_pre_ptr, rows_wdw_ptr,
                                         stats_ptr):
        """dsp_icpc_compressed on two codec.EncodedWaveforms sets in host memory (decode_data on the device)"""
        import numpy as np
        w = (C.c_int32 * 8)(*[int(v) for ab in aux_windows for v in ab])
        keep = [np.ascontiguousarray(x) for x in (enc_pre.data, enc_pre.offsets, enc_wdw.data, enc_wdw.offsets)]
        self._check(self._lib.lgdsp_icpc_compressed_run_encoded(
            self._h, C.byref(p_pre) if p_pre is not None else None, C.byref(p_wdw) if p_wdw is not None else None,
            int(enc_pre.codec), C.c_void_p(keep[0].ctypes.data), C.c_void_p(keep[1].ctypes.data), int(enc_pre.shift),
            int(enc_pre.sample_bytes), int(enc_wdw.codec), C.c_void_p(keep[2].ctypes.data), C.c_void_p(keep[3].ctypes.data),
            int(enc_wdw.shift), int(enc_wdw.sample_bytes), float(presum_rate), w, len(enc_pre), C.c_void_p(rows_pre_ptr),
            C.c_void_p(rows_wdw_ptr), C.c_void_p(stats_ptr)))

    def window_stats_host(self, wf_ptr, sample_bytes, n_events, n_samples, ld, t_first_ns, dt_ns, shift_ptr, windows, out_ptr):
        """signalstats on `windows` ([(from, until), ...] 0-based inclusive) of every waveform; out double[n][nw][5]"""
        w = (C.c_int32 * (2 * len(windows)))(*[int(v) for ab in windows for v in ab])
        self._check(self._lib.lgdsp_window_stats_run(self._h, C.c_void_p(wf_ptr), int(sample_bytes), int(n_events), int(n_samples),
                                                     int(ld), float(t_first_ns), float(dt_ns),
                                                     C.c_void_p(shift_ptr) if shift_ptr else None, w, len(windows),
                                                     C.c_void_p(out_ptr)))

    def window_stats_device(self, d_wf_ptr, sample_bytes, n_events, n_samples, ld, t_first_ns, dt_ns, d_shift_ptr, windows,
                            d_out_ptr):
        w = (C.c_int32 * (2 * len(windows)))(*[int(v) for ab in windows for v in ab])
        self._check(self._lib.lgdsp_window_stats_run_device(self._h, C.c_void_p(d_wf_ptr), int(sample_bytes), int(n_events),
                                                            int(n_samples), int(ld), float(t_first_ns), float(dt_ns),
                                                            C.c_void_p(d_shift_ptr) if d_shift_ptr else None, w, len(windows),
                                                            C.c_void_p(d_out_ptr)))

    def _compressed(self, fn, p_pre, p_wdw, pre_ptr, pre_bytes, ld_pre, wdw_ptr, wdw_bytes, ld_wdw, presum_rate, aux_windows,
                    n_events, rows_pre_ptr, rows_wdw_ptr, stats_ptr):
        w = (C.c_int32 * 8)(*[int(v) for ab in aux_windows for v in ab])
        self._check(fn(self._h, C.byref(p_pre) if p_pre is not None else None, C.byref(p_wdw) if p_wdw is not None else None,
                       C.c_void_p(pre_ptr), int(pre_bytes), int(ld_pre), C.c_void_p(wdw_ptr), int(wdw_bytes), int(ld_wdw),
                       float(presum_rate), w, int(n_events), C.c_void_p(rows_pre_ptr), C.c_void_p(rows_wdw_ptr),
                       C.c_void_p(stats_ptr)))

    def icpc_compressed_run_host(self, *a):
        """dsp_icpc_compressed on host buffers: see lgdsp_icpc_compressed_run (include/lgdsp_b200.h)"""
        self._compressed(self._lib.lgdsp_icpc_compressed_run, *a)

    def icpc_compressed_run_device(self, *a):
        self._compressed(self._lib.lgdsp_icpc_compressed_run_device, *a)

    # ---- dsp_sipm ----
    def sipm_run_host(self, params, wf_ptr, n_events, ld, rows_ptr, trig_ptr):
        self._check(self._lib.lgdsp_sipm_run(self._h, C.byref(params), C.c_void_p(wf_ptr), int(n_events), int(ld),
                                             C.c_void_p(rows_ptr), C.c_void_p(trig_ptr)))

    def sipm_run_device(self, params, d_wf_ptr, n_events, ld, d_rows_ptr, d_trig_ptr):
        self._check(self._lib.lgdsp_sipm_run_device(self._h, C.byref(params) if params is not None else None,
                                                    C.c_void_p(d_wf_ptr), int(n_events), int(ld), C.c_void_p(d_rows_ptr),
                                                    C.c_void_p(d_trig_ptr)))

    def sipm_list_pointers_device(self, d_rows_ptr, n_events, lst, cap, d_elem_ptr):
        """element pointers of trigger list `lst` (device int64[n_events + 1]); returns the total number of triggers"""
        tot = C.c_int64(0)
        self._check(self._lib.lgdsp_sipm_list_pointers_device(self._h, C.c_void_p(d_rows_ptr), int(n_events), int(lst), int(cap),
                                                              C.c_void_p(d_elem_ptr), C.byref(tot)))
        return tot.value

    def sipm_list_gather_device(self, d_trig_ptr, n_events, lst, cap, d_elem_ptr, d_flat_ptr, flat_stride):
        self._check(self._lib.lgdsp_sipm_list_gather_device(self._h, C.c_void_p(d_trig_ptr), int(n_events), int(lst), int(cap),
                                                            C.c_void_p(d_elem_ptr), C.c_void_p(d_flat_ptr), int(flat_stride)))

    def thresholdstats(self, y, mn, mx, mad):
        import numpy as np
        y = np.ascontiguousarray(y, dtype=np.float64)
        out = C.c_double(0.0)
        self._check(self._lib.lgdsp_thresholdstats(self._h, C.c_void_p(y.ctypes.data), y.size, float(mn), float(mx),
                                                   1 if mad else 0, C.byref(out)))
        return out.value

    def intersect_maximum(self, y, t_first_ns, dt_ns, thr, min_n, max_n, cap):
        import numpy as np
        y = np.ascontiguousarray(y, dtype=np.float64)
        out = [np.zeros(cap) for _ in range(4)]
        n = C.c_int32(0)
        self._check(self._lib.lgdsp_intersect_maximum(self._h, C.c_void_p(y.ctypes.data), y.size, float(t_first_ns), float(dt_ns),
                                                      float(thr), int(min_n), int(max_n), int(cap),
                                                      *[C.c_void_p(o.ctypes.data) for o in out], C.byref(n)))
        m = min(n.value, cap)
        return {"x": out[0][:m], "x_high": out[1][:m], "x_tot": out[2][:m], "max": out[3][:m], "multiplicity": n.value}

    def wfstats_run_host(self, params, wf_ptr, thr_ptr, n_events, ld, rows_ptr, lists_ptr):
        """the per-waveform primitives selected in params.what on host buffers (lgdsp_wfstats_run)"""
        self._check(self._lib.lgdsp_wfstats_run(self._h, C.byref(params), C.c_void_p(wf_ptr), C.c_void_p(thr_ptr) if thr_ptr else None,
                                                int(n_events), int(ld), C.c_void_p(rows_ptr),
                                                C.c_void_p(lists_ptr) if lists_ptr else None))

    def wfstats_run_device(self, params, d_wf_ptr, d_thr_ptr, n_events, ld, d_rows_ptr, d_lists_ptr):
        self._check(self._lib.lgdsp_wfstats_run_device(self._h, C.byref(params), C.c_void_p(d_wf_ptr),
                                                       C.c_void_p(d_thr_ptr) if d_thr_ptr else None, int(n_events), int(ld),
                                                       C.c_void_p(d_rows_ptr), C.c_void_p(d_lists_ptr) if d_lists_ptr else None))

    def multi_intersect_host(self, params, y_ptr, n_events, ld, x_ptr, flags_ptr):
        self._check(self._lib.lgdsp_multi_intersect_run(self._h, C.byref(params), C.c_void_p(y_ptr), int(n_events), int(ld),
                                                        C.c_void_p(x_ptr), C.c_void_p(flags_ptr)))

    def multi_intersect_device(self, params, d_y_ptr, n_events, ld, d_x_ptr, d_flags_ptr):
        self._check(self._lib.lgdsp_multi_intersect_run_device(self._h, C.byref(params), C.c_void_p(d_y_ptr), int(n_events),
                                                               int(ld), C.c_void_p(d_x_ptr), C.c_void_p(d_flags_ptr)))

    # ---- sweeps ----
    def sweep_run_host(self, sparams, wf_ptr, n_events, ld, variants, out_ptr):
        self._check(self._lib.lgdsp_trap_sweep_run(self._h, C.byref(sparams), C.c_void_p(wf_ptr), int(n_events), int(ld),
                                                   variants, len(variants), C.c_void_p(out_ptr)))

    def sweep_run_device(self, sparams, d_wf_ptr, n_events, ld, variants, d_out_ptr):
        self._check(self._lib.lgdsp_trap_sweep_run_device(self._h, C.byref(sparams), C.c_void_p(d_wf_ptr), int(n_events),
                                                          int(ld), variants, len(variants), C.c_void_p(d_out_ptr)))

    def gsweep_run_host(self, sparams, wf_ptr, n_events, ld, variants, out_ptr, aux_ptr=None):
        """general sweep (lgdsp_sweep_run): variants = ctypes array of _abi.SweepVariant"""
        self._check(self._lib.lgdsp_sweep_run(self._h, C.byref(sparams), C.c_void_p(wf_ptr), int(n_events), int(ld),
                                              variants, len(variants), C.c_void_p(out_ptr),
                                              C.c_void_p(aux_ptr) if aux_ptr else None))

    def gsweep_run_device(self, sparams, d_wf_ptr, n_events, ld, variants, d_out_ptr, d_aux_ptr=None):
        self._check(self._lib.lgdsp_sweep_run_device(self._h, C.byref(sparams), C.c_void_p(d_wf_ptr), int(n_events), int(ld),
                                                     variants, len(variants), C.c_void_p(d_out_ptr),
                                                     C.c_void_p(d_aux_ptr) if d_aux_ptr else None))

    def gsweep_run_ext_host(self, sparams, wf_ptr, sample_bytes, baseline_ptr, n_events, ld, variants, out_ptr, aux_ptr=None):
        """general sweep on uint16 / uint32 samples with an optional external per-event baseline (lgdsp_sweep_run_ext)"""
        self._check(self._lib.lgdsp_sweep_run_ext(self._h, C.byref(sparams), C.c_void_p(wf_ptr), int(sample_bytes),
                                                  C.c_void_p(baseline_ptr) if baseline_ptr else None, int(n_events), int(ld),
                                                  variants, len(variants), C.c_void_p(out_ptr),
                                                  C.c_void_p(aux_ptr) if aux_ptr else None))

    def gsweep_run_ext_device(self, sparams, d_wf_ptr, sample_bytes, d_baseline_ptr, n_events, ld, variants, d_out_ptr,
                              d_aux_ptr=None):
        self._check(self._lib.lgdsp_sweep_run_ext_device(self._h, C.byref(sparams), C.c_void_p(d_wf_ptr), int(sample_bytes),
                                                         C.c_void_p(d_baseline_ptr) if d_baseline_ptr else None, int(n_events),
                                                         int(ld), variants, len(variants), C.c_void_p(d_out_ptr),
                                                         C.c_void_p(d_aux_ptr) if d_aux_ptr else None))

    # ---- synthetic input ----
    def synth_device(self, sp, first_event, n_events, ld, d_wf_ptr):
        self._check(self._lib.lgdsp_synth_generate_device(self._h, C.byref(sp), int(first_event), int(n_events), int(ld),
                                                          C.c_void_p(d_wf_ptr)))
