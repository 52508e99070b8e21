"""`dsp_sipm(data, config, pars_optimization)` -- host-side mirror of the reference's SiPM trigger chain
(/root/reference/src/dsp_sipm.jl:47-158) on top of the C ABI (`lgdsp_sipm_run`), plus the in-tree primitives it is built
from: `IntersectMaximum` (src/intersect_maximum.jl:24-119), `thresholdstats` / `thresholdstats_mad`
(src/thresholdstats.jl:19-41, 61-71).  All arithmetic runs in the CUDA library; there is no CPU path."""
from __future__ import annotations

import ctypes as C
import math
from collections import OrderedDict
from typing import Any, Dict, Mapping, Optional

import numpy as np

from . import _abi
from ._lib import Handle
from .config import (Q, RddspPolicy, DEFAULT_POLICY, LibBuilders, ns, us, julia_round, _ratio, _fill_sg, _trap, _min_n)
from .dsp_icpc import RDWaveforms, _as_waveforms, get_handle
from .stats import wf_samples, wfstats_params, wfstats_rows


def example_sipm_config() -> Dict[str, Any]:
    """make_sipm_config()  /root/reference/test/test_dsp_sipm.jl:40-68, as data"""
    return {
        "t0_hpge_window": (us(47.0), us(53.0)),
        "sg_flt_degree": 3,
        "filters": {
            "sg": {"n_σ_threshold": 3.0, "min_threshold": -1.0, "max_threshold": 1.0,
                   "n_σ_dc_threshold": 5.0, "min_dc_threshold": -4.0, "max_dc_threshold": 4.0,
                   "min_tot_intersect": ns(70.0), "max_tot_intersect": ns(150.0)},
            "trap": {"rt": ns(100.0), "ft": ns(50.0), "pz_tau": us(3.0),
                     "n_σ_threshold": 3.5, "min_threshold": -1.5, "max_threshold": 1.5,
                     "n_σ_dc_threshold": 5.0, "min_dc_threshold": -3.0, "max_dc_threshold": 3.0,
                     "min_tot_intersect": ns(48.0), "max_tot_intersect": ns(250.0)},
        },
    }


def resolve_sipm_params(config: Mapping[str, Any], pars_optimization: Mapping[str, Any], *, n_samples: int,
                        t_first: Q = ns(0.0), step: Q = ns(16.0), sample_kind: str = "u16", max_triggers: int = 64,
                        policy: RddspPolicy = DEFAULT_POLICY, builders=None) -> _abi.SipmParams:
    """what dsp_sipm (src/dsp_sipm.jl:47-139) derives from (config, pars_optimization) and the time axis, in samples"""
    if builders is None:
        builders = LibBuilders()
    sgc, trc = config["filters"]["sg"], config["filters"]["trap"]
    P = _abi.SipmParams()
    P.struct_size = C.sizeof(_abi.SipmParams)
    P.version = _abi.LGDSP_PARAMS_VERSION
    n = int(n_samples)
    P.n_samples = n
    P.sample_kind = {"u16": _abi.SAMPLE_U16, "f32": _abi.SAMPLE_F32}[sample_kind]
    P.t_first_ns, P.dt_ns = t_first.ns(), step.ns()
    # TruncateFilter(first(t0_hpge_window)..last(t0_hpge_window)) [RDDSP]: the samples whose time lies in the closed interval
    lo, hi = config["t0_hpge_window"]
    a = max(0, math.ceil(_ratio(lo - t_first, step) - 1e-9))
    b = min(n - 1, math.floor(_ratio(hi - t_first, step) + 1e-9))
    if a > b:
        raise AssertionError("t0_hpge_window selects no sample of the waveform")
    P.trunc_from, P.trunc_until = a, b
    _fill_sg(P.sg, pars_optimization["sg"]["wl"], int(config["sg_flt_degree"]), step, policy, builders)       # :99
    if P.sg.n_taps > n:
        raise ValueError("Savitzky-Golay window longer than the waveform")
    # IntersectMaximum: max(1, round(Int, tot / step))  src/intersect_maximum.jl:21-22
    P.sg_min_n, P.sg_max_n = _min_n(sgc["min_tot_intersect"], step), _min_n(sgc["max_tot_intersect"], step)
    P.sg_min_thr, P.sg_max_thr, P.sg_nsigma = float(sgc["min_threshold"]), float(sgc["max_threshold"]), float(sgc["n_σ_threshold"])
    P.sg_min_dc, P.sg_max_dc, P.sg_nsigma_dc = (float(sgc["min_dc_threshold"]), float(sgc["max_dc_threshold"]),
                                                 float(sgc["n_σ_dc_threshold"]))
    P.trap = _trap(trc["rt"], trc["ft"], step)                                                               # :129
    if P.trap.navg < 1 or P.trap.ngap < 0 or P.trap.length > n - P.sg.n_taps + 1:
        raise ValueError(f"trapezoidal filter {P.trap.as_tuple()} does not fit the Savitzky-Golay trace")
    RC = _ratio(trc["pz_tau"], step)                                                                         # :125
    P.pz_km1 = 1.0 / (RC / (RC + 1.0)) - 1.0
    P.trap_min_n, P.trap_max_n = _min_n(trc["min_tot_intersect"], step), _min_n(trc["max_tot_intersect"], step)
    P.trap_min_thr, P.trap_max_thr, P.trap_nsigma = (float(trc["min_threshold"]), float(trc["max_threshold"]),
                                                      float(trc["n_σ_threshold"]))
    P.trap_min_dc, P.trap_max_dc, P.trap_nsigma_dc = (float(trc["min_dc_threshold"]), float(trc["max_dc_threshold"]),
                                                       float(trc["n_σ_dc_threshold"]))
    if not (1 <= int(max_triggers) <= _abi.SIPM_MAX_TRIGGERS):
        raise ValueError("max_triggers outside 1..%d" % _abi.SIPM_MAX_TRIGGERS)
    P.max_triggers = int(max_triggers)
    return P


# reference column order, src/dsp_sipm.jl:141-157: (name, source) with source = pass-through input column, scalar row
# column, or (list, field) of the trigger lists
SIPM_TABLE = OrderedDict(
    [("blfc", "baseline"), ("timestamp", "timestamp"), ("eventID_fadc", "eventnumber"), ("e_fc", "daqenergy")]
    + [(c, c) for c in ("t_max", "t_min", "t_max_lar", "t_min_lar", "e_max", "e_min", "e_max_lar", "e_min_lar",
                        "blmean", "blsigma", "blslope", "bloffset", "wfmean", "wfsigma", "wfslope", "wfoffset",
                        "threshold", "threshold_DC")]
    + [("trig_pos", (0, 0)), ("trig_max", (0, 3)), ("trig_pos_DC", (1, 0)), ("trig_max_DC", (1, 3)),
       ("threshold_trap", "threshold_trap"), ("threshold_DC_trap", "threshold_DC_trap"),
       ("trig_pos_trap", (2, 0)), ("trig_pos_high_trap", (2, 1)), ("trig_pos_tot_trap", (2, 2)), ("trig_max_trap", (2, 3)),
       ("trig_pos_DC_trap", (3, 0)), ("trig_pos_high_DC_trap", (3, 1)), ("trig_pos_tot_DC_trap", (3, 2)),
       ("trig_max_DC_trap", (3, 3))])
_PASS = ("blfc", "timestamp", "eventID_fadc", "e_fc")
_COUNT = ("n_trig", "n_trig_DC", "n_trig_trap", "n_trig_DC_trap")


class VectorOfVectors:
    """flat data + element pointers (ArraysOfArrays.VectorOfVectors, the reference's type for trigger lists)"""

    def __init__(self, data: np.ndarray, elem_ptr: np.ndarray):
        self.data, self.elem_ptr = data, elem_ptr

    def __len__(self):
        return len(self.elem_ptr) - 1

    def __getitem__(self, i):
        return self.data[self.elem_ptr[i]:self.elem_ptr[i + 1]]


def _sipm_signal(sig):
    a = np.asarray(sig)
    if a.ndim != 2:
        raise ValueError("waveform signals must be a 2-D array [n_events, n_samples]")
    if np.issubdtype(a.dtype, np.floating):
        a, kind = a.astype(np.float32, copy=False), "f32"
    elif np.issubdtype(a.dtype, np.integer):
        if a.dtype != np.uint16:
            if a.size and (a.min() < 0 or a.max() > 65535):
                raise ValueError("samples outside the UInt16 range")
            a = a.astype(np.uint16)
        kind = "u16"
    else:
        raise TypeError("unsupported sample type %s" % a.dtype)
    if a.strides[1] != a.dtype.itemsize:
        a = np.ascontiguousarray(a)
    return a, kind


def sipm_rows(signal, params: _abi.SipmParams, *, device: int = 0, handle: Optional[Handle] = None):
    """resolved params in, (rows[n_events, SIPM_NCOL], trig[n_events, 4, 4, max_triggers]) out; the call is repeated with
    a larger capacity when a trigger list did not fit"""
    sig, _ = _sipm_signal(signal)
    h = handle or get_handle(device)
    n_events = sig.shape[0]
    while True:
        cap = params.max_triggers
        rows = np.zeros((n_events, _abi.SIPM_NCOL))
        trig = np.zeros((n_events, _abi.SIPM_NLIST, _abi.SIPM_NFIELD, cap))
        h.sipm_run_host(params, sig.ctypes.data, n_events, sig.strides[0] // sig.dtype.itemsize, rows.ctypes.data, trig.ctypes.data)
        most = int(rows[:, [_abi.SIPM_COL[c] for c in _COUNT]].max()) if n_events else 0
        if most <= cap:
            return rows, trig
        if cap >= _abi.SIPM_MAX_TRIGGERS:
            raise RuntimeError(f"an event has {most} triggers, more than LGDSP_SIPM_MAX_TRIGGERS")
        params.max_triggers = min(_abi.SIPM_MAX_TRIGGERS, max(2 * cap, most))


def sipm_to_table(rows, trig, data: Optional[Mapping[str, Any]] = None) -> "OrderedDict[str, Any]":
    out: "OrderedDict[str, Any]" = OrderedDict()
    for name, src in SIPM_TABLE.items():
        if name in _PASS:
            if data is not None and src in data:
                out[name] = np.asarray(data[src])
        elif isinstance(src, tuple):
            lst, field = src
            cnt = rows[:, _abi.SIPM_COL[_COUNT[lst]]].astype(np.int64)
            ptr = np.concatenate(([0], np.cumsum(cnt)))
            mask = np.arange(trig.shape[3])[None, :] < cnt[:, None]
            out[name] = VectorOfVectors(trig[:, lst, field, :][mask], ptr)
        else:
            out[name] = np.ascontiguousarray(rows[:, _abi.SIPM_COL[src]])
    return out


def dsp_sipm(data: Mapping[str, Any], config: Mapping[str, Any], pars_optimization: Mapping[str, Any], *, device: int = 0,
             handle: Optional[Handle] = None, policy: RddspPolicy = DEFAULT_POLICY, builders=None, max_triggers: int = 64):
    """DSP routine for SiPM data: the reference's `dsp_sipm(data, config, pars_optimization)` (src/dsp_sipm.jl:47-158).
    `data["waveform"]`: RDWaveforms (raw UInt16 ADC samples, or floats -> processed as Float32)."""
    w = _as_waveforms(data["waveform"])
    sig, kind = _sipm_signal(w.signal)
    P = resolve_sipm_params(config, pars_optimization, n_samples=sig.shape[1], t_first=w.t_first, step=w.step,
                            sample_kind=kind, max_triggers=max_triggers, policy=policy, builders=builders)
    rows, trig = sipm_rows(sig, P, device=device, handle=handle)
    return sipm_to_table(rows, trig, data)


def dsp_sipm_compressed(data: Mapping[str, Any], config: Mapping[str, Any], pars_optimization: Mapping[str, Any], **kw):
    """`dsp_sipm_compressed(data, config, pars_optimization)` (src/dsp_sipm.jl:207-318): `dsp_sipm` on
    `decode_data(data.waveform_bit_drop)` -- the two functions differ in that line only.  The codec is outside the
    reference tree: `data["waveform_bit_drop"]` holds the DECODED samples."""
    d = dict(data)
    d["waveform"] = d["waveform_bit_drop"]
    return dsp_sipm(d, config, pars_optimization, **kw)


# ---- the in-tree primitives on single traces or, for a 2-D signal [n_events, n_samples], on every row (GPU, through the C ABI) ----
def _thresholdstats_rows(signal, mn, mx, what, col, device, handle):
    sig, kind, _ = wf_samples(signal)
    P = wfstats_params(sig.shape[1], kind, what, ns(0.0), ns(1.0))
    P.thr_min, P.thr_max = float(mn), float(mx)
    return wfstats_rows(sig, P, device=device, handle=handle)[:, _abi.WFSTAT_COL[col]]


def thresholdstats(signal, min: float = -np.inf, max: float = np.inf, *, device: int = 0, handle: Optional[Handle] = None):
    """standard deviation of the samples inside [min, max]  (src/thresholdstats.jl:19-41); one value per row of a 2-D signal"""
    if np.ndim(signal) == 2:
        return _thresholdstats_rows(signal, min, max, _abi.WFSTAT_THRESHOLDSTATS, "thr_sigma", device, handle)
    return (handle or get_handle(device)).thresholdstats(np.ascontiguousarray(signal, dtype=np.float64), min, max, mad=False)


def thresholdstats_mad(signal, min: float = -np.inf, max: float = np.inf, *, device: int = 0, handle: Optional[Handle] = None):
    """1.4826 * MAD of the samples inside [min, max]  (src/thresholdstats.jl:61-71); one value per row of a 2-D signal"""
    if np.ndim(signal) == 2:
        return _thresholdstats_rows(signal, min, max, _abi.WFSTAT_THRESHOLDSTATS_MAD, "thr_mad", device, handle)
    return (handle or get_handle(device)).thresholdstats(np.ascontiguousarray(signal, dtype=np.float64), min, max, mad=True)


class IntersectMaximum:
    """IntersectMaximum(mintot, maxtot)(waveform, threshold)  (src/intersect_maximum.jl:12-23): result dict with
    x, x_high, x_tot, max (arrays, times in ns) and multiplicity.  A 2-D signal [n_events, n_samples] takes a scalar or a
    per-row threshold and gives x, x_high, x_tot, max as VectorOfVectors and multiplicity as int64[n_events]."""

    def __init__(self, mintot: Q, maxtot: Q):
        self.mintot, self.maxtot = mintot, maxtot

    def __call__(self, signal, threshold: float, *, t_first: Q = ns(0.0), step: Q = ns(16.0), device: int = 0,
                 handle: Optional[Handle] = None, max_triggers: int = 256):
        min_n, max_n = _min_n(self.mintot, step), _min_n(self.maxtot, step)
        if np.ndim(signal) == 2:
            return self._rows(signal, threshold, t_first, step, min_n, max_n, device, handle, max_triggers)
        y = np.ascontiguousarray(signal, dtype=np.float64)
        h = handle or get_handle(device)
        while True:
            r = h.intersect_maximum(y, t_first.ns(), step.ns(), float(threshold), min_n, max_n, max_triggers)
            if r["multiplicity"] <= max_triggers:
                return r
            max_triggers = r["multiplicity"]

    @staticmethod
    def _rows(signal, threshold, t_first, step, min_n, max_n, device, handle, cap):
        sig, kind, _ = wf_samples(signal)
        thr = np.asarray(threshold, dtype=np.float64)
        if thr.ndim not in (0, 1) or (thr.ndim == 1 and len(thr) != sig.shape[0]):
            raise ValueError("threshold: a scalar or one value per waveform")
        P = wfstats_params(sig.shape[1], kind, _abi.WFSTAT_INTERSECT_MAXIMUM, t_first, step)
        P.im_min_n, P.im_max_n = min_n, max_n
        while True:
            P.max_triggers = min(int(cap), _abi.WFSTAT_MAX_TRIGGERS)
            rows, lists = wfstats_rows(sig, P, thr, device=device, handle=handle)
            cnt = rows[:, _abi.WFSTAT_COL["multiplicity"]].astype(np.int64)
            most = int(cnt.max()) if len(cnt) else 0
            if most <= P.max_triggers:
                break
            if P.max_triggers >= _abi.WFSTAT_MAX_TRIGGERS:
                raise RuntimeError(f"a waveform has {most} triggers, more than {_abi.WFSTAT_MAX_TRIGGERS}")
            cap = max(2 * P.max_triggers, most)
        ptr = np.concatenate(([0], np.cumsum(cnt)))
        keep = np.arange(lists.shape[2])[None, :] < cnt[:, None]
        out = {k: VectorOfVectors(lists[:, f, :][keep], ptr) for f, k in enumerate(("x", "x_high", "x_tot", "max"))}
        out["multiplicity"] = cnt
        return out


class MultiIntersect:
    """MultiIntersect(threshold_ratios, mintot, n, d, sampling_rate)(waveforms)  (src/multi_intersect.jl:10-34): the
    times [ns] at which every waveform first exceeds ratio * maximum, x[n_events, n_ratios] (a single trace gives x[n_ratios])"""

    def __init__(self, threshold_ratios=None, mintot: Q = ns(64.0), n: int = 1, d: int = 1, sampling_rate: int = 1):
        self.threshold_ratios = (np.arange(1, 91) * 0.01 if threshold_ratios is None      # collect(0.01:0.01:0.9)
                                 else np.asarray(threshold_ratios, dtype=np.float64))
        self.mintot, self.n, self.d, self.sampling_rate = mintot, int(n), int(d), int(sampling_rate)

    def params(self, n_samples: int, t_first: Q, step: Q, builders=None) -> _abi.MultiIntersectParams:
        if builders is None:
            builders = LibBuilders()
        r = self.threshold_ratios
        if not (1 <= len(r) <= _abi.MI_MAX_THR):
            raise ValueError("number of threshold ratios outside 1..%d" % _abi.MI_MAX_THR)
        if not (1 <= self.n <= _abi.MI_MAX_HALF) or not (0 <= self.d <= _abi.LGDSP_MAX_DNI_DEG) or self.d >= 2 * self.n \
                or self.sampling_rate < 1 or 2 * self.n * self.sampling_rate > 256:
            raise ValueError("polynomial window / degree / sampling rate outside the supported range")
        P = _abi.MultiIntersectParams()
        P.struct_size, P.version = C.sizeof(_abi.MultiIntersectParams), _abi.LGDSP_PARAMS_VERSION
        P.n_samples, P.n_thresholds = int(n_samples), len(r)
        P.t_first_ns, P.dt_ns = t_first.ns(), step.ns()
        P.min_n = _min_n(self.mintot, step)                       # max(1, round(Int, mintot / step))  :29-30
        P.half_window, P.degree, P.rate = self.n, self.d, self.sampling_rate
        for j, v in enumerate(r):
            P.ratios[j] = float(v)
        A = builders.lsq_fit_matrix(2 * self.n, self.d)           # _lsq_fit_matrix(0:2n-1, degree)  :80
        for i, v in enumerate(np.asarray(A).reshape(-1)):
            P.A[i] = float(v)
        return P

    def __call__(self, signal, *, t_first: Q = ns(0.0), step: Q = ns(16.0), device: int = 0, handle: Optional[Handle] = None,
                 builders=None):
        y = np.asarray(signal, dtype=np.float64)
        single = y.ndim == 1
        y = np.ascontiguousarray(y.reshape(1, -1) if single else y)
        if y.shape[1] == 0:                                       # isempty(Y) && return intersect_x  :50
            x = np.zeros((y.shape[0], len(self.threshold_ratios)))
            return x[0] if single else x
        P = self.params(y.shape[1], t_first, step, builders)
        x = np.zeros((y.shape[0], P.n_thresholds))
        flags = np.zeros(y.shape[0], dtype=np.int32)
        (handle or get_handle(device)).multi_intersect_host(P, y.ctypes.data, y.shape[0], y.shape[1], x.ctypes.data, flags.ctypes.data)
        if flags.any():
            raise AssertionError("cannot interpolate intersect on left boundary")       # :85-88
        return x[0] if single else x
