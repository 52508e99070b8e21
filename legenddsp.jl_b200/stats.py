"""LegendDSP's per-waveform primitives as broadcasts over waveform arrays, `f.(wvfs, start, stop)`:
`extremestats` (src/extremestats.jl:14-40), `saturation` (src/saturation.jl:12-65), `tailstats` (src/tailstats.jl:13-72) and
`get_wvf_maximum` (src/interpolation.jl:21-46).

Every function takes `RDWaveforms` (the time axis comes from the waveforms) or a 2-D sample array [n_events, n_samples]
(time axis from `t_first` / `step`) and returns one value per waveform; a 1-D trace gives scalars.  Time windows resolve to
sample indices as the reference does, `round(Int, (t - first(X)) / step(X))` with ties to even, and a window outside the
trace raises AssertionError (the reference's @assert, src/tailstats.jl:23-25).  Times are in ns.  All arithmetic runs in the
CUDA library (lgdsp_wfstats_run, one pass over every waveform); there is no CPU path."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np

from . import _abi
from ._lib import Handle
from .config import Q, ns, _sub_over_step
from .dsp_icpc import RDWaveforms, get_handle

_KIND = {np.dtype(np.uint16): _abi.SAMPLE_U16, np.dtype(np.float32): _abi.SAMPLE_F32, np.dtype(np.float64): _abi.SAMPLE_F64}


def wf_samples(signal) -> Tuple[np.ndarray, int, bool]:
    """(samples[n_events, n_samples], LGDSP_SAMPLE_* kind, input was a single trace).  uint16 / float32 / float64 rows that
    are contiguous go to the library as they are (any row stride); other float types become float32 and other integer
    types uint16 (range-checked), as dsp_sipm's inputs do."""
    a = np.asarray(signal)
    single = a.ndim == 1
    if single:
        a = a.reshape(1, -1)
    if a.ndim != 2:
        raise ValueError("waveform signals must be a 1-D trace or a 2-D array [n_events, n_samples]")
    if a.dtype not in _KIND:
        if np.issubdtype(a.dtype, np.floating):
            a = a.astype(np.float32)
        elif np.issubdtype(a.dtype, np.integer):
            if a.size and (a.min() < 0 or a.max() > 65535):
                raise ValueError("samples outside the UInt16 range")
            a = a.astype(np.uint16)
        else:
            raise TypeError("unsupported sample type %s" % a.dtype)
    isz = a.dtype.itemsize
    if a.shape[1] > 1 and a.strides[1] != isz or a.strides[0] < 0 or a.strides[0] % isz or a.strides[0] // isz < a.shape[1]:
        a = np.ascontiguousarray(a)
    return a, _KIND[a.dtype], single


def _axis(wvfs, t_first: Optional[Q], step: Optional[Q]):
    if isinstance(wvfs, RDWaveforms) or (hasattr(wvfs, "signal") and hasattr(wvfs, "step")):
        return wvfs.signal, getattr(wvfs, "t_first", ns(0.0)), wvfs.step
    return wvfs, (t_first if t_first is not None else ns(0.0)), (step if step is not None else ns(16.0))


def window(start: Optional[Q], stop: Optional[Q], n: int, t_first: Q, step: Q) -> Tuple[int, int]:
    """0-based inclusive sample range of the time window [start, stop] (None: the whole trace)"""
    a = 0 if start is None else _sub_over_step(start, t_first, step)
    b = n - 1 if stop is None else _sub_over_step(stop, t_first, step)
    if not (0 <= a <= b <= n - 1):
        raise AssertionError(f"window {a}:{b} outside the waveform (0:{n - 1})")
    return a, b


def wfstats_params(n: int, kind: int, what: int, t_first: Q, step: Q) -> _abi.WfstatsParams:
    P = _abi.WfstatsParams()
    P.struct_size, P.version = C.sizeof(_abi.WfstatsParams), _abi.LGDSP_PARAMS_VERSION
    P.n_samples, P.sample_kind, P.what = int(n), int(kind), int(what)
    P.t_first_ns, P.dt_ns = t_first.ns(), step.ns()
    P.thr_min, P.thr_max = -np.inf, np.inf
    return P


def wfstats_rows(sig: np.ndarray, P: _abi.WfstatsParams, thresholds=None, *, device: int = 0, handle: Optional[Handle] = None):
    """rows[n_events, WFSTAT_NCOL] (and lists[n_events, 4, max_triggers] when IntersectMaximum is selected) of the samples
    prepared by wf_samples"""
    h = handle or get_handle(device)
    n_ev = sig.shape[0]
    rows = np.zeros((n_ev, _abi.WFSTAT_NCOL))
    im = bool(P.what & _abi.WFSTAT_INTERSECT_MAXIMUM)
    lists = np.zeros((n_ev, 4, P.max_triggers)) if im else None
    thr = np.ascontiguousarray(np.broadcast_to(np.asarray(thresholds, dtype=np.float64), (n_ev,))) if im else None
    h.wfstats_run_host(P, sig.ctypes.data, thr.ctypes.data if im else None, n_ev, sig.strides[0] // sig.dtype.itemsize,
                       rows.ctypes.data, lists.ctypes.data if im else None)
    return (rows, lists) if im else rows


def _run(wvfs, what, start, stop, cols, *, t_first=None, step=None, setup=None, device=0, handle=None):
    sig, t0, dt = _axis(wvfs, t_first, step)
    sig, kind, single = wf_samples(sig)
    P = wfstats_params(sig.shape[1], kind, what, t0, dt)
    frm, until = window(start, stop, sig.shape[1], t0, dt)
    if setup is not None:
        setup(P, frm, until)
    rows = wfstats_rows(sig, P, device=device, handle=handle)
    out = tuple(rows[:, _abi.WFSTAT_COL[c]] for c in cols)
    return tuple(o[0] for o in out) if single else out


def extremestats(wvfs, start: Optional[Q] = None, stop: Optional[Q] = None, *, t_first: Optional[Q] = None,
                 step: Optional[Q] = None, device: int = 0, handle: Optional[Handle] = None):
    """extremestats.(wvfs[, start, stop]) -> (min, max, tmin, tmax): extrema and the times [ns] of their FIRST occurrence"""
    def setup(P, a, b):
        P.ext_from, P.ext_until = a, b
    return _run(wvfs, _abi.WFSTAT_EXTREMESTATS, start, stop, ("min", "max", "tmin", "tmax"), t_first=t_first, step=step,
                setup=setup, device=device, handle=handle)


def saturation(wvfs, low: int, high: int, start: Optional[Q] = None, stop: Optional[Q] = None, *, t_first: Optional[Q] = None,
               step: Optional[Q] = None, device: int = 0, handle: Optional[Handle] = None):
    """saturation.(wvfs, low, high[, start, stop]) -> (low, high, max_cons_low, max_cons_high) as int64: the number of raw
    UInt16 samples equal to `low` / `high` and the longest runs of them"""
    def setup(P, a, b):
        P.sat_from, P.sat_until, P.sat_low, P.sat_high = a, b, int(low), int(high)
    r = _run(wvfs, _abi.WFSTAT_SATURATION, start, stop, ("sat_low", "sat_high", "sat_max_cons_low", "sat_max_cons_high"),
             t_first=t_first, step=step, setup=setup, device=device, handle=handle)
    return tuple(np.int64(v) if np.ndim(v) == 0 else v.astype(np.int64) for v in r)


def tailstats(wvfs, start: Q, stop: Q, *, t_first: Optional[Q] = None, step: Optional[Q] = None, device: int = 0,
              handle: Optional[Handle] = None):
    """tailstats.(wvfs, start, stop) -> (mean, sigma, τ [ns]) of log(y) over the window; (0, 0, 0) where a sample is <= 0"""
    def setup(P, a, b):
        P.tail_from, P.tail_until = a, b
    return _run(wvfs, _abi.WFSTAT_TAILSTATS, start, stop, ("tail_mean", "tail_sigma", "tail_tau"), t_first=t_first, step=step,
                setup=setup, device=device, handle=handle)


def get_wvf_maximum(wvfs, start: Q, stop: Q, *, t_first: Optional[Q] = None, step: Optional[Q] = None, device: int = 0,
                    handle: Optional[Handle] = None):
    """get_wvf_maximum.(wvfs, start, stop): the maximum inside the window, refined by a parabola through its neighbours when
    it lies strictly inside the window"""
    def setup(P, a, b):
        P.max_from, P.max_until = a, b
    return _run(wvfs, _abi.WFSTAT_WVF_MAXIMUM, start, stop, ("wvf_max",), t_first=t_first, step=step, setup=setup, device=device,
                handle=handle)[0]
