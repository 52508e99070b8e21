"""The shortcuts of the two fastest bench workloads against the CPU oracle, under random configurations with a non-zero time
of the first sample:

A  the lean PZ-trapezoid group (LGDSP_GROUP_PZTRAP_LEAN, icpc_prefix_kernel + icpc_extract_kernel): e_10410 is a coarse-to-fine
   maximum pruned by a Lipschitz bound, the prefix kernel forms only the t50 mask, t0 runs without t0_inv; traces whose
   (10 us, 4 us) trapezoid peaks between the coarse points (every 33rd output) would lose their maximum to a bound that is
   too tight.  Lean == fused kernel bit for bit, == O.pz_trap, independent of the sub-batching, 32-bit == 16-bit samples.
B  fixed pick-off trapezoid sweeps (dsp_trap_rt_optimization): without aux outputs the warp kernel skips max(y), the threshold
   mask and the crossing and streams only the samples [0, stream_n) that the host derives from dni_window's arithmetic
   (t_first, clamping at both trace ends, the baseline window).  Every path, output type and entry point gives the same
   numbers, and they are the oracle's.
C  the full dsp_icpc chain with t_first != 0 (every interpolated time, bloffset, the window arithmetic).
D  the tail log-regression of the split prefix kernel: four accuracy classes per warp (degree-5 / degree-9 series, log1p
   series, full log with re-referencing) chosen by an integer pre-pass; tails that put the largest |u| of the runs just below
   and above each class boundary, the non-positive-sample sentinel, against an independent float64 reference.

LGDSP_FUZZ_SEEDS_LEAN / _RT / _TFIRST widen parts A / B / C."""
import copy
import math
import os

import numpy as np
import pytest

from parity import TOL, compare_rows
from test_gpu_fuzz import _draw
from test_gpu_icpc import assert_parity_with_ties
from test_gpu_split import _identical, _rows
from test_gpu_sweep_warp import _pathological, sweep_path

pytestmark = pytest.mark.gpu

CH = 33   # coarse grid of the pruned trapezoid maxima: outputs 33*k (one per thread of the extract kernel)
LEAN_COLUMNS = ("blmean", "t0", "t50", "e_trap", "e_10410", "e_max", "e_min", "n_sat_high")   # include/lgdsp_b200.h:105-107
PZ_TRAP_COLUMNS = ("blmean", "t0", "t50", "e_trap", "e_10410")                               # O.pz_trap's five


def _t_first(L, rng, cfg):
    """a non-zero time of the first sample, up to +-20 us and up to 0.4 of the baseline window's end (the in-trace pile-up
    window starts at leftendpoint(bl_window) + first(time), src/dsp_routines.jl:75: it has to stay on the trace), on a multiple
    of 1/2 ns: a pick-off half a sample after a sample time then stays an exact binary fraction through (pick - t_first)/dt"""
    lim = min(20000.0, 0.4 * cfg.bl_window[1].ns())
    v = 0.0
    while abs(v) < 100.0:
        v = round(rng.uniform(-lim, lim) * 2.0) / 2.0
    return L.ns(v)


def _shifted(cfg, t_first):
    """the config with its baseline / tail / current windows moved by t_first (the same samples on the shifted time axis);
    before a negative t_first the baseline window keeps its start at 0, which then lies -t_first into the trace"""
    c = copy.copy(cfg)
    for name in ("bl_window", "tail_window", "current_window"):
        a, b = getattr(c, name)
        setattr(c, name, (a if (name == "bl_window" and t_first.ns() < 0) else a + t_first, b + t_first))
    return c


# ---------------------------------------------------------------------------------------------------------------------
# A. lean PZ-trapezoid group
# ---------------------------------------------------------------------------------------------------------------------
def _from_pz(y, km1, base):
    """uint16 trace whose pole-zero corrected form (y_i = w_i + km1 * sum_{j<=i} w_j, w = x - base) is y, up to the rounding of
    each sample (fed back, so that it does not accumulate)"""
    x = np.empty(len(y), dtype=np.int64)
    S = 0.0
    for i, yi in enumerate(y):
        w = (yi - km1 * S) / (1.0 + km1)
        x[i] = int(round(base + w))
        S += float(x[i] - base)
    assert x.min() >= 0 and x.max() <= 65535
    return x.astype(np.uint16)


def _offgrid_rows(P, n, first_sample):
    """Traces whose (10 us, 4 us) trapezoid T peaks between two coarse points.

    Returns (rows, checked): `checked` are the rows built so that the interval holding the peak has both end points below the
    largest coarse value elsewhere -- a bound that ignored the slope between the coarse points would skip that interval.
    T(j) = mean(y[j+a+g .. j+L-1]) - mean(y[j .. j+a-1]).  A step of height A at sample p gives T a rise of slope A/b ending
    at j = p-a-g and a flat top (value A) over j = p-a-g .. p-a; a negative spike -h at sample s adds +h/a to T over
    j = s-a+1 .. s.  With s = 33k + 16 on the rise, D outputs before the top, and A*D < h*b/a < A*(D + 16), the peak T(s)
    lies 8 A/b above the top while the coarse points s-16 and s+17 lie below it."""
    tr = P.trap_10410
    a, g, b = tr.navg, tr.ngap, tr.navg2
    Lt = a + g + b
    km1 = P.pz_km1
    base = 30000.0
    rows, checked = [], []
    s = (n - Lt - 60 - g - 24) // CH * CH + 16
    if s - a + 1 > 0 and s > first_sample:
        for A, D in ((400.0, 40), (300.0, 60)):
            p = s + D + a + g
            y = np.zeros(n)
            y[p:] = A
            y[s] -= A * (D + 8) * a / b
            checked.append(len(rows))
            rows.append(_from_pz(y, km1, base))
    # a short rectangular pulse and a single-sample spike at 33k + 16
    for width, height in ((5, 2000.0), (1, 9000.0)):
        q = max(first_sample + 1, (n // 2) // CH * CH + 16)
        y = np.zeros(n)
        y[q:q + width] = height
        rows.append(_from_pz(y, km1, base))
    # steps whose trapezoid peaks in the first and in the last 33 outputs
    for p in (a + g + 16, n - 20):
        if first_sample < p < n:
            y = np.zeros(n)
            y[p:] = 3000.0
            rows.append(_from_pz(y, km1, base))
    # a ripple with a period near 66 samples on a flat top
    p = max(first_sample + 1, n // 3)
    y = np.zeros(n)
    k = np.arange(n - p)
    y[p:] = 5000.0 + 400.0 * np.sin(2.0 * np.pi * k / 65.7) + 0.05 * k
    rows.append(_from_pz(y, km1, base))
    return np.stack(rows), checked


def _assert_offgrid(O, P, wf, checked):
    """the constructed traces do what they are for (oracle arithmetic): peak off the coarse grid, its interval's end points
    below the largest coarse value"""
    tr = P.trap_10410
    for r in checked:
        m = O.signalstats(wf[r].astype(np.float64), P.t_first_ns, P.dt_ns, P.bl_from, P.bl_until)["mean"]
        T = O.trap(O.invcr(wf[r].astype(np.float64) - m, P.pz_km1), tr.navg, tr.ngap, tr.navg2)
        j = int(np.argmax(T))
        coarse = T[::CH].max()
        k = j // CH
        assert j % CH != 0 and T[j] > coarse + 1.0, (r, j, T[j], coarse)
        assert T[k * CH] < coarse - 1.0 and (k + 1) * CH < len(T) and T[(k + 1) * CH] < coarse - 1.0, (r, j)


@pytest.mark.parametrize("seed", list(range(int(os.environ.get("LGDSP_FUZZ_SEEDS_LEAN", "4")))))
def test_lean_pz_trap_randomised(L, O, handle, seed):
    cfg, tau, pars_filter, n, step = _draw(L, 500 + seed)
    rng = np.random.default_rng(21000 + seed)
    t_first = _t_first(L, rng, cfg)
    cfg = _shifted(cfg, t_first)
    B = O.OracleBuilders()
    kw = dict(n_samples=n, t_first=t_first, step=step, builders=B)
    P_lean = L.resolve_icpc_params(cfg, tau, pars_filter, groups=L._abi.GROUP_PZTRAP_LEAN, **kw)
    P_full = L.resolve_icpc_params(cfg, tau, pars_filter, groups=L._abi.GROUP_PZTRAP, **kw)
    gen = L.synth.generate_host(160, first_event=13000 * (seed + 1))[:, :n]
    clean = L.synth.generate_host(4, mode=1)[:, :n]
    patho = _pathological(8192)[:, :n]
    off, checked = _offgrid_rows(P_lean, n, P_lean.bl_until)
    wf = np.ascontiguousarray(np.concatenate([gen, clean, patho, off]))
    n_gen, n_off0 = len(gen) + len(clean), len(gen) + len(clean) + len(patho)
    assert len(checked) > 0, "no off-grid trace fits this draw"
    _assert_offgrid(O, P_lean, wf, [n_off0 + r for r in checked])
    c = L.COL

    # 1. lean (split) == fused kernel with the same groups and no lean bit, on every promised column
    fused = _rows(L, handle, wf, P_full, "fused")
    lean = _rows(L, handle, wf, P_lean, "split")
    for name in LEAN_COLUMNS:
        x, y = lean[:, c[name]], fused[:, c[name]]
        bad = np.nonzero(~((x == y) | (np.isnan(x) & np.isnan(y))))[0]
        assert bad.size == 0, (name, bad[:8], x[bad[:8]], y[bad[:8]])

    # 2. lean == O.pz_trap (the pathological traces: flat / periodic ones cross their thresholds anywhere -- only the
    #    well-defined columns)
    ref = O.pz_trap(P_lean, wf)
    for i, name in enumerate(PZ_TRAP_COLUMNS):
        rows = slice(None) if name in ("blmean", "t50", "e_10410") else np.r_[0:n_gen, n_off0:len(wf)]
        res = compare_rows(lean[rows][:, [c[name]]], ref[rows][:, [i]], [name])
        assert res[name][1] == 0, (name, res[name])
    assert (ref[:n_gen, 1] > 0).sum() > 4 and np.isfinite(ref[:n_gen, 3]).all()

    # 3. sub-batches and streams: ring slots are reused across sub-batches, the rows must not change
    for batch, streams in ((257, 3), (64, 1), (17, 2)):
        again = _rows(L, handle, wf, P_lean, "split", batch, streams)
        for name in LEAN_COLUMNS:
            assert np.array_equal(again[:, c[name]], lean[:, c[name]], equal_nan=True), (batch, streams, name)

    # 4. 32-bit samples (the generic prefix-kernel instantiation, n <= LGDSP_MAX_SAMPLES / 2) == 16-bit samples
    n4 = 4096
    dt = step.ns()
    cfg4 = copy.copy(cfg)
    cfg4.current_window = (t_first + L.ns(2700 * dt), t_first + L.ns(3500 * dt))
    cfg4.tail_window = (t_first + L.ns(3600 * dt), t_first + L.ns(4000 * dt))
    P4 = L.resolve_icpc_params(cfg4, tau, pars_filter, groups=L._abi.GROUP_PZTRAP_LEAN, n_samples=n4, t_first=t_first,
                               step=step, builders=B)
    w16 = np.ascontiguousarray(wf[:n_off0, :n4])
    w32 = w16.astype(np.uint32)
    r16 = L.dsp_icpc_rows(w16, P4, handle=handle)
    r32 = np.zeros_like(r16)
    handle.icpc_run_ext_host(P4, w32.ctypes.data, 4, None, len(w32), n4, r32.ctypes.data)
    for name in LEAN_COLUMNS:
        assert np.array_equal(r32[:, c[name]], r16[:, c[name]], equal_nan=True), name


# ---------------------------------------------------------------------------------------------------------------------
# B. fixed pick-off trapezoid sweeps
# ---------------------------------------------------------------------------------------------------------------------
def _last_lookup(pick_ns, Lv, n, n_w, t0, dt):
    """one past the last sample a fixed pick-off reads: dni_window on the trapezoid output (clamped at both ends)"""
    nout = n - Lv + 1
    pc = (pick_ns - (t0 + (Lv - 1) * dt)) / dt
    pc = min(max(pc, 0.0), nout - 1.0)
    f = min(max(int(np.rint(pc)) - n_w // 2, 0), nout - n_w)
    return f + Lv + n_w


def _pickoff_sets(L, S, rts, fts, step, t_first, n, rng):
    """(name, pick-off, rise times) of one seed: one set per pick-off group"""
    dt, t0, n_w = step.ns(), t_first.ns(), S.sig_dni.n_w
    lens = lambda rs: [t.trap.navg + t.trap.ngap + t.trap.navg2
                       for t in L.trap_variants(rs, fts, step, mode="rt", pickoff=L.ns(0.0))]
    Lmax = max(lens(rts))
    lo, hi = Lmax + n_w, n - n_w
    s_in = int(rng.integers(lo, hi)) if hi > lo else (lo + hi) // 2
    s_half = int(rng.integers(lo, hi)) if hi > lo else (lo + hi) // 2
    sets = [("inside", L.ns(t0 + (s_in + float(rng.uniform(0.0, 1.0))) * dt), rts),
            ("beyond the end", L.ns(t0 + (n + float(rng.uniform(1.0, 300.0))) * dt), rts),
            ("before the start", L.ns(t0 - float(rng.uniform(0.0, 60.0)) * dt), rts),
            ("half sample", L.ns(t0 + (s_half + 0.5) * dt), rts)]
    # before bl_until: every look-up ends early enough that the integer pass must run on to the baseline window's end; the
    # look-ups stay below the 512-sample step that holds bl_until + 1 (the pass keeps its prefix sums per such step)
    limit = (S.bl_until + 1) // 512 * 512 - 48
    short = [r for r in rts if max(lens([r])) + n_w <= limit]
    if short:
        s_b = max(0, min(limit - n_w // 2 - 2, int(rng.integers(0, max(1, limit - n_w // 2 - 1)))))
        pick = L.ns(t0 + s_b * dt)
        assert max(_last_lookup(pick.ns(), Lv, n, n_w, t0, dt) for Lv in lens(short)) <= limit
        sets.append(("before bl_until", pick, short))
    else:   # (short traces: no trapezoid ends before the baseline window does)
        sets.append(("before bl_until", L.ns(t0 + S.bl_until * dt * 0.5), rts))
    return sets


def _warp_runs(L, handle, S64, S32, wf, W, cfg, tau, var, tvar):
    """every way of running one fixed pick-off set: returns (f64 result, aux of the warp path, aux of the CTA path) after
    checking that all runs agree bit for bit"""
    from legenddsp.jl_b200.dsp_filter_optimization import _run_general
    ne, n = wf.shape
    with sweep_path("warp"):
        base = _run_general(W, cfg, tau, var, f64=True, handle=handle)                 # truncated stream (no aux)
        a_w, aux_w = _run_general(W, cfg, tau, var, f64=True, want_aux=True, handle=handle)
        f32 = _run_general(W, cfg, tau, var, f64=False, handle=handle)
        t32 = np.zeros((ne, len(tvar)), dtype=np.float32)                             # lgdsp_trap_sweep_run
        handle.sweep_run_host(S32, wf.ctypes.data, ne, n, tvar, t32.ctypes.data)
        wide = np.zeros((ne, n + 24), dtype=np.uint16)                                # ld > n
        wide[:, :n] = wf
        strided = np.zeros((ne, len(var)))
        handle.gsweep_run_host(S64, wide.ctypes.data, ne, n + 24, var.array, strided.ctypes.data)
    with sweep_path("cta"):
        a_c, aux_c = _run_general(W, cfg, tau, var, f64=True, want_aux=True, handle=handle)
        c32 = _run_general(W, cfg, tau, var, f64=False, handle=handle)
    default = _run_general(W, cfg, tau, var, f64=True, handle=handle)
    for name, v in (("warp + aux", a_w), ("strided", strided), ("cta", a_c), ("default dispatch", default)):
        assert np.array_equal(v, base, equal_nan=True), (name, np.nanmax(np.abs(v - base)))
    b32 = base.astype(np.float32)
    for name, v in (("f32", f32), ("lgdsp_trap_sweep_run", t32), ("cta f32", c32)):
        assert np.array_equal(v, b32, equal_nan=True), name
    return base, aux_w, aux_c


@pytest.mark.parametrize("seed", list(range(int(os.environ.get("LGDSP_FUZZ_SEEDS_RT", "6")))))
def test_fixed_pickoff_sweeps_randomised(L, O, handle, seed):
    cfg, tau, _, n0, step = _draw(L, 700 + seed)
    rng = np.random.default_rng(31000 + seed)
    t_first = _t_first(L, rng, cfg)
    n = int(rng.choice([8192, 7000, 6144, 4104, 1024, 264]))
    dt = step.ns()
    full = np.concatenate([L.synth.generate_host(150, first_event=17000 * (seed + 1)), L.synth.generate_host(6, mode=1)])
    n_gen = len(full)
    if n >= 6144:
        cfg = _shifted(cfg, t_first)
        wf = np.ascontiguousarray(np.concatenate([full, _pathological(8192)])[:, :n])
        sc = dt / 16.0
        rts = np.sort(np.r_[rng.uniform(0.3, 2.0), rng.uniform(0.3, 10.0, int(rng.integers(2, 31)))]) * sc
        fts = np.sort(rng.uniform(0.1, 3.0, int(rng.integers(1, 4)))) * sc
    else:
        # short traces (windowed waveforms): the baseline window and the filters scale with the trace, the pulse is in it
        span = n * dt / 1000.0
        cfg = copy.copy(cfg)
        cfg.bl_window = (t_first, t_first + L.us(span * 0.2))
        a0 = max(0, 3400 - n // 2) // 8 * 8
        wf = np.ascontiguousarray(np.concatenate([full[:, a0:a0 + n], _pathological(n)]))
        rts = np.sort(np.r_[rng.uniform(0.005, 0.02), rng.uniform(0.02, 0.17, int(rng.integers(2, 31)))]) * span
        fts = np.sort(rng.uniform(0.01, 0.05, int(rng.integers(1, 4)))) * span
    rts = [L.ns(float(v) * 1000.0) for v in rts]
    fts = [L.ns(float(v) * 1000.0) for v in fts]
    W = L.RDWaveforms(wf, t_first, step)
    # (the direct calls use the library's fit matrices as _run_general does: bit-identical runs; the oracle gets its own)
    S64 = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True)
    S32 = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step)
    So = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, builders=O.OracleBuilders(), out_f64=True)
    gen = slice(0, n_gen)
    for name, pick, rs in _pickoff_sets(L, S64, rts, fts, step, t_first, n, rng):
        var = L.trap_sweep_variants(rs, fts, step, mode="rt", pickoff=pick)
        tvar = L.trap_variants(rs, fts, step, mode="rt", pickoff=pick)
        base, aux_w, aux_c = _warp_runs(L, handle, S64, S32, wf, W, cfg, tau, var, tvar)
        ref, raux = O.sweep(So, wf, var.array, want_aux=True)
        assert np.allclose(base, ref, rtol=1e-8, atol=1e-6, equal_nan=True), (name, np.nanmax(np.abs(base - ref)))
        # t50 of the aux outputs: the warp path's own crossing equals the CTA path's; the oracle's on the generator events
        # (the flat and periodic pathological traces cross half their maximum anywhere)
        assert np.array_equal(aux_w, aux_c, equal_nan=True), (name, np.nanmax(np.abs(aux_w - aux_c)))
        assert np.allclose(aux_w[gen], raux[gen], rtol=1e-9, atol=1e-9, equal_nan=True), name
        assert np.isfinite(base[gen]).mean() > 0.9, name
    # a set with both pick-off modes: the default dispatch runs it on the CTA path (the warp path refuses it)
    mixed = L.trap_sweep_variants(rts[:3], fts, step, mode="rt", pickoff=L.ns(t_first.ns() + 0.5 * n * dt))
    ft = L.trap_sweep_variants(rts[:3], fts, step, mode="ft")
    from legenddsp.jl_b200.config import SweepVariants
    from legenddsp.jl_b200.dsp_filter_optimization import _run_general
    var = SweepVariants(len(mixed) + len(ft))
    for i in range(len(mixed)):
        var.array[i] = mixed.array[i]
    for i in range(len(ft)):
        var.array[len(mixed) + i] = ft.array[i]
    with sweep_path("warp"):
        with pytest.raises(Exception, match="LGDSP_SWEEP_PATH=warp"):
            _run_general(W, cfg, tau, var, f64=True, handle=handle)
    with sweep_path("cta"):
        b = _run_general(W, cfg, tau, var, f64=True, handle=handle)
    a = _run_general(W, cfg, tau, var, f64=True, handle=handle)
    assert np.array_equal(a, b, equal_nan=True)
    ref = O.sweep(So, wf, var.array)
    assert np.allclose(a[gen], ref[gen], rtol=1e-8, atol=1e-6, equal_nan=True), np.nanmax(np.abs(a[gen] - ref[gen]))


# ---------------------------------------------------------------------------------------------------------------------
# C. the full chain with a non-zero t_first
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", list(range(int(os.environ.get("LGDSP_FUZZ_SEEDS_TFIRST", "4")))))
def test_random_configurations_with_t_first(L, O, handle, seed):
    cfg, tau, pars_filter, n, step = _draw(L, 900 + seed)
    t_first = _t_first(L, np.random.default_rng(41000 + seed), cfg)
    cfg = _shifted(cfg, t_first)
    P = L.resolve_icpc_params(cfg, tau, pars_filter, n_samples=n, t_first=t_first, step=step, builders=O.OracleBuilders())
    assert P.t_first_ns == t_first.ns() != 0.0
    wf = np.ascontiguousarray(L.synth.generate_host(160, first_event=23000 * (seed + 1))[:, :n])
    got = L.dsp_icpc_rows(wf, P, handle=handle)
    ref, _ = O.dsp_icpc(P, wf)
    assert_parity_with_ties(L, O, P, wf, got, ref, max_ties=8)
    c = L.COL
    assert np.isfinite(ref[:, c["e_trap"]]).sum() > 100 and (ref[:, c["t0"]] > 0).sum() > 4


# ---------------------------------------------------------------------------------------------------------------------
# D. tail log-regression classes
# ---------------------------------------------------------------------------------------------------------------------
NT = 256   # threads of the split prefix kernel: thread t takes the run of q consecutive tail samples from tail_from + t*q


def _tail_population(P, n):
    """(name, trace, sentinel) rows.  Constant integer baseline B (m == B exactly), a pulse of
    amplitude c from sample 3000 on; inside the tail window every thread's run starts at B + c (x_ref) and holds one sample
    B + c +- d, so the largest |u| = |x - x_ref| / (x_ref - m) of every run is d / c."""
    cnt = P.bl_until - P.bl_from + 1
    Bl = next(v for v in range(8000, 8100) if float(v * cnt) * (1.0 / cnt) == v)   # m = sum * (1/count) == Bl exactly
    a, b = P.tail_from, P.tail_until
    q = (b - a + 1 + NT - 1) // NT
    runs = [(a + t * q, min(a + t * q + q - 1, b)) for t in range(NT) if a + t * q <= b]

    def pulse(c):
        x = np.full(n, Bl, dtype=np.int64)
        x[3000:] = Bl + c
        return x

    def one_per_run(c, d, only=None):
        x = pulse(c)
        for r, (i0, i1) in enumerate(runs):
            if i1 > i0 and (only is None or r == only):
                x[i0 + 1 + r % (i1 - i0)] = Bl + c + (d if r % 2 == 0 else -d)
        return x

    c = 40960
    out = []
    # just below / above 2^-10, 2^-6, 2^-3 (classes 0 | 1 | 2 | 3)
    for d, what in ((39, "|u| < 2^-10"), (41, "|u| > 2^-10"), (639, "|u| < 2^-6"), (641, "|u| > 2^-6"), (5119, "|u| < 2^-3"),
                    (5121, "|u| > 2^-3")):
        out.append((what, one_per_run(c, d), False))
    out.append(("one run |u| < 2^-3, the others 0", one_per_run(c, 5119, only=77), False))
    out.append(("one run |u| > 2^-3, the others 0", one_per_run(c, 5121, only=140), False))
    x = one_per_run(c, 639)
    i0, i1 = runs[130]
    x[(i0 + i1) // 2] = Bl
    out.append(("a sample equal to m", x, True))
    x = one_per_run(c, 39)
    i0, i1 = runs[200]
    x[i0 + 3] = Bl - 5
    out.append(("a negative sample inside one run", x, True))
    x = one_per_run(c, 39)
    i0, _ = runs[40]
    x[i0] = Bl
    out.append(("a run that starts at m and recovers", x, True))
    x = one_per_run(c, 39)
    i0, _ = runs[41]
    x[i0] = Bl + 1
    x[i0 + 1] = Bl + 2
    out.append(("a run that starts one count above m and recovers", x, False))
    # m not an integer: alternating baseline; floor(m) is non-positive, floor(m) + 1 is not
    for off, sentinel in ((0, True), (1, False)):
        x = one_per_run(c, 39)
        x[P.bl_from:P.bl_until + 1:2] = Bl + 1
        i0, i1 = runs[90]
        x[(i0 + i1) // 2] = Bl + off
        out.append((f"m not an integer, a sample at floor(m) + {off}", x, sentinel))
    # small amplitude: every run beyond 1/8, the full logarithm everywhere
    rng = np.random.default_rng(5)
    x = pulse(7)
    x[a:b + 1] += rng.integers(-2, 3, b - a + 1)
    out.append(("amplitude 7 +- 2", x, False))
    # a decaying tail with noise (the classes mixed as in real events)
    k = np.arange(n)
    x = pulse(0)
    x[3000:] = Bl + np.rint(20000.0 * np.exp(-(k[3000:] - 3000) / 31250.0) + rng.normal(0.0, 3.0, n - 3000)).astype(np.int64)
    out.append(("decaying tail", x, False))
    return out


def _tail_reference(x, m, t_first, dt, a, b):
    """tail_mean / tail_sigma / -1/tail_tau of src/tailstats.jl from the exact float64 values x - m: np.log (< 1 ulp),
    correctly rounded sums (math.fsum) and the least-squares line in closed form about the mean time"""
    w = x[a:b + 1].astype(np.float64) - m
    lg = np.log(w)
    N = len(lg)
    mean = math.fsum(lg) / N
    dl = lg - mean
    X = t_first + np.arange(a, b + 1, dtype=np.float64) * dt
    Xc = X - math.fsum(X) / N
    slope = math.fsum(Xc * dl) / math.fsum(Xc * Xc)
    sigma = math.sqrt(math.fsum(dl * dl) / N)
    return mean, sigma, slope


def test_tail_log_regression_classes(L, O, handle):
    t_first = L.ns(-4000.0)
    cfg = _shifted(L.example_config(), t_first)
    P = L.resolve_icpc_params(cfg, L.us(500.0), n_samples=8192, t_first=t_first, builders=O.OracleBuilders())
    pop = _tail_population(P, 8192)
    wf = np.stack([x for _, x, _ in pop]).astype(np.uint16)
    split = _rows(L, handle, wf, P, "split")
    fused = _rows(L, handle, wf, P, "fused")
    ref, _ = O.dsp_icpc(P, wf)
    c = L.COL
    cols = ("blmean", "tail_mean", "tail_sigma", "tail_tau")
    idx = [c[k] for k in cols]
    bad = _identical(split[:, idx], fused[:, idx], cols)
    assert not bad, bad
    for got in (split, fused):
        res = compare_rows(got[:, idx], ref[:, idx], cols)
        assert all(v[1] == 0 for v in res.values()), res
    for e, (what, x, sentinel) in enumerate(pop):
        if sentinel:
            for got in (split, fused, ref):
                assert (got[e, idx[1:]] == 0.0).all(), (what, got[e, idx[1:]])
            continue
        mean, sigma, slope = _tail_reference(x, ref[e, c["blmean"]], P.t_first_ns, P.dt_ns, P.tail_from, P.tail_until)
        for got in (split, fused):
            # Each logarithm of the kernels is within a few ulp (the series of every class reach 1e-16 inside their range),
            # and their sums of <= 2 501 same-signed terms of similar size go through runs of <= 10 and binary trees: a few
            # dozen roundings of 1.1e-16 relative.  1e-14 relative holds that with room; a series used outside its class
            # range is off by its first dropped term (u^6/6 = 6e-7 at |u| = 1/8 for the degree-5 series) in every run.
            # (The oracle's bound, 1e-12, is set by its serial sum over the whole window.)
            assert abs(got[e, c["tail_mean"]] - mean) <= 1e-14 * abs(mean) + 1e-15, (what, got[e, c["tail_mean"]] - mean)
            rtol, atol = TOL["tail_sigma"]
            assert abs(got[e, c["tail_sigma"]] - sigma) <= atol + rtol * sigma, (what, got[e, c["tail_sigma"]], sigma)
            s = -1.0 / got[e, c["tail_tau"]]
            rtol, atol = TOL["tail_tau"]
            assert abs(s - slope) <= atol + rtol * abs(slope), (what, s, slope)
