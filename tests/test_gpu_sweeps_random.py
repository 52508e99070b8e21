"""The general sweep kernel's FIR (CUSP / ZAC, kind 1) and Savitzky-Golay (kind 2) variants against the CPU oracle under random
configurations (src/dsp_filter_optimization.jl:145-231, 286-375, 393-441):

1  CUSP / ZAC rt and ft sweeps through the public wrappers on `_draw` configs with a non-zero t_first, a random RddspPolicy
   and random grids and pick-offs; one hand-built set per trace length / PolynomialDNI that puts pick-offs before the trace,
   beyond it and on half samples, the longest FIR (LGDSP_MAX_FIR taps) and FIRs that leave exactly n_w outputs.
2  Savitzky-Golay sweeps with 1..33 taps (underdetermined fits included), windows at both ends of the SG trace, one- and
   two-sample windows and a window that ends on the rising edge of the current pulse (maximum on its last sample, no
   parabola); every mismatch must be an argmax tie.  The sweep's SG variant equals the chain's a_sg.
3  mixed trapezoid / FIR / SG sets of 1 .. 1024 variants (the trapezoid loop strides by the block size, the FIR / SG loop by
   the warp count, both write the same output buffer).
4  uint32 samples above 65535 with an external baseline, float32 output, the NaN rows of 32-bit waveforms whose sum leaves
   32 bits.
5  the accept / reject boundaries of the host validation of kinds 1 and 2.

The oracle side (configurations, variant tables, oracle outputs, tolerances) runs without a GPU: test_oracle_side_of_the_sweeps
checks that each tolerance is small enough that one dropped tap or a pick-off moved by one sample would fail.
LGDSP_FUZZ_SEEDS_GSWEEP widens parts 1 and 2."""
import copy
import os

import numpy as np
import pytest

from test_gpu_fastpaths import _shifted, _t_first
from test_gpu_fuzz import _draw
from test_gpu_sweep_warp import sweep_path

gpu = pytest.mark.gpu
SEEDS = list(range(int(os.environ.get("LGDSP_FUZZ_SEEDS_GSWEEP", "3"))))
U = 2.0 ** -53            # float64 unit roundoff


# ---------------------------------------------------------------------------------------------------------------------
# error bounds
# ---------------------------------------------------------------------------------------------------------------------
# The kernel forms a FIR output as sum_{k=0}^{L} g[k] TT[j+L-k] (g = first difference of the taps, TT = prefix sums of the
# pole-zero corrected waveform) and an SG trace value as sum_{k=0}^{T} gg[k] TT[j+k].  Each TT entry is one fma of exact
# integer prefix sums and the baseline mean (rounding <= u |TT|, u |Sd|, u km1 |SS| with Sd = cumsum(x - m), SS = cumsum(Sd)),
# and an fma chain of L+1 terms adds at most (L+1) u sum|g| max|TT|.  The oracle filters the IIR output y directly
# (L u sum|c| max|y|) after a recursion whose error grows by u (|y| + 2|x - m|) per sample.  Both sides take their taps and
# fit matrices from different builders (the product's and the oracle's own): sum|c_lib - c_orc| max|y| and the same for the
# PolynomialDNI matrix.  The fit evaluates sum_j u'^j sum_i A[i, j] val_i at u' = pc - from in [0, n_w]: errors of the window
# values pass through the linear map val -> result, at most amp = max_u' sum_i |sum_j A[i, j] u'^j| times the largest, and its
# own roundings (n_w per coefficient, one per Horner step) are at most (n_w + 4) u amp_abs max|val| with
# amp_abs = max_u' sum_j (sum_i |A[i, j]|) u'^j, |val| <= sum|c| max|y|.  Each bound is first order and summed term by term,
# not scaled by a safety factor.
def _dni_matrix(S):
    nw, m = S.sig_dni.n_w, S.sig_dni.degree + 1
    return np.array(S.sig_dni.A[:nw * m]).reshape(nw, m)


def _amp(A):
    """(amp, amp_abs) of the fit matrix A over u' in [0, n_w]"""
    nw, m = A.shape
    up = np.linspace(0.0, float(nw), 8 * nw + 1)[:, None] ** np.arange(m)
    return float(np.abs(up @ A.T).sum(axis=1).max()), float((up * np.abs(A).sum(axis=0)).sum(axis=1).max())


def _coeffs(v):
    return np.ctypeslib.as_array(v.coeffs, (v.n_taps,)).copy()


def event_scales(O, S, wf, baseline=None):
    """per event of wf: (m, y, T = max(|TT|, |Sd|, km1 |SS|), max|y|, n (max|y| + 2 max|x - m|)) in the oracle's arithmetic"""
    n, km1 = S.n_samples, S.pz_km1
    out = []
    for e, row in enumerate(wf):
        x = row[:n].astype(np.float64)
        m = float(baseline[e]) if baseline is not None else O.signalstats(x, S.t_first_ns, S.dt_ns, S.bl_from, S.bl_until)["mean"]
        w = x - m
        y = O.invcr(w, km1)
        Sd = np.cumsum(w)
        T = max(np.abs(np.cumsum(y)).max(), np.abs(Sd).max(), km1 * np.abs(np.cumsum(Sd)).max())
        ym = np.abs(y).max()
        out.append((m, y, T, ym, n * (ym + 2.0 * np.abs(w).max())))
    return out


def fir_tolerance(scales, S_lib, S_orc, v_lib, v_orc):
    """[n_events] bound on |kernel - oracle| of one FIR variant (v_lib: the product's taps, v_orc: the oracle's)"""
    c, cl = _coeffs(v_orc), _coeffs(v_lib)
    Lf = len(c)
    sg = np.abs(np.r_[cl[0], np.diff(cl), -cl[-1]]).sum()
    sc, dc = np.abs(c).sum(), np.abs(cl - c).sum()
    A, Al = _dni_matrix(S_orc), _dni_matrix(S_lib)
    (amp, amp_abs), damp, nw = _amp(A), _amp(Al - A)[0], A.shape[0]
    T = np.array([s[2] for s in scales])
    ym = np.array([s[3] for s in scales])
    drift = np.array([s[4] for s in scales])
    return (amp * ((Lf + 5) * U * sg * T + sc * ((Lf + 1) * U * ym + U * drift) + dc * ym)
            + ((nw + 4) * U * amp_abs + damp) * sc * ym)


def sg_tolerance(scale, v_lib, v_orc):
    """bound on |kernel - oracle| of one SG trace value of one event"""
    h, hl = _coeffs(v_orc), _coeffs(v_lib)
    nt = len(h)
    sgg = np.abs(np.r_[-hl[0], hl[:-1] - hl[1:], hl[-1]]).sum()
    _, _, T, ym, drift = scale
    return (nt + 5) * U * sgg * T + np.abs(h).sum() * ((nt + 1) * U * ym + U * drift) + np.abs(hl - h).sum() * ym


def _peak(win, j, d):
    """get_wvf_maximum's value if its argmax were j (window values win), and its bound when every window value is off by
    <= d: the parabola y1 - a^2 / D (a = y3 - 4 y2 + 3 y1, D = 8 (y3 - 2 y2 + y1)) moves by <= |grad| d plus its roundings"""
    if not 0 < j < len(win) - 1:
        return win[j], d
    y1, y2, y3 = win[j - 1], win[j], win[j + 1]
    a, D = y3 - 4.0 * y2 + 3.0 * y1, 8.0 * (y3 - 2.0 * y2 + y1)
    if D == 0.0:
        return np.nan, np.inf
    q = a * a / D
    g1 = 1.0 - (6.0 * a * D - 8.0 * a * a) / (D * D)
    g2 = -(-8.0 * a * D + 16.0 * a * a) / (D * D)
    g3 = -(2.0 * a * D - 8.0 * a * a) / (D * D)
    return y1 - q, (abs(g1) + abs(g2) + abs(g3)) * d + 8.0 * U * (abs(y1) + abs(q))


def sg_explained(win, got, d):
    """error / bound (<= 1 when explained) of a kernel SG value `got` on the oracle's SG trace values `win` of the window: each
    is within d of the kernel's, so the kernel's first argmax can be any sample within 2 d of the maximum -- an argmax tie --
    and the value must be get_wvf_maximum's at one of them"""
    best = np.inf
    for j in np.nonzero(win >= win.max() - 2.0 * d)[0]:
        v, t = _peak(win, j, d)
        if np.isfinite(v):
            best = min(best, _ratio(abs(got - v), t))
    return best


def _ratio(err, bound):
    return 0.0 if err == 0.0 else err / bound


def check_fir(got, ref, tol, what):
    """returns the largest error / tolerance ratio"""
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(got), nan), (what, np.nonzero(np.isnan(got) != nan))
    r = np.abs(got[~nan] - ref[~nan]) / tol[~nan]
    assert r.size == 0 or r.max() <= 1.0, (what, int(np.argmax(r)), float(r.max()), got[~nan][np.argmax(r)], ref[~nan][np.argmax(r)])
    return float(r.max()) if r.size else 0.0


def sg_window_trace(O, scale, v_orc):
    h = _coeffs(v_orc)
    return O.corr_valid(scale[1][v_orc.win_from:v_orc.win_until + len(h)], h)


def check_sg(O, scales, got, ref, v_lib, v_orc, what):
    """every row equals the oracle within its bound, or is explained sample by sample as an argmax tie; returns (largest
    error / bound of the rows that are not ties, number of ties)"""
    worst, ties = 0.0, 0
    for e in range(len(got)):
        d = sg_tolerance(scales[e], v_lib, v_orc)
        win = sg_window_trace(O, scales[e], v_orc)
        v, t = _peak(win, int(np.argmax(win)), d)          # the oracle's own answer (first argmax) and its bound
        assert abs(v - ref[e]) <= t, (what, e, v, ref[e])
        if abs(got[e] - v) <= t:
            worst = max(worst, _ratio(abs(got[e] - v), t))
            continue
        r = sg_explained(win, got[e], d)
        assert r <= 1.0, (what, e, got[e], ref[e], r)
        ties += 1
    return worst, ties


# ---------------------------------------------------------------------------------------------------------------------
# variant tables
# ---------------------------------------------------------------------------------------------------------------------
def concat_variants(L, parts):
    """one SweepVariants from (SweepVariants, index) pairs (the coefficient arrays stay alive in the result)"""
    out = L.SweepVariants(len(parts))
    for i, (v, k) in enumerate(parts):
        out.array[i] = v.array[k]
        out._keep += v._keep
    return out


def _policy(L, rng):
    return L.RddspPolicy(sg_even_length=str(rng.choice(["up", "down"])), sg_time_axis=str(rng.choice(["center", "trailing"])),
                         cuspzac_norm=str(rng.choice(["beta_over_len", "beta"])))


def _fir(L, B, cfg, kind, taps, rt, ft, step, pol, pick_ns, mode):
    """one CUSP / ZAC variant with `taps` taps for the product (builders None) or the oracle (builders B)"""
    c = copy.copy(cfg)
    length = L.ns(taps * step.ns())
    ft = L.ns(min(ft.ns(), 0.25 * taps * step.ns()))          # (the flat top must stay inside the filter)
    if kind == "cusp":
        c.flt_length_cusp = length
    else:
        c.flt_length_zac = length
    v = L.cuspzac_sweep_variants(c, kind, [rt], [ft], step, mode="rt", policy=pol, builders=B)
    assert v.array[0].n_taps == taps
    v.array[0].pickoff_ns, v.array[0].pickoff_mode = pick_ns, mode
    return v


def _short_traces(L, full, n, cfg, t_first):
    """n-sample windows of the generator's 8 192-sample events around the pulse (windowed waveforms); the baseline window
    scales with the trace"""
    a0 = max(0, 3400 - n // 2) // 8 * 8
    wf = np.ascontiguousarray(full[:, a0:a0 + n])
    c = copy.copy(cfg)
    span = n * 16.0 / 1000.0
    c.bl_window = (t_first, t_first + L.us(span * 0.2))
    return wf, c


def _with_dni(cfg, degree, n_w, step):
    c = copy.copy(cfg)
    c.kwargs_pars = dict(cfg.kwargs_pars)
    c.kwargs_pars["sig_interpolation_order"] = degree
    c.kwargs_pars["sig_interpolation_length"] = type(step)(n_w * step.val, step.unit)
    return c


# ---------------------------------------------------------------------------------------------------------------------
# 1. CUSP / ZAC
# ---------------------------------------------------------------------------------------------------------------------
def cuspzac_case(L, O, seed):
    """a draw, its grids / pick-off / policy, the product's and the oracle's variant tables, the oracle's outputs and bounds"""
    cfg, tau, _, n, step = _draw(L, 1200 + seed)
    rng = np.random.default_rng(61000 + seed)
    t_first = _t_first(L, rng, cfg)
    cfg = _shifted(cfg, t_first)
    pol = _policy(L, rng)
    kind = str(rng.choice(["cusp", "zac"]))
    dt, sc = step.ns(), step.ns() / 16.0
    n_rt, n_ft = int(rng.integers(2, 12)), int(rng.integers(1, 8))
    r0, rs = rng.uniform(0.5, 3.0) * sc, rng.uniform(0.2, 1.5) * sc
    f0, fs = rng.uniform(0.3, 2.0) * sc, rng.uniform(0.1, 0.5) * sc
    grid_rt = (L.us(r0), L.us(rs), L.us(r0 + (n_rt - 1) * rs))
    grid_ft = (L.us(f0), L.us(fs), L.us(f0 + (n_ft - 1) * fs))
    where = str(rng.choice(["inside", "inside", "before the start", "beyond the end", "half sample"]))
    t0 = t_first.ns()
    pick = {"inside": t0 + rng.uniform(0.3, 0.9) * n * dt, "before the start": t0 - rng.uniform(0.0, 60.0) * dt,
            "beyond the end": t0 + (n + rng.uniform(1.0, 300.0)) * dt,
            "half sample": t0 + (int(rng.integers(n // 3, n - n // 4)) + 0.5) * dt}[where]
    if kind == "cusp":
        cfg.e_grid_rt_cusp, cfg.e_grid_ft_cusp, cfg.enc_pickoff_cusp = grid_rt, grid_ft, L.ns(pick)
    else:
        cfg.e_grid_rt_zac, cfg.e_grid_ft_zac, cfg.enc_pickoff_zac = grid_rt, grid_ft, L.ns(pick)
    ft_fixed, rt_fixed = L.us(rng.uniform(0.5, 3.0) * sc), L.us(rng.uniform(1.0, 10.0) * sc)
    rts, fts = L.grid_values(grid_rt), L.grid_values(grid_ft)
    B = O.OracleBuilders()
    S_lib = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True)
    S_orc = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True, builders=B)
    wf = np.ascontiguousarray(np.concatenate([L.synth.generate_host(60, first_event=19000 * (seed + 1)),
                                              L.synth.generate_host(4, mode=1)])[:, :n])
    scales = event_scales(O, S_orc, wf)
    sets = {}
    for mode, rs_, fs_ in (("rt", rts, [ft_fixed]), ("ft", [rt_fixed], fts)):
        vl = L.cuspzac_sweep_variants(cfg, kind, rs_, fs_, step, mode=mode, policy=pol)
        vo = L.cuspzac_sweep_variants(cfg, kind, rs_, fs_, step, mode=mode, policy=pol, builders=B)
        ref = O.sweep(S_orc, wf, vo.array)
        tol = np.stack([fir_tolerance(scales, S_lib, S_orc, vl.array[i], vo.array[i]) for i in range(len(vo))], axis=1)
        sets[mode] = (vl, vo, ref, tol)
    return dict(cfg=cfg, tau=tau, n=n, step=step, t_first=t_first, pol=pol, kind=kind, where=where, ft_fixed=ft_fixed,
                rt_fixed=rt_fixed, wf=wf, S_lib=S_lib, S_orc=S_orc, scales=scales, sets=sets)


@gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_cuspzac_sweeps_randomised(L, O, handle, seed):
    k = cuspzac_case(L, O, seed)
    W = L.RDWaveforms(k["wf"], k["t_first"], k["step"])
    ne = len(k["wf"])
    f_rt = L.dsp_cusp_rt_optimization if k["kind"] == "cusp" else L.dsp_zac_rt_optimization
    f_ft = L.dsp_cusp_ft_optimization if k["kind"] == "cusp" else L.dsp_zac_ft_optimization
    got = f_rt(W, k["cfg"], k["tau"], ft=k["ft_fixed"], policy=k["pol"], handle=handle)
    vl, vo, ref, tol = k["sets"]["rt"]
    assert got.shape == (len(vo), ne) and got.dtype == np.float64
    r_rt = check_fir(got.T, ref, tol, ("rt", k["kind"], k["where"]))
    got = f_ft(W, k["cfg"], k["tau"], k["rt_fixed"], policy=k["pol"], handle=handle)
    vl, vo, ref, tol = k["sets"]["ft"]
    assert got.shape == (len(vo), ne) and got.dtype == np.float32
    # float32 output: the kernel's float64 value rounded once, i.e. within half a float32 spacing of it
    r_ft = check_fir(got.T.astype(np.float64), ref, tol + np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64),
                     ("ft", k["kind"]))
    print(f"seed {seed} {k['kind']} {k['where']}: largest error / bound rt {r_rt:.3g}, ft {r_ft:.3g}")


# (n, PolynomialDNI degree, n_w): n_w <= 32 runs the lane loop once; 4 104 = 4 096 + 9 - 1 holds the longest FIR with exactly
# n_w outputs
EDGE_CASES = [(1024, 0, 7), (2048, 3, 44), (4104, 3, 9), (8192, 1, 32), (8192, 2, 33), (8192, 3, 64)]


def cuspzac_edge_case(L, O, n, degree, n_w):
    cfg, tau, _, _, step = _draw(L, 1400 + n + 10 * n_w + degree)
    step = L.ns(16.0)
    rng = np.random.default_rng(n * 100 + n_w * 10 + degree)
    t_first = L.ns(float(rng.choice([-3000.0, 0.0, 2500.5])))
    full = np.concatenate([L.synth.generate_host(40, first_event=5000 + n), L.synth.generate_host(2, mode=1)])
    if n == 8192:
        wf, cfg = np.ascontiguousarray(full), _shifted(cfg, t_first)
    else:
        wf, cfg = _short_traces(L, full, n, cfg, t_first)
    cfg = _with_dni(cfg, degree, n_w, step)
    pol = _policy(L, rng)
    B = O.OracleBuilders()
    dt, t0 = step.ns(), t_first.ns()
    longest = n - n_w + 1
    taps = sorted({min(longest, L._abi.LGDSP_MAX_FIR), int(rng.integers(8, min(longest, 3000))), int(rng.integers(8, 200))})
    if longest <= L._abi.LGDSP_MAX_FIR:
        assert longest in taps                               # an FIR that leaves exactly n_w outputs
    picks = [(t0 - rng.uniform(0.0, 60.0) * dt, 0), (t0 + (n + rng.uniform(1.0, 300.0)) * dt, 0),
             (t0 + (int(rng.integers(0, n)) + 0.5) * dt, 0), (t0 + rng.uniform(0.0, n) * dt, 0),
             (t0 + float(rng.integers(0, n)) * dt, 0), (rng.uniform(0.0, 0.5) * n * dt, 1), (1.1 * n * dt, 1)]
    specs = [(kind, t, pk) for kind in ("cusp", "zac") for t in taps for pk in picks]
    rt, ft = L.us(rng.uniform(1.0, 8.0)), L.us(rng.uniform(0.5, 3.0))
    vl = concat_variants(L, [(_fir(L, None, cfg, kind, t, rt, ft, step, pol, *pk), 0) for kind, t, pk in specs])
    vo = concat_variants(L, [(_fir(L, B, cfg, kind, t, rt, ft, step, pol, *pk), 0) for kind, t, pk in specs])
    S_lib = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True)
    S_orc = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True, builders=B)
    assert (S_orc.sig_dni.n_w, S_orc.sig_dni.degree) == (n_w, degree)
    scales = event_scales(O, S_orc, wf)
    ref = O.sweep(S_orc, wf, vo.array)
    tol = np.stack([fir_tolerance(scales, S_lib, S_orc, vl.array[i], vo.array[i]) for i in range(len(vo))], axis=1)
    return dict(wf=wf, S_lib=S_lib, S_orc=S_orc, vl=vl, vo=vo, ref=ref, tol=tol, scales=scales, specs=specs)


@gpu
@pytest.mark.parametrize("n,degree,n_w", EDGE_CASES)
def test_cuspzac_edge_set(L, O, handle, n, degree, n_w):
    k = cuspzac_edge_case(L, O, n, degree, n_w)
    wf = k["wf"]
    got = np.zeros((len(wf), len(k["vl"])))
    handle.gsweep_run_host(k["S_lib"], wf.ctypes.data, len(wf), n, k["vl"].array, got.ctypes.data)
    r = check_fir(got, k["ref"], k["tol"], (n, degree, n_w))
    assert np.isfinite(got).all()
    print(f"n {n} degree {degree} n_w {n_w}: largest error / bound {r:.3g}")


# ---------------------------------------------------------------------------------------------------------------------
# 2. Savitzky-Golay
# ---------------------------------------------------------------------------------------------------------------------
def sg_case(L, O, seed):
    cfg, tau, pf, n, step = _draw(L, 1300 + seed)
    rng = np.random.default_rng(71000 + seed)
    t_first = _t_first(L, rng, cfg)
    cfg = _shifted(cfg, t_first)
    pol = _policy(L, rng)
    dt = step.ns()
    # a window-length grid from 1 to 33 samples (1 and 33 taps always; steps of 1 sample also give even lengths, which the
    # policy rounds up / down); degree 2 / 3 of the draw: fits with fewer taps than coefficients are underdetermined
    ks = int(rng.choice([1, 2, 4, 8, 16, 32]))
    cfg.a_grid_wl_sg = (L.ns(dt), L.ns(ks * dt), L.ns(33 * dt))
    wls = L.grid_values(cfg.a_grid_wl_sg)
    B = O.OracleBuilders()
    kw = dict(n_samples=n, t_first=t_first, step=step, policy=pol)
    gl, go = L.sg_sweep_variants(cfg, wls, **kw), L.sg_sweep_variants(cfg, wls, builders=B, **kw)
    wf = np.ascontiguousarray(np.concatenate([L.synth.generate_host(60, first_event=29000 * (seed + 1)),
                                              L.synth.generate_host(4, mode=1)])[:, :n])
    S_lib = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True)
    S_orc = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True, builders=B)
    scales = event_scales(O, S_orc, wf)
    # the rising edge of the current pulse of the four noise-free events (one pulse, a flat current from its first sample on):
    # every SG trace whose kernel reaches that first sample still rises there
    dy = np.diff(scales[60][1])
    edge = int(np.nonzero(dy > 0.5 * dy.max())[0][0]) + 1
    windows = []                        # (grid variant, win_from, win_until, what)
    for i in range(len(gl)):
        last = n - gl.array[i].n_taps
        k, j = int(rng.integers(2, 400)), int(rng.integers(0, last))
        ee = edge - gl.array[i].sg_offset
        windows += [(i, 0, k, "[0, k]"), (i, last - k, last, "ends at n - T"), (i, 0, last, "whole trace"),
                    (i, j, j, "one sample"), (i, j, j + 1, "two samples"), (i, last - 1, last, "last two samples"),
                    (i, ee - 300, ee, "rising edge")]
    vl = concat_variants(L, [(gl, i) for i in range(len(gl))] + [(gl, w[0]) for w in windows])
    vo = concat_variants(L, [(go, i) for i in range(len(go))] + [(go, w[0]) for w in windows])
    for q, (_, a, b, _) in enumerate(windows):
        for v in (vl, vo):
            v.array[len(gl) + q].win_from, v.array[len(gl) + q].win_until = a, b
    ref = O.sweep(S_orc, wf, vo.array)
    what = ["grid"] * len(gl) + [w[3] for w in windows]
    return dict(cfg=cfg, tau=tau, pf=pf, n=n, step=step, t_first=t_first, pol=pol, wf=wf, S_lib=S_lib, S_orc=S_orc,
                scales=scales, vl=vl, vo=vo, ref=ref, n_grid=len(gl), what=what)


@gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_sg_sweeps_randomised(L, O, handle, seed):
    k = sg_case(L, O, seed)
    wf, vl, vo, ref, scales = k["wf"], k["vl"], k["vo"], k["ref"], k["scales"]
    got = np.zeros((len(wf), len(vl)))
    handle.gsweep_run_host(k["S_lib"], wf.ctypes.data, len(wf), k["n"], vl.array, got.ctypes.data)
    assert np.isfinite(got).all()
    worst, ties = 0.0, 0
    for v in range(len(vl)):
        w, t = check_sg(O, scales, got[:, v], ref[:, v], vl.array[v], vo.array[v], (seed, v, k["what"][v]))
        worst, ties = max(worst, w), ties + t
    # the public wrapper on the draw's own grid runs the same variants (with the energy variant in front)
    tab = L.dsp_sg_optimization(L.RDWaveforms(wf, k["t_first"], k["step"]), k["cfg"], k["tau"], k["pf"], policy=k["pol"],
                                handle=handle)
    with np.errstate(divide="ignore", invalid="ignore"):
        assert np.array_equal(tab["aoe"], got[:, :k["n_grid"]] / tab["energy"][:, None], equal_nan=True)
    # the chain's a_sg (current maximum of the SG filter of window length pars_filter.sg.wl) is the sweep's variant at that
    # window length
    from parity import TOL
    from test_gpu_icpc import _argmax_tie_ok
    P = L.resolve_icpc_params(k["cfg"], k["tau"], k["pf"], n_samples=k["n"], t_first=k["t_first"], step=k["step"],
                              policy=k["pol"])
    rows = L.dsp_icpc_rows(wf, P, handle=handle)
    one = L.sg_sweep_variants(k["cfg"], [k["pf"]["sg"]["wl"]], n_samples=k["n"], t_first=k["t_first"], step=k["step"],
                              policy=k["pol"])
    assert (one.array[0].win_from, one.array[0].win_until) == (P.cur_from[0], P.cur_until[0])
    val = np.zeros((len(wf), 1))
    handle.gsweep_run_host(k["S_lib"], wf.ctypes.data, len(wf), k["n"], one.array, val.ctypes.data)
    a_sg = rows[:, L.COL["a_sg"]]
    rtol, atol = TOL["a_sg"]            # (the chain's a_sg tolerance against the oracle; the sweep's value is far tighter)
    for e in np.nonzero(np.abs(val[:, 0] - a_sg) > atol + rtol * np.abs(a_sg))[0]:
        assert _argmax_tie_ok(L, O, P, wf[e], val[e, 0], "a_sg") and _argmax_tie_ok(L, O, P, wf[e], a_sg[e], "a_sg"), \
            (e, val[e, 0], a_sg[e])
    print(f"seed {seed}: largest error / bound {worst:.3g}, argmax ties {ties}")


# ---------------------------------------------------------------------------------------------------------------------
# 3. mixed and large variant sets
# ---------------------------------------------------------------------------------------------------------------------
MIXED = [1, 255, 256, 257, 1024]


def _short_cfg(L, seed, n, t_first):
    cfg, tau, _, _, step = _draw(L, seed)
    full = np.concatenate([L.synth.generate_host(23, first_event=3000 * seed), L.synth.generate_host(1, mode=1)])
    wf, cfg = _short_traces(L, full, n, cfg, t_first)
    span = n * 16.0 / 1000.0
    cfg.current_window = (t_first + L.us(span * 0.3), t_first + L.us(span * 0.7))
    return cfg, tau, L.ns(16.0), wf


def mixed_case(L, O, nvar):
    n, t_first = 2048, L.ns(-1000.0)
    cfg, tau, step, wf = _short_cfg(L, 1500 + nvar, n, t_first)
    rng = np.random.default_rng(81000 + nvar)
    pol = _policy(L, rng)
    B = O.OracleBuilders()
    dt, t0 = step.ns(), t_first.ns()
    traps = L.trap_sweep_variants([L.us(v) for v in np.sort(rng.uniform(1.0, 6.0, 8))],
                                  [L.us(v) for v in np.sort(rng.uniform(0.5, 2.0, 4))], step, mode="ft")
    specs = [(str(rng.choice(["cusp", "zac"])), int(rng.integers(50, 300)), L.us(rng.uniform(0.5, 4.0)), L.us(rng.uniform(0.2, 1.5)),
              *((t0 + rng.uniform(-0.1, 1.1) * n * dt, 0) if q % 2 else (rng.uniform(0.0, 4000.0), 1))) for q in range(12)]
    firs = [[_fir(L, b, cfg, kind, t, rt, ft, step, pol, pk, mode) for kind, t, rt, ft, pk, mode in specs] for b in (None, B)]
    kw = dict(n_samples=n, t_first=t_first, step=step, policy=pol)
    wls = [L.ns(k * dt) for k in (1, 3, 5, 9, 16, 21, 30, 33)]
    sgs = [L.sg_sweep_variants(cfg, wls, **kw), L.sg_sweep_variants(cfg, wls, builders=B, **kw)]
    kinds = np.array([1]) if nvar == 1 else rng.permutation(np.r_[[0, 1, 2], rng.integers(0, 3, nvar - 3)])
    if nvar > 256:
        kinds[-1] = 0                   # a trapezoid variant beyond the first pass of the one-thread-per-variant loop
    pick = [int(rng.integers(0, [len(traps), len(specs), len(wls)][k])) for k in kinds]
    parts = [[(traps, i) if k == 0 else ((firs[s][i], 0) if k == 1 else (sgs[s], i)) for k, i in zip(kinds, pick)] for s in (0, 1)]
    vl, vo = concat_variants(L, parts[0]), concat_variants(L, parts[1])
    S_lib = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True)
    S_orc = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True, builders=B)
    scales = event_scales(O, S_orc, wf)
    ref = O.sweep(S_orc, wf, vo.array)
    tol = {v: fir_tolerance(scales, S_lib, S_orc, vl.array[v], vo.array[v]) for v in np.nonzero(kinds == 1)[0]}
    trap_only = concat_variants(L, [(traps, i) for k, i in zip(kinds, pick) if k == 0] or [(traps, 0)])
    return dict(cfg=cfg, tau=tau, n=n, t_first=t_first, step=step, wf=wf, kinds=kinds, vl=vl, vo=vo, S_lib=S_lib, S_orc=S_orc,
                scales=scales, ref=ref, tol=tol, trap_only=trap_only)


@gpu
@pytest.mark.parametrize("nvar", MIXED)
def test_mixed_variant_sets(L, O, handle, nvar):
    from legenddsp.jl_b200.dsp_filter_optimization import _run_general
    k = mixed_case(L, O, nvar)
    W = L.RDWaveforms(k["wf"], k["t_first"], k["step"])
    got, aux = _run_general(W, k["cfg"], k["tau"], k["vl"], f64=True, want_aux=True, handle=handle)
    kinds, ref, vl, vo = k["kinds"], k["ref"], k["vl"], k["vo"]
    assert got.shape == (len(k["wf"]), nvar)
    worst = {0: 0.0, 1: 0.0, 2: 0.0}
    for v in range(nvar):
        if kinds[v] == 1:
            worst[1] = max(worst[1], check_fir(got[:, v], ref[:, v], k["tol"][v], ("fir", nvar, v)))
        elif kinds[v] == 2:
            worst[2] = max(worst[2], check_sg(O, k["scales"], got[:, v], ref[:, v], vl.array[v], vo.array[v], ("sg", nvar, v))[0])
    # the trapezoid variants: the oracle's (as tests/test_gpu_fastpaths.py B: the four look-ups per output are exact to
    # ~1e-9 relative), and bit for bit the same variants run alone -- on the warp path, which refuses any other set
    t = kinds == 0
    with sweep_path("warp"):
        alone, aux_alone = _run_general(W, k["cfg"], k["tau"], k["trap_only"], f64=True, want_aux=True, handle=handle)
    if t.any():
        assert np.allclose(got[:, t], ref[:, t], rtol=1e-8, atol=1e-6, equal_nan=True), np.nanmax(np.abs(got[:, t] - ref[:, t]))
        assert np.array_equal(got[:, t], alone, equal_nan=True)
    assert np.array_equal(aux, aux_alone)
    print(f"n_variants {nvar}: {int(t.sum())} trapezoid, {int((kinds == 1).sum())} FIR, {int((kinds == 2).sum())} SG; "
          f"largest error / bound FIR {worst[1]:.3g}, SG {worst[2]:.3g}")


# ---------------------------------------------------------------------------------------------------------------------
# 4. sample types
# ---------------------------------------------------------------------------------------------------------------------
def wide_case(L, O):
    """uint32 samples above 65535 (n = 4096, the largest the 32-bit instantiation takes) with an external baseline; the last
    three rows sum to 2^32 - 1 (exact), 2^32 and far beyond (NaN rows)"""
    n, t_first = 4096, L.ns(2000.0)
    cfg, tau, step, wf16 = _short_cfg(L, 1600, n, t_first)
    rng = np.random.default_rng(1600)
    pol = _policy(L, rng)
    B = O.OracleBuilders()
    flat = np.full(n, 1048575, np.uint32)                   # 4096 * 1048575 = 2^32 - 4096
    wrap = [flat.copy(), flat.copy(), np.full(n, 3000000, np.uint32)]
    wrap[0][:8] += 512
    wrap[0][0] -= 1                                          # sum 2^32 - 1
    wrap[1][:8] += 512                                       # sum 2^32
    wf = np.ascontiguousarray(np.concatenate([wf16.astype(np.uint32) * 3 + 20000, np.stack(wrap)]))
    sums = wf.astype(np.uint64).sum(axis=1)
    assert int(sums[-3]) == 2 ** 32 - 1 and int(sums[-2]) == 2 ** 32 and wf.max() > 65535
    own = np.array([O.signalstats(x.astype(np.float64), t_first.ns(), 16.0, 0, 200)["mean"] for x in wf])
    bl = np.ascontiguousarray(own + rng.normal(0.0, 20.0, len(wf)))
    dt, t0 = step.ns(), t_first.ns()
    specs = [("cusp", 1500, L.us(4.0), L.us(1.0), t0 + 0.35 * n * dt, 0), ("zac", 700, L.us(2.0), L.us(0.5), 6000.0, 1),
             ("cusp", 100, L.us(0.5), L.us(0.2), t0 + (0.6 * n + 0.5) * dt, 0)]
    kw = dict(n_samples=n, t_first=t_first, step=step, policy=pol)
    wls = [L.ns(k * dt) for k in (1, 7, 33)]
    traps = L.trap_sweep_variants([L.us(3.0)], [L.us(1.0)], step, mode="ft")
    out = []
    for b in (None, B):
        sgv = L.sg_sweep_variants(cfg, wls, builders=b, **kw)
        out.append(concat_variants(L, [(_fir(L, b, cfg, *s[:4], step, pol, *s[4:]), 0) for s in specs]
                                   + [(sgv, i) for i in range(len(wls))] + [(traps, 0)]))
    vl, vo = out
    S_lib = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True, external_baseline=True)
    S_orc = L.resolve_sweep_params(cfg, tau, n_samples=n, t_first=t_first, step=step, out_f64=True, external_baseline=True, builders=B)
    ok = slice(0, len(wf) - 2)
    scales = event_scales(O, S_orc, wf[ok], baseline=bl[ok])
    ref = O.sweep_ext(S_orc, wf, vo.array, baseline=bl)
    tol = {v: fir_tolerance(scales, S_lib, S_orc, vl.array[v], vo.array[v]) for v in range(len(specs))}
    return dict(wf=wf, bl=bl, vl=vl, vo=vo, S_lib=S_lib, S_orc=S_orc, scales=scales, ref=ref, tol=tol, n_fir=len(specs),
                n_sg=len(wls), ok=ok, cfg=cfg, tau=tau, t_first=t_first, step=step)


@gpu
def test_uint32_samples_external_baseline_and_float32(L, O, handle):
    k = wide_case(L, O)
    wf, bl, vl, vo, ref, ok = k["wf"], k["bl"], k["vl"], k["vo"], k["ref"], k["ok"]
    ne, n, nv = wf.shape[0], wf.shape[1], len(vl)
    got = np.zeros((ne, nv))
    handle.gsweep_run_ext_host(k["S_lib"], wf.ctypes.data, 4, bl.ctypes.data, ne, n, vl.array, got.ctypes.data, None)
    S32 = L.resolve_sweep_params(k["cfg"], k["tau"], n_samples=n, t_first=k["t_first"], step=k["step"], external_baseline=True)
    got32 = np.zeros((ne, nv), np.float32)
    handle.gsweep_run_ext_host(S32, wf.ctypes.data, 4, bl.ctypes.data, ne, n, vl.array, got32.ctypes.data, None)
    # waveforms whose samples sum to 2^32 or more: NaN in every variant kind (the uint32 prefix sums would have wrapped);
    # 2^32 - 1 is still exact
    assert np.isnan(got[-2:]).all() and np.isnan(got32[-2:]).all() and np.isfinite(got[:-2]).all()
    assert np.array_equal(got32, got.astype(np.float32), equal_nan=True)
    worst = 0.0
    for v in range(k["n_fir"]):
        worst = max(worst, check_fir(got[ok, v], ref[ok, v], k["tol"][v], ("uint32 fir", v)))
        r32 = ref[ok, v]
        check_fir(got32[ok, v].astype(np.float64), r32, k["tol"][v] + np.spacing(np.abs(r32).astype(np.float32)).astype(np.float64),
                  ("uint32 fir float32", v))
    for v in range(k["n_fir"], k["n_fir"] + k["n_sg"]):
        check_sg(O, k["scales"], got[ok, v], ref[ok, v], vl.array[v], vo.array[v], ("uint32 sg", v))
    v = nv - 1                                               # the trapezoid variant
    assert np.allclose(got[ok, v], ref[ok, v], rtol=1e-8, atol=1e-6)
    print(f"uint32: largest FIR error / bound {worst:.3g}")


# ---------------------------------------------------------------------------------------------------------------------
# 5. validation boundaries of kinds 1 and 2
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_fir_and_sg_validation_boundaries(L, handle):
    cfg, tau = L.example_config(), L.us(500.0)
    wf = L.synth.generate_host(2)

    def run(v, n=8192):
        S = L.resolve_sweep_params(cfg, tau, n_samples=n, out_f64=True, external_baseline=True)
        out = np.zeros((2, max(1, len(v))))
        handle.gsweep_run_host(S, wf.ctypes.data, 2, 8192, v.array, out.ctypes.data)
        return out

    def fir(taps):
        v = L.SweepVariants(1)
        v.array[0].kind, v.array[0].pickoff_ns = 1, 40000.0
        v.set_coeffs(0, np.full(taps, 1.0 / taps))
        return v

    def sg(taps, offset, a, b):
        v = L.SweepVariants(1)
        v.array[0].kind, v.array[0].sg_offset, v.array[0].win_from, v.array[0].win_until = 2, offset, a, b
        v.set_coeffs(0, np.linspace(-1.0, 1.0, taps))
        return v

    def accepted(v, n=8192):
        assert np.isfinite(run(v, n)).all()

    def rejected(v, n=8192):
        with pytest.raises(L.LgdspError):
            run(v, n)

    nw = L.resolve_sweep_params(cfg, tau).sig_dni.n_w
    accepted(fir(L._abi.LGDSP_MAX_FIR))
    rejected(fir(L._abi.LGDSP_MAX_FIR + 1))
    accepted(fir(1024 - nw + 1), n=1024)                  # n - L + 1 == n_w
    rejected(fir(1024 - nw + 2), n=1024)                  # n - L + 1 == n_w - 1
    accepted(sg(33, 16, 3000, 3100))
    rejected(sg(34, 16, 3000, 3100))
    accepted(sg(9, 8, 3000, 3100))                         # sg_offset T - 1
    rejected(sg(9, 9, 3000, 3100))                         # sg_offset T
    accepted(sg(9, 4, 8000, 8192 - 9))                     # win_until n - T
    rejected(sg(9, 4, 8000, 8192 - 9 + 1))
    accepted(sg(9, 4, 3000, 3000))
    rejected(sg(9, 4, 3001, 3000))                         # win_from > win_until
    rejected(L.SweepVariants(0))                           # n_variants 0 and 1025 (1024 runs in test_mixed_variant_sets)
    rejected(L.trap_sweep_variants([L.us(4.0)] * 1025, [L.us(2.0)], L.ns(16.0), mode="ft"))


# ---------------------------------------------------------------------------------------------------------------------
# the oracle side, without a GPU
# ---------------------------------------------------------------------------------------------------------------------
def _moved(L, vo, v, taps=None, dpick=0.0, win_until=None):
    """a copy of variant v of vo with other taps, its pick-off moved or its window shortened"""
    out = concat_variants(L, [(vo, v)])
    if taps is not None:
        out.set_coeffs(0, taps)
    out.array[0].pickoff_ns += dpick
    if win_until is not None:
        out.array[0].win_until = win_until
    return out


@pytest.mark.parametrize("seed", SEEDS)
def test_oracle_side_of_the_sweeps(L, O, seed):
    """the draws, variant tables and oracle outputs of the GPU tests above build without a GPU, and each tolerance is tight
    enough: one dropped tap or a pick-off one sample away moves the oracle by more than the bound, and the rising-edge
    windows do put the maximum on their last sample, where a scan one sample short would miss it"""
    k = cuspzac_case(L, O, seed)
    wf, S, dt = k["wf"], k["S_orc"], k["step"].ns()
    gen = slice(0, 60)
    for mode, (vl, vo, ref, tol) in k["sets"].items():
        assert np.isfinite(ref).all() and (tol > 0).all()
        for v in range(len(vo)):
            c = _coeffs(vo.array[v])
            c[-1] = 0.0
            drop = O.sweep(S, wf, _moved(L, vo, v, taps=c).array)[:, 0]
            assert (np.abs(drop - ref[:, v]) > tol[:, v])[gen].mean() > 0.95, (mode, v, "dropped tap")
            if mode == "ft" or k["where"] in ("inside", "half sample"):
                for d in (-dt, dt):
                    moved = O.sweep(S, wf, _moved(L, vo, v, dpick=d).array)[:, 0]
                    assert (np.abs(moved - ref[:, v]) > tol[:, v])[gen].mean() > 0.9, (mode, v, "pick-off", d)
    k = sg_case(L, O, seed)
    rising = [v for v, w in enumerate(k["what"]) if w == "rising edge"]
    for v in rising:
        vo = k["vo"].array[v]
        if not _coeffs(vo).any():            # (one tap: the derivative of a constant fit is 0 everywhere)
            continue
        at_end = [e for e in range(len(k["wf"])) if int(np.argmax(sg_window_trace(O, k["scales"][e], vo))) == vo.win_until - vo.win_from]
        assert set(range(60, 64)) <= set(at_end), (v, at_end)
        short = O.sweep(k["S_orc"], k["wf"], _moved(L, k["vo"], v, win_until=vo.win_until - 1).array)[:, 0]
        d = np.array([sg_tolerance(k["scales"][e], k["vl"].array[v], vo) for e in at_end])
        assert (np.abs(short[at_end] - k["ref"][at_end, v]) > 2.0 * d).all(), v
    assert np.isfinite(k["ref"]).all()


@pytest.mark.parametrize("n,degree,n_w", EDGE_CASES)
def test_oracle_side_of_the_edge_sets(L, O, n, degree, n_w):
    k = cuspzac_edge_case(L, O, n, degree, n_w)
    assert np.isfinite(k["ref"]).all() and (k["tol"] > 0).all()
    taps = {t for _, t, _ in k["specs"]}
    assert (n - n_w + 1 in taps) == (n - n_w + 1 <= L._abi.LGDSP_MAX_FIR)
    assert (L._abi.LGDSP_MAX_FIR in taps) == (n - n_w + 1 >= L._abi.LGDSP_MAX_FIR)


def test_oracle_side_of_the_mixed_and_wide_sets(L, O):
    for nvar in MIXED:
        k = mixed_case(L, O, nvar)
        assert len(k["vo"]) == nvar and np.isfinite(k["ref"]).all()
        if nvar > 256:
            assert (k["kinds"][256:] == 0).any() and (k["kinds"][:256] != 0).any()
    k = wide_case(L, O)
    assert np.isfinite(k["ref"]).all()
