"""The one-warp-per-waveform trapezoid sweep kernel (csrc/lgdsp_sweep_warp.cuh) against the one-CTA-per-waveform kernel
(bit for bit, LGDSP_SWEEP_PATH selects the path) and against the CPU oracle; src/dsp_filter_optimization.jl:102-133, 241-274."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


class sweep_path:
    def __init__(self, which):
        self.which = which

    def __enter__(self):
        self.old = os.environ.get("LGDSP_SWEEP_PATH")
        os.environ["LGDSP_SWEEP_PATH"] = self.which

    def __exit__(self, *a):
        if self.old is None:
            os.environ.pop("LGDSP_SWEEP_PATH", None)
        else:
            os.environ["LGDSP_SWEEP_PATH"] = self.old


def _pathological(n):
    rows = [np.full(n, 12000, np.uint16), (np.arange(n) * 7 % 65521).astype(np.uint16),
            np.where(np.arange(n) % 2 == 0, 100, 60000).astype(np.uint16), np.full(n, 65520, np.uint16), np.zeros(n, np.uint16),
            np.clip(9000 + np.arange(n) * 6, 0, 65520).astype(np.uint16)]
    for at in (40, n // 2, n - 200, n - 20):   # steps at the trace ends: clamped pick-off windows, second window of the warp path
        s = np.full(n, 10000, np.uint16)
        s[at:] = 50000
        rows.append(s)
    neg = np.full(n, 30000, np.uint16)
    neg[n // 3:] = 5000
    rows.append(neg)
    return np.stack(rows)


def _both(L, handle, W, cfg, tau, var, f64, want_aux=True):
    from legenddsp.jl_b200.dsp_filter_optimization import _run_general
    with sweep_path("warp"):
        a = _run_general(W, cfg, tau, var, f64=f64, want_aux=want_aux, handle=handle)
    with sweep_path("cta"):
        b = _run_general(W, cfg, tau, var, f64=f64, want_aux=want_aux, handle=handle)
    return a, b


def _grid(L):
    rts = [L.us(1.0 + 0.75 * i) for i in range(20)]
    fts = [L.us(1.0 + 0.3 * i) for i in range(10)]
    return rts, fts


def test_warp_path_equals_cta_path_and_oracle_on_the_grid(L, O, handle):
    cfg, tau = L.example_config(), L.us(500.0)
    wf = np.concatenate([L.synth.generate_host(700, first_event=4242), L.synth.generate_host(40, mode=1), _pathological(8192)])
    W = L.RDWaveforms(wf)
    rts, fts = _grid(L)
    var = L.trap_sweep_variants(rts, fts, L.ns(16.0), mode="ft")
    for f64 in (True, False):
        (a, aa), (b, ba) = _both(L, handle, W, cfg, tau, var, f64)
        assert np.array_equal(a, b, equal_nan=True), np.nanmax(np.abs(a.astype(np.float64) - b))
        assert np.array_equal(aa, ba, equal_nan=True)
    so = L.resolve_sweep_params(cfg, tau, builders=O.OracleBuilders(), out_f64=True)
    sub = np.r_[0:120, 700:len(wf)]
    ref, raux = O.sweep(so, wf[sub], var.array, want_aux=True)
    (a, aa), _ = _both(L, handle, L.RDWaveforms(wf[sub]), cfg, tau, var, True)
    nat = slice(0, 160)   # generator events: tight; the pathological traces have ties everywhere (flat y: any crossing)
    assert np.allclose(a[nat], ref[nat], rtol=1e-8, atol=1e-6, equal_nan=True), np.nanmax(np.abs(a[nat] - ref[nat]))
    assert np.allclose(aa[nat], raux[nat], rtol=1e-9, atol=1e-9, equal_nan=True)


@pytest.mark.parametrize("n_samples", [264, 1024, 4104, 6000, 8192])
def test_warp_path_ragged_lengths(L, O, handle, n_samples):
    cfg, tau = L.example_config(), L.us(500.0)
    full = L.synth.generate_host(96, first_event=77)
    a0 = max(0, 3400 - n_samples // 2) // 8 * 8
    wf = np.ascontiguousarray(full[:, a0:a0 + n_samples])
    W = L.RDWaveforms(wf)
    # short filters so that they fit the short traces
    span = min(n_samples, 4800) * 16.0 / 1000.0   # (longer filters than ~13 us leave the warp path's window capacity)
    rts = [L.us(span * f) for f in (0.02, 0.05, 0.11, 0.17)]
    fts = [L.us(span * f) for f in (0.01, 0.04)]
    from legenddsp.jl_b200.config import DSPConfig, example_config_dict
    d = example_config_dict()
    d["bl_window"] = {"min": L.us(0.0), "max": L.us(span * 0.2)}
    cfgs = DSPConfig.from_dict(d)
    var = L.trap_sweep_variants(rts, fts, L.ns(16.0), mode="ft")
    (a, aa), (b, ba) = _both(L, handle, W, cfgs, tau, var, True)
    assert np.array_equal(a, b, equal_nan=True)
    assert np.array_equal(aa, ba, equal_nan=True)
    so = L.resolve_sweep_params(cfgs, tau, n_samples=n_samples, builders=O.OracleBuilders(), out_f64=True)
    ref = O.sweep(so, wf, var.array)
    assert np.allclose(a, ref, rtol=1e-8, atol=1e-6, equal_nan=True)


def test_rt_sweep_with_fixed_pickoff_and_ineligible_sets(L, O, handle):
    cfg, tau = L.example_config(), L.us(500.0)
    wf = L.synth.generate_host(200, first_event=9)
    W = L.RDWaveforms(wf)
    from legenddsp.jl_b200.dsp_filter_optimization import _run_general
    # fixed pick-off (mode 0): the warp path skips max(y) / the crossing and reads only the samples up to the last look-up
    var = L.trap_sweep_variants(L.grid_values(cfg.e_grid_rt_trap), [L.us(2.0)], L.ns(16.0), mode="rt", pickoff=cfg.enc_pickoff_trap)
    with sweep_path("cta"):
        b = _run_general(W, cfg, tau, var, f64=True, handle=handle)
    with sweep_path("warp"):   # the example grid (1 .. 16 us at ft = 2 us, pick-off 40 us) reaches 2 176 samples: eligible
        a = _run_general(W, cfg, tau, var, f64=True, handle=handle)
    assert np.array_equal(a, b, equal_nan=True)
    ref = O.sweep(L.resolve_sweep_params(cfg, tau, builders=O.OracleBuilders(), out_f64=True), wf, var.array)
    assert np.allclose(a, ref, rtol=1e-8, atol=1e-6, equal_nan=True)
    a = _run_general(W, cfg, tau, var, f64=True, handle=handle)   # default dispatch: whichever path, same numbers
    assert np.array_equal(a, b, equal_nan=True)
    # with the aux outputs the fixed pick-off set needs t50 after all (without them the warp path skips max(y) / the crossing)
    (a2, aa2), (b2, ba2) = _both(L, handle, W, cfg, tau, var, True)
    assert np.array_equal(a2, b2, equal_nan=True) and np.array_equal(aa2, ba2, equal_nan=True) and np.array_equal(a2, b, equal_nan=True)
    # CUSP variants are never eligible: demanding the warp path is an error, the default dispatch runs them
    cvar = L.cuspzac_sweep_variants(cfg, "cusp", [L.us(6.0)], [L.us(2.0)], L.ns(16.0), mode="ft")
    with sweep_path("warp"):
        with pytest.raises(Exception, match="LGDSP_SWEEP_PATH=warp"):
            _run_general(W, cfg, tau, cvar, f64=True, handle=handle)
    assert np.isfinite(_run_general(W, cfg, tau, cvar, f64=True, handle=handle)).all()


def test_warp_path_large_batch_determinism(L, handle):
    import torch
    cfg, tau = L.example_config(), L.us(500.0)
    n = 20000
    d = torch.empty((n, 8192), dtype=torch.int16, device="cuda")
    L.synth.generate_device(handle, d.data_ptr(), n, first_event=31337)
    S = L.resolve_sweep_params(cfg, tau)
    rts, fts = _grid(L)
    var = L.trap_variants(rts, fts, L.ns(16.0), mode="ft")
    outs = []
    for which in ("warp", "warp", "cta"):
        o = torch.zeros((n, 200), dtype=torch.float32, device="cuda")
        with sweep_path(which):
            handle.sweep_run_device(S, d.data_ptr(), n, 8192, var, o.data_ptr())
        handle.synchronize()
        outs.append(o.cpu().numpy())
    assert np.array_equal(outs[0], outs[1], equal_nan=True)
    assert np.array_equal(outs[0], outs[2], equal_nan=True)


@pytest.mark.parametrize("seed", list(range(int(os.environ.get("LGDSP_FUZZ_SEEDS_SWEEP", "6")))))
def test_warp_path_fuzz_against_cta_path(L, O, handle, seed):
    """random configurations (sampling step 16 / 8 / 12.5 ns -> both forms of the division by dt, PolynomialDNI windows of 8 .. 60
    samples and degree 1 .. 3 -> the run-time-sized pick-off loop, trace lengths 6144 .. 8192, random baseline windows and decay
    times) and random (rt, ft) lists that fit the warp path's window: every output and the aux columns bit for bit"""
    from test_gpu_fuzz import _draw
    from legenddsp.jl_b200.dsp_filter_optimization import _run_general
    cfg, tau, _, n, step = _draw(L, 300 + seed)
    rng = np.random.default_rng(9000 + seed)
    sc = step.ns() / 16.0
    rts = [L.ns(float(v) * 1000.0 * sc) for v in np.sort(rng.uniform(0.3, 14.0, int(rng.integers(3, 24))))]
    fts = [L.ns(float(v) * 1000.0 * sc) for v in np.sort(rng.uniform(0.1, 4.0, int(rng.integers(2, 12))))]
    wf = np.ascontiguousarray(np.concatenate([L.synth.generate_host(150, first_event=900 * (seed + 1)),
                                              L.synth.generate_host(10, mode=1), _pathological(8192)])[:, :n])
    W = L.RDWaveforms(wf, L.ns(0.0), step)
    var = L.trap_sweep_variants(rts, fts, step, mode="ft")
    f64 = bool(seed % 2)
    with sweep_path("warp"):
        a, aa = _run_general(W, cfg, tau, var, f64=f64, want_aux=True, handle=handle)
    with sweep_path("cta"):
        b, ba = _run_general(W, cfg, tau, var, f64=f64, want_aux=True, handle=handle)
    assert np.array_equal(a, b, equal_nan=True), np.nanmax(np.abs(a.astype(np.float64) - b))
    assert np.array_equal(aa, ba, equal_nan=True)
    assert np.isfinite(a).mean() > 0.9
