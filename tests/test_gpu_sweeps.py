"""GPU parity of the general sweeps (lgdsp_sweep_run) against the CPU oracle: CUSP / ZAC rise- and flat-top-time sweeps
and the Savitzky-Golay window-length sweep (src/dsp_filter_optimization.jl:145-231, 286-375, 393-441)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _oracle(L, O, cfg, tau, wf, variants, want_aux=False):
    so = L.resolve_sweep_params(cfg, tau, builders=O.OracleBuilders(), out_f64=True)
    return O.sweep(so, wf, variants.array, want_aux=want_aux)


@pytest.mark.parametrize("kind", ["cusp", "zac"])
def test_cuspzac_rt_and_ft_sweeps(L, O, handle, kind):
    cfg = L.example_config()
    tau = L.us(500.0)
    wf = L.synth.generate_host(48, first_event=321)
    W = L.RDWaveforms(wf)
    step = L.ns(16.0)
    # rise-time sweep at ft = 2 us, fixed pick-off enc_pickoff_*: Float64 [n_rt, n_events]
    f_rt = L.dsp_cusp_rt_optimization if kind == "cusp" else L.dsp_zac_rt_optimization
    got = f_rt(W, cfg, tau, ft=L.us(2.0), handle=handle)
    rts = L.grid_values(cfg.e_grid_rt_cusp if kind == "cusp" else cfg.e_grid_rt_zac)
    var = L.cuspzac_sweep_variants(cfg, kind, rts, [L.us(2.0)], step, mode="rt", builders=O.OracleBuilders())
    ref = _oracle(L, O, cfg, tau, wf, var).T
    assert got.shape == (len(rts), 48) and got.dtype == np.float64
    assert np.allclose(got, ref, rtol=1e-8, atol=1e-6, equal_nan=True), np.nanmax(np.abs(got - ref))
    # flat-top sweep at rt = 6 us, pick-off t50 + flt_length/2: Float32 [n_ft, n_events]
    f_ft = L.dsp_cusp_ft_optimization if kind == "cusp" else L.dsp_zac_ft_optimization
    got = f_ft(W, cfg, tau, L.us(6.0), handle=handle)
    fts = L.grid_values(cfg.e_grid_ft_cusp if kind == "cusp" else cfg.e_grid_ft_zac)
    var = L.cuspzac_sweep_variants(cfg, kind, [L.us(6.0)], fts, step, mode="ft", builders=O.OracleBuilders())
    ref = _oracle(L, O, cfg, tau, wf, var).T
    assert got.shape == (len(fts), 48) and got.dtype == np.float32
    assert np.allclose(got, ref.astype(np.float32), rtol=1e-6, atol=1e-4, equal_nan=True)
    # the (rt, ft) point of the default filter equals e_cusp / e_zac of the full chain up to the t50 convention
    # (the chain thresholds at half the PRE-PZ maximum, the sweeps at half the PZ maximum): compare the scale only
    P = L.resolve_icpc_params(cfg, tau, builders=O.OracleBuilders())
    rows = L.dsp_icpc_rows(wf, P, handle=handle)
    drt, dft = L.get_fltpars({}, kind, cfg)
    var1 = L.cuspzac_sweep_variants(cfg, kind, [drt], [dft], step, mode="ft")
    one = _oracle(L, O, cfg, tau, wf, var1)[:, 0]
    big = rows[:, L.COL["e_max"]] > 500
    assert np.allclose(one[big], rows[big, L.COL["e_" + kind]], rtol=2e-3)


def test_sg_optimization(L, O, handle):
    # the example grid starts at 30 ns = 2 samples -> 3 taps with degree 3: the underdetermined fit takes the
    # minimum-norm coefficients (lgdsp_sg_coeffs); the grid runs as it is
    from importlib import import_module
    cfgm = import_module("legenddsp.jl_b200.config")
    d = cfgm.example_config_dict()
    ex = L.dsp_sg_optimization(L.RDWaveforms(L.synth.generate_host(2)), L.example_config(), L.us(500.0), {}, handle=handle)
    assert ex["aoe"].shape == (2, 11) and np.isfinite(ex["aoe"]).all()
    d["a_grid_wl_sg"] = {"start": L.ns(80.0), "stop": L.ns(350.0), "step": L.ns(32.0)}
    cfg = cfgm.DSPConfig.from_dict(d)
    tau = L.us(500.0)
    wf = L.synth.generate_host(200, first_event=999)
    W = L.RDWaveforms(wf)
    pf = {"trap": {"rt": L.us(6.0), "ft": L.us(2.0)}}
    tab = L.dsp_sg_optimization(W, cfg, tau, pf, handle=handle)
    assert tuple(tab.keys()) == ("aoe", "energy", "blmean", "blslope", "t50", "qc_label")
    wls = L.grid_values(cfg.a_grid_wl_sg)
    assert tab["aoe"].shape == (200, len(wls)) and (tab["qc_label"] == -1).all()
    # oracle: the energy variant + every window length, and the aux columns
    sgv = L.sg_sweep_variants(cfg, wls, n_samples=8192, t_first=L.ns(0.0), step=L.ns(16.0), builders=O.OracleBuilders())
    ev = L.trap_sweep_variants([L.us(6.0)], [L.us(2.0)], L.ns(16.0), mode="ft")
    allv = L.SweepVariants(1 + len(wls))
    allv.array[0] = ev.array[0]
    for i in range(len(wls)):
        allv.array[1 + i] = sgv.array[i]
    allv._keep = sgv._keep
    ref, aux = _oracle(L, O, cfg, tau, wf, allv, want_aux=True)
    assert np.allclose(tab["energy"], ref[:, 0], rtol=1e-9, atol=1e-7)
    assert np.array_equal(tab["blmean"], aux[:, 0])
    assert np.allclose(tab["blslope"], aux[:, 1], rtol=1e-9, atol=1e-15)
    assert np.allclose(tab["t50"], aux[:, 2], rtol=0, atol=1e-7)
    # aoe is the window-length variants' current maximum over the energy; every current maximum equals the oracle's within
    # its error bound or is an argmax tie, sample by sample (tests/test_gpu_sweeps_random.py)
    from legenddsp.jl_b200.dsp_filter_optimization import _run_general
    from test_gpu_sweeps_random import check_sg, event_scales
    sgl = L.sg_sweep_variants(cfg, wls, n_samples=8192, t_first=L.ns(0.0), step=L.ns(16.0))
    raw = _run_general(W, cfg, tau, sgl, f64=True, handle=handle)
    with np.errstate(divide="ignore", invalid="ignore"):
        assert np.array_equal(tab["aoe"], raw / tab["energy"][:, None], equal_nan=True)
    scales = event_scales(O, L.resolve_sweep_params(cfg, tau, builders=O.OracleBuilders(), out_f64=True), wf)
    for i in range(len(wls)):
        check_sg(O, scales, raw[:, i], ref[:, 1 + i], sgl.array[i], sgv.array[i], ("wl", i))
    # the first window length equals the chain's a_sg when the same window length is the default
    P = L.resolve_icpc_params(cfg, tau, {"sg": {"wl": wls[2]}}, builders=O.OracleBuilders())
    rows = L.dsp_icpc_rows(wf, P, handle=handle)
    cur = tab["aoe"][:, 2] * tab["energy"]
    ok = np.isfinite(cur)
    assert np.allclose(cur[ok], rows[ok, L.COL["a_sg"]], rtol=1e-8, atol=1e-7)


def test_general_sweep_errors_and_empty(L, O, handle):
    cfg = L.example_config()
    S = L.resolve_sweep_params(cfg, L.us(500.0), out_f64=True)
    wf = L.synth.generate_host(4)
    v = L.SweepVariants(1)
    v.array[0].kind = 7
    out = np.zeros((4, 1))
    with pytest.raises(L.LgdspError):
        handle.gsweep_run_host(S, wf.ctypes.data, 4, 8192, v.array, out.ctypes.data)
    v.array[0].kind = 1      # FIR without coefficients
    with pytest.raises(L.LgdspError):
        handle.gsweep_run_host(S, wf.ctypes.data, 4, 8192, v.array, out.ctypes.data)
    ok = L.trap_sweep_variants([L.us(4.0)], [L.us(2.0)], L.ns(16.0), mode="ft")
    handle.gsweep_run_host(S, wf.ctypes.data, 0, 8192, ok.array, out.ctypes.data)   # empty table in, nothing written
    assert (out == 0).all()


def test_dsp_puls_and_decay_times(L, O, handle):
    """dsp_puls (src/dsp_puls.jl:29-66: no pole-zero correction, t50 with the default 1000 ns mintot, e_10410) and
    dsp_decay_times (src/dsp_decaytime.jl:11-26) are subsets of the chain served by the same kernel"""
    n = 256
    wf = L.synth.generate_host(n, first_event=31337)
    data = {"waveform": L.RDWaveforms(wf, L.ns(0.0), L.ns(16.0)), "baseline": np.arange(n, dtype=np.float32),
            "timestamp": np.arange(n, dtype=np.uint64), "eventnumber": np.arange(n, dtype=np.uint32),
            "daqenergy": np.arange(n, dtype=np.uint16)}
    tab = L.dsp_puls(data, L.example_config(), handle=handle)
    assert tuple(tab.keys()) == L.PULS_COLUMNS
    P = L.resolve_puls_params(L.example_config(), builders=O.OracleBuilders())
    assert P.pz_km1 == 0.0 and P.tx_min_n == 62       # round(1000/16 = 62.5) ties to even
    ref, _ = O.dsp_icpc(P, wf)
    for name, tol in (("blmean", 0), ("blsigma", 1e-9), ("blslope", 1e-15), ("bloffset", 1e-8), ("t50", 1e-7), ("e_max", 0),
                      ("e_10410", 1e-7)):
        a, b = tab[name], ref[:, L.COL[name]]
        assert np.all(np.abs(a - b) <= tol + 1e-9 * np.abs(b)), name
    assert np.array_equal(tab["blfc"], data["baseline"]) and np.array_equal(tab["e_fc"], data["daqenergy"])
    # without pole-zero correction e_10410 sits below the PZ-corrected one for real pulses
    Pz = L.resolve_icpc_params(L.example_config(), L.us(500.0), builders=O.OracleBuilders())
    full = L.dsp_icpc_rows(wf, Pz, handle=handle)
    big = full[:, L.COL["e_max"]] > 1000
    assert (tab["e_10410"][big] < full[big, L.COL["e_10410"]]).mean() > 0.9
    # decay times in us, both call forms
    tau = L.dsp_decay_times(L.RDWaveforms(wf), L.example_config(), handle=handle)
    cfg = L.example_config()
    tau2 = L.dsp_decay_times(L.RDWaveforms(wf), cfg.bl_window, cfg.tail_window, handle=handle)
    assert np.array_equal(tau, tau2)
    ref_full, _ = O.dsp_icpc(Pz, wf)            # (the pulser parameter block carries a placeholder tail window)
    ref_tau = ref_full[:, L.COL["tail_tau"]] * 1e-3
    inv = lambda t: np.where(t == 0, 0.0, 1.0 / np.where(t == 0, 1.0, t))
    assert np.allclose(inv(tau), inv(ref_tau), rtol=1e-7, atol=1e-10)
    good = (full[:, L.COL["e_max"]] > 5000) & (full[:, L.COL["n_sat_high"]] == 0) & (full[:, L.COL["inTrace_n"]] == 1)
    assert abs(np.median(tau[good]) - 500.0) < 5.0       # the generator's decay constant


def test_qc_and_qdrift_flt_optimization(L, O, handle):
    """dsp_qc_flt_optimization without a classifier (src/dsp_filter_optimization.jl:12-14, 31-70) and
    dsp_qdrift_flt_optimization (:72-90, external baseline) against the oracle"""
    cfg, tau = L.tiefree_config(), L.us(500.0)
    wf = L.synth.generate_host(300, first_event=4321)
    W = L.RDWaveforms(wf)
    tbl = L.dsp_qc_flt_optimization(W, cfg, tau, None, handle=handle)
    assert list(tbl.keys()) == ["energy", "blmean", "blslope", "t50", "qc_label"] and (tbl["qc_label"] == -1).all()
    S = L.resolve_sweep_params(cfg, tau, builders=O.OracleBuilders(), out_f64=True)
    rt, ft = cfg.default_flt_param["trap"]["rt"], cfg.default_flt_param["trap"]["ft"]
    var = L.trap_sweep_variants([rt], [ft], L.ns(16.0), mode="ft")
    ref, aux = O.sweep(S, wf, var.array, want_aux=True)
    assert np.allclose(tbl["energy"], ref[:, 0], rtol=1e-9, atol=1e-7)
    assert np.array_equal(tbl["blmean"], aux[:, 0]) and np.allclose(tbl["blslope"], aux[:, 1], rtol=1e-9, atol=1e-15)
    assert np.allclose(tbl["t50"], aux[:, 2], rtol=0, atol=1e-7)
    # Q-drift with the baseline of a previous pass (here: blmean + an offset, so that the external value matters)
    bl = tbl["blmean"] + np.linspace(-1.5, 1.5, len(wf))
    q = L.dsp_qdrift_flt_optimization(W, bl, cfg, tau, handle=handle, builders=O.OracleBuilders())
    P = L.resolve_icpc_params(cfg, tau, builders=O.OracleBuilders())
    qref, t0ref = O.qdrift_flt_optimization(P, wf, bl)
    assert np.allclose(q, qref, rtol=1e-9, atol=1e-3)
    assert (t0ref > 0).sum() > 200
    with pytest.raises(ValueError):
        L.dsp_qdrift_flt_optimization(W, bl[:-1], cfg, tau, handle=handle)


def test_compressed_entry_points_of_the_subset_chains(L, O, handle):
    """dsp_puls_compressed (src/dsp_puls.jl:98-134), dsp_sipm_compressed (src/dsp_sipm.jl:207-318) and
    dsp_qc_flt_optimization_compressed without a classifier (src/dsp_filter_optimization.jl:26-28) differ from their
    plain counterparts only in the input column / decode_data: same kernels on the decoded samples"""
    from test_gpu_sipm import sipm_population
    n = 128
    wf = L.synth.generate_host(n, first_event=777)
    # presummed waveform (rate 4) stored as 32-bit sums divided back to the ADC scale: 2048 samples of 64 ns
    pre = (wf.astype(np.uint32).reshape(n, -1, 4).sum(axis=2) // 4).astype(np.uint32)
    step = L.ns(64.0)
    data = {"waveform_presummed": L.RDWaveforms(pre, L.ns(0.0), step), "baseline": np.zeros(n, np.float32),
            "timestamp": np.arange(n, dtype=np.uint64), "eventnumber": np.arange(n, dtype=np.uint32),
            "daqenergy": np.zeros(n, np.uint16)}
    tab = L.dsp_puls_compressed(data, L.example_config(), handle=handle)
    assert tuple(tab.keys()) == L.PULS_COLUMNS
    P = L.resolve_puls_params(L.example_config(), n_samples=2048, step=step, builders=O.OracleBuilders())
    ref, _ = O.dsp_icpc(P, pre.astype(np.uint16))
    for name, tol in (("blmean", 0), ("blsigma", 1e-9), ("blslope", 1e-15), ("bloffset", 1e-8), ("t50", 1e-7), ("e_max", 0),
                      ("e_10410", 1e-7)):
        a, b = tab[name], ref[:, L.COL[name]]
        assert np.all(np.abs(a - b) <= tol + 1e-9 * np.abs(b)), name
    # the same samples as uint16 go through the 16-bit instantiation: identical table
    data16 = dict(data, waveform_presummed=L.RDWaveforms(pre.astype(np.uint16), L.ns(0.0), step))
    tab16 = L.dsp_puls_compressed(data16, L.example_config(), handle=handle)
    assert all(np.array_equal(tab[k], tab16[k]) for k in tab)
    # true 32-bit sums (values above 65535): every linear column scales by the presum rate
    data32 = dict(data, waveform_presummed=L.RDWaveforms(pre * 4, L.ns(0.0), step))
    tab32 = L.dsp_puls_compressed(data32, L.example_config(), handle=handle)
    assert int((pre * 4).max()) > 65535
    for name in ("blmean", "blsigma", "e_max", "e_10410"):
        assert np.allclose(tab32[name], 4.0 * tab[name], rtol=1e-12, atol=1e-9), name
    assert np.allclose(tab32["t50"], tab["t50"], rtol=0, atol=1e-9)

    # dsp_sipm_compressed == dsp_sipm on the decoded bit-drop waveform
    swf = sipm_population(32, seed=5)
    cfg = L.example_sipm_config()
    cfg["filters"]["sg"].update(min_threshold=-3.0, max_threshold=3.0, min_dc_threshold=-40.0, max_dc_threshold=40.0)
    cfg["filters"]["trap"].update(min_threshold=-15.0, max_threshold=15.0, min_dc_threshold=-30.0, max_dc_threshold=30.0)
    po = {"sg": {"wl": L.ns(200.0)}}
    common = {"baseline": np.zeros(32, np.float32), "timestamp": np.zeros(32, np.uint64),
              "eventnumber": np.arange(32, dtype=np.uint32), "daqenergy": np.zeros(32, np.uint16)}
    a = L.dsp_sipm(dict(common, waveform=L.RDWaveforms(swf)), cfg, po, handle=handle)
    b = L.dsp_sipm_compressed(dict(common, waveform_bit_drop=L.RDWaveforms(swf)), cfg, po, handle=handle)
    assert list(a.keys()) == list(b.keys())
    for k in a:
        if isinstance(a[k], L.VectorOfVectors):
            assert np.array_equal(a[k].data, b[k].data) and np.array_equal(a[k].elem_ptr, b[k].elem_ptr), k
        else:
            assert np.array_equal(a[k], b[k]), k

    # dsp_qc_flt_optimization_compressed(wvfs, config, tau, missing) == dsp_qc_flt_optimization(...)
    W = L.RDWaveforms(wf)
    q1 = L.dsp_qc_flt_optimization(W, L.example_config(), L.us(500.0), handle=handle)
    q2 = L.dsp_qc_flt_optimization_compressed(W, L.example_config(), L.us(500.0), handle=handle)
    assert all(np.array_equal(q1[k], q2[k], equal_nan=True) for k in q1)


@pytest.mark.parametrize("presum", [8, 2, 1])
def test_sg_optimization_compressed(L, O, handle, presum):
    """dsp_sg_optimization_compressed (src/dsp_filter_optimization.jl:460-511) through lgdsp_sweep_run_ext (32-bit presummed
    samples; windowed waveform with the external baseline blmean / presum_rate) against the oracle's restatement"""
    from test_gpu_compressed import _data
    cfg = L.tiefree_config()
    tau = L.us(500.0)
    n = 192
    data = _data(L, n, 4000, presum)
    wp, ww = data["waveform_presummed"], data["waveform_windowed"]
    assert wp.signal.dtype == (np.uint32 if presum > 1 else np.uint16)
    pf = {"trap": {"rt": L.us(6.0), "ft": L.us(2.0)}}
    tab = L.dsp_sg_optimization_compressed(ww, wp, cfg, tau, pf, presum_rate=float(presum), handle=handle)
    assert list(tab.keys()) == ["aoe", "energy", "blmean", "blslope", "t50", "qc_label"] and (tab["qc_label"] == -1).all()
    wls = L.grid_values(cfg.a_grid_wl_sg)
    assert tab["aoe"].shape == (n, len(wls))
    B = O.OracleBuilders()
    S_pre = L.resolve_sweep_params(cfg, tau, n_samples=wp.signal.shape[1], t_first=wp.t_first, step=wp.step, builders=B, out_f64=True)
    S_wdw = L.resolve_sweep_params(cfg, tau, n_samples=ww.signal.shape[1], t_first=ww.t_first, step=ww.step, builders=B, out_f64=True,
                                   external_baseline=True)
    ev = L.trap_sweep_variants([pf["trap"]["rt"]], [pf["trap"]["ft"]], wp.step, mode="ft")
    sgv = L.sg_sweep_variants(cfg, wls, n_samples=ww.signal.shape[1], t_first=ww.t_first, step=ww.step, builders=B)
    ref = O.dsp_sg_optimization_compressed(S_pre, S_wdw, wp.signal, ww.signal, ev.array, sgv.array, presum)
    assert np.array_equal(tab["blmean"], ref["blmean"])
    assert np.allclose(tab["blslope"], ref["blslope"], rtol=1e-9, atol=1e-15)
    assert np.allclose(tab["t50"], ref["t50"], rtol=0, atol=1e-7)
    assert np.allclose(tab["energy"], ref["energy"], rtol=1e-9, atol=1e-6, equal_nan=True)
    ok = np.abs(ref["energy"]) > 50.0 * presum            # (events with a pulse)
    assert ok.sum() > n // 2
    # the current maxima on the windowed waveform, shifted by blmean / presum_rate: each equals the oracle's within its error
    # bound or is an argmax tie, sample by sample (tests/test_gpu_sweeps_random.py)
    from test_gpu_sweeps_random import check_sg, event_scales
    sgl = L.sg_sweep_variants(cfg, wls, n_samples=ww.signal.shape[1], t_first=ww.t_first, step=ww.step)
    sw = np.ascontiguousarray(ww.signal)
    bl = np.ascontiguousarray(tab["blmean"] / float(presum))
    raw = np.zeros((n, len(wls)))
    handle.gsweep_run_ext_host(L.resolve_sweep_params(cfg, tau, n_samples=sw.shape[1], t_first=ww.t_first, step=ww.step,
                                                      out_f64=True, external_baseline=True),
                               sw.ctypes.data, sw.dtype.itemsize, bl.ctypes.data, n, sw.shape[1], sgl.array, raw.ctypes.data, None)
    with np.errstate(divide="ignore", invalid="ignore"):
        assert np.array_equal(tab["aoe"], raw / tab["energy"][:, None], equal_nan=True)
    raw_ref = O.sweep_ext(S_wdw, sw, sgv.array, baseline=bl)
    scales = event_scales(O, S_wdw, sw, baseline=bl)
    for i in range(len(wls)):
        check_sg(O, scales, raw[:, i], raw_ref[:, i], sgl.array[i], sgv.array[i], ("wl", i))
    if presum == 1:
        # presum_rate 1 with the full trace as "window": the compressed sweep equals dsp_sg_optimization on that trace
        wf = L.synth.generate_host(64, first_event=4000)
        W = L.RDWaveforms(wf)
        a = L.dsp_sg_optimization(W, cfg, tau, pf, handle=handle)
        b = L.dsp_sg_optimization_compressed(W, W, cfg, tau, pf, presum_rate=1.0, handle=handle)
        for k in ("energy", "blmean", "blslope", "t50"):
            assert np.array_equal(a[k], b[k], equal_nan=True), k
        assert np.array_equal(a["aoe"], b["aoe"], equal_nan=True)
    # 32-bit copies of 16-bit samples give the same sweep as the 16-bit kernel
    if presum == 1:
        S = L.resolve_sweep_params(cfg, tau, out_f64=True)
        v = L.trap_sweep_variants([L.us(4.0), L.us(8.0)], [L.us(1.0), L.us(3.0)], L.ns(16.0), mode="ft")
        o16 = np.zeros((64, 4)); o32 = np.zeros((64, 4))
        handle.gsweep_run_ext_host(S, wf.ctypes.data, 2, None, 64, 8192, v.array, o16.ctypes.data, None)
        half = np.ascontiguousarray(wf[:, :4096].astype(np.uint32))
        S4 = L.resolve_sweep_params(cfg, tau, n_samples=4096, out_f64=True)
        h16 = np.ascontiguousarray(wf[:, :4096])
        o16h = np.zeros((64, 4))
        handle.gsweep_run_ext_host(S4, h16.ctypes.data, 2, None, 64, 4096, v.array, o16h.ctypes.data, None)
        handle.gsweep_run_ext_host(S4, half.ctypes.data, 4, None, 64, 4096, v.array, o32.ctypes.data, None)
        assert np.array_equal(o16h, o32, equal_nan=True)
        with pytest.raises(L.LgdspError):       # 32-bit samples: at most 4096 per waveform
            big = np.zeros((2, 8192), np.uint32)
            handle.gsweep_run_ext_host(S, big.ctypes.data, 4, None, 2, 8192, v.array, o32.ctypes.data, None)
