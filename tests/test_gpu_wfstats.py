"""The per-waveform primitives on waveform arrays (lgdsp_wfstats_run): the reference's known-answer tests through the batched
entry point, every primitive against the oracle on synthetic ICPC, SiPM-like and degenerate populations (staged in shared
memory and read from global memory), the identities that tie the masks, the single-trace entries, the host and device
paths and the batch order together, the list capacity and the validation rules."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from test_gpu_sipm import sipm_population
from test_sipm_cpu import _signal, check_intersect_maximum_case

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
T0, DT = 8.0, 16.0


@pytest.fixture(scope="module")
def kat():
    with open(os.path.join(HERE, "golden", "kat_reference_tests.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def icpc_u16(L, handle):
    """2048 synthetic ICPC events from the device generator, with saturated, empty and pile-up events present"""
    import torch
    n_ev, n = 2048, 8192
    d = torch.zeros((n_ev, n), dtype=torch.int16, device="cuda")
    torch.cuda.synchronize()
    L.synth.generate_device(handle, d.data_ptr(), n_ev, first_event=4096)
    handle.synchronize()
    wf = d.cpu().numpy().view(np.uint16)
    span = wf.max(axis=1).astype(np.int64) - wf.min(axis=1)
    assert (wf == 65520).any(axis=1).sum() >= 10                      # over-range pulses clip at the ADC ceiling
    assert (span < 80).sum() >= 10                                   # empty traces: noise only
    y = wf.astype(np.int64)
    rise = (y[:, 64:] - y[:, :-64]) > 300                            # steep rising edges
    starts = rise[:, 1:] & ~rise[:, :-1]
    n_edges = np.array([np.sum(np.diff(np.flatnonzero(s)) > 200) + (1 if s.any() else 0) for s in starts])
    assert (n_edges >= 2).sum() >= 5                                 # in-trace pile-up
    return wf


def _params(L, n, kind, what, **kw):
    P = L.stats.wfstats_params(n, kind, what, L.ns(T0), L.ns(DT))
    P.sat_from, P.sat_until, P.ext_from, P.ext_until = 0, n - 1, 0, n - 1
    P.tail_from, P.tail_until, P.max_from, P.max_until = 0, n - 1, 0, n - 1
    P.im_min_n, P.im_max_n, P.max_triggers = 2, 20, 64
    for k, v in kw.items():
        setattr(P, k, v)
    return P


def _kind(L, a):
    return {np.dtype(np.uint16): L._abi.SAMPLE_U16, np.dtype(np.float32): L._abi.SAMPLE_F32,
            np.dtype(np.float64): L._abi.SAMPLE_F64}[a.dtype]


def _run(L, handle, wf, P, thr=None):
    wf = np.asarray(wf)
    thr = np.zeros(wf.shape[0]) if thr is None else np.ascontiguousarray(thr, dtype=np.float64)
    rows = np.zeros((wf.shape[0], L._abi.WFSTAT_NCOL))
    lists = np.zeros((wf.shape[0], 4, max(P.max_triggers, 1)))
    handle.wfstats_run_host(P, wf.ctypes.data, thr.ctypes.data, wf.shape[0], wf.strides[0] // wf.itemsize, rows.ctypes.data,
                            lists.ctypes.data)
    return rows, lists


def _sigma_close(got, ref, y):
    """a standard deviation from sums in another order: the variance E[y^2] - E[y]^2 is exact up to n*eps*E[y^2]"""
    tol = 1e-12 * max(float(np.mean(np.square(y, dtype=np.float64))), 1e-300)
    return abs(got * got - ref * ref) <= 1e-9 * ref * ref + tol or (np.isnan(got) and np.isnan(ref))


def _check_against_oracle(L, O, handle, wf, windows, thr_bounds=(-np.inf, np.inf), im=(2, 20), im_thr=None, sat=(0, 65535),
                          what=None):
    """every selected primitive, row by row, against the oracle; wf may be a strided view"""
    n_ev, n = wf.shape
    kind = _kind(L, wf)
    if what is None:
        what = L._abi.WFSTAT_ALL if kind == L._abi.SAMPLE_U16 else L._abi.WFSTAT_ALL & ~L._abi.WFSTAT_SATURATION
    (sf, su), (ef, eu), (tf, tu), (mf, mu) = windows
    P = _params(L, n, kind, what, sat_from=sf, sat_until=su, ext_from=ef, ext_until=eu, tail_from=tf, tail_until=tu,
                max_from=mf, max_until=mu, sat_low=sat[0], sat_high=sat[1], thr_min=thr_bounds[0], thr_max=thr_bounds[1],
                im_min_n=im[0], im_max_n=im[1], max_triggers=4096)
    thr = np.zeros(n_ev) if im_thr is None else np.broadcast_to(np.asarray(im_thr, dtype=np.float64), (n_ev,))
    rows, lists = _run(L, handle, wf, P, thr)
    c = L._abi.WFSTAT_COL
    A = L._abi
    for e in range(n_ev):
        y = wf[e].astype(np.float64)
        r = rows[e]
        if what & A.WFSTAT_SATURATION:
            s = O.saturation(wf[e, sf:su + 1], sat[0], sat[1])
            assert [r[c["sat_low"]], r[c["sat_high"]], r[c["sat_max_cons_low"]], r[c["sat_max_cons_high"]]] == \
                [s["low"], s["high"], s["max_cons_low"], s["max_cons_high"]], e
        if what & A.WFSTAT_EXTREMESTATS:
            s = O.extremestats(y, T0, DT, ef, eu)
            np.testing.assert_array_equal(r[[c["min"], c["max"], c["tmin"], c["tmax"]]], [s["min"], s["max"], s["tmin"], s["tmax"]])
        if what & A.WFSTAT_WVF_MAXIMUM:
            np.testing.assert_array_equal(r[c["wvf_max"]], O.get_wvf_maximum(y, mf, mu))
        if what & A.WFSTAT_TAILSTATS:
            s = O.tailstats(y, T0, DT, tf, tu)
            assert np.isclose(r[c["tail_mean"]], s["mean"], rtol=1e-9, atol=0, equal_nan=True), e
            yw = np.log(np.maximum(y[tf:tu + 1], 1e-300))
            assert _sigma_close(r[c["tail_sigma"]], s["sigma"], yw), e
            # tau = -1/slope, slope = cov(X, log y) / var(X): exact up to eps * E[X]E[Y] / var(X) (cancellation in cov)
            x = T0 + np.arange(tf, tu + 1) * DT
            vx = max(float(np.var(x)), 1e-300)
            slope_tol = 1e-12 * abs(np.mean(x)) * (abs(np.mean(yw)) + np.std(yw)) / vx
            if s["tau"] == 0.0 or np.isnan(s["tau"]):
                np.testing.assert_array_equal(r[c["tail_tau"]], s["tau"])
            else:
                assert abs(-1.0 / r[c["tail_tau"]] + 1.0 / s["tau"]) <= 1e-9 * abs(1.0 / s["tau"]) + slope_tol, e
        if what & A.WFSTAT_THRESHOLDSTATS:
            sel = y[(y >= thr_bounds[0]) & (y <= thr_bounds[1])]
            assert _sigma_close(r[c["thr_sigma"]], O.thresholdstats(y, *thr_bounds), sel if len(sel) else y), e
        if what & A.WFSTAT_THRESHOLDSTATS_MAD:
            assert r[c["thr_mad"]] == O.thresholdstats_mad(y, *thr_bounds), e
        if what & A.WFSTAT_INTERSECT_MAXIMUM:
            ref = O.intersect_maximum(y, T0, DT, thr[e], im[0], im[1], cap=4096)
            m = ref["multiplicity"]
            assert r[c["multiplicity"]] == m, e
            k = min(m, 4096)
            for f, name in enumerate(("x", "x_high", "x_tot")):
                np.testing.assert_array_equal(lists[e, f, :k], ref[name])
            assert np.allclose(lists[e, 3, :k], ref["max"], rtol=1e-13, atol=1e-13)
            assert not lists[e, :, k:].any()
    return rows


# ---- 1. known-answer tests of the reference through the batched entry point ----
def test_kat_batched(L, handle, kat):
    A, c = L._abi, L._abi.WFSTAT_COL
    k = kat["intersect_maximum"]
    cases = k["cases"]
    by_max = {}
    for cs in cases:
        by_max.setdefault(cs["max_n"], []).append(cs)
    for max_n, group in by_max.items():
        Y = np.stack([_signal(k["n"], cs) for cs in group]).astype(np.float64)
        f = L.IntersectMaximum(L.ns(k["min_n"] * k["dt"]), L.ns(max_n * k["dt"]))
        res = f(Y, k["thr"], step=L.ns(k["dt"]), handle=handle)
        for i, cs in enumerate(group):
            r = {kk: np.asarray(res[kk][i]) for kk in ("x", "x_high", "x_tot", "max")}
            r["multiplicity"] = int(res["multiplicity"][i])
            check_intersect_maximum_case(r, cs)
    empty = L.IntersectMaximum(L.ns(32.0), L.ns(1600.0))(np.zeros((3, 0)), 0.4, handle=handle)
    assert list(empty["multiplicity"]) == [0, 0, 0] and len(empty["x"].data) == 0          # :85-93
    # thresholdstats_mad cases, batched where the lengths agree
    by_len = {}
    for cs in kat["thresholdstats_mad"]["cases"]:
        by_len.setdefault((len(cs["signal"]), float(cs["min"]), float(cs["max"])), []).append(cs)
    for (n, mn, mx), group in by_len.items():
        v = L.thresholdstats_mad(np.array([cs["signal"] for cs in group], dtype=np.float64).reshape(len(group), n), mn, mx,
                                 handle=handle)
        for cs, got in zip(group, v):
            if "expect" in cs:
                assert abs(got - cs["expect"]) <= cs["atol"], cs["name"]
            else:
                assert got < cs["lt"], cs["name"]
    kt = kat["thresholdstats"]
    rng = np.random.default_rng(kt["seed"])
    sigma = 10.0 * rng.random()
    y = sigma * rng.standard_normal(kt["n"])
    got = L.thresholdstats(np.stack([y, 2 * y, y]), handle=handle)
    assert np.isclose(got[0], sigma, rtol=0.05) and np.isclose(got[0], np.std(y, ddof=1), rtol=kt["rtol_all"])
    assert got[0] == got[2] and np.isclose(got[1], 2 * got[0], rtol=1e-12)
    # extremestats (test/test_stats.jl:12-30): the three windows of one trace in one batch of three rows
    ke = kat["extremestats"]
    y = np.array(ke["signal"], dtype=np.float64)
    for cs in ke["cases"]:
        P = _params(L, len(y), A.SAMPLE_F64, A.WFSTAT_EXTREMESTATS, ext_from=cs["from"], ext_until=cs["until"], t_first_ns=ke["t0"],
                    dt_ns=ke["dt"])
        rows, _ = _run(L, handle, np.stack([y, y, y]), P)
        for r in rows:
            assert (r[c["min"]], r[c["max"]], r[c["tmin"]], r[c["tmax"]]) == (cs["min"], cs["max"], cs["tmin"], cs["tmax"])
        w = L.RDWaveforms(np.stack([y, y]), L.ns(ke["t0"]), L.ns(ke["dt"]))
        mn, mx, tmin, tmax = L.extremestats(w, L.ns(ke["t0"] + cs["from"] * ke["dt"]), L.ns(ke["t0"] + cs["until"] * ke["dt"]),
                                            handle=handle)
        assert list(tmin) == [cs["tmin"]] * 2 and list(tmax) == [cs["tmax"]] * 2 and list(mx) == [cs["max"]] * 2
    # get_wvf_maximum (test/test_interpolation.jl:6-45): the cases share n, one batch per window
    for cs in kat["get_wvf_maximum"]["cases"]:
        yy = _signal(cs["n"], cs)
        got = L.get_wvf_maximum(np.stack([yy, yy]), L.ns(cs["from"] * 16.0), L.ns(cs["until"] * 16.0), handle=handle)
        assert (got == cs["exact"]).all() and ((cs["ge"] <= got) & (got < cs["lt"])).all(), cs["name"]


# ---- 2. against the oracle, each primitive on its own ----
def test_icpc_population_u16(L, O, handle, icpc_u16):
    wf = icpc_u16[:256]
    bl = wf[:, :2000].mean(axis=1)
    for bit in (0x01, 0x02, 0x04, 0x08, 0x10, 0x20, 0x40):
        _check_against_oracle(L, O, handle, wf, ((0, 8191), (100, 8000), (5000, 8191), (2900, 3400)), thr_bounds=(8000.0, 16000.0),
                              im=(3, 40), im_thr=bl + 0.5 * (wf.max(axis=1) - bl), sat=(0, 65520), what=bit)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_icpc_population_baseline_subtracted(L, O, handle, icpc_u16, dtype):
    wf = icpc_u16[256:512].astype(np.float64)
    wf = (wf - wf[:, :2000].mean(axis=1, keepdims=True)).astype(dtype)
    amp = wf.max(axis=1)
    for bit in (0x02, 0x04, 0x08, 0x10, 0x20, 0x40):
        _check_against_oracle(L, O, handle, wf, ((0, 8191), (0, 8191), (4000, 8191), (2800, 3600)), thr_bounds=(-20.0, 20.0),
                              im=(2, 30), im_thr=np.maximum(0.3 * amp, 10.0), what=bit)


def test_sipm_population(L, O, handle):
    wf = sipm_population(96, n=6250, seed=11)
    y = wf.astype(np.float64)
    for bit in (0x01, 0x02, 0x04, 0x08, 0x10, 0x20, 0x40):
        _check_against_oracle(L, O, handle, wf, ((0, 6249), (2900, 3400), (10, 6000), (0, 6249)), thr_bounds=(1990.0, 2010.0),
                              im=(2, 10), im_thr=np.median(y, axis=1) + 12.0, sat=(2000, 1990), what=bit)
    yf = (y - 2000.0)
    for bit in (0x10, 0x20, 0x40):
        _check_against_oracle(L, O, handle, yf, ((0, 6249),) * 4, thr_bounds=(-6.0, 6.0), im=(3, 12), im_thr=8.0, what=bit)


def test_degenerate_traces(L, O, handle):
    rng = np.random.default_rng(3)
    n = 500
    wf = np.stack([np.full(n, 1234, np.uint16), np.zeros(n, np.uint16), np.full(n, 65535, np.uint16),
                   rng.integers(0, 3, n).astype(np.uint16),                                  # heavy ties
                   np.tile(np.array([0, 0, 65535, 65535, 65535, 7, 0], np.uint16), 72)[:n],   # alternating saturation runs
                   np.concatenate([np.full(250, 65535, np.uint16), np.zeros(250, np.uint16)])])
    for bit in (0x01, 0x02, 0x04, 0x08, 0x10, 0x20, 0x40):
        _check_against_oracle(L, O, handle, wf, ((0, n - 1), (0, n - 1), (0, n - 1), (0, n - 1)), thr_bounds=(-np.inf, np.inf),
                              im=(1, 3), im_thr=1.0, what=bit)
    # 768 = 256 chunks of 3 samples: the longest run is the trailing run of the last thread's chunk, and that chunk also
    # holds another sample
    tail = np.zeros((2, 768), np.uint16)
    tail[0, -2:] = 65535
    tail[0, 100:700:7] = 65535
    tail[1, -2:] = 5
    tail[1, 1:600:3] = 5
    for bit in (0x01, 0x02, 0x08):
        _check_against_oracle(L, O, handle, tail, ((0, 767),) * 4, im_thr=1.0, sat=(5, 65535), what=bit)
    one = np.array([[7], [0], [65535]], np.uint16)
    for bit in (0x01, 0x02, 0x04, 0x08, 0x10, 0x20, 0x40):
        _check_against_oracle(L, O, handle, one, ((0, 0),) * 4, im=(1, 1), im_thr=1.0, what=bit)


def test_strided_rows_and_windows_at_the_ends(L, O, handle, icpc_u16):
    big = np.zeros((64, 8192 + 40), np.uint16)
    big[:, :8192] = icpc_u16[512:576]
    wf = big[:, :8192]                                # ld_samples = 8232 > n_samples
    assert not wf.flags.c_contiguous
    for win in ((0, 2), (8189, 8191), (0, 8191), (4095, 4096)):
        _check_against_oracle(L, O, handle, wf, (win,) * 4, thr_bounds=(0.0, 70000.0), im=(2, 5), sat=(0, 65520),
                              im_thr=wf.mean(axis=1) + 100.0)


@pytest.mark.parametrize("n", [8192, 20000])
def test_staged_and_global_paths(L, O, handle, n):
    """8192 samples are staged in shared memory, 20000 are read from global memory (thresholdstats_mad on uint16 / float32
    through the CTA's converted copy)"""
    rng = np.random.default_rng(n)
    n_ev = 48
    y = rng.normal(0, 3.0, (n_ev, n)) + 500.0
    for e in range(n_ev):
        for _ in range(int(rng.integers(0, 12))):
            a = int(rng.integers(0, n - 100))
            y[e, a:a + int(rng.integers(5, 90))] += rng.uniform(20, 300)
    y[::7, :: 5] = 65535.0
    wins = ((0, n - 1), (10, n - 20), (n // 2, n - 1), (100, n - 100))
    u16 = np.clip(np.rint(y), 0, 65535).astype(np.uint16)
    for arr in (u16, u16.astype(np.float32), u16.astype(np.float64) - 500.0):
        _check_against_oracle(L, O, handle, arr, wins, thr_bounds=(-50.0, 550.0), im=(3, 30), im_thr=float(np.median(arr)) + 15.0)


# ---- 3. identities ----
def test_every_mask_is_the_union_of_single_bits(L, handle, icpc_u16):
    wf = icpc_u16[:40]
    n = wf.shape[1]
    thr = wf.mean(axis=1) + 50.0
    kw = dict(sat_low=0, sat_high=65520, sat_from=10, sat_until=n - 1, ext_from=5, ext_until=8000, tail_from=4000, tail_until=n - 1, max_from=2900,
              max_until=3500, thr_min=8000.0, thr_max=16000.0, im_min_n=3, im_max_n=25, max_triggers=32)
    single = {}
    for b in range(7):
        single[1 << b] = _run(L, handle, wf, _params(L, n, L._abi.SAMPLE_U16, 1 << b, **kw), thr)
    for what in range(1, 128):
        rows, lists = _run(L, handle, wf, _params(L, n, L._abi.SAMPLE_U16, what, **kw), thr)
        expect = sum(single[1 << b][0] for b in range(7) if what & (1 << b))
        assert np.array_equal(rows.view(np.int64), expect.view(np.int64)), what
        if what & 0x40:
            assert np.array_equal(lists, single[0x40][1]), what


def test_batch_rows_equal_the_single_trace_entries(L, handle):
    rng = np.random.default_rng(5)
    Y = rng.normal(0, 1, (24, 3001))
    Y[:, 100:140] += 4.0
    Y[::3, 2000:2003] += 9.0
    P = _params(L, 3001, L._abi.SAMPLE_F64, 0x70, thr_min=-1.5, thr_max=2.5, im_min_n=2, im_max_n=9, max_triggers=64)
    thr = rng.uniform(1.0, 2.5, 24)
    rows, lists = _run(L, handle, Y, P, thr)
    c = L._abi.WFSTAT_COL
    for e in range(24):
        assert rows[e, c["thr_sigma"]] == handle.thresholdstats(Y[e], -1.5, 2.5, mad=False)
        assert rows[e, c["thr_mad"]] == handle.thresholdstats(Y[e], -1.5, 2.5, mad=True)
        r = handle.intersect_maximum(Y[e], T0, DT, thr[e], 2, 9, 64)
        m = r["multiplicity"]
        assert rows[e, c["multiplicity"]] == m
        for f, name in enumerate(("x", "x_high", "x_tot", "max")):
            assert np.array_equal(lists[e, f, :min(m, 64)], r[name])


def test_host_paths_equal_the_device_path(L, handle):
    """pageable and page-locked host memory, more events than one chunk, against the device entry"""
    import torch
    n_ev, n, cap = 20000, 2000, 16
    wf = sipm_population(200, n=n, seed=9)
    wf = np.tile(wf, (n_ev // 200, 1))
    wf[::13] = 0
    rng = np.random.default_rng(1)
    thr = np.median(wf, axis=1).astype(np.float64) + rng.uniform(5.0, 20.0, n_ev)
    P = _params(L, n, L._abi.SAMPLE_U16, L._abi.WFSTAT_ALL, sat_low=0, sat_high=2000, thr_min=1990.0, thr_max=2010.0,
                tail_from=500, im_min_n=2, im_max_n=12, max_triggers=cap)
    rows_p, lists_p = _run(L, handle, wf, P, thr)                               # pageable
    pin_wf = torch.from_numpy(wf.view(np.int16)).pin_memory()
    pin_thr = torch.from_numpy(thr).pin_memory()
    pin_rows = torch.zeros((n_ev, L._abi.WFSTAT_NCOL), dtype=torch.float64).pin_memory()
    pin_lists = torch.zeros((n_ev, 4, cap), dtype=torch.float64).pin_memory()
    handle.wfstats_run_host(P, pin_wf.data_ptr(), pin_thr.data_ptr(), n_ev, n, pin_rows.data_ptr(), pin_lists.data_ptr())
    d_wf, d_thr = pin_wf.cuda(), pin_thr.cuda()
    d_rows = torch.zeros((n_ev, L._abi.WFSTAT_NCOL), dtype=torch.float64, device="cuda")
    d_lists = torch.zeros((n_ev, 4, cap), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    handle.wfstats_run_device(P, d_wf.data_ptr(), d_thr.data_ptr(), n_ev, n, d_rows.data_ptr(), d_lists.data_ptr())
    handle.synchronize()
    rows_d, lists_d = d_rows.cpu().numpy(), d_lists.cpu().numpy()
    for r, l in ((rows_p, lists_p), (pin_rows.numpy(), pin_lists.numpy())):
        assert np.array_equal(r.view(np.int64), rows_d.view(np.int64))
        assert np.array_equal(l.view(np.int64), lists_d.view(np.int64))
    assert (rows_d[:, L._abi.WFSTAT_COL["multiplicity"]] > 0).sum() > n_ev // 2


def test_permuted_batch_gives_permuted_rows(L, handle, icpc_u16):
    rng = np.random.default_rng(2)
    wf = np.tile(icpc_u16[:300], (4, 1))                                        # 1200 events > resident CTAs
    perm = rng.permutation(len(wf))
    thr = wf.mean(axis=1) + 40.0
    P = _params(L, 8192, L._abi.SAMPLE_U16, L._abi.WFSTAT_ALL, sat_high=65520, thr_min=8000.0, thr_max=16000.0, tail_from=5000, max_from=2900,
                max_until=3500, im_min_n=3, im_max_n=30, max_triggers=48)
    r1, l1 = _run(L, handle, wf, P, thr)
    r2, l2 = _run(L, handle, np.ascontiguousarray(wf[perm]), P, thr[perm])
    assert np.array_equal(r1[perm].view(np.int64), r2.view(np.int64)) and np.array_equal(l1[perm], l2)
    assert np.array_equal(r1[:300].view(np.int64), r1[300:600].view(np.int64))


# ---- 4. capacity ----
def test_capacity(L, O, handle):
    y = np.tile(np.array([0.0, 0.0, 3.0, 3.0, 3.0, 0.0]), 100)
    Y = np.stack([y, np.concatenate([y[:300], np.zeros(300)]), np.zeros(600)])
    P = _params(L, 600, L._abi.SAMPLE_F64, L._abi.WFSTAT_INTERSECT_MAXIMUM, im_min_n=2, im_max_n=5, max_triggers=7)
    rows, lists = _run(L, handle, Y, P, np.ones(3))
    c = L._abi.WFSTAT_COL["multiplicity"]
    assert list(rows[:, c]) == [100, 50, 0]
    ref = O.intersect_maximum(y, T0, DT, 1.0, 2, 5, cap=1024)
    assert np.array_equal(lists[0, 0], ref["x"][:7]) and np.array_equal(lists[0, 1], ref["x_high"][:7])
    assert not lists[2].any()
    res = L.IntersectMaximum(L.ns(2 * DT), L.ns(5 * DT))(Y, 1.0, t_first=L.ns(T0), step=L.ns(DT), handle=handle, max_triggers=7)
    assert list(res["multiplicity"]) == [100, 50, 0]
    assert np.array_equal(res["x"][0], ref["x"]) and np.array_equal(res["x_high"][0], ref["x_high"])
    assert np.array_equal(res["x"][1], ref["x"][:50]) and len(res["x"][2]) == 0


# ---- 5. validation: documented codes, nothing launched ----
def test_validation(L, handle):
    A = L._abi
    lib = handle._lib
    wf = np.zeros((4, 100), np.uint16)
    thr = np.zeros(4)
    rows = np.zeros((4, A.WFSTAT_NCOL))
    lists = np.zeros((4, 4, 8))

    def call(P, wf_p=wf.ctypes.data, thr_p=thr.ctypes.data, n_ev=4, ld=100, lists_p=lists.ctypes.data):
        before = handle.launch_count
        rc = lib.lgdsp_wfstats_run(handle._h, C.byref(P), C.c_void_p(wf_p) if wf_p else None, C.c_void_p(thr_p) if thr_p else None,
                                   n_ev, ld, C.c_void_p(rows.ctypes.data), C.c_void_p(lists_p) if lists_p else None)
        assert handle.launch_count == before or rc == 0
        return rc

    def P(what=A.WFSTAT_ALL, **kw):
        return _params(L, 100, A.SAMPLE_U16, what, **dict(dict(max_triggers=8), **kw))
    assert call(P()) == 0
    inv, uns = A.LGDSP_ERR_INVALID_ARG, A.LGDSP_ERR_UNSUPPORTED
    assert call(P(struct_size=8)) == inv
    assert call(P(version=A.LGDSP_PARAMS_VERSION + 1)) == inv
    assert call(P(what=0)) == inv
    assert call(P(what=0x80)) == inv
    assert call(P(sample_kind=3)) == uns
    assert call(P(sample_kind=A.SAMPLE_F32)) == uns                                   # saturation needs raw UInt16
    wf32 = np.zeros((4, 100), np.float32)
    assert call(P(sample_kind=A.SAMPLE_F32, what=A.WFSTAT_ALL & ~A.WFSTAT_SATURATION), wf_p=wf32.ctypes.data) == 0
    assert call(P(n_samples=-1)) == uns
    assert call(P(n_samples=65537)) == uns
    for f in ("sat", "ext", "tail", "max"):
        for a, b in ((-1, 10), (5, 4), (0, 100)):
            assert call(P(**{f + "_from": a, f + "_until": b})) == inv, (f, a, b)
        bit = {"sat": 0x01, "ext": 0x02, "tail": 0x04, "max": 0x08}[f]
        assert call(P(what=A.WFSTAT_ALL & ~bit, **{f + "_from": 5, f + "_until": 4})) == 0   # unselected: not checked
    assert call(P(im_min_n=0)) == inv
    assert call(P(im_max_n=0)) == inv
    assert call(P(max_triggers=0)) == inv
    assert call(P(max_triggers=65537)) == inv
    assert call(P(), thr_p=None) == inv
    assert call(P(what=0x3F), thr_p=None, lists_p=None) == 0
    assert call(P(), ld=99) == inv
    assert call(P(), wf_p=None) == inv
    before = handle.launch_count
    assert call(P(), n_ev=0) == 0 and handle.launch_count == before
