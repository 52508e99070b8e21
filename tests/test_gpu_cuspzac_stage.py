"""The CUSP / ZAC stage of the split pipeline (select kernel + finish kernel, whose recurrences read prefix sums staged in
shared memory) against the fused kernel, bit for bit on the six CUSP / ZAC columns, for populations that reach every
branch of the staging: noise-only events (every chunk a candidate: the finish kernel's helper warps and their combine),
pulses at the very start and end of the trace (candidate chunks whose streams clamp at the trace ends), two structured
passes (unequal CUSP / ZAC lengths), short traces and a row stride larger than the trace."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CZ_COLS = ("e_cusp_max", "t_cusp_max", "e_cusp", "e_zac_max", "t_zac_max", "e_zac")


def _rows(L, h, wf, P, path):
    h.set_icpc_path(path, 0, 0)
    try:
        return L.dsp_icpc_rows(wf, P, handle=h)
    finally:
        h.set_icpc_path("split")


def _assert_identical(L, a, b):
    for name in CZ_COLS:
        j = L.COL[name]
        x, y = a[:, j], b[:, j]
        same = (x == y) | (np.isnan(x) & np.isnan(y))
        assert same.all(), (name, int((~same).sum()), int(np.nonzero(~same)[0][0]))


def _population(L, n, rng, first_event):
    """generator events, noise-only traces and exponential pulses whose edge sits in the first or last 40 samples"""
    gen = L.synth.generate_host(96, first_event=first_event, n_samples=n)
    i = np.arange(n)
    noise = 12000.0 + rng.normal(0.0, 3.0, (40, n))
    edges = np.r_[rng.integers(1, 40, 20), n - rng.integers(2, 40, 20)]
    amp = rng.uniform(200.0, 20000.0, 40)
    step = np.where(i[None, :] >= edges[:, None], np.exp(-(i[None, :] - edges[:, None]) / 31250.0), 0.0)
    pulses = 9000.0 + amp[:, None] * step + rng.normal(0.0, 3.0, (40, n))
    made = np.clip(np.rint(np.concatenate([noise, pulses])), 0, 65535).astype(np.uint16)
    return np.concatenate([gen, made])


def _short_config(L, n):
    """the example config with the windows and filter lengths scaled to an n-sample trace (16 ns samples)"""
    from importlib import import_module
    cfgm = import_module("legenddsp.jl_b200.config")
    d = cfgm.example_config_dict()
    us = cfgm.us
    span = n * 0.016
    d["bl_window"] = {"min": us(0.0), "max": us(0.25 * span)}
    d["current_window"] = {"min": us(0.3 * span), "max": us(0.5 * span)}
    d["tail_window"] = {"min": us(0.6 * span), "max": us(0.9 * span)}
    d["flt_length_cusp"] = d["flt_length_zac"] = us(0.06 * span)
    d["flt_defaults"]["trap"] = d["flt_defaults"]["cusp"] = d["flt_defaults"]["zac"] = {"rt": us(0.02 * span), "ft": us(0.01 * span)}
    return cfgm.DSPConfig.from_dict(d)


def test_stage_full_traces(L, O, handle):
    """8192 samples, one structured pass (equal CUSP / ZAC lengths)"""
    P = L.resolve_icpc_params(L.example_config(), L.us(500.0))
    wf = _population(L, 8192, np.random.default_rng(5), 40000)
    _assert_identical(L, _rows(L, handle, wf, P, "split"), _rows(L, handle, wf, P, "fused"))


def test_stage_two_passes(L, O, handle):
    """unequal CUSP / ZAC lengths: the select kernel runs two structured passes and the finish kernel two rounds"""
    cfg = L.example_config()
    pars = {"cusp": {"rt": L.us(3.0), "ft": L.us(1.0)}, "zac": {"rt": L.us(4.0), "ft": L.us(2.0)}}
    P = L.resolve_icpc_params(cfg, L.us(300.0), pars)
    wf = _population(L, 8192, np.random.default_rng(6), 41000)
    _assert_identical(L, _rows(L, handle, wf, P, "split"), _rows(L, handle, wf, P, "fused"))


@pytest.mark.parametrize("n", [1600, 2504, 4104, 6144])
def test_stage_short_traces_ragged_rows(L, O, handle, n):
    """short traces, read from rows of a wider array (row stride n + 37 samples)"""
    P = L.resolve_icpc_params(_short_config(L, n), L.us(500.0), n_samples=n)
    wf = _population(L, n, np.random.default_rng(n), 42000 + n)
    wide = np.zeros((wf.shape[0], n + 37), dtype=np.uint16)
    wide[:, :n] = wf
    ragged = wide[:, :n]
    assert ragged.strides[0] == 2 * (n + 37)
    split = _rows(L, handle, ragged, P, "split")
    _assert_identical(L, split, _rows(L, handle, wf, P, "fused"))
    assert np.isfinite(split[:, L.COL["e_cusp_max"]]).any()
