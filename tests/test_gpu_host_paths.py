"""Every chunked host entry point against its _device counterpart on the same inputs, bit for bit (NaN equals NaN): pageable
and page-locked input and output, strided input (ld > n), and at least three chunks with a ragged tail."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N_FIXED = 2 * 8192 + 77      # sweep, SiPM and window statistics run in chunks of 8 192 events
N_MI = 2 * 4096 + 33         # MultiIntersect: chunks of 4 096 traces
N_ICPC = 3 * 1500 + 401      # dsp_icpc / compressed on a handle with 1 500 (pageable) / 1 000 (page-locked) events per chunk


def pinned(a):
    """a page-locked copy of a numpy array"""
    import torch
    a = np.ascontiguousarray(a)
    return torch.from_numpy(a.reshape(-1).view(np.uint8)).pin_memory().numpy().view(a.dtype).reshape(a.shape)


def strided(a, pad=8):
    """the same rows `pad` samples further apart (ld = n + pad)"""
    w = np.zeros((a.shape[0], a.shape[1] + pad), a.dtype)
    w[:, :a.shape[1]] = a
    return w[:, :a.shape[1]]


def kinds(a):
    """the three forms of an input: pageable, page-locked, strided pageable"""
    return {"pageable": a, "pinned": pinned(a), "strided": strided(a)}


def ld(a):
    return a.strides[0] // a.itemsize


class Dev:
    """device copies of inputs and device outputs, read back after the handle's stream is synchronised"""

    def __init__(self, handle):
        import torch
        self.torch, self.handle, self.inputs, self.outputs = torch, handle, [], []

    def put(self, a):
        t = self.torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8)).cuda()
        self.torch.cuda.synchronize()
        self.inputs.append(t)
        return t.data_ptr()

    def out(self, shape, dtype):
        t = self.torch.empty(int(np.prod(shape)) * np.dtype(dtype).itemsize, dtype=self.torch.uint8, device="cuda")
        self.outputs.append((t, shape, dtype))
        return t.data_ptr()

    def get(self):
        self.handle.synchronize()
        return [t.cpu().numpy().view(dt).reshape(sh) for t, sh, dt in self.outputs]


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and a.dtype == b.dtype
    if a.dtype.kind == "f":
        nan = np.isnan(a)
        if not np.array_equal(nan, np.isnan(b)):
            return False
        a, b = np.where(nan, 0, a), np.where(nan, 0, b)
        it = np.int64 if a.itemsize == 8 else np.int32
        return np.array_equal(a.view(it), b.view(it))
    return np.array_equal(a, b)


def outputs(pin, *specs):
    """output arrays (shape, dtype), filled with a sentinel; page-locked when pin"""
    out = [np.full(sh, 7.25 if np.dtype(dt).kind == "f" else 77, dt) for sh, dt in specs]
    return [pinned(o) for o in out] if pin else out


def cfg4096(L):
    from importlib import import_module
    cfgm = import_module("legenddsp.jl_b200.config")
    d = cfgm.example_config_dict()
    us = cfgm.us
    d["bl_window"] = {"min": us(0.0), "max": us(19.5)}
    d["tail_window"] = {"min": us(35.0), "max": us(55.0)}
    d["current_window"] = {"min": us(21.5), "max": us(31.0)}
    d["flt_length_cusp"] = d["flt_length_zac"] = us(8.0)
    d["flt_defaults"]["trap"] = d["flt_defaults"]["cusp"] = d["flt_defaults"]["zac"] = {"rt": us(1.0), "ft": us(0.5)}
    return cfgm.DSPConfig.from_dict(d)


@pytest.fixture(scope="module")
def small_chunks(L):
    keep = {k: os.environ.get(k) for k in ("LGDSP_HOST_CHUNK", "LGDSP_HOST_CHUNK_DIRECT")}
    os.environ["LGDSP_HOST_CHUNK"], os.environ["LGDSP_HOST_CHUNK_DIRECT"] = "1500", "1000"
    try:
        h = L.Handle(0)
    finally:
        for k, v in keep.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    yield h
    h.close()


@pytest.fixture(scope="module")
def icpc_pool(L):
    wf = L.synth.generate_host(N_ICPC, first_event=52000)
    P = L.resolve_icpc_params(L.example_config(), L.us(500.0))
    P4 = L.resolve_icpc_params(cfg4096(L), L.us(500.0), n_samples=4096)
    wf4 = L.synth.generate_host(N_ICPC, first_event=9000, n_samples=4096).astype(np.uint32) * 3
    bl = 3 * 15000.0 + np.random.default_rng(3).normal(0, 30.0, N_ICPC)
    return wf, P, wf4, P4, bl


@pytest.mark.parametrize("kind", ["pageable", "pinned", "strided"])
@pytest.mark.parametrize("pin_out", [False, True])
def test_icpc_run(L, small_chunks, icpc_pool, kind, pin_out):
    h = small_chunks
    wf, P, _, _, _ = icpc_pool
    dev = Dev(h)
    h.icpc_run_device(P, dev.put(wf), len(wf), wf.shape[1], dev.out((len(wf), L.NCOL), np.float64))
    ref, = dev.get()
    src = kinds(wf)[kind]
    rows, = outputs(pin_out, ((len(wf), L.NCOL), np.float64))
    h.icpc_run_host(P, src.ctypes.data, len(wf), ld(src), rows.ctypes.data)
    assert same(rows, ref)


@pytest.mark.parametrize("kind", ["pageable", "pinned", "strided"])
def test_icpc_run_ext_wide_samples_and_baseline(L, small_chunks, icpc_pool, kind):
    h = small_chunks
    _, _, wf4, P4, bl = icpc_pool
    dev = Dev(h)
    h.icpc_run_ext_device(P4, dev.put(wf4), 4, dev.put(bl), len(wf4), wf4.shape[1], dev.out((len(wf4), L.NCOL), np.float64))
    ref, = dev.get()
    src = kinds(wf4)[kind]
    b = pinned(bl) if kind == "pinned" else bl
    rows, = outputs(kind == "pinned", ((len(wf4), L.NCOL), np.float64))
    h.icpc_run_ext_host(P4, src.ctypes.data, 4, b.ctypes.data, len(wf4), ld(src), rows.ctypes.data)
    assert same(rows, ref)


@pytest.mark.parametrize("pin", [False, True])
def test_icpc_run_encoded(L, small_chunks, icpc_pool, pin):
    h = small_chunks
    wf, P, _, _, _ = icpc_pool
    dev = Dev(h)
    h.icpc_run_device(P, dev.put(wf), len(wf), wf.shape[1], dev.out((len(wf), L.NCOL), np.float64))
    ref, = dev.get()
    enc = L.encode_waveforms(wf)
    data, off = (pinned(enc.data), pinned(enc.offsets)) if pin else (enc.data, enc.offsets)
    rows, = outputs(pin, ((len(wf), L.NCOL), np.float64))
    h.icpc_run_encoded_host(P, enc.codec, data.ctypes.data, off.ctypes.data, enc.shift, 2, None, len(wf), rows.ctypes.data)
    assert same(rows, ref)


@pytest.fixture(scope="module")
def compressed_pool(L, icpc_pool):
    wf = icpc_pool[0]
    pre, wdw = L.synth.compress(wf, 8, (2600, 1400))
    Pp, Pw, aux = L.resolve_compressed_params(L.tiefree_config(), L.us(500.0), None, presum_rate=8, n_pre=pre.shape[1],
                                              step_pre=L.ns(128.0), n_wdw=wdw.shape[1], t_first_wdw=L.ns(16.0 * 2600),
                                              step_wdw=L.ns(16.0))
    return pre, wdw, Pp, Pw, aux


def _compressed_ref(L, h, pool):
    pre, wdw, Pp, Pw, aux = pool
    n = len(pre)
    dev = Dev(h)
    h.icpc_compressed_run_device(Pp, Pw, dev.put(pre), 4, pre.shape[1], dev.put(wdw), 2, wdw.shape[1], 8.0, aux, n,
                                 dev.out((n, L.NCOL), np.float64), dev.out((n, L.NCOL), np.float64), dev.out((n, 5, 5), np.float64))
    return dev.get()


@pytest.mark.parametrize("kind", ["pageable", "pinned", "strided"])
def test_compressed_run(L, small_chunks, compressed_pool, kind):
    h = small_chunks
    pre, wdw, Pp, Pw, aux = compressed_pool
    ref = _compressed_ref(L, h, compressed_pool)
    n = len(pre)
    p, w = kinds(pre)[kind], kinds(wdw)[kind]
    got = outputs(kind == "pinned", ((n, L.NCOL), np.float64), ((n, L.NCOL), np.float64), ((n, 5, 5), np.float64))
    h.icpc_compressed_run_host(Pp, Pw, p.ctypes.data, 4, ld(p), w.ctypes.data, 2, ld(w), 8.0, aux, n, *[g.ctypes.data for g in got])
    for g, r in zip(got, ref):
        assert same(g, r)


@pytest.mark.parametrize("pin", [False, True])
def test_compressed_run_encoded(L, small_chunks, compressed_pool, pin):
    h = small_chunks
    pre, wdw, Pp, Pw, aux = compressed_pool
    ref = _compressed_ref(L, h, compressed_pool)
    n = len(pre)
    ep, ew = L.encode_waveforms(pre, L.ULEB128_ZIGZAG_DIFF), L.encode_waveforms(wdw)
    if pin:
        ep.data, ep.offsets, ew.data, ew.offsets = (pinned(x) for x in (ep.data, ep.offsets, ew.data, ew.offsets))
    got = outputs(pin, ((n, L.NCOL), np.float64), ((n, L.NCOL), np.float64), ((n, 5, 5), np.float64))
    h.icpc_compressed_run_encoded_host(Pp, Pw, ep, ew, 8.0, aux, *[g.ctypes.data for g in got])
    for g, r in zip(got, ref):
        assert same(g, r)


@pytest.fixture(scope="module")
def fixed_pool(L):
    rng = np.random.default_rng(11)
    wf = L.synth.generate_host(N_FIXED, first_event=77000, n_samples=1024)
    return wf, rng.normal(12000.0, 40.0, N_FIXED)


@pytest.mark.parametrize("kind", ["pageable", "pinned", "strided"])
def test_sweep_run_ext_baseline_and_aux(L, handle, fixed_pool, kind):
    wf, bl = fixed_pool
    n = len(wf)
    S = L.resolve_sweep_params(L.example_config(), L.us(500.0), n_samples=1024, out_f64=True, external_baseline=True)
    trap = L.trap_sweep_variants([L.us(1.0), L.us(2.0)], [L.us(0.5), L.us(1.0)], L.ns(16.0), mode="ft")
    # one FIR (CUSP, 500 taps) and one Savitzky-Golay variant (window set on the 1 024-sample trace) besides the trapezoids
    fir = L.cuspzac_sweep_variants(cfg4096(L), "cusp", [L.us(1.0)], [L.us(0.5)], L.ns(16.0), mode="ft")
    sg = L.sg_sweep_variants(cfg4096(L), [L.ns(200.0)], n_samples=4096, t_first=L.ns(0.0), step=L.ns(16.0))
    sg.array[0].win_from, sg.array[0].win_until = 300, 700
    from test_gpu_sweeps_random import concat_variants
    var = concat_variants(L, [(trap, i) for i in range(len(trap))] + [(fir, 0), (sg, 0)])
    dev = Dev(handle)
    handle.gsweep_run_ext_device(S, dev.put(wf), 2, dev.put(bl), n, 1024, var.array, dev.out((n, len(var)), np.float64),
                                 dev.out((n, 4), np.float64))
    ref, ref_aux = dev.get()
    src = kinds(wf)[kind]
    b = pinned(bl) if kind == "pinned" else bl
    out, aux = outputs(kind == "pinned", ((n, len(var)), np.float64), ((n, 4), np.float64))
    handle.gsweep_run_ext_host(S, src.ctypes.data, 2, b.ctypes.data, n, ld(src), var.array, out.ctypes.data, aux.ctypes.data)
    assert same(out, ref) and same(aux, ref_aux)


@pytest.mark.parametrize("kind", ["pageable", "pinned", "strided"])
def test_trap_sweep_run(L, handle, fixed_pool, kind):
    wf, _ = fixed_pool
    n = len(wf)
    S = L.resolve_sweep_params(L.example_config(), L.us(500.0), n_samples=1024, external_baseline=True)
    var = L.trap_variants([L.us(1.0), L.us(3.0)], [L.us(0.5)], L.ns(16.0), mode="rt", pickoff=L.us(9.0))
    dev = Dev(handle)
    handle.sweep_run_device(S, dev.put(wf), n, 1024, var, dev.out((n, len(var)), np.float32))
    ref, = dev.get()
    src = kinds(wf)[kind]
    out, = outputs(kind == "pinned", ((n, len(var)), np.float32))
    handle.sweep_run_host(S, src.ctypes.data, n, ld(src), var, out.ctypes.data)
    assert same(out, ref)


@pytest.mark.parametrize("kind", ["pageable", "pinned", "strided"])
def test_sipm_run(L, handle, kind):
    from test_gpu_sipm import sipm_population
    base = sipm_population(64, n=6250, seed=5)
    wf = np.tile(base, (N_FIXED // 64 + 1, 1))[:N_FIXED]
    wf = (wf + np.random.default_rng(6).integers(0, 3, wf.shape, dtype=np.uint16)).astype(np.uint16)
    cfg = L.example_sipm_config()
    cfg["filters"]["sg"].update(min_threshold=-3.0, max_threshold=3.0)
    P = L.resolve_sipm_params(cfg, {"sg": {"wl": L.ns(200.0)}}, n_samples=6250, max_triggers=16)
    n, A = len(wf), L._abi
    tshape = (n, A.SIPM_NLIST, A.SIPM_NFIELD, 16)
    dev = Dev(handle)
    handle.sipm_run_device(P, dev.put(wf), n, 6250, dev.out((n, A.SIPM_NCOL), np.float64), dev.out(tshape, np.float64))
    ref, ref_trig = dev.get()
    assert (ref[:, A.SIPM_COL["n_trig"]] > 0).any()
    src = kinds(wf)[kind]
    rows, trig = outputs(kind == "pinned", ((n, A.SIPM_NCOL), np.float64), (tshape, np.float64))
    handle.sipm_run_host(P, src.ctypes.data, n, ld(src), rows.ctypes.data, trig.ctypes.data)
    assert same(rows, ref) and same(trig, ref_trig)


@pytest.mark.parametrize("kind", ["pageable", "pinned", "strided"])
def test_multi_intersect_run(L, handle, kind):
    rng = np.random.default_rng(8)
    k = np.arange(1024)
    s0, rise, amp = rng.integers(200, 600, N_MI), rng.integers(10, 120, N_MI), rng.uniform(50, 5000, N_MI)
    Y = amp[:, None] * np.clip((k[None, :] - s0[:, None]) / rise[:, None], 0, 1) + rng.normal(0, 1.0, (N_MI, 1024))
    Y[::7, :40] += 3 * amp[::7, None]        # starts above the thresholds: flagged traces
    P = L.MultiIntersect(mintot=L.ns(32.0), n=2, d=2, sampling_rate=4).params(1024, L.ns(0.0), L.ns(16.0))
    n, m = len(Y), P.n_thresholds
    dev = Dev(handle)
    handle.multi_intersect_device(P, dev.put(Y), n, 1024, dev.out((n, m), np.float64), dev.out((n,), np.int32))
    ref, ref_flags = dev.get()
    src = kinds(Y)[kind]
    x, flags = outputs(kind == "pinned", ((n, m), np.float64), ((n,), np.int32))
    handle.multi_intersect_host(P, src.ctypes.data, n, ld(src), x.ctypes.data, flags.ctypes.data)
    assert same(x, ref) and same(flags, ref_flags)


@pytest.mark.parametrize("kind", ["pageable", "pinned", "strided"])
def test_window_stats_run(L, handle, fixed_pool, kind):
    wf, bl = fixed_pool
    n = len(wf)
    wins = [(0, 155), (156, 304), (547, 702), (10, 73), (0, 1023)]
    dev = Dev(handle)
    handle.window_stats_device(dev.put(wf), 2, n, 1024, 1024, 5.0, 16.0, dev.put(bl), wins, dev.out((n, len(wins), 5), np.float64))
    ref, = dev.get()
    src = kinds(wf)[kind]
    b = pinned(bl) if kind == "pinned" else bl
    out, = outputs(kind == "pinned", ((n, len(wins), 5), np.float64))
    handle.window_stats_host(src.ctypes.data, 2, n, 1024, ld(src), 5.0, 16.0, b.ctypes.data, wins, out.ctypes.data)
    assert same(out, ref)


@pytest.mark.parametrize("pin_out", [False, True])
def test_decode_data_into_strided_rows(L, handle, pin_out):
    """8 192 + 517 events of 1 400 samples decoded into rows 1 408 samples apart: the rows equal the original samples and
    the 8 padding samples of every row keep the caller's sentinel"""
    wf = L.synth.generate_host(8192 + 517, first_event=123, n_samples=1400)
    enc = L.encode_waveforms(wf)
    out, = outputs(pin_out, ((len(wf), 1408), np.uint16))
    out[:] = 0xBEEF
    handle.decode_data_host(enc.codec, enc.data.ctypes.data, enc.offsets.ctypes.data, len(wf), 1400, enc.shift, out.ctypes.data, 2, 1408)
    assert np.array_equal(out[:, :1400], wf)
    assert (out[:, 1400:] == 0xBEEF).all()
