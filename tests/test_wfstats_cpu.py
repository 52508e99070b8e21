"""The per-waveform primitives on waveform arrays without a GPU: the ctypes mirror of lgdsp_wfstats_params against the header,
window resolution, sample-type handling, and that the compute calls fail loudly (no CPU fallback)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("struct_size", "version", "n_samples", "sample_kind", "what", "reserved0", "t_first_ns", "dt_ns", "sat_from", "sat_until",
          "ext_from", "ext_until", "tail_from", "tail_until", "max_from", "max_until", "sat_low", "sat_high", "thr_min", "thr_max",
          "im_min_n", "im_max_n", "max_triggers", "reserved1")


def _c_layout():
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "lgdsp_b200.h"', 'int main(void) {',
             'printf("sizeof %zu\\n", sizeof(lgdsp_wfstats_params));']
    lines += ['printf("%s %%zu\\n", offsetof(lgdsp_wfstats_params, %s));' % (f, f) for f in FIELDS]
    lines += ['printf("ncol %d\\n", (int)LGDSP_WFSTAT_NCOL);', 'printf("f64 %d\\n", LGDSP_SAMPLE_F64);',
              'printf("all %u\\n", LGDSP_WFSTAT_ALL);', 'printf("col_mult %d\\n", (int)LGDSP_WFSTAT_multiplicity);',
              'printf("col_wvf %d\\n", (int)LGDSP_WFSTAT_wvf_max);', 'return 0; }']
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "w.c"), os.path.join(d, "w")
        open(src, "w").write("\n".join(lines) + "\n")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.run([cc, "-I", os.path.join(ROOT, "include"), src, "-o", exe], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    return dict((l.split()[0], int(l.split()[1])) for l in out.strip().splitlines())


def test_wfstats_params_mirror_matches_header(L):
    c = _c_layout()
    A = L._abi
    assert C.sizeof(A.WfstatsParams) == c["sizeof"]
    assert [f for f, _ in A.WfstatsParams._fields_] == list(FIELDS)
    for f in FIELDS:
        assert getattr(A.WfstatsParams, f).offset == c[f], f
    assert c["ncol"] == A.WFSTAT_NCOL == len(A.WFSTAT_COLUMNS)
    assert c["f64"] == A.SAMPLE_F64 and c["all"] == A.WFSTAT_ALL
    assert c["col_mult"] == A.WFSTAT_COL["multiplicity"] and c["col_wvf"] == A.WFSTAT_COL["wvf_max"]


def test_window_resolution(L):
    w = L.stats.window
    assert w(None, None, 100, L.ns(0.0), L.ns(16.0)) == (0, 99)
    assert w(L.ns(32.0), L.ns(160.0), 100, L.ns(0.0), L.ns(16.0)) == (2, 10)
    # round(Int, x) is ties-to-even: 24/16 = 1.5 -> 2, 40/16 = 2.5 -> 2, 56/16 = 3.5 -> 4
    assert w(L.ns(24.0), L.ns(40.0), 100, L.ns(0.0), L.ns(16.0)) == (2, 2)
    assert w(L.ns(56.0), None, 100, L.ns(0.0), L.ns(16.0)) == (4, 99)
    # time axis that does not start at 0, window in another unit
    assert w(L.us(1.0), L.us(2.0), 1000, L.ns(200.0), L.ns(8.0)) == (100, 225)


@pytest.mark.parametrize("start,stop", [(-16.0, 160.0), (0.0, 1600.0), (320.0, 160.0)])
def test_window_outside_the_trace_raises(L, start, stop):
    with pytest.raises(AssertionError):
        L.stats.window(L.ns(start), L.ns(stop), 100, L.ns(0.0), L.ns(16.0))
    wf = np.zeros((3, 100), np.uint16)
    with pytest.raises(AssertionError):        # resolved before any device is touched
        L.tailstats(wf, L.ns(start), L.ns(stop))
    with pytest.raises(AssertionError):
        L.get_wvf_maximum(L.RDWaveforms(wf, L.ns(0.0), L.ns(16.0)), L.ns(start), L.ns(stop))
    with pytest.raises(AssertionError):
        L.extremestats(np.zeros(0), L.ns(0.0), L.ns(0.0))


def test_sample_types(L):
    S = L.stats
    for dt, kind in ((np.uint16, L._abi.SAMPLE_U16), (np.float32, L._abi.SAMPLE_F32), (np.float64, L._abi.SAMPLE_F64)):
        a = np.arange(60, dtype=dt).reshape(3, 20)
        got, k, single = S.wf_samples(a)
        assert k == kind and not single and np.shares_memory(got, a)
        # rows of a wider buffer: no copy, the row stride becomes ld_samples
        wide = np.zeros((4, 32), dtype=dt)
        got, _, _ = S.wf_samples(wide[:, :20])
        assert np.shares_memory(got, wide) and got.strides[0] == 32 * np.dtype(dt).itemsize
    got, k, single = S.wf_samples(np.arange(7, dtype=np.float64))
    assert single and got.shape == (1, 7) and k == L._abi.SAMPLE_F64
    # other integers -> uint16 (range-checked), other floats -> float32, column-strided views -> contiguous copy
    got, k, _ = S.wf_samples(np.array([[1, 2], [65535, 0]], dtype=np.int64))
    assert got.dtype == np.uint16 and k == L._abi.SAMPLE_U16 and got.tolist() == [[1, 2], [65535, 0]]
    with pytest.raises(ValueError):
        S.wf_samples(np.array([[70000]], dtype=np.int32))
    with pytest.raises(ValueError):
        S.wf_samples(np.array([[-1]], dtype=np.int32))
    got, k, _ = S.wf_samples(np.ones((2, 3), dtype=np.float16))
    assert got.dtype == np.float32 and k == L._abi.SAMPLE_F32
    a = np.arange(40.0).reshape(4, 10)
    got, _, _ = S.wf_samples(a[:, ::2])
    assert got.flags.c_contiguous and np.array_equal(got, a[:, ::2])
    with pytest.raises(TypeError):
        S.wf_samples(np.ones((2, 2), dtype=np.complex128))
    with pytest.raises(ValueError):
        S.wf_samples(np.ones((2, 2, 2)))


def test_new_functions_fail_loudly_without_a_device(L):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    wf = np.full((4, 64), 100, np.uint16)
    calls = [lambda: L.extremestats(wf), lambda: L.saturation(wf, 0, 65535), lambda: L.tailstats(wf, L.ns(0.0), L.ns(160.0)),
             lambda: L.get_wvf_maximum(wf, L.ns(0.0), L.ns(160.0)), lambda: L.thresholdstats(wf.astype(float)),
             lambda: L.thresholdstats_mad(wf.astype(float)),
             lambda: L.IntersectMaximum(L.ns(16.0), L.ns(64.0))(wf.astype(float), 1.0)]
    for f in calls:
        with pytest.raises(L.LgdspError) as ei:
            f()
        assert ei.value.code == L._abi.LGDSP_ERR_NO_DEVICE
