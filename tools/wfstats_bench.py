"""Throughput of lgdsp_wfstats_run (the per-waveform primitives on waveform arrays), one JSON document.

Device entry, CUDA events around each call (lgdsp_last_kernel_ms), on a resident batch of 131 072 x 8192 synthetic ICPC
waveforms (2.1 GB as uint16, 8.6 GB as float64: every pass streams from HBM, the batch is > 16x the 126 MB L2), for every
primitive alone and all seven together, uint16 and float64 input.  Reported: waveforms/s and the algorithmic bytes (samples
+ thresholds + rows + lists) over the kernel time against the HBM bandwidth of MEASURED_PEAKS.json (data-sheet 7.7 TB/s when
that file is absent).  Then 1 000 host traces of 8192 float64 samples through the per-trace loop of the single-trace entries
(lgdsp_intersect_maximum + lgdsp_thresholdstats, one call each per trace) against one batched call on the same traces.
GPU name, power limit and SM clock are read in the same run.

    python tools/wfstats_bench.py [--events 131072] [--reps 3] [--out FILE]   (without --out the JSON goes to stdout, progress to stderr)
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PRIMS = (("saturation", 0x01), ("extremestats", 0x02), ("tailstats", 0x04), ("get_wvf_maximum", 0x08), ("thresholdstats", 0x10),
         ("thresholdstats_mad", 0x20), ("intersect_maximum", 0x40), ("all", 0x7F))


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except Exception as e:   # the numbers are still reported; the card description is then missing
        return {"error": str(e)}


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:
        return 7700.0, "data sheet (HGX B200, one GPU)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", type=int, default=131072)
    ap.add_argument("--samples", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cap", type=int, default=16)
    ap.add_argument("--loop-traces", type=int, default=1000)
    ap.add_argument("--out", default=None, help="write the JSON document to this file (default: stdout)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("wfstats_bench needs a CUDA device")
    import legenddsp.jl_b200 as L
    A = L._abi
    h = L.Handle(0)
    n_ev, n, cap = a.events, a.samples, a.cap
    info = {"gpu_before": gpu_info()}
    d_u16 = torch.zeros((n_ev, n), dtype=torch.int16, device="cuda")
    torch.cuda.synchronize()
    L.synth.generate_device(h, d_u16.data_ptr(), n_ev, n_samples=n)
    h.synchronize()
    d_f64 = (d_u16.to(torch.int32) & 0xFFFF).to(torch.float64)
    d_thr = d_f64[:, :2000].mean(dim=1) + 50.0
    d_rows = torch.zeros((n_ev, A.WFSTAT_NCOL), dtype=torch.float64, device="cuda")
    d_lists = torch.zeros((n_ev, 4, cap), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    peak, peak_src = hbm_peak()
    res = []
    for dname, d_wf, kind, sb in (("uint16", d_u16, A.SAMPLE_U16, 2), ("float64", d_f64, A.SAMPLE_F64, 8)):
        for pname, what in PRIMS:
            if kind != A.SAMPLE_U16:             # saturation compares raw ADC samples: uint16 only
                if what == A.WFSTAT_SATURATION:
                    continue
                what &= ~A.WFSTAT_SATURATION
            P = L.stats.wfstats_params(n, kind, what, L.ns(0.0), L.ns(16.0))
            P.sat_from, P.sat_until, P.sat_low, P.sat_high = 0, n - 1, 0, 65535
            P.ext_from, P.ext_until, P.tail_from, P.tail_until = 0, n - 1, 4000, n - 1
            P.max_from, P.max_until = 2900, 3500
            P.thr_min, P.thr_max = 8000.0, 16000.0
            P.im_min_n, P.im_max_n, P.max_triggers = 3, 40, cap
            im = bool(what & A.WFSTAT_INTERSECT_MAXIMUM)
            run = lambda: h.wfstats_run_device(P, d_wf.data_ptr(), d_thr.data_ptr() if im else None, n_ev, n, d_rows.data_ptr(),
                                               d_lists.data_ptr() if im else None)
            run()
            h.synchronize()
            ms = []
            for _ in range(a.reps):
                run()
                h.synchronize()
                ms.append(h.last_kernel_ms())
            t = float(np.median(ms)) * 1e-3
            nbytes = n_ev * (n * sb + A.WFSTAT_NCOL * 8 + ((8 + 4 * cap * 8) if im else 0))
            res.append({"input": dname, "primitives": pname, "what": what, "ms": [round(x, 4) for x in ms],
                        "wf_per_s": n_ev / t, "algorithmic_bytes": nbytes, "gb_per_s": nbytes / t / 1e9,
                        "hbm_fraction": nbytes / t / 1e9 / peak})
            print(f"{dname:8s} {pname:20s} {t * 1e3:9.3f} ms  {n_ev / t / 1e6:8.2f} M wf/s  {nbytes / t / 1e9:8.1f} GB/s", file=sys.stderr, flush=True)
    del d_u16, d_f64, d_rows, d_lists
    torch.cuda.empty_cache()

    # per-trace loop of the single-trace entries against one batched host call, same traces, from host memory
    m = a.loop_traces
    rng = np.random.default_rng(1)
    Y = rng.normal(0, 1.0, (m, n))
    for e in range(m):
        for _ in range(int(rng.integers(0, 20))):
            s0 = int(rng.integers(0, n - 60))
            Y[e, s0:s0 + int(rng.integers(1, 60))] += rng.uniform(2, 6)
    thr = np.full(m, 3.0)
    h.intersect_maximum(Y[0], 0.0, 16.0, 3.0, 2, 20, 256)
    t0 = time.perf_counter()
    loop = [(h.intersect_maximum(Y[e], 0.0, 16.0, thr[e], 2, 20, 256), h.thresholdstats(Y[e], -2.0, 2.0, True)) for e in range(m)]
    t_loop = time.perf_counter() - t0
    P = L.stats.wfstats_params(n, A.SAMPLE_F64, A.WFSTAT_INTERSECT_MAXIMUM | A.WFSTAT_THRESHOLDSTATS_MAD, L.ns(0.0), L.ns(16.0))
    P.thr_min, P.thr_max, P.im_min_n, P.im_max_n, P.max_triggers = -2.0, 2.0, 2, 20, 256
    L.stats.wfstats_rows(Y, P, thr, handle=h)          # warm-up of the same shape: grows the pinned staging once
    t0 = time.perf_counter()
    rows, lists = L.stats.wfstats_rows(Y, P, thr, handle=h)
    t_batch = time.perf_counter() - t0
    same = all(rows[e, A.WFSTAT_COL["thr_mad"]] == loop[e][1] and rows[e, A.WFSTAT_COL["multiplicity"]] == loop[e][0]["multiplicity"]
               and np.array_equal(lists[e, 0, :len(loop[e][0]["x"])], loop[e][0]["x"]) for e in range(m))
    info["gpu_after"] = gpu_info()
    doc = {"tool": "tools/wfstats_bench.py", "events": n_ev, "samples": n, "max_triggers": cap, "reps": a.reps,
           "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "device": info, "device_entry": res,
           "single_trace_loop": {"traces": m, "samples": n, "primitives": "intersect_maximum + thresholdstats_mad",
                                 "loop_s": t_loop, "batched_s": t_batch, "speedup": t_loop / t_batch, "same_results": bool(same)}}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)
        print(json.dumps(doc["single_trace_loop"]), file=sys.stderr, flush=True)
    else:
        print(json.dumps(doc, indent=1), flush=True)
    h.close()


if __name__ == "__main__":
    main()
