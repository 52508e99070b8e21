"""Time split of the three launches of dsp_icpc_compressed (presummed pass, window statistics, windowed pass).
usage (GPU box): python tools/compressed_split.py [n_events]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import importlib
import numpy as np
import torch
L = importlib.import_module("legenddsp.jl_b200")
n = int(sys.argv[1]) if len(sys.argv) > 1 else 32768
cfg, tau = L.tiefree_config(), L.us(500.0)
Pp, Pw, aux = L.resolve_compressed_params(cfg, tau, None, presum_rate=8, n_pre=1024, step_pre=L.ns(128.0), n_wdw=1400,
                                          t_first_wdw=L.ns(16.0 * 2600), step_wdw=L.ns(16.0))
h = L.Handle(0)
wf = L.synth.generate_host(n, first_event=0)
pre, wdw = L.synth.compress(wf, 8, (2600, 1400))
d_pre = torch.from_numpy(pre.view(np.int32)).cuda()
d_wdw = torch.from_numpy(wdw.view(np.int16)).cuda()
rows = torch.empty((n, L.NCOL), dtype=torch.float64, device="cuda")
rows_w = torch.empty((n, L.NCOL), dtype=torch.float64, device="cuda")
bl = torch.full((n,), 1500.0, dtype=torch.float64, device="cuda")
st = torch.empty((n, 5, 5), dtype=torch.float64, device="cuda")
for rep in range(2):
    h.icpc_run_ext_device(Pp, d_pre.data_ptr(), 4, None, n, 1024, rows.data_ptr()); h.synchronize(); t_pre = h.last_kernel_ms()
    h.icpc_run_ext_device(Pw, d_wdw.data_ptr(), 2, bl.data_ptr(), n, 1400, rows_w.data_ptr()); h.synchronize(); t_wdw = h.last_kernel_ms()
    h.window_stats_device(d_pre.data_ptr(), 4, n, 1024, 1024, 0.0, 128.0, bl.data_ptr(), aux + [(0, 304)], st.data_ptr()); h.synchronize()
    t_st = h.last_kernel_ms()
print(f"{n} events: presummed pass {t_pre:.3f} ms ({n / t_pre / 1e3:.2f} M ev/s), windowed pass {t_wdw:.3f} ms ({n / t_wdw / 1e3:.2f} M ev/s), "
      f"window stats {t_st:.3f} ms")
