#!/usr/bin/env python
"""bench.py -- throughput of the dsp_icpc hot path (waveforms/s, 8192-sample UInt16 ICPC waveforms).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload W] [--batch B] [--dump-outputs DIR]

One "step" = one pass of the chain over one batch of synthetic waveforms.
  value            the batch is already resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e              the same through the reference-facing host C-ABI call with PINNED host buffers: H2D of the raw UInt16
                   samples + kernels + D2H of the 49-column rows inside the timed region
  e2e_pageable     the same from pageable numpy memory (what a Julia `flatview(wvfs.signal)` is): staged through the library's
                   pinned ring by LGDSP_COPY_THREADS host threads
  e2e_encoded      the same with radware-sigcompress ENCODED waveforms in pinned host memory (the on-disk form of LEGEND
                   waveforms): only the encoded bytes cross the host link, decode_data runs on the GPU
  value_with_gather  (config 5 of BASELINE.json) the device-resident step plus the gather of every rank's output table on rank 0
                   (NCCL gather over NVLink, then one D2H into pinned host memory) inside the timed region
  extra_workloads  BASELINE configs[1] (PZ + trapezoid energy / t0 only) and configs[3] (20 x 10 trapezoid sweep), a few steps each
Workloads: dsp_icpc (default; full 49-column chain incl. CUSP/ZAC = BASELINE.json configs[2]/[4]), pz_trap (configs[1]),
trap_sweep (configs[3]), compressed (dsp_icpc_compressed, SURVEY 8f rank 1; e2e on ENCODED bytes), sipm.
Multi-GPU: one process per GPU under torchrun, events sharded, no collective on the data path ("weak" scaling: per-GPU
batch fixed).  `--impl reference` times the CPU port of the reference algorithm (oracle/, -O3 build) on rank 0; it does
not load the product library.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_IN = 8192 * 2
NCOL = 49
# DRAM traffic per waveform from the committed ncu capture of the split pipeline (profiles/r02_ncu_launches_split.txt:
# dram__bytes_read.sum + dram__bytes_write.sum of prefix + extract + CUSP/ZAC select + finish, per event).  The prefix sums
# (65.6 KB per event) are written once and read by the two consumers through L2/HBM: that is the price of running the chain
# as kernels with their own occupancy; algorithmic bytes are 16 776 B per waveform.
NCU_DRAM_BYTES_PER_WF = {"dsp_icpc": 223.9e3,
                         # sweep_warp_kernel (profiles/r02_sweep_warp_kernel_ncu_full.txt): 309.0 MB read + 9.9 MB written per 16 384 events
                         "trap_sweep": 19.46e3}


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "of measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "of fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """host cores this process may use (torchrun exports OMP_NUM_THREADS=1, so ask the scheduler, not OpenMP)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


PRESUM, WDW_FROM, WDW_N = 8, 2600, 1400   # the compressed workload: 1024 presummed uint32 + 1400 windowed uint16 samples


def compressed_setup(L, cfg, tau, builders=None):
    return L.resolve_compressed_params(cfg, tau, None, presum_rate=PRESUM, n_pre=8192 // PRESUM, step_pre=L.ns(16.0 * PRESUM),
                                       n_wdw=WDW_N, t_first_wdw=L.ns(16.0 * WDW_FROM), step_wdw=L.ns(16.0), builders=builders)


SIPM_N, SIPM_CAP = 6250, 32


def sipm_setup(L, builders=None):
    cfg = L.example_sipm_config()
    cfg["filters"]["sg"].update(min_threshold=-3.0, max_threshold=3.0, min_dc_threshold=-40.0, max_dc_threshold=40.0)
    cfg["filters"]["trap"].update(min_threshold=-15.0, max_threshold=15.0, min_dc_threshold=-30.0, max_dc_threshold=30.0)
    return L.resolve_sipm_params(cfg, {"sg": {"wl": L.ns(200.0)}}, n_samples=SIPM_N, builders=builders, max_triggers=SIPM_CAP)


def sipm_events(torch, n_events, seed, device):
    """raw UInt16 SiPM-like traces (baseline 2000 ADC, white noise sigma 2, 0..6 photo-electron pulses): int16 bit patterns"""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    k = torch.arange(SIPM_N, device=device, dtype=torch.float32)[None, :]
    y = 2000.0 + 2.0 * torch.randn((n_events, SIPM_N), generator=g, device=device)
    for q in range(6):
        on = (torch.rand((n_events, 1), generator=g, device=device) < 0.5).float()
        s0 = 100.0 + (SIPM_N - 500.0) * torch.rand((n_events, 1), generator=g, device=device)
        amp = 15.0 + 105.0 * torch.rand((n_events, 1), generator=g, device=device)
        d = (k - s0).clamp(min=0.0)
        y += on * amp * (k >= s0).float() * (1.0 - torch.exp(-d / 3.0)) * torch.exp(-d / 30.0)
    return y.round().clamp(0, 65535).to(torch.int32).to(torch.int16)


def sweep_variants(L):
    rts = [L.us(1.0 + 0.75 * i) for i in range(20)]
    fts = [L.us(1.0 + 0.3 * i) for i in range(10)]
    return L.trap_variants(rts, fts, L.ns(16.0), mode="ft")


class CpuArm:
    """the CPU port of the reference algorithm (oracle/, the -O3 -march=native build that also pays for the reference's
    second ZAC pass) on all host cores; its own event generator -- nothing of the product library is loaded"""

    def __init__(self, L, workload, cfg, tau, groups, threads):
        from oracle import oracle as O
        O.use_fast_build(True)
        self.O, self.L, self.workload, self.threads = O, L, workload, threads
        self.kind = "port"
        b = O.OracleBuilders()
        if workload == "compressed":
            self.P = compressed_setup(L, cfg, tau, b)
        elif workload == "sipm":
            self.P = sipm_setup(L, b)
        else:
            self.P = L.resolve_icpc_params(cfg, tau, groups=groups or L._abi.GROUP_ALL, builders=b)
        if workload == "trap_sweep":
            self.sp = L.resolve_sweep_params(cfg, tau, builders=b)
            self.variants = sweep_variants(L)

    def events(self, n):
        if self.workload == "sipm":
            import torch
            return sipm_events(torch, n, 99, "cpu").numpy().view("uint16")
        wf = self.O.synth_generate(n, first_event=10_000_000)
        if self.workload == "compressed":
            import numpy as np
            pre = wf.reshape(n, 8192 // PRESUM, PRESUM).sum(axis=2, dtype=np.uint32)
            return pre, np.ascontiguousarray(wf[:, WDW_FROM:WDW_FROM + WDW_N])
        return wf

    def step(self, ev):
        O, t = self.O, self.threads
        if self.workload == "sipm":
            O.dsp_sipm(self.P, ev, n_threads=t)
        elif self.workload == "compressed":
            Pp, Pw, aux = self.P
            O.dsp_icpc_compressed(Pp, Pw, ev[0], ev[1], PRESUM, aux, n_threads=t)
        elif self.workload == "trap_sweep":
            O.trap_sweep(self.sp, ev, self.variants, n_threads=t)
        elif self.workload == "pz_trap":
            O.pz_trap(self.P, ev, n_threads=t)
        else:
            O.dsp_icpc(self.P, ev, n_threads=t)

    def throughput(self, n, reps=1):
        ev = self.events(n)
        best = None
        for _ in range(reps):
            t0 = time.perf_counter()
            self.step(ev)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        return n / best

    def describe(self, n):
        what = {"pz_trap": "only the steps that produce blmean, t0, t50, e_trap, e_10410 (src/dsp_icpc.jl:102-163)",
                "trap_sweep": "one full trapezoid pass per (rt, ft) variant as the reference does"}.get(
                    self.workload, "float64, one materialised intermediate per step, direct-form CUSP/ZAC FIRs, ZAC applied twice as "
                                   "src/dsp_icpc.jl:175,177")
        return (f"{n} waveforms of the same synthetic stream; CPU restatement of the reference algorithm (oracle/, gcc -O3 "
                f"-march=native -fopenmp, OpenMP over events): {what}; not Julia")


DUMP_BYTES = 64_000_000


def dump_outputs(torch, outdir, arrays, seed=0):
    """np.save each device array of `arrays` (events on axis 0) as outdir/<name>.npy with its non-finite entries set to 0, and
    beside it outdir/<name>_nonfinite.npy (float32, same shape): 0 finite, 1 NaN, 2 +inf, 3 -inf.  The chain's NaN / inf
    results are real outputs; this keeps every file finite without losing them.  When the files together would exceed
    DUMP_BYTES, each keeps the same seeded sample of events, in event order"""
    import numpy as np
    first = next(iter(arrays.values()))
    n = first.shape[0]
    per_event = sum(a[0].numel() * (a.element_size() + 4) for a in arrays.values())
    keep = min(n, (DUMP_BYTES - 2 * 1024 * len(arrays)) // per_event)   # 1 KB per file for the .npy header
    idx = None
    if keep < n:
        idx = torch.from_numpy(np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))).to(first.device)
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        a = a if idx is None else a.index_select(0, idx)
        code = torch.zeros(a.shape, dtype=torch.float32, device=a.device)
        code[torch.isnan(a)] = 1.0
        code[torch.isposinf(a)] = 2.0
        code[torch.isneginf(a)] = 3.0
        np.save(os.path.join(outdir, name + ".npy"), torch.where(code == 0, a, torch.zeros_like(a)).cpu().numpy())
        np.save(os.path.join(outdir, name + "_nonfinite.npy"), code.cpu().numpy())


WL_NAME = {"dsp_icpc": "full dsp_icpc, 49 columns incl. CUSP+ZAC (BASELINE configs[2]/[4])",
           "pz_trap": "pole-zero + trapezoid energy / t0 only: blmean, t0, t50, e_trap, e_10410 (BASELINE configs[1])",
           "trap_sweep": "20x10 trapezoid (rt, ft) sweep, 200 variants (BASELINE configs[3])",
           "sipm": "dsp_sipm trigger chain on 6250-sample UInt16 SiPM traces (SURVEY 8f rank 3)",
           "compressed": "dsp_icpc_compressed: 1024 presummed uint32 (x8) + 1400 windowed uint16 samples per event "
                         "(SURVEY 8f rank 1)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="dsp_icpc", choices=["dsp_icpc", "pz_trap", "trap_sweep", "compressed", "sipm"])
    ap.add_argument("--batch", type=int, default=131072, help="waveforms per step per GPU (131072 = 2.1 GB >> L2)")
    ap.add_argument("--pool", type=int, default=8, help="distinct resident batches cycled by the steps")
    ap.add_argument("--direct", action="store_true", help="CUSP/ZAC as direct 2375-tap FIRs (validation mode)")
    ap.add_argument("--path", default="split", choices=["split", "fused"], help="dsp_icpc execution path")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-sample", type=int, default=0, help="events of the cpu_baseline sample (0: auto)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip extra_workloads / e2e variants / value_with_gather")
    ap.add_argument("--groups", default=None, help="override the column-group mask (hex), for per-stage timing experiments")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output arrays of the last timed step (rank 0) as DIR/<name>.npy with non-finite entries "
                         "as 0 and their kind in DIR/<name>_nonfinite.npy; above 64 MB in all, the same fixed seeded sample "
                         "of events from every array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    import importlib
    L = importlib.import_module("legenddsp.jl_b200")

    cfg = L.tiefree_config()
    tau = L.us(500.0)
    groups = {"dsp_icpc": L._abi.GROUP_ALL, "pz_trap": L._abi.GROUP_PZTRAP_LEAN, "trap_sweep": 0, "compressed": 0, "sipm": 0}[args.workload]
    wl_name = WL_NAME[args.workload]
    if args.groups is not None:
        groups = int(args.groups, 16)
        wl_name += f" [experimental group mask {groups:#x}]"
    out_bytes = {"dsp_icpc": NCOL * 8, "pz_trap": 5 * 8, "trap_sweep": 200 * 4, "compressed": 65 * 8,
                 "sipm": (24 + 16 * SIPM_CAP) * 8}[args.workload]
    bytes_in = {"compressed": (8192 // PRESUM) * 4 + WDW_N * 2, "sipm": SIPM_N * 2}.get(args.workload, BYTES_IN)
    bytes_per_wf = bytes_in + out_bytes

    # ------------------------------------------------------------------------------------------
    # reference arm: the CPU port of the reference algorithm (the reference itself is Julia and cannot be
    # installed here -- DESIGN.md section 2), all host threads, bounded sample per step
    # ------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return 0
        threads = host_threads()
        arm = CpuArm(L, args.workload, cfg, tau, groups, threads)
        n_s = args.cpu_sample or {"pz_trap": 512 * threads, "trap_sweep": 16 * threads}.get(args.workload, 32 * threads)
        ev = arm.events(n_s)
        for _ in range(args.warmup):
            arm.step(ev)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            arm.step(ev)
        dt = time.perf_counter() - t0
        val = n_s * args.steps / dt
        print(json.dumps({
            "impl": "reference", "metric": "waveforms/sec for dsp_icpc (8192-sample)", "value": val,
            "unit": "waveforms/s", "n_gpus": 0, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl_name, "n_samples": 8192, "events_per_step": n_s,
                       "note": "CPU restatement of the reference algorithm (oracle/), not Julia: no Julia toolchain in this image"},
            "cpu_baseline": {"value": val, "unit": "waveforms/s", "cores": threads, "kind": arm.kind, "sample": arm.describe(n_s)},
            "e2e": {"value": val, "unit": "waveforms/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return 0

    # ------------------------------------------------------------------------------------------
    # our arm
    # ------------------------------------------------------------------------------------------
    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: the communicator initialisation prints "NCCL version ..." to fd 1, so fd 1
        # points at stderr while the process group and its communicator come up
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    # a dedicated (non-default) torch stream shared with the library, so torch's CUDA events time our kernels
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    h = L.Handle(local_rank, stream=stream.cuda_stream)
    h.set_icpc_path(args.path)

    P = L.resolve_icpc_params(cfg, tau, groups=groups or L._abi.GROUP_ALL, cuspzac_direct=args.direct)
    variants = sparams = None
    if args.workload == "trap_sweep":
        sparams = L.resolve_sweep_params(cfg, tau)
        variants = sweep_variants(L)
    elif args.workload == "compressed":
        Pp, Pw, aux = compressed_setup(L, cfg, tau)
    elif args.workload == "sipm":
        Ps = sipm_setup(L)
    else:
        h.icpc_set_params(P)

    B = args.batch
    n_pool = max(1, args.pool)
    # resident pool of distinct batches, generated on the device (each rank its own slice of the event stream)
    if args.workload == "sipm":
        pool = torch.stack([sipm_events(torch, B, 1000 + rank * n_pool + k, dev) for k in range(n_pool)])
        out_t = torch.empty((B, 4, 4, SIPM_CAP), dtype=torch.float64, device=dev)
    else:
        pool = torch.empty((n_pool, B, 8192), dtype=torch.int16, device=dev)
        for k in range(n_pool):
            L.synth.generate_device(h, pool[k].data_ptr(), B, first_event=(rank * n_pool + k) * B)
    if args.workload == "trap_sweep":
        out = torch.empty((B, 200), dtype=torch.float32, device=dev)
    else:
        out = torch.empty((B, NCOL), dtype=torch.float64, device=dev)
    h.synchronize()
    if args.workload == "compressed":
        # the DAQ's compressed format made from the full traces (input generation, outside the timed region); only the
        # compressed buffers stay resident
        torch.cuda.synchronize()
        full = pool.view(n_pool, B, 8192).to(torch.int32) & 0xFFFF
        c_pre = full.view(n_pool, B, 8192 // PRESUM, PRESUM).sum(dim=3, dtype=torch.int32).contiguous()
        c_wdw = pool[:, :, WDW_FROM:WDW_FROM + WDW_N].contiguous()
        del full, pool
        out_w = torch.empty((B, NCOL), dtype=torch.float64, device=dev)
        out_s = torch.empty((B, 5, 5), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        h.icpc_compressed_run_device(Pp, Pw, c_pre[0].data_ptr(), 4, 8192 // PRESUM, c_wdw[0].data_ptr(), 2, WDW_N, float(PRESUM),
                                     aux, B, out.data_ptr(), out_w.data_ptr(), out_s.data_ptr())
        h.synchronize()

    def step(k):
        if args.workload == "sipm":
            h.sipm_run_device(Ps, pool[k % n_pool].data_ptr(), B, SIPM_N, out.data_ptr(), out_t.data_ptr())
        elif args.workload == "compressed":
            h.icpc_compressed_run_device(None, None, c_pre[k % n_pool].data_ptr(), 4, 8192 // PRESUM, c_wdw[k % n_pool].data_ptr(),
                                         2, WDW_N, float(PRESUM), aux, B, out.data_ptr(), out_w.data_ptr(), out_s.data_ptr())
        elif args.workload == "trap_sweep":
            h.sweep_run_device(sparams, pool[k % n_pool].data_ptr(), B, 8192, variants, out.data_ptr())
        else:
            h.icpc_run_device(None, pool[k % n_pool].data_ptr(), B, 8192, out.data_ptr())

    def timed(fn, steps, warmup, finish=None):
        """device ms (CUDA events on the launching stream, max over ranks) and kernel launches of `steps` calls;
        finish() (optional) makes the launching stream wait for side-stream work before the end event"""
        for k in range(warmup):
            fn(k)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        l0 = h.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for k in range(steps):
            fn(k)
        if finish is not None:
            finish()
        e1.record(stream)
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), h.launch_count - l0

    sampler = ClockSampler(local_rank)
    for k in range(args.warmup):
        step(k)
    torch.cuda.synchronize()
    if rank == 0:
        sampler.start()
    ms_max, launches = timed(step, args.steps, 0)
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / (ms_max * 1e-3)
    if args.dump_outputs and rank == 0:
        # before anything below reuses the output buffers
        if args.workload == "sipm":
            arrays = {"rows": out.view(-1)[:B * L._abi.SIPM_NCOL].view(B, L._abi.SIPM_NCOL), "triggers": out_t}
        elif args.workload == "compressed":
            arrays = {"rows_presummed": out, "rows_windowed": out_w, "window_stats": out_s}
        elif args.workload == "trap_sweep":
            arrays = {"trap_sweep": out}
        else:
            arrays = {"rows": out}
        dump_outputs(torch, args.dump_outputs, arrays)

    # ---- e2e through the host C-ABI call (H2D + kernels + D2H inside the timed region) ----
    Be = min(B, 131072)

    def wall(fn, steps):
        fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return float(te.item())

    e2e_extra = {}
    if args.workload == "compressed":
        # the reference-facing call takes the ENCODED waveform sets (decode_data, src/dsp_icpc.jl:313-314, runs on the device)
        pre_h = (c_pre[0][:Be].cpu().numpy().view(np.uint32))
        wdw_h = (c_wdw[0][:Be].cpu().numpy().view(np.uint16))
        enc_p = L.encode_waveforms(pre_h, L.ULEB128_ZIGZAG_DIFF)
        enc_w = L.encode_waveforms(wdw_h, L.RADWARE_SIGCOMPRESS)
        pins = [torch.from_numpy(a).pin_memory() for a in (enc_p.data, enc_p.offsets, enc_w.data, enc_w.offsets)]
        enc_p.data, enc_p.offsets, enc_w.data, enc_w.offsets = [p.numpy() for p in pins]
        host_out = torch.empty((Be, NCOL), dtype=torch.float64).pin_memory()
        host_out_w = torch.empty((Be, NCOL), dtype=torch.float64).pin_memory()
        host_out_s = torch.empty((Be, 25), dtype=torch.float64).pin_memory()
        h.icpc_compressed_run_encoded_host(Pp, Pw, enc_p, enc_w, float(PRESUM), aux, host_out.data_ptr(), host_out_w.data_ptr(),
                                           host_out_s.data_ptr())

        def e2e_step():
            h.icpc_compressed_run_encoded_host(None, None, enc_p, enc_w, float(PRESUM), aux, host_out.data_ptr(), host_out_w.data_ptr(),
                                               host_out_s.data_ptr())
        h2d_bytes = enc_p.nbytes + enc_w.nbytes + 2 * (Be + 1) * 8
        e2e_note = (f"ENCODED host input: ULEB128 zig-zag diff (presummed) + radware-sigcompress (windowed), "
                    f"{(enc_p.nbytes + enc_w.nbytes) / Be:.0f} B/event instead of {bytes_in} B decoded; decode_data on the device")
        # the decoded-input variant for comparison
        hp = torch.from_numpy(pre_h.view(np.int32)).pin_memory()
        hw = torch.from_numpy(wdw_h.view(np.int16)).pin_memory()

        def e2e_raw():
            h.icpc_compressed_run_host(None, None, hp.data_ptr(), 4, 8192 // PRESUM, hw.data_ptr(), 2, WDW_N, float(PRESUM), aux, Be,
                                       host_out.data_ptr(), host_out_w.data_ptr(), host_out_s.data_ptr())
        if not args.no_extra:
            s = wall(e2e_raw, args.e2e_steps)
            e2e_extra["e2e_decoded_input"] = {"value": world * Be * args.e2e_steps / s, "unit": "waveforms/s",
                                              "h2d_bytes_per_step": Be * bytes_in}
    else:
        host_in = torch.empty((Be, SIPM_N if args.workload == "sipm" else 8192), dtype=torch.int16).pin_memory()
        host_in.copy_(pool[0][:Be])
        host_out_t = torch.empty((Be, 16 * SIPM_CAP), dtype=torch.float64).pin_memory() if args.workload == "sipm" else None
        host_out = (torch.empty((Be, 200), dtype=torch.float32) if args.workload == "trap_sweep"
                    else torch.empty((Be, NCOL), dtype=torch.float64)).pin_memory()

        def e2e_step():
            if args.workload == "sipm":
                h.sipm_run_host(Ps, host_in.data_ptr(), Be, SIPM_N, host_out.data_ptr(), host_out_t.data_ptr())
            elif args.workload == "trap_sweep":
                h.sweep_run_host(sparams, host_in.data_ptr(), Be, 8192, variants, host_out.data_ptr())
            else:
                h.icpc_run_host(None, host_in.data_ptr(), Be, 8192, host_out.data_ptr())
        h2d_bytes = Be * bytes_in
        e2e_note = "pinned host buffers, raw UInt16 samples"
    e2e_s = wall(e2e_step, args.e2e_steps)
    e2e_val = world * Be * args.e2e_steps / e2e_s
    ho = host_out.double()
    checksum = float(ho[torch.isfinite(ho)].sum().item())  # the result is really read on the host

    if args.workload == "dsp_icpc" and not args.no_extra:
        # (a) pageable caller memory (numpy): staged through the library's pinned ring
        pg_in = host_in.numpy().copy()
        pg_out = np.empty((Be, NCOL))
        s = wall(lambda: h.icpc_run_host(None, pg_in.ctypes.data, Be, 8192, pg_out.ctypes.data), args.e2e_steps)
        e2e_extra["e2e_pageable"] = {"value": world * Be * args.e2e_steps / s, "unit": "waveforms/s", "h2d_bytes_per_step": Be * bytes_in,
                                     "note": "pageable numpy buffers packed into the pinned staging ring by host threads; bound by the "
                                             "host's memcpy bandwidth (tools/h2d_peak.py)"}
        same = np.array_equal(np.nan_to_num(pg_out), np.nan_to_num(host_out.numpy()))
        # (b) radware-sigcompress encoded waveforms in pinned memory: decode_data on the device
        enc = L.encode_waveforms(pg_in.view(np.uint16), L.RADWARE_SIGCOMPRESS)
        pe, po = torch.from_numpy(enc.data).pin_memory(), torch.from_numpy(enc.offsets).pin_memory()
        s = wall(lambda: h.icpc_run_encoded_host(None, enc.codec, pe.data_ptr(), po.data_ptr(), enc.shift, 2, None, Be,
                                                 host_out.data_ptr()), args.e2e_steps)
        same = same and np.array_equal(np.nan_to_num(pg_out), np.nan_to_num(host_out.numpy()))
        e2e_extra["e2e_encoded"] = {"value": world * Be * args.e2e_steps / s, "unit": "waveforms/s",
                                    "h2d_bytes_per_step": enc.nbytes + (Be + 1) * 8, "bytes_per_event": enc.nbytes / Be,
                                    "note": "RadwareSigcompress(-32768) encoded UInt16 waveforms in pinned host memory (the on-disk form "
                                            "of LEGEND waveforms); decode_data (src/dsp_icpc.jl:313-314) on the device",
                                    "rows_identical_to_e2e": bool(same)}

    # ---- config 5: device-resident step + gather of every rank's output table on rank 0 inside the timed region ----
    gather = None
    if args.workload == "dsp_icpc" and not args.no_extra:
        gsteps = min(args.steps, 10)
        table = torch.empty((world, B, NCOL), dtype=torch.float64, device=dev) if rank == 0 else None
        host_tab = [torch.empty((world * B, NCOL), dtype=torch.float64).pin_memory() for _ in range(2)] if rank == 0 else None

        # double-buffered: the gather + D2H of step k run on a side stream under the kernels of step k+1
        outs2 = [out, torch.empty_like(out)]
        gs = torch.cuda.Stream(device=dev)
        ev_done = [torch.cuda.Event(), torch.cuda.Event()]
        ev_free = [torch.cuda.Event(), torch.cuda.Event()]
        used = [False, False]

        def gstep(k, compute=True):
            b = k & 1
            if compute:
                if used[b]:
                    stream.wait_event(ev_free[b])   # the previous gather out of this buffer is done
                h.icpc_run_device(None, pool[k % n_pool].data_ptr(), B, 8192, outs2[b].data_ptr())
            ev_done[b].record(stream)
            with torch.cuda.stream(gs):
                gs.wait_event(ev_done[b])
                if world > 1:
                    dist.gather(outs2[b], list(table.unbind(0)) if rank == 0 else None, dst=0)
                    src = table
                else:
                    src = outs2[b]
                if rank == 0:
                    host_tab[b].copy_(src.view(-1, NCOL), non_blocking=True)
                ev_free[b].record(gs)
            used[b] = True

        def gfinish():
            for b in range(2):
                if used[b]:
                    stream.wait_event(ev_free[b])

        ms_g, _ = timed(gstep, gsteps, 1, gfinish)
        ms_only, _ = timed(lambda k: gstep(k, False), gsteps, 1, gfinish)
        gather = {"value_with_gather": world * B * gsteps / (ms_g * 1e-3), "unit": "waveforms/s", "steps": gsteps,
                  "gather_ms_per_step": ms_only / gsteps, "d2h_bytes_per_step_rank0": world * B * NCOL * 8,
                  "how": "per step: kernels, NCCL gather of the 392-byte rows to rank 0 (NVLink; no-op at N=1), one D2H of the "
                         "gathered table into pinned host memory; two output buffers: the gather + D2H of step k run on a side "
                         "stream under the kernels of step k+1, the timed region ends when the last table is in host memory; "
                         "gather_ms_per_step is the gather + D2H timed alone"}

    # ---- the other two single-GPU configurations of BASELINE.json, a few steps each ----
    extra = []
    peaks, peak_kind = _peaks()
    if args.workload == "dsp_icpc" and not args.no_extra and args.groups is None:
        xs = min(args.steps, 8)
        P2 = L.resolve_icpc_params(cfg, tau, groups=L._abi.GROUP_PZTRAP_LEAN)
        h.icpc_set_params(P2)
        ms2, _ = timed(step, xs, 2)
        h.icpc_set_params(P)
        b2 = BYTES_IN + 5 * 8
        extra.append({"workload": WL_NAME["pz_trap"], "value": world * B * xs / (ms2 * 1e-3), "unit": "waveforms/s", "ms_per_step": ms2 / xs,
                      "roofline": {"frac": B * b2 / (ms2 * 1e-3 / xs) / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes_per_waveform": b2},
                      "kernel": "icpc_prefix_kernel + icpc_extract_kernel (LGDSP_GROUP_PZTRAP_LEAN)"})
        sp3, v3 = L.resolve_sweep_params(cfg, tau), sweep_variants(L)
        out3 = torch.empty((B, 200), dtype=torch.float32, device=dev)
        ms3, _ = timed(lambda k: h.sweep_run_device(sp3, pool[k % n_pool].data_ptr(), B, 8192, v3, out3.data_ptr()), xs, 2)
        b3 = BYTES_IN + 200 * 4
        extra.append({"workload": WL_NAME["trap_sweep"], "value": world * B * xs / (ms3 * 1e-3), "unit": "waveforms/s", "ms_per_step": ms3 / xs,
                      "roofline": {"frac": B * b3 / (ms3 * 1e-3 / xs) / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes_per_waveform": b3},
                      "kernel": "sweep_warp_kernel (one warp per waveform; LGDSP_SWEEP_PATH=cta: sweep_kernel)"})
        # the reference's own rise-time sweep: e_grid_rt_trap (31 rise times at ft = 2 us), fixed pick-off enc_pickoff_trap, Float64 grid
        # (src/dsp_filter_optimization.jl:102-133); nothing in it depends on t50, so the warp kernel skips max(y) and the crossing
        sp4 = L.resolve_sweep_params(cfg, tau, out_f64=True)
        v4 = L.trap_sweep_variants(L.grid_values(cfg.e_grid_rt_trap), [L.us(2.0)], L.ns(16.0), mode="rt", pickoff=cfg.enc_pickoff_trap)
        nv4 = len(v4.array)
        out4 = torch.empty((B, nv4), dtype=torch.float64, device=dev)
        ms_rt, _ = timed(lambda k: h.gsweep_run_device(sp4, pool[k % n_pool].data_ptr(), B, 8192, v4.array, out4.data_ptr()), xs, 2)
        # bytes the computation needs: the samples up to the last look-up of the set (fixed windows: the same for every event; the
        # kernel reads no sample behind it) + the outputs.  frac_whole_waveform counts all 16 384 input bytes as the other workloads do
        n_w4 = sp4.sig_dni.n_w
        last4 = sp4.bl_until + 1
        for i in range(nv4):
            t4 = v4.array[i].trap
            L4 = t4.navg + t4.ngap + t4.navg2
            nout4 = 8192 - L4 + 1
            pc4 = min(max((v4.array[i].pickoff_ns - (sp4.t_first_ns + (L4 - 1) * sp4.dt_ns)) / sp4.dt_ns, 0.0), nout4 - 1.0)
            f4 = min(max(int(round(pc4)) - n_w4 // 2, 0), nout4 - n_w4)
            last4 = max(last4, f4 + L4 + n_w4)
        b4 = 2 * min(8192, last4 + 8) + nv4 * 8
        rate4 = B / (ms_rt * 1e-3 / xs) / 1e9 / peaks["hbm_gbs"]
        extra.append({"workload": f"dsp_trap_rt_optimization: {nv4} rise times, fixed pick-off (src/dsp_filter_optimization.jl:102-133)",
                      "value": world * B * xs / (ms_rt * 1e-3), "unit": "waveforms/s", "ms_per_step": ms_rt / xs,
                      "roofline": {"frac": rate4 * b4, "algorithmic_bytes_per_waveform": b4,
                                   "frac_whole_waveform": rate4 * (BYTES_IN + nv4 * 8)},
                      "kernel": "sweep_warp_kernel"})

    kernel_ms = None
    if args.workload == "dsp_icpc" and args.path == "split" and not args.no_extra and rank == 0:
        nprof = min(B, 16384)
        ms4 = h.icpc_profile_device(pool[0].data_ptr(), nprof, 8192, out.data_ptr())
        kernel_ms = {"events": nprof, "icpc_prefix_kernel": ms4[0], "icpc_extract_kernel": ms4[1], "icpc_cuspzac_kernel": ms4[2],
                     "icpc_cuspzac_finish_kernel": ms4[3],
                     "note": "one batch run serially with CUDA events between the kernels; in the timed steps the batches of "
                             "four stream pairs overlap"}
        tot4 = sum(ms4) or 1.0
        names4 = ("icpc_prefix_kernel", "icpc_extract_kernel", "icpc_cuspzac_kernel", "icpc_cuspzac_finish_kernel")
        top = max(range(4), key=lambda i: ms4[i])
        kernel_ms["dominant"] = {"kernel": names4[top], "share_of_serial_pipeline": ms4[top] / tot4,
                                 "share_in_ncu_launch_list": "profiles/r02_ncu_launches_split.txt"}

    if rank == 0:
        achieved = B * bytes_per_wf / (ms_max * 1e-3 / args.steps) / 1e9
        kern = {"trap_sweep": "sweep_warp_kernel", "sipm": "sipm_kernel"}.get(
            args.workload, ("icpc_kernel (fused)" if args.path == "fused" else
                            "split pipeline: icpc_prefix_kernel -> icpc_extract_kernel || icpc_cuspzac_kernel -> icpc_cuspzac_finish_kernel")
            + (" x2 (presummed + windowed) + window_stats_kernel" if args.workload == "compressed" else ""))
        line = {
            "metric": "waveforms/sec for dsp_icpc (8192-sample)", "value": value, "unit": "waveforms/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl_name, "n_samples": {"compressed": [8192 // PRESUM, WDW_N], "sipm": SIPM_N}.get(args.workload, 8192),
                       "events_per_step_per_gpu": B, "resident_pool_batches": n_pool,
                       "events_timed_per_gpu": B * args.steps, "resident_pool_events_per_gpu": B * n_pool,
                       "size_note": "BASELINE configs[2] names 10 M events from a 4 M-event pool: the timed region here is "
                                    f"{B * args.steps / 1e6:.1f} M events cycling a {B * n_pool / 1e6:.2f} M-event resident pool (same workload, "
                                    "sample count and dtype; --steps 80 --pool 32 gives the named size)",
                       "dsp_config": "reference example config (test/test_dsp_icpc.jl:50-161), tie-free windows, tau=500us, default filter pars",
                       "cuspzac": "direct FIR" if args.direct else "structured", "path": args.path,
                       "l2": f"inputs larger than L2: each step reads a different {B * bytes_in / 1e9:.1f} GB batch",
                       "parallelism": f"event-sharded x{world}, no data-path collective"},
            "clocks": clocks,
            "gpu_launches": int(launches),
            "e2e": {"value": e2e_val, "unit": "waveforms/s", "h2d_bytes_per_step": int(h2d_bytes),
                    "d2h_bytes_per_step": Be * (out_bytes if args.workload != "compressed" else (2 * NCOL + 25) * 8),
                    "events_per_step_per_gpu": Be, "steps": args.e2e_steps, "input": e2e_note, "checksum": checksum},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / peaks["hbm_gbs"],
                         "traffic": (NCU_DRAM_BYTES_PER_WF[args.workload] * B if args.workload in NCU_DRAM_BYTES_PER_WF
                                     and args.groups is None and args.path == "split" else None),
                         "traffic_unit": "bytes per step (ncu dram__bytes_read.sum + dram__bytes_write.sum of the pipeline's kernels, "
                                         "scaled by events)",
                         "peak_source": peak_kind, "algorithmic_bytes_per_waveform": bytes_per_wf, "kernel": kern,
                         "kernel_ms": kernel_ms},
        }
        line.update(e2e_extra)
        if gather:
            line["value_with_gather"] = gather
        if extra:
            line["extra_workloads"] = extra
        if not args.no_cpu and world == 1:
            threads = host_threads()
            arm = CpuArm(L, args.workload, cfg, tau, groups, threads)
            n_s = args.cpu_sample or {"pz_trap": 8192 * threads, "trap_sweep": 64 * threads}.get(args.workload, 512 * threads)
            v = arm.throughput(n_s)
            line["cpu_baseline"] = {"value": v, "unit": "waveforms/s", "cores": threads, "kind": arm.kind, "sample": arm.describe(n_s)}
        print(json.dumps(line))
    h.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
