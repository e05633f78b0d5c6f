#!/usr/bin/env python
"""bench.py -- headline benchmark of bundler_sfm_b200 (contract: see the task prompt / DESIGN.md section 6).

Workload selection (`--workload auto`, the default; both arms apply the same rule):
  1 GPU   -> BA, BASELINE.json configs[2]: 1000 cameras / 500,000 points / 3,000,000 observations (the configuration the
             metric is quoted on and the one that needs the tensor-core reduced solve); one "step" = one full
             run_sfm-equivalent LM solve; metric LM iterations / second.  configs[1] (50 / 20k / 100k) rides along as the
             "ba_config2" object and KeyMatchFull config 4 as the "match" object.
  N > 1   -> MATCH, BASELINE.json configs[3]: all pairs of 500 images x 5000 SIFT keys sharded over the N ranks with an
             NCCL all-gather of the match table (the path that shards: `scaling: strong`); BA replicas (configs[1]) ride
             along as "ba_replicas".
  value : inputs already resident in HBM when the timed region starts
  e2e   : the reference-facing C-ABI call (bsfm_run_sfm / keydb create+run+fetch) with HOST buffers, copies inside the timing
`--workload ba2|ba3|match` forces one.  `--impl reference` times the unmodified reference CPU code (oracle/_ref, built
from /root/reference) on the host cores this process may use (sched_getaffinity and the cgroup quota).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BA_CFGS = {"ba2": dict(num_cameras=50, num_points=20000, views_per_point=5),
           "ba3": dict(num_cameras=1000, num_points=500000, views_per_point=6)}
BA_CFG = BA_CFGS["ba2"]
MATCH_CFG = dict(num_images=500, keys_per_image=5000)
# the `config.workload` strings are shared by both arms (the driver compares them)
WORKLOAD_STR = {
    "ba2": "synthetic BA: 50 cams, 20k points, 100k obs (BASELINE.json configs[1]); one step = one full LM solve",
    "ba3": "synthetic BA: 1000 cams, 500k points, 3M obs (BASELINE.json configs[2]); one step = one full LM solve",
    "match": "KeyMatchFull config 4: all pairs of 500 images x 5000 SIFT keys, exact 2-NN + ratio 0.6 (BASELINE.json configs[3])",
}
METRIC_STR = {"ba": "LM iterations/s (sparse bundle adjustment solve)", "match": "descriptor-pairs/s (all-pairs SIFT match, KeyMatchFull)"}


def measure_device_peaks(torch, dev):
    """measured on THIS box, in this process, before the timed runs (each takes a few tens of ms):
      int8 tensor pipe : a plain tcgen05.mma kind::i8 loop of the library (bsfm_measure_int8_peak; N = 256 and N = 128 tiles)
      fp64             : cuBLAS DGEMM through torch.matmul, 6144^3, best of 5"""
    from bundler_sfm_b200 import _lib
    lib = _lib.load_library()
    out = {}
    try:
        out["int8_tops_n256"] = max(lib.bsfm_measure_int8_peak(256, 20000) for _ in range(2))
        out["int8_tops_n128"] = max(lib.bsfm_measure_int8_peak(128, 40000) for _ in range(2))
    except Exception as e:      # noqa: BLE001 -- never fake a peak
        out["int8_error"] = str(e)
    try:
        n = 6144
        a = torch.randn(n, n, dtype=torch.float64, device=dev)
        b = torch.randn(n, n, dtype=torch.float64, device=dev)
        best = 0.0
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); c = a @ b; e1.record(); torch.cuda.synchronize()
            best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        out["fp64_dgemm_tflops"] = best
        del a, b, c
    except Exception as e:      # noqa: BLE001
        out["fp64_error"] = str(e)
    return out


def usable_cores():
    """host cores this process may really use: the scheduler affinity mask, capped by the cgroup CPU quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except (OSError, ValueError, IndexError):
            pass
    return max(1, n)


def pick_workload(args):
    if args.workload in ("ba2", "ba3", "match"):
        return args.workload
    if args.workload == "ba":
        return "ba3"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return "match" if (args.gpus > 1 or world > 1) else "ba3"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region through NVML in-process (the same counters
    `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints; an external `nvidia-smi -lms 100` loop was
    measured to slow the host-side CUDA calls of the timed loop by ~4x, so it is not used)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index, period_s=0.05):
        self.gpu = gpu_index
        self.period = period_s
        self.samples = []
        self.stop_flag = False
        self.thread = None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # map the CUDA device to its NVML handle through the PCI bus id (CUDA_VISIBLE_DEVICES safe)
            import torch
            bus = torch.cuda.get_device_properties(self.gpu).pci_bus_id if hasattr(torch.cuda.get_device_properties(self.gpu), "pci_bus_id") else None
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.gpu) if bus is None else None
            if self.handle is None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    h = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(h).bus == bus:
                        self.handle = h
                        break
                if self.handle is None:
                    self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        except Exception as e:   # NVML missing: report it, never fake a clock
            self.nvml = None
            self.err = str(e)

    def _run(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
                rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((sm, mx, rs))
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        if self.nvml is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.stop_flag = True
        self.thread.join(timeout=2)
        sm = [s[0] for s in self.samples]
        reasons = set()
        for _, _, rs in self.samples:
            for bit, name in self.REASONS.items():
                if rs & bit:
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(s[1] for s in self.samples)) if sm else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------------------
# reference arm: the unmodified reference on the host cores
# ------------------------------------------------------------------------------------------------
def _ref_ba_worker(args):
    seed, nsolves = args
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    from bundler_sfm_b200 import synth
    from oracle import loader
    scene = synth.ba_scene(seed=seed, **BA_CFGS["ba2"])
    its = 0
    t0 = time.perf_counter()
    for _ in range(nsolves):
        out = loader.run_sfm_oracle(scene)
        its += int(out["info"][5])
    return its, time.perf_counter() - t0


def run_reference_ba2(steps, warmup, procs):
    """`procs` independent reference processes (the reference is single-threaded and not re-entrant,
    SURVEY.md F6), each solving the config-2 scene `steps` times: aggregate LM iterations / s."""
    import multiprocessing as mp
    os.environ["OPENBLAS_NUM_THREADS"] = "1"    # before anything loads OpenBLAS: one BLAS thread per process
    kind = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_sba.so")) else "port"
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        if warmup > 0:
            pool.map(_ref_ba_worker, [(1234 + r, 1) for r in range(procs)])
        t0 = time.perf_counter()
        res = pool.map(_ref_ba_worker, [(1234 + r, steps) for r in range(procs)])
        wall = time.perf_counter() - t0
    its = sum(r[0] for r in res)
    return its / wall, wall, kind, its


def run_reference_ba3(lm_iterations, threads, scene=None):
    """The reference on config 3 is ONE process (sba is single-threaded; only dpotrf runs on `threads` OpenBLAS
    threads): a bounded sample = the unmodified run_sfm stopped after `lm_iterations` LM iterations (REF_SBA_ITMAX
    changes the itmax argument of the call, nothing in the reference).  -> (LM it/s, seconds, kind, iterations)"""
    os.environ["OPENBLAS_NUM_THREADS"] = str(threads)
    os.environ["REF_SBA_ITMAX"] = str(lm_iterations)
    from bundler_sfm_b200 import synth
    from oracle import loader
    if loader.ref_sba() is None:
        return None
    if scene is None:
        scene = synth.ba_scene(seed=1234, **BA_CFGS["ba3"])
    t0 = time.perf_counter()
    out = loader.run_sfm_ref(scene)
    dt = time.perf_counter() - t0
    os.environ.pop("REF_SBA_ITMAX")
    its = int(out["info"][5])
    return its / dt, dt, "reference", its


def _ref_match_worker(args):
    seed, npairs = args
    from bundler_sfm_b200 import synth
    from oracle import loader
    imgs = synth.sift_like_descriptors(2, MATCH_CFG["keys_per_image"], seed=seed)
    lib = loader.ref_match()
    t0 = time.perf_counter()
    for _ in range(npairs):
        if lib is not None:
            loader.match_pair_ref(imgs[0], imgs[1], 0.6, 200)     # stock KeyMatchFull: ANN priority search, 200-visit cap
        else:
            loader.match_pair_port(imgs[0], imgs[1], 0.6)
    return npairs, time.perf_counter() - t0


def run_reference_match(pairs_per_proc, procs, warmup=1):
    import multiprocessing as mp
    kind = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_match.so")) else "port"
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        if warmup > 0:
            pool.map(_ref_match_worker, [(7 + r, 1) for r in range(procs)])
        t0 = time.perf_counter()
        res = pool.map(_ref_match_worker, [(7 + r, pairs_per_proc) for r in range(procs)])
        wall = time.perf_counter() - t0
    npairs = sum(r[0] for r in res)
    K = MATCH_CFG["keys_per_image"]
    return npairs * K * K / wall, npairs / wall, wall, kind, npairs


def main_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    procs = usable_cores()
    wl = pick_workload(args)
    if wl == "match":
        # one step = `pairs` image pairs per process (one process per usable core); the run is sized to ~1-2 minutes
        pairs = 4
        steps = max(1, min(args.steps, 6))
        dps, ips, wall, kind, npairs = run_reference_match(pairs * steps, procs, warmup=min(args.warmup, 1))
        line = {"impl": "reference", "metric": METRIC_STR["match"], "value": dps, "unit": "descriptor-pairs/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * wall / steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": WORKLOAD_STR["match"], **MATCH_CFG},
                "cpu_baseline": {"value": dps, "unit": "descriptor-pairs/s", "cores": procs, "kind": kind,
                                 "sample": f"{npairs} image pairs of 5000x5000 keys ({pairs} per process and step), stock ANN kd-tree priority search "
                                           f"(200-visit cap, the reference's default), one single-threaded process per usable core"},
                "e2e": {"value": dps, "unit": "descriptor-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "image_pairs_per_s": ips}
    elif wl == "ba3":
        # 835 s for the full solve (tests/golden/ba_config3_ref.json): a step = the same solve stopped after 2 LM iterations
        res = run_reference_ba3(2, procs)
        if res is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref_sba.so not built (needs /root/reference at build time)"}), flush=True)
            return
        ips, wall, kind, its = res
        line = {"impl": "reference", "metric": METRIC_STR["ba"], "value": ips, "unit": "LM iterations/s",
                "n_gpus": args.gpus, "steps": 1, "warmup": 0, "ms_per_step": 1e3 * wall, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": WORKLOAD_STR["ba3"], **BA_CFGS["ba3"]},
                "cpu_baseline": {"value": ips, "unit": "LM iterations/s", "cores": procs, "kind": kind,
                                 "sample": f"one run_sfm call of the unmodified reference stopped after {its} LM iterations ({wall:.1f} s incl. the initial "
                                           f"error evaluation); sba is single-threaded, dpotrf uses {procs} OpenBLAS threads; the full 20-iteration solve took "
                                           f"835 s in the build container (tests/golden/ba_config3_ref.json)"},
                "e2e": {"value": ips, "unit": "LM iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    else:
        steps = max(1, min(args.steps, 3))
        ips, wall, kind, its = run_reference_ba2(steps, min(args.warmup, 1), procs)
        line = {"impl": "reference", "metric": METRIC_STR["ba"], "value": ips, "unit": "LM iterations/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * wall / steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": WORKLOAD_STR["ba2"], **BA_CFGS["ba2"]},
                "cpu_baseline": {"value": ips, "unit": "LM iterations/s", "cores": procs, "kind": kind,
                                 "sample": f"{steps} full run_sfm solves per process, {procs} independent single-threaded processes (one per usable core)"},
                "e2e": {"value": ips, "unit": "LM iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def pinned_view(torch, arr):
    """the array in page-locked host memory (the e2e contract: inputs are copied from pinned host memory); returns
    (numpy view, tensor that owns the memory) and falls back to the pageable array if pinning is not possible"""
    try:
        t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
        return t.numpy(), t
    except Exception:     # noqa: BLE001 -- measurement convenience only
        return arr, None


def flush_l2(torch, buf):
    buf.add_(1)   # 512 MB read+write > 126 MB L2


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every array as out_dir/<name>.npy in float64, so that two builds can be compared output for output.
    When they would take more than DUMP_LIMIT_BYTES in all, every array of more than 1 MB is replaced by a fixed, seeded
    sample of its rows, whose indices go to <name>_rows.npy (a row takes at least as many bytes as its index)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    large = sum(a.nbytes for a in arrays.values() if a.nbytes > (1 << 20))
    small = sum(a.nbytes for a in arrays.values()) - large
    for name, a in arrays.items():
        if small + large > DUMP_LIMIT_BYTES and a.nbytes > (1 << 20):
            keep = max(1, int(a.shape[0] * (DUMP_LIMIT_BYTES - small) / (2 * large)))
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def bench_ba(args, torch, dist, rank, world, dev, cfg_key, steps, warmup, scene=None, dump_dir=None):
    from bundler_sfm_b200 import bundle, synth
    os.environ.setdefault("BSFM_BA_VERBOSE", "0")
    cfg = BA_CFGS[cfg_key]
    if scene is None:
        scene = synth.ba_scene(seed=1234 + rank, **cfg)
    n, m = scene["vmask"].shape
    nvis = scene["projections"].shape[0]
    p0, cnp = bundle.pack_params(scene)
    d_vmask = torch.from_numpy(np.ascontiguousarray(scene["vmask"], np.int8)).to(dev)
    d_x = torch.from_numpy(np.ascontiguousarray(scene["projections"])).to(dev)
    d_p0 = torch.from_numpy(p0).to(dev)
    d_p = d_p0.clone()
    flush = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    R_init, f_fixed = scene["R"], scene["f"]
    devnull = os.open(os.devnull, os.O_WRONLY)

    def solve_resident():
        d_p.copy_(d_p0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        its, info = bundle.levmar_model(n, m, d_vmask.data_ptr(), d_p.data_ptr(), d_x.data_ptr(), cnp, R_init, f_fixed)
        return its, time.perf_counter() - t0, bundle.last_timing(), info

    vm_pin, _keep_vm = pinned_view(torch, scene["vmask"])
    pr_pin, _keep_pr = pinned_view(torch, scene["projections"])
    scene_e2e = dict(scene, vmask=vm_pin, projections=pr_pin)

    def solve_e2e():
        t0 = time.perf_counter()
        out = bundle.run_sfm(scene_e2e)
        return int(out["info"][5]), time.perf_counter() - t0, out

    # silence the reference-compatible stdout chatter of the solver ("max_pct_change: ...")
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(devnull, 1)
    try:
        for _ in range(warmup):
            solve_resident(); solve_e2e()
        lib = bundle.load_library()
        launches0 = lib.bsfm_kernel_launches()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(torch.cuda.current_device()); sampler.start()
        its_sum, dev_ms, wall = 0, 0.0, 0.0
        for _ in range(steps):
            flush_l2(torch, flush)
            its, w, tm, info = solve_resident()
            its_sum += its; wall += w; dev_ms += tm["total_ms"]
        torch.cuda.synchronize()
        launches = lib.bsfm_kernel_launches() - launches0
        if dump_dir is not None:     # the last timed solve: refined parameters (cameras, then points) and info[10]
            p = d_p.cpu().numpy()
            dumped = {"cameras": p[:m * cnp].reshape(m, cnp), "points": p[m * cnp:].reshape(n, 3), "info": info}
        if dist is not None:
            dist.barrier()
        e_its, e_wall = 0, 0.0
        for _ in range(steps):
            flush_l2(torch, flush)
            its, w, out = solve_e2e()
            e_its += its; e_wall += w
        torch.cuda.synchronize()
        clocks = sampler.stop()
        # one more solve with per-phase events and (large systems) per-kernel-class events of the dense Cholesky
        os.environ["BSFM_BA_TIMING"] = "1"
        lib.bsfm_ba_chol_profile(1)
        _, _, tm, _ = solve_resident()
        os.environ.pop("BSFM_BA_TIMING")
        pms = (ctypes.c_float * 4)(); pl = (ctypes.c_int * 4)(); ops = ctypes.c_double(); fl = ctypes.c_double()
        lib.bsfm_ba_chol_profile_read(pms, pl, ctypes.byref(ops), ctypes.byref(fl))
        lib.bsfm_ba_chol_profile(0)
    finally:
        os.dup2(saved, 1)
        os.close(saved)
    if dump_dir is not None:
        dump_outputs(dump_dir, dumped)
    rmse = float(np.sqrt(out["info"][1] / nvis))
    # max over ranks (device-event time of the solves), sum of iterations
    t = torch.tensor([dev_ms * 1e-3, e_wall, float(its_sum), float(e_its)], dtype=torch.float64, device=dev)
    if dist is not None:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dev_s, e_s, its_all, e_its_all = tmax[0].item(), tmax[1].item(), tsum[2].item(), tsum[3].item()
    else:
        dev_s, e_s, its_all, e_its_all = t[0].item(), t[1].item(), t[2].item(), t[3].item()
    # the dense n x m visibility mask of the reference interface is uploaded as it is, unless BSFM_BA_MASK_HOST_MIN enables the
    # library's host-side compression (ba_solver.cu, host_scan_vmask: CRS, 4 (n + 1) + 4 nvis bytes; measured slower end to end here)
    host_min = os.environ.get("BSFM_BA_MASK_HOST_MIN")
    mask_bytes = (4 * (n + 1) + 4 * nvis) if (host_min is not None and n * m >= int(host_min)) else n * m
    h2d = mask_bytes + nvis * 16 + m * ctypes.sizeof(bundle.CameraParams) + n * 24
    d2h = (m * cnp + 3 * n) * 8
    # algorithmic HBM bytes per LM iteration (SURVEY.md 8d / DESIGN.md): ~0.7 KB per observation + 16 (9m)^2
    alg_bytes = 0.7e3 * nvis + 16.0 * (9 * m) ** 2
    iters_one = tm["iterations"]
    res = {
        "value": its_all / dev_s, "ms_per_step": 1e3 * dev_s / steps, "e2e_value": e_its_all / e_s,
        "h2d": h2d, "d2h": d2h, "launches": int(launches), "clocks": clocks, "rmse": rmse, "iterations_per_solve": iters_one,
        "phase_ms": {k: v for k, v in tm.items()},
        "roofline_achieved_gbs": alg_bytes * iters_one / (tm["total_ms"] * 1e-3) / 1e9,
        "steps": steps, "warmup": warmup,
    }
    if pl[2] > 0 and pms[2] > 0:      # large system: the tensor-core trailing update is the dominant kernel
        res["chol"] = {
            "kernel_ms_one_solve": {"diag_block": pms[0], "panel_solve": pms[1], "trailing_update_tcgen05": pms[2], "back_substitution": pms[3]},
            "launches_one_solve": {"diag_block": pl[0], "panel_solve": pl[1], "trailing_update_tcgen05": pl[2], "back_substitution": pl[3]},
            "trailing_int8_tops": ops.value / (pms[2] * 1e-3) / 1e12, "trailing_fp64_equiv_tflops": fl.value / (pms[2] * 1e-3) / 1e12,
            "trailing_avg_launch_ms": pms[2] / pl[2], "int8_ops_per_launch": ops.value / pl[2],
        }
    return res


def bench_match(args, torch, dist, rank, world, dev, num_images, keys_per_image, steps, warmup, dump_dir=None):
    from bundler_sfm_b200 import keymatch, synth
    imgs = synth.sift_like_descriptors(num_images, keys_per_image, seed=7)
    keys, key_off = keymatch.concat_keys(imgs)
    sizes = [keys_per_image] * num_images
    b, e = keymatch.shard_images(sizes, -1, world)[rank]
    d_keys = torch.from_numpy(keys).to(dev)
    db = keymatch.KeyDatabase(None, key_off, device_ptr=d_keys.data_ptr())

    # N > 1: the library's own NCCL communicator (one rank per process; the unique id travels through torch.distributed once,
    # like init_process_group -- outside the timed regions).  The table all-gather runs inside the library over NVLink.
    comm = keymatch.Comm.from_torch(device=dev) if dist is not None else None

    def gather():
        if comm is None:
            return db.result_dev()[3]
        return db.allgather(comm)

    from bundler_sfm_b200 import _lib
    lib = _lib.load_library()
    for _ in range(warmup):
        db.run(b, e, -1, 0.6); gather()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = lib.bsfm_kernel_launches()
    sampler = ClockSampler(torch.cuda.current_device()); sampler.start()
    # device time: the library times its launches with CUDA events on ITS stream (bsfm_match_last_timing); the NCCL table
    # all-gather (also on the library's stream, synchronised before it returns) is timed around the call; wall clock of the
    # whole pass is kept as a cross-check
    search_ms, dev_ms, total_matches = 0.0, 0.0, 0
    t0 = time.perf_counter()
    for _ in range(steps):
        db.run(b, e, -1, 0.6)
        tm = db.timing()
        tg = time.perf_counter()
        total_matches = gather()          # host-synchronous (the library synchronises its stream): wall clock = device time + launch latency
        gather_ms = 1e3 * (time.perf_counter() - tg)
        search_ms += tm["search_ms"]
        dev_ms += tm["total_ms"] + gather_ms
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = lib.bsfm_kernel_launches() - launches0
    if dump_dir is not None and rank == 0:     # the table of the last timed pass (all ranks' shards when gathered)
        c_last, m_last = db.fetch() if comm is None else db.gathered_fetch()
        dump_outputs(dump_dir, {"pair_counts": c_last, "matches": m_last})
    if dist is not None:
        dist.barrier()
    # e2e: host descriptors (pinned) -> upload -> run -> gather -> table on the host
    keys_pin, _keep_keys = pinned_view(torch, keys)
    # one untimed end-to-end pass first (NCCL sets up its large-message channels on first use, the allocator warms up), then
    # `e2e_steps` timed passes; every pass starts from host descriptors and ends with the whole table on the host
    e2e_steps = max(1, min(steps, 3))
    e2e_wall, e2e_parts, e2e_matches = 0.0, None, 0
    for it in range(1 + e2e_steps):
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        db2 = keymatch.KeyDatabase(keys_pin, key_off, comm=comm)      # N > 1: every rank uploads and prepares 1/N of the images
        t1 = time.perf_counter()
        db2.run(b, e, -1, 0.6)
        t2 = time.perf_counter()
        if comm is not None:
            db2.allgather(comm)
            t3 = time.perf_counter()
            c_host, m_host = db2.gathered_fetch()                    # the whole table on the host of every rank
        else:
            t3 = time.perf_counter()
            c_host, m_host = db2.fetch()
        torch.cuda.synchronize()
        t4 = time.perf_counter()
        db2.close()
        if it > 0:
            e2e_wall += (t4 - t0) / e2e_steps
            e2e_parts = {"database_build_ms": 1e3 * (t1 - t0), "search_ms": 1e3 * (t2 - t1), "table_allgather_ms": 1e3 * (t3 - t2), "fetch_ms": 1e3 * (t4 - t3)}
        e2e_matches = int(m_host.shape[0])
    t = torch.tensor([dev_ms * 1e-3, search_ms * 1e-3, e2e_wall, wall], dtype=torch.float64, device=dev)
    parts_all = [e2e_parts]
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        pt = torch.tensor([e2e_parts[k] for k in ("database_build_ms", "search_ms", "table_allgather_ms", "fetch_ms")], dtype=torch.float64, device=dev)
        gathered = [torch.zeros_like(pt) for _ in range(world)]
        dist.all_gather(gathered, pt)
        parts_all = [dict(zip(("database_build_ms", "search_ms", "table_allgather_ms", "fetch_ms"), [round(float(x), 2) for x in g.tolist()])) for g in gathered]
    dev_s, search_s, e2e_wall, wall = t[0].item(), t[1].item(), t[2].item(), t[3].item()
    npairs = num_images * (num_images - 1) // 2
    dp = float(npairs) * keys_per_image * keys_per_image
    db.close()
    if comm is not None:
        comm.close()
    assert e2e_matches == int(total_matches), (e2e_matches, total_matches)
    return {"desc_pairs_per_s": dp * steps / dev_s, "image_pairs_per_s": npairs * steps / dev_s, "ms_per_pass": 1e3 * dev_s / steps,
            "wall_ms_per_pass": 1e3 * wall / steps, "launches": int(launches), "clocks": clocks,
            "search_kernel_ms_per_pass_max_rank": 1e3 * search_s / steps, "int8_tops_search_kernel": dp * 256 / world / (search_s / steps) / 1e12,
            "e2e_desc_pairs_per_s": dp / e2e_wall, "matches": int(total_matches), "h2d_bytes": int(keys.nbytes), "images": num_images, "keys_per_image": keys_per_image,
            "pairs": npairs, "shard": [int(b), int(e)], "steps": steps, "warmup": warmup, "e2e_breakdown_ms_per_rank": parts_all}


def cpu_baseline_ba2():
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    from bundler_sfm_b200 import synth
    from oracle import loader
    scene = synth.ba_scene(seed=1234, **BA_CFGS["ba2"])
    t0 = time.perf_counter()
    out = loader.run_sfm_oracle(scene)
    dt = time.perf_counter() - t0
    kind = "reference" if loader.ref_sba() is not None else "port"
    return {"value": out["info"][5] / dt, "unit": "LM iterations/s", "cores": 1, "kind": kind,
            "sample": f"one full run_sfm solve of the config ({int(out['info'][5])} LM iterations, {dt:.1f} s), single thread"}


def cpu_baseline_ba3(scene):
    """bounded live sample of the reference on config 3: run_sfm stopped after ONE LM iteration (~40-60 s)"""
    cores = usable_cores()
    res = run_reference_ba3(1, cores, scene)
    if res is None:
        stored = json.load(open(os.path.join(ROOT, "tests", "golden", "ba_config3_ref.json")))
        return {"value": stored["info"][5] / stored["seconds"], "unit": "LM iterations/s", "cores": 8, "kind": "reference",
                "sample": "oracle/_ref not available on this box: stored summary of the full reference solve in the build container "
                          "(tests/golden/ba_config3_ref.json: 20 LM iterations in 835 s, 8 OpenBLAS threads for dpotrf)"}
    ips, dt, kind, its = res
    return {"value": ips, "unit": "LM iterations/s", "cores": cores, "kind": kind,
            "sample": f"the unmodified run_sfm on this scene stopped after {its} LM iteration(s): {dt:.1f} s incl. the initial error evaluation "
                      f"(sba single-threaded, dpotrf on {cores} OpenBLAS threads); stored full solve: 20 iterations in 835 s (tests/golden/ba_config3_ref.json)"}


def cpu_baseline_match(budget_s=12.0):
    """single-thread reference MatchKeys (ANN kd-tree, stock 200-visit cap) on pairs of the workload's image size"""
    from bundler_sfm_b200 import synth
    from oracle import loader
    K = MATCH_CFG["keys_per_image"]
    imgs = synth.sift_like_descriptors(2, K, seed=7)
    ref = loader.ref_match() is not None
    n, t0 = 0, time.perf_counter()
    while True:
        if ref:
            loader.match_pair_ref(imgs[0], imgs[1], 0.6, 200)
        else:
            loader.match_pair_port(imgs[0], imgs[1], 0.6)
        n += 1
        dt = time.perf_counter() - t0
        if dt > budget_s:
            break
    return {"value": n * K * K / dt, "unit": "descriptor-pairs/s", "cores": 1, "kind": "reference" if ref else "port",
            "sample": f"{n} image pairs of {K} x {K} keys through the reference MatchKeys (kd-tree build + 200-visit priority search), "
                      f"{dt:.1f} s, single thread"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "ba", "ba2", "ba3", "match"])
    ap.add_argument("--match-images", type=int, default=MATCH_CFG["num_images"])
    ap.add_argument("--no-side", action="store_true", help="skip the side objects (ba_config2 / match / ba_replicas)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the headline path computed in its last step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.impl == "reference":
        return main_reference(args)

    import torch
    rank, world, local = dist_env()
    dist = None
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist_mod
        dist_mod.init_process_group("nccl", device_id=dev)
        dist = dist_mod
    args.warmup = max(args.warmup, 3)
    peaks = load_peaks()
    wl = pick_workload(args)
    dpk = measure_device_peaks(torch, dev)
    if dpk.get("int8_tops_n256", 0) > 0:
        i8_peak = dpk["int8_tops_n256"]
        i8_src = ("measured on this GPU by a plain tcgen05.mma kind::i8 loop (M128 N256, operands resident in shared memory; "
                  f"N128 tiles reach {dpk.get('int8_tops_n128', 0):.0f}); 2 x bf16 dense of MEASURED_PEAKS.json would be {2.0 * peaks['bf16_tflops']:.0f}")
    else:
        i8_peak = 2.0 * peaks["bf16_tflops"]
        i8_src = "2 x bf16 dense, " + peaks["source"]

    def ba_object(ba, key):
        """the BA fields of a JSON line (headline or side object)"""
        obj = {"metric": METRIC_STR["ba"], "value": ba["value"], "unit": "LM iterations/s", "steps": ba["steps"], "warmup": ba["warmup"],
               "ms_per_step": ba["ms_per_step"], "dtype": "f64",
               "config": {"workload": WORKLOAD_STR[key], **BA_CFGS[key],
                          "note": "N>1 = N independent replicas (BA does not shard); L2 flushed between timed steps (256 MB buffer)", "jacobian": "finite-difference (reference-compatible)", "lm_iterations_per_solve": ba["iterations_per_solve"],
                          "final_rmse_px": ba["rmse"]},
               "e2e": {"value": ba["e2e_value"], "unit": "LM iterations/s", "h2d_bytes_per_step": ba["h2d"], "d2h_bytes_per_step": ba["d2h"]},
               "gpu_launches": ba["launches"], "clocks": ba["clocks"], "ba_phase_ms_one_solve": ba["phase_ms"]}
        if "chol" in ba:
            c = ba["chol"]
            obj["roofline"] = {"bound": "tensor", "achieved": c["trailing_int8_tops"], "peak": i8_peak, "unit": "TOP/s (int8)",
                               "frac": c["trailing_int8_tops"] / i8_peak, "traffic": None,
                               "kernel": "tc_syrk_kernel (tcgen05 kind::i8 int8-slice trailing update of the reduced-camera Cholesky)",
                               "fp64_equivalent_tflops": c["trailing_fp64_equiv_tflops"],
                               "fp64_dgemm_tflops_measured": dpk.get("fp64_dgemm_tflops"),
                               "note": "dominant kernel of the solve; achieved = algorithmic int8 ops (28 slice products x 2 x lower-triangle MACs) / CUDA-event "
                                       "time of its launches in one solve; fp64_equivalent_tflops = the same update counted as fp64 FLOPs, next to this "
                                       "GPU's cuBLAS DGEMM rate; peak = " + i8_src}
            obj["cholesky_kernels"] = c
        else:
            obj["roofline"] = {"bound": "hbm", "achieved": ba["roofline_achieved_gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                               "frac": ba["roofline_achieved_gbs"] / peaks["hbm_gbs"], "traffic": None,
                               "note": "whole LM iteration: algorithmic bytes 0.7 KB/obs + 16(9m)^2 per iteration / device time; latency-bound at this size; peak " + peaks["source"]}
        return obj

    def match_object(match):
        return {"metric": METRIC_STR["match"], "value": match["desc_pairs_per_s"], "unit": "descriptor-pairs/s",
                "steps": match["steps"], "warmup": match["warmup"], "ms_per_step": match["ms_per_pass"], "dtype": "u8",
                "config": {"workload": WORKLOAD_STR["match"], **MATCH_CFG, "note": "descriptors (320 MB) exceed L2"},
                "e2e": {"value": match["e2e_desc_pairs_per_s"], "unit": "descriptor-pairs/s", "h2d_bytes_per_step": match["h2d_bytes"],
                        "d2h_bytes_per_step": match["matches"] * 8},
                "gpu_launches": match["launches"], "clocks": match["clocks"],
                "roofline": {"bound": "tensor", "achieved": match["int8_tops_search_kernel"], "peak": i8_peak, "unit": "TOP/s (int8)",
                             "frac": match["int8_tops_search_kernel"] / i8_peak, "traffic": None,
                             "note": "tcgen05 kind::i8 search kernel per GPU; 256 int8 ops per descriptor pair; peak = " + i8_src},
                "match_detail": match}

    line, cpu = None, None
    if wl in ("ba2", "ba3"):
        from bundler_sfm_b200 import synth
        scene = synth.ba_scene(seed=1234 + rank, **BA_CFGS[wl])
        ba = bench_ba(args, torch, dist, rank, world, dev, wl, steps=args.steps, warmup=args.warmup, scene=scene,
                      dump_dir=args.dump_outputs if rank == 0 else None)
        line = {"n_gpus": world, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic", **ba_object(ba, wl)}
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline_ba3(scene) if wl == "ba3" else cpu_baseline_ba2()
        del scene
        if not args.no_side:
            if wl == "ba3":
                side = bench_ba(args, torch, dist, rank, world, dev, "ba2", steps=min(args.steps, 10), warmup=3)
                line["ba_config2"] = ba_object(side, "ba2")
                if rank == 0 and world == 1 and not args.no_cpu_baseline:
                    line["ba_config2"]["cpu_baseline"] = cpu_baseline_ba2()
            m = bench_match(args, torch, dist, rank, world, dev, args.match_images, MATCH_CFG["keys_per_image"], steps=max(1, min(args.steps, 3)), warmup=1)
            line["match"] = match_object(m)
    else:
        # the headline of this workload: EXACTLY --steps timed passes behind --warmup (>= 3) untimed ones (a pass is 0.05-0.35 s)
        m = bench_match(args, torch, dist, rank, world, dev, args.match_images, MATCH_CFG["keys_per_image"], steps=max(1, args.steps), warmup=args.warmup,
                        dump_dir=args.dump_outputs)
        line = {"n_gpus": world, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "data": "synthetic", **match_object(m)}
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline_match()
        if not args.no_side:
            side = bench_ba(args, torch, dist, rank, world, dev, "ba2", steps=min(args.steps, 10), warmup=3)
            line["ba_replicas"] = {"scaling": "weak", **ba_object(side, "ba2")}

    if rank == 0:
        # key order of the contract first
        head = {k: line[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                                     "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline")}
        head.update({k: v for k, v in line.items() if k not in head})
        if cpu is not None:
            head["cpu_baseline"] = cpu
        head["measured_peaks_this_run"] = dpk
        print(json.dumps(head), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
