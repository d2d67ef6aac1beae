#!/usr/bin/env python
"""Benchmark of the SPART forward hot path (BASELINE.json metric: simulations / second).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|3|4|5] [--impl ours|reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic parameter sets.  The headline line is
BASELINE.json configs[1] (`--config 2`, the default): 1M-sample PROSPECT-5D + SAILH look-up table,
Sentinel2A-MSI bands, fixed geometry (sza 40, vza 0, raa 0), FP64; every rank processes its own 1M-sample
shard (weak scaling, no data-path collective), the timed region is bracketed by a barrier + synchronize and
the reported time is the max over ranks.  The other BASELINE configurations ride on the same line under
`configs` (value, roofline fraction, e2e each): 3 = 1M PROSPECT-PRO + random angles on LANDSAT8-OLI (weak),
4 = 10M samples on the 2001-band full-spectrum sensor (strong: 10M / N per rank, chunked output buffer),
5 = 100M samples for Sentinel-2A + -2B (strong: 100M / N per rank, FP64 and FP32, chunked, gathered).

Keys of the JSON line:
  value              whole-job simulations/s with parameters already resident in HBM (compute only)
  value_with_gather  N > 1: the same step followed by its only collective, the gather of every rank's
                     [n, nb, 3] result on rank 0, issued chunk by chunk on a side stream so that chunk i
                     travels while chunk i + 1 is computed; verified on rank 0 against a recomputation of
                     every rank's shard from its seed.  `gather` lists the variants (full / compact / FP32)
                     with the NVLink GB/s into rank 0.
  e2e                the same metric through the public host-buffer API (run_batch_params on pinned host
                     arrays, broadcast rows, compact result): H2D of the parameters and D2H of the result
                     inside the timed region.  e2e_variants: full [n, nb, 3] result, pageable NumPy arrays,
                     float32 I/O.
  roofline           the dominant kernel against the FP64 pipe (the path is FP64-arithmetic bound, ~20 flop/B);
                     `peak` is a DFMA-chain micro-benchmark measured live in this run, `frac_clock_peak` uses
                     148 SM x 64 DFMA/clk x 2 x the SM clock; `step_frac` is the share-weighted whole step.
                     roofline_hbm gives the same kernel against the measured HBM copy bandwidth,
                     roofline_fp32 the FP32 mode against the measured FFMA peak.
  cpu_baseline       the UNMODIFIED reference (oracle/_ref, SPART(...).run() per sample, one fresh object
                     each, all host cores) on a bounded sample; the NumPy oracle port's rate is kept beside it.

--dump-outputs DIR writes, after the timed steps of the headline config, the [rows, nb, 3] FP64 band results
(R_TOC, R_TOA, L_TOA) its last step left in each sensor's output buffer as DIR/bands_<sensor>.npy (rank 0; for
the chunked configs 4 / 5 the buffer holds the last chunk).  The parameters are generated from fixed seeds, so
the same arguments give the same inputs on every run and two builds can be compared output for output.  The
JSON line's `dump_outputs` key records the files, their shapes and which samples they hold.
"""
import argparse
import json
import multiprocessing as mp
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "spart-python_b200"))

METRIC = "SPART simulations/sec (full RT + SRF)"
ROW = dict(CDM=1, PROT=7, CBC=8, SMC=13, FILM=14, SZA=19, VZA=20, RAA=21)

# BASELINE.json configs[1..4].  bcast: parameter rows that are constant over the batch (broadcast rows)
CONFIGS = {
    2: dict(sensors=["Sentinel2A-MSI"], n=1_000_000, scaling="weak", bcast=(7, 8, 13, 14, 19, 20, 21),
            workload="configs[1]: 1M-sample PROSPECT-5D+SAILH LUT, Sentinel2A-MSI (13 bands), fixed geometry, FP64"),
    3: dict(sensors=["LANDSAT8-OLI"], n=1_000_000, scaling="weak", bcast=(1, 13, 14),
            workload="configs[2]: 1M-sample PROSPECT-PRO (CBC/PROT) LUT, random sun/view angles, LANDSAT8-OLI (9 bands)"),
    4: dict(sensors=["SYNTH2001"], n=10_000_000, scaling="strong", bcast=(7, 8, 13, 14, 19, 20, 21), chunk=32768,
            workload="configs[3]: 10M-sample full 1 nm 400-2400 nm R_TOC/R_TOA/L_TOA (2001-band synthetic sensor), "
                     "sharded, output buffer reused per 32768-sample chunk"),
    5: dict(sensors=["Sentinel2A-MSI", "Sentinel2B-MSI"], n=100_000_000, scaling="strong",
            bcast=(7, 8, 13, 14, 19, 20, 21), chunk=1 << 20,
            workload="configs[4]: 100M-sample Sentinel2A+2B retrieval LUT (26 bands), sharded, output buffer reused "
                     "per 1Mi-sample chunk, gathered on rank 0"),
}
KERNELS = ("lidf_kernel", "geometry_kernel", "band_kernel")
DUMP_BYTES = 48 << 20      # --dump-outputs: larger outputs are reduced to a fixed, seeded sample of rows


def kernel_source_sha():
    """Identity of the build the executed-flop counts in profiles/flop_per_sample.json belong to: a
    hash of the SASS of the band-path kernels; falls back to a hash of the CUDA sources without cuobjdump."""
    import hashlib
    import re
    import shutil
    import subprocess
    h = hashlib.sha256()
    lib = ROOT / "spart-python_b200" / "spart_b200" / "lib" / "libspart_b200.so"
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    try:
        txt = subprocess.run([cuobjdump, "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
        keep = False
        for line in txt.splitlines():
            m = re.search(r"Function : (\S+)", line)
            if m:
                keep = bool(re.search(r"lidf_kernel|geometry_kernel|band_kernel", m.group(1)))
            if keep:
                h.update(re.sub(r"/\*[0-9a-f]{16}\*/", "", line).encode())     # drop the encoding column
        return "sass:" + h.hexdigest()[:16]
    except Exception:
        for f in sorted((ROOT / "spart-python_b200" / "csrc").glob("*")):
            if f.suffix in (".cu", ".cuh", ".h"):
                h.update(f.read_bytes())
        return "src:" + h.hexdigest()[:16]


def load_flop_counts():
    """profiles/flop_per_sample.json: executed FP64 flop per simulation (FMA = 2) per kernel and config,
    from ncu's smsp__sass_thread_inst_executed_op_{dadd,dmul,dfma}_pred_on (tools/collect_profiles.sh);
    'fp32' holds FP32 flop + 16 x MUFU per simulation of the FP32 mode.  Returns (counts, note)."""
    p = ROOT / "profiles" / "flop_per_sample.json"
    if not p.exists():
        return {}, "no profiles/flop_per_sample.json"
    d = json.loads(p.read_text())
    sha = d.pop("src_sha", None)
    note = None
    if sha != kernel_source_sha():
        note = f"flop counts measured on kernel build {sha}, current build {kernel_source_sha()}"
    return d, note


# ----------------------------------------------------------------------------- helpers
def synthetic_params_torch(n, config, seed, device, dtype=None):
    """Synthetic parameter block [27, n] generated on the device (distributions of SURVEY.md section
    8(d); same ranges as oracle.synthetic_params)."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    u = lambda lo, hi: torch.rand(n, generator=g, device=device, dtype=torch.float64) * (hi - lo) + lo
    P = torch.empty((27, n), dtype=torch.float64, device=device)
    P[0] = u(5, 80); P[1] = u(0.002, 0.02); P[2] = u(0.005, 0.05); P[3] = u(0, 0.5)
    P[4] = u(1, 25); P[5] = u(0, 10); P[6] = u(1, 3); P[7] = 0.0; P[8] = 0.0
    P[9] = u(0.2, 0.8); P[10] = u(0, 25); P[11] = u(90, 115)
    smp = u(5, 55)
    dry = u(0, 1) < 0.05
    P[12] = torch.where(dry, u(0, 5), smp); P[13] = 25.0; P[14] = 0.015
    P[15] = u(0.1, 8); P[16] = u(-0.5, 0.5); P[17] = u(-0.5, 0.5); P[18] = u(0.01, 0.2)
    P[19] = 40.0; P[20] = 0.0; P[21] = 0.0
    P[22] = u(0.05, 0.6); P[23] = u(0.25, 0.45); P[24] = u(0.5, 4); P[25] = u(900, 1030)
    P[26] = torch.randint(1, 366, (n,), generator=g, device=device).to(torch.float64)
    if config == 3:      # PROSPECT-PRO leaves, random sun / view angles
        P[1] = 0.0
        P[7] = u(0, 0.003)
        P[8] = u(0, 0.01)
        P[19], P[20], P[21] = u(0, 65), u(0, 40), u(0, 180)
    return P if dtype is None else P.to(dtype)


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML from before the warm-up to the end of the GPU legs;
    the summary uses the samples that fall into the marked (timed) windows."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        self.windows, self.error = [], None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            }
            while not self.stop_flag:
                t = time.perf_counter()
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((t, mhz, tuple(name for bit, name in names.items() if r & bit)))
                time.sleep(0.001)
        except Exception as e:  # NVML missing: report that instead of failing the bench
            self.error = f"nvml_unavailable:{type(e).__name__}"

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def summary(self):
        inside = [s for s in self.samples if any(a <= s[0] <= b for a, b in self.windows)]
        mhz = sorted(s[1] for s in inside)
        reasons = sorted({r for s in inside for r in s[2]})
        if self.error:
            reasons.append(self.error)
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(mhz),
                "window": "the timed K steps of the headline config plus a 0.3 s continuation of the same loop"}


# ------------------------------------------------------------------- CPU baselines
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def _oracle_worker(args):
    n, seed, config, sensor = args
    sys.path.insert(0, str(ROOT / "oracle"))
    import spart_oracle as so
    P = so.synthetic_params(n, config, seed=seed)
    out = so.spart_bands(P, sensor)
    return float(out[0, 0, 0])


def time_oracle(total, cores, config=2, sensor="Sentinel2A-MSI", chunk=512, pool=None):
    """Times the NumPy oracle port over `total` samples split into `chunk`-sample tasks on `cores`
    worker processes; returns (simulations/s, samples actually run)."""
    tasks = [(chunk, 1000 + i, config, sensor) for i in range(max(1, total // chunk))]
    own = pool is None
    if own:
        pool = mp.get_context("fork").Pool(cores)
        pool.map(_oracle_worker, [(8, 1, config, sensor)] * cores)           # import + table load outside timing
    t0 = time.perf_counter()
    pool.map(_oracle_worker, tasks, chunksize=1)
    dt = time.perf_counter() - t0
    if own:
        pool.close()
    return len(tasks) * chunk / dt, len(tasks) * chunk


REF_DIR = ROOT / "oracle" / "_ref"        # installed by build() (tools/install_reference.py)


def reference_available():
    return (REF_DIR / "SPART" / "SPART.py").exists()


def _reference_worker(args):
    """One process of the reference arm: the unmodified reference's own per-sample loop -- five fresh
    parameter objects and a fresh SPART object per sample, run() (SPART.py:162-269)."""
    seeds, config, sensor = args
    if str(REF_DIR) not in sys.path:
        sys.path.insert(0, str(REF_DIR))
    sys.path.insert(1, str(ROOT / "oracle"))
    import contextlib
    import io
    import warnings
    import numpy as np
    import SPART
    import spart_oracle as so       # only its seeded parameter generator (the same distribution as the GPU arm)
    assert Path(SPART.__file__).resolve().parent == (REF_DIR / "SPART").resolve()
    f = np.float64
    acc = 0.0
    with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
        warnings.simplefilter("ignore")
        for seed in seeds:
            p = so.synthetic_params(1, config, seed=seed)[0]
            leaf = SPART.LeafBiology(*[f(v) for v in p[0:9]])
            soil = SPART.SoilParameters(*[f(v) for v in p[9:15]])
            canopy = SPART.CanopyStructure(*[f(v) for v in p[15:19]])
            angles = SPART.Angles(*[f(v) for v in p[19:22]])
            atm = SPART.AtmosphericProperties(*[f(v) for v in p[22:26]])
            df = SPART.SPART(soil, leaf, canopy, atm, angles, sensor, int(p[26])).run()
            acc += float(df["R_TOC"].iloc[0])
    return acc


def time_reference(per_core, cores, config=2, sensor="Sentinel2A-MSI", pool=None, seed0=5000):
    """Times SPART(...).run() of the unmodified reference over per_core * cores samples on `cores`
    processes; returns (simulations/s, samples run)."""
    own = pool is None
    if own:
        pool = mp.get_context("fork").Pool(cores)
        pool.map(_reference_worker, [([1], config, sensor)] * cores)         # imports + pickles outside timing
    tasks = [([seed0 + c * per_core + i for i in range(per_core)], config, sensor) for c in range(cores)]
    t0 = time.perf_counter()
    pool.map(_reference_worker, tasks, chunksize=1)
    dt = time.perf_counter() - t0
    if own:
        pool.close()
    return per_core * cores / dt, per_core * cores


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on all host cores, on the
    headline config's synthetic distribution; each step is a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    sensor = cfg["sensors"][0] if cfg["sensors"][0] != "SYNTH2001" else "Sentinel2A-MSI"
    cores = host_cores()
    real = reference_available()
    pool = mp.get_context("fork").Pool(cores)
    if real:
        # ~0.46 s per sample and core: keep the whole run (warm-up + steps) around a minute
        per_core = max(1, min(4, int(60.0 / (0.5 * (args.steps + args.warmup)))))
        pool.map(_reference_worker, [([1], args.config, sensor)] * cores)
        step = lambda i: time_reference(per_core, cores, args.config, sensor, pool=pool, seed0=9000 + 1000 * i)
        kind, per_step = "reference", per_core * cores
        sample = (f"{per_step} samples/step ({per_core} per core) of the same synthetic distribution through the "
                  f"unmodified reference (oracle/_ref: fresh LeafBiology / SoilParameters / CanopyStructure / Angles / "
                  f"AtmosphericProperties / SPART object per sample, run()), {cores} processes")
    else:
        per_step = 512 * cores * 2
        pool.map(_oracle_worker, [(8, 1, args.config, sensor)] * cores)
        step = lambda i: time_oracle(per_step, cores, args.config, sensor, pool=pool)
        kind = "port"
        sample = (f"{per_step} samples/step, NumPy oracle port (oracle/spart_oracle.py) in {cores} processes; "
                  "oracle/_ref is missing (build() installs it where the reference checkout of BASELINE.json is readable)")
    for i in range(args.warmup):
        step(-1 - i)
    t0 = time.perf_counter()
    done = 0
    for i in range(args.steps):
        _, n = step(i)
        done += n
    dt = time.perf_counter() - t0
    pool.close()
    value = done / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value,
        "unit": "simulations/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["workload"], "samples_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": "simulations/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "simulations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ our arm
class Ctx:
    """Per-process state of the GPU arm."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import spart_b200
        self.torch, self.dist, self.sb, self.args = torch, dist, spart_b200, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        # keep this rank (and the pinned host buffers it first-touches) on the CPUs next to its GPU;
        # the original affinity is restored before the CPU baseline leg
        self.full_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
        try:
            import pynvml
            pynvml.nvmlInit()
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(self.local))
        except Exception:
            pass
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        self.eng = spart_b200.default_engine(self.dev)
        self.flops, self.flop_note = load_flop_counts()
        self.peaks = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, warmup, sampler=None):
        """W untimed + exactly K timed calls of fn between barrier + synchronize, CUDA events on the
        launching stream, max over ranks -> ms per step."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        t1 = time.perf_counter()
        if sampler is not None:
            sampler.mark(t0, t1)
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps

    def sensor(self, name):
        return self.sb.synthetic_fullspectrum_sensorinfo() if name == "SYNTH2001" else name

    def seed(self, config, rank=None):
        return 20261018 + config + 7919 * (self.rank if rank is None else rank)


def rooflines(cx, tag, kern_ms, n_launch, step_ms, nb_total, cfg_bytes):
    """Roofline entries of one configuration from the per-kernel CUDA-event times (ms per launch set)."""
    peaks = cx.peaks
    flop = cx.flops.get(tag) or {}
    clock_peak = 148 * 64 * 2 * 1.965e9 / 1e12         # 148 SMs x 64 DFMA/clk x 2 flop x max SM clock
    dominant = max(kern_ms, key=kern_ms.get)
    per = {}
    for k in KERNELS:
        f = flop.get(k)
        per[k] = (f * n_launch / (kern_ms[k] * 1e-3) / 1e12 / peaks["fp64_tflops"]) if (f and kern_ms[k] > 0) else None
    tot_flop = sum(flop.get(k, 0.0) for k in KERNELS)
    tot_ms = sum(kern_ms.values())
    ach = (flop.get(dominant, 0.0) * n_launch / (kern_ms[dominant] * 1e-3) / 1e12) or None
    rl = {
        "kernel": dominant, "bound": "fp64", "achieved": ach, "peak": peaks["fp64_tflops"], "unit": "TFLOP/s",
        "frac": (ach / peaks["fp64_tflops"]) if ach else None,
        "frac_clock_peak": (ach / clock_peak) if ach else None, "clock_peak": clock_peak,
        "traffic": None,
        "peak_source": "DFMA-chain micro-benchmark measured live in this run (spart_measure_peaks); clock_peak = "
                       "148 SM x 64 DFMA/clk x 2 x 1.965 GHz",
        "kernel_ms": kern_ms, "kernel_frac": per, "share_of_step": kern_ms[dominant] / step_ms,
        "step_frac": (tot_flop * n_launch / (tot_ms * 1e-3) / 1e12 / peaks["fp64_tflops"]) if tot_flop else None,
        "step_frac_clock_peak": (tot_flop * n_launch / (tot_ms * 1e-3) / 1e12 / clock_peak) if tot_flop else None,
        # the FP64 issue ceiling of dependent chains on register operands (FP64 instructions of different warps
        # issue every 3 cycles on the B200): measured live, ~2/3 of the DFMA-chain peak
        "register_chain_peak": peaks.get("fp64_register_chain_tflops"),
        "frac_register_chain_peak": (ach / peaks["fp64_register_chain_tflops"])
        if (ach and peaks.get("fp64_register_chain_tflops")) else None,
        "step_frac_register_chain_peak": (tot_flop * n_launch / (tot_ms * 1e-3) / 1e12 / peaks["fp64_register_chain_tflops"])
        if (tot_flop and peaks.get("fp64_register_chain_tflops")) else None,
        "flop_per_simulation": {k: flop.get(k) for k in KERNELS}, "flop_count_note": cx.flop_note,
        "kernel_build": kernel_source_sha(),
    }
    mp_file = ROOT / "MEASURED_PEAKS.json"
    hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
    if mp_file.exists():
        hbm_peak, hbm_src = float(json.loads(mp_file.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    nbytes = cfg_bytes[dominant] * n_launch
    ach_gb = nbytes / (kern_ms[dominant] * 1e-3) / 1e9
    rl_hbm = {"kernel": dominant, "bound": "hbm", "achieved": ach_gb, "peak": hbm_peak, "unit": "GB/s",
              "frac": ach_gb / hbm_peak, "traffic": None, "peak_source": hbm_src,
              "algorithmic_bytes_per_simulation": cfg_bytes}
    tr = ROOT / "profiles" / "dram_traffic.json"
    if tr.exists():
        t = json.loads(tr.read_text()).get(tag) or {}
        rl["traffic"] = rl_hbm["traffic"] = t.get(dominant)
    return rl, rl_hbm


def algorithmic_bytes(nb, n_rows_read):
    """HBM bytes per simulation and kernel: leaf angles read 2 parameter rows and write 12 cumulative
    values; geometry reads those 12 + its parameter rows and writes the 32-double record; the band kernel
    reads the record + its parameter rows and writes nb x 3 results (broadcast rows cost nothing)."""
    return {"lidf_kernel": (2 + 12) * 8, "geometry_kernel": (12 + min(n_rows_read, 12) + 32) * 8,
            "band_kernel": (32 + min(n_rows_read, 12)) * 8 + nb * 3 * 8}


def measure_resident(cx, config, steps, warmup, sampler=None, precision="fp64", n=None):
    """Resident-input throughput of one configuration on this rank's shard; returns a dict with value,
    ms_per_step and per-kernel times.  Configs 4 / 5 evaluate their shard in chunks that reuse one output
    buffer (their full output would be 480 GB / 62 GB)."""
    torch, eng = cx.torch, cx.eng
    cfg = CONFIGS[config]
    sensors = [cx.sensor(s) for s in cfg["sensors"]]
    nbs = [eng.sensor(s)[1].n_bands for s in sensors]
    n_rank = n or (cfg["n"] if cfg["scaling"] == "weak" else cfg["n"] // cx.world)
    chunk = min(cfg.get("chunk", n_rank), n_rank)
    params = synthetic_params_torch(n_rank, config, cx.seed(config), cx.dev)
    outs = [torch.empty((chunk, nb, 3), dtype=torch.float64, device=cx.dev) for nb in nbs]
    ws = eng.workspace(chunk)
    bounds = [(lo, min(lo + chunk, n_rank)) for lo in range(0, n_rank, chunk)]

    def step():
        for lo, hi in bounds:
            p = params[:, lo:hi]
            for i, s in enumerate(sensors):
                eng.forward_bands(p, s, out=outs[i][:hi - lo], precision=precision, broadcast_rows=cfg["bcast"],
                                  reuse_record=i > 0, workspace=ws)

    prof_sensor = sensors[0]
    for _ in range(warmup):
        step()
    cx.barrier()
    for s in sensors:
        eng.profile_enable(s, True)
    launches0 = eng.launch_count()
    ms = cx.timed(step, steps, 0, sampler)
    launches = eng.launch_count() - launches0
    kern = {k: 0.0 for k in KERNELS}
    calls = 0
    for s in sensors:
        pr = eng.profile_read(s)
        eng.profile_enable(s, False)
        kern["lidf_kernel"] += pr["lidf_ms"]
        kern["geometry_kernel"] += pr["geometry_ms"]
        kern["band_kernel"] += pr["band_ms"]
        calls += pr["calls"]
    kern = {k: v / steps for k, v in kern.items()}          # ms per step on this rank
    total = n_rank * cx.world
    res = {"value": total / (ms * 1e-3), "ms_per_step": ms, "samples_per_gpu_per_step": n_rank, "chunk": chunk,
           "kernel_ms": kern, "gpu_launches": launches, "bands": sum(nbs), "scaling": cfg["scaling"],
           "workload": cfg["workload"]}
    return res, params, outs, (prof_sensor, nbs)


def dump_outputs(directory, names, outs, n, chunk):
    """--dump-outputs: the rows of each sensor's output buffer that the last step wrote (the last chunk starts at
    sample (n - 1) // chunk * chunk) as float64 <directory>/bands_<sensor>.npy; beyond DUMP_BYTES in all, a
    sorted row sample drawn with a fixed seed, so that every run with the same arguments keeps the same rows.
    Returns what was written, for the JSON line."""
    import numpy as np
    import torch
    directory = Path(directory)
    directory.mkdir(parents=True, exist_ok=True)
    rows = n - (n - 1) // chunk * chunk
    files, sampled = {}, False
    for name, o in zip(names, outs):
        o = o[:rows]
        keep = DUMP_BYTES // len(outs) // (o[0].numel() * o.element_size())
        if keep < rows:
            sampled = True
            idx = np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
            o = o[torch.from_numpy(idx).to(o.device)]
        np.save(directory / f"bands_{name}.npy", o.cpu().numpy())
        files[f"bands_{name}.npy"] = list(o.shape)
    return {"dir": str(directory), "files": files, "rank": 0, "first_sample": n - rows, "samples": rows,
            "rows": "sorted sample numpy.random.default_rng(0).choice(samples, rows, replace=False)" if sampled
                    else "all"}


def measure_e2e(cx, config, params_dev, n, variant, steps=5, precision="fp64"):
    """End to end through run_batch_params on host buffers: H2D of the parameters + kernels + D2H of the
    result inside the timed region.  variant: 'compact' (pinned, broadcast rows, compact result),
    'full' (pinned, [n, nb, 3]), 'pageable' (plain NumPy arrays, full result), 'f32' (pinned float32 I/O,
    compact)."""
    import numpy as np
    torch, sb = cx.torch, cx.sb
    cfg = CONFIGS[config]
    sensors = [cx.sensor(s) for s in cfg["sensors"]]
    nbs = [cx.eng.sensor(s)[1].n_bands for s in sensors]
    f32 = variant == "f32"
    compact = variant in ("compact", "f32")
    dt = torch.float32 if f32 else torch.float64
    host_in = torch.empty((27, n), dtype=dt)
    if variant != "pageable":
        host_in = host_in.pin_memory()
    host_in.copy_(params_dev[:, :n].to(dt))
    outs = []
    for nb in nbs:
        o = torch.empty(n * nb * 2 + n if compact else (n, nb, 3), dtype=dt)
        outs.append(o if variant == "pageable" else o.pin_memory())
    src = host_in.numpy() if variant == "pageable" else host_in
    dst = [o.numpy() if variant == "pageable" else o for o in outs]
    prec = "fp32" if f32 else precision

    def step():
        for s, o in zip(sensors, dst):
            sb.run_batch_params(src, s, out=o, precision=prec, broadcast_rows=cfg["bcast"], compact=compact)

    for _ in range(2):
        step()
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    dt_s = cx.max_over_ranks(time.perf_counter() - t0)
    esz = 4 if f32 else 8
    rows = 27 - len(cfg["bcast"])
    h2d = (rows * n + len(cfg["bcast"])) * esz * len(sensors)
    d2h = sum((n * nb * 2 + n if compact else n * nb * 3) * esz for nb in nbs)
    return {"value": cx.world * n * steps / dt_s, "unit": "simulations/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "steps": steps, "samples_per_gpu_per_step": n,
            "api": f"spart_b200.run_batch_params({'pageable NumPy' if variant == 'pageable' else 'pinned host'} "
                   f"{'float32' if f32 else 'float64'} [27,n], broadcast_rows={list(cfg['bcast'])}, compact={compact}"
                   f"{', precision=fp32' if f32 else ''}) -> host result"}, dst


def measure_copy_ceiling(cx, h2d_bytes, d2h_bytes, pieces=16, reps=6):
    """What the host link of this box sustains for the bytes of one end-to-end step, copies only: h2d_bytes from
    and d2h_bytes into pinned host memory, both directions at once on two streams, in `pieces` pieces each.  No
    implementation of the step can be faster; `e2e.value / ceiling` says how close the pipeline gets."""
    torch = cx.torch
    hin = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    hout = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    din = torch.empty(h2d_bytes, dtype=torch.uint8, device=cx.dev)
    dout = torch.empty(d2h_bytes, dtype=torch.uint8, device=cx.dev)
    s1, s2 = torch.cuda.Stream(device=cx.dev), torch.cuda.Stream(device=cx.dev)

    def both():
        a, b = h2d_bytes // pieces, d2h_bytes // pieces
        with torch.cuda.stream(s1):
            for i in range(pieces):
                din[i * a:(i + 1) * a].copy_(hin[i * a:(i + 1) * a], non_blocking=True)
        with torch.cuda.stream(s2):
            for i in range(pieces):
                hout[i * b:(i + 1) * b].copy_(dout[i * b:(i + 1) * b], non_blocking=True)

    best = None
    for r in range(reps + 1):
        torch.cuda.synchronize()
        cx.barrier()
        t0 = time.perf_counter()
        both()
        torch.cuda.synchronize()
        dt = cx.max_over_ranks(time.perf_counter() - t0)
        if r > 0:
            best = dt if best is None else min(best, dt)
    return best


def measure_with_gather(cx, config, params, steps, warmup, variant, n_chunks=4):
    """N > 1: the step followed by the gather of every rank's result on rank 0, chunk-pipelined on a side
    stream (spart_b200.distributed.gather_pipelined) and verified on rank 0.  variant: 'full' (FP64
    [n, nb, 3]), 'compact' (FP64 R_TOC / R_TOA + ET scale), 'f32' (FP32 mode, float32 I/O, compact)."""
    torch, eng = cx.torch, cx.eng
    from spart_b200.distributed import gather_pipelined
    from spart_b200.engine import out_elems
    cfg = CONFIGS[config]
    sensors = [cx.sensor(s) for s in cfg["sensors"]]
    nbs = [eng.sensor(s)[1].n_bands for s in sensors]
    f32 = variant == "f32"
    compact = variant != "full"
    dt = torch.float32 if f32 else torch.float64
    prec = "fp32" if f32 else "fp64"
    P = params.to(dt) if f32 else params
    n = P.shape[1]
    chunk = min(cfg.get("chunk", (n + n_chunks - 1) // n_chunks), n)
    bounds = [(lo, min(lo + chunk, n)) for lo in range(0, n, chunk)]
    # one block per (chunk, sensor): every block is gathered as soon as its kernels are done
    blocks, plan = [], []
    for lo, hi in bounds:
        for i, nb in enumerate(nbs):
            blocks.append(out_elems(hi - lo, nb, compact))
            plan.append((lo, hi, i))
    ws = eng.workspace(chunk)
    total = sum(blocks)
    local = torch.empty(total, dtype=dt, device=cx.dev)
    recv = torch.empty((cx.world, total), dtype=dt, device=cx.dev) if cx.rank == 0 else None

    def compute(c, view):
        lo, hi, i = plan[c]
        nb = nbs[i]
        eng.forward_bands(P[:, lo:hi], sensors[i], out=view if compact else view.view(hi - lo, nb, 3), precision=prec,
                          broadcast_rows=cfg["bcast"], compact=compact, reuse_record=i > 0, workspace=ws)

    def step():
        gather_pipelined(compute, blocks, dt, cx.dev, dst=0, local=local, recv=recv)

    ms = cx.timed(step, steps, warmup)
    # verification: rank 0 recomputes every rank's shard from its seed and compares bit for bit
    ok = None
    if cx.rank == 0:
        ok = True
        for r in range(cx.world):
            Pr = synthetic_params_torch(n, config, cx.seed(config, r), cx.dev)
            Pr = Pr.to(dt) if f32 else Pr
            chk = torch.empty(total, dtype=dt, device=cx.dev)
            off = 0
            for c, e in enumerate(blocks):
                lo, hi, i = plan[c]
                eng.forward_bands(Pr[:, lo:hi], sensors[i], out=chk[off:off + e] if compact else
                                  chk[off:off + e].view(hi - lo, nbs[i], 3), precision=prec, broadcast_rows=cfg["bcast"],
                                  compact=compact, reuse_record=i > 0)
                off += e
            ok = ok and bool(torch.equal(chk, recv[r]))
            del Pr, chk
    nbytes = (cx.world - 1) * total * (4 if f32 else 8)
    return {"value_with_gather": cx.world * n / (ms * 1e-3), "ms_per_step": ms, "bytes_into_rank0_per_step": nbytes,
            "nvlink_gb_per_s_into_rank0": nbytes / (ms * 1e-3) / 1e9, "chunk_samples": chunk, "blocks_per_step": len(blocks),
            "verified_on_rank0": ok, "op": "nccl gather to rank 0 per block on a side stream (gather_pipelined)"}


def measure_retrieval(cx, steps=3):
    """The consumer of config 5 without its 62 GB gather: the look-up table stays sharded (1M entries of 13
    bands per GPU here), 100k observations are searched on every GPU against its own slice and the per-observation
    (cost, index) words are min-reduced with one NCCL all-reduce of 8 bytes per observation
    (spart_b200.lut.nearest_sharded)."""
    torch = cx.torch
    from spart_b200 import lut
    g = torch.Generator(device=cx.dev).manual_seed(77 + cx.rank)
    n_local, m, nb = 1_000_000, 100_000, 13
    L = torch.rand((n_local, nb), generator=g, device=cx.dev, dtype=torch.float32)
    O = torch.rand((m, nb), generator=torch.Generator(device=cx.dev).manual_seed(5), device=cx.dev, dtype=torch.float32)
    if cx.world > 1:
        fn = lambda: lut.nearest_sharded(L, O, index_offset=cx.rank * n_local)
    else:
        fn = lambda: lut.nearest(L, O)
    ms = cx.timed(fn, steps, 2)
    fn_tc = (lambda: lut.nearest_sharded(L, O, index_offset=cx.rank * n_local, method="tensor")) if cx.world > 1 else (
        lambda: lut.nearest(L, O, method="tensor"))
    ms_tc = cx.timed(fn_tc, steps, 2)
    agree = float((fn_tc()[0] == fn()[0]).float().mean().item())
    idx, cost = fn()
    # every rank must hold the same global answer
    same = True
    if cx.world > 1:
        ref = idx.clone()
        cx.dist.broadcast(ref, 0)
        same = bool(torch.equal(ref, idx))
    pairs = float(cx.world) * n_local * m
    return {"ms_per_search": ms, "pairs_per_s": pairs / (ms * 1e-3), "entries_total": cx.world * n_local,
            "observations": m, "bands": nb, "allreduce_bytes": 8 * m if cx.world > 1 else 0,
            "same_result_on_all_ranks": same,
            "tensor_core_variant": {"ms_per_search": ms_tc, "pairs_per_s": pairs / (ms_tc * 1e-3),
                                    "same_entry_as_exact_search": agree,
                                    "note": "3xTF32 mma.sync comparison + exact FP32 re-costing of the winner"},
            "note": "table sharded over the GPUs, never gathered; FP32 SIMT search + ncclMin of packed (cost, index) words"}


def run_ours(args):
    import numpy as np
    cx = Ctx(args)
    torch, eng, world, rank = cx.torch, cx.eng, cx.world, cx.rank
    config = args.config
    cfg = CONFIGS[config]
    sampler = ClockSampler(cx.local)
    sampler.start()
    cx.peaks = eng.measure_peaks()

    # --- headline: resident-input timing of the chosen config --------------------------------------
    res, params, outs, (sensor0, nbs) = measure_resident(cx, config, args.steps, args.warmup, sampler, n=args.n)
    n = res["samples_per_gpu_per_step"]
    nb = res["bands"]
    dump = dump_outputs(args.dump_outputs, cfg["sensors"], outs, n, res["chunk"]) if (args.dump_outputs and
                                                                                    rank == 0) else None
    # keep the same loop busy for another 0.3 s so that the NVML sampler sees the clocks under this load
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < 0.3:
        eng.forward_bands(params[:, :min(n, 1 << 20)], cx.sensor(cfg["sensors"][0]), out=outs[0][:min(n, 1 << 20)],
                          broadcast_rows=cfg["bcast"])
        torch.cuda.synchronize()
    sampler.mark(t0, time.perf_counter())
    tag = f"cfg{config}"
    rl, rl_hbm = rooflines(cx, tag, res["kernel_ms"], n, res["ms_per_step"], nb,
                           algorithmic_bytes(nb, 27 - len(cfg["bcast"])))

    # --- FP32 mode on the same batch ----------------------------------------------------------------
    fp32 = None
    if config in (2, 3):
        s0 = cx.sensor(cfg["sensors"][0])
        out32 = torch.empty_like(outs[0])
        eng.profile_enable(s0, True)
        ms32 = cx.timed(lambda: eng.forward_bands(params, s0, out=out32, broadcast_rows=cfg["bcast"], precision="fp32"),
                        args.steps, args.warmup)
        pr = eng.profile_read(s0)
        eng.profile_enable(s0, False)
        eng.forward_bands(params, s0, out=outs[0], broadcast_rows=cfg["bcast"])
        err32 = float(((out32 - outs[0]).abs() / outs[0].abs()).max().item())
        P32 = params.float()
        o32 = torch.empty(n * nb * 2 + n, dtype=torch.float32, device=cx.dev)
        ms32io = cx.timed(lambda: eng.forward_bands(P32, s0, out=o32, broadcast_rows=cfg["bcast"], precision="fp32",
                                                    compact=True), args.steps, args.warmup)
        k32 = {"geometry_kernel_f32": pr["geometry_ms"] / max(pr["calls"], 1),
               "band_kernel_f32": pr["band_ms"] / max(pr["calls"], 1)}
        f32c = cx.flops.get(f"{tag}_fp32") or {}
        fp32 = {"value": world * n / (ms32 * 1e-3), "unit": "simulations/s", "ms_per_step": ms32,
                "max_rel_err_vs_fp64": err32, "kernel_ms": k32,
                "value_f32_io_compact": world * n / (ms32io * 1e-3), "ms_per_step_f32_io_compact": ms32io}
        if f32c:
            # FP32-mode roofline: executed FP32 flop (FMA = 2) against the measured FFMA peak; the SFU
            # (MUFU) instruction rate against 16 / clk / SM; FP64 flop of the mixed-precision parts
            tot = sum(k32.values()) * 1e-3
            fl = sum(v.get("fp32_flop", 0.0) for v in f32c.values())
            mufu = sum(v.get("mufu", 0.0) for v in f32c.values())
            d64 = sum(v.get("fp64_flop", 0.0) for v in f32c.values())
            fp32["roofline_fp32"] = {
                "bound": "fp32 issue", "achieved": fl * n / tot / 1e12, "peak": cx.peaks["fp32_tflops"], "unit": "TFLOP/s",
                "frac": fl * n / tot / 1e12 / cx.peaks["fp32_tflops"],
                "sfu_frac": mufu * n / tot / (148 * 16 * 1.965e9),
                "fp64_frac": d64 * n / tot / 1e12 / cx.peaks["fp64_tflops"],
                "per_simulation": f32c, "peak_source": "FFMA-chain micro-benchmark measured live in this run"}
        del out32, P32, o32

    # --- N > 1: the step with its gather -------------------------------------------------------------
    gather = None
    if world > 1:
        gather = {}
        for variant in ("full", "compact", "f32"):
            gather[variant] = measure_with_gather(cx, config, params, max(3, min(args.steps, 10)), 3, variant)

    # --- end to end through the public host-buffer API -----------------------------------------------
    e2e_n = n if config in (2, 3) else min(n, 1 << 21 if config == 5 else 1 << 15)
    e2e_steps = max(1, min(args.steps, 5))
    e2e, got = measure_e2e(cx, config, params, e2e_n, "compact", e2e_steps)
    t_copy = measure_copy_ceiling(cx, e2e["h2d_bytes_per_step"], e2e["d2h_bytes_per_step"])
    e2e["copy_only_ceiling"] = {
        "value": cx.world * e2e_n / t_copy, "unit": "simulations/s", "ms_per_step": t_copy * 1e3,
        "frac": e2e["value"] / (cx.world * e2e_n / t_copy),
        "note": "the same bytes moved between pinned host memory and the GPU in both directions at once, 16 pieces "
                "each, no kernels: the host link's ceiling for this step on this box"}
    # same bits as the device path
    chk = eng.forward_bands(params[:, :e2e_n], cx.sensor(cfg["sensors"][0]), broadcast_rows=cfg["bcast"], compact=True)
    assert torch.equal(got[0].to(cx.dev), chk.buf), "host-buffer path disagrees with the device path"
    del chk
    e2e_variants = {}
    for variant in ("full", "pageable", "f32"):
        if config == 4 and variant == "pageable":
            continue
        e2e_variants[variant], _ = measure_e2e(cx, config, params, e2e_n, variant, e2e_steps)
    del got

    # --- the other BASELINE configurations (extra keys of the same line) ---------------------------------
    extras = {}
    if config == 2 and not args.no_extras:
        del params, outs
        torch.cuda.empty_cache()
        for c in (3, 4, 5):
            k = 3 if c in (4, 5) else max(3, min(args.steps, 10))
            r, p, o, _ = measure_resident(cx, c, k, 2)
            nr = r["samples_per_gpu_per_step"]
            r_rl, r_hbm = rooflines(cx, f"cfg{c}", r["kernel_ms"], nr, r["ms_per_step"], r["bands"],
                                    algorithmic_bytes(r["bands"], 27 - len(CONFIGS[c]["bcast"])))
            r["roofline"] = {k2: r_rl[k2] for k2 in ("kernel", "frac", "frac_clock_peak", "step_frac", "kernel_frac",
                                                     "share_of_step", "achieved", "peak", "unit")}
            r["roofline_hbm_frac"] = r_hbm["frac"]
            if c == 4:
                r["output_gb_per_s"] = nr * world * 2001 * 3 * 8 / (r["ms_per_step"] * 1e-3) / 1e9
            if c in (4, 5):       # FP32 mode of the same workload
                r32, _, _, _ = measure_resident(cx, c, 3, 2, precision="fp32")
                r["fp32_mode"] = {"value": r32["value"], "ms_per_step": r32["ms_per_step"]}
            en = nr if c == 3 else (1 << 21 if c == 5 else 1 << 15)
            en = min(en, nr)
            r["e2e"], _ = measure_e2e(cx, c, p, en, "compact", 3)
            r["e2e_f32"], _ = measure_e2e(cx, c, p, en, "f32", 3)
            if world > 1 and c in (3, 5):
                r["gather"] = {v: measure_with_gather(cx, c, p, 3, 2, v) for v in (("compact", "f32") if c == 5
                                                                                   else ("full", "compact", "f32"))}
            extras[str(c)] = r
            del p, o
            torch.cuda.empty_cache()

    retrieval = measure_retrieval(cx) if (config == 2 and not args.no_extras) else None
    sampler.stop_flag = True
    sampler.join(2)
    if rank != 0:
        if world > 1:
            cx.dist.destroy_process_group()
        return

    # --- CPU baseline: the unmodified reference on all host cores, bounded sample --------------------
    if cx.full_affinity is not None:
        os.sched_setaffinity(0, cx.full_affinity)
    cores = host_cores()
    cpu = None
    if not args.no_cpu:
        sensor_name = cfg["sensors"][0] if cfg["sensors"][0] != "SYNTH2001" else "Sentinel2A-MSI"
        port_rate, port_ran = time_oracle(512 * cores * 8, cores, config, sensor_name)
        if reference_available():
            rate, ran = time_reference(48, cores, config, sensor_name)       # ~22 s of reference work per core
            cpu = {"value": rate, "unit": "simulations/s", "cores": cores, "kind": "reference",
                   "sample": f"{ran} samples of the same synthetic distribution through the unmodified reference "
                             f"(oracle/_ref, one fresh SPART object per sample, run()), {cores} processes",
                   "port_value": port_rate,
                   "port_sample": f"{port_ran} samples, NumPy oracle port (oracle/spart_oracle.py), {cores} processes"}
        else:
            cpu = {"value": port_rate, "unit": "simulations/s", "cores": cores, "kind": "port",
                   "sample": f"{port_ran} samples of the same synthetic distribution, NumPy oracle port "
                             f"(oracle/spart_oracle.py), {cores} processes; oracle/_ref is missing"}

    line = {
        "metric": METRIC, "value": res["value"], "unit": "simulations/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["workload"], "samples_per_gpu_per_step": n, "sensor": "+".join(cfg["sensors"]),
                   "bands": nb, "broadcast_rows": list(cfg["bcast"]), "chunk": res["chunk"],
                   "l2": "working set per step (params + workspace + output, >= 0.8 GB) exceeds the 126 MB L2"},
        "e2e": e2e, "e2e_variants": e2e_variants,
        "gpu_launches": res["gpu_launches"],
        "clocks": sampler.summary(),
        "roofline": rl, "roofline_hbm": rl_hbm,
        "cpu_baseline": cpu,
        "peaks": cx.peaks,
        "fp32_mode": fp32,
        "gather": gather,
        "value_with_gather": gather["full"]["value_with_gather"] if gather else None,
        "configs": extras,
        "lut_retrieval": retrieval,
        "dump_outputs": dump,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        cx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json configs[config-1]")
    ap.add_argument("--n", type=int, default=None, help="samples per GPU per step (default: the config's)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs 3/4/5 riding on the default line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the band results of the last timed step of the headline config to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
