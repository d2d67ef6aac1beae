#!/usr/bin/env python
"""Cost of a retrieval by bounded Levenberg-Marquardt on the GPU, split into the forward model and the rest.

Setup: Sentinel-2A R_TOC, FP64, P = 7 varied rows (Cab, Cw, Cdm, N, LAI, SMp, LIDFa; the other rows fixed, sun /
view angles 40 / 0 / 0), m = 10^5 noise-free observations of random truth, S = 4 starts per observation from
`lut.nearest_k` on a 2^20-entry `space.sample` LUT, default tolerances and chunk (2^16 tracks).  After a warm-up
call on 4096 observations:
  whole    one `invert` call, host clock around it ending in a device synchronise: ms, observations/s, forward
           runs and forward runs/s;
  phases   the same call with stand-ins that record CUDA events around design, forward, step and finish, and
           events around the whole call; "rest_of_call" is the remainder of the call's span: the active lists
           (compaction), the host's read of their size, the time the device waits idle for the next launch after
           that read, and each chunk's state initialisation.  ms per phase summed, and the share of design + step +
           rest_of_call + finish in the forward time.  The design and step spans also hold such idle time: a span
           opens when the host records its first event, and the device may wait there for the launch;
  kernels  design, forward and step on one full chunk (2^16 tracks, all active) run back to back with no host
           synchronisation in between, CUDA events around each, median of 10: the kernels' own cost per
           iteration;
  forward  `forward_bands` alone on one full chunk's batch (2^16 tracks x 8 samples), median of 10: runs/s;
  quality  the fraction recovered to 1e-6 in u, the statuses and the forward calls of the winning tracks.
Card name and power limit are read in the same process.

    python tools/invert_bench.py --out DIR        -> DIR/invert.json
"""
import argparse
import json
import statistics
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT / "spart-python_b200", ROOT / "tools"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

from spart_b200 import default_engine, inversion, lut, sensitivity     # noqa: E402
from soil_library_bench import device_info                              # noqa: E402

SENSOR = "Sentinel2A-MSI"
BASE = np.array([40, 0.01, 0.02, 0.1, 10, 1, 1.5, 0, 0, 0.5, 10, 100, 20, 25, 0.015, 3, -0.35, -0.15, 0.05,
                 40, 0, 0, 0.3, 0.35, 1.5, 1013, 180], dtype=np.float64)
VARY = {"Cab": (5, 80), "Cw": (0.005, 0.05), "Cdm": (0.002, 0.02), "N": (1, 3), "LAI": (0.1, 8), "SMp": (5, 55),
        "LIDFa": (-0.5, 0.5)}


def setup(m, S, n_lut, seed=1):
    sp = sensitivity.ParameterSpace(BASE, VARY)
    eng = default_engine()
    table = sp.sample(n_lut, seed=seed)
    tab = lut.generate(table, SENSOR, column=0)
    rng = np.random.default_rng(seed)
    truth = rng.uniform(0.02, 0.98, (m, sp.d))
    X = np.tile(BASE, (m, 1))
    X[:, sp.rows] = sp.lo + (sp.hi - sp.lo) * truth
    batch = torch.from_numpy(np.ascontiguousarray(X.T)).cuda()
    obs = eng.forward_bands(batch, SENSOR, broadcast_rows=sp.broadcast_rows)[..., 0].contiguous()
    idx, _ = lut.nearest_k(tab, obs.float(), S)
    start = inversion.starts(table, idx, sp)
    del tab, table
    return sp, truth, obs, start


def timed_phases(sp, obs, start):
    eng = default_engine()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    marks = {"design": [], "forward": [], "step": [], "finish": []}
    buf = {}

    def wrap(name, fn):
        def run(*a):
            e0, e1 = ev(), ev()
            e0.record()
            out = fn(*a)
            e1.record()
            marks[name].append((e0, e1))
            return out
        return run

    def design(prob, state, active):
        n = prob.n_tracks * (prob.P + 1)
        if "b" not in buf or buf["b"].shape[1] < n:
            buf["b"] = torch.empty((27, n), dtype=torch.float64, device="cuda")
        return inversion._design(prob, state, active, buf["b"])
    fwd = lambda p: eng.forward_bands(p, SENSOR, broadcast_rows=sp.broadcast_rows)
    torch.cuda.synchronize()
    e0, e1 = ev(), ev()
    e0.record()
    res = inversion.invert(obs, SENSOR, sp, start, design=wrap("design", design), forward=wrap("forward", fwd),
                           step=wrap("step", inversion._step), finish=wrap("finish", inversion._finish))
    e1.record()
    torch.cuda.synchronize()
    ms = {k: sum(a.elapsed_time(b) for a, b in v) for k, v in marks.items()}
    # everything else on the stream: the active lists, the host's read of their size and the gap it leaves
    # before the next launch, and the state initialisation of each chunk
    ms["rest_of_call"] = e0.elapsed_time(e1) - sum(ms.values())
    ms["iterations"] = len(marks["forward"])
    return ms, res


def full_chunk_kernels(sp, obs, start, reps=10):
    """ms of design, forward and step on one full chunk with every track active, queued back to back."""
    eng = default_engine()
    S = start.shape[1]
    mc = 2 ** 16 // S
    P = sp.d
    prob = inversion.Problem(sp.rows, sp.lo, sp.hi, sp.base, np.zeros(0, dtype=np.int32),
                             torch.empty((0, mc), dtype=torch.float64, device="cuda"), obs[:mc].contiguous(), None, S,
                             0, inversion.FTOL, inversion.XTOL, inversion.MAX_ITERATIONS, False, sp.broadcast_rows)
    state0 = inversion.init_state(prob, start[:mc])
    active = torch.arange(mc * S, dtype=torch.int32, device="cuda")
    buf = torch.empty((27, mc * S * (P + 1)), dtype=torch.float64, device="cuda")
    times = {"design": [], "forward": [], "step": []}
    for r in range(reps + 1):
        state = state0.clone()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record()
        batch = inversion._design(prob, state, active, buf)
        e[1].record()
        f = eng.forward_bands(batch, SENSOR, broadcast_rows=sp.broadcast_rows)
        e[2].record()
        inversion._step(prob, f, state, active)
        e[3].record()
        torch.cuda.synchronize()
        if r:                                       # the first round is a warm-up
            for k, (a, b) in zip(times, zip(e, e[1:])):
                times[k].append(a.elapsed_time(b))
    out = {k: statistics.median(v) for k, v in times.items()}
    out["tracks"] = mc * S
    out["design_plus_step_share_of_forward"] = (out["design"] + out["step"]) / out["forward"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles"))
    ap.add_argument("--m", type=int, default=10 ** 5)
    ap.add_argument("--starts", type=int, default=4)
    ap.add_argument("--lut", type=int, default=2 ** 20)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    info = device_info()
    sp, truth, obs, start = setup(a.m, a.starts, a.lut)
    inversion.invert(obs[:4096], SENSOR, sp, start[:4096])                    # warm-up
    torch.cuda.synchronize()
    whole = []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        res = inversion.invert(obs, SENSOR, sp, start)
        torch.cuda.synchronize()
        whole.append((time.perf_counter() - t0) * 1e3)
    runs = int(res.n_forward.sum().item())
    phase = [timed_phases(sp, obs, start)[0] for _ in range(a.reps)]
    med = {k: statistics.median(p[k] for p in phase) for k in phase[0]}
    other = med["design"] + med["step"] + med["rest_of_call"] + med["finish"]
    # forward alone on one full chunk's batch
    eng = default_engine()
    n = (2 ** 16) * (sp.d + 1)
    X = np.tile(BASE, (n, 1))
    X[:, sp.rows] = sp.lo + (sp.hi - sp.lo) * np.random.default_rng(2).uniform(0, 1, (n, sp.d))
    batch = torch.from_numpy(np.ascontiguousarray(X.T)).cuda()
    eng.forward_bands(batch, SENSOR, broadcast_rows=sp.broadcast_rows)
    fw = []
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.forward_bands(batch, SENSOR, broadcast_rows=sp.broadcast_rows)
        e1.record()
        torch.cuda.synchronize()
        fw.append(e0.elapsed_time(e1))
    u = (res.x.cpu().numpy() - sp.lo) / (sp.hi - sp.lo)
    status = res.status.cpu().numpy()
    iters = res.iterations.cpu().numpy()
    out = {
        **info,
        "setup": {"sensor": SENSOR, "column": "R_TOC", "precision": "fp64", "varied": list(sp.names),
                  "m": a.m, "starts": a.starts, "lut_entries": a.lut, "chunk_tracks": 2 ** 16,
                  "ftol": inversion.FTOL, "xtol": inversion.XTOL, "max_iter": inversion.MAX_ITERATIONS},
        "whole_ms": whole, "whole_ms_median": statistics.median(whole),
        "observations_per_s": a.m / statistics.median(whole) * 1e3,
        "forward_runs": runs, "forward_runs_per_s": runs / statistics.median(whole) * 1e3,
        "phases_ms_median": med,
        "full_chunk_kernels_ms_median": full_chunk_kernels(sp, obs, start),
        "non_forward_share_of_forward": other / med["forward"],
        "forward_only_ms_per_chunk_batch": statistics.median(fw), "forward_only_samples": n,
        "forward_only_runs_per_s": n / statistics.median(fw) * 1e3,
        "recovered_1e-6": float((np.abs(u - truth).max(1) <= 1e-6).mean()),
        "recovered_1e-9": float((np.abs(u - truth).max(1) <= 1e-9).mean()),
        "status_counts": {inversion.STATUS_NAMES[i]: int((status == i).sum()) for i in range(6)},
        "winning_track_forward_calls": {"median": float(np.median(iters)), "p99": float(np.quantile(iters, 0.99)),
                                        "max": int(iters.max())},
    }
    Path(a.out).mkdir(parents=True, exist_ok=True)
    (Path(a.out) / "invert.json").write_text(json.dumps(out, indent=2) + "\n")
    print(json.dumps(out, indent=2))


if __name__ == "__main__":
    main()
