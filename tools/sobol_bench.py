#!/usr/bin/env python
"""Cost of a Sobol' sensitivity analysis on the GPU, split into design, forward model and estimator.

The space is bench.py's configuration 2: the 19 continuous rows `bench.synthetic_params_torch` draws are varied
over the same ranges (SMp over the union [0, 55) of its wet and dry draws), PROT = CBC = 0, SMC = 25, film = 0.015,
sun / view angles 40 / 0 / 0 and DOY = 180 are fixed, sensor Sentinel-2A, FP64.  For N = 2^16 and 2^20 base
points (N (d + 2) = 1.4 M and 22 M forward runs) `sensitivity.sobol` runs with its default chunk of 2^15 base
points (688 K samples, 148 MB of parameters and 215 MB of outputs per chunk: above the 126 MB L2).  After a
warm-up call at each N, `reps` repetitions each time
  phases  the loop of `sobol` with CUDA events between design, forward and accumulate of every chunk (+ finish),
          summed over the chunks: ms per phase, and design + estimator as a share of the forward time;
  whole   one `sobol` call, CUDA events around it (host copy of the results included): ms and runs/s.
Card name and power limit are read in the same process.

    python tools/sobol_bench.py --out DIR        -> DIR/sobol.json
"""
import argparse
import json
import statistics
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT / "spart-python_b200", ROOT / "tools"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

from spart_b200 import default_engine, sensitivity     # noqa: E402
from soil_library_bench import device_info              # noqa: E402

SENSOR = "Sentinel2A-MSI"
VARY = {"Cab": (5, 80), "Cdm": (0.002, 0.02), "Cw": (0.005, 0.05), "Cs": (0, 0.5), "Cca": (1, 25), "Cant": (0, 10),
        "N": (1, 3), "B": (0.2, 0.8), "lat": (0, 25), "lon": (90, 115), "SMp": (0, 55), "LAI": (0.1, 8),
        "LIDFa": (-0.5, 0.5), "LIDFb": (-0.5, 0.5), "q": (0.01, 0.2), "aot550": (0.05, 0.6), "uo3": (0.25, 0.45),
        "uh2o": (0.5, 4), "Pa": (900, 1030)}
FIXED = {"PROT": 0.0, "CBC": 0.0, "SMC": 25.0, "film": 0.015, "sol_angle": 40.0, "obs_angle": 0.0,
         "rel_angle": 0.0, "DOY": 180.0}
CHUNK = 2 ** 15


def space():
    base = np.zeros(27)
    for k, v in FIXED.items():
        base[sensitivity.ROW_NAMES.index(k)] = v
    return sensitivity.ParameterSpace(base, VARY)


def phases(sp, n):
    """The loop of `sobol` with an event after each phase; returns summed ms (design, forward, estimator)."""
    eng = default_engine()
    d = sp.d
    fwd = lambda p: eng.forward_bands(p, SENSOR, broadcast_rows=sp.broadcast_rows)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    marks = []
    torch.cuda.synchronize()
    ref = fwd(sp.design(1)).reshape(d + 2, -1)
    acc = sensitivity._new_acc(ref.shape[1], d, ref.device)
    for c0 in range(0, n, CHUNK):
        m = min(CHUNK, n - c0)
        e = [ev() for _ in range(4)]
        e[0].record()
        P = sp.design(m, first=c0)
        e[1].record()
        F = fwd(P)
        e[2].record()
        sensitivity._accumulate(F, m, d, ref, acc)
        e[3].record()
        marks.append(e)
        del P, F
    e = [ev(), ev()]
    e[0].record()
    sensitivity._finish(acc, ref, n, d)
    e[1].record()
    torch.cuda.synchronize()
    des = sum(a.elapsed_time(b) for a, b, _, _ in marks)
    fw = sum(b.elapsed_time(c) for _, b, c, _ in marks)
    est = sum(c.elapsed_time(dd) for _, _, c, dd in marks) + e[0].elapsed_time(e[1])
    return des, fw, est


def whole(sp, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    sensitivity.sobol(sp, SENSOR, n, chunk=CHUNK)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "sobol_bench measures on the GPU"
    torch.cuda.set_device(0)
    info = device_info()
    print(json.dumps(info), flush=True)
    sp = space()
    res = {"card": info, "sensor": SENSOR, "precision": "fp64", "d": sp.d, "chunk": CHUNK,
           "varied": list(sp.names), "fixed": FIXED, "sizes": {}}
    for n in (2 ** 16, 2 ** 20):
        whole(sp, n)                                  # warm-up of every shape the timed windows use
        phases(sp, n)
        ph = [phases(sp, n) for _ in range(args.reps)]
        wh = [whole(sp, n) for _ in range(args.reps)]
        des, fw, est = (statistics.median(x[i] for x in ph) for i in range(3))
        runs = n * (sp.d + 2)
        w = statistics.median(wh)
        r = {"base_points": n, "forward_runs": runs, "design_ms": des, "forward_ms": fw,
             "accumulate_finish_ms": est, "design_share_of_forward": des / fw, "estimator_share_of_forward": est / fw,
             "design_plus_estimator_share_of_forward": (des + est) / fw,
             "forward_ns_per_run": 1e6 * fw / runs, "sobol_call_ms": w, "runs_per_s": runs / (w * 1e-3),
             "reps_phases_ms": ph, "reps_sobol_call_ms": wh}
        res["sizes"][str(n)] = r
        print(n, json.dumps(r), flush=True)
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "sobol.json").write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
