#!/usr/bin/env python
"""Cost of per-sample dry-soil spectra (SPART_FLAG_SOIL_LIBRARY) on one GPU.

For each configuration the variants GSV soil (B / lat / lon), one user spectrum (soil_spectrum) and soil
libraries of k = 1, 64, 4096, 65536 spectra with uniformly random per-sample indices run in one process.  Every
variant is warmed up first; then the variants alternate, each repetition timing every variant once:
  band_ms  band-kernel time per call (CUDA events of spart_profile_enable / spart_profile_read)
  call_ms  end-to-end time per forward_bands call on device-resident params (CUDA events around the calls)
Configurations: config 2 (1 Mi samples, Sentinel-2A, one sun / view geometry) in FP64 and FP32, config 3
(1 Mi samples, random geometry, Landsat-8) and the SRF band mode (131 072 samples, TerraAqua-MODIS).

    python tools/soil_library_bench.py --out DIR        -> DIR/soil_library.json
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT / "spart-python_b200", ROOT):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import spart_b200 as sb                      # noqa: E402
from bench import synthetic_params_torch     # noqa: E402

LIBRARY_SIZES = (1, 64, 4096, 65536)
CONFIGS = {
    "cfg2_fp64": dict(sensor="Sentinel2A-MSI", config=2, n=1 << 20, precision="fp64", uniform_geometry=True),
    "cfg2_fp32": dict(sensor="Sentinel2A-MSI", config=2, n=1 << 20, precision="fp32", uniform_geometry=True),
    "cfg3_fp64": dict(sensor="LANDSAT8-OLI", config=3, n=1 << 20, precision="fp64"),
    "srf_fp64": dict(sensor="TerraAqua-MODIS", config=2, n=131072, precision="fp64", band_mode="srf",
                     uniform_geometry=True),
}


def device_info():
    """Name, power limit and max SM clock of cuda:0, read in the same process as the measurement."""
    info = {"device": torch.cuda.get_device_name(0), "power_limit_w": None, "max_sm_clock_mhz": None}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True).stdout
        pw, clk = (x.strip() for x in q.strip().splitlines()[0].split(","))
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(pw), float(clk)
    except Exception as e:                   # keep the measurement; say why the card data is missing
        info["query_error"] = repr(e)
    return info


def synthetic_library(k, seed):
    rng = np.random.default_rng(seed)
    x = np.linspace(0.0, 1.0, 2001)
    a, b = rng.uniform(0.05, 0.2, (k, 1)), rng.uniform(0.1, 0.4, (k, 1))
    return sb.SoilLibrary(a + b * x ** 0.7)


def variants(params, n, libs):
    """name -> (params, soil keyword arguments)."""
    g = torch.Generator(device=params.device).manual_seed(7)
    out = {"gsv": (params, {}), "spectrum": (params, {"soil_spectrum": libs[LIBRARY_SIZES[1]].spectra[0]})}
    for k in LIBRARY_SIZES:
        p = params.clone()
        p[9] = torch.randint(0, k, (n,), generator=g, device=params.device).to(p.dtype)
        out[f"lib{k}"] = (p, {"soil_library": libs[k]})
    return out


def time_variant(eng, cfg, params, soil, out, calls):
    kw = dict(precision=cfg["precision"], band_mode=cfg.get("band_mode", "interp"),
              uniform_geometry=cfg.get("uniform_geometry", False))
    handle, _ = eng.sensor(cfg["sensor"], **soil)
    # band-kernel time
    sb._lib.check(eng.lib.spart_profile_enable(handle, 1), "spart_profile_enable")
    for _ in range(calls):
        eng.forward_bands(params, cfg["sensor"], out=out, **kw, **soil)
    ms = (sb._lib.c_double * sb._lib.NKERNELS)()
    c = sb._lib.c_int64()
    sb._lib.check(eng.lib.spart_profile_read(handle, ms, sb._lib.byref(c)), "spart_profile_read")
    sb._lib.check(eng.lib.spart_profile_enable(handle, 0), "spart_profile_enable")
    band_ms = ms[2] / c.value
    # end-to-end call time, profiling off
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(calls):
        eng.forward_bands(params, cfg["sensor"], out=out, **kw, **soil)
    e1.record()
    e1.synchronize()
    return band_ms, e0.elapsed_time(e1) / calls


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--calls", type=int, default=5, help="calls per timing")
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    torch.cuda.set_device(0)
    eng = sb.default_engine()
    info = device_info()
    print(json.dumps(info), flush=True)
    libs = {k: synthetic_library(k, seed=k) for k in LIBRARY_SIZES}
    res = {"info": info, "reps": args.reps, "calls": args.calls, "library_sizes": list(LIBRARY_SIZES), "configs": {}}
    for name in args.configs.split(","):
        cfg = CONFIGS[name]
        n = cfg["n"]
        params = synthetic_params_torch(n, cfg["config"], seed=11, device=eng.device)
        if cfg["precision"] == "fp32":
            params = params.float()                      # float in, float out (SPART_FLAG_F32_IO)
        var = variants(params, n, libs)
        _, st = eng.sensor(cfg["sensor"])
        out = torch.empty((n, st.n_bands, 3), dtype=params.dtype, device=eng.device)
        for v, (p, soil) in var.items():                 # warm every shape and context
            time_variant(eng, cfg, p, soil, out, 1)
        rows = {v: {"band_ms": [], "call_ms": []} for v in var}
        for _ in range(args.reps):
            for v, (p, soil) in var.items():
                b, c = time_variant(eng, cfg, p, soil, out, args.calls)
                rows[v]["band_ms"].append(b)
                rows[v]["call_ms"].append(c)
        base = np.median(rows["spectrum"]["band_ms"])
        for v in rows:
            rows[v]["band_vs_spectrum"] = float(np.median(rows[v]["band_ms"]) / base)
        res["configs"][name] = {"sensor": cfg["sensor"], "n": n, "precision": cfg["precision"],
                                "band_mode": cfg.get("band_mode", "interp"),
                                "uniform_geometry": cfg.get("uniform_geometry", False), "variants": rows}
        print(name, json.dumps({v: [round(x, 3) for x in r["band_ms"]] + [round(r["band_vs_spectrum"], 4)]
                                for v, r in rows.items()}), flush=True)
        del var, out, params
        torch.cuda.empty_cache()
    res["finished"] = time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime())
    out_dir = Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    (out_dir / "soil_library.json").write_text(json.dumps(res, indent=1) + "\n")
    eng.close()


if __name__ == "__main__":
    main()
