#!/usr/bin/env python
"""Throughput of the k-nearest LUT search (spart_lut_topk) against the single-best search (spart_lut_nearest).

The retrieval shape of bench.py: 10^5 observations x 2^20 entries x 13 bands, uniform random FP32 values.  Every
variant is warmed up first; then the variants alternate, each repetition timing every variant once with CUDA events
around `calls` calls (device-resident inputs, outputs allocated by the call as a user sees it):
  search   spart_lut_nearest (lut.nearest) and spart_lut_topk (lut.nearest_k) at k = 1, 10, 32, 50, 128: ms per call and
           pairs/s (pairs = observations x entries)
  merge    spart_lut_topk_merge (lut.merge_k) alone, on the [L][m][k] lists a search at that m leaves (L = its
           slice count), at m = 1, 10^3, 10^5 and k = 10, 128; beside it the whole nearest_k call at that m
  estimate lut.estimate (two moment passes + finish) for P = 27 float64 parameters of the 2^20 entries, k = 10, 50
A torch.profiler pass at the end, outside the timed windows, splits each nearest_k call into the search kernel and
the merge kernel (device times).

    python tools/lut_topk_bench.py --out DIR        -> DIR/lut_topk.json
"""
import argparse
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
for p in (ROOT / "spart-python_b200", ROOT / "tools"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

from spart_b200 import _lib, lut                 # noqa: E402
from soil_library_bench import device_info       # noqa: E402

N, M, NB = 1 << 20, 100_000, 13
KS = (1, 10, 32, 50, 128)


def timed(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / calls


def alternate(variants, reps, calls):
    """name -> list of ms per call, one per repetition; every variant warmed up, then all alternated."""
    for fn in variants.values():
        fn()
    out = {name: [] for name in variants}
    for _ in range(reps):
        for name, fn in variants.items():
            out[name].append(timed(fn, calls))
    return out


def sorted_lists(L, m, k, g):
    """[L, m, k] ascending packed words with positive costs and distinct indices."""
    cost = torch.rand((L, m, k), generator=g, device="cuda").sort(-1).values
    idx = torch.arange(L * k, device="cuda").reshape(L, 1, k).expand(L, m, k)
    return (cost.view(torch.int32).to(torch.int64) << 32) | idx


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=3, help="calls per timing")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    torch.cuda.set_device(0)
    info = device_info()
    print(json.dumps(info), flush=True)
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(77)
    L = torch.rand((N, NB), generator=g, device="cuda")
    O = torch.rand((M, NB), generator=torch.Generator(device="cuda").manual_seed(5), device="cuda")
    res = {"info": info, "shape": {"observations": M, "entries": N, "bands": NB}, "reps": args.reps,
           "calls": args.calls}

    # search: nearest and top-k alternated
    variants = {"nearest": lambda: lut.nearest(L, O)}
    variants.update({f"topk_k{k}": (lambda k=k: lut.nearest_k(L, O, k)) for k in KS})
    ms = alternate(variants, args.reps, args.calls)
    search = {}
    for name, t in ms.items():
        best = min(t)
        search[name] = {"ms": [round(x, 3) for x in t], "best_ms": round(best, 3), "pairs_per_s": M * N / (best * 1e-3)}
    for name in search:
        search[name]["vs_nearest"] = round(search[name]["pairs_per_s"] / search["nearest"]["pairs_per_s"], 4)
        print(name, json.dumps(search[name]), flush=True)
    res["search"] = search
    # the top-k results agree with nearest at k = 1
    i1, c1 = lut.nearest(L, O)
    ik, ck = lut.nearest_k(L, O, 1)
    res["k1_equals_nearest"] = bool(torch.equal(ik[:, 0], i1) and torch.equal(ck[:, 0].view(torch.int32),
                                                                                c1.view(torch.int32)))

    # merge alone, at the list count a search at that m leaves
    merge = {}
    for m in (1, 1000, M):
        for k in (10, 128):
            n_lists = lib.spart_lut_topk_workspace_bytes(N, m, k) // (8 * m * k)
            lists = sorted_lists(n_lists, m, k, g)
            Om = O[:m].contiguous()
            t = alternate({"merge": lambda: lut.merge_k(lists), "nearest_k": lambda: lut.nearest_k(L, Om, k)},
                          args.reps, args.calls)
            merge[f"m{m}_k{k}"] = {"lists": n_lists, "merge_ms": round(min(t["merge"]), 4),
                                   "nearest_k_ms": round(min(t["nearest_k"]), 4)}
            print("merge", m, k, json.dumps(merge[f"m{m}_k{k}"]), flush=True)
            del lists
    res["merge"] = merge

    # estimate, P = 27 float64 parameters of the 2^20 entries
    params = torch.rand((27, N), generator=g, device="cuda", dtype=torch.float64)
    est = {}
    for k in (10, 50):
        idx, _ = lut.nearest_k(L, O, k)
        t = alternate({"estimate": lambda: lut.estimate(params, idx)}, args.reps, args.calls)
        est[f"k{k}"] = {"ms": round(min(t["estimate"]), 4)}
        print("estimate", k, json.dumps(est[f"k{k}"]), flush=True)
    res["estimate_p27"] = est

    # device time of the search and merge kernels inside one nearest_k call (profiler pass, not timed above)
    from torch.profiler import ProfilerActivity, profile
    split = {}
    for k in KS:
        lut.nearest_k(L, O, k)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            lut.nearest_k(L, O, k)
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            for key in ("lut_topk_kernel", "lut_topk_merge_kernel"):
                if key in ev.key and ("merge" in key) == ("merge" in ev.key):
                    kern[key] = kern.get(key, 0.0) + ev.device_time_total / 1e3
        split[f"k{k}"] = {name: round(v, 4) for name, v in kern.items()}
        print("split", k, json.dumps(split[f"k{k}"]), flush=True)
    res["kernel_ms"] = split

    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "lut_topk.json").write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
