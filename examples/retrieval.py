"""Retrieval of Sentinel-2A canopy parameters: a quasi-random look-up table gives each observation its 8 nearest
entries, and a bounded Levenberg-Marquardt fit from those entries refines it past the table's grid, with a
standard deviation per parameter.  Everything runs on the GPU.

Run from the repository root (needs a GPU and the built library):
    PYTHONPATH=spart-python_b200 python examples/retrieval.py
"""
import numpy as np
import torch

import spart_b200
from spart_b200.inversion import STATUS_NAMES, invert, starts
from spart_b200.sensitivity import ParameterSpace

SENSOR = "Sentinel2A-MSI"
# fixed values: the reference's README example (geometry 40 / 0 / 0, DOY 100)
base = np.array([40, 0.01, 0.02, 0, 10, 10, 1.5, 0, 0, 0.5, 0, 100, 20, 25, 0.015, 3, -0.35, -0.15, 0.05,
                 40, 0, 0, 0.325, 0.35, 1.41, 1013.25, 100], dtype=np.float64)
space = ParameterSpace(base, {"Cab": (5, 80), "Cw": (0.005, 0.05), "Cdm": (0.002, 0.02), "N": (1, 3),
                              "LAI": (0.1, 8), "SMp": (5, 55)})

# the table: 2^16 scrambled Sobol' points of the space, R_TOC of every band
params = space.sample(2 ** 16, seed=3)
table = spart_b200.lut.generate(params, SENSOR, column=0)

# observations: R_TOC of 1000 random parameter sets, with 1e-4 noise
rng = np.random.default_rng(0)
m, sigma = 1000, 1e-4
truth = space.lo + (space.hi - space.lo) * rng.uniform(0, 1, (m, space.d))
X = np.tile(base, (m, 1))
X[:, space.rows] = truth
clean = spart_b200.default_engine().forward_bands(torch.from_numpy(np.ascontiguousarray(X.T)).cuda(), SENSOR)[..., 0]
obs = (clean + sigma * torch.from_numpy(rng.standard_normal(clean.shape)).cuda()).contiguous()

idx, _ = spart_b200.lut.nearest_k(table, obs.float(), 8)        # the 8 nearest entries
x0 = starts(params, idx, space)                                  # their parameters as starts [m, 8, P]
res = invert(obs, SENSOR, space, x0, weights=np.full(obs.shape[1], sigma ** -2), absolute_sigma=True)

x, sd = res.x.cpu().numpy(), res.std.cpu().numpy()
lut_x = x0[:, 0].cpu().numpy()
print(f"{'':>5} {'LUT |err|':>10} {'fit |err|':>10} {'fit std':>10}   (medians over {m} observations)")
for i, n in enumerate(res.names):
    print(f"{n:>5} {np.median(np.abs(lut_x[:, i] - truth[:, i])):10.3g} {np.median(np.abs(x[:, i] - truth[:, i])):10.3g}"
          f" {np.median(sd[:, i]):10.3g}")
status = res.status.cpu().numpy()
print("status:", {STATUS_NAMES[s]: int((status == s).sum()) for s in np.unique(status)})
print(f"forward runs per observation: {res.n_forward.double().mean().item():.0f}")
