"""Which parameters drive which Sentinel-2A band: Sobol' indices of a forward-model box, all on the GPU, then a
quasi-random look-up table that varies only the rows that matter.

Run from the repository root (needs a GPU and the built library):
    PYTHONPATH=spart-python_b200 python examples/sensitivity.py
"""
import numpy as np

import spart_b200
from spart_b200.sensitivity import ParameterSpace, ROW_NAMES, sobol

# fixed values: the reference's README example (geometry 40 / 0 / 0, DOY 100)
base = np.array([40, 0.01, 0.02, 0, 10, 10, 1.5, 0, 0, 0.5, 0, 100, 20, 25, 0.015, 3, -0.35, -0.15, 0.05,
                 40, 0, 0, 0.325, 0.35, 1.41, 1013.25, 100], dtype=np.float64)
space = ParameterSpace(base, {"Cab": (5, 80), "Cdm": (0.002, 0.02), "Cw": (0.005, 0.05), "Cs": (0, 0.5),
                              "N": (1, 3), "SMp": (5, 55), "LAI": (0.1, 8), "LIDFa": (-0.5, 0.5),
                              "aot550": (0.05, 0.6), "uh2o": (0.5, 4)})
res = sobol(space, "Sentinel2A-MSI", 2 ** 14, seed=1)      # 2^14 (d + 2) = 196,608 forward runs
print(f"R_TOA total indices, N = {res.n} base points (standard error <= {res.total_se[:, 1].max():.3f})")
print("band " + " ".join(f"{n:>7}" for n in res.names))
for b in range(res.total.shape[0]):
    print(f"{b:4d} " + " ".join(f"{x:7.3f}" for x in res.total[b, 1]))

# keep the rows whose total index reaches 5 % in some band; fix the others at their base value
keep = {n: (space.lo[i], space.hi[i]) for i, n in enumerate(res.names) if res.total[:, 1, i].max() >= 0.05}
print("varied in the LUT:", ", ".join(keep))
lut_space = ParameterSpace(base, keep)
params = lut_space.sample(2 ** 16, seed=7)                 # scrambled Sobol' points, every row filled
table = spart_b200.lut.generate(params, "Sentinel2A-MSI", column=1)
print("LUT", tuple(table.shape), "rows varied:", [ROW_NAMES[r] for r in lut_space.rows])
