"""Shared pytest configuration.

`-m "not gpu"` runs on the CPU build container: oracle vs golden fixtures, host logic,
C-ABI symbol checks, gloo world_size-2 sharding.  `-m gpu` runs on a B200 and compares the
CUDA path (through the C-ABI) with the oracle and with the golden fixtures.
"""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
GOLDEN = ROOT / "tests" / "golden"
for p in (ROOT / "spart-python_b200", ROOT / "oracle", ROOT):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


def load_golden(name):
    with np.load(GOLDEN / name, allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


def golden_columns(a, g):
    """The wavelength columns of spectra `a` (last axis 2001 or 2162) that golden file `g` stores: its sorted
    `wl_idx` (tools/make_golden.py::thin_spectra), cut to the width of `a`."""
    idx = g["wl_idx"]
    return a[..., idx[idx < a.shape[-1]]]


def relerr(a, b):
    """max |a-b| / |b| with NaN == NaN treated as equal."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    both_nan = np.isnan(a) & np.isnan(b)
    with np.errstate(all="ignore"):
        e = np.abs(a - b) / np.abs(b)
    e = np.where(both_nan, 0.0, e)
    e = np.where((a == b), 0.0, e)
    return float(np.nanmax(np.where(np.isnan(e), np.inf, e))) if e.size else 0.0


@pytest.fixture(scope="session")
def optical():
    import spart_oracle
    return spart_oracle.load_optical()
