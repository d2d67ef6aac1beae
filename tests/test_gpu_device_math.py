"""Accuracy of the device math functions every physics result rests on, asserted against 50-digit mpmath.

tests/device_math_harness.cu is compiled at test time with the library's NVCC_FLAGS into a shared library
and evaluates one function of spart_device.cuh / spart_device_f32.cuh per call on device arrays.  The FP64
bounds are the ones DESIGN.md section 4 states; the FP32 bounds are those of the CUDA intrinsics the FP32
mode uses (CUDA C Programming Guide, intrinsic functions) and of the plate-function generator."""
import ctypes
import importlib.util
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
CSRC = ROOT / "spart-python_b200" / "csrc"
HARNESS = Path(__file__).resolve().parent / "device_math_harness.cu"
F64 = dict(exp_fast=0, exp_clamp=1, exp_neg=2, exp_bounded=3, log_fast=4, rcp_fast=5, sqrt_fast=6, sin=7, cos=8,
           plate_tau=9)
F32 = dict(one_minus_tau=0, fexp=1, flog=2, rcp=3, fsqrt=4, tau=5)
TINY = 2.0 ** -1074


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    import torch
    assert torch.cuda.is_available()
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).exists():
        pytest.skip("nvcc is not installed: the device-math harness is compiled at test time")
    spec = importlib.util.spec_from_file_location("spart_build", ROOT / "spart-python_b200" / "build.py")
    build = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(build)
    so = tmp_path_factory.mktemp("devmath") / "libdevmath.so"
    subprocess.run([nvcc] + build.NVCC_FLAGS + ["-I", str(CSRC), "-o", str(so), str(HARNESS)], check=True)
    lib = ctypes.CDLL(str(so))
    for f in (lib.dm_eval64, lib.dm_eval32):
        f.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]
        f.restype = ctypes.c_int
    torch.cuda.init()
    torch.zeros(1, device="cuda")            # the primary context, shared with the harness's runtime
    assert lib.dm_init() == 0

    def run(fn, x):
        x = np.ascontiguousarray(x)
        dt = torch.float64 if x.dtype == np.float64 else torch.float32
        xd = torch.from_numpy(x).cuda()
        yd = torch.empty_like(xd)
        torch.cuda.synchronize()
        f, code = (lib.dm_eval64, F64[fn]) if dt == torch.float64 else (lib.dm_eval32, F32[fn])
        assert f(code, xd.data_ptr(), yd.data_ptr(), x.size) == 0
        return yd.cpu().numpy()
    return run


def mp():
    import mpmath
    mpmath.mp.dps = 50
    return mpmath


def ulp_errors(got, x, f):
    """|got - f(x)| in units in the last place of the double nearest f(x), f evaluated in 50-digit mpmath."""
    m = mp()
    out = np.empty(len(x))
    for i, (g, v) in enumerate(zip(got, x)):
        ref = f(m.mpf(float(v)))
        e = max(int(m.frexp(ref)[1]) - 1, -1022) if ref != 0 else -1022
        out[i] = float(abs(m.mpf(float(g)) - ref) / m.mpf(2) ** (e - 52))
    return out


def rng_mix(seed, n, lo, hi):
    rng = np.random.default_rng(seed)
    return rng.uniform(lo, hi, n)


def test_exp_fast(harness):
    m = mp()
    x = np.concatenate([rng_mix(1, 6000, -745.1, 709.7), rng_mix(2, 3000, -2, 2), rng_mix(3, 2000, -745.1, -708),
                        [0.0, -0.0, 1e-300, -1e-300, 709.78, -708.39, -744.4, -745.13]])
    got = harness("exp_fast", x)
    e = ulp_errors(got, x, m.exp)
    sub = np.exp(x) < 2.0 ** -1022
    print(f"exp_fast: {e[~sub].max():.3f} ulp, subnormal results {e[sub].max():.3f} ulp")
    assert sub.sum() > 500                                   # subnormal results are part of the sample
    assert e[~sub].max() <= 1.1, f"exp_fast {e[~sub].max():.3f} ulp"
    # subnormal results, in units of the subnormal grid
    assert e[sub].max() <= 1.1, f"exp_fast subnormal {e[sub].max():.3f} ulp"
    sp = harness("exp_fast", np.array([np.nan, np.inf, -np.inf, 710.0, 1000.0, -746.0, -1000.0]))
    assert np.isnan(sp[0]) and sp[1] == np.inf and sp[2] == 0 and sp[3] == np.inf and sp[4] == np.inf
    assert sp[5] == 0 and sp[6] == 0


@pytest.mark.parametrize("fn", ["exp_clamp", "exp_neg", "exp_bounded"])
def test_exp_clamped_variants(harness, fn):
    m = mp()
    x = np.concatenate([rng_mix(4, 6000, -700, 700 if fn != "exp_neg" else 50), [-700.0, 0.0, -1e-300]])
    if fn != "exp_neg":
        x = np.append(x, 700.0)
    got = harness(fn, x)
    e = ulp_errors(got, x, m.exp)
    print(f"{fn}: {e.max():.3f} ulp")
    assert e.max() <= 1.1, f"{fn} {e.max():.3f} ulp"
    if fn == "exp_bounded":
        return
    e700, em700 = float(m.exp(700)), float(m.exp(-700))
    lo = harness(fn, np.array([-700.5, -746.0, -1e4, -np.inf, np.nan]))
    assert (np.abs(lo[:4] / em700 - 1) < 2e-16).all() and np.isnan(lo[4]), lo
    if fn == "exp_clamp":
        hi = harness(fn, np.array([700.5, 710.0, 1e4, np.inf]))
        assert (np.abs(hi / e700 - 1) < 2e-16).all(), hi


def test_log_fast(harness):
    m = mp()
    rng = np.random.default_rng(5)
    x = np.concatenate([
        np.exp(rng.uniform(np.log(2.0 ** -1021), np.log(1.7e308), 6000)),
        rng.uniform(0.5, 2.0, 3000),
        1.0 + rng.uniform(-1e-6, 1e-6, 500),
        # the sqrt(2) mantissa switch: mantissas on either side of 0x3ff6a09f..., at several exponents
        np.ldexp(np.array([np.nextafter(np.sqrt(2), 0), np.sqrt(2), np.nextafter(np.sqrt(2), 2),
                           1.4142, 1.41422, 1.4142133, 1.41421342])[:, None], np.arange(-20, 21)[None, :]).ravel(),
        [1.0, 2.0, 0.5, 2.0 ** -1022, 1.7976931348623157e308]])
    got = harness("log_fast", x)
    e = ulp_errors(got, x, m.log)
    print(f"log_fast: {e.max():.3f} ulp")
    assert e.max() <= 2.5, f"log_fast {e.max():.3f} ulp at {x[np.argmax(e)]!r}"
    sp = harness("log_fast", np.array([0.0, -0.0, -1.0, -np.inf, np.inf, np.nan]))
    assert sp[0] == -np.inf and sp[1] == -np.inf and np.isnan(sp[2]) and np.isnan(sp[3])
    assert sp[4] == np.inf and np.isnan(sp[5])


@pytest.mark.parametrize("fn", ["rcp_fast", "sqrt_fast"])
def test_rcp_sqrt(harness, fn):
    m = mp()
    rng = np.random.default_rng(6)
    x = np.exp(rng.uniform(np.log(2.0 ** -1020), np.log(2.0 ** 1020), 8000))
    x = np.concatenate([x, rng.uniform(0.5, 4, 4000), 2.0 ** np.arange(-1020, 1021, 40)])
    if fn == "rcp_fast":
        x = np.concatenate([x, -x[:2000]])
    f = (lambda v: 1 / v) if fn == "rcp_fast" else m.sqrt
    e = ulp_errors(harness(fn, x), x, f)
    print(f"{fn}: {e.max():.3f} ulp")
    assert e.max() <= 1.0, f"{fn} {e.max():.3f} ulp"
    if fn == "sqrt_fast":
        sp = harness(fn, np.array([0.0, -1.0, np.nan]))
        assert sp[0] == 0 and np.isnan(sp[1]) and np.isnan(sp[2])


@pytest.mark.parametrize("fn", ["sin", "cos"])
def test_sincos_small(harness, fn):
    """|x| up to 8 (the leaf-angle iteration works on [0, 2 pi] plus its steps)."""
    m = mp()
    k = np.arange(-5, 6)[:, None] * (np.pi / 2)
    near = (k + np.array([-1e-3, -1e-9, 0.0, 1e-9, 1e-3])[None, :]).ravel()
    x = np.concatenate([rng_mix(7, 8000, -8, 8), rng_mix(8, 2000, -1e-3, 1e-3), near])
    x = x[np.abs(x) <= 8]
    e = ulp_errors(harness(fn, x), x, getattr(m, fn))
    print(f"{fn}: {e.max():.3f} ulp")
    assert e.max() <= 1.6, f"{fn} {e.max():.3f} ulp at {x[np.argmax(e)]!r}"


def tau_exact(K):
    """(1 - K) e^-K + K^2 E1(K) (prospect_5d.py:182-196) in 50-digit arithmetic."""
    m = mp()
    k = m.mpf(float(K))
    return (1 - k) * m.exp(-k) + k * k * m.e1(k)


def tau_arguments():
    rng = np.random.default_rng(9)
    dense = np.exp(rng.uniform(np.log(1e-12), np.log(1e3), 3000))
    edges = [1.0] + [2.0 ** j for j in range(1, 7)]
    around = [v for b in edges for v in (np.nextafter(b, 0), b, np.nextafter(b, np.inf))]
    return np.concatenate([dense, around, [1e-12, 0.5, 0.999, 63.99, 64.0, 100.0, 700.0, 708.0, 744.0, 745.0,
                                           746.0, 800.0, 1e3, 1e4]])


def test_plate_tau(harness):
    """plate_tau through the shared-memory table of load_tau_table: relative error <= 2e-15 on every piece,
    2^j +- 1 ulp at the piece boundaries; where tau is subnormal or underflows (K >= ~700) within two units of
    the subnormal grid."""
    K = tau_arguments()
    got = harness("plate_tau", K)
    ref = np.array([float(tau_exact(k)) for k in K])
    assert (got >= 0).all() and np.isfinite(got).all()
    normal = ref >= 2.0 ** -1022
    rel = np.abs(got[normal] - ref[normal]) / ref[normal]
    worst = np.argmax(rel)
    print(f"plate_tau: relative {rel.max():.3e} at K = {K[normal][worst]!r}")
    assert rel.max() <= 2e-15, f"plate_tau rel {rel.max():.3e} at K = {K[normal][worst]!r}"
    assert (np.abs(got[~normal] - ref[~normal]) <= 2 * TINY).all()
    assert (~normal).sum() >= 4 and (got[K >= 746] == 0).all()
    pieces = np.where(K < 1, 0, np.minimum(np.floor(np.log2(np.maximum(K, 1))) + 1, 7)).astype(int)
    assert (np.bincount(pieces[normal], minlength=8) > 30).all()


def test_plate_tau_f(harness):
    """FP32 plate function (plate_tau_f, spart_device_f32.cuh): tau and 1 - tau, each against 50 digits.
    tau is formed directly for K >= 1, so it keeps its relative accuracy where it is far below float resolution
    of 1 (7e-11 at K = 21, the largest K of the input domain); its error there is that of __expf(-K)."""
    K = tau_arguments()
    K = np.unique(K[(K >= 2.0 ** -126) & (K < 3e38)].astype(np.float32))
    exact = [tau_exact(float(k)) for k in K]
    omt = harness("one_minus_tau", K).astype(np.float64)
    ref = np.array([float(1 - t) for t in exact])
    rel = np.abs(omt - ref) / ref
    worst = np.argmax(rel)
    print(f"1 - tau (fp32): relative {rel.max():.3e} at K = {K[worst]!r}")
    assert rel.max() <= ONE_MINUS_TAU_F_BOUND, f"1 - tau (fp32) rel {rel.max():.3e} at K = {K[worst]!r}"
    tau = harness("tau", K).astype(np.float64)
    ref = np.array([float(t) for t in exact])
    live = K <= 87.0                        # __expf(-K) is a normal float
    rel = np.abs(tau[live] - ref[live]) / ref[live]
    bound = np.where(K[live] < 1, ONE_MINUS_TAU_F_BOUND, (4 + 1.173 * K[live]) * 2.0 ** -23 + 2e-7)
    worst = np.argmax(rel / bound)
    print(f"tau (fp32): relative {rel.max():.3e}, {(rel / bound).max():.2f} of the bound at K = {K[live][worst]!r}")
    assert (rel <= bound).all(), f"tau (fp32) rel {rel[worst]:.3e} at K = {K[live][worst]!r}"
    assert (tau[(K >= 1) & live] > 0).all() and (tau >= 0).all()


# FP32 mode: the generator's float-coefficient interpolants are good to 9e-8 relative (tools/gen_tau_coeffs.py);
# 1 - tau adds __expf and __logf.  Measured on a B200: 7.0e-7 at K = 0.0515, just above the switch from the
# series of 1 - e^-K to 1 - __expf(-K), whose absolute error (~1e-7) is then relative to 1 - tau ~ 0.1.
# For K >= 1, __expf(-K) is good to 2 + floor(1.173 K) ulp (CUDA C Programming Guide), which bounds tau there.
ONE_MINUS_TAU_F_BOUND = 1e-6


def float_ulps(got, ref):
    """|got - ref| in float ulps of ref (ref in float64)."""
    e = np.floor(np.log2(np.abs(ref)))
    return np.abs(got.astype(np.float64) - ref) / 2.0 ** (np.maximum(e, -126) - 23)


def test_fp32_intrinsics(harness):
    """fexp (__expf): <= 2 + floor(1.173 |x|) ulp (+1 for the float argument rounding of x in the rule);
    flog (__logf): 2^-21.41 absolute on [0.5, 2], else 3 ulp; rcp (rcp.approx.ftz.f32) and fsqrt
    (sqrt.approx.ftz.f32): 2 ulp on normal numbers."""
    rng = np.random.default_rng(10)
    x = rng.uniform(-80, 80, 20000).astype(np.float32)
    e = float_ulps(harness("fexp", x), np.exp(x.astype(np.float64)))
    assert (e <= 2 + np.floor(1.173 * np.abs(x)) + 1).all(), f"fexp {e.max():.2f} ulp"
    x = np.exp(rng.uniform(np.log(1.2e-38), np.log(3e38), 20000)).astype(np.float32)
    x = np.concatenate([x, rng.uniform(0.5, 2, 5000).astype(np.float32)])
    got, ref = harness("flog", x).astype(np.float64), np.log(x.astype(np.float64))
    mid = (x >= 0.5) & (x <= 2)
    assert (np.abs(got - ref)[mid] <= 2.0 ** -21.41).all()
    assert (float_ulps(got[~mid], ref[~mid]) <= 3).all(), f"flog {float_ulps(got[~mid], ref[~mid]).max():.2f} ulp"
    x = np.exp(rng.uniform(np.log(1.2e-38), np.log(8e37), 20000)).astype(np.float32)
    x64 = x.astype(np.float64)
    assert float_ulps(harness("rcp", x), 1 / x64).max() <= 2
    assert float_ulps(harness("fsqrt", x), np.sqrt(x64)).max() <= 2
