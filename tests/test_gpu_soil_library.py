"""Per-sample dry-soil spectra from a soil library (SPART_FLAG_SOIL_LIBRARY).

Every sample's result must equal bit for bit the same sample run with soil_spectrum = its library row, in every
mode; the library path inherits the reference parity of the user-spectrum path from that."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from conftest import load_golden, relerr  # noqa: E402

RTOL64 = 1e-9
SOIL_B = 9


@pytest.fixture(scope="module")
def env():
    import torch
    import spart_b200
    import spart_oracle as so
    assert torch.cuda.is_available()
    return torch, spart_b200, so


def golden_rdry():
    return [load_golden(f"soilfile_{s}.npz")["rdry"] for s in ("Sentinel2A", "TerraAqua")]


def synthetic_spectra(k, seed=0):
    """k smooth dry-soil spectra in [0.02, 0.7]."""
    rng = np.random.default_rng(seed)
    x = np.linspace(0.0, 1.0, 2001)
    a, b, c, d = (rng.uniform(lo, hi, (k, 1)) for lo, hi in ((0.05, 0.2), (0.1, 0.4), (2.0, 9.0), (0.0, 0.05)))
    return np.clip(a + b * x ** 0.7 + d * np.sin(c * x), 0.02, 0.7)


@pytest.fixture(scope="module")
def library(env):
    _, sb, _ = env
    return sb.SoilLibrary(np.concatenate([np.stack(golden_rdry()), synthetic_spectra(6)]))


def with_index(P, idx):
    """[n, 27] oracle-layout params with row 9 (B) replaced by the library index."""
    P = np.array(P, dtype=np.float64)
    P[:, SOIL_B] = idx
    return P


def to_dev(torch, P, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    return t if dtype is None else t.to(dtype)


def assert_groups_bit_identical(run, P, idx, lib):
    """run(P, **soil) -> numpy [n, ...]: the library run equals, per index group, the soil_spectrum run."""
    got = run(P, soil_library=lib)
    for i in np.unique(idx):
        rows = idx == i
        want = run(P, soil_spectrum=lib.spectra[int(i)])
        assert np.array_equal(got[rows], want[rows]), f"library index {i}"
    return got


def band_runner(env, sensor, **kw):
    torch, sb, _ = env

    def run(P, **soil):
        dtype = torch.float32 if kw.get("f32_io") else None
        extra = {k: v for k, v in kw.items() if k != "f32_io"}
        out = sb.run_batch_params(to_dev(torch, P, dtype), sensor, **extra, **soil)
        if kw.get("compact"):         # one row per sample: (R_TOC, R_TOA) of every band, then etscale
            out = torch.cat([out.R.reshape(out.n, -1), out.etscale[:, None]], dim=1)
        torch.cuda.synchronize()
        return out.cpu().numpy()
    return run


@pytest.mark.parametrize("sensor,cfg,kw", [
    ("Sentinel2A-MSI", 2, dict(uniform_geometry=True)),
    ("Sentinel2A-MSI", 2, dict()),
    ("LANDSAT8-OLI", 3, dict()),
    ("TerraAqua-MODIS", 3, dict()),
    ("Sentinel3A-OLCI", 3, dict()),
    ("TerraAqua-MODIS", 3, dict(band_mode="srf")),
    ("Sentinel2A-MSI", 2, dict(precision="fp32", uniform_geometry=True)),
    ("LANDSAT8-OLI", 3, dict(precision="fp32")),
    ("LANDSAT8-OLI", 3, dict(precision="fp32", f32_io=True)),
    ("Sentinel2A-MSI", 3, dict(compact=True)),
    ("Sentinel2A-MSI", 2, dict(precision="fp32", f32_io=True, compact=True, uniform_geometry=True)),
])
def test_bit_identical_to_soil_spectrum(env, library, sensor, cfg, kw):
    _, _, so = env
    rng = np.random.default_rng(cfg * 7 + len(kw))
    idx = rng.integers(0, len(library), 5000).astype(np.float64)
    P = with_index(so.synthetic_params(5000, cfg, seed=300 + cfg), idx)
    got = assert_groups_bit_identical(band_runner(env, sensor, **kw), P, idx, library)
    assert np.isfinite(got).all()


def test_spectrum_planes_bit_identical(env, library):
    torch, sb, so = env
    idx = np.random.default_rng(5).integers(0, len(library), 400).astype(np.float64)
    P = with_index(so.synthetic_params(400, 3, seed=31), idx)
    eng = sb.default_engine()

    def run(P, **soil):
        out = eng.forward_spectrum(to_dev(torch, P), **soil)
        torch.cuda.synchronize()
        return out.cpu().numpy()
    got = assert_groups_bit_identical(run, P, idx, library)
    # plane 4 is the library spectrum, its 2400 nm value beyond 2400 nm
    i = idx.astype(int)
    assert np.array_equal(got[:, 4, :2001], library.spectra[i])
    assert np.array_equal(got[:, 4, 2001:], np.repeat(library.spectra[i, -1:], 161, axis=1))


def test_user_lidf_bit_identical(env, library):
    torch, sb, so = env
    n = 3000
    idx = np.random.default_rng(6).integers(0, len(library), n).astype(np.float64)
    P = with_index(so.synthetic_params(n, 3, seed=32), idx)
    lidf = np.random.default_rng(7).dirichlet(np.ones(13), n)

    def run(P, **soil):
        out = sb.run_batch_params(to_dev(torch, P), "LANDSAT8-OLI", lidf=lidf, **soil)
        torch.cuda.synchronize()
        return out.cpu().numpy()
    assert_groups_bit_identical(run, P, idx, library)


@pytest.mark.parametrize("name,at", [("soilfile_Sentinel2A", 0), ("soilfile_TerraAqua", 1)])
def test_reference_goldens_inside_mixed_library(env, library, name, at):
    """The user-spectrum goldens of the reference, their rows interleaved with other samples and indices."""
    torch, sb, so = env
    g = load_golden(f"{name}.npz")
    assert np.array_equal(library.spectra[at], g["rdry"])
    G, m = g["params"], g["params"].shape[0]
    other = so.synthetic_params(3 * m, 3, seed=33)
    P = np.empty((4 * m, 27))
    P[0::4], P[1::4], P[2::4], P[3::4] = G, other[0::3], other[1::3], other[2::3]
    idx = np.random.default_rng(8).integers(0, len(library), 4 * m).astype(np.float64)
    idx[0::4] = at
    got = sb.run_batch_params(to_dev(torch, with_index(P, idx)), str(g["sensor"]), soil_library=library)
    got = got.cpu().numpy()[0::4]
    assert relerr(got, g["O2"]) < RTOL64
    assert relerr(got, g["O1"]) < 5e-8


def test_oracle_per_index_group(env, library):
    torch, sb, so = env
    n = 20000
    idx = np.random.default_rng(9).integers(0, len(library), n).astype(np.float64)
    P = with_index(so.synthetic_params(n, 3, seed=34), idx)
    got = sb.run_batch_params(to_dev(torch, P), "LANDSAT8-OLI", soil_library=library).cpu().numpy()
    for i in range(len(library)):
        rows = idx == i
        want = so.spart_bands(P[rows], "LANDSAT8-OLI", soil_rdry=library.spectra[i])
        assert relerr(got[rows], want) < RTOL64, f"library index {i}"


def test_host_path(env, library):
    torch, sb, so = env
    n = 300001                       # several spans of the host path plus a ragged tail
    idx = np.random.default_rng(10).integers(0, len(library), n).astype(np.float64)
    P = np.ascontiguousarray(with_index(so.synthetic_params(n, 3, seed=35), idx).T)
    dev = sb.run_batch_params(torch.from_numpy(P).cuda(), "Sentinel2A-MSI", soil_library=library).cpu().numpy()
    assert np.array_equal(sb.run_batch_params(P, "Sentinel2A-MSI", soil_library=library), dev)
    pinned = torch.from_numpy(P).pin_memory()
    assert np.array_equal(sb.run_batch_params(pinned, "Sentinel2A-MSI", soil_library=library), dev)
    # row 9 as a broadcast row: the whole batch takes one library spectrum
    Q = P[:, :20000].copy()
    Q[SOIL_B] = 3.0
    one = sb.run_batch_params(Q, "Sentinel2A-MSI", soil_library=library, broadcast_rows=[SOIL_B])
    assert np.array_equal(one, sb.run_batch_params(Q, "Sentinel2A-MSI", soil_spectrum=library.spectra[3]))
    b = np.array(Q)
    b[SOIL_B, 1:] = np.nan              # never read: only element 0 of a broadcast row is
    assert np.array_equal(sb.run_batch_params(b, "Sentinel2A-MSI", soil_library=library, broadcast_rows=[SOIL_B]), one)


def test_multi_sensor_reuses_record(env, library):
    torch, sb, so = env
    idx = np.random.default_rng(11).integers(0, len(library), 5000).astype(np.float64)
    dev = to_dev(torch, with_index(so.synthetic_params(5000, 5, seed=36), idx))
    for prec in ("fp64", "fp32"):
        a, b = sb.run_batch_params(dev, ["Sentinel2A-MSI", "Sentinel2B-MSI"], precision=prec, soil_library=library)
        assert torch.equal(a, sb.run_batch_params(dev, "Sentinel2A-MSI", precision=prec, soil_library=library))
        assert torch.equal(b, sb.run_batch_params(dev, "Sentinel2B-MSI", precision=prec, soil_library=library))


@pytest.mark.parametrize("kw", [dict(), dict(uniform_geometry=True), dict(band_mode="srf"), dict(precision="fp32"),
                                dict(precision="fp32", f32_io=True)])
def test_invalid_indices_poison_only_their_samples(env, library, kw):
    torch, sb, so = env
    n, k = 4000, len(library)
    idx = np.random.default_rng(12).integers(0, k, n).astype(np.float64)
    P = with_index(so.synthetic_params(n, 2, seed=37), idx)
    bad = np.arange(5, n, 97)
    Pbad = P.copy()
    Pbad[bad, SOIL_B] = np.resize([-1.0, float(k), 2.5, np.nan], bad.size)
    run = band_runner(env, "TerraAqua-MODIS", **kw)
    got, ref = run(Pbad, soil_library=library), run(P, soil_library=library)
    assert np.isnan(got[bad]).all()
    keep = np.setdiff1d(np.arange(n), bad)
    assert np.array_equal(got[keep], ref[keep])


def test_invalid_indices_spectrum_planes(env, library):
    torch, sb, so = env
    P = with_index(so.synthetic_params(8, 3, seed=38), [0, -1, 1, len(library), 2, 0.5, np.nan, 3])
    out = sb.default_engine().forward_spectrum(to_dev(torch, P), soil_library=library).cpu().numpy()
    bad = [1, 3, 5, 6]
    assert np.isfinite(out[:, 0:3]).all()                 # leaf planes do not depend on the soil
    assert np.isnan(out[bad, 3:]).all()
    assert np.isfinite(np.delete(out, bad, axis=0)).all()


def test_flag_rules(env, library):
    torch, sb, so = env
    from spart_b200 import _lib
    eng = sb.default_engine()
    dev = to_dev(torch, so.synthetic_params(16, 2, seed=39))
    with pytest.raises(ValueError):
        eng.forward_bands(dev, "Sentinel2A-MSI", soil_library=library, soil_spectrum=library.spectra[0])
    handle, _ = eng.sensor("Sentinel2A-MSI")                     # no library in this context
    ws, out = eng.workspace(16), torch.empty((16, 13, 3), dtype=torch.float64, device=dev.device)
    rc = eng.lib.spart_forward_bands(handle, 0, dev.data_ptr(), 16, 16, 0, _lib.FP64, _lib.FLAG_SOIL_LIBRARY,
                                     ws.data_ptr(), out.data_ptr(), None)
    assert rc == -1 and b"soil library" in eng.lib.spart_last_error()
    handle, _ = eng.sensor("Sentinel2A-MSI", soil_library=library)
    rc = eng.lib.spart_forward_bands(handle, 0, dev.data_ptr(), 16, 16, 0, _lib.FP64,
                                     _lib.FLAG_SOIL_LIBRARY | _lib.FLAG_SOIL_SPECTRUM, ws.data_ptr(), out.data_ptr(),
                                     None)
    assert rc == -1 and b"exclude each other" in eng.lib.spart_last_error()


def test_run_batch_and_lut_generate(env, library, tmp_path):
    torch, sb, so = env
    n = 3000
    P = so.synthetic_params(n, 2, seed=40)
    idx = np.random.default_rng(13).integers(0, len(library), n)
    got = sb.run_batch(P[:, 0:9], P[:, 9:15], P[:, 15:19], P[:, 19:22], P[:, 22:26], P[:, 26], "Sentinel2A-MSI",
                       soil_library=library, soil_index=idx)
    want = sb.run_batch_params(np.ascontiguousarray(with_index(P, idx).T), "Sentinel2A-MSI", soil_library=library)
    assert np.array_equal(got, want)
    one = sb.run_batch(P[:, 0:9], P[:, 9:15], P[:, 15:19], P[:, 19:22], P[:, 22:26], P[:, 26], "Sentinel2A-MSI",
                       soil_library=library, soil_index=4)
    assert np.array_equal(one, sb.run_batch_params(np.ascontiguousarray(P.T), "Sentinel2A-MSI",
                                                   soil_spectrum=library.spectra[4]))
    lut = sb.lut.generate(with_index(P, idx).T, "Sentinel2A-MSI", column=0, path=tmp_path / "lut.npz",
                          soil_library=library, out_dtype=torch.float64)
    assert np.array_equal(lut.cpu().numpy(), want[..., 0])
    assert np.array_equal(np.load(tmp_path / "lut.npz")["params"][:, SOIL_B], idx.astype(np.float32))


def test_scale_4096_spectra(env):
    """1 M config-2 samples over k = 4096 spectra: per-group bit identity on 100 000 rows, determinism, and the
    folded-geometry kernels against the general ones."""
    torch, sb, so = env
    n, k = 1 << 20, 4096
    lib = sb.SoilLibrary(synthetic_spectra(k, seed=1))
    idx = np.random.default_rng(14).integers(0, k, n).astype(np.float64)
    P = with_index(so.synthetic_params(n, 2, seed=41), idx)
    dev = to_dev(torch, P)
    a = sb.run_batch_params(dev, "Sentinel2A-MSI", soil_library=lib, uniform_geometry=True)
    b = sb.run_batch_params(dev, "Sentinel2A-MSI", soil_library=lib, uniform_geometry=True)
    assert torch.equal(a, b)
    general = sb.run_batch_params(dev, "Sentinel2A-MSI", soil_library=lib)
    assert relerr(general.cpu().numpy(), a.cpu().numpy()) < 1e-12
    a = a.cpu().numpy()
    groups = np.unique(idx)[:410]                 # about 100 000 rows
    checked = 0
    for i in groups:
        rows = np.nonzero(idx == i)[0]
        want = sb.run_batch_params(to_dev(torch, P[rows]), "Sentinel2A-MSI", soil_spectrum=lib.spectra[int(i)],
                                   uniform_geometry=True).cpu().numpy()
        assert np.array_equal(a[rows], want), f"library index {i}"
        checked += rows.size
    assert checked >= 95000
