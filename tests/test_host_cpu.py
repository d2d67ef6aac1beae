"""CPU-only checks of the host side: C-ABI symbols, loud failure without a GPU, host table
folding against the oracle, parameter packing, world_size-2 gloo sharding."""
import json
import os
import re
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

import spart_oracle as so
from conftest import ROOT, relerr


def test_capi_exports_every_declared_symbol():
    from spart_b200 import _lib
    lib = _lib.load()
    header = (ROOT / "include" / "spart_b200.h").read_text()
    declared = set(re.findall(r"\b(spart_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.EXPORTS)
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.spart_abi_version() == _lib.ABI_VERSION
    assert isinstance(lib.spart_device_count(), int)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_fails_loudly_without_gpu():
    import spart_b200
    from spart_b200 import _lib
    with pytest.raises(spart_b200.SpartError):
        spart_b200.run_batch_params(np.zeros((27, 4)), "Sentinel2A-MSI")
    lib = _lib.load()
    a, b = _lib.c_double(), _lib.c_double()
    assert lib.spart_measure_peaks(0, _lib.byref(a), _lib.byref(b)) == -2      # SPART_ENODEV
    assert b"no CUDA device" in lib.spart_last_error()


def test_product_never_imports_oracle():
    for py in (ROOT / "spart-python_b200").rglob("*.py"):
        txt = py.read_text()
        assert "spart_oracle" not in txt and "oracle" not in txt.replace("oracle/", ""), py


def test_host_tables_match_oracle(optical):
    from spart_b200 import tables as T
    lc = T.leaf_soil_constants()
    nr, nw = optical["nr"][:, 0], optical["nw"][:, 0]
    assert np.array_equal(lc[8], so.calculate_tav(40, nr))
    assert np.array_equal(lc[9], so.calculate_tav(90, nr))
    assert np.array_equal(lc[14], so.calculate_tav(90, 2 / nw) / so.calculate_tav(90, 2))
    assert np.array_equal(lc[15], 1 - so.calculate_tav(90, nw) / nw ** 2)
    for name in T.SENSOR_NAMES:
        info = T.load_sensor_info(name)
        st = T.build_sensor(name, info)
        assert np.array_equal(st.srf_index, so.closest_index(info["wl_srf_smac"], optical["wl_Ea"]))
        lo, hi, frac = so.band_sample_points(info["wl_smac"].T[0])
        assert np.array_equal(st.wl_lo, lo) and np.array_equal(st.wl_hi, hi) and np.array_equal(st.wl_frac, frac)
        # ET convolution: linear in Ea, so conv_ea * scale == faithful per-sample convolution
        P = so.synthetic_params(3, 3, seed=1)
        La = so.et_band_radiance(P[:, so.DOY], P[:, so.SZA], optical, info)
        scale = so.et_correction(P[:, so.DOY:so.DOY + 1]) * np.cos(P[:, so.SZA:so.SZA + 1] * np.pi / 180) / np.pi
        assert relerr(st.conv_ea[None, :] * scale, La) < 1e-14
        # folded SMAC constants keep the coefficients' dtype semantics
        c = info["SMAC_coef"]
        ak2 = (1 - c["wo"]) * (3 - c["wo"] * 3 * c["gc"])
        assert np.array_equal(st.smac[T.SMAC_ROWS.index("ak2")], ak2[0].astype(np.float64))
        assert ak2.dtype == c["wo"].dtype


def test_reference_install(tmp_path, monkeypatch):
    """tools/install_reference.py (run by build()): copies src/SPART of a reference checkout unchanged plus the
    nvtx stand-in; a missing checkout, or one below a directory this user may not read, installs nothing."""
    import importlib.util
    import pathlib
    spec = importlib.util.spec_from_file_location("install_reference", ROOT / "tools" / "install_reference.py")
    inst = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(inst)
    pkg = tmp_path / "checkout" / "src" / "SPART"
    (pkg / "model_parameters").mkdir(parents=True)
    (pkg / "SPART.py").write_text("class SPART:\n    pass\n")
    (pkg / "model_parameters" / "optical_params.pkl").write_bytes(bytes(range(256)))
    dest = tmp_path / "_ref"
    target = inst.install(str(tmp_path / "checkout"), dest)
    assert target == dest / "SPART" and (dest / "nvtx.py").is_file()
    assert (target / "SPART.py").read_bytes() == (pkg / "SPART.py").read_bytes()
    assert (target / "model_parameters" / "optical_params.pkl").read_bytes() == bytes(range(256))
    assert inst.install(str(tmp_path / "missing"), tmp_path / "none") is None
    assert not (tmp_path / "none").exists()

    def unreadable(self):
        raise PermissionError(13, "Permission denied", str(self))
    monkeypatch.setattr(pathlib.Path, "is_dir", unreadable)
    assert inst.install(str(tmp_path / "checkout"), tmp_path / "none") is None
    assert not (tmp_path / "none").exists()
    assert inst.default_source() == json.loads((ROOT / "BASELINE.json").read_text())["reference_path"]


def test_unknown_sensor_raises_filenotfound():
    from spart_b200 import tables as T
    with pytest.raises(FileNotFoundError):
        T.load_sensor_info("NoSuch-Sensor")


def test_param_holders_mirror_reference():
    import spart_b200 as sb
    with pytest.warns(UserWarning):
        soil = sb.SoilParameters(0.5, 0, 100, 15)
    assert soil.SMC == 25 and soil.film == 0.015 and soil.rdry_set is False
    leaf = sb.LeafBiology(40, 10, 0.02, 0.01, 0, 10, 1.5)
    assert (leaf.Cdm, leaf.Cs, leaf.Cca, leaf.PROT, leaf.CBC, leaf.rho_thermal) == (10, 0.01, 0, 0.0, 0.0, 0.01)
    atm = sb.AtmosphericProperties(0.3, 0.35, 1.4)
    assert atm.Pa == 1013.25
    atm2 = sb.AtmosphericProperties(0.3, 0.35, 1.4, alt_m=1000, temp_k=288.0)
    assert atm2.Pa == pytest.approx(1013.25 * np.exp(-(9.80665 * 1000 * 0.02896968 / (288.0 * 8.314462618))))
    can = sb.CanopyStructure(3, -0.35, -0.15, 0.05)
    assert (can.nlayers, can.nlincl, can.nlazi) == (60, 13, 36)
    p = sb.pack_params(soil, leaf, can, atm, sb.Angles(40, 0, 0), 100)
    assert p.shape == (27, 1) and p[so.CDM, 0] == 10 and p[so.SMC, 0] == 25 and p[so.DOY, 0] == 100


def test_soil_parameters_from_file(tmp_path):
    """JPL spectral-library text format (bsm.py:201-226): 21 header lines, wavelength in
    micrometres (descending), reflectance in percent."""
    import spart_b200 as sb
    wl_um = np.arange(2.5, 0.3995, -0.0005)                 # 0.5 nm steps, descending
    refl_pct = 10 + 20 * (wl_um - 0.4)
    f = tmp_path / "soil.txt"
    with open(f, "w") as fh:
        fh.write("\n".join(f"header {i}" for i in range(21)) + "\n")
        for w, r in zip(wl_um, refl_pct):
            fh.write(f"{w:.4f}\t{r:.6f}\n")
    soil = sb.SoilParametersFromFile(str(f), 20, 25, 0.015)
    assert soil.rdry_set and soil.rdry.shape == (2001, 1)
    want = (10 + 20 * (np.arange(400, 2401) / 1000 - 0.4)) / 100
    # positional interpolation (like the reference) is off by up to a quarter sample spacing
    assert np.allclose(soil.rdry[:, 0], want, atol=1e-4)
    with pytest.warns(UserWarning):
        soil2 = sb.SoilParametersFromFile(want.copy(), 20)
    assert soil2.SMC == 25 and soil2.film == 0.015 and soil2.rdry is not None
    p = sb.pack_params(soil2, sb.LeafBiology(40, 0.01, 0.02, 0, 10, 10, 1.5), sb.CanopyStructure(3, -0.35, -0.15, 0.05),
                       sb.AtmosphericProperties(0.3, 0.35, 1.4), sb.Angles(40, 0, 0), 100)
    assert p[so.SMP, 0] == 20 and p[so.SOIL_B, 0] == 0


def test_pack_batch_layout():
    import spart_b200 as sb
    P = so.synthetic_params(50, 3, seed=4)
    block = sb.pack_batch(P[:, 0:9], P[:, 9:15], P[:, 15:19], P[:, 19:22], P[:, 22:26], P[:, 26])
    assert np.array_equal(block, P.T)
    block = sb.pack_batch(P[:, 0:7], P[:, 9:13], P[:, 15:19], [40, 0, 0], P[:, 22:26], 100)
    assert block.shape == (27, 50) and (block[so.SZA] == 40).all() and (block[so.DOY] == 100).all()
    assert (block[so.SMC] == 25).all() and (block[so.FILM] == 0.015).all() and (block[so.PROT] == 0).all()
    tb = sb.pack_batch(torch.from_numpy(P[:, 0:9]), torch.from_numpy(P[:, 9:15]), torch.from_numpy(P[:, 15:19]),
                       torch.from_numpy(P[:, 19:22]), torch.from_numpy(P[:, 22:26]), torch.from_numpy(P[:, 26]))
    assert torch.equal(tb, torch.from_numpy(P.T.copy()))


def test_shard_bounds_cover_batch():
    from spart_b200.distributed import shard_bounds
    for n in (0, 1, 7, 8, 1000003):
        for w in (1, 2, 3, 8):
            b = [shard_bounds(n, w, r) for r in range(w)]
            assert b[0][0] == 0 and b[-1][1] == n
            assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))
            sizes = [hi - lo for lo, hi in b]
            assert max(sizes) - min(sizes) <= 1


def _gloo_worker(rank, world, port, n, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    sys.path.insert(0, str(ROOT / "spart-python_b200"))
    sys.path.insert(0, str(ROOT / "oracle"))
    from spart_b200.distributed import run_batch_sharded
    import spart_oracle as so2
    dist.init_process_group("gloo", rank=rank, world_size=world)
    P = torch.from_numpy(so2.synthetic_params(n, 3, seed=11).T.copy())

    def compute(p, sensor, precision):          # stand-in for the CUDA path (test only)
        return torch.from_numpy(so2.spart_bands(p.numpy().T, sensor))

    full = run_batch_sharded(P, "LANDSAT8-OLI", group=None, dst=None, compute=compute)
    root_only = run_batch_sharded(P, "LANDSAT8-OLI", group=None, dst=0, compute=compute)
    q.put((rank, full.numpy(), None if root_only is None else root_only.numpy()))
    dist.destroy_process_group()


def test_sharded_gather_gloo_world2():
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    n, world = 37, 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, n, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        rank, full, root = q.get(timeout=120)
        res[rank] = (full, root)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    want = so.spart_bands(so.synthetic_params(n, 3, seed=11), "LANDSAT8-OLI")
    for rank in range(world):
        assert np.array_equal(res[rank][0], want)
    assert np.array_equal(res[0][1], want) and res[1][1] is None


@pytest.mark.parametrize("tool,header", [("gen_math_coeffs.py", "math_coeffs.h"), ("gen_tau_coeffs.py", "tau_coeffs.h")])
def test_generated_coefficient_headers_are_reproducible(tmp_path, tool, header):
    """The polynomial / quadrature / E1 coefficient headers compiled into the kernels are exactly
    what their generators produce (multi-precision arithmetic, accuracy asserted inside the tools)."""
    import subprocess
    pytest.importorskip("mpmath")
    out = tmp_path / header
    subprocess.run([sys.executable, str(ROOT / "tools" / tool), "--out", str(out)], check=True,
                   capture_output=True, timeout=300)
    committed = ROOT / "spart-python_b200" / "csrc" / header
    assert out.read_text() == committed.read_text()


def _gloo_pipeline_worker(rank, world, port, n_local, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    sys.path.insert(0, str(ROOT / "spart-python_b200"))
    sys.path.insert(0, str(ROOT / "oracle"))
    from spart_b200 import lut
    from spart_b200.distributed import run_batch_sharded_pipelined
    import spart_oracle as so2
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sensor = "LANDSAT8-OLI"
    P = torch.from_numpy(so2.synthetic_params(n_local, 3, seed=100 + rank).T.copy())

    def compute(p, view):                        # stand-in for the CUDA path (test only)
        view.view(p.shape[1], 9, 3).copy_(torch.from_numpy(so2.spart_bands(p.numpy().T, sensor)))
    compute.n_bands = 9
    res = run_batch_sharded_pipelined(P, sensor, chunk=7, dst=0, compute=compute)
    got = None if res is None else [torch.cat(per).numpy() for per in res]

    # sharded retrieval: each rank owns a slice of the table; stand-in search in NumPy, real reduction
    table = np.random.default_rng(5).random((40, 4)).astype(np.float32)
    obs = torch.from_numpy(np.random.default_rng(6).random((11, 4)).astype(np.float32))
    lo, hi = (0, 17) if rank == 0 else (17, 40)

    def search(l, o, w, off):
        d = ((o.numpy()[:, None, :] - l.numpy()[None, :, :]) ** 2).sum(-1).astype(np.float32)
        i = d.argmin(1)
        bits = d[np.arange(d.shape[0]), i].view(np.uint32).astype(np.int64)
        return torch.from_numpy((bits << 32) | (i + off))

    def unpack(words):
        w = words.numpy()
        return torch.from_numpy(w & 0xffffffff), torch.from_numpy((w >> 32).astype(np.uint32).view(np.float32))
    idx, cost = lut.nearest_sharded(torch.from_numpy(table[lo:hi]), obs, search=search, unpack_words=unpack)
    q.put((rank, got, idx.numpy(), cost.numpy()))
    dist.destroy_process_group()


def test_pipelined_gather_and_sharded_retrieval_gloo_world2():
    """World-size-2 run of the chunk-pipelined gather (ragged last chunk) and of the sharded table search
    with its 8-byte-per-observation min-all-reduce; the CUDA kernels are replaced by NumPy stand-ins."""
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    n_local, world = 19, 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_pipeline_worker, args=(r, world, port, n_local, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        rank, got, idx, cost = q.get(timeout=120)
        res[rank] = (got, idx, cost)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert res[1][0] is None
    for r in range(world):
        want = so.spart_bands(so.synthetic_params(n_local, 3, seed=100 + r), "LANDSAT8-OLI")
        assert np.array_equal(res[0][0][r], want)
    table = np.random.default_rng(5).random((40, 4)).astype(np.float32)
    obs = np.random.default_rng(6).random((11, 4)).astype(np.float32)
    d = ((obs[:, None, :] - table[None, :, :]) ** 2).sum(-1).astype(np.float32)
    for r in range(world):
        assert np.array_equal(res[r][1], d.argmin(1))
        assert np.array_equal(res[r][2], d.min(1))


def test_compact_bands_rebuilds_l_toa():
    """CompactBands on host arrays: L_TOA = (conv_ea * etscale) * R_TOA in the arithmetic type of the run."""
    from spart_b200.engine import CompactBands, out_elems
    rng = np.random.default_rng(0)
    n, nb = 5, 3
    conv = rng.random(nb) * 1000
    for dt, fp32 in ((np.float64, False), (np.float32, True), (np.float64, True)):
        buf = rng.random(out_elems(n, nb, True)).astype(dt)
        c = CompactBands(buf, n, nb, conv, fp32)
        R, ets = buf[:n * nb * 2].reshape(n, nb, 2), buf[n * nb * 2:]
        at = np.float32 if fp32 else np.float64
        want = ((conv.astype(at)[None, :] * ets.astype(at)[:, None]) * R[..., 1].astype(at)).astype(dt)
        assert np.array_equal(c.L_TOA, want) and c.full().shape == (n, nb, 3) and c.full().dtype == dt
        assert np.array_equal(c.full()[..., :2], R)
