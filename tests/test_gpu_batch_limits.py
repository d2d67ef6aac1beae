"""Every entry point past its launch and index limits.

The band path accepts at most MAX = 65535 * 128 samples per C call (band-kernel grid.y), so
`Engine.forward_bands` splits a larger batch into calls; the spectrum and SAILH entry points loop over
grid.y slices of 65535 samples; outputs of the documented workloads pass 2^31 elements; the LUT search
splits its table into slices of whole 128-entry tiles and packs (cost, index) into one 64-bit word.
Each test here runs at those sizes and checks the samples at every boundary (first / last of each call
or slice, +-1 and +-2 around each split, the last sample) plus a few hundred random ones: against the
oracle at 1e-9 (FP64) or 1e-4 on physically valid outputs (FP32), and bit for bit against a small batch
of the same samples run with the same flags and kernels -- samples are independent, so a sample's bits
must not depend on where it sits in the batch.  Big outputs are compared on the device; only the selected
rows are copied to the host.  The tests allocate up to ~25 GB at a time and free it at the end."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import spart_oracle as so  # noqa: E402
from conftest import relerr  # noqa: E402
from test_gpu_domain import check_close  # noqa: E402
from test_gpu_soil_library import synthetic_spectra  # noqa: E402

MAX = 65535 * 128                 # samples per spart_forward_bands call
N_SPLIT = 2 * MAX + 1000          # two full calls and a ragged tail
RTOL64 = 1e-9
RTOL32 = 1e-4
NO_ENTRY = 2 ** 32 - 1
GB = 1 << 30


@pytest.fixture(scope="module")
def env():
    import torch
    import spart_b200
    assert torch.cuda.is_available()
    yield torch, spart_b200
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def need(torch, nbytes):
    """Skip (with the byte counts) when the device has less free memory than the test needs."""
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"needs {nbytes} bytes of free device memory, {free} free")


def release(torch):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def same_bits(torch, a, b):
    """Bitwise equality of two float tensors (NaN payloads included)."""
    it = torch.int64 if a.dtype == torch.float64 else torch.int32
    return a.shape == b.shape and a.dtype == b.dtype and bool(torch.equal(a.contiguous().view(it),
                                                                          b.contiguous().view(it)))


def boundaries(n, splits):
    s = {0, 1, n - 2, n - 1}
    for b in splits:
        s |= {b - 2, b - 1, b, b + 1, b + 2}
    return sorted(i for i in s if 0 <= i < n)


def pick(n, splits, k=300, seed=0, extra=()):
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate([boundaries(n, splits), list(extra),
                                     rng.choice(n, min(k, n), replace=False)]).astype(np.int64))


# ------------------------------------------------------------------------- A. band paths past one launch
BC_GEN = [7, 8, 13, 14]                       # PROT, CBC, SMC, film
BC_GEO = [19, 20, 21]                         # one geometry: the uniform kernels
MODES = {
    # name: sensor, synthetic config, broadcast rows, forward_bands keywords, soil source, float32 I/O
    "fp64_general": ("LANDSAT8-OLI", 3, BC_GEN + [16, 17], {}, None, False),
    "fp64_uniform": ("Sentinel2A-MSI", 2, BC_GEN + BC_GEO, {}, None, False),
    "srf": ("LANDSAT8-OLI", 3, BC_GEN, {"band_mode": "srf"}, None, False),
    "fp32_double_io": ("LANDSAT8-OLI", 3, BC_GEN, {"precision": "fp32"}, None, False),
    "fp32_float_io": ("Sentinel2A-MSI", 2, BC_GEN + BC_GEO, {"precision": "fp32"}, None, True),
    "soil_spectrum": ("Sentinel2A-MSI", 2, BC_GEN + BC_GEO, {}, "spectrum", False),
    "soil_library": ("LANDSAT8-OLI", 3, BC_GEN, {}, "library", False),
    "soil_library_row9": ("Sentinel2A-MSI", 2, BC_GEN + [9] + BC_GEO, {}, "library", False),
}
# library indices that are not a whole number in [0, 8), placed on the split columns
BAD_INDEX = {MAX - 1: -1.0, MAX: 8.0, MAX + 1: 2.5, 2 * MAX - 1: float("nan"), 2 * MAX: 1e300, 2 * MAX + 1: 7.5}


@pytest.fixture(scope="module")
def split_params(env):
    """Device [27, N_SPLIT] float64 batches of configs 2 and 3 (built once).  The rows some modes broadcast are
    made constant (their element 0), so a run with them as broadcast rows is the same model as one without."""
    torch, _ = env
    cache = {}

    def get(cfg):
        if cfg not in cache:
            need(torch, 4 * 27 * 8 * N_SPLIT + 12 * GB)
            P = torch.from_numpy(np.ascontiguousarray(so.synthetic_params(N_SPLIT, cfg, seed=70 + cfg).T)).cuda()
            for r in BC_GEN + ([16, 17] if cfg == 3 else BC_GEO):
                P[r].fill_(float(P[r, 0]))
            cache[cfg] = P
        return cache[cfg]
    yield get
    cache.clear()
    release(torch)


def oracle(P, sensor, band_mode="interp", soil=None, lib=None):
    """[n, nb, 3] oracle outputs and the (0, 1) canopy mask; lib: per-sample library index in row 9 (invalid -> NaN)."""
    kw = dict(band_mode=band_mode, return_canopy=True)
    if lib is None:
        want, rv = so.spart_bands(P, sensor, soil_rdry=soil, **kw)
    else:
        k = P[:, 9]
        nb = len(so.load_sensor(sensor)["wl_smac"])
        want, rv = np.full((P.shape[0], nb, 3), np.nan), np.full((P.shape[0], nb, 4), np.nan)
        for j in range(lib.shape[0]):
            sel = k == j
            if sel.any():
                want[sel], rv[sel] = so.spart_bands(P[sel], sensor, soil_rdry=lib[j], **kw)
    return want, ((rv > 0) & (rv < 1)).all(axis=2)


def check_rows(got, want, ok, fp32, what):
    if not fp32:
        assert relerr(got, want) < RTOL64, what
        return
    valid = np.broadcast_to(ok[..., None], got.shape)
    assert valid.mean() > 0.95, what
    with np.errstate(all="ignore"):
        e = np.abs(got - want) / np.abs(want)
    assert e[valid].max() < RTOL32, what


@pytest.mark.parametrize("mode", list(MODES))
def test_band_paths_past_one_launch(env, split_params, mode):
    """n = 2 MAX + 1000 (three calls, the last ragged): boundary and random samples against the oracle and against
    a small batch; the same batch with every broadcast row NaN after element 0 gives the same bits (each call must
    read the batch's element 0, not the first column of its own slice)."""
    torch, sb = env
    sensor, cfg, bc, kw, soil, f32 = MODES[mode]
    eng = sb.default_engine()
    base = split_params(cfg)
    need(torch, 2 * 27 * 8 * N_SPLIT + 3 * N_SPLIT * 13 * 3 * 8 + 4 * GB)
    row9 = base[9].clone()
    extra = {}
    lib = None
    try:
        if soil == "spectrum":
            extra["soil_spectrum"] = synthetic_spectra(1, seed=5)[0]
        elif soil == "library":
            lib = synthetic_spectra(8, seed=6)
            extra["soil_library"] = sb.SoilLibrary(lib)
            if 9 in bc:
                base[9].fill_(5.0)
            else:
                g = torch.Generator(device="cuda").manual_seed(9)
                base[9].copy_(torch.randint(0, 8, (N_SPLIT,), generator=g, device="cuda").double())
                for i, v in BAD_INDEX.items():
                    base[9, i] = v
        P = base.float() if f32 else base
        a = eng.forward_bands(P, sensor, broadcast_rows=bc, **kw, **extra)
        Pn = P.clone()
        Pn[bc, 1:] = float("nan")
        b = eng.forward_bands(Pn, sensor, broadcast_rows=bc, **kw, **extra)
        torch.cuda.synchronize()
        assert same_bits(torch, a, b), f"{mode}: broadcast rows read beyond element 0"
        del Pn, b
        idx = pick(N_SPLIT, (MAX, 2 * MAX), seed=len(mode), extra=list(BAD_INDEX) if lib is not None else ())
        tidx = torch.from_numpy(idx).cuda()
        small = eng.forward_bands(P[:, tidx].contiguous(), sensor, broadcast_rows=bc, **kw, **extra)
        got = a[tidx]
        assert same_bits(torch, small, got), f"{mode}: a sample's bits depend on its position in the batch"
        Ph = P[:, tidx].double().T.cpu().numpy()
        if 9 in bc:
            Ph[:, 9] = Ph[0, 9]
        want, ok = oracle(Ph, sensor, kw.get("band_mode", "interp"), extra.get("soil_spectrum"),
                          None if lib is None else lib)
        if lib is not None and 9 not in bc:
            assert np.isnan(want[np.isin(idx, list(BAD_INDEX))]).all()
        check_rows(got.double().cpu().numpy(), want, ok, "precision" in kw, mode)
    finally:
        base[9].copy_(row9)
        a = b = small = got = P = None
        release(torch)


def test_band_path_at_one_launch(env, split_params):
    """n = MAX (one call, grid.y = 65535) and MAX + 1 (a second call of one sample), as column views of a wider
    batch (ld > n): the same bits as the three-call run's first samples, and the oracle at the edges."""
    torch, sb = env
    eng = sb.default_engine()
    P = split_params(3)
    bc = BC_GEN + [16, 17]
    ref = eng.forward_bands(P[:, :MAX + 2], "LANDSAT8-OLI", broadcast_rows=bc)
    for n in (MAX, MAX + 1):
        got = eng.forward_bands(P[:, :n], "LANDSAT8-OLI", broadcast_rows=bc)
        torch.cuda.synchronize()
        assert same_bits(torch, got, ref[:n]), n
        idx = torch.tensor(boundaries(n, (MAX,)), device="cuda")
        want = so.spart_bands(P[:, idx].T.cpu().numpy(), "LANDSAT8-OLI")
        assert relerr(got[idx].cpu().numpy(), want) < RTOL64, n
    del ref, got
    release(torch)


# ------------------------------------------------------------------------------- B. refusals at the limit
def test_refusals_past_the_call_limit(env):
    torch, sb = env
    from spart_b200 import _lib
    eng = sb.default_engine()
    n = MAX + 1
    need(torch, 27 * 8 * n + n * 13 * 2 * 8 + GB)
    P = torch.zeros((27, n), dtype=torch.float64, device="cuda")
    for kw in (dict(compact=True), dict(reuse_record=True), dict(lidf=np.full(13, 1 / 13))):
        with pytest.raises(ValueError):
            eng.forward_bands(P, "Sentinel2A-MSI", **kw)
    with pytest.raises(ValueError):
        eng.forward_bands_multi(P, ["Sentinel2A-MSI", "Sentinel2B-MSI"])
    del P
    release(torch)
    # direct C calls with dummy buffers: the size check rejects them before anything is read
    lib = _lib.load()
    handle, _ = eng.sensor("Sentinel2A-MSI")
    buf = torch.zeros(64, dtype=torch.float64, device="cuda")
    p, s = buf.data_ptr(), torch.cuda.current_stream().cuda_stream
    calls = {
        "spart_forward_bands": lambda: lib.spart_forward_bands(handle, 0, p, n, n, 0, _lib.FP64, 0, p, p, s),
        "spart_forward_bands_bc": lambda: lib.spart_forward_bands_bc(handle, 0, p, p, n, n, 0, _lib.FP64, 0, p, p, s),
        "spart_smac": lambda: lib.spart_smac(handle, 0, p, n, n, p, p, s),
        "spart_sailh": lambda: lib.spart_sailh(handle, p, n, n, p, p, p, 0, p, p, s),
        "spart_forward_spectrum": lambda: lib.spart_forward_spectrum(handle, p, n, n, 0, 0.01, 0.01, p, p, s),
    }
    for name, call in calls.items():
        assert call() == -1, name                                     # SPART_EINVAL
        msg = lib.spart_last_error().decode()
        assert "split the batch" in msg, (name, msg)
    assert lib.spart_forward_bands(handle, 0, p, n - 1, n, 0, _lib.FP64, 0, 0, p, s) == -1     # null workspace
    assert "null argument" in lib.spart_last_error().decode()
    assert lib.spart_forward_bands_bc(handle, 0, p, None, 1, 1, 0, _lib.FP64, 0, p, p, s) == -1
    assert "null broadcast base" in lib.spart_last_error().decode()


# ------------------------------------------------------------- C. full-spectrum paths past 65535 samples / 2^31
SPEC_NAMES = ["leaf_refl", "leaf_tran", "kChlrel", "soil_refl", "soil_refl_dry", "rso", "rdo", "rsd", "rdd"]


def check_spectra(got, want, names, what):
    rv = np.stack([want[k] for k in ("rso", "rdo", "rsd", "rdd")], axis=2)
    canopy_ok = ((rv > 0) & (rv < 1)).all(axis=2)
    for i, k in enumerate(names):
        w = want[k]
        scale = None
        if k in ("rso", "rdo", "rsd", "rdd"):
            scale = np.where(canopy_ok, np.abs(w), np.maximum(np.abs(w), 1.0))
        check_close(got[:, i, :w.shape[1]], w, RTOL64, scale, f"{what} {k}")


def test_forward_spectrum_three_slices(env):
    """n = 2 * 65535 + 3: three grid.y slices, 20 GB of output; element 2^31 falls in sample 110 365."""
    torch, sb = env
    n = 2 * 65535 + 3
    need(torch, n * 9 * 2162 * 8 + 4 * GB)
    assert (n * 9 * 2162) > 2 ** 31 and 110365 * 9 * 2162 <= 2 ** 31 < 110366 * 9 * 2162
    P = so.synthetic_params(n, 3, seed=81)
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    eng = sb.default_engine()
    out = eng.forward_spectrum(dev)
    idx = pick(n, (65535, 131070), k=200, extra=(110364, 110365, 110366))
    tidx = torch.from_numpy(idx).cuda()
    got = out[tidx]
    del out
    release(torch)
    small = eng.forward_spectrum(dev[:, tidx].contiguous())
    assert same_bits(torch, small, got)
    check_spectra(got.cpu().numpy(), so.canopy_spectra(P[idx]), SPEC_NAMES, "forward_spectrum")
    del dev, got, small
    release(torch)


@pytest.mark.parametrize("per_sample", [False, True])
def test_sailh_past_one_slice(env, per_sample):
    """n = 65537: two grid.y slices, shared spectra and per-sample [n, 2162] spectra."""
    torch, sb = env
    n = 65537
    need(torch, n * 2162 * 8 * 7 + 2 * GB)
    P = so.synthetic_params(n, 3, seed=82)
    eng = sb.default_engine()
    base = so.canopy_spectra(so.synthetic_params(64, 3, seed=83))
    spec = [torch.from_numpy(base[k]).cuda() for k in ("soil_refl", "leaf_refl", "leaf_tran")]
    which = np.arange(n) % 64 if per_sample else np.zeros(n, dtype=np.int64)
    if per_sample:
        tw = torch.from_numpy(which).cuda()
        args = [s[tw].contiguous() for s in spec]
    else:
        args = [s[0].contiguous() for s in spec]
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    out = eng.sailh(dev, *args)
    idx = pick(n, (65535,), k=200)
    tidx = torch.from_numpy(idx).cuda()
    got = out[tidx]
    del out
    sargs = [a[tidx].contiguous() for a in args] if per_sample else args
    small = eng.sailh(dev[:, tidx].contiguous(), *sargs)
    assert same_bits(torch, small, got)
    w = which[idx]
    with np.errstate(all="ignore"):
        want = so.sailh(base["soil_refl"][w], base["leaf_refl"][w], base["leaf_tran"][w],
                        P[idx, so.LAI:so.HOT_Q + 1], P[idx, so.SZA:so.RAA + 1])
    check_spectra(got.cpu().numpy(), dict(zip(("rso", "rdo", "rsd", "rdd"), want)), ["rso", "rdo", "rsd", "rdd"],
                  "sailh")
    del dev, args, sargs, got, small
    release(torch)


def test_fullspectrum_sensor_fp64_past_2_31(env):
    """The synthetic 2001-band sensor in FP64 at n = 360 000 (17 GB): element 2^31 falls in sample 357 735."""
    torch, sb = env
    n, nb = 360_000, 2001
    need(torch, n * nb * 3 * 8 + 4 * GB)
    assert 357735 * nb * 3 <= 2 ** 31 < 357736 * nb * 3
    info = sb.synthetic_fullspectrum_sensorinfo()
    P = so.synthetic_params(n, 4, seed=84)
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    eng = sb.default_engine()
    out = eng.forward_bands(dev, info)
    idx = pick(n, (), k=200, extra=(357734, 357735, 357736))
    tidx = torch.from_numpy(idx).cuda()
    got = out[tidx]
    del out
    release(torch)
    small = eng.forward_bands(dev[:, tidx].contiguous(), info)
    assert same_bits(torch, small, got)
    assert relerr(got.cpu().numpy(), so.spart_bands(P[idx], info)) < RTOL64
    del dev, got, small
    release(torch)


def test_fullspectrum_sensor_fp32_compact_past_2_31(env):
    """FP32 with float I/O and compact output at n = 540 000: the [n][nb][2] part passes 2^31 elements at sample
    536 602, and the whole etscale tail (from element 2.16e9) lies beyond 2^31."""
    torch, sb = env
    n, nb = 540_000, 2001
    need(torch, (n * nb * 2 + n) * 4 + 4 * GB)
    assert 536602 * nb * 2 <= 2 ** 31 < 536603 * nb * 2 and n * nb * 2 > 2 ** 31
    info = sb.synthetic_fullspectrum_sensorinfo()
    P = so.synthetic_params(n, 4, seed=85).astype(np.float32)
    dev = torch.from_numpy(np.ascontiguousarray(P.T)).cuda()
    eng = sb.default_engine()
    res = eng.forward_bands(dev, info, precision="fp32", compact=True)
    idx = pick(n, (), k=200, extra=(536601, 536602, 536603))
    tidx = torch.from_numpy(idx).cuda()
    R, ets = res.R[tidx], res.etscale[tidx]
    del res
    release(torch)
    small = eng.forward_bands(dev[:, tidx].contiguous(), info, precision="fp32", compact=True)
    assert same_bits(torch, small.R, R) and same_bits(torch, small.etscale, ets)
    got = small.full().double().cpu().numpy()
    want, ok = oracle(P[idx].astype(np.float64), info)
    check_rows(got, want, ok, True, "fp32 compact 2001 bands")
    del dev, R, ets, small
    release(torch)


# -------------------------------------------------------------- D. host path and pipelined sharding past the split
def test_host_path_past_the_split(env, split_params):
    """forward_bands_host at n = MAX + 1000 with broadcast rows NaN after element 0: the device path's bits."""
    torch, sb = env
    n = MAX + 1000
    bc = BC_GEN + BC_GEO
    need(torch, 27 * 8 * n + 2 * n * 13 * 3 * 8 + 4 * GB)
    eng = sb.default_engine()
    P = split_params(2)[:, :n].contiguous()
    dev = eng.forward_bands(P, "Sentinel2A-MSI", broadcast_rows=bc)
    Ph = P.cpu().numpy()
    del P
    Ph[bc, 1:] = np.nan
    host = eng.forward_bands_host(Ph, "Sentinel2A-MSI", broadcast_rows=bc)
    assert same_bits(torch, torch.from_numpy(host).cuda(), dev)
    del dev, host, Ph
    release(torch)


def test_pipelined_sharding_reads_the_shard_broadcast_base(env, tmp_path):
    """run_batch_sharded_pipelined on a world-size-1 NCCL group, chunk < n_local with a one-sample last chunk,
    broadcast rows NaN after element 0: equal to one forward_bands run on full rows."""
    torch, sb = env
    import torch.distributed as dist
    from spart_b200.distributed import run_batch_sharded_pipelined
    n, chunk = 10 * 4096 + 1, 4096
    bc = BC_GEN + BC_GEO
    P = torch.from_numpy(np.ascontiguousarray(so.synthetic_params(n, 2, seed=86).T)).cuda()
    want = sb.default_engine().forward_bands(P, "Sentinel2A-MSI", broadcast_rows=bc)
    Pn = P.clone()
    Pn[bc, 1:] = float("nan")
    dist.init_process_group("nccl", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1,
                            device_id=torch.device("cuda", torch.cuda.current_device()))
    try:
        res = run_batch_sharded_pipelined(Pn, "Sentinel2A-MSI", chunk=chunk, dst=0, broadcast_rows=bc)
        torch.cuda.synchronize()
        assert len(res) == 1 and len(res[0]) == 11 and res[0][-1].shape[0] == 1
        assert same_bits(torch, torch.cat(res[0]), want)
    finally:
        dist.destroy_process_group()
    del P, Pn, want, res
    release(torch)


# ------------------------------------------------------------------------ E. LUT search at its size and index limits
def retrieval_case(torch, n, m, nb, seed):
    """A table of smooth-ish rows and observations that are noisy copies of random rows (near neighbours, near
    ties), every 17th observation uniform random."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    L = torch.rand((n, nb), generator=g, device="cuda", dtype=torch.float32)
    pick_ = torch.randint(0, n, (m,), generator=g, device="cuda")
    O = (L[pick_] + 1e-3 * torch.randn((m, nb), generator=g, device="cuda")).float()
    O[::17] = torch.rand((O[::17].shape[0], nb), generator=g, device="cuda")
    return L, O


def checked_obs(m):
    """Observations verified against the brute force: all of them up to 600, otherwise the block edges and 300 more."""
    if m <= 600:
        return np.arange(m)
    return pick(m, (128, 256, 512, m - 128), k=300, seed=m)


def fp32_cost(torch, O, L):
    """The kernels' FP32 cost of each (observation, entry) row pair, unweighted: d = o - l in float, even bands
    fused-multiply-added into c0, odd ones into c1, then c0 + c1 (d * d is exact in double, so one rounding of
    the double sum to float is the fma)."""
    d = (O - L).double()
    c = [torch.zeros(O.shape[0], dtype=torch.float64, device=O.device) for _ in range(2)]
    for b in range(O.shape[1]):
        c[b & 1] = (d[:, b] * d[:, b] + c[b & 1]).float().double()
    return (c[0].float() + c[1].float())


def brute_min(torch, L, Oc):
    """float64 minimum of sum_b (o_b - l_b)^2 over the whole table, chunked."""
    best = torch.full((Oc.shape[0],), float("inf"), dtype=torch.float64, device=L.device)
    Od = Oc.double()
    for s0 in range(0, L.shape[0], 1 << 20):
        d = torch.cdist(Od, L[s0:s0 + (1 << 20)].double(), compute_mode="donot_use_mm_for_euclid_dist")
        best = torch.minimum(best, d.min(dim=1).values ** 2)
    return best


def check_search(torch, L, O, idx, cost, method, what, sel=None, best=None):
    """The chosen entries of the checked observations against the float64 brute force: within FP32 rounding of the
    minimum (exact) or within the 3xTF32 bound of test_gpu_abi5 (tensor); the reported cost is the entry's FP32
    cost bit for bit.  best: precomputed brute_min of O[sel]."""
    sel = torch.from_numpy(checked_obs(O.shape[0]) if sel is None else sel).cuda()
    Oc, i = O[sel], idx[sel]
    assert bool(((i >= 0) & (i < L.shape[0])).all()), what
    Lc = L[i]
    chosen = ((Oc.double() - Lc.double()) ** 2).sum(1)
    if best is None:
        best = brute_min(torch, L, Oc)
    nb = L.shape[1]
    if method == "exact":
        ok = chosen <= best * (1 + (nb + 2) * 2.0 ** -22)
    else:
        scale = Oc.double().norm(dim=1).max() * L.double().norm(dim=1).max()
        ok = chosen <= best + 4e-6 * scale
    assert bool(ok.all()), f"{what}: {int((~ok).sum())} observations with a worse entry"
    assert same_bits(torch, cost[sel], fp32_cost(torch, Oc, Lc)), f"{what}: reported cost is not the entry's FP32 cost"


N_GRID = [1, 127, 128, 129, 128 * 1184 - 1, 128 * 1184 + 1, 2 ** 24 + 3]
M_GRID = [1, 255, 256, 257, 65537]
NB_GRID = [1, 4, 5, 13, 26, 30, 32]


@pytest.mark.parametrize("n", N_GRID)
def test_lut_shape_grid(env, n):
    """Both methods over m x nb (nb = 32 exact only): m = 1 gives the search the most table slices, large m one."""
    torch, sb = env
    from spart_b200 import lut
    need(torch, n * 32 * 4 * 3 + 4 * GB)
    every = np.unique(np.concatenate([checked_obs(m) for m in M_GRID]))
    for nb in NB_GRID:
        L, O = retrieval_case(torch, n, max(M_GRID), nb, seed=n + nb)
        best = brute_min(torch, L, O[torch.from_numpy(every).cuda()])      # once for the observations of every m
        for m in M_GRID:
            sel = checked_obs(m)
            b = best[torch.from_numpy(np.searchsorted(every, sel)).cuda()]
            for method in (("exact",) if nb > 30 else ("exact", "tensor")):
                idx, cost = lut.nearest(L, O[:m].contiguous(), method=method)
                check_search(torch, L, O[:m], idx, cost, method, f"n={n} m={m} nb={nb} {method}", sel, b)
        del L, O, best
    release(torch)


@pytest.mark.parametrize("method", ["exact", "tensor"])
def test_lut_weighted_search_at_scale(env, method):
    torch, sb = env
    from spart_b200 import lut
    n, m, nb = 128 * 1184 + 1, 4099, 13
    L, O = retrieval_case(torch, n, m, nb, seed=7)
    w = torch.rand(nb, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8)) + 0.1
    idx, cost = lut.nearest(L, O, w, method=method)
    sw = w.sqrt()
    sel = torch.from_numpy(checked_obs(m)).cuda()
    # in the scaled space (entries and observations times sqrt(w), as the kernels form them) the search is unweighted
    Ls, Os = L.double() * sw.double(), O[sel].double() * sw.double()
    chosen = ((Os - Ls[idx[sel]]) ** 2).sum(1)
    best = brute_min(torch, Ls.float(), Os.float())
    # the kernels round o sqrt(w) and l sqrt(w) to float: each difference d_b moves by up to 2^-22 |o_b| or so, the
    # cost by up to 2 |d| |delta| <= 2^-21 sqrt(cost) |o| (Cauchy-Schwarz)
    rnd = 2.0 ** -21 * Os.norm(dim=1)
    if method == "exact":
        tol = 1e-5 * best + 2 * rnd * best.sqrt() + 1e-12
    else:
        tol = 4e-6 * Os.norm(dim=1).max() * Ls.norm(dim=1).max()
    assert bool((chosen <= best + tol).all())
    c = cost[sel].double()
    assert bool(((c - chosen).abs() <= 1e-4 * chosen + rnd * chosen.sqrt() + 1e-12).all())


@pytest.mark.parametrize("method", ["exact", "tensor"])
@pytest.mark.parametrize("m", [1, 300, 5000])
def test_lut_ties_go_to_the_first_copy(env, method, m):
    """Three stacked copies of one table: the index found lies in the first copy and is the one-copy result; with
    small m the copies lie in different table slices."""
    torch, sb = env
    from spart_b200 import lut
    T, O = retrieval_case(torch, 1000, m, 13, seed=m)
    O[: min(m, 64)] = T[: min(m, 64)]                       # exact self-matches, cost 0 in every copy
    one = lut.nearest(T, O, method=method)
    three = lut.nearest(torch.cat([T, T, T]).contiguous(), O, method=method)
    assert torch.equal(three[0], one[0]) and same_bits(torch, three[1], one[1])
    assert bool((three[0] < 1000).all())


@pytest.mark.parametrize("method", ["exact", "tensor"])
def test_lut_index_limit(env, method):
    """index_offset + n = 2^32 - 1 is accepted and returns index_offset + local; 2^32 is refused."""
    torch, sb = env
    from spart_b200 import lut
    L, O = retrieval_case(torch, 1000, 300, 13, seed=3)
    idx0, cost0 = lut._search(L, O, None, 0, packed=False, method=method)
    off = 2 ** 32 - 1 - 1000
    idx, cost = lut._search(L, O, None, off, packed=False, method=method)
    assert torch.equal(idx, idx0 + off) and same_bits(torch, cost, cost0)
    assert int(idx.max()) <= 2 ** 32 - 2
    with pytest.raises(sb.SpartError):
        lut._search(L, O, None, off + 1, packed=False, method=method)


@pytest.mark.parametrize("method", ["exact", "tensor"])
def test_lut_nan_rows_and_no_entry(env, method):
    """NaN table rows are never chosen; an observation with a NaN, or against an all-NaN table, gets the documented
    "no entry" result (index 2^32 - 1, cost NaN) -- also when the table ends in a partial tile."""
    torch, sb = env
    from spart_b200 import lut
    L, O = retrieval_case(torch, 5000, 700, 13, seed=4)
    nan_rows = torch.zeros(5000, dtype=torch.bool, device="cuda")
    nan_rows[::7] = True
    nan_rows[L[:, 0] > 0.9] = True
    Ln = L.clone()
    Ln[nan_rows, 3] = float("nan")
    O[5, 2] = float("nan")
    idx, cost = lut.nearest(Ln, O, method=method)
    keep = torch.nonzero(~nan_rows)[:, 0]
    idx_c, cost_c = lut.nearest(L[keep].contiguous(), O, method=method)
    live = torch.ones(700, dtype=torch.bool, device="cuda")
    live[5] = False
    assert int(idx[5]) == NO_ENTRY and bool(torch.isnan(cost[5]))
    assert not bool(nan_rows[idx[live]].any())
    if method == "exact":
        assert torch.equal(idx[live], keep[idx_c[live]]) and same_bits(torch, cost[live], cost_c[live])
    else:
        check_search(torch, L[keep].contiguous(), O[live], torch.searchsorted(keep, idx[live]), cost[live], method,
                     "nan rows")
    for n in (128, 129, 1000):
        idx, cost = lut.nearest(torch.full((n, 13), float("nan"), device="cuda"), O, method=method)
        assert bool((idx == NO_ENTRY).all()) and bool(torch.isnan(cost).all()), n


@pytest.mark.parametrize("method", ["exact", "tensor"])
def test_lut_all_nan_shard_loses_the_reduction(env, method):
    """Packed pieces of a sharded search on one GPU: an all-NaN piece next to a valid one gives the valid piece's
    entry after the signed min-reduction, and "no entry" where neither piece has one."""
    torch, sb = env
    from spart_b200 import lut
    L, O = retrieval_case(torch, 3000, 400, 13, seed=5)
    O[7, 0] = float("nan")
    bad = torch.full((1001, 13), float("nan"), device="cuda")
    w0 = lut.for_min_reduction(lut._search(bad, O, None, 0, packed=True, method=method))
    w1 = lut.for_min_reduction(lut._search(L, O, None, 1001, packed=True, method=method))
    idx, cost = lut.unpack(torch.minimum(w0, w1))
    i1, c1 = lut.nearest(L, O, method=method)
    live = torch.ones(400, dtype=torch.bool, device="cuda")
    live[7] = False
    assert torch.equal(idx[live], i1[live] + 1001) and same_bits(torch, cost[live], c1[live])
    assert int(idx[7]) == NO_ENTRY and bool(torch.isnan(cost[7]))
