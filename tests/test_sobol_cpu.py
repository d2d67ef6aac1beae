"""CPU checks of the sensitivity analysis: the refusals of `ParameterSpace`, the C-ABI symbols, the design rule
restated in NumPy (from the direction numbers the kernel compiles in) against scipy.stats.qmc.Sobol, and the
reduction of `sobol(group=...)` over gloo at world size 2, with NumPy stand-ins for the design, forward and
estimator kernels.  The NumPy restatement of the scrambled design here is also the reference of the GPU tests."""
import os
import re
import socket
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

sys.path.insert(0, str(ROOT / "spart-python_b200"))

DIRS_H = ROOT / "spart-python_b200" / "csrc" / "sobol_dirs.h"
GAMMA = 0x9E3779B97F4A7C15
M64 = (1 << 64) - 1


def direction_numbers():
    """SPART_SOBOL_V of the generated header, uint32 [64, 32]."""
    words = re.findall(r"0x([0-9a-f]{8})u", DIRS_H.read_text())
    return np.array([int(w, 16) for w in words], dtype=np.uint32).reshape(64, 32)


def _splitmix(state):
    state = (state + GAMMA) & M64
    z = state
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return state, z ^ (z >> 31)


def scramble(v, seed, dim):
    """(L_dim v, s_dim): dimension dim draws words 32 dim .. 32 dim + 31 of the SplitMix64 stream of seed."""
    state = (seed + 32 * dim * GAMMA) & M64
    row = [1 << 31]
    for r in range(1, 32):
        state, w = _splitmix(state)
        row.append(((w & ((1 << r) - 1)) << (32 - r)) | (1 << (31 - r)))
    state, w = _splitmix(state)
    out = [sum((bin(rw & int(x)).count("1") & 1) << (31 - r) for r, rw in enumerate(row)) for x in v]
    return np.array(out, dtype=np.uint32), np.uint32(w & 0xFFFFFFFF)


def points(v, shift, first, count):
    """k_d(i) for i = first .. first + count - 1: uint32 [count, D] from v [D, 32] and shift [D]."""
    i = np.arange(first, first + count, dtype=np.uint64)
    g = i ^ (i >> np.uint64(1))
    k = np.tile(np.asarray(shift, dtype=np.uint32), (count, 1))
    for j in range(32):
        on = ((g >> np.uint64(j)) & np.uint64(1)).astype(bool)
        k[on] ^= v[:, j]
    return k


def values(k, lo, hi):
    """lo + (hi - lo) u, u = k 2^-32, moved below hi if it rounds up to it."""
    lo, hi = np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)
    x = lo + (hi - lo) * (k.astype(np.float64) * 2.0 ** -32)
    return np.where(x < hi, x, np.nextafter(hi, lo))


def design_np(rows, lo, hi, seed, scramble_on, first, count, saltelli):
    """The varied rows the design kernel writes: dict row -> float64 [count] (saltelli 0) or [(d + 2) count]."""
    d = len(rows)
    D = 2 * d if saltelli else d
    v = direction_numbers()[:D].copy()
    s = np.zeros(D, dtype=np.uint32)
    if scramble_on:
        for dim in range(D):
            v[dim], s[dim] = scramble(v[dim], seed, dim)
    k = points(v, s, first, count)
    xa = values(k[:, :d], lo, hi)
    if not saltelli:
        return {r: xa[:, p] for p, r in enumerate(rows)}
    xb = values(k[:, d:], lo, hi)
    out = {}
    for p, r in enumerate(rows):
        out[r] = np.concatenate([xa[:, p], xb[:, p]] + [xb[:, p] if i == p else xa[:, p] for i in range(d)])
    return out


# ---- ParameterSpace ------------------------------------------------------------------------------------------

BASE = np.array([40, 0.01, 0.02, 0.1, 10, 1, 1.5, 0, 0, 0.5, 10, 100, 20, 25, 0.015, 3, -0.35, -0.15, 0.05,
                 40, 0, 0, 0.3, 0.35, 1.5, 1013, 180], dtype=np.float64)


@pytest.mark.parametrize("vary, match", [
    ({"Chl": (1, 2)}, "unknown parameter row"),
    ({27: (1, 2)}, "unknown parameter row"),
    ({-1: (1, 2)}, "unknown parameter row"),
    ({"Cab": (10, 80), 0: (5, 6)}, "varied twice"),
    ({"Cab": (80, 10)}, "lo < hi"),
    ({"Cab": (10, 10)}, "lo < hi"),
    ({"Cab": (10, np.inf)}, "lo < hi"),
    ({"Cab": (np.nan, 1)}, "lo < hi"),
    ({"LIDFa": (-0.9, 0.5)}, "LIDFa"),                         # 0.9 + |fixed LIDFb| 0.15 > 1
    ({"LIDFa": (-0.5, 0.5), "LIDFb": (-0.6, 0.2)}, "LIDFa"),
    ({}, "1 to 27"),
    ({**{n: (0, 1) for n in range(27)}, "DOY": (1, 2)}, "1 to 27"),    # 28 entries
])
def test_parameter_space_refusals(vary, match):
    from spart_b200.sensitivity import ParameterSpace
    with pytest.raises(ValueError, match=match):
        ParameterSpace(BASE, vary)


def test_parameter_space_accepts_and_describes():
    from spart_b200.sensitivity import ParameterSpace
    sp = ParameterSpace(BASE[:, None], {"LAI": (0.1, 8), 0: (5, 80), "LIDFa": (-0.5, 0.5), "LIDFb": (-0.5, 0.5)})
    assert sp.names == ("LAI", "Cab", "LIDFa", "LIDFb") and sp.d == 4
    assert list(sp.rows) == [15, 0, 16, 17]
    assert sp.broadcast_rows == ((1 << 27) - 1) & ~((1 << 15) | 1 | (1 << 16) | (1 << 17))
    with pytest.raises(ValueError, match="27 parameter rows"):
        ParameterSpace(BASE[:26], {"LAI": (0, 1)})
    with pytest.raises(ValueError, match="finite"):
        ParameterSpace(np.where(np.arange(27) == 3, np.nan, BASE), {"LAI": (0, 1)})
    ParameterSpace(np.where(np.arange(27) == 3, np.nan, BASE), {"Cs": (0, 1)})     # a varied row's base is unused


def test_exports_declare_the_sobol_entry_points():
    from spart_b200 import _lib
    header = (ROOT / "include" / "spart_b200.h").read_text()
    lib = _lib.load()
    for sym in ("spart_sobol_design", "spart_sobol_acc_elems", "spart_sobol_accumulate", "spart_sobol_finish"):
        assert sym in _lib.EXPORTS and re.search(rf"\b{sym}\s*\(", header) and hasattr(lib, sym)
    assert lib.spart_sobol_acc_elems(39, 19) == 128 * 20 * 39 * 8
    assert lib.spart_sobol_acc_elems(39, 28) == 0 and lib.spart_sobol_acc_elems(0, 3) == 0


# ---- design rule ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("first", [0, 12345, 2 ** 20 + 3])
def test_unscrambled_rule_equals_scipy(first):
    from scipy.stats import qmc
    v = direction_numbers()
    for D in range(2, 55):
        eng = qmc.Sobol(D, scramble=False, bits=32)
        if first:
            eng.fast_forward(first)
        want = eng.random(512)
        got = points(v[:D], np.zeros(D, dtype=np.uint32), first, 512).astype(np.float64) * 2.0 ** -32
        assert np.array_equal(got, want), D


def test_scramble_rule_is_per_dimension_and_keeps_nets():
    v = direction_numbers()
    a, sa = scramble(v[5], 7, 5)
    assert not np.array_equal(a, v[5])
    # L is unit lower-triangular: the leading bit of each column is unchanged
    for x, y in zip(v[5], a):
        assert int(x).bit_length() == int(y).bit_length()
    # the design of d parameters is a prefix of the design of more: dimension d's scramble ignores D
    one = design_np([0, 4], [0, 0], [1, 1], 99, True, 0, 64, 0)
    two = design_np([0, 4, 9], [0, 0, 0], [1, 1, 1], 99, True, 0, 64, 0)
    assert np.array_equal(one[0], two[0]) and np.array_equal(one[4], two[4])
    # net property: the first 2^m points fall one per interval of width 2^-m
    u = design_np([0, 1, 2], [0] * 3, [1] * 3, 3, True, 0, 1024, 0)
    for x in u.values():
        for m in range(11):
            assert np.array_equal(np.sort(np.floor(x[:2 ** m] * 2 ** m)), np.arange(2 ** m))


# ---- sharded reduction over gloo -----------------------------------------------------------------------------

ROWS = [0, 15, 22]
LO, HI = np.array([-np.pi] * 3), np.array([np.pi] * 3)
NB = 2


def _space():
    from spart_b200.sensitivity import ParameterSpace
    return ParameterSpace(BASE, {r: (-np.pi, np.pi) for r in ROWS})


def _design(space, count, seed, first):
    d = space.d
    P = np.full((27, (d + 2) * count), np.nan)
    P[:, 0] = space.base
    for r, x in design_np(ROWS, LO, HI, seed, True, first, count, 1).items():
        P[r] = x
    return torch.from_numpy(P)


def _forward(P):
    """An Ishigami-like model with NB bands x 3 outputs."""
    x = P.numpy()[ROWS]
    f = np.sin(x[0]) + 7 * np.sin(x[1]) ** 2 + 0.1 * x[2] ** 4 * np.sin(x[0])
    out = np.stack([f, 2 * f + x[1], f - 3, x[0], f * f, np.cos(x[2])], axis=-1)
    return torch.from_numpy(out.reshape(-1, NB, 3).copy())


def _accumulate(f, n, d, ref, acc):
    """NumPy stand-in: acc[:n_out * (2 + 2 d)] holds per output the sums of f and f^2, then per parameter those
    of f_B D and D^2 (D = f_ABi - f_A).  Unshifted: the stand-in values are O(1)."""
    F = f.numpy().reshape(d + 2, n, -1)
    n_out = F.shape[2]
    a = acc.numpy()[:n_out * (2 + 4 * d)].reshape(n_out, 2 + 4 * d)
    fab = np.concatenate([F[0], F[1]])
    a[:, 0] += fab.sum(0)
    a[:, 1] += (fab * fab).sum(0)
    for i in range(d):
        D = F[2 + i] - F[0]
        a[:, 2 + 4 * i:6 + 4 * i] += np.stack([(F[1] * D).sum(0), D.sum(0), (D * D).sum(0), (D ** 4).sum(0)], -1)


def _finish(acc, ref, N, d):
    n_out = ref.shape[1]
    a = acc.numpy()[:n_out * (2 + 4 * d)].reshape(n_out, 2 + 4 * d)
    mean = a[:, 0] / (2 * N)
    V = a[:, 1] / (2 * N) - mean ** 2
    s = a[:, 2:].reshape(n_out, d, 4) / N
    first = (s[..., 0] - mean[:, None] * s[..., 1]) / V[:, None]
    total = s[..., 2] / (2 * V[:, None])
    nan = np.full_like(first, np.nan)                   # the stand-in skips the standard errors
    return [torch.from_numpy(np.ascontiguousarray(x)) for x in (mean, V, first, total, nan, nan)]


STAND_INS = dict(design=_design, forward=_forward, accumulate=_accumulate, finish=_finish)
N_BASE, CHUNK = 1024, 96


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    sys.path.insert(0, str(ROOT / "spart-python_b200"))
    from spart_b200 import sensitivity
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        # a refused call on both ranks enters no collective, so the next call's collectives still pair up
        try:
            sensitivity.sobol(_space(), None, N_BASE, chunk=0, group=dist.group.WORLD, **STAND_INS)
            refused = False
        except ValueError:
            refused = True
        res = sensitivity.sobol(_space(), None, N_BASE, seed=11, chunk=CHUNK, group=dist.group.WORLD, **STAND_INS)
        q.put((rank, [res.mean, res.var, res.first, res.total, res.first_se, res.total_se, refused]))
    finally:
        dist.destroy_process_group()


def test_sharded_sobol_gloo_world2_equals_one_rank():
    import torch.multiprocessing as mp
    from scipy.stats import sobol_indices
    from spart_b200 import sensitivity
    one = sensitivity.sobol(_space(), None, N_BASE, seed=11, chunk=CHUNK, **STAND_INS)
    assert one.names == ("Cab", "LAI", "aot550") and one.first.shape == (NB, 3, 3) and one.mean.shape == (NB, 3)
    # the stand-in run is the Saltelli estimator of the whole design
    f = _forward(_design(_space(), N_BASE, 11, 0)).numpy().reshape(5, N_BASE, -1).transpose(0, 2, 1)
    want = sobol_indices(func={"f_A": f[0], "f_B": f[1], "f_AB": f[2:]}, n=N_BASE)
    np.testing.assert_allclose(one.first.reshape(-1, 3), want.first_order, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(one.total.reshape(-1, 3), want.total_order, rtol=1e-9, atol=1e-12)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    ref = [one.mean, one.var, one.first, one.total, one.first_se, one.total_se]
    for r in (0, 1):
        assert res[r].pop() is True
        for got, want in zip(res[r], ref):
            np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-15)    # atol: means near 0
        for a, b in zip(res[r], res[0]):
            assert np.array_equal(a, b, equal_nan=True)     # the same result on every rank


@pytest.mark.parametrize("kw, match", [
    (dict(n=0), "1 <= n"), (dict(n=2 ** 32 + 1), "1 <= n"), (dict(chunk=0), "chunk"),
    (dict(precision="fp16"), "precision"), (dict(band_mode="box"), "band_mode"), (dict(seed=-1), "seed"),
    (dict(soil_library=object()), "soil_library"),
])
def test_sobol_refuses_before_any_collective(kw, match):
    """Refused on every rank before the first collective.  No process group exists here, so reaching one would
    fail with another error."""
    from spart_b200 import sensitivity
    args = dict(n=64, chunk=16) | kw
    with pytest.raises(ValueError, match=match):
        sensitivity.sobol(_space(), None, group=object(), **args, **STAND_INS)
