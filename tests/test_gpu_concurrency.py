"""The stream, thread and context-lifetime contract of every entry point.

include/spart_b200.h promises that the device entry points enqueue all their work on the caller's stream and
never allocate or synchronise per call, that a context may be used from several host threads at once, and that
the error text and the launch counter are per thread; `Engine` promises that its cached contexts stay valid for
the calls that use them.  On torch's legacy default stream with a synchronise after each call, none of this is
visible, so the tests here run on non-blocking side streams behind a GPU delay (`torch.cuda._sleep`, calibrated
with CUDA events to at least 100 ms) and from several host threads:

  A. stream order: inputs start as decoys (valid parameters of another seed); on the side stream s the delay,
     the copy of the real inputs, a NaN fill of the output, the call, a clone of the output and the decoys again
     are enqueued.  Work on any other stream would read decoys, write before the NaN fill or read after the
     overwrite.  Two controls show the harness sees a misordering.
  B. asynchrony: a warmed-up device call returns while s is still asleep (no host synchronise, no cudaMalloc /
     cudaFree on the call path).
  C. threads: a shuffled mix of the A jobs from 7 threads on one Engine, host-path jobs among them, argument
     errors on one thread, launch counts and profile counts per context; the SRF kernels' shared-memory cap.
  D. context lifetime: eviction while a call uses the context, and destruction with work still queued.
  E. the pipelined gather and the sharded search on a side stream.
  F. threads on two GPUs.

Every result must equal, bit for bit (NaN payloads included), the same call run serially on the default stream;
the oracle only checks that those serial baselines are sane (1e-9 in FP64, 1e-4 on valid FP32 outputs)."""
import ctypes
import random
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import spart_oracle as so  # noqa: E402
from test_gpu_batch_limits import check_rows, oracle  # noqa: E402
from test_gpu_soil_library import synthetic_spectra  # noqa: E402

N = 256                 # samples of a band job
N_SPEC = 24             # samples of a spectrum / SAILH job ([n, 9 or 4, 2162] outputs)
NAN = float("nan")
L8, S2A = "LANDSAT8-OLI", "Sentinel2A-MSI"


@pytest.fixture(scope="module")
def env():
    import torch
    import spart_b200
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    yield torch, spart_b200
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def cycles(env):
    """torch.cuda._sleep cycles of a delay of at least 100 ms, measured with CUDA events (the clock is not
    assumed)."""
    torch, _ = env
    c = 1 << 20
    for _ in range(12):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.cuda._sleep(c)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= 120.0:
            return c
        c = int(c * min(max(150.0 / max(ms, 1e-3), 1.5), 64.0))
    pytest.fail(f"torch.cuda._sleep({c}) lasted {ms:.1f} ms, not 100 ms")


def bits(t):
    """The integer view of a tensor (NaN-aware bit comparison)."""
    import torch
    t = t.contiguous()
    return t.view({torch.float64: torch.int64, torch.float32: torch.int32}.get(t.dtype, t.dtype))


def same(a, b):
    import torch
    return a.shape == b.shape and a.dtype == b.dtype and bool(torch.equal(bits(a), bits(b)))


def dev_params(torch, n, cfg, seed, rows_const=(), f32=False):
    P = np.ascontiguousarray(so.synthetic_params(n, cfg, seed=seed).T)
    for r in rows_const:
        P[r] = P[r, 0]
    t = torch.from_numpy(P).cuda()
    return t.float() if f32 else t


# ----------------------------------------------------------------------------------------------------------- jobs
class Job:
    """One entry-point call with buffers of its own.  `real` / `decoy`: device tensors that are only read;
    `bufs`: what the call reads (real or decoy values are copied in); `outs`: the result buffers it writes
    (NaN-filled before the call).  call(bufs, outs) enqueues the call on the current stream and returns the result
    tensors.  `base`, `launches`: result and spart_launch_count() delta of a serial run; `l8_calls`: forward_bands
    calls on the plain LANDSAT8-OLI context."""

    def __init__(self, name, real, decoy, outs, call, l8_calls=0):
        self.name, self.real, self.decoy, self.call, self.l8_calls = name, real, decoy, call, l8_calls
        self.bufs = [d.clone() for d in decoy]
        self.outs = outs
        self.base = self.launches = None

    def fresh(self):
        """A copy with buffers of its own (for another thread)."""
        j = Job(self.name, self.real, self.decoy, [o.clone() for o in self.outs], self.call, self.l8_calls)
        j.base, j.launches = self.base, self.launches
        return j

    def load(self, src):
        for b, x in zip(self.bufs, src):
            b.copy_(x)

    def enqueue(self, after_call=None):
        """Real inputs in, NaN outputs, the call, a snapshot, decoys in -- all on the current stream."""
        self.load(self.real)
        for o in self.outs:
            o.fill_(NAN)
        res = self.call(self.bufs, self.outs)
        if after_call is not None:
            after_call()
        snap = [r.clone() for r in res]
        self.load(self.decoy)
        return snap

    def matches(self, snap):
        return len(snap) == len(self.base) and all(same(a, b) for a, b in zip(snap, self.base))


def make_jobs(torch, sb, eng):
    from spart_b200 import lut
    lib = eng.lib
    nb = {s: eng.sensor(s)[1].n_bands for s in (L8, S2A, "Sentinel2B-MSI")}
    spec = synthetic_spectra(1, seed=31)[0]
    soils = sb.SoilLibrary(synthetic_spectra(5, seed=32))
    jobs = []

    def pair(n, cfg, seed, **kw):
        return dev_params(torch, n, cfg, seed, **kw), dev_params(torch, n, cfg, seed + 1000, **kw)

    def bands(name, sensor, cfg, seed, l8=0, f32=False, rows_const=(), compact=False, post=None, **kw):
        real, decoy = pair(N, cfg, seed, rows_const=rows_const, f32=f32)
        if post is not None:
            post(real, decoy)
        dt = torch.float32 if f32 else torch.float64
        o = torch.empty((N * nb[sensor] * 2 + N,) if compact else (N, nb[sensor], 3), dtype=dt, device="cuda")

        def call(b, outs):
            r = eng.forward_bands(b[0], sensor, out=outs[0], compact=compact, **kw)
            return [r.buf if compact else r]
        jobs.append(Job(name, [real], [decoy], [o], call, l8))

    bands("fp64_general", L8, 3, 1, l8=1)
    bands("uniform_broadcast_rows", S2A, 2, 2, rows_const=(19, 20, 21), broadcast_rows=[19, 20, 21])
    bands("srf", L8, 3, 3, l8=1, band_mode="srf")
    bands("fp32_double_io", L8, 3, 4, l8=1, precision="fp32")
    bands("fp32_float_io_compact", S2A, 2, 5, f32=True, compact=True, precision="fp32")
    bands("soil_spectrum", S2A, 2, 6, soil_spectrum=spec)

    def lib_index(real, decoy):
        real[9].copy_(torch.arange(N, device="cuda") % 5)
        decoy[9].copy_((torch.arange(N, device="cuda") + 2) % 5)
    bands("soil_library", L8, 3, 7, post=lib_index, soil_library=soils)

    # lidf= as a CUDA tensor: spart_set_lidf and SPART_FLAG_USER_LIDF
    P, Pd = pair(N, 3, 8)
    lidf = [torch.from_numpy(eng.leafangles(so.synthetic_params(N, 3, seed=sd)[:, 16:18])).cuda() for sd in (108, 1108)]
    o = torch.empty((N, nb[L8], 3), dtype=torch.float64, device="cuda")
    jobs.append(Job("user_lidf", [P, lidf[0]], [Pd, lidf[1]], [o],
                    lambda b, outs: [eng.forward_bands(b[0], L8, out=outs[0], lidf=b[1])], 1))

    # one record, two sensors (SPART_FLAG_REUSE_RECORD)
    P, Pd = pair(N, 2, 9)
    outs = [torch.empty((N, nb[s], 3), dtype=torch.float64, device="cuda") for s in (S2A, "Sentinel2B-MSI")]
    jobs.append(Job("multi_sensor", [P], [Pd], outs,
                    lambda b, outs: eng.forward_bands_multi(b[0], [S2A, "Sentinel2B-MSI"], outs=outs)))

    P, Pd = pair(N_SPEC, 3, 10)
    o = torch.empty((N_SPEC, 9, 2162), dtype=torch.float64, device="cuda")
    jobs.append(Job("spectrum", [P], [Pd], [o], lambda b, outs: [eng.forward_spectrum(b[0], out=outs[0])]))

    P, Pd = pair(N, 3, 11)
    o = torch.empty((N, 9, nb[S2A]), dtype=torch.float64, device="cuda")
    jobs.append(Job("smac", [P], [Pd], [o], lambda b, outs: [eng.smac(b[0], S2A, out=outs[0])]))

    g = torch.Generator(device="cuda").manual_seed(12)
    for shared in (True, False):
        shape = (2162,) if shared else (N_SPEC, 2162)
        P, Pd = pair(N_SPEC, 3, 13 + shared)
        spectra = [[0.05 + 0.4 * torch.rand(shape, generator=g, device="cuda", dtype=torch.float64)
                    for _ in range(3)] for _ in range(2)]
        o = torch.empty((N_SPEC, 4, 2162), dtype=torch.float64, device="cuda")
        jobs.append(Job("sailh_shared" if shared else "sailh_per_sample", [P] + spectra[0], [Pd] + spectra[1], [o],
                        lambda b, outs: [eng.sailh(b[0], b[1], b[2], b[3], out=outs[0])]))

    # spart_leafangles through the C ABI on device buffers (Engine.leafangles returns host data)
    P, Pd = pair(N, 3, 15)
    ab = [x[16:18].contiguous() for x in (P, Pd)]
    o = torch.empty((N, 13), dtype=torch.float64, device="cuda")

    def leafangles(b, outs):
        s = torch.cuda.current_stream().cuda_stream
        rc = lib.spart_leafangles(b[0].data_ptr(), N, N, outs[0].data_ptr(), s)
        assert rc == 0, lib.spart_last_error()
        return [outs[0]]
    jobs.append(Job("leafangles_c_abi", [ab[0]], [ab[1]], [o], leafangles))

    tabs = []
    for seed in (16, 17):
        gl = torch.Generator(device="cuda").manual_seed(seed)
        L = torch.rand((4096, 13), generator=gl, device="cuda")
        O = (L[torch.randint(0, 4096, (512,), generator=gl, device="cuda")]
             + 1e-3 * torch.randn((512, 13), generator=gl, device="cuda"))
        tabs.append((L, O))
    for method in ("exact", "tensor"):
        jobs.append(Job(f"lut_nearest_{method}", list(tabs[0]), list(tabs[1]), [],
                        lambda b, outs, m=method: list(lut.nearest(b[0], b[1], method=m))))
    jobs.append(Job("lut_packed_unpack", list(tabs[0]), list(tabs[1]), [],
                    lambda b, outs: (lambda w: [w, *lut.unpack(w)])(lut._search(b[0], b[1], None, 0, packed=True))))

    for j in jobs:                   # serial baselines on the default stream
        j.load(j.real)
        c0 = lib.spart_launch_count()
        res = j.call(j.bufs, j.outs)
        j.launches = lib.spart_launch_count() - c0
        torch.cuda.synchronize()
        j.base = [r.clone() for r in res]
        j.load(j.decoy)
    torch.cuda.synchronize()
    return {j.name: j for j in jobs}, spec, soils


@pytest.fixture(scope="module")
def eng(env):
    torch, sb = env
    e = sb.Engine(0)
    yield e
    torch.cuda.synchronize()
    e.close()


@pytest.fixture(scope="module")
def jobs(env, eng):
    torch, sb = env
    return make_jobs(torch, sb, eng)


DEVICE_JOBS = ["fp64_general", "uniform_broadcast_rows", "srf", "fp32_double_io", "fp32_float_io_compact",
               "soil_spectrum", "soil_library", "user_lidf", "multi_sensor", "spectrum", "smac", "sailh_shared",
               "sailh_per_sample", "leafangles_c_abi", "lut_nearest_exact", "lut_nearest_tensor", "lut_packed_unpack"]


def test_serial_baselines_are_sane(env, eng, jobs):
    """The band baselines against the oracle (1e-9 in FP64, 1e-4 on valid FP32 outputs); the library and LUT
    baselines against their definitions."""
    torch, sb = env
    js, spec, soils = jobs
    for name, sensor, kw in (("fp64_general", L8, {}), ("uniform_broadcast_rows", S2A, {}),
                             ("srf", L8, {"band_mode": "srf"}), ("fp32_double_io", L8, {}),
                             ("fp32_float_io_compact", S2A, {}), ("soil_spectrum", S2A, {"soil": spec}),
                             ("soil_library", L8, {"lib": soils.spectra}), ("user_lidf", L8, {})):
        j = js[name]
        P = j.real[0].double().T.cpu().numpy()
        if name == "user_lidf":
            want = so.spart_bands(P, sensor, lidf=j.real[1].cpu().numpy())
            ok = np.ones(want.shape[:2], bool)
        else:
            want, ok = oracle(P, sensor, **kw)
        got = j.base[0]
        if name == "fp32_float_io_compact":
            nb = want.shape[1]
            got = sb.CompactBands(got, N, nb, eng.sensor(S2A)[1].conv_ea, True).full()
        check_rows(got.double().cpu().numpy(), want, ok, name.startswith("fp32"), name)
    for k, s in enumerate((S2A, "Sentinel2B-MSI")):
        want, ok = oracle(js["multi_sensor"].real[0].T.cpu().numpy(), s)
        check_rows(js["multi_sensor"].base[k].cpu().numpy(), want, ok, False, s)
    ab = js["leafangles_c_abi"].real[0].cpu().numpy()
    assert np.abs(js["leafangles_c_abi"].base[0].cpu().numpy() - so.leafangles(ab[0], ab[1])).max() < 1e-12
    L, O = js["lut_nearest_exact"].real
    idx, cost = js["lut_nearest_exact"].base
    full = ((O[:, None, :] - L[None, :, :]) ** 2).sum(-1)
    assert bool((full.gather(1, idx[:, None])[:, 0] <= full.min(1).values * (1 + 1e-5) + 1e-12).all())
    words, i2, c2 = js["lut_packed_unpack"].base
    assert same(i2, idx) and same(c2, cost)


# -------------------------------------------------------------------------------------------------- A. stream order
def ordered(torch, job, s, cycles, query=False):
    """The A protocol on side stream s.  Returns (snapshot, whether s was still busy when the call returned)."""
    busy = []
    job.load(job.decoy)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(cycles)
        snap = job.enqueue(after_call=lambda: busy.append(not s.query()))
    s.synchronize()
    return snap, busy[0]


def test_default_stream_runs_beside_a_sleeping_side_stream(env, cycles):
    """Canary: torch's side streams are non-blocking here, so work on the legacy default stream is not ordered
    behind them -- which is what lets the A tests see work enqueued on the wrong stream."""
    torch, _ = env
    s = torch.cuda.Stream()
    x = torch.zeros(1, device="cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(cycles)
    x.add_(1)
    torch.cuda.default_stream().synchronize()
    assert not s.query(), "the default stream waited for the side stream"
    s.synchronize()
    assert float(x) == 1.0


def test_call_on_another_stream_is_seen(env, eng, jobs, cycles):
    """Negative control: spart_forward_bands given a different stream's handle than the one the protocol runs on
    reads the decoys (or writes before the NaN fill), so the result differs from the baseline."""
    torch, _ = env
    j = jobs[0]["fp64_general"].fresh()
    other = torch.cuda.Stream()
    handle, st = eng.sensor(L8)
    ws = eng.workspace(N)

    def wrong(b, outs):
        rc = eng.lib.spart_forward_bands(handle, 0, b[0].data_ptr(), N, N, 0, 64, 0, ws.data_ptr(),
                                         outs[0].data_ptr(), other.cuda_stream)
        assert rc == 0
        return [outs[0]]
    j.call = wrong
    snap, _ = ordered(torch, j, torch.cuda.Stream(), cycles)
    torch.cuda.synchronize()
    assert not j.matches(snap)


@pytest.mark.parametrize("name", DEVICE_JOBS)
def test_stream_order(env, jobs, cycles, name):
    """Every device entry point (and mode) reads its inputs and writes its outputs in the order of the caller's
    stream: twice on a fresh side stream, each bit-equal to the serial baseline."""
    torch, _ = env
    j = jobs[0][name].fresh()
    s = torch.cuda.Stream()
    for _ in range(2):
        snap, _ = ordered(torch, j, s, cycles)
        assert j.matches(snap), name


# -------------------------------------------------------------------------------------------------- B. asynchrony
@pytest.mark.parametrize("name", DEVICE_JOBS)
def test_call_returns_before_its_stream_runs(env, jobs, cycles, name):
    """After a warm-up on the same stream, the call returns while its stream is still asleep: no host synchronise
    and no cudaMalloc / cudaFree on the call path."""
    torch, _ = env
    j = jobs[0][name].fresh()
    s = torch.cuda.Stream()
    ordered(torch, j, s, 1000)
    snap, busy = ordered(torch, j, s, cycles)
    assert busy, f"{name} waited for its stream"
    assert j.matches(snap)


# ------------------------------------------------------------------------------------------------------ C. threads
def host_jobs(torch, eng):
    """(name, call, baseline, launches) of host-path calls: pageable and pinned on the Sentinel-2A context, and
    pageable on a second context (TerraAqua-MODIS)."""
    P = np.ascontiguousarray(so.synthetic_params(3000, 2, seed=40).T)
    pinned = torch.from_numpy(P).pin_memory()
    nb = eng.sensor(S2A)[1].n_bands
    specs = [("host_pageable", lambda out=None: eng.forward_bands_host(P, S2A, out=out), (3000, nb, 3)),
             ("host_pinned", lambda out=None: eng.forward_bands_host(pinned, S2A, out=out), None),
             ("host_modis", lambda out=None: eng.forward_bands_host(P, "TerraAqua-MODIS", out=out), None)]
    res = []
    for name, call, _ in specs:
        c0 = eng.lib.spart_launch_count()
        base = call()
        res.append((name, call, base, eng.lib.spart_launch_count() - c0))
    return res


def run_threads(fns):
    errors = []

    def wrap(fn):
        def go():
            try:
                fn()
            except BaseException as e:      # noqa: BLE001 -- reported by the main thread
                errors.append(e)
        return go
    ts = [threading.Thread(target=wrap(f)) for f in fns]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    if errors:
        raise errors[0]


def test_threads_share_one_engine(env, eng, jobs):
    """Seven threads, each with its own stream and buffers, run shuffled rounds of every device and host job on
    one Engine; one of them also makes argument errors.  Every result equals its baseline, each thread's launch
    count grows by the sum of its jobs' serial counts, each error text names its own call, and the profiled
    context counts exactly the forward_bands calls all threads made on it."""
    torch, sb = env
    js = jobs[0]
    hjobs = host_jobs(torch, eng)
    lib = eng.lib
    eng.profile_enable(L8)
    l8_calls = [0] * 7
    failures = []
    rounds = 3

    def worker(t):
        rng = random.Random(t)
        mine = [js[n].fresh() for n in DEVICE_JOBS]
        s = torch.cuda.Stream()
        pinned_out = torch.empty(hjobs[1][2].shape, dtype=torch.float64).pin_memory()
        # valid buffers for the invalid calls: they are refused before anything is read
        e_par = torch.zeros((27, 1), dtype=torch.float64, device="cuda")
        e_ws, e_out = eng.workspace(1), torch.empty(64, dtype=torch.float64, device="cuda")
        c0 = lib.spart_launch_count()
        want = 0
        errs = 0
        for _ in range(rounds):
            order = list(range(len(mine))) + [-1 - k for k in range(len(hjobs))] + ([None] * 4 if t == 0 else [])
            rng.shuffle(order)
            for k in order:
                if k is None:                             # argument errors on this thread only
                    errs += 1
                    handle, _ = eng.sensor(S2A)
                    flag_err = errs % 2 == 0
                    rc = lib.spart_forward_bands(handle, 0, e_par.data_ptr(), 1, 1, 0, 64 if flag_err else 7,
                                                 (1 << 20) if flag_err else 0, e_ws.data_ptr(), e_out.data_ptr(),
                                                 s.cuda_stream)
                    try:
                        sb._lib.check(rc, f"error call {errs}")
                        failures.append("an invalid call succeeded")
                    except sb.SpartError as e:
                        text = str(e)
                        expect = "unknown flag bit" if flag_err else "precision must be"
                        if not (text.startswith(f"error call {errs}:") and expect in text):
                            failures.append(f"error text of call {errs}: {text}")
                elif k < 0:
                    name, call, base, launches = hjobs[-1 - k]
                    got = call(pinned_out).numpy() if name == "host_pinned" else call()
                    want += launches
                    if not np.array_equal(got.view(np.int64), base.view(np.int64)):
                        failures.append(f"thread {t}: {name}")
                else:
                    j = mine[k]
                    with torch.cuda.stream(s):
                        snap = j.enqueue()
                    s.synchronize()
                    want += j.launches
                    l8_calls[t] += j.l8_calls
                    if not j.matches(snap):
                        failures.append(f"thread {t}: {j.name}")
        got = lib.spart_launch_count() - c0
        if got != want:
            failures.append(f"thread {t}: {got} launches counted, {want} made")

    try:
        run_threads([lambda t=t: worker(t) for t in range(7)])
        prof = eng.profile_read(L8)
    finally:
        eng.profile_enable(L8, on=False)
    assert not failures, failures[:10]
    assert prof["calls"] == sum(l8_calls) == 7 * rounds * 4


SRF_SENSORS = ["TerraAqua-MODIS", "Sentinel2B-MSI", "Sentinel2A-MSI", "Sentinel3A-OLCI"]


def test_srf_calls_of_different_sensors_from_four_threads(env, eng):
    """band_kernel_srf's dynamic shared memory differs per sensor (4 KB per accumulator slot); its cap belongs to
    the kernel and device, so one thread's smaller plan must not lower it under another thread's launch.  Four
    threads, one sensor each (the MODIS thread also runs the soil-library twin, soillib_srf), n = 128 so that host
    time dominates, 300 calls each: no error and every result bit-equal to its baseline."""
    torch, sb = env
    soils = sb.SoilLibrary(synthetic_spectra(3, seed=50))
    P = dev_params(torch, 128, 3, 51)
    Plib = P.clone()
    Plib[9].copy_(torch.arange(128, device="cuda") % 3)
    base = {s: eng.forward_bands(P, s, band_mode="srf") for s in SRF_SENSORS}
    base["lib"] = eng.forward_bands(Plib, SRF_SENSORS[0], band_mode="srf", soil_library=soils)
    torch.cuda.synchronize()
    results = {}

    def worker(t):
        s = torch.cuda.Stream()
        sensor = SRF_SENSORS[t]
        outs = []
        with torch.cuda.stream(s):
            for i in range(300):
                if t == 0 and i % 2:
                    outs.append(("lib", eng.forward_bands(Plib, sensor, band_mode="srf", soil_library=soils)))
                else:
                    outs.append((sensor, eng.forward_bands(P, sensor, band_mode="srf")))
        s.synchronize()
        results[t] = outs

    run_threads([lambda t=t: worker(t) for t in range(4)])
    for t, outs in results.items():
        assert len(outs) == 300
        bad = [k for k, o in outs if not same(o, base[k])]
        assert not bad, f"thread {t}: {len(bad)} results differ"


# ----------------------------------------------------------------------------------------------- D. context lifetime
CTX_CALLS = ("spart_forward_bands", "spart_forward_bands_bc", "spart_forward_bands_host", "spart_forward_spectrum",
             "spart_smac", "spart_sailh", "spart_profile_enable", "spart_profile_read", "spart_destroy")


class DeadHandleProxy:
    """Stands in for the ctypes library of an Engine: records the handles passed to spart_destroy and refuses,
    without calling into C, any call that passes a destroyed handle (counted in `dead_calls`).  A handle value
    that spart_create returns again is live again."""

    def __init__(self, lib):
        self._lib, self._mu = lib, threading.Lock()
        self.dead, self.destroyed, self.dead_calls = set(), {}, []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if name in ("spart_create", "spart_create_with_soils"):
            def create(*a):
                rc = fn(*a)
                with self._mu:
                    self.dead.discard(a[-1]._obj.value)
                return rc
            return create
        if name not in CTX_CALLS:
            return fn

        def guarded(h, *a):
            v = h.value if isinstance(h, ctypes.c_void_p) else h
            with self._mu:
                if v in self.dead:
                    self.dead_calls.append(name)
                    raise RuntimeError(f"{name} called with destroyed context {v:#x}")
                if name == "spart_destroy":
                    self.dead.add(v)
                    self.destroyed[v] = self.destroyed.get(v, 0) + 1
            return fn(h, *a)
        return guarded


def test_eviction_while_a_call_uses_the_context(env, monkeypatch):
    """forward_bands obtains its context, then (inside the call) MAX_CONTEXTS other soil-spectrum contexts are
    created, which evicts it.  The call must still run on a live context and give the baseline's bits; the evicted
    context is destroyed once, when the call ends, and the cache stays bounded."""
    torch, sb = env
    from spart_b200.engine import MAX_CONTEXTS
    eng = sb.Engine(0)
    try:
        P = dev_params(torch, N, 3, 60)
        base = eng.forward_bands(P, L8)
        torch.cuda.synchronize()
        eng.lib = proxy = DeadHandleProxy(eng.lib)
        handle = eng.sensor(L8)[0].value
        spectra = synthetic_spectra(MAX_CONTEXTS, seed=61)
        prep, first = eng._prep, [True]

        def prep_and_evict(*a, **k):
            if first.pop() if first else False:
                for sp in spectra:
                    eng.sensor(S2A, soil_spectrum=sp)
            return prep(*a, **k)
        monkeypatch.setattr(eng, "_prep", prep_and_evict)
        got = eng.forward_bands(P, L8)
        torch.cuda.synchronize()
        assert proxy.dead_calls == []
        assert same(got, base)
        assert proxy.destroyed.get(handle) == 1, "the evicted context was not destroyed after the call"
        assert len(eng._ctx) <= MAX_CONTEXTS
    finally:
        eng.close()


def test_eviction_from_other_threads(env):
    """Two threads create 40 distinct soil-spectrum contexts between them (the cache holds 32) while four others
    run band, spectrum and host-path jobs whose contexts are evicted and re-created under them: no call ever
    reaches the library with a destroyed context, and every result equals its baseline."""
    torch, sb = env
    eng = sb.Engine(0)
    try:
        P = dev_params(torch, N, 3, 70)
        Ps = dev_params(torch, N_SPEC, 3, 71)
        Ph = np.ascontiguousarray(so.synthetic_params(2000, 2, seed=72).T)
        spectra = synthetic_spectra(40, seed=73)
        base_b = eng.forward_bands(P, L8)
        base_s = eng.forward_spectrum(Ps)
        base_h = eng.forward_bands_host(Ph, S2A)
        base_x = eng.forward_bands(P, S2A, soil_spectrum=spectra[0])
        torch.cuda.synchronize()
        eng.lib = proxy = DeadHandleProxy(eng.lib)
        failures = []

        def creator(t):
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                for i in range(t, 40, 2):
                    got = eng.forward_bands(P, S2A, soil_spectrum=spectra[i])
                    if i == 0:
                        s.synchronize()
                        if not same(got, base_x):
                            failures.append("soil spectrum")
            s.synchronize()

        def user(kind):
            s = torch.cuda.Stream()
            for _ in range(30):
                if kind == "host":
                    if not np.array_equal(eng.forward_bands_host(Ph, S2A).view(np.int64), base_h.view(np.int64)):
                        failures.append(kind)
                    continue
                with torch.cuda.stream(s):
                    got = eng.forward_bands(P, L8) if kind == "bands" else eng.forward_spectrum(Ps)
                s.synchronize()
                if not same(got, base_b if kind == "bands" else base_s):
                    failures.append(kind)

        run_threads([lambda: creator(0), lambda: creator(1), lambda: user("bands"), lambda: user("bands"),
                     lambda: user("spectrum"), lambda: user("host")])
        assert proxy.dead_calls == []
        assert not failures, failures[:10]
        assert len(proxy.destroyed) >= 8, "the cache evicted less than the test meant it to"
    finally:
        eng.close()


@pytest.mark.parametrize("how", ["evict", "close"])
def test_destroy_with_work_still_queued(env, cycles, how):
    """forward_bands enqueued behind a delay on a side stream, then its context evicted (or the Engine closed) at
    once: spart_destroy waits for the device before freeing the tables, so the result is still correct."""
    torch, sb = env
    from spart_b200.engine import MAX_CONTEXTS
    eng = sb.Engine(0)
    try:
        P = dev_params(torch, N, 3, 80)
        spec = synthetic_spectra(1, seed=81)[0]
        base = eng.forward_bands(P, L8, soil_spectrum=spec)
        torch.cuda.synchronize()
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            torch.cuda._sleep(cycles)
            got = eng.forward_bands(P, L8, soil_spectrum=spec)
        if how == "evict":
            for sp in synthetic_spectra(MAX_CONTEXTS, seed=82):
                eng.sensor(S2A, soil_spectrum=sp)
        else:
            eng.close()
        s.synchronize()
        assert same(got, base)
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------- E. pipelined gather
@pytest.fixture(scope="module")
def nccl_world1(env, tmp_path_factory):
    torch, _ = env
    import torch.distributed as dist
    dist.init_process_group("nccl", store=dist.FileStore(str(tmp_path_factory.mktemp("nccl") / "store"), 1),
                            rank=0, world_size=1, device_id=torch.device("cuda", 0))
    yield dist
    dist.destroy_process_group()


def test_pipelined_gather_waits_for_each_chunk(env, nccl_world1, cycles):
    """gather_pipelined on a side stream, each chunk written only after a delay: the gather of chunk c (on its
    own stream) must wait for chunk c, so recv equals the chunks."""
    torch, _ = env
    from spart_b200.distributed import gather_pipelined
    g = torch.Generator(device="cuda").manual_seed(90)
    chunks = [torch.randn(e, generator=g, device="cuda", dtype=torch.float64) for e in (5000, 5000, 5000, 17)]
    s = torch.cuda.Stream()

    def compute_chunk(c, view):
        torch.cuda._sleep(cycles // 4)
        view.copy_(chunks[c])
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        local, recv = gather_pipelined(compute_chunk, [c.numel() for c in chunks], torch.float64, "cuda:0", dst=0)
        snap = recv.clone()
    s.synchronize()
    assert same(snap[0], torch.cat(chunks)) and same(local, torch.cat(chunks))


def test_sharded_search_on_a_side_stream(env, nccl_world1, jobs, cycles):
    """nearest_sharded (search, NCCL min-reduction, unpack) enqueued behind a delay on a side stream equals the
    single-GPU search."""
    torch, _ = env
    from spart_b200 import lut
    j = jobs[0]["lut_nearest_exact"]
    L, O = j.real
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(cycles)
        idx, cost = lut.nearest_sharded(L, O)
        snap = [idx.clone(), cost.clone()]
    s.synchronize()
    assert j.matches(snap)


# ---------------------------------------------------------------------------------------------------- F. two GPUs
def test_threads_on_two_gpus(env):
    """A thread per device (two per device) runs band calls on its own device's Engine: results equal the
    device's serial baseline and each thread's current device never changes."""
    torch, sb = env
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    base, params, engines = {}, {}, {}
    for d in (0, 1):
        with torch.cuda.device(d):
            engines[d] = sb.default_engine(d)
            params[d] = torch.from_numpy(np.ascontiguousarray(so.synthetic_params(N, 3, seed=95).T)).cuda(d)
            base[d] = engines[d].forward_bands(params[d], L8)
            torch.cuda.synchronize(d)
    failures = []

    def worker(d):
        torch.cuda.set_device(d)
        s = torch.cuda.Stream(d)
        for _ in range(50):
            with torch.cuda.stream(s):
                got = engines[d].forward_bands(params[d], L8)
            if torch.cuda.current_device() != d:
                failures.append(f"device changed to {torch.cuda.current_device()} on a device-{d} thread")
            s.synchronize()
            if not same(got, base[d]):
                failures.append(f"device {d}")

    run_threads([lambda d=d: worker(d) for d in (0, 1, 0, 1)])
    assert not failures, failures[:10]
    assert same(base[0].cpu(), base[1].cpu())
