"""Host-side driver of the CUDA path: one `Engine` per GPU.

PyTorch is used for device memory, streams and (in distributed.py) NCCL only; all
arithmetic happens in libspart_b200.so.  A context (immutable device tables) is created
lazily per sensor and cached (bounded, least recently used first out).
"""
import hashlib
import threading
from collections import OrderedDict
from contextlib import contextmanager

import numpy as np
import torch

from . import _lib
from . import tables as T
from .params import SoilLibrary

NPAR = 27
NOUT = 3
NSPEC = 9
NWL_S = 2162
MAX_SAMPLES_PER_CALL = 65535 * 128    # grid.y limit of band_kernel, see spart_forward_bands
MAX_CONTEXTS = 32                     # cached (sensor, soil spectrum or library) contexts per engine

_PRECISION = {"fp64": _lib.FP64, 64: _lib.FP64, "fp32": _lib.FP32, 32: _lib.FP32}


def _require_cuda():
    if not torch.cuda.is_available():
        raise _lib.SpartError("spart_b200 needs a CUDA device (B200); there is no CPU fallback")


def out_elems(n, nb, compact):
    """Elements of a result buffer (SPART_OUT_ELEMS of include/spart_b200.h)."""
    return n * nb * 2 + n if compact else n * nb * NOUT


class CompactBands:
    """Result of a `compact=True` run: `R` [n, nb, 2] = (R_TOC, R_TOA) and `etscale` [n], both views of
    one flat buffer (SPART_FLAG_COMPACT_OUT), plus the sensor's SRF-convolved extraterrestrial
    irradiance `conv_ea` [nb].  `L_TOA` is rebuilt bit for bit as the kernels form it:
    (conv_ea[b] * etscale[s]) * R_TOA[s, b] (SPART.py:252) in the buffer's dtype."""

    def __init__(self, buf, n, nb, conv_ea, fp32=False):
        self.buf, self.n, self.nb = buf, n, nb
        self.R = buf[:n * nb * 2].reshape(n, nb, 2)
        self.etscale = buf[n * nb * 2:n * nb * 2 + n]
        # the arithmetic type the kernels formed L_TOA in: float in FP32 mode, whatever the storage type
        self.fp32 = bool(fp32) or (buf.dtype in (torch.float32, np.float32))
        self.conv_ea_f64 = np.asarray(conv_ea, dtype=np.float64)
        self._conv_ea = None

    @property
    def conv_ea(self):
        """conv_ea in the arithmetic type of the run, on the buffer's device (built on first use: creating a
        CompactBands must not touch the GPU, the gather pipeline creates one per chunk)."""
        if self._conv_ea is None:
            if isinstance(self.buf, torch.Tensor):
                self._conv_ea = torch.as_tensor(self.conv_ea_f64).to(torch.float32 if self.fp32 else self.buf.dtype).to(
                    self.buf.device)
            else:
                self._conv_ea = self.conv_ea_f64.astype(np.float32 if self.fp32 else self.buf.dtype)
        return self._conv_ea

    @property
    def R_TOC(self):
        return self.R[..., 0]

    @property
    def R_TOA(self):
        return self.R[..., 1]

    @property
    def L_TOA(self):
        if self.fp32 and self.buf.dtype not in (torch.float32, np.float32):      # FP32 mode with double I/O
            f = (lambda x: x.float()) if isinstance(self.buf, torch.Tensor) else (lambda x: x.astype(np.float32))
            lt = (self.conv_ea[None, :] * f(self.etscale)[:, None]) * f(self.R[..., 1])
            return lt.double() if isinstance(self.buf, torch.Tensor) else lt.astype(np.float64)
        return (self.conv_ea[None, :] * self.etscale[:, None]) * self.R[..., 1]

    def full(self):
        """[n, nb, 3] = (R_TOC, R_TOA, L_TOA), identical to a non-compact run."""
        if isinstance(self.buf, torch.Tensor):
            return torch.cat([self.R, self.L_TOA[..., None]], dim=2)
        return np.concatenate([self.R, self.L_TOA[..., None]], axis=2)


class _Context:
    """A cached C context: its handle and tables, the host arrays it was built from, the number of calls
    using it (`Engine._use`) and whether it has left the cache (then the last user destroys it)."""
    __slots__ = ("handle", "st", "keep", "uses", "retired")

    def __init__(self, handle, st, keep):
        self.handle, self.st, self.keep, self.uses, self.retired = handle, st, keep, 0, False


def _sensor_digest(info):
    """Content hash of everything the hot path uses of a sensorinfo dict."""
    h = hashlib.sha1()
    for k in ("wl_smac", "wl_srf_smac", "p_srf_smac"):
        a = np.ascontiguousarray(np.asarray(info[k]))
        h.update(k.encode() + str(a.dtype).encode() + str(a.shape).encode() + a.tobytes())
    for k in sorted(info["SMAC_coef"]):
        a = np.ascontiguousarray(np.asarray(info["SMAC_coef"][k]))
        h.update(k.encode() + str(a.dtype).encode() + a.tobytes())
    h.update("\x1f".join(str(b) for b in info["band_id_smac"]).encode())
    return h.hexdigest()


class Engine:
    """Owns the C contexts of one GPU."""

    def __init__(self, device=None):
        _require_cuda()
        self.lib = _lib.load()
        if self.lib.spart_device_count() <= 0:
            raise _lib.SpartError("libspart_b200: no CUDA device visible")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else
                                   (device.index if isinstance(device, torch.device) else int(device)))
        self._opt = T.load_optical()
        self._lc = T.leaf_soil_constants(self._opt)
        self._ctx = OrderedDict()   # key -> (ctx handle, SensorTables, keep-alive arrays); LRU order
        self._lock = threading.Lock()

    # ---- contexts ------------------------------------------------------------------
    def sensor(self, sensor, soil_spectrum=None, soil_library=None):
        """(ctx, SensorTables) for a shipped sensor name or a reference-style sensorinfo dict.
        Custom dicts are keyed by the content of every array the hot path uses (so an edited dict
        is a new sensor).  soil_spectrum: optional user dry-soil reflectance [2001]
        (SoilParametersFromFile); such a context carries the spectrum as its first soil vector and
        must be run with SPART_FLAG_SOIL_SPECTRUM.  soil_library: optional SoilLibrary, uploaded once
        into the context (spart_create_with_soils) for runs with SPART_FLAG_SOIL_LIBRARY; keyed by its
        content digest.  At most MAX_CONTEXTS contexts are kept; the least recently used one is
        destroyed (its device tables are freed) when a new one is needed.  The returned handle is
        therefore valid only until the cache evicts it: any later `sensor()` call that creates a context,
        from this thread or another one, may destroy it.  The Engine's own methods hold their context
        for the whole call (see `_use`)."""
        e = self._entry(sensor, soil_spectrum, soil_library, pin=False)
        return e.handle, e.st

    @contextmanager
    def _use(self, sensor, soil_spectrum=None, soil_library=None):
        """(ctx, SensorTables) pinned for the duration of the `with` block: eviction (by any thread)
        retires a pinned context instead of destroying it, and the last user's exit destroys it."""
        e = self._entry(sensor, soil_spectrum, soil_library, pin=True)
        try:
            yield e.handle, e.st
        finally:
            with self._lock:
                e.uses -= 1
                if e.retired and e.uses == 0:
                    self.lib.spart_destroy(e.handle)

    def _retire(self, e):
        """Called under _lock for an entry leaving the cache: destroy it now unless a call is using it."""
        e.retired = True
        if e.uses == 0:
            self.lib.spart_destroy(e.handle)

    def _entry(self, sensor, soil_spectrum, soil_library, pin):
        skey = sensor if isinstance(sensor, str) else ("custom", _sensor_digest(sensor))
        soil = None
        if soil_spectrum is not None and soil_library is not None:
            raise ValueError("soil_spectrum and soil_library exclude each other")
        if soil_library is not None and not isinstance(soil_library, SoilLibrary):
            raise TypeError("soil_library must be a SoilLibrary")
        if soil_spectrum is not None:
            soil = np.ascontiguousarray(np.asarray(soil_spectrum, dtype=np.float64).reshape(-1))
            if soil.shape[0] != T.NWL:
                raise ValueError("soil_spectrum must have 2001 values (400..2400 nm)")
        if soil_library is not None:
            key = (skey, ("lib", soil_library.digest))
        else:
            key = (skey, None if soil is None else hashlib.sha1(soil.tobytes()).hexdigest())
        with self._lock:
            e = self._ctx.get(key)
            if e is not None:
                self._ctx.move_to_end(key)
                e.uses += pin
                return e
            info = T.load_sensor_info(sensor) if isinstance(sensor, str) else sensor
            st = T.build_sensor(sensor if isinstance(sensor, str) else "custom", info, self._opt)
            lc = self._lc
            if soil is not None:
                lc = self._lc.copy()
                lc[11], lc[12], lc[13] = soil, 0.0, 0.0
            tabs = _lib.SpartTables(n_wl=T.NWL, lc=_lib.as_double_ptr(lc))
            smac = np.ascontiguousarray(st.smac)
            cs = _lib.SpartSensor(n_bands=st.n_bands, wl_lo=_lib.as_int32_ptr(st.wl_lo),
                                  wl_hi=_lib.as_int32_ptr(st.wl_hi), wl_frac=_lib.as_double_ptr(st.wl_frac),
                                  smac=_lib.as_double_ptr(smac), conv_ea=_lib.as_double_ptr(st.conv_ea),
                                  srf_len=_lib.as_int32_ptr(st.srf_len), srf_idx=_lib.as_int32_ptr(st.srf_idx),
                                  srf_w=_lib.as_double_ptr(st.srf_w))
            handle = _lib.c_void_p()
            if soil_library is None:
                _lib.check(self.lib.spart_create(_lib.byref(tabs), _lib.byref(cs), 1, self.device.index,
                                                 _lib.byref(handle)), "spart_create")
            else:
                lib_rows = soil_library.spectra
                _lib.check(self.lib.spart_create_with_soils(_lib.byref(tabs), _lib.byref(cs), 1,
                                                            _lib.as_double_ptr(lib_rows), lib_rows.shape[0],
                                                            self.device.index, _lib.byref(handle)),
                           "spart_create_with_soils")
            while len(self._ctx) >= MAX_CONTEXTS:
                self._retire(self._ctx.popitem(last=False)[1])
            e = self._ctx[key] = _Context(handle, st, (smac, lc))
            e.uses += pin
            return e

    def close(self):
        """Destroy every cached context; one that a call is using is destroyed when that call ends."""
        with self._lock:
            for e in self._ctx.values():
                self._retire(e)
            self._ctx.clear()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- device path ---------------------------------------------------------------
    def _prep(self, params, allow_f32=False):
        ok = (isinstance(params, torch.Tensor) and params.is_cuda and params.dim() == 2 and params.shape[0] == NPAR
              and (params.shape[1] <= 1 or params.stride(1) == 1)
              and (params.dtype == torch.float64 or (allow_f32 and params.dtype == torch.float32)))
        if not ok:
            raise ValueError("params must be a CUDA float64 tensor [27, n] with contiguous rows"
                             " (float32 is accepted with precision='fp32')")
        if params.device != self.device:
            raise ValueError(f"params on {params.device}, engine on {self.device}")
        # a [27, 1] view of a wider batch keeps that batch's row stride, which is its ld
        return params, params.shape[1], (params.stride(0) if params.shape[1] >= 1 else 1)

    def _geometry_mask(self, params, n, mask, uniform_geometry):
        """uniform_geometry=True is checked, not trusted: unless the three angle rows already are
        broadcast rows they must be constant over the batch (one small reduction and a
        synchronisation); they are then passed as broadcast rows, which is what selects the
        folded-geometry kernels."""
        if not uniform_geometry or (mask & _lib.GEOMETRY_ROWS) == _lib.GEOMETRY_ROWS or n == 0:
            return mask
        ang = params[19:22, :n]
        same = bool((ang == ang[:, :1]).all().item()) if isinstance(params, torch.Tensor) else bool(
            (ang == ang[:, :1]).all())
        if not same:
            raise _lib.SpartError("uniform_geometry=True, but the sun / observer angle rows 19..21 vary over the batch")
        return mask | _lib.GEOMETRY_ROWS

    @staticmethod
    def _flags(soil_spectrum, band_mode, f32_io=False, compact=False, reuse=False, soil_library=None):
        if band_mode not in ("interp", "srf"):
            raise ValueError("band_mode must be 'interp' or 'srf'")
        return ((_lib.FLAG_SOIL_SPECTRUM if soil_spectrum is not None else 0)
                | (_lib.FLAG_SOIL_LIBRARY if soil_library is not None else 0)
                | (_lib.FLAG_SRF_BANDS if band_mode == "srf" else 0)
                | (_lib.FLAG_F32_IO if f32_io else 0) | (_lib.FLAG_COMPACT_OUT if compact else 0)
                | (_lib.FLAG_REUSE_RECORD if reuse else 0))

    def workspace(self, n):
        """Device scratch for a batch of n samples (spart_workspace_bytes)."""
        return torch.empty(max(self.lib.spart_workspace_bytes(None, n) // 8, 1), dtype=torch.float64, device=self.device)

    def _set_lidf(self, lidf, n, ws, stream):
        """Store a caller-supplied leaf inclination distribution [n, 13] in the workspace (spart_set_lidf)."""
        lidf = torch.as_tensor(lidf, dtype=torch.float64).to(self.device).reshape(-1, 13)
        if lidf.shape[0] == 1 and n > 1:
            lidf = lidf.expand(n, 13)
        if lidf.shape[0] != n:
            raise ValueError("lidf must have one row of 13 values per sample (or a single row for the whole batch)")
        lidf = lidf.contiguous()
        _lib.check(self.lib.spart_set_lidf(lidf.data_ptr(), n, ws.data_ptr(), stream), "spart_set_lidf")
        return lidf                       # keep alive until the stream has consumed it

    def forward_bands(self, params, sensor, out=None, precision="fp64", uniform_geometry=False,
                      soil_spectrum=None, band_mode="interp", broadcast_rows=0, compact=False,
                      reuse_record=False, workspace=None, lidf=None, soil_library=None, broadcast_base=None):
        """params: CUDA float64 [27, n] -> CUDA float64 [n, nb, 3] = (R_TOC, R_TOA, L_TOA).
        Asynchronous on the current torch stream.

        broadcast_rows: bit mask / iterable of rows that are constant over the batch (only their
        element 0 is read).  uniform_geometry=True: the three angle rows are verified to be constant
        and passed as broadcast rows (raises SpartError otherwise).  soil_spectrum: dry soil
        reflectance [2001] used instead of the B/lat/lon soil vectors.  soil_library: a SoilLibrary;
        row 9 (B) then holds each sample's index into it (a broadcast row 9 gives the whole batch one
        spectrum) and rows 10, 11 are ignored; an index that is not a whole number in [0, k) gives NaN
        soil-dependent outputs.  Excludes soil_spectrum.  band_mode: "interp" (the
        reference: np.interp at the band centre) or "srf" (SRF-weighted band means).
        precision="fp32" with float32 params: float32 in, float32 out (SPART_FLAG_F32_IO).
        compact=True: returns a CompactBands (R_TOC, R_TOA + etscale; two thirds of the bytes).
        `out`: result buffer to fill ([n, nb, 3], or flat with out_elems(n, nb, True) elements when
        compact).
        lidf: a leaf inclination distribution [n, 13] (or one row for the whole batch) used instead of the one
        derived from LIDFa / LIDFb -- the reference's assigned `CanopyStructure.lidf`; FP64 only.
        broadcast_base: the tensor whose column 0 holds the broadcast rows' values (default `params`): a
        CUDA tensor [27, >= 1] of the params' dtype and row stride, typically the batch that `params` is a
        column slice of.  A batch of more than MAX_SAMPLES_PER_CALL samples is split into calls, and every
        call reads the broadcast rows from this column 0, never from its own first column."""
        prec = _PRECISION[precision]
        with self._use(sensor, soil_spectrum, soil_library) as (handle, st):
            params, n, ld = self._prep(params, allow_f32=(prec == _lib.FP32))
            f32_io = params.dtype == torch.float32
            mask = self._geometry_mask(params, n, _lib.row_mask(broadcast_rows), uniform_geometry)
            flags = self._flags(soil_spectrum, band_mode, f32_io, compact, reuse_record, soil_library)
            if lidf is not None:
                if prec != _lib.FP64 or reuse_record or n > MAX_SAMPLES_PER_CALL:
                    raise ValueError("lidf= needs precision='fp64', no reuse_record and at most "
                                     f"{MAX_SAMPLES_PER_CALL} samples per call")
                flags |= _lib.FLAG_USER_LIDF
            nb = st.n_bands
            elems = out_elems(n, nb, compact)
            if out is None:
                out = torch.empty(elems if compact else (n, nb, NOUT), dtype=params.dtype, device=self.device)
            elif not (out.is_cuda and out.dtype == params.dtype and out.is_contiguous() and out.numel() == elems
                      and (compact or tuple(out.shape) == (n, nb, NOUT))):
                raise ValueError("out must be a contiguous CUDA tensor of the params' dtype: [n, nb, 3], or flat with"
                                 " n*nb*2 + n elements when compact")
            if n > MAX_SAMPLES_PER_CALL and (compact or reuse_record):
                raise ValueError(f"compact / reuse_record runs handle at most {MAX_SAMPLES_PER_CALL} samples per"
                                 " call")
            bc = params if broadcast_base is None else broadcast_base
            if broadcast_base is not None and not (
                    isinstance(bc, torch.Tensor) and bc.device == params.device and bc.dtype == params.dtype
                    and bc.dim() == 2 and bc.shape[0] == NPAR and bc.shape[1] >= 1 and bc.stride(0) == ld):
                raise ValueError("broadcast_base must be a tensor [27, >= 1] on the params' device with their dtype and"
                                 " row stride")
            esz = params.element_size()
            with torch.cuda.device(self.device):
                stream = torch.cuda.current_stream(self.device).cuda_stream
                for s0 in range(0, n, MAX_SAMPLES_PER_CALL):
                    m = min(MAX_SAMPLES_PER_CALL, n - s0)
                    ws = workspace if (workspace is not None and s0 == 0 and m == n) else self.workspace(m)
                    keep = self._set_lidf(lidf, n, ws, stream) if lidf is not None else None      # noqa: F841
                    # every call reads the broadcast rows from column 0 of the batch, not from its own first column
                    _lib.check(self.lib.spart_forward_bands_bc(handle, 0, params.data_ptr() + esz * s0, bc.data_ptr(),
                                                               m, ld, mask, prec, flags, ws.data_ptr(),
                                                               out.data_ptr() + esz * s0 * nb * NOUT, stream),
                               "spart_forward_bands")
            return CompactBands(out, n, nb, st.conv_ea, prec == _lib.FP32) if compact else out

    def forward_bands_multi(self, params, sensors, outs=None, precision="fp64", uniform_geometry=False,
                            soil_spectrum=None, band_mode="interp", broadcast_rows=0, compact=False,
                            soil_library=None):
        """One batch evaluated for several sensors: the sensor-independent per-sample kernels run
        once and every further sensor only runs the band kernel (SPART_FLAG_REUSE_RECORD).
        Returns a list of results as forward_bands would."""
        n = params.shape[1]
        if n > MAX_SAMPLES_PER_CALL:
            raise ValueError(f"forward_bands_multi handles at most {MAX_SAMPLES_PER_CALL} samples per call")
        mask = self._geometry_mask(params, n, _lib.row_mask(broadcast_rows), uniform_geometry)
        ws = self.workspace(n)
        res = []
        for i, s in enumerate(sensors):
            res.append(self.forward_bands(params, s, out=None if outs is None else outs[i], precision=precision,
                                          soil_spectrum=soil_spectrum, soil_library=soil_library,
                                          band_mode=band_mode, broadcast_rows=mask,
                                          compact=compact, reuse_record=i > 0, workspace=ws))
        return res

    def forward_spectrum(self, params, out=None, soil_spectrum=None, rho_thermal=0.01, tau_thermal=0.01, lidf=None,
                         soil_library=None):
        """params: CUDA float64 [27, n] -> CUDA float64 [n, 9, 2162]: leaf refl, leaf tran,
        kChlrel, soil refl, soil refl dry, rso, rdo, rsd, rdd.  rho_thermal / tau_thermal: leaf
        reflectance / transmittance beyond 2400 nm (LeafBiology.rho_thermal / tau_thermal).
        soil_spectrum / soil_library as in forward_bands."""
        # any context carries the wavelength tables
        with self._use("Sentinel2A-MSI", soil_spectrum, soil_library) as (handle, _):
            params, n, ld = self._prep(params)
            if out is None:
                out = torch.empty((n, NSPEC, NWL_S), dtype=torch.float64, device=self.device)
            ws = self.workspace(n)
            flags = self._flags(soil_spectrum, "interp", soil_library=soil_library)
            with torch.cuda.device(self.device):
                stream = torch.cuda.current_stream(self.device).cuda_stream
                if lidf is not None:
                    keep = self._set_lidf(lidf, n, ws, stream)      # noqa: F841
                    flags |= _lib.FLAG_USER_LIDF
                _lib.check(self.lib.spart_forward_spectrum(handle, params.data_ptr(), n, ld, flags,
                                                           float(rho_thermal), float(tau_thermal), ws.data_ptr(),
                                                           out.data_ptr(), stream), "spart_forward_spectrum")
            return out

    def smac(self, params, sensor, out=None):
        """SMAC alone.  params: CUDA float64 [27, n] (angle and atmosphere rows used)
        -> CUDA float64 [n, 9, nb]: Ta_s, Ta_o, Tg, Ra_dd, Ra_so, Ta_ss, Ta_sd, Ta_oo, Ta_do."""
        with self._use(sensor) as (handle, st):
            params, n, ld = self._prep(params)
            if out is None:
                out = torch.empty((n, 9, st.n_bands), dtype=torch.float64, device=self.device)
            ws = self.workspace(n)
            with torch.cuda.device(self.device):
                stream = torch.cuda.current_stream(self.device).cuda_stream
                _lib.check(self.lib.spart_smac(handle, 0, params.data_ptr(), n, ld, ws.data_ptr(), out.data_ptr(),
                                               stream), "spart_smac")
            return out

    def sailh(self, params, soil_refl, leaf_refl, leaf_tran, out=None):
        """SAILH on caller-supplied spectra.  params: CUDA float64 [27, n] (canopy and angle rows
        used); spectra: CUDA float64 [2162] (shared by all samples) or [n, 2162].
        -> CUDA float64 [n, 4, 2162] = rso, rdo, rsd, rdd."""
        with self._use("Sentinel2A-MSI") as (handle, _):
            params, n, ld = self._prep(params)
            specs = [soil_refl, leaf_refl, leaf_tran]
            shared = all(x.dim() == 1 for x in specs)
            for x in specs:
                ok = x.is_cuda and x.dtype == torch.float64 and x.is_contiguous() and (
                    tuple(x.shape) == (NWL_S,) if shared else tuple(x.shape) == (n, NWL_S))
                if not ok:
                    raise RuntimeError("Parameter leafopt.refl must be of len 2162 i.e. include thermal specturm "
                                       "(CUDA float64, all three spectra [2162] or all [n, 2162])")
            if out is None:
                out = torch.empty((n, 4, NWL_S), dtype=torch.float64, device=self.device)
            ws = self.workspace(n)
            with torch.cuda.device(self.device):
                stream = torch.cuda.current_stream(self.device).cuda_stream
                _lib.check(self.lib.spart_sailh(handle, params.data_ptr(), n, ld, soil_refl.data_ptr(),
                                                leaf_refl.data_ptr(), leaf_tran.data_ptr(), 0 if shared else NWL_S,
                                                ws.data_ptr(), out.data_ptr(), stream), "spart_sailh")
            return out

    def leafangles(self, ab):
        """[n, 2] (LIDFa, LIDFb) host array -> [n, 13] lidf host array."""
        ab = np.ascontiguousarray(np.asarray(ab, dtype=np.float64).reshape(-1, 2).T)
        n = ab.shape[1]
        with torch.cuda.device(self.device):
            d = torch.from_numpy(ab).to(self.device)
            out = torch.empty((n, 13), dtype=torch.float64, device=self.device)
            stream = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(self.lib.spart_leafangles(d.data_ptr(), n, n, out.data_ptr(), stream), "spart_leafangles")
            return out.cpu().numpy()

    # ---- host path -----------------------------------------------------------------
    def forward_bands_host(self, params, sensor, out=None, precision="fp64", uniform_geometry=False,
                           soil_spectrum=None, band_mode="interp", broadcast_rows=0, compact=False,
                           soil_library=None):
        """params: host float64 [27, n] (NumPy array or CPU tensor; float32 with precision="fp32") ->
        host array [n, nb, 3] of the same dtype (CompactBands when compact).  H2D, kernels and D2H are
        pipelined inside the C library; pinned memory is DMA'd directly, pageable memory is staged
        by the library's copy threads.  Other arguments as forward_bands."""
        prec = _PRECISION[precision]
        with self._use(sensor, soil_spectrum, soil_library) as (handle, st):
            p = params.numpy() if isinstance(params, torch.Tensor) else np.asarray(params)
            okdt = p.dtype == np.float64 or (p.dtype == np.float32 and prec == _lib.FP32)
            if not okdt or p.ndim != 2 or p.shape[0] != NPAR or (p.shape[1] > 1 and p.strides[1] != p.itemsize):
                raise ValueError("params must be a host float64 array [27, n] with contiguous rows"
                                 " (float32 is accepted with precision='fp32')")
            n, nb = p.shape[1], st.n_bands
            ld = p.strides[0] // p.itemsize if n >= 1 else 1
            mask = self._geometry_mask(p, n, _lib.row_mask(broadcast_rows), uniform_geometry)
            flags = self._flags(soil_spectrum, band_mode, p.dtype == np.float32, compact, soil_library=soil_library)
            elems = out_elems(n, nb, compact)
            if out is None:
                out = np.empty(elems if compact else (n, nb, NOUT), dtype=p.dtype)
            o = out.numpy() if isinstance(out, torch.Tensor) else out
            if o.dtype != p.dtype or not o.flags.c_contiguous or o.size != elems or not (
                    compact or o.shape == (n, nb, NOUT)):
                raise ValueError("out must be a C-contiguous host array of the params' dtype: [n, nb, 3], or flat with"
                                 " n*nb*2 + n elements when compact")
            _lib.check(self.lib.spart_forward_bands_host(handle, 0, p.ctypes.data, n, ld, mask, prec, flags,
                                                         o.ctypes.data), "spart_forward_bands_host")
            return CompactBands(out, n, nb, st.conv_ea, prec == _lib.FP32) if compact else out

    def profile_enable(self, sensor, on=True):
        with self._use(sensor) as (handle, _):
            _lib.check(self.lib.spart_profile_enable(handle, 1 if on else 0), "spart_profile_enable")

    def profile_read(self, sensor):
        """Summed CUDA-event durations of the three kernels since the last read:
        {'lidf_ms', 'geometry_ms', 'band_ms', 'calls'}."""
        with self._use(sensor) as (handle, _):
            ms = (_lib.c_double * _lib.NKERNELS)()
            c = _lib.c_int64()
            _lib.check(self.lib.spart_profile_read(handle, ms, _lib.byref(c)), "spart_profile_read")
            return {"lidf_ms": ms[0], "geometry_ms": ms[1], "band_ms": ms[2], "calls": c.value}

    def measure_peaks(self):
        a, b = _lib.c_double(), _lib.c_double()
        _lib.check(self.lib.spart_measure_peaks(self.device.index, _lib.byref(a), _lib.byref(b)),
                   "spart_measure_peaks")
        c = _lib.c_double()
        _lib.check(self.lib.spart_measure_fp64_chain(self.device.index, _lib.byref(c)), "spart_measure_fp64_chain")
        return {"fp64_tflops": a.value, "fp32_tflops": b.value, "fp64_register_chain_tflops": c.value}

    def launch_count(self):
        return int(self.lib.spart_launch_count())


_default = {}
_default_lock = threading.Lock()


def default_engine(device=None):
    """Process-wide engine of a device (created on first use)."""
    _require_cuda()
    idx = torch.cuda.current_device() if device is None else (
        device.index if isinstance(device, torch.device) else int(device))
    with _default_lock:
        if idx not in _default:
            _default[idx] = Engine(idx)
        return _default[idx]
