"""Batched entry point: the drop-in for a loop over `SPART(...).run()`.

    out = run_batch(leaf, soil, canopy, angles, atm, doy, "Sentinel2A-MSI")   # [n, nb, 3]

replaces (reference src/SPART/SPART.py:83-95, 162-269)

    for i in range(n):
        out[i] = SPART(SoilParameters(*soil[i]), LeafBiology(*leaf[i]), CanopyStructure(*canopy[i]),
                       AtmosphericProperties(*atm[i]), Angles(*angles[i]), sensor, doy[i]).run()[...]

with one fresh model object per sample (the reference's dirty-flag cache is not reproduced,
SURVEY.md section 3.2).
"""
import warnings

import numpy as np
import pandas as pd
import torch

from .engine import NPAR, CompactBands, default_engine

_GROUPS = (("leaf", 9), ("soil", 6), ("canopy", 4), ("angles", 3), ("atm", 4), ("doy", 1))


def pack_batch(leaf, soil, canopy, angles, atm, doy, device=None):
    """Assemble the [27, n] float64 parameter block (layout of include/spart_b200.h).

    leaf [n, 9] (or [n, 7]: PROT = CBC = 0), soil [n, 6] (or [n, 4]: SMC = 25, film = 0.015),
    canopy [n, 4], angles [n, 3] or [3], atm [n, 4], doy [n] or scalar.  NumPy arrays give a
    NumPy block, torch tensors give a torch block on `device` (or on the tensors' device).
    """
    use_torch = any(isinstance(x, torch.Tensor) for x in (leaf, soil, canopy, angles, atm, doy))
    if use_torch:
        dev = device
        for x in (leaf, soil, canopy, angles, atm, doy):
            if isinstance(x, torch.Tensor) and dev is None:
                dev = x.device
        as2d = lambda x: torch.as_tensor(x, dtype=torch.float64, device=dev).reshape(-1, 1) if (
            torch.as_tensor(x).dim() <= 1) else torch.as_tensor(x, dtype=torch.float64, device=dev)
        cat, full, empty = torch.cat, (lambda n, w, v: torch.full((n, w), v, dtype=torch.float64, device=dev)), None
    else:
        as2d = lambda x: np.asarray(x, dtype=np.float64).reshape(-1, 1) if np.ndim(x) <= 1 else np.asarray(
            x, dtype=np.float64)
        cat = lambda xs, dim: np.concatenate(xs, axis=dim)
        full = lambda n, w, v: np.full((n, w), v, dtype=np.float64)

    leaf, soil, canopy, atm = as2d(leaf), as2d(soil), as2d(canopy), as2d(atm)
    n = leaf.shape[0]
    if leaf.shape[1] == 7:
        leaf = cat([leaf, full(n, 2, 0.0)], 1)
    if soil.shape[1] == 4:
        soil = cat([soil, full(n, 1, 25.0), full(n, 1, 0.015)], 1)
    ang = as2d(angles)
    if ang.shape[0] == 3 and ang.shape[1] == 1:          # shared geometry [3]
        ang = ang.reshape(1, 3).expand(n, 3) if use_torch else np.broadcast_to(ang.reshape(1, 3), (n, 3))
    d = as2d(doy)
    if d.shape[0] == 1 and n != 1:
        d = d.expand(n, 1) if use_torch else np.broadcast_to(d, (n, 1))
    cols = [leaf, soil, canopy, ang, atm, d]
    for (name, width), c in zip(_GROUPS, cols):
        if c.shape != (n, width):
            raise ValueError(f"{name}: expected shape ({n}, {width}), got {tuple(c.shape)}")
    block = cat(cols, 1)                                   # [n, 27]
    return block.t().contiguous() if use_torch else np.ascontiguousarray(block.T)


_warned = set()


def _warn_once(key, text):
    """The reference prints / warns per object (prospect_5d.py:150-154, bsm.py:274-286); a batch of a
    million samples says it once per process."""
    if key not in _warned:
        _warned.add(key)
        warnings.warn(text, stacklevel=3)


def _pro_warning(params):
    """PROSPECT-PRO switch (prospect_5d.py:148-155): PROT / CBC > 0 together with Cdm > 0 sets Cdm = 0."""
    if "pro" in _warned or params.shape[1] == 0:
        return
    pro = (params[7] > 0) | (params[8] > 0)
    hit = (pro & (params[1] > 0)).any()
    if bool(hit.item() if isinstance(hit, torch.Tensor) else hit):
        _warn_once("pro", "WARNING: When setting PROT and/or CBC > 0. we assume that PROSPECT-PRO was called. "
                          "Cdm will be therefore set to zero (Cdm = PROT + CBC)")


def run_batch_params(params, sensor, precision="fp64", device=None, out=None, uniform_geometry=False,
                     soil_spectrum=None, band_mode="interp", broadcast_rows=0, compact=False, warn=False,
                     lidf=None, soil_library=None):
    """params: [27, n] float64 (float32 with precision="fp32": float32 in, float32 out).  CUDA tensor
    in -> CUDA tensor [n, nb, 3] out (asynchronous on the current stream); NumPy array / CPU tensor
    in -> NumPy array out (copies pipelined in the C library).

    broadcast_rows: rows (bit mask or indices) that are constant over the batch; only their first
    element is read and, on the host path, copied.  uniform_geometry=True: the angle rows 19..21 are
    verified to be constant over the batch (SpartError otherwise) and treated as broadcast rows; the
    result is the same to a few ulp, only faster.
    soil_spectrum: dry-soil reflectance [2001] shared by the batch (the reference's
    SoilParametersFromFile, bsm.py:155-226); the B / lat / lon rows are then ignored.
    soil_library: a SoilLibrary of measured dry-soil spectra, one selected per sample: row 9 (B) holds the
    sample's 0-based index into the library (a broadcast row 9 selects one spectrum for the batch), rows 10, 11
    are ignored.  An index that is not a whole number in [0, k) gives NaN soil-dependent outputs.
    band_mode="srf" replaces the reference's np.interp band sampling of the canopy reflectances by
    the sensor's spectral-response-weighted band means (FP64 only).
    compact=True returns a CompactBands (R_TOC, R_TOA and the per-sample ET scale; L_TOA is rebuilt
    bit for bit on demand): two thirds of the bytes on every copy.
    warn=True emits the reference's PROSPECT-PRO warning once if the batch triggers it.
    lidf: leaf inclination distribution [n, 13] (or 13 values for the whole batch) used instead of the one
    derived from LIDFa / LIDFb, like an assigned `CanopyStructure.lidf` in the reference (FP64, one sensor)."""
    if warn:
        _pro_warning(params)
    kw = dict(precision=precision, uniform_geometry=uniform_geometry, soil_spectrum=soil_spectrum,
              soil_library=soil_library, band_mode=band_mode, broadcast_rows=broadcast_rows, compact=compact)
    if isinstance(sensor, (list, tuple)):      # several sensors on one batch (e.g. Sentinel-2A + -2B)
        if not (isinstance(params, torch.Tensor) and params.is_cuda):
            eng = default_engine(device)
            dev_params = torch.as_tensor(np.ascontiguousarray(params) if not isinstance(params, torch.Tensor)
                                         else params).to(eng.device)
            outs = eng.forward_bands_multi(dev_params, list(sensor), **kw)
            if compact:
                return [CompactBands(o.buf.cpu().numpy(), o.n, o.nb, o.conv_ea_f64, o.fp32) for o in outs]
            return [o.cpu().numpy() for o in outs]
        return default_engine(params.device).forward_bands_multi(params, list(sensor), outs=out, **kw)
    if lidf is not None and isinstance(sensor, (list, tuple)):
        raise ValueError("lidf= takes one sensor per call")
    if isinstance(params, torch.Tensor) and params.is_cuda:
        return default_engine(params.device).forward_bands(params, sensor, out=out, lidf=lidf, **kw)
    if lidf is not None:         # host arrays with an explicit distribution: through the device path
        eng = default_engine(device)
        dev = torch.as_tensor(np.ascontiguousarray(params) if not isinstance(params, torch.Tensor) else params).to(eng.device)
        res = eng.forward_bands(dev, sensor, lidf=lidf, **kw)
        if compact:
            return CompactBands(res.buf.cpu().numpy(), res.n, res.nb, res.conv_ea_f64, res.fp32)
        return res.cpu().numpy()
    return default_engine(device).forward_bands_host(params, sensor, out=out, **kw)


def run_batch(leaf, soil, canopy, angles, atm, doy, sensor, precision="fp64", device=None, out=None,
              soil_spectrum=None, band_mode="interp", compact=False, soil_library=None, soil_index=None):
    """Batched SPART forward run -> [n, nb, 3] ordered (R_TOC, R_TOA, L_TOA).  Arguments given in
    their short forms (angles [3], scalar doy, leaf [n, 7], soil [n, 4]) become broadcast rows.
    soil_library (a SoilLibrary) with soil_index ([n] 0-based indices, or one index for the whole batch):
    every sample takes its dry-soil spectrum from the library; soil's B / lat / lon columns are then ignored."""
    if (soil_library is None) != (soil_index is None):
        raise ValueError("soil_library and soil_index go together")
    ndim = lambda x: x.dim() if hasattr(x, "dim") else np.ndim(x)
    width = lambda x: x.shape[1] if ndim(x) == 2 else None
    rows = []
    if ndim(angles) == 1:
        rows += [19, 20, 21]
    if ndim(doy) == 0:
        rows += [26]
    if width(leaf) == 7:
        rows += [7, 8]                 # PROT = CBC = 0
    if width(soil) == 4:
        rows += [13, 14]               # SMC = 25, film = 0.015
        _warn_once("smc", "BSM soil model: SMC not supplied, set to default of 25 %")
        _warn_once("film", "BSM soil model: water film optical thickness not supplied, set to default of 0.0150 cm")
    params = pack_batch(leaf, soil, canopy, angles, atm, doy, device)
    if soil_index is not None:
        if ndim(soil_index) == 0:
            rows += [9]
        if isinstance(params, torch.Tensor):
            params[9] = torch.as_tensor(soil_index, dtype=torch.float64, device=params.device)
        else:
            params[9] = np.asarray(soil_index, dtype=np.float64)
    return run_batch_params(params, sensor, precision, device, out, soil_spectrum=soil_spectrum,
                            soil_library=soil_library, band_mode=band_mode, broadcast_rows=rows, compact=compact,
                            warn=True)


def row_as_dataframe(out_row, sensor, engine=None):
    """One row [nb, 3] of a batch result as the DataFrame `SPART.run()` returns
    (SPART.py:254-260): columns Band, L_TOA, R_TOA, R_TOC indexed by band-centre wavelength."""
    _, st = (engine or default_engine()).sensor(sensor)
    r = out_row.detach().cpu().numpy() if isinstance(out_row, torch.Tensor) else np.asarray(out_row)
    return pd.DataFrame(zip(st.band_id, r[:, 2], r[:, 1], r[:, 0]), index=st.wl_smac,
                        columns=["Band", "L_TOA", "R_TOA", "R_TOC"])
