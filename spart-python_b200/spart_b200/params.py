"""Parameter holders with the names, argument order, defaults, warnings and attributes of
the reference's classes, so that user scripts written for wirrell/SPART-python run unchanged.

  LeafBiology            reference src/SPART/prospect_5d.py:19-83
  SoilParameters         reference src/SPART/bsm.py:229-287
  SoilParametersFromFile reference src/SPART/bsm.py:155-226   (dry spectrum supplied by the user)
  SoilLibrary            (new) many such spectra, one selected per sample of a batch
  CanopyStructure        reference src/SPART/sailh.py:304-348
  Angles                 reference src/SPART/sailh.py:275-301
  AtmosphericProperties  reference src/SPART/smac.py:275-330
"""
import hashlib
import math
import warnings
from dataclasses import dataclass

import numpy as np


@dataclass
class LeafBiology:
    """Leaf biochemistry for PROSPECT-5D / PROSPECT-PRO (positional order as in the reference:
    Cab, Cdm, Cw, Cs, Cca, Cant, N, PROT, CBC)."""
    Cab: float
    Cdm: float
    Cw: float
    Cs: float
    Cca: float
    Cant: float
    N: float
    PROT: float = 0.0
    CBC: float = 0.0
    rho_thermal: float = 0.01
    tau_thermal: float = 0.01

    def as_row(self):
        return [self.Cab, self.Cdm, self.Cw, self.Cs, self.Cca, self.Cant, self.N, self.PROT, self.CBC]


class SoilParameters:
    """BSM soil: brightness B, spectral coordinates lat/lon, moisture SMp [%], carrying
    capacity SMC (default 25, with the reference's warning) and film thickness (default
    0.015 cm, with the reference's warning)."""

    def __init__(self, B, lat, lon, SMp, SMC=None, film=None):
        self.B = B
        self.lat = lat
        self.lon = lon
        self.SMp = SMp
        if SMC is None:
            warnings.warn("BSM soil model: SMC not supplied, set to default of 25 %")
            SMC = 25
        self.SMC = SMC
        if film is None:
            warnings.warn("BSM soil model: water film optical thickness not supplied, set to default of 0.0150 cm")
            film = 0.0150
        self.film = film
        self.rdry_set = False

    def as_row(self):
        return [self.B, self.lat, self.lon, self.SMp, self.SMC, self.film]


class SoilParametersFromFile:
    """Dry-soil reflectance supplied by the user: a JPL spectral-library text file
    (https://speclib.jpl.nasa.gov/) or an array with the 2001 values for 400..2400 nm
    (reference bsm.py:155-226).  SMp / SMC / film as in SoilParameters."""

    def __init__(self, soil_file, SMp, SMC=None, film=None):
        if SMC is None:
            warnings.warn("BSM soil model: SMC not supplied, set to default of 25 %")
            SMC = 25
        self.SMC = SMC
        if film is None:
            warnings.warn("BSM soil model: water film optical thickness not supplied,")
            warnings.warn("\t set to default of 0.0150 cm")
            film = 0.0150
        self.film = film
        self.rdry = soil_file if isinstance(soil_file, np.ndarray) else self._load_jpl_soil_refl(soil_file)
        self.SMp = SMp
        self.rdry_set = True

    @staticmethod
    def _load_jpl_soil_refl(file_path):
        """JPL file: 21 header lines, then tab-separated wavelength [um] / reflectance [% or
        fraction] in descending wavelength order.  Returns [2001, 1] on the 1 nm grid; like the
        reference, missing integer wavelengths are filled by pandas' positional linear
        interpolation (bsm.py:201-226)."""
        import pandas as pd
        refl = pd.read_csv(file_path, sep="\t", skiprows=21, index_col=0, header=None)
        refl.index = refl.index * 1000
        if (refl.loc[:, 1] > 1).any():
            refl = refl / 100
        refl = refl.sort_index().loc[400:2401]       # label slice (the files list wavelengths descending)
        wls = np.arange(400, 2401, 1)
        missing = [wl for wl in wls if wl not in refl.index]
        if missing:
            refl = pd.concat([refl, pd.DataFrame({1: np.nan}, index=missing)])
        refl = refl.sort_index().interpolate("linear")
        return refl.loc[wls].to_numpy()

    def as_row(self):
        return [0.0, 0.0, 0.0, self.SMp, self.SMC, self.film]      # B, lat, lon are not used


class SoilLibrary:
    """A library of k measured dry-soil spectra on the 400..2400 nm grid, for batches in which every sample
    takes its own spectrum -- e.g. a look-up table whose entries each use one soil of the library, where the
    reference builds one SoilParametersFromFile per SPART object.  Passed as `soil_library=` to the batched
    entry points; row 9 (B) of the parameter block then holds each sample's 0-based index into the library
    (rows 10, 11 are ignored).  An index that is not a whole number in [0, k) gives NaN soil outputs.

    spectra: [k, 2001], or [k, 2001, 1] as stacked SoilParametersFromFile.rdry arrays; 1 <= k <= 2^24.
    The library keeps a read-only float64 copy (`spectra`) and its content digest (`digest`)."""

    MAX_SPECTRA = 1 << 24         # F32_IO carries the index as a float, which is exact for whole numbers up to 2^24

    def __init__(self, spectra):
        a = np.asarray(spectra, dtype=np.float64)
        if a.ndim == 3 and a.shape[2] == 1:
            a = a[:, :, 0]
        if a.ndim != 2 or a.shape[1] != 2001:
            raise ValueError(f"soil library spectra must be [k, 2001] (or [k, 2001, 1]), got {a.shape}")
        if not 1 <= a.shape[0] <= self.MAX_SPECTRA:
            raise ValueError(f"a soil library holds 1 to 2^24 spectra, got {a.shape[0]}")
        a = np.array(a, dtype=np.float64, order="C")          # own copy
        a.flags.writeable = False
        self.spectra = a
        self.digest = hashlib.sha1(a.tobytes()).hexdigest()

    def __len__(self):
        return self.spectra.shape[0]

    @classmethod
    def from_files(cls, paths):
        """One spectrum per JPL spectral-library text file, read as SoilParametersFromFile does."""
        return cls(np.stack([SoilParametersFromFile._load_jpl_soil_refl(p) for p in paths]))

    @classmethod
    def from_per_sample(cls, spectra):
        """spectra [n, 2001] (one dry-soil spectrum per sample, e.g. the rdry of one SoilParametersFromFile per
        sample) -> (library of the distinct spectra, index [n] float64) with library.spectra[index] == spectra."""
        a = np.asarray(spectra, dtype=np.float64)
        if a.ndim == 3 and a.shape[2] == 1:
            a = a[:, :, 0]
        if a.ndim != 2 or a.shape[1] != 2001:
            raise ValueError(f"per-sample spectra must be [n, 2001], got {a.shape}")
        uniq, index = np.unique(np.ascontiguousarray(a), axis=0, return_inverse=True)
        return cls(uniq), index.reshape(-1).astype(np.float64)


class CanopyStructure:
    """SAILH canopy: LAI, leaf-inclination parameters LIDFa / LIDFb, hot-spot parameter q.
    `nlayers`, `nlincl`, `nlazi` are the SAIL assumptions 60 / 13 / 36.  `lidf` (the
    13-class leaf inclination distribution the reference computes in its constructor) is
    evaluated on the GPU on first access; an assigned `lidf` replaces it, as in the reference."""

    def __init__(self, LAI, LIDFa, LIDFb, q):
        self.LAI = LAI
        self.LIDFa = LIDFa
        self.LIDFb = LIDFb
        self.q = q
        self.nlayers = 60
        self.nlincl = 13
        self.nlazi = 36
        self._lidf = None
        self.lidf_set = False          # True once a distribution has been assigned (it then replaces LIDFa / LIDFb)

    @property
    def lidf(self):
        if self._lidf is None:
            from .engine import default_engine
            self._lidf = default_engine().leafangles(np.array([[self.LIDFa, self.LIDFb]], dtype=np.float64))[0][:, None]
        return self._lidf

    @lidf.setter
    def lidf(self, value):
        # the reference uses an assigned distribution as is (sailh.py:81-97 read canopy.lidf); so does the GPU
        # path (SPART_FLAG_USER_LIDF): LIDFa / LIDFb are then ignored
        v = np.asarray(value, dtype=np.float64).reshape(-1)
        if v.shape[0] != 13:
            raise ValueError("lidf must hold the 13 leaf-inclination classes of sailh.py:49")
        self._lidf = v[:, None].copy()
        self.lidf_set = True

    def as_row(self):
        return [self.LAI, self.LIDFa, self.LIDFb, self.q]


class Angles:
    """Solar zenith, observer zenith and relative azimuth angle in degrees."""

    def __init__(self, sol_angle, obs_angle, rel_angle):
        self.sol_angle = sol_angle
        self.obs_angle = obs_angle
        self.rel_angle = rel_angle

    def as_row(self):
        return [self.sol_angle, self.obs_angle, self.rel_angle]


def _pressure_from_altitude(alt_m, temp_k):
    """Barometric formula used when Pa is not given (smac.py:320-330)."""
    g, M, R0, Pa0 = 9.80665, 0.02896968, 8.314462618, 1013.25
    return Pa0 * math.exp(-(g * alt_m * M / (temp_k * R0)))


class AtmosphericProperties:
    """SMAC atmosphere: aot550, ozone uo3 [cm-atm], water vapour uh2o [g cm-2] and surface
    pressure Pa [hPa] (default 1013.25, or derived from alt_m + temp_k)."""

    def __init__(self, aot550, uo3, uh2o, Pa=None, alt_m=None, temp_k=None):
        self.aot550 = aot550
        self.uo3 = uo3
        self.uh2o = uh2o
        if Pa is None:
            if alt_m is not None and temp_k is not None:
                Pa = _pressure_from_altitude(alt_m, temp_k)
            else:
                Pa = 1013.25
        self.Pa = Pa

    def as_row(self):
        return [self.aot550, self.uo3, self.uh2o, self.Pa]


def pack_params(soilpar, leafbio, canopy, atm, angles, DOY):
    """One sample as a [27, 1] float64 column in the batch layout of include/spart_b200.h."""
    row = leafbio.as_row() + soilpar.as_row() + canopy.as_row() + angles.as_row() + atm.as_row() + [DOY]
    return np.asarray(row, dtype=np.float64).reshape(27, 1)
