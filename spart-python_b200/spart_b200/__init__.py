"""spart_b200 -- B200-native batched SPART forward model.

Public surface = the reference's (`LeafBiology`, `SoilParameters`, `CanopyStructure`,
`Angles`, `AtmosphericProperties`, `SPART(...).run()`; reference src/SPART/__init__.py:1-5)
plus the batched entry points `run_batch` / `run_batch_params`.
"""
from ._lib import SpartError
from .batch import pack_batch, row_as_dataframe, run_batch, run_batch_params
from . import inversion, lut, sensitivity
from .engine import CompactBands, Engine, default_engine
from .model import SPART, SpectralBands, load_optical_parameters, load_sensor_info
from .params import (Angles, AtmosphericProperties, CanopyStructure, LeafBiology, SoilParameters,
                     SoilLibrary, SoilParametersFromFile, pack_params)
from .stages import (BSM, PROSPECT_5D, SAILH, SMAC, bsm_batch, prospect_batch, sailh_batch, smac_batch,
                     set_leaf_refl_trans_assumptions, set_soil_refl_trans_assumptions)
from .tables import SENSOR_NAMES, synthetic_fullspectrum_sensorinfo

__all__ = [
    "SPART", "SpectralBands", "LeafBiology", "SoilParameters", "SoilParametersFromFile", "SoilLibrary",
    "CanopyStructure", "Angles",
    "AtmosphericProperties", "run_batch", "run_batch_params", "pack_batch", "pack_params",
    "row_as_dataframe", "lut", "sensitivity", "inversion", "Engine", "CompactBands", "default_engine", "SpartError", "SENSOR_NAMES",
    "load_optical_parameters", "load_sensor_info", "synthetic_fullspectrum_sensorinfo",
    "PROSPECT_5D", "BSM", "SAILH", "SMAC", "prospect_batch", "bsm_batch", "sailh_batch", "smac_batch",
    "set_leaf_refl_trans_assumptions", "set_soil_refl_trans_assumptions",
]
