"""CPU-only checks of the soil library (SoilLibrary, SPART_FLAG_SOIL_LIBRARY): shapes, loading, the per-sample
migration path, argument rules and the flag's value in the C header."""
import re

import numpy as np
import pytest
import torch

from conftest import ROOT


def spectra(k, seed=0):
    return np.random.default_rng(seed).uniform(0.05, 0.6, (k, 2001))


def test_soil_library_shapes():
    import spart_b200 as sb
    a = spectra(5)
    lib = sb.SoilLibrary(a)
    assert len(lib) == 5 and lib.spectra.dtype == np.float64 and np.array_equal(lib.spectra, a)
    assert not lib.spectra.flags.writeable
    a[0, 0] = -1.0                                       # the library keeps its own copy
    assert lib.spectra[0, 0] != -1.0
    assert sb.SoilLibrary(lib.spectra[:, :, None]).digest == lib.digest      # stacked SoilParametersFromFile.rdry
    assert sb.SoilLibrary(spectra(5, seed=1)).digest != lib.digest
    for bad in (np.zeros((3, 2000)), np.zeros(2001), np.zeros((0, 2001)), np.zeros((2, 2001, 2))):
        with pytest.raises(ValueError):
            sb.SoilLibrary(bad)
    assert sb.SoilLibrary.MAX_SPECTRA == 2 ** 24


def test_soil_library_from_files(tmp_path):
    """JPL spectral-library text files, read as SoilParametersFromFile reads them."""
    import spart_b200 as sb
    wl_um = np.arange(2.5, 0.3995, -0.0005)
    paths = []
    for j, slope in enumerate((20.0, 35.0)):
        f = tmp_path / f"soil{j}.txt"
        with open(f, "w") as fh:
            fh.write("\n".join(f"header {i}" for i in range(21)) + "\n")
            for w, r in zip(wl_um, 10 + slope * (wl_um - 0.4)):
                fh.write(f"{w:.4f}\t{r:.6f}\n")
        paths.append(str(f))
    lib = sb.SoilLibrary.from_files(paths)
    assert lib.spectra.shape == (2, 2001)
    for j, p in enumerate(paths):
        assert np.array_equal(lib.spectra[j], sb.SoilParametersFromFile(p, 20, 25, 0.015).rdry[:, 0])


def test_soil_library_from_per_sample_round_trip():
    import spart_b200 as sb
    base = spectra(4)
    rng = np.random.default_rng(2)
    pick = rng.integers(0, 4, 50)
    per_sample = base[pick]
    lib, index = sb.SoilLibrary.from_per_sample(per_sample)
    assert len(lib) == 4 and index.shape == (50,) and index.dtype == np.float64
    assert np.array_equal(lib.spectra[index.astype(int)], per_sample)
    lib3, index3 = sb.SoilLibrary.from_per_sample(per_sample[:, :, None])
    assert lib3.digest == lib.digest and np.array_equal(index3, index)


def test_flag_matches_header_and_exports():
    from spart_b200 import _lib
    header = (ROOT / "include" / "spart_b200.h").read_text()
    assert int(re.search(r"SPART_FLAG_SOIL_LIBRARY\s*=\s*(\d+)", header).group(1)) == _lib.FLAG_SOIL_LIBRARY == 128
    assert "spart_create_with_soils" in _lib.EXPORTS
    assert int(re.search(r"#define SPART_ABI_VERSION (\d+)", header).group(1)) == _lib.ABI_VERSION == 5


def test_soil_library_exported_from_spart_alias():
    import SPART
    import spart_b200
    assert SPART.SoilLibrary is spart_b200.SoilLibrary


def test_run_batch_soil_arguments_go_together():
    import spart_b200 as sb
    P = np.zeros((4, 27))
    args = (P[:, 0:9], P[:, 9:15], P[:, 15:19], P[:, 19:22], P[:, 22:26], P[:, 26], "Sentinel2A-MSI")
    with pytest.raises(ValueError):
        sb.run_batch(*args, soil_index=np.zeros(4))
    with pytest.raises(ValueError):
        sb.run_batch(*args, soil_library=sb.SoilLibrary(spectra(2)))


def test_soil_spectrum_and_library_exclude_each_other():
    """Checked before any context is created, so without a GPU too."""
    import spart_b200 as sb
    from spart_b200.engine import Engine
    lib = sb.SoilLibrary(spectra(2))
    eng = Engine.__new__(Engine)            # argument checks of sensor() run before it touches the device
    with pytest.raises(ValueError):
        eng.sensor("Sentinel2A-MSI", soil_spectrum=lib.spectra[0], soil_library=lib)
    with pytest.raises(TypeError):
        eng.sensor("Sentinel2A-MSI", soil_library=lib.spectra)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_soil_library_fails_loudly_without_gpu():
    import spart_b200 as sb
    from spart_b200 import _lib
    lib = sb.SoilLibrary(spectra(2))
    with pytest.raises(sb.SpartError):
        sb.run_batch_params(np.zeros((27, 4)), "Sentinel2A-MSI", soil_library=lib)
    tabs = _lib.SpartTables(n_wl=2001, lc=_lib.as_double_ptr(np.zeros((17, 2001))))
    handle = _lib.c_void_p()
    rc = _lib.load().spart_create_with_soils(_lib.byref(tabs), None, 0, _lib.as_double_ptr(lib.spectra), 2, 0,
                                             _lib.byref(handle))
    assert rc == -2 and b"no CUDA device" in _lib.load().spart_last_error()
