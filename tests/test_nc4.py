"""The package's own netCDF-4 (HDF5) reader, smmregrid_b200/nc4.py -- CPU only.

Pinned on files the real netCDF library wrote (two data files of the reference's test suite,
tests/golden/data/, copied by tests/golden/make_golden.py netcdf4) and, for the old on-disk style
(superblock 0, symbol tables) and for weight-shaped files, on tests/golden/h5mini.py."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
DATA = os.path.join(HERE, "golden", "data")


def test_files_written_by_the_netcdf_library():
    from smmregrid_b200 import nc4
    with nc4.File(os.path.join(DATA, "regional.nc")) as f:
        assert f.dimensions == {"time": 1, "lon": 61, "lat": 90} and f.unlimited == {"time"}
        assert f.attrs["Conventions"] == "CF-1.6" and f.attrs["history"].startswith("Fri May 19 14:01:46 2023: cdo sellonlatbox")
        assert set(f.variables) == {"time", "lon", "lat", "pr"}
        pr = f.variables["pr"]
        assert pr.dims == ("time", "lat", "lon") and pr.shape == (1, 90, 61) and pr.dtype == np.float32
        assert pr.attrs["units"] == "mm/month" and pr.attrs["_FillValue"] == np.float32(-9999.0)
        assert np.array_equal(f.variables["lon"][...], np.arange(61.0))
        assert np.array_equal(f.variables["lat"][...], np.arange(90.0) - 19.5)
        assert f.variables["lat"].attrs == {"long_name": "latitude", "axis": "Y", "standard_name": "latitude",
                                            "units": "degrees_north"}
        a = pr[...]
        assert float(a.astype(np.float64).sum()) == 288627.2366672754          # deflate + shuffle + chunking undone
        assert abs(float(a.min()) - 0.158886) < 1e-6 and abs(float(a.max()) - 271.514) < 1e-3
        assert np.array_equal(pr.decoded(), a)                                 # no fill values in this cut
        assert f.variables["time"].attrs["units"] == "days since 2004-01-15 00:00:00"
    with nc4.File(os.path.join(DATA, "healpix_0.nc")) as f:
        assert f.dimensions == {"level_full": 90, "time": 2, "x": 12}
        assert f.variables["ta"].dims == ("time", "level_full", "x") and f.variables["ta"].dtype == np.float32
        assert f.variables["tas"].dims == ("time", "x")
        assert np.array_equal(f.variables["level_full"][...], np.arange(1, 91, dtype=np.int32))
        assert int(f.variables["time"][...].astype(np.int64).sum()) == 3159216000 and f.variables["time"].dtype == np.int32
        assert float(f.variables["ta"][...].astype(np.float64).sum()) == 523979.29876708984
        assert f.variables["tas"].attrs["units"] == "K" and f.variables["tas"].attrs["grid_mapping"] == "crs"
        assert "NCO" in f.attrs


def _weights_file(tmp_path, three_d):
    import h5mini
    from smmregrid_b200 import synth
    if three_d:
        lev = np.array([0.5, 10.0, 100.0, 1000.0])
        w = synth.ocean3d_weights(36, 18, 12, 6, n_levels=4, seed=3, level_values=lev)
    else:
        w = synth.conservative_latlon(36, 18, 12, 6)
    path = str(tmp_path / ("w3d.nc" if three_d else "w2d.nc"))
    h5mini.write_weights(path, w)
    return path, w


@pytest.mark.parametrize("three_d", [False, True])
def test_weights_from_a_netcdf4_file(tmp_path, three_d):
    """CdoWeights.from_file on an HDF5 weights file (old on-disk style, as h5py / h5netcdf write):
    every variable equal to its source, the level dimension found through DIMENSION_LIST, the level
    values from its coordinate variable, global attributes kept."""
    from smmregrid_b200 import CdoWeights, nc4
    path, w = _weights_file(tmp_path, three_d)
    assert nc4.is_hdf5(path)
    back = CdoWeights.from_file(path)
    for k in ("src_address", "dst_address", "remap_matrix", "src_grid_imask", "dst_grid_imask", "dst_grid_frac",
              "dst_grid_dims", "src_grid_dims", "dst_grid_center_lat"):
        assert np.array_equal(np.asarray(back[k]), np.asarray(w[k]).reshape(np.asarray(back[k]).shape)), k
        assert np.asarray(back[k]).dtype == np.asarray(w[k]).dtype or k.endswith("dims") or k.endswith("address"), k
    assert back.attrs["map_method"] == "Conservative remapping"
    if three_d:
        assert back.mask_dim == "depth_full" and np.array_equal(back.levels, [0.5, 10.0, 100.0, 1000.0])
        assert np.array_equal(back["link_length"], w["link_length"])
    else:
        assert back.mask_dim is None
    with nc4.File(path) as f:
        assert f.variables["remap_matrix"].dims[-2:] == ("num_links", "num_wgts")
        assert f.dimensions["num_links"] == np.asarray(w["src_address"]).shape[-1]
        assert f.variables["remap_matrix"].attrs == {"units": "1"}


def test_damaged_files_are_reported(tmp_path):
    from smmregrid_b200 import CdoWeights, nc4
    bad = str(tmp_path / "bad.nc")
    with open(bad, "wb") as f:
        f.write(nc4.MAGIC + b"\0" * 64)
    with pytest.raises(OSError):
        CdoWeights.from_file(bad)
    good = open(os.path.join(DATA, "regional.nc"), "rb").read()
    cut = str(tmp_path / "cut.nc")
    with open(cut, "wb") as f:
        f.write(good[:len(good) // 3])
    with pytest.raises(OSError):
        with nc4.File(cut) as f:
            f.variables["pr"][...]
    with pytest.raises(ValueError):
        other = str(tmp_path / "x.bin")
        open(other, "wb").write(b"hello world, not a weights file")
        CdoWeights.from_file(other)
