"""SURVEY 8b-2: the reference's OWN Python package on the B200 path.

build/reference_bindings/pyrichdem/ (built by oracle/Makefile where the reference's sources are available; git-ignored)
holds
  * `_richdem.so`    -- the reference's pybind11 binding source (wrappers/pyrichdem/src/pywrapper.cpp), unmodified,
                        compiled with include/richdem_b200.hpp in front of it (tests/pyrichdem_module.cpp), so that
                        rdFillDepressionsD8 / rdResolveFlatsEpsilon / FA_* / FM_* / FlowAccumulation on float32 rasters
                        are the explicit specialisations that call librichdem_b200.so;
  * `richdem/__init__.pyc` -- the byte-compiled, unmodified wrappers/pyrichdem/richdem/__init__.py.
The tests drive `richdem.FillDepressions / ResolveFlats / FlowAccumulation / FlowProportions / FlowAccumFromProps`
exactly as a pyrichdem user would (reference __init__.py:381,461,490,650,599) and compare with the golden outputs of
the unmodified CPU reference."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(os.path.dirname(HERE), "build", "reference_bindings", "pyrichdem")
ND = -9999.0


@pytest.fixture(scope="module")
def rdref():
    if not os.path.exists(os.path.join(PKG, "richdem", "__init__.pyc")) or not any(
            f.startswith("_richdem") for f in os.listdir(PKG)):
        pytest.skip("build/reference_bindings/pyrichdem not built (reference tree absent at build time)")
    sys.path.insert(0, PKG)
    try:
        import richdem  # the reference package, unmodified
    finally:
        sys.path.remove(PKG)
    assert os.path.dirname(richdem.__file__).startswith(PKG)
    # pkg_resources.require("richdem") needs an installed distribution (reference __init__.py:26-31); the
    # package is imported from a build directory here
    richdem._RichDEMVersion = lambda: "RichDEM (reference Python layer over librichdem_b200)"
    return richdem


def test_module_binds_the_b200_library(rdref):
    import _richdem
    with open("/proc/self/maps") as f:
        maps = f.read()
    assert "librichdem_b200.so" in maps, "the reference binding must have pulled in the B200 library"
    assert _richdem.rdHash() == "b200"


def test_reference_python_api_on_beauford_crop(rdref, golden):
    rd = rdref
    g = golden["beauford_crop"]
    dem = rd.rdarray(g["dem"].copy(), no_data=ND)
    filled = rd.FillDepressions(dem, in_place=False)            # reference __init__.py:381
    assert type(filled) is rd.rdarray and np.array_equal(np.asarray(filled), g["filled"])
    assert np.array_equal(np.asarray(dem), g["dem"]), "in_place=False leaves the input alone"
    resolved = rd.ResolveFlats(filled, in_place=False)          # :461
    assert np.array_equal(np.asarray(resolved), g["resolved"])
    acc = rd.FlowAccumulation(resolved, method="D8")            # :490
    assert acc.dtype == np.float64 and acc.no_data == -1
    assert np.array_equal(np.asarray(acc), g["fa_d8"])
    accinf = rd.FlowAccumulation(resolved, method="Dinf")
    np.testing.assert_allclose(np.asarray(accinf), g["fa_dinf"], rtol=5e-7, atol=0)  # the unit-weight D-infinity walk may use packed fixed-point sums (< 2^-23)
    props = rd.FlowProportions(resolved, method="Dinf")         # :650
    assert props.shape == g["resolved"].shape + (9,)
    got = np.asarray(props).reshape(-1, 9)[::7]
    assert np.array_equal(got > 0, g["fm_dinf_nz"] > 0)
    assert np.abs(got.view(np.int32).astype(np.int64) - g["fm_dinf_nz"].view(np.int32).astype(np.int64)).max() <= 1
    acc2 = rd.FlowAccumFromProps(props)                         # :599
    np.testing.assert_allclose(np.asarray(acc2), g["fa_dinf"], rtol=1e-6, atol=0)
    # in-place variants mutate the caller's array (reference semantics)
    d2 = rd.rdarray(g["dem"].copy(), no_data=ND)
    assert rd.FillDepressions(d2, in_place=True) is None
    assert np.array_equal(np.asarray(d2), g["filled"])
    assert "FillDepressions" in d2.metadata["PROCESSING_HISTORY"]


def test_reference_python_api_weights_and_other_methods(rdref, golden):
    rd = rdref
    g = golden["flow_metrics_ref"]
    dem = rd.rdarray(golden["beauford_crop"]["resolved"].copy(), no_data=ND)
    for m, e in (("D4", None), ("Quinn", None), ("Holmgren", 2.5), ("Freeman", 1.1)):
        acc = rd.FlowAccumulation(dem, method=m, exponent=e)
        np.testing.assert_allclose(np.asarray(acc)[::3, ::3], g[f"beauford__{m}_{e}__fa"], rtol=1e-6, atol=0, err_msg=m)
    w = rd.rdarray(np.full(dem.shape, 2.0), no_data=-1)
    acc = rd.FlowAccumulation(dem, method="D8", weights=w)
    assert np.array_equal(np.asarray(acc)[np.asarray(dem) != ND], 2.0 * golden["beauford_crop"]["fa_d8"][np.asarray(dem) != ND])
    with pytest.raises(Exception, match="requires an exponent"):
        rd.FlowAccumulation(dem, method="Holmgren")


def test_other_dtypes_keep_the_reference_cpu_templates(rdref, golden):
    """float64 rasters are outside the drop-in (only float is specialised): same module, reference CPU code, same answer."""
    rd = rdref
    g = golden["fill_testdem1"]
    f64 = rd.rdarray(g["dem"].astype(np.float64), no_data=float(g["nodata"]))
    assert np.array_equal(np.asarray(rd.FillDepressions(f64)), g["expected"].astype(np.float64))


def test_reference_terrain_attribute_runs_on_the_b200(rdref, golden):
    """richdem.TerrainAttribute (reference __init__.py:735-794) -> TA_x<float> (pywrapper.hpp:46-53) -> the explicit
    specialisations of include/richdem_b200.hpp -> rdb200_terrain_attribute_f32."""
    rd = rdref
    g = golden["terrain_attributes_ref"]
    dem = rd.rdarray(golden["beauford_crop"]["dem"].copy(), no_data=ND, geotransform=[0, 30.0, 0, 0, 0, -20.0])
    for attrib in ("slope_riserun", "slope_percentage", "curvature", "planform_curvature", "profile_curvature"):
        out = rd.TerrainAttribute(dem, attrib, zscale=2.5)
        assert out.dtype == np.float32 and out.no_data == -9999
        assert np.array_equal(np.asarray(out)[::3, ::3].view(np.uint32), g[f"beauford__{attrib}__2.5"].view(np.uint32)), attrib
    for attrib in ("slope_degrees", "slope_radians", "aspect"):
        got = np.asarray(rd.TerrainAttribute(dem, attrib, zscale=2.5))[::3, ::3]
        ref = g[f"beauford__{attrib}__2.5"]
        assert np.abs(got.view(np.int32).astype(np.int64) - ref.view(np.int32).astype(np.int64)).max() <= 1, attrib
