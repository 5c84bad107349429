"""CPU-side checks: the C-ABI library builds/loads and exports every symbol the header declares,
the Python mirror of the reference API validates arguments like the reference does, and compute
calls fail loudly (no CPU fallback) when no B200 is visible."""
import ctypes
import os
import re

import numpy as np
import pytest


import richdem_b200 as rd
from richdem_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _has_gpu():
    import torch
    return torch.cuda.is_available()


def test_library_builds_and_exports_every_declared_symbol():
    path = build.build()
    assert os.path.exists(path)
    header = open(os.path.join(ROOT, "include", "richdem_b200.h")).read()
    declared = set(re.findall(r"RDB200_API[^;]*?\b(rdb200_\w+)\s*\(", header))
    assert len(declared) >= 30
    L = ctypes.CDLL(path)
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/richdem_b200.h but not exported"
    # and the ctypes table covers the whole header
    assert declared == set(_lib.SIGNATURES) | set(_lib.OTHER_SYMBOLS)
    assert _lib.lib().rdb200_version() == 100


def test_sass_contains_tma_and_no_legacy_paths():
    """The fill sweep stages tiles with TMA (UTMALDG in SASS, B200_PROFILING.md) and the library
    is built for sm_100a only."""
    import subprocess
    out = subprocess.run(["cuobjdump", "-sass", build.build()], capture_output=True, text=True).stdout
    assert "UTMALDG" in out
    assert "SM100a" in out or "sm_100a" in out
    archs = set(re.findall(r"arch = (sm_\w+)", out))
    assert archs == {"sm_100a"}, archs


def test_rdarray_semantics():
    a = rd.rdarray(np.zeros((4, 5), np.float32), no_data=-9999)
    assert a.no_data == -9999 and a.shape == (4, 5)
    b = a.copy()
    assert b.no_data == -9999 and type(b) is rd.rdarray
    with pytest.raises(Exception, match="no_data value must be specified"):
        rd.rdarray(np.zeros((2, 2)))
    c = rd.rdarray(np.ones((3, 3)), meta_obj=a, no_data=-1)
    assert c.no_data == -1
    p = rd.rd3array(np.zeros((3, 3, 9)), no_data=-2)
    assert p.dtype == np.float32


def test_argument_validation_matches_reference_behaviour():
    raw = np.zeros((8, 8), np.float32)
    dem = rd.rdarray(raw, no_data=-9999)
    with pytest.raises(Exception, match="rdarray or numpy.ndarray is required"):
        rd.FillDepressions(raw)
    with pytest.raises(Exception, match="Unknown topology"):
        rd.FillDepressions(dem, topology="D6")
    with pytest.raises(Exception, match="rdarray or numpy.ndarray is required"):
        rd.ResolveFlats(raw)
    with pytest.raises(Exception, match="Invalid FlowAccumulation method"):
        rd.FlowAccumulation(dem, method="nope")
    with pytest.raises(Exception, match="outside the B200 hot path"):
        rd.FlowAccumulation(dem, method="Rho8")
    with pytest.raises(Exception, match="requires an exponent"):
        rd.FlowAccumulation(dem, method="Holmgren")
    with pytest.raises(Exception, match="must be of type 'float64'"):
        rd.FlowAccumulation(dem, method="D8", weights=rd.rdarray(np.ones((8, 8), np.float32), no_data=-1))
    with pytest.raises(Exception, match="Invalid FlowProportions method"):
        rd.FlowProportions(dem, method=None)
    with pytest.raises(Exception, match="rd3array"):
        rd.FlowAccumFromProps(dem)
    with pytest.raises(Exception, match="float32"):
        rd.FillDepressions(rd.rdarray(np.zeros((8, 8), np.float64), no_data=-1))


@pytest.mark.skipif(_has_gpu(), reason="only meaningful on a box without a GPU")
def test_no_cpu_fallback_compute_fails_loudly():
    dem = rd.rdarray(np.arange(64, dtype=np.float32).reshape(8, 8), no_data=-9999)
    for call in (lambda: rd.FillDepressions(dem), lambda: rd.ResolveFlats(dem),
                 lambda: rd.FlowAccumulation(dem, method="D8"), lambda: rd.FlowProportions(dem, method="Dinf")):
        with pytest.raises(rd.RichdemB200Error, match="no CPU fallback|no CUDA"):
            call()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "richdem_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "liboracle" not in src, f


def test_product_never_reaches_the_kernel_emulation():
    """tests/emu (the CPU model of the kernels) is test infrastructure like the oracle: nothing shipped, benchmarked or
    smoke-tested may name it, and the loader's only mention of it is the refusal to load such a build."""
    names = ("librdb200_emu_test", "tests/emu", "cuda_emu", "build_emu")
    files = [os.path.join(ROOT, "bench.py"), os.path.join(ROOT, "__graft_entry__.py")]
    for dirpath, _, fs in os.walk(os.path.join(ROOT, "richdem_b200")):
        files += [os.path.join(dirpath, f) for f in fs if f.endswith((".py", ".cu", ".cuh", ".inc", ".h", ".hpp"))]
    for dirpath, _, fs in os.walk(os.path.join(ROOT, "include")):
        files += [os.path.join(dirpath, f) for f in fs]
    for f in files:
        src = open(f).read()
        for n in names:
            if f.endswith("_lib.py") and n == "tests/emu":
                continue  # the comment next to the loader's refusal
            assert n not in src, (f, n)
    lib_src = open(os.path.join(ROOT, "richdem_b200", "_lib.py")).read()
    assert lib_src.count("rdb200_emulated") == 1 and "no CPU fallback" in lib_src


def test_cxx_dropin_header_links_and_fails_loudly_without_gpu():
    """include/richdem_b200.hpp specialises the reference templates; the check binary (built by oracle/Makefile against
    the reference's headers into build/reference_bindings/) must route every call into librichdem_b200 -- on a machine without a GPU
    that means 9 std::runtime_errors, no CPU fallback."""
    import subprocess
    exe = os.path.join(ROOT, "build", "reference_bindings", "cxx_dropin_check")
    if not os.path.exists(exe):
        pytest.skip("build/reference_bindings/cxx_dropin_check not built (reference headers absent at build time)")
    if _has_gpu():
        pytest.skip("GPU present: covered by the gpu-marked test")
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-2000:]
    assert "calls=9 thrown=9" in out.stdout


def test_header_and_ctypes_table_agree_on_arity():
    """Every prototype in include/richdem_b200.h has as many parameters as its ctypes signature."""
    header = open(os.path.join(ROOT, "include", "richdem_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    protos = re.findall(r"RDB200_API\s+[\w\s\*]+?\b(rdb200_\w+)\s*\(([^;]*?)\)\s*;", header, flags=re.S)
    assert len(protos) >= 40
    for name, params in protos:
        params = params.strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        if name in _lib.SIGNATURES:
            assert n == len(_lib.SIGNATURES[name]), (name, n, len(_lib.SIGNATURES[name]))


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` runs on CPU only and prints one JSON line with the contract keys."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--size", "384",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "Mcells/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"]


def test_scoped_param_restores_what_the_process_had_set():
    """sharded.py's Python band protocol leashes the fill's rounds per run through a process-wide switch; the switch must be
    back to what the process had (or to the library's default) when the call is over (ADVICE r1)."""
    from richdem_b200 import _lib
    _lib.reset_params()
    try:
        with _lib.scoped_param("fill_band_rounds", 64):
            assert _lib._param_values["fill_band_rounds"] == 64
        assert "fill_band_rounds" not in _lib._param_values  # never set before: back to the default, not recorded as set
        _lib.set_param("fill_band_rounds", 7)
        with _lib.scoped_param("fill_band_rounds", 64):
            with _lib.scoped_param("fill_band_rounds", 3):
                assert _lib._param_values["fill_band_rounds"] == 3
            assert _lib._param_values["fill_band_rounds"] == 64
        assert _lib._param_values["fill_band_rounds"] == 7
        with pytest.raises(_lib.RichdemB200Error, match="unknown parameter"):
            _lib.set_param("no_such_switch", 1)
    finally:
        _lib.reset_params()
    assert _lib._param_values == {}


def test_native_cache_format_round_trips_with_the_reference(tmp_path):
    """SURVEY 8f-4: SaveNative / LoadNative speak richdem::Array2D's cache format (common/Array2D.hpp:209-281): a file
    written by the reference (tests/golden/native_cache_ref.rd, make_golden.py::native_cache) is read here, and a file
    written here is byte-identical to it, so the reference reads it back as it reads its own, metadata included."""
    import oracle
    import richdem_b200 as rd
    dem = oracle.fbm_terrain(37, 53, seed=3)
    dem[5:9, 7:20] = -9999.0
    gt = [100.0, 30.0, 0.0, 2000.0, 0.0, -20.0]
    a = os.path.join(ROOT, "tests", "golden", "native_cache_ref.rd")
    got = rd.LoadNative(a)
    assert got.dtype == np.float32 and got.shape == dem.shape and np.array_equal(np.asarray(got).view(np.uint32), dem.view(np.uint32))
    assert got.no_data == -9999.0 and list(got.geotransform) == gt and got.projection == "EPSG:26915"
    b = str(tmp_path / "from_python.rd")
    src = rd.rdarray(dem.copy(), no_data=-9999.0, geotransform=gt)
    src.projection = "EPSG:26915"
    rd.SaveNative(src, b)
    with open(a, "rb") as fa, open(b, "rb") as fb:
        assert fa.read() == fb.read(), "byte-identical files (the reference has not counted the data cells either)"
    with pytest.raises(RuntimeError, match="truncated"):
        with open(b, "rb") as fb:
            blob = fb.read()
        with open(b, "wb") as fb:
            fb.write(blob[:-100])
        rd.LoadNative(b)
