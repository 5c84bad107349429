"""TEST INFRASTRUCTURE ONLY -- CPU oracles for the fill -> flats -> flow-accumulation path.

Two interchangeable back ends with the same Python surface:

* ``port``  -- ``oracle/liboracle.so``: the plain-C restatement in ``oracle/oracle.c``
  (always buildable; this is what travels to the GPU box).
* ``ref``   -- ``oracle/_ref/libref_richdem.so``: the UNMODIFIED reference headers from
  ``/root/reference/include`` compiled by ``oracle/Makefile`` (``ref_shim.cpp``).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  ``richdem_b200`` never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_PORT_PATH = os.path.join(_HERE, "liboracle.so")
_REF_PATH = os.path.join(_HERE, "_ref", "libref_richdem.so")

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_i8p = np.ctypeslib.ndpointer(np.int8, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")


def build(force: bool = False) -> None:
    """Compile the C port (and the reference shim when /root/reference exists)."""
    if force or not os.path.exists(_PORT_PATH) or (
        os.path.getmtime(_PORT_PATH) < os.path.getmtime(os.path.join(_HERE, "oracle.c"))
    ):
        subprocess.check_call(["make", "-C", _HERE, "liboracle.so"], stdout=subprocess.DEVNULL)
    if os.path.isdir("/root/reference/include/richdem") and (
        force or not os.path.exists(_REF_PATH)
        or os.path.getmtime(_REF_PATH) < os.path.getmtime(os.path.join(_HERE, "ref_shim.cpp"))
    ):
        subprocess.check_call(["make", "-C", _HERE, "ref"], stdout=subprocess.DEVNULL,
                              stderr=subprocess.DEVNULL)


def build_bindings() -> None:
    """Compile the reference's C++ drop-in check and its Python module over librichdem_b200.so into
    build/reference_bindings/ (oracle/Makefile `bindings`; nothing happens where the reference's sources are absent).
    Compiler errors reach stderr."""
    import sys
    subprocess.check_call(["make", "-C", _HERE, "bindings", f"PYTHON={sys.executable}"], stdout=subprocess.DEVNULL)


def have_ref() -> bool:
    return os.path.exists(_REF_PATH)


class _Backend:
    """numpy front end over one of the two shared libraries."""

    def __init__(self, path: str, names: dict):
        self.lib = C.CDLL(path)
        self.kind = names["kind"]
        n = names
        self._fill = self._sig(n["fill"], [_f32p, C.c_int, C.c_int])
        self._find_flats = self._sig(n["find_flats"], [_f32p, C.c_int, C.c_int, C.c_float, _i8p])
        self._flat_mask = self._sig(n["flat_mask"], [_f32p, C.c_int, C.c_int, C.c_float, _i32p, _i32p])
        self._resolve = self._sig(n["resolve"], [_f32p, C.c_int, C.c_int, C.c_float])
        self._dirs = self._sig(n["dirs"], [_f32p, C.c_int, C.c_int, C.c_float, _u8p])
        self._d8acc_u8 = self._sig(n["d8acc_u8"], [_u8p, C.c_int, C.c_int, _i32p])
        self._d8acc_i32 = self._sig(n["d8acc_i32"], [_i32p, C.c_int, C.c_int, C.c_int32, _i32p])
        self._fm_d8 = self._sig(n["fm_d8"], [_f32p, C.c_int, C.c_int, C.c_float, _f32p])
        self._fm_dinf = self._sig(n["fm_dinf"], [_f32p, C.c_int, C.c_int, C.c_float, _f32p])
        self._facc = self._sig(n["facc"], [_f32p, C.c_int, C.c_int, _f64p])
        self._fa_d8 = self._sig(n["fa_d8"], [_f32p, C.c_int, C.c_int, C.c_float, _f64p])
        self._fa_dinf = self._sig(n["fa_dinf"], [_f32p, C.c_int, C.c_int, C.c_float, _f64p])
        self._fm_method = self._sig(n["fm_method"], [C.c_int, _f32p, C.c_int, C.c_int, C.c_float, C.c_double, _f32p])
        self._fa_method = self._sig(n["fa_method"], [C.c_int, _f32p, C.c_int, C.c_int, C.c_float, C.c_double, _f64p])
        self._ta = self._sig(n["terrain_attribute"], [C.c_int, _f32p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float,
                                                      C.c_double, C.c_double, _f32p])
        self._extra = {}
        for k in ("fill_zhou", "fill_barnes", "fill_original", "fill_d4"):
            if k in n:
                self._extra[k] = self._sig(n[k], [_f32p, C.c_int, C.c_int])

    def _sig(self, name, argtypes):
        f = getattr(self.lib, name)
        f.argtypes = argtypes
        f.restype = None
        return f

    @staticmethod
    def _dem(dem):
        a = np.ascontiguousarray(dem, dtype=np.float32)
        assert a.ndim == 2
        return a

    # -- a1/a2
    def fill_depressions(self, dem, variant: str | None = None):
        out = self._dem(dem).copy()
        h, w = out.shape
        f = self._fill if variant is None else self._extra[variant]
        f(out, w, h)
        return out

    # -- a3
    def find_flats(self, dem, nodata):
        d = self._dem(dem)
        h, w = d.shape
        out = np.empty((h, w), np.int8)
        self._find_flats(d, w, h, nodata, out)
        return out

    # -- a4..a7
    def flat_mask(self, dem, nodata):
        d = self._dem(dem)
        h, w = d.shape
        mask = np.zeros((h, w), np.int32)
        labels = np.zeros((h, w), np.int32)
        self._flat_mask(d, w, h, nodata, mask, labels)
        return mask, labels

    # -- a8
    def resolve_flats(self, dem, nodata):
        out = self._dem(dem).copy()
        h, w = out.shape
        self._resolve(out, w, h, nodata)
        return out

    # -- a12
    def d8_flow_directions(self, dem, nodata):
        d = self._dem(dem)
        h, w = d.shape
        out = np.empty((h, w), np.uint8)
        self._dirs(d, w, h, nodata, out)
        return out

    # -- a13
    def d8_flow_accum(self, dirs, nodata=None):
        dirs = np.ascontiguousarray(dirs)
        h, w = dirs.shape
        out = np.empty((h, w), np.int32)
        if dirs.dtype == np.uint8:
            self._d8acc_u8(dirs, w, h, out)
        else:
            self._d8acc_i32(np.ascontiguousarray(dirs, np.int32), w, h,
                            -1 if nodata is None else int(nodata), out)
        return out

    # -- a9 / a10
    def fm_d8(self, dem, nodata):
        d = self._dem(dem)
        h, w = d.shape
        out = np.empty((h, w, 9), np.float32)
        self._fm_d8(d, w, h, nodata, out.reshape(-1))
        return out

    def fm_dinf(self, dem, nodata):
        d = self._dem(dem)
        h, w = d.shape
        out = np.empty((h, w, 9), np.float32)
        self._fm_dinf(d, w, h, nodata, out.reshape(-1))
        return out

    # -- f1: the remaining flow metrics.  method: "D4", "Quinn", "Holmgren", "Freeman" (also "D8", "Dinf")
    METHOD_IDS = {"D8": 0, "Dinf": 1, "D4": 2, "Quinn": 3, "Holmgren": 3, "Freeman": 4}

    def fm_method(self, dem, nodata, method, exponent=None):
        d = self._dem(dem)
        h, w = d.shape
        out = np.empty((h, w, 9), np.float32)
        x = 1.0 if method == "Quinn" else float(exponent or 0.0)
        self._fm_method(self.METHOD_IDS[method], d, w, h, nodata, x, out.reshape(-1))
        return out

    def fa_method(self, dem, nodata, method, exponent=None, weights=None):
        d = self._dem(dem)
        h, w = d.shape
        acc = np.ones((h, w), np.float64) if weights is None else np.array(weights, np.float64, order="C")
        x = 1.0 if method == "Quinn" else float(exponent or 0.0)
        self._fa_method(self.METHOD_IDS[method], d, w, h, nodata, x, acc)
        return acc

    # -- f4: terrain attributes (methods/terrain_attributes.hpp:370-538)
    TA_IDS = {"slope_riserun": 0, "slope_percentage": 1, "slope_degrees": 2, "slope_radians": 3, "aspect": 4,
              "curvature": 5, "planform_curvature": 6, "profile_curvature": 7}

    def terrain_attribute(self, dem, attrib, nodata=-9999.0, zscale=1.0, cell=(1.0, 1.0), nodata_out=-9999.0):
        d = self._dem(dem)
        h, w = d.shape
        out = np.empty((h, w), np.float32)
        self._ta(self.TA_IDS[attrib], d, w, h, nodata, nodata_out, zscale, float(cell[0]), float(cell[1]), out)
        return out

    # -- f4: the native cache format, written / read by the reference itself (common/Array2D.hpp:209-281)
    def save_native(self, path, dem, nodata, geotransform, projection=""):
        assert self.kind == "reference"
        d = self._dem(dem)
        h, w = d.shape
        f = self.lib.ref_save_native_f32
        f.argtypes = [C.c_char_p, _f32p, C.c_int, C.c_int, C.c_float, np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS"), C.c_char_p]
        f.restype = None
        f(path.encode(), d, w, h, nodata, np.ascontiguousarray(geotransform, np.float64), projection.encode())

    def load_native(self, path):
        assert self.kind == "reference"
        f = self.lib.ref_load_native_f32
        f.argtypes = [C.c_char_p, C.c_void_p, np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS"), C.POINTER(C.c_float),
                      np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS"), C.c_char_p, C.c_int]
        f.restype = C.c_int
        dims = np.zeros(2, np.int32)
        nd = C.c_float()
        gt = np.zeros(6, np.float64)
        proj = C.create_string_buffer(4096)
        f(path.encode(), None, dims, C.byref(nd), gt, proj, 4096)
        data = np.empty((int(dims[1]), int(dims[0])), np.float32)
        f(path.encode(), data.ctypes.data_as(C.c_void_p), dims, C.byref(nd), gt, proj, 4096)
        return data, float(nd.value), gt, proj.value.decode()

    # -- f2: direction-grid flat resolution (reference backend only: flats/flat_resolution.hpp:588-607)
    def d8_flow_directions_flats(self, dem, nodata):
        """(directions, mask, labels) of barnes_flat_resolution_d8(dem, dirs, alter=false)."""
        d = self._dem(dem)
        h, w = d.shape
        if self.kind == "reference":
            f = self.lib.ref_barnes_flat_resolution_d8_f32
            f.argtypes = [_f32p, C.c_int, C.c_int, C.c_float, _u8p, _i32p, _i32p]
            f.restype = None
            dirs = np.empty((h, w), np.uint8)
            m = np.empty((h, w), np.int32)
            l = np.empty((h, w), np.int32)
            f(d, w, h, nodata, dirs, m, l)
            return dirs, m, l
        # the C port: d8_flow_directions, GetFlatMask's mask / labels (identical to resolve_flats_barnes' wherever the
        # NoData value lies below the data, as -9999 does: pinned by tests/test_oracle.py against the reference and
        # the golden fixtures) and the masked direction stencil (flat_resolution.hpp:37-63, 97-116)
        dirs = self.d8_flow_directions(d, nodata)
        m, l = self.flat_mask(d, nodata)
        out = dirs.copy()
        d8x = [0, -1, -1, 0, 1, 1, 1, 0, -1]
        d8y = [0, 0, -1, -1, -1, 0, 1, 1, 1]
        ys, xs = np.nonzero(dirs[1:-1, 1:-1] == 0)
        for y, x in zip(ys + 1, xs + 1):
            minimum, flowdir = m[y, x], 0
            for n in range(1, 9):
                ny, nx = y + d8y[n], x + d8x[n]
                if l[ny, nx] != l[y, x]:
                    continue
                if m[ny, nx] < minimum or (m[ny, nx] == minimum and flowdir > 0 and flowdir % 2 == 0 and n % 2 == 1):
                    minimum, flowdir = m[ny, nx], n
            out[y, x] = flowdir
        return out, m, l

    # -- a11
    def flow_accumulation(self, props, weights=None):
        p = np.ascontiguousarray(props, np.float32)
        h, w, nine = p.shape
        assert nine == 9
        acc = np.ones((h, w), np.float64) if weights is None else np.array(weights, np.float64, order="C")
        self._facc(p.reshape(-1), w, h, acc)
        return acc

    def fa_d8(self, dem, nodata, weights=None):
        d = self._dem(dem)
        h, w = d.shape
        acc = np.ones((h, w), np.float64) if weights is None else np.array(weights, np.float64, order="C")
        self._fa_d8(d, w, h, nodata, acc)
        return acc

    def fa_dinf(self, dem, nodata, weights=None):
        d = self._dem(dem)
        h, w = d.shape
        acc = np.ones((h, w), np.float64) if weights is None else np.array(weights, np.float64, order="C")
        self._fa_dinf(d, w, h, nodata, acc)
        return acc


_PORT_NAMES = dict(
    kind="port",
    fill="orc_fill_depressions_d8_f32", find_flats="orc_find_flats_f32",
    flat_mask="orc_get_flat_mask_f32", resolve="orc_resolve_flats_epsilon_f32",
    dirs="orc_d8_flow_directions_f32", d8acc_u8="orc_d8_flow_accum_u8_i32",
    d8acc_i32="orc_d8_flow_accum_i32", fm_d8="orc_fm_d8_f32", fm_dinf="orc_fm_tarboton_f32",
    facc="orc_flow_accumulation_props_f64", fa_d8="orc_fa_d8_f32_f64",
    fa_dinf="orc_fa_tarboton_f32_f64", fm_method="orc_fm_method_f32", fa_method="orc_fa_method_f32_f64",
    terrain_attribute="orc_terrain_attribute_f32",
    fill_d4="orc_fill_depressions_d4_f32",
)
_REF_NAMES = dict(
    kind="reference",
    fill="ref_fill_depressions_d8_f32", find_flats="ref_find_flats_f32",
    flat_mask="ref_get_flat_mask_f32", resolve="ref_resolve_flats_epsilon_f32",
    dirs="ref_d8_flow_directions_f32", d8acc_u8="ref_d8_flow_accum_u8_i32",
    d8acc_i32="ref_d8_flow_accum_i32_i32", fm_d8="ref_fm_d8_f32", fm_dinf="ref_fm_tarboton_f32",
    facc="ref_flow_accumulation_props_f64", fa_d8="ref_fa_d8_f32_f64",
    fa_dinf="ref_fa_tarboton_f32_f64", fm_method="ref_fm_method_f32", fa_method="ref_fa_method_f32_f64",
    terrain_attribute="ref_terrain_attribute_f32",
    fill_zhou="ref_priority_flood_zhou2016_f32", fill_barnes="ref_priority_flood_barnes2014_f32",
    fill_original="ref_priority_flood_original_f32", fill_d4="ref_fill_depressions_d4_f32",
)

_port = None
_ref = None


def port() -> _Backend:
    """The C restatement (oracle.c)."""
    global _port
    if _port is None:
        build()
        _port = _Backend(_PORT_PATH, _PORT_NAMES)
    return _port


def ref() -> _Backend:
    """The unmodified reference, compiled (raises if oracle/_ref was never built)."""
    global _ref
    if _ref is None:
        if not have_ref():
            build()
        if not have_ref():
            raise RuntimeError("oracle/_ref/libref_richdem.so absent (reference tree not available)")
        _ref = _Backend(_REF_PATH, _REF_NAMES)
    return _ref


def best() -> _Backend:
    """Reference when it was built here, else the port."""
    return ref() if have_ref() else port()


def digest(a) -> str:
    """SHA-256 of an array's dtype, shape and C-order bytes: how tests/golden/reference_digests.json pins whole outputs
    of the reference that would be too large to store."""
    import hashlib
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str} {a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def device_fbm(h: int, w: int, seed: int = 42, octaves: int = 12, quantum: float = 0.0, y0: int = 0) -> np.ndarray:
    """The benchmark raster: bit-identical CPU restatement (oracle.c: orc_generate_fbm_f32) of the device generator
    rdb200_dev_generate_fbm_f32 (rows y0 .. y0+h of the raster), multi-threaded."""
    build()
    lib = C.CDLL(_PORT_PATH)
    f = lib.orc_generate_fbm_f32
    f.argtypes = [_f32p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_float]
    f.restype = None
    out = np.empty((h, w), np.float32)
    f(out, w, h, y0, seed, octaves, quantum)
    return out


# ---------------------------------------------------------------------------------------
# seeded synthetic terrain for tests (numpy; the bench uses the device generator instead)
def fbm_terrain(h: int, w: int, seed: int = 42, octaves: int | None = None, hurst: float = 0.75,
                amplitude: float = 1000.0, quantum: float | None = None) -> np.ndarray:
    """Value-noise fractional-Brownian terrain, float32, no NaN / NoData."""
    rng = np.random.default_rng(seed)
    size = max(h, w)
    if octaves is None:
        octaves = max(1, int(np.log2(size)) - 1)
    out = np.zeros((h, w), np.float64)
    yy = np.arange(h, dtype=np.float64)[:, None]
    xx = np.arange(w, dtype=np.float64)[None, :]
    cell = float(2 ** int(np.ceil(np.log2(size)) - 1))
    amp = 1.0
    for _ in range(octaves):
        gh = int(h / cell) + 3
        gw = int(w / cell) + 3
        g = rng.random((gh, gw))
        fy = yy / cell
        fx = xx / cell
        iy = np.floor(fy).astype(np.int64)
        ix = np.floor(fx).astype(np.int64)
        ty = fy - iy
        tx = fx - ix
        ty = ty * ty * ty * (ty * (ty * 6 - 15) + 10)
        tx = tx * tx * tx * (tx * (tx * 6 - 15) + 10)
        v00 = g[iy, ix]
        v01 = g[iy, ix + 1]
        v10 = g[iy + 1, ix]
        v11 = g[iy + 1, ix + 1]
        out += amp * ((v00 * (1 - tx) + v01 * tx) * (1 - ty) + (v10 * (1 - tx) + v11 * tx) * ty)
        amp *= 2.0 ** (-hurst)
        cell /= 2.0
        if cell < 1.0:
            break
    out -= out.min()
    out *= amplitude / max(out.max(), 1e-30)
    if quantum:
        out = np.round(out / quantum) * quantum
    return out.astype(np.float32)
