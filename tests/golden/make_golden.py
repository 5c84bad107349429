"""Regenerates the golden fixtures under tests/golden/ (run in the build container only).

Sources, all under /root/reference (never copied as source; only test DATA is re-encoded):
  * tests/depressions/testdem1.dem -> testdem1.all.out   known-answer fill (tests/tests.cpp:238-271)
  * tests/flow_accum/*.d8 -> *.out                        known-answer d8_flow_accum (tests/tests.cpp:135-146)
  * data/*.dem                                             hand-made flat-resolution / D-infinity inputs
  * docs/imgs/beauford.npz                                 the Beauford DEM (crop with NoData)
and outputs of the UNMODIFIED reference implementation (oracle/_ref, built by oracle/Makefile from
/root/reference/include) on those inputs and on seeded synthetic DEMs.
"""
import glob
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402

REF = "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))


def read_ascii_grid(path):
    """ESRI ASCII grid: 6 header lines then rows."""
    with open(path) as f:
        toks = f.read().split()
    hdr = {toks[2 * i].lower(): float(toks[2 * i + 1]) for i in range(6)}
    ncols, nrows = int(hdr["ncols"]), int(hdr["nrows"])
    vals = np.array(toks[12:12 + ncols * nrows], dtype=np.float64).reshape(nrows, ncols)
    return vals, hdr["nodata_value"]


def main():
    R = oracle.ref()

    # 1. fill known-answer
    dem, nd = read_ascii_grid(f"{REF}/tests/depressions/testdem1.dem")
    exp, _ = read_ascii_grid(f"{REF}/tests/depressions/testdem1.all.out")
    np.savez_compressed(f"{OUT}/fill_testdem1.npz", dem=dem.astype(np.float32), expected=exp.astype(np.float32),
                        nodata=np.float32(nd))

    # 2. d8_flow_accum known-answers
    names, d8s, outs, nds = [], [], [], []
    for p in sorted(glob.glob(f"{REF}/tests/flow_accum/*.d8")):
        o = p[:-3] + ".out"
        if not os.path.exists(o):
            continue
        a, nda = read_ascii_grid(p)
        b, _ = read_ascii_grid(o)
        names.append(os.path.basename(p)[:-3])
        d8s.append(a.astype(np.int32))
        outs.append(b.astype(np.int32))
        nds.append(int(nda))
    fa = {"names": np.array(names), "d8_nodata": np.array(nds, np.int32)}
    for nm, a, b in zip(names, d8s, outs):
        fa[nm + "__d8"] = a
        fa[nm + "__out"] = b
    np.savez_compressed(f"{OUT}/flow_accum_fixtures.npz", **fa)

    # 3. hand-made flats / dinf inputs with reference outputs
    flat_cases = {}
    for p in sorted(glob.glob(f"{REF}/data/*.dem")):
        a, nda = read_ascii_grid(p)
        a32 = a.astype(np.float32)
        key = os.path.basename(p)[:-4]
        flat_cases[key + "__dem"] = a32
        flat_cases[key + "__nodata"] = np.float32(nda)
        flat_cases[key + "__resolved"] = R.resolve_flats(a32, float(nda))
        m, l = R.flat_mask(a32, float(nda))
        flat_cases[key + "__mask"] = m
        flat_cases[key + "__labeled"] = (l != 0)
        flat_cases[key + "__filled"] = R.fill_depressions(a32)
        flat_cases[key + "__dirs"] = R.d8_flow_directions(a32, float(nda))
        flat_cases[key + "__fm_d8"] = R.fm_d8(a32, float(nda))
        flat_cases[key + "__fm_dinf"] = R.fm_dinf(a32, float(nda))
    np.savez_compressed(f"{OUT}/data_dems.npz", **flat_cases)

    # 4. Beauford crop (has NoData = -9999) through the whole reference pipeline
    b = np.load(f"{REF}/docs/imgs/beauford.npz")["beauford"]
    crop = np.ascontiguousarray(b[300:620, 300:700])
    nd = -9999.0
    filled = R.fill_depressions(crop, "fill_zhou")
    resolved = R.resolve_flats(filled, nd)
    np.savez_compressed(
        f"{OUT}/beauford_crop.npz", dem=crop, nodata=np.float32(nd), filled=filled, resolved=resolved,
        dirs=R.d8_flow_directions(resolved, nd), fa_d8=R.fa_d8(resolved, nd), fa_dinf=R.fa_dinf(resolved, nd),
        fm_dinf_nz=np.float32(R.fm_dinf(resolved, nd)).reshape(-1, 9)[::7],  # every 7th cell's 9 slots
    )

    # 5. seeded synthetic DEMs (inputs are regenerated at test time from the seed)
    syn = {}
    for seed, (h, w), q in [(101, (180, 260), None), (102, (200, 150), 0.5), (103, (256, 256), 2.0)]:
        dem = oracle.fbm_terrain(h, w, seed=seed, quantum=q)
        f = R.fill_depressions(dem)
        r = R.resolve_flats(f, -9999.0)
        k = f"s{seed}"
        syn[k + "__shape"] = np.array([h, w])
        syn[k + "__quantum"] = np.float64(q if q else 0)
        syn[k + "__dem"] = dem
        syn[k + "__filled"] = f
        syn[k + "__resolved"] = r
        syn[k + "__dirs"] = R.d8_flow_directions(r, -9999.0)
        syn[k + "__fa_d8"] = R.fa_d8(r, -9999.0)
        syn[k + "__fa_dinf"] = R.fa_dinf(r, -9999.0)
    np.savez_compressed(f"{OUT}/synthetic_ref.npz", **syn)
    metrics()
    flowdirs_flats()
    terrain_attributes()
    reference_digests()
    epsilon_fill()
    native_cache()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


def flowdirs_flats():
    """7. direction-grid flat resolution (SURVEY 8f-2): barnes_flat_resolution_d8(dem, dirs, alter=false) of the unmodified
    reference (flats/flat_resolution.hpp:588-607) on the filled Beauford crop and a seeded synthetic DEM."""
    R = oracle.ref()
    g = np.load(f"{OUT}/beauford_crop.npz")
    out = {}
    for name, dem in (("beauford", g["filled"]), ("s105", R.fill_depressions(oracle.fbm_terrain(160, 230, seed=105, quantum=0.5)))):
        out[name + "__dirs"] = R.d8_flow_directions_flats(dem, -9999.0)[0]
        if name != "beauford":
            out[name + "__dem"] = dem
    np.savez_compressed(f"{OUT}/flowdirs_flats_ref.npz", **out)


METRIC_CASES = [("D4", None), ("Quinn", None), ("Holmgren", 2.5), ("Holmgren", 0.7), ("Freeman", 1.1), ("Freeman", 4.0)]


def metrics():
    """6. the remaining flow metrics (SURVEY 8f-1): FM_D4 / FM_Quinn / FM_Holmgren / FM_Freeman proportions and the FA_*
    accumulations of the unmodified reference on the resolved Beauford crop (NoData) and one seeded synthetic DEM."""
    R = oracle.ref()
    g = np.load(f"{OUT}/beauford_crop.npz")
    out = {}
    syn = R.resolve_flats(R.fill_depressions(oracle.fbm_terrain(150, 210, seed=104, quantum=0.25)), -9999.0)
    for name, dem in (("beauford", g["resolved"]), ("s104", syn)):
        for m, e in METRIC_CASES:
            k = f"{name}__{m}_{e}"
            out[k + "__fm"] = R.fm_method(dem, -9999.0, m, e).reshape(-1, 9)[::11]  # every 11th cell's 9 slots
            out[k + "__fa"] = R.fa_method(dem, -9999.0, m, e)[::3, ::3]             # every 3rd row / column
    out["s104__resolved"] = syn
    np.savez_compressed(f"{OUT}/flow_metrics_ref.npz", **out)


TA_CASES = [(1.0, (1.0, 1.0)), (2.5, (30.0, 20.0))]


def terrain_attributes():
    """8. terrain attributes (SURVEY 8f-4): TA_* of the unmodified reference (methods/terrain_attributes.hpp:370-538) on the
    Beauford crop (NoData) and a seeded synthetic DEM, unit cells / zscale 1 and 30 x 20 cells / zscale 2.5."""
    R = oracle.ref()
    g = np.load(f"{OUT}/beauford_crop.npz")
    syn = oracle.fbm_terrain(140, 190, seed=106, quantum=0.5)  # quantised: exact zero gradients exist
    out = {"s106__dem": syn}
    for name, dem in (("beauford", g["dem"]), ("s106", syn)):
        for attrib in R.TA_IDS:
            for zs, cell in TA_CASES:
                out[f"{name}__{attrib}__{zs}"] = R.terrain_attribute(dem, attrib, -9999.0, zs, cell)[::3, ::3]
    np.savez_compressed(f"{OUT}/terrain_attributes_ref.npz", **out)


ND = -9999.0
PORT_CASES = [(7, (97, 133), None, False), (8, (160, 120), 0.5, True), (9, (300, 300), 4.0, False)]
D4_CASES = [(7, (97, 133), None), (8, (160, 120), 0.5), (9, (300, 300), 4.0)]
TA_LIVE_CASES = [(1.0, (1.0, 1.0), -9999.0), (0.3048, (10.0, 10.0), -1.0), (3.0, (5.0, 7.5), -9999.0)]


def reference_digests():
    """9. whole outputs of the unmodified reference on the seeded synthetic DEMs of tests/test_oracle.py and on the 8192^2
    benchmark raster of tests/test_gpu_parity.py, as oracle.digest() values (the arrays themselves are megabytes): the
    inputs are regenerated at test time from their seeds and the C port / the GPU must reproduce every digest."""
    import json
    R = oracle.ref()
    dg = oracle.digest
    out = {}
    for seed, shape, q, patch in PORT_CASES:
        dem = oracle.fbm_terrain(*shape, seed=seed, quantum=q)
        if patch:
            dem[20:50, 30:70] = ND
            dem[:9, :13] = ND
        f = R.fill_depressions(dem)
        m, l = R.flat_mask(f, ND)
        r = R.resolve_flats(f, ND)
        d = R.d8_flow_directions(r, ND)
        wts = np.random.default_rng(seed).random(shape)
        out[f"port_s{seed}"] = {
            "dem": dg(dem), **{f"fill_{v}": dg(R.fill_depressions(dem, v)) for v in (None, "fill_zhou", "fill_barnes", "fill_original")},
            "find_flats": dg(R.find_flats(f, ND)), "flat_mask": dg(m), "flat_labeled": dg(l != 0), "resolved": dg(r),
            "dirs": dg(d), "d8_flow_accum": dg(R.d8_flow_accum(d)), "fm_d8": dg(R.fm_d8(r, ND)), "fm_dinf": dg(R.fm_dinf(r, ND)),
            "fa_d8": dg(R.fa_d8(r, ND)), "fa_dinf": dg(R.fa_dinf(r, ND)), "fa_dinf_weighted": dg(R.fa_dinf(r, ND, wts))}
    dem = oracle.fbm_terrain(140, 190, seed=21, quantum=0.5)
    dem[20:40, 30:70] = ND
    wts = np.random.default_rng(3).random(dem.shape)
    out["metrics_s21"] = {"dem": dg(dem)}
    for m, e in METRIC_CASES:
        out["metrics_s21"][f"{m}_{e}"] = {"fm": dg(R.fm_method(dem, ND, m, e)), "fa": dg(R.fa_method(dem, ND, m, e)),
                                          "fa_weighted": dg(R.fa_method(dem, ND, m, e, wts))}
    for seed, shape, q in D4_CASES:
        dem = oracle.fbm_terrain(*shape, seed=seed, quantum=q)
        dem[20:40, 30:60] = ND
        out[f"fill_d4_s{seed}"] = {"dem": dg(dem), "fill_d4": dg(R.fill_depressions(dem, "fill_d4"))}
    dem = R.fill_depressions(oracle.fbm_terrain(180, 150, seed=33, quantum=1.0))
    dem[60:80, 40:70] = ND
    dirs, m, l = R.d8_flow_directions_flats(dem, ND)
    out["flowdirs_flats_s33"] = {"dem": dg(dem), "dirs": dg(dirs), "mask": dg(m), "labeled": dg(l != 0)}
    dem = oracle.fbm_terrain(150, 211, seed=23, quantum=0.5)
    dem[20:40, 30:70] = ND
    dem[0, :9] = ND
    out["terrain_s23"] = {"dem": dg(dem)}
    for attrib in R.TA_IDS:
        for zs, cell, nd_out in TA_LIVE_CASES:
            out["terrain_s23"][f"{attrib}__{zs}"] = dg(R.terrain_attribute(dem, attrib, ND, zs, cell, nd_out))
    dem = oracle.device_fbm(8192, 8192, seed=42)
    f = R.fill_depressions(dem)
    out["bench_8192"] = {"dem": dg(dem), "filled": dg(f), "fa_d8": dg(R.fa_d8(f, ND))}
    with open(f"{OUT}/reference_digests.json", "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")


def epsilon_fill():
    """10. PriorityFloodEpsilon_Barnes2014 (depressions/Barnes2014.hpp:336-420) of the unmodified reference on three seeded
    60 x 80 synthetic DEMs, whole (tests/test_oracle.py::test_epsilon_fill_depends_on_the_queue_order)."""
    import ctypes as C
    R = oracle.ref()
    f = R.lib.ref_priority_flood_epsilon_f32
    f.argtypes = [np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS"), C.c_int, C.c_int, C.c_float]
    f.restype = None
    out = {}
    for seed in (2, 5, 7):
        z = oracle.fbm_terrain(60, 80, seed=seed, quantum=0.5)
        ref = z.copy()
        f(ref, 80, 60, ND)
        out[f"s{seed}__dem"], out[f"s{seed}__epsilon_filled"] = z, ref
    np.savez_compressed(f"{OUT}/epsilon_fill_ref.npz", **out)


def native_cache():
    """11. a file in richdem::Array2D's native cache format (common/Array2D.hpp:209-281) written by the unmodified
    reference; the reference reads it back bit for bit, metadata included."""
    R = oracle.ref()
    dem = oracle.fbm_terrain(37, 53, seed=3)
    dem[5:9, 7:20] = ND
    gt = [100.0, 30.0, 0.0, 2000.0, 0.0, -20.0]
    path = f"{OUT}/native_cache_ref.rd"
    R.save_native(path, dem, ND, gt, "EPSG:26915")
    data, nd, gt2, proj = R.load_native(path)
    assert np.array_equal(data.view(np.uint32), dem.view(np.uint32)) and nd == ND and list(gt2) == gt and proj == "EPSG:26915"


if __name__ == "__main__":
    if "--metrics-only" in sys.argv:
        metrics()
    elif "--flowdirs-flats-only" in sys.argv:
        flowdirs_flats()
    elif "--terrain-attributes-only" in sys.argv:
        terrain_attributes()
    elif "--reference-digests-only" in sys.argv:
        reference_digests()
        epsilon_fill()
        native_cache()
    else:
        main()
