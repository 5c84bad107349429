"""Pins the CPU oracle (oracle/oracle.c) before anything trusts it:
  * against the reference's own known-answer fixtures (re-encoded in tests/golden/),
  * against stored outputs of the unmodified reference on real + synthetic terrain,
  * against digests of whole outputs of the unmodified reference on seeded synthetic terrain
    (tests/golden/reference_digests.json, written by tests/golden/make_golden.py from oracle/_ref).
No GPU involved."""
import json
import os

import numpy as np
import pytest

import oracle

ND = -9999.0
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
with open(os.path.join(GOLDEN, "reference_digests.json")) as _f:
    REF = json.load(_f)


def assert_digests(expected, **arrays):
    """Each array's oracle.digest() equals the stored digest of the reference's output of the same name.  Only digests
    are stored, so a failure names the outputs and what they hold; tests/golden/make_golden.py::reference_digests shows
    the reference call that produced each one, for a cell-by-cell comparison where the reference is at hand."""
    bad = []
    for k, a in arrays.items():
        got = oracle.digest(a)
        if got != expected[k]:
            a = np.asarray(a)
            what = f"{a.dtype} {a.shape}" + (f", min {a.min()}, max {a.max()}" if a.size else "")
            if a.dtype == bool:
                what += f", {np.count_nonzero(a)} set"
            elif a.dtype.kind == "f":
                what += f", {np.count_nonzero(~np.isfinite(a))} non-finite"
            bad.append(f"{k}: {what}; digest {got[:16]} instead of the reference's {expected[k][:16]}")
    assert not bad, "differs from the reference:\n  " + "\n  ".join(bad)


def test_fill_known_answer(port, golden):
    g = golden["fill_testdem1"]  # reference tests/tests.cpp:238-271
    assert np.array_equal(port.fill_depressions(g["dem"]), g["expected"])


def test_d8_flow_accum_known_answers(port, golden):
    g = golden["flow_accum_fixtures"]  # reference tests/tests.cpp:135-146
    assert len(g["names"]) == 24
    for name, nd in zip(g["names"], g["d8_nodata"]):
        got = port.d8_flow_accum(g[f"{name}__d8"], nodata=int(nd))
        assert np.array_equal(got, g[f"{name}__out"]), name


def test_data_dems_against_reference_outputs(port, golden):
    g = golden["data_dems"]
    keys = sorted({k.split("__")[0] for k in g.files})
    assert {"pit", "multi_flat", "garbrecht", "dinf_test"} <= set(keys)
    for k in keys:
        dem, nd = g[f"{k}__dem"], float(g[f"{k}__nodata"])
        assert np.array_equal(port.fill_depressions(dem), g[f"{k}__filled"]), k
        assert np.array_equal(port.resolve_flats(dem, nd), g[f"{k}__resolved"]), k
        m, l = port.flat_mask(dem, nd)
        assert np.array_equal(m, g[f"{k}__mask"]), k
        assert np.array_equal(l != 0, g[f"{k}__labeled"]), k
        assert np.array_equal(port.d8_flow_directions(dem, nd), g[f"{k}__dirs"]), k
        assert np.array_equal(port.fm_d8(dem, nd), g[f"{k}__fm_d8"]), k
        assert np.array_equal(port.fm_dinf(dem, nd), g[f"{k}__fm_dinf"]), k


def test_beauford_crop_pipeline(port, golden):
    g = golden["beauford_crop"]
    dem, nd = g["dem"], float(g["nodata"])
    assert (dem == nd).mean() > 0.05  # the crop exercises the NoData branches
    filled = port.fill_depressions(dem)
    assert np.array_equal(filled, g["filled"])
    resolved = port.resolve_flats(filled, nd)
    assert np.array_equal(resolved, g["resolved"])
    assert np.array_equal(port.d8_flow_directions(resolved, nd), g["dirs"])
    assert np.array_equal(port.fa_d8(resolved, nd), g["fa_d8"])
    assert np.array_equal(port.fa_dinf(resolved, nd), g["fa_dinf"])
    assert np.array_equal(port.fm_dinf(resolved, nd).reshape(-1, 9)[::7], g["fm_dinf_nz"])


def test_synthetic_against_reference_outputs(port, golden):
    g = golden["synthetic_ref"]
    for seed in (101, 102, 103):
        k = f"s{seed}"
        h, w = (int(v) for v in g[f"{k}__shape"])
        q = float(g[f"{k}__quantum"]) or None
        dem = oracle.fbm_terrain(h, w, seed=seed, quantum=q)
        assert np.array_equal(dem, g[f"{k}__dem"]), "terrain generator drifted"
        f = port.fill_depressions(dem)
        assert np.array_equal(f, g[f"{k}__filled"])
        r = port.resolve_flats(f, ND)
        assert np.array_equal(r, g[f"{k}__resolved"])
        assert np.array_equal(port.d8_flow_directions(r, ND), g[f"{k}__dirs"])
        assert np.array_equal(port.fa_d8(r, ND), g[f"{k}__fa_d8"])
        assert np.array_equal(port.fa_dinf(r, ND), g[f"{k}__fa_dinf"])


@pytest.mark.parametrize("seed,shape,q,nodata_patch", [(7, (97, 133), None, False), (8, (160, 120), 0.5, True),
                                                       (9, (300, 300), 4.0, False)])
def test_port_matches_compiled_reference_live(port, seed, shape, q, nodata_patch):
    """The whole pipeline, bit for bit, against the reference's outputs (tests/golden/make_golden.py::reference_digests;
    the fill against all four of the reference's Priority-Flood variants)."""
    D = REF[f"port_s{seed}"]
    dem = oracle.fbm_terrain(*shape, seed=seed, quantum=q)
    if nodata_patch:
        dem[20:50, 30:70] = ND
        dem[:9, :13] = ND
    assert_digests(D, dem=dem)
    f = port.fill_depressions(dem)
    assert_digests(D, **{f"fill_{v}": f for v in (None, "fill_zhou", "fill_barnes", "fill_original")})
    m, l = port.flat_mask(f, ND)
    assert_digests(D, find_flats=port.find_flats(f, ND), flat_mask=m, flat_labeled=l != 0)
    r = port.resolve_flats(f, ND)
    d = port.d8_flow_directions(r, ND)
    wts = np.random.default_rng(seed).random(shape)
    assert_digests(D, resolved=r, dirs=d, d8_flow_accum=port.d8_flow_accum(d), fm_d8=port.fm_d8(r, ND),
                   fm_dinf=port.fm_dinf(r, ND), fa_d8=port.fa_d8(r, ND), fa_dinf=port.fa_dinf(r, ND),
                   fa_dinf_weighted=port.fa_dinf(r, ND, wts))


def test_fill_is_min_over_paths_of_max(port):
    """Independent definition check on a tiny raster: brute-force Jacobi iteration of
    W = max(Z, min_nbrs W) from +inf (SURVEY 8a'-1)."""
    dem = oracle.fbm_terrain(23, 31, seed=5, quantum=5.0)
    h, w = dem.shape
    W = np.full((h + 2, w + 2), np.inf, np.float32)
    Z = np.full((h + 2, w + 2), np.inf, np.float32)
    Z[1:-1, 1:-1] = dem
    border = np.zeros((h + 2, w + 2), bool)
    border[1, 1:-1] = border[-2, 1:-1] = border[1:-1, 1] = border[1:-1, -2] = True
    W[border] = Z[border]
    for _ in range(10 * (h + w)):
        m = np.full_like(W, np.inf)
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                if dy or dx:
                    m[1:-1, 1:-1] = np.minimum(m[1:-1, 1:-1], W[1 + dy:h + 1 + dy, 1 + dx:w + 1 + dx])
        new = np.minimum(W, np.maximum(Z, m))
        new[border] = Z[border]
        if np.array_equal(new, W):
            break
        W = new
    assert np.array_equal(W[1:-1, 1:-1], port.fill_depressions(dem))


METRIC_CASES = [("D4", None), ("Quinn", None), ("Holmgren", 2.5), ("Holmgren", 0.7), ("Freeman", 1.1), ("Freeman", 4.0)]


def test_remaining_flow_metrics_against_reference_outputs(port, golden):
    """SURVEY 8f-1: FM_D4 / FM_Quinn / FM_Holmgren / FM_Freeman and their FA_* against stored outputs of the
    unmodified reference (tests/golden/make_golden.py::metrics)."""
    g = golden["flow_metrics_ref"]
    dems = {"beauford": golden["beauford_crop"]["resolved"], "s104": g["s104__resolved"]}
    for name, dem in dems.items():
        for m, e in METRIC_CASES:
            k = f"{name}__{m}_{e}"
            assert np.array_equal(port.fm_method(dem, ND, m, e).reshape(-1, 9)[::11], g[k + "__fm"]), k
            assert np.array_equal(port.fa_method(dem, ND, m, e)[::3, ::3], g[k + "__fa"]), k


@pytest.mark.parametrize("method,exponent", METRIC_CASES)
def test_remaining_flow_metrics_port_matches_compiled_reference_live(port, method, exponent):
    dem = oracle.fbm_terrain(140, 190, seed=21, quantum=0.5)
    dem[20:40, 30:70] = ND
    assert_digests(REF["metrics_s21"], dem=dem)
    wts = np.random.default_rng(3).random(dem.shape)
    assert_digests(REF["metrics_s21"][f"{method}_{exponent}"], fm=port.fm_method(dem, ND, method, exponent),
                   fa=port.fa_method(dem, ND, method, exponent), fa_weighted=port.fa_method(dem, ND, method, exponent, wts))


@pytest.mark.parametrize("seed,shape,q", [(7, (97, 133), None), (8, (160, 120), 0.5), (9, (300, 300), 4.0)])
def test_d4_fill_port_matches_compiled_reference_live(port, seed, shape, q):
    """FillDepressions<Topology::D4> (depressions/depressions.hpp:16-17)."""
    dem = oracle.fbm_terrain(*shape, seed=seed, quantum=q)
    dem[20:40, 30:60] = ND
    d4 = port.fill_depressions(dem, "fill_d4")
    assert_digests(REF[f"fill_d4_s{seed}"], dem=dem, fill_d4=d4)
    assert (d4 >= port.fill_depressions(dem)).all() and (d4 > port.fill_depressions(dem)).any(), "D4 fills at least as high as D8"


def test_direction_grid_flat_resolution_against_reference_outputs(port, golden):
    """SURVEY 8f-2: barnes_flat_resolution_d8 (flats/flat_resolution.hpp:588-607)."""
    g = golden["flowdirs_flats_ref"]
    for name, dem in (("beauford", golden["beauford_crop"]["filled"]), ("s105", g["s105__dem"])):
        dirs, m, l = port.d8_flow_directions_flats(dem, ND)
        assert np.array_equal(dirs, g[name + "__dirs"]), name
        inner = np.zeros(dirs.shape, bool)
        inner[1:-1, 1:-1] = True
        assert not ((dirs == 0) & inner & (l != 0)).any(), "every cell of a drainable flat received a direction"


def test_direction_grid_flat_resolution_port_matches_compiled_reference_live(port):
    dem = port.fill_depressions(oracle.fbm_terrain(180, 150, seed=33, quantum=1.0))
    dem[60:80, 40:70] = ND
    dirs, m, l = port.d8_flow_directions_flats(dem, ND)
    assert_digests(REF["flowdirs_flats_s33"], dem=dem, dirs=dirs, mask=m, labeled=l != 0)


# ---- SURVEY 8f-4: terrain attributes --------------------------------------------------------------------------------------
TA_CASES = [(1.0, (1.0, 1.0)), (2.5, (30.0, 20.0))]


def test_terrain_attributes_against_reference_outputs(port, golden):
    """TA_* (methods/terrain_attributes.hpp:370-538) against stored outputs of the unmodified reference
    (tests/golden/make_golden.py::terrain_attributes): the restatement is bit-identical, libm calls included."""
    g = golden["terrain_attributes_ref"]
    for name, dem in (("beauford", golden["beauford_crop"]["dem"]), ("s106", g["s106__dem"])):
        for attrib in port.TA_IDS:
            for zs, cell in TA_CASES:
                got = port.terrain_attribute(dem, attrib, ND, zs, cell)[::3, ::3]
                assert np.array_equal(got.view(np.uint32), g[f"{name}__{attrib}__{zs}"].view(np.uint32)), (name, attrib, zs)


def test_terrain_attributes_port_matches_compiled_reference_live(port):
    dem = oracle.fbm_terrain(150, 211, seed=23, quantum=0.5)
    dem[20:40, 30:70] = ND
    dem[0, :9] = ND
    assert_digests(REF["terrain_s23"], dem=dem)
    for attrib in port.TA_IDS:
        for zs, cell, nd_out in ((1.0, (1.0, 1.0), -9999.0), (0.3048, (10.0, 10.0), -1.0), (3.0, (5.0, 7.5), -9999.0)):
            a = port.terrain_attribute(dem, attrib, ND, zs, cell, nd_out)
            assert_digests(REF["terrain_s23"], **{f"{attrib}__{zs}": a})
            assert np.all(a[dem == ND] == nd_out)


# ---- SURVEY 8f-3: why the epsilon fill is not on the B200 path -----------------------------------------------------------
def test_epsilon_fill_depends_on_the_queue_order(golden):
    """PriorityFloodEpsilon_Barnes2014 (depressions/Barnes2014.hpp:336-420) drains its FIFO "pit" queue before it looks at the
    priority queue again (:377-392), so a pit cell can be closed from a neighbour that is not its cheapest one: the result is
    NOT the order-free fixed point W = max(Z, min_n nextafter(W_n)) a parallel relaxation converges to -- it lies up to a few
    float ulps above it in a few cells.  A bit-exact GPU version would have to replay the serial queue order; the row stays
    on the reference's CPU template (DESIGN.md section 0, f3).  The reference's results are stored whole
    (tests/golden/make_golden.py::epsilon_fill)."""
    import heapq
    g = golden["epsilon_fill_ref"]

    def fixed_point(z):  # Dijkstra on the cost max(Z(c), nextafter(cost of the predecessor))
        h, w = z.shape
        W = np.full((h, w), np.inf, np.float32)
        done = np.zeros((h, w), bool)
        pq = []
        for y in range(h):
            for x in range(w):
                if y in (0, h - 1) or x in (0, w - 1):
                    W[y, x] = z[y, x]
                    heapq.heappush(pq, (float(z[y, x]), y, x))
        while pq:
            v, y, x = heapq.heappop(pq)
            if done[y, x]:
                continue
            done[y, x] = True
            up = np.nextafter(np.float32(v), np.float32(np.inf))
            for yy in range(max(0, y - 1), min(h, y + 2)):
                for xx in range(max(0, x - 1), min(w, x + 2)):
                    if not done[yy, xx]:
                        c = max(z[yy, xx], up)
                        if c < W[yy, xx]:
                            W[yy, xx] = c
                            heapq.heappush(pq, (float(c), yy, xx))
        return W

    above, cells = 0, 0
    for seed in (2, 5, 7):
        z = oracle.fbm_terrain(60, 80, seed=seed, quantum=0.5)
        assert np.array_equal(z, g[f"s{seed}__dem"]), "terrain generator drifted"
        ref = g[f"s{seed}__epsilon_filled"]
        fp = fixed_point(z)
        d = ref.view(np.int32).astype(np.int64) - fp.view(np.int32).astype(np.int64)
        below = np.argwhere(d < 0)
        assert not len(below), f"seed {seed}: the serial result is never below the order-free fixed point ({len(below)} cells, first {below[0]})"
        assert d.max() <= 16, f"seed {seed}: {d.max()} ulps above the fixed point at {np.unravel_index(d.argmax(), d.shape)}"
        above += int((d > 0).sum())
        cells += z.size
        assert np.array_equal(ref >= z, np.ones_like(z, bool))
    assert 0 < above < cells // 100, (above, cells)
