"""GPU parity tests (run on the B200 box with -m gpu).  Every call goes through the C ABI of
librichdem_b200.so (via the Python mirror of the reference API) and is compared with the CPU
checker on the same inputs: bit-exact for filled elevations, flat masks, resolved elevations,
direction grids, FM_D8 proportions and unit-weight D8 accumulation; <= 1 float ulp for D-infinity
proportions; 1e-9 relative (north_star allows 1e-5) for weighted / D-infinity accumulation."""
import json
import os

import numpy as np
import pytest

import oracle
import richdem_b200 as rd
from richdem_b200 import _lib

pytestmark = pytest.mark.gpu
ND = -9999.0
ACC_RTOL = 1e-9  # north_star tolerance is 1e-5 relative; only atomic-add ordering differs
# unit-weight D-infinity may carry its sums as 56-bit fixed point with 24 fractional bits (csrc/accum.cu,
# accum_walk_dinf_lanes_kernel; chosen when many cells have no receiver, always with accum_dinf_packed=1): relative error
# < 2^-23 ~ 1.2e-7 by construction; north_star allows 1e-5.  accum_dinf_packed=0 (double atomics) is held to ACC_RTOL.
DINF_UNIT_RTOL = 5e-7


def R(a, nd=ND):
    return rd.rdarray(np.ascontiguousarray(a), no_data=nd)


def ulp_diff(a, b):
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64))


def check_pipeline(dem, nd, O, accum_weights=None, dinf_rtol=None):
    filled = np.asarray(rd.FillDepressions(R(dem, nd)))
    f_ref = O.fill_depressions(dem)
    assert np.array_equal(filled, f_ref), f"fill: {(filled != f_ref).sum()} cells differ"
    m, l = rd.FlatMask(R(f_ref, nd))
    m_ref, l_ref = O.flat_mask(f_ref, nd)
    assert np.array_equal(l != 0, l_ref != 0), "flat labels (membership) differ"
    assert np.array_equal(m, m_ref), f"flat mask: {(m != m_ref).sum()} cells differ"
    # same partition: label pairs must be in bijection
    pairs = np.unique(np.stack([l[l != 0], l_ref[l_ref != 0]]), axis=1)
    assert len(np.unique(pairs[0])) == pairs.shape[1] == len(np.unique(pairs[1]))
    res = np.asarray(rd.ResolveFlats(R(f_ref, nd)))
    r_ref = O.resolve_flats(f_ref, nd)
    assert np.array_equal(res.view(np.uint32), r_ref.view(np.uint32)), "resolve_flats bits differ"
    assert np.array_equal(np.asarray(rd.FlowDirectionsD8(R(r_ref, nd))), O.d8_flow_directions(r_ref, nd))
    dirs = O.d8_flow_directions(r_ref, nd)
    assert np.array_equal(np.asarray(rd.D8FlowAccum(dirs)), O.d8_flow_accum(dirs))
    assert np.array_equal(np.asarray(rd.FlowProportions(R(r_ref, nd), "D8")), O.fm_d8(r_ref, nd))
    pg, pr = np.asarray(rd.FlowProportions(R(r_ref, nd), "Dinf")), O.fm_dinf(r_ref, nd)
    assert np.array_equal(pg > 0, pr > 0), "D-infinity facet choice differs"
    assert ulp_diff(pg, pr).max() <= 1
    a = rd.FlowAccumulation(R(r_ref, nd), "D8")
    assert a.no_data == -1 and a.dtype == np.float64
    assert np.array_equal(np.asarray(a), O.fa_d8(r_ref, nd)), "unit-weight D8 accumulation must be exact"
    np.testing.assert_allclose(np.asarray(rd.FlowAccumulation(R(r_ref, nd), "Dinf")), O.fa_dinf(r_ref, nd),
                               rtol=dinf_rtol or DINF_UNIT_RTOL, atol=0)
    if accum_weights is not None:
        w = R(accum_weights, -1)
        np.testing.assert_allclose(np.asarray(rd.FlowAccumulation(R(r_ref, nd), "D8", weights=w)),
                                   O.fa_d8(r_ref, nd, accum_weights), rtol=ACC_RTOL, atol=0)
        np.testing.assert_allclose(np.asarray(rd.FlowAccumulation(R(r_ref, nd), "Tarboton", weights=w)),
                                   O.fa_dinf(r_ref, nd, accum_weights), rtol=ACC_RTOL, atol=0)
    np.testing.assert_allclose(np.asarray(rd.FlowAccumFromProps(rd.rd3array(pr, no_data=-2))),
                               O.flow_accumulation(pr), rtol=ACC_RTOL, atol=0)
    pd8 = O.fm_d8(r_ref, nd)
    assert np.array_equal(np.asarray(rd.FlowAccumFromProps(rd.rd3array(pd8, no_data=-2))), O.flow_accumulation(pd8))


# ---- golden fixtures -------------------------------------------------------------------------
def test_fill_known_answer(golden):
    g = golden["fill_testdem1"]
    assert np.array_equal(np.asarray(rd.FillDepressions(R(g["dem"], float(g["nodata"])))), g["expected"])


def test_d8_flow_accum_known_answers(golden):
    g = golden["flow_accum_fixtures"]
    for name, nd in zip(g["names"], g["d8_nodata"]):
        d = g[f"{name}__d8"]
        u8 = np.where(d == nd, 255, d).astype(np.uint8)
        assert np.array_equal(np.asarray(rd.D8FlowAccum(u8)), g[f"{name}__out"]), name


def test_data_dems(golden):
    g = golden["data_dems"]
    for k in sorted({k.split("__")[0] for k in g.files}):
        dem, nd = g[f"{k}__dem"], float(g[f"{k}__nodata"])
        assert np.array_equal(np.asarray(rd.FillDepressions(R(dem, nd))), g[f"{k}__filled"]), k
        assert np.array_equal(np.asarray(rd.ResolveFlats(R(dem, nd))), g[f"{k}__resolved"]), k
        m, l = rd.FlatMask(R(dem, nd))
        assert np.array_equal(m, g[f"{k}__mask"]) and np.array_equal(l != 0, g[f"{k}__labeled"]), k
        assert np.array_equal(np.asarray(rd.FlowDirectionsD8(R(dem, nd))), g[f"{k}__dirs"]), k
        assert np.array_equal(np.asarray(rd.FlowProportions(R(dem, nd), "D8")), g[f"{k}__fm_d8"]), k
        assert ulp_diff(np.asarray(rd.FlowProportions(R(dem, nd), "Dinf")), g[f"{k}__fm_dinf"]).max() <= 1, k


def test_beauford_crop_golden(golden):
    g = golden["beauford_crop"]
    dem, nd = g["dem"], float(g["nodata"])
    filled = rd.FillDepressions(R(dem, nd))
    assert np.array_equal(np.asarray(filled), g["filled"])
    resolved = rd.ResolveFlats(filled)
    assert np.array_equal(np.asarray(resolved), g["resolved"])
    assert np.array_equal(np.asarray(rd.FlowDirectionsD8(resolved)), g["dirs"])
    assert np.array_equal(np.asarray(rd.FlowAccumulation(resolved, "D8")), g["fa_d8"])
    np.testing.assert_allclose(np.asarray(rd.FlowAccumulation(resolved, "Dinf")), g["fa_dinf"], rtol=DINF_UNIT_RTOL)


def test_synthetic_golden(golden):
    g = golden["synthetic_ref"]
    for seed in (101, 102, 103):
        k = f"s{seed}"
        filled = rd.FillDepressions(R(g[f"{k}__dem"]))
        assert np.array_equal(np.asarray(filled), g[f"{k}__filled"])
        resolved = rd.ResolveFlats(filled)
        assert np.array_equal(np.asarray(resolved), g[f"{k}__resolved"])
        assert np.array_equal(np.asarray(rd.FlowAccumulation(resolved, "D8")), g[f"{k}__fa_d8"])


# ---- oracle comparisons on seeded inputs -----------------------------------------------------
@pytest.mark.parametrize("shape,seed,q,patch", [
    ((150, 220), 1, None, False), ((257, 131), 2, 0.5, False), ((400, 500), 3, 2.0, True),
    ((65, 129), 4, 1.0, False), ((64, 64), 5, 10.0, False), ((63, 200), 6, None, True),
    ((1024, 1024), 7, None, False), ((777, 1025), 8, 1.0, True),
])
def test_pipeline_vs_oracle(checker, shape, seed, q, patch):
    dem = oracle.fbm_terrain(*shape, seed=seed, quantum=q)
    if patch:
        h, w = shape
        dem[h // 4: h // 4 + h // 8, w // 3: w // 3 + w // 6] = ND
        dem[0: h // 10, 0: w // 10] = ND
    wts = np.random.default_rng(seed).random(shape)
    check_pipeline(dem, ND, checker, accum_weights=wts)


def test_pipeline_vs_oracle_large(checker):
    dem = oracle.fbm_terrain(2048, 3000, seed=21, quantum=0.5)
    check_pipeline(dem, ND, checker)


@pytest.mark.parametrize("shape", [(1, 1), (1, 7), (2, 2), (3, 3), (3, 64), (5, 1), (4, 130)])
def test_degenerate_shapes(checker, shape):
    dem = (np.random.default_rng(3).random(shape) * 10).astype(np.float32)
    check_pipeline(dem, ND, checker)


def test_special_rasters(checker):
    flat = np.full((70, 90), 5.0, np.float32)                 # one big undrainable flat
    check_pipeline(flat, ND, checker)
    allnd = np.full((40, 50), ND, np.float32)                 # everything NoData
    check_pipeline(allnd, ND, checker)
    bowl = np.fromfunction(lambda y, x: (y - 40) ** 2 + (x - 50) ** 2, (81, 101)).astype(np.float32)
    check_pipeline(bowl, ND, checker)                         # one deep pit -> big drainable flat
    neg = -oracle.fbm_terrain(100, 100, seed=9, quantum=1.0)  # negative elevations and zeros
    check_pipeline(neg - neg.max() / 2, ND, checker)
    tiny = (oracle.fbm_terrain(90, 90, seed=10, quantum=50.0) * 1e-42).astype(np.float32)  # denormals
    check_pipeline(tiny, ND, checker)


def test_non_tma_staging_gives_identical_fill(checker):
    dem = oracle.fbm_terrain(500, 700, seed=12)
    a = np.asarray(rd.FillDepressions(R(dem)))
    _lib.set_param("fill_use_tma", 0)
    try:
        b = np.asarray(rd.FillDepressions(R(dem)))
    finally:
        _lib.set_param("fill_use_tma", 1)
    assert np.array_equal(a, b) and np.array_equal(a, checker.fill_depressions(dem))


def test_capped_in_tile_iterations_converge_to_same_answer(checker):
    dem = oracle.fbm_terrain(600, 600, seed=13)
    _lib.set_param("fill_max_iters", 2)
    try:
        a = np.asarray(rd.FillDepressions(R(dem)))
    finally:
        _lib.set_param("fill_max_iters", 0)
    assert np.array_equal(a, checker.fill_depressions(dem))


def test_in_place_and_copy_semantics():
    dem = R(oracle.fbm_terrain(128, 128, seed=14))
    orig = np.array(dem)
    out = rd.FillDepressions(dem)
    assert out is not dem and np.array_equal(np.asarray(dem), orig)
    assert rd.FillDepressions(dem, in_place=True) is None
    assert np.array_equal(np.asarray(dem), np.asarray(out))
    assert "FillDepressions" in out.metadata["PROCESSING_HISTORY"]
    w = R(np.full((128, 128), 2.0), -1)
    acc = rd.FlowAccumulation(dem, "D8", weights=w, in_place=True)
    assert np.shares_memory(acc, w)


# ---- size-independent properties at a size the CPU oracle would need minutes for ----------------
def test_properties_at_8192():
    import torch
    N = 8192
    L = _lib.lib()
    d = torch.empty((N, N), dtype=torch.float32, device="cuda")
    _lib.check(L.rdb200_dev_generate_fbm_f32(d.data_ptr(), N, N, 0, 77, 12, 0.0))
    z = d.clone()
    _lib.check(L.rdb200_dev_fill_depressions_d8_f32(d.data_ptr(), N, N))
    assert bool((d >= z).all()), "fill never lowers a cell"
    assert bool(torch.isfinite(d).all())
    for sl in (np.s_[0, :], np.s_[-1, :], np.s_[:, 0], np.s_[:, -1]):
        assert torch.equal(d[sl], z[sl]), "border cells are pinned"
    raised = float((d > z).float().mean())
    assert 0.05 < raised < 0.6
    again = d.clone()
    _lib.check(L.rdb200_dev_fill_depressions_d8_f32(again.data_ptr(), N, N))
    assert torch.equal(again, d), "fill is idempotent"
    # every interior cell has a neighbour that is not higher (no pits left)
    pad = torch.nn.functional.pad(d[None, None], (1, 1, 1, 1), value=float("inf"))
    nmin = -torch.nn.functional.max_pool2d(-pad, 3, stride=1)[0, 0]
    inner = torch.ones_like(d, dtype=torch.bool)
    inner[0, :] = inner[-1, :] = False
    inner[:, 0] = inner[:, -1] = False
    # nmin includes the centre; a pit would have all 8 neighbours strictly higher -> check via
    # second-smallest is overkill: use the definition W = max(Z, min8(W)) instead
    p = torch.nn.functional.pad(d[None, None], (1, 1, 1, 1), value=float("inf"))[0, 0]
    m8 = torch.full_like(d, float("inf"))
    for dy in (0, 1, 2):
        for dx in (0, 1, 2):
            if dy == 1 and dx == 1:
                continue
            m8 = torch.minimum(m8, p[dy:dy + N, dx:dx + N])
    assert torch.equal(d[inner], torch.maximum(z, m8)[inner]), "fixed-point equation holds everywhere"
    del pad, nmin, p, m8, again
    # D8 accumulation: flow is conserved -- the accumulation of all outlets sums to the cell count
    acc = torch.empty((N, N), dtype=torch.float64, device="cuda")
    _lib.check(L.rdb200_dev_fa_d8_f32_f64(d.data_ptr(), acc.data_ptr(), N, N, ND, 1))
    props = torch.empty((N, N, 9), dtype=torch.float32, device="cuda")
    _lib.check(L.rdb200_dev_fm_d8_f32(d.data_ptr(), props.data_ptr(), N, N, ND))
    outlet = props[..., 0] == -1.0
    assert float(acc[outlet].sum()) == float(N * N)
    assert float(acc.min()) == 1.0
    acc2 = torch.empty_like(acc)
    _lib.check(L.rdb200_dev_fa_d8_f32_f64(d.data_ptr(), acc2.data_ptr(), N, N, ND, 1))
    assert torch.equal(acc, acc2), "unit-weight D8 accumulation is deterministic"
    # generic props path agrees with the fused path
    acc3 = torch.ones_like(acc)
    _lib.check(L.rdb200_dev_flow_accumulation_props_f64(props.data_ptr(), acc3.data_ptr(), N, N))
    assert torch.equal(acc, acc3)


def test_cxx_dropin_matches_reference_cpu_templates():
    """The C++ drop-in header: RichDEM call sites on Array2D<float> run on the GPU and agree with
    the reference's own CPU templates instantiated for double (in-process oracle inside the binary)."""
    import os
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "build", "reference_bindings", "cxx_dropin_check")
    if not os.path.exists(exe):
        pytest.skip("build/reference_bindings/cxx_dropin_check not built (reference headers absent at build time)")
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-3000:]
    assert "thrown=0 mismatches=0 dim_mismatch_throws=1" in out.stdout, out.stdout[-3000:]


# ---- alternative code paths must give identical results ------------------------------------------
VARIANTS = [  # every switch is a schedule / layout choice (rdb200_set_param); none may change a result
    {"fill_ordered": 0, "fill_multigrid": 0}, {"fill_multigrid": 0}, {"fill_vcycle": 0}, {"fill_multigrid": 4, "fill_vcycle": 4},
    {"fill_multigrid": 8, "fill_multigrid_min": 256, "fill_vcycle": 2}, {"fill_multigrid": 3, "fill_multigrid_min": 128, "fill_vcycle": 0},
    {"flats_tiled": 0}, {"flats_uf_tiled": 0}, {"flats_fused_classify": 0}, {"flats_pair": 0}, {"accum_packed": 0}, {"accum_fused_prep": 0}, {"accum_walk_lanes": 0},
    {"accum_fused_prep": 0, "accum_walk_lanes": 0}, {"accum_walk_scan": 1}, {"accum_walk_scan": 2}, {"flowmet_tarboton_filter": 0}, {"flowdirs_rolling": 0}, {"accum_dinf_packed": 0}, {"accum_dinf_packed": 1}, {"accum_dinf_packed": 1, "accum_dinf_share": 0}, {"accum_dinf_packed": 1, "accum_dinf_share": 64}, {},
]


@pytest.mark.parametrize("cfg", VARIANTS, ids=lambda c: ",".join(f"{k}={v}" for k, v in c.items()) or "defaults")
@pytest.mark.parametrize("shape,q", [((1500, 2040), 0.5), ((777, 1028), 2.0)])
def test_algorithm_variants_agree(checker, cfg, shape, q):
    """Round-1 kernels vs the round-2 defaults (multigrid start + V-cycles, fused D8 preparation, persistent-lane
    walk, tiled union-find, rolling-window direction kernel): same bits, and equal to the checker."""
    dem = oracle.fbm_terrain(*shape, seed=shape[0], quantum=q)
    dem[shape[0] // 4: shape[0] // 4 + 40, shape[1] // 3: shape[1] // 3 + 60] = ND
    f_ref = checker.fill_depressions(dem)
    r_ref = checker.resolve_flats(f_ref, ND)
    try:
        for k, v in cfg.items():
            _lib.set_param(k, v)
        f = np.asarray(rd.FillDepressions(R(dem)))
        r = np.asarray(rd.ResolveFlats(R(f_ref)))
        a = np.asarray(rd.FlowAccumulation(R(r_ref), "D8"))
        a2 = np.asarray(rd.FlowAccumulation(R(f_ref), "D8"))
        d = np.asarray(rd.FlowDirectionsD8(R(r_ref)))
        ai = np.asarray(rd.FlowAccumulation(R(r_ref), "Dinf"))
    finally:
        _lib.reset_params()
    assert np.array_equal(f, f_ref)
    assert np.array_equal(r.view(np.uint32), r_ref.view(np.uint32))
    assert np.array_equal(a, checker.fa_d8(r_ref, ND))
    assert np.array_equal(a2, checker.fa_d8(f_ref, ND))
    assert np.array_equal(d, checker.d8_flow_directions(r_ref, ND))
    np.testing.assert_allclose(ai, checker.fa_dinf(r_ref, ND), rtol=ACC_RTOL if cfg.get("accum_dinf_packed") == 0 else DINF_UNIT_RTOL,
                               atol=0)


def walled_lake_case():
    """ADVICE round 1: a lake whose wall sits inside a coarse block next to a tile seam.  The prolongation of a V-cycle
    lowers cells on a tile edge; the neighbouring tile (whose own cells lie in blocks with a high maximum) must be
    woken as well, or 336 cells keep the level 20 instead of 1."""
    dem = np.full((64, 192), 20.0, np.float32)
    dem[8:56, 57:191] = 0.0
    dem[32, 191] = 1.0
    return dem


def test_vcycle_prolongation_wakes_neighbouring_tiles(checker):
    dem = walled_lake_case()
    expected = checker.fill_depressions(dem)
    assert (expected == 1.0).sum() > 6000
    try:
        for cfg in ({"fill_multigrid": 8, "fill_multigrid_min": 32, "fill_vcycle": 1},
                    {"fill_multigrid": 8, "fill_multigrid_min": 32, "fill_vcycle": 1, "fill_use_tma": 0},
                    {"fill_multigrid": 4, "fill_multigrid_min": 32, "fill_vcycle": 2}):
            _lib.reset_params()
            for k, v in cfg.items():
                _lib.set_param(k, v)
            assert np.array_equal(np.asarray(rd.FillDepressions(R(dem))), expected), cfg
    finally:
        _lib.reset_params()


def test_unit_weight_d8_on_width_not_multiple_of_4(checker):
    """W % 4 != 0 takes the scalar (non-vectorised, non-packed) kernels."""
    dem = checker.fill_depressions(oracle.fbm_terrain(301, 403, seed=19, quantum=0.5))
    assert np.array_equal(np.asarray(rd.FlowAccumulation(R(dem), "D8")), checker.fa_d8(dem, ND))


# ---- SURVEY 8f-1: FM_D4 / FM_Quinn / FM_Holmgren / FM_Freeman and their FA_* ----------------------------
METRIC_CASES = [("D4", None), ("Quinn", None), ("Holmgren", 2.5), ("Holmgren", 0.7), ("Freeman", 1.1), ("Freeman", 4.0)]
MFD_ACC_RTOL = 1e-6  # north_star: 1e-5 relative; proportions may differ by 1 float ulp where pow() is involved


def check_metric(dem, nd, m, e, fm_ref, fa_ref, fm_sel=None, fa_sel=None):
    p = np.asarray(rd.FlowProportions(R(dem, nd), m, exponent=e))
    p = p if fm_sel is None else fm_sel(p)
    if m in ("D4", "Quinn"):  # no transcendental involved: bit-identical
        assert np.array_equal(p, fm_ref), (m, e)
    else:
        assert np.array_equal(p > 0, fm_ref > 0), (m, e)
        assert ulp_diff(p, fm_ref).max() <= 1, (m, e, int(ulp_diff(p, fm_ref).max()))
    a = rd.FlowAccumulation(R(dem, nd), m, exponent=e)
    assert a.no_data == -1 and a.dtype == np.float64
    a = np.asarray(a) if fa_sel is None else fa_sel(np.asarray(a))
    np.testing.assert_allclose(a, fa_ref, rtol=MFD_ACC_RTOL if m not in ("D4",) else ACC_RTOL, atol=0, err_msg=f"{m} {e}")


def test_remaining_flow_metrics_golden(golden):
    g = golden["flow_metrics_ref"]
    dems = {"beauford": golden["beauford_crop"]["resolved"], "s104": g["s104__resolved"]}
    for name, dem in dems.items():
        for m, e in METRIC_CASES:
            k = f"{name}__{m}_{e}"
            check_metric(dem, ND, m, e, g[k + "__fm"], g[k + "__fa"], fm_sel=lambda p: p.reshape(-1, 9)[::11],
                         fa_sel=lambda a: a[::3, ::3])


@pytest.mark.parametrize("method,exponent", METRIC_CASES)
def test_remaining_flow_metrics_vs_oracle(checker, method, exponent):
    dem = oracle.fbm_terrain(700, 900, seed=31, quantum=0.25)
    dem[100:140, 300:420] = ND
    dem = checker.resolve_flats(checker.fill_depressions(dem), ND)
    check_metric(dem, ND, method, exponent, checker.fm_method(dem, ND, method, exponent),
                 checker.fa_method(dem, ND, method, exponent))
    wts = np.random.default_rng(4).random(dem.shape)
    a = rd.FlowAccumulation(R(dem), method, exponent=exponent, weights=R(wts, -1))
    np.testing.assert_allclose(np.asarray(a), checker.fa_method(dem, ND, method, exponent, wts), rtol=MFD_ACC_RTOL, atol=0)


def test_exponent_methods_require_an_exponent():
    dem = R(oracle.fbm_terrain(40, 50, seed=1))
    for m in ("Holmgren", "Freeman"):
        with pytest.raises(Exception, match="requires an exponent"):
            rd.FlowAccumulation(dem, m)
        with pytest.raises(Exception, match="requires an exponent"):
            rd.FlowProportions(dem, m)
    with pytest.raises(Exception, match="outside the B200 hot path"):
        rd.FlowAccumulation(dem, "Rho8")


# ---- the benchmark raster and the benchmark size -----------------------------------------------------------
def test_device_terrain_generator_equals_its_cpu_restatement():
    """bench.py --impl reference runs the reference on oracle.device_fbm(...): it must be the raster the GPU arm uses."""
    import torch
    L = _lib.lib()
    for (h, w, y0, seed, q) in ((700, 1000, 0, 42, 0.0), (513, 4100, 12345, 7, 0.0), (300, 260, 70000, 42, 0.5)):
        d = torch.empty((h, w), dtype=torch.float32, device="cuda")
        _lib.check(L.rdb200_dev_generate_fbm_f32(d.data_ptr(), w, h, y0, seed, 12, q))
        assert np.array_equal(d.cpu().numpy().view(np.uint32), oracle.device_fbm(h, w, seed=seed, quantum=q, y0=y0).view(np.uint32))


def test_fill_and_d8_accumulation_vs_reference_at_8192():
    """The benchmark workload at 8192^2 (67 Mcells) against the reference: fill bit-exact, FA_D8 bit-exact (digests of the
    reference's whole outputs, tests/golden/make_golden.py::reference_digests)."""
    N = 8192
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")) as f:
        D = json.load(f)["bench_8192"]
    dem = oracle.device_fbm(N, N, seed=42)
    assert oracle.digest(dem) == D["dem"], "benchmark raster drifted"
    filled = np.asarray(rd.FillDepressions(R(dem)))
    assert oracle.digest(filled) == D["filled"]
    assert oracle.digest(np.asarray(rd.FlowAccumulation(R(filled), "D8"))) == D["fa_d8"]


# ---- FillDepressions<Topology::D4> ---------------------------------------------------------------------------
@pytest.mark.parametrize("shape,seed,q", [((150, 220), 1, None), ((400, 500), 3, 2.0), ((64, 64), 5, 10.0), ((1500, 2040), 7, 0.5),
                                          ((3, 3), 9, None), ((1, 17), 10, None)])
def test_d4_fill_vs_oracle(checker, shape, seed, q):
    dem = oracle.fbm_terrain(*shape, seed=seed, quantum=q)
    if shape[0] > 100:
        dem[shape[0] // 4: shape[0] // 4 + 20, shape[1] // 3: shape[1] // 3 + 30] = ND
    got = np.asarray(rd.FillDepressions(R(dem), topology="D4"))
    assert np.array_equal(got, checker.fill_depressions(dem, "fill_d4"))


def test_d4_fill_variants(checker):
    dem = oracle.fbm_terrain(1100, 1300, seed=23, quantum=1.0)
    expected = checker.fill_depressions(dem, "fill_d4")
    try:
        for cfg in ({}, {"fill_multigrid": 0}, {"fill_multigrid": 4, "fill_multigrid_min": 128, "fill_vcycle": 2}, {"fill_ordered": 0, "fill_multigrid": 0}):
            _lib.reset_params()
            for k, v in cfg.items():
                _lib.set_param(k, v)
            assert np.array_equal(np.asarray(rd.FillDepressions(R(dem), topology="D4")), expected), cfg
    finally:
        _lib.reset_params()


# ---- SURVEY 8f-2: direction-grid flat resolution (barnes_flat_resolution_d8, the pipeline of rd_d8_flowdirs) ----------
def test_flow_directions_with_resolved_flats_golden(golden):
    g = golden["flowdirs_flats_ref"]
    for name, dem in (("beauford", golden["beauford_crop"]["filled"]), ("s105", g["s105__dem"])):
        d = R(dem.copy())
        got = np.asarray(rd.FlowDirectionsD8Resolved(d))
        assert np.array_equal(got, g[name + "__dirs"]), name
        assert np.array_equal(np.asarray(d), dem), "alter=False leaves the elevations alone"


@pytest.mark.parametrize("shape,seed,q", [((300, 420), 2, 0.5), ((777, 1028), 4, 2.0), ((64, 70), 5, 10.0)])
def test_flow_directions_with_resolved_flats_vs_oracle(checker, shape, seed, q):
    dem = oracle.fbm_terrain(*shape, seed=seed, quantum=q)
    dem[shape[0] // 3: shape[0] // 3 + 12, shape[1] // 4: shape[1] // 4 + 25] = ND
    filled = checker.fill_depressions(dem)
    expected = checker.d8_flow_directions_flats(filled, ND)[0]
    assert np.array_equal(np.asarray(rd.FlowDirectionsD8Resolved(R(filled.copy()))), expected)
    # alter=True: the elevations take the increments and plain D8 directions on them drain every drainable flat
    d = R(filled.copy())
    dirs_alt = np.asarray(rd.FlowDirectionsD8Resolved(d, alter=True))
    assert np.array_equal(np.asarray(d).view(np.uint32), checker.resolve_flats(filled, ND).view(np.uint32))
    assert np.array_equal(dirs_alt, checker.d8_flow_directions(np.asarray(d), ND))


# ---- SURVEY 8f-4: terrain attributes (TA_*, methods/terrain_attributes.hpp:370-538) ------------------------------------
TA_EXACT = ("slope_riserun", "slope_percentage", "curvature", "planform_curvature", "profile_curvature")
TA_LIBM = ("slope_degrees", "slope_radians", "aspect")  # through atan / atan2: <= 1 float ulp
TA_CASES = [(1.0, (1.0, 1.0)), (2.5, (30.0, 20.0))]


def check_terrain_attribute(got, ref, attrib, where):
    assert got.dtype == np.float32 and got.shape == ref.shape
    if attrib in TA_EXACT:
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), (where, attrib, int((got != ref).sum()))
    else:
        d = ulp_diff(got, ref)
        assert d.max() <= 1, (where, attrib, int(d.max()))
        assert (d != 0).mean() < 1e-3, (where, attrib, float((d != 0).mean()))  # a rounding-boundary rarity, not a bias


def test_terrain_attributes_golden(golden):
    g = golden["terrain_attributes_ref"]
    for name, dem in (("beauford", golden["beauford_crop"]["dem"]), ("s106", g["s106__dem"])):
        for attrib in TA_EXACT + TA_LIBM:
            for zs, cell in TA_CASES:
                d = R(dem)
                d.geotransform = [0.0, cell[0], 0.0, 0.0, 0.0, -cell[1]]
                out = rd.TerrainAttribute(d, attrib, zscale=zs)
                assert out.no_data == -9999
                check_terrain_attribute(np.asarray(out)[::3, ::3], g[f"{name}__{attrib}__{zs}"], attrib, (name, zs))


@pytest.mark.parametrize("shape", [(517, 1031), (1, 9), (7, 1), (2, 2), (130, 129), (16, 128), (17, 257)])
def test_terrain_attributes_vs_oracle(checker, shape):
    """Shapes around the 128 x 16 window of the kernel, degenerate rasters, NoData patches and NoData on the border."""
    dem = oracle.fbm_terrain(*shape, seed=shape[0] + shape[1], quantum=0.25)
    if shape[0] > 40:
        dem[10:30, 20:90] = ND
        dem[0, :7] = ND
        dem[-1, -5:] = ND
    for attrib in TA_EXACT + TA_LIBM:
        d = R(dem)
        d.geotransform = [100.0, 10.0, 0.0, 200.0, 0.0, -10.0]
        got = np.asarray(rd.TerrainAttribute(d, attrib, zscale=0.3048))
        ref = checker.terrain_attribute(dem, attrib, ND, 0.3048, (10.0, 10.0))
        check_terrain_attribute(got, ref, attrib, shape)


def test_terrain_attribute_rejects_unknown_names():
    with pytest.raises(Exception, match="Invalid TerrainAttributes attribute"):
        rd.TerrainAttribute(R(oracle.fbm_terrain(8, 8, seed=1)), "spi")
