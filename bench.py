#!/usr/bin/env python
"""bench.py -- Priority-Flood fill + D8 flow accumulation on a synthetic fractal DEM.

Metric (BASELINE.json): "Priority-Flood + D8 flow-accum Mcells/s on 32768^2 DEM; HBM GB/s vs peak".
One step = FillDepressions<D8> followed by FA_D8 (unit weights) over one 32768 x 32768 float32
DEM (1.07 Gcells; 4 GiB, far larger than the 126 MB L2, so no cache flush is needed between
steps).  `value` = cells / device time with the DEM resident in HBM; `e2e` = the same two calls
through the host-pointer C ABI (pinned host buffers, H2D/D2H inside the timed region).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--size 32768] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step computed, the filled DEM (DIR/filled.npy, float32) and its D8
accumulation (DIR/fa_d8.npy, float64): whole rasters up to DUMP_CELLS cells, above that the same seeded sample of
DUMP_CELLS cells in every run of a size, so that two builds (or, at the same raster size, the GPU path and
--impl reference) can be compared output for output.

After the timed loop the result of the last step is VERIFIED on the device (fixed-point equation of the fill,
pinned border, conservation of the D8 accumulation) and position-weighted 64-bit checksums of the filled raster and
of the accumulation are printed; they are all-reduced over the ranks, so the line of every N carries the same two
numbers when the sharded results equal the single-GPU ones.

`configs` in the JSON line times the other BASELINE.json configurations once each (they are not the metric):
4096^2 fill; 16384^2 fill + flat resolution + FA_D8; 32768^2 fill + FA_Dinf (N = 1, 2, 4); 65536^2 fill + flat
resolution + FA_D8 (N = 8; the reference cannot represent that raster, Array2D.hpp:98-101).

N > 1 (launched by torchrun, one rank per GPU): the raster is row-sharded; fill and accumulation exchange one-row
halos over NCCL (richdem_b200/sharded.py); strong scaling (total work fixed).
`--impl reference` times the reference's own CPU implementation (oracle/_ref when it was compiled from
/root/reference, else the C port) on the SAME raster (the device generator's CPU restatement, bit-identical).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Priority-Flood fill + D8 flow accumulation throughput"
UNIT = "Mcells/s"
ND = -9999.0
SEED = 42


def BAND_FILL_KW(row0, height):
    """The band's place in the raster for sharded.fill_band (the C++ band driver takes the multigrid settings from the
    library switches fill_multigrid / fill_vcycle; RDB200_PARAMS presets them for experiments)."""
    return {"row0": row0, "height": height}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index: int = 0):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(float(s[0])) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = max((int(float(s[1])) for s in self.samples if s[1].replace(".", "").isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if len(s) > 2 + i and s[2 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons,
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------
def cpu_reference_run(n: int, steps: int, warmup: int, budget_s: float = 1e9, dump_dir=None):
    """Times the CPU implementation (reference if compiled, else port) on the n x n benchmark raster (the device
    generator's bit-identical CPU restatement).  Stops early (after >= 1 timed step) when `budget_s` is spent.
    dump_dir: write the last step's outputs there as --dump-outputs does for the GPU path."""
    import oracle
    O = oracle.best()
    kind = "reference" if O.kind == "reference" else "port"
    cores = os.cpu_count() if kind == "reference" else 1
    t_gen = time.perf_counter()
    dem = oracle.device_fbm(n, n, seed=SEED)
    t_gen = time.perf_counter() - t_gen
    times = []
    t_start = time.perf_counter()
    for i in range(warmup + steps):
        f = a = None
        t = time.perf_counter()
        f = O.fill_depressions(dem)
        t1 = time.perf_counter()
        a = O.fa_d8(f, ND)
        t2 = time.perf_counter()
        if i >= warmup:
            times.append((t2 - t, t1 - t, t2 - t1))
        if times and time.perf_counter() - t_start > budget_s:
            break
    if dump_dir:
        idx = dump_indices(n, n)
        save_dump(dump_dir, "filled", f.reshape(-1)[idx], n, n)
        save_dump(dump_dir, "fa_d8", a.reshape(-1)[idx], n, n)
    del a, f
    tot = sum(t[0] for t in times) / len(times)
    return {
        "value": n * n / tot / 1e6, "unit": UNIT, "cores": cores, "kind": kind,
        "sample": f"{n}x{n} benchmark fBm DEM (seed {SEED}; CPU restatement of the device generator, bit-identical), "
                  f"FillDepressions<D8> + FA_D8, mean of {len(times)} run(s); fill "
                  f"{sum(t[1] for t in times) / len(times):.2f}s + accum {sum(t[2] for t in times) / len(times):.2f}s; "
                  f"the flood and the accumulation wavefront are serial in the reference (OpenMP only parallelises "
                  f"FM_D8); raster generated in {t_gen:.1f}s (not timed)",
        "seconds_per_run": tot, "steps_run": len(times),
    }


def _host_mem_available_gib():
    try:
        import psutil
        return psutil.virtual_memory().available / 2 ** 30
    except Exception:
        return 0.0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.size
    # the reference's FA_D8 materialises a 36 B/cell Array3D (flow_accumulation.hpp:27) next to the 4 + 4 + 8 + 1 B/cell
    # rasters: ~56 B/cell; halve the raster until that fits comfortably in host memory
    need = lambda m: 60.0 * m * m / 2 ** 30
    avail = _host_mem_available_gib()
    while n > 2048 and avail > 0 and need(n) > 0.8 * avail:
        n //= 2
    if args.ref_size:
        n = args.ref_size
    # one full-size step costs minutes of serial CPU: cap the number of steps by wall time, not the raster
    cb = cpu_reference_run(n, max(1, args.steps), 0 if n >= 8192 else max(0, min(args.warmup, 1)), budget_s=args.ref_budget_s,
                           dump_dir=args.dump_outputs)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["seconds_per_run"] * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.size}x{args.size} synthetic fBm float32 DEM (seed {SEED}, 12 octaves), "
                               f"FillDepressions<D8> + FA_D8 unit weights", "seed": SEED,
                   "timed_raster": f"{n}x{n}", "same_config": n == args.size, "steps_run": cb["steps_run"],
                   "note": "steps are capped by wall time (one 32768^2 step is minutes of serial CPU work); the raster is "
                           "the GPU arm's raster, bit for bit"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print("\n" + json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
def _checksum(t, row0, width):
    """Position-weighted 64-bit checksum (wraps mod 2^64): sum_i bits(v_i) * (1 + (i mod 1000003)), i = global cell
    index.  Order-independent, so ranks can add their parts; any changed / moved cell changes it."""
    import torch
    h = t.shape[0]
    tot = torch.zeros((), dtype=torch.int64, device=t.device)
    step = max(1, (1 << 26) // max(width, 1))
    for y in range(0, h, step):
        blk = t[y:y + step]
        bits = blk.view(torch.int32).to(torch.int64) if blk.dtype == torch.float32 else blk.view(torch.int64)
        idx = (torch.arange(blk.numel(), device=t.device, dtype=torch.int64) + (row0 + y) * width) % 1000003 + 1
        tot += (bits.reshape(-1) * idx).sum()
    return tot


DUMP_CELLS = 1 << 22  # at most 16 MiB of elevations + 32 MiB of accumulation


def dump_indices(N, W):
    """Flat cell indices --dump-outputs writes: all N * W when they are at most DUMP_CELLS, else the sorted, seeded
    sample np.unique(default_rng(SEED).integers(0, N * W, DUMP_CELLS)), the same in every run of a size."""
    import numpy as np
    cells = N * W
    return np.arange(cells) if cells <= DUMP_CELLS else np.unique(np.random.default_rng(SEED).integers(0, cells, DUMP_CELLS))


def save_dump(out_dir, name, values, N, W):
    """values (at dump_indices(N, W)) -> out_dir/<name>.npy, as the N x W raster when it is whole."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), values.reshape(N, W) if N * W <= DUMP_CELLS else values)


def dump_outputs(out_dir, filled, acc, r0, r1, gt, N, W, world, rank):
    """Writes filled.npy and fa_d8.npy of the GPU path (see --dump-outputs).  filled / acc are local rasters (gt ghost
    rows + rows r0 .. r1 of the raster + ghost rows); ranks add their cells."""
    import numpy as np
    import torch
    import torch.distributed as dist
    idx = dump_indices(N, W)
    rows = idx // W
    mine = np.nonzero((rows >= r0) & (rows < r1))[0]
    src = torch.from_numpy((rows[mine] - r0 + gt) * W + idx[mine] % W).cuda()
    dst = torch.from_numpy(mine).cuda()
    for name, t in (("filled", filled), ("fa_d8", acc)):
        v = torch.zeros(len(idx), dtype=t.dtype, device="cuda")
        v[dst] = t.reshape(-1)[src]
        if world > 1:
            dist.all_reduce(v)
        if rank == 0:
            save_dump(out_dir, name, v.cpu().numpy(), N, W)


def verify_band(z_loc, w_loc, acc_loc, gt, gb, r0, r1, H, W):
    """Checks on the device, band by band of rows (so that temporaries stay small):
       fill:  W >= Z, finite, raster border pinned, W = max(Z, min8 W) on every interior cell (the fixed-point equation;
              ghost rows supply the neighbours across a seam);
       FA_D8: accumulation >= 1, and the accumulation of the cells without a receiver (raster edge, or no strictly
              lower neighbour) sums to the number of cells -- returned as a partial sum for the all-reduce.
       z_loc / w_loc / acc_loc are local rasters (gt + owned + gb rows)."""
    import torch
    inf = float("inf")
    ok = {"w_ge_z": True, "finite": True, "border_pinned": True, "fixed_point": True, "acc_ge_1": True}
    outlet_sum = torch.zeros((), dtype=torch.float64, device=w_loc.device)
    hloc = w_loc.shape[0]
    CH = max(64, (1 << 27) // W)
    for y0 in range(gt, hloc - gb, CH):
        y1 = min(hloc - gb, y0 + CH)
        a0, a1 = max(0, y0 - 1), min(hloc, y1 + 1)  # with one halo row where it exists
        wv = w_loc[a0:a1]
        p = torch.nn.functional.pad(wv[None, None], (1, 1, 1, 1), value=inf)[0, 0]
        if a0 == y0:   # no row above inside the local raster: this is the raster's first row
            pass
        m8 = torch.full((y1 - y0, W), inf, dtype=torch.float32, device=w_loc.device)
        off = y0 - a0  # row of wv that is the first checked row
        for dy in (0, 1, 2):
            for dx in (0, 1, 2):
                if dy == 1 and dx == 1:
                    continue
                m8 = torch.minimum(m8, p[off + dy:off + dy + (y1 - y0), dx:dx + W])
        wc, zc = w_loc[y0:y1], z_loc[y0:y1]
        gy = torch.arange(r0 + (y0 - gt), r0 + (y1 - gt), device=w_loc.device)[:, None]
        gx = torch.arange(W, device=w_loc.device)[None, :]
        edge = (gy == 0) | (gy == H - 1) | (gx == 0) | (gx == W - 1)
        ok["w_ge_z"] &= bool((wc >= zc).all())
        ok["finite"] &= bool(torch.isfinite(wc).all())
        ok["border_pinned"] &= bool((wc[edge] == zc[edge]).all())
        ok["fixed_point"] &= bool((wc == torch.maximum(zc, m8))[~edge].all())
        if acc_loc is not None:
            ac = acc_loc[y0:y1]
            ok["acc_ge_1"] &= bool((ac >= 1.0).all())
            outlet = edge | (m8 >= wc)
            outlet_sum += ac[outlet].sum()
        del p, m8
    return ok, outlet_sum


def run_b200(args):
    import torch
    import torch.distributed as dist
    from richdem_b200 import _lib, sharded

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    _lib.init(local_rank)
    L = _lib.lib()
    N = args.size
    W = N
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    _lib.set_stream(stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gmax(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    r0, r1, gt, gb = sharded.local_rows(N, world, rank)
    hloc = (r1 - r0) + gt + gb
    dem0 = torch.empty((hloc, W), dtype=torch.float32, device="cuda")
    _lib.check(L.rdb200_dev_generate_fbm_f32(dem0.data_ptr(), W, hloc, r0 - gt, SEED, 12, 0.0))
    work = torch.empty_like(dem0)
    acc = torch.empty((hloc, W), dtype=torch.float64, device="cuda") if world == 1 else None
    torch.cuda.synchronize()

    agg = {"launches": 0, "sweep_ms": 0.0, "visits": 0, "tile_cells": 4096, "rounds": 0, "iters": 0,
           "fill_ms": 0.0, "acc_ms": 0.0, "exchange_rounds": 0}
    last = {}

    def one_step(record: bool):
        work.copy_(dem0)
        if world == 1:
            _lib.check(L.rdb200_dev_fill_depressions_d8_f32(work.data_ptr(), W, hloc))
            s1 = _lib.stats()
            _lib.check(L.rdb200_dev_fa_d8_f32_f64(work.data_ptr(), acc.data_ptr(), W, hloc, ND, 1))
            s2 = _lib.stats()
            last["filled"], last["acc"] = work, acc
            if record:
                agg["launches"] += s1["kernel_launches"] + s2["kernel_launches"] + 1
                agg["sweep_ms"] += s1["ms_main_kernel"]
                agg["visits"] += s1["fill_tile_visits"]
                agg["rounds"] += s1["fill_rounds"]
                agg["iters"] += s1["fill_tile_iters"]
                agg["fill_ms"] += s1["ms_total"]
                agg["acc_ms"] += s2["ms_total"]
        else:
            # rdb200_mgpu_* (the C++ band drivers over NCCL) report per-call counters like the single-GPU entry points
            ta = time.perf_counter()
            filled, rounds, st = sharded.fill_band(work, gt, gb, return_stats=True, **BAND_FILL_KW(r0 - gt, N))
            torch.cuda.synchronize()
            tb = time.perf_counter()
            res, rounds2, st2 = sharded.fa_band(filled, gt, gb, ND, dinf=False, rank_rows=(r0, r1, N), return_stats=True)
            torch.cuda.synchronize()
            tc = time.perf_counter()
            last["filled"], last["acc"] = filled, res
            if record:
                agg["fill_ms"] += (tb - ta) * 1e3
                agg["acc_ms"] += (tc - tb) * 1e3
                agg["fill_xr"] = agg.get("fill_xr", 0) + rounds
                agg["acc_xr"] = agg.get("acc_xr", 0) + rounds2
                agg["launches"] += st["kernel_launches"] + st2["kernel_launches"] + 1
                agg["sweep_ms"] += st["ms_main_kernel"]
                agg["visits"] += st["fill_tile_visits"]
                agg["rounds"] += st["fill_rounds"]
                agg["iters"] += st["fill_tile_iters"]
                agg["exchange_rounds"] += rounds + rounds2

    for _ in range(args.warmup):
        one_step(False)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        e0.record(stream)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            one_step(True)
        e1.record(stream)
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
    dev_ms = e0.elapsed_time(e1)
    t = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms = float(t[0]), float(t[1])
    ms_per_step = dev_ms / args.steps
    cells = float(N) * float(N)
    value = cells / (ms_per_step * 1e-3) / 1e6

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last["filled"], last["acc"], r0, r1, gt, N, W, world, rank)

    # ---- verification of what was just timed (the last step's outputs), at every N ----
    verification = None
    if not args.no_verify:
        filled, accr = last["filled"], last["acc"]
        zsrc = dem0
        if world > 1:  # ghost rows of the input hold the neighbours' rows already (generated with the band)
            pass
        ok, outlet_sum = verify_band(zsrc, filled, accr, gt, gb, r0, r1, N, W)
        own = slice(gt, gt + (r1 - r0))
        cs = torch.stack([_checksum(filled[own], r0, W), _checksum(accr[own], r0, W)])
        flags = torch.tensor([int(v) for v in ok.values()], dtype=torch.int32, device="cuda")
        osum = outlet_sum.reshape(1).clone()
        if world > 1:
            dist.all_reduce(cs, op=dist.ReduceOp.SUM)
            dist.all_reduce(flags, op=dist.ReduceOp.MIN)
            dist.all_reduce(osum, op=dist.ReduceOp.SUM)
        verification = {k: bool(int(f)) for k, f in zip(ok.keys(), flags.tolist())}
        verification["fa_d8_outlets_sum_to_cell_count"] = float(osum[0]) == cells
        verification["checksum_filled"] = f"{int(cs[0]) & 0xFFFFFFFFFFFFFFFF:016x}"
        verification["checksum_fa_d8"] = f"{int(cs[1]) & 0xFFFFFFFFFFFFFFFF:016x}"
        verification["all_ok"] = all(v for k, v in verification.items() if isinstance(v, bool))
        verification["note"] = ("device-side checks of the last timed step; the checksums are position-weighted sums over "
                                "all cells, all-reduced over ranks: equal across N <=> identical rasters")

    # ---- e2e: the reference-facing calls with HOST buffers (N=1: whole raster; N>1: per-rank band) ----
    e2e = None
    if not args.no_e2e:
        try:
            own_rows = r1 - r0
            hrows = own_rows if world > 1 else hloc
            h_dem = torch.empty((hrows, W), dtype=torch.float32, pin_memory=True)
            h_acc = torch.empty((hrows, W), dtype=torch.float64, pin_memory=True)
            src = dem0[gt:gt + own_rows] if world > 1 else dem0
            h_src = torch.empty((hrows, W), dtype=torch.float32, pin_memory=True)
            h_src.copy_(src)
            torch.cuda.synchronize()
            e2e_steps = max(1, min(args.steps, args.e2e_steps))
            times = []
            if world == 1:
                for i in range(1 + e2e_steps):
                    h_dem.copy_(h_src)  # host-side reset of the in/out buffer (not timed)
                    barrier()
                    ts = time.perf_counter()
                    _lib.check(L.rdb200_fill_depressions_d8_f32(h_dem.data_ptr(), W, hrows))
                    _lib.check(L.rdb200_fa_d8_f32_f64(h_dem.data_ptr(), h_acc.data_ptr(), W, hrows, ND, 1))
                    float(h_acc[hrows // 2, W // 2])  # read the result on the host
                    te = time.perf_counter()
                    if i >= 1:
                        times.append(te - ts)
                e2e_s = sum(times) / len(times)
                e2e = {"value": cells / e2e_s / 1e6, "unit": UNIT,
                       "h2d_bytes_per_step": int(2 * cells * 4), "d2h_bytes_per_step": int(cells * 4 + cells * 8),
                       "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
                       "note": "rdb200_fill_depressions_d8_f32 + rdb200_fa_d8_f32_f64 on pinned host buffers"}
            else:
                for i in range(1 + e2e_steps):
                    barrier()
                    ts = time.perf_counter()
                    loc = torch.empty((hloc, W), dtype=torch.float32, device="cuda")
                    loc[gt:gt + own_rows].copy_(h_src, non_blocking=True)
                    sharded.exchange_rows(loc, gt, gb)  # ghost rows of elevation come from the neighbours
                    filled, _ = sharded.fill_band(loc, gt, gb, **BAND_FILL_KW(r0 - gt, N))
                    res, _ = sharded.fa_band(filled, gt, gb, ND, dinf=False, rank_rows=(r0, r1, N))
                    h_dem.copy_(filled[gt:gt + own_rows], non_blocking=True)
                    h_acc.copy_(res[gt:gt + own_rows], non_blocking=True)
                    barrier()
                    float(h_acc[hrows // 2, W // 2])
                    te = time.perf_counter()
                    if i >= 1:
                        times.append(te - ts)
                e2e_s = gmax(sum(times) / len(times))
                e2e = {"value": cells / e2e_s / 1e6, "unit": UNIT,
                       "h2d_bytes_per_step": int(cells * 4), "d2h_bytes_per_step": int(cells * 4 + cells * 8),
                       "ms_per_step": e2e_s * 1e3, "steps": e2e_steps,
                       "note": "per-rank pinned host band -> sharded fill + FA_D8 -> pinned host band"}
            del h_dem, h_acc, h_src
        except Exception as exc:  # never lose the headline line because the host-side leg failed
            if world > 1:
                raise
            e2e = {"value": None, "unit": UNIT, "error": repr(exc)[:300]}

    # ---- the other BASELINE.json configurations, once each (not the metric) ----
    configs = None
    if not args.no_configs:
        configs = {}
        try:
            del acc
            last.clear()
            configs.update(run_configs(args, world, rank, N, W, dem0, work, barrier, gmax))
        except Exception as exc:
            if world > 1:
                raise
            configs["error"] = repr(exc)[:400]

    if world > 1:
        tot = torch.tensor([agg["launches"], agg["visits"], agg["sweep_ms"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        launches_all = int(tot[0])
    else:
        launches_all = agg["launches"]

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_hbm_peak()
    # roofline of the dominant kernel (fill_sweep_kernel): algorithmic bytes = 12 B per cell swept
    # (read W, read Z, write W -- SURVEY 8d) x cells of the tiles it visited, / its device time.  N > 1: rank 0's band.
    sweep_bytes = 12.0 * agg["visits"] * agg["tile_cells"]
    achieved = sweep_bytes / (agg["sweep_ms"] * 1e-3) / 1e9 if agg["sweep_ms"] > 0 else 0.0
    launches_per_step_kernel = agg["rounds"] / args.steps if args.steps else 0
    roofline = {
        "bound": "hbm", "kernel": "fill_sweep_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "peak_source": peak_src, "traffic": args.traffic,
        "traffic_of": "the dominant launch (first sweep round of the finest level): dram read + write of one ncu --set full "
                      "capture, profiles/traffic.json; its algorithmic bytes are 12.88 GB",
        "dominant_launch": args.dominant_launch,
        "algorithmic_bytes_per_launch": sweep_bytes / max(agg["rounds"], 1),
        "avg_launch_ms": agg["sweep_ms"] / max(agg["rounds"], 1),
        "sweep_share_of_step": agg["sweep_ms"] / dev_ms,
        "tile_visits_per_step": agg["visits"] / args.steps, "full_raster_equivalents_per_step":
            agg["visits"] * agg["tile_cells"] / args.steps / (cells / world),
        "in_tile_passes_per_visit": agg["iters"] / max(agg["visits"], 1),
        "sweep_launches_per_step": launches_per_step_kernel,
        "scope": "whole raster (all multigrid levels)" if world == 1 else "rank 0's band",
        "end_to_end_fill_fraction_8B_per_cell": (8.0 * cells / world) / (agg["fill_ms"] / args.steps * 1e-3) / 1e9 / peak
        if agg["fill_ms"] > 0 else None,
    }
    cb = None
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_reference_run(min(N, args.cpu_sample), 1, 0)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{N}x{N} synthetic fBm float32 DEM (seed {SEED}, 12 octaves), FillDepressions<D8> "
                               f"+ FA_D8 unit weights", "l2": "inputs (4 B/cell DEM + 8 B/cell accumulation) exceed "
                               "the 126 MB L2; no flush needed", "sharding": f"{world} row band(s)",
                   "wall_ms_per_step": wall_ms / args.steps},
        "stages_ms_per_step": {"fill": agg["fill_ms"] / args.steps, "fa_d8": agg["acc_ms"] / args.steps}
        if world == 1 else {"fill_rank0_wall": agg["fill_ms"] / args.steps, "fa_d8_rank0_wall": agg["acc_ms"] / args.steps,
                            "fill_exchange_rounds": agg.get("fill_xr", 0) / args.steps,
                            "fa_exchange_rounds": agg.get("acc_xr", 0) / args.steps},
        "pipeline_ms": (configs or {}).get("pipeline_this_size", {}).get("ms"),
        "verification": verification,
        "configs": configs,
        "roofline": roofline,
        "cpu_baseline": cb,
        "e2e": e2e,
        "gpu_launches": launches_all,
        "clocks": clk.summary(),
    }
    # (the compiled reference writes progress-bar control codes without a newline: keep the JSON on a line of its own)
    print("\n" + json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_configs(args, world, rank, N, W, dem0, work, barrier, gmax):
    """The other BASELINE.json configurations (configs[1..4]) timed once each after one untimed pass: device time,
    max over ranks.  Returns {name: {...}}."""
    import torch
    import torch.distributed as dist
    from richdem_b200 import _lib, sharded
    L = _lib.lib()
    out = {}

    def timed(fn, reps=1):
        fn()  # warm-up / allocation
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(torch.cuda.current_stream())
        for _ in range(reps):
            fn()
        e1.record(torch.cuda.current_stream())
        barrier()
        return gmax(e0.elapsed_time(e1) / reps)

    r0, r1, gt, gb = sharded.local_rows(N, world, rank)
    hloc = (r1 - r0) + gt + gb
    cells = float(N) * float(N)
    stage = {}

    if world == 1:
        # full pipeline at the benchmark size: fill -> flats -> FA_D8 (the headline omits the flat resolution)
        def pipe():
            work.copy_(dem0)
            _lib.check(L.rdb200_dev_fill_depressions_d8_f32(work.data_ptr(), W, hloc))
            stage["fill"] = _lib.stats()["ms_total"]
            _lib.check(L.rdb200_dev_resolve_flats_epsilon_f32(work.data_ptr(), W, hloc, ND))
            s = _lib.stats()
            stage["flats"] = s["ms_total"]
            stage["flats_rounds"] = s["flat_bfs_levels"]
            _lib.check(L.rdb200_dev_fa_d8_f32_f64(work.data_ptr(), acc.data_ptr(), W, hloc, ND, 1))
            stage["fa_d8"] = _lib.stats()["ms_total"]
        acc = torch.empty((hloc, W), dtype=torch.float64, device="cuda")
        ms = timed(pipe)
        out["pipeline_this_size"] = {"workload": f"{N}x{N} fill + flat resolution + FA_D8", "ms": ms,
                                     "mcells_per_s": cells / ms / 1e3, "stages_ms": dict(stage)}

        # config 4 (N=1 leg): fill + FA_Dinf at the benchmark size
        def fill_dinf():
            work.copy_(dem0)
            _lib.check(L.rdb200_dev_fill_depressions_d8_f32(work.data_ptr(), W, hloc))
            stage["fill"] = _lib.stats()["ms_total"]
            _lib.check(L.rdb200_dev_fa_tarboton_f32_f64(work.data_ptr(), acc.data_ptr(), W, hloc, ND, 1))
            s = _lib.stats()
            stage["fa_dinf"] = s["ms_total"]
            stage["fa_dinf_levels"] = s["accum_rounds"]
        stage.clear()
        ms = timed(fill_dinf)
        out[f"fill_dinf{N}"] = {"workload": f"{N}x{N} fill + FA_Dinf (BASELINE config 4, 1-GPU leg)", "ms": ms,
                                "mcells_per_s": cells / ms / 1e3, "stages_ms": dict(stage)}
        # d8_flow_directions once
        dirs = torch.empty((hloc, W), dtype=torch.uint8, device="cuda")
        ms = timed(lambda: _lib.check(L.rdb200_dev_d8_flow_directions_f32(work.data_ptr(), dirs.data_ptr(), W, hloc, ND)))
        out["d8_flow_directions"] = {"workload": f"{N}x{N} d8_flow_directions", "ms": ms, "mcells_per_s": cells / ms / 1e3}
        # terrain attributes (SURVEY 8f-4): one 3x3 stencil pass, 4 B in + 4 B out per cell
        ta = torch.empty((hloc, W), dtype=torch.float32, device="cuda")
        for ta_name, ta_id in (("slope_riserun", 0), ("aspect", 4), ("profile_curvature", 7)):
            ms = timed(lambda: _lib.check(L.rdb200_dev_terrain_attribute_f32(ta_id, work.data_ptr(), ta.data_ptr(), W, hloc, ND, ND,
                                                                              1.0, 1.0, 1.0)))
            out["terrain_" + ta_name] = {"workload": f"{N}x{N} TA_{ta_name}", "ms": ms, "mcells_per_s": cells / ms / 1e3,
                                         "gb_per_s": 8.0 * cells / ms / 1e6}
        del dirs, acc, ta

        # configs 2 and 3 on their own rasters
        for name, n2, with_flats in (("fill4096", 4096, False), ("pipeline16384", 16384, True)):
            if n2 > N:
                continue
            d2 = torch.empty((n2, n2), dtype=torch.float32, device="cuda")
            _lib.check(L.rdb200_dev_generate_fbm_f32(d2.data_ptr(), n2, n2, 0, SEED, 12, 0.0))
            w2 = torch.empty_like(d2)
            a2 = torch.empty((n2, n2), dtype=torch.float64, device="cuda") if with_flats else None
            st2 = {}

            def run2():
                w2.copy_(d2)
                _lib.check(L.rdb200_dev_fill_depressions_d8_f32(w2.data_ptr(), n2, n2))
                st2["fill"] = _lib.stats()["ms_total"]
                if with_flats:
                    _lib.check(L.rdb200_dev_resolve_flats_epsilon_f32(w2.data_ptr(), n2, n2, ND))
                    st2["flats"] = _lib.stats()["ms_total"]
                    _lib.check(L.rdb200_dev_fa_d8_f32_f64(w2.data_ptr(), a2.data_ptr(), n2, n2, ND, 1))
                    st2["fa_d8"] = _lib.stats()["ms_total"]
            ms = timed(run2, reps=3)
            out[name] = {"workload": f"{n2}x{n2} " + ("fill + flat resolution + FA_D8 (BASELINE config 3)" if with_flats
                                                     else "Priority-Flood fill (BASELINE config 2)"),
                         "ms": ms, "mcells_per_s": n2 * n2 / ms / 1e3, "stages_ms": dict(st2)}
            del d2, w2, a2
    else:
        # config 4: fill + FA_Dinf, row-sharded
        def fill_dinf_sharded():
            work.copy_(dem0)
            filled, xr = sharded.fill_band(work, gt, gb, **BAND_FILL_KW(r0 - gt, N))
            res, xr2 = sharded.fa_band(filled, gt, gb, ND, dinf=True, rank_rows=(r0, r1, N))
            stage["fill_exchange_rounds"], stage["fa_exchange_rounds"] = xr, xr2
        ms = timed(fill_dinf_sharded)
        out[f"fill_dinf{N}"] = {"workload": f"{N}x{N} fill + FA_Dinf over {world} row bands (BASELINE config 4)", "ms": ms,
                                "mcells_per_s": cells / ms / 1e3, "exchange_rounds": dict(stage)}

        # config 3 / 5 shape: fill + flat resolution + FA_D8, row-sharded, at the benchmark size
        def pipe_sharded():
            work.copy_(dem0)
            filled, xr = sharded.fill_band(work, gt, gb, **BAND_FILL_KW(r0 - gt, N))
            filled = filled.contiguous()
            sharded.resolve_flats_band(filled, gt, gb, ND)
            sharded.exchange_rows(filled, gt, gb)
            res, xr2 = sharded.fa_band(filled, gt, gb, ND, dinf=False, rank_rows=(r0, r1, N))
        ms = timed(pipe_sharded)
        out["pipeline_this_size"] = {"workload": f"{N}x{N} fill + flat resolution + FA_D8 over {world} row bands", "ms": ms,
                                     "mcells_per_s": cells / ms / 1e3}

        # config 5: 65536^2 full pipeline on 8 GPUs (the reference cannot represent this raster: int32 cell indices)
        if world == 8 and not args.no_65536:
            n5 = 65536
            q0, q1, qt, qb = sharded.local_rows(n5, world, rank)
            h5 = (q1 - q0) + qt + qb
            del work
            torch.cuda.empty_cache()
            d5 = torch.empty((h5, n5), dtype=torch.float32, device="cuda")
            _lib.check(L.rdb200_dev_generate_fbm_f32(d5.data_ptr(), n5, h5, q0 - qt, SEED, 12, 0.0))
            w5 = torch.empty_like(d5)
            st5 = {}

            def pipe5():
                w5.copy_(d5)
                ta = time.perf_counter()
                filled, xr = sharded.fill_band(w5, qt, qb, **BAND_FILL_KW(q0 - qt, n5))
                filled = filled.contiguous()
                torch.cuda.synchronize()
                tb = time.perf_counter()
                sharded.resolve_flats_band(filled, qt, qb, ND)
                sharded.exchange_rows(filled, qt, qb)
                torch.cuda.synchronize()
                tc = time.perf_counter()
                res, xr2 = sharded.fa_band(filled, qt, qb, ND, dinf=False, rank_rows=(q0, q1, n5))
                torch.cuda.synchronize()
                td = time.perf_counter()
                st5.update({"fill_rank0_wall": (tb - ta) * 1e3, "flats_rank0_wall": (tc - tb) * 1e3,
                            "fa_d8_rank0_wall": (td - tc) * 1e3, "fill_exchange_rounds": xr, "fa_exchange_rounds": xr2})
            ms = timed(pipe5)
            out["pipeline65536"] = {"workload": "65536x65536 fill + flat resolution + FA_D8 over 8 row bands (BASELINE config 5)",
                                    "ms": ms, "mcells_per_s": float(n5) * n5 / ms / 1e3, "stages_ms": dict(st5),
                                    "cpu_note": "not representable in the reference (Array2D xy_t/i_t are int32: 2^32 cells); "
                                                "its CPU time extrapolates linearly from cpu_baseline"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--size", type=int, default=32768)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=8192, help="edge of the bounded CPU sample DEM (cpu_baseline)")
    ap.add_argument("--ref-size", type=int, default=0, help="--impl reference: raster edge (default: --size, memory permitting)")
    ap.add_argument("--ref-budget-s", type=float, default=200.0, help="--impl reference: stop after the step that passes this")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--no-65536", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--traffic", type=float, default=None,
                    help="dram bytes per sweep launch from the committed ncu capture (default: profiles/traffic.json)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's filled DEM and D8 accumulation as DIR/<name>.npy (see the module doc)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.dominant_launch = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        args.dominant_launch = tj.get("dominant_launch")
        if args.traffic is None:
            args.traffic = float(tj["dram_bytes_per_launch"])
    except Exception:
        pass
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
