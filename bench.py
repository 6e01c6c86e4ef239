#!/usr/bin/env python
"""bench.py -- cell-timesteps/s of the fused surface-energy-balance path on B200.

Headline workload (BASELINE.json configs[1], "C2"): 2048 x 2048 synthetic 10 m DEM + 5 albedo maps,
one ablation season of hourly AWS rows (2200 steps), potential insolation computed in the kernel
without shadows.  A "step" of this benchmark is ONE PASS OF THE WHOLE SEASON over the raster.
With N > 1 GPUs the raster grows to (N*2048) x 2048 and is cut into N row bands, one per rank
(weak scaling); the only exchange is one NCCL all-reduce of the per-step area statistics.

  value  whole-job cell-timesteps/s, inputs resident in HBM, CUDA events on the launching stream
  e2e    the same through the public API from pinned HOST buffers: upload of every raster + forcing,
         pre-pass, kernels, download of the three state rasters + statistics, every pass
  configs.f64        the same workload in float64 (value, roofline)
  configs.c3_shadow  BASELINE configs[2]: 8192 x 8192 with topographic shading, STRONG scaling -- the
         raster is fixed, N row bands; the shading sweep shards by sub-step, an all-to-all over NVLink
         delivers every band its mask rows, the fused kernels run per band (parallel.ShardedShading)
  configs.c4_stations BASELINE configs[3]: 4096 x 4096, 15-minute rows, AWS + 3 stations blended per cell, cloud
         attenuation of the shortwave (specification ours: the reference has one AWS)
  configs.c5         BASELINE configs[4]: parameter ensemble on 4096 x 4096, 8 members per GPU; four members
         per pass of the fused kernel (enrgy_run_members)
  --impl reference   the UNMODIFIED reference (oracle/_ref, copied by __graft_entry__.build()) run
         through oracle/ref_harness.py on the host cores -- per-step np.load of the insolation
         and CSV appends included -- one process per core on row bands, on a bounded sample of C2;
         without a copy of the reference, the NumPy oracle, reported as kind "port".
  --dump-outputs DIR  the statistics and the glacier cells of the final state rasters of the headline's
         last timed pass as .npy files (dump_outputs); the inputs are seeded, so two builds can be
         compared output for output
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CELLS = 2048
N_STEPS = 2200
# Algorithmic work per glacier cell-step.  SURVEY.md 8(d): energy-balance core 93 FLOP (+ 2 exp, not
# counted) + 12 FLOP per insolation sub-step; C2 has 4 sub-steps per step -> 141 FLOP.  That is the
# REFERENCE's arithmetic after hoisting per-cell invariants; the kernel executes less (DESIGN.md 4.1:
# ez = e, exp(0) = 1, one reciprocal per quantity, analytic longwave sum, daily albedo blend, flux
# scalars folded into the balance FMA chain).  Counted in the SASS of the hot basic block (insolation +
# balance + statistics of one step for the 8 cells of a thread, profiles/r02_sass.txt: 373 instructions,
# of them FFMA2 96, FADD2 50, FMUL2 36, scalar FMUL 8, FADD 8): (96 x 4 + 50 x 2 + 36 x 2 + 16) / 8 = 71.5
# FLOP, (182 x 2 + 16) / 8 = 47.5 FP32-pipe lane-operations and 373 / 8 = 46.6 issue slots per cell-step
# (rows that take the analytic direct-beam path execute 40 packed instructions fewer, not credited here).
# Both are reported; `roofline.frac` uses the SURVEY figure as the contract asks.
FLOP_PER_CELL_STEP = 141.0
FLOP_EXECUTED_PER_CELL_STEP = 71.5
FP32_PIPE_OPS_PER_CELL_STEP = 47.5       # lane-operations on the FMA pipe (a packed FFMA2 is two)
ISSUE_SLOTS_PER_CELL_STEP = 46.6         # thread-instructions of the hot block per cell-step
# Shading sweep (shade.cu), per terrain cell and sunlit sub-step: 4 B of terrain read + 1 bit of mask
# written; executed thread-instructions from the SASS of the sweep loop (DESIGN.md 4.2)
SWEEP_BYTES_PER_CELL_SUB = 4.0 + 1.0 / 8.0
SWEEP_SLOTS_PER_CELL_SUB = 11.0
METRIC = "cell-timesteps/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


_JSON_FD = None


def claim_stdout():
    """Keeps fd 1 for the ONE JSON line: everything else written to stdout by this process or by
    native libraries (NCCL prints its version banner there) is sent to stderr."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML during the timed region."""

    def __init__(self, index, period=0.05):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:          # pragma: no cover
            log("clock sampler unavailable:", e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------
class Ctx:
    """Process-wide bits every leg needs."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            log("warning: WORLD_SIZE=%d but --gpus=%d; using WORLD_SIZE" % (self.world, args.gpus))
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.stream = torch.cuda.Stream()
        peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
        self.hbm_peak = json.load(open(peaks_file))["hbm_gbs"] if os.path.isfile(peaks_file) else 6650.0
        self.hbm_source = "MEASURED_PEAKS.json" if os.path.isfile(peaks_file) else "fallback (B200_PROFILING.md)"

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, values):
        """[world][len(values)] list of per-rank numbers on every rank."""
        t = self.torch.tensor([float(v) for v in values], dtype=self.torch.float64, device="cuda")
        if self.world == 1:
            return [t.cpu().tolist()]
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [o.cpu().tolist() for o in out]

    def timed(self, one_pass, warmup, steps):
        """`steps` passes after `warmup`, CUDA events on the launching stream, barrier + synchronize on
        both sides, max over ranks: ms per pass."""
        torch = self.torch
        for _ in range(warmup):
            one_pass()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            one_pass()
        e1.record(self.stream)
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps


def build_engine(case, dem_full, precision, device, shadow=False):
    from enrgy_b200 import _lib
    from enrgy_b200.engine import Engine
    from enrgy_b200.forcing import build_forcing
    m = case.meta
    eng = Engine(m["rows_full"], case.dem.shape[1], precision=precision, device=device)
    eng.set_params(cell_size=case.cell, elev_aws=case.elev_aws, aws_row=case.aws_rc[0],
                   aws_col=case.aws_rc[1], sensor_z=1.6, zm=1e-3, z_h_or_e=1e-4, emissivity=0.98,
                   insol_mode=_lib.INSOL_COMPUTED, shadow=shadow, lat=case.lat, lon=case.lon,
                   band_row0=m["band_row0"], band_rows=case.dem.shape[0])
    keys = list(case.albedo_maps)
    table = build_forcing(case.aws_rows, keys)
    upload(eng, case, dem_full, table)
    return eng, table


def upload(eng, case, dem_full, table, pinned=None):
    """Everything a user's Energy.model() call moves to the device, from (pinned) host memory."""
    src = pinned if pinned is not None else {
        "dem": dem_full, "swe": case.swe, "alb": [case.albedo_maps[k] for k in case.albedo_maps]}
    eng.set_dem(src["dem"])
    eng.set_forcing(table)            # the host pre-pass starts here and overlaps the raster uploads
    eng.set_albedo_maps(src["alb"])
    eng.set_swe(src["swe"])
    eng.prepass()


def pin(arr):
    import torch
    t = torch.empty(arr.shape, dtype=torch.float32, pin_memory=True)
    t.numpy()[...] = arr
    return t


# ---------------------------------------------------------------------------------------------
def bench_c2(ctx, args, dtype, headline):
    """C2 (weak scaling over row bands).  headline: clocks, e2e, launch count, pipe peaks."""
    torch, dist = ctx.torch, ctx.dist
    from enrgy_b200 import _lib
    from enrgy_b200._lib import check
    from enrgy_b200.synthetic import make_band_case
    n, T, world = args.n, args.t, ctx.world
    case, dem_full = make_band_case(n, T, world=world, rank=ctx.rank)
    precision = _lib.F32 if dtype == "f32" else _lib.F64
    t_setup = time.time()
    eng, table = build_engine(case, dem_full, precision, ctx.local_rank)
    eng.set_stream(ctx.stream.cuda_stream)
    stats = torch.zeros((T, _lib.S_COUNT), dtype=torch.float64, device="cuda")
    eng.snapshot(save=True)

    def one_pass():
        eng.snapshot(save=False)                       # rewind the season (device-to-device)
        eng.run_async(0, T, stats.data_ptr(), None)    # fused kernel + statistics finalize
        if world > 1:
            with torch.cuda.stream(ctx.stream):
                dist.all_reduce(stats)                 # glacier-wide sums (NCCL)

    one_pass()
    ctx.barrier()
    log("rank %d: C2 %s setup %.1f s, kernel %s" % (ctx.rank, dtype, time.time() - t_setup, eng.kernel_info()))
    steps = args.steps if headline else max(3, min(args.steps, 6))
    sampler = None
    if headline:
        sampler = ClockSampler(ctx.local_rank, period=0.02)
        for _ in range(max(args.warmup - 1, 0)):
            one_pass()
        ctx.barrier()
        sampler.start()
        l0 = eng.launch_count()
        ms_step = ctx.timed(one_pass, 0, steps)
        clocks = sampler.stop()
        launches = eng.launch_count() - l0 + (steps if world > 1 else 0)
    else:
        ms_step = ctx.timed(one_pass, max(args.warmup - 1, 2), steps)
        clocks, launches = None, None
    kernel_ms = eng.last_kernel_ms()                   # fused kernel alone, last pass
    cell_steps = float(n) * n * world * T
    value = cell_steps / (ms_step * 1e-3)
    stats_host = stats.cpu().numpy()
    if headline and args.dump_outputs and ctx.rank == 0:
        # before the e2e leg below, which uploads and runs the season again
        dump_outputs(args.dump_outputs, stats_host, eng.state(np.float32 if precision == _lib.F32 else np.float64),
                     ~np.isnan(case.dem))
    n_valid = float(np.count_nonzero(~np.isnan(case.dem)))
    bytes_per_launch = algorithmic_bytes(case, precision)
    peak = eng.microbench(0 if dtype == "f32" else 1) if ctx.rank == 0 else None
    out = {"value": value, "ms_per_step": ms_step, "kernel_ms": kernel_ms, "steps": steps, "dtype": dtype,
           "kernel": eng.kernel_info(), "band_rows": [b[1] for b in case.meta["bands"]],
           "check": {"mean_melt_flux_last_step": float(stats_host[-1, _lib.S_MELT] / stats_host[-1, _lib.S_NVALID])}}
    if ctx.rank == 0:
        achieved = FLOP_PER_CELL_STEP * n_valid * T / (kernel_ms * 1e-3) / 1e12
        executed = FLOP_EXECUTED_PER_CELL_STEP * n_valid * T / (kernel_ms * 1e-3) / 1e12
        out["roofline"] = {
            "bound": "fp32" if dtype == "f32" else "fp64",
            "bound_note": "no dense contraction and 0.03 B of HBM traffic per cell-step: neither 'tensor' nor 'hbm' binds; the FP32 (FP64) pipe does",
            "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
            "traffic": measured_traffic(dtype),
            "peak_source": "enrgy_microbench FMA loop on this GPU (MEASURED_PEAKS.json has no FP32/FP64 pipe peak)",
            "flop_per_cell_step": FLOP_PER_CELL_STEP, "kernel_ms": kernel_ms,
            "flop_source": "SURVEY.md 8(d): 93 (core) + 4 x 12 (insolation sub-steps), glacier cells only",
            "as_executed": {"flop_per_cell_step": FLOP_EXECUTED_PER_CELL_STEP, "achieved": executed,
                            "frac": executed / peak if peak else None},
            "glacier_cell_fraction": n_valid / float(case.dem.size),
            "hbm": {"achieved": bytes_per_launch / (kernel_ms * 1e-3) / 1e9, "peak": ctx.hbm_peak, "unit": "GB/s",
                    "frac": bytes_per_launch / (kernel_ms * 1e-3) / 1e9 / ctx.hbm_peak, "peak_source": ctx.hbm_source},
        }
        if clocks is not None:
            out["roofline"]["pipes"] = issue_roofline(n_valid * T, kernel_ms, clocks, dtype)
    if headline:
        # ---- end to end through the public API from pinned host buffers -----------------------
        pinned_t = {"dem": pin(dem_full), "swe": pin(case.swe), "alb": [pin(case.albedo_maps[k]) for k in case.albedo_maps]}
        pinned = {"dem": pinned_t["dem"].numpy(), "swe": pinned_t["swe"].numpy(), "alb": [t.numpy() for t in pinned_t["alb"]]}
        out_state = [torch.empty(case.dem.shape, dtype=torch.float32, pin_memory=True) for _ in range(3)]
        stats_h = torch.empty((T, _lib.S_COUNT), dtype=torch.float64, pin_memory=True)

        def e2e_pass():
            upload(eng, case, dem_full, table, pinned)
            check(eng.lib.enrgy_run(eng.h, 0, T, stats_h.numpy().ctypes.data))
            check(eng.lib.enrgy_get_state(eng.h, 32, *[o.numpy().ctypes.data for o in out_state]))
            if world > 1:
                g = stats_h.cuda(non_blocking=True)
                dist.all_reduce(g)
                stats_h.copy_(g)
        eng.set_stream(None)
        e2e_steps = max(1, min(args.steps, 5))
        e2e_pass()
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_pass()
        ctx.barrier()
        e2e_s = ctx.max_over_ranks((time.perf_counter() - t0) / e2e_steps)
        m = case.meta
        # without shading only the band of the DEM (+ one row either side) goes up
        dem_rows_up = min(dem_full.shape[0], m["band_row0"] + case.dem.shape[0] + 1) - max(0, m["band_row0"] - 1)
        h2d = dem_rows_up * dem_full.shape[1] * 4 + case.swe.nbytes + sum(a.nbytes for a in case.albedo_maps.values()) + table.nbytes
        d2h = 3 * case.dem.size * 4 + stats_h.numel() * 8
        out["e2e"] = {"value": cell_steps / e2e_s, "unit": "cell-timesteps/s", "h2d_bytes_per_step": int(h2d),
                      "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_s * 1e3, "steps": e2e_steps}
        out["clocks"] = clocks
        out["gpu_launches"] = int(launches)
        out["bytes_per_launch"] = bytes_per_launch
    eng.close()
    return out


def bench_c3(ctx, args):
    """C3: fixed 8192 x 8192 raster with shading, strong scaling over N row bands."""
    torch, dist = ctx.torch, ctx.dist
    from enrgy_b200 import _lib
    from enrgy_b200.parallel import ShardedShading
    from enrgy_b200.synthetic import make_band_case
    n, T, world = args.c3_n, args.c3_t, ctx.world
    t_setup = time.time()
    case, dem_full = make_band_case(n, T, world=world, rank=ctx.rank, rows_full=n)
    eng, table = build_engine(case, dem_full, _lib.F32, ctx.local_rank, shadow=True)
    eng.set_stream(ctx.stream.cuda_stream)
    stats = torch.zeros((T, _lib.S_COUNT), dtype=torch.float64, device="cuda")
    eng.snapshot(save=True)
    sub_counts = eng.point_scalars()[:, _lib.P_NSUB].astype(int)
    sh = ShardedShading(eng, case.meta["bands"], ctx.rank, world, exchange=os.environ.get("ENRGY_SHADE_EXCHANGE") or None)

    def one_pass():
        eng.snapshot(save=False)
        sh.run(0, T, stats.data_ptr(), ctx.stream, sub_counts)      # sweep (1/N of the sub-steps) -> all-to-all -> fused
        if world > 1:
            with torch.cuda.stream(ctx.stream):
                dist.all_reduce(stats)

    one_pass()
    ctx.barrier()
    log("rank %d: C3 setup %.1f s, kernel %s" % (ctx.rank, time.time() - t_setup, eng.kernel_info()))
    steps = max(3, min(args.steps, 5))
    ms_step = ctx.timed(one_pass, 2, steps)
    per_rank = ctx.gather([eng.last_sweep_ms(), eng.last_kernel_ms(), case.dem.shape[0]])
    n_sub = int(sub_counts.sum())
    cell_steps = float(n) * n * T
    out = {"value": cell_steps / (ms_step * 1e-3), "unit": "cell-timesteps/s", "scaling": "strong", "ms_per_step": ms_step,
           "steps": steps, "dtype": "f32",
           "workload": "C3: %dx%d 10 m synthetic DEM + 5 albedo maps (fixed), %d hourly steps, %d sunlit sub-steps with "
                       "topographic shading; %d row bands" % (n, n, T, n_sub, world),
           "sweep_ms_per_rank": [p[0] for p in per_rank], "fused_ms_per_rank": [p[1] for p in per_rank],
           "band_rows": [int(p[2]) for p in per_rank],
           "exchange": sh.exchange, "exchange_bytes_per_pass_per_rank": int(sh.bytes_sent_last_run),
           "chunks_per_pass": len(sh.chunks(0, T, sub_counts)), "sub_steps": n_sub,
           "per_rank_times": "sweep / fused kernel time of the LAST chunk of a pass (%d sub-steps swept by rank 0)" % sh.subs_last_scan,
           "check": {"melt_flux_sum_W_m2_cells": float(stats.cpu().numpy()[:, _lib.S_MELT].sum())}}
    if ctx.rank == 0:
        sweep_ms = max(p[0] for p in per_rank)
        mhz = 1965.0
        swept = float(n) * n * sh.subs_last_scan        # cell-sub-steps of the scan that sweep_ms times (the last chunk's)
        out["roofline_sweep"] = {
            "bound": "issue", "kernel_ms": sweep_ms,
            "issue_slots": {"achieved": SWEEP_SLOTS_PER_CELL_SUB * swept / (sweep_ms * 1e-3) / 1e12,
                            "peak": 148 * 128 * mhz * 1e6 / 1e12, "unit": "Tera thread-instr/s",
                            "slots_per_cell_sub_step": SWEEP_SLOTS_PER_CELL_SUB},
            "hbm": {"achieved": SWEEP_BYTES_PER_CELL_SUB * swept / (sweep_ms * 1e-3) / 1e9, "peak": ctx.hbm_peak, "unit": "GB/s",
                    "bytes_per_cell_sub_step": SWEEP_BYTES_PER_CELL_SUB,
                    "note": "algorithmic bytes (terrain read once per sub-step + mask bit); concurrent sub-steps share the terrain rows in L2/L1, so DRAM traffic is far lower"},
        }
        r = out["roofline_sweep"]
        r["issue_slots"]["frac"] = r["issue_slots"]["achieved"] / r["issue_slots"]["peak"]
        r["hbm"]["frac"] = r["hbm"]["achieved"] / r["hbm"]["peak"]
    eng.close()
    del sh
    torch.cuda.empty_cache()
    return out


def bench_c5(ctx, args):
    """C5: parameter ensemble (albedo offset, roughness lengths), 8 members per GPU on 4096 x 4096."""
    from enrgy_b200 import _lib
    from enrgy_b200.ensemble import make_members, run_members, shard
    from enrgy_b200.synthetic import make_band_case
    n, T, world = args.c5_n, args.t, ctx.world
    per_gpu = args.c5_members
    case, dem_full = make_band_case(n, T, world=1, rank=0)
    eng, _ = build_engine(case, dem_full, _lib.F32, ctx.local_rank)
    members = make_members(per_gpu * world, seed=0)
    mine = shard(members, world, ctx.rank)
    # three ways to run this rank's members, same inputs: one pass of the kernel per member; fused passes
    # (four members per pass share terrain, insolation, meteorology, net longwave) with the per-step
    # statistics of every member; fused passes without them (season totals from the final rasters)
    out = {}
    for name, kw in (("one_pass_per_member", dict(fused=False)), ("fused_with_step_statistics", dict(fused=True)),
                     ("fused", dict(fused=True, want_stats=False))):
        run_members(eng, members, mine, **kw)            # warm-up (the same kernels, buffers and tables)
        ctx.barrier()
        t0 = time.perf_counter()
        res = run_members(eng, members, mine, **kw)
        ctx.torch.cuda.synchronize()
        wall = ctx.max_over_ranks(time.perf_counter() - t0)
        out[name] = {"seconds": wall, "value": float(n) * n * T * per_gpu * world / wall,
                     "mean_ice_melt_range_m": [float(min(res[i]["mean_ice"] for i in mine)), float(max(res[i]["mean_ice"] for i in mine))]}
    eng.close()
    best = out["fused"]
    return {"value": best["value"], "unit": "member-cell-timesteps/s", "scaling": "weak",
            "members": per_gpu * world, "members_per_gpu": per_gpu, "seconds": best["seconds"],
            "workload": "C5: %d members (albedo offset N(0, 0.03), zm log-uniform) x %dx%d x %d hourly steps, member axis "
                        "sharded over %d GPUs; DEM, terrain, albedo maps and forcing stay resident; four members per pass "
                        "of the fused kernel (enrgy_run_members), season totals from the final rasters"
                        % (per_gpu * world, n, n, T, world),
            "timing": "wall clock around all members incl. the host pre-pass of each and the download of the totals, max over ranks",
            "variants": out, "mean_ice_melt_range_m": best["mean_ice_melt_range_m"]}


def bench_c4(ctx, args):
    """C4: 4096 x 4096 per GPU, 15-minute rows, three extra weather stations blended per cell and
    Beer-Lambert cloud attenuation of the shortwave (enrgy_set_stations); weak scaling over row bands."""
    torch, dist = ctx.torch, ctx.dist
    from enrgy_b200 import _lib
    from enrgy_b200.forcing import build_station_series
    from enrgy_b200.synthetic import make_band_case, make_station_rows
    n, T, world = args.c4_n, args.c4_t, ctx.world
    # (the library takes rasters up to 32767 rows: the Q16 shear of the shading sweep is int32 arithmetic;
    # eight bands of 4096 rows are cut from 32752)
    rows_total = min(n * world, 32767 // 16 * 16)
    case, dem_full = make_band_case(n, T, world=world, rank=ctx.rank, step_s=900, rows_full=rows_total)
    eng, _ = build_engine(case, dem_full, _lib.F32, ctx.local_rank)
    rows_full = case.meta["rows_full"]
    spots = [(0.2 * rows_full, 0.3 * n, 150.0, 41), (0.75 * rows_full, 0.7 * n, -80.0, 42), (0.5 * rows_full, 0.9 * n, 60.0, 43)]
    eng.set_stations([(r, c, case.elev_aws + dz) for (r, c, dz, _) in spots],
                     [build_station_series(make_station_rows(case, case.elev_aws + dz, seed=sd)) for (_, _, dz, sd) in spots],
                     cloud_k=0.7)
    eng.prepass()
    eng.set_stream(ctx.stream.cuda_stream)
    stats = torch.zeros((T, _lib.S_COUNT), dtype=torch.float64, device="cuda")
    eng.snapshot(save=True)

    def one_pass():
        eng.snapshot(save=False)
        eng.run_async(0, T, stats.data_ptr(), None)
        if world > 1:
            with torch.cuda.stream(ctx.stream):
                dist.all_reduce(stats)

    ms_step = ctx.timed(one_pass, 2, max(3, min(args.steps, 5)))
    kernel_ms = eng.last_kernel_ms()
    info = eng.kernel_info()
    st = stats.cpu().numpy()
    eng.close()
    return {"value": float(rows_full) * n * T / (ms_step * 1e-3), "unit": "cell-timesteps/s", "scaling": "weak",
            "ms_per_step": ms_step, "kernel_ms": kernel_ms, "dtype": "f32", "kernel": info,
            "raster": [int(rows_full), int(n)],
            "workload": "C4: %dx%d per GPU (%d row bands), %d rows of 15 minutes, the AWS + 3 extra weather stations blended "
                        "per cell (inverse squared distance, lapse-rate reduction), Beer-Lambert cloud attenuation k = 0.7, "
                        "in-kernel insolation (one sun position per row), no shading" % (n, n, world, T),
            "check": {"mean_melt_flux_last_step": float(st[-1, _lib.S_MELT] / st[-1, _lib.S_NVALID])}}


def run_ours(args):
    claim_stdout()
    ctx = Ctx(args)
    head = bench_c2(ctx, args, args.dtype, headline=True)
    configs = {}
    if args.configs:
        other = "f64" if args.dtype == "f32" else "f32"
        for name, fn in (("c2_" + other, lambda: bench_c2(ctx, args, other, headline=False)),
                         ("c3_shadow", lambda: bench_c3(ctx, args)),
                         ("c4_stations", lambda: bench_c4(ctx, args)),
                         ("c5", lambda: bench_c5(ctx, args))):
            if args.only is not None and name != args.only:
                continue
            try:
                t0 = time.time()
                configs[name] = fn()
                configs[name]["bench_seconds"] = time.time() - t0
            except Exception as e:                      # a side config must never take the headline down
                import traceback
                traceback.print_exc(file=sys.stderr)
                configs[name] = {"error": "%s: %s" % (type(e).__name__, e)}
                ctx.torch.cuda.synchronize()
    result = None
    if ctx.rank == 0:
        n, T, world = args.n, args.t, ctx.world
        result = {
            "metric": METRIC, "value": head["value"], "unit": "cell-timesteps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": "C2: %dx%d 10 m synthetic DEM + 5 albedo maps per GPU, %d hourly steps, "
                                   "in-kernel insolation (4 sub-steps/step), no shading" % (n, n, T),
                       "raster": [n * world, n], "steps_per_pass": T, "parallelism": "row bands x%d, balanced by visited tiles" % world,
                       "band_rows": head["band_rows"],
                       "l2": "per-pass inputs ~%.0f MB > 126 MB L2, no flush" % (head["bytes_per_launch"] / 1e6)},
            "roofline": head["roofline"],
            "e2e": head["e2e"],
            "gpu_launches": head["gpu_launches"],
            "clocks": head["clocks"],
            "kernel": head["kernel"],
            "check": head["check"],
            "configs": configs,
        }
        if args.cpu_baseline and world == 1:
            result["cpu_baseline"] = cpu_baseline(n, args.cpu_sample_steps, cores=1)
    if ctx.world > 1:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()
    if ctx.rank == 0:
        emit(result)


DUMP_BYTES = 64 * 10 ** 6
DUMP_SEED = 0


def dump_outputs(path, stats, state, valid):
    """--dump-outputs: what the last timed pass hands its caller, as <path>/<name>.npy -- the per-step
    area statistics (float64 [T, S_COUNT], all-reduced over ranks) and rank 0's final swe, total_snow and
    total_ice rasters in the run's precision, at the glacier cells `valid` only (ascending cell index):
    off the glacier the rasters are NaN by definition (model.py:258), and the DEM alone decides where.
    Cells that would take the files over DUMP_BYTES are cut to the same seeded sample in every raster,
    so two builds can be compared file by file."""
    os.makedirs(path, exist_ok=True)
    state = [a[valid] for a in state]
    cells = state[0].size
    room = (DUMP_BYTES - stats.nbytes - 4096) // (len(state) * state[0].itemsize)     # (4096: .npy headers)
    if room < 1:
        raise ValueError("--dump-outputs: the statistics alone (%d bytes) fill the %d-byte budget" % (stats.nbytes, DUMP_BYTES))
    idx = None
    if cells > room:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(cells, room, replace=False))
    np.save(os.path.join(path, "stats.npy"), stats)
    for name, a in zip(("swe", "total_snow", "total_ice"), state):
        np.save(os.path.join(path, name + ".npy"), a if idx is None else a[idx])
    log("outputs of the last timed pass written to %s%s" % (path, "" if idx is None else " (%d of %d cells)" % (room, cells)))


def issue_roofline(cell_steps, kernel_ms, clocks, dtype):
    """The binding resources of the fused kernel (ncu: DRAM < 1 %): FP32-pipe lane-operations per
    second against 128 lanes x SMs x clock, and instruction issue slots against 4 schedulers x 32
    lanes x SMs x clock, both at the SM clock sampled during the run.  float32 figures (the packed
    path); float64 runs the same algorithm on the FP64 pipe (64 lanes per SM)."""
    mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
    lanes = 128 if dtype == "f32" else 64
    peak = 148 * lanes * mhz * 1e6 / 1e12
    pipe = FP32_PIPE_OPS_PER_CELL_STEP * cell_steps / (kernel_ms * 1e-3) / 1e12
    slots = ISSUE_SLOTS_PER_CELL_STEP * cell_steps / (kernel_ms * 1e-3) / 1e12
    issue_peak = 148 * 128 * mhz * 1e6 / 1e12
    return {"fp_pipe": {"achieved": pipe, "peak": peak, "unit": "Tera lane-ops/s", "frac": pipe / peak,
                        "ops_per_cell_step": FP32_PIPE_OPS_PER_CELL_STEP},
            "issue_slots": {"achieved": slots, "peak": issue_peak, "unit": "Tera thread-instr/s", "frac": slots / issue_peak,
                            "slots_per_cell_step": ISSUE_SLOTS_PER_CELL_STEP,
                            "note": "float32: two cells per packed instruction (FFMA2/FADD2/FMUL2)"},
            "sm_mhz": mhz}


def measured_traffic(dtype):
    """dram__bytes_read.sum + dram__bytes_write.sum of the fused kernel for this workload, from the
    committed ncu --set full capture (profiles/*_traffic.json, newest round), or None."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")), reverse=True):
        v = json.load(open(path)).get(dtype)
        if v is not None:
            return v
    return None


def algorithmic_bytes(case, precision):
    """HBM bytes one pass has to move: DEM + 3 normals + 5 albedo maps + 3 state rasters in and 3 out."""
    cells = case.dem.size
    r = 4 if precision == 32 else 8
    return cells * (4 + 3 * r + 5 * 4 + 3 * r + 3 * r)


# ---------------------------------------------------------------------------------------------
# CPU arm: the unmodified reference (oracle/_ref) through oracle/ref_harness.py, or -- if that copy
# is absent -- the NumPy oracle (a restatement pinned bit-identically against the reference).
_SAMPLE = {}


def cpu_sample(n, steps):
    """The C2 raster with the insolation rasters of its first `steps` rows (computed once per process
    by the insolation oracle: the reference itself cannot compute them, SURVEY F2)."""
    key = (n, steps)
    if key not in _SAMPLE:
        from enrgy_b200.synthetic import make_band_case
        from oracle import insolation_oracle as I
        from oracle.enrgy_oracle import time_step_seconds
        case, dem_full = make_band_case(n, steps, world=1, rank=0)
        normals = I.terrain_normals(case.dem, case.cell)
        pot = np.empty((steps,) + case.dem.shape, dtype=np.float32)
        for i, row in enumerate(case.aws_rows):
            pot[i] = I.potential_insolation(case.dem, case.cell, case.lat, case.lon, I.to_unix(row["DATE"]),
                                            time_step_seconds(case.aws_rows, i), shadow=False, normals=normals)
        _SAMPLE[key] = (case, pot)
    return _SAMPLE[key]


def _cpu_band(job):
    """One process: the CPU implementation on a row band of the sample (cells are independent given
    the AWS-cell scalars; every band carries the AWS cell's row in front so the point sampling of
    raster_utils.py:85-89 sees the same cell).  Returns the seconds of the model run."""
    import dataclasses
    kind, case, pot, sl = job
    ar = case.aws_rc[0]
    if sl is not None:
        def band(a):
            return np.concatenate([a[ar:ar + 1], a[sl]], axis=0)
        gt = list(case.geotransform)
        gt[3] = case.xy_aws[1] + 0.5 * case.cell          # the AWS row becomes row 0 of the band
        case = dataclasses.replace(case, dem=band(case.dem), geotransform=tuple(gt), swe=band(case.swe),
                                   albedo_maps={k: band(a) for k, a in case.albedo_maps.items()},
                                   aws_rc=(0, case.aws_rc[1]))
        pot = np.concatenate([pot[:, ar:ar + 1], pot[:, sl]], axis=1)
    if kind == "reference":
        from oracle import ref_harness
        r = ref_harness.run_reference(case, pot, f64=False, z=1.6, zm=1e-3, z_h_or_e=1e-4, emissivity=0.98,
                                      keep_steps=(), res=10)
        return r["model_seconds"]
    from oracle import enrgy_oracle as O
    alb = {}
    for k, a in case.albedo_maps.items():
        a = a.copy(); a[a < 0] = 0.001; a[a > 1] = 1
        alb[k] = a
    cfg = O.ModelConfig(z=1.6, elev_aws=case.elev_aws, xy_aws=case.xy_aws, zm=1e-3, z_h_or_e=1e-4, emissivity=0.98)
    t0 = time.perf_counter()
    O.run_model(case.dem, case.geotransform, case.aws_rows, pot, cfg, swe=case.swe, albedo_arrays=alb,
                state_dtype=np.float32)
    return time.perf_counter() - t0


def cpu_baseline(n, steps, cores):
    """Times the CPU path on a bounded sample: the C2 raster for the first `steps` hourly rows.
    kind "reference": the unmodified reference's Energy.model (model.py:155-286), its per-step np.load
    of the insolation raster (model.py:481, files on the box's /tmp) and CSV appends included."""
    import multiprocessing as mp
    from oracle import ref_harness
    kind = "reference" if ref_harness.reference_available() else "port"
    case, pot = cpu_sample(n, steps)
    rows_total = case.dem.shape[0]
    if cores <= 1:
        jobs = [(kind, case, pot, None)]
    else:
        edges = np.linspace(0, rows_total, cores + 1).astype(int)
        jobs = [(kind, case, pot, slice(edges[b], edges[b + 1])) for b in range(cores)]
    t0 = time.perf_counter()
    if cores <= 1:
        secs = [_cpu_band(jobs[0])]
    else:
        with mp.get_context("fork").Pool(cores) as pool:
            secs = pool.map(_cpu_band, jobs)
    wall = time.perf_counter() - t0
    model_s = max(secs)                                  # the slowest process bounds the job
    cell_steps = float(rows_total) * case.dem.shape[1] * steps
    return {"value": cell_steps / model_s, "unit": "cell-timesteps/s", "cores": cores, "kind": kind,
            "sample": "%dx%d raster, first %d hourly rows of the season, float32 as shipped; %s; %.1f s in Energy.model "
                      "(slowest of %d processes), %.1f s wall with start-up and writing the insolation files"
                      % (rows_total, case.dem.shape[1], steps,
                         "unmodified reference incl. per-step np.load + CSV appends" if kind == "reference"
                         else "NumPy port (oracle/enrgy_oracle.py), insolation in memory", model_s, cores, wall),
            "model_seconds": model_s}


def run_reference(args):
    """--impl reference: the CPU path on all host cores (rank 0 only).  A "step" of this arm is one
    run of the bounded sample; value = cell-timesteps/s of the sample."""
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n, T = args.n, args.t
    vals, secs = [], []
    last = None
    cpu_sample(n, args.cpu_sample_steps)                 # (untimed: building the sample)
    for _ in range(args.warmup + args.steps):
        last = cpu_baseline(n, args.cpu_sample_steps, cores)
        vals.append(last["value"])
        secs.append(last["model_seconds"])
    n_warm = args.warmup
    timed, tsecs = vals[n_warm:], secs[n_warm:]
    value = float(np.mean(timed))
    one = cpu_baseline(n, args.cpu_sample_steps, 1) if args.single_core else None
    cb = dict(last)
    cb["value"] = value
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "cell-timesteps/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": len(timed), "warmup": n_warm,
        "ms_per_step": float(np.mean(tsecs)) * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C2: %dx%d 10 m synthetic DEM + 5 albedo maps, %d hourly steps; each step of this arm is the "
                               "bounded sample: the first %d rows" % (n, n, T, args.cpu_sample_steps),
                   "sample_cell_steps": float(n) * n * args.cpu_sample_steps},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "cell-timesteps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if one is not None:
        out["cpu_single_process"] = one
    emit(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--n", type=int, default=N_CELLS, help="raster edge per GPU")
    ap.add_argument("--t", type=int, default=N_STEPS, help="AWS rows per pass")
    ap.add_argument("--cpu-sample-steps", type=int, default=24)
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-configs", dest="configs", action="store_false", help="headline only")
    ap.add_argument("--no-single-core", dest="single_core", action="store_false")
    ap.add_argument("--only", default=None, help="run the headline and only this side config (c2_f64, c3_shadow, c4_stations, c5)")
    ap.add_argument("--c3-n", type=int, default=8192)
    ap.add_argument("--c3-t", type=int, default=1536)
    ap.add_argument("--c4-n", type=int, default=4096)
    ap.add_argument("--c4-t", type=int, default=2200)
    ap.add_argument("--c5-n", type=int, default=4096)
    ap.add_argument("--c5-members", type=int, default=8, help="ensemble members per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the statistics and state rasters of the last timed pass as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        log("note: the timing rules ask for >= 3 warm-up passes")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
