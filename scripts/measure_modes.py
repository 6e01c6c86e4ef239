#!/usr/bin/env python
"""Side measurements for profiles/: streamed-insolation mode, sub-surface model, strong scaling of
the shading path on a fixed raster.  Not part of the bench contract.

  python scripts/measure_modes.py streamed|msm
  python scripts/measure_modes.py msm --stations 3 [--no-msm]    (the station blend of bench.py's C4)
  torchrun ... scripts/measure_modes.py strong --n 8192 --t 96
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from enrgy_b200 import _lib                                   # noqa: E402
from enrgy_b200.engine import Engine                          # noqa: E402
from enrgy_b200.forcing import build_forcing                  # noqa: E402
from enrgy_b200.parallel import row_bands                     # noqa: E402
from enrgy_b200.synthetic import make_band_case, make_dem, make_albedo_maps, make_aws_rows  # noqa: E402


def timed(eng, t, passes=3):
    eng.snapshot(save=True)
    best = 1e30
    for _ in range(passes + 1):
        eng.snapshot(save=False)
        eng.run(0, t, want_stats=False)
        best = min(best, eng.last_kernel_ms())
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=["streamed", "msm", "strong", "ensemble"])
    ap.add_argument("--members", type=int, default=8)
    ap.add_argument("--size", dest="n", type=int, default=2048)
    ap.add_argument("--nsteps", dest="t", type=int, default=256)
    ap.add_argument("--dtype", default="f32")
    ap.add_argument("--sequential", action="store_true", help="ensemble: one run per member instead of fused passes")
    ap.add_argument("--shadow", action="store_true", help="ensemble: with topographic shading")
    ap.add_argument("--nostats", action="store_true", help="ensemble: fused passes without per-step statistics")
    ap.add_argument("--stations", type=int, default=0,
                    help="msm: blend this many extra weather stations (bench.py C4's spots, cloud_k = 0.7)")
    ap.add_argument("--no-msm", action="store_true", help="msm: the same run without the sub-surface model")
    a = ap.parse_args()
    prec = _lib.F32 if a.dtype == "f32" else _lib.F64
    if a.mode == "ensemble":
        # config C5: members share DEM / terrain / maps / forcing on the device; under torchrun the
        # member axis is sharded over the ranks (members are independent: no collective except the
        # gather of the per-member totals)
        from enrgy_b200.ensemble import make_members, run_members, shard
        world = int(os.environ.get("WORLD_SIZE", "1"))
        rank = int(os.environ.get("RANK", "0"))
        local = int(os.environ.get("LOCAL_RANK", "0"))
        if world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        case, dem = make_band_case(a.n, a.t)
        keys = list(case.albedo_maps)
        eng = Engine(a.n, a.n, precision=prec, device=local)
        eng.set_params(cell_size=10.0, elev_aws=case.elev_aws, aws_row=case.aws_rc[0], aws_col=case.aws_rc[1],
                       sensor_z=1.6, zm=1e-3, z_h_or_e=1e-4, emissivity=0.98, lat=case.lat, lon=case.lon,
                       insol_mode=_lib.INSOL_COMPUTED, shadow=a.shadow)
        eng.set_dem(dem)
        eng.set_albedo_maps([case.albedo_maps[k] for k in keys])
        eng.set_swe(case.swe)
        eng.set_forcing(build_forcing(case.aws_rows, keys))
        members = make_members(a.members)
        mine = shard(members, world, rank)
        run_members(eng, members, indices=mine, fused=not a.sequential, want_stats=not a.nostats)   # warm-up (and the sunlit masks)
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()
        t0 = time.perf_counter()
        out = run_members(eng, members, indices=mine, fused=not a.sequential, want_stats=not a.nostats)
        totals = np.zeros(a.members, dtype=np.float64)
        for i, o in out.items():
            totals[i] = o["mean_ice"]
        if world > 1:
            tt = torch.from_numpy(totals).cuda()
            dist.all_reduce(tt)                                      # gather of the per-member totals
            totals = tt.cpu().numpy()
            dist.barrier()
        wall = time.perf_counter() - t0
        cells = float(a.n) * a.n * a.t * a.members
        if rank == 0:
            print(json.dumps({"mode": "ensemble", "fused": not a.sequential, "stats": not a.nostats, "lib": os.path.basename(_lib.LIB_PATH), "shadow": a.shadow, "dtype": a.dtype,
                              "kernel": eng.kernel_info(), "last_kernel_ms": eng.last_kernel_ms(), "last_sweep_ms": eng.last_sweep_ms(),
                              "members": a.members, "gpus": world, "n": a.n, "t": a.t, "wall_s": wall,
                              "member_cell_steps_per_s": cells / wall,
                              "mean_ice_spread": float(np.std(totals))}))
        eng.close()
        if world > 1:
            dist.destroy_process_group()
        return
    if a.mode in ("streamed", "msm"):
        case, dem = make_band_case(a.n, a.t)
        keys = list(case.albedo_maps)
        eng = Engine(a.n, a.n, precision=prec)
        kw = dict(cell_size=10.0, elev_aws=case.elev_aws, aws_row=case.aws_rc[0], aws_col=case.aws_rc[1],
                  sensor_z=1.6, zm=1e-3, z_h_or_e=1e-4, emissivity=0.98, lat=case.lat, lon=case.lon)
        msm = a.mode == "msm" and not a.no_msm
        if a.mode == "streamed":
            eng.set_params(insol_mode=_lib.INSOL_STREAMED, **kw)
        else:
            eng.set_params(insol_mode=_lib.INSOL_COMPUTED, msm_depths=[0.1, 0.1, 0.3, 0.5, 0.5, 0.5, 3.0] if msm else None, **kw)
        eng.set_dem(dem)
        if msm:
            eng.set_msm([-6.9, -6.93, -7.025, -7.31, -6.93, -7.12, -7.0, -5.57], 275.0)
        eng.set_albedo_maps([case.albedo_maps[k] for k in keys])
        eng.set_swe(case.swe)
        eng.set_forcing(build_forcing(case.aws_rows, keys))
        if a.mode == "msm" and a.stations > 0:
            from enrgy_b200.forcing import build_station_series
            from enrgy_b200.synthetic import make_station_rows
            spots = [(0.2 * a.n, 0.3 * a.n, 150.0, 41), (0.75 * a.n, 0.7 * a.n, -80.0, 42), (0.5 * a.n, 0.9 * a.n, 60.0, 43)]
            spots = spots[:a.stations]
            eng.set_stations([(r, c, case.elev_aws + dz) for (r, c, dz, _) in spots],
                             [build_station_series(make_station_rows(case, case.elev_aws + dz, seed=sd)) for (_, _, dz, sd) in spots],
                             cloud_k=0.7)
        if a.mode == "streamed":
            rng = np.random.default_rng(0)
            field = (0.6 + 0.4 * rng.random((a.n, a.n))).astype(np.float32)
            field[np.isnan(dem)] = np.nan
            chunk = 32
            # all steps resident: upload in chunks into one window is not supported by the ABI, so
            # the whole [T, H, W] block is built on the host once
            pot = np.empty((a.t, a.n, a.n), dtype=np.float32)
            for i in range(a.t):
                hour = i % 24
                pot[i] = field * max(0.0, 0.3 * np.sin((hour - 4) / 24.0 * 2 * np.pi) + 0.15)
            eng.set_insolation(0, pot)
            del pot
        eng.prepass()
        ms = timed(eng, a.t)
        cells = float(a.n) * a.n * a.t
        print(json.dumps({"mode": a.mode, "msm": msm, "stations": a.stations if a.mode == "msm" else 0,
                          "dtype": a.dtype, "n": a.n, "t": a.t, "kernel_ms": ms,
                          "cell_steps_per_s": cells / (ms * 1e-3), "kernel": eng.kernel_info(),
                          "streamed_GBps": (cells * 0.70 * 4 / (ms * 1e-3) / 1e9) if a.mode == "streamed" else None}))
        eng.close()
        return
    # strong scaling of the shading path: one n x n raster, bands balanced by glacier cells
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dem = make_dem(a.n, a.n, seed=0)
    valid_per_row = (~np.isnan(dem)).sum(axis=1)
    bands = row_bands(a.n, world, align=16, valid_per_row=valid_per_row)
    dates = ["20220520", "20220915"]
    aws = make_aws_rows(a.t)
    r, c = a.n // 2, a.n // 2
    stream = torch.cuda.Stream()
    stats = torch.zeros((a.t, _lib.S_COUNT), dtype=torch.float64, device="cuda")

    def measure(bands):
        """One engine on this rank's band; returns (max-over-ranks ms per pass, this rank's kernel ms)."""
        r0, rows = bands[rank]
        alb = make_albedo_maps(rows, a.n, dates, seed=1, nan_like=dem[r0:r0 + rows], row0=r0)
        eng = Engine(a.n, a.n, precision=prec, device=local)
        eng.set_params(cell_size=10.0, elev_aws=float(dem[r, c]), aws_row=r, aws_col=c, sensor_z=1.6, zm=1e-3,
                       z_h_or_e=1e-4, emissivity=0.98, insol_mode=_lib.INSOL_COMPUTED, shadow=True, lat=77.98,
                       lon=14.1, band_row0=r0, band_rows=rows)
        eng.set_dem(dem)
        eng.set_forcing(build_forcing(aws, dates))
        eng.set_albedo_maps([alb[k] for k in dates])
        eng.prepass()
        eng.set_stream(stream.cuda_stream)
        eng.snapshot(save=True)

        def one():
            eng.snapshot(save=False)
            eng.run_async(0, a.t, stats.data_ptr(), None)
            if world > 1:
                with torch.cuda.stream(stream):
                    dist.all_reduce(stats)
        one()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(2):
            one()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / 2], dtype=torch.float64, device="cuda")
        mine = torch.zeros(world, dtype=torch.float64, device="cuda")
        mine[rank] = eng.last_kernel_ms()
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(mine)
        eng.close()
        return float(ms.item()), mine.cpu().numpy()

    rounds = []
    for it in range(3 if world > 1 else 1):
        ms, per_rank = measure(bands)
        rounds.append({"ms_per_pass": ms, "cell_steps_per_s": float(a.n) * a.n * a.t / (ms * 1e-3),
                       "band_rows": [b[1] for b in bands], "kernel_ms_per_rank": [round(float(x), 2) for x in per_rank]})
        # next round: bands re-cut from the measured kernel times (parallel.rebalance_bands)
        from enrgy_b200.parallel import rebalance_bands
        bands = rebalance_bands(bands, per_rank, valid_per_row, align=16)
    if rank == 0:
        best = min(rounds, key=lambda x: x["ms_per_pass"])
        print(json.dumps({"mode": "strong", "n": a.n, "t": a.t, "gpus": world, "ms_per_pass": best["ms_per_pass"],
                          "cell_steps_per_s": best["cell_steps_per_s"], "band_rows": best["band_rows"],
                          "rounds": rounds}), file=sys.stderr)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
