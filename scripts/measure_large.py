#!/usr/bin/env python
"""Shading-path timings for the large-raster bound, one JSON line per measurement (with the card's name and
power limit read in the same call).

  ab     libraries compared on one square case (default 8192^2, 96 hourly rows, float32, computed insolation
         with shading): the sweep and the mask-fed fused kernel per pass, the libraries alternated --reps
         times, each run in a process of its own (ENRGY_B200_LIB) on inputs generated once;
  large  one large case (default 40 000 x 40 000, 24 hourly rows, constant albedo): cell-steps/s, sweep ms
         per sub-step and the device memory in use at the end of the run (cudaMemGetInfo, whole device).

  python scripts/measure_large.py ab --libs scratch/variants/parent.so enrgy_b200/csrc/libenrgy_b200.so --out profiles/x.jsonl
  python scripts/measure_large.py large --out profiles/y.jsonl"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [s.strip() for s in q.split(",")]
    return dict(gpu=name, power_limit=power)


def emit(rec, out):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(line + "\n")


def one(a):
    """Child of `ab`: one library, inputs from the cache, best of --passes (every pass sweeps afresh)."""
    import numpy as np
    import torch
    from enrgy_b200 import _lib
    from enrgy_b200.engine import Engine
    z = np.load(os.path.join(a.cache, "case.npz"), allow_pickle=True)
    meta = z["meta"].item()
    eng = Engine(a.size, a.size, precision=_lib.F32)
    eng.set_params(cell_size=10.0, elev_aws=meta["elev_aws"], aws_row=meta["aws_rc"][0], aws_col=meta["aws_rc"][1],
                   sensor_z=1.6, zm=1e-3, z_h_or_e=1e-4, emissivity=0.98, lat=meta["lat"], lon=meta["lon"],
                   insol_mode=_lib.INSOL_COMPUTED, shadow=True)
    eng.set_dem(z["dem"])
    eng.set_albedo_maps(list(z["albedo"]))
    eng.set_swe(z["swe"])
    eng.set_forcing(z["forcing"])
    eng.prepass()
    eng.snapshot(save=True)
    s0, s1 = eng.sub_range(0, a.nsteps)
    masks = torch.empty((s1 - s0) * eng.mask_words(a.size), dtype=torch.int32, device="cuda")
    stats = torch.zeros((a.nsteps, _lib.S_COUNT), dtype=torch.float64, device="cuda")
    sweep, fused = [], []
    for _ in range(a.passes):
        eng.snapshot(save=False)
        eng.shade_scan(s0, s1, [(0, a.size, masks.data_ptr())])
        eng.run_masked(0, a.nsteps, masks.data_ptr(), stats.data_ptr())
        eng.synchronize()
        sweep.append(eng.last_sweep_ms())
        fused.append(eng.last_kernel_ms())
    chk = float(np.nansum(stats.cpu().numpy()[:, _lib.S_MELT]))
    eng.close()
    print(json.dumps(dict(sweep_ms=min(sweep), fused_ms=min(fused), subs=s1 - s0, melt_check=chk)))


def ab(a):
    import numpy as np
    from enrgy_b200.forcing import build_forcing
    from enrgy_b200.synthetic import make_band_case
    info = gpu_info()
    with tempfile.TemporaryDirectory() as tmp:
        case, dem = make_band_case(a.size, a.nsteps)
        keys = list(case.albedo_maps)
        np.savez(os.path.join(tmp, "case.npz"), dem=dem, albedo=np.stack([case.albedo_maps[k] for k in keys]),
                 swe=case.swe, forcing=build_forcing(case.aws_rows, keys),
                 meta=np.array(dict(elev_aws=case.elev_aws, aws_rc=case.aws_rc, lat=case.lat, lon=case.lon)))
        del case, dem
        for rep in range(a.reps):
            for lib in a.libs:
                env = dict(os.environ, ENRGY_B200_LIB=os.path.abspath(lib))
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "one", "--cache", tmp, "--size",
                                    str(a.size), "--nsteps", str(a.nsteps), "--passes", str(a.passes)],
                                   env=env, capture_output=True, text=True, check=True)
                rec = json.loads(r.stdout.strip().splitlines()[-1])
                rec.update(mode="ab", lib=os.path.basename(lib), rep=rep, size=a.size, nsteps=a.nsteps, **info)
                emit(rec, a.out)


def large(a):
    import numpy as np
    import torch
    from enrgy_b200 import _lib
    from enrgy_b200.engine import Engine
    from enrgy_b200.forcing import build_forcing
    from enrgy_b200.synthetic import make_aws_rows
    info = gpu_info()
    n = a.size
    free0, total = torch.cuda.mem_get_info()
    dem = np.empty((n, n), dtype=np.float32)
    c = np.arange(n, dtype=np.float32)[None, :]
    for r0 in range(0, n, 2048):
        r = np.arange(r0, min(r0 + 2048, n), dtype=np.float32)[:, None]
        dem[r0:r0 + r.shape[0]] = (800.0 - 600.0 * r / n + 50.0 * np.cos(r / 23.0) * np.sin(c / 17.0)
                                   + 20.0 * np.sin(r / 7.3 + c / 11.0))
    aws = (n // 2, n // 2)
    eng = Engine(n, n, precision=_lib.F32)
    eng.set_params(cell_size=10.0, elev_aws=float(dem[aws]), aws_row=aws[0], aws_col=aws[1], sensor_z=1.6, zm=1e-3,
                   z_h_or_e=1e-4, emissivity=0.98, const_albedo=(0.35, 0.75), insol_mode=_lib.INSOL_COMPUTED,
                   shadow=True, lat=77.98, lon=14.10)
    eng.set_dem(dem)
    eng.set_forcing(build_forcing(make_aws_rows(a.nsteps)))
    eng.prepass()
    eng.snapshot(save=True)
    s0, s1 = eng.sub_range(0, a.nsteps)
    masks = torch.empty((s1 - s0) * eng.mask_words(n), dtype=torch.int32, device="cuda")
    stats = torch.zeros((a.nsteps, _lib.S_COUNT), dtype=torch.float64, device="cuda")
    for p in range(a.passes):
        eng.snapshot(save=False)
        torch.cuda.synchronize()
        t = time.perf_counter()
        eng.shade_scan(s0, s1, [(0, n, masks.data_ptr())])
        eng.run_masked(0, a.nsteps, masks.data_ptr(), stats.data_ptr())
        eng.synchronize()
        wall = time.perf_counter() - t
        sweep, fused = eng.last_sweep_ms(), eng.last_kernel_ms()
        free1, _ = torch.cuda.mem_get_info()
        st = stats.cpu().numpy()
        emit(dict(mode="large", rows=n, cols=n, nsteps=a.nsteps, subs=s1 - s0, pass_=p, wall_s=wall,
                  cell_steps_per_s=float(n) * n * a.nsteps / wall, sweep_ms=sweep, sweep_ms_per_sub=sweep / (s1 - s0),
                  fused_ms=fused, device_mem_in_use_gb=(total - free1) / 1e9,
                  device_mem_in_use_before_gb=(total - free0) / 1e9, finite=bool(np.isfinite(st).all()),
                  melt_check=float(np.nansum(st[:, _lib.S_MELT])), **info), a.out)
    eng.close()


ap = argparse.ArgumentParser()
ap.add_argument("mode", choices=["ab", "one", "large"])
ap.add_argument("--libs", nargs="+", default=[])
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--passes", type=int, default=3)
ap.add_argument("--size", type=int, default=None)
ap.add_argument("--nsteps", type=int, default=None)
ap.add_argument("--cache")
ap.add_argument("--out")
a = ap.parse_args()
if a.size is None:
    a.size = 40000 if a.mode == "large" else 8192
if a.nsteps is None:
    a.nsteps = 24 if a.mode == "large" else 96
{"ab": ab, "one": one, "large": large}[a.mode](a)
