"""CPU-side tests: the C ABI library loads and exports every declared symbol; the host mirror of
the reference's row logic (forcing table) matches the oracle's reading of the same rows."""
import ctypes
import json
import os
import re

import numpy as np
import pytest

from enrgy_b200 import _lib
from enrgy_b200.forcing import build_forcing, get_closest_dates, heuristic_unit_guesser
from enrgy_b200.geo import coords_to_index, utm_to_latlon
from enrgy_b200.synthetic import make_case
from oracle import enrgy_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "enrgy_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(enrgy_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), "libenrgy_b200.so lacks %s" % n
        assert n in _lib.EXPORTED_SYMBOLS, "ctypes binding lacks %s" % n
    assert lib.enrgy_abi_version() == 1


def test_params_struct_layout_matches_header():
    # field order of struct enrgy_params in the header == ctypes Structure
    text = open(os.path.join(ROOT, "include", "enrgy_b200.h")).read()
    body = text[text.index("typedef struct enrgy_params {"):text.index("} enrgy_params;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"\b(?:double|int32_t)\s+([a-z_0-9]+)(?:\[[A-Z_]+\])?;", body)
    assert fields == [f[0] for f in _lib.Params._fields_]
    assert ctypes.sizeof(_lib.Params) % 8 == 0


def test_no_cpu_fallback():
    """Without a CUDA device a context cannot be created -- there is no CPU path behind the ABI."""
    lib = _lib.load()
    if lib.enrgy_device_count() > 0:
        pytest.skip("a GPU is visible")
    h = ctypes.c_void_p()
    rc = lib.enrgy_create(0, 16, 16, 32, ctypes.byref(h))
    assert rc == _lib.ERR_NODEVICE
    assert b"no CPU fallback" in lib.enrgy_last_error()


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "enrgy_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".sh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "from oracle" not in src and "import oracle" not in src, f
                assert "/root/reference" not in src, f
                assert "from tests" not in src and "import tests" not in src, f      # (tests import the oracle)
    # ... and following the imports: loading every module of the package pulls in neither
    import subprocess
    import sys
    code = ("import sys, pkgutil, importlib, enrgy_b200\n"
            "for m in pkgutil.walk_packages(enrgy_b200.__path__, 'enrgy_b200.'):\n"
            "    importlib.import_module(m.name)\n"
            "bad = [k for k in sys.modules if k == 'oracle' or k.startswith('oracle.') or k == 'tests' or k.startswith('tests.')]\n"
            "assert not bad, bad\n")
    subprocess.run([sys.executable, "-c", code], check=True, cwd=ROOT)


def test_forcing_matches_reference_row_logic():
    case = make_case(32, 30, seed=4, calm_every=7, with_gradient=True, step_s=1800)
    keys = list(case.albedo_maps)
    t = build_forcing(case.aws_rows, keys, temp_lapse_rate="GRADIENT", cloud_corr=0.3, last_snowfall="20220530")
    for i, row in enumerate(case.aws_rows):
        assert t[i, _lib.F_DT] == O.time_step_seconds(case.aws_rows, i)
        assert t[i, _lib.F_RH] == O.unit_guess(float(row["HUMID"]), 100)
        assert t[i, _lib.F_CLOUD] == min(1.0, max(0.0, float(row["CLOUDINESS"]) + 0.3))
        assert t[i, _lib.F_LAPSE] == float(row["GRADIENT"])
        d, before, after = O.albedo_bracket(keys, row["DATE"])
        assert keys[int(t[i, _lib.F_ALB_I0])] == before.strftime("%Y%m%d")
        assert keys[int(t[i, _lib.F_ALB_I1])] == after.strftime("%Y%m%d")
        assert t[i, _lib.F_ALB_DAYS] == (d - before).days and t[i, _lib.F_ALB_SPAN] == (after - before).days
    assert t[-1, _lib.F_DT] == t[-2, _lib.F_DT] == 1800          # last row repeats the previous step
    assert t[0, _lib.F_SNOW_DAYS] == 2                            # 20220601 - 20220530
    with pytest.raises(ValueError):
        heuristic_unit_guesser(130.0, 100)
    with pytest.raises(ValueError):                               # date outside the albedo maps
        from datetime import datetime
        get_closest_dates(keys, datetime(2021, 1, 1))


def test_geo_helpers():
    gt = (470000.0, 10.0, 0.0, 8660000.0, 0.0, -10.0)
    assert coords_to_index(gt, 470000.0 + 10 * 7 + 5, 8660000.0 - 10 * 3 - 5) == (3, 7)
    lat, lon = utm_to_latlon(478342, 8655635)                     # the reference's AWS (model.py:557)
    assert abs(lat - 77.974) < 5e-3 and abs(lon - 14.069) < 5e-3


def test_raster_roundtrip_and_config(tmp_path):
    from enrgy_b200.raster_utils import export_array_as_geotiff, have_gdal, load_raster, save_npy_raster
    a = np.arange(12, dtype=np.float32).reshape(3, 4)
    a[0, 0] = np.nan
    a[1, 1] = -0.5
    a[2, 2] = 1.5
    gt = (1.0, 10.0, 0.0, 2.0, 0.0, -10.0)
    p = save_npy_raster(str(tmp_path / "r.npy"), a, gt)
    arr, gt2, _ = load_raster(p, None, 10, remove_outliers=True, v=False)
    assert tuple(gt2) == gt and arr.dtype == np.float32
    assert arr[1, 1] == np.float32(0.001) and arr[2, 2] == 1.0 and np.isnan(arr[0, 0])
    if not have_gdal():
        out = export_array_as_geotiff(a, gt, "x", str(tmp_path / "o.tiff"))
        back = np.load(out)
        assert back[0, 0] == -9999.0


def test_insolation_tables_match_oracle():
    """The product's pre-pass (C++, libm) and the oracle (Python math, libm) derive the same sun
    vectors and Q16 ray directions -- checked through the exported prototype? No GPU is needed for
    the oracle side; the product side is checked on the GPU in test_gpu_shading.py."""
    from oracle import insolation_oracle as I
    rows = I.substep_table(I.to_unix("20220601 10:00:00"), 3600, 77.98, 14.1, 10.0)
    assert len(rows) == 4
    for r in rows:
        assert abs(r["E"] ** 2 + r["N"] ** 2 + r["U"] ** 2 - 1.0) < 1e-12
        assert max(abs(r["dc_fix"]), abs(r["dr_fix"])) == 65536


REGIME_VARIANTS = ["polar_night", "polar_dawn", "polar_dusk", "cold_unstable", "extremes", "irregular_time"]


@pytest.mark.parametrize("f64", [True, False])
@pytest.mark.parametrize("variant", ["default", "andreas", "gradient_calm"] + REGIME_VARIANTS)
def test_host_prepass_matches_oracle(f64, variant):
    """The library's host pre-pass (C++: Monin-Obukhov solve, CH, shortwave factor; csrc/prepass.cu,
    reached through enrgy_host_prepass WITHOUT a device) against the oracle's per-row scalars, which are
    the reference's own (turbo.py:88-137, model.py:500-530).  No GPU, no kernel: host logic only.
    The weather regimes of tests/regimes.py (with their insolation, dark where the sun is down) reach the
    unstable branch of the Monin-Obukhov solve and the neutral row (L = +inf), gales, calm air, dry and
    saturated air, a station at 600-660 hPa and rows of 10 min to 63.75 h."""
    from enrgy_b200.engine import host_prepass
    from oracle import insolation_oracle as I
    from tests import parity as P
    from tests import regimes as G
    kw = {}
    case_kw = {}
    if variant == "andreas":
        kw = dict(andreas=True)
    if variant == "gradient_calm":
        case_kw = dict(with_gradient=True, calm_every=5)     # GRADIENT column, WIND_SPEED 0 -> 0.1
        kw = dict(temp_lapse_rate="GRADIENT")
    if variant in REGIME_VARIANTS:
        case = G.make_regime_case(variant)
        pot = I.insolation_series(case, shadow=False).astype(np.float32)
    else:
        case = make_case(48, 30, w=56, seed=17, **case_kw)
        pot = P.random_insolation(case, 30)
    ora = P.run_oracle(case, pot, f64, **kw)
    alb = P.clipped_albedo(case, np.float32)
    table = build_forcing(case.aws_rows, list(alb), temp_lapse_rate=kw.get("temp_lapse_rate", -0.006))
    pot_aws = np.asarray(pot, dtype=np.float64 if f64 else np.float32)[:, case.aws_rc[0], case.aws_rc[1]].astype(np.float64)
    point = host_prepass(case.dem, table, precision=_lib.F64 if f64 else _lib.F32, pot_aws=pot_aws,
                         cell_size=case.cell, elev_aws=case.elev_aws, aws_row=case.aws_rc[0], aws_col=case.aws_rc[1],
                         sensor_z=1.6, zm=1e-3, z_h_or_e=1e-4, emissivity=0.98, andreas=kw.get("andreas", False),
                         insol_mode=_lib.INSOL_STREAMED, lat=case.lat, lon=case.lon)
    L_ref = np.array([r["L"] for r in ora["rows"]])
    f_ref = np.array([r["factor"] for r in ora["rows"]])
    assert P.l_rel_err(point[:, _lib.P_L], L_ref) < (1e-9 if f64 else 1e-5)
    assert np.max(np.abs(point[:, _lib.P_SW_FACTOR] - f_ref) / np.maximum(np.abs(f_ref), 1e-12)) < (1e-12 if f64 else 1e-6)
    if variant == "cold_unstable":
        # both branches and the neutral row really occur
        assert (L_ref < 0).sum() >= 10 and (L_ref > 0).any() and np.isposinf(L_ref).sum() >= 3
    if variant == "polar_night":
        assert np.all(f_ref == 1.0)                          # potential insolation 0 -> factor 1
    if variant in ("polar_dawn", "polar_dusk"):
        assert f_ref.max() > 3.0                             # a faint SWD over a sun at the horizon


def test_host_prepass_computed_insolation_and_errors():
    """In-kernel insolation: the pre-pass's potential insolation at the AWS cell and its sub-step
    counts against the insolation oracle (with and without the shading ray of the AWS cell); bad
    input is refused with the library's error codes."""
    from enrgy_b200.engine import host_prepass
    from enrgy_b200._lib import EnrgyError
    from oracle import insolation_oracle as I
    from oracle.enrgy_oracle import time_step_seconds
    from datetime import datetime, timedelta
    case = make_case(64, 12, w=72, seed=19)
    table = build_forcing(case.aws_rows, list(case.albedo_maps))
    base = dict(cell_size=case.cell, elev_aws=case.elev_aws, aws_row=case.aws_rc[0], aws_col=case.aws_rc[1],
                sensor_z=1.6, zm=1e-3, z_h_or_e=1e-4, insol_mode=_lib.INSOL_COMPUTED, lat=case.lat, lon=case.lon)
    for shadow in (False, True):
        point = host_prepass(case.dem, table, shadow=shadow, **base)
        for i, row in enumerate(case.aws_rows):
            dt = time_step_seconds(case.aws_rows, i)
            want = I.potential_insolation(case.dem, case.cell, case.lat, case.lon, I.to_unix(row["DATE"]), dt,
                                          shadow=shadow)[case.aws_rc]
            got_kwh = point[i, _lib.P_POT_AWS] * dt / 3.6e6                 # W m-2 over the step -> kWh m-2
            assert abs(got_kwh - want) <= 1e-9 * max(abs(want), 1e-6), (shadow, i)
            n_sub = len(I.substep_table(I.to_unix(row["DATE"]), dt, case.lat, case.lon, case.cell))
            assert int(point[i, _lib.P_NSUB]) == n_sub
    # dark, dawn and irregular rows: 0 .. 255 sunlit sub-steps, partial last sub-steps
    from tests import regimes as G
    for name in ("polar_night", "polar_dawn", "polar_dusk", "irregular_time"):
        rc = G.make_regime_case(name)
        t_rc = build_forcing(rc.aws_rows, list(rc.albedo_maps))
        b_rc = dict(base, elev_aws=rc.elev_aws, aws_row=rc.aws_rc[0], aws_col=rc.aws_rc[1])
        counts = []
        for shadow in (False, True):
            point = host_prepass(rc.dem, t_rc, shadow=shadow, **b_rc)
            for i, row in enumerate(rc.aws_rows):
                dt = time_step_seconds(rc.aws_rows, i)
                n_sub = len(I.substep_table(I.to_unix(row["DATE"]), dt, rc.lat, rc.lon, rc.cell))
                assert int(point[i, _lib.P_NSUB]) == n_sub, (name, i)
                if not shadow:
                    counts.append(n_sub)
                want = I.potential_insolation(rc.dem, rc.cell, rc.lat, rc.lon, I.to_unix(row["DATE"]), dt,
                                              shadow=shadow)[rc.aws_rc]
                assert abs(point[i, _lib.P_POT_AWS] * dt / 3.6e6 - want) <= 1e-9 * max(abs(want), 1e-6), (name, shadow, i)
        if name == "polar_night":
            assert set(counts) == {0}
        elif name == "irregular_time":
            assert {0, 1, 4, 12, 28, 255} <= set(counts)
        else:
            assert 0 in counts and 4 in counts and any(0 < k < 4 for k in counts)
    # at most 255 sunlit sub-steps in one row: 63.75 h of midnight sun pass, 64 h are refused
    for hours, ok in ((63.75, True), (64.0, False)):
        rows = G.make_regime_case("irregular_time").aws_rows[:2]
        rows = [dict(rows[0], DATE="20220620 00:00:00"),
                dict(rows[1], DATE=(datetime(2022, 6, 20) + timedelta(hours=hours)).strftime("%Y%m%d %H:%M:%S"))]
        t_b = build_forcing(rows, ["20220601", "20220701"])
        if ok:
            assert list(host_prepass(case.dem, t_b, **base)[:, _lib.P_NSUB]) == [255, 255]
        else:
            with pytest.raises(EnrgyError) as err:
                host_prepass(case.dem, t_b, **base)
            assert err.value.code == _lib.ERR_RANGE
    with pytest.raises(EnrgyError):
        host_prepass(case.dem, table, **dict(base, aws_row=999))
    bad = table.copy()
    bad[3, _lib.F_RH] = 55.0                                                   # per cent instead of a fraction
    with pytest.raises(EnrgyError):
        host_prepass(case.dem, bad, **base)


def test_extra_station_host_logic(tmp_path):
    """add_station / add_cloud_transmissivity (BASELINE config C4): real-world coordinates -> cell units of
    the model grid (cell centres), the station's own file -> the series table; argument checks."""
    import csv
    from enrgy_b200 import Energy, _lib
    from enrgy_b200.forcing import build_station_series
    from enrgy_b200.raster_utils import save_npy_raster
    from enrgy_b200.synthetic import make_station_rows
    case = make_case(40, 9, w=56, seed=3)
    d = str(tmp_path)
    dem = save_npy_raster(os.path.join(d, "dem.npy"), case.dem, case.geotransform)
    e = Energy(dem, None, os.path.join(d, "out"), res=10)
    ul_x, x_dist, _, ul_y, _, y_dist = case.geotransform
    rows = make_station_rows(case, case.elev_aws + 80.0, seed=4)
    path = os.path.join(d, "st.csv")
    with open(path, "w", newline="") as f:
        w = csv.DictWriter(f, fieldnames=list(rows[0]))
        w.writeheader()
        w.writerows(rows)
    # the centre of cell (row 7, col 30) and a point a quarter of a cell off it
    e.add_station(path, (ul_x + 30.5 * x_dist, ul_y + 7.5 * y_dist), case.elev_aws + 80.0)
    e.add_station(path, (ul_x + 12.75 * x_dist, ul_y + 33.25 * y_dist), 512.0)
    e.add_cloud_corr(0.2)
    pos, series = e._station_setup(9)
    assert np.allclose(pos, [(7.0, 30.0, case.elev_aws + 80.0), (32.75, 12.25, 512.0)], atol=1e-9)
    want = build_station_series(rows, cloud_corr=0.2)
    assert want.shape == (9, _lib.ST_COUNT) and np.array_equal(series[0], want)
    assert np.all(want[:, _lib.ST_RH] <= 1.0) and np.all((want[:, _lib.ST_CLOUD] >= 0) & (want[:, _lib.ST_CLOUD] <= 1))
    assert want[0, _lib.ST_T_AIR] == float(rows[0]["T_AIR"]) and want[3, _lib.ST_PRESSURE] == float(rows[3]["PRESSURE"])
    with pytest.raises(ValueError):
        e._station_setup(10)                       # another number of rows than the main AWS file
    e.add_station(path, (ul_x, ul_y), 1.0)
    with pytest.raises(ValueError):
        e.add_station(path, (ul_x, ul_y), 1.0)     # a fourth one
    with pytest.raises(ValueError):
        e.add_cloud_transmissivity(-0.1)
    e.add_cloud_transmissivity(0.7)
    assert e.cloud_k == 0.7


def test_sharded_shading_chunk_plan():
    """Chunks of the multi-GPU shading run: whole steps, inside the memory budget, and -- several ranks -- at
    least 192 sub-steps per rank and launch (a smaller sweep launch leaves the GPU half empty in its tail)
    unless the budget forbids it."""
    from enrgy_b200.parallel import ShardedShading, plan_step_chunks, split_even

    class Stub:
        def mask_words(self, rows):
            return (rows + 7) // 8 * 8 * 256          # 8192 columns
    sub = np.array([4] * 300 + [0] * 84 + [4] * 384)   # a stretch of night rows in between
    for world in (1, 2, 8):
        bands = [(i * (8192 // world), 8192 // world) for i in range(world)]
        sh = ShardedShading(Stub(), bands, 0, world)
        plan = sh.chunks(0, sub.size, sub)
        assert plan[0][0] == 0 and plan[-1][1] == sub.size and all(a[1] == b[0] for a, b in zip(plan, plan[1:]))
        counts = [int(sub[a:b].sum()) for a, b in plan]
        per_sub = 4 * (sum(sh.words) // world + max(sh.words)) * 2 + 1
        assert all(c * per_sub <= sh.budget + 4 * per_sub for c in counts)
        if world > 1:
            assert all(c >= min(192 * world, sh.budget // per_sub) - 4 for c in counts[:-1]), (world, counts)
    assert split_even(10, 27, 4) == [(10, 15), (15, 19), (19, 23), (23, 27)] or sum(b - a for a, b in split_even(10, 27, 4)) == 17
    assert plan_step_chunks(sub, 0, 10, 3) == [(t, t + 1) for t in range(10)]       # a step is never cut
    with pytest.raises(ValueError):
        ShardedShading(Stub(), [(0, 100), (100, 92)], 0, 2)                          # band starts off the 8-row grid
    with pytest.raises(ValueError):
        ShardedShading(Stub(), [(0, 96), (96, 96)], 0, 2, exchange="pigeon")


def test_ensemble_members_and_sharding():
    """Seeded member perturbations (SURVEY 8d C5) and their round-robin sharding over ranks."""
    from enrgy_b200.ensemble import make_members, shard
    a, b = make_members(64, seed=0), make_members(64, seed=0)
    assert a == b and len(a) == 64
    off = np.array([m["albedo_offset"] for m in a])
    zm = np.array([m["zm"] for m in a])
    assert abs(off.mean()) < 0.02 and 0.015 < off.std() < 0.045                 # N(0, 0.03)
    assert (zm >= 3e-4).all() and (zm <= 3e-3).all()                            # log-uniform [3e-4, 3e-3]
    assert all(abs(m["z_h_or_e"] - m["zm"] / 10.0) < 1e-18 for m in a)
    assert make_members(4, seed=1) != make_members(4, seed=2)
    parts = [shard(a, 8, r) for r in range(8)]
    assert sorted(i for p in parts for i in p) == list(range(64)) and all(len(p) == 8 for p in parts)
    assert shard(a[:5], 8, 7) == [] and shard(a[:5], 2, 1) == [1, 3]


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: the glacier cells of the rasters (off it they are NaN by definition), all of
    them while they fit the byte budget, else the same seeded sample of cells from every raster, the same
    on every call; finite float32/float64 values only."""
    import bench
    rng = np.random.default_rng(5)
    stats = rng.random((30, _lib.S_COUNT))
    cells = 64 * 80
    valid = (np.arange(cells) % 7 != 3).reshape(64, 80)
    for dtype in (np.float32, np.float64):
        # every value is its raster's number times `cells` plus its cell index; NaN off the glacier
        state = tuple(np.where(valid, (np.arange(cells) + q * cells).reshape(64, 80), np.nan).astype(dtype)
                      for q in range(3))
        bench.dump_outputs(str(tmp_path / "whole"), stats, state, valid)
        for name, a in zip(("swe", "total_snow", "total_ice"), state):
            assert np.array_equal(np.load(tmp_path / "whole" / (name + ".npy")), a[valid])
        assert np.array_equal(np.load(tmp_path / "whole" / "stats.npy"), stats)
        monkeypatch.setattr(bench, "DUMP_BYTES", 40000)
        runs = []
        for k in range(2):
            d = tmp_path / ("sample%d" % k)
            bench.dump_outputs(str(d), stats, state, valid)
            files = {f.name: np.load(f) for f in d.iterdir()}
            assert sum(f.stat().st_size for f in d.iterdir()) <= 40000
            assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in files.values())
            runs.append(files)
        monkeypatch.undo()
        assert runs[0].keys() == runs[1].keys() == {"stats.npy", "swe.npy", "total_snow.npy", "total_ice.npy"}
        assert all(np.array_equal(runs[0][k], runs[1][k]) for k in runs[0])
        swe = runs[0]["swe.npy"]
        assert swe.dtype == dtype and 0 < swe.size < valid.sum() and np.all(np.diff(swe) > 0)
        assert valid.ravel()[swe.astype(int)].all()                             # glacier cells only
        assert np.array_equal(runs[0]["total_snow.npy"], swe + cells)          # the same cells in each raster
        assert np.array_equal(runs[0]["total_ice.npy"], swe + 2 * cells)
        monkeypatch.setattr(bench, "DUMP_BYTES", stats.nbytes)                  # no room left for any cell
        with pytest.raises(ValueError):
            bench.dump_outputs(str(tmp_path / "full"), stats, state, valid)
        monkeypatch.undo()


def test_header_is_plain_c(tmp_path):
    """include/enrgy_b200.h is the drop-in boundary: it must compile as C11 and as C++17 on its own, and the
    calls INTEGRATION.md shows must match its prototypes."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "use.c"
    src.write_text(
        '#include <stddef.h>\n#include "enrgy_b200.h"\n'
        "int f(enrgy_ctx* h, int n, const double* series, double* stats, float* a, float* b, float* c) {\n"
        "  double row[3] = {1, 2, 3}, col[3] = {1, 2, 3}, elev[3] = {1, 2, 3}, off[8] = {0}, zm[8] = {0}, zhe[8] = {0}, tot[8][4];\n"
        "  struct enrgy_params p; (void)p;\n"
        "  if (enrgy_set_stations(h, 3, row, col, elev, series, 0.7) != ENRGY_OK) return 1;\n"
        "  if (enrgy_set_insolation_aws(h, 0, n, series) != ENRGY_OK) return 1;\n"
        "  enrgy_prepass(h); enrgy_run(h, 0, n, stats);\n"
        "  if (enrgy_run_members(h, 8, off, zm, zhe, 0, n, NULL, &tot[0][0]) != ENRGY_OK) return (int)(size_t)enrgy_last_error();\n"
        "  return enrgy_get_member_state(h, 3, 32, a, b, c);\n}\n")
    inc = os.path.join(ROOT, "include")
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-fsyntax-only", "-I", inc, str(src)], check=True)
    subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-x", "c++", "-I", inc, str(src)], check=True)
