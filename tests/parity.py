"""Shared helpers of the parity tests: run the oracle and the CUDA engine on the same inputs."""
from __future__ import annotations

import numpy as np

from enrgy_b200 import _lib
from enrgy_b200.engine import Engine
from enrgy_b200.forcing import build_forcing
from oracle import enrgy_oracle as O
from oracle import insolation_oracle as I

FLUX_FIELDS = ("rs", "lwd", "lwu", "sens", "lat", "atmo", "mf", "g")


def clipped_albedo(case, dtype):
    """load_raster(..., remove_outliers=True), reference raster_utils.py:48-50."""
    out = {}
    for k, a in case.albedo_maps.items():
        a = a.astype(dtype).copy()
        a[a < 0] = 0.001
        a[a > 1] = 1
        out[k] = a
    return out


def oracle_config(case, **kw):
    return O.ModelConfig(z=kw.get("z", 1.6), elev_aws=case.elev_aws, xy_aws=case.xy_aws,
                         zm=kw.get("zm", 1e-3), z_h_or_e=kw.get("z_h_or_e", 1e-4),
                         andreas=kw.get("andreas", False), const_albedo=kw.get("const_albedo"),
                         temp_lapse_rate=kw.get("temp_lapse_rate", -0.006),
                         last_snowfall=kw.get("last_snowfall"), max_ice_albedo=kw.get("max_ice_albedo"),
                         emissivity=kw.get("emissivity", 0.98), cloud_corr=kw.get("cloud_corr"),
                         sensible_corr=kw.get("sensible_corr", 1), latent_corr=kw.get("latent_corr", 1),
                         msm=kw.get("msm"), snow_density=kw.get("snow_density"))


def run_oracle(case, pot, f64, keep_steps=None, **kw):
    dt = np.float64 if f64 else np.float32
    cfg = oracle_config(case, **kw)
    alb = None if kw.get("const_albedo") else clipped_albedo(case, dt)
    return O.run_model(case.dem.astype(dt), case.geotransform, case.aws_rows,
                       pot if callable(pot) else np.asarray(pot, dtype=dt), cfg,
                       swe=case.swe.astype(dt) if kw.get("use_swe", True) else None,
                       albedo_arrays=alb, state_dtype=dt, keep_steps=keep_steps, want_means=True,
                       stations=kw.get("stations"), cloud_k=kw.get("cloud_k"))


def run_oracle_arrays(case, pot, f64, **kw):
    """Like run_oracle, but the case's albedo maps are taken as they are (already clipped)."""
    dt = np.float64 if f64 else np.float32
    cfg = oracle_config(case, **kw)
    alb = None if kw.get("const_albedo") else {k: a.astype(dt) for k, a in case.albedo_maps.items()}
    return O.run_model(case.dem.astype(dt), case.geotransform, case.aws_rows, np.asarray(pot, dtype=dt), cfg,
                       swe=case.swe.astype(dt), albedo_arrays=alb, state_dtype=dt, want_means=True)


def make_engine(case, f64, pot=None, computed=False, shadow=False, device=0, band=None, **kw):
    """band = (row0, rows): the engine of one row band of the case (every band-local raster is cut here)."""
    h, w = case.shape
    r0, nr = band if band is not None else (0, h)
    rows = slice(r0, r0 + nr)
    eng = Engine(h, w, precision=_lib.F64 if f64 else _lib.F32, device=device)
    eng.set_params(cell_size=case.cell, elev_aws=case.elev_aws, aws_row=case.aws_rc[0],
                   aws_col=case.aws_rc[1], sensor_z=kw.get("z", 1.6), zm=kw.get("zm", 1e-3),
                   z_h_or_e=kw.get("z_h_or_e", 1e-4), andreas=kw.get("andreas", False),
                   sensible_corr=kw.get("sensible_corr", 1), latent_corr=kw.get("latent_corr", 1),
                   emissivity=kw.get("emissivity", 0.98), const_albedo=kw.get("const_albedo"),
                   max_ice_albedo=kw.get("max_ice_albedo"), snow_density=kw.get("snow_density"),
                   msm_depths=kw["msm"]["depths"] if kw.get("msm") else None,
                   insol_mode=_lib.INSOL_COMPUTED if computed else _lib.INSOL_STREAMED,
                   shadow=shadow, lat=case.lat, lon=case.lon,
                   band_row0=r0 if band is not None else 0, band_rows=nr if band is not None else 0)
    eng.set_dem(case.dem)
    if kw.get("msm"):
        eng.set_msm(kw["msm"]["temperatures"], kw["msm"]["elev"])
    keys = None
    if not kw.get("const_albedo"):
        alb = clipped_albedo(case, np.float32)
        keys = list(alb)
        eng.set_albedo_maps([alb[k][rows] for k in keys])
    if kw.get("use_swe", True):
        eng.set_swe(case.swe[rows])
    table = build_forcing(case.aws_rows, keys, temp_lapse_rate=kw.get("temp_lapse_rate", -0.006),
                          cloud_corr=kw.get("cloud_corr"), last_snowfall=kw.get("last_snowfall"))
    eng.set_forcing(table)
    if kw.get("stations") is not None:          # BASELINE config C4: extra weather stations, cloud attenuation
        from enrgy_b200.forcing import build_station_series
        st = kw["stations"]
        eng.set_stations([(s_["row"], s_["col"], s_["elev"]) for s_ in st],
                         [build_station_series(s_["rows"], cloud_corr=kw.get("cloud_corr")) for s_ in st],
                         cloud_k=kw.get("cloud_k"))
    if not computed:
        eng.set_insolation(0, np.ascontiguousarray(np.asarray(pot, dtype=np.float32)[:, rows]))
        if band is not None:
            eng.set_insolation_aws(0, np.asarray(pot, dtype=np.float32)[:, case.aws_rc[0], case.aws_rc[1]])
    if kw.get("msm") and band is not None:
        # the sub-surface pre-pass integrates the AWS cell on every band (as Energy.model hands it over)
        ar, ac = case.aws_rc
        eng.set_aws_cell([float(alb[k][ar, ac]) for k in keys] if keys else None, float(case.swe[ar, ac]))
    eng.prepass()
    return eng


def rel_err(got, ref, floor):
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(ref)), "NaN masks differ"
    with np.errstate(invalid="ignore"):
        e = np.abs(got - ref) / np.maximum(np.abs(ref), floor)
    return e


def max_rel_err(got, ref, floor):
    e = rel_err(got, ref, floor)
    return float(np.nanmax(e)) if np.isfinite(e).any() else 0.0


def l2_rel_err(got, ref):
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    m = ~np.isnan(ref)
    den = np.sqrt(np.sum(ref[m] ** 2))
    return float(np.sqrt(np.sum((got[m] - ref[m]) ** 2)) / den) if den > 0 else 0.0


def means_from_stats(stats):
    """[T, 13] area means laid out like oracle run_model(want_means=True)."""
    s = stats
    nv = s[:, _lib.S_NVALID]
    with np.errstate(invalid="ignore", divide="ignore"):
        cols = [s[:, _lib.S_RS] / nv, (s[:, _lib.S_LWD] - s[:, _lib.S_LWU]) / nv, s[:, _lib.S_LWD] / nv,
                s[:, _lib.S_SENS] / nv, s[:, _lib.S_LAT] / nv, s[:, _lib.S_ATMO] / nv, s[:, _lib.S_G] / nv,
                s[:, _lib.S_MELT] / nv, s[:, _lib.S_SNOW] / nv, s[:, _lib.S_ICE] / nv,
                s[:, _lib.S_SWE] / s[:, _lib.S_NSWE], s[:, _lib.S_NSNOW], s[:, _lib.S_NSWE]]
    return np.stack(cols, axis=1)


def random_insolation(case, n_steps, seed=5, f32=True):
    rng = np.random.default_rng(seed)
    h, w = case.shape
    pot = 0.2 * rng.random((n_steps, h, w))
    pot[0] = 0.0                                 # potential == 0 -> factor 1 (model.py:523-524)
    pot = pot.astype(np.float32)
    pot[:, np.isnan(case.dem)] = np.nan
    return pot


def oracle_insolation(case, pot, computed, shadow, f64):
    """The insolation the oracle runs on: `pot` when it is streamed, else the specification's series."""
    if not computed:
        return pot
    pot_o = I.insolation_series(case, shadow=shadow, dtype=np.float64)
    return pot_o if f64 else pot_o.astype(np.float32)


def oracle_band_sums(ora, rows, valid):
    """[T, S_COUNT] statistics of the rows `rows` of the raster, as float64 sums of the oracle's per-step
    rasters (flux sums over glacier cells, SWE sums and counts over its non-NaN cells, before the update)."""
    v = valid[rows]
    out = np.zeros((len(ora["rows"]), _lib.S_COUNT))
    cols = ((_lib.S_RS, "rs"), (_lib.S_LWD, "lwd"), (_lib.S_LWU, "lwu"), (_lib.S_SENS, "sens"),
            (_lib.S_LAT, "lat"), (_lib.S_ATMO, "atmo"), (_lib.S_G, "g"), (_lib.S_MELT, "mf"))
    for i, (r, (snow, ice, swe)) in enumerate(zip(ora["rows"], ora["melt"])):
        for col, name in cols:
            out[i, col] = np.nansum(np.asarray(r[name], dtype=np.float64)[rows][v])
        out[i, _lib.S_SNOW] = np.nansum(np.asarray(snow, dtype=np.float64)[rows][v])
        out[i, _lib.S_ICE] = np.nansum(np.asarray(ice, dtype=np.float64)[rows][v])
        swe = np.asarray(swe, dtype=np.float64)[rows]
        out[i, _lib.S_SWE] = np.nansum(swe)
        out[i, _lib.S_NSNOW] = np.count_nonzero(swe > 0)
        out[i, _lib.S_NSWE] = np.count_nonzero(~np.isnan(swe))
        out[i, _lib.S_NVALID] = np.count_nonzero(v)
    return out


def compare_run(case, f64, pot=None, computed=False, shadow=False, band=None, ora=None, skip=(), **kw):
    """Runs oracle and engine; returns dict of worst relative errors.
    skip: (row, field) pairs of the per-step flux rasters left out of res[field]; their worst error is
    res["skipped"] (only with skip).
    band = (row0, rows): the engine runs that row band; its rasters are compared with those rows of the
    whole-raster oracle and its statistics with the oracle's float64 sums over them ("band_sums"; the
    glacier-wide means only exist for the whole raster).  ora: run_oracle's result for these inputs, for
    callers that compare several bands against one oracle run."""
    n = len(case.aws_rows)
    r0, nr = band if band is not None else (0, case.shape[0])
    rows = slice(r0, r0 + nr)
    if ora is None:
        ora = run_oracle(case, oracle_insolation(case, pot, computed, shadow, f64), f64, **kw)
    eng = make_engine(case, f64, pot=pot, computed=computed, shadow=shadow, band=band, **kw)
    try:
        dump = eng.dump_steps(0, n)
        stats = eng.run(0, n)
        swe, tsn, tic = eng.state(np.float64)
        point = eng.point_scalars()
        layers = eng.layer_temps() if kw.get("msm") else None
    finally:
        eng.close()
    ff, mfl, tfl = (1e-3, 1e-7, 1e-6) if f64 else (1.0, 1e-3, 1e-3)
    msm_floor = 5.0
    if kw.get("msm") and not f64:
        # The bound for the melt gate in float32 is tied to the reference's OWN float32-vs-float64 gap on this
        # very case (SURVEY 8c): the as-shipped reference deviates from its float64-injected self by a few
        # 1e-3 W m-2 in the melt flux (the gate carries the cold content of the surface layer, which integrates
        # the float32 round-off of every earlier step).  1e-4 x 5 W m-2 = 5e-4 W m-2 must not be looser than that.
        # Where nothing melts (a cold regime), mf is exactly 0 in both runs and the reference has no such
        # error to measure: the bound then rests on the cases that melt.
        if any(np.nanmax(r["mf"]) > 0 for r in ora["rows"]):
            ora64 = run_oracle(case, oracle_insolation(case, pot, computed, shadow, True), True, **kw)
            own_gap = max(float(np.nanmax(np.abs(np.asarray(a["mf"], dtype=np.float64) - b["mf"])))
                          for a, b in zip(ora["rows"], ora64["rows"]))
            assert 1e-4 * msm_floor <= own_gap, ("the float32 melt-flux bound is looser than the reference's own "
                                                 "float32 error on this case", own_gap)
    res = {}
    skipped = 0.0
    off = np.isnan(case.dem)[rows]
    for name in FLUX_FIELDS:
        idx = _lib.DUMP_NAMES.index(name)
        worst = 0.0
        for i in range(n):
            ref = np.array(ora["rows"][i][name], dtype=np.float64)[rows]
            if name == "g" and not kw.get("msm"):
                ref[off] = np.nan       # np.zeros(atmo.shape): finite off-glacier (model.py:434)
            if name == "lwu" and not kw.get("msm"):
                # without the sub-surface model the reference's surface temperature raster is
                # zeros EVERYWHERE (np.zeros_like(dem), SURVEY F9), so its lwu is finite off-glacier
                # too; the debug view only covers glacier cells.
                ref[off] = np.nan
            floor = ff
            if kw.get("msm") and not f64 and name in ("mf", "g"):
                # float32 + sub-surface model: the melt gate qm = full - q0 carries the cold content
                # of the surface layer, which integrates the float32 round-off of every earlier
                # step's fluxes (3e-5 W m-2 per term, in the as-shipped reference too): the
                # per-step melt flux agrees to ~5e-4 W m-2, the melt TOTALS to 1e-4 relative.
                floor = msm_floor
            e = max_rel_err(dump[i, idx], ref, floor)
            if (i, name) in skip:
                skipped = max(skipped, e)
            else:
                worst = max(worst, e)
        res[name] = worst
    if skip:
        res["skipped"] = skipped
    worst = 0.0
    for i in range(n):
        ref = np.array(ora["rows"][i]["albedo"], dtype=np.float64)[rows]
        ref[off] = np.nan           # constant-albedo rasters are finite off-glacier (model.py:332)
        worst = max(worst, max_rel_err(dump[i, _lib.D_ALBEDO], ref, 1e-3))
    res["albedo"] = worst
    res["snow"] = max(max_rel_err(dump[i, _lib.D_SNOW], ora["melt"][i][0][rows], mfl) for i in range(n))
    res["ice"] = max(max_rel_err(dump[i, _lib.D_ICE], ora["melt"][i][1][rows], mfl) for i in range(n))
    if layers is not None:
        res["layer_t"] = max(max_rel_err(layers[l], ora["layer_temperatures"][l][rows], 1e-3 if f64 else 1.0)
                             for l in range(layers.shape[0]))
    res["swe"] = max_rel_err(swe, ora["swe"][rows], tfl)
    res["total_snow"] = max_rel_err(tsn, ora["total_snow"][rows], tfl)
    res["total_ice"] = max_rel_err(tic, ora["total_ice"][rows], tfl)
    res["total_ice_l2"] = l2_rel_err(tic, ora["total_ice"][rows])
    res["total_snow_l2"] = l2_rel_err(tsn, ora["total_snow"][rows])
    if band is None:
        m_e = means_from_stats(stats)
        m_o = ora["means"]
        floors = np.array([ff, ff, ff, ff, ff, ff, ff, ff, mfl, mfl, tfl, 0.5, 0.5])
        res["means"] = float(np.max(np.abs(m_e - m_o) / np.maximum(np.abs(m_o), floors)))
    else:
        s_o = oracle_band_sums(ora, rows, ~np.isnan(case.dem))
        # the per-cell floors, times the cells a sum runs over
        floors = np.full(_lib.S_COUNT, ff)
        if kw.get("msm") and not f64:
            floors[[_lib.S_MELT, _lib.S_G]] = msm_floor
        floors[[_lib.S_SNOW, _lib.S_ICE]] = mfl
        floors[_lib.S_SWE] = tfl
        floors[[_lib.S_NSNOW, _lib.S_NSWE, _lib.S_NVALID]] = 0.5
        scale = np.maximum(s_o[:, [_lib.S_NVALID]], 1.0)
        res["band_sums"] = float(np.max(np.abs(stats - s_o) / np.maximum(np.abs(s_o), floors * scale)))
    res["L"] = l_rel_err(point[:, _lib.P_L], [r["L"] for r in ora["rows"]])
    return res


def l_rel_err(got, ref):
    """Worst relative error of the Monin-Obukhov lengths.  A neutral row (air at the surface temperature:
    Qh = 0) has L = +inf; an infinity matched by the same infinity counts as exact, any other value
    against it as an infinite error."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        e = np.abs(got - ref) / np.abs(ref)
    e = np.where(np.isinf(ref) & (got == ref), 0.0, e)
    return float(np.max(np.where(np.isnan(e), np.inf, e)))
