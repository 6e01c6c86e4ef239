"""Seeded AWS weather for named regimes that the summer series of synthetic.make_aws_rows never reaches.

make_aws_rows is June to September at 78 N in fixed hourly rows, with air at 1-9 degC over a 0 degC
surface: the sun never sets, the Monin-Obukhov solve stays on its stable branch and every row has the same
number of insolation sub-steps.  The regimes here cover the rest:

  polar_night     78 N from 10 December: no sunlit sub-step at all, cold air, SWD 0
  polar_dawn      78 N around 20 February: hourly rows with 0, 2 or 4 sunlit sub-steps and a faint SWD,
                  so the observed / potential shortwave factor is large
  polar_dusk      the same around 20 October
  cold_unstable   air from -30 to -0.01 degC (unstable over the 0 degC surface), rows of exactly 0.00 degC
                  (neutral: Qh = 0, L = +inf) and +-0.01 degC; a negative balance, no melt
  extremes        calm rows under warm air (strong stability), gales of 25-40 m/s, humidity of 100 and
                  10 %, cloudiness 0 and 1, on a DEM raised by 3000 m with the station at 600-660 hPa
  irregular_time  rows of 10 min, 50 min, 1 h and 3 h, a 7 h logger gap and one 63.75 h row: 0 to 255
                  sub-steps in one run, partial last sub-steps, a row exactly on an albedo map date
                  (interpolation span 0) and the last snowfall inside the run
  msm_season      about 2200 hourly rows from mid-August at 78 N: polar sunset and freeze-up, for the
                  sub-surface model over a season

The rows carry the reference's CSV columns formatted as make_aws_rows formats them.  make_regime_case
builds the matching SyntheticCase (albedo map dates that span the run, the DEM shift of `extremes`) and
REGIME_KW holds the model options each regime needs (last_snowfall, the sub-surface stack)."""
from __future__ import annotations

import math
from datetime import datetime, timedelta

import numpy as np

from enrgy_b200.synthetic import (DEFAULT_LAT, DEFAULT_LON, DEFAULT_ULX, DEFAULT_ULY, SyntheticCase, make_albedo_maps,
                                  make_dem, make_swe)

FMT = "%Y%m%d %H:%M:%S"

# the 7-layer stack of test_gpu_parity
MSM7 = dict(depths=[0.1, 0.1, 0.3, 0.5, 0.5, 0.5, 3.0],
            temperatures=[-6.9, -6.93, -7.025, -7.31, -6.93, -7.12, -7.0, -5.57], elev=275.0)


def _row(t, t_air, wind, pres, hum, cld, swd):
    return {"DATE": t.strftime(FMT), "T_AIR": "%.2f" % t_air, "WIND_SPEED": "%.2f" % wind,
            "PRESSURE": "%.1f" % pres, "HUMID": "%.1f" % hum, "CLOUDINESS": "%.2f" % cld, "SWD": "%.1f" % swd}


def _sun_up(t):
    """sin(sun elevation) at the middle of the hour starting at t, 78 N (the almanac of the insolation
    specification, so that SWD > 0 exactly where the sun can be up)."""
    from oracle import insolation_oracle as I
    return I.sun_vector(I.to_unix(t.strftime(FMT)) + 1800.0, DEFAULT_LAT, DEFAULT_LON)[2]


def _hourly(start, n):
    t0 = datetime.strptime(start, FMT)
    return [t0 + timedelta(hours=i) for i in range(n)]


def polar_night(n=48, seed=31):
    rng = np.random.default_rng(seed)
    rows = []
    for i, t in enumerate(_hourly("20221210 00:00:00", n)):
        t_air = -18.0 + 9.0 * math.sin(i / 7.0) + 1.0 * rng.standard_normal()
        t_air = min(max(t_air, -28.0), -8.0)
        wind = float(np.clip(7.5 + 7.5 * math.sin(i / 5.0 + 0.3) + rng.standard_normal(), 0.0, 15.0))
        rows.append(_row(t, t_air, wind, 998.0 + 12.0 * math.sin(i / 17.0), float(np.clip(70 + 30 * math.sin(i / 9.0), 40, 100)),
                         float(np.clip(0.5 + 0.5 * math.sin(i / 6.0), 0, 1)), 0.0))
    return rows


def polar_dawn(n=48, start="20220219 12:00:00", seed=32):
    """Hourly rows around the first (February) or last (October) sunrises of 78 N: the sun stands a
    degree or two above the horizon for a few hours around noon.  SWD is a few W m-2 while it is up (several
    times the clear-sky potential of a sun that low) and 1 W m-2 of twilight while it is just below."""
    rng = np.random.default_rng(seed)
    rows = []
    for i, t in enumerate(_hourly(start, n)):
        u = _sun_up(t)
        swd = 3.0 + 1500.0 * u + 0.3 * rng.random() if u > 0 else (1.0 if u > -0.06 else 0.0)
        t_air = -14.0 + 3.0 * math.sin(i / 9.0) + 0.8 * rng.standard_normal()
        wind = float(np.clip(4.0 + 3.0 * math.sin(i / 6.0) + rng.standard_normal(), 0.0, 14.0))
        rows.append(_row(t, t_air, wind, 1003.0 + 6.0 * math.sin(i / 13.0), float(np.clip(75 + 20 * math.sin(i / 7.0), 30, 100)),
                         float(np.clip(0.4 + 0.6 * math.sin(i / 8.0 + 1.0), 0, 1)), swd))
    return rows


def cold_unstable(n=40, seed=33):
    """Air colder than the 0 degC surface in most rows, the neutral row 0.00 and +-0.01 among them."""
    rng = np.random.default_rng(seed)
    special = {3: 0.0, 4: -0.01, 9: 0.0, 10: 0.01, 17: 0.0, 23: -0.01, 30: 0.0, 31: 0.01, 38: 0.0}
    rows = []
    for i, t in enumerate(_hourly("20220405 00:00:00", n)):
        t_air = special.get(i, -0.01 - 29.99 * rng.random() ** 1.5)
        wind = float(np.clip(5.0 + 4.0 * math.sin(i / 4.0) + rng.standard_normal(), 0.0, 18.0))
        if i % 11 == 7:
            wind = 0.0
        u = _sun_up(t)
        swd = max(0.0, 60.0 * u) if u > 0 else 0.0
        rows.append(_row(t, t_air, wind, 990.0 + 15.0 * math.sin(i / 11.0), float(np.clip(60 + 35 * math.sin(i / 5.0), 20, 100)),
                         float(np.clip(0.5 + 0.5 * math.sin(i / 3.0), 0, 1)), swd))
    return rows


def extremes(n=36, seed=34):
    """Cycles through calm warm air, gales, saturated and dry air, clear and overcast sky; the station
    stands high (600-660 hPa; the case's DEM is raised by 3000 m to match)."""
    rng = np.random.default_rng(seed)
    rows = []
    for i, t in enumerate(_hourly("20220710 00:00:00", n)):
        kind = i % 6
        t_air = 2.0 + 3.0 * rng.random()
        wind = 3.0 + 4.0 * rng.random()
        hum = 40.0 + 50.0 * rng.random()
        cld = rng.random()
        if kind == 0:                       # calm (0 -> 0.1 m/s) under warm air: strongly stable
            t_air, wind = 10.0 + 5.0 * rng.random(), 0.0
        elif kind == 1:                     # gale
            wind = 25.0 + 15.0 * rng.random()
        elif kind == 2:
            hum = 100.0
        elif kind == 3:
            hum = 10.0
        elif kind == 4:
            cld = 0.0
        else:
            cld = 1.0
        if i % 7 == 3:
            wind = 40.0 if i % 2 else 25.0
        u = _sun_up(t)
        swd = max(0.0, 700.0 * u * (1.0 - 0.7 * cld))
        rows.append(_row(t, t_air, wind, 630.0 + 30.0 * math.sin(i / 5.0), hum, cld, swd))
    return rows


# the time steps of irregular_time after its first (63.75 h) row, repeated: 10 min, 50 min, 1 h, 3 h and a
# 7 h logger gap -- 12 h, so that the rows keep landing on midnight (and on the albedo map date)
IRREGULAR_CYCLE_S = (600, 3000, 3600, 10800, 25200)


def irregular_time(cycles=16, seed=35):
    """One 63.75 h row in the midnight sun (255 sunlit sub-steps), then rows of mixed lengths into the
    first nights of late August (sub-steps 0 .. 28, partial last sub-steps)."""
    rng = np.random.default_rng(seed)
    t = datetime.strptime("20220817 08:15:00", FMT)
    times = [t]
    t += timedelta(hours=63.75)
    for _ in range(cycles):
        for dt in IRREGULAR_CYCLE_S:
            times.append(t)
            t += timedelta(seconds=dt)
    times.append(t)
    rows = []
    for i, t in enumerate(times):
        u = _sun_up(t)
        swd = max(0.0, 550.0 * u * (0.8 + 0.2 * rng.random())) if u > 0 else 0.0
        rows.append(_row(t, 1.0 + 4.0 * math.sin(i / 6.0) + 0.5 * rng.standard_normal(),
                         float(np.clip(4.0 + 3.0 * math.sin(i / 4.0), 0.0, 12.0)), 995.0 + 5.0 * math.sin(i / 9.0),
                         float(np.clip(80.0 + 15.0 * math.sin(i / 5.0), 30, 100)), float(np.clip(0.5 + 0.5 * math.sin(i / 3.0), 0, 1)),
                         swd))
    return rows


def msm_season(n=2200, seed=36):
    """Hourly rows from 15 August: the last midnight sun, polar sunset (late October), freeze-up."""
    rng = np.random.default_rng(seed)
    rows = []
    for i, t in enumerate(_hourly("20220815 00:00:00", n)):
        days = i / 24.0
        u = _sun_up(t)
        t_air = 2.0 - 0.22 * days + 3.0 * math.sin(2.0 * math.pi * (t.hour - 9.0) / 24.0) * max(0.0, 1.0 - days / 60.0) \
            + 2.0 * math.sin(i / 61.0) + 0.6 * rng.standard_normal()
        wind = float(np.clip(5.0 + 3.5 * math.sin(i / 37.0) + rng.standard_normal(), 0.0, 20.0))
        if i % 41 == 40:
            wind = 0.0
        cld = float(np.clip(0.5 + 0.5 * math.sin(i / 41.0 + 2.0), 0.0, 1.0))
        swd = max(0.0, 650.0 * u * (1.0 - 0.6 * cld)) if u > 0 else 0.0
        rows.append(_row(t, t_air, wind, 995.0 + 9.0 * math.sin(i / 61.0), float(np.clip(78 + 17 * math.sin(i / 29.0 + 1.0), 30, 100)),
                         cld, swd))
    return rows


def _albedo_dates(rows, inner=()):
    """Map dates bracketing the run (a day before the first row, a day after the last) plus `inner` ones."""
    first = datetime.strptime(rows[0]["DATE"], FMT) - timedelta(days=1)
    last = datetime.strptime(rows[-1]["DATE"], FMT) + timedelta(days=1)
    return sorted({first.strftime("%Y%m%d"), last.strftime("%Y%m%d"), *inner})


REGIMES = {
    "polar_night": (polar_night, ()),
    "polar_dawn": (polar_dawn, ()),
    "polar_dusk": (lambda: polar_dawn(start="20221019 12:00:00", seed=37), ()),
    "cold_unstable": (cold_unstable, ("20220406",)),
    "extremes": (extremes, ()),
    "irregular_time": (irregular_time, ("20220825",)),     # a row at 20220825 00:00:00: span 0
    "msm_season": (msm_season, ("20220915", "20221101")),
}

# model options of each regime (parity.compare_run keywords)
REGIME_KW = {
    "polar_night": dict(),
    "polar_dawn": dict(),
    "polar_dusk": dict(),
    "cold_unstable": dict(),
    "extremes": dict(),
    "irregular_time": dict(last_snowfall="20220822"),
    "msm_season": dict(msm=MSM7, snow_density=350.0, last_snowfall="20220901"),
}

# the DEM shift of a regime [m] (extremes: a high glacier, 600-660 hPa at the station)
DEM_SHIFT = {"extremes": 3000.0}


def make_regime_case(name, h=48, w=56, seed=17, rows=None):
    """SyntheticCase of a regime: make_case's DEM, albedo maps and SWE on an h x w raster, the regime's rows
    (or `rows`), albedo map dates that span them, the AWS cell in the middle of the raster at 78 N."""
    make_rows, inner = REGIMES[name]
    rows = make_rows() if rows is None else rows
    cell = 10.0
    dem = make_dem(h, w, seed=seed, cell=cell)
    dem = (dem.astype(np.float64) + DEM_SHIFT.get(name, 0.0)).astype(np.float32)
    gt = (DEFAULT_ULX, cell, 0.0, DEFAULT_ULY, 0.0, -cell)
    albedo = make_albedo_maps(h, w, _albedo_dates(rows, inner), seed=seed + 1, nan_like=dem)
    swe = make_swe(dem, seed=seed + 2)
    r, c = h // 2, w // 2
    if np.isnan(dem[r, c]):
        raise ValueError("AWS cell is off-glacier")
    return SyntheticCase(dem=dem, geotransform=gt, cell=cell, albedo_maps=albedo, swe=swe, aws_rows=rows,
                         elev_aws=float(np.float32(dem[r, c])), xy_aws=(gt[0] + (c + 0.5) * cell, gt[3] - (r + 0.5) * cell),
                         aws_rc=(r, c), meta={"regime": name, "n_steps": len(rows), "seed": seed})
