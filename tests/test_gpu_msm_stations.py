"""The sub-surface model together with the station blend and the cloud attenuation of the shortwave
(BASELINE config C4 with msm.use) through the C ABI, against the specification in oracle/enrgy_oracle.py:
the blended T, p and e feed the flux sum that drives the conduction step, and the surface temperature of the
point solve is sampled from the distributed (blended) layer temperatures at the AWS cell."""
import csv
import dataclasses
import os

import numpy as np
import pytest

from enrgy_b200 import Energy, _lib
from enrgy_b200.raster_utils import save_npy_raster
from enrgy_b200.synthetic import make_case, make_station_rows
from oracle import insolation_oracle as I
from tests import parity as P
from tests.test_gpu_launch_paths import _chunk_into

pytestmark = pytest.mark.gpu

LAYERS = dict(depths=[0.1, 0.1, 0.3, 0.5, 0.5, 0.5, 3.0],
              temperatures=[-6.9, -6.93, -7.025, -7.31, -6.93, -7.12, -7.0, -5.57], elev=275.0)
MSM = dict(msm=LAYERS, snow_density=350.0, last_snowfall="20220522")
MODES = {"streamed": dict(), "computed": dict(computed=True), "shadow": dict(computed=True, shadow=True)}


def _case(n_steps):
    # (on this case the float32 oracle's own melt-flux gap to its float64 self is at least 6e-4 W m-2 in every
    # mode and station set below, above the 5e-4 that compare_run's float32 sub-surface floor requires)
    return make_case(80, n_steps, w=96, seed=9)


def _stations(case, n):
    h, w = case.shape
    spots = [(0.18 * h, 0.30 * w, 140.0, 11), (0.80 * h + 0.37, 0.62 * w + 0.5, -90.0, 12), (0.45 * h, 0.85 * w, 60.0, 13)]
    return [dict(row=r, col=c, elev=case.elev_aws + dz, rows=make_station_rows(case, case.elev_aws + dz, seed=sd))
            for (r, c, dz, sd) in spots[:n]]


def _oracle_layers_at_aws(case, pot, **kw):
    """[T, layers + 1] float64 oracle boundary temperatures at the AWS cell before each row's tick.  Row m >= 2
    is the final state of the oracle run over the first m rows (on this uniform time base the last row of the
    shorter table takes the same time step as in the full one); row 0 is the initial state.  A one-row table
    has no time step, so row 1 carries only its surface value, the point_t_surf of the full run."""
    n = len(case.aws_rows)
    r, c = case.aws_rc
    full = P.run_oracle(case, pot, True, **kw)
    out = np.full((n, len(LAYERS["depths"]) + 1), np.nan)
    out[:, 0] = [row["point_t_surf"] for row in full["rows"]]
    for m in range(2, n):
        part = P.run_oracle(dataclasses.replace(case, aws_rows=case.aws_rows[:m]), pot[:m], True, **kw)
        out[m] = [float(t[r, c]) for t in part["layer_temperatures"]]
    d = np.asarray(case.dem, dtype=np.float64)[r, c] - LAYERS["elev"]
    out[0] = [min(t + d * -0.006, 0.0) for t in LAYERS["temperatures"]]
    return full, out


@pytest.mark.parametrize("f64", [True, False])
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("n_extra,cloud_k", [(1, None), (1, 0.5), (3, None), (3, 0.7)])
def test_msm_with_stations_against_the_oracle(f64, mode, n_extra, cloud_k):
    """Per-step flux rasters, melt, final state, layer temperatures, the area means and the Monin-Obukhov
    length: 1e-9 (float64) / 1e-4 (float32, with the sub-surface floors of compare_run)."""
    case = _case(30)
    pot = P.random_insolation(case, 30) if mode == "streamed" else None
    res = P.compare_run(case, f64, pot=pot, stations=_stations(case, n_extra), cloud_k=cloud_k, **MODES[mode], **MSM)
    tol = 1e-9 if f64 else 1e-4
    bad = {k: v for k, v in res.items() if v >= tol and not k.endswith("_l2")}
    assert not bad, bad


def _close_sums(a, b, rtol):
    """Area sums that agree to rounding: relative to the value or, for columns that cross zero, to the
    column's largest value."""
    scale = np.abs(b).max(axis=0, keepdims=True)
    return bool((np.abs(a - b) <= rtol * (np.abs(b) + scale)).all())


@pytest.mark.parametrize("f64", [True, False])
@pytest.mark.parametrize("mode", list(MODES))
def test_msm_with_the_primary_station_alone_equals_plain_msm(f64, mode):
    """No extra station: the blend instance (weights, folded vapour-pressure factors, exp(0) cloud factor,
    one pair of cells per thread) gives the plain sub-surface run's rasters and layer temperatures -- bit for
    bit in float32, to a few ulp in float64 -- and the pre-pass integrates the AWS cell identically."""
    case = _case(20)
    pot = P.random_insolation(case, 20) if mode == "streamed" else None
    out = []
    for st in (None, []):
        eng = P.make_engine(case, f64, pot=pot, stations=st, cloud_k=0.8, **MODES[mode], **MSM)
        try:
            stats = eng.run(0, 20)
            out.append((eng.state(np.float64) + (eng.layer_temps(),), stats, eng.point_scalars(), eng.point_layers()))
        finally:
            eng.close()
    (plain, s_plain, pt_plain, pl_plain), (blend, s_blend, pt_blend, pl_blend) = out
    for a, b in zip(blend, plain):
        if f64:
            # (float64 reciprocals are Newton steps from a hardware seed, scheduled differently per instance)
            assert np.array_equal(np.isnan(a), np.isnan(b)) and np.allclose(a, b, rtol=1e-13, atol=1e-15, equal_nan=True)
        else:
            assert np.array_equal(a, b, equal_nan=True)
    # (the longwave area sum comes from the kernel instead of the DEM moments; float32 sums in another order)
    assert _close_sums(s_blend, s_plain, 1e-11 if f64 else 3e-6)
    assert np.array_equal(pt_blend, pt_plain) and np.array_equal(pl_blend, pl_plain)


def test_aws_cell_integrates_the_blend():
    """float64: the pre-pass integrates the AWS cell in the blended meteorology of that cell, so its boundary
    temperatures before every row (enrgy_get_point_layers) and the surface temperature of the point solve
    (ENRGY_P_TSURF_AWS) are the oracle's, sampled from the distributed field, within 1e-9."""
    case = _case(16)
    pot = P.random_insolation(case, 16)
    kw = dict(stations=_stations(case, 3), cloud_k=0.7, **MSM)
    ora, want = _oracle_layers_at_aws(case, pot, **kw)
    eng = P.make_engine(case, True, pot=pot, **kw)
    try:
        layers = eng.point_layers()
        point = eng.point_scalars()
    finally:
        eng.close()
    have = ~np.isnan(want)
    assert have.sum() == want.size - (want.shape[1] - 1)
    assert P.max_rel_err(layers[have], want[have], 1e-3) < 1e-9
    assert P.max_rel_err(point[:, _lib.P_TSURF_AWS], [r["point_t_surf"] for r in ora["rows"]], 1e-3) < 1e-9
    # the distributed fluxes at the AWS cell that debug_point_output prints
    r, c = case.aws_rc
    for col, name in ((_lib.P_SENS_AWS, "sens"), (_lib.P_LAT_AWS, "lat")):
        assert P.max_rel_err(point[:, col], [float(row[name][r, c]) for row in ora["rows"]], 1e-3) < 1e-9, name


def test_msm_with_stations_on_row_bands():
    """float32 with shading: two row bands, one of them without the AWS cell (it gets that cell's values by
    enrgy_set_aws_cell), give the whole run's rasters and layer temperatures bit for bit, the same pre-pass,
    and area sums that add up."""
    case = _case(20)
    kw = dict(computed=True, shadow=True, stations=_stations(case, 3), cloud_k=0.7, **MSM)
    whole = P.make_engine(case, False, **kw)
    try:
        s_whole = whole.run(0, 20)
        st_whole = whole.state(np.float32) + (whole.layer_temps(),)
        pre_whole = (whole.point_scalars(), whole.point_layers())
    finally:
        whole.close()
    assert case.aws_rc[0] < 48
    total = np.zeros_like(s_whole)
    for r0, nr in ((0, 48), (48, 32)):
        eng = P.make_engine(case, False, band=(r0, nr), **kw)
        try:
            total += eng.run(0, 20)
            part = eng.state(np.float32) + (eng.layer_temps(),)
            pre = (eng.point_scalars(), eng.point_layers())
        finally:
            eng.close()
        for a, b in zip(part, st_whole):
            assert np.array_equal(a, b[..., r0:r0 + nr, :], equal_nan=True)
        assert all(np.array_equal(a, b) for a, b in zip(pre, pre_whole))
    cols = [_lib.S_RS, _lib.S_LWD, _lib.S_LWU, _lib.S_SENS, _lib.S_LAT, _lib.S_G, _lib.S_MELT, _lib.S_SNOW, _lib.S_ICE]
    assert _close_sums(total[1:, cols], s_whole[1:, cols], 3e-6)


@pytest.mark.parametrize("f64", [True, False])
def test_msm_with_stations_cut_into_mask_chunks(f64):
    """With shading, a run cut into at least three mask chunks: float64 equals the run in one piece bit for bit
    (statistics, state, layer temperatures); float32 is held to the oracle (its plain sub-surface path
    already differs from the one-piece run in the last bits when cut, test_gpu_launch_paths)."""
    n = 16
    case = _case(n)
    kw = dict(computed=True, shadow=True, stations=_stations(case, 2), cloud_k=0.7, **MSM)
    out = {}
    for cut in ((False, True) if f64 else (True,)):
        eng = P.make_engine(case, f64, **kw)
        try:
            if cut:
                _chunk_into(eng, 3)
            stats = eng.run(0, n)
            out[cut] = (stats, eng.state(np.float64), eng.layer_temps())
        finally:
            eng.close()
    if f64:
        assert np.array_equal(out[True][0], out[False][0])
        for a, b in zip(out[True][1] + (out[True][2],), out[False][1] + (out[False][2],)):
            assert np.array_equal(a, b, equal_nan=True)
        return
    stats, (swe, tsn, tic), layers = out[True]
    ora = P.run_oracle(case, P.oracle_insolation(case, None, True, True, False), False, **kw)
    for got, want in ((swe, ora["swe"]), (tsn, ora["total_snow"]), (tic, ora["total_ice"])):
        assert P.max_rel_err(got, want, 1e-3) < 1e-4
    for got, want in zip(layers, ora["layer_temperatures"]):
        assert P.max_rel_err(got, want, 1.0) < 1e-4
    floors = np.array([1.0] * 8 + [1e-3, 1e-3, 1e-3, 0.5, 0.5])
    m_e, m_o = P.means_from_stats(stats), ora["means"]
    assert float(np.max(np.abs(m_e - m_o) / np.maximum(np.abs(m_o), floors))) < 1e-4


def test_energy_class_with_msm_and_stations(tmp_path):
    """Through the reference-shaped class: add_msm, two add_station files, add_cloud_transmissivity and
    debug_point_output with msm_xy at the AWS cell.  The printed layer temperatures and fluxes at the AWS cell
    are the oracle's to the printed precision; the ice melt is the oracle's and measurably not the one of the
    sub-surface run without the extra stations."""
    case = _case(16)
    d = str(tmp_path)
    dem = save_npy_raster(os.path.join(d, "dem.npy"), case.dem, case.geotransform)
    swe = save_npy_raster(os.path.join(d, "swe.npy"), case.swe, case.geotransform)
    alb = {k: save_npy_raster(os.path.join(d, "alb_%s.npy" % k), a, case.geotransform) for k, a in case.albedo_maps.items()}
    aws = case.write_aws_csv(os.path.join(d, "aws.csv"))
    e = Energy(dem, None, os.path.join(d, "out"), res=10, precision="f64")
    e.lat, e.lon = case.lat, case.lon
    e.add_snow(swe)
    e.add_msm(LAYERS["depths"], LAYERS["temperatures"], LAYERS["elev"])
    e.msm_xy = case.xy_aws
    e.debug_point_output = "point.csv"
    ul_x, x_dist, _, ul_y, _, y_dist = case.geotransform
    stations = _stations(case, 2)
    for k, st in enumerate(stations):
        path = os.path.join(d, "station%d.csv" % k)
        with open(path, "w", newline="") as f:
            wr = csv.DictWriter(f, fieldnames=list(st["rows"][0]))
            wr.writeheader()
            wr.writerows(st["rows"])
        e.add_station(path, (ul_x + (st["col"] + 0.5) * x_dist, ul_y + (st["row"] + 0.5) * y_dist), st["elev"])
    e.add_cloud_transmissivity(0.6)
    e.model(aws_file=aws, albedo_maps=alb, z=1.6, elev_aws=case.elev_aws, xy_aws=case.xy_aws, zm=1e-3,
            z_h_or_e=1e-4, emissivity=0.98, last_snowfall="20220522", v=False)
    pot = I.insolation_series(case, shadow=True, dtype=np.float64)
    okw = dict(msm=LAYERS, last_snowfall="20220522")
    ora, want = _oracle_layers_at_aws(case, pot, stations=stations, cloud_k=0.6, **okw)
    # (the class keeps its state rasters in float32 like the reference, model.py:76-80)
    assert P.max_rel_err(e.total_ice_melt_array, ora["total_ice"], 1e-3) < 2e-7
    plain = P.run_oracle(case, pot, True, **okw)
    assert P.max_rel_err(e.total_ice_melt_array, plain["total_ice"], 1e-3) > 1e-3
    lines = open(os.path.join(d, "out", "point.csv")).read().split("\n")
    depth, header = 0.0, "0.0,"
    for x in LAYERS["depths"]:
        depth += x
        header += "%s," % depth
    assert lines[0] == header + "SENSIBLE,LATENT"
    assert len(lines) == 1 + len(case.aws_rows)
    r, c = case.aws_rc
    for i, line in enumerate(lines[1:]):
        f = line.split(",")
        assert f[0] == case.aws_rows[i]["DATE"]
        vals = [float(x) for x in f[1:]]
        for got, ref in zip(vals[:-2], want[i]):
            assert np.isnan(ref) or abs(got - ref) <= 0.0051, (i, got, ref)
        assert abs(vals[-2] - float(ora["rows"][i]["sens"][r, c])) <= 0.0501
        assert abs(vals[-1] - float(ora["rows"][i]["lat"][r, c])) <= 0.0501


def test_run_members_refuses_msm_with_stations():
    case = make_case(40, 6, w=56, seed=3)
    eng = P.make_engine(case, True, pot=P.random_insolation(case, 6), stations=_stations(case, 1), cloud_k=0.5, **MSM)
    try:
        with pytest.raises(_lib.EnrgyError) as err:
            eng.run_members([0.0, 0.1])
        assert err.value.code == _lib.ERR_ARG
        assert np.isfinite(eng.run(0, 6)).all()
    finally:
        eng.close()
