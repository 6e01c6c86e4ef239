"""Rasters of more than 32 767 (and 65 535) rows or columns, up to the 2^20 bound of enrgy_create.

Narrow rasters keep the oracle affordable while the long axis passes the points where 32-bit arithmetic or
launch dimensions used to break: the Q16 shear u * dfix of the shading sweep passes 2^31 (any sun more
than ~25 degrees off an axis on 70 000 cells), and set-up kernels that gave a grid row to each raster row
(or row tile) passed CUDA's grid.y limit of 65 535.  The tall case keeps its AWS cell beyond row 65 536.
"""
import dataclasses

import numpy as np
import pytest

from enrgy_b200 import _lib
from enrgy_b200.engine import Engine
from enrgy_b200.ensemble import make_members, run_members
from enrgy_b200.forcing import build_forcing
from enrgy_b200.synthetic import make_aws_rows, make_case
from oracle import insolation_oracle as I
from oracle.enrgy_oracle import time_step_seconds
from tests import parity as P
from tests.test_gpu_parity import VARIANTS
from tests.test_gpu_stations import _stations

pytestmark = pytest.mark.gpu

LONG = 70_000
NARROW = 64
AWS_ROW = 66_000                      # beyond row 65 536
T = 4


def _tall_case(n_steps=T, rows=LONG, seed=7):
    case = make_case(rows, n_steps, w=NARROW, seed=seed)
    r, c = AWS_ROW, NARROW // 2
    assert not np.isnan(case.dem[r, c])
    gt = case.geotransform
    return dataclasses.replace(case, aws_rc=(r, c), elev_aws=float(case.dem[r, c]),
                               xy_aws=(gt[0] + (c + 0.5) * case.cell, gt[3] - (r + 0.5) * case.cell))


@pytest.fixture(scope="module")
def tall():
    return _tall_case()


@pytest.mark.parametrize("shape", [(LONG, NARROW), (NARROW, LONG)], ids=["tall", "wide"])
def test_masks_bit_exact(shape):
    """enrgy_shade_masks = the specification's masks bit for bit, every sub-step of eight rows three hours
    apart (a day at 78 N: the sun goes all the way round), with shears past 2^31."""
    case = make_case(shape[0], 24, w=shape[1], seed=3)
    eng = P.make_engine(case, False, computed=True, shadow=True)
    try:
        octants = set()
        for step in range(24):
            for s in eng.substeps(step):
                row_type, sigma, dfix = I.line_geometry(int(s[5]), int(s[6]))
                octants.add((row_type, sigma, dfix > 0))
        assert len(octants) == 8, octants
        valid = ~np.isnan(case.dem)
        big = 0
        for step in range(0, 24, 3):
            row = case.aws_rows[step]
            table = I.substep_table(I.to_unix(row["DATE"]), time_step_seconds(case.aws_rows, step), case.lat,
                                    case.lon, case.cell)
            subs = eng.substeps(step)
            masks = eng.shade_masks(step, max_sub=len(subs))
            assert masks.shape[0] == len(table) == len(subs)
            for j, (s, sub) in enumerate(zip(subs, table)):
                assert (int(s[5]), int(s[6])) == (sub["dc_fix"], sub["dr_fix"])
                row_type, _, dfix = I.line_geometry(int(s[5]), int(s[6]))
                na = shape[0] if row_type else shape[1]
                big = max(big, (na - 1) * abs(dfix))        # |u| runs up to na - 1 along the sweep axis
                lit = I.shadow_mask(case.dem, sub["dc_fix"], sub["dr_fix"], sub["dz"])
                assert np.array_equal(masks[j][valid], lit[valid]), (step, j)
        assert big >= 2 ** 31
    finally:
        eng.close()


ORACLE_RUNS = {
    "streamed_f32": (False, dict(streamed=True)),
    "streamed_f64": (True, dict(streamed=True)),
    "computed_f64": (True, dict(computed=True)),
    "shadow_f32": (False, dict(computed=True, shadow=True)),
    "shadow_f64": (True, dict(computed=True, shadow=True)),
    "msm_f64": (True, dict(streamed=True, **VARIANTS["msm"])),
    "stations_f64": (True, dict(streamed=True, stations=2, cloud_k=0.7)),
    "stations_f32": (False, dict(computed=True, shadow=True, stations=3, cloud_k=0.9)),
}


@pytest.mark.parametrize("name", list(ORACLE_RUNS))
def test_energy_balance_against_oracle(tall, name):
    """The tall raster against the oracle at the usual bars (float64 1e-9, float32 1e-4): streamed,
    computed and shaded insolation, the sub-surface model in float64 (2-row tiles: msm_init over 70 000
    rows), the station blend with cloud attenuation; the AWS cell lies beyond row 65 536."""
    f64, kw = ORACLE_RUNS[name]
    kw = dict(kw)
    pot = P.random_insolation(tall, T) if kw.pop("streamed", False) else None
    if "stations" in kw:
        kw["stations"] = _stations(tall, kw["stations"])
    res = P.compare_run(tall, f64, pot=pot, **kw)
    tol = 1e-9 if f64 else 1e-4
    bad = {k: v for k, v in res.items() if v >= tol and not k.endswith("_l2")}
    assert not bad, bad


def test_row_bands_with_shading():
    """Row bands of a 100 000-row raster with shading (one engine per band): a cut above row 32 768 and a
    band of more than 65 535 rows give the whole raster's state bit for bit; so does a band beyond row
    65 536 whose masks the caller sweeps by enrgy_shade_scan and feeds to enrgy_run_masked."""
    import torch
    case = make_case(100_000, T, w=NARROW, seed=9)
    whole = P.make_engine(case, False, computed=True, shadow=True)
    try:
        whole.run(0, T)
        ref = whole.state(np.float64)
    finally:
        whole.close()
    for band in ((0, 32_776), (32_776, 67_224)):
        eng = P.make_engine(case, False, computed=True, shadow=True, band=band)
        try:
            eng.run(0, T)
            got = eng.state(np.float64)
        finally:
            eng.close()
        for a, b in zip(got, ref):
            assert np.array_equal(a, b[band[0]:band[0] + band[1]], equal_nan=True), band
    band = (65_544, 100_000 - 65_544)
    eng = P.make_engine(case, False, computed=True, shadow=True, band=band)
    try:
        s0, s1 = eng.sub_range(0, T)
        buf = torch.zeros(max(s1 - s0, 1) * eng.mask_words(band[1]), dtype=torch.int32, device="cuda")
        eng.shade_scan(s0, s1, [(band[0], band[1], buf.data_ptr())])
        eng.run_masked(0, T, buf.data_ptr())
        eng.synchronize()
        got = eng.state(np.float64)
    finally:
        eng.close()
    for a, b in zip(got, ref):
        assert np.array_equal(a, b[band[0]:], equal_nan=True)


def test_fused_members_on_tall_raster(tall):
    """Fused ensemble members on the tall raster equal one run per member bit for bit."""
    members = make_members(5, seed=3, albedo_sigma=0.08)
    eng = P.make_engine(tall, False, pot=P.random_insolation(tall, T))
    try:
        one = run_members(eng, members, keep_rasters=True, fused=False, want_stats=False)
        eng.snapshot(save=False)
        fused = run_members(eng, members, keep_rasters=True, fused=True, want_stats=False)
    finally:
        eng.close()
    for i in range(len(members)):
        for k in ("swe", "total_snow", "total_ice"):
            assert np.array_equal(one[i][k], fused[i][k], equal_nan=True), (i, k)
    assert not np.array_equal(fused[0]["total_ice"], fused[1]["total_ice"], equal_nan=True)


def test_size_limits():
    """2^20 rows are accepted and run (computed insolation with shading, float32: 131 072 row tiles of the
    fused kernel, 2^20 rows of terrain normals); one row or column more is refused with ENRGY_ERR_ARG."""
    n = 1 << 20
    for shape in ((n + 1, NARROW), (NARROW, n + 1)):
        with pytest.raises(_lib.EnrgyError) as e:
            Engine(*shape)
        assert e.value.code == _lib.ERR_ARG
    r = np.arange(n, dtype=np.float64)[:, None]
    c = np.arange(NARROW, dtype=np.float64)[None, :]
    dem = (500.0 + 40.0 * np.sin(r / 37.0) * np.cos(c / 11.0) + 200.0 * np.sin(r / 5000.0)).astype(np.float32)
    dem[:, :3] = np.nan
    aws = (n - 5, NARROW // 2)
    eng = Engine(n, NARROW, precision=_lib.F32)
    try:
        eng.set_params(cell_size=10.0, elev_aws=float(dem[aws]), aws_row=aws[0], aws_col=aws[1], sensor_z=1.6,
                       zm=1e-3, z_h_or_e=1e-4, const_albedo=(0.35, 0.75), insol_mode=_lib.INSOL_COMPUTED,
                       shadow=True, lat=77.98, lon=14.10)
        eng.set_dem(dem)
        eng.set_forcing(build_forcing(make_aws_rows(3, start="20220601 10:00:00")))
        eng.prepass()
        stats = eng.run(0, 3)
        swe, tsn, tic = eng.state(np.float32)
    finally:
        eng.close()
    assert np.isfinite(stats).all()
    assert stats[:, _lib.S_NVALID].min() == np.count_nonzero(~np.isnan(dem))
    for a in (swe, tsn, tic):
        assert a.shape == dem.shape
        assert np.isfinite(a[~np.isnan(dem)]).all()
