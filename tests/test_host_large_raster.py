"""Rasters of more than 32 767 rows or columns on the host: the pre-pass's shading ray of the AWS cell.

enrgy_host_prepass runs without a device.  With computed insolation and shading it marches the ray of
the AWS cell along its Q16 scan line; the shear u * dfix of that line passes 2^31 once u * |dfix| does,
which on a raster of 70 000 rows happens for any sun more than ~25 degrees off an axis.  The raster here
is flat up to two rows past the AWS cell and a 3000 m plateau beyond, in the direction of one chosen
sub-step: the AWS cell sits where that sub-step's shear crosses 2^31 between the cell and its neighbour,
so a 32-bit shear would lose the plateau behind the crossing and read the cell as sunlit.  Every row's
potential insolation and shortwave factor at the AWS cell is checked against the oracle's traced ray.
"""
import numpy as np
import pytest

from enrgy_b200 import _lib
from enrgy_b200.engine import host_prepass
from enrgy_b200.forcing import build_forcing
from enrgy_b200.synthetic import make_aws_rows
from oracle import insolation_oracle as I
from oracle.enrgy_oracle import time_step_seconds

LONG = 70_000                         # cells along the long axis
SHORT = 24
CELL = 10.0
LAT, LON = 77.98, 14.10
KEYS = ["20220520", "20220615"]


def _tables(rows):
    out = []
    for i, row in enumerate(rows):
        dt = time_step_seconds(rows, i)
        out.append((I.to_unix(row["DATE"]), dt, I.substep_table(I.to_unix(row["DATE"]), dt, LAT, LON, CELL)))
    return out


def _case(tall):
    """(dem, aws (row, col), aws_rows, the chosen sub-step's dfix): scan lines along the long axis
    (row type on the tall raster, column type on the wide one) with sigma = +1, i.e. u = index along that
    axis and the sun toward growing indices."""
    aws_rows = make_aws_rows(24)
    subs = [s for _, _, table in _tables(aws_rows) for s in table]
    cand = []
    for s in subs:
        row_type, sigma, dfix = I.line_geometry(s["dc_fix"], s["dr_fix"])
        if row_type == tall and sigma == 1 and dfix > 0 and dfix * (LONG - 16) > 2 ** 31:
            cand.append(dfix)
    assert cand, "no sub-step of the day shears past 2^31 on this raster"
    dfix = min(cand)                                    # the AWS cell as far along the axis as fits
    u_aws = (2 ** 31 - 32768 - 1) // dfix               # u * dfix + 32768 < 2^31 <= (u + 1) * dfix + 32768
    assert u_aws * dfix + 32768 < 2 ** 31 <= (u_aws + 1) * dfix + 32768
    assert 32768 < u_aws < LONG - 3
    dem = np.zeros((LONG, SHORT), dtype=np.float32)
    dem[u_aws + 2:] = 3000.0
    aws = (u_aws, SHORT // 2)
    if not tall:
        dem = np.ascontiguousarray(dem.T)
        aws = aws[::-1]
    return dem, aws, aws_rows, dfix


@pytest.mark.parametrize("tall", [True, False], ids=["tall", "wide"])
def test_aws_ray_beyond_32768_cells(tall):
    dem, (r, c), aws_rows, dfix = _case(tall)
    table = build_forcing(aws_rows, KEYS)
    point = host_prepass(dem, table, precision=_lib.F64, cell_size=CELL, elev_aws=0.0, aws_row=r, aws_col=c,
                         sensor_z=1.6, zm=1e-3, z_h_or_e=1e-4, insol_mode=_lib.INSOL_COMPUTED, shadow=True,
                         lat=LAT, lon=LON)
    big = 0
    shaded_at_crossing = False
    for i, (t, dt, subs) in enumerate(_tables(aws_rows)):
        want = I.potential_insolation_window(dem, CELL, LAT, LON, t, dt, (r, r + 1, c, c + 1), shadow=True)[0, 0]
        got = point[i, _lib.P_POT_AWS] * dt / 3.6e6                     # W m-2 over the step -> kWh m-2
        assert abs(got - want) <= 1e-9 * max(abs(want), 1e-6), (i, got, want)
        pot_w = want * 3.6e6 / dt
        f_ref = 1.0 if pot_w == 0 else float(aws_rows[i]["SWD"]) / pot_w
        assert abs(point[i, _lib.P_SW_FACTOR] - f_ref) <= 1e-9 * max(abs(f_ref), 1e-12), (i, point[i, _lib.P_SW_FACTOR], f_ref)
        assert int(point[i, _lib.P_NSUB]) == len(subs)
        for s in subs:
            row_type, sigma, d = I.line_geometry(s["dc_fix"], s["dr_fix"])
            u1 = sigma * (r if row_type else c) + 1                     # first cell of the ray past the AWS cell
            big = max(big, abs(u1 * d))
            if d == dfix and row_type == tall and sigma == 1:
                lit = I.trace_cells(dem, np.array([r]), np.array([c]), s["dc_fix"], s["dr_fix"], s["dz"])[0]
                shaded_at_crossing |= not lit
    # a 32-bit shear overflows on this case, and the plateau behind the crossing shades the AWS cell
    assert big >= 2 ** 31
    assert shaded_at_crossing


def test_host_prepass_size_bound():
    """1 .. 2^20 cells a side: the largest raster is accepted (streamed insolation: no ray), one more
    row or column is refused with ENRGY_ERR_ARG."""
    n = 1 << 20
    table = build_forcing(make_aws_rows(2), KEYS)
    base = dict(cell_size=CELL, elev_aws=0.0, sensor_z=1.6, zm=1e-3, z_h_or_e=1e-4, insol_mode=_lib.INSOL_STREAMED,
                lat=LAT, lon=LON)
    pot = np.full(2, 100.0)
    point = host_prepass(np.zeros((n, 1), np.float32), table, pot_aws=pot, aws_row=n - 1, aws_col=0, **base)
    assert np.all(np.isfinite(point[:, _lib.P_SW_FACTOR]))
    point = host_prepass(np.zeros((1, n), np.float32), table, pot_aws=pot, aws_row=0, aws_col=n - 1, **base)
    assert np.all(np.isfinite(point[:, _lib.P_SW_FACTOR]))
    for shape, aws in (((n + 1, 1), (0, 0)), ((1, n + 1), (0, 0))):
        with pytest.raises(_lib.EnrgyError) as e:
            host_prepass(np.zeros(shape, np.float32), table, pot_aws=pot, aws_row=aws[0], aws_col=aws[1], **base)
        assert e.value.code == _lib.ERR_ARG
