"""The station-blend specification together with the sub-surface model (oracle/enrgy_oracle.py, "several
weather stations" and msm.py): with no extra station the blend must BE the reference-pinned sub-surface
path, bit for bit, in both dtype configurations."""
import numpy as np
import pytest

from enrgy_b200.synthetic import make_case
from tests import parity as P

MSM = dict(msm=dict(depths=[0.1, 0.1, 0.3, 0.5, 0.5, 0.5, 3.0],
                    temperatures=[-6.9, -6.93, -7.025, -7.31, -6.93, -7.12, -7.0, -5.57], elev=275.0),
           snow_density=350.0, last_snowfall="20220522")


@pytest.mark.parametrize("f64", [False, True])
def test_msm_with_the_primary_station_alone_is_plain_msm_bit_for_bit(f64):
    case = make_case(40, 12, w=56, seed=3)
    pot = P.random_insolation(case, 12)
    ref = P.run_oracle(case, pot, f64, **MSM)
    got = P.run_oracle(case, pot, f64, stations=[], cloud_k=0.8, **MSM)
    for k in ("swe", "total_snow", "total_ice"):
        assert np.array_equal(ref[k], got[k], equal_nan=True), k
    for a, b in zip(ref["layer_temperatures"], got["layer_temperatures"]):
        assert a.dtype == b.dtype and np.array_equal(a, b, equal_nan=True)
    assert ref["stats_csv"] == got["stats_csv"]
    for a, b in zip(ref["rows"], got["rows"]):
        assert a["point_t_surf"] == b["point_t_surf"] and a["L"] == b["L"]
        for fld in P.FLUX_FIELDS:
            assert a[fld].dtype == b[fld].dtype and np.array_equal(a[fld], b[fld], equal_nan=True), fld
