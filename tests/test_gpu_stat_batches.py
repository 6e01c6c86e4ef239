"""The fused kernel sums its per-step area statistics over a warp in batches of steps (kernels.cu,
StatBatchFor: up to 4 entries in float32, 2 in float64 and with sunlit masks; with fused members a batch
holds (step, member) pairs; the sub-surface model reduces every step).  A batch that a run, a time block
or the start of a run cuts short is summed on its own; these runs make every such cut and check that the
statistics and state rasters do not depend on where a batch ends, bit for bit."""
import numpy as np
import pytest

from enrgy_b200.ensemble import make_members
from enrgy_b200.synthetic import make_case
from tests import parity as P

pytestmark = pytest.mark.gpu

MSM = dict(msm=dict(depths=[0.25, 0.5, 1.0], temperatures=[-2.0, -3.0, -4.0, -5.0], elev=400.0),
           snow_density=350.0, last_snowfall="20220522")
# runs shorter than, one short of, one past and 2 S + 3 past a batch of S = 1, 2 or 4 entries
PREFIXES = (1, 2, 3, 4, 5, 7, 9, 11)
# time blocks: hourly rows with shading fill 64-step blocks (a season of 64 + 3 steps ends in a block of
# 3); daily rows (96 sub-steps each) cut a block after two steps
FORCINGS = {"hourly": dict(n_steps=67, step_s=3600), "daily": dict(n_steps=13, step_s=86400)}


def _case(forcing):
    f = FORCINGS[forcing]
    return make_case(40, f["n_steps"], w=72, seed=17, step_s=f["step_s"], start="20220620 00:00:00")


def _split_state_equal(got, want, f64):
    # swe and total_ice are carried step by step; total_snow is added once per run as swe(start) - swe(end),
    # so a run cut in pieces rounds it differently in the last bit (as test_gpu_edge_cases states)
    assert np.array_equal(got[0], want[0], equal_nan=True)
    assert np.array_equal(got[2], want[2], equal_nan=True)
    assert np.allclose(got[1], want[1], rtol=1e-13 if f64 else 1e-6, atol=0, equal_nan=True)


@pytest.mark.parametrize("forcing", sorted(FORCINGS))
@pytest.mark.parametrize("mode", ["plain", "msm"])
@pytest.mark.parametrize("f64", [False, True])
def test_runs_cut_at_any_step(f64, mode, forcing):
    """A run of n steps gives the first n statistic rows of the whole run; a run cut at steps 5 and 30 (no
    multiple of any batch size) gives the whole run's statistics and rasters."""
    case = _case(forcing)
    n = len(case.aws_rows)
    kw = MSM if mode == "msm" else {}
    eng = P.make_engine(case, f64, computed=True, shadow=forcing == "hourly", **kw)
    try:
        eng.snapshot(save=True)
        whole = eng.run(0, n)
        whole_state = eng.state(np.float64)
        for k in PREFIXES:
            eng.snapshot(save=False)
            assert np.array_equal(eng.run(0, k), whole[:k]), k
        # (float32 sub-surface model: a launch restarts the float64 accumulator of the top boundary
        # temperature from its float32 raster, so a run cut in pieces differs in the last bits anyway)
        if mode == "msm" and not f64:
            return
        a, b = 5, min(30, n - 1)
        eng.snapshot(save=False)
        cut = np.concatenate([eng.run(0, a), eng.run(a, b), eng.run(b, n)])
        assert np.array_equal(cut, whole)
        _split_state_equal(eng.state(np.float64), whole_state, f64)
    finally:
        eng.close()


@pytest.mark.parametrize("forcing", sorted(FORCINGS))
@pytest.mark.parametrize("f64", [False, True])
def test_fused_members_runs_of_any_length(f64, forcing):
    """Three fused members: a run of n steps gives the first n statistic rows of every member's whole run,
    and the member rasters equal those of the pass without statistics (no batch).  (A members run starts
    every member from the handle's state, so it cannot be cut and continued.)"""
    case = _case(forcing)
    n = len(case.aws_rows)
    members = make_members(3, seed=5, albedo_sigma=0.05)
    off = [m["albedo_offset"] for m in members]
    zm = [m["zm"] for m in members]
    zh = [m["z_h_or_e"] for m in members]
    eng = P.make_engine(case, f64, computed=True, shadow=forcing == "hourly")
    try:
        whole, _ = eng.run_members(off, zm, zh, 0, n)
        rasters = [eng.member_state(k, np.float64) for k in range(len(members))]
        eng.run_members(off, zm, zh, 0, n, want_stats=False)
        for k in range(len(members)):
            for a, b in zip(eng.member_state(k, np.float64), rasters[k]):
                assert np.array_equal(a, b, equal_nan=True), k
        for k in PREFIXES:
            stats, _ = eng.run_members(off, zm, zh, 0, k)
            assert np.array_equal(stats, whole[:, :k]), k
    finally:
        eng.close()
