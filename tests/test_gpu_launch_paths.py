"""Launch paths of the fused kernel that must not change a result: runs cut into chunks by the sunlit-mask
budget (fused members, the station blend, the sub-surface model), a debug dump that reuses masks cached
by a run, and the masked run fed chunk by chunk by the caller.  The comparisons are bit for bit unless a
test says otherwise."""
import numpy as np
import pytest

from enrgy_b200 import _lib
from enrgy_b200.ensemble import make_members
from enrgy_b200.synthetic import make_case, make_station_rows
from tests import parity as P

pytestmark = pytest.mark.gpu

N_STEPS = 16
MSM = dict(msm=dict(depths=[0.25, 0.5, 1.0], temperatures=[-2.0, -3.0, -4.0, -5.0], elev=400.0),
           snow_density=350.0, last_snowfall="20220522")


def _case():
    return make_case(64, N_STEPS, w=96, seed=41)


def _engine(case, f64, **kw):
    return P.make_engine(case, f64, computed=True, shadow=True, **kw)


def _chunk_into(eng, n_chunks):
    """Sets a mask budget that cuts a run of all steps into at least n_chunks chunks (the greedy cut of
    the library: whole steps, as many as fit the budget); returns the number of chunks."""
    rows, cols = eng.band_rows, eng.cols
    per_sub = 4 * (eng.mask_words(rows) + cols * (((rows + 31) // 32 + 7) // 8 * 8))
    counts = [int(x) for x in eng.point_scalars()[:, _lib.P_NSUB]]
    max_subs = max(max(counts), sum(counts) // (n_chunks + 1))
    eng.set_mask_budget(max_subs * per_sub)
    chunks, held = 0, None
    for k in counts:
        if held is None or held + k > max_subs:
            chunks, held = chunks + 1, 0
        held += k
    assert chunks >= n_chunks, chunks
    return chunks


def _assert_same_state(got, want):
    for a, b in zip(got, want):
        assert np.array_equal(a, b, equal_nan=True)


def _stations(case):
    h, w = case.shape
    spots = [(0.18 * h, 0.30 * w, 140.0, 11), (0.80 * h + 0.37, 0.62 * w + 0.5, -90.0, 12)]
    return [dict(row=r, col=c, elev=case.elev_aws + dz, rows=make_station_rows(case, case.elev_aws + dz, seed=sd))
            for (r, c, dz, sd) in spots]


@pytest.mark.parametrize("f64", [False, True])
def test_fused_members_cut_into_chunks(f64):
    """Five members (a group of four, a pair with a padding copy) over at least three mask chunks: the
    member rasters and per-step statistics equal the members run in one piece bit for bit; the rasters
    also equal one enrgy_run per member bit for bit (its statistics sum in another order, so they agree to
    rounding, as in test_gpu_ensemble)."""
    case = _case()
    members = make_members(5, seed=7, albedo_sigma=0.06)
    off = [m["albedo_offset"] for m in members]
    zm = [m["zm"] for m in members]
    zh = [m["z_h_or_e"] for m in members]
    out = {}
    for cut in (False, True):
        eng = _engine(case, f64)
        try:
            if cut:
                _chunk_into(eng, 3)
            stats, totals = eng.run_members(off, zm, zh, 0, N_STEPS)
            out[cut] = (stats, totals, [eng.member_state(k, np.float64) for k in range(len(members))])
        finally:
            eng.close()
    assert np.array_equal(out[True][0], out[False][0])
    assert np.array_equal(out[True][1], out[False][1], equal_nan=True)
    for k in range(len(members)):
        _assert_same_state(out[True][2][k], out[False][2][k])
    eng = _engine(case, f64)
    try:
        eng.snapshot(save=True)
        for k, m in enumerate(members):
            eng.snapshot(save=False)
            eng.set_member(m["albedo_offset"], m["zm"], m["z_h_or_e"])
            eng.prepass()
            stats = eng.run(0, N_STEPS)
            _assert_same_state(out[True][2][k], eng.state(np.float64))
            assert np.allclose(out[True][0][k], stats, rtol=1e-12 if f64 else 2e-6, atol=1e-9 if f64 else 1e-3), k
    finally:
        eng.close()


@pytest.mark.parametrize("mode,f64", [
    ("stations", False), ("stations", True), ("msm", True),
    pytest.param("msm", False, marks=pytest.mark.xfail(
        strict=True, reason="float32 sub-surface model with shading: the SWE raster and its sums differ in the "
                            "last bits when the run is cut into mask chunks"))])
def test_runs_cut_into_chunks(mode, f64):
    """The station blend and the sub-surface model with shading, cut into mask chunks, equal the run in one
    piece bit for bit: statistics, state rasters and (sub-surface model) the layer temperatures."""
    case = _case()
    kw = dict(stations=_stations(case), cloud_k=0.7) if mode == "stations" else MSM
    out = {}
    for cut in (False, True):
        eng = _engine(case, f64, **kw)
        try:
            if cut:
                _chunk_into(eng, 3)
            stats = eng.run(0, N_STEPS)
            out[cut] = (stats, eng.state(np.float64), eng.layer_temps() if mode == "msm" else None)
        finally:
            eng.close()
    assert np.array_equal(out[True][0], out[False][0])
    _assert_same_state(out[True][1], out[False][1])
    if mode == "msm":
        assert np.array_equal(out[True][2], out[False][2], equal_nan=True)


@pytest.mark.parametrize("f64", [False, True])
def test_dump_reuses_masks_cached_by_a_run(f64):
    """enrgy_dump_steps over steps whose masks a run has cached (so the dump reads them at an offset into
    the cache) equals the same dump on a fresh handle, and leaves kernel_info() alone."""
    case = _case()
    eng = _engine(case, f64)
    fresh = _engine(case, f64)
    try:
        eng.snapshot(save=True)
        eng.run(0, N_STEPS)
        info = eng.kernel_info()
        eng.snapshot(save=False)
        got = eng.dump_steps(5, 11)
        assert eng.kernel_info() == info
        want = fresh.dump_steps(5, 11)
        assert np.array_equal(got, want, equal_nan=True)
    finally:
        eng.close()
        fresh.close()


@pytest.mark.parametrize("f64", [False, True])
def test_masked_run_fed_chunk_by_chunk(f64):
    """enrgy_run_masked over chunks of steps, each with masks the caller swept by enrgy_shade_scan, with
    enrgy_defer_snow_total around the chunks (as parallel.ShardedShading runs them), equals enrgy_run."""
    import torch
    case = _case()
    ref = _engine(case, f64)
    eng = _engine(case, f64)
    try:
        want_stats = ref.run(0, N_STEPS)
        want_state = ref.state(np.float64)
        cuts = [(0, 4), (4, 9), (9, 10), (10, N_STEPS)]
        stats = torch.zeros((N_STEPS, _lib.S_COUNT), dtype=torch.float64, device="cuda")
        bufs = []
        eng.defer_snow_total(True)
        for k, (c0, c1) in enumerate(cuts):
            s0, s1 = eng.sub_range(c0, c1)
            buf = torch.zeros(max(s1 - s0, 1) * eng.mask_words(eng.band_rows), dtype=torch.int32, device="cuda")
            bufs.append(buf)
            eng.shade_scan(s0, s1, [(0, eng.band_rows, buf.data_ptr())])
            if k == len(cuts) - 1:
                eng.defer_snow_total(False)
            eng.run_masked(c0, c1, buf.data_ptr(), stats.data_ptr() + 8 * _lib.S_COUNT * c0)
        eng.synchronize()
        assert np.array_equal(stats.cpu().numpy(), want_stats)
        _assert_same_state(eng.state(np.float64), want_state)
    finally:
        eng.close()
        ref.close()
