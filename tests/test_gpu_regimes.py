"""The energy balance against the oracle in the weather regimes of tests/regimes.py: polar night, polar
dawn and dusk, cold and unstable air with neutral rows, extremes (calm, gales, dry and saturated air, clear
and overcast sky, a high glacier), rows of irregular length (0 to 255 sub-steps in one run) and a season
with the sub-surface model.

Bars as in test_gpu_parity: 1e-9 relative in float64, 1e-4 in float32, against max(|ref|, floor).

Runs with shading over rows where the sun stays down (polar night) have no sunlit sub-step: no mask is
swept and the kernel reads none.  Every entry point must run them, and their rasters must equal the same
run without shading bit for bit (in such a row the direct beam is 0 whichever insolation instance of the
kernel computes it, and the diffuse part is the same pre-pass value)."""
import os

import numpy as np
import pytest

from enrgy_b200 import _lib
from oracle import insolation_oracle as I
from tests import parity as P
from tests import regimes as G

pytestmark = pytest.mark.gpu

SHORT = ["polar_night", "polar_dawn", "polar_dusk", "cold_unstable", "extremes", "irregular_time"]
MODES = ["streamed", "computed", "shaded"]


def _tol(f64):
    return 1e-9 if f64 else 1e-4


def _assert_within(res, f64):
    for k, v in res.items():
        assert v < _tol(f64), (k, v)


def _pot(case):
    """The specification's insolation of the case (shaded; dark where the sun is down), as streamed rasters."""
    return I.insolation_series(case).astype(np.float32)


def _compare(name, f64, mode, **extra):
    case = G.make_regime_case(name)
    kw = dict(G.REGIME_KW[name], **extra)
    if mode == "streamed":
        return P.compare_run(case, f64, pot=_pot(case), **kw)
    return P.compare_run(case, f64, computed=True, shadow=mode == "shaded", **kw)


# float32 extremes: the (row, field) slices where the kernel misses the float32 oracle by more than 1e-4 of the
# floor (measured on a B200).  All are cells where a flux or the whole balance crosses zero between terms of
# hundreds of W m-2:
#   rows 7, 17, 19, 31   gales of 31-40 m/s: sensible and latent fluxes of 300-400 W m-2, latent flux or balance
#                        near 0 at a few cells; kernel 1.1e-4 to 2.4e-4 off the float32 oracle
#   row 15 (sub-surface) 10 % humidity: balance 0.29 W m-2 = 315 (lwd) - 310 (lwu) - 90 (lat) + ...; 1.0e-4 to
#                        1.2e-4 at one cell
# At these rows the reference's own float32 run is as far from its float64 run as the kernel is (both 2e-4 to
# 1.1e-3 of the 1 W m-2 floor), so two float32 implementations that round in another order cannot agree to 1e-4
# there.  Everything else of the float32 extremes, the sub-surface model included, is held to 1e-4.
F32_EXTREMES_SLICE = {
    False: {(17, "atmo"), (17, "mf"), (19, "atmo"), (19, "mf")},
    True: {(7, "lat"), (19, "lat"), (15, "atmo"), (31, "atmo")},
}


def _skip(name, f64, msm):
    return F32_EXTREMES_SLICE[msm] if name == "extremes" and not f64 else ()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("f64", [True, False])
@pytest.mark.parametrize("name", SHORT)
def test_regime_parity(name, f64, mode):
    res = _compare(name, f64, mode, skip=_skip(name, f64, False))
    res.pop("skipped", None)
    print(name, f64, mode, res)
    _assert_within(res, f64)


@pytest.mark.parametrize("mode", ["streamed", "shaded"])
@pytest.mark.parametrize("f64", [True, False])
@pytest.mark.parametrize("name", ["cold_unstable", "extremes"])
def test_regime_parity_msm(name, f64, mode):
    """The sub-surface model (the 7-layer stack) in cold, unstable air (no melt: the float32 melt-flux
    bound cannot be tied to the reference's own float32 error there) and in the extremes (melt)."""
    res = _compare(name, f64, mode, msm=G.MSM7, snow_density=350.0, skip=_skip(name, f64, True))
    res.pop("skipped", None)
    print(name, f64, mode, res)
    _assert_within(res, f64)


@pytest.mark.xfail(strict=True, reason="float32 fluxes at their zero crossings in gales (and one dry-air cell with "
                                       "the sub-surface model): the kernel and the float32 oracle round differently "
                                       "by more than 1e-4 of the 1 W m-2 floor")
@pytest.mark.parametrize("mode,msm", [("streamed", False), ("computed", False), ("shaded", False),
                                      ("streamed", True), ("shaded", True)])
def test_extremes_f32_slice(mode, msm):
    """The slices F32_EXTREMES_SLICE leaves out of the float32 extremes, at the 1e-4 bar."""
    extra = dict(msm=G.MSM7, snow_density=350.0) if msm else {}
    res = _compare("extremes", False, mode, skip=F32_EXTREMES_SLICE[msm], **extra)
    print(mode, msm, res["skipped"])
    assert res["skipped"] < 1e-4


# ---- dark ranges with shading ---------------------------------------------------------------------
def _night():
    return G.make_regime_case("polar_night")


def _engine(case, f64, shadow=True):
    return P.make_engine(case, f64, computed=True, shadow=shadow)


def _unshaded_run(case, f64):
    eng = _engine(case, f64, shadow=False)
    try:
        stats = eng.run(0, len(case.aws_rows))
        return stats, eng.state(np.float64)
    finally:
        eng.close()


def _assert_same_state(got, want):
    for a, b in zip(got, want):
        assert np.array_equal(a, b, equal_nan=True)


def _assert_matches_oracle(case, f64, state, stats=None, ora=None):
    """Final state rasters (and glacier-wide per-step means) against the oracle, floors of compare_run."""
    ora = ora or P.run_oracle(case, I.insolation_series(case, dtype=np.float64 if f64 else np.float32), f64)
    ff, mfl, tfl = (1e-3, 1e-7, 1e-6) if f64 else (1.0, 1e-3, 1e-3)
    for got, key in zip(state, ("swe", "total_snow", "total_ice")):
        assert P.max_rel_err(got, ora[key], tfl) < _tol(f64), key
    if stats is not None:
        floors = np.array([ff] * 8 + [mfl, mfl, tfl, 0.5, 0.5])
        m = P.means_from_stats(stats)
        assert float(np.max(np.abs(m - ora["means"]) / np.maximum(np.abs(ora["means"]), floors))) < _tol(f64)
    return ora


@pytest.mark.parametrize("f64", [True, False])
def test_dark_range_run(f64):
    """enrgy_run with shading on a fresh handle over rows without a sunlit sub-step (no masks allocated)."""
    case = _night()
    n = len(case.aws_rows)
    eng = _engine(case, f64)
    try:
        assert eng.point_scalars()[:, _lib.P_NSUB].sum() == 0
        stats = eng.run(0, n)
        state = eng.state(np.float64)
    finally:
        eng.close()
    _assert_matches_oracle(case, f64, state, stats)
    want_stats, want_state = _unshaded_run(case, f64)
    _assert_same_state(state, want_state)
    assert np.array_equal(stats, want_stats)


@pytest.mark.parametrize("f64", [True, False])
def test_dark_range_dump(f64):
    """enrgy_dump_steps with shading on a fresh handle over dark rows equals the unshaded dump."""
    case = _night()
    n = len(case.aws_rows)
    got = []
    for shadow in (True, False):
        eng = _engine(case, f64, shadow=shadow)
        try:
            got.append(eng.dump_steps(0, n))
        finally:
            eng.close()
    assert np.array_equal(got[0], got[1], equal_nan=True)
    assert np.all(np.nan_to_num(got[0][:, _lib.D_POT]) >= 0)
    ora = P.run_oracle(case, I.insolation_series(case, dtype=np.float64 if f64 else np.float32), f64)
    floor = 1e-3 if f64 else 1.0
    for name in ("rs", "lwd", "sens", "lat", "atmo"):
        idx = _lib.DUMP_NAMES.index(name)
        worst = max(P.max_rel_err(got[0][i, idx], ora["rows"][i][name], floor) for i in range(n))
        assert worst < _tol(f64), (name, worst)


@pytest.mark.parametrize("f64", [True, False])
def test_dark_range_members(f64):
    """enrgy_run_members with shading on a fresh handle over dark rows: the members equal those of an
    unshaded handle bit for bit; the member without perturbation equals the oracle."""
    case = _night()
    n = len(case.aws_rows)
    off = [0.0, 0.03, -0.05]
    out = []
    for shadow in (True, False):
        eng = _engine(case, f64, shadow=shadow)
        try:
            stats, totals = eng.run_members(off, None, None, 0, n)
            out.append((stats, totals, [eng.member_state(k, np.float64) for k in range(len(off))]))
        finally:
            eng.close()
    assert np.array_equal(out[0][0], out[1][0])
    assert np.array_equal(out[0][1], out[1][1], equal_nan=True)
    for k in range(len(off)):
        _assert_same_state(out[0][2][k], out[1][2][k])
    _assert_matches_oracle(case, f64, out[0][2][0], out[0][0][0])


@pytest.mark.parametrize("f64", [True, False])
def test_dark_range_run_masked_without_masks(f64):
    """enrgy_run_masked with d_masks = NULL over rows without a sunlit sub-step; still refused where the
    rows have one."""
    import torch
    case = _night()
    n = len(case.aws_rows)
    eng = _engine(case, f64)
    try:
        assert eng.sub_range(0, n) == (0, 0)
        d_stats = torch.zeros((n, _lib.S_COUNT), dtype=torch.float64, device="cuda")
        eng.run_masked(0, n, None, d_stats.data_ptr())
        eng.synchronize()
        stats = d_stats.cpu().numpy()
        state = eng.state(np.float64)
    finally:
        eng.close()
    want_stats, want_state = _unshaded_run(case, f64)
    _assert_same_state(state, want_state)
    assert np.array_equal(stats, want_stats)
    _assert_matches_oracle(case, f64, state, stats)
    day = G.make_regime_case("polar_dawn")
    eng = _engine(day, f64)
    try:
        with pytest.raises(_lib.EnrgyError, match="d_masks is null"):
            eng.run_masked(0, len(day.aws_rows), None)
    finally:
        eng.close()


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_dark_range_energy_class(tmp_path, precision):
    """The Energy class with shading and a checkpoint that makes its first range of rows dark."""
    from enrgy_b200 import Energy
    from enrgy_b200.raster_utils import save_npy_raster
    case = _night()
    f64 = precision == "f64"
    d = str(tmp_path)
    dem = save_npy_raster(os.path.join(d, "dem.npy"), case.dem, case.geotransform)
    swe = save_npy_raster(os.path.join(d, "swe.npy"), case.swe, case.geotransform)
    alb = {k: save_npy_raster(os.path.join(d, "alb_%s.npy" % k), a, case.geotransform) for k, a in case.albedo_maps.items()}
    aws = case.write_aws_csv(os.path.join(d, "aws.csv"))
    e = Energy(dem, None, os.path.join(d, "out"), res=10, precision=precision)
    e.lat, e.lon = case.lat, case.lon
    e.add_snow(swe)
    e.add_checkpoints(["20221210"])                 # rows [0, 13) end at 20221210 12:00:00: all dark
    e.model(aws_file=aws, albedo_maps=alb, z=1.6, elev_aws=case.elev_aws, xy_aws=case.xy_aws, zm=1e-3,
            z_h_or_e=1e-4, emissivity=0.98, v=False)
    assert any("20221210 12:00:00 total_melt_ice" in f for f in os.listdir(os.path.join(d, "out")))
    # (the class hands its rasters back as float32, as the reference keeps them)
    state = (e.swe_array, e.total_snow_melt_array, e.total_ice_melt_array)
    _assert_matches_oracle(case, f64, state, e.stats)


@pytest.mark.parametrize("f64", [True, False])
def test_dark_range_sharded_shading(f64):
    """parallel.ShardedShading with one rank over dark rows: its chunk has no sunlit sub-step."""
    import torch
    from enrgy_b200.parallel import ShardedShading
    case = _night()
    n = len(case.aws_rows)
    eng = _engine(case, f64)
    try:
        stream = torch.cuda.Stream()
        eng.set_stream(stream.cuda_stream)
        d_stats = torch.zeros((n, _lib.S_COUNT), dtype=torch.float64, device="cuda")
        sh = ShardedShading(eng, [(0, case.shape[0])], 0, 1)
        sh.run(0, n, d_stats.data_ptr(), stream, eng.point_scalars()[:, _lib.P_NSUB].astype(int))
        stream.synchronize()
        stats = d_stats.cpu().numpy()
        eng.set_stream(None)
        state = eng.state(np.float64)
    finally:
        eng.close()
    want_stats, want_state = _unshaded_run(case, f64)
    _assert_same_state(state, want_state)
    assert np.array_equal(stats, want_stats)
    _assert_matches_oracle(case, f64, state, stats)


def _greedy_chunks(counts, max_subs):
    """The cut of a run into mask chunks that enrgy_run and ShardedShading make: whole rows, as many as fit
    max_subs sunlit sub-steps, at least one row per chunk."""
    out, t = [], 0
    while t < len(counts):
        e, s = t, 0
        while e < len(counts) and (e == t or s + counts[e] <= max_subs):
            s += counts[e]
            e += 1
        out.append((t, e, s))
        t = e
    return out


def _sweep_launches(eng, steps):
    """Launches of one sweep over the sunlit sub-steps of `steps` (shade.cu launch_sweep): one for the
    row-type scan lines, two (sweep and transpose) for the column-type ones."""
    row_type = [I.line_geometry(int(s[5]), int(s[6]))[0] for t in steps for s in eng.substeps(t)]
    return (1 if any(row_type) else 0) + (2 if not all(row_type) else 0)


@pytest.mark.parametrize("f64", [True, False])
@pytest.mark.parametrize("name", ["polar_dawn", "polar_dusk"])
def test_dark_into_day_chunked(name, f64):
    """From day into night and back under a mask budget of one sub-step: every sunlit row is a chunk of its
    own and the nights between are chunks without a sunlit sub-step.  enrgy_run and ShardedShading (one rank,
    the same budget) equal the run in one piece bit for bit.  The launch count pins the cut enrgy_run made:
    per chunk one fused kernel, one finalize and the sweep of its sub-step (none for a dark chunk), plus the
    first run's off-glacier pass."""
    import torch
    from enrgy_b200.parallel import ShardedShading
    case = G.make_regime_case(name)
    n = len(case.aws_rows)
    out = {}
    for how in ("whole", "chunked", "sharded"):
        eng = _engine(case, f64)
        try:
            counts = [int(x) for x in eng.point_scalars()[:, _lib.P_NSUB]]
            plan = _greedy_chunks(counts, 1)
            assert any(s == 0 for _, _, s in plan[1:]) and sum(s > 0 for _, _, s in plan) >= 4, plan
            before = eng.launch_count()
            if how == "chunked":
                eng.set_mask_budget(1)            # fewer bytes than one sub-step's masks: max_subs = 1
                stats = eng.run(0, n)
                want = 1 + sum(2 + (_sweep_launches(eng, range(a, b)) if s else 0) for a, b, s in plan)
                assert eng.launch_count() - before == want
            elif how == "sharded":
                stream = torch.cuda.Stream()
                eng.set_stream(stream.cuda_stream)
                d_stats = torch.zeros((n, _lib.S_COUNT), dtype=torch.float64, device="cuda")
                sh = ShardedShading(eng, [(0, case.shape[0])], 0, 1, budget_bytes=4 * eng.mask_words(case.shape[0]) * 2 + 1)
                assert [c[:2] for c in plan] == sh.chunks(0, n, counts)
                sh.run(0, n, d_stats.data_ptr(), stream, counts)
                stream.synchronize()
                stats = d_stats.cpu().numpy()
                eng.set_stream(None)
            else:
                stats = eng.run(0, n)
                assert eng.launch_count() - before == 1 + 2 + _sweep_launches(eng, range(n))
            out[how] = (stats, eng.state(np.float64))
        finally:
            eng.close()
    for how in ("chunked", "sharded"):
        assert np.array_equal(out[how][0], out["whole"][0]), how
        _assert_same_state(out[how][1], out["whole"][1])


# ---- runs split at the dark/day boundary and at the logger gap ------------------------------------
def _splits(name, counts):
    if name == "irregular_time":
        gaps = [i for i, r in enumerate(G.make_regime_case(name).aws_rows) if r["DATE"].endswith("17:00:00")]
        dark = [i for i in range(1, len(counts)) if counts[i - 1] > 0 and counts[i] == 0]
        return sorted({1, gaps[2], gaps[2] + 1, dark[-1]})
    # dusk and dawn: the first dark row, the first sunlit row after the night
    first_dark = next(i for i in range(1, len(counts)) if counts[i] == 0 and counts[i - 1] > 0)
    first_day = next(i for i in range(first_dark, len(counts)) if counts[i] > 0)
    return [first_dark, first_day]


@pytest.mark.parametrize("mode", ["streamed", "shaded"])
@pytest.mark.parametrize("name", ["polar_dawn", "irregular_time"])
def test_split_at_dark_and_gap(name, mode):
    """A float64 run split into runs at the dark/day boundaries (and, irregular rows, at the 63.75 h row and
    around a 7 h logger gap) equals the run in one piece: statistics, swe and total_ice bit for bit,
    total_snow (added once per run as swe(start) - swe(end)) to 1e-13."""
    case = G.make_regime_case(name)
    n = len(case.aws_rows)
    kw = G.REGIME_KW[name]
    pot = _pot(case) if mode == "streamed" else None

    def engine():
        if mode == "streamed":
            return P.make_engine(case, True, pot=pot, **kw)
        return P.make_engine(case, True, computed=True, shadow=True, **kw)
    counts = [len(I.substep_table(I.to_unix(r["DATE"]), P.O.time_step_seconds(case.aws_rows, i), case.lat, case.lon,
                                  case.cell)) for i, r in enumerate(case.aws_rows)]
    cuts = [0] + _splits(name, counts) + [n]
    one = engine()
    try:
        s_all = one.run(0, n)
        ref = one.state(np.float64)
    finally:
        one.close()
    eng = engine()
    try:
        parts = [eng.run(a, b) for a, b in zip(cuts, cuts[1:])]
        got = eng.state(np.float64)
    finally:
        eng.close()
    assert np.array_equal(np.concatenate(parts), s_all)
    assert np.array_equal(got[0], ref[0], equal_nan=True) and np.array_equal(got[2], ref[2], equal_nan=True)
    assert np.allclose(got[1], ref[1], rtol=1e-13, atol=0, equal_nan=True)


# ---- the sub-surface model over a season -----------------------------------------------------------
SEASON_SHAPE = (32, 40)
# first rows of 4-row dump windows; rows 36-39 (noon of 16 August) melt on most of the glacier
SEASON_DUMPS = (0, 36, 240, 700, 1130, 1600, 2000, 2196)


def _season_flux_errors(f64, dump, t, ora_rows, floor_mf):
    """Worst relative error of the dumped fluxes of rows t, t + 1, ... against the oracle's."""
    ff = 1e-3 if f64 else 1.0
    res = {}
    for name in P.FLUX_FIELDS:
        idx = _lib.DUMP_NAMES.index(name)
        floor = floor_mf if name in ("mf", "g") else ff
        res[name] = max(P.max_rel_err(dump[k, idx], ora_rows[t + k][name], floor) for k in range(dump.shape[0]))
    return res


@pytest.mark.parametrize("f64,mode", [(True, "streamed"), (False, "streamed"), (True, "computed"),
                                      (False, "computed"), (True, "shaded")])
def test_msm_season(f64, mode, capsys):
    """About 2200 hourly rows from mid-August at 78 N (polar sunset, freeze-up) with the 7-layer sub-surface
    stack: the final layer temperatures and state, every row's glacier-wide means, and the dumped rasters of
    eight 4-row windows (the state run up to each window on a second handle) against the oracle."""
    case = G.make_regime_case("msm_season", *SEASON_SHAPE)
    n = len(case.aws_rows)
    kw = G.REGIME_KW["msm_season"]
    computed, shadow = mode != "streamed", mode == "shaded"
    pot = _pot(case) if mode == "streamed" else None
    keep = {t + k for t in SEASON_DUMPS for k in range(4) if t + k < n}
    ora = P.run_oracle(case, P.oracle_insolation(case, pot, computed, shadow, f64), f64, keep_steps=keep, **kw)
    ff, mfl, tfl = (1e-3, 1e-7, 1e-6) if f64 else (1.0, 1e-3, 1e-3)
    floor_mf = ff
    if not f64:
        # as compare_run: the float32 melt gate carries the cold content of the surface layer, so mf and g
        # are held to 1e-4 of 5 W m-2, which must not be looser than the reference's own float32 error
        floor_mf = 5.0
        ora64 = P.run_oracle(case, P.oracle_insolation(case, pot, computed, shadow, True), True, keep_steps=keep, **kw)
        assert any(np.nanmax(ora["rows"][t]["mf"]) > 0 for t in keep)        # the dumped rows include melt
        gap = max(float(np.nanmax(np.abs(np.asarray(ora["rows"][t]["mf"], dtype=np.float64) - ora64["rows"][t]["mf"])))
                  for t in sorted(keep))
        assert 1e-4 * floor_mf <= gap, ("the float32 melt-flux bound is looser than the reference's own float32 "
                                        "error on this case", gap)
        drift = max(float(np.nanmax(np.abs(a - b))) for a, b in zip(ora["layer_temperatures"], ora64["layer_temperatures"]))
        with capsys.disabled():
            print("\nmsm_season %s: the oracle's own float32 - float64 gap: melt flux %.3g W m-2 at the dumped rows, "
                  "layer temperatures %.3g K at the end" % (mode, gap, drift))
    eng = P.make_engine(case, f64, pot=pot, computed=computed, shadow=shadow, **kw)
    try:
        stats = eng.run(0, n)
        swe, tsn, tic = eng.state(np.float64)
        layers = eng.layer_temps()
    finally:
        eng.close()
    res = {}
    res["layer_t"] = max(P.max_rel_err(layers[l], ora["layer_temperatures"][l], 1e-3 if f64 else 1.0)
                         for l in range(layers.shape[0]))
    res["swe"] = P.max_rel_err(swe, ora["swe"], tfl)
    res["total_snow"] = P.max_rel_err(tsn, ora["total_snow"], tfl)
    res["total_ice"] = P.max_rel_err(tic, ora["total_ice"], tfl)
    floors = np.array([ff] * 8 + [mfl, mfl, tfl, 0.5, 0.5])
    res["means"] = float(np.max(np.abs(P.means_from_stats(stats) - ora["means"]) / np.maximum(np.abs(ora["means"]), floors)))
    eng = P.make_engine(case, f64, pot=pot, computed=computed, shadow=shadow, **kw)
    try:
        t_done = 0
        for t in SEASON_DUMPS:
            eng.run(t_done, t)
            t_done = t
            dump = eng.dump_steps(t, min(t + 4, n))
            for k, v in _season_flux_errors(f64, dump, t, ora["rows"], floor_mf).items():
                res[k] = max(res.get(k, 0.0), v)
            for k in range(dump.shape[0]):
                snow, ice, _ = ora["melt"][t + k]
                res["snow"] = max(res.get("snow", 0.0), P.max_rel_err(dump[k, _lib.D_SNOW], snow, mfl))
                res["ice"] = max(res.get("ice", 0.0), P.max_rel_err(dump[k, _lib.D_ICE], ice, mfl))
    finally:
        eng.close()
    if not f64:
        lt64 = ora64["layer_temperatures"]
        with capsys.disabled():
            print("msm_season %s float32 kernel: final layer temperatures off the float64 oracle by at most %.3g K "
                  "(surface %.3g K)" % (mode, max(float(np.nanmax(np.abs(layers[l] - lt64[l]))) for l in range(layers.shape[0])),
                                         float(np.nanmax(np.abs(layers[0] - lt64[0])))))
    print(f64, mode, res)
    _assert_within(res, f64)
