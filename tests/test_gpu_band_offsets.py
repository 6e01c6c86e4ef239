"""Row bands that start anywhere, against the oracle and against the whole raster.

Bands are how the library runs on several GPUs (`Energy.model` under torchrun, `ShardedShading`, any C
caller that sets band_row0 / band_rows).  The raster here is ragged (77 x 131) and the bands start on odd
rows, on multiples of 8 that are no multiple of 16 and on multiples of 16; some are lower than one patch
of the fused kernel (8 rows, 4 with stations), some hold the AWS cell (row 38) and some do not.  A band's
state equals the whole run's rows bit for bit, except where DESIGN.md says rounding may differ (float32
analytic direct beam at cuts off the 8-row grid; float64 stations).  With shading, a band must start on
a multiple of 8 rows (the sweep writes the masks in 8-row groups): other starts are refused.  The last
test sweeps more sub-steps in one chunk than one launch of the sweep takes.
"""
import numpy as np
import pytest

from enrgy_b200 import _lib
from enrgy_b200.ensemble import make_members, run_members
from enrgy_b200.synthetic import make_case
from oracle import insolation_oracle as I
from oracle.enrgy_oracle import time_step_seconds
from tests import parity as P
from tests.test_gpu_parity import VARIANTS
from tests.test_gpu_stations import _stations

pytestmark = pytest.mark.gpu

T = 24
UNALIGNED = [(0, 5), (5, 19), (24, 9), (33, 31), (64, 13), (76, 1)]
UNALIGNED_TILING = UNALIGNED[:5]                  # (76, 1) lies inside (64, 13)
SHADED = [(0, 8), (8, 16), (24, 40), (64, 13), (40, 1), (72, 5)]
SHADED_TILING = SHADED[:4]


@pytest.fixture(scope="module")
def case():
    # 78 N, 24 hourly rows of 1 June: the sun goes all the way round, so every scan-line family occurs
    return make_case(77, T, w=131, seed=3)


@pytest.fixture(scope="module")
def pot(case):
    return P.random_insolation(case, T)


def _diff(a, b):
    d = np.abs(np.asarray(a, dtype=np.float64) - b)
    return dict(cells=int(np.count_nonzero(d > 0)), max_abs=float(np.nanmax(d)) if d.size else 0.0)


def _check_bands(case, f64, bands, tiling, pot=None, computed=False, shadow=False, **kw):
    """Every band against the sliced whole-raster oracle (compare_run, one oracle run for all bands), its
    final state against the whole-raster engine's rows, and the statistics of the tiling bands against the
    whole run's."""
    tol = 1e-9 if f64 else 1e-4
    ora = P.run_oracle(case, P.oracle_insolation(case, pot, computed, shadow, f64), f64, **kw)
    whole = P.make_engine(case, f64, pot=pot, computed=computed, shadow=shadow, **kw)
    try:
        stats_w = whole.run(0, T)
        state_w = whole.state(np.float64)
    finally:
        whole.close()
    total = np.zeros_like(stats_w)
    for band in bands:
        res = P.compare_run(case, f64, pot=pot, computed=computed, shadow=shadow, band=band, ora=ora, **kw)
        bad = {k: v for k, v in res.items() if v >= tol and not k.endswith("_l2")}
        assert not bad, (band, bad)
        eng = P.make_engine(case, f64, pot=pot, computed=computed, shadow=shadow, band=band, **kw)
        try:
            stats = eng.run(0, T)
            state = eng.state(np.float64)
        finally:
            eng.close()
        r0, n = band
        # float32 with insolation computed in the kernel and no shading: a patch (8 rows x 32 columns) takes
        # the analytic form of the direct beam in the steps where the sun stands above every slope of the
        # patch, and the two forms differ in the last bits -- a band with an edge off the 8-row grid groups
        # other rows into its patches (row_bands cuts on it)
        patches_differ = computed and not shadow and not f64 and (r0 % 8 or ((r0 + n) % 8 and r0 + n < case.shape[0]))
        for name, a, b in zip(("swe", "total_snow", "total_ice"), state, state_w):
            b = b[r0:r0 + n]
            if f64 and kw.get("stations") is not None:
                # (float64 stations: reciprocals by Newton steps, scheduled per instantiation -- a few ulp,
                # tests/test_gpu_stations.py)
                assert np.array_equal(np.isnan(a), np.isnan(b)) and np.allclose(a, b, rtol=1e-13, atol=1e-15,
                                                                                equal_nan=True), (band, name)
            elif patches_differ:
                assert np.array_equal(np.isnan(a), np.isnan(b)) and np.allclose(a, b, rtol=1e-6, atol=1e-9,
                                                                                equal_nan=True), (band, name, _diff(a, b))
            else:
                assert np.array_equal(a, b, equal_nan=True), (band, name, _diff(a, b))
        if band in tiling:
            total += stats
    # (float32: the per-CTA statistic rows are float32 sums, and bands change which cells a CTA adds up)
    assert np.allclose(total, stats_w, rtol=1e-12 if f64 else 3e-6, atol=1e-9 if f64 else 1e-3), \
        float(np.max(np.abs(total - stats_w) / np.maximum(np.abs(stats_w), 1e-9)))


UNSHADED_MODES = {
    "streamed_maps": dict(),
    "streamed_const": dict(const_albedo=(0.35, 0.75)),
    "computed": dict(computed=True),                   # float32: the analytic direct beam on gentle patches
    "msm": VARIANTS["msm"],                            # bands without the AWS cell get it by set_aws_cell
    "stations": dict(stations=3, cloud_k=0.8),
}


def _mode_kw(case, kw):
    kw = dict(kw)
    if "stations" in kw:
        kw["stations"] = _stations(case, kw["stations"])
    return kw


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("mode", list(UNSHADED_MODES))
def test_unaligned_bands_without_shading(case, pot, mode, f64):
    kw = _mode_kw(case, UNSHADED_MODES[mode])
    _check_bands(case, f64, UNALIGNED, UNALIGNED_TILING, pot=None if kw.get("computed") else pot, **kw)


SHADED_MODES = {
    "computed": dict(),                                # the masked kernel (one-barrier path in float32)
    "msm": VARIANTS["msm"],
    "stations": dict(stations=3, cloud_k=0.8),
}


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("mode", list(SHADED_MODES))
def test_shaded_bands(case, mode, f64):
    _check_bands(case, f64, SHADED, SHADED_TILING, computed=True, shadow=True, **_mode_kw(case, SHADED_MODES[mode]))


def test_shaded_band_masks_bit_exact(case):
    """shade_masks of every band = the rows of the specification's whole-raster masks, every sub-step of
    the day; the day holds all eight scan-line families (row / column type, both sweep directions, both
    signs of the shear)."""
    valid = ~np.isnan(case.dem)
    want, seen = [], set()
    for step in range(T):
        table = I.substep_table(I.to_unix(case.aws_rows[step]["DATE"]), time_step_seconds(case.aws_rows, step),
                                case.lat, case.lon, case.cell)
        want.append([I.shadow_mask(case.dem, s["dc_fix"], s["dr_fix"], s["dz"]) for s in table])
        seen.update((rt, sg, df > 0) for rt, sg, df in (I.line_geometry(s["dc_fix"], s["dr_fix"]) for s in table))
    assert len(seen) == 8, seen
    for r0, n in SHADED:
        eng = P.make_engine(case, False, computed=True, shadow=True, band=(r0, n))
        try:
            v = valid[r0:r0 + n]
            for step in range(T):
                masks = eng.shade_masks(step)
                assert masks.shape == (len(want[step]), n, case.shape[1])
                for j, lit in enumerate(want[step]):
                    assert np.array_equal(masks[j][v], lit[r0:r0 + n][v]), ((r0, n), step, j)
        finally:
            eng.close()


@pytest.mark.parametrize("f64", [False, True])
def test_fused_members_on_shaded_bands(case, f64):
    """Four fused members on every band = one run per member on the whole raster: states bit for bit, the
    statistics of the tiling bands add up to the whole run's."""
    members = make_members(4, seed=2, albedo_sigma=0.05)
    whole = P.make_engine(case, f64, computed=True, shadow=True)
    try:
        ref = run_members(whole, members, keep_rasters=True, fused=False)
    finally:
        whole.close()
    total = [np.zeros_like(ref[i]["stats"]) for i in range(len(members))]
    for r0, n in SHADED:
        eng = P.make_engine(case, f64, computed=True, shadow=True, band=(r0, n))
        try:
            got = run_members(eng, members, keep_rasters=True, fused=True)
        finally:
            eng.close()
        for i in range(len(members)):
            for k in ("swe", "total_snow", "total_ice"):
                a, b = got[i][k], ref[i][k][r0:r0 + n]
                assert np.array_equal(a, b, equal_nan=True), (i, k, (r0, n), _diff(a, b))
            if (r0, n) in SHADED_TILING:
                total[i] += got[i]["stats"]
    for i in range(len(members)):
        assert np.allclose(total[i], ref[i]["stats"], rtol=1e-12 if f64 else 3e-6, atol=1e-9 if f64 else 1e-3), i


@pytest.mark.parametrize("r0", [4, 84])
def test_shaded_band_off_the_8_row_grid_is_refused(r0):
    """With shading a band must start on a multiple of 8 rows; the same band without shading runs."""
    case = make_case(100, T, w=72, seed=3)        # 100 rows: where row_bands(100, 2) once cut at row 84
    band = (r0, 16)
    with pytest.raises(_lib.EnrgyError) as e:
        P.make_engine(case, False, computed=True, shadow=True, band=band)
    assert e.value.code == _lib.ERR_ARG
    res = P.compare_run(case, False, computed=True, band=band)
    bad = {k: v for k, v in res.items() if v >= 1e-4 and not k.endswith("_l2")}
    assert not bad, bad


def test_sweep_over_more_sub_steps_than_one_launch_takes():
    """Five years of daily rows on a 24 x 40 raster at the equator: one chunk of the default mask budget
    holds more than 65535 column-type sub-steps, more than one launch of the sweep takes (grid limits).
    The masks of ~30 steps spread over the run (the last one, and the sub-steps at both ends of the
    second launch, among them) are bit-exact, and the run equals one whose chunks stay far below the limit."""
    import torch
    n_steps = 1826
    case = make_case(24, n_steps, w=40, seed=7, step_s=86400, start="20180101 00:00:00")
    case.lat = 0.0                                 # the sun crosses from east to west: mostly column type
    kw = dict(computed=True, shadow=True, const_albedo=(0.35, 0.75))
    eng = P.make_engine(case, False, **kw)
    ref = P.make_engine(case, False, **kw)
    try:
        # the precondition, from the engine's own sub-step table
        subs = [eng.substeps(t, max_sub=128) for t in range(n_steps)]
        s0, s1 = eng.sub_range(0, n_steps)
        assert (s0, s1) == (0, sum(len(s) for s in subs))
        first = np.cumsum([0] + [len(s) for s in subs])
        col = []                                   # (sigma, dfix, sub-step) of the column-type sub-steps
        for t, ss in enumerate(subs):
            for j, s in enumerate(ss):
                if np.isfinite(s[7]) and (s[5] != 0 or s[6] != 0):
                    row_type, sigma, dfix = I.line_geometry(int(s[5]), int(s[6]))
                    if not row_type:
                        col.append((sigma, dfix, int(first[t]) + j))
        assert len(col) > 65535, len(col)
        per_sub = 4 * (eng.mask_words(24) + 40 * 8)     # masks + transposed temporary, bytes per sub-step
        assert s1 * per_sub < 1 << 30                    # one chunk of the default budget holds them all
        # the launches take the column-type sub-steps in direction order (api.cu sweep_range)
        second = [c[2] for c in sorted(col, key=lambda c: (c[0], c[1]))[65535:]]
        step_of = np.searchsorted(first, second, side="right") - 1
        steps = sorted(set(np.linspace(0, n_steps - 1, 30).astype(int).tolist()) | {int(step_of.min()), int(step_of.max())})

        buf = torch.zeros(s1 * eng.mask_words(24), dtype=torch.int32, device="cuda")
        eng.shade_scan(0, s1, [(0, 24, buf.data_ptr())])
        eng.synchronize()
        words = 128 // 32                                # pitch = round_up(40, 128)
        raw = buf.cpu().numpy().view(np.uint32).reshape(s1, -1, words, 8)     # [sub][rows / 8][word][row % 8]
        valid = ~np.isnan(case.dem)
        second = set(second)
        n_second = 0
        for t in steps:
            for j, s in enumerate(subs[t]):
                k = int(first[t]) + j
                w = np.ascontiguousarray(raw[k].transpose(0, 2, 1)).reshape(-1, words)     # [row][word]
                got = np.unpackbits(w.view(np.uint8), axis=-1, bitorder="little")[:24, :40].astype(bool)
                lit = I.shadow_mask(case.dem, int(s[5]), int(s[6]), np.float32(s[7]))
                assert np.array_equal(got[valid], lit[valid]), (t, j)
                n_second += k in second
        assert n_second > 0

        stats = eng.run(0, n_steps)
        state = eng.state(np.float64)
        ref.set_mask_budget(8000 * per_sub)              # chunks of at most 8000 sub-steps
        want = ref.run(0, n_steps)
        assert np.array_equal(stats, want)
        for a, b in zip(state, ref.state(np.float64)):
            assert np.array_equal(a, b, equal_nan=True)
    finally:
        eng.close()
        ref.close()
