"""World-size-2 test of the N>1 host path on the CPU (gloo): row-band partition, per-band
statistics as SUMS + counts, one all-reduce, means formed after -- must equal the single-process
result on the whole raster.  The per-band numbers come from the NumPy oracle here (the CUDA kernel
needs a GPU); what is under test is the partition and the reduction plumbing bench.py and
Energy use on the GPUs."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from enrgy_b200 import _lib
from enrgy_b200.parallel import allreduce_stats, means_from_sums, rebalance_bands, row_bands, tile_cost_per_row
from enrgy_b200.synthetic import make_case
from oracle import enrgy_oracle as O
from tests import parity as P


def _band_sums(case, pot, r0, n, kw):
    """Oracle on rows [r0, r0+n) (+ the AWS row in front so the point sampling is unchanged)."""
    ar = case.aws_rc[0]
    sl = slice(r0, r0 + n)

    def band(a):
        return np.concatenate([a[ar:ar + 1], a[sl]], axis=0)
    gt = list(case.geotransform)
    gt[3] = case.xy_aws[1] + 0.5 * case.cell
    cfg = P.oracle_config(case, **kw)
    alb = {k: band(a) for k, a in P.clipped_albedo(case, np.float64).items()}
    out = O.run_model(band(case.dem.astype(np.float64)), tuple(gt), case.aws_rows,
                      np.concatenate([pot[:, ar:ar + 1], pot[:, sl]], axis=1).astype(np.float64), cfg,
                      swe=band(case.swe.astype(np.float64)), albedo_arrays=alb, state_dtype=np.float64,
                      keep_steps=None)
    T = len(case.aws_rows)
    s = np.zeros((T, _lib.S_COUNT))
    for i in range(T):
        row, melt = out["rows"][i], out["melt"][i]
        cut = lambda a: np.asarray(a)[1:]          # drop the duplicated AWS row
        s[i, _lib.S_RS] = np.nansum(cut(row["rs"]))
        s[i, _lib.S_LWD] = np.nansum(cut(row["lwd"]))
        s[i, _lib.S_LWU] = np.nansum(np.where(np.isnan(cut(row["lwd"])), np.nan, cut(row["lwu"])))
        s[i, _lib.S_SENS] = np.nansum(cut(row["sens"]))
        s[i, _lib.S_LAT] = np.nansum(cut(row["lat"]))
        s[i, _lib.S_ATMO] = np.nansum(cut(row["atmo"]))
        s[i, _lib.S_MELT] = np.nansum(cut(row["mf"]))
        s[i, _lib.S_SNOW] = np.nansum(cut(melt[0]))
        s[i, _lib.S_ICE] = np.nansum(cut(melt[1]))
        swe = cut(melt[2])
        s[i, _lib.S_SWE] = np.nansum(swe)
        s[i, _lib.S_NSNOW] = np.sum(swe > 0)
        s[i, _lib.S_NSWE] = np.count_nonzero(~np.isnan(swe))
        s[i, _lib.S_NVALID] = np.count_nonzero(~np.isnan(cut(row["atmo"])))
    return s


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        case = make_case(64, 6, seed=31, w=48)
        pot = P.random_insolation(case, 6, seed=2)
        valid_per_row = (~np.isnan(case.dem)).sum(axis=1)
        bands = row_bands(case.dem.shape[0], world, align=8, valid_per_row=valid_per_row)
        r0, n = bands[rank]
        sums = torch.from_numpy(_band_sums(case, pot, r0, n, {}))
        allreduce_stats(sums)
        if rank == 0:
            np.save(os.path.join(out_dir, "reduced.npy"), sums.numpy())
            np.save(os.path.join(out_dir, "bands.npy"), np.array(bands))
    finally:
        dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_two_rank_band_reduction(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    reduced = np.load(tmp_path / "reduced.npy")
    bands = np.load(tmp_path / "bands.npy")
    assert bands[0][0] == 0 and bands[-1][0] + bands[-1][1] == 64 and bands[1][0] % 8 == 0
    case = make_case(64, 6, seed=31, w=48)
    pot = P.random_insolation(case, 6, seed=2)
    whole = P.run_oracle(case, pot, True)
    got = means_from_sums(reduced)
    want = whole["means"]
    # oracle means: rs, rl, lwd, sens, lat, atmo, g, melt, snow, ice, swe, n_snow, n_swe
    assert np.allclose(got[1:, :11], want[1:, :11], rtol=1e-11, atol=1e-12)
    cover = np.round(want[1:, 11] / want[1:, 12] * 100)
    assert np.array_equal(got[1:, 11], cover)
    # first row: the reference counts EVERY non-NaN SWE cell, off-glacier included -- identical here
    # because the synthetic SWE raster is NaN off-glacier
    assert np.allclose(got[0, :11], want[0, :11], rtol=1e-11, atol=1e-12)


def test_row_bands_properties():
    for rows, world in ((2048, 8), (100, 3), (64, 4), (8192, 8)):
        b = row_bands(rows, world)
        assert b[0][0] == 0 and sum(n for _, n in b) == rows
        assert all(b[i][0] + b[i][1] == b[i + 1][0] for i in range(world - 1))
        assert all(n > 0 for _, n in b)
    # no empty bands, ever: an empty band reads as "whole raster" at the C ABI
    for rows, world in ((16, 4), (100, 8)):
        with pytest.raises(ValueError):
            row_bands(rows, world, align=16)
    w = np.zeros(512)
    w[200:216] = 1.0                                 # the glacier occupies sixteen rows only
    b = row_bands(512, 4, align=16, valid_per_row=w)
    assert all(n >= 16 for _, n in b) and sum(n for _, n in b) == 512
    assert rebalance_bands(b, [1.0, 0.0, 0.0, 0.0], w) and all(n >= 16 for _, n in rebalance_bands(b, [1.0, 0.0, 0.0, 0.0], w))
    w = np.zeros(256)
    w[64:192] = 1.0                                  # glacier only in the middle half
    b = row_bands(256, 2, align=16, valid_per_row=w)
    assert b[0] == (0, 128) and b[1] == (128, 128)
    w[64:96] = 5.0
    b = row_bands(256, 2, align=16, valid_per_row=w)
    assert b[1][0] < 128                             # the heavy rows pull the cut north


def test_rebalance_bands_moves_rows_to_the_fast_ranks():
    """Bands rebalanced from measured times: a band that took twice as long as the others gives rows
    away; total rows and alignment are kept; equal times leave the cuts where they are."""
    rows, world = 1024, 4
    w = np.full(rows, 100.0)
    bands = row_bands(rows, world, align=16, valid_per_row=w)
    assert rebalance_bands(bands, [1.0, 1.0, 1.0, 1.0], w) == bands
    nb = rebalance_bands(bands, [1.0, 2.0, 1.0, 1.0], w)
    assert sum(n for _, n in nb) == rows and all(r0 % 16 == 0 for r0, _ in nb)
    assert nb[1][1] < bands[1][1] and nb[0][1] > bands[0][1] and nb[3][1] > bands[3][1]
    # estimated cost of the new bands is equal to within the alignment
    cost = np.concatenate([np.full(n, t / n) for (_, n), t in zip(bands, [1.0, 2.0, 1.0, 1.0])])
    shares = [cost[r0:r0 + n].sum() for r0, n in nb]
    assert max(shares) - min(shares) < 0.1


def test_tile_cost_weights():
    """Bands cut by visited tiles: a ragged glacier margin (one valid cell per tile) weighs as much as
    a filled interior, so the band holding it gets fewer rows than a cut by glacier cells gives it."""
    valid = np.zeros((256, 512), dtype=bool)
    valid[:128, :] = True                          # interior: every cell
    valid[128:, ::128] = True                      # margin: one cell per 128-column tile
    w = tile_cost_per_row(valid, tile_h=8, tile_w=128)
    assert w.shape == (256,) and np.allclose(w, 4 / 8.0)          # 4 tiles per 8-row group everywhere
    by_tiles = row_bands(256, 2, align=16, valid_per_row=w)
    by_cells = row_bands(256, 2, align=16, valid_per_row=valid.sum(axis=1))
    assert by_tiles == [(0, 128), (128, 128)]
    assert by_cells[0][1] < 128                                    # cells alone would starve rank 0 of rows


def test_band_cuts_properties_randomised():
    """row_bands / rebalance_bands on random weights and times: bands tile the raster without gaps or
    overlaps, edges are aligned, no band is empty, and re-cutting with the times a perfectly
    uniform cost model would have produced leaves the bands unchanged.  Raster heights need not be a
    multiple of the alignment (the weight in the bottom rows pulls the cuts against the upper bound)."""
    from hypothesis import example, given, settings, strategies as st

    @settings(max_examples=60, deadline=None)
    @given(st.integers(1, 8), st.integers(1, 40), st.integers(0, 15), st.integers(0, 2**31 - 1),
           st.sampled_from([1, 8, 16]), st.booleans())
    @example(2, 6, 4, 0, 16, True)                   # rows = 100: once cut at row 84
    @example(3, 16, 1, 0, 16, True)                  # rows = 257: once cut at rows 225 and 241
    def check(world, groups, extra, seed, align, bottom):
        rows = groups * 16 + extra
        rng = np.random.default_rng(seed)
        w = rng.integers(0, 200, rows).astype(float)
        w[rng.random(rows) < 0.3] = 0.0
        if bottom:
            w[:rows - min(rows, 16)] = 0.0           # all the weight in the last rows
        if rows < world * align:
            with pytest.raises(ValueError):
                row_bands(rows, world, align=align, valid_per_row=w)
            return
        bands = row_bands(rows, world, align=align, valid_per_row=w)
        assert len(bands) == world and bands[0][0] == 0
        assert all(n >= align for _, n in bands) and sum(n for _, n in bands) == rows
        assert all(bands[i][0] + bands[i][1] == bands[i + 1][0] for i in range(world - 1))
        assert all(r0 % align == 0 for r0, _ in bands[1:])
        # times proportional to the weights the bands were cut with -> same cuts again
        secs = [max(w[r0:r0 + n].sum(), 0.0) for r0, n in bands]
        if min(secs) > 0:
            again = rebalance_bands(bands, secs, w, align=align)
            assert sum(n for _, n in again) == rows
            assert max(abs(a[0] - b[0]) for a, b in zip(again, bands)) <= align
    check()


# ---- Energy.model over two ranks (gloo), the per-band numbers from an oracle-backed engine stand-in ----
def _energy_worker(rank, world, port, d):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from enrgy_b200 import Energy
        from tests.fake_engine import FakeEngine
        case = make_case(96, 8, seed=31, w=48)
        pot = np.load(os.path.join(d, "pot.npy"))
        keys = list(case.albedo_maps)

        def factory(rows, cols, precision, device):
            f = FakeEngine(rows, cols, precision, device)
            f.aws_rows, f.geotransform, f.xy_aws, f.albedo_keys = case.aws_rows, case.geotransform, case.xy_aws, keys
            # (the AWS-cell insolation reaches the engine through Energy.model -> set_insolation_aws)
            return f
        e = Energy(os.path.join(d, "dem.npy"), None, os.path.join(d, "out"), res=10, precision="f64")
        e._engine_factory = factory
        e.debug_views = False
        e.use_precomputed = True
        e.add_pickle_dir(os.path.join(d, "pickle"))
        e.add_snow(os.path.join(d, "swe.npy"))
        e.add_checkpoints(["20220601"])
        e.model(aws_file=os.path.join(d, "aws.csv"), albedo_maps={k: os.path.join(d, "alb_%s.npy" % k) for k in keys},
                z=1.6, elev_aws=case.elev_aws, xy_aws=case.xy_aws, zm=1e-3, z_h_or_e=1e-4, emissivity=0.98, v=False)
        np.save(os.path.join(d, "ice_rank%d.npy" % rank), e.total_ice_melt_array)
        np.save(os.path.join(d, "swe_rank%d.npy" % rank), e.swe_array)
        if rank == 0:
            np.save(os.path.join(d, "bands.npy"), np.array(e.bands))
    finally:
        dist.destroy_process_group()


def test_energy_model_two_ranks(tmp_path):
    """`Energy.model` under a 2-rank process group: bands cut by visited tiles, each rank feeds its band,
    statistics all-reduced, rank 0 writes heat_fluxes.csv, every rank ends with the full rasters --
    equal to the single-process oracle on the whole raster."""
    from enrgy_b200.raster_utils import save_npy_raster
    d = str(tmp_path)
    case = make_case(96, 8, seed=31, w=48)
    pot = P.random_insolation(case, 8, seed=2)
    np.save(os.path.join(d, "pot.npy"), pot)
    save_npy_raster(os.path.join(d, "dem.npy"), case.dem, case.geotransform)
    save_npy_raster(os.path.join(d, "swe.npy"), case.swe, case.geotransform)
    for k, a in case.albedo_maps.items():
        save_npy_raster(os.path.join(d, "alb_%s.npy" % k), a, case.geotransform)
    case.write_aws_csv(os.path.join(d, "aws.csv"))
    os.makedirs(os.path.join(d, "pickle", "10"))
    for i, row in enumerate(case.aws_rows):
        np.save(os.path.join(d, "pickle", "10", "%s_total.sdat.npy" % row["DATE"]), pot[i])
    world = 2
    mp.spawn(_energy_worker, args=(world, _free_port(), d), nprocs=world, join=True)
    bands = np.load(os.path.join(d, "bands.npy"))
    assert len(bands) == 2 and bands[0][0] == 0 and bands[1][0] % 16 == 0 and bands[1][0] + bands[1][1] == 96
    whole = P.run_oracle(case, pot, True)
    for rank in range(world):
        ice = np.load(os.path.join(d, "ice_rank%d.npy" % rank))
        swe = np.load(os.path.join(d, "swe_rank%d.npy" % rank))
        assert ice.shape == case.dem.shape and ice.dtype == np.float32
        assert P.max_rel_err(ice, whole["total_ice"], 1e-6) < 1e-6
        assert P.max_rel_err(swe, whole["swe"], 1e-6) < 1e-6
    text = open(os.path.join(d, "out", "heat_fluxes.csv")).read()
    got = [line.split(",") for line in text.split("\n") if line[:2] == "20"]
    want = [line.split(",") for line in whole["stats_csv"].split("\n") if line[:2] == "20"]
    assert len(got) == len(want) == 8
    for g, w in zip(got, want):
        assert g[0] == w[0]
        lim = [0.1001] * 8 + [0.0101] + [0.00011] * 3 + [1.001]
        assert all(abs(float(x) - float(y)) <= l for x, y, l in zip(g[1:], w[1:], lim)), (g, w)
    files = os.listdir(os.path.join(d, "out"))
    # one export (the final one, written by rank 0 only; without GDAL a .npy + its side-car json)
    assert sum("remaining_snow_cover" in f and f.endswith(".npy") for f in files) == 1
