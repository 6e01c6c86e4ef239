"""Multi-GPU plumbing: one process per GPU, the raster cut into row bands (SURVEY.md 8e).

Cells are independent once the AWS-cell pre-pass has produced the per-step scalars, so the energy
balance needs NO collective: every rank runs the fused kernel on its own band of the albedo / SWE /
state rasters, and the only exchange is the sum of the per-step area statistics (`[T, S_COUNT]`
float64 sums and counts) -- one all-reduce per pass, NCCL for CUDA tensors (NVLink/NVSwitch), gloo on
the CPU in the tests.

Topographic shading is the one step that is NOT local to a band: a scan line runs through the whole
raster, so the sunlit mask of a band depends on terrain in every other band.  The sweep therefore
shards along a different axis -- the sunlit SUB-STEPS, which are independent of each other and cost
the same whatever the terrain: every rank sweeps the full (replicated) terrain for 1/N of the
sub-steps and an all-to-all over NVLink hands every rank the rows of its own band
(`ShardedShading`).  Per cell and sub-step that exchange moves one bit.
"""
from __future__ import annotations

import numpy as np

from . import _lib


def row_bands(rows, world, align=16, valid_per_row=None):
    """[(row0, n_rows)] for `world` ranks.  Band edges are multiples of `align` (the tile height of
    the fused kernel).  With `valid_per_row` (glacier cells per raster row) the bands are balanced
    by glacier cells instead of rows -- off-glacier tiles cost nothing (load balance, SURVEY 7)."""
    if world < 1:
        raise ValueError("world must be >= 1")
    if valid_per_row is None:
        weights = np.ones(rows, dtype=np.float64)
    else:
        weights = np.asarray(valid_per_row, dtype=np.float64)
        if weights.shape != (rows,):
            raise ValueError("valid_per_row must have one entry per raster row")
    if rows < world * align:
        # (an empty band would read as "whole raster" at the C ABI and double count the statistics)
        raise ValueError("%d rows cannot give %d bands of at least %d rows" % (rows, world, align))
    cum = np.concatenate([[0.0], np.cumsum(weights)])
    total = cum[-1]
    edges = [0]
    for r in range(1, world):
        target = total * r / world
        e = int(np.searchsorted(cum, target))
        e = int(round(e / align)) * align
        # every band keeps at least `align` rows, also where the glacier occupies a few rows only; the
        # upper bound is rounded down to a multiple of `align` too (rows need not be one)
        e = min(max(e, edges[-1] + align), (rows // align - (world - r)) * align)
        edges.append(e)
    edges.append(rows)
    return [(edges[i], edges[i + 1] - edges[i]) for i in range(world)]


def tile_cost_per_row(valid, tile_h=8, tile_w=128):
    """Cost weights for row_bands(valid_per_row=...) in units of VISITED TILES: the fused kernel walks
    tiles of tile_h x tile_w cells and a tile with one glacier cell costs as much as a full one, so a
    band along the glacier margin is more expensive than its glacier-cell count says.  `valid` is the
    boolean glacier mask [rows, cols]; every row gets 1 / tile_h of the tiles its row group touches."""
    valid = np.asarray(valid, dtype=bool)
    rows, cols = valid.shape
    hp, wp = -(-rows // tile_h) * tile_h, -(-cols // tile_w) * tile_w
    v = np.zeros((hp, wp), dtype=bool)
    v[:rows, :cols] = valid
    tiles = v.reshape(hp // tile_h, tile_h, wp // tile_w, tile_w).any(axis=(1, 3)).sum(axis=1)
    return np.repeat(tiles / float(tile_h), tile_h)[:rows]


def rebalance_bands(bands, seconds, valid_per_row, align=16):
    """New band edges from MEASURED per-band times, for runs whose cost per glacier cell is not uniform
    (tiles on the margin cost as much as full ones; streamed rasters).  The
    measured time of every band is spread over its rows in proportion to their glacier cells
    (piecewise-constant cost per glacier cell), and the cuts are placed at equal shares of that
    estimate.  One or two rounds settle (scripts/measure_modes.py strong)."""
    w = np.asarray(valid_per_row, dtype=np.float64)
    rows = w.shape[0]
    if len(bands) != len(seconds):
        raise ValueError("one measured time per band")
    cost = np.zeros(rows, dtype=np.float64)
    for (r0, n), t in zip(bands, seconds):
        tot = w[r0:r0 + n].sum()
        if n > 0:
            cost[r0:r0 + n] = (w[r0:r0 + n] * (float(t) / tot)) if tot > 0 else 0.0
    return row_bands(rows, len(bands), align=align, valid_per_row=cost)


def split_even(lo, hi, parts):
    """[lo, hi) cut into `parts` contiguous ranges whose sizes differ by at most one."""
    n = hi - lo
    edges = [lo + (n * p) // parts for p in range(parts + 1)]
    return [(edges[p], edges[p + 1]) for p in range(parts)]


def plan_step_chunks(sub_counts, t0, t1, max_subs):
    """Steps [t0, t1) cut into chunks of at most max_subs sunlit sub-steps (at least one step each)."""
    out, t = [], t0
    while t < t1:
        e, n = t, 0
        while e < t1 and (e == t or n + sub_counts[e] <= max_subs):
            n += sub_counts[e]
            e += 1
        out.append((t, e))
        t = e
    return out


class ShardedShading:
    """Row-band run WITH shading over `world` ranks (one Engine per rank, every one loaded with the
    full terrain and its own band).  Per chunk of rows
      1. rank p sweeps sub-steps p/N .. (p+1)/N of the chunk over the full raster and writes the rows of
         band q for rank q (enrgy_shade_scan with one destination segment per rank),
      2. every rank ends up with the masks of ITS band for all sub-steps of the chunk, already in the
         order the fused kernel reads them,
      3. the fused kernels run on the band with these masks (enrgy_run_masked).
    Step 2, three ways (`exchange`):
      "copy" (default)  bulk peer-to-peer copies into the peers' receive buffers (torch symmetric memory)
                        on a side stream, bracketed by two stream-ordered barriers: the copy engines move
                        the masks over NVLink while the SMs run the kernels of the neighbouring chunks;
      "all_to_all"      one all_to_all_single (NCCL) on the side stream -- its kernels take SMs from the
                        persistent fused kernel in flight (2.8 ms per chunk on 8 GPUs); also the fallback
                        where symmetric memory is not available;
      "p2p"             ONE KERNEL WITH STEP 1: the sweep stores the mask words straight into the peers'
                        receive buffers (whole 32-byte sectors); stores over NVLink slow the sweep by 10 %.
    Measured on 8192^2, 8 GPUs (profiles/r02_summary.md).
    Chunks are double-buffered: the sweep (and exchange) of chunk k + 1 is enqueued before the fused
    kernels of chunk k, so the exchange hides behind them.
    With world == 1 the sweep writes straight into the receive buffer.  Nothing synchronises the host."""

    def __init__(self, engine, bands, rank, world, group=None, budget_bytes=8 << 30, p2p=False, exchange=None):
        import torch
        self.torch = torch
        self.eng, self.bands, self.rank, self.world, self.group = engine, list(bands), int(rank), int(world), group
        if len(self.bands) != self.world:
            raise ValueError("one band per rank")
        if any(r0 % 8 for r0, _ in self.bands):
            raise ValueError("band starts must be multiples of 8 rows")
        self.words = [engine.mask_words(n) for _, n in self.bands]       # uint32 per sub-step and band
        self.budget = int(budget_bytes)
        self.slots = [dict(send=None, recv=None, peers=None, ready=None) for _ in range(2)]
        # exchange: "all_to_all" (NCCL kernels), "p2p" (the sweep stores into the peers' buffers), "copy" (bulk
        # peer-to-peer copies by the copy engines into the peers' buffers: no SM of the kernels in flight is taken)
        self.exchange = "none" if self.world == 1 else (exchange or ("p2p" if p2p else "copy"))
        if self.exchange not in ("none", "all_to_all", "p2p", "copy"):
            raise ValueError("exchange must be all_to_all, p2p or copy")
        self.comm = None                          # side stream of the exchange, made at the first run
        self.bytes_sent_last_run = 0
        self.subs_last_scan = 0
        self._flag = None                         # one word for the stream-ordered barriers
        self._symm_failed = False

    # ---- buffers ---------------------------------------------------------------------------------
    def _recv(self, slot, n_words):
        """Receive buffer of a slot: symmetric memory (peer-addressable) for the p2p exchange."""
        torch = self.torch
        sl = self.slots[slot]
        if sl["recv"] is not None and sl["recv"].numel() >= n_words:
            return sl
        if self.exchange in ("p2p", "copy"):
            try:
                import torch.distributed as dist
                import torch.distributed._symmetric_memory as symm
                # every rank must allocate the same size: the largest band times the sub-steps of a chunk
                t = symm.empty(int(n_words), dtype=torch.int32, device=torch.device("cuda", torch.cuda.current_device()))
                hdl = symm.rendezvous(t, self.group if self.group is not None else dist.group.WORLD)
                sl["recv"], sl["peers"] = t, [int(p) for p in hdl.buffer_ptrs]
                sl["hdl"] = hdl
                # the peers' receive buffers as tensors (bulk copies of the "copy" exchange)
                sl["peer_tensors"] = [hdl.get_buffer(q, (int(n_words),), torch.int32) for q in range(self.world)]
                return sl
            except Exception as e:                                    # pragma: no cover  (needs several GPUs)
                import sys
                print("symmetric memory unavailable (%s: %s); falling back to all_to_all" % (type(e).__name__, e), file=sys.stderr)
                self.exchange = "all_to_all"
                self._symm_failed = True
        sl["recv"] = torch.empty(max(int(n_words), 1), dtype=torch.int32, device="cuda")
        sl["peers"] = None
        return sl

    def _send(self, slot, n_words):
        sl = self.slots[slot]
        if sl["send"] is None or sl["send"].numel() < n_words:
            sl["send"] = self.torch.empty(max(int(n_words), 1), dtype=self.torch.int32, device="cuda")
        return sl["send"]

    def chunks(self, t0, t1, sub_counts):
        """Chunks of rows: within the memory budget, and (several ranks) at least a few of them so that the
        exchange of one chunk hides behind the kernels of its neighbours."""
        per_sub = 4 * (sum(self.words) // self.world + max(self.words)) * 2 + 1
        total = int(sum(sub_counts[t0:t1]))
        max_subs = max(1, self.budget // per_sub)
        if self.world > 1:
            # a rank sweeps 1/world of a chunk's sub-steps in one launch, and a launch of fewer than ~200
            # sub-steps leaves the GPU half empty in its tail (measured on 8192^2: 64 sub-steps per launch
            # run at 6.2e11 cell-sub-steps/s, 192 at 1.05e12)
            max_subs = min(max_subs, max(192 * self.world, -(-total // 4)))
        return plan_step_chunks(sub_counts, t0, t1, max_subs)

    def _barrier(self, stream):
        """Stream-ordered barrier over the ranks (a one-word all-reduce)."""
        import torch.distributed as dist
        with self.torch.cuda.stream(stream):
            dist.all_reduce(self._flag, group=self.group)

    # ---- the run ---------------------------------------------------------------------------------
    def run(self, t0, t1, d_stats_ptr, stream, sub_counts):
        """Steps [t0, t1): statistics of this band into the device array at d_stats_ptr ([t1 - t0, S_COUNT]
        float64, NOT yet reduced over ranks).  `stream` is the torch.cuda.Stream everything runs on."""
        torch = self.torch
        eng, me, world = self.eng, self.rank, self.world
        sp = stream.cuda_stream
        if world > 1 and self.comm is None:
            self.comm = torch.cuda.Stream()
            self._flag = torch.zeros(1, dtype=torch.int32, device="cuda")
        plan = self.chunks(t0, t1, sub_counts)
        if len(plan) > 1:
            eng.defer_snow_total(True)            # the rasters must not depend on where the run is cut
        # every rank needs the same receive size (symmetric allocation): largest band x largest chunk
        max_chunk_subs = 0
        for (c0, c1) in plan:
            s0, s1 = eng.sub_range(c0, c1)
            max_chunk_subs = max(max_chunk_subs, s1 - s0)
        recv_words = max(self.words) * max_chunk_subs
        self.bytes_sent_last_run = 0
        staged = {}

        def stage(k):
            """Sweep of chunk k (and its exchange) into slot k % 2."""
            c0, c1 = plan[k]
            s0, s1 = eng.sub_range(c0, c1)
            shares = split_even(s0, s1, world)
            a, b = shares[me]
            sl = self._recv(k % 2, recv_words)
            self.subs_last_scan = b - a           # (last_sweep_ms() of the engine times the last scan only)
            if world == 1:
                if b > a:
                    eng.shade_scan(a, b, [(self.bands[0][0], self.bands[0][1], sl["recv"].data_ptr())], sp)
            elif self.exchange == "p2p":
                # all ranks are done with this slot (fused kernels of chunk k - 2) before anybody writes into it
                if k >= 2:
                    self._barrier(stream)
                segs = [(r0, n, sl["peers"][q] + 4 * (a - s0) * self.words[q]) for q, (r0, n) in enumerate(self.bands)]
                if b > a:
                    eng.shade_scan(a, b, segs, sp)
                self._barrier(stream)             # every rank's stores have landed
                self.bytes_sent_last_run += 4 * (b - a) * (sum(self.words) - self.words[me])
            elif self.exchange == "copy":
                # sweep into the local send buffer (one segment per destination band), then bulk copies into
                # the peers' receive buffers on the side stream: copy engines over NVLink, no kernel
                in_split = [(b - a) * w for w in self.words]
                send = self._send(k % 2, sum(in_split))
                segs, off, offs = [], 0, []
                for (r0, n), w in zip(self.bands, in_split):
                    segs.append((r0, n, send.data_ptr() + 4 * off))
                    offs.append(off)
                    off += w
                if k >= 2:
                    self._barrier(stream)         # every rank has finished the fused kernels that read this slot
                if b > a:
                    eng.shade_scan(a, b, segs, sp)
                swept = torch.cuda.Event()
                swept.record(stream)
                with torch.cuda.stream(self.comm):
                    self.comm.wait_event(swept)
                    for dq in range(world):
                        q = (me + dq) % world     # start with myself, then round the ring: no two ranks hit one peer at once
                        n_w = in_split[q]
                        if n_w:
                            dst0 = (a - s0) * self.words[q]
                            sl["peer_tensors"][q][dst0:dst0 + n_w].copy_(send[offs[q]:offs[q] + n_w], non_blocking=True)
                    self._barrier(self.comm)      # every rank's copies have landed
                    done = torch.cuda.Event()
                    done.record(self.comm)
                sl["ready"] = done
                self.bytes_sent_last_run += 4 * (sum(in_split) - in_split[me])
            else:
                in_split = [(b - a) * w for w in self.words]                         # what I send to rank q
                out_split = [(hi - lo) * self.words[me] for lo, hi in shares]        # what rank p sends me
                send = self._send(k % 2, sum(in_split))
                segs, off = [], 0
                for (r0, n), w in zip(self.bands, in_split):
                    segs.append((r0, n, send.data_ptr() + 4 * off))
                    off += w
                if b > a:
                    eng.shade_scan(a, b, segs, sp)
                swept = torch.cuda.Event()
                swept.record(stream)
                import torch.distributed as dist
                with torch.cuda.stream(self.comm):
                    self.comm.wait_event(swept)
                    dist.all_to_all_single(sl["recv"][:sum(out_split)], send[:sum(in_split)], out_split, in_split,
                                           group=self.group)
                    done = torch.cuda.Event()
                    done.record(self.comm)
                sl["ready"] = done
                self.bytes_sent_last_run += 4 * (sum(in_split) - in_split[me])
            staged[k] = sl

        stage(0)
        for k, (c0, c1) in enumerate(plan):
            if k + 1 < len(plan):
                stage(k + 1)
            sl = staged.pop(k)
            if self.exchange in ("all_to_all", "copy"):
                stream.wait_event(sl["ready"])
            if len(plan) > 1 and k == len(plan) - 1:
                eng.defer_snow_total(False)
            stats_ptr = None if d_stats_ptr is None else d_stats_ptr + 8 * _lib.S_COUNT * (c0 - t0)
            # a chunk without a sunlit sub-step (polar night) needs no masks
            s0, s1 = eng.sub_range(c0, c1)
            eng.run_masked(c0, c1, sl["recv"].data_ptr() if s1 > s0 else None, stats_ptr, sp)


def allreduce_stats(stats):
    """In-place SUM of a [T, S_COUNT] statistics tensor over all ranks (torch.distributed)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    return stats


def means_from_sums(stats):
    """Area means laid out like the reference's CSV columns (var_classes.py:45-56, model.py:246-252)
    from the summed statistics: [T, 12] = rs, rl, lwd, sens, lat, atmo, g, melt, snow, ice, swe,
    snow cover per cent."""
    s = np.asarray(stats, dtype=np.float64)
    nv = s[:, _lib.S_NVALID]
    with np.errstate(invalid="ignore", divide="ignore"):
        cover = np.round(s[:, _lib.S_NSNOW] / s[:, _lib.S_NSWE] * 100)
        cols = [s[:, _lib.S_RS] / nv, (s[:, _lib.S_LWD] - s[:, _lib.S_LWU]) / nv, s[:, _lib.S_LWD] / nv,
                s[:, _lib.S_SENS] / nv, s[:, _lib.S_LAT] / nv, s[:, _lib.S_ATMO] / nv, s[:, _lib.S_G] / nv,
                s[:, _lib.S_MELT] / nv, s[:, _lib.S_SNOW] / nv, s[:, _lib.S_ICE] / nv,
                s[:, _lib.S_SWE] / s[:, _lib.S_NSWE], cover]
    return np.stack(cols, axis=1)
