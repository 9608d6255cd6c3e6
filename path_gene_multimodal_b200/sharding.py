"""Multi-GPU partitioning of the hot path (SURVEY 8e): one process per GPU.

* slide-parallel (BASELINE config 4): slides are independent, exactly like the reference's one-slide-per-LSF-job
  model (/root/reference/main.py:322-335) - ``assign_slides`` / ``slide_parallel``; no data-path collective,
  only a final gather of per-slide statistics.
* spatial strips of one giant slide (config 5): each rank owns the nuclei with x in [lo, hi) and all ranks
  exchange the points near strip edges with ONE all-gather (counts first, then a max-padded payload of 24-byte
  records packed by pg_halo_pack) over NCCL / NVLink.  Radius graph: halo width r.  kNN: halo width h with the
  per-point completeness test of pg_knn (k-th distance inside the region whose points are all present); the
  undirected union additionally queries the ghosts within h (halo 2h) so that every reverse edge into an owned
  row is seen locally - no second exchange.  Rows are emitted only for owned points with GLOBAL ids and the
  (d^2, global id) tie-break, so concatenating the ranks' outputs reproduces the single-GPU result bit for bit.

The algorithms are written as generators that ``yield`` their collectives; ``run`` drives one with
torch.distributed (NCCL on GPUs, gloo in the CPU tests), ``run_emulated`` steps several ranks in lockstep inside
one process (single-GPU tests of "sharded == single").
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from functools import partial

import numpy as np
import torch

_INF = float("inf")


# ------------------------------------------------------------------------------------------ slides
def assign_slides(n_slides: int, world: int, sizes=None) -> list[list[int]]:
    """Slides per rank: round-robin, or longest-processing-time-first when nuclei counts are known."""
    out = [[] for _ in range(world)]
    if sizes is None:
        for s in range(n_slides):
            out[s % world].append(s)
        return out
    load = [0] * world
    for s in sorted(range(n_slides), key=lambda i: (-int(sizes[i]), i)):
        r = min(range(world), key=lambda q: (load[q], q))
        out[r].append(s)
        load[r] += int(sizes[s])
    return [sorted(x) for x in out]


def slide_parallel(n_slides: int, fn, rank: int = 0, world: int = 1, sizes=None, group=None) -> dict:
    """Run ``fn(slide_index)`` for this rank's slides and gather every rank's results: {slide: result}.

    ``fn`` results must be small picklable summaries (statistics, counts, paths) - graphs stay on the
    rank that built them, as each LSF job of the reference keeps its own slide's outputs."""
    mine = assign_slides(n_slides, world, sizes)[rank]
    local = {s: fn(s) for s in mine}
    if world == 1:
        return local
    import torch.distributed as dist

    gathered = [None] * world
    dist.all_gather_object(gathered, local, group=group)
    merged = {}
    for d in gathered:
        merged.update(d)
    return merged


# ------------------------------------------------------------------------------------------ strips
@dataclass
class Strip:
    lo: float
    hi: float
    is_first: bool
    is_last: bool

    @property
    def x_lo(self):
        return -_INF if self.is_first else self.lo

    @property
    def x_hi(self):
        return _INF if self.is_last else self.hi


def strips_from_edges(edges) -> list[Strip]:
    w = len(edges) - 1
    return [Strip(float(edges[i]), float(edges[i + 1]), i == 0, i == w - 1) for i in range(w)]


def equal_count_edges(x: torch.Tensor, world: int, x_min: float, x_max: float, bins: int = 8192):
    """Generator: strip edges with ~equal nuclei counts from a global histogram of x (one all-reduce).

    Edges fall on histogram-bin boundaries so every rank derives identical values."""
    width = (x_max - x_min) / bins if x_max > x_min else 1.0
    b = torch.clamp(((x - x_min) / width).floor().long(), 0, bins - 1)
    hist = torch.bincount(b, minlength=bins).to(torch.int64)
    hist = yield ("all_reduce_sum", hist)
    cum = torch.cumsum(hist, 0).cpu().numpy()
    total = int(cum[-1])
    edges = [x_min]
    for q in range(1, world):
        target = total * q / world
        i = int(np.searchsorted(cum, target, side="left"))
        edges.append(x_min + (i + 1) * width)
    edges.append(x_max)
    for i in range(1, len(edges)):   # monotone even for degenerate histograms
        edges[i] = max(edges[i], edges[i - 1])
    return np.asarray(edges, dtype=np.float64)


def partition_by_strips(eng, xy: torch.Tensor, types: torch.Tensor, gid: torch.Tensor, edges, rank: int, world: int):
    """Generator: move every point to the rank owning its strip (one all-to-all of 24-byte records).

    Used when the table is not born partitioned; returns (xy, types, gid) of this rank's strip. The send buffer -
    records grouped by destination strip, input order kept - and the send counts come from pg_strip_partition
    (count / scan / place kernels); ONE host read (send + receive counts together) sizes the exchange."""
    recs, totals = eng.strip_partition(xy, types, gid, [float(e) for e in edges[1:-1]])
    send_counts = totals.to(torch.int64)
    recv_counts = yield ("all_to_all_counts", send_counts)
    both = torch.stack([send_counts, recv_counts]).tolist()   # the host synchronisation of this exchange
    got = yield ("all_to_all_v", recs.contiguous(), both[0], both[1])
    meta = got[:, 2].contiguous().view(torch.int32).reshape(-1, 2)
    return got[:, :2].contiguous(), meta[:, 1].contiguous(), meta[:, 0].contiguous()


def spatial_sort(eng, xy, types, gid, cell_size: float, bounds=None):
    """The strip's points in the cell order of a ``cell_size`` grid (one grid build + pg_grid_export).

    A strip owns its row order - its outputs are keyed by global id - so it may as well be the order in which the
    query kernels walk the points: the per-row records of the radius walk then land coalesced, the gather reads its
    parked entries in sequence, and the kNN union finds its neighbours' lists next to its own instead of at random
    places of a gigabyte-sized array. Returns (xy, types, gid) reordered."""
    if int(xy.shape[0]) == 0:
        return xy, types, gid
    eng.grid_build(xy, types, gid, cell_size, bounds)
    return eng.grid_export()


# ------------------------------------------------------------------------------------------ halo
def exchange_halo(eng, xy, types, gid, strip: Strip, width: float, rank: int, world: int):
    """Generator: pack this rank's edge points (pg_halo_pack), all-gather counts then the padded payload.

    Returns (all_recs float64 [world * max_cnt, 3] (24-byte records, padding rows are NaN), max_cnt). One host
    read per exchange: the gathered counts (they size the padded payload); the pack kernel cannot overflow, its
    capacity is the number of points."""
    n = int(xy.shape[0])
    if world == 1:
        return torch.empty((0, 3), dtype=torch.float64, device=xy.device), 0
    recs, count = eng.halo_pack(xy, types, gid, strip.x_lo + width, strip.x_hi - width, capacity=max(n, 1))
    counts = yield ("all_gather", count)                    # [world, 1] int32
    counts = counts.reshape(-1).tolist()                    # host sync: sizes the padded payload
    max_cnt = max(max(counts), 1)
    payload = torch.full((max_cnt, 3), float("nan"), dtype=torch.float64, device=xy.device)
    payload[:counts[rank]] = recs[:counts[rank]]
    all_recs = yield ("all_gather", payload)                # [world, max_cnt, 3]
    return all_recs.reshape(world * max_cnt, 3).contiguous(), max_cnt


def _append_ghosts(xy, types, gid, ghost_cap: int, ranges, unpack):
    """The owned points copied to the front of arrays with room for ``ghost_cap`` ghosts, behind which
    ``unpack(ranges, xy_all, types_all, gid_all, n_owned)`` (Engine.halo_unpack_multi / _slab with the source bound)
    appends the ghosts of each range. Returns (xy_all, types_all, gid_all, [count per range]) trimmed to the points
    present. One host read; none when ``unpack`` is None (nothing to append)."""
    n = int(xy.shape[0])
    cap = n + ghost_cap
    xy_all = torch.empty((cap, 2), dtype=torch.float64, device=xy.device)
    ty_all = torch.empty((cap,), dtype=torch.int32, device=xy.device)
    gid_all = torch.empty((cap,), dtype=torch.int32, device=xy.device)
    xy_all[:n] = xy
    ty_all[:n] = types
    gid_all[:n] = gid
    if unpack is None:
        return xy_all[:n], ty_all[:n], gid_all[:n], [0] * len(ranges)
    got = unpack(ranges, xy_all, ty_all, gid_all, n).tolist()   # host sync: the grid build needs the point count
    base = n + sum(got)
    return xy_all[:base], ty_all[:base], gid_all[:base], got


def merge_halo(eng, xy, types, gid, all_recs, max_cnt, rank, ranges):
    """Append to the owned points the gathered records whose x lies in each [a, b) of ``ranges`` (in that
    order), skipping this rank's own contribution. Returns (xy_all, types_all, gid_all, [count per range]).
    One enqueue for all ranges (pg_halo_unpack_multi) and one host read of the counts."""
    n_recs = int(all_recs.shape[0])
    unpack = partial(eng.halo_unpack_multi, all_recs, n_recs, rank * max_cnt, (rank + 1) * max_cnt) if n_recs else None
    return _append_ghosts(xy, types, gid, n_recs, ranges, unpack)


class PeerHalo:
    """This rank's halo receive slab, mapped into every rank of the group over NVLink (torch symmetric memory):
    ``world x cap`` 24-byte records followed by ``world`` int32 counts. With it the halo exchange is ONE kernel that
    packs and stores into the peers' slabs (pg_halo_push) between two device-side barriers - no NCCL call, no padded
    payload and no host read to size it. ``cap`` bounds the records one rank may contribute per exchange; exceeding
    it raises on every rank (all of them see every count)."""

    def __init__(self, cap: int, device, group=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm

        group = group if group is not None else dist.group.WORLD
        self.world, self.rank, self.cap = dist.get_world_size(group), dist.get_rank(group), int(cap)
        nbytes = self.world * self.cap * 24 + 8 * ((self.world * 4 + 7) // 8)
        self.buf = symm.empty(nbytes, dtype=torch.uint8, device=device)
        self.hdl = symm.rendezvous(self.buf, group)
        self.ptrs_dev = int(self.hdl.buffer_ptrs_dev)
        self.buf.zero_()
        torch.cuda.synchronize(device)
        self.hdl.barrier(channel=0)

    def exchange(self, eng, xy, types, gid, strip: "Strip", width: float, ranges, ghost_cap: int | None = None):
        """Push this rank's edge points to every peer, then append the received records of each x-range to the owned
        points. Same return as merge_halo. One host read (the unpack counts + the overflow flag)."""
        self.hdl.barrier(channel=0)                             # every peer is done reading the previous exchange
        eng.halo_push(xy, types, gid, strip.x_lo + width, strip.x_hi - width, self.ptrs_dev, self.world, self.rank, self.cap)
        self.hdl.barrier(channel=0)                             # all records and counts have landed
        ghost_cap = int(ghost_cap) if ghost_cap is not None else min(self.world - 1, 4) * self.cap
        out = _append_ghosts(xy, types, gid, ghost_cap, ranges,
                             partial(eng.halo_unpack_slab, self.buf, self.world, self.rank, self.cap))
        try:
            eng.check_overflow()
        except RuntimeError as exc:
            if getattr(exc, "code", None) != -4:      # PG_ERR_CAPACITY; anything else (a non-finite input ...) as it is
                raise
            raise RuntimeError(f"PeerHalo: a rank packed more than cap={self.cap} halo records (or more than {ghost_cap} "
                               "ghosts arrived here); build the PeerHalo with a larger cap") from exc
        return out


def _halo(eng, xy, types, gid, strip: Strip, width: float, rank: int, world: int, ranges, peer):
    """Generator: the owned points and the ghosts of each x-range, as merge_halo returns them. The halo of ``width``
    travels through ``peer``'s slabs when it is given and there are peers, else through exchange_halo."""
    if peer is not None and world > 1:
        return peer.exchange(eng, xy, types, gid, strip, width, ranges)
    all_recs, max_cnt = yield from exchange_halo(eng, xy, types, gid, strip, width, rank, world)
    return merge_halo(eng, xy, types, gid, all_recs, max_cnt, rank, ranges)


def sharded_radius_graph(eng, xy, types, gid, r: float, strip: Strip, rank: int, world: int, n_types: int = 5,
                         upper: bool = True, bounds=None, peer: PeerHalo | None = None):
    """Generator: radius graph rows of this rank's strip, columns in global ids.

    Returns the dict of Engine.radius_graph (row_ptr / col / dist32 / edges / degree / nbr_count / stats / hist)
    over the owned rows, plus ``row_gid`` (global id of each row) and ``n_ghost``."""
    from .engine import radius_cell

    ranges = [(strip.x_lo - r, strip.x_hi + r)]
    xy_all, ty_all, gid_all, got = yield from _halo(eng, xy, types, gid, strip, r, rank, world, ranges, peer)
    n_own = int(xy.shape[0])
    eng.grid_build(xy_all, ty_all, gid_all, radius_cell(r), bounds, n_query=n_own)
    g = eng.radius_graph(r, upper=upper, n_types=n_types, want_dist32=True, want_dist64=True, want_edges=upper)
    g["row_gid"] = gid
    g["n_ghost"] = got[0]
    return g


def _strip_bounds(strip: Strip, width: float, bounds):
    """Bounding box of a strip + halo when the slide's box is known: no reduction over the points, no host read."""
    if bounds is None:
        return None
    x0, y0, x1, y1 = (float(v) for v in bounds)
    lo = max(x0, strip.x_lo - width)
    hi = min(x1, strip.x_hi + width)
    return (lo, y0, max(hi, lo), y1)


def sharded_knn_graph(eng, xy, types, gid, k: int, strip: Strip, rank: int, world: int, n_global: int,
                      n_types: int = 5, union: bool = True, h0: float | None = None, density: float | None = None,
                      bounds=None, max_rounds: int = 8, peer: PeerHalo | None = None):
    """Generator: kNN lists (and the undirected union / composition) for this rank's strip, bit-exact with
    the single-GPU result. The halo width starts at ``h0`` (default 3 sqrt(k / (pi rho))) and doubles until
    every rank's completeness test passes (all-reduced), so a too-small guess costs a retry, never an error.

    ``bounds`` = (x0, y0, x1, y1) of the whole slide lets every rank derive its grid box without touching the
    points. Host reads per round: the gathered halo counts, the unpack counts, the all-reduced verdict."""
    from .engine import default_knn_cell

    n_own = int(xy.shape[0])
    if h0 is None:
        rho = density if density else 3.72e-4
        h0 = 3.0 * math.sqrt(k / (math.pi * rho))
    h = float(h0)
    for _ in range(max_rounds):
        width = 2.0 * h if union else h
        lo1, hi1 = strip.x_lo - h, strip.x_hi + h
        ranges = [(lo1, hi1)]
        if union:
            ranges += [(strip.x_lo - 2 * h, lo1), (hi1, strip.x_hi + 2 * h)]
        xy_all, ty_all, gid_all, got = yield from _halo(eng, xy, types, gid, strip, width, rank, world, ranges, peer)
        n_q = n_own + (got[0] if union else 0)
        n_all = int(xy_all.shape[0])
        kn = None
        red = torch.zeros((2,), dtype=torch.float64, device=xy.device)     # [all complete?, -max k-th distance]
        if k >= n_all:
            if world == 1:
                raise ValueError(f"k={k} must be smaller than the number of points ({n_all})")
        else:
            box = _strip_bounds(strip, width, bounds)
            if box is not None:
                area = max(box[2] - box[0], 1e-9) * max(box[3] - box[1], 1e-9)
            else:
                ext = torch.stack([xy_all.amax(0) - xy_all.amin(0)]).reshape(-1).tolist()
                area = max(ext[0], 1e-9) * max(ext[1], 1e-9)
            eng.grid_build(xy_all, ty_all, gid_all, default_knn_cell(n_all, area, k), box, n_query=n_q)
            kn = eng.knn(k, dist_dtype=torch.float64, x_lo=strip.x_lo - width, x_hi=strip.x_hi + width, check_halo=True)
            red[0] = kn["halo_ok"][0].to(torch.float64)
            if n_own:
                red[1] = -kn["dist"][:n_own, k - 1].max()
        red = yield ("all_reduce_min", red)
        verdict = red.tolist()                                   # the host synchronisation of the round
        ok, d_global = verdict[0] >= 1.0, -verdict[1]
        if ok and (not union or d_global <= h):
            break
        h = max(2.0 * h, d_global * 1.01)
    else:
        raise RuntimeError("sharded_knn_graph: halo did not converge")
    out = {"knn_idx": kn["knn_idx"][:n_own], "dist": kn["dist"][:n_own], "row_gid": gid, "halo": h,
           "n_ghost": int(xy_all.shape[0]) - n_own}
    if union:
        # rows address their neighbours by global id: dense id -> row / id -> type maps (pg_gid_maps), then the fused
        # union (pg_knn_union_*: CSR + i<j edge list + composition + degree in one rank pass) over own + ghost rows;
        # the owned rows are a prefix of every output
        id_map, type_by_gid = eng.gid_maps(gid_all, ty_all, n_q, n_global)
        u = eng.knn_union(kn["knn_idx"], kn["dist"], types=type_by_gid, n_types=n_types, row_id=gid_all[:n_q].contiguous(),
                          id_map=id_map, hist_len=0)
        ends = torch.stack([u["row_ptr"][n_own], u["up_ptr"][n_own]]).tolist()
        e_own, eu_own = int(ends[0]), int(ends[1])
        row_ptr = u["row_ptr"][:n_own + 1]
        st = eng.compose_degree(row_ptr.contiguous(), None, None, 1, compose=False)     # statistics over the owned rows only
        out.update({"row_ptr": row_ptr, "col": u["col"][:e_own], "w": u["w"][:e_own], "edges": u["edges"][:eu_own],
                    "weight": u["edge_w"][:eu_own], "degree": u["degree"][:n_own], "nbr_count": u["nbr_count"][:n_own],
                    "stats": st["stats"], "hist": st["hist"]})
    return out


# ------------------------------------------------------------------------------------------ drivers
class TorchComm:
    """Collectives of the generators above on a torch.distributed group (NCCL on GPUs, gloo on CPU)."""

    def __init__(self, group=None):
        import torch.distributed as dist

        self.dist, self.group = dist, group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)

    def execute(self, req):
        kind = req[0]
        d = self.dist
        if kind == "all_gather":
            t = req[1].contiguous()
            flat = torch.empty((self.world * t.numel(),), dtype=t.dtype, device=t.device)
            d.all_gather_into_tensor(flat, t.reshape(-1), group=self.group)
            return flat.reshape((self.world,) + tuple(t.shape))
        if kind in ("all_reduce_sum", "all_reduce_min"):
            t = req[1].clone()
            d.all_reduce(t, op=d.ReduceOp.SUM if kind == "all_reduce_sum" else d.ReduceOp.MIN, group=self.group)
            return t
        if kind == "all_to_all_counts":
            t = req[1].contiguous()
            out = torch.empty_like(t)
            d.all_to_all_single(out, t, group=self.group)
            return out
        if kind == "all_to_all_v":
            rec, send, recv = req[1], req[2], req[3]
            out = torch.empty((int(sum(recv)),) + tuple(rec.shape[1:]), dtype=rec.dtype, device=rec.device)
            d.all_to_all_single(out, rec.contiguous(), output_split_sizes=list(recv), input_split_sizes=list(send), group=self.group)
            return out
        raise ValueError(f"unknown collective {kind}")


class LocalComm:
    """The collectives of a one-rank world (the generators then run unchanged on a single GPU)."""

    world, rank = 1, 0

    def execute(self, req):
        kind = req[0]
        if kind == "all_gather":
            return req[1].contiguous().unsqueeze(0)
        if kind in ("all_reduce_sum", "all_reduce_min", "all_to_all_counts", "all_to_all_v"):
            return req[1]
        raise ValueError(f"unknown collective {kind}")


def run(gen, comm: TorchComm | None = None):
    """Drive one generator to completion, executing the collectives it yields."""
    try:
        req = next(gen)
        while True:
            if comm is None:
                raise RuntimeError("a collective was requested but no communicator was given")
            req = gen.send(comm.execute(req))
    except StopIteration as stop:
        return stop.value


def run_emulated(gens: list):
    """Step the generators of all ranks in lockstep inside one process (ranks emulated one after another)."""
    world = len(gens)
    results = [None] * world
    reqs = [None] * world
    live = [True] * world
    for q, g in enumerate(gens):
        try:
            reqs[q] = next(g)
        except StopIteration as stop:
            results[q], live[q] = stop.value, False
    while any(live):
        assert all(live), "ranks must issue the same collectives"
        kind = reqs[0][0]
        assert all(r[0] == kind for r in reqs)
        if kind == "all_gather":
            stacked = torch.stack([r[1] for r in reqs])
            answers = [stacked.clone() for _ in range(world)]
        elif kind == "all_reduce_sum":
            tot = torch.stack([r[1] for r in reqs]).sum(0)
            answers = [tot.clone() for _ in range(world)]
        elif kind == "all_reduce_min":
            tot = torch.stack([r[1] for r in reqs]).min(0).values
            answers = [tot.clone() for _ in range(world)]
        elif kind == "all_to_all_counts":
            m = torch.stack([r[1] for r in reqs])      # m[src, dst]
            answers = [m[:, q].clone() for q in range(world)]
        elif kind == "all_to_all_v":
            answers = []
            for q in range(world):
                parts = []
                for src in range(world):
                    send = reqs[src][2]
                    off = int(sum(send[:q]))
                    parts.append(reqs[src][1][off:off + int(send[q])])
                answers.append(torch.cat(parts))
        else:
            raise ValueError(kind)
        for q, g in enumerate(gens):
            try:
                reqs[q] = g.send(answers[q])
            except StopIteration as stop:
                results[q], live[q] = stop.value, False
    return results
