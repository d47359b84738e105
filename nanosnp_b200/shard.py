"""Region sharding of the s1+s2 path across GPUs (SURVEY.md section 8e).

Every site depends only on reads overlapping [c-16, c+16], so contigs are cut into fixed regions [s, e);
each region is computed on [s-16, e+16) and emits the sites with s <= c < e.  Regions are independent:
there is no data-path collective.  Per-rank call lists are gathered to rank 0 (torch.distributed
gather_object: NCCL/gloo plumbing only) and concatenated in (contig, position) order BEFORE the record
logic runs in 1000-site batches per contig, because predict.py's output depends on batch composition
(SURVEY 8a, row P13).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Sequence, Tuple

import numpy as np

FLANK = 16


@dataclass(frozen=True)
class Region:
    contig: str
    contig_index: int
    contig_len: int
    emit_start: int      # sites with emit_start <= c < emit_end belong to this region
    emit_end: int

    @property
    def start(self) -> int:          # computed span = emitted span + halo
        return max(0, self.emit_start - FLANK)

    @property
    def end(self) -> int:
        return min(self.contig_len, self.emit_end + FLANK)

    @property
    def length(self) -> int:
        return self.end - self.start


def plan_regions(contigs: Sequence[Tuple[str, int]], region_len: int) -> List[Region]:
    """Cuts each (name, length) contig into regions of at most region_len emitted positions."""
    out = []
    for ci, (name, L) in enumerate(contigs):
        n = max(1, -(-L // region_len))
        step = -(-L // n)
        for k in range(n):
            s, e = k * step, min(L, (k + 1) * step)
            if s < e:
                out.append(Region(name, ci, L, s, e))
    return out


def plan_target_units(contigs: Sequence[Tuple[str, int]], targets: Dict[str, np.ndarray],
                      region_len: int) -> Tuple[List[Region], List[np.ndarray]]:
    """Work units of a targeted run.  targets: contig -> merged, sorted [k, 2] [start, end) intervals.  An interval longer
    than region_len is cut like plan_regions cuts a contig; consecutive intervals (or pieces) share a unit while the unit's
    emitted span [first start, last end) stays <= region_len.  Units have disjoint emit spans in contig order.  Returns the
    units and, aligned with them, each unit's intervals as int64 [k, 2] (kept out of the hashed Region)."""
    units: List[Region] = []
    unit_iv: List[np.ndarray] = []
    for ci, (name, L) in enumerate(contigs):
        iv = targets.get(name)
        if iv is None or len(iv) == 0:
            continue
        pieces = []
        for s, e in np.asarray(iv, np.int64).reshape(-1, 2).tolist():
            n = max(1, -(-(e - s) // region_len))
            step = -(-(e - s) // n)
            pieces += [(s + k * step, min(e, s + (k + 1) * step)) for k in range(n) if s + k * step < e]
        cur: List[Tuple[int, int]] = []
        for s, e in pieces + [(None, None)]:
            if cur and (s is None or e - cur[0][0] > region_len):
                units.append(Region(name, ci, L, cur[0][0], cur[-1][1]))
                unit_iv.append(np.array(cur, np.int64))
                cur = []
            if s is not None:
                cur.append((s, e))
    return units, unit_iv


def listed_tiles(region: Region, intervals: np.ndarray, tile: int = 1024) -> np.ndarray:
    """The tiles (indices from region.start) the GPU computes for a unit: those holding any position of [start-16, end+16)
    of an interval, clipped to the unit's computed span."""
    iv = np.asarray(intervals, np.int64).reshape(-1, 2)
    a = np.maximum(iv[:, 0] - FLANK, region.start) - region.start
    b = np.minimum(iv[:, 1] + FLANK, region.end) - region.start
    keep = a < b
    n_tiles = -(-region.length // tile)
    diff = np.zeros(n_tiles + 1, np.int64)
    np.add.at(diff, a[keep] // tile, 1)
    np.add.at(diff, (b[keep] - 1) // tile + 1, -1)
    return np.nonzero(np.cumsum(diff[:n_tiles]) > 0)[0]


def fetch_ranges(region: Region, intervals: np.ndarray) -> np.ndarray:
    """[start-16, end+16) of every interval, clipped to the contig and merged: the reference ranges whose reads a unit needs."""
    out: List[List[int]] = []
    for s, e in np.asarray(intervals, np.int64).reshape(-1, 2).tolist():
        s, e = max(0, s - FLANK), min(region.contig_len, e + FLANK)
        if out and s <= out[-1][1]:
            out[-1][1] = max(out[-1][1], e)
        else:
            out.append([s, e])
    return np.array(out, np.int64).reshape(-1, 2)


def assign_lpt(regions: Sequence[Region], world_size: int, weights: Sequence[int] = None) -> List[List[int]]:
    """Longest-processing-time-first assignment of regions to ranks (balances 25 unequal contigs).  weights: optional cost of
    each region (a targeted run passes its listed tiles); default: the computed span.
    Deterministic; returns per-rank lists of region indices, each in (contig, position) order."""
    w = [rg.length for rg in regions] if weights is None else [int(x) for x in weights]
    order = sorted(range(len(regions)), key=lambda i: (-w[i], i))
    load = [0] * world_size
    mine: List[List[int]] = [[] for _ in range(world_size)]
    for i in order:
        r = min(range(world_size), key=lambda k: (load[k], k))
        load[r] += w[i]
        mine[r].append(i)
    for m in mine:
        m.sort()
    return mine


def read_range_for_region(read_pos: np.ndarray, max_span: int, region: Region) -> Tuple[int, int]:
    """Conservative [lo, hi) slice of a position-sorted read array that can overlap the region's computed span.
    Reads spanning a boundary are handed to both neighbours (at most one read length of duplication)."""
    lo = int(np.searchsorted(read_pos, region.start - max_span, side="left"))
    hi = int(np.searchsorted(read_pos, region.end, side="left"))
    return lo, hi


def merge_site_lists(parts: Sequence[Dict[str, np.ndarray]]) -> Dict[str, np.ndarray]:
    """Concatenates per-region results {contig_index, pos, ...} and orders them by (contig_index, pos)."""
    parts = [p for p in parts if p is not None and len(p["pos"])]
    if not parts:
        return {}
    keys = parts[0].keys()
    cat = {k: np.concatenate([p[k] for p in parts]) for k in keys}
    order = np.lexsort((cat["pos"], cat["contig_index"]))
    return {k: v[order] for k, v in cat.items()}


def gather_to_rank0(local_parts: List[Dict[str, np.ndarray]]):
    """torch.distributed plumbing: returns the merged site list on rank 0, None elsewhere."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return merge_site_lists(local_parts)
    gathered = [None] * dist.get_world_size() if dist.get_rank() == 0 else None
    dist.gather_object(local_parts, gathered, dst=0)
    if dist.get_rank() != 0:
        return None
    flat = [p for parts in gathered for p in parts]
    return merge_site_lists(flat)
