"""Target intervals of a restricted run: `--bed FILE` and `--region CTG[:START-END]` of `python -m nanosnp_b200.predict`.

Both feed one list: per contig of the reference index, sorted, merged, 0-based half-open [start, end) intervals clipped to
the contig.  A site at 0-based position c is kept iff c lies in an interval (shard.plan_target_units, runner.run_device).
"""
from __future__ import annotations

import sys
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np


def merge_intervals(iv: Iterable[Tuple[int, int]], length: int) -> np.ndarray:
    """Clips to [0, length), drops empty intervals, merges overlapping and adjacent ones: int64 [k, 2], ascending."""
    out: List[List[int]] = []
    for s, e in sorted((max(0, s), min(length, e)) for s, e in iv):
        if s >= e:
            continue
        if out and s <= out[-1][1]:
            out[-1][1] = max(out[-1][1], e)
        else:
            out.append([s, e])
    return np.array(out, np.int64).reshape(-1, 2)


def parse_bed(lines: Iterable[str], name: str = "BED") -> List[Tuple[str, int, int]]:
    """(contig, start, end) of every interval line: the first three whitespace-separated fields, 0-based half-open.  Blank
    lines and `#` / `track` / `browser` lines are skipped.  A malformed line raises ValueError naming its line number."""
    out = []
    for no, line in enumerate(lines, 1):
        f = line.split()
        if not f or f[0].startswith("#") or f[0] in ("track", "browser"):
            continue
        try:
            if len(f) < 3:
                raise ValueError("fewer than three fields")
            s, e = int(f[1]), int(f[2])
            if s < 0:
                raise ValueError("negative start")
            if e < s:
                raise ValueError("end before start")
        except ValueError as err:
            raise ValueError(f"{name} line {no}: {err}: {line.rstrip()!r}") from None
        out.append((f[0], s, e))
    return out


def parse_region(spec: str, lengths: Dict[str, int]) -> Tuple[str, int, int]:
    """`CTG` or `CTG:START-END` (1-based inclusive, commas allowed) -> (contig, start, end) 0-based half-open.  A string that
    is a contig name of the index as a whole is that contig (names may contain ':')."""
    if spec in lengths:
        return spec, 0, lengths[spec]
    ctg, sep, rng = spec.rpartition(":")
    a, dash, b = rng.replace(",", "").partition("-")
    try:
        if not sep or not ctg or not dash:
            raise ValueError
        s, e = int(a), int(b)
    except ValueError:
        raise ValueError(f"--region {spec!r}: expected CTG or CTG:START-END") from None
    if s < 1 or e < s:
        raise ValueError(f"--region {spec!r}: need 1 <= START <= END")
    return ctg, s - 1, e


def build_targets(contigs: Sequence[Tuple[str, int]], bed: Optional[str] = None, regions: Sequence[str] = (),
                  report=sys.stderr) -> Dict[str, np.ndarray]:
    """The union of a BED file and --region strings, per contig of the reference index (contigs without an interval are
    absent).  Intervals on contigs outside the index are skipped; their number is reported once on `report`."""
    lengths = dict(contigs)
    raw: List[Tuple[str, int, int]] = []
    if bed is not None:
        with open(bed) as f:
            raw += parse_bed(f, bed)
    raw += [parse_region(r, lengths) for r in regions]
    per: Dict[str, List[Tuple[int, int]]] = {}
    skipped = 0
    for c, s, e in raw:
        if c not in lengths:
            skipped += 1
            continue
        per.setdefault(c, []).append((s, e))
    if skipped and report is not None:
        print(f"nanosnp_b200: skipped {skipped} target interval(s) on contigs that are not in the reference index", file=report)
    out = {}
    for c, iv in per.items():
        m = merge_intervals(iv, lengths[c])
        if len(m):
            out[c] = m
    return out


def in_targets(pos0: np.ndarray, iv: Optional[np.ndarray]) -> np.ndarray:
    """Boolean mask: 0-based positions inside the sorted disjoint intervals iv."""
    pos0 = np.asarray(pos0, np.int64)
    if iv is None or len(iv) == 0:
        return np.zeros(len(pos0), bool)
    k = np.searchsorted(iv[:, 1], pos0, side="right")
    inside = k < len(iv)
    inside[inside] &= iv[k[inside], 0] <= pos0[inside]
    return inside
