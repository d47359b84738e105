"""Target intervals of a restricted run: `--bed FILE` and `--region CTG[:START-END]` of `python -m nanosnp_b200.predict`.

Both feed one list: per contig of the reference index, sorted, merged, 0-based half-open [start, end) intervals clipped to
the contig.  A site at 0-based position c is kept iff c lies in an interval (shard.plan_target_units, runner.run_device).
`--sites FILE` (a VCF of given sites) uses the same representation: runs of consecutive listed positions are one interval.
"""
from __future__ import annotations

import gzip
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


def site_intervals(pos0: np.ndarray) -> np.ndarray:
    """Sorted, merged intervals of a set of 0-based positions: every run of consecutive positions is one [start, end)."""
    u = np.unique(np.asarray(pos0, np.int64))
    if len(u) == 0:
        return np.zeros((0, 2), np.int64)
    brk = np.nonzero(np.diff(u) != 1)[0]
    return np.stack([u[np.r_[0, brk + 1]], u[np.r_[brk, len(u) - 1]] + 1], axis=1)


def parse_sites(lines: Iterable[str], name: str = "VCF") -> List[Tuple[str, int]]:
    """(CHROM, POS) of every data line of a VCF, POS as written (1-based).  `#` lines and blank lines are skipped; the other
    columns are ignored.  A line with fewer than two columns or a non-integer POS raises ValueError naming its line number."""
    out = []
    for no, line in enumerate(lines, 1):
        if line.startswith("#") or not line.strip():
            continue
        f = line.split()
        try:
            if len(f) < 2:
                raise ValueError("fewer than two columns")
            p = int(f[1])
        except ValueError as err:
            raise ValueError(f"{name} line {no}: {err}: {line.rstrip()!r}") from None
        out.append((f[0], p))
    return out


def load_sites_vcf(path: str, contigs: Sequence[Tuple[str, int]], report=sys.stderr) -> Dict[str, np.ndarray]:
    """The sites of a VCF (plain, or gzip / bgzip by its magic bytes) per contig of the reference index, as merged int64
    [k, 2] intervals of 0-based positions c = POS - 1 (contigs without a site are absent).  Duplicates collapse; sites on
    contigs outside the index or outside [1, contig length] are skipped, and their number is reported once on `report`."""
    lengths = dict(contigs)
    with open(path, "rb") as f:
        gz = f.read(2) == b"\x1f\x8b"
    with (gzip.open(path, "rt") if gz else open(path)) as f:
        raw = parse_sites(f, path)
    per: Dict[str, List[int]] = {}
    skipped = 0
    for c, p in raw:
        if c not in lengths or not 1 <= p <= lengths[c]:
            skipped += 1
            continue
        per.setdefault(c, []).append(p - 1)
    if skipped and report is not None:
        print(f"nanosnp_b200: skipped {skipped} site(s) on contigs that are not in the reference index or outside the contig",
              file=report)
    return {c: site_intervals(p) for c, p in per.items()}


def intersect_targets(a: Dict[str, np.ndarray], b: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
    """Per contig, the positions in both sets of sorted merged intervals, as sorted merged intervals (contigs left empty
    are absent): the sites of `--sites` that lie inside `--bed` / `--region` targets."""
    out = {}
    for c in a.keys() & b.keys():
        x, y = np.asarray(a[c], np.int64).reshape(-1, 2), np.asarray(b[c], np.int64).reshape(-1, 2)
        # every interval of x against the intervals of y it overlaps: y[lo:hi] with y.end > x.start and y.start < x.end
        lo = np.searchsorted(y[:, 1], x[:, 0], side="right")
        hi = np.searchsorted(y[:, 0], x[:, 1], side="left")
        n = np.maximum(hi - lo, 0)
        xi = np.repeat(np.arange(len(x)), n)
        yi = np.arange(n.sum()) - np.repeat(np.cumsum(n) - n, n) + np.repeat(lo, n)
        s, e = np.maximum(x[xi, 0], y[yi, 0]), np.minimum(x[xi, 1], y[yi, 1])
        keep = s < e
        if keep.any():                                  # pieces of merged inputs never touch: the result is merged too
            out[c] = np.stack([s[keep], e[keep]], axis=1)
    return out
