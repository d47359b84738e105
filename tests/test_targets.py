"""Target intervals (`--bed` / `--region`) on the host: parsing, unit planning, the tile rule, multi-range BAM fetch."""
import io

import numpy as np
import pytest

from nanosnp_b200.shard import FLANK, Region, fetch_ranges, listed_tiles, plan_regions, plan_target_units
from nanosnp_b200.targets import build_targets, in_targets, merge_intervals, parse_bed, parse_region

CONTIGS = [("chr1", 10_000), ("chr2", 5_000), ("HLA-A*01:01:01:01", 3_000)]


def _bed(tmp_path, text):
    p = tmp_path / "t.bed"
    p.write_text(text)
    return str(p)


def test_bed_comments_whitespace_extra_columns(tmp_path):
    bed = _bed(tmp_path, "# header\ntrack name=x\nbrowser position chr1:1-100\n\n"
                         "chr1\t100\t200\tname\t0\t+\n"
                         "chr1 300   400 extra\n"
                         "  \t\n"
                         "chr2\t0\t10\n")
    t = build_targets(CONTIGS, bed, report=None)
    assert set(t) == {"chr1", "chr2"}
    assert t["chr1"].tolist() == [[100, 200], [300, 400]] and t["chr2"].tolist() == [[0, 10]]


def test_bed_unsorted_overlapping_adjacent_duplicate_empty(tmp_path):
    bed = _bed(tmp_path, "chr1\t500\t600\nchr1\t100\t200\nchr1\t150\t250\nchr1\t250\t260\nchr1\t100\t200\n"
                         "chr1\t700\t700\nchr1\t900\t950\nchr1\t950\t951\nchr2\t7\t7\n")
    t = build_targets(CONTIGS, bed, report=None)
    assert t["chr1"].tolist() == [[100, 260], [500, 600], [900, 951]]
    assert "chr2" not in t                                   # only an empty interval


def test_bed_clip_and_unknown_contig(tmp_path):
    bed = _bed(tmp_path, "chr2\t4990\t9000\nchr2\t6000\t7000\nchrUn\t1\t5\nchrUn\t8\t9\nchr1\t0\t1\n")
    err = io.StringIO()
    t = build_targets(CONTIGS, bed, report=err)
    assert t["chr2"].tolist() == [[4990, 5000]] and t["chr1"].tolist() == [[0, 1]]
    msg = err.getvalue()
    assert msg.count("\n") == 1 and "skipped 2 " in msg


@pytest.mark.parametrize("line,what", [("chr1\t1.5\t10", "line 3"), ("chr1\t-1\t10", "negative"), ("chr1\t20\t10", "end before start"),
                                       ("chr1\t20", "fewer than three"), ("chr1\tx\t10", "line 3")])
def test_bed_malformed_names_line(tmp_path, line, what):
    bed = _bed(tmp_path, f"# c\nchr1\t1\t2\n{line}\n")
    with pytest.raises(ValueError) as e:
        build_targets(CONTIGS, bed, report=None)
    assert "line 3" in str(e.value) and what in str(e.value)


def test_region_strings():
    L = dict(CONTIGS)
    assert parse_region("chr1", L) == ("chr1", 0, 10_000)
    assert parse_region("chr1:1-1", L) == ("chr1", 0, 1)
    assert parse_region("chr1:1,001-2,000", L) == ("chr1", 1000, 2000)
    assert parse_region("HLA-A*01:01:01:01", L) == ("HLA-A*01:01:01:01", 0, 3000)        # a whole name that contains ':'
    assert parse_region("HLA-A*01:01:01:01:11-20", L) == ("HLA-A*01:01:01:01", 10, 20)
    for bad in ("chr1:0-5", "chr1:9-5", "chr1:5", "chr1:a-b", "nosuch"):
        with pytest.raises(ValueError):
            parse_region(bad, L)


def test_bed_and_region_union(tmp_path):
    bed = _bed(tmp_path, "chr1\t100\t200\n")
    t = build_targets(CONTIGS, bed, ["chr1:201-300", "chr2", "chrX:1-5"], report=None)
    assert t["chr1"].tolist() == [[100, 300]] and t["chr2"].tolist() == [[0, 5000]]
    assert build_targets(CONTIGS, _bed(tmp_path, "# nothing\n"), report=None) == {}


def test_in_targets():
    iv = np.array([[3, 5], [10, 11]])
    assert in_targets(np.arange(13), iv).nonzero()[0].tolist() == [3, 4, 10]
    assert not in_targets(np.arange(5), None).any()


def _random_targets(rng, L, n, max_len):
    s = rng.integers(0, L, n)
    e = s + rng.integers(0, max_len, n)
    return merge_intervals(zip(s.tolist(), e.tolist()), L)


@pytest.mark.parametrize("region_len", [1, 50, 1000, 7_777, 100_000])
def test_plan_target_units_invariants(region_len):
    rng = np.random.default_rng(region_len)
    contigs = [("a", 60_000), ("b", 3_000), ("c", 250_000)]
    for trial in range(6):
        targets = {nm: _random_targets(rng, L, int(rng.integers(0, 300)), int(rng.choice([2, 40, 3000, 30_000]))) for nm, L in contigs}
        units, ivs = plan_target_units(contigs, targets, region_len)
        assert len(units) == len(ivs)
        for ci, (nm, L) in enumerate(contigs):
            mine = [(u, iv) for u, iv in zip(units, ivs) if u.contig == nm]
            hit = np.zeros(L, np.int32)
            for u, iv in mine:
                assert u.contig_index == ci and u.contig_len == L
                assert u.emit_end - u.emit_start <= region_len and u.length <= region_len + 2 * FLANK
                assert iv[0, 0] == u.emit_start and iv[-1, 1] == u.emit_end
                assert (iv[:, 0] < iv[:, 1]).all() and (iv[1:, 0] >= iv[:-1, 1]).all()
                for s, e in iv:
                    hit[s:e] += 1
            for (u, _), (v, _) in zip(mine, mine[1:]):
                assert u.emit_end <= v.emit_start                  # sorted and disjoint emit spans
            want = np.zeros(L, np.int32)
            for s, e in targets.get(nm, np.zeros((0, 2), np.int64)):
                want[s:e] = 1
            assert (hit == want).all()                            # every target position is emitted by exactly one unit


def test_whole_contig_targets_plan_like_plan_regions():
    contigs = [("a", 1_000_003), ("b", 77)]
    for rl in (10_000, 333_333, 2_000_000):
        units, _ = plan_target_units(contigs, {nm: np.array([[0, L]]) for nm, L in contigs}, rl)
        assert units == plan_regions(contigs, rl)


def test_listed_tiles_rule_at_the_pileup_tile():
    tile = 1024                                                   # the pileup kernel's position tile (kTile, pileup.cu)
    rng = np.random.default_rng(tile)
    for trial in range(40):
        L = int(rng.integers(1, 40_000))
        iv = _random_targets(rng, L, int(rng.integers(1, 30)), int(rng.choice([1, 20, 2000])))
        if not len(iv):
            continue
        rg = Region("x", 0, L, int(iv[0, 0]), int(iv[-1, 1]))
        near = np.zeros(rg.length, bool)                          # positions of [start-16, end+16) inside the computed span
        for s, e in iv:
            a, b = max(s - FLANK, rg.start), min(e + FLANK, rg.end)
            near[a - rg.start:b - rg.start] = True
        want = sorted({p // tile for p in np.nonzero(near)[0].tolist()})
        assert listed_tiles(rg, iv).tolist() == want


def test_fetch_ranges_halo_merge():
    rg = Region("x", 0, 1000, 10, 900)
    assert fetch_ranges(rg, np.array([[10, 20], [40, 50], [100, 110], [890, 900]])).tolist() == [[0, 66], [84, 126], [874, 916]]
    assert fetch_ranges(Region("x", 0, 1000, 0, 1000), np.array([[0, 1000]])).tolist() == [[0, 1000]]


def test_bam_fetch_ranges(tmp_path):
    from nanosnp_b200.bam import BamReader, write_bam
    from nanosnp_b200.reads import max_reference_span
    from nanosnp_b200.synth import SynthConfig, generate_host
    refs, reads = {}, {}
    for i, (name, L) in enumerate([("c1", 1_500_000), ("c2", 200_000)]):
        cfg = SynthConfig(contig_len=L, coverage=12.0, contig=name, seed_ref=3 + i, seed_var=5 + i, seed_reads=7 + i, len_median=3000, len_min=200)
        refs[name], reads[name] = generate_host(cfg)
    path = str(tmp_path / "x.bam")
    write_bam(path, [(n, len(r)) for n, r in refs.items()], reads, index=True)
    rd = reads["c1"]
    ends = rd.pos.astype(np.int64) + np.maximum(max_reference_span_each(rd), 1)
    rng = np.random.default_rng(0)
    for ranges in ([[0, 10]], [[1000, 2000], [2000, 2500], [700_000, 700_001], [1_499_000, 1_500_000]],
                   [[s, s + 50] for s in range(5_000, 1_500_000, 97_000)], [[0, 1_500_000]],
                   sorted([[int(s), int(s) + 300] for s in rng.choice(np.arange(0, 1_499_000, 20_000), 12, replace=False)])):
        r_np = np.array(ranges)
        sel = np.zeros(rd.n_reads, bool)
        for s, e in ranges:
            sel |= (rd.pos < e) & (ends > s)
        with BamReader(path) as r:
            got = r.fetch_ranges(0, ranges)
        assert got.n_reads == int(sel.sum())
        assert (got.pos == rd.pos[sel]).all()                     # each once, in file order
        want_cig = np.concatenate([rd.cigar[rd.cigar_off[i]:rd.cigar_off[i + 1]] for i in np.nonzero(sel)[0]] or [np.zeros(0, rd.cigar.dtype)])
        assert (got.cigar.astype(np.uint32) == want_cig.astype(np.uint32)).all()
        assert r_np.shape[1] == 2
    sparse = [[s, s + 100] for s in (10_000, 600_000, 1_200_000)]
    with BamReader(path) as r:
        r.fetch(0, 10_000, 1_200_100)
        union = r.inflated_bytes
    with BamReader(path) as r:
        r.fetch_ranges(0, sparse)
        part = r.inflated_bytes
    assert part < 0.5 * union
    with BamReader(path) as r:
        for bad in ([[10, 5]], [[0, 10], [5, 20]], [[-1, 3]]):
            with pytest.raises(ValueError):
                r.fetch_ranges(0, bad)
        assert r.fetch_ranges(1, np.zeros((0, 2))).n_reads == 0


def max_reference_span_each(rd):
    """Reference span of every read (M D N = X)."""
    op = rd.cigar.astype(np.uint32) & 15
    ln = (rd.cigar.astype(np.uint32) >> 4).astype(np.int64)
    consume = np.isin(op, [0, 2, 3, 7, 8])
    cs = np.concatenate([[0], np.cumsum(np.where(consume, ln, 0))])
    return cs[rd.cigar_off[1:]] - cs[rd.cigar_off[:-1]]
