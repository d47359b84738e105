"""`--sites FILE`: parsing of the site VCF, merging of 1-bp runs into intervals and intersection with BED targets (CPU)."""
import gzip
import io

import numpy as np
import pytest

from nanosnp_b200.targets import (build_targets, in_targets, intersect_targets, load_sites_vcf, merge_intervals, parse_sites,
                                  site_intervals)

CONTIGS = [("chr1", 1000), ("chr2", 50)]
VCF = ("##fileformat=VCFv4.2\n"
       "##contig=<ID=chr1,length=1000>\n"
       "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"
       "chr1\t10\trs1\tA\tG\t.\t.\t.\n"
       "chr1\t11\t.\tC\tT,G\t.\t.\t.\n"                 # multi-allelic: only CHROM / POS count
       "chr1\t12\t.\tCTT\tC\t.\t.\t.\n"                 # indel record
       "chr1\t10\trs1\tA\tG\t.\t.\t.\n"                 # duplicate
       "chr1\t500\n"                                     # two columns are enough
       "chrX\t5\t.\tA\tG\t.\t.\t.\n"                    # contig not in the index
       "chr1\t1001\t.\tA\tG\t.\t.\t.\n"                 # past the contig end
       "chr1\t0\t.\tA\tG\t.\t.\t.\n"                    # POS 0
       "\n"
       "chr2\t50\t.\tA\tG\t.\t.\t.\n"
       "chr1\t1000\t.\tA\tG\t.\t.\t.\n")
WANT = {"chr1": np.array([[9, 12], [499, 500], [999, 1000]]), "chr2": np.array([[49, 50]])}


def _eq(got, want):
    assert set(got) == set(want)
    for c in want:
        assert got[c].dtype == np.int64 and np.array_equal(got[c], want[c]), (c, got[c], want[c])


@pytest.mark.parametrize("form", ["plain", "crlf", "gzip", "bgzip"])
def test_load_sites_vcf_forms(tmp_path, form):
    from nanosnp_b200.bam import bgzf_compress
    text = VCF.replace("\n", "\r\n") if form == "crlf" else VCF
    raw = text.encode()
    p = tmp_path / ("s.vcf.gz" if form in ("gzip", "bgzip") else "s.vcf")
    p.write_bytes(gzip.compress(raw) if form == "gzip" else bgzf_compress(raw) if form == "bgzip" else raw)
    rep = io.StringIO()
    _eq(load_sites_vcf(str(p), CONTIGS, report=rep), WANT)
    msg = rep.getvalue()
    assert msg.count("\n") == 1 and "skipped 3 site(s)" in msg


def test_bgzip_of_many_blocks(tmp_path):
    from nanosnp_b200.bam import bgzf_compress
    pos = np.arange(1, 200_001, 3)
    raw = ("#CHROM\tPOS\n" + "".join(f"chr1\t{p}\t.\tA\tG\n" for p in pos)).encode()
    assert len(raw) > 3 * 65536                                      # several BGZF members
    blob = bgzf_compress(raw)
    (tmp_path / "m.vcf.gz").write_bytes(blob)
    got = load_sites_vcf(str(tmp_path / "m.vcf.gz"), [("chr1", 300_000)], report=None)
    assert np.array_equal(got["chr1"], np.stack([pos - 1, pos], axis=1))


@pytest.mark.parametrize("line,why", [("chr1\n", "fewer than two columns"), ("chr1\tx12\tA\n", "x12"),
                                      ("chr1\t1.5\tA\n", "1.5")])
def test_malformed_line_names_it(line, why):
    with pytest.raises(ValueError) as e:
        parse_sites(["#h\n", "chr1\t5\n", line], "my.vcf")
    assert "my.vcf line 3" in str(e.value) and why in str(e.value)


def test_no_report_without_skips_and_empty_lists(tmp_path):
    p = tmp_path / "e.vcf"
    p.write_text("##x\n#CHROM\tPOS\n")
    rep = io.StringIO()
    assert load_sites_vcf(str(p), CONTIGS, report=rep) == {} and rep.getvalue() == ""
    p.write_text("chrZ\t3\n")
    assert load_sites_vcf(str(p), CONTIGS, report=rep) == {} and "skipped 1 site(s)" in rep.getvalue()


def test_runs_merge_into_intervals():
    assert site_intervals([]).shape == (0, 2)
    assert np.array_equal(site_intervals([7]), [[7, 8]])
    assert np.array_equal(site_intervals([5, 3, 4, 4, 9, 11, 10, 20]), [[3, 6], [9, 12], [20, 21]])
    rng = np.random.default_rng(1)
    for _ in range(200):
        pos = rng.integers(0, 300, rng.integers(0, 120))
        iv = site_intervals(pos)
        assert np.array_equal(iv, merge_intervals([(int(p), int(p) + 1) for p in pos], 300))
        covered = np.zeros(300, bool)
        covered[pos] = True
        assert np.array_equal(in_targets(np.arange(300), iv), covered)
    dense = site_intervals(np.arange(1000, 201_000))
    assert np.array_equal(dense, [[1000, 201_000]])


def test_intersection_with_bed(tmp_path):
    bed = tmp_path / "t.bed"
    bed.write_text("chr1\t0\t10\nchr1\t11\t500\nchr2\t0\t10\n")
    t = build_targets(CONTIGS, str(bed), report=None)
    sites = {"chr1": np.array([[9, 12], [499, 500], [999, 1000]]), "chr2": np.array([[49, 50]])}
    _eq(intersect_targets(sites, t), {"chr1": np.array([[9, 10], [11, 12], [499, 500]])})
    _eq(intersect_targets(sites, build_targets(CONTIGS, None, ["chr1"], report=None)), {"chr1": sites["chr1"]})
    assert intersect_targets(sites, {}) == {} and intersect_targets({}, t) == {}


def test_intersection_matches_masks():
    rng = np.random.default_rng(2)
    L = 400
    for _ in range(300):
        a = site_intervals(rng.integers(0, L, rng.integers(0, 150)))
        b = merge_intervals([(int(s), int(s + rng.integers(1, 40))) for s in rng.integers(0, L, rng.integers(0, 10))], L)
        got = intersect_targets({"c": a}, {"c": b})
        want = site_intervals(np.nonzero(in_targets(np.arange(L), a) & in_targets(np.arange(L), b))[0])
        assert np.array_equal(got.get("c", np.zeros((0, 2), np.int64)), want)
