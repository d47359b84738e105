"""GPU s1 and s4 on long-read alignment geometry (tests/test_long_cigars.long_fixture): kilobase D / N, long clips and
insertions, tiles inside one op, deletion- and skip-only tiles, ultra-long reads that make low-depth tiles deep, a read with more
than 65 535 CIGAR ops.

s1 (counts of covered rows, flags, candidates, windows) is bit-exact against the oracle chain: whole contig with 32- and 16-bit
CIGAR words, region shards whose boundaries fall inside long ops (directly and through the host read slicing), target
intervals inside deletion- and skip-only tiles, and the depth cap at 8 / 144 / off.  The CLI over plain and indexed BAMs (the
long read in CG:B,I) writes the oracle's VCF rows.  s4 read matrices with group columns inside long D / N equal the
pysam-emulator restatement.
"""
import os
import re
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

pytestmark = pytest.mark.gpu

CTG = "ctg1"


def _s1(engine, reads, ref, **kw):
    """candidate_windows -> host (pos0, windows, counts, flags)."""
    import torch
    rd = reads.to_torch(engine.device)
    rf = torch.from_numpy(np.ascontiguousarray(ref)).to(engine.device)
    pos, _, x, counts, flags = engine.candidate_windows(rd, rf, **kw)
    torch.cuda.synchronize()
    return pos.cpu().numpy(), x.cpu().numpy(), counts.cpu().numpy(), flags.cpu().numpy()


def _compare(res, pos, x, counts, flags, lo=0, hi=None):
    """Covered bits, count rows of covered positions, zero rows elsewhere, gate bits (test_gpu_deep._compare)."""
    hi = len(res.flags) if hi is None else hi
    exp_flags = res.flags[lo:hi]
    cov = (exp_flags & 1).astype(bool)
    bad = np.nonzero((flags & 1) != (exp_flags & 1))[0]
    assert bad.size == 0, f"covered differs at {bad[:10] + lo}"
    d = np.nonzero((counts[cov] != res.counts[lo:hi][cov]).any(1))[0]
    if d.size:
        p = np.nonzero(cov)[0][d[0]]
        raise AssertionError(f"counts differ at 0-based {p + lo}: gpu {counts[p]} oracle {res.counts[lo + p]} ({d.size} rows)")
    assert (counts[~cov] == 0).all()
    bad = np.nonzero(flags != exp_flags)[0]
    assert bad.size == 0, f"gate differs at {bad[:10] + lo}"


def _params(max_depth):
    from nanosnp_b200 import _lib
    p = _lib.default_params()
    p.max_depth = max_depth
    return p


@pytest.fixture(scope="module")
def engine():
    import torch
    from nanosnp_b200.pipeline import PileupEngine
    assert torch.cuda.is_available()
    return PileupEngine("cuda:0")


@pytest.fixture(scope="module")
def fx():
    from test_long_cigars import long_fixture
    return long_fixture()


@pytest.fixture(scope="module")
def fx16():
    from test_long_cigars import long_fixture
    return long_fixture(cigar16=True)


@pytest.fixture(scope="module")
def oracle_res(fx, fx16, orc, tmp_path_factory):
    """(fixture name, max_depth) -> oracle S1Result, built on first use."""
    d = tmp_path_factory.mktemp("long_oracle")
    cache = {}

    def get(name, max_depth=144):
        key = (name, max_depth)
        if key not in cache:
            ref, rd, _ = fx if name == "fx" else fx16
            mp = str(d / f"{name}_{max_depth}.mpileup")
            orc.mpileup_text(rd, CTG, mp, max_depth=max_depth)
            cache[key] = orc.s1_restate(mp, CTG, ref, pd_path=str(d / f"{name}_{max_depth}.pd"))
        return cache[key]
    return get


# ------------------------------------------------------------------------------------------------ s1
def test_whole_contig_bit_exact(engine, fx, fx16, oracle_res):
    """32-bit CIGAR words; the cigar16 variant as 16- and 32-bit words gives the same bytes; all equal the oracle chain."""
    from nanosnp_b200.reads import cigar16
    ref, rd, _ = fx
    res = oracle_res("fx")
    assert len(res.positions) > 500
    pos, x, counts, flags = _s1(engine, rd, ref)
    _compare(res, pos, x, counts, flags)
    assert np.array_equal(pos + 1, res.positions) and np.array_equal(x, res.windows)
    ref16, rd16, _ = fx16
    res16 = oracle_res("fx16")
    a = _s1(engine, rd16, ref16)
    c16 = cigar16(rd16)
    assert c16.cigar.dtype == np.uint16
    b = _s1(engine, c16, ref16)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)
    _compare(res16, *b)
    assert np.array_equal(b[0] + 1, res16.positions) and np.array_equal(b[1], res16.windows)


SHARDS = (0, 130_000, 244_500, 270_001)          # first base after a 70 kb S; inside a 5 kb N; inside a 20 kb D


def test_region_shards_with_halos(engine, fx, oracle_res):
    """Emit boundaries inside a 20 kb D, inside a 5 kb N and on the first base after a 70 kb S; 16-bp halos.  Run on the whole
    read set and on the host slice (max_reference_span / read_range_for_region): the union equals the whole-contig run."""
    from nanosnp_b200.reads import max_reference_span, slice_reads
    from nanosnp_b200.shard import Region, read_range_for_region
    from test_long_cigars import CONTIG_LEN, read_geometry
    ref, rd, tags = fx
    g = read_geometry(rd)
    res = oracle_res("fx")
    # the boundaries sit where they claim
    d20 = tags.index("D20000"); n5 = tags.index("N5000"); s70 = tags.index("S70000lead")
    sel = lambda r, op, L: (g["rid"] == r) & (g["op"] == op) & (g["ln"] == L)          # noqa: E731
    rs_d, rs_n = int(g["rs"][sel(d20, 2, 20_000)][0]), int(g["rs"][sel(n5, 3, 5000)][0])
    assert rs_d < SHARDS[3] < rs_d + 20_000 and rs_n < SHARDS[2] < rs_n + 5000 and int(rd.pos[s70]) == SHARDS[1]
    span = max_reference_span(rd) + 1
    bounds = list(SHARDS) + [CONTIG_LEN]
    for sliced in (False, True):
        got_pos, got_x = [], []
        for s, e in zip(bounds[:-1], bounds[1:]):
            rg = Region(CTG, 0, CONTIG_LEN, s, e)
            reads = slice_reads(rd, *read_range_for_region(rd.pos, span, rg)) if sliced else rd
            pos, x, counts, flags = _s1(engine, reads, ref, region_start=rg.start, region_len=rg.length, emit_start=s, emit_end=e)
            _compare(res, pos, x, counts, flags, rg.start, rg.end)
            got_pos.append(pos); got_x.append(x)
        assert np.array_equal(np.concatenate(got_pos) + 1, res.positions) and np.array_equal(np.concatenate(got_x), res.windows)


def test_targets_in_deletion_and_skip_only_tiles(engine, fx, oracle_res):
    """One-base intervals inside deletion-only and skip-only tiles, inside tiles that lie within one op, and at tile edges:
    positions equal the oracle's inside the targets, the listed tiles' rows equal the unrestricted run's."""
    import torch
    from nanosnp_b200.shard import Region, listed_tiles
    from nanosnp_b200.targets import in_targets, merge_intervals
    from test_long_cigars import CONTIG_LEN, tile_classes
    ref, rd, _ = fx
    res = oracle_res("fx")
    tc = tile_classes(rd)
    del_only = np.nonzero(tc["dele"] & ~tc["aln"] & ~tc["skip"])[0]
    skip_only = np.nonzero(tc["skip"] & ~tc["aln"] & ~tc["dele"])[0]
    inside = np.nonzero(tc["inside"])[0]
    assert del_only.size and skip_only.size and inside.size
    pts = []
    for t in list(del_only) + list(skip_only) + list(inside[::7]):
        pts += [1024 * t + 511]
    cand = res.positions.astype(np.int64) - 1
    for t in np.unique(np.concatenate([cand[::25] // 1024, inside[::5]])):
        pts += [1024 * int(t) - 1, 1024 * int(t), 1024 * int(t) + 1]                  # tile edges
    pts += list(cand[::9])                                                            # some certain hits
    iv = merge_intervals([(int(p), int(p) + 1) for p in pts if 0 <= p < CONTIG_LEN], CONTIG_LEN)
    rg = Region(CTG, 0, CONTIG_LEN, 0, CONTIG_LEN)
    rf = torch.from_numpy(ref).cuda()
    rdt = rd.to_torch("cuda")
    c_all, f_all = engine.pileup_counts(rdt, rf, 0, CONTIG_LEN)
    c_t, f_t = engine.pileup_counts(rdt, rf, 0, CONTIG_LEN, targets=iv)
    tl = listed_tiles(rg, iv)
    assert np.isin(del_only, tl).all() and np.isin(skip_only, tl).all()
    on = np.zeros(CONTIG_LEN, bool)
    for t in tl:
        on[t * 1024:(t + 1) * 1024] = True
    on_t = torch.from_numpy(on).cuda()
    assert torch.equal(c_t[on_t], c_all[on_t]) and torch.equal(f_t[on_t], f_all[on_t])
    assert int(f_t[~on_t].abs().sum()) == 0
    pos, n_dev = engine.select(f_t, rf, 0, 0, CONTIG_LEN, 65536, targets=iv)
    n = int(n_dev.item())
    engine.check_status()
    x, _, _ = engine.gather(c_t, rf, 0, pos, n_dev, n)
    p = pos[:n].cpu().numpy().astype(np.int64)
    want = cand[in_targets(cand, iv)]
    assert len(want) > 50 and np.array_equal(p, want)
    assert np.array_equal(x[:n].cpu().numpy(), res.windows[np.isin(cand, p)])
    # the deletion- and skip-only rows themselves equal the oracle's
    for t in list(del_only) + list(skip_only):
        sl = slice(1024 * t, 1024 * (t + 1))
        cov = (res.flags[sl] & 1).astype(bool)
        assert cov.all()
        assert np.array_equal(c_t[sl].cpu().numpy()[cov], res.counts[sl][cov])


@pytest.mark.parametrize("max_depth", [8, 144, 0])
def test_depth_cap_with_ultra_long_reads(fx, orc, oracle_res, max_depth):
    """Pool entries that live for 150-350 kb, same-start bursts after them: the GPU drops what orc.depth_cap drops and the
    rows, candidates and windows equal the chain's."""
    from nanosnp_b200.pipeline import PileupEngine
    ref, rd, _ = fx
    dropped = orc.depth_cap(rd, max_depth=max_depth) if max_depth else np.zeros(rd.n_reads, np.uint8)
    if max_depth == 8:
        assert dropped.sum() > 200
    elif max_depth == 144:
        assert dropped.sum() > 20
    res = oracle_res("fx", max_depth)
    eng = PileupEngine("cuda:0", _params(max_depth))
    pos, x, counts, flags = _s1(eng, rd, ref)
    _compare(res, pos, x, counts, flags)
    assert np.array_equal(pos + 1, res.positions) and np.array_equal(x, res.windows)


# ------------------------------------------------------------------------------------------------ end to end
def test_predict_cli_plain_and_indexed_bam(fx, oracle_res, golden_weights, tmp_path):
    """`python -m nanosnp_b200.predict` over a plain and an indexed BAM (the >65 535-op read stored in CG:B,I): the VCF equals the
    oracle chain's windows through the float64 model and the reference record logic."""
    import torch
    from nanosnp_b200 import predict as P
    from nanosnp_b200.bam import bgzf_decompress, write_bam
    from oracle.pyoracle import write_fasta
    from oracle.s2_restate import PileupModelOracle, predict_vcf, vcf_header
    from test_gpu_targets import _compare_vcf
    ref, rd, _ = fx
    res = oracle_res("fx")
    assert np.diff(rd.cigar_off).max() > 65_535
    fa = str(tmp_path / "ref.fa")
    write_fasta(fa, {CTG: ref})
    plain, idx = str(tmp_path / "plain.bam"), str(tmp_path / "idx.bam")
    write_bam(plain, [(CTG, len(ref))], {CTG: rd})
    write_bam(idx, [(CTG, len(ref))], {CTG: rd}, index=True)
    assert b"CGBI" in bgzf_decompress(plain)
    torch.set_num_threads(os.cpu_count() or 1)
    model64 = PileupModelOracle(*golden_weights)
    up = np.char.upper(ref[res.positions - 1].view("S1")).view(np.uint8)
    want = vcf_header(open(fa + ".fai").read().splitlines()) + predict_vcf(model64, CTG, res.positions, up, res.windows)
    cfg = str(Path(P.__file__).parent / "config" / "ont_pileup.yaml")
    outs = []
    for bam, region_len in ((plain, 100_000_000), (idx, 50_000)):
        out = str(tmp_path / (Path(bam).stem + ".vcf"))
        P.main(["-config", cfg, "-model_path", str(ROOT / "tests" / "golden" / "ont_pileup_weights.npz"), "-data", bam,
                "-reference", fa, "-output", out, "--region_len", str(region_len)])
        outs.append(open(out).read())
    assert outs[0] == outs[1]
    assert outs[0].count("\n") > 100
    _compare_vcf(outs[0], want)


# ------------------------------------------------------------------------------------------------ s4 read matrices
def _hap_input(seed=23, L=60_000):
    """A 60 kb contig at ~15x from two haplotypes, het sites every ~250 bp; reads with kilobase D and N over groups of sites,
    10 kb+ soft clips, and two ~50 kb reads.  Records as oracle.pysam_emul.Segment takes them."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    ref = acgt[rng.integers(0, 4, L)].copy()
    sites = np.cumsum(rng.integers(120, 380, L // 120))
    sites = sites[(sites > 300) & (sites < L - 300)]
    alt = (np.searchsorted(acgt, ref[sites]) + rng.integers(1, 4, len(sites))) % 4
    which = rng.integers(0, 2, len(sites))
    haps = [ref.copy(), ref.copy()]
    for h in range(2):
        haps[h][sites[which == h]] = acgt[alt[which == h]]
    vcf = [(CTG, int(p) + 1, chr(ref[p]), chr(acgt[a]), round(float(rng.uniform(5, 60)), 2), "0/1") for p, a in zip(sites, alt)]
    recs = []

    def add(pos, ops, h, flag=0):
        seq, x = [], pos
        for ln, op in ops:
            if op == "M":
                s = haps[h][x:x + ln].copy()
                e = rng.random(ln) < 0.03
                s[e] = acgt[rng.integers(0, 4, int(e.sum()))]
                seq.append(s); x += ln
            elif op in "IS":
                seq.append(acgt[rng.integers(0, 4, ln)])
            elif op in "DN":
                x += ln
        assert x <= L
        seq = np.concatenate(seq).tobytes().decode()
        qual = [(7 * (j // 11) + 3 * len(recs)) % 41 + 1 for j in range(len(seq))]
        hp = h + 1 if rng.random() < 0.7 else None
        recs.append([f"r{len(recs)}", pos, flag | (16 if rng.random() < 0.5 else 0), 60, "".join(f"{a}{b}" for a, b in ops), seq, qual, hp])

    def body(ref_len):
        ops, r = [], 0
        while r < ref_len:
            m = int(min(ref_len - r, rng.integers(3, 30)))
            ops.append((m, "M")); r += m
            if r < ref_len and rng.random() < 0.3:
                if rng.random() < 0.5:
                    d = int(rng.integers(1, 4)); ops.append((d, "D")); r += d
                else:
                    ops.append((int(rng.integers(1, 4)), "I"))
        if ops[-1][1] != "M":
            ops.append((3, "M"))
        return ops
    cov = 0
    while cov < 15 * L:
        span = int(rng.integers(2000, 6000))
        p = int(rng.integers(0, L - span))
        add(p, body(span), int(rng.integers(0, 2)))
        cov += span
    # long D / N over sites: windows and groups inside, or straddling, the op
    for k, p in enumerate(range(3_000, L - 12_000, 4_500)):
        op = "DN"[k % 2]
        ln = [1200, 2500, 4096, 5000][k % 4]
        add(p, body(1500) + [(ln, op)] + body(1500), k % 2)
    for k, p in enumerate(range(5_000, L - 10_000, 9_000)):                           # 10 kb+ soft clips, both ends
        add(p, [(10_000 + 37 * k, "S")] + body(3000), k % 2)
        add(p + 50, body(3000) + [(12_000 + 11 * k, "S")], (k + 1) % 2)
    add(1_000, body(20_000) + [(3000, "D")] + body(26_000), 0)                      # two ~50 kb reads
    add(8_000, body(15_000) + [(2000, "N")] + body(33_000), 1)
    order = sorted(range(len(recs)), key=lambda i: recs[i][1])
    recs = [recs[i] for i in order]
    for i, r in enumerate(recs):
        r[0] = f"r{i}"
    return ref, recs, sorted(vcf, key=lambda v: v[1])


def test_hap_group_matrices_inside_long_ops(tmp_path):
    """HaplotypeModel read matrices for groups whose 11 sites and 33-column windows lie inside or straddle long D / N, reads with
    10 kb+ clips and two ~50 kb reads: equal to the pysam-emulator restatement, from uploaded arrays and through a BAM round
    trip with auxiliary fields."""
    from nanosnp_b200 import hap_groups as hg
    from nanosnp_b200.bam import write_bam
    from oracle import pysam_emul
    from oracle.hap_groups_restate import canonical_rows, subgroup_matrices
    from test_hap_groups import packed
    sys.path.insert(0, str(ROOT / "tests" / "golden"))
    import make_golden_hapgroups as M
    ref, recs, vcf = _hap_input()
    vpath = tmp_path / "p.vcf"; vpath.write_text(M.vcf_text(vcf))
    groups = hg.select_snp_multiprocess(str(vpath), 19, 5, 14, nthreads=1)
    g = groups[CTG]
    # some groups span a long D / N of some read
    long_ops = []
    for r in recs:
        x = r[1]
        for ln, op in re.findall(r"(\d+)([MIDNSH])", r[4]):
            ln = int(ln)
            if op in "DN" and ln >= 1000:
                long_ops.append((x, x + ln))
            if op in "MDN":
                x += ln
    inside = sum(any(a <= gg[0] - 1 and gg[-1] - 1 < b for a, b in long_ops) for gg in g)
    straddle = sum(any(a < gg[5] - 1 - 16 < b or a < gg[5] - 1 + 16 < b for a, b in long_ops) for gg in g)
    assert inside >= 3 and straddle >= 3, (inside, straddle)
    sam = pysam_emul.AlignmentFile(CTG, [pysam_emul.Segment(*r) for r in recs])
    rd, aux = packed(recs)
    assert max(len(r[5]) for r in recs) > 45_000
    bam = str(tmp_path / "h.bam")
    write_bam(bam, [(CTG, len(ref))], {CTG: rd}, aux={CTG: aux})
    subs = hg.plan_subgroups(g)
    want = []
    for a, b in subs:
        want += subgroup_matrices(sam, CTG, g[a:b], 150, 16)
    n_checked = 0
    for al in (hg.upload_alignments(rd, aux), hg.load_contig(bam, CTG)):
        gm = hg.group_matrices(al, g, subs, 150, 16)
        assert [list(p) for p in gm.positions] == [w["positions"] for w in want]
        hap = [h.cpu().numpy() for h in gm.hap]; pile = [p.cpu().numpy() for p in gm.pile]
        for i, w in enumerate(want):
            d = w["hap"][0].shape[0]
            assert gm.depth[i] == d
            if d == 0:
                continue
            for got, exp, centre in (([m[i, :d] for m in hap], w["hap"], 5), ([m[i, :d] for m in pile], w["pile"], 16)):
                for x, y in zip(canonical_rows(*got, centre), canonical_rows(*exp, centre)):
                    np.testing.assert_array_equal(x, y)
            n_checked += 1
    assert n_checked > 80

