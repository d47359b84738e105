"""Stage s1 away from the default parameters, against the oracle chain run with the same values.

Every other s1 test runs with nsnp_default_params (AF 0.12 / 0.12, coverage 6, MAPQ 20, flags 2316, cap 144 or 0).  Here:

  * a hand-built AF-boundary fixture: for every depth 1..300 and a few deeper ones, and every AF threshold used below, columns
    whose top non-reference allele (a SNP, an insertion class or a deletion class) sits one below and exactly at the smallest
    passing count.  Ten (snp_min_af, indel_min_af) sets -- unequal, exact fractions, 0, 1, above 1, NaN -- and six coverage
    limits: counts, flags, candidates and windows bit-exact, the stand-alone regate, region shards, a short candidate buffer;
  * a plain Python statement of the gate (tensor_maker.cpp:195-228, main.cpp:196) decides each fixture column; a CPU test holds
    the oracle to it on every machine;
  * the read filters (min_mapq x excl_flags) on a hand-built read set with every flag bit and on a synthetic contig;
  * the depth cap at limits from 1 to 8000 on a synthetic contig, short deep reads and a pile of same-start bursts.
"""
import math

import numpy as np
import pytest

NAN = float("nan")
# (snp_min_af, indel_min_af)
AF_SETS = [(0.12, 0.12), (0.25, 0.5), (0.5, 0.25), (0.1, 0.3), (1 / 3, 0.2), (0.0, 1.0), (1.0, 0.0), (0.9, 0.9), (1.5, 1.5),
           (NAN, NAN)]
COVERAGES = [0, 1, 6, 7, 33, 1000]
# (snp_min_af, indel_min_af, min_coverage) of every oracle run on the boundary fixture
GATE_SETS = [(s, i, 6) for s, i in AF_SETS] + [(0.12, 0.12, c) for c in COVERAGES if c != 6]
DEPTHS = list(range(1, 301)) + [383, 511, 512, 1000, 2000]
SNP, INS, DEL = 0, 1, 2
READ_LEN = 80
TILE = 1024
MAX_OVERLAP = 16_383                  # reads over one tile (pileup.cu kMaxOverlap)
CAP_STRIDE = 16                       # cap_kernel samples every 16th read (pileup.cu kCapStride)


def _set_id(s):
    return "-".join("nan" if x != x else f"{x:.4g}" for x in s)


def _params(snp=0.12, indel=0.12, min_coverage=6, min_mapq=20, excl_flags=2316, max_depth=144):
    from nanosnp_b200 import _lib
    p = _lib.default_params()
    p.snp_min_af, p.indel_min_af, p.min_coverage = snp, indel, min_coverage
    p.min_mapq, p.excl_flags, p.max_depth = min_mapq, excl_flags, max_depth
    return p


def _engine(**kw):
    import torch
    from nanosnp_b200.pipeline import PileupEngine
    assert torch.cuda.is_available()
    return PileupEngine("cuda:0", params=_params(**kw))


def oracle_chain(orc, reads, ref, path, snp=0.12, indel=0.12, min_coverage=6, min_mapq=20, excl_flags=2316, max_depth=144):
    """mpileup restatement -> s1 restatement with all six parameters."""
    orc.mpileup_text(reads, "ctg1", path, min_mapq=min_mapq, excl_flags=excl_flags, max_depth=max_depth)
    return orc.s1_restate(path, "ctg1", ref, snp_min_af=snp, indel_min_af=indel, min_coverage=min_coverage)


def _gpu_s1(engine, reads, ref, **kw):
    import torch
    rd = reads.to_torch(engine.device)
    rf = torch.from_numpy(np.ascontiguousarray(ref)).to(engine.device)
    pos, refbase, x, counts, flags = engine.candidate_windows(rd, rf, **kw)
    torch.cuda.synchronize()
    return pos.cpu().numpy(), x.cpu().numpy(), counts.cpu().numpy(), flags.cpu().numpy()


def _assert_s1_equal(res, pos, x, counts, flags):
    """Counts and both flag bits at every position, candidate positions and windows: bit for bit."""
    bad = np.nonzero((counts != res.counts).any(1))[0]
    assert bad.size == 0, f"counts differ at 0-based {bad[:5]}: gpu {counts[bad[0]]} oracle {res.counts[bad[0]]} ({bad.size} rows)"
    for bit, name in ((1, "COVERED"), (2, "GATE")):
        bad = np.nonzero((flags & bit) != (res.flags & bit))[0]
        assert bad.size == 0, f"{name} differs at 0-based {bad[:10]} ({bad.size} positions)"
    assert np.array_equal(pos + 1, res.positions), (len(pos), len(res.positions))
    assert np.array_equal(x, res.windows)


# ------------------------------------------------------------------------------------------------ read packing
def pack_reads(pos, flag, mapq, cig, ncig, codes):
    """PackedReads from per-read arrays: cig [n, K] CIGAR words of which the first ncig[i] are used, codes [n, W] bases
    (0..3 = ACGT, 4 = N; W a multiple of 16, one slot per read).  Vectorised: the fixtures below hold millions of reads."""
    from nanosnp_b200.reads import PackedReads
    n, W = codes.shape
    assert W % 16 == 0
    cigar = cig[np.arange(cig.shape[1])[None, :] < ncig[:, None]].astype(np.uint32)
    cigar_off = np.concatenate([[0], np.cumsum(ncig)]).astype(np.int64)
    flat = codes.reshape(-1, 4)
    b = flat & 3
    seq2 = (b[:, 0] | (b[:, 1] << 2) | (b[:, 2] << 4) | (b[:, 3] << 6)).astype(np.uint8)
    nmask = np.packbits(codes.reshape(-1) == 4, bitorder="little")
    pad = np.zeros(16, np.uint8)
    return PackedReads(np.asarray(pos, np.int32), np.asarray(flag, np.uint16), np.asarray(mapq, np.uint8), cigar_off, cigar,
                       np.arange(n, dtype=np.int64) * W, np.concatenate([seq2, pad]), np.concatenate([nmask, pad]))


def _ref_codes(ref):
    lut = np.full(256, 4, np.uint8)
    for k, ch in enumerate(b"ACGT"):
        lut[ch] = k
        lut[ch + 32] = k
    return lut[ref]


# ------------------------------------------------------------------------------------------------ AF-boundary fixture
def min_count(t, d):
    """Smallest count c with c / d >= t in IEEE double (Python float division), or None when no count in 0..d reaches t."""
    if not t <= 1.0:                                         # above 1 or NaN
        return None
    c = max(0, math.floor(t * d) - 1)
    while c > 0 and (c - 1) / d >= t:
        c -= 1
    while c / d < t:
        c += 1
    return c


def thresholds(kind):
    return sorted({(s if kind == SNP else i) for s, i in AF_SETS if not math.isnan(s)})


def boundary_columns():
    """(kind, depth, alt count) of every fixture column: for each kind, depth and threshold t of that kind, the counts c*-1 and
    c* around the smallest passing count c*.  A column without alternative reads is the same for every kind (SNP)."""
    cols = set()
    for kind in (SNP, INS, DEL):
        for d in DEPTHS:
            for t in thresholds(kind):
                c = min_count(t, d)
                if c is None:
                    continue
                for cc in (c - 1, c):
                    if cc >= 0:
                        cols.add((SNP if cc == 0 else kind, d, cc))
    return sorted(cols, key=lambda k: (k[1], k[0], k[2]))


def gate_statement(kind, d, c, ref_code, alt_code, snp, indel, min_coverage):
    """GATE of a fixture column, stated plainly: entries of the pileup dict with a count sorted by count, ties in key order
    A < C < D < G < I < T (std::map order + stable sort); the top entry is not the reference base, or a non-reference SNP /
    indel class reaches its AF; and depth >= min_coverage.  Depth counts A/C/G/T and deletion stars: d at every column."""
    key = {"A": 0, "C": 1, "D": 2, "G": 3, "I": 4, "T": 5}
    ref_key = key["ACGT"[ref_code]]
    tally = {ref_key: d - c if kind == SNP else d}
    alt_key = key["ACGT"[alt_code]] if kind == SNP else key["I"] if kind == INS else key["D"]
    if c > 0:
        tally[alt_key] = c
    entries = sorted((k for k in tally if tally[k] > 0), key=lambda k: (-tally[k], k))
    top_other = bool(entries) and entries[0] != ref_key
    af = snp if kind == SNP else indel
    af_pass = c > 0 and c / d >= af
    return (top_other or af_pass) and d >= min_coverage


class BoundaryFixture:
    def __init__(self, seed=2024):
        rng = np.random.default_rng(seed)
        cols = boundary_columns()
        self.kind = np.array([k for k, _, _ in cols], np.int64)
        self.depth = np.array([d for _, d, _ in cols], np.int64)
        self.count = np.array([c for _, _, c in cols], np.int64)
        spacing = np.where(self.depth >= 1500, 256, 128)     # under 16 383 reads over any 1 024-bp tile
        self.col = (200 + np.concatenate([[0], np.cumsum(spacing[:-1])])).astype(np.int64)
        L = int(self.col[-1]) + 200
        self.ref = np.frombuffer(bytes(rng.choice(list(b"ACGT"), L).astype(np.uint8)), np.uint8).copy()
        rc = _ref_codes(self.ref)
        self.ref_code = rc[self.col].astype(np.int64)
        self.alt_code = (self.ref_code + rng.integers(1, 4, len(cols))) % 4            # SNP columns
        self.indel_len = rng.integers(1, 4, len(cols))                                   # indel columns: 1..3 bp
        ins_seqs = rng.integers(0, 4, (len(cols), 2, 3))                                 # two insertion sequences per column

        # one row per read
        ci = np.repeat(np.arange(len(cols)), self.depth)
        j = np.arange(len(ci)) - np.repeat(np.cumsum(self.depth) - self.depth, self.depth)   # index inside the column
        X = self.col[ci]
        start = X - 40 + (j * 5) % 8                       # the column is base 33..40 of an 80-bp reference span
        kind = np.where(j < self.count[ci], self.kind[ci], -1)   # the first c reads of a column carry its allele
        k = self.indel_len[ci]
        a = X - start + 1                                   # aligned bases up to and including the column
        ins, dele = kind == INS, kind == DEL
        n = len(ci)
        order = np.argsort(start, kind="stable")
        W = 96
        codes = np.empty((n, W), np.uint8)
        m = np.arange(W, dtype=np.int32)[None, :]
        for lo in range(0, n, 1 << 18):                     # query base m -> reference base or inserted base, in slices
            o = order[lo:lo + (1 << 18)]
            ko, ao, so = k[o][:, None].astype(np.int32), a[o][:, None].astype(np.int32), start[o][:, None]
            io, do = ins[o][:, None], dele[o][:, None]
            src = m + np.where(io & (m >= ao), -ko, 0) + np.where(do & (m >= ao), ko, 0)
            cd = rc[np.minimum(so + src, L - 1)]
            in_ins = io & (m >= ao) & (m < ao + ko)
            iv = ins_seqs[ci[o][:, None], (j[o] % 2)[:, None], np.clip(m - ao, 0, 2)].astype(np.uint8)
            cd = np.where(in_ins, iv, cd)
            sn = np.nonzero(kind[o] == SNP)[0]
            cd[sn, (X - start)[o][sn]] = self.alt_code[ci[o][sn]]
            qlen = READ_LEN + np.where(io, ko, 0) - np.where(do, ko, 0)
            codes[lo:lo + len(o)] = np.where(m < qlen, cd, 0)
        cig = np.zeros((n, 3), np.uint32)
        ncig = np.where(ins | dele, 3, 1)
        cig[:, 0] = np.where(ins | dele, a, READ_LEN) << 4
        cig[:, 1] = (k << 4) | np.where(ins, 1, 2)
        cig[:, 2] = np.where(ins, READ_LEN - a, READ_LEN - a - k) << 4
        flag = 16 * (j % 2)
        self.reads = pack_reads(start[order], flag[order], np.full(n, 60), cig[order], ncig[order], codes)
        self.n_reads = n
        # reads over each 1 024-bp tile
        t0, t1 = start // TILE, (start + READ_LEN - 1) // TILE
        self.tile_overlap = np.bincount(t0, minlength=L // TILE + 1) + np.bincount(t1[t1 != t0], minlength=L // TILE + 1)

    def expected_gate(self, snp, indel, min_coverage):
        return np.array([gate_statement(k, d, c, r, a, snp, indel, min_coverage) for k, d, c, r, a in
                         zip(self.kind, self.depth, self.count, self.ref_code, self.alt_code)], bool)


@pytest.fixture(scope="module")
def boundary(orc, tmp_path_factory):
    """The fixture, its mpileup text (cap off) and the oracle's flags / positions per parameter set, computed once.  The count
    rows do not depend on the AF / coverage parameters: they are kept once."""
    fx = BoundaryFixture()
    mp = str(tmp_path_factory.mktemp("boundary") / "ctg1.mpileup")
    orc.mpileup_text(fx.reads, "ctg1", mp, max_depth=0)
    fx.oracle_counts = None
    cache = {}

    def get(s):
        if s not in cache:
            res = orc.s1_restate(mp, "ctg1", fx.ref, snp_min_af=s[0], indel_min_af=s[1], min_coverage=s[2], want_windows=False)
            if fx.oracle_counts is None:
                fx.oracle_counts = res.counts
            else:
                assert np.array_equal(res.counts, fx.oracle_counts)
            cache[s] = (res.flags, res.positions)
        return cache[s]
    fx.oracle = get
    return fx


def _oracle_result(fx, s):
    """S1Result-like view of the cached oracle run: windows are rows of the count array (test_oracle_pinning)."""
    from oracle.pyoracle import S1Result
    flags, positions = fx.oracle(s)
    c = positions.astype(np.int64) - 1
    win = fx.oracle_counts[c[:, None] + np.arange(-16, 17)[None, :]] if len(c) else np.zeros((0, 33, 18), np.int32)
    return S1Result(positions, win, None, fx.oracle_counts, flags)


# ------------------------------------------------------------------------------------------------ CPU: the oracle's gate
def test_boundary_fixture_shape(boundary):
    """Both sides of every boundary exist for every threshold in (0, 1] and every kind, including the depths 255 / 256 / 257
    where the 1/3 threshold steps from 85 to 86 (the seam of the kernel's table and its divide); no tile is over its read limit."""
    fx = boundary
    have = set(zip(fx.kind.tolist(), fx.depth.tolist(), fx.count.tolist()))
    for kind in (SNP, INS, DEL):
        for t in thresholds(kind):
            if not 0.0 < t <= 1.0:
                continue
            below = above = 0
            for d in DEPTHS:
                c = min_count(t, d)
                below += (SNP if c - 1 == 0 else kind, d, c - 1) in have
                above += (kind, d, c) in have
            assert below == len(DEPTHS) and above == len(DEPTHS), (kind, t, below, above)
    assert min_count(1 / 3, 255) == 85 and min_count(1 / 3, 256) == 86 and min_count(1 / 3, 257) == 86
    assert fx.tile_overlap.max() < MAX_OVERLAP
    assert (fx.tile_overlap > 255).any() and (fx.tile_overlap[fx.tile_overlap > 0] <= 255).any()    # deep and shallow tiles


@pytest.mark.parametrize("s", GATE_SETS, ids=_set_id)
def test_oracle_gate_matches_plain_statement(boundary, s):
    """The oracle's GATE bit equals the plain statement at every fixture column, and is clear everywhere else; the columns of
    each kind and threshold fall on both sides of it."""
    fx = boundary
    flags, positions = fx.oracle(s)
    want = fx.expected_gate(*s)
    got = (flags[fx.col] & 2) != 0
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, [(int(fx.kind[i]), int(fx.depth[i]), int(fx.count[i]), bool(got[i])) for i in bad[:10]]
    others = np.ones(len(flags), bool)
    others[fx.col] = False
    assert not (flags[others] & 2).any()
    assert np.array_equal(positions - 1, fx.col[want])              # every gated column is also a candidate (33 rows covered)
    # both sides of the boundary are present wherever the thresholds make one
    for kind, t in ((SNP, s[0]), (INS, s[1]), (DEL, s[1])):
        if not 0.0 < t <= 1.0:
            continue
        sel = fx.kind == kind
        af = fx.count[sel] / fx.depth[sel]
        assert (af >= t).any() and (af < t).any()


# ------------------------------------------------------------------------------------------------ GPU: AF and coverage
@pytest.fixture(scope="module")
def boundary_dev(boundary):
    import torch
    return boundary.reads.to_torch("cuda:0"), torch.from_numpy(boundary.ref).to("cuda:0")


def _gpu_s1_dev(engine, rd, rf, **kw):
    import torch
    pos, refbase, x, counts, flags = engine.candidate_windows(rd, rf, **kw)
    torch.cuda.synchronize()
    return pos.cpu().numpy(), x.cpu().numpy(), counts.cpu().numpy(), flags.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("s", GATE_SETS, ids=_set_id)
def test_boundary_bit_exact(boundary, boundary_dev, s):
    """Counts, both flag bits, candidates and windows equal the oracle for every AF / coverage set; the stand-alone select with
    recompute_gate rebuilds the fused epilogue's GATE bits and positions from the count rows alone."""
    import torch
    fx = boundary
    rd, rf = boundary_dev
    eng = _engine(snp=s[0], indel=s[1], min_coverage=s[2], max_depth=0)
    res = _oracle_result(fx, s)
    _assert_s1_equal(res, *_gpu_s1_dev(eng, rd, rf))
    counts, flags = eng.pileup_counts(rd, rf)
    flags2 = flags & 1
    L = len(fx.ref)
    pos, n_dev = eng.select(flags2, rf, 0, 0, L, L, counts=counts, recompute_gate=True)
    n = int(n_dev.item())
    eng.check_status()
    assert np.array_equal(pos[:n].cpu().numpy() + 1, res.positions)
    assert torch.equal(flags2, flags)


@pytest.mark.gpu
def test_boundary_shards_non_default(boundary, boundary_dev):
    """Three region shards with 16-bp halos at (snp 0.25, indel 0.5, coverage 7) give the oracle's candidates (cap off, so the
    halo caveat of the depth cap does not apply)."""
    fx = boundary
    rd, rf = boundary_dev
    s = (0.25, 0.5, 7)
    eng = _engine(snp=s[0], indel=s[1], min_coverage=s[2], max_depth=0)
    res = _oracle_result(fx, s)
    L = len(fx.ref)
    cuts = [0, L // 3 + 5, 2 * L // 3 - 11, L]
    got = []
    for s0, e0 in zip(cuts[:-1], cuts[1:]):
        rs, re_ = max(0, s0 - 16), min(L, e0 + 16)
        pos, x, counts, flags = _gpu_s1_dev(eng, rd, rf, region_start=rs, region_len=re_ - rs, emit_start=s0, emit_end=e0)
        assert np.array_equal(counts, res.counts[rs:re_]) and np.array_equal(flags, res.flags[rs:re_])
        sel = (res.positions - 1 >= s0) & (res.positions - 1 < e0)
        assert np.array_equal(x, res.windows[sel])
        got.append(pos)
    assert np.array_equal(np.concatenate(got) + 1, res.positions)


@pytest.mark.gpu
def test_select_capacity_overflow(boundary, boundary_dev):
    """A candidate buffer shorter than the site count: n_dev holds the full count, the first `capacity` positions are the
    oracle's, the status reports NSNP_E_OVERFLOW once, and the next call on the engine succeeds.  f32 windows are the int32
    windows cast."""
    import torch
    from nanosnp_b200 import _lib
    fx = boundary
    rd, rf = boundary_dev
    eng = _engine(max_depth=0)
    res = _oracle_result(fx, (0.12, 0.12, 6))
    counts, flags = eng.pileup_counts(rd, rf)
    L = len(fx.ref)
    n = len(res.positions)
    assert n > 100
    for cap in (0, 1, n // 2, n - 1):
        pos, n_dev = eng.select(flags, rf, 0, 0, L, cap)
        assert int(n_dev.item()) == n
        assert np.array_equal(pos[:cap].cpu().numpy() + 1, res.positions[:cap])
        with pytest.raises(_lib.NsnpError) as e:
            eng.check_status()
        assert e.value.code == _lib.E_OVERFLOW
        pos, n_dev = eng.select(flags, rf, 0, 0, L, n)
        eng.check_status()
        assert int(n_dev.item()) == n and np.array_equal(pos.cpu().numpy() + 1, res.positions)
    x32, xf, refbase = eng.gather(counts, rf, 0, pos, n_dev, n, want_f32=True)
    torch.cuda.synchronize()
    assert torch.equal(xf, x32.float())
    assert np.array_equal(x32.cpu().numpy(), res.windows)


# ------------------------------------------------------------------------------------------------ GPU: coverage on a contig
@pytest.mark.gpu
@pytest.mark.parametrize("min_coverage", COVERAGES)
def test_min_coverage_synthetic(orc, tmp_path, min_coverage):
    from nanosnp_b200.synth import SynthConfig, generate_host
    cfg = SynthConfig(contig_len=120_000, coverage=30.0, seed_ref=71, seed_var=72, seed_reads=73, len_median=3000, len_min=200)
    ref, reads = generate_host(cfg)
    res = oracle_chain(orc, reads, ref, str(tmp_path / "c.mpileup"), min_coverage=min_coverage)
    _assert_s1_equal(res, *_gpu_s1(_engine(min_coverage=min_coverage), reads, ref))
    if min_coverage == 1000:
        assert len(res.positions) == 0
    elif min_coverage <= 7:
        assert len(res.positions) > 100


# ------------------------------------------------------------------------------------------------ GPU: read filters
MAPQS = [0, 1, 19, 20, 21, 59, 60, 255]
MIN_MAPQS = [0, 1, 20, 21, 60, 255]
EXCL_FLAGS = [0, 4, 256, 1796, 2316, 3844, 0xFFFF]


def filter_reads(seed=31):
    """Every single flag bit (0..15) at every MAPQ of MAPQS, plus plain reads so that every position stays covered: each read
    carries its own mismatches and indels, so dropping any one of them changes some count row."""
    from nanosnp_b200.reads import from_records
    rng = np.random.default_rng(seed)
    L = 3000
    ref = np.frombuffer(bytes(rng.choice(list(b"ACGT"), L).astype(np.uint8)), np.uint8).copy()
    specs = [(1 << b, q) for b in range(16) for q in MAPQS] + [(16 * (i % 2), 60) for i in range(60)]
    recs = []
    for f, q in specs:
        p = int(rng.integers(0, L - 500))
        parts, seq, r = [], [], p
        for _ in range(3):
            mlen = int(rng.integers(40, 100))
            s = bytearray(ref[r:r + mlen])
            for k in rng.choice(mlen, 3, replace=False):
                s[k] = b"ACGT"[(b"ACGT".index(s[k]) + int(rng.integers(1, 4))) % 4]
            parts.append(f"{mlen}M"); seq.append(s.decode()); r += mlen
            il = int(rng.integers(1, 4))
            if rng.random() < 0.5:
                parts.append(f"{il}I"); seq.append("".join("ACGT"[v] for v in rng.integers(0, 4, il)))
            else:
                parts.append(f"{il}D"); r += il
        mlen = int(rng.integers(40, 100))
        parts.append(f"{mlen}M"); seq.append(ref[r:r + mlen].tobytes().decode())
        recs.append((p, f, q, "".join(parts), "".join(seq)))
    recs.sort(key=lambda t: t[0])
    return ref, from_records(recs)


@pytest.fixture(scope="module")
def filter_inputs():
    from nanosnp_b200.synth import SynthConfig, generate_host
    hand = filter_reads()
    cfg = SynthConfig(contig_len=60_000, coverage=25.0, seed_ref=81, seed_var=82, seed_reads=83, len_median=3000, len_min=200,
                      lowmapq_frac=0.15, secondary_frac=0.08, supp_frac=0.08)
    ref, reads = generate_host(cfg)
    mq = reads.mapq.copy()                                   # MAPQs at and around every limit of the grid
    for k, v in enumerate((1, 20, 21, 59, 255)):
        mq[k::11] = v
    reads.mapq = mq
    return {"hand": hand, "synthetic": (ref, reads)}


@pytest.mark.gpu
@pytest.mark.parametrize("excl_flags", EXCL_FLAGS)
@pytest.mark.parametrize("min_mapq", MIN_MAPQS)
@pytest.mark.parametrize("name", ["hand", "synthetic"])
def test_read_filters(orc, tmp_path, filter_inputs, name, min_mapq, excl_flags):
    """min_mapq x excl_flags against the oracle given the same values (cap off on the hand-built set, 144 on the contig).
    Unmapped reads (flag 4) are dropped whatever excl_flags says."""
    ref, reads = filter_inputs[name]
    md = 0 if name == "hand" else 144
    res = oracle_chain(orc, reads, ref, str(tmp_path / "f.mpileup"), min_mapq=min_mapq, excl_flags=excl_flags, max_depth=md)
    _assert_s1_equal(res, *_gpu_s1(_engine(min_mapq=min_mapq, excl_flags=excl_flags, max_depth=md), reads, ref))


# ------------------------------------------------------------------------------------------------ GPU: depth cap
CAP_GRID = [1, 2, 3, 17, 18, 19, 20, 50, 143, 144, 145, 1000, 8000]


def burst_pile(seed=41):
    """Bursts of reads sharing a start position, burst sizes 1..300 in shuffled order, 37 bp apart; reads of 80, 120 or 160 bp,
    both strands, every 13th read below MAPQ 20.  Reads are prepended (far from the bursts) until the read with the largest
    pool -- earlier passing reads whose end reaches its start -- has an index that is not a multiple of 16, so the sampled bound
    of cap_kernel does not see the maximum.  Returns (ref, reads, pool size per read)."""
    import bisect
    rng = np.random.default_rng(seed)
    sizes = rng.permutation(np.arange(1, 301))
    starts = np.repeat(1000 + 37 * np.arange(len(sizes)), sizes)
    lens = 80 + 40 * (np.arange(len(starts)) % 3)
    L = int(starts[-1] + 400)
    ref = np.frombuffer(bytes(rng.choice(list(b"ACGT"), L).astype(np.uint8)), np.uint8).copy()
    for lead in range(CAP_STRIDE):
        p = np.concatenate([np.arange(lead) * 5, starts]).astype(np.int64)
        ln = np.concatenate([np.full(lead, 60), lens]).astype(np.int64)
        mapq = np.full(len(p), 60)
        mapq[lead::13] = 10
        ends, pool = [], np.zeros(len(p), np.int64)      # pool[i]: earlier passing reads with exclusive end >= p[i]
        for i in range(len(p)):
            pool[i] = len(ends) - bisect.bisect_left(ends, p[i])
            if mapq[i] >= 20:
                bisect.insort(ends, p[i] + ln[i])
        passing = np.where(mapq >= 20, pool, -1)
        imax = int(np.argmax(passing))
        if imax % CAP_STRIDE and pool[::CAP_STRIDE].max() < pool[imax] and (passing == pool[imax]).sum() == 1:
            pool = passing
            break
    else:
        raise AssertionError("no lead-in puts the largest pool off the sampled reads")
    rc = _ref_codes(ref)
    n = len(p)
    W = 176
    codes = rc[np.minimum(p[:, None] + np.arange(W)[None, :], L - 1)]
    snp = rng.random((n, W)) < 0.03                             # a few substitutions, so that dropped reads change counts
    codes = np.where(snp, (codes + rng.integers(1, 4, (n, W))) % 4, codes)
    codes = np.where(np.arange(W)[None, :] < ln[:, None], codes, 0).astype(np.uint8)
    cig = (ln << 4).astype(np.uint32)[:, None]
    reads = pack_reads(p, 16 * (np.arange(n) % 2), mapq, cig, np.ones(n, np.int64), codes)
    return ref, reads, pool


@pytest.fixture(scope="module")
def cap_inputs():
    from nanosnp_b200.synth import SynthConfig, generate_host
    out = {"synthetic": generate_host(SynthConfig(contig_len=200_000, coverage=30.0, seed_ref=91, seed_var=92, seed_reads=93)),
           "deep_short_reads": generate_host(SynthConfig(contig_len=30_000, coverage=100.0, len_median=600, len_min=100, len_sigma=0.4,
                                                         seed_ref=7, seed_var=8, seed_reads=9))}
    ref, reads, pool = burst_pile()
    out["bursts"] = (ref, reads)
    out["bursts_pool"] = pool
    return out


def _cap_case(orc, tmp_path, ref, reads, md):
    res = oracle_chain(orc, reads, ref, str(tmp_path / "cap.mpileup"), max_depth=md)
    _assert_s1_equal(res, *_gpu_s1(_engine(max_depth=md), reads, ref))
    return orc.depth_cap(reads, max_depth=md)


@pytest.mark.gpu
@pytest.mark.parametrize("md", CAP_GRID)
@pytest.mark.parametrize("name", ["synthetic", "deep_short_reads", "bursts"])
def test_depth_cap_grid(orc, tmp_path, cap_inputs, name, md):
    """Counts, flags, candidates and windows bit-exact against the oracle chain with the same --max-depth.  The inputs with
    reads that share start positions lose reads at the small limits, so the one-thread replay of cap_kernel runs."""
    ref, reads = cap_inputs[name]
    dropped = _cap_case(orc, tmp_path, ref, reads, md)
    if (name == "deep_short_reads" and md <= 20) or (name == "bursts" and md <= 145):
        assert dropped.sum() > 0
    if md >= 8000:
        assert dropped.sum() == 0


@pytest.mark.gpu
def test_depth_cap_between_sampled_reads(orc, tmp_path, cap_inputs):
    """The pile's largest pool falls between two sampled reads.  At a limit of (largest pool + 1) exactly that one read is
    dropped, although the pool of every sampled read is smaller; one more and nothing is dropped."""
    ref, reads = cap_inputs["bursts"]
    pool = cap_inputs["bursts_pool"]
    top = int(pool.max())
    assert int(np.argmax(pool)) % CAP_STRIDE != 0 and pool[::CAP_STRIDE].max() < top
    dropped = _cap_case(orc, tmp_path, ref, reads, top + 1)
    assert np.array_equal(np.nonzero(dropped)[0], [int(np.argmax(pool))])
    assert _cap_case(orc, tmp_path, ref, reads, top + 2).sum() == 0
