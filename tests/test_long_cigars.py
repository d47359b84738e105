"""Long-read alignment geometry: kilobase deletions and reference skips, long soft clips and insertions, ultra-long reads.

The seeded fixture built here (`long_fixture`) puts every long-op path of the s1 kernels to work: ops on both sides of the
packed 16-bit prefix-scan switch (1024 for the two-ops-per-lane walk, 2048 for a one-op-per-lane walk), ops longer than a tile,
tiles that lie wholly inside one read's D or N, a stretch covered only by deletions and skips, ultra-long reads whose index
range makes ordinary low-depth tiles deep, and one read with more than 65 535 CIGAR ops (stored in CG:B,I in a BAM).

CPU: the fixture holds what it claims (path choices decided from the CIGARs on the host); a plain NumPy statement of the
long-op semantics (interval arithmetic over each read's ops) equals the oracle's count rows; and, where the reference's
own tools are built, the oracle equals them on a slice of the fixture.  tests/test_gpu_long_cigars.py runs the GPU side.
"""
import numpy as np
import pytest

CONTIG_LEN = 409_600                                  # 400 tiles of 1024
GAP = (360_448, 380_928)                              # no background reads: covered only by a few reads' D and N
THRESH_DN = (61, 1023, 1024, 1025, 2047, 2048, 2049, 4095, 4096, 5000, 20_000, 70_000)
THRESH_S = (1023, 1024, 4095, 4096, 65_535, 65_536, 100_000)
THRESH_I = (61, 1024, 4096, 70_000)
THRESH_M = (1024, 4096, 70_000)
TILE = 1024
KREADLIST = 1024                                      # pileup.cu kReadList: more candidate reads than this -> deep tile
REF_OPS, QRY_OPS, ALN_OPS = (0, 2, 3, 7, 8), (0, 1, 4, 7, 8), (0, 7, 8)
PASS_EXCL, PASS_MAPQ = 2316, 20


# ------------------------------------------------------------------------------------------------ fixture
class _Builder:
    def __init__(self, ref, rng, max_op):
        self.ref, self.rng, self.max_op = ref, rng, max_op
        self.recs, self.tags = [], []

    def seq_for(self, pos, ops):
        """Read bases: the reference under M (3 % substitutions), random bases under I and S."""
        op = np.array([o for _, o in ops]); ln = np.array([x for x, _ in ops], np.int64)
        rl = np.where(np.isin(op, list("MDN")), ln, 0)
        rs = pos + np.cumsum(rl) - rl
        ql = np.where(np.isin(op, list("MIS")), ln, 0)
        oid = np.repeat(np.arange(len(ops)), ql)
        within = np.arange(int(ql.sum())) - np.repeat(np.cumsum(ql) - ql, ql)
        acgt = np.frombuffer(b"ACGT", np.uint8)
        seq = acgt[self.rng.integers(0, 4, len(oid))]
        m = (op[oid] == "M") & (self.rng.random(len(oid)) >= 0.03)
        seq[m] = self.ref[rs[oid[m]] + within[m]]
        return seq.tobytes().decode()

    def add(self, pos, ops, tag=None, strand=None, flag=0, mapq=60):
        """ops: [(length, op)]; reads with an op of max_op or longer are left out (the cigar16 variant)."""
        if any(ln >= self.max_op for ln, _ in ops):
            return False
        assert all(ln > 0 for ln, _ in ops) and pos >= 0
        span = sum(ln for ln, op in ops if op in "MDN")
        assert pos + span <= len(self.ref), (tag, pos, span)
        strand = int(self.rng.integers(0, 2)) if strand is None else strand
        self.recs.append((pos, flag | 16 * strand, mapq, "".join(f"{ln}{op}" for ln, op in ops), self.seq_for(pos, ops)))
        self.tags.append(tag)
        return True


def _short_ops(rng, ref_len):
    """ONT-like alignment body of about ref_len reference bases: short M runs between 1- to 6-base I / D."""
    n = ref_len // 8 + 16
    m, u = rng.integers(3, 30, n).tolist(), rng.random(n).tolist()
    d, i = rng.choice([1, 1, 2, 3, 6], n).tolist(), rng.choice([1, 1, 2, 4], n).tolist()
    ops, r, k = [], 0, 0
    while r < ref_len:
        if k == n:
            return ops + _short_ops(rng, ref_len - r)
        mm = min(ref_len - r, m[k])
        ops.append((mm, "M")); r += mm
        if r >= ref_len:
            break
        if u[k] < 0.3:
            ops.append((d[k], "D")); r += d[k]
        elif u[k] < 0.6:
            ops.append((i[k], "I"))
        k += 1
    if ops[-1][1] != "M":
        ops.append((5, "M"))
    return ops


def _merge(ops):
    out = []
    for ln, op in ops:
        if out and out[-1][1] == op:
            out[-1] = (out[-1][0] + ln, op)
        else:
            out.append((ln, op))
    return out


def long_fixture(cigar16=False, seed=2024):
    """(ref uint8[CONTIG_LEN], PackedReads, tags) -- tags[i] names the feature read i carries (None: background).
    cigar16=True drops every read with an op of 4096 or longer (the 1024-4095 ops stay), so the reads fit 16-bit CIGAR words."""
    from nanosnp_b200.reads import from_records
    rng = np.random.default_rng(seed)
    ref = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, CONTIG_LEN)].copy()
    b = _Builder(ref, rng, 4096 if cigar16 else 1 << 28)
    M = lambda n: (n, "M")                                                                # noqa: E731
    # background: ~20x, 3-20 kb (median 5 kb), none touching the gap
    cov = 0
    while cov < 20 * CONTIG_LEN:
        span = int(np.clip(np.exp(rng.normal(np.log(5000), 0.5)), 3000, 20_000))
        p = int(rng.integers(0, CONTIG_LEN - span))
        if p < GAP[1] and p + span > GAP[0]:
            continue
        ops = _short_ops(rng, span)
        if rng.random() < 0.2:
            ops = [(int(rng.integers(5, 300)), "S")] + ops
        if rng.random() < 0.2:
            ops = ops + [(int(rng.integers(5, 300)), "S")]
        u = rng.random()
        b.add(p, ops, flag=256 if u < 0.02 else 1024 if u < 0.04 else 0, mapq=5 if 0.04 <= u < 0.07 else 60)
        cov += span
    # threshold lengths of D and N, between two 2 kb bodies
    for i, L in enumerate(THRESH_DN):
        for j, op in enumerate("DN"):
            p = 150_000 + 10_000 * j if L == 70_000 else 20_000 + 24_000 * i + 4_000 * j
            b.add(p, [M(2000), (L, op), M(2000)], tag=f"{op}{L}")
    # soft clips at both ends, with and without hard clips outside
    for i, L in enumerate(THRESH_S):
        p = 15_000 + 9_000 * i
        b.add(p, [(L, "S")] + _short_ops(rng, 3000), tag=f"S{L}lead")
        b.add(p + 100, _short_ops(rng, 3000) + [(L, "S")], tag=f"S{L}trail")
        b.add(p + 200, [(7, "H"), (L, "S")] + _short_ops(rng, 3000) + [(L, "S"), (9, "H")], tag=f"S{L}both_H")
    b.add(130_000, [(70_000, "S")] + _short_ops(rng, 4000), tag="S70000lead")          # a shard boundary sits on its first base
    # long insertions and long aligned runs
    for i, L in enumerate(THRESH_I):
        b.add(40_000 + 50_000 * i, [M(2000), (L, "I"), M(2000)], tag=f"I{L}")
    for i, L in enumerate(THRESH_M):
        b.add(45_000 + 90_000 * i, _short_ops(rng, 500) + [(2, "D"), M(L), (1, "I")] + _short_ops(rng, 500), tag=f"M{L}")
    # long D / N exactly on, and one base either side of, tile edges of 1024 and 2048: tiles wholly inside one op
    k = 0
    for op in "DN":
        for A in (1024, 2048):
            for ds in (-1, 0, 1):
                for de in (-1, 0, 1):
                    s = A * ((8_000 + 9_500 * k) // A) + ds
                    e = s - ds + 3 * A + de
                    b.add(s - 1500, [M(1500), (e - s, op), M(1500)], tag=f"edge{op}{A}{ds:+d}{de:+d}")
                    k += 1
    # adjacency
    b.add(300_000, [M(1000), (500, "D"), (700, "N"), M(1000)], tag="MDNM")
    b.add(301_000, [M(1000), (700, "N"), (500, "D"), M(1000)], tag="MNDM")
    b.add(302_000, [M(1000), (30, "I"), (2000, "N"), M(1000)], tag="MINM")
    b.add(305_000, [(200, "S"), (1300, "D")] + _short_ops(rng, 2000), tag="SD")
    b.add(306_000, _short_ops(rng, 2000) + [(1500, "N"), (300, "S")], tag="NS")
    # chunk geometry: long ops at op index 0, 31, 32, 63, 64 (slot 0 / slot 1 of a lane of the 64-op walk)
    ops = [(int(x), "M") if i % 2 == 0 else (1, "ID"[i % 4 == 1]) for i, x in enumerate(rng.integers(3, 20, 89))]
    ops[0], ops[31], ops[32], ops[63], ops[64] = M(1500), (1500, "D"), M(1200), (2500, "N"), M(1030)
    b.add(310_000, ops, tag="chunkpos")
    # one 64-op chunk at the packed-scan limit (all ops 1000-1023: the 64 reference lengths sum just below 65 536) ...
    lens = np.full(64, 1023); lens[rng.choice(64, 3, replace=False)] = 1000
    b.add(2_000, [(int(x), "MDMN"[i % 4]) for i, x in enumerate(lens)] + [M(100)], tag="packed_limit")
    # ... and one whose ops are all 1024-4095 and sum past 65 536
    lens = rng.integers(1024, 1100, 64)
    b.add(232_000, [(int(x), "MDMN"[i % 4]) for i, x in enumerate(lens)] + [M(100)], tag="unpacked_chunk")
    # the gap: a few reads whose D and N (and one another's M) cover it
    b.add(357_000, [M(3448), (12_288, "D"), (10_000, "N"), M(1000)], tag="gap_MDNM")          # D tile-exact, then N
    b.add(355_000, [M(5000), (3000, "N"), (2000, "D"), M(1500)], tag="gap_MNDM", strand=1)
    b.add(378_000, [M(1500), (4000, "N"), M(1500)], tag="gap_N", strand=0)
    b.add(359_000, [(80, "S"), M(800), (2000, "D"), (20, "I"), (7000, "N"), (150, "S")], tag="gap_MDINS", strand=1)
    # ultra-long reads: 150-350 kb spans; the first has more than 65 535 ops and query bases
    many = []
    while len(many) < 70_000:
        many += [(int(rng.integers(1, 8)), "M"), (int(rng.integers(1, 3)), "ID"[len(many) % 4 == 2])]
    many = _merge(many + [M(10)])
    assert 2 * sum(ln for ln, op in many if op in "MD") < 350_000
    ul = [(4_000, _merge(many + [M(2000)] + _short_ops(rng, 350_000 - sum(ln for ln, op in many if op in "MD") - 2000)))]
    for p, span in ((11_000, 300_000), (20_000, 150_000), (37_000, 220_000), (55_000, 250_000)):
        ul.append((p, [M(3000), (2500, "N")] + _short_ops(rng, span - 5500)))
    for i, (p, ops) in enumerate(ul):
        b.add(p, ops, tag=f"ultra{i}")
    # same-start bursts of short reads after them: long-lived entries in the depth cap's pool
    for j, (p, n) in enumerate(((80_000, 40), (150_000, 12), (150_001, 12), (200_000, 170), (240_500, 60))):
        for _ in range(n):
            b.add(p, _short_ops(rng, int(rng.integers(300, 900))), tag=f"burst{j}")
    order = sorted(range(len(b.recs)), key=lambda i: b.recs[i][0])
    return ref, from_records([b.recs[i] for i in order]), [b.tags[i] for i in order]


# ------------------------------------------------------------------------------------------------ host-side geometry
def read_geometry(reads):
    """Per op: read id, op, length, reference start; per read: end (exclusive), passing filter bit."""
    cig = reads.cigar.astype(np.int64)
    op, ln = cig & 15, cig >> 4
    n = reads.n_reads
    rid = np.repeat(np.arange(n), np.diff(reads.cigar_off))
    rl = np.where(np.isin(op, REF_OPS), ln, 0)
    cum = np.cumsum(rl) - rl
    rs = reads.pos[rid].astype(np.int64) + cum - cum[reads.cigar_off[:-1]][rid]
    rend = reads.pos.astype(np.int64).copy()
    np.add.at(rend, rid, rl)
    passing = ((reads.flag & 4) == 0) & ((reads.flag & PASS_EXCL) == 0) & (reads.mapq >= PASS_MAPQ)
    return dict(rid=rid, op=op, ln=ln, rs=rs, rend=rend, passing=passing)


def window_scans(reads, width, threshold):
    """For every walk window of `width` ops starting at a 32-op checkpoint: (max op length, sum of reference lengths).  The
    kernel leaves the packed 16-bit scan for a window with any op >= threshold (64 / 1024 for the two-ops-per-lane walk,
    32 / 2048 for a one-op-per-lane walk)."""
    g = read_geometry(reads)
    out = []
    for r in range(reads.n_reads):
        c0, c1 = int(reads.cigar_off[r]), int(reads.cigar_off[r + 1])
        if c1 - c0 > 4096:
            continue                                                       # ultra-long reads: short ops only
        for k in range(c0, c1, 32):
            sl = slice(k, min(k + width, c1))
            out.append((r, int(g["ln"][sl].max()), int(np.where(np.isin(g["op"][sl], REF_OPS), g["ln"][sl], 0).sum()),
                        int(np.where(np.isin(g["op"][sl], QRY_OPS), g["ln"][sl], 0).sum())))
    return np.array(out, np.int64)


def tile_classes(reads, L=CONTIG_LEN, tile=TILE, leave_out=()):
    """Per tile: candidate-range width (tile_hi - tile_lo of read_scan_kernel), reads really overlapping, and whether a passing
    read covers it with one D / N op alone (inside), aligned bases present, deletion / skip coverage present."""
    g = read_geometry(reads)
    n_t = (L + tile - 1) // tile
    lo = np.full(n_t, np.iinfo(np.int64).max); hi = np.zeros(n_t, np.int64)
    over = np.zeros(n_t, np.int64)
    for r in range(reads.n_reads):
        a, e = int(reads.pos[r]), int(g["rend"][r])
        if e <= a or r in leave_out:
            continue
        t0, t1 = a // tile, (min(e, L) - 1) // tile
        lo[t0:t1 + 1] = np.minimum(lo[t0:t1 + 1], r); hi[t0:t1 + 1] = np.maximum(hi[t0:t1 + 1], r + 1)
        over[t0:t1 + 1] += 1
    keep = g["passing"][g["rid"]]
    diff = {k: np.zeros(L + 1, np.int64) for k in ("aln", "del", "skip")}
    for key, ops in (("aln", ALN_OPS), ("del", (2,)), ("skip", (3,))):
        m = keep & np.isin(g["op"], ops)
        np.add.at(diff[key], g["rs"][m], 1); np.add.at(diff[key], np.minimum(g["rs"][m] + g["ln"][m], L), -1)
    cov = {k: np.cumsum(v)[:L] > 0 for k, v in diff.items()}
    tl = lambda x: x.reshape(n_t, tile) if L % tile == 0 else None                      # noqa: E731
    m = keep & np.isin(g["op"], (2, 3))
    inside = np.zeros(n_t, bool)
    for s, ln in zip(g["rs"][m], g["ln"][m]):
        t0, t1 = -(-int(s) // tile), (int(s + ln)) // tile                                # tiles wholly inside [s, s + ln)
        inside[t0:t1] = True
    return dict(width=np.where(hi > 0, hi - lo, 0), over=over, inside=inside, aln=tl(cov["aln"]).any(1),
                dele=tl(cov["del"]).any(1), skip=tl(cov["skip"]).any(1))


def long_op_rows(reads, L, dropped=None):
    """The long-op semantics in plain NumPy, by interval arithmetic over each passing read's ops:
    covered  -- an aligned base, a deletion or a reference skip of some read lies on p
    star     -- [fwd, rev] deletions spanning p (the '*' / '#' channels)
    aligned  -- [fwd, rev] aligned bases on p (ACGT reads: the reference channel holds minus this, tensor_maker.cpp:230-246)"""
    g = read_geometry(reads)
    keep = g["passing"] & (True if dropped is None else dropped == 0)
    k = keep[g["rid"]]
    strand = ((reads.flag >> 4) & 1)[g["rid"]]
    out = {}
    for key, ops in (("aligned", ALN_OPS), ("star", (2,)), ("any", REF_OPS)):
        d = np.zeros((2, L + 1), np.int64)
        m = k & np.isin(g["op"], ops)
        np.add.at(d, (strand[m], np.minimum(g["rs"][m], L)), 1)
        np.add.at(d, (strand[m], np.minimum(g["rs"][m] + g["ln"][m], L)), -1)
        out[key] = np.cumsum(d, axis=1)[:, :L]
    return out["any"].sum(0) > 0, out["star"], out["aligned"]


# ------------------------------------------------------------------------------------------------ CPU tests
@pytest.fixture(scope="module")
def fx():
    return long_fixture()


@pytest.fixture(scope="module")
def fx16():
    return long_fixture(cigar16=True)


def test_fixture_exercises_long_geometry(fx, fx16):
    from nanosnp_b200.reads import cigar16, max_reference_span
    ref, rd, tags = fx
    g = read_geometry(rd)
    have = set(t for t in tags if t)
    for L in THRESH_DN:
        assert {f"D{L}", f"N{L}"} <= have
        for op in (2, 3):
            assert ((g["op"] == op) & (g["ln"] == L)).any(), (op, L)
    for L in THRESH_S:
        assert {f"S{L}lead", f"S{L}trail", f"S{L}both_H"} <= have
        assert ((g["op"] == 4) & (g["ln"] == L)).sum() >= 4
    for L in THRESH_I:
        assert ((g["op"] == 1) & (g["ln"] == L)).any()
    for L in THRESH_M:
        assert ((g["op"] == 0) & (g["ln"] == L)).any()
    # clips at both ends, inside hard clips
    first, last = rd.cigar_off[:-1], rd.cigar_off[1:] - 1
    assert ((g["op"][first] == 5) & (g["op"][first + 1] == 4) & (g["ln"][first + 1] == 100_000)).any()
    assert ((g["op"][last] == 5) & (g["op"][last - 1] == 4) & (g["ln"][last - 1] == 100_000)).any()
    # long D / N on tile edges of 1024 and 2048, and one base either side
    dn = np.isin(g["op"], (2, 3)) & (g["ln"] >= 3000)
    for A in (1024, 2048):
        for off in (-1, 0, 1):
            for op in (2, 3):
                sel = dn & (g["op"] == op)
                assert ((g["rs"][sel] - off) % A == 0).any() and ((g["rs"][sel] + g["ln"][sel] - off) % A == 0).any(), (A, off, op)
    # adjacency
    seq = lambda r: "".join("MIDNSHP=X"[o] for o in g["op"][rd.cigar_off[r]:rd.cigar_off[r + 1]])    # noqa: E731
    ops_text = [seq(r) for r in range(rd.n_reads)]
    for pat in ("MDNM", "MNDM", "MINM"):
        assert any(pat in s for s in ops_text), pat
    assert any(s.startswith("SD") for s in ops_text) and any(s.endswith("NS") for s in ops_text)
    # long ops at op index 0, 31, 32, 63, 64 of one read (slot 0 and slot 1 of a lane)
    r = tags.index("chunkpos")
    c0 = int(rd.cigar_off[r])
    for i in (0, 31, 32, 63, 64):
        assert g["ln"][c0 + i] >= 1024, i
    # the packed-scan switch, decided on the host: windows at the limit stay packed, others leave it
    w2 = window_scans(rd, 64, 1024)
    packed = w2[:, 1] < 1024
    assert (packed & (w2[:, 2] > 65_000) & (w2[:, 2] < 65_536)).any()              # the packed scan at its limit
    assert (~packed & (w2[:, 2] > 65_536)).any()                                    # 64 ops of 1024-4095 summing past 2^16
    r_un = tags.index("unpacked_chunk")
    c0 = int(rd.cigar_off[r_un])
    assert (g["ln"][c0:c0 + 64] >= 1024).all() and (g["ln"][c0:c0 + 64] < 4096).all()
    w1 = window_scans(rd, 32, 2048)
    assert (w1[:, 1] >= 2048).any() and ((w1[:, 1] < 2048) & (w1[:, 1] >= 1024)).any()
    assert (w2[packed][:, 2:] < 65_536).all()                                       # the packed halves never carry
    # tiles: inside a single op, deletion-only and skip-only, deep only through an ultra-long read
    tc = tile_classes(rd)
    assert tc["inside"].sum() >= 40
    del_only = tc["dele"] & ~tc["aln"] & ~tc["skip"]
    skip_only = tc["skip"] & ~tc["aln"] & ~tc["dele"]
    assert del_only.sum() >= 3 and skip_only.sum() >= 3, (np.nonzero(del_only)[0], np.nonzero(skip_only)[0])
    deep_by_range = (tc["width"] > KREADLIST) & (tc["over"] < 256)
    ul = [i for i, t in enumerate(tags) if t and t.startswith("ultra")]
    without = tile_classes(rd, leave_out=set(ul))["width"]
    assert (deep_by_range & (without <= KREADLIST)).sum() >= 20, (deep_by_range.sum(), tc["width"].max(), without.max())
    # the ultra-long reads: 150-350 kb; one holds more than 65 535 ops and query bases (CG:B,I in a BAM)
    spans = g["rend"] - rd.pos
    assert len(ul) == 5 and all(150_000 <= spans[i] <= 351_000 for i in ul)
    n_ops = np.diff(rd.cigar_off)
    big = [i for i in ul if n_ops[i] > 65_535]
    assert big and int(np.where(np.isin(g["op"], QRY_OPS) & (g["rid"] == big[0]), g["ln"], 0).sum()) > 65_535
    assert max_reference_span(rd) >= 350_000
    # the cigar16 variant: every op below 4096, the 1024-4095 ops kept
    _, rd16, tags16 = fx16
    assert cigar16(rd16).cigar.dtype == np.uint16 and cigar16(rd).cigar.dtype == np.uint32
    ln16 = rd16.cigar >> 4
    for L in (1023, 1024, 1025, 2047, 2048, 2049, 4095):
        assert (ln16 == L).any(), L
    assert "unpacked_chunk" in tags16 and "packed_limit" in tags16


def test_numpy_long_op_semantics_equal_oracle_rows(fx, orc, tmp_path):
    """Covered bit, '*' / '#' per strand, aligned depth per strand (reference channels) from interval arithmetic over the ops
    equal the oracle's count rows at every position of the contig (cap off)."""
    ref, rd, _ = fx
    mp = str(tmp_path / "ctg1.mpileup")
    orc.mpileup_text(rd, "ctg1", mp, max_depth=0)
    res = orc.s1_restate(mp, "ctg1", ref, want_windows=False)
    covered, star, aligned = long_op_rows(rd, CONTIG_LEN)
    got_cov = (res.flags & 1).astype(bool)
    bad = np.nonzero(got_cov != covered)[0]
    assert bad.size == 0, bad[:10]
    c = res.counts
    assert np.array_equal(c[:, 8], star[0])
    assert np.array_equal(c[:, 17], star[1])
    rc = np.searchsorted(np.frombuffer(b"ACGT", np.uint8), ref)                  # ACGT contig: 0..3
    fwd = -c[np.arange(CONTIG_LEN), rc]
    rev = -c[np.arange(CONTIG_LEN), 9 + rc]
    for got, want, what in ((fwd, aligned[0], "fwd"), (rev, aligned[1], "rev")):
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, (what, bad[:10], got[bad[:3]], want[bad[:3]])
    # the features are really there in the rows: deletion-only and skip-only stretches, kilobase '*' runs
    assert ((star.sum(0) > 0) & (aligned.sum(0) == 0)).sum() > 3000
    assert (covered & (star.sum(0) == 0) & (aligned.sum(0) == 0)).sum() > 3000     # covered by skips alone


def test_count_row_encoding_hand_case(orc, tmp_path):
    """tensor_maker.cpp:230-246 on a hand case: the reference channel of each strand holds minus the strand's aligned (ACGT)
    bases, mismatches their own channel, deletions '*' / '#'; a reference skip covers without counting."""
    from nanosnp_b200.reads import from_records
    ref = np.frombuffer(b"ACGTACGTACGTACGTACGT", np.uint8)
    recs = [(2, 0, 60, "3M4D3M", "GTAGTA"), (2, 16, 60, "2M5N3M", "GTTAC"), (3, 0, 60, "2M", "TA"), (4, 16, 60, "3M", "AAG")]
    mp = str(tmp_path / "h.mpileup")
    orc.mpileup_text(from_records(recs), "ctg1", mp, max_depth=0)
    res = orc.s1_restate(mp, "ctg1", ref, want_windows=False, min_coverage=1)
    c = res.counts
    # p = 4 (A): read0 A fwd, read1 skip, read2 A fwd, read3 A rev -> A = -2, a = -1
    assert c[4, 0] == -2 and c[4, 9] == -1 and c[4, 8] == 0 and c[4, 17] == 0
    # p = 5 (C): read0 deletion fwd, read1 skip, read3 A rev (mismatch) -> '*' = 1, a = 1, c = -1
    assert c[5, 8] == 1 and c[5, 9] == 1 and c[5, 10] == -1 and c[5, 1] == 0
    covered, star, aligned = long_op_rows(from_records(recs), len(ref))
    assert np.array_equal(covered, (res.flags & 1).astype(bool))
    assert np.array_equal(star[0], c[:, 8]) and np.array_equal(star[1], c[:, 17])


def test_oracle_pinned_to_reference_tools_on_a_slice(fx, orc, tmp_path):
    """On a ~100 kb slice of the fixture (gap, tile-edge deletions, clipped and ultra-long reads), the oracle's tensor and
    predict data equal those of the reference's own compiled tools run on the same mpileup text."""
    from oracle.pyoracle import have_ref_binaries, s1_reference, write_fasta
    if not have_ref_binaries():
        pytest.skip("the reference's own tools are not built (oracle/_ref)")
    ref, rd, _ = fx
    lo, hi = 300_000, 400_000
    mp_all = str(tmp_path / "all.mpileup")
    orc.mpileup_text(rd, "ctg1", mp_all)
    d = tmp_path / "pile"; d.mkdir()
    mp = str(d / "ctg1.mpileup")
    with open(mp_all) as f, open(mp, "w") as out:
        n = 0
        for line in f:
            if lo < int(line.split("\t", 2)[1]) <= hi:
                out.write(line); n += 1
    assert n > 90_000
    fa = str(tmp_path / "ref.fa")
    write_fasta(fa, {"ctg1": ref})
    t_ref, pd_ref = s1_reference(mp, fa, "ctg1", str(tmp_path / "w"))
    t_orc, pd_orc = str(tmp_path / "o.tensor"), str(tmp_path / "o.pd")
    orc.s1_restate(mp, "ctg1", ref, tensor_path=t_orc, pd_path=pd_orc)
    assert open(t_orc, "rb").read() == open(t_ref, "rb").read()
    assert open(pd_orc, "rb").read() == open(pd_ref, "rb").read()
