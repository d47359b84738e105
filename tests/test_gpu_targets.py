"""Calling restricted to target intervals (`--bed` / `--region`) on the GPU, against the oracle chain run on whole contigs
and filtered to the targets, and against the unrestricted GPU path."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CONTIGS = [("ctgA", 300_000), ("ctgB", 90_000), ("ctgC", 170_000)]
NOREADS = ("ctgD", 40_000)


def _compare_vcf(got_text, ref_text):
    """QUAL within its last printed digit on at most 3 % of the records, everything else identical."""
    got = [l for l in got_text.splitlines() if not l.startswith("#")]
    ref = [l for l in ref_text.splitlines() if not l.startswith("#")]
    assert [l for l in got_text.splitlines() if l.startswith("#")] == [l for l in ref_text.splitlines() if l.startswith("#")]
    assert len(got) == len(ref)
    nq = 0
    for a, b in zip(got, ref):
        fa, fb = a.split("\t"), b.split("\t")
        assert fa[:5] == fb[:5] and fa[6:9] == fb[6:9], (a, b)
        sa, sb = fa[9].split(":"), fb[9].split(":")
        assert sa[0] == sb[0] and sa[2:] == sb[2:], (a, b)
        if fa[5] != fb[5]:
            nq += 1
            assert abs(float(fa[5]) - float(fb[5])) <= 0.0101
    assert nq <= 0.03 * max(1, len(ref))


def _coverage(reads, L):
    from nanosnp_b200.reads import max_reference_span
    op = reads.cigar.astype(np.uint32) & 15
    ln = (reads.cigar.astype(np.uint32) >> 4).astype(np.int64)
    cs = np.concatenate([[0], np.cumsum(np.where(np.isin(op, [0, 2, 3, 7, 8]), ln, 0))])
    end = reads.pos + (cs[reads.cigar_off[1:]] - cs[reads.cigar_off[:-1]])
    d = np.zeros(L + 1, np.int64)
    np.add.at(d, np.clip(reads.pos, 0, L), 1)
    np.add.at(d, np.clip(end, 0, L), -1)
    assert max_reference_span(reads) > 0
    return np.cumsum(d[:L])


def _seeded_bed(rng, refs, reads):
    """A few hundred intervals of 1 bp to 20 kb with every edge case of the contract."""
    lines = []
    for name, L in CONTIGS:
        for _ in range(150):
            s = int(rng.integers(0, L if name != "ctgC" else 30_000))           # ctgC 40-160 kb: short intervals only (below)
            ln = int(rng.choice([1, 2, 17, 300, 2_000, 20_000]))
            lines.append((name, s, min(L, s + ln)))
        lines += [(name, 0, 20), (name, L - 20, L)]                               # contig ends
        for t in (5, 17, 61):                                                      # tile boundaries +- 1 (tile 1024)
            b = 1024 * t
            if b + 2 < L:
                lines += [(name, b - 1, b + 1), (name, b + 1, b + 40), (name, b - 60, b)]
        lines += [(name, 1000, 1100), (name, 1100, 1200), (name, 1150, 1300), (name, 1000, 1100)]   # adjacent, overlapping, duplicate
    lines += [("ctgC", p, p + 1 + p % 3) for p in range(40_000, 160_000, 400)]       # hundreds of short intervals in one unit
    cov = _coverage(reads["ctgA"], CONTIGS[0][1])
    gap = np.nonzero(cov == 0)[0]
    gap = gap[(gap > 2000) & (gap < CONTIGS[0][1] - 2000)]
    assert len(gap), "the synthetic contig needs a coverage gap"
    lines.append(("ctgA", int(gap[len(gap) // 2]) - 30, int(gap[len(gap) // 2]) + 30))   # inside a coverage gap
    lines += [(NOREADS[0], 100, 5000), ("chrUnknown", 1, 100)]                      # no reads; not in the index
    order = rng.permutation(len(lines))
    return "track name=t\n# seeded\n" + "".join("%s\t%d\t%d\tx\n" % lines[i] for i in order)


@pytest.fixture(scope="module")
def case(tmp_path_factory, golden):
    from nanosnp_b200.bam import write_bam
    from nanosnp_b200.dataset import save_reads_npz
    from nanosnp_b200.synth import SynthConfig, generate_host
    from nanosnp_b200.targets import build_targets
    from oracle.pyoracle import write_fasta
    d = tmp_path_factory.mktemp("targets")
    refs, reads = {}, {}
    for i, (name, L) in enumerate(CONTIGS):
        cfg = SynthConfig(contig_len=L, coverage=22.0, contig=name, seed_ref=31 + i, seed_var=41 + i, seed_reads=51 + i, len_median=4000,
                          len_min=300, gap_period=100_000 if name == "ctgA" else 0, gap_len=12_000 if name == "ctgA" else 0)
        refs[name], reads[name] = generate_host(cfg)
    refs[NOREADS[0]] = generate_host(SynthConfig(contig_len=NOREADS[1], coverage=1.0, contig=NOREADS[0], seed_ref=9))[0]
    fa = str(d / "ref.fa")
    write_fasta(fa, refs)
    plain = str(d / "plain.bam"); write_bam(plain, [(n, len(r)) for n, r in refs.items()], reads)
    idx = str(d / "idx.bam"); write_bam(idx, [(n, len(r)) for n, r in refs.items()], reads, index=True)
    npz = d / "npz"; npz.mkdir()
    for name, _ in CONTIGS:
        save_reads_npz(str(npz / f"{name}.reads.npz"), reads[name], name, len(refs[name]))
    bed = str(d / "t.bed")
    with open(bed, "w") as f:
        f.write(_seeded_bed(np.random.default_rng(7), refs, reads))
    contigs = [(n, len(r)) for n, r in refs.items()]
    return dict(dir=d, refs=refs, reads=reads, fa=fa, plain=plain, idx=idx, npz=str(npz), bed=bed, contigs=contigs,
                targets=build_targets(contigs, bed, report=None), golden=golden)


@pytest.fixture(scope="module")
def oracle_res(case, orc):
    out = {}
    (case["dir"] / "pd").mkdir(exist_ok=True)
    for name, _ in CONTIGS:
        mp = str(case["dir"] / f"{name}.mpileup")
        orc.mpileup_text(case["reads"][name], name, mp)
        out[name] = orc.s1_restate(mp, name, case["refs"][name], pd_path=str(case["dir"] / "pd" / f"{name}.pd"))
    return out


@pytest.fixture(scope="module")
def model64(golden_weights):
    import torch
    from oracle.s2_restate import PileupModelOracle
    torch.set_num_threads(os.cpu_count() or 1)
    return PileupModelOracle(*golden_weights)


def _expected_vcf(case, oracle_res, model64, targets):
    from nanosnp_b200.targets import in_targets
    from oracle.s2_restate import predict_vcf, vcf_header
    text = vcf_header(open(case["fa"] + ".fai").read().splitlines())
    for name, _ in CONTIGS:
        res = oracle_res[name]
        keep = in_targets(res.positions.astype(np.int64) - 1, targets.get(name))
        if keep.any():
            pos = res.positions[keep]
            up = np.char.upper(case["refs"][name][pos - 1].view("S1")).view(np.uint8)
            text += predict_vcf(model64, name, pos, up, res.windows[keep])
    return text


def _run(case, data, out, *extra, region_len=50_000):
    from nanosnp_b200 import predict as P
    cfg = str(P.__file__).replace("predict.py", "config/ont_pileup.yaml")
    P.main(["-config", cfg, "-model_path", str(case["golden"] / "ont_pileup_weights.npz"), "-reference", case["fa"],
            "--region_len", str(region_len), "-data", data, "-output", str(out), *extra])
    return open(out, "rb").read()


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
def test_bed_oracle_parity_every_input(case, oracle_res, model64, precision):
    d = case["dir"]
    pd_dir = d / "pd"                                     # the oracle's .pd text of every whole contig, filtered on the host
    args = ("--bed", case["bed"], "--precision", precision)
    a = _run(case, case["plain"], d / f"p_{precision}.vcf", *args)
    b = _run(case, case["idx"], d / f"i_{precision}.vcf", *args)
    c = _run(case, case["npz"], d / f"n_{precision}.vcf", *args)
    p = _run(case, str(pd_dir), d / f"d_{precision}.vcf", *args)
    assert a == b == c == p
    assert a.count(b"\n") > 300
    _compare_vcf(a.decode(), _expected_vcf(case, oracle_res, model64, case["targets"]))


@pytest.mark.parametrize("region_len", [300, 20_000, 10_000_000])
def test_s1_bit_exact_inside_targets(case, oracle_res, region_len):
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupEngine
    from nanosnp_b200.reads import max_reference_span, slice_reads
    from nanosnp_b200.shard import listed_tiles, plan_target_units, read_range_for_region
    from nanosnp_b200.targets import in_targets
    eng = PileupEngine("cuda")
    units, ivs = plan_target_units(case["contigs"], case["targets"], region_len)
    per_unit = [len(iv) for iv in ivs]
    assert max(per_unit) >= (1 if region_len < 1000 else 3)
    if region_len == 10_000_000:
        assert max(per_unit) >= 100                       # hundreds of intervals in one unit
    for name, L in CONTIGS:
        res = oracle_res[name]
        reads = case["reads"][name]
        ref = torch.from_numpy(case["refs"][name]).cuda()
        span = max_reference_span(reads) + 1
        got_pos = []
        for rg, iv in zip(units, ivs):
            if rg.contig != name:
                continue
            rd = slice_reads(reads, *read_range_for_region(reads.pos, span, rg)).to_torch("cuda")
            c_all, f_all = eng.pileup_counts(rd, ref, rg.start, rg.length)
            c_t, f_t = eng.pileup_counts(rd, ref, rg.start, rg.length, targets=iv)
            tl = listed_tiles(rg, iv)
            on = np.zeros(rg.length, bool)
            for t in tl:
                on[t * 1024:(t + 1) * 1024] = True
            on_t = torch.from_numpy(on).cuda()
            assert torch.equal(c_t[on_t], c_all[on_t]) and torch.equal(f_t[on_t], f_all[on_t])
            assert int(f_t[~on_t].abs().sum()) == 0                            # unlisted tiles: flags 0
            pos, n_dev = eng.select(f_t, ref, rg.start, rg.emit_start, rg.emit_end, max(1024, rg.emit_end - rg.emit_start), targets=iv)
            n = int(n_dev.item())
            eng.check_status()
            x, _, _ = eng.gather(c_t, ref, rg.start, pos, n_dev, n)
            p = pos[:n].cpu().numpy().astype(np.int64)
            sel = np.isin(res.positions.astype(np.int64) - 1, p)
            assert (res.positions[sel].astype(np.int64) - 1 == p).all()
            assert np.array_equal(x[:n].cpu().numpy(), res.windows[sel])
            got_pos.append(p)
        want = res.positions.astype(np.int64) - 1
        want = want[in_targets(want, case["targets"].get(name))]
        got = np.concatenate(got_pos) if got_pos else np.zeros(0, np.int64)
        assert np.array_equal(got, want)


def test_bad_intervals_return_invalid(case):
    import ctypes as C
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupEngine
    from nanosnp_b200.reads import slice_reads
    eng = PileupEngine("cuda")
    ref = torch.from_numpy(case["refs"]["ctgB"]).cuda()
    rd = slice_reads(case["reads"]["ctgB"], 0, 50).to_torch("cuda")
    for bad in ([[10, 5]], [[0, 10], [5, 20]], [[20, 30], [0, 10]], [[-1, 3]], [[0, 5000]], [[7, 7]]):
        with pytest.raises(_lib.NsnpError) as e:
            eng.pileup_counts(rd, ref, 1000, 2000, targets=np.array(bad))
        assert e.value.code == _lib.E_INVALID
        flags = torch.zeros(2000, dtype=torch.uint8, device="cuda")
        with pytest.raises(_lib.NsnpError) as e:
            eng.select(flags, ref, 1000, 1000, 3000, 4096, targets=np.array(bad))
        assert e.value.code == _lib.E_INVALID
    lib = _lib.load()
    st = rd.as_struct()
    counts = torch.empty((100, 18), dtype=torch.int32, device="cuda")
    ws = torch.empty(lib.nsnp_pileup_targets_workspace_bytes(st.n_reads, st.n_cigar, 100, 3), dtype=torch.uint8, device="cuda")
    assert lib.nsnp_pileup_counts_targets(C.byref(st), ref.data_ptr(), ref.shape[0], 0, 100, None, 3, C.byref(eng.params),
                                          counts.data_ptr(), flags.data_ptr(), ws.data_ptr(), ws.numel(), eng.status.data_ptr(),
                                          0) == _lib.E_INVALID


def test_whole_contig_targets_identical(case):
    d = case["dir"]
    whole = d / "whole.bed"
    whole.write_text("".join(f"{n}\t0\t{L}\n" for n, L in case["contigs"]))
    regs = [a for n, _ in case["contigs"] for a in ("--region", n)]
    for data in (case["plain"], case["idx"], case["npz"]):
        base = _run(case, data, d / "w0.vcf")
        assert _run(case, data, d / "w1.vcf", "--bed", str(whole)) == base
        assert _run(case, data, d / "w2.vcf", *regs) == base


def test_two_ranks_with_bed(case):
    from nanosnp_b200 import predict as P
    d = case["dir"]
    one = _run(case, case["idx"], d / "r1.vcf", "--bed", case["bed"])
    cfg = str(P.__file__).replace("predict.py", "config/ont_pileup.yaml")
    env = dict(os.environ, NSNP_DIST_BACKEND="gloo", PYTHONPATH=str(case["golden"].parent.parent))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29551", "-m", "nanosnp_b200.predict", "-config", cfg, "-model_path",
           str(case["golden"] / "ont_pileup_weights.npz"), "-reference", case["fa"], "--region_len", "50000", "-data", case["idx"],
           "-output", str(d / "r2.vcf"), "--bed", case["bed"]]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert open(d / "r2.vcf", "rb").read() == one


def test_many_tiny_intervals(case, oracle_res, model64):
    import io
    import torch
    from nanosnp_b200.caller import call_contig_text
    from nanosnp_b200.pipeline import PileupEngine, PileupModelForward, PileupModelWeights
    from nanosnp_b200.runner import RegionRunner
    from nanosnp_b200.shard import plan_target_units
    from nanosnp_b200.targets import merge_intervals
    from oracle.s2_restate import load_weights_npz
    rng = np.random.default_rng(3)
    name, L = CONTIGS[0]
    pts = np.sort(rng.choice(L // 2, 20_000, replace=False) * 2)                     # even positions: no two adjacent
    pts[:50] = np.sort(oracle_res[name].positions[:50].astype(np.int64) - 1)        # some certain hits
    iv = merge_intervals([(int(p), int(p) + 1) for p in np.unique(pts)], L)
    enc, fwd = load_weights_npz(case["golden"] / "ont_pileup_weights.npz")
    runner = RegionRunner(PileupEngine("cuda"), PileupModelForward(PileupModelWeights(enc, fwd), 2), records=True)
    import ctypes as C
    from nanosnp_b200 import _lib
    lib = _lib.load()

    def run(targets, sink):
        # s1 launches from the library's own launch counters; the model and text launches scale with the sites instead
        runner.launches = 0
        torch.cuda.synchronize()
        _lib.check(lib.nsnp_profile_read(None, None))             # drop what earlier profiled calls left
        lib.nsnp_profile_enable(1)
        call_contig_text(runner, case["reads"][name], case["refs"][name], name, sink, 1000, 50_000, units, None, targets)
        torch.cuda.synchronize()
        ms = (C.c_double * len(_lib.PROF_SLOTS))(); ln = (C.c_int64 * len(_lib.PROF_SLOTS))()
        _lib.check(lib.nsnp_profile_read(ms, ln))
        lib.nsnp_profile_enable(0)
        return runner.launches, {k: int(ln[i]) for i, k in enumerate(_lib.PROF_SLOTS) if k in ("read_scan_kernel", "pileup_tile_kernel", "select_kernels")}
    units, ivs = plan_target_units([(name, L)], {name: iv}, 50_000)
    assert sum(len(u) for u in ivs) == len(iv) >= 19_900
    sink = io.BytesIO()
    many, s1_many = run(ivs, sink)
    one, s1_one = run([np.array([[u.emit_start, u.emit_end]]) for u in units], io.BytesIO())
    assert s1_many == s1_one and s1_many["pileup_tile_kernel"] == len(units)
    assert many <= one
    want = _expected_vcf(case, oracle_res, model64, {name: iv})
    header = want[:want.index("\n", want.index("#CHROM")) + 1]
    assert want.count("\n") > header.count("\n") + 50
    _compare_vcf(header + sink.getvalue().decode(), want)


def test_depth_cap_inside_targets(tmp_path, orc, golden):
    """A 250x contig: the cap at 144 drops reads.  In-memory input with targets is bit-exact with the oracle (cap 144)."""
    import torch
    from nanosnp_b200.pipeline import PileupEngine
    from nanosnp_b200.reads import max_reference_span, slice_reads
    from nanosnp_b200.shard import plan_target_units, read_range_for_region
    from nanosnp_b200.synth import SynthConfig, generate_host
    from nanosnp_b200.targets import in_targets, merge_intervals
    L = 60_000
    ref_h, reads = generate_host(SynthConfig(contig_len=L, coverage=250.0, contig="ctg1", seed_ref=5, seed_var=6, seed_reads=7,
                                             len_median=1500, len_min=200))
    assert (np.bincount(reads.pos)[np.bincount(reads.pos) > 1]).size > 0        # same-start reads exist
    mp = str(tmp_path / "c.mpileup")
    orc.mpileup_text(reads, "ctg1", mp, max_depth=144)
    res = orc.s1_restate(mp, "ctg1", ref_h)
    iv = merge_intervals([(1000, 1400), (9_990, 10_010), (30_000, 36_000), (59_900, 60_000)], L)
    eng = PileupEngine("cuda")
    ref = torch.from_numpy(ref_h).cuda()
    span = max_reference_span(reads) + 1
    units, ivs = plan_target_units([("ctg1", L)], {"ctg1": iv}, 8_000)
    got = []
    for rg, u in zip(units, ivs):
        rd = slice_reads(reads, *read_range_for_region(reads.pos, span, rg)).to_torch("cuda")
        c, f = eng.pileup_counts(rd, ref, rg.start, rg.length, targets=u)
        pos, n_dev = eng.select(f, ref, rg.start, rg.emit_start, rg.emit_end, 65536, targets=u)
        n = int(n_dev.item())
        eng.check_status()
        x, _, _ = eng.gather(c, ref, rg.start, pos, n_dev, n)
        p = pos[:n].cpu().numpy().astype(np.int64)
        sel = np.isin(res.positions.astype(np.int64) - 1, p)
        assert np.array_equal(x[:n].cpu().numpy(), res.windows[sel])
        got.append(p)
    want = res.positions.astype(np.int64) - 1
    assert np.array_equal(np.concatenate(got), want[in_targets(want, iv)])


def test_empty_and_unknown_only_bed_give_header_only(case):
    d = case["dir"]
    (d / "empty.bed").write_text("# nothing\n")
    (d / "unk.bed").write_text("chrZ\t1\t100\n")
    head = _run(case, case["plain"], d / "h0.vcf", "--bed", str(d / "empty.bed"))
    assert head.endswith(b"Sample\n") and all(l.startswith(b"#") for l in head.splitlines())
    assert _run(case, case["idx"], d / "h1.vcf", "--bed", str(d / "unk.bed")) == head


def test_f16x1_with_targets_same_calls(case):
    d = case["dir"]
    a = _run(case, case["npz"], d / "x3.vcf", "--bed", case["bed"], "--precision", "f16x3").decode().splitlines()
    b = _run(case, case["npz"], d / "x1.vcf", "--bed", case["bed"], "--precision", "f16x1").decode().splitlines()
    assert len(a) == len(b)
    for la, lb in zip(a, b):
        if la.startswith("#"):
            assert la == lb
            continue
        fa, fb = la.split("\t"), lb.split("\t")
        assert fa[:5] == fb[:5] and fa[6] == fb[6] and fa[9].split(":")[0] == fb[9].split(":")[0], (la, lb)     # same calls
