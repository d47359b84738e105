"""Genotyping given sites (`--sites VCF`) on the GPU, against the oracle chain's count rows and float64 model, and against the
unrestricted GPU path.

Expectation: a listed 0-based site c is called iff rows c-16 .. c+16 all exist in the oracle's mpileup and the centre
reference base is ACGT (either case); its window is the oracle's count rows c-16 .. c+16.  The AF gate and min_coverage do
not apply, so the expectation is built from the rows directly rather than from the oracle's candidates."""
import io
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CONTIGS = [("ctgA", 300_000), ("ctgB", 90_000), ("ctgC", 170_000)]
NOREADS = ("ctgD", 40_000)
AF = 0.12


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


def _tallies(counts, ref):
    v = counts.astype(np.int64)
    code = np.full(256, 4, np.int64)
    for i, b in enumerate(b"ACGT"):
        code[b] = code[b + 32] = i
    rc = code[ref]
    chr_ = np.where(rc < 4, rc, 0)
    idx = np.arange(len(v))
    depth = -v[idx, chr_] - v[idx, 9 + chr_] + v[:, 8] + v[:, 17]
    snp = v[:, 0:4] + v[:, 9:13]
    snp[idx, chr_] = 0
    return depth, snp.max(1), np.maximum(v[:, 4] + v[:, 13], v[:, 6] + v[:, 15]), rc


def _min_count(depth):
    """Smallest count k with k / depth >= AF (the gate's float64 comparison)."""
    d = np.maximum(depth, 1).astype(np.float64)
    k = np.ceil(AF * d).astype(np.int64)
    k = np.where((k - 1) / d >= AF, k - 1, k)
    return np.where(k / d < AF, k + 1, k)


def _expected_sites(case, oracle_res, listed):
    """contig -> 0-based called sites of the listed positions, by the rule of the module docstring."""
    out = {}
    for name, L in CONTIGS:
        c = np.asarray(listed.get(name, []), np.int64)
        c = np.unique(c[(c >= 16) & (c < L - 16)])
        cov = np.concatenate([[0], np.cumsum(oracle_res[name].flags & 1, dtype=np.int64)])
        full = cov[c + 17] - cov[c - 16] == 33
        acgt = np.isin(case["refs"][name][c], np.frombuffer(b"ACGTacgt", np.uint8))
        out[name] = c[full & acgt]
    return out


def _windows(oracle_res, name, c):
    return oracle_res[name].counts[np.asarray(c, np.int64)[:, None] + np.arange(-16, 17)]


def _expected_vcf(case, oracle_res, model64, called):
    from oracle.s2_restate import predict_vcf, vcf_header
    text = vcf_header(open(case["fa"] + ".fai").read().splitlines())
    for name, _ in CONTIGS:
        c = called[name]
        if len(c):
            up = np.char.upper(case["refs"][name][c].view("S1")).view(np.uint8)
            text += predict_vcf(model64, name, c + 1, up, _windows(oracle_res, name, c))
    return text


def _write_sites(path, listed, extra=()):
    """A site VCF of the 0-based positions; records cycle through SNP, multi-allelic and indel forms, every tenth is repeated."""
    forms = ["A\tG", "C\tT,G", "CTT\tC", "A\tAGG"]
    lines = ["##fileformat=VCFv4.2\n", "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"]
    for name, pos in listed.items():
        for i, c in enumerate(np.asarray(pos, np.int64).tolist()):
            rec = f"{name}\t{c + 1}\t.\t{forms[i % 4]}\t.\t.\t.\n"
            lines.append(rec)
            if i % 10 == 0:
                lines.append(rec)
    lines += list(extra)
    with open(path, "w") as f:
        f.write("".join(lines))
    return str(path)


@pytest.fixture(scope="module")
def case(tmp_path_factory, golden):
    from nanosnp_b200.bam import write_bam
    from nanosnp_b200.dataset import save_reads_npz
    from nanosnp_b200.synth import SynthConfig, generate_host
    from oracle.pyoracle import write_fasta
    d = tmp_path_factory.mktemp("sites")
    refs, reads = {}, {}
    for i, (name, L) in enumerate(CONTIGS):
        cfg = SynthConfig(contig_len=L, coverage=22.0, contig=name, seed_ref=61 + i, seed_var=71 + i, seed_reads=81 + i, len_median=4000,
                          len_min=300, gap_period=100_000 if name == "ctgA" else 0, gap_len=12_000 if name == "ctgA" else 0,
                          ref_n_period=9_000 if name == "ctgB" else 0, ref_n_len=25 if name == "ctgB" else 0,
                          ref_lower_period=7_000 if name == "ctgB" else 0, ref_lower_len=200 if name == "ctgB" else 0)
        refs[name], reads[name] = generate_host(cfg)
    refs[NOREADS[0]] = generate_host(SynthConfig(contig_len=NOREADS[1], coverage=1.0, contig=NOREADS[0], seed_ref=9))[0]
    fa = str(d / "ref.fa")
    write_fasta(fa, refs)
    plain = str(d / "plain.bam"); write_bam(plain, [(n, len(r)) for n, r in refs.items()], reads)
    idx = str(d / "idx.bam"); write_bam(idx, [(n, len(r)) for n, r in refs.items()], reads, index=True)
    npz = d / "npz"; npz.mkdir()
    for name, _ in CONTIGS:
        save_reads_npz(str(npz / f"{name}.reads.npz"), reads[name], name, len(refs[name]))
    return dict(dir=d, refs=refs, reads=reads, fa=fa, plain=plain, idx=idx, npz=str(npz), golden=golden,
                contigs=[(n, len(r)) for n, r in refs.items()])


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


@pytest.fixture(scope="module")
def mixed(case, oracle_res):
    """The seeded site list of the parity tests: every kind of position a list of known sites can hold."""
    rng = np.random.default_rng(11)
    listed, kinds = {}, {}
    for name, L in CONTIGS:
        res, ref = oracle_res[name], case["refs"][name]
        depth, snp, indel, rc = _tallies(res.counts, ref)
        cov = (res.flags & 1) == 1
        gate = (res.flags & 2) == 2
        k = _min_count(depth)
        pick = lambda m, n: rng.choice(np.nonzero(m)[0], min(n, int(m.sum())), replace=False) if m.any() else np.zeros(0, np.int64)
        kind = {
            "gate": pick(gate, 40),
            "zero_alt": pick(cov & (depth > 0) & (snp == 0) & (indel == 0) & (rc < 4), 150),
            "below_af": pick(cov & ~gate & (rc < 4) & (k > 1) & ((snp == k - 1) | (indel == k - 1)), 120),
            "low_depth": pick(cov & (depth >= 1) & (depth <= 5), 120),
            "ends": np.r_[0:21, L - 21:L],
            "n_base": pick(rc == 4, 40),
            "lower": pick((ref >= ord("a")) & (ref <= ord("z")), 60),
        }
        if name == "ctgA":
            gap = np.nonzero(~cov)[0]
            gap = gap[(gap > 2000) & (gap < L - 2000)]
            lo, hi = int(gap[0]), int(gap[np.searchsorted(gap, gap[0] + 20_000) - 1])
            kind["gap"] = np.r_[lo - 40:lo + 20, hi - 20:hi + 40, (lo + hi) // 2]
        listed[name] = np.unique(np.concatenate([np.asarray(v, np.int64) for v in kind.values()]))
        kinds[name] = kind
    listed[NOREADS[0]] = np.array([100, 5000, 20_000])
    path = _write_sites(case["dir"] / "mixed.vcf", listed,
                        extra=["chrUnknown\t5\t.\tA\tG\t.\t.\t.\n", f"ctgB\t{CONTIGS[1][1] + 1}\t.\tA\tG\t.\t.\t.\n",
                               f"ctgB\t{CONTIGS[1][1] + 500}\t.\tA\tG\t.\t.\t.\n"])
    return dict(path=path, listed=listed, kinds=kinds, called=_expected_sites(case, oracle_res, listed))


def _run(case, data, out, *extra, region_len=50_000):
    from nanosnp_b200 import predict as P
    cfg = str(P.__file__).replace("predict.py", "config/ont_pileup.yaml")
    P.main(["-config", cfg, "-model_path", str(case["golden"] / "ont_pileup_weights.npz"), "-reference", case["fa"],
            "--region_len", str(region_len), "-data", data, "-output", str(out), *extra])
    return open(out, "rb").read()


def test_site_list_covers_every_kind(case, oracle_res, mixed):
    """The parity list holds each kind of position, and the called set holds those that have a full window."""
    called = {n: set(c.tolist()) for n, c in mixed["called"].items()}
    got = {}
    for name, _ in CONTIGS:
        res = oracle_res[name]
        depth = _tallies(res.counts, case["refs"][name])[0]
        for kind, pos in mixed["kinds"][name].items():
            n_called = sum(int(p) in called[name] for p in pos)
            got[kind] = got.get(kind, 0) + n_called
        gate = set((res.positions.astype(np.int64) - 1).tolist())
        got["not_gate"] = got.get("not_gate", 0) + len(called[name] - gate)
        got["depth_lt6"] = got.get("depth_lt6", 0) + int((depth[mixed["called"][name]] < 6).sum())
    assert got["n_base"] == 0
    for kind in ("gate", "zero_alt", "below_af", "low_depth", "lower", "gap", "depth_lt6"):
        assert got[kind] > 0, (kind, got)
    assert got["not_gate"] > 300


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
def test_sites_oracle_parity_every_input(case, oracle_res, model64, mixed, precision):
    d = case["dir"]
    args = ("--sites", mixed["path"], "--precision", precision)
    err = io.StringIO()
    from contextlib import redirect_stderr
    with redirect_stderr(err):
        a = _run(case, case["plain"], d / f"p_{precision}.vcf", *args)
    assert "skipped 3 site(s)" in err.getvalue()
    b = _run(case, case["idx"], d / f"i_{precision}.vcf", *args)
    c = _run(case, case["npz"], d / f"n_{precision}.vcf", *args)
    assert a == b == c
    assert a.count(b"\n") > 400
    _compare_vcf(a.decode(), _expected_vcf(case, oracle_res, model64, mixed["called"]))


@pytest.mark.parametrize("region_len", [300, 20_000, 10_000_000])
def test_s1_bit_exact_per_unit(case, oracle_res, mixed, region_len):
    import torch
    from nanosnp_b200.pipeline import PileupEngine
    from nanosnp_b200.reads import max_reference_span, slice_reads
    from nanosnp_b200.shard import listed_tiles, plan_target_units, read_range_for_region
    from nanosnp_b200.targets import load_sites_vcf
    eng = PileupEngine("cuda")
    targets = load_sites_vcf(mixed["path"], case["contigs"], report=None)
    units, ivs = plan_target_units(case["contigs"], targets, region_len)
    per_unit = [int((iv[:, 1] - iv[:, 0]).sum()) for iv in ivs]
    assert min(per_unit) >= 1 and max(per_unit) >= (1 if region_len < 1000 else 3 if region_len < 100_000 else 300)
    for name, L in CONTIGS:
        reads = case["reads"][name]
        ref = torch.from_numpy(case["refs"][name]).cuda()
        span = max_reference_span(reads) + 1
        got = []
        for rg, iv in zip(units, ivs):
            if rg.contig != name:
                continue
            rd = slice_reads(reads, *read_range_for_region(reads.pos, span, rg)).to_torch("cuda")
            c_all, f_all = eng.pileup_counts(rd, ref, rg.start, rg.length)
            c_t, f_t = eng.pileup_counts(rd, ref, rg.start, rg.length, targets=iv)
            on = np.zeros(rg.length, bool)
            for t in listed_tiles(rg, iv):
                on[t * 1024:(t + 1) * 1024] = True
            on_t = torch.from_numpy(on).cuda()
            assert torch.equal(c_t[on_t], c_all[on_t]) and torch.equal(f_t[on_t], f_all[on_t])
            cap = max(1, int((iv[:, 1] - iv[:, 0]).sum()))
            pos, n_dev = eng.select(f_t, ref, rg.start, rg.emit_start, rg.emit_end, cap, targets=iv, sites=True)
            n = int(n_dev.item())
            eng.check_status()
            x, _, _ = eng.gather(c_t, ref, rg.start, pos, n_dev, n)
            p = pos[:n].cpu().numpy().astype(np.int64)
            want = mixed["called"][name]
            assert np.array_equal(p, want[(want >= rg.emit_start) & (want < rg.emit_end)])
            assert np.array_equal(x[:n].cpu().numpy(), _windows(oracle_res, name, p))
            got.append(p)
        assert np.array_equal(np.concatenate(got), mixed["called"][name])


def test_candidate_positions_as_sites_identical(case, oracle_res):
    """Listing exactly the unrestricted run's candidates (the .pd positions) reproduces its VCF byte for byte."""
    d = case["dir"]
    listed = {name: oracle_res[name].positions.astype(np.int64) - 1 for name, _ in CONTIGS}
    path = _write_sites(d / "cands.vcf", listed)
    for data in (case["plain"], case["idx"], case["npz"]):
        base = _run(case, data, d / "c0.vcf")
        assert _run(case, data, d / "c1.vcf", "--sites", path) == base


def test_sites_with_bed_is_the_intersection(case, mixed):
    from nanosnp_b200.targets import build_targets, intersect_targets, load_sites_vcf
    d = case["dir"]
    bed = d / "t.bed"
    bed.write_text("ctgA\t0\t5000\nctgA\t90000\t150000\nctgB\t10\t40000\nctgC\t100000\t170000\nctgD\t0\t100\nchrQ\t0\t9\n")
    inter = intersect_targets(load_sites_vcf(mixed["path"], case["contigs"], report=None),
                              build_targets(case["contigs"], str(bed), report=None))
    path = _write_sites(d / "inter.vcf", {c: np.concatenate([np.arange(s, e) for s, e in iv]) for c, iv in inter.items()})
    a = _run(case, case["npz"], d / "sb.vcf", "--sites", mixed["path"], "--bed", str(bed))
    assert a == _run(case, case["npz"], d / "si.vcf", "--sites", path)
    assert a.count(b"\n") > 100 and a != _run(case, case["npz"], d / "s.vcf", "--sites", mixed["path"])
    assert _run(case, case["idx"], d / "sr.vcf", "--sites", mixed["path"], "--region", "ctgA:1-5000", "--region",
                "ctgA:90001-150000", "--region", "ctgB:11-40000", "--region", "ctgC:100001-170000",
                "--region", "ctgD:1-100") == a


def test_dense_list(case, oracle_res, model64):
    """Every position of a 200 kb interval (across the coverage gap of ctgA): the oracle's answer, no candidate overflow (50,000
    sites per unit), and the same s1 launches as one site per work unit."""
    import ctypes as C
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.caller import call_contig_text
    from nanosnp_b200.pipeline import PileupEngine, PileupModelForward, PileupModelWeights
    from nanosnp_b200.runner import RegionRunner
    from nanosnp_b200.shard import plan_target_units
    from nanosnp_b200.targets import site_intervals
    from oracle.s2_restate import load_weights_npz
    name, L = CONTIGS[0]
    dense = site_intervals(np.arange(50_000, 250_000))
    enc, fwd = load_weights_npz(case["golden"] / "ont_pileup_weights.npz")
    runner = RegionRunner(PileupEngine("cuda"), PileupModelForward(PileupModelWeights(enc, fwd), 1), records=True)
    lib = _lib.load()
    units, ivs = plan_target_units([(name, L)], {name: dense}, 50_000)
    assert len(units) == 4 and all(int((iv[:, 1] - iv[:, 0]).sum()) == 50_000 for iv in ivs)

    def run(targets, sink):
        torch.cuda.synchronize()
        _lib.check(lib.nsnp_profile_read(None, None))             # drop what earlier profiled calls left
        lib.nsnp_profile_enable(1)
        call_contig_text(runner, case["reads"][name], case["refs"][name], name, sink, 1000, 50_000, units, None, targets, True)
        torch.cuda.synchronize()
        ms = (C.c_double * len(_lib.PROF_SLOTS))(); ln = (C.c_int64 * len(_lib.PROF_SLOTS))()
        _lib.check(lib.nsnp_profile_read(ms, ln))
        lib.nsnp_profile_enable(0)
        return {k: int(ln[i]) for i, k in enumerate(_lib.PROF_SLOTS)
                                 if k in ("read_scan_kernel", "pileup_tile_kernel", "select_kernels")}
    sink = io.BytesIO()
    s1_many = run(ivs, sink)
    called = _expected_sites(case, oracle_res, {name: np.arange(50_000, 250_000)})
    assert len(called[name]) > 150_000
    one_each = []
    for u in units:                                           # one called site per unit
        c = called[name][(called[name] >= u.emit_start) & (called[name] < u.emit_end)]
        one_each.append(np.array([[c[len(c) // 2], c[len(c) // 2] + 1]]))
    s1_one = run(one_each, io.BytesIO())
    assert s1_many == s1_one and s1_many["pileup_tile_kernel"] == len(units)
    want = _expected_vcf(case, oracle_res, model64, {**{n: np.zeros(0, np.int64) for n, _ in CONTIGS}, **called})
    header = want[:want.index("\n", want.index("#CHROM")) + 1]
    _compare_vcf(header + sink.getvalue().decode(), want)


def test_two_ranks_with_sites(case, mixed):
    from nanosnp_b200 import predict as P
    d = case["dir"]
    one = _run(case, case["idx"], d / "r1.vcf", "--sites", mixed["path"])
    cfg = str(P.__file__).replace("predict.py", "config/ont_pileup.yaml")
    env = dict(os.environ, NSNP_DIST_BACKEND="gloo", PYTHONPATH=str(case["golden"].parent.parent))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29561", "-m", "nanosnp_b200.predict", "-config", cfg, "-model_path",
           str(case["golden"] / "ont_pileup_weights.npz"), "-reference", case["fa"], "--region_len", "50000", "-data", case["idx"],
           "-output", str(d / "r2.vcf"), "--sites", mixed["path"]]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert open(d / "r2.vcf", "rb").read() == one


def test_pd_refused_and_empty_lists(case, oracle_res, mixed):
    d = case["dir"]
    with pytest.raises(ValueError, match="--sites needs read inputs"):
        _run(case, str(d / "pd"), d / "pd.vcf", "--sites", mixed["path"])
    (d / "empty.vcf").write_text("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")
    (d / "unk.vcf").write_text("chrZ\t1\t.\tA\tG\t.\t.\t.\nchrZ\t7\t.\tA\tG\t.\t.\t.\n")
    head = _run(case, case["plain"], d / "h0.vcf", "--sites", str(d / "empty.vcf"))
    assert head.endswith(b"Sample\n") and all(l.startswith(b"#") for l in head.splitlines())
    assert _run(case, case["idx"], d / "h1.vcf", "--sites", str(d / "unk.vcf")) == head
    assert _run(case, case["npz"], d / "h2.vcf", "--sites", str(d / "unk.vcf")) == head


def test_bad_site_intervals_return_invalid(case):
    import ctypes as C
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupEngine
    eng = PileupEngine("cuda")
    ref = torch.from_numpy(case["refs"]["ctgB"]).cuda()
    flags = torch.zeros(2000, dtype=torch.uint8, device="cuda")
    for bad in ([[10, 5]], [[0, 10], [5, 20]], [[20, 30], [0, 10]], [[-1, 3]], [[1000, 3001]], [[7, 7]]):
        with pytest.raises(_lib.NsnpError) as e:
            eng.select(flags, ref, 1000, 1000, 3000, 4096, targets=np.array(bad), sites=True)
        assert e.value.code == _lib.E_INVALID
    lib = _lib.load()
    pos = torch.empty(16, dtype=torch.int32, device="cuda")
    n = torch.zeros(1, dtype=torch.int32, device="cuda")
    ws = torch.empty(lib.nsnp_select_sites_workspace_bytes(2000, 3), dtype=torch.uint8, device="cuda")
    args = (flags.data_ptr(), ref.data_ptr(), ref.shape[0], 1000, 2000, 1000, 3000)
    tail = (pos.data_ptr(), 16, n.data_ptr(), ws.data_ptr(), ws.numel(), eng.status.data_ptr(), 0)
    assert lib.nsnp_select_candidates_sites(*args, None, 3, *tail) == _lib.E_INVALID         # no interval array
    iv = np.array([[1000, 1001]], np.int32)
    assert lib.nsnp_select_candidates_sites(*args, iv.ctypes.data, -1, *tail) == _lib.E_INVALID
    assert lib.nsnp_select_candidates_sites(flags.data_ptr(), None, *args[2:], iv.ctypes.data, 1, *tail) == _lib.E_INVALID
    assert lib.nsnp_select_candidates_sites(*args, iv.ctypes.data, 1, *tail) == _lib.OK
    assert lib.nsnp_select_candidates_sites(*args, None, 0, *tail) == _lib.OK
    eng.check_status()
    assert int(n.item()) == 0


def test_f16x1_with_sites_same_calls(case, mixed):
    d = case["dir"]
    a = _run(case, case["npz"], d / "x3.vcf", "--sites", mixed["path"], "--precision", "f16x3").decode().splitlines()
    b = _run(case, case["npz"], d / "x1.vcf", "--sites", mixed["path"], "--precision", "f16x1").decode().splitlines()
    assert len(a) == len(b) and len(a) > 400
    for la, lb in zip(a, b):
        if la.startswith("#"):
            assert la == lb
            continue
        fa, fb = la.split("\t"), lb.split("\t")
        assert fa[:5] == fb[:5] and fa[6] == fb[6] and fa[9].split(":")[0] == fb[9].split(":")[0], (la, lb)
