"""GPU parity at high read depth: a chrM-like contig (16 569 bp) at 300x to 8000x, one tile under 16 383 reads, and the model
on counts above 2048 (where an fp16 count is no longer exact, so the lo operand of layer 0 carries real bits).

s1 must stay bit-exact against the oracle chain whatever the number of indel events in a tile (deep tiles chain every event,
including the 1- and 2-base ones); the model must stay within its tolerances against the float64 network, in every precision;
records and VCF text must agree with the oracle's rows; the CLI must run a BAM holding such a contig to the end.
"""
import io

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

CHRM_LEN = 16_569
TILE = 1024
SLAB_EVENTS = 32768                   # per-tile event slab of pileup_tile_kernel (pileup.cu kSlabCapMax)
F16X3_ATOL = 5e-5
FP32_ATOL = 2e-5
F16X1_ATOL = 5e-3

# nominal coverage, --max-depth
DEEP = {"300x": (300.0, 144), "1000x": (1000.0, 144), "8000x": (8000.0, 144), "8000x_nocap": (8000.0, 0)}


def chrm_cfg(coverage):
    from nanosnp_b200.synth import SynthConfig
    return SynthConfig(contig_len=CHRM_LEN, coverage=coverage, contig="chrM", snp_rate=1e-2, seed_ref=61, seed_var=62, seed_reads=63)


def _params(max_depth):
    from nanosnp_b200 import _lib
    p = _lib.default_params()
    p.max_depth = max_depth
    return p


@pytest.fixture(scope="module")
def engines():
    import torch
    from nanosnp_b200.pipeline import PileupEngine
    assert torch.cuda.is_available()
    return {md: PileupEngine("cuda:0", _params(md)) for md in (144, 0)}


@pytest.fixture(scope="module")
def deep_case(orc, tmp_path_factory):
    """name -> (ref, reads, oracle S1Result, max_depth); each contig and its oracle chain is built once per module."""
    from nanosnp_b200.synth import generate_host
    cache = {}
    d = tmp_path_factory.mktemp("deep")

    def get(name):
        if name not in cache:
            cov, md = DEEP[name]
            ref, reads = generate_host(chrm_cfg(cov))
            mp = str(d / f"{name}.mpileup")
            orc.mpileup_text(reads, "chrM", mp, max_depth=md)
            cache[name] = (ref, reads, orc.s1_restate(mp, "chrM", ref), md)
        return cache[name]
    return get


@pytest.fixture(scope="module")
def weights(golden_weights):
    from nanosnp_b200.pipeline import PileupModelWeights
    return PileupModelWeights(*golden_weights, device="cuda:0")


@pytest.fixture(scope="module")
def model64(golden_weights):
    import os
    import torch
    from oracle.s2_restate import PileupModelOracle
    torch.set_num_threads(os.cpu_count() or 1)
    return PileupModelOracle(*golden_weights)


# ------------------------------------------------------------------------------------------------ host-side helpers
def _events_per_tile(reads, dropped, region_start, region_len):
    """Indel events anchored in each tile of [region_start, region_start + region_len), counted with the kernel's rules (passing
    reads the cap keeps, length <= NSNP_MAX_INDEL, not leading, anchor = reference position before the op), and the number of
    passing reads overlapping each tile."""
    cig = reads.cigar.astype(np.int64)
    op, ln = cig & 15, cig >> 4
    n = reads.n_reads
    rid = np.repeat(np.arange(n), np.diff(reads.cigar_off))
    rl = np.where(np.isin(op, (0, 2, 3, 7, 8)), ln, 0)
    cum = np.cumsum(rl) - rl                                   # exclusive, over the whole array
    rs = reads.pos[rid].astype(np.int64) + cum - cum[reads.cigar_off[:-1]][rid]
    rend = np.zeros(n, np.int64)
    np.add.at(rend, rid, rl)
    rend += reads.pos
    passing = ((reads.flag & 4) == 0) & ((reads.flag & 2316) == 0) & (reads.mapq >= 20) & (dropped == 0)
    ev = passing[rid] & np.isin(op, (1, 2)) & (ln <= 60) & (rs > reads.pos[rid]) & (rs - 1 >= region_start) & (rs - 1 < region_start + region_len)
    n_tiles = (region_len + TILE - 1) // TILE
    per_tile = np.bincount((rs[ev] - 1 - region_start) // TILE, minlength=n_tiles)
    over = np.zeros(n_tiles, np.int64)
    for t in range(n_tiles):
        ts, te = region_start + t * TILE, min(region_start + (t + 1) * TILE, region_start + region_len)
        over[t] = int((passing & (reads.pos < te) & (rend > ts)).sum())
    return per_tile, over


def _gpu_s1(engine, reads, ref, **kw):
    import torch
    rd = reads.to_torch(engine.device)
    rf = torch.from_numpy(np.ascontiguousarray(ref)).to(engine.device)
    pos, refbase, x, counts, flags = engine.candidate_windows(rd, rf, **kw)
    torch.cuda.synchronize()
    return pos.cpu().numpy(), x.cpu().numpy(), counts.cpu().numpy(), flags.cpu().numpy()


def _compare(res, pos, x, counts, flags, lo=0, hi=None):
    """test_gpu_s1._compare: covered bits, count rows of covered positions, zero rows elsewhere, gate bits."""
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


# ------------------------------------------------------------------------------------------------ s1 at depth
@pytest.mark.parametrize("name", list(DEEP))
def test_deep_contig_s1_bit_exact(engines, orc, deep_case, name):
    """Whole contig, then three shards whose boundaries and 16-bp halos cut through deep tiles: counts, flags, candidate
    positions and windows equal the oracle chain bit for bit."""
    ref, reads, res, md = deep_case(name)
    eng = engines[md]
    dropped = orc.depth_cap(reads, max_depth=md) if md else np.zeros(reads.n_reads, np.uint8)
    per_tile, over = _events_per_tile(reads, dropped, 0, CHRM_LEN)
    assert over.max() > 255                                            # every case runs deep tiles
    if name != "300x":
        assert per_tile.max() > SLAB_EVENTS, per_tile.max()            # more indel events in one tile than one slab holds
    assert len(res.positions) > 100
    pos, x, counts, flags = _gpu_s1(eng, reads, ref)
    _compare(res, pos, x, counts, flags)
    assert np.array_equal(pos + 1, res.positions) and np.array_equal(x, res.windows)
    # region shards with halos (SURVEY 8e): tile boundaries of a shard start at its halo, not at multiples of 1024
    got = []
    for s, e in ((0, 5_001), (5_001, 11_333), (11_333, CHRM_LEN)):
        rs, re_ = max(0, s - 16), min(CHRM_LEN, e + 16)
        pos, x, counts, flags = _gpu_s1(eng, reads, ref, region_start=rs, region_len=re_ - rs, emit_start=s, emit_end=e)
        _compare(res, pos, x, counts, flags, rs, re_)
        sel = (res.positions - 1 >= s) & (res.positions - 1 < e)
        assert np.array_equal(x, res.windows[sel])
        got.append(pos)
    assert np.array_equal(np.concatenate(got) + 1, res.positions)


def _one_tile_reads(n, seed=17):
    """n reads that all overlap tile 0 of a 2 000-bp contig: starts in [0, 600), 150-400 bp, three or four indels each
    (1- and 2-base ones as well as longer ones), both strands, a few N bases."""
    rng = np.random.default_rng(seed)
    recs = []
    for i in range(n):
        p = int(rng.integers(0, 600))
        parts, q = [], 0
        for k in range(int(rng.integers(3, 5))):
            m = int(rng.integers(20, 80))
            parts.append(f"{m}M"); q += m
            il = int(rng.choice([1, 1, 2, 3, 7]))
            if rng.random() < 0.5:
                parts.append(f"{il}I"); q += il
            else:
                parts.append(f"{il}D")
        m = int(rng.integers(20, 80))
        parts.append(f"{m}M"); q += m
        seq = "".join("ACGTN"[b] for b in rng.choice(5, q, p=[0.2495, 0.2495, 0.2495, 0.2495, 0.002]))
        recs.append((p, 16 * int(rng.integers(0, 2)), 60, "".join(parts), seq))
    recs.sort(key=lambda r: r[0])
    return recs


def test_tile_overlap_limit(engines, orc, tmp_path):
    """16 383 reads over one tile (the most the biased 16-bit depth deltas hold) are bit-exact against the oracle with the cap
    off; one read more is a clean NSNP_E_OVERFLOW, and the engine keeps working afterwards."""
    from nanosnp_b200 import _lib
    from nanosnp_b200.reads import from_records
    eng = engines[0]
    rng = np.random.default_rng(5)
    ref = np.frombuffer(bytes(rng.choice(list(b"ACGT"), 2000).astype(np.uint8)), np.uint8)
    recs = _one_tile_reads(16_384)
    keep = sorted(recs[:8000] + recs[8001:], key=lambda r: r[0])          # 16 383 reads
    rd = from_records(keep)
    per_tile, over = _events_per_tile(rd, np.zeros(rd.n_reads, np.uint8), 0, len(ref))
    assert over[0] == 16_383 and per_tile[0] > SLAB_EVENTS, (over, per_tile)
    mp = str(tmp_path / "t.mpileup")
    orc.mpileup_text(rd, "ctg1", mp, max_depth=0)
    res = orc.s1_restate(mp, "ctg1", ref)
    first = _gpu_s1(eng, rd, ref)
    pos, x, counts, flags = first
    _compare(res, pos, x, counts, flags)
    assert np.array_equal(pos + 1, res.positions) and np.array_equal(x, res.windows)
    assert counts[:, [0, 1, 2, 3]].min() < -2048                        # one strand alone is thousands deep
    with pytest.raises(_lib.NsnpError) as e:
        _gpu_s1(eng, from_records(recs), ref)
    assert e.value.code == _lib.E_OVERFLOW
    again = _gpu_s1(eng, rd, ref)                                        # the status word was cleared
    for a, b in zip(first, again):
        assert np.array_equal(a, b)


# ------------------------------------------------------------------------------------------------ model at deep counts
def _col_order():
    n = np.arange(256)
    return ((n >> 2) & 3) * 64 + (n >> 5) * 8 + ((n >> 4) & 1) * 4 + (n & 3)


def _col_scale():
    n = np.arange(256)
    return np.where(((n >> 2) & 3) == 2, -2.0, -1.0) * np.log2(np.e)


def _onehot_rows(n, seed):
    """Every (site, window row) has one channel set to an odd value in (2048, 16383] (either sign), the others zero: the fp16
    hi part of such a count drops 1-7, which only the lo operand carries."""
    rng = np.random.default_rng(seed)
    x = np.zeros((n, 33, 18), np.int32)
    ch = rng.integers(0, 18, (n, 33))
    v = 2 * rng.integers(1025, 8192, (n, 33)) + 1
    sign = np.where(rng.random((n, 33)) < 0.5, -1, 1)
    np.put_along_axis(x, ch[..., None], (sign * v)[..., None].astype(np.int32), axis=2)
    return x


def _dense_rows(n, seed):
    """Every channel nonzero, shaped like a deep pile-up: a reference channel per strand at -(2049..16383), odd; mismatch and
    indel channels up to a few hundred."""
    rng = np.random.default_rng(seed)
    x = rng.integers(1, 400, (n, 33, 18)).astype(np.int32)
    x[:, :, [0, 9]] = -(2 * rng.integers(1025, 8192, (n, 33, 2)) + 1)
    return x


@pytest.fixture(scope="module")
def deep_inputs(deep_case):
    """4 097 windows: one-hot deep rows, the 8000x contig's real windows, dense random deep rows, shuffled together."""
    _, _, res, _ = deep_case("8000x_nocap")
    real = res.windows
    assert np.abs(real).max() > 2048 and ((np.abs(real) > 2048) & (real % 2 != 0)).sum() > 100
    onehot = _onehot_rows(2048, 3)
    x = np.concatenate([onehot, real, _dense_rows(4097 - 2048 - len(real), 4)])
    perm = np.random.default_rng(9).permutation(len(x))
    return {"x": np.ascontiguousarray(x[perm]), "onehot": onehot}


@pytest.mark.parametrize("cg", [2])
def test_layer0_gates_at_deep_counts(weights, golden_weights, deep_inputs, cg):
    """Raw layer-0 accumulators of step 0 (both directions) against float64, relative to sum |x w|: the three passes over the
    input k-blocks are exact enough that dropping the lo pass would exceed the bound by far on the one-hot rows."""
    import torch
    from nanosnp_b200 import _lib
    lib = _lib.load()
    enc, _ = golden_weights
    for name, x in (("onehot", deep_inputs["onehot"]), ("mixed", deep_inputs["x"])):
        m = len(x)
        xi = torch.from_numpy(x).cuda()
        for d in (0, 1):
            sfx = "_reverse" if d else ""
            out = torch.full((m, 256), float("nan"), device="cuda")
            _lib.check(lib.nsnp_debug_lstm_tc_gates(weights.blob.data_ptr(), xi.data_ptr(), 0, d, cg, 0, out.data_ptr(), m,
                                                    torch.cuda.current_stream().cuda_stream))
            torch.cuda.synchronize()
            w = enc[f"lstm.weight_ih_l0{sfx}"].astype(np.float64)
            b = (enc[f"lstm.bias_ih_l0{sfx}"] + enc[f"lstm.bias_hh_l0{sfx}"]).astype(np.float64)
            xt = x[:, 0 if d == 0 else 32, :].astype(np.float64)
            ref = (xt @ w.T + b)[:, _col_order()] * _col_scale()
            mag = (np.abs(xt) @ np.abs(w).T + np.abs(b))[:, _col_order()] * np.abs(_col_scale())
            err = np.abs(out.cpu().numpy().astype(np.float64) - ref)
            assert np.isfinite(err).all()
            worst = float((err / (mag + 1.0)).max())
            assert worst < 1e-5, (name, d, worst)
            # what the lo operand contributes: x - fp16(x), times the weights
            lo = xt - xt.astype(np.float16).astype(np.float64)
            lo_term = np.abs((lo @ w.T)[:, _col_order()] * _col_scale())
            if name == "onehot":
                big = lo_term > 1e-2
                assert big.mean() > 0.5
                assert (err[big] < 0.1 * lo_term[big]).all(), (name, d, float((err[big] / lo_term[big]).max()))


def _argmax_where_clear(p, p64, tol):
    top = np.sort(p64, axis=1)[:, -2:]
    clear = (top[:, 1] - top[:, 0]) > 2 * tol
    return np.array_equal(p.argmax(1)[clear], p64.argmax(1)[clear])


def test_model_precisions_at_deep_counts(weights, model64, deep_inputs, deep_case):
    """F16X3 within 5e-5 and FP32 within 2e-5 of the float64 network on deep windows, int32 and float32 input, n = 1, 129,
    4 097, and through the fused read from a count tensor; the argmax agrees wherever the float64 margin exceeds the tolerance."""
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupModelForward
    x = deep_inputs["x"]
    g64, z64 = (t.numpy() for t in model64.predict64(x))
    for prec, tol in ((_lib.PREC_F16X3, F16X3_ATOL), (_lib.PREC_FP32, FP32_ATOL)):
        fwd = PileupModelForward(weights, prec)
        for n in (1, 129, 4097):
            for dt in (torch.int32, torch.float32):
                g, z = fwd(torch.from_numpy(x[:n]).cuda().to(dt))
                g, z = g.cpu().numpy(), z.cpu().numpy()
                err = max(float(np.abs(g - g64[:n]).max()), float(np.abs(z - z64[:n]).max()))
                assert err < tol, (prec, n, dt, err)
                assert _argmax_where_clear(g, g64[:n], tol) and _argmax_where_clear(z, z64[:n], tol), (prec, n, dt)
    # fused read: windows are row spans of a deep count tensor (the 8000x contig, cap off)
    _, _, res, _ = deep_case("8000x_nocap")
    counts = torch.from_numpy(res.counts).cuda()
    pos = torch.from_numpy((res.positions - 1).astype(np.int32)).cuda()
    n = len(res.positions)
    gr, zr = (t.numpy() for t in model64.predict64(res.windows))
    # and a synthetic count tensor of deep rows (one-hot and dense), sites anywhere in it
    rng = np.random.default_rng(21)
    syn = np.concatenate([_onehot_rows(300, 22).reshape(-1, 18), _dense_rows(300, 23).reshape(-1, 18)])
    syn = np.ascontiguousarray(syn[rng.permutation(len(syn))])
    spos = np.sort(rng.choice(np.arange(16, len(syn) - 16), 4097, replace=False)).astype(np.int32)
    sw = syn[spos[:, None] + np.arange(-16, 17)]
    gs, zs = (t.numpy() for t in model64.predict64(sw))
    fwd = PileupModelForward(weights, _lib.PREC_F16X3)
    for cnt, p, nn, g0, z0 in ((counts, pos, n, gr, zr), (torch.from_numpy(syn).cuda(), torch.from_numpy(spos).cuda(), 4097, gs, zs)):
        g, z = fwd.from_counts(cnt, 0, p, nn)
        g, z = g.cpu().numpy(), z.cpu().numpy()
        err = max(float(np.abs(g - g0).max()), float(np.abs(z - z0).max()))
        assert err < F16X3_ATOL, err
        assert _argmax_where_clear(g, g0, F16X3_ATOL) and _argmax_where_clear(z, z0, F16X3_ATOL)


def test_single_pass_mode_at_deep_counts(weights, deep_inputs, small_case):
    """NSNP_PREC_F16X1 (the single pass drops the low bits of counts above 2048): with a few thousand deep windows among ordinary
    ones every argmax equals the three-pass path's, |dp| < 5e-3, and the deep sites carry the three-pass values (they are
    re-evaluated); with more deep windows than one call re-evaluates, the call reports NSNP_E_OVERFLOW.  A silent flip fails."""
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupModelForward
    tc = PileupModelForward(weights, _lib.PREC_F16X3)
    base = np.tile(small_case["windows"], (5, 1, 1))[:20_001]
    assert np.abs(base).max() <= 2048
    slots = np.zeros(len(base), bool)
    slots[np.random.default_rng(31).choice(len(base), 3000, replace=False)] = True
    base[slots] = np.tile(deep_inputs["x"], (2, 1, 1))[:3000]
    deep = (np.abs(base) > 2048).any(axis=(1, 2))                       # some real 8000x windows stay below 2048
    assert 2500 < deep.sum() <= 3000
    x = torch.from_numpy(base).cuda().contiguous()
    g3, z3 = tc(x)
    dm = torch.from_numpy(deep).cuda()
    for inp in (x, x.float()):
        x1 = PileupModelForward(weights, _lib.PREC_F16X1)
        g1, z1 = x1(inp)
        assert int(deep.sum()) <= x1.reevaluated() <= 4096
        assert torch.equal(g1.argmax(1), g3.argmax(1)) and torch.equal(z1.argmax(1), z3.argmax(1))
        err = max(float((g1 - g3).abs().max()), float((z1 - z3).abs().max()))
        assert 1e-5 < err < F16X1_ATOL, err
        assert torch.equal(g1[dm], g3[dm]) and torch.equal(z1[dm], z3[dm])
    # all deep: more sites to re-evaluate than one call takes
    xd = torch.from_numpy(np.tile(deep_inputs["x"], (5, 1, 1))[:20_001]).cuda().contiguous()
    x1 = PileupModelForward(weights, _lib.PREC_F16X1)
    x1(xd)
    with pytest.raises(_lib.NsnpError) as e:
        x1.reevaluated()
    assert e.value.code == _lib.E_OVERFLOW


# ------------------------------------------------------------------------------------------------ records and VCF text
def _oracle_rows(model64, contig, ref, res):
    from oracle.s2_restate import predict_vcf
    up = np.char.upper(ref[res.positions - 1].view("S1")).view(np.uint8)
    return predict_vcf(model64, contig, res.positions, up, res.windows).splitlines()


def _compare_rows(got, ref):
    """test_gpu_dropin._compare_vcf on record lines: CHROM POS ID REF ALT FILTER INFO FORMAT, GT DP AF identical; QUAL within
    the last printed digit on at most 3 % of the rows."""
    assert len(got) == len(ref), (len(got), len(ref))
    nq = 0
    for a, b in zip(got, ref):
        fa, fb = a.split("\t"), b.split("\t")
        assert fa[:5] == fb[:5] and fa[6:9] == fb[6:9], (a, b)
        sa, sb = fa[9].split(":"), fb[9].split(":")
        assert sa[0] == sb[0] and sa[2:] == sb[2:], (a, b)
        if fa[5] != fb[5]:
            nq += 1
            assert abs(float(fa[5]) - float(fb[5])) <= 0.0101
    assert nq <= 0.03 * len(ref)


@pytest.mark.parametrize("name", ["1000x", "8000x_nocap"])
def test_deep_records_and_text(engines, weights, model64, deep_case, name):
    """RegionRunner(records=True), fused and unfused, one region and several: GPU text == host text of the same records, and the
    rows equal the oracle's (DP in the thousands)."""
    from nanosnp_b200.caller import call_contig, call_contig_text
    from nanosnp_b200.pipeline import PileupModelForward
    from nanosnp_b200.runner import RegionRunner
    ref, reads, res, md = deep_case(name)
    want = _oracle_rows(model64, "chrM", ref, res)
    assert max(int(l.split("\t")[9].split(":")[2]) for l in want) > 300
    outs = []
    for fused in (True, False):
        runner = RegionRunner(engines[md], PileupModelForward(weights, 1), records=True, fused=fused)
        for region_len in (1 << 30, 5_000):
            host = io.BytesIO()
            call_contig(runner, reads, ref, "chrM", host, 1000, region_len)
            text = io.BytesIO()
            info = call_contig_text(runner, reads, ref, "chrM", text, 1000, region_len)
            assert text.getvalue() == host.getvalue(), (fused, region_len)
            assert info["sites"] == len(res.positions)
            outs.append(host.getvalue())
    assert all(o == outs[0] for o in outs)
    _compare_rows(outs[0].decode().splitlines(), want)


def test_predict_cli_bam_with_deep_contig(tmp_path, model64, deep_case):
    """`python -m nanosnp_b200.predict` over a BAM holding a 30x contig and the 1000x chrM-like contig runs to the end and writes
    the oracle's rows for both."""
    from nanosnp_b200 import predict as P
    from nanosnp_b200.bam import write_bam
    from nanosnp_b200.synth import SynthConfig, generate_host
    from oracle import pyoracle
    ref_m, reads_m, res_m, _ = deep_case("1000x")
    cfg = SynthConfig(contig_len=120_000, coverage=30.0, contig="ctg30", seed_ref=71, seed_var=72, seed_reads=73, len_median=4000, len_min=300)
    ref_a, reads_a = generate_host(cfg)
    mp = str(tmp_path / "a.mpileup")
    pyoracle.mpileup_text(reads_a, "ctg30", mp)
    res_a = pyoracle.s1_restate(mp, "ctg30", ref_a)
    fa = str(tmp_path / "ref.fa")
    pyoracle.write_fasta(fa, {"ctg30": ref_a, "chrM": ref_m})
    bam = str(tmp_path / "reads.bam")
    write_bam(bam, [("ctg30", len(ref_a)), ("chrM", len(ref_m))], {"ctg30": reads_a, "chrM": reads_m})
    out = str(tmp_path / "out.vcf")
    cfgp = str(P.__file__).replace("predict.py", "config/ont_pileup.yaml")
    P.main(["-config", cfgp, "-model_path", str(GOLDEN / "ont_pileup_weights.npz"), "-data", bam, "-reference", fa, "-output", out])
    rows = [l for l in open(out).read().splitlines() if not l.startswith("#")]
    for ctg, ref, res in (("ctg30", ref_a, res_a), ("chrM", ref_m, res_m)):
        _compare_rows([l for l in rows if l.split("\t")[0] == ctg], _oracle_rows(model64, ctg, ref, res))
