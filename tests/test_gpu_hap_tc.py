"""HaplotypeModel s5 on the tensor cores (precision "f16x3", csrc/haplotype_tc.cu) against the float64 oracle network and the fp32
CUDA path.  Weights are the seeded oracle's (the shipped checkpoints are missing).  With the golden seed the probabilities are
nearly uniform (max gt ~0.11), so every accuracy check also runs with all weights x 4, which saturates gates and spreads them."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

TOL = 5e-5


def _lib():
    from nanosnp_b200 import _lib as L
    return L


def weight_sets(seed):
    from oracle.hap_restate import HaplotypeModelOracle
    m = HaplotypeModelOracle(seed=seed)
    sd = m.state_dict()
    return {"seed": sd, "x4": {k: v * 4 for k, v in sd.items()}}


def oracle64(sd, xp, xh):
    """float64 evaluation of the oracle network on the device (inputs: device tensors)."""
    import torch
    from oracle.hap_restate import HaplotypeModelOracle
    m = HaplotypeModelOracle()
    m.load_state_dict(sd)
    m = m.to(xp.device)
    g, z = [], []
    for s in range(0, xp.shape[0], 256):
        a, b = m.predict(xp[s:s + 256], xh[s:s + 256], dtype=torch.float64)
        g.append(a); z.append(b)
    return torch.cat(g), torch.cat(z)


def net(sd, precision):
    from nanosnp_b200 import haplotype as G
    n = G.LSTMNetwork(precision=precision).to("cuda")
    n.load_state_dict(sd)
    return n


def maxdiff(a, b):
    return max(float((x - y).abs().max()) for x, y in zip(a, b))


def assert_rows_match(got: str, want: str):
    """same ctg, pos and GT; QUAL within 0.01 (it is printed with two decimals)"""
    g = [r.split("\t") for r in got.splitlines()]; w = [r.split("\t") for r in want.splitlines()]
    assert len(g) == len(w) > 0
    for a, b in zip(g, w):
        assert a[:3] == b[:3], (a, b)
        assert abs(float(a[3]) - float(b[3])) <= 0.0100001, (a, b)


@pytest.fixture(scope="module")
def hap():
    return np.load(GOLDEN / "hap_small.npz")


@pytest.fixture(scope="module")
def golden_feats(hap):
    from nanosnp_b200 import haplotype as G
    pref = np.stack([G.reference_codes(hap["ref"], np.arange(p - 16, p + 17)) for p in hap["pos"]])
    href = np.stack([G.reference_codes(hap["ref"], q) for q in hap["hap_pos"]])
    fp = G.frequency_features(hap["pileup_seq"], hap["pileup_bq"], hap["pileup_mq"], hap["pileup_hp"], pref)
    fh = G.frequency_features(hap["haplotype_seq"], hap["haplotype_bq"], hap["haplotype_mq"], hap["haplotype_hp"], href)
    return fp, fh


def write_bins(hap, tmp_path):
    d = tmp_path / "bins"; d.mkdir()
    np.savez(d / "ctgH_1_5000.npz", pileup_sequences=hap["pileup_seq"], pileup_hap=hap["pileup_hp"], pileup_baseq=hap["pileup_bq"],
             pileup_mapq=hap["pileup_mq"], haplotype_sequences=hap["haplotype_seq"], haplotype_hap=hap["haplotype_hp"],
             haplotype_baseq=hap["haplotype_bq"], haplotype_mapq=hap["haplotype_mq"],
             candidate_positions=np.array(["ctgH:%d" % p for p in hap["pos"]]),
             haplotype_positions=np.array([["ctgH:%d" % q for q in row] for row in hap["hap_pos"]]))
    fa = tmp_path / "ref.fa"
    fa.write_bytes(b">ctgH some description\n" + bytes(hap["ref"]) + b"\n")
    return d, fa


# ------------------------------------------------------------------------------------------------------------------ CPU
def test_precision_is_validated():
    from nanosnp_b200.haplotype import LSTMNetwork
    with pytest.raises(ValueError):
        LSTMNetwork(precision="f16x1")
    assert LSTMNetwork().precision == "fp32"


def test_tc_symbols_load():
    lib = _lib().load()
    for name in ("nsnp_hap_model_tc_blob_bytes", "nsnp_hap_model_tc_pack_weights", "nsnp_hap_model_tc_workspace_bytes",
                 "nsnp_hap_model_tc_forward", "nsnp_debug_hap_tc_gates"):
        assert name in _lib().SYMBOLS and getattr(lib, name)
    assert lib.nsnp_abi_version() == 2
    assert lib.nsnp_hap_model_tc_blob_bytes() > lib.nsnp_hap_model_blob_bytes()
    assert lib.nsnp_hap_model_tc_workspace_bytes(129) > lib.nsnp_hap_model_tc_workspace_bytes(128) > 0


def test_tc_pack_weights_on_the_host():
    from nanosnp_b200.haplotype import LSTMNetwork
    from oracle.hap_restate import HaplotypeModelOracle
    L = _lib(); lib = L.load()
    nb = lib.nsnp_hap_model_tc_blob_bytes()
    buf = np.zeros(nb, np.uint8)
    assert lib.nsnp_hap_model_tc_pack_weights(C.byref(L.HapWeights()), buf.ctypes.data, nb) == L.E_INVALID    # missing tensors
    n = LSTMNetwork(precision="f16x3")
    n.load_state_dict(HaplotypeModelOracle(seed=1).state_dict())
    with pytest.raises(L.NsnpError):
        n.predict(None, None)                                  # packing needs .to('cuda') first: there is no CPU fallback


def test_tc_forward_without_device():
    import torch
    L = _lib(); lib = L.load()
    if lib.nsnp_device_count() > 0 and torch.cuda.is_available():
        pytest.skip("a GPU is present")
    buf = (C.c_char * 4096)()
    a = C.addressof(buf)
    assert lib.nsnp_hap_model_tc_forward(a, a, a, 4, a, a, a, 1 << 40, None) == L.E_NO_DEVICE
    assert lib.nsnp_debug_hap_tc_gates(a, a, 0, 0, a, 4, None) == L.E_NO_DEVICE
    assert lib.nsnp_hap_model_tc_forward(a, a, a, 0, a, a, a, 0, None) == L.OK
    assert lib.nsnp_hap_model_tc_forward(a, None, a, 4, a, a, a, 1 << 40, None) == L.E_INVALID


# ------------------------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("wset", ["seed", "x4"])
def test_gpu_golden_set_against_float64(hap, golden_feats, wset, tmp_path):
    import torch
    from nanosnp_b200 import haplotype as G
    fp, fh = golden_feats
    sd = weight_sets(int(hap["seed"]))[wset]
    gt, zy = net(sd, "f16x3").predict(fp, fh)
    g64, z64 = oracle64(sd, fp, fh)
    err = maxdiff((gt, zy), (g64.to(gt.device), z64.to(gt.device)))
    assert err < TOL, err
    assert torch.equal(gt.argmax(1).cpu(), g64.argmax(1).cpu()) and torch.equal(zy.argmax(1).cpu(), z64.argmax(1).cpu())
    if wset == "seed":
        assert np.abs(gt.cpu().numpy() - hap["gt"]).max() < TOL and np.abs(zy.cpu().numpy() - hap["zy"]).max() < TOL
        d, fa = write_bins(hap, tmp_path)
        out = tmp_path / "haplotype.csv"
        assert G.predict(net(sd, "f16x3"), str(d), str(fa), 20, 33, 11, str(out), "cuda") == len(hap["pos"])
        assert_rows_match(out.read_text(), (GOLDEN / "hap_small.csv").read_text())


def deep_features(seed=11, depth=40000):
    """features of read matrices 40,000 rows deep with qualities up to 93: every sum channel passes fp16's 65504"""
    import torch
    from nanosnp_b200 import haplotype as G
    g = torch.Generator().manual_seed(seed)
    out = []
    for L in (33, 11):
        n = 3
        seq = torch.randint(1, 5, (n, depth, L), generator=g, dtype=torch.int32)
        seq[torch.rand((n, depth, L), generator=g) < 0.05] = -1
        bq = torch.randint(60, 94, (n, depth, L), generator=g, dtype=torch.int32)
        mq = torch.randint(60, 94, (n, depth, L), generator=g, dtype=torch.int32)
        hp = torch.randint(1, 4, (n, depth, 1), generator=g, dtype=torch.int32).expand(n, depth, L).contiguous()
        seq[1, depth // 2:] = -2                                 # a shallower site: pad rows
        ref = torch.randint(0, 5, (n, L), generator=g, dtype=torch.int32)
        out.append(G.frequency_features(seq, bq, mq, hp, ref))
    fp, fh = out
    big_p = fp[:1].clone(); big_h = fh[:1].clone()              # hand-set rows: channel values up to 1e7
    big_p[0, 5:26] = torch.rand((21, 33), generator=g).to(fp.device) * 1e7
    big_h[0, 5:26] = torch.rand((21, 11), generator=g).to(fh.device) * 1e7
    return torch.cat([fp, big_p]), torch.cat([fh, big_h])


@pytest.mark.gpu
@pytest.mark.parametrize("wset", ["seed", "x4"])
def test_gpu_range_layer0_gates_and_probabilities(wset):
    import torch
    xp, xh = deep_features()
    for x in (xp, xh):
        assert float(x[:3, 10:14].min()) > 65504 and float(x[:3, 18:22].min()) > 65504    # every quality / MAPQ sum beyond fp16
    sd = weight_sets(1)[wset]
    n = net(sd, "f16x3")
    gt, zy = n.predict(xp, xh)
    L = _lib(); lib = L.load()
    for e, (x, pre) in enumerate(((xp, "pileup_encoder"), (xh, "haplotype_encoder"))):
        x = x.contiguous()
        m = x.shape[0]
        for d, sfx in enumerate(("", "_reverse")):
            w = sd[f"{pre}.lstm.weight_ih_l0{sfx}"].double().to(x.device)
            b = (sd[f"{pre}.lstm.bias_ih_l0{sfx}"] + sd[f"{pre}.lstm.bias_hh_l0{sfx}"]).double().to(x.device)
            xt = x[:, :, 0 if d == 0 else x.shape[2] - 1].double()
            want = xt @ w.T + b
            bound = (xt.abs() @ w.abs().T) + b.abs()
            got = torch.empty((m, 1024), dtype=torch.float32, device=x.device)
            L.check(lib.nsnp_debug_hap_tc_gates(n._blob.data_ptr(), x.data_ptr(), e, d, got.data_ptr(), m,
                                                torch.cuda.current_stream().cuda_stream))
            torch.cuda.synchronize()
            rel = float(((got.double() - want).abs() / (bound + 1e-30)).max())
            assert rel < 1e-5, (e, d, rel)
    g64, z64 = oracle64(sd, xp, xh)
    err = maxdiff((gt, zy), (g64.to(gt.device), z64.to(gt.device)))
    assert err < TOL, err


def bench_contig_features(mb=2.0, cov=30.0):
    """the s4 path as tools/hap_bench.py builds it: synthetic contig, random HP tags and qualities, a group about every kb"""
    import torch
    from nanosnp_b200 import hap_groups as hg
    from nanosnp_b200 import haplotype as G
    from nanosnp_b200.synth import SynthConfig, generate_device
    dev = torch.device("cuda:0")
    L = int(mb * 1e6)
    ref, reads = generate_device(SynthConfig(contig_len=L, coverage=cov, seed_ref=1000, seed_var=1001, seed_reads=1002), dev)
    g = torch.Generator(device="cpu"); g.manual_seed(7)
    qual = torch.randint(1, 42, (reads.n_bases,), dtype=torch.uint8, generator=g).to(dev)
    hp = torch.randint(0, 3, (reads.n_reads,), dtype=torch.uint8, generator=g).to(dev)
    end, end_pm, ck = hg.read_ends(reads, dev)
    al = hg.ContigAlignments(reads, qual, hp, end, end_pm, ck, None, None, dev)
    rng = np.random.default_rng(3)
    pos = np.cumsum(rng.integers(600, 1400, size=L // 1000)); pos = pos[pos < L - 100].astype(np.int64)
    q = rng.uniform(2, 60, len(pos)); het = np.ones(len(pos), bool)
    groups = hg.find_adjacent_sites(pos, het, q, 5, 19, 14)
    gm = hg.group_matrices(al, groups, hg.plan_subgroups(groups), 150, 16)
    refh = ref.cpu().numpy()
    cand = gm.positions[:, 5]
    pref = G.reference_codes(refh, cand[:, None] + np.arange(-16, 17)[None, :]); href = G.reference_codes(refh, gm.positions)
    d = min(gm.hap[0].shape[1], int(3 * cov))
    return (G.frequency_features(gm.pile[0][:, :d], gm.pile[2][:, :d], gm.pile[3][:, :d], gm.pile[1][:, :d], pref, dev),
            G.frequency_features(gm.hap[0][:, :d], gm.hap[2][:, :d], gm.hap[3][:, :d], gm.hap[1][:, :d], href, dev))


@pytest.fixture(scope="module")
def contig_feats():
    return bench_contig_features()


@pytest.mark.gpu
@pytest.mark.parametrize("wset", ["seed", "x4"])
def test_gpu_realistic_scale_against_fp32_and_float64(contig_feats, wset):
    import torch
    xp, xh = contig_feats
    n = xp.shape[0]
    assert n > 500
    sd = weight_sets(1)[wset]
    gt, zy = net(sd, "f16x3").predict(xp, xh)
    g32, z32 = net(sd, "fp32").predict(xp, xh)
    assert maxdiff((gt, zy), (g32, z32)) < TOL
    assert torch.equal(gt.argmax(1), g32.argmax(1)) and torch.equal(zy.argmax(1), z32.argmax(1))
    idx = torch.arange(0, n, max(1, n // 160), device=xp.device)
    assert len(idx) >= 128
    g64, z64 = oracle64(sd, xp[idx], xh[idx])
    assert maxdiff((gt[idx], zy[idx]), (g64.to(gt.device), z64.to(gt.device))) < TOL


@pytest.mark.gpu
def test_gpu_batch_invariance_and_ragged_sizes(golden_feats):
    import torch
    fp, fh = golden_feats
    total = 2 * 4096 + 300                                     # more than two 4096-site chunks
    rep = (total + fp.shape[0] - 1) // fp.shape[0]
    noise = torch.Generator(device="cpu").manual_seed(2)
    xp = (fp.repeat(rep, 1, 1)[:total] * (1 + 0.01 * torch.rand((total, 1, 1), generator=noise)).to(fp.device)).contiguous()
    xh = (fh.repeat(rep, 1, 1)[:total] * (1 + 0.01 * torch.rand((total, 1, 1), generator=noise)).to(fh.device)).contiguous()
    n = net(weight_sets(1)["x4"], "f16x3")
    gt, zy = n.predict(xp, xh)
    g2, z2 = n.predict(xp, xh)
    assert torch.equal(gt, g2) and torch.equal(zy, z2)         # two identical calls, identical bits
    for k in (1, 127, 128, 129, 1000, 4095, 4097, total):
        for off in (0, 77):
            if off + k > total:
                continue
            gk, zk = n.predict(xp[off:off + k], xh[off:off + k])
            assert torch.equal(gk, gt[off:off + k]) and torch.equal(zk, zy[off:off + k]), (k, off)


@pytest.mark.gpu
def test_gpu_fused_s4_s5_f16x3_equals_fp32(tmp_path):
    from nanosnp_b200 import haplotype as G
    from nanosnp_b200.bam import write_bam
    from test_hap_groups import GOLD, packed, records, vcf_file
    gold = np.load(GOLD, allow_pickle=False)
    lens = dict(zip([str(c) for c in gold["contigs"]], [int(l) for l in gold["contig_lens"]]))
    bdir = tmp_path / "bams"; bdir.mkdir()
    fa = tmp_path / "ref.fa"
    with open(fa, "wb") as f:
        for ctg in lens:
            rd, aux = packed(records(gold, ctg))
            write_bam(str(bdir / f"{ctg}.bam"), [(ctg, lens[ctg])], {ctg: rd}, aux={ctg: aux})
            f.write(b">" + ctg.encode() + b"\n" + bytes(gold[f"ref_{ctg}"]) + b"\n")
    vcf = vcf_file(gold, tmp_path)
    sd = weight_sets(5)["seed"]
    outs = []
    for prec in ("fp32", "f16x3"):
        out = tmp_path / f"{prec}.csv"
        G.predict_from_bams(net(sd, prec), vcf, str(bdir), str(fa), str(out), batch_size=7, max_depth=24, threads=3)
        outs.append("\n".join(sorted(out.read_text().splitlines())))
    assert_rows_match(outs[1], outs[0])


@pytest.mark.gpu
def test_gpu_errors_and_cli(hap, golden_feats, tmp_path):
    import subprocess
    import torch
    fp, fh = golden_feats
    L = _lib(); lib = L.load()
    sd = weight_sets(int(hap["seed"]))["seed"]
    n = net(sd, "f16x3")
    n.predict(fp[:1], fh[:1])                                  # packs the blob
    m = fp.shape[0]
    need = lib.nsnp_hap_model_tc_workspace_bytes(m)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    gt = torch.empty((m, 10), device="cuda"); zy = torch.empty((m, 3), device="cuda")
    args = [n._blob.data_ptr(), fp.data_ptr(), fh.data_ptr(), m, gt.data_ptr(), zy.data_ptr(), ws.data_ptr()]
    assert lib.nsnp_hap_model_tc_forward(*args, need - 1, None) == L.E_WORKSPACE
    for i in (0, 1, 2, 4, 5, 6):
        bad = list(args); bad[i] = None
        assert lib.nsnp_hap_model_tc_forward(*bad, need, None) == L.E_INVALID
    assert lib.nsnp_hap_model_tc_forward(*args[:3], 0, *args[4:], 0, None) == L.OK
    assert lib.nsnp_hap_model_tc_forward(*args[:3], -1, *args[4:], need, None) == L.E_INVALID
    assert lib.nsnp_hap_model_tc_forward(*args, need, None) == L.OK
    torch.cuda.synchronize()
    # the CLI with --precision f16x3 writes the golden rows
    d, fa = write_bins(hap, tmp_path)
    ckpt = tmp_path / "model.pt"
    torch.save(sd, ckpt)
    cfg = tmp_path / "hap.yaml"
    cfg.write_text("model:\n  pileup_dim: 105\n  haplotype_dim: 105\n  pileup_length: 33\n  haplotype_length: 11\n  hidden_size: 256\n"
                   "  lstm_layers: 3\n  gt_num_class: 10\n  zy_num_class: 3\n")
    out = tmp_path / "cli.csv"
    env = dict(os.environ, PYTHONPATH=str(ROOT))
    subprocess.run([sys.executable, "-m", "nanosnp_b200.haplotype", "-config", str(cfg), "-model_path", str(ckpt), "-bin_paths", str(d),
                    "-reference_path", str(fa), "-output", str(out), "-batch_size", "20", "--precision", "f16x3"], check=True, env=env, cwd=str(ROOT))
    assert_rows_match(out.read_text(), (GOLDEN / "hap_small.csv").read_text())
