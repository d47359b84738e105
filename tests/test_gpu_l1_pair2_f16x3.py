"""The two-group three-pass layer-1 kernel (lstm1_pair2x3_kernel) against pinned bytes: every probability must stay the same.

lstm1_pair2x3_kernel replaced a one-group kernel that computed the same MMA order and cell arithmetic.  The SHA-256
digests below were recorded from both kernels on the same seeded inputs, and the two agreed on every array, so they pin
the bytes of that reference.  Covered: batch sizes around the 128-site tile, the 512-site tile quad of a cluster and the
75 776-site host chunk; a whole 12.5 Mb region of the bench workload through the fused count-tensor entry point
(nsnp_pileup_model_forward_sites); and NSNP_PREC_F16X1 (lstm1_pair2_kernel) on a batch whose low-margin sites are
re-evaluated by a three-pass batch.
"""
import hashlib
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
SIZES = (1, 127, 128, 129, 511, 512, 513, 4096, 75_775, 75_776, 75_777)
# SHA-256 of dtype, shape and bytes of each output (_digest)
DIGESTS = {
    "gt_1": "81def334a83f8b81d6a02b2a9198df2814c9b123e5e4e76160931f4ab86a3dd5",
    "zy_1": "69ca434dc7cd8b6c0937af22583cab1f213b5dfe60fa10e397bb05adde5a684a",
    "gt_127": "7d8b09c22fc67cf986b13540eaacfd3ebc9ee3d54d0f7b5060b17201e2dbbe91",
    "zy_127": "451a27faada7a7196736796752db8dfddd2dc078ff41cdc6480a24d4c84639e6",
    "gt_128": "d631f8ba9e4543a7eab100057db078836377421c6988872e0997641a5d4809f2",
    "zy_128": "3a5075430b8aceb5f73414b883a004bc3f4880d226c2278f5d19bfa971ab8db8",
    "gt_129": "5b3d8d7075a8bcec3dfe555a263ce57a860928065908fb678edaf662490f5e50",
    "zy_129": "c358f02813d3fadf1a6d14b5c779b6827077c657338db68aba717d5f53dde3c2",
    "gt_511": "f3c5ea7fe44bd1f7f0c7161c46c2e6a692531ad17fb0ad31020e6f433cf31085",
    "zy_511": "73ad81167dc14807367b0da3203536d9807f7599e694282719fbd361c65d1e3c",
    "gt_512": "9586c2d06a21a39ec2e709c27286a2d5a08fc7069110294914eaf92ad58e2e06",
    "zy_512": "833bad4c036115e7ea6ad1e1814721666be0739e6c6d19df662e410b80057169",
    "gt_513": "ef4ec0eb5157e30adeb67eaa1cb7e9980d4b84e93764eba0ba7267f8ab52a3de",
    "zy_513": "d1aa93d9363300cbcdcfc6bc16cb02ca2d62c82c00c6156e9392dac7d2a4d4f7",
    "gt_4096": "30be5ccb5c8cce932c63c7a53896e3c1684966f06e419779b05326a38502329a",
    "zy_4096": "f373467db02d08c92301acc217efb575fd502099550a7d317581e1556e8fd535",
    "gt_75775": "e351634a63b4ee5371465fc8f0e1ffad2736a8a8b7039991c66b2d0e86c36d0c",
    "zy_75775": "254fe2ba042c170893eda98b8aece9275087b6a28c2a6ad7a2d0c40b19435e76",
    "gt_75776": "583c0b4a9e39fc28d4ed0d28c7d13cf8697e8182c5a7cd5cf753c36ed2e23892",
    "zy_75776": "caa4ef9268241823696b6b23400f4c9692a79ac2d79ad388f4e855dbff5deeb6",
    "gt_75777": "4af28b2ed44c93fbccc55b6a5d44108bd42e0e9085e6040daf1778ab154929be",
    "zy_75777": "95c72f029fb17cae74158134bfa3eef05b6e1288db2ae1a40eac2ef761aa702c",
    "region_gt": "fb9c5a4d57327f0cb30d86576bc7447a3ba4b411a415563494a386d130f1dff2",
    "region_zy": "3a4d379eea516b8fde0f0315b298c48b3babec2b093ad6cc4a23fe3c240af2e5",
    "x1_gt": "f1416f6b978ec91445f0f20fe48a32f9f9381052d48db58411a2d349b42ffec7",
    "x1_zy": "cd139774fe480626f7a8cb4c3973bf756e8ca5b3b93bd23d086c4b3e5e465045",
}
X1_LOW = 4                            # low-margin sites of the f16x1 batch, re-evaluated in three passes


def _windows(golden, n, seed=None):
    """n int32 windows: the golden small case's windows, repeated; with a seed, plus count noise so that every site differs."""
    base = np.load(golden / "s1_small.npz")["windows"].astype(np.int32)
    x = np.tile(base, ((n + len(base) - 1) // len(base), 1, 1))[:n]
    return x if seed is None else x + np.random.default_rng(seed).integers(0, 4, size=x.shape, dtype=np.int32)


def _same_bytes(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def _digest(a):
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def outputs():
    """Every output this file checks, on the seeded inputs the digests were recorded from."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupEngine, PileupModelForward, PileupModelWeights
    from nanosnp_b200.runner import RegionRunner
    from nanosnp_b200.shard import plan_regions
    from nanosnp_b200.synth import generate_device
    from oracle.s2_restate import load_weights_npz
    from test_gpu_scale import bench_cfg, region_reads

    golden = ROOT / "tests" / "golden"
    w = PileupModelWeights(*load_weights_npz(golden / "ont_pileup_weights.npz"), device="cuda:0")
    tc = PileupModelForward(w, _lib.PREC_F16X3)
    res = {}
    x = torch.from_numpy(_windows(golden, max(SIZES), seed=5)).cuda()
    for n in SIZES:
        g, z = tc(x[:n].contiguous())
        res[f"gt_{n}"], res[f"zy_{n}"] = g.cpu().numpy(), z.cpu().numpy()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        tc(x[:4096].contiguous())
        torch.cuda.synchronize()
    res["kernels"] = " ".join(sorted({e.key for e in prof.key_averages()}))
    # single pass + three-pass re-evaluation of the low-margin sites; the real windows of the small case keep the
    # low-margin count within the re-evaluation batch
    x1 = PileupModelForward(w, _lib.PREC_F16X1)
    g, z = x1(torch.from_numpy(_windows(golden, 20_001)).cuda())
    res["x1_gt"], res["x1_zy"], res["x1_low"] = g.cpu().numpy(), z.cpu().numpy(), x1.reevaluated()
    # region 0 of the bench workload, windows read straight from the count tensor
    eng = PileupEngine("cuda:0")
    cfg = bench_cfg()
    ref, reads = generate_device(cfg, eng.device)
    rg = plan_regions([(cfg.contig, cfg.contig_len)], 12_500_000)[0]
    rd = region_reads(reads, reads.pos.cpu().numpy(), rg, int(cfg.len_max * 1.3) + 1000)
    out = RegionRunner(eng, tc, records=True).run_device(rd, ref, rg)
    res["region_gt"], res["region_zy"] = out.gt[:out.n].cpu().numpy(), out.zy[:out.n].cpu().numpy()
    return res


def test_runs_the_two_group_kernel(outputs):
    assert "lstm1_pair2x3_kernel" in outputs["kernels"], outputs["kernels"]


@pytest.mark.parametrize("n", SIZES)
def test_batch_sizes_bit_identical(outputs, n):
    for k in (f"gt_{n}", f"zy_{n}"):
        assert _digest(outputs[k]) == DIGESTS[k], k
    assert np.isfinite(outputs[f"gt_{n}"]).all()


def test_bench_region_bit_identical(outputs):
    assert outputs["region_gt"].shape[0] > 400_000
    for k in ("region_gt", "region_zy"):
        assert _digest(outputs[k]) == DIGESTS[k], k


def test_single_pass_reevaluation_bit_identical(outputs):
    assert int(outputs["x1_low"]) == X1_LOW > 0
    for k in ("x1_gt", "x1_zy"):
        assert _digest(outputs[k]) == DIGESTS[k], k
