"""The two-group three-pass layer-1 kernel (lstm1_pair2x3_kernel, the default) against the one-group kernel it replaces
(lstm_tc_kernel<1,2,4>, NSNP_L1_VARIANT=0): every probability must be the same bytes.

The variant is read once per process, so each variant runs this file as a script in its own process on the same seeded
inputs and writes its outputs to a .npz; the tests compare the two files.  Covered: batch sizes around the 128-site tile,
the 512-site tile quad of a cluster and the 75 776-site host chunk; a whole 12.5 Mb region of the bench workload through
the fused count-tensor entry point (nsnp_pileup_model_forward_sites); and NSNP_PREC_F16X1 on a batch whose low-margin sites
are re-evaluated by a three-pass batch.
"""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
SIZES = (1, 127, 128, 129, 511, 512, 513, 4096, 75_775, 75_776, 75_777)


def _windows(golden, n, seed=None):
    """n int32 windows: the golden small case's windows, repeated; with a seed, plus count noise so that every site differs."""
    base = np.load(golden / "s1_small.npz")["windows"].astype(np.int32)
    x = np.tile(base, ((n + len(base) - 1) // len(base), 1, 1))[:n]
    return x if seed is None else x + np.random.default_rng(seed).integers(0, 4, size=x.shape, dtype=np.int32)


def _run(out_path):
    """One process, one layer-1 variant: write every output this file compares to out_path."""
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
    res["kernels"] = np.array(sorted({e.key for e in prof.key_averages()}))
    # single pass + three-pass re-evaluation of the low-margin sites (that batch runs the variant under test); the real
    # windows of the small case keep the low-margin count within the re-evaluation batch
    x1 = PileupModelForward(w, _lib.PREC_F16X1)
    g, z = x1(torch.from_numpy(_windows(golden, 20_001)).cuda())
    res["x1_gt"], res["x1_zy"], res["x1_low"] = g.cpu().numpy(), z.cpu().numpy(), np.array(x1.reevaluated())
    # region 0 of the bench workload, windows read straight from the count tensor
    eng = PileupEngine("cuda:0")
    cfg = bench_cfg()
    ref, reads = generate_device(cfg, eng.device)
    rg = plan_regions([(cfg.contig, cfg.contig_len)], 12_500_000)[0]
    rd = region_reads(reads, reads.pos.cpu().numpy(), rg, int(cfg.len_max * 1.3) + 1000)
    out = RegionRunner(eng, tc, records=True).run_device(rd, ref, rg)
    res["region_gt"], res["region_zy"] = out.gt[:out.n].cpu().numpy(), out.zy[:out.n].cpu().numpy()
    np.savez(out_path, **res)


@pytest.fixture(scope="module")
def variants(tmp_path_factory):
    d = tmp_path_factory.mktemp("l1_variants")
    res = {}
    for v in ("0", "1"):
        env = dict(os.environ, NSNP_L1_VARIANT=v, PYTHONPATH=str(ROOT))
        r = subprocess.run([sys.executable, __file__, str(d / f"v{v}.npz")], env=env, capture_output=True, text=True, timeout=1200)
        assert r.returncode == 0, r.stderr[-3000:]
        res[v] = dict(np.load(d / f"v{v}.npz"))
    return res


def _same_bytes(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def test_each_variant_runs_its_own_kernel(variants):
    old, new = (" ".join(variants[v]["kernels"]) for v in ("0", "1"))
    assert "lstm_tc_kernel" in old and "lstm1_pair2x3_kernel" not in old
    assert "lstm1_pair2x3_kernel" in new and "lstm_tc_kernel" not in new


@pytest.mark.parametrize("n", SIZES)
def test_batch_sizes_bit_identical(variants, n):
    for k in (f"gt_{n}", f"zy_{n}"):
        assert _same_bytes(variants["0"][k], variants["1"][k]), k
    assert np.isfinite(variants["1"][f"gt_{n}"]).all()


def test_bench_region_bit_identical(variants):
    assert variants["1"]["region_gt"].shape[0] > 400_000
    for k in ("region_gt", "region_zy"):
        assert _same_bytes(variants["0"][k], variants["1"][k]), k


def test_single_pass_reevaluation_bit_identical(variants):
    assert int(variants["0"]["x1_low"]) == int(variants["1"]["x1_low"]) > 0
    for k in ("x1_gt", "x1_zy"):
        assert _same_bytes(variants["0"][k], variants["1"][k]), k


if __name__ == "__main__":
    _run(sys.argv[1])
