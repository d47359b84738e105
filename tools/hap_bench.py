#!/usr/bin/env python
"""BASELINE configs[4] measurement: HaplotypeModel s4 (read matrices) + s5 (features, model) on one synthetic contig.
usage: tools/hap_bench.py [mb] [coverage] [reps]   -> one JSON line (groups/s per stage, device-timed; the model at both
precisions, fp32 and the tensor-core f16x3, timed alternately after warm-up)"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from nanosnp_b200 import hap_groups as hg
from nanosnp_b200 import haplotype as G
from nanosnp_b200 import _lib
from nanosnp_b200.synth import SynthConfig, generate_device
import ctypes as C

mb = float(sys.argv[1]) if len(sys.argv) > 1 else 12.5
cov = float(sys.argv[2]) if len(sys.argv) > 2 else 30.0
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
dev = torch.device("cuda:0")
L = int(mb * 1e6)
cfg = SynthConfig(contig_len=L, coverage=cov, seed_ref=1000, seed_var=1001, seed_reads=1002)
ref, reads = generate_device(cfg, dev)
n = reads.n_reads
g = torch.Generator(device="cpu"); g.manual_seed(7)
qual = torch.randint(1, 42, (reads.n_bases,), dtype=torch.uint8, generator=g).to(dev)
hp = torch.randint(0, 3, (n,), dtype=torch.uint8, generator=g).to(dev)
end, end_pm, ck = hg.read_ends(reads, dev)
al = hg.ContigAlignments(reads, qual, hp, end, end_pm, ck if os.environ.get("HAP_NO_CK") is None else None, None, None, dev)

# sites every ~1 kb, a third of them low-quality candidates (human: ~1 het SNP per kb)
rng = np.random.default_rng(3)
pos = np.cumsum(rng.integers(600, 1400, size=L // 1000)); pos = pos[pos < L - 100].astype(np.int64)
q = rng.uniform(2, 60, len(pos)); het = np.ones(len(pos), bool)
groups = hg.find_adjacent_sites(pos, het, q, 5, 19, 14)
subs = hg.plan_subgroups(groups)

def timed(f):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize(); e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter(); e0.record(); r = f(); e1.record(); torch.cuda.synchronize()
        ts.append((e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))
    return r, min(t[0] for t in ts), min(t[1] for t in ts)

gm, ms_mat, wall_mat = timed(lambda: hg.group_matrices(al, groups, subs, 150, 16))
G_ = len(gm.positions)
refh = ref.cpu().numpy()
cand = gm.positions[:, 5]
pref = G.reference_codes(refh, cand[:, None] + np.arange(-16, 17)[None, :]); href = G.reference_codes(refh, gm.positions)
d = min(gm.hap[0].shape[1], int(3 * cov))
def feats():
    return (G.frequency_features(gm.pile[0][:, :d], gm.pile[2][:, :d], gm.pile[3][:, :d], gm.pile[1][:, :d], pref, dev),
            G.frequency_features(gm.hap[0][:, :d], gm.hap[2][:, :d], gm.hap[3][:, :d], gm.hap[1][:, :d], href, dev))
(xp, xh), ms_feat, _ = timed(feats)
from oracle.hap_restate import HaplotypeModelOracle          # weights only (random init: the checkpoint is not shipped)
sd = HaplotypeModelOracle(seed=1).state_dict()
net = G.LSTMNetwork().to(dev); net.load_state_dict(sd)
net_tc = G.LSTMNetwork(precision="f16x3").to(dev); net_tc.load_state_dict(sd)
# both precisions in the same run: warm up each, then alternate the timed calls
(g32, z32), (gtc, ztc) = net.predict(xp, xh), net_tc.predict(xp, xh)
ms32, mstc = [], []
for _ in range(reps):
    ms32.append(timed(lambda: net.predict(xp, xh))[1]); mstc.append(timed(lambda: net_tc.predict(xp, xh))[1])
ms_model, ms_tc = min(ms32), min(mstc)
dp = max(float((gtc - g32).abs().max()), float((ztc - z32).abs().max()))
# pruned multiply-adds per site: every LSTM step the model needs (the last layer stops at the centre) plus the tail
mac = sum(steps * 2 * 1024 * (in_dim + 256) for Lx in (33, 11) for steps, in_dim in ((Lx, 105), (Lx, 512), (Lx // 2 + 1, 512)))
mac += 2 * 256 * 512 + 256 * 512 + 13 * 256
try:
    import subprocess
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
except OSError:
    power = "unknown"
out = {"workload": f"synthetic {mb} Mb contig at {cov}x, HP tags + qualities random, 1 site / kb, QUAL<19 candidates", "reads": n,
       "groups": int(len(groups)), "groups_out": int(G_), "rows_cap": int(gm.hap[0].shape[1]), "mean_depth": float(gm.depth.mean()),
       "s4_matrices_ms": ms_mat, "s4_matrices_wall_ms": wall_mat, "s5_features_ms": ms_feat, "s5_model_ms": ms_model,
       "groups_per_s_s4": G_ / (wall_mat * 1e-3), "groups_per_s_s4_s5": G_ / ((wall_mat + ms_feat + ms_model) * 1e-3),
       "s5_model_tc_ms": ms_tc, "tc_speedup": ms_model / ms_tc, "mac_per_site_pruned": mac,
       "tflops_fp32": 2 * mac * G_ / (ms_model * 1e-3) / 1e12, "tflops_tc": 2 * mac * G_ / (ms_tc * 1e-3) / 1e12,
       "max_abs_dp_tc_vs_fp32": dp, "gpu": torch.cuda.get_device_name(dev), "power_limit": power}
print(json.dumps(out))
