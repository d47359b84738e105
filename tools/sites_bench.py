"""Genotyping given sites (`--sites`) on the bench workload: device-resident step time per site list, alternated with the
unrestricted step in the same run.

    python tools/sites_bench.py [--steps 5] [--warmup 2] [--out profiles/r03_sites.json]

Workload: bench.py's 100 Mb / 30x synthetic contig (same generator and seeds, bench.synth_cfg), 12.5 Mb regions, f16x3,
device-resident reads (bench.region_slices).  Site lists: (a) one site per 30 bp on average (dbSNP-like density, ~3.3 M
sites), (b) one per kb, (c) a 500-site panel.  A site list is a set of 1-bp intervals, so every unit hands the GPU its
sites as intervals and the GPU computes only the pileup tiles near them.  Stage times come from CUDA events around each
stage (runner.StageTimer); sites/s counts the called sites (listed sites with a full 33-row window and an ACGT centre).
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def site_lists(L, seed=23):
    from nanosnp_b200.targets import site_intervals
    rng = np.random.default_rng(seed)
    return {"a_per_30bp": site_intervals(rng.choice(L, L // 30, replace=False)),
            "b_per_kb": site_intervals(np.arange(0, L, 1000) + rng.integers(0, 1000, -(-L // 1000))),
            "c_panel_500": site_intervals(rng.choice(L, 500, replace=False))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--contig-mb", type=float, default=100.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupEngine, PileupModelForward, PileupModelWeights
    from nanosnp_b200.runner import RegionRunner, StageTimer
    from nanosnp_b200.shard import listed_tiles, plan_regions, plan_target_units
    from nanosnp_b200.synth import generate_device
    from target_bench import gpu_info
    if not torch.cuda.is_available():
        raise SystemExit("sites_bench.py: no CUDA device (there is no CPU path)")
    dev = torch.device("cuda", 0)
    bargs = argparse.Namespace(coverage=30.0)
    L = int(args.contig_mb * 1e6)
    region_len = 12_500_000
    cfg = bench.synth_cfg(bargs, 0, L)
    ref, reads = generate_device(cfg, dev)
    enc, fwd = bench.load_weights(None)
    runner = RegionRunner(PileupEngine(dev), PileupModelForward(PileupModelWeights(enc, fwd, device=dev), _lib.PREC_F16X3), records=True)
    alg = {"pileup": 0.0, "n_bases": 0, "n_cigar": 0, "n_reads": 0}
    full_regions = plan_regions([(cfg.contig, L)], region_len)
    work = {None: [(rg, rd, None) for rg, rd in zip(full_regions, bench.region_slices(reads, full_regions, cfg, dev, alg))]}
    lists = site_lists(L)
    tiles = {}
    for name, iv in lists.items():
        units, ivs = plan_target_units([(cfg.contig, L)], {cfg.contig: iv}, region_len)
        slices = bench.region_slices(reads, units, cfg, dev, dict(alg))
        work[name] = [(rg, rd, u) for rg, rd, u in zip(units, slices, ivs)]
        tiles[name] = int(sum(len(listed_tiles(rg, u)) for rg, _, u in work[name]))
    del reads
    torch.cuda.empty_cache()
    gpu = gpu_info()                        # card name and power limit, read in the same run as the timings

    def step(key, timer=None):
        n = 0
        for rg, rd, u in work[key]:
            n += runner.run_device(rd, ref, rg, timer, targets=u, sites=key is not None).n
        return n

    res = {name: {"ms": [], "stage_ms": None} for name in [None] + list(lists)}
    for key in res:
        for _ in range(args.warmup):
            step(key)
    torch.cuda.synchronize()
    # alternate: every list once per round, forward on even rounds and reversed on odd ones (as tools/target_bench.py)
    for it in range(args.steps):
        for key in (list(res) if it % 2 == 0 else list(res)[::-1]):
            tm = StageTimer(True)
            l0 = runner.launches
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n = step(key, tm)
            e1.record()
            torch.cuda.synchronize()
            r = res[key]
            r["ms"].append(e0.elapsed_time(e1))
            r["sites"], r["launches"] = n, runner.launches - l0
            st = tm.totals_ms()
            r["stage_ms"] = {k: r["stage_ms"][k] + st[k] for k in st} if r["stage_ms"] else st
    out = {"gpu": gpu, "workload": {"contig_mb": args.contig_mb, "coverage": 30.0, "seeds": "bench.synth_cfg rank 0",
                                    "region_len": region_len, "precision": "f16x3", "steps": args.steps,
                                    "timing": "CUDA events around a device-resident step (reads already on the GPU)"},
           "lists": {}}
    base = float(np.median(res[None]["ms"]))
    for key, r in res.items():
        name = "unrestricted" if key is None else key
        iv = None if key is None else lists[key]
        ms = float(np.median(r["ms"]))
        out["lists"][name] = {
            "ms_per_step_median": ms, "ms_per_step": [round(x, 3) for x in r["ms"]], "ratio_to_unrestricted": ms / base,
            "listed_sites": None if iv is None else int((iv[:, 1] - iv[:, 0]).sum()), "called_sites": r["sites"],
            "called_sites_per_s": r["sites"] / (ms / 1e3), "launches_per_step": r["launches"], "units": len(work[key]),
            "listed_tiles": None if key is None else tiles[key],
            "stage_ms_per_step": {k: v / args.steps for k, v in r["stage_ms"].items() if k in ("pileup", "select", "gather", "model")}}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
