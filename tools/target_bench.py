"""Targeted calling (`--bed` / `--region`) on the bench workload: device-resident step time per target set, alternated with
the unrestricted step in the same run, plus one indexed-BAM run from BAM to VCF.

    python tools/target_bench.py [--steps 5] [--warmup 3] [--out profiles/r03_targets.json]

Workload: bench.py's 100 Mb / 30x synthetic contig (same generator and seeds, bench.synth_cfg), 12.5 Mb regions, f16x3,
device-resident reads (bench.region_slices).  Target sets: (a) one whole-contig interval, (b) exon-like 100-400 bp intervals
about 10 kb apart (~2 % of positions), (c) a 20-gene panel (~0.1 %), (d) 100,000 single positions.  Stage times come from
CUDA events around each stage (runner.StageTimer).
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def target_sets(L, seed=17):
    from nanosnp_b200.targets import merge_intervals
    rng = np.random.default_rng(seed)
    starts = np.arange(0, L - 500, 10_000) + rng.integers(0, 5_000, (L - 500 + 9_999) // 10_000)
    exon = merge_intervals(zip(starts.tolist(), (starts + rng.integers(100, 401, len(starts))).tolist()), L)
    genes = np.sort(rng.choice(L // 10_000 - 1, 20, replace=False)) * 10_000
    panel = merge_intervals([(int(g), int(g) + L // 1000 // 20) for g in genes], L)
    pts = np.sort(rng.choice(L, 100_000, replace=False))
    points = merge_intervals([(int(p), int(p) + 1) for p in pts], L)
    return {"a_whole": np.array([[0, L]], np.int64), "b_exon": exon, "c_panel": panel, "d_points": points}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:          # the measurement itself still needs the GPU; only the label is missing
        return {"name": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--contig-mb", type=float, default=100.0)
    ap.add_argument("--bam-mb", type=float, default=12.5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupEngine, PileupModelForward, PileupModelWeights
    from nanosnp_b200.runner import RegionRunner, StageTimer
    from nanosnp_b200.shard import listed_tiles, plan_regions, plan_target_units
    from nanosnp_b200.synth import generate_device
    if not torch.cuda.is_available():
        raise SystemExit("target_bench.py: no CUDA device (there is no CPU path)")
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
    full_reads = bench.region_slices(reads, full_regions, cfg, dev, alg)
    sets = target_sets(L)
    work = {None: [(rg, rd, None) for rg, rd in zip(full_regions, full_reads)]}
    tiles = {}
    for name, iv in sets.items():
        units, ivs = plan_target_units([(cfg.contig, L)], {cfg.contig: iv}, region_len)
        slices = bench.region_slices(reads, units, cfg, dev, dict(alg))
        work[name] = [(rg, rd, u) for rg, rd, u in zip(units, slices, ivs)]
        tiles[name] = int(sum(len(listed_tiles(rg, u)) for rg, _, u in work[name]))
    del reads
    torch.cuda.empty_cache()

    def step(key, timer=None, keep=None):
        n = 0
        for rg, rd, u in work[key]:
            o = runner.run_device(rd, ref, rg, timer, targets=u)
            n += o.n
            if keep is not None:
                keep.append(o.rec.clone())
        return n

    res = {name: {"ms": [], "stage_ms": None} for name in [None] + list(sets)}
    for key in res:
        for _ in range(args.warmup):
            step(key)
    torch.cuda.synchronize()
    # alternate: every set once per round, in forward order on even rounds and reversed on odd ones, so that no set always
    # follows the same neighbour (a heavy step heats the card and lowers the clock of the next one)
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
    # (a) must give the same records as the unrestricted step
    ka, kn = [], []
    step("a_whole", keep=ka); step(None, keep=kn)
    torch.cuda.synchronize()
    same_a = all(torch.equal(x, y) for x, y in zip(ka, kn)) and len(ka) == len(kn)
    out = {"gpu": gpu_info(), "workload": {"contig_mb": args.contig_mb, "coverage": 30.0, "seeds": "bench.synth_cfg rank 0",
                                            "region_len": region_len, "precision": "f16x3", "steps": args.steps},
           "a_whole_records_identical_to_unrestricted": bool(same_a), "sets": {}}
    base = float(np.median(res[None]["ms"]))
    for key, r in res.items():
        name = "unrestricted" if key is None else key
        iv = None if key is None else sets[key]
        out["sets"][name] = {
            "ms_per_step_median": float(np.median(r["ms"])), "ms_per_step": [round(x, 3) for x in r["ms"]],
            "ratio_to_unrestricted": float(np.median(r["ms"])) / base, "sites": r["sites"], "launches_per_step": r["launches"],
            "listed_tiles": None if key is None else tiles[key], "intervals": None if iv is None else int(len(iv)),
            "target_fraction": None if iv is None else float((iv[:, 1] - iv[:, 0]).sum() / L), "units": len(work[key]),
            "stage_ms_per_step": {k: v / args.steps for k, v in r["stage_ms"].items() if k in ("pileup", "select", "gather", "model")}}
    out["indexed_bam_panel"] = bam_run(args, bargs)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


def bam_run(args, bargs):
    """BAM -> VCF through `python -m nanosnp_b200.predict` machinery in this process: (c)-like panel on a 12.5 Mb / 30x
    indexed BAM, against the run without targets (wall time and bytes inflated by the BAM reader)."""
    import bench
    from nanosnp_b200 import predict as P
    from nanosnp_b200.bam import BamReader, write_bam
    from nanosnp_b200.model import LSTMNetwork
    from nanosnp_b200.synth import generate_host
    from oracle.pyoracle import write_fasta
    import torch
    import yaml
    from nanosnp_b200.utils import AttrDict
    L = int(args.bam_mb * 1e6)
    cfg = bench.synth_cfg(bargs, 0, L)
    ref, reads = generate_host(cfg)
    d = tempfile.mkdtemp(prefix="nsnp_tb_")
    fa = os.path.join(d, "ref.fa")
    write_fasta(fa, {cfg.contig: ref})
    bam = os.path.join(d, "x.bam")
    write_bam(bam, [(cfg.contig, L)], {cfg.contig: reads}, index=True)
    panel = {cfg.contig: target_sets(L)["c_panel"]}
    conf = AttrDict(yaml.load(open(os.path.join(ROOT, "nanosnp_b200", "config", "ont_pileup.yaml")), Loader=yaml.FullLoader))
    model = LSTMNetwork(conf.model, precision="f16x3").to("cuda")
    z = np.load(os.path.join(ROOT, "tests", "golden", "ont_pileup_weights.npz"))
    model.encoder.load_state_dict({k[8:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("encoder.")})
    model.forward_layer.load_state_dict({k[14:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("forward_layer.")})
    out = {"bam_mb": args.bam_mb, "panel_fraction": float((panel[cfg.contig][:, 1] - panel[cfg.contig][:, 0]).sum() / L)}
    readers = []
    orig = BamReader.__init__

    def init(self, *a, **k):                           # keep the readers predict() opens: their inflated byte counts
        orig(self, *a, **k)
        readers.append(self)
    BamReader.__init__ = init
    try:
        for name, t in (("warmup", None), ("unrestricted", None), ("panel", panel), ("panel2", panel), ("unrestricted2", None)):
            o = os.path.join(d, name + ".vcf")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            P.predict(model, [bam], fa + ".fai", 1000, o, torch.device("cuda"), reference=fa, targets=t)
            torch.cuda.synchronize()
            if name != "warmup":
                out[name] = {"wall_s": time.perf_counter() - t0, "inflated_bytes": readers[-1].inflated_bytes,
                             "records": sum(1 for l in open(o) if not l.startswith("#"))}
    finally:
        BamReader.__init__ = orig
        shutil.rmtree(d, ignore_errors=True)
    return out


if __name__ == "__main__":
    main()
