#!/usr/bin/env python
"""bench.py -- candidate sites/sec of the s1+s2 hot path (BASELINE.json metric) on synthetic ONT-like reads.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (N>1: launched under torchrun)
  python bench.py --impl reference [--steps K] [--warmup W]      the reference's CPU path on a bounded sample

One "step" = one pass of pileup -> candidate select -> window gather -> PileupModel forward over the workload:
  N = 1   BASELINE.json configs[1]: one synthetic 100 Mb contig at 30x
  N > 1   BASELINE.json configs[3]: the whole-genome-shaped 3.1 Gb input (chr1-22,X,Y,M lengths) at 30x, cut into regions
          with 16-bp halos, LPT-assigned to the N GPUs (STRONG scaling, the north-star split), through the product's
          sharded path; a weak-scaling line (one 100 Mb contig per rank) is reported as the secondary key "weak"
  value  device-resident inputs, CUDA-event timed, max over ranks; --dump-outputs DIR writes what the last timed step
         returned (see dump_outputs) so that two builds can be compared on the same seeded inputs
  e2e    same work through the host-buffer API: pinned host arrays -> H2D -> kernels -> VCF text on the GPU -> D2H of the
         text (N > 1: every rank writes its segments of ONE ordered VCF file; only counts / batch heads are all-reduced)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "candidate sites/sec (s1+s2)"
FLOP_PER_SITE = 6.22e6           # exact-output minimal PileupModel FLOPs, SURVEY 8(d)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--contig-mb", type=float, default=100.0)
    ap.add_argument("--coverage", type=float, default=30.0)
    ap.add_argument("--region-mb", type=float, default=12.5)
    ap.add_argument("--cpu-sample-kb", type=float, default=500.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--precision", default="f16x3", choices=["fp32", "f16x3"])
    ap.add_argument("--weights", default=None, help="checkpoint: the reference's .chkpt or a flat .npz (default: the committed fixture of the shipped one)")
    ap.add_argument("--genome-scale", type=float, default=1.0, help="N > 1: shrink every contig of the 3.1 Gb genome (smoke runs)")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the secondary weak-scaling line")
    ap.add_argument("--no-selfcheck", action="store_true")
    ap.add_argument("--no-fast-mode", action="store_true", help="skip the secondary NSNP_PREC_F16X1 measurement")
    ap.add_argument("--write-vcf", action="store_true", help="N > 1: also place the text segments into ONE file on /dev/shm inside the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (rank 0's regions) as DIR/<name>.npy")
    return ap.parse_args()


def synth_cfg(args, rank, contig_len):
    from nanosnp_b200.synth import SynthConfig
    return SynthConfig(contig_len=int(contig_len), coverage=args.coverage, contig=f"ctg{rank + 1}",
                       seed_ref=1000 + rank, seed_var=2000 + rank, seed_reads=3000 + rank)


def load_weights(path=None):
    """The committed checkpoint fixture (flat .npz of the shipped ont_pileup.chkpt), or --weights: a .npz of that form or the
    reference's own .chkpt (torch.save of {'encoder': ..., 'forward_layer': ...}, PileupModel/utils.py:67-77)."""
    from nanosnp_b200.utils import load_weights_npz
    if path and not str(path).endswith(".npz"):
        import torch
        ck = torch.load(path, map_location="cpu")
        return tuple({k: v.detach().cpu().numpy() for k, v in ck[part].items()} for part in ("encoder", "forward_layer"))
    return load_weights_npz(path or ROOT / "tests" / "golden" / "ont_pileup_weights.npz")


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_reference_run(args, steps, warmup):
    """Times the reference's CPU s1+s2 path (oracle/_ref binaries + CPU predict logic) on a bounded sample."""
    from nanosnp_b200.synth import generate_host
    from oracle.cpu_path import run_cpu_path
    cores = os.cpu_count() or 1
    cfg = synth_cfg(args, 0, args.cpu_sample_kb * 1e3)
    ref, reads = generate_host(cfg)
    weights = load_weights(args.weights)
    times, res = [], None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        res = run_cpu_path(reads, ref, cfg.contig, weights, cores)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    mean = sum(times) / len(times)
    return {"value": res["n_sites"] / mean, "seconds_per_step": mean, "cores": cores, "kind": res["kind"],
            "n_sites": res["n_sites"], "stage_s": res["stage_s"],
            "sample": f"{args.cpu_sample_kb:.0f} kb synthetic contig at {args.coverage:g}x (same generator/config as the GPU workload), "
                      f"{res['n_sites']} sites; stages: mpileup restatement (ours, not samtools) + reference DNA_CreateCanSnpTensor/"
                      f"DNA_CreatePredictData ({res['kind']}) + text->int32 + predict.py logic on torch CPU fp32"}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args, args.steps, min(args.warmup, 1) if args.warmup else 0)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "sites/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["seconds_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32 counts + fp32 model", "data": "synthetic",
            "config": {"workload": f"synthetic contig at {args.coverage:g}x, s1+s2 on host CPU; bounded sample", "sample_kb": args.cpu_sample_kb,
                       "extrapolated": True},
            "cpu_baseline": {"value": r["value"], "unit": "sites/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                             "stage_s": r["stage_s"]},
            "e2e": {"value": r["value"], "unit": "sites/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ our arm
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        """Samples taken inside [t_begin, t_end] (the timed region); nvidia-smi needs a few hundred ms to start, so the
        sampler is started before the warm-up and, if the timed region is shorter than one sampling period, the
        samples of the load immediately before it (same kernels, same clocks) are used and the window says so."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        window = "timed region"
        lines = [l for (t, l) in self.lines if t_begin is None or (t_begin <= t <= t_end + 0.12)]
        if not lines and t_begin is not None:
            lines = [l for (t, l) in self.lines if t <= t_end + 0.12][-5:]
            window = "warm-up + timed region (timed region shorter than the sampling period)"
        self.window = window
        for l in lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nme, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


GRCH38 = [("chr1", 248956422), ("chr2", 242193529), ("chr3", 198295559), ("chr4", 190214555), ("chr5", 181538259),
          ("chr6", 170805979), ("chr7", 159345973), ("chr8", 145138636), ("chr9", 138394717), ("chr10", 133797422),
          ("chr11", 135086622), ("chr12", 133275309), ("chr13", 114364328), ("chr14", 107043718), ("chr15", 101991189),
          ("chr16", 90338345), ("chr17", 83257441), ("chr18", 80373285), ("chr19", 58617616), ("chr20", 64444167),
          ("chr21", 46709983), ("chr22", 50818468), ("chrX", 156040895), ("chrY", 57227415), ("chrM", 16569)]


def region_slices(reads, regions, cfg, dev, alg):
    """Device slices of one contig's reads for some of its regions (what a host decoder hands over per region)."""
    import torch
    from nanosnp_b200.reads import PackedReads
    from nanosnp_b200.shard import read_range_for_region
    pos_host = reads.pos.cpu().numpy()
    max_span = int(cfg.len_max * 1.3) + 1000
    n_total = reads.n_reads
    total_bases = int(reads.seq2.numel()) * 4
    pad = torch.zeros(16, dtype=torch.uint8, device=dev)
    out = []
    for rg in regions:
        lo, hi = read_range_for_region(pos_host, max_span, rg)
        c0, c1 = int(reads.cigar_off[lo].item()), int(reads.cigar_off[hi].item())
        b0 = int(reads.seq_off[lo].item()) if lo < n_total else total_bases
        b1 = int(reads.seq_off[hi].item()) if hi < n_total else total_bases - 64
        out.append(PackedReads(reads.pos[lo:hi].clone(), reads.flag[lo:hi].clone(), reads.mapq[lo:hi].clone(),
                               (reads.cigar_off[lo:hi + 1] - c0), reads.cigar[c0:c1].clone(), (reads.seq_off[lo:hi] - b0),
                               torch.cat([reads.seq2[b0 // 4:(b1 + 3) // 4], pad]),
                               None if reads.nmask is None else torch.cat([reads.nmask[b0 // 8:(b1 + 7) // 8], pad])))
        alg["n_bases"] += b1 - b0; alg["n_cigar"] += c1 - c0; alg["n_reads"] += hi - lo
        alg["pileup"] += 0.25 * (b1 - b0) + 4.0 * (c1 - c0) + 23.0 * (hi - lo) + 74.0 * rg.length     # SURVEY 8(d) B_A (+ ref byte)
    return out


DUMP_SITES = 1 << 16             # sites sampled by --dump-outputs: ~15 MB of .npy files


def dump_outputs(out_dir, outputs):
    """--dump-outputs: what RegionRunner.run_device returned to the caller in the last timed step, for comparing two builds
    output for output.  outputs: [(pos0, gt, zy, rec)] per region, in region order.  Writes region_sites (site count of
    every region) and, for a sample of DUMP_SITES sites drawn with a fixed seed from the concatenation of all regions,
    site_index (index into that concatenation), pos0 (0-based contig position), gt [k,21] and zy [k,3] (probabilities)
    and records [k,32] (the bytes of the compact site records).  Integers are stored exactly as float64 / float32."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    pos0, gt, zy, rec = (torch.cat([o[i] for o in outputs]) for i in range(4))
    n = pos0.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_SITES), replace=False))
    ti = torch.from_numpy(idx).to(pos0.device)
    arrays = {"region_sites": np.array([o[0].shape[0] for o in outputs], np.float64), "site_index": idx.astype(np.float64),
              "pos0": pos0[ti].cpu().numpy().astype(np.float64), "gt": gt[ti].cpu().numpy(), "zy": zy[ti].cpu().numpy(),
              "records": rec[ti].cpu().numpy().astype(np.float32)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main_ours(args):
    import ctypes as C
    import hashlib
    import numpy as np
    import torch
    import torch.distributed as dist
    from nanosnp_b200 import _lib
    from nanosnp_b200.caller import ShardedVcfWriter
    from nanosnp_b200.pipeline import PileupEngine, PileupModelForward, PileupModelWeights
    from nanosnp_b200.predict_io import ContigVcfAssembler
    from nanosnp_b200.reads import FIELDS, PackedReads, cigar16
    from nanosnp_b200.runner import RegionRunner, StageTimer
    from nanosnp_b200.shard import assign_lpt, plan_regions
    from nanosnp_b200.synth import SynthConfig, generate_device
    from nanosnp_b200.vcf_text import GpuVcfText

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GPU path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version on stdout while the communicator is created: route that to stderr so that stdout carries
        # the one JSON line only
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    K, W = args.steps, max(args.warmup, 3)
    lib = _lib.load()
    eng = PileupEngine(dev)
    enc, fwd = load_weights(args.weights)
    prec = _lib.PREC_FP32 if args.precision == "fp32" else _lib.PREC_F16X3
    model = PileupModelForward(PileupModelWeights(enc, fwd, device=dev), precision=prec)
    runner = RegionRunner(eng, model, records=True)        # device-resident result = compact site records (fused s1 -> s2 hand-off)
    # few host cores per rank: host waits sleep on blocking events instead of spinning in cudaStreamSynchronize
    runner_e2e = RegionRunner(eng, model, records=True, blocking_sync=(os.cpu_count() or 1) <= 4 * world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def pinned(rd):
        rd = cigar16(rd)                                       # host hand-off ships uint16 CIGAR words (every length < 4096 here)
        return PackedReads(*[None if getattr(rd, f) is None else getattr(rd, f).cpu().pin_memory() for f in FIELDS])

    def time_device(work, steps, timer=None, profile=False, keep=None):
        """work: [(Region, device reads, device ref)].  Returns (ms_total, sites of one step, t_begin, t_end).
        keep: a list that receives device copies of (pos0, gt, zy, rec) of every region of the last timed step (the runner
        reuses its buffers from region to region)."""
        def step(tm=None, keep=None):
            n = 0
            for rg, rd, rf in work:
                o = runner.run_device(rd, rf, rg, tm)
                n += o.n
                if keep is not None:
                    keep.append((o.pos0.clone(), o.gt.clone(), o.zy.clone(), o.rec.clone()))
            return n
        for _ in range(W):
            n_sites = step()
        barrier()
        if profile:
            lib.nsnp_profile_enable(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t_begin = time.time()
        e0.record()
        for i in range(steps):
            n_sites = step(timer, keep if i == steps - 1 else None)
        e1.record()
        barrier()
        return e0.elapsed_time(e1), n_sites, t_begin, time.time()

    def time_e2e(step_host, steps):
        step_host()                                            # warm-up: buffers, pinned staging, text kernels
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        f0.record()
        for _ in range(steps):
            n = step_host()
        f1.record()
        barrier()
        return max(f0.elapsed_time(f1), (time.perf_counter() - t0) * 1e3), n

    def reduce_max_sum(vals):
        v = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world == 1:
            return v.tolist(), v.tolist()
        mx = v.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = v.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        return mx.tolist(), sm.tolist()

    alg = {"pileup": 0.0, "n_bases": 0, "n_cigar": 0, "n_reads": 0}
    selfcheck = None
    weak = None
    sampler = ClockSampler(local)
    sampler.start()

    # ================================================================ one 100 Mb contig per rank (N = 1 headline; N > 1: "weak")
    def contig_workload(steps, with_e2e, with_selfcheck, alg_acc, keep=None):
        L = int(args.contig_mb * 1e6)
        cfg = synth_cfg(args, rank, L)
        ref, reads = generate_device(cfg, dev)
        regions = plan_regions([(cfg.contig, L)], int(args.region_mb * 1e6))
        dev_regions = region_slices(reads, regions, cfg, dev, alg_acc)
        del reads
        torch.cuda.empty_cache()
        work = [(rg, rd, ref) for rg, rd in zip(regions, dev_regions)]
        timer = StageTimer(True)
        ms_total, n_sites, t_begin, t_end = time_device(work, steps, timer, profile=True, keep=keep)
        res = {"cfg": cfg, "regions": regions, "ms_total": ms_total, "n_sites": n_sites, "t": (t_begin, t_end), "timer": timer, "e2e": None}
        kms = (C.c_double * len(_lib.PROF_SLOTS))(); kln = (C.c_int64 * len(_lib.PROF_SLOTS))()
        _lib.check(lib.nsnp_profile_read(kms, kln))
        lib.nsnp_profile_enable(0)
        res["kernel_ms"] = {k: kms[i] for i, k in enumerate(_lib.PROF_SLOTS)}
        res["kernel_launches"] = {k: int(kln[i]) for i, k in enumerate(_lib.PROF_SLOTS)}
        if rank == 0:
            # the window-gather kernel of the dataset seam (B2), timed alone on the first region: it is no longer on the fused path
            rgath = RegionRunner(eng, model, keep_windows=True)
            o = rgath.run_device(dev_regions[0], ref, regions[0])
            cnt = rgath._bufs["counts"][: regions[0].length * 18].view(regions[0].length, 18)
            xg = torch.empty((o.n, 33, 18), dtype=torch.int32, device=dev); rb = torch.empty(o.n, dtype=torch.uint8, device=dev)
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for it in range(4):
                if it == 1:
                    g0.record()
                eng.gather(cnt, ref, regions[0].start, o.pos0, None, o.n, x_i32=xg, refbase=rb)
            g1.record(); torch.cuda.synchronize()
            res["gather_standalone"] = {"ms": g0.elapsed_time(g1) / 3, "sites": o.n}
            del rgath, o, cnt, xg, rb
            torch.cuda.empty_cache()
        if with_e2e:
            host_regions = [pinned(rd) for rd in dev_regions]
            h2d = sum(h.nbytes() for h in host_regions)
            sha = [None]
            nbytes = [0]

            def step_host(keep_hash=False):
                gen = GpuVcfText(dev, cfg.contig, 1000)
                h = hashlib.sha256() if keep_hash else None
                nbytes[0] = 0

                def write(mv):
                    nbytes[0] += len(mv)
                    if h is not None:
                        h.update(mv)
                n = runner_e2e.run_host_text(host_regions, regions, ref, gen, write)
                if h is not None:
                    sha[0] = h.hexdigest()
                return n
            e2e_ms, n_e2e = time_e2e(step_host, steps)
            res["e2e"] = {"ms": e2e_ms, "sites": n_e2e, "h2d": h2d, "d2h": nbytes[0], "vcf_bytes": nbytes[0]}
            if with_selfcheck:
                # outside the timed region: (1) the tensor-core probabilities of one region against the fp32 FFMA path on
                # every site, (2) the bytes of the GPU-text e2e path against the host text assembly of the same step's
                # records (run_host_many + nsnp_vcf_format_contig_records)
                rk = RegionRunner(eng, model, keep_windows=True)
                o = rk.run_device(dev_regions[0], ref, regions[0])
                f32 = PileupModelForward(model.w, _lib.PREC_FP32)
                g32, z32 = f32(o.x)
                dp = max(float((o.gt - g32).abs().max()), float((o.zy - z32).abs().max()))
                flips = int((o.gt.argmax(1) != g32.argmax(1)).sum()) + int((o.zy.argmax(1) != z32.argmax(1)).sum())
                del rk, o, g32, z32, f32
                step_host(keep_hash=True)
                capn = max(1024, max(rg.emit_end - rg.emit_start for rg in regions) // 3)
                host_outs = tuple({"rec": torch.empty((capn, 32), dtype=torch.uint8).pin_memory()} for _ in range(2))
                h2 = hashlib.sha256()

                class Sink:
                    def write(self, b):
                        h2.update(b)
                asm = ContigVcfAssembler(cfg.contig, 1000, max(1, (os.cpu_count() or 1) // world), Sink())
                runner_e2e.run_host_many(host_regions, regions, ref, host_outs, lambda k, r: asm.add_records(r["rec"].numpy()))
                asm.close()
                ok = dp < 5e-5 and sha[0] == h2.hexdigest()
                res["selfcheck"] = {"f16x3_vs_fp32_max_abs_dp": dp, "argmax_flips": flips, "tolerance": 5e-5,
                                    "vcf_sha256_gpu_text": sha[0], "vcf_sha256_host_text": h2.hexdigest(), "ok": bool(ok)}
                if not ok:
                    raise SystemExit(f"bench.py self-check failed: {res['selfcheck']}")
            del host_regions
        if with_selfcheck and not args.no_fast_mode and args.precision == "f16x3":
            # secondary, outside the timed region of the headline: the opt-in single-pass mode (NSNP_PREC_F16X1: one fp16 MMA per
            # product, low-margin sites re-evaluated with the three-pass path) on the same device-resident workload, and its
            # records of one region against the headline path's: calls must be identical, QUAL may drift
            x1 = PileupModelForward(model.w, _lib.PREC_F16X1)
            r1 = RegionRunner(eng, x1, records=True)

            def step1():
                return sum(r1.run_device(rd, rf, rg).n for rg, rd, rf in work)
            step1()
            torch.cuda.synchronize()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record()
            for _ in range(steps):
                n1 = step1()
            q1.record(); torch.cuda.synchronize()
            ms1 = q0.elapsed_time(q1)
            rec3 = runner.run_device(dev_regions[0], ref, regions[0]).rec.clone().cpu().numpy()
            rec1 = r1.run_device(dev_regions[0], ref, regions[0]).rec.clone().cpu().numpy()
            n_low = x1.reevaluated()
            same_calls = bool(rec1.shape == rec3.shape and (rec1[:, [0, 1, 3]] == rec3[:, [0, 1, 3]]).all() and ((rec1[:, 2] & 1) == (rec3[:, 2] & 1)).all()
                              and (rec1[:, 4:8] == rec3[:, 4:8]).all() and (rec1[:, 16:24] == rec3[:, 16:24]).all())
            qa = np.ascontiguousarray(rec1[:, 8:16]).view(np.int32).astype(np.int64); qb = np.ascontiguousarray(rec3[:, 8:16]).view(np.int32).astype(np.int64)
            res["fast_mode"] = {"precision": "f16x1: one fp16 tensor-core pass per product, fp32 accumulate; sites with a top-2 margin < 0.02 re-evaluated with the three-pass path",
                                "value": n1 * steps / (ms1 * 1e-3), "unit": "sites/s", "ms_per_step": ms1 / steps, "steps": steps,
                                "calls_identical_to_headline_path": same_calls, "qual_drift_max": float(np.abs(qa - qb).max()) / 100.0,
                                "records_with_other_qual_pct": float(((qa != qb).any(axis=1)).mean() * 100.0),
                                "reevaluated_sites_in_region0": int(n_low), "sites_in_region0": int(rec3.shape[0]),
                                "note": "opt-in (LSTMNetwork(precision='f16x1') / --precision f16x1); not the headline: QUAL text differs from the three-pass path on ~3 % of the records (by at most 0.06)"}
            if not same_calls:
                raise SystemExit(f"bench.py: single-pass mode changed a call: {res['fast_mode']}")
            del x1, r1, rec1, rec3
        return res

    # ================================================================ genome-shaped strong scaling (N > 1)
    def genome_workload(steps, keep=None):
        contigs = [(n, max(2000, int(L * args.genome_scale))) for n, L in GRCH38]
        regions = plan_regions(contigs, int(args.region_mb * 1e6))
        mine = assign_lpt(regions, world)[rank]
        t_gen = time.perf_counter()
        work, idx = [], []
        for ci in sorted({regions[i].contig_index for i in mine}):
            name, L = contigs[ci]
            cfg = SynthConfig(contig_len=L, coverage=args.coverage, contig=name, seed_ref=100 + ci, seed_var=200 + ci, seed_reads=300 + ci)
            ref, reads = generate_device(cfg, dev)
            ii = [i for i in mine if regions[i].contig_index == ci]
            for i, rd in zip(ii, region_slices(reads, [regions[i] for i in ii], cfg, dev, alg)):
                work.append((regions[i], rd, ref)); idx.append(i)
            del reads
            torch.cuda.empty_cache()
        torch.cuda.synchronize()
        t_gen = time.perf_counter() - t_gen
        timer = StageTimer(True)
        ms_total, n_sites, t_begin, t_end = time_device(work, steps, timer, profile=True, keep=keep)
        kms = (C.c_double * len(_lib.PROF_SLOTS))(); kln = (C.c_int64 * len(_lib.PROF_SLOTS))()
        _lib.check(lib.nsnp_profile_read(kms, kln))
        lib.nsnp_profile_enable(0)
        res = {"regions": [w[0] for w in work], "all_regions": len(regions), "contigs": contigs, "ms_total": ms_total, "n_sites": n_sites,
               "t": (t_begin, t_end), "timer": timer, "e2e": None, "t_gen": t_gen,
               "kernel_ms": {k: kms[i] for i, k in enumerate(_lib.PROF_SLOTS)}, "kernel_launches": {k: int(kln[i]) for i, k in enumerate(_lib.PROF_SLOTS)}}
        if not args.no_e2e:
            host_regions = [pinned(w[1]) for w in work]
            h2d = sum(h.nbytes() for h in host_regions)
            refs = [w[2] for w in work]
            rgs = [w[0] for w in work]
            out_path = f"/dev/shm/nsnp_bench_{os.environ.get('MASTER_PORT', '0')}.vcf"
            header = b"##fileformat=VCFv4.3\n" + b"".join(f"##contig=<ID={n},length={L}>\n".encode() for n, L in contigs)
            info = {}
            writer = ShardedVcfWriter(contigs, regions, 1000, dev)

            def step_host(to_file=args.write_vcf):
                # the text of region k is made (deferred batch heads) and copied to the host while region k+1 computes
                writer.begin()
                ns = runner_e2e.run_host_collect(host_regions, rgs, refs, on_region=lambda k, o: writer.add_region(idx[k], o.rec))
                info.update(writer.finish(out_path if to_file else None, header))
                return sum(ns)
            e2e_ms, n_e2e = time_e2e(step_host, steps)
            step_host(True)                                     # outside the timed region: the file, for the checksum below
            res["e2e"] = {"ms": e2e_ms, "sites": n_e2e, "h2d": h2d, "d2h": 0, "vcf_bytes": info.get("vcf_bytes", 0)}
            if rank == 0:
                with open(out_path, "rb") as f:
                    hsh = hashlib.sha256()
                    for blk in iter(lambda: f.read(1 << 24), b""):
                        hsh.update(blk)
                res["vcf_sha256"] = hsh.hexdigest()
                os.unlink(out_path)
        return res

    outputs = [] if args.dump_outputs and rank == 0 else None
    if world == 1:
        main_res = contig_workload(K, not args.no_e2e, not args.no_selfcheck and not args.no_e2e, alg, keep=outputs)
        scaling = "weak"
    else:
        main_res = genome_workload(K, keep=outputs)
        scaling = "strong"
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
        del outputs
    clocks = sampler.stop(*main_res["t"])
    if world > 1 and not args.no_weak:
        wk = contig_workload(max(1, min(K, 2)), not args.no_e2e, False, {"pileup": 0.0, "n_bases": 0, "n_cigar": 0, "n_reads": 0})
        mxw, smw = reduce_max_sum([wk["ms_total"], float(wk["n_sites"]), wk["e2e"]["ms"] if wk["e2e"] else 0.0, float(wk["e2e"]["sites"]) if wk["e2e"] else 0.0])
        ks = max(1, min(K, 2))
        weak = {"scaling": "weak", "workload": f"one synthetic {args.contig_mb:g} Mb contig at {args.coverage:g}x per GPU", "steps": ks,
                "value": smw[1] / (mxw[0] * 1e-3) * ks, "ms_per_step": mxw[0] / ks,
                "e2e_value": (smw[3] / (mxw[2] * 1e-3) * ks) if mxw[2] > 0 else None}

    ms_total, n_sites = main_res["ms_total"], main_res["n_sites"]
    e2e = main_res["e2e"]
    stage_ms = main_res["timer"].totals_ms()
    stage_calls = main_res["timer"].counts()
    kernel_ms, kernel_launches = main_res["kernel_ms"], main_res["kernel_launches"]
    # kernels of this library launched inside the timed region, counted by the library itself (select / text slots are three kernels each)
    launches = sum(kernel_launches.values()) + 2 * kernel_launches.get("select_kernels", 0) + 2 * kernel_launches.get("vcf_text_kernels", 0)

    # ---- reduce over ranks: max time, total sites / bytes ----
    mx, sm = reduce_max_sum([ms_total, float(n_sites), e2e["ms"] if e2e else 0.0, float(e2e["sites"]) if e2e else 0.0,
                             float(e2e["h2d"]) if e2e else 0.0, float(e2e["d2h"]) if e2e else 0.0, float(alg["pileup"]), float(launches)])
    ms_total, sites_all = mx[0], sm[1]
    e2e_ms, e2e_sites, h2d_all, d2h_all = mx[2], sm[3], sm[4], sm[5]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    pk_path = ROOT / "MEASURED_PEAKS.json"
    if pk_path.exists():
        peaks = json.loads(pk_path.read_text())
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tf_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    ms_step = ms_total / K
    regions = main_res["regions"]

    traffic = {}
    tr_path = ROOT / "profiles" / "traffic.json"
    if tr_path.exists():
        traffic = json.loads(tr_path.read_text())

    def hbm(stage, bytes_per_step, traffic_bytes=None):
        ms = stage_ms[stage] / K
        a = bytes_per_step / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        return {"bound": "hbm", "achieved": a, "peak": hbm_peak, "unit": "GB/s", "frac": a / hbm_peak, "ms_per_step": ms,
                "launches_per_step": stage_calls[stage] // K, "algorithmic_bytes_per_step": bytes_per_step, "traffic": traffic_bytes}
    Lr = sum(rg.length for rg in regions)
    stages = {
        "pileup": hbm("pileup", alg["pileup"], traffic.get("pileup_tile_kernel", {}).get("dram_bytes_per_position", 0) * Lr or None),
        "select": hbm("select", 1.0 * Lr + 4.0 * n_sites),
    }
    if main_res.get("gather_standalone"):
        gs = main_res["gather_standalone"]
        a = 4753.0 * gs["sites"] / (gs["ms"] * 1e-3) / 1e9
        stages["gather"] = {"bound": "hbm", "achieved": a, "peak": hbm_peak, "unit": "GB/s", "frac": a / hbm_peak, "ms_per_launch": gs["ms"],
                            "sites_per_launch": gs["sites"], "algorithmic_bytes_per_launch": 4753.0 * gs["sites"],
                            "traffic": traffic.get("gather_kernel", {}).get("dram_bytes_per_site", 0) * gs["sites"] or None,
                            "note": "the dataset-seam kernel (nsnp_gather_windows), timed alone on one region outside the timed step: the fused "
                                    "path reads windows straight from the count tensor and never launches it"}
    # ---- roofline of the dominant kernel (largest share of the timed region), timed live with CUDA events around
    #      each of its launches on the launching stream (nsnp_profile_*); rank 0's kernels ----
    flop_per_site = {"lstm_layer0": 2 * 1385472.0, "lstm_layer1": 2 * 1671168.0, "tail_kernel": 2 * 55296.0}     # SURVEY 8(d)
    kernels = {}
    for name in _lib.PROF_SLOTS:
        ms = kernel_ms[name] / K
        ent = {"ms_per_step": ms, "launches_per_step": kernel_launches[name] // K, "share_of_step": ms / ms_step}
        if name in flop_per_site and ms > 0:
            tf = flop_per_site[name] * n_sites / (ms * 1e-3) / 1e12
            ent.update({"bound": "tensor" if name != "tail_kernel" else "fp32", "achieved": tf, "unit": "TFLOP/s", "peak": tf_peak, "frac": tf / tf_peak})
            if name in traffic:
                ent["traffic"] = traffic[name]["dram_bytes_per_site"] * n_sites / max(1, kernel_launches[name] // K)
        kernels[name] = ent
    dom = max(("lstm_layer0", "lstm_layer1", "pileup_tile_kernel"), key=lambda k: kernel_ms[k])
    if dom == "pileup_tile_kernel":
        d = kernels[dom]; a = alg["pileup"] / (d["ms_per_step"] * 1e-3) / 1e9
        roofline = {"kernel": "pileup_tile_kernel", "bound": "hbm", "achieved": a, "peak": hbm_peak, "unit": "GB/s", "frac": a / hbm_peak,
                    "traffic": traffic.get(dom, {}).get("dram_bytes_per_position", 0) * Lr / max(1, len(regions)) or None}
    else:
        d = kernels[dom]
        roofline = {"kernel": {"lstm_layer0": "lstm0_pair2_kernel (layer-0 BiLSTM, tcgen05 cta_group::2, two alternating site groups per CTA)",
                               "lstm_layer1": "lstm_tc_kernel<1,2,4> (layer-1 BiLSTM, tcgen05 cta_group::2)"}[dom] if args.precision != "fp32" else dom,
                    "bound": "tensor", "achieved": d["achieved"], "peak": tf_peak, "unit": "TFLOP/s", "frac": d["frac"],
                    "traffic": d.get("traffic"), "traffic_note": "DRAM bytes per launch, scaled from the ncu capture in profiles/traffic.json",
                    "ms_per_step": d["ms_per_step"], "launches_per_step": d["launches_per_step"], "share_of_step": d["share_of_step"],
                    "peak_source": peak_src,
                    "note": ("fp32 FFMA path (no tensor cores): algorithmic FLOPs over the bf16 sustained peak" if args.precision == "fp32" else
                             "algorithmic (exact-minimal) FLOPs of this layer over the measured sustained bf16 peak; every algorithmic MAC "
                             "costs three fp16 MMAs (hi/lo split), so frac <= 1/3 by construction; rank 0's kernels (DESIGN.md 4.4)")}
    model_ms = stage_ms["model"] / K
    tfs = FLOP_PER_SITE * n_sites / (model_ms * 1e-3) / 1e12 if model_ms > 0 else 0.0
    stages["model"] = {"bound": "tensor", "achieved": tfs, "peak": tf_peak, "unit": "TFLOP/s", "frac": tfs / tf_peak, "ms_per_step": model_ms,
                       "algorithmic_flop_per_site": FLOP_PER_SITE}
    if world == 1:
        cfg = main_res["cfg"]
        config = {"workload": f"synthetic {args.contig_mb:g} Mb contig at {args.coverage:g}x on 1 GPU: pileup tensor build + candidate filter + PileupModel inference",
                  "contig_mb": args.contig_mb, "coverage": args.coverage, "region_mb": args.region_mb, "regions_per_gpu": len(regions),
                  "sites_per_gpu_step": n_sites, "reads": alg["n_reads"], "aligned_bases": alg["n_bases"], "cigar_ops": alg["n_cigar"],
                  "weights": "shipped ont_pileup.chkpt (fp32)", "l2": "inputs (>3 GB per step) exceed the 126 MB L2; no explicit flush",
                  "seeds": [cfg.seed_ref, cfg.seed_var, cfg.seed_reads], "parallelism": "1 GPU, regions of one contig in sequence"}
    else:
        total_len = sum(L for _, L in main_res["contigs"])
        config = {"workload": f"whole-genome-shaped synthetic {total_len / 1e9:.2f} Gb (chr1-22,X,Y,M lengths) at {args.coverage:g}x: "
                              f"{main_res['all_regions']} regions of <= {args.region_mb:g} Mb + 16-bp halo, LPT-assigned to {world} GPUs "
                              "(BASELINE configs[3]); pileup tensor build + candidate filter + PileupModel inference + one ordered VCF",
                  "genome_scale": args.genome_scale, "coverage": args.coverage, "region_mb": args.region_mb, "regions_total": main_res["all_regions"],
                  "regions_rank0": len(regions), "sites_total_step": sites_all, "pileup_algorithmic_bytes_total": sm[6],
                  "weights": "shipped ont_pileup.chkpt (fp32)", "l2": "per-rank inputs (>10 GB per step) exceed the 126 MB L2; no explicit flush",
                  "seeds": "seed_ref/var/reads = 100/200/300 + contig index", "setup_generate_s_rank0": main_res["t_gen"],
                  "parallelism": f"region shards x{world}, no data-path collective; all-reduce of per-region counts, batch heads (10 B per 1000 sites) "
                                 "and text lengths only", "vcf_sha256": main_res.get("vcf_sha256")}
    line = {
        "metric": METRIC, "value": sites_all / (ms_total * 1e-3) * K, "unit": "sites/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "int32 counts, fp64 AF gate, " + ("fp32 model" if args.precision == "fp32" else "fp16 hi/lo split x3 tensor-core model (fp32 accumulate)"),
        "data": "synthetic", "config": config,
        "clocks": clocks, "gpu_launches": int(sm[7]),
        "roofline": roofline, "roofline_stages": stages, "kernels": kernels,
        "stage_ms_per_step": {k: v / K for k, v in stage_ms.items()},
    }
    if e2e:
        line["e2e"] = {"value": e2e_sites / (e2e_ms * 1e-3) * K, "unit": "sites/s", "h2d_bytes_per_step": h2d_all,
                       "d2h_bytes_per_step": d2h_all if world == 1 else e2e["vcf_bytes"], "ms_per_step": e2e_ms / K, "vcf_bytes_per_step": e2e["vcf_bytes"],
                       "note": ("pinned host read arrays -> H2D -> kernels (incl. site_record_kernel and the VCF text kernels: record lengths -> scan -> "
                                "write) -> D2H of the VCF text through RegionRunner.run_host_text; the host only patches the flagged QUAL rounding ties "
                                "(~4 per million records); copies overlap the kernels of the neighbouring regions; reference FASTA and weights resident"
                                if world == 1 else
                                "per rank: pinned host read arrays (uint16 CIGAR words) -> H2D -> kernels -> site records -> VCF text kernels with deferred "
                                "batch heads -> D2H of region k's text while region k+1 computes; after the last region: all-reduce of region site counts, "
                                "batch heads and text lengths, one-character ALT fix-ups and QUAL tie fix-ups on the host: the timed region ends when "
                                "every rank holds its ordered text segments and their file offsets in pinned host memory (the same end point as at N = 1, "
                                "where the text chunks are handed to the caller's write()); placing them into ONE file (caller.ShardedVcfWriter, shared "
                                "mapping) is timed only with --write-vcf; the file of one step is still produced and checksummed (config.vcf_sha256); "
                                "barrier on both sides, max over ranks"), "file_in_timed_region": bool(args.write_vcf)}
    else:
        line["e2e"] = None
    if weak is not None:
        line["weak"] = weak
    if main_res.get("selfcheck"):
        line["selfcheck"] = main_res["selfcheck"]
    if main_res.get("fast_mode"):
        line["fast_mode"] = main_res["fast_mode"]
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(args, 1, 0)
        line["cpu_baseline"] = {"value": r["value"], "unit": "sites/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                                "stage_s": r["stage_s"], "extrapolated": True,
                                "note": f"rate of a {args.cpu_sample_kb:g} kb sample of the same generator/config, not the full 100 Mb run"}
    else:
        line["cpu_baseline"] = None
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        main_reference(a)
    else:
        main_ours(a)
