"""Runs the whole s1+s2 GPU path for one region: reads -> counts -> candidates -> windows -> probabilities.

Used by bench.py (device-resident and host-buffer modes) and by the predict.py drop-in.  Buffers are
allocated once and grown on demand; the only host synchronisation per region is the site count.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from .pipeline import PileupEngine, PileupModelForward
from .reads import FIELDS, PackedReads
from .shard import Region

COV_CHANNELS = [0, 1, 2, 3, 9, 10, 11, 12]           # predict.py:63


@dataclass
class RegionOutput:
    n: int
    pos0: torch.Tensor        # int32 [n]
    refbase: torch.Tensor     # uint8 [n]
    cov8: torch.Tensor        # float32 [n,8] centre counts of [A C G T a c g t]
    gt: torch.Tensor          # float32 [n,21]
    zy: torch.Tensor          # float32 [n,3]
    x: Optional[torch.Tensor] = None
    rec: Optional[torch.Tensor] = None    # uint8 [n,32] compact site records (records mode)


class StageTimer:
    """CUDA-event timing of the stages of one step on the launching stream (bench.py roofline numbers)."""
    STAGES = ("h2d", "pileup", "select", "gather", "model", "d2h")

    def __init__(self, enabled: bool):
        self.enabled = enabled
        self.pairs = {s: [] for s in self.STAGES}
        self._open = None

    def start(self, stage: str):
        if not self.enabled:
            return
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        self._open = (stage, ev)

    def stop(self):
        if not self.enabled or self._open is None:
            return
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        self.pairs[self._open[0]].append((self._open[1], ev))
        self._open = None

    def totals_ms(self) -> Dict[str, float]:
        torch.cuda.synchronize()
        return {s: float(sum(a.elapsed_time(b) for a, b in p)) for s, p in self.pairs.items()}

    def counts(self) -> Dict[str, int]:
        return {s: len(p) for s, p in self.pairs.items()}


class RegionRunner:
    def __init__(self, engine: PileupEngine, model: PileupModelForward, keep_windows: bool = False, records: bool = False,
                 blocking_sync: bool = False, fused: bool = True):
        """blocking_sync: host waits sleep on a blocking CUDA event instead of spinning in cudaStreamSynchronize.  A
        spinning wait costs one host core per GPU for the whole run; with few cores per GPU (8 ranks on 16 cores) that
        core is better spent on VCF text assembly.  Spinning wakes up a little faster, so it stays the default."""
        self.blocking_sync = blocking_sync
        self.eng = engine
        self.model = model
        self.device = engine.device
        self.keep_windows = keep_windows
        self.records = records            # numeric record logic on the GPU: 32 bytes/site leave the device instead of 133
        self.fused = fused                # records mode: no window tensor between s1 and s2 (windows are row spans of the counts)
        self._bufs: Dict[str, torch.Tensor] = {}
        self.launches = 0          # kernels of this library launched so far

    def _buf(self, key: str, shape, dtype) -> torch.Tensor:
        n = int(np.prod(shape))
        t = self._bufs.get(key)
        if t is None or t.numel() < n or t.dtype != dtype:
            t = torch.empty(int(n * 1.2) + 64, dtype=dtype, device=self.device)
            self._bufs[key] = t
        return t[:n].view(*shape)

    def run_device(self, reads: PackedReads, ref: torch.Tensor, region: Region, timer: Optional[StageTimer] = None,
                   targets: Optional[np.ndarray] = None, sites: bool = False) -> RegionOutput:
        """targets: the unit's [k, 2] sorted disjoint [start, end) intervals (contig coordinates, inside the emit span), or None
        for every position of the region.  With targets only the tiles near them are computed and only sites inside them
        are kept; the launch count does not depend on k.  sites: the targets are a list of given sites (`--sites`): each
        listed position with a full window and an ACGT centre base is called, whether it passes the gate or not."""
        eng = self.eng
        rlen = region.length
        timer = timer or StageTimer(False)
        counts = self._buf("counts", (rlen, _lib.CHANNELS), torch.int32)
        flags = self._buf("flags", (rlen,), torch.uint8)
        timer.start("pileup")
        eng.pileup_counts(reads, ref, region.start, rlen, counts=counts, flags=flags, targets=targets)
        timer.stop()
        self.launches += (2 if reads.n_reads else 1) + (targets is not None)
        if sites:                                 # at most one candidate per listed position
            cap = max(1024, int(np.subtract(targets[:, 1], targets[:, 0], dtype=np.int64).sum()))
        else:
            cap = max(1024, region.emit_end - region.emit_start)
        pos = self._buf("pos", (cap,), torch.int32)
        n_dev = self._buf("n", (1,), torch.int32)
        timer.start("select")
        eng.select(flags, ref, region.start, region.emit_start, region.emit_end, cap, pos=pos, n_dev=n_dev, targets=targets, sites=sites)
        timer.stop()
        self.launches += 3
        if self.blocking_sync:
            if not hasattr(self, "_n_host"):
                self._n_host = torch.empty(1, dtype=torch.int32).pin_memory()
                self._n_ev = torch.cuda.Event(blocking=True)
            self._n_host.copy_(n_dev, non_blocking=True)
            self._n_ev.record()
            self._n_ev.synchronize()
            n = int(self._n_host[0])
        else:
            n = int(n_dev.item())                # the one host sync per region
        eng.check_status()
        gt = self._buf("gt", (max(n, 1), _lib.GT_CLASSES), torch.float32)[:n]
        zy = self._buf("zy", (max(n, 1), _lib.ZY_CLASSES), torch.float32)[:n]
        # fused s1 -> s2 hand-off: the model (and the record kernel) read each site's rows straight from the count tensor, the
        # [n,33,18] window tensor of the dataset seam is only materialised when the caller wants it (keep_windows) or for the
        # fp32 parity path
        fused = self.fused and self.records and not self.keep_windows and self.model.tensor_core
        if fused:
            if n:
                timer.start("model")
                self.model.from_counts(counts, region.start, pos, n, gt=gt, zy=zy)
                timer.stop()
                chunks = -(-n // 75776)
                self.launches += 2 * chunks + 1 + (6 if (self.model.precision == _lib.PREC_F16X1 and n > 16384) else 0)   # + margin, gather, 2 LSTM, tail, scatter
            rec = self._buf("rec", (max(n, 1), 32), torch.uint8)[:n]
            if n:
                eng.site_records_from_counts(gt, zy, counts, region.start, ref, pos, n, rec=rec)
                self.launches += 1
            return RegionOutput(n, pos[:n], None, None, gt, zy, None, rec)
        x = self._buf("x", (max(n, 1), _lib.WINDOW, _lib.CHANNELS), torch.int32)[:n]
        refbase = self._buf("refbase", (max(n, 1),), torch.uint8)[:n]
        if n:
            timer.start("gather")
            eng.gather(counts, ref, region.start, pos, n_dev, n, x_i32=x, refbase=refbase)
            timer.stop()
            timer.start("model")
            self.model(x, gt=gt, zy=zy)
            timer.stop()
            chunks = -(-n // 75776)
            self.launches += 1 + (2 * chunks + 1 + (6 if (self.model.precision == _lib.PREC_F16X1 and n > 16384) else 0) if self.model.tensor_core else 3 * chunks)   # gather + LSTM layers per chunk + tail
        if self.records:
            rec = self._buf("rec", (max(n, 1), 32), torch.uint8)[:n]
            if n:
                eng.site_records(gt, zy, x, refbase, pos, n, rec=rec)
                self.launches += 1
            return RegionOutput(n, pos[:n], refbase, None, gt, zy, x if self.keep_windows else None, rec)
        cov8 = x[:, 16, COV_CHANNELS].to(torch.float32) if n else torch.empty((0, 8), dtype=torch.float32, device=self.device)
        return RegionOutput(n, pos[:n], refbase, cov8, gt, zy, x if self.keep_windows else None)

    # ---- host-buffer mode, pipelined: H2D of region k+1 and D2H of region k-1 overlap the kernels of region k ----
    def run_host_many(self, host_regions, regions, ref: torch.Tensor, host_outs, consume=None, targets=None):
        """host_regions: PackedReads of pinned host tensors, one per region; host_outs: two dicts of pinned result
        buffers (double buffered).  consume(k, result_dict) is called on the host once region k's results have landed
        (e.g. VCF formatting); it runs while the GPU works on later regions.  targets: optional per-region intervals (run_device).
        Returns the total site count."""
        dev = self.device
        main = torch.cuda.current_stream(dev)
        if not hasattr(self, "_copy_streams"):
            self._copy_streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
        up_s, down_s = self._copy_streams
        n_reg = len(regions)
        up_done = [None] * n_reg
        comp_done = [None] * n_reg
        down_done = [None] * n_reg
        results = [None] * n_reg
        dev_reads = [None] * n_reg

        def start_upload(k):
            with torch.cuda.stream(up_s):
                if k >= 2:
                    up_s.wait_event(comp_done[k - 2])            # buffer set k%2 is free once region k-2 has been computed
                dev_reads[k] = self.upload(host_regions[k], key=f"reads{k % 2}")
                ev = torch.cuda.Event(); ev.record(up_s); up_done[k] = ev

        handles = [None] * n_reg

        def finish(k):
            down_done[k].synchronize()
            if consume is not None:
                handles[k] = consume(k, results[k])             # may return a future (background host work on the pinned buffers)

        def release(k):
            if k >= 0 and handles[k] is not None and hasattr(handles[k], "result"):
                handles[k].result()
                handles[k] = None

        up_s.wait_stream(main)
        start_upload(0)
        total = 0
        for k in range(n_reg):
            if k + 1 < n_reg:
                if k + 1 >= 2 and comp_done[k - 1] is None:
                    raise RuntimeError("pipeline order")
                start_upload(k + 1)
            main.wait_event(up_done[k])
            out = self.run_device(dev_reads[k], ref, regions[k], targets=None if targets is None else targets[k])
            ev = torch.cuda.Event(); ev.record(main); comp_done[k] = ev
            # results: device -> device staging (so the next region can reuse the work buffers) -> pinned host
            ho = host_outs[k % 2]
            release(k - 2)                                        # the consumer of region k-2 is done with this pinned buffer set
            with torch.cuda.stream(down_s):
                down_s.wait_event(ev)
                res = {"n": out.n}
                for name in (("rec",) if self.records else ("pos0", "refbase", "cov8", "gt", "zy")):
                    t = getattr(out, name)
                    if ho[name].shape[0] < out.n:
                        raise _lib.NsnpError(_lib.E_WORKSPACE, f"host result buffer '{name}' too small for {out.n} sites")
                    h = ho[name][: out.n]
                    h.copy_(t, non_blocking=True)
                    res[name] = h
                ev2 = torch.cuda.Event(blocking=self.blocking_sync); ev2.record(down_s); down_done[k] = ev2
            main.wait_event(ev2)                                  # run_device's buffers are reused by region k+1
            results[k] = res
            total += out.n
            if k >= 1:
                finish(k - 1)                                     # host-side consumer of the previous region
        finish(n_reg - 1)
        release(n_reg - 2); release(n_reg - 1)
        return total

    # ---- host-buffer mode with the VCF text assembled on the GPU ---------------------------------------------------------
    def run_host_text(self, host_regions, regions, ref: torch.Tensor, textgen, write, targets=None, sites: bool = False) -> int:
        """Pinned host read arrays of consecutive regions of ONE contig -> H2D -> kernels -> compact records -> VCF text on
        the GPU (vcf_text.GpuVcfText, which carries partial 1000-site batches across regions) -> D2H of the text.
        write(memoryview) receives the text chunks in order.  H2D of region k+1 and D2H of chunk k-1 overlap the kernels of
        region k; the host does no per-record work.  targets, sites: optional per-region intervals and their mode (run_device).
        Returns the site count."""
        assert self.records, "run_host_text needs a RegionRunner(records=True)"
        dev = self.device
        main = torch.cuda.current_stream(dev)
        if not hasattr(self, "_copy_streams"):
            self._copy_streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
        up_s, down_s = self._copy_streams
        n_reg = len(regions)
        up_done = [None] * n_reg
        comp_done = [None] * n_reg
        dev_reads = [None] * n_reg

        def start_upload(k):
            with torch.cuda.stream(up_s):
                if k >= 2:
                    up_s.wait_event(comp_done[k - 2])
                dev_reads[k] = self.upload(host_regions[k], key=f"reads{k % 2}")
                ev = torch.cuda.Event(); ev.record(up_s); up_done[k] = ev

        up_s.wait_stream(main)
        if n_reg:
            start_upload(0)
        total = 0
        pending = None
        for k in range(n_reg):
            if k + 1 < n_reg:
                start_upload(k + 1)
            main.wait_event(up_done[k])
            out = self.run_device(dev_reads[k], ref, regions[k], targets=None if targets is None else targets[k], sites=sites)
            chunk = textgen.push(out.rec) if out.n else None        # copies the records: the work buffers are free again
            self.launches += 3 if chunk is not None else 0
            ev = torch.cuda.Event(); ev.record(main); comp_done[k] = ev
            total += out.n
            if pending is not None:                                   # its kernels finished before run_device's site-count sync
                write(textgen.fetch(pending, down_s))
            pending = chunk
        if pending is not None:
            write(textgen.fetch(pending, down_s))
        last = textgen.flush()
        if last is not None:
            self.launches += 3
            write(textgen.fetch(last, down_s))
        return total

    # ---- host-buffer mode, records kept on the device (multi-GPU: the text is made after the count / head exchange) ----------
    def run_host_collect(self, host_regions, regions, refs, on_region=None, targets=None) -> list:
        """Pinned host reads of arbitrary regions (refs[k]: the device reference of region k's contig) -> H2D -> kernels ->
        compact records, returned as one device tensor per region -- or handed to on_region(k, RegionOutput) right after region
        k's kernels were enqueued (e.g. ShardedVcfWriter.add_region).  The H2D of region k+1 overlaps the kernels of region k."""
        assert self.records
        dev = self.device
        main = torch.cuda.current_stream(dev)
        if not hasattr(self, "_copy_streams"):
            self._copy_streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
        up_s, _ = self._copy_streams
        n_reg = len(regions)
        up_done, comp_done, dev_reads, out = [None] * n_reg, [None] * n_reg, [None] * n_reg, [None] * n_reg

        def start_upload(k):
            with torch.cuda.stream(up_s):
                if k >= 2:
                    up_s.wait_event(comp_done[k - 2])
                dev_reads[k] = self.upload(host_regions[k], key=f"reads{k % 2}")
                ev = torch.cuda.Event(); ev.record(up_s); up_done[k] = ev

        up_s.wait_stream(main)
        if n_reg:
            start_upload(0)
        for k in range(n_reg):
            if k + 1 < n_reg:
                start_upload(k + 1)
            main.wait_event(up_done[k])
            o = self.run_device(dev_reads[k], refs[k], regions[k], targets=None if targets is None else targets[k])
            if on_region is not None:
                on_region(k, o)
                out[k] = o.n
            else:
                out[k] = o.rec.clone()
            ev = torch.cuda.Event(); ev.record(main); comp_done[k] = ev
        return out

    # ---- host-buffer mode: what a caller holding decoded reads in (pinned) host memory pays -------------
    def upload(self, host_reads: PackedReads, key: str = "reads") -> PackedReads:
        out = []
        for f in FIELDS:
            a = getattr(host_reads, f)
            if a is None:
                out.append(None)
                continue
            d = self._buf(f"{key}.{f}", tuple(a.shape), a.dtype)
            d.copy_(a, non_blocking=True)
            out.append(d)
        return PackedReads(*out)

    def run_host(self, host_reads: PackedReads, ref: torch.Tensor, region: Region, host_out: Optional[dict] = None,
                 timer: Optional[StageTimer] = None):
        timer = timer or StageTimer(False)
        timer.start("h2d")
        rd = self.upload(host_reads)
        timer.stop()
        out = self.run_device(rd, ref, region, timer)
        timer.start("d2h")
        res = {}
        for k in ("pos0", "refbase", "cov8", "gt", "zy"):
            t = getattr(out, k)
            if host_out is not None and k in host_out and host_out[k].shape[0] >= out.n:
                h = host_out[k][: out.n]
                h.copy_(t, non_blocking=True)
            else:
                h = t.to("cpu", non_blocking=False)
            res[k] = h
        timer.stop()
        res["n"] = out.n
        return res
