"""Whole-contig driver of the GPU s1+s2 path: regions with 16-bp halos -> RegionRunner -> per-contig VCF assembler.

This is what `predict.py` uses for read inputs (BAM / packed reads): it replaces make_predict_data.sh steps 1-5 and the
model + record loop of PileupModel/predict.py for one contig, keeping the reference's 1000-site batch composition.
"""
from __future__ import annotations

import os
from typing import Optional

import numpy as np
import torch

from .predict_io import ContigVcfAssembler
from .reads import PackedReads, max_reference_span, slice_reads
from .runner import RegionRunner
from .shard import assign_lpt, gather_to_rank0, plan_regions, read_range_for_region


def _pinned(reads: PackedReads) -> PackedReads:
    return reads.to_torch("cpu", pin=True)


def call_contig(runner: RegionRunner, reads: PackedReads, ref: np.ndarray, contig: str, sink, batch_size: int = 1000,
                region_len: int = 12_500_000, n_threads: int = 0, regions=None, targets=None) -> dict:
    """reads: numpy PackedReads of one contig (coordinate sorted).  Writes VCF records to `sink` (binary file-like).
    targets: optional per-region intervals, aligned with `regions` (shard.plan_target_units)."""
    L = int(len(ref))
    ref_dev = torch.from_numpy(np.ascontiguousarray(ref)).to(runner.device)
    regions = regions if regions is not None else plan_regions([(contig, L)], region_len)
    span = max_reference_span(reads) + 1
    host_regions = []
    for rg in regions:
        lo, hi = read_range_for_region(reads.pos, span, rg)
        host_regions.append(_pinned(slice_reads(reads, lo, hi)))
    cap = max(4096, max(rg.emit_end - rg.emit_start for rg in regions))

    def pinned_out():
        if runner.records:
            return {"rec": torch.empty((cap, 32), dtype=torch.uint8).pin_memory()}
        return {"pos0": torch.empty(cap, dtype=torch.int32).pin_memory(), "refbase": torch.empty(cap, dtype=torch.uint8).pin_memory(),
                "cov8": torch.empty((cap, 8), dtype=torch.float32).pin_memory(), "gt": torch.empty((cap, 21), dtype=torch.float32).pin_memory(),
                "zy": torch.empty((cap, 3), dtype=torch.float32).pin_memory()}
    host_outs = (pinned_out(), pinned_out())
    asm = ContigVcfAssembler(contig, batch_size, n_threads, sink)

    def consume(k, res):
        if runner.records:
            asm.add_records(res["rec"].numpy())
        else:
            asm.add(res["pos0"].numpy(), res["refbase"].numpy(), res["gt"].numpy(), res["zy"].numpy(), res["cov8"].numpy())
        return None
    n = runner.run_host_many(host_regions, regions, ref_dev, host_outs, consume, targets)
    nbytes = asm.close()
    return {"sites": n, "vcf_bytes": nbytes, "regions": len(regions)}


def call_contig_text(runner: RegionRunner, reads: PackedReads, ref: np.ndarray, contig: str, sink, batch_size: int = 1000,
                     region_len: int = 12_500_000, regions=None, region_reads=None, targets=None) -> dict:
    """call_contig with the VCF text assembled on the GPU (csrc/vcf_dev.cu): the host only writes the bytes.
    region_reads: optional ready-made per-region PackedReads (e.g. BamReader.fetch); else `reads` is sliced.
    targets: optional per-region intervals, aligned with `regions` (shard.plan_target_units)."""
    from .vcf_text import GpuVcfText
    L = int(len(ref))
    ref_dev = torch.from_numpy(np.ascontiguousarray(ref)).to(runner.device)
    regions = regions if regions is not None else plan_regions([(contig, L)], region_len)
    if region_reads is None:
        span = max_reference_span(reads) + 1
        region_reads = [slice_reads(reads, *read_range_for_region(reads.pos, span, rg)) for rg in regions]
    host_regions = [_pinned(r) for r in region_reads]
    gen = GpuVcfText(runner.device, contig, batch_size)
    nbytes = [0]

    def write(mv):
        nbytes[0] += len(mv)
        if sink is not None:
            sink.write(mv)
    n = runner.run_host_text(host_regions, regions, ref_dev, gen, write, targets)
    return {"sites": n, "vcf_bytes": nbytes[0], "regions": len(regions)}


def records_of_regions(runner: RegionRunner, reads: PackedReads, ref: np.ndarray, regions) -> list:
    """Compact site records (uint8 [n, 32] copies, one array per region) of some regions of one contig."""
    assert runner.records, "records_of_regions needs a RegionRunner(records=True)"
    if not regions:
        return []
    ref_dev = torch.from_numpy(np.ascontiguousarray(ref)).to(runner.device)
    span = max_reference_span(reads) + 1
    host_regions = []
    for rg in regions:
        lo, hi = read_range_for_region(reads.pos, span, rg)
        host_regions.append(_pinned(slice_reads(reads, lo, hi)))
    cap = max(4096, max(rg.emit_end - rg.emit_start for rg in regions))
    host_outs = tuple({"rec": torch.empty((cap, 32), dtype=torch.uint8).pin_memory()} for _ in range(2))
    out = [None] * len(regions)

    def consume(k, res):
        out[k] = res["rec"].numpy().copy()            # the pinned buffer is reused two regions later
        return None
    runner.run_host_many(host_regions, regions, ref_dev, host_outs, consume)
    return out


def call_contigs_sharded(contigs, produce, sink, batch_size: int = 1000, region_len: int = 12_500_000, n_threads: int = 0) -> dict:
    """Multi-GPU driver (one process per GPU, torch.distributed already initialised or a single process).

    contigs: [(name, length)] in output order.  Every rank plans the same regions, takes its LPT share and calls
    produce(contig_index, regions_of_that_contig) -> [records per region].  The per-region records are gathered to
    rank 0, put back into (contig, position) order and only then cut into the reference's 1000-site batches per contig
    (predict.py's record logic depends on the batch composition), so the text is identical to a single-GPU run.
    Only rank 0 writes to `sink`; it returns the totals, the other ranks return None."""
    import torch.distributed as dist
    from .predict_io import RECORD_DTYPE
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    regions = plan_regions(contigs, region_len)
    mine = assign_lpt(regions, world)[rank]
    parts = []
    for ci in sorted({regions[i].contig_index for i in mine}):
        rgs = [regions[i] for i in mine if regions[i].contig_index == ci]
        for rec in produce(ci, rgs):
            rec = np.ascontiguousarray(rec)
            view = rec.view(RECORD_DTYPE).reshape(-1) if rec.dtype != RECORD_DTYPE else rec
            parts.append({"contig_index": np.full(len(view), ci, np.int32), "pos": view["pos1"].astype(np.int64), "rec": view})
    merged = gather_to_rank0(parts)
    if rank != 0:
        return None
    sites = nbytes = 0
    if merged:
        for ci, (name, _) in enumerate(contigs):
            sel = merged["rec"][merged["contig_index"] == ci]
            if len(sel) == 0:
                continue
            asm = ContigVcfAssembler(name, batch_size, n_threads, sink)
            asm.add_records(sel)
            nbytes += asm.close()
            sites += len(sel)
    return {"sites": sites, "vcf_bytes": nbytes, "regions": len(regions), "world": world}


# ---- multi-GPU: records stay on the rank that computed them; only counts, batch heads and text lengths are exchanged ----------
def _all_reduce(t, op):
    """t: CPU tensor.  NCCL needs device tensors: round-trip through the current device."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return t
    if dist.get_backend() == "nccl":
        d = t.cuda()
        dist.all_reduce(d, op=op)
        return d.cpu()
    dist.all_reduce(t, op=op)
    return t


class ShardedVcfWriter:
    """Every rank holds the compact site records of ITS regions and writes their text itself, at the right place of ONE
    ordered file (see write()).  Buffers (device text / workspaces / batch-head table, pinned host text) persist across calls."""

    def __init__(self, contigs, regions, batch_size: int = 1000, device=None):
        from . import _lib
        self.lib = _lib.load()
        self.contigs, self.regions, self.batch, self.device = list(contigs), list(regions), int(batch_size), device
        self._dev = {}
        self._host = {}
        self._pool = None
        self.write_threads = max(1, min(16, (os.cpu_count() or 1) // max(1, int(os.environ.get("WORLD_SIZE", "1")))))

    def _dbuf(self, key, nbytes, dtype=torch.uint8):
        t = self._dev.get(key)
        if t is None or t.numel() * t.element_size() < nbytes:
            t = torch.empty(int(nbytes * 1.15) // torch.empty((), dtype=dtype).element_size() + 64, dtype=dtype, device=self.device)
            self._dev[key] = t
        return t

    def _hbuf(self, key, n, dtype=torch.uint8):
        t = self._host.get(key)
        if t is None or t.numel() < n:
            t = torch.empty(int(n * 1.15) + 64, dtype=dtype).pin_memory()
            self._host[key] = t
        return t

    def write(self, out_path: Optional[str], header: bytes, records_by_region: dict) -> dict:
        """out_path None: stop once every rank holds its text segments in pinned host memory and knows their file offsets
        (self.segments: [(memoryview, offset)]); the caller places them.  records_by_region: region index -> uint8 [n,32] torch tensor on `device`, or a host RECORD_DTYPE / uint8 array.

          1. SUM all-reduce of the per-region site counts  -> every region's first site index inside its contig file;
          2. MIN all-reduce of the batch-head table        -> the genotype argmax of the first ten sites of every 1000-site batch
                                                              of every contig (what predict.py's `gt_output[ti]` reads; 10 B per batch);
          3. each rank formats its regions (GPU kernels for device records, all regions enqueued back to back; the host twin
             otherwise) -- byte-identical to one process formatting the merged list, because batches are counted from the
             contig's first site either way;
          4. SUM all-reduce of the per-region text lengths -> file offsets; every rank pwrite()s its segments, rank 0 the header.

        No record ever crosses ranks (the r01 path pickled all of them to rank 0 and formatted there)."""
        import ctypes as C
        import torch.distributed as dist
        from . import _lib
        from .predict_io import RECORD_DTYPE
        lib, regions, contigs, batch = self.lib, self.regions, self.contigs, self.batch
        import time
        tr = [("start", time.perf_counter())]
        mark = lambda name: tr.append((name, time.perf_counter()))
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        rank = dist.get_rank() if world > 1 else 0
        n_reg = len(regions)
        counts = torch.zeros(n_reg, dtype=torch.int64)
        for i, rec in records_by_region.items():
            counts[i] = int(rec.shape[0])
        counts = _all_reduce(counts, dist.ReduceOp.SUM if world > 1 else None)
        mark("counts")
        first = [0] * n_reg                                        # first site index of each region inside its contig
        tot = {}
        for i, rg in enumerate(regions):
            first[i] = tot.get(rg.contig_index, 0)
            tot[rg.contig_index] = first[i] + int(counts[i])
        nb = {ci: (n + batch - 1) // batch for ci, n in tot.items()}
        hoff, o = {}, 0
        for ci in sorted(nb):
            hoff[ci] = o; o += nb[ci]
        mine = sorted(records_by_region)
        on_gpu = any(isinstance(r, torch.Tensor) and r.is_cuda for r in records_by_region.values())
        texts = {}                                                 # region index -> memoryview / bytes
        if on_gpu:
            stream = torch.cuda.current_stream(self.device).cuda_stream
            heads = self._dbuf("heads", max(o, 1) * 10)[: max(o, 1) * 10].view(-1, 10)
            heads.fill_(255)
            with torch.cuda.device(self.device):
                for i in mine:
                    rec = records_by_region[i]
                    ci = regions[i].contig_index
                    if rec.shape[0]:
                        _lib.check(lib.nsnp_vcf_batch_heads(rec.data_ptr(), int(rec.shape[0]), 0, first[i], batch,
                                                            heads[hoff[ci]:].data_ptr(), stream))
            if world > 1:
                if dist.get_backend() == "nccl":
                    dist.all_reduce(heads, op=dist.ReduceOp.MIN)
                else:
                    heads.copy_(_all_reduce(heads.cpu(), dist.ReduceOp.MIN))
            mark("heads")
            # all text kernels of my regions back to back, each into its own slice of one device buffer
            caps = [int(lib.nsnp_vcf_text_capacity(int(records_by_region[i].shape[0]), contigs[regions[i].contig_index][0].encode())) for i in mine]
            wss = [(int(lib.nsnp_vcf_text_workspace_bytes(int(records_by_region[i].shape[0]))) + 255) // 256 * 256 for i in mine]
            toff = np.concatenate([[0], np.cumsum(caps)]).astype(np.int64)
            woff = np.concatenate([[0], np.cumsum(wss)]).astype(np.int64)
            text_dev = self._dbuf("text", int(toff[-1]) + 256)
            ws_dev = self._dbuf("ws", int(woff[-1]) + 256)
            meta_dev = self._dbuf("meta", 8 * (len(mine) + 1), torch.int64)
            tie_cnt_off, tie_ent_off = [], []
            with torch.cuda.device(self.device):
                for k, i in enumerate(mine):
                    rec = records_by_region[i]
                    ci = regions[i].contig_index
                    n = int(rec.shape[0])
                    wp = ws_dev.data_ptr() + int(woff[k])
                    _lib.check(lib.nsnp_vcf_text_records(contigs[ci][0].encode(), rec.data_ptr() if n else 0, n, 0, first[i], batch,
                                                         heads[hoff[ci]:].data_ptr(), text_dev.data_ptr() + int(toff[k]), caps[k],
                                                         meta_dev.data_ptr() + 8 * k, wp, wss[k], stream))
                    cp = C.c_void_p(); ep = C.c_void_p(); cap = C.c_int32(0)
                    lib.nsnp_vcf_text_ties(wp, n, C.byref(cp), C.byref(ep), C.byref(cap))
                    tie_cnt_off.append((cp.value or wp) - ws_dev.data_ptr()); tie_ent_off.append((ep.value or wp) - ws_dev.data_ptr())
            meta_h = self._hbuf("meta", len(mine) + 1, torch.int64)
            ties_n = self._hbuf("ties_n", len(mine) + 1, torch.int32)
            meta_h[:len(mine)].copy_(meta_dev[:len(mine)], non_blocking=True)
            for k, i in enumerate(mine):
                if records_by_region[i].shape[0]:
                    ties_n[k:k + 1].copy_(ws_dev[tie_cnt_off[k]:tie_cnt_off[k] + 4].view(torch.int32), non_blocking=True)
                else:
                    ties_n[k] = 0
            torch.cuda.current_stream(self.device).synchronize()
            mark("text kernels")
            lens = [int(meta_h[k]) if records_by_region[i].shape[0] else 0 for k, i in enumerate(mine)]
            for k, ln in enumerate(lens):
                if ln > caps[k]:
                    raise _lib.NsnpError(_lib.E_WORKSPACE, "VCF text buffer too small")
            slack = 64                                             # a tie fix-up can lengthen a record by a digit
            hoffs = np.concatenate([[0], np.cumsum([ln + slack for ln in lens])]).astype(np.int64)
            text_h = self._hbuf("text", int(hoffs[-1]) + 64)
            ties_h = self._hbuf("ties", 64 * 4096 * max(1, sum(1 for k in range(len(mine)) if int(ties_n[k]) > 0)))
            tie_slot = {}
            for k, ln in enumerate(lens):
                if ln:
                    text_h[int(hoffs[k]):int(hoffs[k]) + ln].copy_(text_dev[int(toff[k]):int(toff[k]) + ln], non_blocking=True)
                nt = int(ties_n[k])
                if nt > 4096:
                    raise _lib.NsnpError(_lib.E_OVERFLOW, f"{nt} rounding-tie records in one region")
                if nt > 0:
                    slot = len(tie_slot) * 64 * 4096
                    tie_slot[k] = slot
                    ties_h[slot:slot + 64 * nt].copy_(ws_dev[tie_ent_off[k]:tie_ent_off[k] + 64 * nt], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            mark("d2h")
            mv = memoryview(text_h.numpy())
            for k, i in enumerate(mine):
                ln = lens[k]
                if k in tie_slot:
                    ci = regions[i].contig_index
                    w = lib.nsnp_vcf_text_patch_ties(contigs[ci][0].encode(), text_h.data_ptr() + int(hoffs[k]), ln, ln + slack,
                                                     ties_h.data_ptr() + tie_slot[k], int(ties_n[k]))
                    if w <= 0 and ln > 0:
                        raise _lib.NsnpError(_lib.E_WORKSPACE, "tie fix-up of the VCF text failed")
                    ln = int(w)
                texts[i] = mv[int(hoffs[k]):int(hoffs[k]) + ln]
        else:
            heads_np = np.full((max(o, 1), 10), 255, np.uint8)
            for i in mine:
                ci = regions[i].contig_index
                r = np.ascontiguousarray(records_by_region[i]).view(RECORD_DTYPE).reshape(-1)
                g = first[i] + np.arange(len(r))
                sel = (g % batch) < 10
                heads_np[hoff[ci] + g[sel] // batch, g[sel] % batch] = r["gt"][sel]
            heads_np = _all_reduce(torch.from_numpy(heads_np), dist.ReduceOp.MIN if world > 1 else None).numpy()
            for i in mine:
                ci = regions[i].contig_index
                r = np.ascontiguousarray(records_by_region[i]).view(RECORD_DTYPE).reshape(-1)
                if len(r) == 0:
                    texts[i] = b""
                    continue
                cap = len(r) * (96 + len(contigs[ci][0])) + 256
                buf = np.empty(cap, np.uint8)
                h = np.ascontiguousarray(heads_np[hoff[ci]:hoff[ci] + nb[ci]])
                w = lib.nsnp_vcf_format_records_at(contigs[ci][0].encode(), r.ctypes.data, len(r), first[i], batch, h.ctypes.data,
                                                   buf.ctypes.data, cap)
                if w < 0:
                    raise _lib.NsnpError(_lib.E_WORKSPACE, "VCF text buffer too small")
                texts[i] = buf[:w].tobytes()
        mark("patch")
        return self._place(out_path, header, texts, counts, n_reg, world, rank, mark, tr)

    def _place(self, out_path, header, texts, counts, n_reg, world, rank, mark=None, tr=None):
        import torch.distributed as dist
        if mark is None:
            import time
            tr = [("start", time.perf_counter())]
            mark = lambda name: tr.append((name, time.perf_counter()))
        # 4. offsets, ordered file
        lens_t = torch.zeros(n_reg, dtype=torch.int64)
        for i, t in texts.items():
            lens_t[i] = len(t)
        lens_t = _all_reduce(lens_t, dist.ReduceOp.SUM if world > 1 else None)
        offs = np.concatenate([[len(header)], len(header) + np.cumsum(lens_t.numpy())])
        mark("lengths")
        self.segments = [(t, int(offs[i])) for i, t in texts.items() if len(t)]
        if out_path is None:
            return {"sites": int(counts.sum()), "vcf_bytes": int(offs[-1]) - len(header), "regions": n_reg, "world": world}
        if rank == 0:
            # an existing file keeps its pages: only its size changes (a fresh tmpfs / page-cache allocation costs more than the copy)
            fd0 = os.open(out_path, os.O_WRONLY | os.O_CREAT, 0o644)
            try:
                os.ftruncate(fd0, int(offs[-1]))
                os.pwrite(fd0, header, 0)
            finally:
                os.close(fd0)
        if world > 1:
            dist.barrier()
        mark("create")
        # every rank copies its segments into a shared mapping of the file: concurrent pwrite()s to one file serialise on the
        # inode lock (3 GB/s for the whole box), page-wise copies into a mapping do not.  ctypes.memmove releases the GIL.
        import ctypes as C2
        import mmap
        segs = [(t, int(offs[i])) for i, t in texts.items() if len(t)]
        if segs:
            fd = os.open(out_path, os.O_RDWR)
            try:
                mm = mmap.mmap(fd, int(offs[-1]), mmap.MAP_SHARED, mmap.PROT_READ | mmap.PROT_WRITE)
            finally:
                os.close(fd)
            try:
                base = C2.addressof(C2.c_char.from_buffer(mm))
                jobs = []
                for t, o_ in segs:
                    src = np.frombuffer(t, np.uint8)
                    for c in range(0, len(src), 8 << 20):
                        jobs.append((base + o_ + c, src[c:c + (8 << 20)]))
                move = lambda j: C2.memmove(j[0], j[1].ctypes.data, j[1].shape[0])
                if len(jobs) > 1 and self.write_threads > 1:
                    from concurrent.futures import ThreadPoolExecutor
                    if self._pool is None:
                        self._pool = ThreadPoolExecutor(self.write_threads)
                    list(self._pool.map(move, jobs))
                else:
                    for j in jobs:
                        move(j)
                del base
            finally:
                mm.close()
        mark("pwrite")
        if world > 1:
            dist.barrier()
        if os.environ.get("NSNP_TRACE") and rank == 0:
            import sys
            print("ShardedVcfWriter " + " ".join(f"{b[0]}={1e3 * (b[1] - a[1]):.1f}ms" for a, b in zip(tr[:-1], tr[1:])), file=sys.stderr)
        return {"sites": int(counts.sum()), "vcf_bytes": int(offs[-1]) - len(header), "regions": n_reg, "world": world}


    # ---- streaming form: text while the regions are still being computed ------------------------------------------------
    # begin() / add_region(i, rec) right after region i's kernels were enqueued / finish(out_path, header).  A region's text is
    # made at once with deferred batch heads (nsnp_vcf_text_records_deferred) and copied to pinned host memory while the next
    # region computes; after the last region only the counts / head table / length all-reduces, the one-character ALT fix-ups
    # and the tie fix-ups remain.  Same bytes as write().
    def begin(self):
        self._st = {"idx": [], "recs": [], "off": [], "len": [], "fix": [], "ties": [], "pending": None, "k": 0, "text_used": 0,
                    "fix_used": 0, "tie_used": 0}
        if not hasattr(self, "_down"):
            self._down = torch.cuda.Stream(self.device)

    def _stage(self, key, used, extra, dtype=torch.uint8):
        """pinned staging that keeps its content when it grows"""
        t = self._host.get(key)
        if t is None or t.numel() < used + extra:
            self._down.synchronize()
            n = max(int((used + extra) * 1.5), 64 << 20 if key == "s_text" else 1 << 20)
            nt = torch.empty(n, dtype=dtype).pin_memory()
            if t is not None and used:
                nt[:used].copy_(t[:used])
            self._host[key] = t = nt
        return t

    def _collect_pending(self):
        st = self._st
        p = st["pending"]
        if p is None:
            return
        st["pending"] = None
        i, n, bufs, ev, cnt_off, ent_off, fcnt_off, fent_off = p
        ev.synchronize()
        meta = self._hbuf("s_meta", 8, torch.int64)
        cnts = self._hbuf("s_cnts", 8, torch.int32)
        with torch.cuda.stream(self._down):
            meta[:1].copy_(bufs["meta"][:1], non_blocking=True)
            cnts[0:1].copy_(bufs["ws"][cnt_off:cnt_off + 4].view(torch.int32), non_blocking=True)
            cnts[1:2].copy_(bufs["ws"][fcnt_off:fcnt_off + 4].view(torch.int32), non_blocking=True)
        self._down.synchronize()
        ln, nt, nf = int(meta[0]), int(cnts[0]), int(cnts[1])
        if ln > bufs["text"].numel() or nt > 4096 or nf > n:
            raise _lib_mod().NsnpError(-4, f"VCF text buffers too small for region {i} ({ln} bytes, {nt} ties, {nf} fix-ups)")
        slack = 64
        text_h = self._stage("s_text", st["text_used"], ln + slack)
        fix_h = self._stage("s_fix", st["fix_used"], 16 * nf)
        tie_h = self._stage("s_tie", st["tie_used"], 64 * nt)
        with torch.cuda.stream(self._down):
            if ln:
                text_h[st["text_used"]:st["text_used"] + ln].copy_(bufs["text"][:ln], non_blocking=True)
            if nf:
                fix_h[st["fix_used"]:st["fix_used"] + 16 * nf].copy_(bufs["ws"][fent_off:fent_off + 16 * nf], non_blocking=True)
            if nt:
                tie_h[st["tie_used"]:st["tie_used"] + 64 * nt].copy_(bufs["ws"][ent_off:ent_off + 64 * nt], non_blocking=True)
            done = torch.cuda.Event(); done.record(self._down)
        bufs["free"] = done                                     # the device buffers may be overwritten once this copy is done
        st["off"].append(st["text_used"]); st["len"].append(ln)
        st["fix"].append((st["fix_used"], nf)); st["ties"].append((st["tie_used"], nt))
        st["text_used"] += ln + slack; st["fix_used"] += 16 * nf; st["tie_used"] += 64 * nt

    def add_region(self, i: int, rec: torch.Tensor):
        """rec: uint8 [n,32] device records of region i, just enqueued on the current stream (the buffer may be reused afterwards)."""
        import ctypes as C
        lib = self.lib
        st = self._st
        self._collect_pending()
        n = int(rec.shape[0])
        st["idx"].append(i)
        st["recs"].append(rec.clone())
        if n == 0:
            st["off"].append(st["text_used"]); st["len"].append(0); st["fix"].append((st["fix_used"], 0)); st["ties"].append((st["tie_used"], 0))
            return
        contig = self.contigs[self.regions[i].contig_index][0].encode()
        bufs = self._dev.setdefault(("stream", st["k"] % 2), {})
        st["k"] += 1
        cap = int(lib.nsnp_vcf_text_capacity(n, contig)); wsb = int(lib.nsnp_vcf_text_workspace_bytes(n))
        if "free" in bufs:
            torch.cuda.current_stream(self.device).wait_event(bufs["free"])
        if "text" not in bufs or bufs["text"].numel() < cap:
            bufs["text"] = torch.empty(int(cap * 1.2) + 256, dtype=torch.uint8, device=self.device)
        if "ws" not in bufs or bufs["ws"].numel() < wsb:
            bufs["ws"] = torch.empty(int(wsb * 1.2) + 256, dtype=torch.uint8, device=self.device)
        if "meta" not in bufs:
            bufs["meta"] = torch.zeros(2, dtype=torch.int64, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            _lib_mod().check(lib.nsnp_vcf_text_records_deferred(contig, st["recs"][-1].data_ptr(), n, 0, bufs["text"].data_ptr(), bufs["text"].numel(),
                                                                bufs["meta"].data_ptr(), bufs["ws"].data_ptr(), bufs["ws"].numel(), stream))
        cp = C.c_void_p(); ep = C.c_void_p(); cap_t = C.c_int32(0); fc = C.c_void_p(); fe = C.c_void_p()
        lib.nsnp_vcf_text_ties(bufs["ws"].data_ptr(), n, C.byref(cp), C.byref(ep), C.byref(cap_t))
        lib.nsnp_vcf_text_fixups(bufs["ws"].data_ptr(), n, C.byref(fc), C.byref(fe))
        base = bufs["ws"].data_ptr()
        ev = torch.cuda.Event(); ev.record(torch.cuda.current_stream(self.device))
        st["pending"] = (i, n, bufs, ev, cp.value - base, ep.value - base, fc.value - base, fe.value - base)

    def finish(self, out_path: Optional[str], header: bytes) -> dict:
        import ctypes as C
        import torch.distributed as dist
        lib, regions, contigs, batch = self.lib, self.regions, self.contigs, self.batch
        st = self._st
        self._collect_pending()
        self._down.synchronize()
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        rank = dist.get_rank() if world > 1 else 0
        n_reg = len(regions)
        counts = torch.zeros(n_reg, dtype=torch.int64)
        for i, rec in zip(st["idx"], st["recs"]):
            counts[i] = int(rec.shape[0])
        counts = _all_reduce(counts, dist.ReduceOp.SUM if world > 1 else None)
        first = [0] * n_reg
        tot = {}
        for i, rg in enumerate(regions):
            first[i] = tot.get(rg.contig_index, 0)
            tot[rg.contig_index] = first[i] + int(counts[i])
        nb = {ci: (n + batch - 1) // batch for ci, n in tot.items()}
        hoff, o = {}, 0
        for ci in sorted(nb):
            hoff[ci] = o; o += nb[ci]
        stream = torch.cuda.current_stream(self.device).cuda_stream
        heads = self._dbuf("heads", max(o, 1) * 10)[: max(o, 1) * 10].view(-1, 10)
        heads.fill_(255)
        with torch.cuda.device(self.device):
            for i, rec in zip(st["idx"], st["recs"]):
                if rec.shape[0]:
                    _lib_mod().check(lib.nsnp_vcf_batch_heads(rec.data_ptr(), int(rec.shape[0]), 0, first[i], batch,
                                                              heads[hoff[regions[i].contig_index]:].data_ptr(), stream))
        if world > 1:
            if dist.get_backend() == "nccl":
                dist.all_reduce(heads, op=dist.ReduceOp.MIN)
            else:
                heads.copy_(_all_reduce(heads.cpu(), dist.ReduceOp.MIN))
        heads_h = heads.cpu().numpy()
        text_h = self._host.get("s_text"); fix_h = self._host.get("s_fix"); tie_h = self._host.get("s_tie")
        mv = memoryview(text_h.numpy()) if text_h is not None else memoryview(b"")
        texts = {}
        for k, i in enumerate(st["idx"]):
            ln = st["len"][k]
            if ln == 0:
                texts[i] = b""
                continue
            ci = regions[i].contig_index
            table = np.ascontiguousarray(heads_h[hoff[ci]:hoff[ci] + nb[ci]])
            base_ptr = text_h.data_ptr() + st["off"][k]
            fo, nf = st["fix"][k]
            drops = C.c_int32(0)
            if nf:
                _lib_mod().check(lib.nsnp_vcf_text_patch_heads(base_ptr, ln, fix_h.data_ptr() + fo, nf, first[i], batch, table.ctypes.data, C.byref(drops)))
            if drops.value:
                # a fix-up record of a batch with fewer than ten sites (the last batch of a contig): format this region exactly
                rec = st["recs"][k]
                g = self._gen_for(ci)
                texts[i] = bytes(g.fetch(g.format_at(rec, first[i], heads[hoff[ci]:hoff[ci] + nb[ci]])))
                continue
            to, nt = st["ties"][k]
            if nt:
                w = lib.nsnp_vcf_text_patch_ties_at(contigs[ci][0].encode(), base_ptr, ln, ln + 64, tie_h.data_ptr() + to, nt, first[i], batch, table.ctypes.data)
                if w <= 0:
                    raise _lib_mod().NsnpError(-3, "tie fix-up of the VCF text failed")
                ln = int(w)
            texts[i] = mv[st["off"][k]:st["off"][k] + ln]
        st["recs"] = []
        return self._place(out_path, header, texts, counts, n_reg, world, rank)

    def _gen_for(self, ci):
        from .vcf_text import GpuVcfText
        if not hasattr(self, "_gens"):
            self._gens = {}
        if ci not in self._gens:
            self._gens[ci] = GpuVcfText(self.device, self.contigs[ci][0], self.batch)
        return self._gens[ci]


def _lib_mod():
    from . import _lib
    return _lib


def write_sharded_vcf(out_path: str, header: bytes, contigs, regions, records_by_region: dict, batch_size: int = 1000, device=None) -> dict:
    """One-shot form of ShardedVcfWriter.write."""
    return ShardedVcfWriter(contigs, regions, batch_size, device).write(out_path, header, records_by_region)
