"""Flat packed read arrays (struct nsnp_reads of include/nanosnp_b200.h).

This is the hand-off format between a host BAM decoder and the GPU path: it replaces the
BAM -> `samtools mpileup` text -> per-contig text files chain of
dna_sv_tensor/src/scripts/make_predict_data.sh:147-176.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _lib

FIELDS = ("pos", "flag", "mapq", "cigar_off", "cigar", "seq_off", "seq2", "nmask")
DTYPES = {"pos": np.int32, "flag": np.uint16, "mapq": np.uint8, "cigar_off": np.int64, "cigar": np.uint32,      # cigar: uint16 when packed by cigar16()
          "seq_off": np.int64, "seq2": np.uint8, "nmask": np.uint8}

CIGAR_OPS = "MIDNSHP=X"


@dataclass
class PackedReads:
    """Reads of one contig, sorted by pos.  Arrays are numpy (host) or torch (host-pinned / device)."""
    pos: object
    flag: object
    mapq: object
    cigar_off: object          # [n+1]
    cigar: object
    seq_off: object            # [n]
    seq2: object
    nmask: Optional[object] = None

    @property
    def n_reads(self) -> int:
        return int(self.pos.shape[0])

    @property
    def n_cigar(self) -> int:
        return int(self.cigar.shape[0])

    @property
    def n_bases(self) -> int:
        return int(self.seq2.shape[0]) * 4

    def is_torch(self) -> bool:
        return not isinstance(self.pos, np.ndarray)

    def nbytes(self) -> int:
        tot = 0
        for f in FIELDS:
            a = getattr(self, f)
            if a is None:
                continue
            tot += a.nbytes if isinstance(a, np.ndarray) else a.numel() * a.element_size()
        return tot

    def _ptr(self, a) -> int:
        if a is None:
            return 0
        if isinstance(a, np.ndarray):
            assert a.flags["C_CONTIGUOUS"]
            return a.ctypes.data
        assert a.is_contiguous()
        return a.data_ptr()

    def as_struct(self) -> _lib.Reads:
        """ctypes view; the caller must keep `self` alive while the struct is in use."""
        r = _lib.Reads()
        r.n_reads = self.n_reads
        for f in FIELDS:
            setattr(r, f, self._ptr(getattr(self, f)))
        r.qual = 0
        r.n_cigar = self.n_cigar
        r.n_bases = self.n_bases
        r.cigar_bits = 16 if self.cigar.dtype in (np.uint16, np.int16) or str(self.cigar.dtype) in ("torch.int16", "torch.uint16") else 32
        return r

    def to_torch(self, device, pin: bool = False, non_blocking: bool = False) -> "PackedReads":
        import torch

        def conv(a):
            if a is None:
                return None
            if isinstance(a, np.ndarray):
                # torch has no uint16/uint32 arithmetic, but storage + data_ptr is all we need
                t = torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a.view(np.int32) if a.dtype == np.uint32 else a)
            else:
                t = a
            if pin and t.device.type == "cpu":
                t = t.pin_memory()
            return t.to(device, non_blocking=non_blocking)
        return PackedReads(*[conv(getattr(self, f)) for f in FIELDS])

    def to_numpy(self) -> "PackedReads":
        def conv(f, a):
            if a is None or isinstance(a, np.ndarray):
                return a
            h = a.detach().cpu().numpy()
            return h.view(np.uint16) if (f == "cigar" and h.dtype == np.int16) else h.view(DTYPES[f])
        return PackedReads(*[conv(f, getattr(self, f)) for f in FIELDS])

    def prefix(self, n: int) -> "PackedReads":
        """First n reads (host arrays only): the bounded CPU-baseline sample of bench.py."""
        assert isinstance(self.pos, np.ndarray)
        nc = int(self.cigar_off[n])
        # bases of the first n reads end where read n starts (reads are laid out in order)
        nb = int(self.seq_off[n]) if n < self.n_reads else self.n_bases
        nb4 = (nb + 3) // 4
        return PackedReads(self.pos[:n], self.flag[:n], self.mapq[:n], self.cigar_off[: n + 1], self.cigar[:nc],
                           self.seq_off[:n], self.seq2[:nb4], None if self.nmask is None else self.nmask[: (nb + 7) // 8])


def slice_reads(reads: "PackedReads", lo: int, hi: int) -> "PackedReads":
    """Reads [lo, hi) as a self-contained PackedReads (numpy): offsets rebased, arrays padded for the kernels' look-ahead."""
    assert isinstance(reads.pos, np.ndarray)
    n = reads.n_reads
    c0, c1 = int(reads.cigar_off[lo]), int(reads.cigar_off[hi])
    nb_total = reads.n_bases
    b0 = int(reads.seq_off[lo]) if lo < n else nb_total
    b1 = int(reads.seq_off[hi]) if hi < n else nb_total
    b0 -= b0 % 16                                   # keep 4-byte alignment of the sliced seq2 / nmask
    pad = np.zeros(16, np.uint8)
    seq2 = np.concatenate([reads.seq2[b0 // 4:(b1 + 3) // 4], pad])
    nmask = None if reads.nmask is None else np.concatenate([reads.nmask[b0 // 8:(b1 + 7) // 8], pad])
    return PackedReads(np.ascontiguousarray(reads.pos[lo:hi]), np.ascontiguousarray(reads.flag[lo:hi]), np.ascontiguousarray(reads.mapq[lo:hi]),
                       reads.cigar_off[lo:hi + 1] - c0, np.ascontiguousarray(reads.cigar[c0:c1]), reads.seq_off[lo:hi] - b0, seq2, nmask)


def canonicalize_cigars(reads: "PackedReads") -> "PackedReads":
    """Merges adjacent CIGAR ops of the same type ("1D2D" -> "3D", "1I2I" -> "3I"): `samtools mpileup` reports such runs as
    ONE indel, and the GPU path refuses unmerged runs (include/nanosnp_b200.h).  nsnp_bam_fill already does this while
    decoding; this is the numpy equivalent for hand-made inputs.  Host arrays only."""
    assert isinstance(reads.pos, np.ndarray)
    cg = reads.cigar.astype(np.uint32)
    if cg.shape[0] == 0:
        return reads
    ops = cg & 15
    first = np.ones(cg.shape[0], bool)
    first[1:] = ops[1:] != ops[:-1]
    first[reads.cigar_off[:-1][reads.cigar_off[:-1] < cg.shape[0]]] = True          # a read's first op always starts a group
    if first.all():
        return reads
    starts = np.nonzero(first)[0]
    lens = np.add.reduceat((cg >> 4).astype(np.int64), starts)
    merged = ((lens << 4) | ops[starts]).astype(np.uint32)
    new_off = np.concatenate([[0], np.cumsum(first)])[reads.cigar_off].astype(np.int64)
    return PackedReads(reads.pos, reads.flag, reads.mapq, new_off, merged, reads.seq_off, reads.seq2, reads.nmask)


def cigar16(reads: "PackedReads") -> "PackedReads":
    """The same reads with the CIGAR words as uint16 (struct nsnp_reads.cigar_bits = 16) when every op length is below 4096
    -- true for ONT / HiFi alignments except the occasional long clip -- else unchanged.  Halves the CIGAR bytes that cross
    PCIe (16 of the 23.5 bytes per reference position at 30x).  numpy or torch (host / device) arrays."""
    c = reads.cigar
    if isinstance(c, np.ndarray):
        if c.dtype == np.uint16 or (c.size and int(c.max()) >= (4096 << 4)):
            return reads
        c16 = c.astype(np.uint16)
    else:
        import torch
        if c.dtype == torch.int16:
            return reads
        if c.numel() and (int(c.max()) >= (4096 << 4) or int(c.min()) < 0):
            return reads
        c16 = c.to(torch.int16)                       # values < 65536: the bit pattern is the uint16 word
    return PackedReads(reads.pos, reads.flag, reads.mapq, reads.cigar_off, c16, reads.seq_off, reads.seq2, reads.nmask)


def max_reference_span(reads: "PackedReads") -> int:
    """Longest reference span of any read (host arrays): bounds how far back a region must look for overlapping reads."""
    ops = reads.cigar & 15
    rl = np.where((ops == 0) | (ops == 2) | (ops == 3) | (ops == 7) | (ops == 8), reads.cigar >> 4, 0).astype(np.int64)
    cs = np.concatenate([[0], np.cumsum(rl)])
    spans = cs[reads.cigar_off[1:]] - cs[reads.cigar_off[:-1]]
    return int(spans.max()) if len(spans) else 0


def reference_span(cigar: np.ndarray) -> int:
    ops = cigar & 15
    lens = cigar >> 4
    return int(lens[(ops == 0) | (ops == 2) | (ops == 3) | (ops == 7) | (ops == 8)].sum())


def from_records(records, with_nmask: bool = True) -> PackedReads:
    """Builds PackedReads from an iterable of (pos0, flag, mapq, cigar_string, seq_string) tuples (tests, small inputs)."""
    import re
    pos, flag, mapq, coff, cig, soff = [], [], [], [0], [], []
    bases = []
    nb = 0
    code = {"A": 0, "C": 1, "G": 2, "T": 3}
    for (p, f, q, cs, seq) in records:
        pos.append(p); flag.append(f); mapq.append(q)
        for m in re.finditer(r"(\d+)([MIDNSHP=X])", cs):
            cig.append((int(m.group(1)) << 4) | CIGAR_OPS.index(m.group(2)))
        coff.append(len(cig))
        soff.append(nb)
        bases.append(seq)
        nb += (len(seq) + 15) // 16 * 16
    # one code per base slot (reads start on 16-base boundaries; padding slots stay 0), 4 = not ACGT -> an nmask bit
    lut = np.full(256, 4, np.uint8)
    for ch, c in code.items():
        lut[ord(ch)] = lut[ord(ch.lower())] = c
    codes = np.zeros(nb + 16, np.uint8)
    for so, seq in zip(soff, bases):
        codes[so:so + len(seq)] = lut[np.frombuffer(seq.encode("latin-1"), np.uint8)]
    isn = codes == 4
    c2 = np.where(isn, 0, codes).astype(np.uint8)[: (nb + 3) // 4 * 4].reshape(-1, 4)
    seq2 = np.zeros((nb + 3) // 4 + 8, np.uint8)
    seq2[: c2.shape[0]] = c2[:, 0] | (c2[:, 1] << 2) | (c2[:, 2] << 4) | (c2[:, 3] << 6)
    nmask = np.zeros((nb + 7) // 8 + 8, np.uint8)
    nmask[: (nb + 7) // 8] = np.packbits(isn[: (nb + 7) // 8 * 8], bitorder="little")
    return PackedReads(np.asarray(pos, np.int32), np.asarray(flag, np.uint16), np.asarray(mapq, np.uint8),
                       np.asarray(coff, np.int64), np.asarray(cig, np.uint32), np.asarray(soff, np.int64), seq2,
                       nmask if with_nmask else None)
