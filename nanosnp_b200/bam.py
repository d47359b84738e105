"""BAM front end: BGZF inflate (zlib) + native record decode -> PackedReads per contig.

Replaces the BAM reading that `samtools mpileup` does for the reference (make_predict_data.sh:151): the host decodes the
BAM into the flat packed arrays the GPU path consumes.  A small BGZF/BAM writer is included for tests and for turning
synthetic reads into a file the reference's own tooling could read.
"""
from __future__ import annotations

import ctypes as C
import struct
import zlib
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import _lib
from .reads import PackedReads

_BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_decompress(path: str) -> bytes:
    """All BGZF members of a file, inflated and concatenated (test utility; the product path is the native streaming
    reader below).  Walks the blocks by their BSIZE field: linear in the file size."""
    with open(path, "rb") as f:
        data = memoryview(f.read())
    out, i, n = [], 0, len(data)
    while i < n:
        if n - i < 18 or data[i] != 31 or data[i + 1] != 139:
            raise ValueError("not a BGZF block")
        xlen = struct.unpack_from("<H", data, i + 10)[0]
        bsize, o = None, 0
        while o + 4 <= xlen:
            si1, si2, slen = struct.unpack_from("<BBH", data, i + 12 + o)
            if si1 == 66 and si2 == 67 and slen == 2:
                bsize = struct.unpack_from("<H", data, i + 16 + o)[0]
            o += 4 + slen
        if bsize is None:
            raise ValueError("BGZF block without a BC field")
        out.append(zlib.decompress(data[i + 12 + xlen:i + bsize + 1 - 8], -15))
        i += bsize + 1
    return b"".join(out)


def bgzf_compress(raw: bytes, level: int = 1, with_offsets: bool = False):
    """Proper BGZF: <= 64 KB blocks, each a gzip member with the BC extra field, plus the EOF marker block.
    with_offsets: also returns the file offset of every block (each holds 0xFF00 uncompressed bytes but the last)."""
    out = []
    offs, fpos = [], 0
    for s in range(0, len(raw), 0xFF00):
        offs.append(fpos)
        chunk = raw[s:s + 0xFF00]
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        comp = co.compress(chunk) + co.flush()
        bsize = len(comp) + 25
        out.append(struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, bsize))
        out.append(comp)
        out.append(struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))
        fpos += bsize + 1
    offs.append(fpos)
    out.append(_BGZF_EOF)
    return (b"".join(out), offs) if with_offsets else b"".join(out)


def parse_header(raw: bytes) -> Tuple[str, List[Tuple[str, int]], int]:
    if raw[:4] != b"BAM\x01":
        raise ValueError("not a BAM stream")
    l_text = struct.unpack_from("<i", raw, 4)[0]
    text = raw[8:8 + l_text].decode(errors="replace")
    o = 8 + l_text
    n_ref = struct.unpack_from("<i", raw, o)[0]; o += 4
    refs = []
    for _ in range(n_ref):
        l_name = struct.unpack_from("<i", raw, o)[0]; o += 4
        name = raw[o:o + l_name - 1].decode(); o += l_name
        l_ref = struct.unpack_from("<i", raw, o)[0]; o += 4
        refs.append((name, l_ref))
    return text, refs, o


@dataclass
class ReadAux:
    """What the HaplotypeModel s4 stage needs beside PackedReads (create_pileup_haplotype.py:105-131): base qualities at the
    reads' seq_off base index, HP tag per read (0 = untagged) and a 64-bit hash of the query name (rows are keyed by name)."""
    qual: np.ndarray                    # uint8 [n_bases]
    hp: np.ndarray                      # uint8 [n_reads]
    qhash: np.ndarray                   # uint64 [n_reads]
    names: Optional[List[str]] = None   # only used by write_bam


def qname_hash(name: str) -> int:
    h = 1469598103934665603
    for c in name.encode():
        h = ((h ^ c) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


class BamReader:
    """Streaming BAM reader (native: csrc/bam_stream.cu).  BGZF blocks are inflated on `threads` host threads 32 MB at a
    time; records are decoded contig by contig, or region by region when a .bai lies next to the file."""

    def __init__(self, path: str, threads: int = 0, keep_aux: bool = False):
        self.lib = _lib.load()
        self.h = self.lib.nsnp_bam_open(path.encode(), int(threads))
        if not self.h:
            raise ValueError(self.lib.nsnp_last_error().decode())
        self.keep_aux = bool(keep_aux)
        self.aux: Optional[ReadAux] = None          # aux data of the contig / region decoded last (keep_aux=True)
        if keep_aux:
            _lib.check(self.lib.nsnp_bam_keep_aux(self.h, 1))
        n = self.lib.nsnp_bam_n_ref(self.h)
        self.refs: List[Tuple[str, int]] = [(self.lib.nsnp_bam_ref_name(self.h, i).decode(), int(self.lib.nsnp_bam_ref_len(self.h, i))) for i in range(n)]
        self.has_index = bool(self.lib.nsnp_bam_has_index(self.h))

    def close(self):
        if self.h:
            self.lib.nsnp_bam_close(self.h)
            self.h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def inflated_bytes(self) -> int:
        return int(self.lib.nsnp_bam_inflated_bytes(self.h))

    def _take(self, n, n_cig, n_bases) -> PackedReads:
        pos = np.empty(n, np.int32); flag = np.empty(n, np.uint16); mapq = np.empty(n, np.uint8)
        cigar_off = np.zeros(n + 1, np.int64); cigar = np.empty(max(1, n_cig), np.uint32); seq_off = np.empty(n, np.int64)
        seq2 = np.zeros(n_bases // 4 + 16, np.uint8); nmask = np.zeros(n_bases // 8 + 16, np.uint8)
        any_n = C.c_int32(0)
        _lib.check(self.lib.nsnp_bam_take(self.h, pos.ctypes.data, flag.ctypes.data, mapq.ctypes.data, cigar_off.ctypes.data, cigar.ctypes.data,
                                          seq_off.ctypes.data, seq2.ctypes.data, nmask.ctypes.data, C.byref(any_n)))
        if self.keep_aux:
            qual = np.zeros(n_bases + 16, np.uint8); hp = np.zeros(n, np.uint8); qh = np.zeros(n, np.uint64)
            _lib.check(self.lib.nsnp_bam_take_aux(self.h, qual.ctypes.data, hp.ctypes.data, qh.ctypes.data))
            self.aux = ReadAux(qual, hp, qh)
        return PackedReads(pos, flag, mapq, cigar_off, cigar[:n_cig], seq_off, seq2, nmask if any_n.value else None)

    def contigs(self, only=None):
        """Yields (ref_id, name, PackedReads) for every reference with reads, in file order; `only`: set of names."""
        want = None
        if only is not None:
            want = np.array([1 if name in only else 0 for name, _ in self.refs], np.int8)
        while True:
            n = C.c_int64(0); nc = C.c_int64(0); nb = C.c_int64(0)
            rid = self.lib.nsnp_bam_next_contig(self.h, 0 if want is None else want.ctypes.data, C.byref(n), C.byref(nc), C.byref(nb))
            if rid == -1:
                return
            if rid < 0:
                raise ValueError(self.lib.nsnp_last_error().decode())
            rd = self._take(n.value, nc.value, nb.value)
            if n.value > 1 and (np.diff(rd.pos) < 0).any():
                raise ValueError(f"reads of {self.refs[rid][0]} are not coordinate sorted")
            yield rid, self.refs[rid][0], rd

    def fetch(self, ref_id: int, beg: int, end: int) -> PackedReads:
        """Reads of one reference that overlap [beg, end) or start inside it (needs the .bai linear index)."""
        n = C.c_int64(0); nc = C.c_int64(0); nb = C.c_int64(0)
        rid = self.lib.nsnp_bam_fetch(self.h, int(ref_id), int(beg), int(end), C.byref(n), C.byref(nc), C.byref(nb))
        if rid < 0:
            raise ValueError(self.lib.nsnp_last_error().decode())
        return self._take(n.value, nc.value, nb.value)


    def fetch_ranges(self, ref_id: int, ranges) -> PackedReads:
        """Reads of one reference that overlap any of the ascending, disjoint [beg, end) ranges, each once, in file order
        (needs the .bai).  Each needed BGZF block is inflated once: the reader walks on between close ranges and seeks
        through the linear index past gaps."""
        rg = np.ascontiguousarray(np.asarray(ranges, dtype=np.int64).reshape(-1, 2))
        n = C.c_int64(0); nc = C.c_int64(0); nb = C.c_int64(0)
        rid = self.lib.nsnp_bam_fetch_ranges(self.h, int(ref_id), rg.ctypes.data, len(rg), C.byref(n), C.byref(nc), C.byref(nb))
        if rid < 0:
            raise ValueError(self.lib.nsnp_last_error().decode())
        return self._take(n.value, nc.value, nb.value)


def read_bam(path: str, contigs=None, threads: int = 0) -> Tuple[List[Tuple[str, int]], Dict[str, PackedReads]]:
    """Returns (reference list, {contig: PackedReads}) for the requested contigs (default: all with reads).  Convenience
    for small files: callers that must bound memory iterate BamReader.contigs() / fetch() instead."""
    with BamReader(path, threads) as r:
        out = {name: rd for _, name, rd in r.contigs(None if contigs is None else set(contigs))}
        return r.refs, out


def _reg2bin(beg: int, end: int) -> int:              # SAM specification section 5.3
    end -= 1
    if beg >> 14 == end >> 14: return ((1 << 15) - 1) // 7 + (beg >> 14)
    if beg >> 17 == end >> 17: return ((1 << 12) - 1) // 7 + (beg >> 17)
    if beg >> 20 == end >> 20: return ((1 << 9) - 1) // 7 + (beg >> 20)
    if beg >> 23 == end >> 23: return ((1 << 6) - 1) // 7 + (beg >> 23)
    if beg >> 26 == end >> 26: return ((1 << 3) - 1) // 7 + (beg >> 26)
    return 0


def _write_bai(path: str, n_ref: int, recs) -> None:
    """recs: (ref_id, beg, end, voffset_begin, voffset_end) per record in file order (tests / interoperability)."""
    bins = [dict() for _ in range(n_ref)]
    lin = [dict() for _ in range(n_ref)]
    for rid, beg, end, v0, v1 in recs:
        if rid < 0:
            continue
        ch = bins[rid].setdefault(_reg2bin(beg, max(end, beg + 1)), [])
        if ch and ch[-1][1] == v0:
            ch[-1][1] = v1
        else:
            ch.append([v0, v1])
        for w in range(beg >> 14, ((max(end, beg + 1) - 1) >> 14) + 1):
            if w not in lin[rid] or v0 < lin[rid][w]:
                lin[rid][w] = v0
    out = [b"BAI\x01", struct.pack("<i", n_ref)]
    for rid in range(n_ref):
        out.append(struct.pack("<i", len(bins[rid])))
        for b, ch in sorted(bins[rid].items()):
            out.append(struct.pack("<Ii", b, len(ch)))
            for v0, v1 in ch:
                out.append(struct.pack("<QQ", v0, v1))
        n_intv = (max(lin[rid]) + 1) if lin[rid] else 0
        out.append(struct.pack("<i", n_intv))
        last = 0
        for w in range(n_intv):
            last = lin[rid].get(w, last)
            out.append(struct.pack("<Q", last))
    with open(path, "wb") as f:
        f.write(b"".join(out))


def write_bam(path: str, refs: List[Tuple[str, int]], reads_by_contig: Dict[str, PackedReads], long_cigar_as_tag: int = 65535,
              index: bool = False, aux: Optional[Dict[str, "ReadAux"]] = None) -> None:
    """Coordinate-sorted BAM from packed reads (tests / interoperability).  Qualities are written as 0xFF (absent) unless `aux`
    carries them (then also query names and HP:C tags).  index=True also writes <path>.bai (bins + 16 kb linear index)."""
    code4 = np.array([1, 2, 4, 8], np.uint8)
    parts = [b"BAM\x01"]
    text = "@HD\tVN:1.6\tSO:coordinate\n" + "".join(f"@SQ\tSN:{n}\tLN:{l}\n" for n, l in refs)
    parts += [struct.pack("<i", len(text)), text.encode(), struct.pack("<i", len(refs))]
    for n, l in refs:
        parts += [struct.pack("<i", len(n) + 1), n.encode() + b"\0", struct.pack("<i", l)]
    rec_info = []
    upos = sum(len(x) for x in parts)
    for rid, (name, _) in enumerate(refs):
        rd = reads_by_contig.get(name)
        if rd is None:
            continue
        for i in range(rd.n_reads):
            cg = rd.cigar[rd.cigar_off[i]:rd.cigar_off[i + 1]].astype(np.uint32)
            ops = cg & 15; lens = (cg >> 4).astype(np.int64)
            l_seq = int(lens[(ops == 0) | (ops == 1) | (ops == 4) | (ops == 7) | (ops == 8)].sum())
            ref_len = int(lens[(ops == 0) | (ops == 2) | (ops == 3) | (ops == 7) | (ops == 8)].sum())
            k = int(rd.seq_off[i]) + np.arange(l_seq)
            c2 = (rd.seq2[k >> 2] >> (2 * (k & 3))) & 3
            c4 = code4[c2]
            if rd.nmask is not None:
                isn = ((rd.nmask[k >> 3] >> (k & 7)) & 1).astype(bool)
                c4 = np.where(isn, 15, c4).astype(np.uint8)
            if l_seq & 1:
                c4 = np.append(c4, 0).astype(np.uint8)
            seq = ((c4[0::2] << 4) | c4[1::2]).astype(np.uint8).tobytes()
            ax = aux.get(name) if aux else None
            rname = (ax.names[i] if (ax is not None and ax.names is not None) else f"r{i}").encode() + b"\0"
            tags = b""
            if ax is not None and int(ax.hp[i]):
                tags += b"HPC" + struct.pack("<B", int(ax.hp[i]))
            qbytes = b"\xff" * l_seq if ax is None else ax.qual[int(rd.seq_off[i]): int(rd.seq_off[i]) + l_seq].tobytes()
            cig_bytes = cg.tobytes(); n_cig = len(cg)
            if n_cig > long_cigar_as_tag:              # SAM spec: real CIGAR in CG:B,I, placeholder <l_seq>S<ref_len>N in the record
                tags += b"CGBI" + struct.pack("<I", n_cig) + cig_bytes
                cig_bytes = struct.pack("<II", (l_seq << 4) | 4, (ref_len << 4) | 3); n_cig = 2
            body = struct.pack("<iiBBHHHIiii", rid, int(rd.pos[i]), len(rname), int(rd.mapq[i]), 4680, n_cig, int(rd.flag[i]), l_seq, -1, -1, 0)
            body += rname + cig_bytes + seq + qbytes + tags
            parts += [struct.pack("<i", len(body)), body]
            rec_info.append((rid, int(rd.pos[i]), int(rd.pos[i]) + ref_len, upos, upos + 4 + len(body)))
            upos += 4 + len(body)
    raw = b"".join(parts)
    comp, block_off = bgzf_compress(raw, with_offsets=True)
    with open(path, "wb") as f:
        f.write(comp)
    if index:
        def voff(u):                                   # uncompressed offset -> BGZF virtual offset
            k = min(u // 0xFF00, len(block_off) - 1)
            return (block_off[k] << 16) | (u - k * 0xFF00)
        _write_bai(path + ".bai", len(refs), [(r, b, e, voff(u0), voff(u1)) for r, b, e, u0, u1 in rec_info])
