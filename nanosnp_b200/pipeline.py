"""Host side of the GPU s1 + s2 path: thin wrappers that own torch tensors and hand raw pointers to the C ABI.

Mirrors the reference stage boundaries so parity can be checked at each of them:
    pileup_counts   <- samtools mpileup + TensorMaker::make_tensor   (tensor_maker.cpp:61-249)
    select          <- create_pileup_tensor gate + window rule        (make_candidate_snp_tensor/main.cpp:174-217)
    gather          <- window emit + DNA_CreatePredictData + make_bin_predict_data.py
    PileupModel     <- LSTMNetwork.predict                            (PileupModel/model.py:114-119)
PyTorch is used for memory ownership and streams only; every computation is a kernel of the C-ABI library.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _lib
from .reads import PackedReads


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(device) -> torch.device:
    device = torch.device(device)
    if device.type != "cuda" or not torch.cuda.is_available():
        raise _lib.NsnpError(_lib.E_NO_DEVICE, "nanosnp_b200 needs a CUDA device: there is no CPU fallback")
    return device


@dataclass
class RegionResult:
    """Everything predict.py needs for the sites of one region (device tensors unless stated)."""
    n: int
    pos0: torch.Tensor          # int32 [n] 0-based centre positions, ascending
    refbase: torch.Tensor       # uint8 [n] upper-cased centre reference base
    x: Optional[torch.Tensor]   # int32 [n,33,18] position_matrix (None when not requested)
    gt: Optional[torch.Tensor]  # float32 [n,21]
    zy: Optional[torch.Tensor]  # float32 [n,3]


def _intervals(targets) -> np.ndarray:
    """[k, 2] int32 host copy of target intervals (the library checks order, overlap and range)."""
    a = np.asarray(targets)
    if a.size and (a.min() < np.iinfo(np.int32).min or a.max() > np.iinfo(np.int32).max):
        raise _lib.NsnpError(_lib.E_INVALID, "target interval outside the int32 contig coordinates")
    return np.ascontiguousarray(a.reshape(-1, 2), dtype=np.int32)


class PileupEngine:
    """One engine per GPU / process.  Buffers are grown on demand and reused across regions."""

    def __init__(self, device="cuda:0", params: Optional[_lib.Params] = None):
        self.lib = _lib.load()
        self.device = require_cuda(device)
        self.params = params if params is not None else _lib.default_params()
        self._ws = {}
        self.status = torch.zeros(4, dtype=torch.int32, device=self.device)

    # -- helpers -----------------------------------------------------------------------------------
    def _workspace(self, key: str, nbytes: int) -> torch.Tensor:
        t = self._ws.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=self.device)
            self._ws[key] = t
        return t

    def check_status(self) -> None:
        _lib.check(self.lib.nsnp_check_status(self.status.data_ptr(), _stream(self.device)))

    # -- s1 step A ---------------------------------------------------------------------------------
    def pileup_counts(self, reads: PackedReads, ref: torch.Tensor, region_start: int = 0, region_len: Optional[int] = None,
                      counts: Optional[torch.Tensor] = None, flags: Optional[torch.Tensor] = None, targets: Optional[np.ndarray] = None):
        """targets: optional [k, 2] sorted disjoint [start, end) contig intervals: only the tiles holding a position within 16 bp
        of an interval are computed; every other position gets flags 0 and an unwritten count row."""
        contig_len = int(ref.shape[0])
        if region_len is None:
            region_len = contig_len - region_start
        if counts is None:
            counts = torch.empty((region_len, _lib.CHANNELS), dtype=torch.int32, device=self.device)
        if flags is None:
            flags = torch.empty(region_len, dtype=torch.uint8, device=self.device)
        st = reads.as_struct()
        if targets is not None:
            iv = _intervals(targets)
            ws = self._workspace("pileup", self.lib.nsnp_pileup_targets_workspace_bytes(st.n_reads, st.n_cigar, region_len, len(iv)))
            with torch.cuda.device(self.device):
                _lib.check(self.lib.nsnp_pileup_counts_targets(C.byref(st), ref.data_ptr(), contig_len, region_start, region_len,
                                                               iv.ctypes.data, len(iv), C.byref(self.params), counts.data_ptr(),
                                                               flags.data_ptr(), ws.data_ptr(), ws.numel(), self.status.data_ptr(),
                                                               _stream(self.device)))
            return counts, flags
        need = self.lib.nsnp_pileup_workspace_bytes(st.n_reads, st.n_cigar, region_len)
        ws = self._workspace("pileup", need)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nsnp_pileup_counts(C.byref(st), ref.data_ptr(), contig_len, region_start, region_len,
                                                   C.byref(self.params), counts.data_ptr(), flags.data_ptr(),
                                                   ws.data_ptr(), ws.numel(), self.status.data_ptr(), _stream(self.device)))
        return counts, flags

    # -- s1 step B ---------------------------------------------------------------------------------
    def select(self, flags: torch.Tensor, ref: torch.Tensor, region_start: int, emit_start: int, emit_end: int,
               capacity: int, counts: Optional[torch.Tensor] = None, recompute_gate: bool = False,
               pos: Optional[torch.Tensor] = None, n_dev: Optional[torch.Tensor] = None, targets: Optional[np.ndarray] = None,
               sites: bool = False):
        """targets: optional [k, 2] sorted disjoint [start, end) contig intervals: only sites inside them are selected.
        sites: every covered position of the targets with an ACGT centre base and a full 33-row window is selected, whether it
        passes the allele-frequency / depth gate or not (`--sites`); needs targets."""
        region_len = int(flags.shape[0])
        if pos is None:
            pos = torch.empty(max(capacity, 1), dtype=torch.int32, device=self.device)
        if n_dev is None:
            n_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
        if sites:
            if targets is None:
                raise ValueError("select(sites=True) needs the site intervals as targets")
            iv = _intervals(targets)
            ws = self._workspace("select", self.lib.nsnp_select_sites_workspace_bytes(region_len, len(iv)))
            with torch.cuda.device(self.device):
                _lib.check(self.lib.nsnp_select_candidates_sites(
                    flags.data_ptr(), ref.data_ptr(), int(ref.shape[0]), region_start, region_len, emit_start, emit_end, iv.ctypes.data,
                    len(iv), pos.data_ptr(), capacity, n_dev.data_ptr(), ws.data_ptr(), ws.numel(), self.status.data_ptr(),
                    _stream(self.device)))
            return pos, n_dev
        if targets is not None:
            iv = _intervals(targets)
            ws = self._workspace("select", self.lib.nsnp_select_targets_workspace_bytes(region_len, len(iv)))
            with torch.cuda.device(self.device):
                _lib.check(self.lib.nsnp_select_candidates_targets(
                    0 if counts is None else counts.data_ptr(), flags.data_ptr(), ref.data_ptr(), int(ref.shape[0]), region_start,
                    region_len, emit_start, emit_end, iv.ctypes.data, len(iv), C.byref(self.params), int(recompute_gate), pos.data_ptr(),
                    capacity, n_dev.data_ptr(), ws.data_ptr(), ws.numel(), self.status.data_ptr(), _stream(self.device)))
            return pos, n_dev
        ws = self._workspace("select", self.lib.nsnp_select_workspace_bytes(region_len))
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nsnp_select_candidates(0 if counts is None else counts.data_ptr(), flags.data_ptr(), ref.data_ptr(),
                                                       int(ref.shape[0]), region_start, region_len, emit_start, emit_end,
                                                       C.byref(self.params), int(recompute_gate), pos.data_ptr(), capacity,
                                                       n_dev.data_ptr(), ws.data_ptr(), ws.numel(), self.status.data_ptr(),
                                                       _stream(self.device)))
        return pos, n_dev

    # -- s1 step C ---------------------------------------------------------------------------------
    def gather(self, counts: torch.Tensor, ref: torch.Tensor, region_start: int, pos: torch.Tensor, n_dev: Optional[torch.Tensor],
               n_max: int, want_i32: bool = True, want_f32: bool = False, x_i32=None, x_f32=None, refbase=None):
        if want_i32 and x_i32 is None:
            x_i32 = torch.empty((n_max, _lib.WINDOW, _lib.CHANNELS), dtype=torch.int32, device=self.device)
        if want_f32 and x_f32 is None:
            x_f32 = torch.empty((n_max, _lib.WINDOW, _lib.CHANNELS), dtype=torch.float32, device=self.device)
        if refbase is None:
            refbase = torch.empty(max(n_max, 1), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nsnp_gather_windows(counts.data_ptr(), ref.data_ptr(), region_start, int(counts.shape[0]),
                                                    pos.data_ptr(), 0 if n_dev is None else n_dev.data_ptr(), n_max,
                                                    0 if x_i32 is None else x_i32.data_ptr(), 0 if x_f32 is None else x_f32.data_ptr(),
                                                    refbase.data_ptr(), _stream(self.device)))
        return x_i32, x_f32, refbase

    # -- s2 numeric record logic ------------------------------------------------------------------
    def site_records(self, gt: torch.Tensor, zy: torch.Tensor, x: torch.Tensor, refbase: torch.Tensor, pos: torch.Tensor, n: int,
                     rec: Optional[torch.Tensor] = None) -> torch.Tensor:
        if rec is None:
            rec = torch.empty((max(n, 1), 32), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nsnp_site_records(gt.data_ptr(), zy.data_ptr(), x.data_ptr(), refbase.data_ptr(), pos.data_ptr(), n, 0,
                                                  rec.data_ptr(), _stream(self.device)))
        return rec[:n]

    def site_records_from_counts(self, gt: torch.Tensor, zy: torch.Tensor, counts: torch.Tensor, region_start: int, ref: torch.Tensor,
                                 pos: torch.Tensor, n: int, rec: Optional[torch.Tensor] = None) -> torch.Tensor:
        """site_records with the centre row read from the count tensor and the reference base from the contig."""
        if rec is None:
            rec = torch.empty((max(n, 1), 32), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nsnp_site_records_sites(gt.data_ptr(), zy.data_ptr(), counts.data_ptr(), region_start, ref.data_ptr(),
                                                        pos.data_ptr(), n, 0, rec.data_ptr(), _stream(self.device)))
        return rec[:n]

    # -- s1 for a whole region ---------------------------------------------------------------------
    def candidate_windows(self, reads: PackedReads, ref: torch.Tensor, region_start: int = 0, region_len: Optional[int] = None,
                          emit_start: Optional[int] = None, emit_end: Optional[int] = None, capacity: Optional[int] = None):
        """reads -> (pos0 int32[n], refbase uint8[n], x int32[n,33,18]).  One host sync (the site count)."""
        contig_len = int(ref.shape[0])
        if region_len is None:
            region_len = contig_len - region_start
        emit_start = region_start if emit_start is None else emit_start
        emit_end = region_start + region_len if emit_end is None else emit_end
        counts, flags = self.pileup_counts(reads, ref, region_start, region_len)
        cap = int(capacity if capacity is not None else max(1024, (emit_end - emit_start)))
        pos, n_dev = self.select(flags, ref, region_start, emit_start, emit_end, cap)
        n = int(n_dev.item())
        self.check_status()
        x, _, refbase = self.gather(counts, ref, region_start, pos, n_dev, n)
        return pos[:n], refbase[:n], x[:n], counts, flags


class PileupModelWeights:
    """Packs a reference checkpoint (utils.py:67-77: ck['encoder'], ck['forward_layer']) into the device blob."""

    def __init__(self, encoder_state: dict, forward_state: dict, device="cuda:0"):
        lib = _lib.load()
        self.device = require_cuda(device)
        keep = []

        def ptr(t):
            a = np.ascontiguousarray(t.detach().cpu().numpy() if hasattr(t, "detach") else t, dtype=np.float32)
            keep.append(a)
            return a.ctypes.data

        w = _lib.ModelWeights()
        for layer in range(2):
            for d, suffix in enumerate(("", "_reverse")):
                i = layer * 2 + d
                w.w_ih[i] = ptr(encoder_state[f"lstm.weight_ih_l{layer}{suffix}"])
                w.w_hh[i] = ptr(encoder_state[f"lstm.weight_hh_l{layer}{suffix}"])
                w.b_ih[i] = ptr(encoder_state[f"lstm.bias_ih_l{layer}{suffix}"])
                w.b_hh[i] = ptr(encoder_state[f"lstm.bias_hh_l{layer}{suffix}"])
        w.proj_w, w.proj_b = ptr(encoder_state["output_proj.weight"]), ptr(encoder_state["output_proj.bias"])
        w.dense_w, w.dense_b = ptr(forward_state["dense.weight"]), ptr(forward_state["dense.bias"])
        w.gt_w, w.gt_b = ptr(forward_state["genotype_layer.weight"]), ptr(forward_state["genotype_layer.bias"])
        w.zy_w, w.zy_b = ptr(forward_state["zygosity_layer.weight"]), ptr(forward_state["zygosity_layer.bias"])
        nbytes = lib.nsnp_model_blob_bytes()
        host = np.zeros(nbytes, np.uint8)
        _lib.check(lib.nsnp_model_pack_weights(C.byref(w), host.ctypes.data, nbytes))
        self.blob = torch.from_numpy(host).to(self.device)


class PileupModelForward:
    """nsnp_pileup_model_forward with reusable workspace."""

    def __init__(self, weights: PileupModelWeights, precision: int = _lib.PREC_FP32):
        self.lib = _lib.load()
        self.w = weights
        self.device = weights.device
        self.precision = precision
        self._ws = None
        self._last_n = 0
        self.tensor_core = precision in (_lib.PREC_F16X3, _lib.PREC_F16X1)

    def __call__(self, x: torch.Tensor, n_dev: Optional[torch.Tensor] = None, gt=None, zy=None):
        assert x.is_cuda and x.is_contiguous() and tuple(x.shape[1:]) == (_lib.WINDOW, _lib.CHANNELS)
        n = int(x.shape[0])
        if gt is None:
            gt = torch.empty((n, _lib.GT_CLASSES), dtype=torch.float32, device=self.device)
        if zy is None:
            zy = torch.empty((n, _lib.ZY_CLASSES), dtype=torch.float32, device=self.device)
        self._last_n = n
        self._workspace(n)
        if x.dtype == torch.int32:
            xi, xf = x.data_ptr(), 0
        elif x.dtype == torch.float32:
            xi, xf = 0, x.data_ptr()
        else:
            raise TypeError("x must be int32 or float32 [N,33,18]")
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nsnp_pileup_model_forward(self.w.blob.data_ptr(), xi, xf, n, 0 if n_dev is None else n_dev.data_ptr(),
                                                          gt.data_ptr(), zy.data_ptr(), self._ws.data_ptr(), self._ws.numel(),
                                                          self.precision, _stream(self.device)))
        return gt, zy

    def reevaluated(self) -> int:
        """NSNP_PREC_F16X1: low-margin sites the last call found and re-ran through the three-pass path (synchronises); raises
        when there were more than the library re-evaluates."""
        if self.precision != _lib.PREC_F16X1 or self._ws is None or self._last_n == 0:
            return 0
        c = C.c_int64(0)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nsnp_model_f16x1_reevaluated(self._ws.data_ptr(), C.byref(c), _stream(self.device)))
        return int(c.value)

    def _workspace(self, n: int) -> torch.Tensor:
        need = self.lib.nsnp_model_workspace_bytes(n)
        if self._ws is None or self._ws.numel() < need:
            if self._ws is not None:
                self.reevaluated()                    # an overflow recorded in the old workspace must not get lost
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
            if self.precision == _lib.PREC_F16X1:
                with torch.cuda.device(self.device):
                    _lib.check(self.lib.nsnp_model_f16x1_reset(self._ws.data_ptr(), _stream(self.device)))
        return self._ws

    def from_counts(self, counts: torch.Tensor, region_start: int, pos: torch.Tensor, n: int, gt=None, zy=None):
        """The same forward pass with every site's window read straight from the region's count tensor [L,18] (a window is the
        contiguous row span counts[pos-16 .. pos+16]): no [n,33,18] tensor is materialised.  Tensor-core path only."""
        assert counts.is_cuda and counts.is_contiguous() and counts.dtype == torch.int32 and self.tensor_core
        if gt is None:
            gt = torch.empty((n, _lib.GT_CLASSES), dtype=torch.float32, device=self.device)
        if zy is None:
            zy = torch.empty((n, _lib.ZY_CLASSES), dtype=torch.float32, device=self.device)
        self._last_n = n
        self._workspace(n)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.nsnp_pileup_model_forward_sites(self.w.blob.data_ptr(), counts.data_ptr(), region_start, int(counts.shape[0]),
                                                                pos.data_ptr(), n, 0, gt.data_ptr(), zy.data_ptr(), self._ws.data_ptr(),
                                                                self._ws.numel(), self.precision, _stream(self.device)))
        return gt, zy
