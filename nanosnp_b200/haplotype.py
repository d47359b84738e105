"""Drop-in for the reference's HaplotypeModel s5 seams (BASELINE configs[4]; SURVEY 8a H4-H6), GPU only:

    net = LSTMNetwork(config).to(device); net.load_state_dict(torch.load(ckpt))     # predict_dev.py:64-65
    gt, zy = net.predict(x_pileup, x_haplotype)                                      # model_dev.py:133-143
    TestDataset(...)[i] -> (position, pileup_feature[105,33], haplotype_feature[105,11])   # dataset_dev.py:323-349
    predict(...) -> `ctg\\tpos\\tGT\\tqual` rows                                        # predict_dev.py:27-48

The reference reads PyTables `.bin` files written by write_to_bins.py (PyTables / pysam are absent here), so the dataset takes the
same eight arrays from an `.npz` (keys as the HDF5 node names; nanosnp_b200.hap_groups writes them from the pileup VCF and the
HP-tagged BAMs: SURVEY 8a H1-H3).  predict_from_bams() runs s4 + s5 without the files in between: group selection on the host,
read matrices, the 105-channel features and the model on the GPU.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from math import e, log
from typing import Optional

import numpy as np
import torch

from . import _lib
from .pipeline import require_cuda

PRECISIONS = ("fp32", "f16x3")
GT10 = ["AA", "AC", "AG", "AT", "CC", "CG", "CT", "GG", "GT", "TT"]                 # HaplotypeModel/options.py:8-17
_ENC = ("pileup_encoder", "haplotype_encoder")


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def required_keys():
    keys = []
    for enc in _ENC:
        for l in range(3):
            for sfx in ("", "_reverse"):
                keys += [f"{enc}.lstm.{k}_l{l}{sfx}" for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
        keys += [f"{enc}.output_proj.weight", f"{enc}.output_proj.bias"]
    keys += [f"forward_layer.{n}.{p}" for n in ("dense", "genotype_layer", "zygosity_layer") for p in ("weight", "bias")]
    return keys


class LSTMNetwork:
    """model_dev.LSTMNetwork for inference: same constructor / load_state_dict / predict; the forward pass is csrc/haplotype.cu.

    precision "fp32" (default, the parity reference): fp32 FFMA.  "f16x3": tcgen05 tensor cores (csrc/haplotype_tc.cu), hi/lo
    split operands with three MMAs per product and fp32 accumulation; probabilities within 5e-5 of a float64 evaluation."""

    def __init__(self, config=None, precision: str = "fp32"):
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {PRECISIONS}, got {precision!r}")
        self.precision = precision
        m = getattr(config, "model", None) if config is not None else None
        if m is not None:
            dims = (m.pileup_dim, m.haplotype_dim, m.pileup_length, m.haplotype_length, m.hidden_size, m.lstm_layers, m.gt_num_class, m.zy_num_class)
            if tuple(dims) != (105, 105, 33, 11, 256, 3, 10, 3):
                raise NotImplementedError(f"the CUDA path is built for ont_haplotype.yaml's architecture, got {dims}")
        self.device: Optional[torch.device] = None
        self._state = None
        self._blob = None
        self._ws = None
        self.lib = _lib.load()

    def to(self, device):
        self.device = require_cuda(device)
        self._blob = None
        return self

    def eval(self):
        return self

    def load_state_dict(self, state, strict: bool = True):
        missing = [k for k in required_keys() if k not in state]
        unexpected = [k for k in state if k not in required_keys()]
        if missing or (strict and unexpected):
            raise RuntimeError(f"Error(s) in loading state_dict: missing keys {missing[:4]}..., unexpected keys {unexpected[:4]}")
        self._state = {k: np.ascontiguousarray(torch.as_tensor(v).detach().to(torch.float32).cpu().numpy()) for k, v in state.items()}
        self._blob = None

    def _pack(self):
        if self._state is None:
            raise RuntimeError("load_state_dict() has not been called")
        if self.device is None:
            raise _lib.NsnpError(_lib.E_NO_DEVICE, "call .to('cuda') first: there is no CPU fallback")
        s = self._state
        w = _lib.HapWeights()
        for ei, enc in enumerate(_ENC):
            for l in range(3):
                for d, sfx in enumerate(("", "_reverse")):
                    i = (ei * 3 + l) * 2 + d
                    w.w_ih[i] = s[f"{enc}.lstm.weight_ih_l{l}{sfx}"].ctypes.data
                    w.w_hh[i] = s[f"{enc}.lstm.weight_hh_l{l}{sfx}"].ctypes.data
                    w.b_ih[i] = s[f"{enc}.lstm.bias_ih_l{l}{sfx}"].ctypes.data
                    w.b_hh[i] = s[f"{enc}.lstm.bias_hh_l{l}{sfx}"].ctypes.data
            w.proj_w[ei] = s[f"{enc}.output_proj.weight"].ctypes.data
            w.proj_b[ei] = s[f"{enc}.output_proj.bias"].ctypes.data
        for name, field in (("dense", "dense"), ("genotype_layer", "gt"), ("zygosity_layer", "zy")):
            setattr(w, field + "_w", s[f"forward_layer.{name}.weight"].ctypes.data)
            setattr(w, field + "_b", s[f"forward_layer.{name}.bias"].ctypes.data)
        tc = self.precision == "f16x3"
        nbytes = (self.lib.nsnp_hap_model_tc_blob_bytes if tc else self.lib.nsnp_hap_model_blob_bytes)()
        host = np.zeros(nbytes, np.uint8)
        _lib.check((self.lib.nsnp_hap_model_tc_pack_weights if tc else self.lib.nsnp_hap_model_pack_weights)(C.byref(w), host.ctypes.data, nbytes))
        self._blob = torch.from_numpy(host).to(self.device)

    def predict(self, pileup_x: torch.Tensor, haplotype_x: torch.Tensor):
        """pileup_x: float [N,105,33], haplotype_x: float [N,105,11] on the device -> softmaxed (gt [N,10], zy [N,3])."""
        if self._blob is None:
            self._pack()
        px = pileup_x.to(self.device, torch.float32).contiguous(); hx = haplotype_x.to(self.device, torch.float32).contiguous()
        n = int(px.shape[0])
        assert tuple(px.shape[1:]) == (105, 33) and tuple(hx.shape) == (n, 105, 11)
        gt = torch.empty((n, 10), dtype=torch.float32, device=self.device)
        zy = torch.empty((n, 3), dtype=torch.float32, device=self.device)
        tc = self.precision == "f16x3"
        need = (self.lib.nsnp_hap_model_tc_workspace_bytes if tc else self.lib.nsnp_hap_model_workspace_bytes)(n)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        forward = self.lib.nsnp_hap_model_tc_forward if tc else self.lib.nsnp_hap_model_forward
        with torch.cuda.device(self.device):
            _lib.check(forward(self._blob.data_ptr(), px.data_ptr(), hx.data_ptr(), n, gt.data_ptr(), zy.data_ptr(),
                               self._ws.data_ptr(), self._ws.numel(), _stream(self.device)))
        return gt, zy


def reference_codes(ref: np.ndarray, positions1: np.ndarray) -> np.ndarray:
    """int32 codes of ref[pos-1] (dataset_dev.py:104-118): A1 C2 G3 T4; N, lower case, other letters and out of range give 0."""
    lut = np.zeros(256, np.int32)
    for ch, v in (("A", 1), ("C", 2), ("G", 3), ("T", 4)):
        lut[ord(ch)] = v
    p = np.asarray(positions1, np.int64) - 1
    ok = (p >= 0) & (p < len(ref))
    out = np.zeros(p.shape, np.int32)
    out[ok] = lut[np.asarray(ref, np.uint8)[p[ok]]]
    return out


def frequency_features(seq, bq, mq, hp, refcode, device="cuda:0") -> torch.Tensor:
    """int32 [n, depth, L] matrices + int32 [n, L] reference codes -> float32 [n, 105, L] on the device."""
    lib = _lib.load()
    device = require_cuda(device)
    arrs = [(a.to(device, torch.int32) if torch.is_tensor(a) else torch.as_tensor(np.ascontiguousarray(a, np.int32)).to(device)).contiguous()
            for a in (seq, bq, mq, hp, refcode)]
    n, depth, L = (int(v) for v in arrs[0].shape)
    out = torch.empty((n, 105, L), dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        _lib.check(lib.nsnp_hap_features(*[a.data_ptr() for a in arrs], n, depth, L, out.data_ptr(), _stream(device)))
    return out


class TestDataset:
    """dataset_dev.TestDataset over an `.npz` holding the arrays write_to_bins.py stores (`pileup_sequences`, `pileup_hap`,
    `pileup_baseq`, `pileup_mapq`, `haplotype_*`, `candidate_positions` (`ctg:pos` strings), `haplotype_positions` ([n,11]
    `ctg:pos` strings).  Features are computed for the whole file at once on the GPU; items come back as host arrays."""
    __test__ = False

    def __init__(self, bin_path: str, references: dict, pileup_length: int = 33, haplotype_length: int = 11, device="cuda:0"):
        z = np.load(bin_path, allow_pickle=False)
        self.positions = [str(s) for s in np.asarray(z["candidate_positions"]).reshape(-1)]
        n = len(self.positions)
        pref = np.zeros((n, pileup_length), np.int32); href = np.zeros((n, haplotype_length), np.int32)
        hpos = np.asarray(z["haplotype_positions"]).reshape(n, -1)
        for i, cp in enumerate(self.positions):
            ctg, pos = cp.split(":")
            ref = references.get(ctg)
            if ref is not None:
                pref[i] = reference_codes(ref, int(pos) + np.arange(-(pileup_length // 2), pileup_length // 2 + 1))
            for j in range(haplotype_length):
                c2, p2 = str(hpos[i, j]).split(":")
                r2 = references.get(c2)
                if r2 is not None:
                    href[i, j] = reference_codes(r2, np.asarray([int(p2)]))[0]
        self.pileup = frequency_features(z["pileup_sequences"], z["pileup_baseq"], z["pileup_mapq"], z["pileup_hap"], pref, device)
        self.haplotype = frequency_features(z["haplotype_sequences"], z["haplotype_baseq"], z["haplotype_mapq"], z["haplotype_hap"], href, device)

    def __len__(self):
        return len(self.positions)

    def __getitem__(self, i):
        return self.positions[i], self.pileup[i].cpu().numpy(), self.haplotype[i].cpu().numpy()


def calculate_score(p) -> float:                              # predict_dev.py:22-25; p is a numpy float32 (float32 arithmetic under NumPy 2)
    tmp = max((-10 * log(e, 10)) * log(((1.0 - p) + 1e-300) / (p + 1e-300)) + 10, 0)
    return float(round(tmp, 2))


def load_reference_file(path: str) -> dict:
    """get_truth.load_reference_file (get_truth.py:88-104): name (first word) -> uint8 sequence."""
    from .dataset import load_fasta
    return load_fasta(path)


def predict(model: LSTMNetwork, test_data: str, reference_path: str, batch_size: int, pileup_length: int, haplotype_length: int,
            output_file: str, device) -> int:
    """predict_dev.predict: every `.npz` of the directory -> `ctg\\tpos\\tGT\\tqual` rows (input of scripts/merge.py)."""
    references = load_reference_file(reference_path)
    n_rows = 0
    model.eval()
    with open(output_file, "w") as fw:
        for name in sorted(os.listdir(test_data)):
            if not name.endswith(".npz"):
                continue
            ds = TestDataset(os.path.join(test_data, name), references, pileup_length, haplotype_length, device)
            for s in range(0, len(ds), batch_size):
                gt, _ = model.predict(ds.pileup[s:s + batch_size], ds.haplotype[s:s + batch_size])
                g = gt.cpu().numpy()
                gp = g.max(axis=1); go = g.argmax(axis=1)
                for j in range(len(go)):
                    ctg, pos = ds.positions[s + j].split(":")
                    fw.write(ctg + "\t" + pos + "\t" + GT10[go[j]] + "\t" + str(calculate_score(gp[j])) + "\n")
                    n_rows += 1
    return n_rows


def predict_from_bams(model: LSTMNetwork, pileup_vcf: str, bams: str, reference_path: str, output_file: str, batch_size: int = 1000,
                      pileup_flanking_size: int = 16, adjacent_size: int = 5, low_quality_threshold: float = 19, hete_support_quality: float = 14,
                      max_coverage: int = 150, max_depth: Optional[int] = None, threads: int = 1, device="cuda:0") -> int:
    """scripts/s4_haplotype_model_feature_generation.sh + s5_haplotype_model_predict.sh in one pass, nothing written in between:
    groups (hap_groups.select_snp_multiprocess) -> read matrices on the GPU (hap_groups.group_matrices; chunking and sub-groups as
    make_predict_bins.py with `threads`) -> 105-channel features -> model -> `ctg\tpos\tGT\tqual` rows.  max_depth = the
    --max_pileup_depth / --max_haplotype_depth cut (3 x coverage in the reference's script)."""
    from . import hap_groups as hg
    device = require_cuda(device)
    references = load_reference_file(reference_path)
    groups = hg.select_snp_multiprocess(pileup_vcf, low_quality_threshold, adjacent_size, hete_support_quality, nthreads=threads)
    n_hap = 2 * adjacent_size + 1
    n_rows = 0
    with open(output_file, "w") as fw:
        for ctg, g in groups.items():
            chunks = hg.plan_chunks(len(g), threads)
            al = hg.load_contig(os.path.join(bams, ctg + ".bam"), ctg, device) if chunks else None
            if al is None:
                continue
            subs = [(lo + a, lo + b) for lo, hi in chunks for a, b in hg.plan_subgroups(g[lo:hi])]
            gm = hg.group_matrices(al, g, subs, max_coverage, pileup_flanking_size)
            if len(gm.positions) == 0:
                continue
            ref = references.get(ctg)
            cand = gm.positions[:, n_hap // 2]
            win = cand[:, None] + np.arange(-pileup_flanking_size, pileup_flanking_size + 1)[None, :]
            pref = reference_codes(ref, win) if ref is not None else np.zeros(win.shape, np.int32)
            href = reference_codes(ref, gm.positions) if ref is not None else np.zeros(gm.positions.shape, np.int32)
            d = gm.hap[0].shape[1] if max_depth is None else min(gm.hap[0].shape[1], max_depth)
            for s in range(0, len(cand), batch_size):
                sl = slice(s, s + batch_size)
                xp = frequency_features(gm.pile[0][sl, :d], gm.pile[2][sl, :d], gm.pile[3][sl, :d], gm.pile[1][sl, :d], pref[sl], device)
                xh = frequency_features(gm.hap[0][sl, :d], gm.hap[2][sl, :d], gm.hap[3][sl, :d], gm.hap[1][sl, :d], href[sl], device)
                gt, _ = model.predict(xp, xh)
                gq = gt.cpu().numpy()
                gp = gq.max(axis=1); go = gq.argmax(axis=1)
                for j in range(len(go)):
                    fw.write(ctg + "\t" + str(int(cand[s + j])) + "\t" + GT10[go[j]] + "\t" + str(calculate_score(gp[j])) + "\n")
                    n_rows += 1
    return n_rows


def main(argv=None):
    import argparse
    import yaml
    from .utils import AttrDict
    ap = argparse.ArgumentParser(description="drop-in for HaplotypeModel/predict_dev.py (GPU only)")
    ap.add_argument("-config", required=True)
    ap.add_argument("-model_path", required=True)
    ap.add_argument("-bin_paths", required=True, help="directory of .npz files (arrays of write_to_bins.py)")
    ap.add_argument("-reference_path", required=True)
    ap.add_argument("-output", required=True)
    ap.add_argument("-batch_size", type=int, default=1000)
    ap.add_argument("--no_cuda", action="store_true")
    ap.add_argument("--precision", choices=PRECISIONS, default="fp32",
                    help="fp32: FFMA parity path (default); f16x3: tensor cores, hi/lo split operands, within 5e-5 of float64")
    opt = ap.parse_args(argv)
    if opt.no_cuda:
        raise SystemExit("nanosnp_b200.haplotype: --no_cuda is not supported (no CPU fallback)")
    config = AttrDict(yaml.load(open(opt.config), Loader=yaml.FullLoader))
    net = LSTMNetwork(config, precision=opt.precision).to("cuda")
    net.load_state_dict(torch.load(opt.model_path, map_location="cpu"))
    predict(net, opt.bin_paths, opt.reference_path, opt.batch_size, config.model.pileup_length, config.model.haplotype_length, opt.output, "cuda")


if __name__ == "__main__":
    main()
