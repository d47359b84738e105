"""ctypes binding of the C-ABI library (include/nanosnp_b200.h).

The library is the only compute path: if it cannot be loaded the import fails loudly -- there is
deliberately no pure-Python / PyTorch fallback for any kernel.
"""
from __future__ import annotations

import os
import ctypes as C
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["NSNP_LIB"]) if os.environ.get("NSNP_LIB") else _HERE / "libnanosnp_b200.so"   # NSNP_LIB: A/B builds

# error codes (include/nanosnp_b200.h)
OK, E_INVALID, E_CUDA, E_WORKSPACE, E_OVERFLOW, E_NO_DEVICE, E_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
CHANNELS, FLANK, WINDOW = 18, 16, 33
GT_CLASSES, ZY_CLASSES = 21, 3
F_COVERED, F_GATE = 1, 2
PREC_FP32, PREC_F16X3, PREC_F16X1 = 0, 1, 2
PROF_SLOTS = ("read_scan_kernel", "pileup_tile_kernel", "select_kernels", "gather_kernel", "lstm_layer0", "lstm_layer1", "tail_kernel", "site_record_kernel", "vcf_text_kernels")


class NsnpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"nanosnp_b200 error {code}: {msg}")
        self.code = code


class Reads(C.Structure):
    _fields_ = [
        ("n_reads", C.c_int64),
        ("pos", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p),
        ("cigar_off", C.c_void_p), ("cigar", C.c_void_p),
        ("seq_off", C.c_void_p), ("seq2", C.c_void_p), ("nmask", C.c_void_p), ("qual", C.c_void_p),
        ("n_cigar", C.c_int64), ("n_bases", C.c_int64), ("cigar_bits", C.c_int32), ("reserved", C.c_int32),
    ]


class Params(C.Structure):
    _fields_ = [
        ("snp_min_af", C.c_double), ("indel_min_af", C.c_double),
        ("min_coverage", C.c_int32), ("min_mapq", C.c_int32),
        ("excl_flags", C.c_uint32), ("max_depth", C.c_int32),
    ]


class ModelWeights(C.Structure):
    _fields_ = [
        ("w_ih", C.c_void_p * 4), ("w_hh", C.c_void_p * 4), ("b_ih", C.c_void_p * 4), ("b_hh", C.c_void_p * 4),
        ("proj_w", C.c_void_p), ("proj_b", C.c_void_p), ("dense_w", C.c_void_p), ("dense_b", C.c_void_p),
        ("gt_w", C.c_void_p), ("gt_b", C.c_void_p), ("zy_w", C.c_void_p), ("zy_b", C.c_void_p),
    ]


class HapWeights(C.Structure):
    _fields_ = [("w_ih", C.c_void_p * 12), ("w_hh", C.c_void_p * 12), ("b_ih", C.c_void_p * 12), ("b_hh", C.c_void_p * 12),
                ("proj_w", C.c_void_p * 2), ("proj_b", C.c_void_p * 2), ("dense_w", C.c_void_p), ("dense_b", C.c_void_p),
                ("gt_w", C.c_void_p), ("gt_b", C.c_void_p), ("zy_w", C.c_void_p), ("zy_b", C.c_void_p)]


class SynthCfg(C.Structure):
    _fields_ = [
        ("seed_ref", C.c_uint64), ("seed_var", C.c_uint64), ("seed_reads", C.c_uint64),
        ("contig_len", C.c_int64), ("n_reads", C.c_int64),
        ("sub_thr", C.c_uint32), ("ins_thr", C.c_uint32), ("del_thr", C.c_uint32), ("snp_thr", C.c_uint32),
        ("lowmapq_thr", C.c_uint32), ("secondary_thr", C.c_uint32), ("supp_thr", C.c_uint32),
        ("nbase_thr", C.c_uint32), ("softclip_thr", C.c_uint32), ("long_indel_thr", C.c_uint32),
        ("len_min", C.c_int32),
        ("ref_n_period", C.c_int32), ("ref_n_len", C.c_int32),
        ("ref_lower_period", C.c_int32), ("ref_lower_len", C.c_int32),
        ("gap_period", C.c_int32), ("gap_len", C.c_int32),
        ("use_eqx", C.c_int32),
        ("len_quantiles", C.c_void_p), ("mrun_cdf", C.c_void_p), ("indel_cdf", C.c_void_p),
    ]


# name -> (restype, argtypes).  Every symbol include/nanosnp_b200.h declares is listed here; the CPU test
# suite checks that the shared object exports each of them.
_P, _I64, _I32, _SZ = C.c_void_p, C.c_int64, C.c_int32, C.c_size_t
SYMBOLS = {
    "nsnp_default_params": (None, [C.POINTER(Params)]),
    "nsnp_abi_version": (C.c_int, []),
    "nsnp_last_error": (C.c_char_p, []),
    "nsnp_device_count": (C.c_int, []),
    "nsnp_pileup_workspace_bytes": (_SZ, [_I64, _I64, _I64]),
    "nsnp_pileup_counts": (C.c_int, [C.POINTER(Reads), _P, _I64, _I64, _I64, C.POINTER(Params), _P, _P, _P, _SZ, _P, _P]),
    "nsnp_select_workspace_bytes": (_SZ, [_I64]),
    "nsnp_select_candidates": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _I64, _I64, C.POINTER(Params), C.c_int, _P, _I64, _P, _P, _SZ, _P, _P]),
    "nsnp_pileup_targets_workspace_bytes": (_SZ, [_I64, _I64, _I64, _I64]),
    "nsnp_pileup_counts_targets": (C.c_int, [C.POINTER(Reads), _P, _I64, _I64, _I64, _P, _I64, C.POINTER(Params), _P, _P, _P, _SZ, _P, _P]),
    "nsnp_select_targets_workspace_bytes": (_SZ, [_I64, _I64]),
    "nsnp_select_candidates_targets": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _I64, _I64, _P, _I64, C.POINTER(Params), C.c_int, _P, _I64, _P,
                                                 _P, _SZ, _P, _P]),
    "nsnp_gather_windows": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _I64, _P, _P, _P, _P]),
    "nsnp_model_blob_bytes": (_SZ, []),
    "nsnp_model_pack_weights": (C.c_int, [C.POINTER(ModelWeights), _P, _SZ]),
    "nsnp_model_workspace_bytes": (_SZ, [_I64]),
    "nsnp_pileup_model_forward": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _P, _SZ, C.c_int, _P]),
    "nsnp_pileup_model_forward_sites": (C.c_int, [_P, _P, _I64, _I64, _P, _I64, _P, _P, _P, _P, _SZ, C.c_int, _P]),
    "nsnp_site_records_sites": (C.c_int, [_P, _P, _P, _I64, _P, _P, _I64, _P, _P, _P]),
    "nsnp_debug_lstm_tc_gates": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _I64, _P]),
    "nsnp_model_f16x1_reset": (C.c_int, [_P, _P]),
    "nsnp_model_f16x1_reevaluated": (C.c_int, [_P, _P, _P]),
    "nsnp_hap_features": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _I32, _P, _P]),
    "nsnp_hap_model_blob_bytes": (_SZ, []),
    "nsnp_hap_model_pack_weights": (C.c_int, [C.POINTER(HapWeights), _P, _SZ]),
    "nsnp_hap_model_workspace_bytes": (_SZ, [_I64]),
    "nsnp_hap_model_forward": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _SZ, _P]),
    "nsnp_hap_model_tc_blob_bytes": (_SZ, []),
    "nsnp_hap_model_tc_pack_weights": (C.c_int, [C.POINTER(HapWeights), _P, _SZ]),
    "nsnp_hap_model_tc_workspace_bytes": (_SZ, [_I64]),
    "nsnp_hap_model_tc_forward": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _SZ, _P]),
    "nsnp_debug_hap_tc_gates": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _I64, _P]),
    "nsnp_hap_checkpoint_count": (_I64, [_I64, _I64]),
    "nsnp_hap_read_ends": (C.c_int, [C.POINTER(Reads), _P, _P, _P]),
    "nsnp_hap_group_matrices": (C.c_int, [C.POINTER(Reads), _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I32, _I32, _I32, _P, _P, _P, _P, _P, _P]),
    "nsnp_profile_enable": (None, [C.c_int]),
    "nsnp_profile_read": (C.c_int, [_P, _P]),
    "nsnp_check_status": (C.c_int, [_P, _P]),
    "nsnp_vcf_format_batch": (_I64, [C.c_char_p, _I64, _P, _P, _P, _P, _P, _P, _I64]),
    "nsnp_site_records": (C.c_int, [_P, _P, _P, _P, _P, _I64, _P, _P, _P]),
    "nsnp_vcf_format_contig_records": (_I64, [C.c_char_p, _I64, _P, _I64, C.c_int, _P, _I64]),
    "nsnp_vcf_format_contig": (_I64, [C.c_char_p, _I64, _P, _P, _P, _P, _P, _I64, C.c_int, _P, _I64]),
    "nsnp_vcf_text_workspace_bytes": (_SZ, [_I64]),
    "nsnp_vcf_text_capacity": (_I64, [_I64, C.c_char_p]),
    "nsnp_vcf_text_records": (C.c_int, [C.c_char_p, _P, _I64, _P, _I64, _I64, _P, _P, _I64, _P, _P, _SZ, _P]),
    "nsnp_vcf_text_ties": (C.c_int, [_P, _I64, _P, _P, _P]),
    "nsnp_vcf_text_records_deferred": (C.c_int, [C.c_char_p, _P, _I64, _P, _P, _I64, _P, _P, _SZ, _P]),
    "nsnp_vcf_text_fixups": (C.c_int, [_P, _I64, _P, _P]),
    "nsnp_vcf_text_patch_heads": (C.c_int, [_P, _I64, _P, _I32, _I64, _I64, _P, _P]),
    "nsnp_vcf_text_patch_ties_at": (_I64, [C.c_char_p, _P, _I64, _I64, _P, _I32, _I64, _I64, _P]),
    "nsnp_vcf_batch_heads": (C.c_int, [_P, _I64, _P, _I64, _I64, _P, _P]),
    "nsnp_vcf_text_patch_ties": (_I64, [C.c_char_p, _P, _I64, _I64, _P, _I32]),
    "nsnp_vcf_format_records_at": (_I64, [C.c_char_p, _P, _I64, _I64, _I64, _P, _P, _I64]),
    "nsnp_bam_count": (_I64, [_P, _I64, _I64, _I32, _P, _P]),
    "nsnp_bam_fill": (_I64, [_P, _I64, _I64, _I32, _P, _P, _P, _P, _P, _P, _P, _P]),
    "nsnp_bam_open": (_P, [C.c_char_p, C.c_int]),
    "nsnp_bam_close": (None, [_P]),
    "nsnp_bam_n_ref": (_I32, [_P]),
    "nsnp_bam_ref_name": (C.c_char_p, [_P, _I32]),
    "nsnp_bam_ref_len": (_I64, [_P, _I32]),
    "nsnp_bam_has_index": (C.c_int, [_P]),
    "nsnp_bam_inflated_bytes": (_I64, [_P]),
    "nsnp_bam_next_contig": (_I32, [_P, _P, _P, _P, _P]),
    "nsnp_bam_fetch": (_I32, [_P, _I32, _I64, _I64, _P, _P, _P]),
    "nsnp_bam_fetch_ranges": (_I32, [_P, _I32, _P, _I64, _P, _P, _P]),
    "nsnp_bam_take": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "nsnp_bam_keep_aux": (C.c_int, [_P, C.c_int]),
    "nsnp_bam_take_aux": (C.c_int, [_P, _P, _P, _P]),
    "nsnp_synth_ref_host": (C.c_int, [C.POINTER(SynthCfg), _P]),
    "nsnp_synth_count_host": (C.c_int, [C.POINTER(SynthCfg), _P, _P, _P, _P, _P]),
    "nsnp_synth_fill_host": (C.c_int, [C.POINTER(SynthCfg), _P, _P, _P, _P, _P]),
    "nsnp_synth_ref_dev": (C.c_int, [C.POINTER(SynthCfg), _P, _P]),
    "nsnp_synth_count_dev": (C.c_int, [C.POINTER(SynthCfg), _P, _P, _P, _P, _P, _P]),
    "nsnp_synth_fill_dev": (C.c_int, [C.POINTER(SynthCfg), _P, _P, _P, _P, _P, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Loads the shared object (building it first if the sources are newer and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        from . import build as _build
        _build.build()
    if not LIB_PATH.exists():
        raise ImportError(f"{LIB_PATH} is missing: run `python -m nanosnp_b200.build` (needs nvcc); there is no CPU fallback")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError here = ABI mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.nsnp_abi_version() != 2:
        raise ImportError("nanosnp_b200: ABI version mismatch between _lib.py and the shared object")
    _lib = lib
    return lib


def check(code: int) -> None:
    if code < 0:
        raise NsnpError(code, load().nsnp_last_error().decode())


def default_params() -> Params:
    p = Params()
    load().nsnp_default_params(C.byref(p))
    return p
