"""The PileupModel past the counts s1 writes, and at other weight scales, against the float64 network.

s1 caps a tile at 16 383 reads, but the model also takes windows that never pass through s1: `.pd` text, the LSTMNetwork
drop-in, float32 windows.  fp16 ends at 65 504, so the tensor-core path stages layer-0 inputs as x 2^-8 (its hi weight halves
carry the 2^8 back): counts up to 65 504 x 2^8 = 16 769 024 (TOP) keep the hi/lo split's accuracy, up to 2 TOP the lo half
carries the excess at fp16 precision, and larger counts saturate at 2 TOP (where every gate they reach is saturated as well).
Covered here:
  - a count ladder (0, +-1 ... 65 519, 65 520 ... TOP, INT32_MAX) in each of the 18 channels (16 and 17 are staged by another
    warp, with the bias column) at steps 0, 16 and 32, and deep-pile-up windows with reference channels at -(65 520 ... 10^6);
  - int32 windows, float32 windows and the count-tensor entry, in fp32, f16x3 and f16x1, with ladder sites first and last in
    batches of 1, 129, 385 and 4 097 sites; the raw step-0 gates of the production layer-0 kernel (debug entry);
  - the shipped weights, a seeded PyTorch init, shipped x4 (saturated gates) and shipped x1/8 (subnormal lo halves);
  - the predict CLI on a `.pd` file holding such windows, in every precision: no record may be dropped;
  - on the CPU: weights whose fp16 halves would not be finite are refused by the packer, naming the tensor.
"""
import ctypes as C
import os
from pathlib import Path

import numpy as np
import pytest

from test_gpu_deep import _argmax_where_clear, _col_order, _col_scale, _compare_rows, _dense_rows, _onehot_rows
from test_gpu_l1_pair2_f16x3 import _same_bytes, _windows
from test_gpu_tc import F16X3_ATOL

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"
FP32_ATOL = 2e-5
F16X1_ATOL = 5e-3
TOP = 65504 * 256                     # the top of the range the tensor-core path stages exactly (x 2^-8 in fp16)
INT32_MAX = 2**31 - 1
LADDER = (1, 2047, 2048, 2049, 4095, 4097, 16383, 16385, 32767, 32769, 65503, 65504, 65519, 65520, 65521, 100_001, 2**20 - 1,
          TOP, INT32_MAX)
VALUES = (0,) + tuple(s * v for v in LADDER for s in (1, -1))
EXTREME = tuple(v for v in VALUES if abs(v) >= 65503)
STEPS = (0, 16, 32)                   # first step of each direction, and the centre


def _ladder():
    """One window per (value, channel, step): an ordinary window of the small case with that one entry set."""
    keys = [(v, c, t) for v in VALUES for c in range(18) for t in STEPS]
    x = _windows(GOLDEN, len(keys), seed=11)
    for i, (v, c, t) in enumerate(keys):
        x[i, t, c] = v
    return x, keys


def _pileup_rows(n, seed):
    """Deep-pile-up-shaped windows past fp16: a reference channel per strand at -(65 520 ... 10^6), the others at a few thousand."""
    rng = np.random.default_rng(seed)
    x = rng.integers(1, 4000, (n, 33, 18)).astype(np.int32)
    x[:, :, [0, 9]] = -rng.integers(65_520, 1_000_001, (n, 33, 2))
    return x


def _staged(x):
    """The count the tensor-core path computes with: x up to TOP (its hi/lo split is exact to 2^-22), 65 504 + the fp16 excess
    (times 2^8) up to 2 TOP, saturated beyond."""
    y = np.asarray(x, np.float64) / 256.0
    hi = np.clip(y, -65504.0, 65504.0)
    lo = np.clip(y - hi, -65504.0, 65504.0).astype(np.float16).astype(np.float64)
    return 256.0 * (hi + lo)


def _counts_entry(x):
    """A synthetic count tensor holding the windows back to back, and the centre row of each: from_counts reads x back."""
    return np.ascontiguousarray(x.reshape(-1, 18)), (np.arange(len(x)) * 33 + 16).astype(np.int32)


def _x1_batch(x):
    """20 001 ordinary windows (above the 16 384 sites where the single pass engages) with the windows x at seeded slots."""
    big = _windows(GOLDEN, 20_001)
    assert np.abs(big).max() <= 2048
    slots = np.sort(np.random.default_rng(41).choice(len(big), len(x), replace=False))
    big[slots] = x
    return big, slots


def _check(what, g, z, g64, z64, tol):
    assert np.isfinite(g).all() and np.isfinite(z).all(), what
    err = max(float(np.abs(g - g64).max()), float(np.abs(z - z64).max()))
    assert err < tol, (what, err)
    assert _argmax_where_clear(g, g64, tol) and _argmax_where_clear(z, z64, tol), what
    return err


def _weights_sets(golden_weights):
    from oracle.s2_restate import PileupModelOracle
    enc, fwd = golden_weights
    scale = lambda k: ({n: v * k for n, v in enc.items()}, {n: v * k for n, v in fwd.items()})
    return {"shipped": golden_weights, "seed77": PileupModelOracle(seed=77).state_dicts(), "x4": scale(4.0), "x1/8": scale(0.125)}


@pytest.fixture(scope="module")
def weights(golden_weights):
    from nanosnp_b200.pipeline import PileupModelWeights
    return PileupModelWeights(*golden_weights, device="cuda:0")


@pytest.fixture(scope="module")
def model64(golden_weights):
    import torch
    from oracle.s2_restate import PileupModelOracle
    torch.set_num_threads(os.cpu_count() or 1)
    return PileupModelOracle(*golden_weights)


@pytest.fixture(scope="module")
def cases(model64):
    """The ladder and 256 deep-pile-up windows, and their float64 probabilities."""
    lad, keys = _ladder()
    x = np.concatenate([lad, _pileup_rows(256, 3)])
    g64, z64 = (t.numpy() for t in model64.predict64(x))
    return {"x": x, "keys": keys, "g64": g64, "z64": z64}


# ------------------------------------------------------------------------------------------------ count ladder
@pytest.mark.gpu
def test_count_ladder_every_entry_point_and_precision(weights, cases):
    """Every ladder and pile-up window, int32 / float32 windows and the count-tensor entry, fp32 and f16x3: within the bars of
    the float64 network, no NaN, equal argmax wherever float64's margin is clear."""
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupModelForward
    x, g64, z64 = cases["x"], cases["g64"], cases["z64"]
    xt = torch.from_numpy(x).cuda()
    for prec, tol in ((_lib.PREC_FP32, FP32_ATOL), (_lib.PREC_F16X3, F16X3_ATOL)):
        fwd = PileupModelForward(weights, prec)
        for dt in (torch.int32, torch.float32):
            g, z = fwd(xt.to(dt).contiguous())
            _check((prec, dt), g.cpu().numpy(), z.cpu().numpy(), g64, z64, tol)
    cnt, pos = _counts_entry(x)
    g, z = PileupModelForward(weights, _lib.PREC_F16X3).from_counts(torch.from_numpy(cnt).cuda(), 0, torch.from_numpy(pos).cuda(), len(x))
    _check("from_counts", g.cpu().numpy(), z.cpu().numpy(), g64, z64, F16X3_ATOL)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 129, 385, 4097])
def test_extreme_counts_first_and_last_in_the_batch(weights, model64, n):
    """Each window with a count of 65 503 or more (18 values x channels 0, 8, 15, 16, 17 x steps 0, 16, 32) sits first or last
    in a batch of n ordinary windows (n = 1, 4 097: an odd tile count, whose padding CTA re-reads the last real tile)."""
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupModelForward
    keys = [(v, c, t) for v in EXTREME for c in (0, 8, 15, 16, 17) for t in STEPS]
    ext = _windows(GOLDEN, len(keys), seed=12)
    for i, (v, c, t) in enumerate(keys):
        ext[i, t, c] = v
    base = _windows(GOLDEN, n, seed=13)
    slots = (0,) if n == 1 else (0, n - 1)
    gb, zb = (t.numpy() for t in model64.predict64(base))
    ge, ze = (t.numpy() for t in model64.predict64(ext))
    batches, g64, z64 = [], [], []
    for k in range(0, len(keys), len(slots)):
        b, g, z = base.copy(), gb.copy(), zb.copy()
        for s, i in zip(slots, range(k, min(k + len(slots), len(keys)))):
            b[s], g[s], z[s] = ext[i], ge[i], ze[i]
        batches.append(b); g64.append(g); z64.append(z)
    g64, z64 = np.concatenate(g64), np.concatenate(z64)
    fwd = {p: PileupModelForward(weights, p) for p in (_lib.PREC_FP32, _lib.PREC_F16X3)}
    got = {k: ([], []) for k in ("fp32", "i32", "f32", "counts")}
    for b in batches:
        xb = torch.from_numpy(b).cuda()
        for key, out in (("fp32", fwd[_lib.PREC_FP32](xb)), ("i32", fwd[_lib.PREC_F16X3](xb)), ("f32", fwd[_lib.PREC_F16X3](xb.float()))):
            got[key][0].append(out[0].cpu().numpy()); got[key][1].append(out[1].cpu().numpy())
        cnt, pos = _counts_entry(b)
        g, z = fwd[_lib.PREC_F16X3].from_counts(torch.from_numpy(cnt).cuda(), 0, torch.from_numpy(pos).cuda(), n)
        got["counts"][0].append(g.cpu().numpy()); got["counts"][1].append(z.cpu().numpy())
    for key, (gs, zs) in got.items():
        _check((n, key), np.concatenate(gs), np.concatenate(zs), g64, z64, FP32_ATOL if key == "fp32" else F16X3_ATOL)


@pytest.mark.gpu
def test_single_pass_mode_carries_three_pass_bytes_above_2048(weights, cases):
    """NSNP_PREC_F16X1 on 20 001 sites holding every ladder and pile-up window: each site with a count above 2048 (2049 and up)
    carries f16x3's bytes, through int32, float32 and the count tensor; the others stay within the single-pass bar."""
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupModelForward
    x, slots = _x1_batch(cases["x"])
    deep = (np.abs(x) > 2048).any(axis=(1, 2))
    at2048 = ~deep & (np.abs(x) == 2048).any(axis=(1, 2))
    assert deep.sum() > 1900 and at2048.sum() > 0
    xt = torch.from_numpy(x).cuda()
    cnt, pos = _counts_entry(x)
    cnt, pos = torch.from_numpy(cnt).cuda(), torch.from_numpy(pos).cuda()
    tc = PileupModelForward(weights, _lib.PREC_F16X3)
    g3, z3 = (t.cpu().numpy() for t in tc(xt))
    assert np.isfinite(g3).all()
    _check("f16x3 ladder slots", g3[slots], z3[slots], cases["g64"], cases["z64"], F16X3_ATOL)
    g3c, z3c = (t.cpu().numpy() for t in tc.from_counts(cnt, 0, pos, len(x)))
    x1 = PileupModelForward(weights, _lib.PREC_F16X1)
    for name, run, ref in (("i32", lambda: x1(xt), (g3, z3)), ("f32", lambda: x1(xt.float()), (g3, z3)),
                           ("counts", lambda: x1.from_counts(cnt, 0, pos, len(x)), (g3c, z3c))):
        g1, z1 = (t.cpu().numpy() for t in run())
        assert deep.sum() <= x1.reevaluated() <= 4096, name
        assert _same_bytes(g1[deep], ref[0][deep]) and _same_bytes(z1[deep], ref[1][deep]), name
        assert np.isfinite(g1).all() and np.array_equal(g1.argmax(1), ref[0].argmax(1)) and np.array_equal(z1.argmax(1), ref[1].argmax(1)), name
        assert max(float(np.abs(g1 - ref[0]).max()), float(np.abs(z1 - ref[1]).max())) < F16X1_ATOL, name


@pytest.mark.gpu
@pytest.mark.parametrize("cg", [2])
def test_layer0_gates_of_the_count_ladder(weights, golden_weights, cases, cg):
    """Raw step-0 layer-0 accumulators (debug entry: lstm0_pair2_kernel, both directions) of the ladder and pile-up windows
    against the float64 product, relative to sum |x w|; counts beyond TOP are taken as staged (_staged: saturated at 2 TOP)."""
    _gates_within_sum_xw(weights.blob, golden_weights[0], cases["x"], cg)


# ------------------------------------------------------------------------------------------------ other weight scales
def _gates_within_sum_xw(blob, enc, x, cg=2):
    """Step-0 layer-0 accumulators of both directions (debug entry) within 1e-5 of sum |x w| of the float64 product (plus, for a
    count past TOP, the fp16 precision of its excess)."""
    import torch
    from nanosnp_b200 import _lib
    lib = _lib.load()
    xi = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    for d in (0, 1):
        sfx = "_reverse" if d else ""
        out = torch.full((len(x), 256), float("nan"), device="cuda")
        _lib.check(lib.nsnp_debug_lstm_tc_gates(blob.data_ptr(), xi.data_ptr(), 0, d, cg, 0, out.data_ptr(), len(x),
                                                torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        w = np.asarray(enc[f"lstm.weight_ih_l0{sfx}"], np.float64)
        b = np.asarray(enc[f"lstm.bias_ih_l0{sfx}"], np.float64) + np.asarray(enc[f"lstm.bias_hh_l0{sfx}"], np.float64)
        xt = _staged(x[:, 0 if d == 0 else 32, :])
        ref = (xt @ w.T + b)[:, _col_order()] * _col_scale()
        mag = (np.abs(xt) @ np.abs(w).T + np.abs(b))[:, _col_order()] * np.abs(_col_scale())
        # Allowed on top of the bound: past TOP the lo half holds the excess itself, so the dropped lo.w_lo term is the excess
        # times w's fp16 rounding error (2^-11 relative, 2^-25 absolute for a subnormal hi half); and a lo weight half below
        # fp16's normal range (2^-14 after its 2^10 pre-scale) keeps w to 2^-35 absolute, times a count of up to millions
        excess = np.abs(xt - np.clip(xt, -TOP, TOP))
        extra = ((excess @ (2.0**-11 * np.abs(w)).T)[:, _col_order()] * np.abs(_col_scale()) + 2.0**-25 * excess.sum(1, keepdims=True)
                 + 2.0**-35 * np.abs(xt).sum(1, keepdims=True))
        got = out.cpu().numpy().astype(np.float64)
        assert np.isfinite(got).all(), (cg, d)
        worst = float((np.maximum(np.abs(got - ref) - extra, 0.0) / (mag + 1.0)).max())
        assert worst < 1e-5, (cg, d, worst)


@pytest.mark.gpu
@pytest.mark.parametrize("wset", ["shipped", "seed77", "x4", "x1/8"])
def test_weight_scales(golden_weights, small_case, wset):
    """The shipped weights, a seeded PyTorch init, the shipped weights x4 (saturated gates: the ex2 / rcp epilogue at inf) and
    x1/8 (lo halves of weights and of h deep in fp16's subnormal range), on the small case's windows, deep windows
    (2049 ... 16 383) and the count ladder: no NaN or inf, and the layer-0 gates within 1e-5 of sum |x w|.  fp32 and f16x3 meet
    their bars of float64 -- except with x4, where the float64 network itself is ill-conditioned: the fp32 path's own error
    on the small case's windows is over 1e-2 (~0.3 on a B200), so no absolute bar can hold there and the gate bound is the check."""
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupModelForward, PileupModelWeights
    from oracle.s2_restate import PileupModelOracle
    torch.set_num_threads(os.cpu_count() or 1)
    enc, fwd = _weights_sets(golden_weights)[wset]
    m64 = PileupModelOracle(enc, fwd)
    w = PileupModelWeights(enc, fwd, device="cuda:0")
    lad, _ = _ladder()
    for name, x in (("small", small_case["windows"][:2000]), ("deep", np.concatenate([_onehot_rows(1024, 3), _dense_rows(1024, 4)])),
                    ("ladder", np.concatenate([lad, _pileup_rows(256, 5)]))):
        _gates_within_sum_xw(w.blob, enc, x)
        g64, z64 = (t.numpy() for t in m64.predict64(x))
        xt = torch.from_numpy(x).cuda()
        for prec, tol in ((_lib.PREC_FP32, FP32_ATOL), (_lib.PREC_F16X3, F16X3_ATOL)):
            g, z = (t.cpu().numpy() for t in PileupModelForward(w, prec)(xt))
            assert np.isfinite(g).all() and np.isfinite(z).all(), (wset, name, prec)
            if wset != "x4":
                _check((wset, name, prec), g, z, g64, z64, tol)
            elif name == "small" and prec == _lib.PREC_FP32:
                assert float(np.abs(g - g64).max()) > 1e-2          # ill-conditioned: fp32 rounding alone moves p by > 1e-2


# ------------------------------------------------------------------------------------------------ end to end
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "f16x3", "f16x1"])
def test_predict_cli_pd_with_counts_past_fp16(tmp_path, golden_weights, model64, small_case, precision):
    """`python -m nanosnp_b200.predict -data x.pd` on the small case's windows, every third one turned into a deep pile-up with
    reference counts of 65 520 ... 10^6: the rows equal the oracle's (predict.py's formatter on float64 probabilities), none dropped."""
    from nanosnp_b200 import predict as P
    from nanosnp_b200.postprocess import write_pd
    from oracle.pyoracle import write_fasta
    from oracle.s2_restate import vcf_records
    ref, pos = small_case["ref"], small_case["site_pos"]
    x = small_case["windows"].copy()
    deep = np.arange(len(x)) % 3 == 0
    x[deep, :, 0] = -np.random.default_rng(51).integers(65_520, 1_000_001, (int(deep.sum()), 33))
    x[deep, :, 9] = -np.random.default_rng(52).integers(65_520, 1_000_001, (int(deep.sum()), 33))
    up = np.char.upper(ref[pos - 1].view("S1")).view(np.uint8)
    keep = np.isin(up, np.frombuffer(b"ACGT", np.uint8))
    d = tmp_path / "pd"; d.mkdir()
    assert write_pd(str(d / "ctg1.pd"), "ctg1", pos, ref, x) == int(keep.sum())
    g64, z64 = (t.numpy() for t in model64.predict64(x[keep]))
    want = vcf_records(["ctg1"] * int(keep.sum()), pos[keep], up[keep], x[keep].astype(np.float32), g64, z64).splitlines()
    assert sum(int(l.split("\t")[9].split(":")[2]) > 65_520 for l in want) > 10
    fa = str(tmp_path / "ref.fa")
    write_fasta(fa, {"ctg1": ref})
    out = str(tmp_path / "out.vcf")
    cfg = str(P.__file__).replace("predict.py", "config/ont_pileup.yaml")
    P.main(["-config", cfg, "-model_path", str(GOLDEN / "ont_pileup_weights.npz"), "-data", str(d), "-reference", fa, "-output", out,
            "--precision", precision])
    _compare_rows([l for l in open(out).read().splitlines() if not l.startswith("#")], want)


# ------------------------------------------------------------------------------------------------ packer (CPU)
def _pack(enc, fwd):
    from nanosnp_b200 import _lib
    lib = _lib.load()
    keep = []

    def ptr(a):
        a = np.ascontiguousarray(a, dtype=np.float32); keep.append(a); return a.ctypes.data
    w = _lib.ModelWeights()
    for layer in range(2):
        for d, sfx in enumerate(("", "_reverse")):
            i = layer * 2 + d
            w.w_ih[i] = ptr(enc[f"lstm.weight_ih_l{layer}{sfx}"]); w.w_hh[i] = ptr(enc[f"lstm.weight_hh_l{layer}{sfx}"])
            w.b_ih[i] = ptr(enc[f"lstm.bias_ih_l{layer}{sfx}"]); w.b_hh[i] = ptr(enc[f"lstm.bias_hh_l{layer}{sfx}"])
    w.proj_w, w.proj_b = ptr(enc["output_proj.weight"]), ptr(enc["output_proj.bias"])
    w.dense_w, w.dense_b = ptr(fwd["dense.weight"]), ptr(fwd["dense.bias"])
    w.gt_w, w.gt_b = ptr(fwd["genotype_layer.weight"]), ptr(fwd["genotype_layer.bias"])
    w.zy_w, w.zy_b = ptr(fwd["zygosity_layer.weight"]), ptr(fwd["zygosity_layer.bias"])
    nbytes = lib.nsnp_model_blob_bytes()
    blob = np.zeros(nbytes, np.uint8)
    rc = lib.nsnp_model_pack_weights(C.byref(w), blob.ctypes.data, nbytes)
    return rc, (lib.nsnp_last_error().decode() if rc else ""), blob


# (tensor, index, value just inside, value just outside): row 130 is a g-gate row (activation scale 2 log2 e); a layer-0 input
# weight or bias meets 2^8 as well, so its limit is 65 520 / 2^8 / (2 log2 e) = 88.7; every other one 65 520 / (2 log2 e) = 22 707
PACK_LIMITS = [
    ("lstm.weight_ih_l0", (130, 5), 88.0, 89.0, "lstm.weight_ih_l0[130][5]"),
    ("lstm.weight_ih_l0_reverse", (130, 17), -88.0, -89.0, "lstm.weight_ih_l0_reverse[130][17]"),
    ("lstm.bias_ih_l0", (130,), 88.0, 89.0, "lstm.bias_ih_l0 + lstm.bias_hh_l0[130]"),
    ("lstm.weight_hh_l0", (130, 3), 22_000.0, 23_000.0, "lstm.weight_hh_l0[130][3]"),
    ("lstm.weight_ih_l1_reverse", (130, 100), 22_000.0, 23_000.0, "lstm.weight_ih_l1_reverse[130][100]"),
    ("lstm.weight_hh_l1", (130, 63), -22_000.0, -23_000.0, "lstm.weight_hh_l1[130][63]"),
]


@pytest.mark.parametrize("tensor,idx,inside,outside,name", PACK_LIMITS)
def test_pack_refuses_weights_outside_fp16(golden_weights, tensor, idx, inside, outside, name):
    """A weight whose fp16 hi or lo operand half would be inf is an error that names the tensor and the element, not a blob
    with inf in it; the same weight just inside the range packs.  (Host-only call: no GPU needed.)"""
    from nanosnp_b200 import _lib
    enc, fwd = golden_weights
    for v, ok in ((inside, True), (outside, False)):
        e = {k: a.copy() for k, a in enc.items()}
        e[tensor][idx] = v
        if tensor.startswith("lstm.bias_ih"):
            e[tensor.replace("bias_ih", "bias_hh")][idx] = 0.0
        rc, msg, blob = _pack(e, fwd)
        if ok:
            assert rc == 0, msg
        else:
            assert rc == _lib.E_INVALID and name in msg, (rc, msg)


def test_pack_refuses_folded_dense_weights_outside_fp16(golden_weights):
    """The tail's folded dense o output_proj weights are split into fp16 halves as well: out of range is refused by name."""
    from nanosnp_b200 import _lib
    enc, fwd = golden_weights
    rc, msg, _ = _pack(enc, fwd)
    assert rc == 0, msg
    f = {k: a.copy() for k, a in fwd.items()}
    f["dense.weight"][7] *= 1e6
    rc, msg, _ = _pack(enc, f)
    assert rc == _lib.E_INVALID and "dense.weight" in msg, (rc, msg)


def test_pack_layer0_input_hi_halves_carry_the_staging_scale(golden_weights):
    """The layer-0 input columns (x and the bias column) hold fp16(w s) 2^8 in their hi half and fp16((w s - hi) 2^10) in their lo
    half; the h columns fp16(w s) and the plain remainder (s = the folded activation scale)."""
    enc, fwd = golden_weights
    rc, msg, blob = _pack(enc, fwd)
    assert rc == 0, msg
    from nanosnp_b200 import _lib
    lib = _lib.load()
    # tensor-core section: after the float blob (rounded up to 256 bytes); L0 d0 hi, L0 d0 lo, each [96/8][256][8] halfs
    n_float = (lib.nsnp_model_blob_bytes() - (4 * 96 + 4 * 192 + 2 * 128) * 256 * 2 - 2 * 256 * 4)
    hi = blob[n_float:n_float + 96 * 256 * 2].view(np.float16).reshape(12, 256, 8).transpose(1, 0, 2).reshape(256, 96)
    lo = blob[n_float + 96 * 256 * 2:n_float + 2 * 96 * 256 * 2].view(np.float16).reshape(12, 256, 8).transpose(1, 0, 2).reshape(256, 96)
    w = np.zeros((256, 96), np.float32)
    w[:, :18] = enc["lstm.weight_ih_l0"]
    w[:, 18] = enc["lstm.bias_ih_l0"] + enc["lstm.bias_hh_l0"]
    w[:, 32:] = enc["lstm.weight_hh_l0"]
    v = w[_col_order()] * _col_scale()[:, None].astype(np.float32)
    h = v.astype(np.float16)
    assert np.array_equal(hi[:, :32], (h[:, :32].astype(np.float32) * 256).astype(np.float16))
    assert np.array_equal(lo[:, :32], ((v[:, :32] - h[:, :32].astype(np.float32)) * 1024).astype(np.float16))
    assert np.array_equal(hi[:, 32:], h[:, 32:]) and np.array_equal(lo[:, 32:], (v[:, 32:] - h[:, 32:].astype(np.float32)).astype(np.float16))

