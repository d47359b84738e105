"""GPU parity of the tcgen05 tensor-core PileupModel path (NSNP_PREC_F16X3, model_tc.cu)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# fp16 hi/lo split operands, fp32 TMEM accumulation, ex2/rcp.approx activations: observed max |dp| ~5e-6 against
# the CPU fp32 oracle (the fp32 FFMA path shows ~1e-6).  Enforced tolerance:
F16X3_ATOL = 5e-5


@pytest.fixture(scope="module")
def weights(golden_weights):
    from nanosnp_b200.pipeline import PileupModelWeights
    return PileupModelWeights(*golden_weights, device="cuda:0")


def _tile_layout(hi, lo):
    """[m][33][128] hi / lo -> layer-1 operand layout [tile][33][hi|lo][chunk 16][row 128][8]"""
    m = hi.shape[0]; tiles = (m + 127) // 128
    out = np.zeros((tiles, 33, 2, 16, 128, 8), np.float16)
    for part, a in enumerate((hi, lo)):
        pad = np.zeros((tiles * 128, 33, 128), np.float16); pad[:m] = a
        out[:, :, part] = pad.reshape(tiles, 128, 33, 16, 8).transpose(0, 2, 3, 1, 4)
    return out


def _col_order():
    n = np.arange(256)
    return ((n >> 2) & 3) * 64 + (n >> 5) * 8 + ((n >> 4) & 1) * 4 + (n & 3)


def _col_scale():
    """Activation scale folded into the packed weights (model_tc.cu): -log2(e) for i, f, o and -2 log2(e) for g."""
    n = np.arange(256)
    return np.where(((n >> 2) & 3) == 2, -2.0, -1.0) * np.log2(np.e)


@pytest.mark.parametrize("layer,cg", [(0, 2), (1, 2)])
def test_umma_operand_layout_first_step_gates(weights, golden_weights, small_case, layer, cg):
    """Raw TMEM accumulators of step 0 == W_ih . in + b (h = 0), from the production kernels (lstm0_pair2_kernel,
    lstm1_pair2x3_kernel) through the debug entry: validates descriptors, operand layout, hi/lo split."""
    import torch
    from nanosnp_b200 import _lib
    lib = _lib.load()
    enc, _ = golden_weights
    m = 300
    rng = np.random.default_rng(1)
    if layer == 0:
        xin = small_case["windows"][:m]
        xi = torch.from_numpy(xin).cuda(); h0 = None
    else:
        h = rng.uniform(-1, 1, size=(m, 33, 128)).astype(np.float32)
        hi = h.astype(np.float16); lo = (h - hi.astype(np.float32)).astype(np.float16)
        h0 = torch.from_numpy(_tile_layout(hi, lo)).cuda(); xi = None
        xin = hi.astype(np.float64) + lo.astype(np.float64)
    for d in (0, 1):
        sfx = "_reverse" if d else ""
        out = torch.full((m, 256), float("nan"), device="cuda")
        _lib.check(lib.nsnp_debug_lstm_tc_gates(weights.blob.data_ptr(), 0 if xi is None else xi.data_ptr(), layer, d, cg,
                                                0 if h0 is None else h0.data_ptr(), out.data_ptr(), m, torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        w = enc[f"lstm.weight_ih_l{layer}{sfx}"].astype(np.float64)
        b = (enc[f"lstm.bias_ih_l{layer}{sfx}"] + enc[f"lstm.bias_hh_l{layer}{sfx}"]).astype(np.float64)
        ref = (xin[:, 0 if d == 0 else 32, :].astype(np.float64) @ w.T + b)[:, _col_order()] * _col_scale()
        assert np.abs(out.cpu().numpy() - ref).max() < 1e-4          # accumulators carry the folded activation scale (up to 2.89x)


def test_tensor_core_forward_matches_oracle(weights, golden, small_case):
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupModelForward
    z = np.load(golden / "s2_small.npz")
    tc = PileupModelForward(weights, _lib.PREC_F16X3)
    f32 = PileupModelForward(weights, _lib.PREC_FP32)
    x = torch.from_numpy(small_case["windows"]).cuda()
    gt, zy = tc(x)
    g32, z32 = f32(x)
    torch.cuda.synchronize()
    assert np.abs(gt.cpu().numpy() - z["gt"]).max() < F16X3_ATOL and np.abs(zy.cpu().numpy() - z["zy"]).max() < F16X3_ATOL
    assert (gt - g32).abs().max().item() < F16X3_ATOL
    assert np.array_equal(gt.cpu().numpy().argmax(1), z["gt"].argmax(1)) and np.array_equal(zy.cpu().numpy().argmax(1), z["zy"].argmax(1))
    # ragged sizes around the 128-site tile and the 2-CTA cluster, float32 input, deep counts
    for n in (1, 127, 128, 129, 255, 256, 257, 1000):
        g, y = tc(x[:n])
        assert (g - gt[:n]).abs().max().item() == 0.0 and (y - zy[:n]).abs().max().item() == 0.0, n
    g, y = tc(x[:500].float())
    assert torch.equal(g, gt[:500])
    big = torch.full((130, 33, 18), 3000, dtype=torch.int32, device="cuda"); big[:, :, 0] = -12000
    g, y = tc(big); g2, y2 = f32(big)
    assert torch.isfinite(g).all() and (g - g2).abs().max().item() < 1e-3


def test_tensor_core_random_weights(small_case):
    import torch
    from oracle.s2_restate import PileupModelOracle
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupModelWeights, PileupModelForward
    m = PileupModelOracle(seed=77)
    tc = PileupModelForward(PileupModelWeights(*m.state_dicts(), device="cuda:0"), _lib.PREC_F16X3)
    x = small_case["windows"][:2000]
    g0, z0 = m.predict64(x)
    g1, z1 = tc(torch.from_numpy(x).cuda())
    assert np.abs(g1.cpu().numpy() - g0.numpy()).max() < F16X3_ATOL and np.abs(z1.cpu().numpy() - z0.numpy()).max() < F16X3_ATOL


def test_single_pass_mode_small_batches(weights, small_case):
    """NSNP_PREC_F16X1 just above its activation threshold (16 384 sites), int32 and float32 windows, with a device-side
    count: calls equal the three-pass path's, the low-margin sites carry its values, <= 16 384 sites are the three-pass path."""
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupModelForward
    tc = PileupModelForward(weights, _lib.PREC_F16X3)
    x1 = PileupModelForward(weights, _lib.PREC_F16X1)
    base = torch.from_numpy(small_case["windows"]).cuda()
    x = base.repeat(4, 1, 1)[:20_001].contiguous()                  # odd tile count, one chunk
    g3, z3 = tc(x)
    for inp in (x, x.float()):
        g1, z1 = x1(inp)
        n_low = x1.reevaluated()
        assert 0 < n_low <= 4096
        assert torch.equal(g1.argmax(1), g3.argmax(1)) and torch.equal(z1.argmax(1), z3.argmax(1))
        err = max(float((g1 - g3).abs().max()), float((z1 - z3).abs().max()))
        assert 1e-5 < err < 5e-3, err
        top = g3.topk(2, dim=1).values
        tight = (top[:, 0] - top[:, 1]) < 0.012
        assert int(tight.sum()) > 0 and torch.equal(g1[tight], g3[tight]) and torch.equal(z1[tight], z3[tight])
    nd = torch.tensor([17_000], dtype=torch.int32, device="cuda")   # device-side count below the host bound
    g1, z1 = x1(x, n_dev=nd)
    assert torch.equal(g1[:17_000].argmax(1), g3[:17_000].argmax(1))
    g1, z1 = x1(x[:16_384].contiguous())
    assert torch.equal(g1, g3[:16_384]) and x1.reevaluated() == 0


def test_single_pass_mode_reports_overflow(golden_weights, small_case):
    """More low-margin sites than the library re-evaluates (zero weights: every head is uniform) must not pass silently: the
    count check raises NSNP_E_OVERFLOW, and keeps raising after later clean calls on the same workspace."""
    import torch
    from nanosnp_b200 import _lib
    from nanosnp_b200.pipeline import PileupModelForward, PileupModelWeights
    enc, fwd = golden_weights
    zero = PileupModelWeights({k: np.zeros_like(v) for k, v in enc.items()}, {k: np.zeros_like(v) for k, v in fwd.items()}, device="cuda:0")
    x1 = PileupModelForward(zero, _lib.PREC_F16X1)
    x = torch.from_numpy(small_case["windows"]).cuda().repeat(4, 1, 1)[:20_000].contiguous()
    g, z = x1(x)
    assert torch.allclose(g, torch.full_like(g, 1 / 21)) and torch.allclose(z, torch.full_like(z, 1 / 3))
    with pytest.raises(_lib.NsnpError) as e:
        x1.reevaluated()
    assert e.value.code == _lib.E_OVERFLOW
    x1(x[:100].contiguous())
    with pytest.raises(_lib.NsnpError):
        x1.reevaluated()
