"""Host-side quantisation of the FP8 evaluator (net.py): e4m3 rounding, weight and activation scales, argument checks.
CPU only; the device kernels use the same rounding (cvt.rn.satfinite.e4m3x2.f32) and are checked in test_fp8_gpu.py."""
import numpy as np
import pytest
import torch

from chinesechesszero_b200 import net as N


def _e4m3_values():
    """Every finite non-negative float8_e4m3fn value by code 0x00..0x7E, decoded from the bit layout (1-4-3, bias 7)."""
    vals = []
    for code in range(0x7F):
        e, m = code >> 3, code & 7
        vals.append(m * 2.0 ** -9 if e == 0 else (1 + m / 8) * 2.0 ** (e - 7))
    return np.array(vals)


def _satfinite_ref(x: float) -> float:
    """Round to nearest e4m3, ties to the even code, magnitudes past 448 saturate to 448."""
    vals = _e4m3_values()
    a = min(abs(x), 448.0)
    i = int(np.searchsorted(vals, a))
    if i < len(vals) and vals[i] == a:
        r = vals[i]
    else:
        lo, hi = vals[i - 1], vals[i]
        r = lo if (a - lo < hi - a or (a - lo == hi - a and (i - 1) % 2 == 0)) else hi
    return float(np.copysign(r, x))


EDGES = [0.0, -0.0, 1.0, 1.0625, 1.1875, 1.125 + 1e-6, 2.0 ** -6, 2.0 ** -9, 2.0 ** -10, 3 * 2.0 ** -10, 2.0 ** -11, 7 * 2.0 ** -10,
         240.0, 248.0, 432.0, 440.0, 447.0, 448.0, 449.0, 464.0, 480.0, 1e4, 3e38, -448.0, -460.0, -1e30, -1.0625, -2.0 ** -10, 0.3, 5.7]


def test_e4m3_quantize_is_satfinite_round_to_nearest_even():
    got = N.e4m3_quantize(torch.tensor(EDGES, dtype=torch.float32), 1.0).float().numpy()
    ref = np.array([_satfinite_ref(float(np.float32(x))) for x in EDGES])
    assert not np.isnan(got).any()
    np.testing.assert_array_equal(got, ref)
    assert got[EDGES.index(1.0625)] == 1.0 and got[EDGES.index(1.1875)] == 1.25  # ties to even
    assert got[EDGES.index(2.0 ** -10)] == 0.0 and got[EDGES.index(3 * 2.0 ** -10)] == 2.0 ** -8  # subnormal ties
    assert got[EDGES.index(1e4)] == 448.0 and got[EDGES.index(-1e30)] == -448.0


def test_e4m3_quantize_applies_the_scale_in_fp32_and_keeps_channels_last():
    x = torch.randn(3, 256, 10, 9).contiguous(memory_format=torch.channels_last) * 10
    inv = torch.tensor([0.37])
    q = N.e4m3_quantize(x, inv)
    assert q.dtype == torch.float8_e4m3fn and q.is_contiguous(memory_format=torch.channels_last)
    ref = np.vectorize(_satfinite_ref)((x.float() * inv).numpy())
    np.testing.assert_array_equal(q.float().numpy(), ref)


def test_weight_scales_are_per_output_channel_amax_over_448():
    torch.manual_seed(0)
    w = torch.randn(256, 256, 3, 3) * torch.linspace(0.01, 2.0, 256).view(-1, 1, 1, 1)
    w[7] = 0.0
    s = N.weight_scales(w)
    amax = w.abs().flatten(1).amax(1)
    assert s.shape == (256,)
    torch.testing.assert_close(s[amax > 0], amax[amax > 0] / 448.0, rtol=0, atol=0)
    assert s[7] == 1.0
    q = N.e4m3_quantize(w, (1.0 / s).view(-1, 1, 1, 1)).float()
    # every live channel uses the top of the e4m3 range and nothing saturates beyond it
    assert torch.all(q.abs().flatten(1).amax(1)[amax > 0] == 448.0)
    rel = ((q * s.view(-1, 1, 1, 1) - w).abs() / amax.clamp_min(1e-30).view(-1, 1, 1, 1)).amax()
    assert rel <= 16.0 / 448  # half an ulp of the top binade (32), relative to the channel's amax


def test_activation_scale_from_calibration_amax():
    amax = torch.tensor([4.48, 0.0, 1000.0, 1e-3])
    s = N.activation_scale(amax)
    torch.testing.assert_close(s, torch.tensor([0.01, 1.0, 1000.0 / 448.0, 1e-3 / 448.0]))
    x = torch.tensor([0.0, 2.24, 4.48, 9.0])
    assert N.e4m3_quantize(x, 1.0 / s[0]).float().tolist() == [0.0, 224.0, 448.0, 448.0]


def test_precision_argument_is_checked():
    net = N.Net(num_channels=32, resblocks_num=1)
    with pytest.raises(ValueError, match="precision"):
        N.BatchedEvaluator(net, device="cpu", precision="fp16")
    with pytest.raises(ValueError, match="fp8"):  # no K9 on the CPU, and a 32-channel net: no silent bf16 fallback
        N.BatchedEvaluator(net, device="cpu", precision="fp8")
    with pytest.raises(ValueError, match="fp8"):
        N.BatchedEvaluator(net, device="cpu", precision="fp8", conv_impl="torch")
