"""K9 (csrc/ccz_conv.cuh): the tcgen05 / TMA-im2col 3x3 convolution with the fused ResBlock epilogue
(net.py:33-41 with eval-mode BN folded) against a plain fp32 torch reference of the same op, through the
C ABI (ccz_conv3x3_c256).  The ragged-batch parity test bounds every element on its own (fp64 reference,
tests/test_forward_stages_gpu.elementwise_bound): fp32 accumulation over K = 2304 bf16 products, the fp32 epilogue and
one bf16 rounding of the output."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _case(n, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    cl = torch.channels_last
    x = torch.randn(n, 256, 10, 9, device="cuda", generator=g).to(torch.bfloat16).contiguous(memory_format=cl)
    skip = torch.randn(n, 256, 10, 9, device="cuda", generator=g).to(torch.bfloat16).contiguous(memory_format=cl)
    w = (torch.randn(256, 256, 3, 3, device="cuda", generator=g) * 0.03).to(torch.bfloat16).contiguous(memory_format=cl)
    bias = torch.randn(256, device="cuda", generator=g) * 0.1
    return x, skip, w, bias


def _ref(x, w, bias, skip):
    y = F.conv2d(x.float(), w.float(), bias, padding=1)
    if skip is not None:
        y = y + skip.float()
    return torch.relu(y)


@pytest.mark.parametrize("n", [1, 3, 37, 128, 300])  # ragged tails: n*90 is rarely a multiple of 128 / 256
@pytest.mark.parametrize("variant", [0, 1, 2, 34, 66])  # default, 1-CTA tiles, CTA pairs, 2 / 4 pairs per cluster
@pytest.mark.parametrize("with_skip", [False, True])
def test_conv_matches_fp32_reference(n, variant, with_skip):
    from chinesechesszero_b200 import _lib

    from tests.test_forward_stages_gpu import K_CONV, conv_reference, conv_y_ratio, gamma_f16

    x, skip, w, bias = _case(n, seed=n)
    sk = skip if with_skip else None
    y = _lib.conv3x3_c256(x, w, bias, sk, variant=variant)
    # fp64 reference of the same operands, per-element bound: fp32 accumulation over K + fp32 epilogue + bf16 output
    pre, wx, babs = conv_reference(x, w, bias, sk)
    assert conv_y_ratio(y, pre, wx, babs, gamma_f16(K_CONV)) <= 1.0
    assert y.is_contiguous(memory_format=torch.channels_last)


def test_conv_halo_is_zero_padding_and_boards_are_independent():
    """One hot pixel at a corner / edge of one board must only reach its 3x3 neighbourhood on that board."""
    from chinesechesszero_b200 import _lib

    _, _, w, bias = _case(1)
    x = torch.zeros(4, 256, 10, 9, device="cuda", dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last)
    x[1, 5, 0, 0] = 1.0   # corner
    x[2, 7, 9, 8] = 2.0   # opposite corner
    x[3, 9, 4, 8] = -1.0  # right edge
    y = _lib.conv3x3_c256(x, w, torch.zeros_like(bias))
    ref = _ref(x, w, torch.zeros_like(bias), None)
    assert (y.float() - ref).abs().max().item() <= 2.0 ** -8 * ref.abs().max().item()
    assert y[0].abs().max().item() == 0.0  # untouched board stays zero (no bleed across boards)


def test_conv_in_place_block_update_and_determinism():
    """out may alias skip (the evaluator updates the block input in place); two runs are bit-identical."""
    from chinesechesszero_b200 import _lib

    x, skip, w, bias = _case(200, seed=5)
    a = _lib.conv3x3_c256(x, w, bias, skip)
    s2 = skip.clone(memory_format=torch.channels_last)
    b = _lib.conv3x3_c256(x, w, bias, s2, out=s2)
    assert b.data_ptr() == s2.data_ptr() and torch.equal(a, b)


def test_conv_rejects_bad_arguments():
    from chinesechesszero_b200 import _lib

    x, skip, w, bias = _case(2)
    with pytest.raises(_lib.CczError):
        _lib.conv3x3_c256(x.contiguous(), w, bias)  # NCHW-contiguous input
    with pytest.raises(_lib.CczError):
        _lib.conv3x3_c256(x, w, bias.to(torch.bfloat16))
    with pytest.raises(_lib.CczError):
        _lib.conv3x3_c256(x, w, bias, out=x)  # output aliasing the input would corrupt halo reads
    with pytest.raises(_lib.CczError):
        _lib.conv3x3_c256(x, w, bias, variant=3)
