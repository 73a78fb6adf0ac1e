"""K9's pixel tiles (variant 128, the bf16 default tiling, csrc/ccz_conv.cuh) against tiles of consecutive pixels (variant 2,
the tiling K9 used before and still the e4m3 default).

A pixel tile multiplies only the filter taps that fall on the board; the k-blocks it drops contribute exact zeros to
every accumulator of the tile, and the taps it keeps are accumulated in the same order.  So the two tilings must agree
bit for bit (compared as int16 / uint8 views), for every batch size around the 128-board rows of a CTA and the 256-board
blocks of a CTA pair, with and without the skip input, through the device-count entry point, and for the e4m3 kernel's
bf16 and e4m3 outputs."""
import pytest
import torch

pytestmark = pytest.mark.gpu

CL = torch.channels_last
SIZES = (1, 2, 127, 128, 129, 255, 256, 257, 300, 3760, 4096)
OLD, NEW = 2, 128  # _lib.CONV_VARIANT_PAIR (tiles of 256 consecutive pixels on CTA pairs), _lib.CONV_VARIANT_PIXEL


@pytest.fixture(scope="module")
def data():
    torch.manual_seed(0)
    n = max(SIZES)
    x = torch.randn(n, 256, 10, 9, device="cuda").relu().to(torch.bfloat16).contiguous(memory_format=CL)
    skip = torch.randn(n, 256, 10, 9, device="cuda").to(torch.bfloat16).contiguous(memory_format=CL)
    w = (torch.randn(256, 256, 3, 3, device="cuda") * 0.03).to(torch.bfloat16).contiguous(memory_format=CL)
    bias = torch.randn(256, device="cuda") * 0.1
    return x, skip, w, bias


def _bits_equal(a, b):
    return torch.equal(a.view(torch.int16), b.view(torch.int16))


@pytest.mark.parametrize("with_skip", [False, True])
def test_pixel_tiles_match_consecutive_tiles(data, with_skip):
    from chinesechesszero_b200 import _lib

    x, skip, w, bias = data
    for n in SIZES:
        xs, ss = x[:n], (skip[:n] if with_skip else None)
        new = _lib.conv3x3_c256(xs, w, bias, ss)
        assert _bits_equal(_lib.conv3x3_c256(xs, w, bias, ss, variant=NEW), new), f"n={n}"
        old = _lib.conv3x3_c256(xs, w, bias, ss, variant=OLD)
        assert _bits_equal(new, old), f"n={n}"
    # a board's output does not depend on its block or CTA row: board 0 alone equals board 0 of the full batch
    assert _bits_equal(_lib.conv3x3_c256(x[:1], w, bias, skip[:1] if with_skip else None), new[:1])


def test_pixel_tiles_in_place_skip(data):
    """The block as net.py runs it: the skip is the output buffer (read and written by the same tile)."""
    from chinesechesszero_b200 import _lib

    x, skip, w, bias = data
    ref = _lib.conv3x3_c256(x[:3760], w, bias, skip[:3760], variant=OLD)
    buf = skip[:3760].clone(memory_format=CL)
    _lib.conv3x3_c256(x[:3760], w, bias, buf, out=buf)
    assert _bits_equal(buf, ref)


@pytest.mark.parametrize("with_skip", [False, True])
def test_pixel_tiles_device_count(data, with_skip):
    """ccz_conv3x3_c256_count with the count below the capacity: the first `count` boards as the host-count launch."""
    from chinesechesszero_b200 import _lib

    x, skip, w, bias = data
    ss = skip if with_skip else None
    for u in (1, 129, 256, 300, 3760):
        count = torch.tensor([u], dtype=torch.int32, device="cuda")
        new = _lib.conv3x3_c256(x, w, bias, ss, count=count)
        old = _lib.conv3x3_c256(x[:u], w, bias, ss[:u] if with_skip else None, variant=OLD)
        assert _bits_equal(new[:u], old), f"u={u}"


@pytest.mark.parametrize("with_skip", [False, True])
def test_pixel_tiles_e4m3(data, with_skip):
    from chinesechesszero_b200 import _lib

    x, skip, w, bias = data
    xq = (x.float() * 4).to(_lib.E4M3).contiguous(memory_format=CL)
    wq = (w.float() * 64).to(_lib.E4M3).contiguous(memory_format=CL)
    deq = torch.full((256,), 1 / 256, device="cuda") * (1 + torch.rand(256, device="cuda"))
    inv = torch.tensor([2.0], device="cuda")

    def run(n, variant, count=None):
        sk = skip[:n] if with_skip else None
        return _lib.conv3x3_c256_e4m3(xq[:n], wq, deq, bias, skip=sk, inv_s_out=inv, count=count, variant=variant)

    for n in SIZES:
        (y0, q0), (y1, q1) = run(n, NEW), run(n, OLD)
        assert _bits_equal(y0, y1) and torch.equal(q0.view(torch.uint8), q1.view(torch.uint8)), f"n={n}"
    for u in (129, 3760):
        count = torch.tensor([u], dtype=torch.int32, device="cuda")
        (y0, q0), (y1, q1) = run(max(SIZES), NEW, count), run(u, OLD)
        assert _bits_equal(y0[:u], y1) and torch.equal(q0[:u].view(torch.uint8), q1.view(torch.uint8)), f"u={u}"
    # yq alone (no bf16 output)
    sk = skip[:300] if with_skip else None
    _, q_only = _lib.conv3x3_c256_e4m3(xq[:300], wq, deq, bias, skip=sk, inv_s_out=inv, y=False, variant=NEW)
    _, q_old = _lib.conv3x3_c256_e4m3(xq[:300], wq, deq, bias, skip=sk, inv_s_out=inv, y=False, variant=OLD)
    assert torch.equal(q_only.view(torch.uint8), q_old.view(torch.uint8))
