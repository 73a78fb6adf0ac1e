"""Every stage of the bf16 and fp8 forward, wired as ``BatchedEvaluator._forward`` wires it, against fp64 references with
a-priori per-element error bounds.

The library entry points the evaluator calls (K10 ``stem_lookup[_e4m3]``, K9 ``conv3x3_c256[_e4m3]``, K11 ``heads_pack``,
K12 ``leaf_unique``) are wrapped while the real forward runs: inputs are cloned before each call (conv2 overwrites its
skip), outputs after it.  Each stage is then checked on the exact operands the evaluator gave it (teacher forcing), so
rounding does not compound over the 80 tower layers and every bound can be tight.

Parameters are teacher-forced too: every weight and bias a call received is first checked element by element against the
net's fp32 parameters folded in fp64 by this file (so folding, storage rounding and which layer's parameters reach which
call are all checked), and the contraction reference then uses those verified operands.  That keeps the e4m3 weight
rounding (2^-4) out of the conv bounds, which is what lets a dropped k-block be caught.

Per-element bound (``elementwise_bound``): ``|got - ref| <= sum(u_r)*(|W|.|x| + |b|) + gamma*|W|.|x| + u_out*(|ref| + ...)``,
``|W|.|x|`` being the same contraction over absolute values.  After a ReLU the pre-activation bound is used.
"""
import inspect
import json

import numpy as np
import pytest
import torch
import torch.nn.functional as F

U_BF16 = 2.0 ** -8   # unit roundoff of bf16 (8-bit significand)
U_E4M3 = 2.0 ** -4   # unit roundoff of e4m3 (4-bit significand)
U_FP32 = 2.0 ** -24
E4M3_SUB = 2.0 ** -10  # half the spacing of e4m3 subnormals (2^-9), in units of the scale
U_FOLD = 2.0 ** -21  # _fold's fp32 arithmetic (sqrt, divide, multiply, add) against the fp64 fold
U_EPI = 2.0 ** -22   # fp32 epilogue: scale, + bias, + skip (three roundings of magnitudes <= |W|.|x| + |b| + |skip|)
K_CONV = 9 * 256


def gamma_f16(k: int) -> float:
    """Accumulation term of a bf16 contraction over ``k`` products with fp32 accumulation (kind::f16, cuBLAS): the fp32
    worst case, whatever the summation order."""
    return k * U_FP32


# Accumulation term of e4m3 K9 (tcgen05.mma kind::f8f6f4), whose accumulator precision is not documented.  Measured by
# test_e4m3_accumulation_error_is_within_gamma on a B200 (1000 W limit): max |err| / (|W|.|x|) = 2.41e-7 = 2^-21.98 over
# 2 x 32 x 256 outputs of K = 2304 contractions.  That is the measurement's resolution (the bf16 rounding of its 2^-14
# offset), so the accumulator itself is at least that good -- no sign of the reduced-precision accumulation of Hopper's FP8
# MMA.  gamma is 4x the figure, far below the 2^-10 cap (dropping one 128-channel k-block moves an output by about 2^-7 of
# |W|.|x|); the fp32 epilogue term U_EPI also covers near-cancelling sums.
MEASURED_E4M3_ACC = 2.412e-7
GAMMA_E4M3 = min(4 * MEASURED_E4M3_ACC, 2.0 ** -10)


def elementwise_bound(ref, wx_abs, u_in=(), b_abs=0.0, u_out=0.0, gamma=0.0):
    """Per-element bound of ``|got - ref|`` for ``got`` = a contraction with operand roundings ``u_in`` (unit roundoffs),
    accumulation term ``gamma`` and an output rounding ``u_out``; ``wx_abs`` = |W|.|x|, ``b_abs`` = |b| (+|skip|).
    Works on numpy arrays and torch tensors."""
    pre = sum(u_in) * (wx_abs + b_abs) + gamma * wx_abs
    return pre + u_out * (abs(ref) + pre)


def worst_ratio(got, ref, bound) -> float:
    """max |got - ref| / bound (elements with a zero bound must be exact; NaN propagates)."""
    err = (got.double() - ref).abs()
    r = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, torch.inf, 0.0).to(err))
    return float(r.max()) if r.numel() else 0.0


def conv3x3_f64(x, w):
    """fp64 conv3x3 pad 1 of ``x`` (n,C,10,9) (any layout) with ``w`` (Co,C,3,3), as nine fp64 GEMMs over NHWC rows."""
    n, c = x.shape[:2]
    xp = F.pad(x.double().permute(0, 2, 3, 1), (0, 0, 1, 1, 1, 1))
    w = w.double()
    out = torch.zeros((n * 90, w.shape[0]), dtype=torch.float64, device=x.device)
    for ky in range(3):
        for kx in range(3):
            out.addmm_(xp[:, ky:ky + 10, kx:kx + 9].reshape(n * 90, c), w[:, :, ky, kx].t())
    return out.view(n, 10, 9, -1).permute(0, 3, 1, 2)


@torch.no_grad()
def fold_f64(conv, bn):
    """(W, B, |B| magnitude) of eval-mode BatchNorm folded into ``conv`` in fp64; the magnitude bounds the fp32 fold's
    bias error through cancellation: |b - mean|*|scale| + |beta|."""
    scale = bn.weight.double() / torch.sqrt(bn.running_var.double() + bn.eps)
    w = conv.weight.double() * scale.view(-1, *([1] * (conv.weight.dim() - 1)))
    bm = conv.bias.double() - bn.running_mean.double()
    return w, bm * scale + bn.bias.double(), (bm * scale).abs() + bn.bias.double().abs()


# ---- the bound helper on the host ----------------------------------------------------------------------------------

def _bf16(a: np.ndarray) -> np.ndarray:
    return torch.from_numpy(a.astype(np.float32)).to(torch.bfloat16).double().numpy()


@pytest.mark.parametrize("k", [16, 256, 2304])
def test_elementwise_bound_holds_for_bf16_dot_products_with_fp32_accumulation(k):
    """bf16 weights (rounded from fp64), bf16 activations, fp32 products accumulated in order in fp32, a bf16 output: never
    outside the bound -- including sums that cancel; and a dropped 64-product block is caught when the weights are exact."""
    rng = np.random.default_rng(k)
    rows = 4000
    x = _bf16(np.maximum(rng.standard_normal((rows, k)), 0) * 3.0)
    w64 = rng.standard_normal((rows, k)) * 0.05
    w64[: rows // 2] -= (w64[: rows // 2] * x[: rows // 2]).sum(1, keepdims=True) / x[: rows // 2].sum(1, keepdims=True)  # ~0 sums
    wb = _bf16(w64)
    b = rng.standard_normal(rows) * 0.1
    prod = (x * wb).astype(np.float32)  # exact: 8x8-bit significands fit fp32
    acc = np.add.accumulate(np.concatenate([b.astype(np.float32)[:, None], prod], 1), axis=1, dtype=np.float32)[:, -1]
    got = _bf16(acc)
    ref = (x * w64).sum(1) + b
    wx = (np.abs(x) * np.abs(w64)).sum(1)
    bound = elementwise_bound(ref, wx, u_in=(U_BF16, U_FP32), b_abs=np.abs(b), u_out=U_BF16, gamma=gamma_f16(k + 1))
    assert np.all(np.abs(got - ref) <= bound)
    assert np.abs(got - ref).max() > 0.01 * bound.max()  # the bound is not vacuous by orders of magnitude
    if k >= 256:  # exact operands: only accumulation + output rounding; a missing 64-product block exceeds it
        ref_exact = (x * wb).sum(1) + b
        bound = elementwise_bound(ref_exact, (np.abs(x) * np.abs(wb)).sum(1), u_in=(U_FP32,), b_abs=np.abs(b), u_out=U_BF16,
                                  gamma=gamma_f16(k + 1))
        assert np.all(np.abs(got - ref_exact) <= bound)
        dropped = ref_exact - (x[:, :64] * wb[:, :64]).sum(1)
        assert np.any(np.abs(got - dropped) > bound)


# ---- recording the real forward --------------------------------------------------------------------------------------

WRAPPED = ("stem_lookup", "stem_lookup_e4m3", "conv3x3_c256", "conv3x3_c256_e4m3", "heads_pack", "leaf_unique")
OUTPUT_ARGS = ("out", "out_q", "operands", "rows", "uniq", "n_unique")


def _clone(v):
    if isinstance(v, torch.Tensor):
        return v.clone()
    if isinstance(v, tuple):
        return tuple(_clone(t) for t in v)
    return v


class Recorder:
    """Wraps the library entry points net.py calls.  While ``calibrating`` (the evaluator's ``refresh``) only the output
    amax of each call is kept; afterwards every call's inputs (cloned before), outputs (cloned after) and pointers."""

    def __init__(self, lib, mp):
        self.calls, self.calib_amax, self.calibrating = [], [], True
        for name in WRAPPED:
            mp.setattr(lib, name, self._wrap(name, getattr(lib, name)))

    def _wrap(self, name, fn):
        sig = inspect.signature(fn)

        def wrapper(*args, **kw):
            if self.calibrating:
                res = fn(*args, **kw)
                self.calib_amax.append((name, res.amax().float().clone()))
                return res
            a = sig.bind(*args, **kw)
            a.apply_defaults()
            inputs = {k: _clone(v) for k, v in a.arguments.items()}
            ptrs = {k: v.data_ptr() for k, v in a.arguments.items() if isinstance(v, torch.Tensor)}
            res = fn(*args, **kw)
            outs = {k: a.arguments[k].clone() for k in OUTPUT_ARGS if isinstance(a.arguments.get(k), torch.Tensor)}
            self.calls.append({"name": name, "in": inputs, "out": outs, "res": _clone(res), "ptr": ptrs})
            return res

        return wrapper


@pytest.fixture(scope="module")
def net():
    from chinesechesszero_b200.net import Net
    from oracle import net_oracle

    torch.manual_seed(11)
    net = Net().eval()
    net_oracle.perturb_(net.state_dict(), seed=3)  # non-trivial BatchNorm: folding matters
    return net.cuda()


@pytest.fixture(scope="module")
def boards():
    """256 distinct positions spread to 384 rows with a seeded duplicate pattern."""
    from chinesechesszero_b200.net import calibration_boards

    cand = calibration_boards(384, seed=5).cpu().numpy()
    seen, keep = set(), []
    for i, r in enumerate(cand):
        if bytes(r[:91]) not in seen:
            seen.add(bytes(r[:91]))
            keep.append(i)
    distinct = cand[keep[:256]]
    assert len(distinct) == 256
    rng = np.random.default_rng(17)
    pick = np.concatenate([np.arange(256), rng.integers(0, 256, size=128)])
    pick = pick[rng.permutation(len(pick))]
    return torch.from_numpy(np.ascontiguousarray(distinct[pick])).cuda()


@pytest.fixture(scope="module")
def calib():
    from chinesechesszero_b200.net import calibration_boards

    return calibration_boards(1024, seed=0)


@pytest.fixture(scope="module")
def folds(net):
    blocks = [(fold_f64(rb.conv1, rb.conv1_bn), fold_f64(rb.conv2, rb.conv2_bn)) for rb in net.res_blocks]
    return {"stem": fold_f64(net.conv_block, net.conv_block_bn), "blocks": blocks,
            "policy": fold_f64(net.policy_conv, net.policy_bn), "value": fold_f64(net.value_conv, net.value_bn)}


_RUNS: dict = {}


@pytest.fixture(scope="module")
def forward_run(net, boards, calib):
    """forward_run(precision, dedup) -> (evaluator, recorder, logits, values), one recorded forward each, cached."""
    from chinesechesszero_b200 import _lib
    from chinesechesszero_b200.net import BatchedEvaluator

    def run(precision, dedup):
        key = (precision, dedup)
        if key not in _RUNS:
            with pytest.MonkeyPatch.context() as mp:
                rec = Recorder(_lib, mp)
                ev = BatchedEvaluator(net, dedup=dedup, precision=precision, calib_boards=calib)
                rec.calibrating = False
                logits, v = ev.forward(None, boards)
                torch.cuda.synchronize()
            _RUNS[key] = (ev, rec, logits, v)
        return _RUNS[key]

    yield run
    _RUNS.clear()


# ---- stage checks (each returns its worst err/bound; exact checks assert) ----------------------------------------------

def check_params_bf16(w, b32, fold):
    W, B, bmag = fold
    return max(worst_ratio(w, W, (U_BF16 + U_FOLD) * W.abs()), worst_ratio(b32, B, U_FOLD * bmag))


def check_params_e4m3(wq, deq, b32, fold, s_in):
    """The weight the conv effectively applies to x = xq*s_in is wq*deq/s_in: within e4m3 rounding of the fp64 fold."""
    W, B, bmag = fold
    s_w = W.abs().flatten(1).amax(1) / 448.0
    w_eff = wq.double() * (deq.double() / s_in).view(-1, 1, 1, 1)
    bound_w = (U_E4M3 + 4 * U_FOLD) * W.abs() + E4M3_SUB * (1 + 2.0 ** -20) * s_w.view(-1, 1, 1, 1)
    return max(worst_ratio(w_eff, W, bound_w), worst_ratio(deq, s_in * s_w, 2 * U_FOLD * s_in * s_w),
               worst_ratio(b32, B, U_FOLD * bmag))


def conv_reference(x, w, bias, skip=None, deq=None, drop_kblock=None):
    """(pre-activation ref, |W|.|x|, |b| + |skip|) of relu(conv(x, w) [* deq] + bias [+ skip]) in fp64.
    ``drop_kblock`` = number of input channels of the centre tap left out (negative control)."""
    w = w.double()
    if drop_kblock:
        w = w.clone()
        w[:, :drop_kblock, 1, 1] = 0
    acc, wx = conv3x3_f64(x, w), conv3x3_f64(x.double().abs(), w.abs())
    if deq is not None:
        d = deq.double().view(1, -1, 1, 1)
        acc, wx = acc * d, wx * d
    babs = bias.double().abs().view(1, -1, 1, 1).expand_as(acc)
    pre = acc + bias.double().view(1, -1, 1, 1)
    if skip is not None:
        pre, babs = pre + skip.double(), babs + skip.double().abs()
    return pre, wx, babs


def conv_y_ratio(y, pre, wx, babs, gamma):
    ref = torch.relu(pre)
    return worst_ratio(y, ref, elementwise_bound(ref, wx, (U_EPI,), babs, U_BF16, gamma))


def conv_yq_ratio(yq, pre, wx, babs, gamma, inv_s):
    """yq = satfinite(relu(f) * inv_s) in e4m3, f within the pre-activation bound of ref: compared in units of the scale
    against the clamped reference (clamping and ReLU are 1-Lipschitz), with the e4m3 output rounding."""
    e = (U_EPI * (wx + babs) + gamma * wx) * inv_s
    t = (torch.relu(pre) * inv_s).clamp(max=448.0)
    bound = e + U_E4M3 * (t + e) + E4M3_SUB + 2.0 ** -23 * (t + e)
    return worst_ratio(yq.float(), t, bound)


def stem_ratio(boards, y, fold, n):
    from chinesechesszero_b200 import _lib

    W, B, bmag = fold
    planes = _lib.movegen_encode(boards[:n].contiguous())[3].view(n, 119, 10, 9)
    ref = torch.relu(conv3x3_f64(planes, W) + B.view(1, -1, 1, 1))
    wx = conv3x3_f64(planes.double().abs(), W.abs())
    # table weights bf16 (from the fp32 fold), bias_turn fp32 sums; output bf16
    bound = elementwise_bound(ref, wx, (U_BF16, U_FOLD), U_FOLD * bmag.view(1, -1, 1, 1), U_BF16, gamma_f16(119 * 9 + 1))
    return worst_ratio(y[:n], ref, bound)


def pack_reference(h, rows, n_games, kp, width):
    """K11 in torch: relu of the bf16 bits (sign set -> +0), policy channel-major at 0, value at kp, zero padding."""
    hb = h.view(torch.int16).view(-1, 90, 32)[rows.long()]
    hb = torch.where(hb < 0, torch.zeros_like(hb), hb)
    out = torch.zeros((n_games, width), dtype=torch.int16, device=h.device)
    out[:, :17 * 90] = hb[:, :, :17].transpose(1, 2).reshape(n_games, -1)
    out[:, kp:kp + 7 * 90] = hb[:, :, 17:24].transpose(1, 2).reshape(n_games, -1)
    return out


@torch.no_grad()
def heads_ratios(ev, net, folds, x_last, h, operands, rows, n, logits, values):
    """1x1 heads GEMM, K11 (exact), policy FC, value FC1 -> ReLU -> FC2 -> tanh.  Returns a dict of worst ratios."""
    r = {}
    hw, hb = ev._heads_gemm
    (Wp, Bp, bmp), (Wv, Bv, bmv) = folds["policy"], folds["value"]
    W = torch.cat([Wp, Wv]).view(24, 256)
    B, bmag = torch.cat([Bp, Bv]), torch.cat([bmp, bmv])
    assert not hw[24:].view(torch.int16).any() and not hb[24:].view(torch.int16).any()
    r["heads_params"] = max(worst_ratio(hw[:24], W, (U_BF16 + U_FOLD) * W.abs()),
                            worst_ratio(hb[:24], B, U_BF16 * B.abs() + 2 * U_FOLD * bmag))  # heads.b is stored in bf16
    X = x_last.permute(0, 2, 3, 1).reshape(-1, 256)[:n * 90].double()
    ref = X @ hw[:24].double().t() + hb[:24].double()
    wx = X.abs() @ hw[:24].double().abs().t()
    bound = elementwise_bound(ref, wx, (U_EPI,), hb[:24].double().abs(), U_BF16, gamma_f16(256))
    r["heads_gemm"] = worst_ratio(h[:n * 90, :24], ref, bound)
    assert not h[:n * 90, 24:].view(torch.int16).any()  # pad columns 24..31 exactly 0
    g, kp = operands.shape[0], ev._kp
    packed = pack_reference(h, rows, g, kp, operands.shape[1])
    assert torch.equal(operands.view(torch.int16), packed)
    assert not operands[:, 17 * 90:kp].view(torch.int16).any() and not operands[:, kp + 7 * 90:].view(torch.int16).any()
    op = packed.view(torch.bfloat16).double()
    # policy FC: bf16 GEMM output, then + the fp32 bias
    wp, bp = ev._fc_pad[0], ev.policy_fc[1]
    Wfc = net.policy_fc.weight.double()
    assert not wp[2086:].view(torch.int16).any() and not wp[:, 1530:].view(torch.int16).any()
    assert torch.equal(bp, net.policy_fc.bias.float())
    pr = worst_ratio(wp[:2086, :1530], Wfc, U_BF16 * Wfc.abs())
    gemm = op[:, :kp] @ wp[:2086].double().t()
    gb = elementwise_bound(gemm, op[:, :kp].abs() @ wp[:2086].double().abs().t(), (), 0.0, U_BF16, gamma_f16(kp))
    ref_l = gemm + bp.double()
    r["policy_fc"] = worst_ratio(logits, ref_l, gb + U_FP32 * (ref_l.abs() + gb))
    # value: FC1 (bf16 weights, bias and output) -> ReLU -> FC2 (fp32) -> tanh
    wv, bv1 = ev._fc_pad[1], ev.value_fc1[1]
    W1 = net.value_fc1.weight.double()
    assert not wv[:, 630:].view(torch.int16).any()
    pr = max(pr, worst_ratio(wv[:, :630], W1, U_BF16 * W1.abs()),
             worst_ratio(bv1, net.value_fc1.bias.double(), U_BF16 * net.value_fc1.bias.double().abs()))
    w2, b2 = ev.value_fc2
    assert torch.equal(w2, net.value_fc2.weight.float()) and torch.equal(b2, net.value_fc2.bias.float())
    opv = op[:, kp:]
    pre1 = opv @ wv.double().t() + bv1.double()
    b1 = elementwise_bound(pre1, opv.abs() @ wv.double().abs().t(), (U_EPI,), bv1.double().abs(), U_BF16, gamma_f16(640))
    v1 = torch.relu(pre1)
    z = v1 @ w2.double().t() + b2.double()
    aw2 = w2.double().abs()
    bz = b1 @ aw2.t() + gamma_f16(257) * ((v1 + b1) @ aw2.t() + b2.double().abs())
    r["value"] = worst_ratio(values, torch.tanh(z).view(-1), (bz + 2.0 ** -21).view(-1))  # tanh' <= 1; fp32 tanh
    r["fc_params"] = pr
    return r


def _conv_calls(rec, name):
    calls = [c for c in rec.calls if c["name"] == name]
    assert len(calls) == 80
    return calls


def _expected_scales(rec):
    """(s_x, s_y) = activation_scale of the amax recorded during refresh(): per chunk the calls are stem, then conv1 and
    conv2 of each block; x_0 is the stem output, x_i the conv2 output of block i-1, y_i the conv1 output of block i."""
    from chinesechesszero_b200.net import activation_scale

    names = [nm for nm, _ in rec.calib_amax]
    per = 81
    assert len(names) % per == 0 and names[0] == "stem_lookup"
    a = torch.stack([v for _, v in rec.calib_amax]).view(-1, per).amax(0)
    amax_x = torch.cat([a[0:1], a[2:per - 1:2]])
    amax_y = a[1:per:2]
    return activation_scale(amax_x), activation_scale(amax_y)


def check_forward(precision, dedup, ev, rec, logits, values, boards, net, folds, s_y_shift=0):
    """All stage checks of one recorded forward.  Returns {stage: worst err/bound}.  ``s_y_shift`` (negative control)
    checks block i with s_y[i + shift]."""
    from chinesechesszero_b200 import _lib

    r = {}
    g = boards.shape[0]
    calls = rec.calls
    if dedup:
        lu = calls[0]
        assert lu["name"] == "leaf_unique"
        U = int(lu["out"]["n_unique"])
        rows, uniq = lu["out"]["rows"], lu["out"]["uniq"]
        assert U == len({bytes(b[:91]) for b in boards.cpu().numpy()}) == 256
        assert int(rows.max()) < U and torch.equal(uniq[rows.long(), :91], boards[:, :91])
        first = [int(np.argmax(rows.cpu().numpy() == u)) for u in range(U)]
        assert first == sorted(first)  # rows numbered in order of first occurrence
        stem_boards = uniq
        counts = [c["in"].get("count") for c in calls[1:]]
        assert all(int(c) == U for c in counts if c is not None)
        assert sum(c is None for c in counts) == 1  # every call but heads_pack takes the device count
    else:
        U, rows, stem_boards = g, torch.arange(g, dtype=torch.int32, device=boards.device), boards
        assert all(c["in"].get("count") is None for c in calls) and calls[0]["name"].startswith("stem")
    fp8 = precision == "fp8"
    stem = [c for c in calls if c["name"].startswith("stem")]
    assert len(stem) == 1 and stem[0]["name"] == ("stem_lookup_e4m3" if fp8 else "stem_lookup")
    stem = stem[0]
    assert torch.equal(stem["in"]["boards"][:U], stem_boards[:U])
    y_stem = stem["res"][0] if fp8 else stem["res"]
    r["stem"] = stem_ratio(stem_boards, y_stem, folds["stem"], U)
    if fp8:
        from chinesechesszero_b200.net import e4m3_quantize

        s_x, s_y = _expected_scales(rec)
        assert torch.equal(ev.fp8_scales["x"], s_x) and torch.equal(ev.fp8_scales["y"], s_y)
        inv_sx, inv_sy = 1.0 / s_x, 1.0 / s_y
        assert torch.equal(stem["in"]["inv_s_out"], inv_sx[0:1])
        assert torch.equal(stem["res"][1][:U].view(torch.uint8), e4m3_quantize(y_stem[:U], inv_sx[0:1]).view(torch.uint8))
        convs = _conv_calls(rec, "conv3x3_c256_e4m3")
    else:
        convs = _conv_calls(rec, "conv3x3_c256")
    x_prev = y_stem  # bf16 x entering the block
    xq_prev = stem["res"][1] if fp8 else None
    worst = {}

    def put(k, v):
        worst[k] = max(worst.get(k, 0.0), v)

    for i in range(40):
        c1, c2 = convs[2 * i], convs[2 * i + 1]
        f1, f2 = folds["blocks"][i]
        a1, a2 = c1["in"], c2["in"]
        assert a1["skip"] is None and a2["skip"] is not None
        assert c2["ptr"]["skip"] == c2["ptr"]["out"]  # the block output overwrites its input
        assert torch.equal(a2["skip"][:U].view(torch.int16), x_prev[:U].view(torch.int16))  # skip = x entering block i
        if fp8:
            j = min(i + s_y_shift, 39)
            assert torch.equal(a1["xq"][:U].view(torch.uint8), xq_prev[:U].view(torch.uint8))
            assert a1["y"] is False and c1["res"][0] is None
            assert torch.equal(a1["inv_s_out"], inv_sy[j:j + 1])
            yq1 = c1["res"][1]
            assert torch.equal(a2["xq"][:U].view(torch.uint8), yq1[:U].view(torch.uint8))
            put("params", check_params_e4m3(a1["wq"], a1["dequant"], a1["bias"], f1, s_x[i]))
            put("params", check_params_e4m3(a2["wq"], a2["dequant"], a2["bias"], f2, s_y[j]))
            pre, wx, babs = conv_reference(a1["xq"][:U], a1["wq"], a1["bias"], deq=a1["dequant"])
            put("conv1_yq", conv_yq_ratio(yq1[:U], pre, wx, babs, GAMMA_E4M3, float(inv_sy[j])))
            pre, wx, babs = conv_reference(a2["xq"][:U], a2["wq"], a2["bias"], a2["skip"][:U], deq=a2["dequant"])
            y2, yq2 = c2["res"]
            put("conv2_y", conv_y_ratio(y2[:U], pre, wx, babs, GAMMA_E4M3))
            if i == 39:
                assert a2["out_q"] is None and a2["inv_s_out"] is None and yq2 is None  # the last block writes no xq
            else:
                assert c2["ptr"]["out_q"] == c1["ptr"]["xq"]  # xq_{l+1} written over xq_l
                assert torch.equal(a2["inv_s_out"], inv_sx[i + 1:i + 2])
                put("conv2_yq", conv_yq_ratio(yq2[:U], pre, wx, babs, GAMMA_E4M3, float(inv_sx[i + 1])))
                xq_prev = yq2
            x_prev = y2
        else:
            assert torch.equal(a1["x"][:U].view(torch.int16), x_prev[:U].view(torch.int16))
            y1 = c1["res"]
            assert torch.equal(a2["x"][:U].view(torch.int16), y1[:U].view(torch.int16))
            put("params", check_params_bf16(a1["w"], a1["bias"], f1))
            put("params", check_params_bf16(a2["w"], a2["bias"], f2))
            pre, wx, babs = conv_reference(a1["x"][:U], a1["w"], a1["bias"])
            put("conv1_y", conv_y_ratio(y1[:U], pre, wx, babs, gamma_f16(K_CONV)))
            pre, wx, babs = conv_reference(a2["x"][:U], a2["w"], a2["bias"], a2["skip"][:U])
            x_prev = c2["res"]
            put("conv2_y", conv_y_ratio(x_prev[:U], pre, wx, babs, gamma_f16(K_CONV)))
    r.update(worst)
    hp = [c for c in calls if c["name"] == "heads_pack"]
    assert len(hp) == 1
    hp = hp[0]
    if dedup:
        assert torch.equal(hp["in"]["rows"], rows)
    else:
        assert hp["in"]["rows"] is None
    r.update(heads_ratios(ev, net, folds, x_prev, hp["in"]["h"], hp["out"]["operands"], rows, U, logits, values))
    return r


_REPORT: dict = {}


@pytest.mark.gpu
@pytest.mark.parametrize("dedup", [True, False])
@pytest.mark.parametrize("precision", ["bf16", "fp8"])
def test_forward_stages_within_elementwise_bounds(forward_run, boards, net, folds, precision, dedup):
    ev, rec, logits, values = forward_run(precision, dedup)
    r = check_forward(precision, dedup, ev, rec, logits, values, boards, net, folds)
    rep = _REPORT.setdefault(precision, {})
    for k, v in r.items():
        rep[k] = max(rep.get(k, 0.0), v)
    assert all(v <= 1.0 for v in r.values()), r


@pytest.mark.gpu
def test_forward_stages_report():
    """One FORWARD_STAGES line: the worst err/bound per stage and precision over the dedup on / off forwards."""
    if len(_REPORT) < 2:
        pytest.skip("needs the forward-stage checks of both precisions in this session")
    print("FORWARD_STAGES " + json.dumps({p: {k: round(v, 4) for k, v in s.items()} for p, s in sorted(_REPORT.items())}))
    assert all(v <= 1.0 for s in _REPORT.values() for v in s.values())


# ---- negative controls: the checks fire on a wrong operand, wiring or scale --------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp8"])
def test_negative_controls_fire(forward_run, boards, net, folds, precision):
    ev, rec, logits, values = forward_run(precision, True)
    fp8 = precision == "fp8"
    U = int(rec.calls[0]["out"]["n_unique"])
    convs = _conv_calls(rec, "conv3x3_c256_e4m3" if fp8 else "conv3x3_c256")
    c2 = convs[2 * 7 + 1]
    a2 = c2["in"]
    y2 = c2["res"][0] if fp8 else c2["res"]
    x_in = a2["xq"] if fp8 else a2["x"]
    w_in = a2["wq"] if fp8 else a2["w"]
    deq = a2["dequant"] if fp8 else None
    gamma = GAMMA_E4M3 if fp8 else gamma_f16(K_CONV)
    pre, wx, babs = conv_reference(x_in[:U], w_in, a2["bias"], a2["skip"][:U], deq=deq)
    assert conv_y_ratio(y2[:U], pre, wx, babs, gamma) <= 1.0
    # two adjacent output channels swapped
    sw = y2[:U].clone()
    sw[:, [40, 41]] = sw[:, [41, 40]]
    assert conv_y_ratio(sw, pre, wx, babs, gamma) > 1.0
    # one input k-block missing from the reference: 64 channels (bf16 BK) or 128 (e4m3 BK) of the centre tap
    p, w_, b_ = conv_reference(x_in[:U], w_in, a2["bias"], a2["skip"][:U], deq=deq, drop_kblock=128 if fp8 else 64)
    assert conv_y_ratio(y2[:U], p, w_, b_, gamma) > 1.0
    # the skip omitted
    p, w_, b_ = conv_reference(x_in[:U], w_in, a2["bias"], None, deq=deq)
    assert conv_y_ratio(y2[:U], p, w_, b_, gamma) > 1.0
    if fp8:  # block i checked with s_y[i+1]
        with pytest.raises(AssertionError):
            check_forward(precision, True, ev, rec, logits, values, boards, net, folds, s_y_shift=1)
        s_x, s_y = _expected_scales(rec)
        assert check_params_e4m3(a2["wq"], a2["dequant"], a2["bias"], folds["blocks"][7][1], s_y[8]) > 1.0
        c1 = convs[2 * 7]
        p, w_, b_ = conv_reference(c1["in"]["xq"][:U], c1["in"]["wq"], c1["in"]["bias"], deq=c1["in"]["dequant"])
        assert conv_yq_ratio(c1["res"][1][:U], p, w_, b_, gamma, float(1.0 / s_y[8])) > 1.0
    # the packed operand shifted by one pixel, and the row map off by one
    hp = [c for c in rec.calls if c["name"] == "heads_pack"][0]
    h, ops, rows = hp["in"]["h"], hp["out"]["operands"], hp["in"]["rows"]
    ref = pack_reference(h, rows, ops.shape[0], ev._kp, ops.shape[1])
    assert torch.equal(ops.view(torch.int16), ref)
    shifted = torch.roll(ops.view(torch.int16)[:, :17 * 90], 1, dims=1)
    assert not torch.equal(shifted, ref[:, :17 * 90])
    assert not torch.equal(ops.view(torch.int16), pack_reference(h, (rows + 1) % U, ops.shape[0], ev._kp, ops.shape[1]))
    x_last = convs[-1]["res"][0] if fp8 else convs[-1]["res"]
    r = heads_ratios(ev, net, folds, x_last, h, ops, rows, U, logits, values)
    assert max(r.values()) <= 1.0
    with pytest.raises(AssertionError):  # the heads checked on the row map off by one
        heads_ratios(ev, net, folds, x_last, h, ops, (rows + 1) % U, U, logits, values)


# ---- the e4m3 accumulation term --------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_e4m3_accumulation_error_is_within_gamma():
    """Measures the accumulation error of e4m3 K9 directly: one board per launch whose activations are constant over the
    board, so every interior pixel has the same exact sum per output channel, and a per-channel bias that cancels it
    (leaving a positive offset of 2^-14 |W|.|x|).  The bf16 output then resolves the accumulator's error at about 2^-22 of
    |W|.|x|.  The same boards with the weights negated give the errors of the opposite sign; an output clipped to 0 by the
    ReLU (an error below -2^-14 |W|.|x|) fails the test."""
    from chinesechesszero_b200 import _lib
    from chinesechesszero_b200.net import e4m3_quantize, weight_scales

    gen = torch.Generator(device="cpu").manual_seed(23)
    w = (torch.randn((256, 256, 3, 3), generator=gen) * 0.03).cuda()
    s_w = weight_scales(w)
    worst = 0.0
    for sign in (1.0, -1.0):
        wq = e4m3_quantize(sign * w, (1.0 / s_w).view(-1, 1, 1, 1)).contiguous(memory_format=torch.channels_last)
        deq = torch.full((256,), 2.0 ** -6, device="cuda")  # a power of two: acc * deq is exact
        wsum, wabs = wq.double().sum((2, 3)), wq.double().abs().sum((2, 3))
        for b in range(32):
            xc = torch.relu(torch.randn((256,), generator=gen)).cuda() * 3.0
            xq1 = e4m3_quantize(xc, 1.0)
            xq = xq1.view(1, 256, 1, 1).expand(1, 256, 10, 9).contiguous(memory_format=torch.channels_last)
            exact = (wsum @ xq1.double()) * 2.0 ** -6
            wx = (wabs @ xq1.double().abs()) * 2.0 ** -6
            bias = (-exact + 2.0 ** -14 * wx).float()
            y, _ = _lib.conv3x3_c256_e4m3(xq, wq, deq, bias)
            got = y[0, :, 1:9, 1:8].double()  # interior pixels see all nine taps
            assert bool((got > 0).all())  # nothing clipped by the ReLU
            err = (got - (exact + bias.double()).view(-1, 1, 1)).abs()
            worst = max(worst, float((err / wx.view(-1, 1, 1)).max()))
    print(f"E4M3_ACCUMULATION max|err|/(|W|.|x|) = {worst:.3e} = 2^{np.log2(max(worst, 1e-300)):.2f}")
    assert GAMMA_E4M3 <= 2.0 ** -10
    assert worst <= GAMMA_E4M3
