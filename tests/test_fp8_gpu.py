"""The FP8 evaluator on the device: e4m3 K9 (csrc/ccz_conv.cuh, T = __nv_fp8_e4m3) and K10's e4m3 copy against torch
references, row independence and dedup bit-identity, accuracy against the fp32 reference Net, and in-place refresh."""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

E4M3 = torch.float8_e4m3fn
CL = torch.channels_last


def _q(x, inv):
    from chinesechesszero_b200.net import e4m3_quantize

    return e4m3_quantize(x, inv)


@pytest.fixture(scope="module")
def operands():
    """e4m3 activations of 300 random boards, an e4m3 weight with per-channel scales, dequant, bias and a bf16 skip."""
    from chinesechesszero_b200.net import weight_scales

    g = torch.Generator(device="cpu").manual_seed(0)
    x = torch.relu(torch.randn((300, 256, 10, 9), generator=g)).cuda().contiguous(memory_format=CL)
    s_x = float(x.amax()) / 448
    xq = _q(x, torch.tensor([1 / s_x], device="cuda"))
    w = (torch.randn((256, 256, 3, 3), generator=g) * torch.linspace(0.2, 2.0, 256).view(-1, 1, 1, 1) * 0.02).cuda()
    s_w = weight_scales(w)
    wq = _q(w, (1 / s_w).view(-1, 1, 1, 1)).contiguous(memory_format=CL)
    deq = (s_x * s_w).float().contiguous()
    bias = (torch.randn(256, generator=g) * 0.3).cuda()
    skip = (torch.randn((300, 256, 10, 9), generator=g) * 0.5).cuda().to(torch.bfloat16).contiguous(memory_format=CL)
    return xq, wq, deq, bias, skip


def _ref(xq, wq, deq, bias, skip):
    """fp64 conv of the dequantised operands: relu(conv(xq, wq) * deq + bias (+ skip))."""
    acc = F.conv2d(xq.double(), wq.double(), padding=1)
    f = acc * deq.double().view(1, -1, 1, 1) + bias.double().view(1, -1, 1, 1)
    if skip is not None:
        f = f + skip.double()
    return torch.relu(f)


@pytest.mark.parametrize("with_skip", [False, True])
@pytest.mark.parametrize("n", [1, 3, 37, 128, 300])
def test_e4m3_k9_matches_dequantized_reference(operands, n, with_skip):
    from chinesechesszero_b200 import _lib

    xq, wq, deq, bias, skip = operands
    xq = xq[:n].contiguous(memory_format=CL)
    sk = skip[:n].contiguous(memory_format=CL) if with_skip else None
    ref = _ref(xq, wq, deq, bias, sk)
    inv = torch.tensor([400.0 / float(ref.max())], device="cuda")
    y, yq = _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, skip=sk, inv_s_out=inv)
    tol = 2.0 ** -8 * float(ref.abs().max()) + 1e-4
    assert float((y.double() - ref).abs().max()) <= tol
    # e4m3 output: at most one code (one ulp) from satfinite(ref * inv); codes of non-negative values are monotone
    rq = _q(ref.float(), inv)
    d = (yq.view(torch.uint8).int() - rq.view(torch.uint8).int()).abs()
    assert int(d.max()) <= 1
    assert float((d > 0).float().mean()) < 0.01
    # each output alone equals the same output of the two-output launch
    y_only, none = _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, skip=sk)
    none2, yq_only = _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, skip=sk, inv_s_out=inv, y=False)
    assert none is None and none2 is None
    assert torch.equal(y_only.view(torch.int16), y.view(torch.int16)) and torch.equal(yq_only.view(torch.uint8), yq.view(torch.uint8))


def test_e4m3_k9_in_place_skip_saturation_and_determinism(operands):
    from chinesechesszero_b200 import _lib

    xq, wq, deq, bias, skip = operands
    y, yq = _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, skip=skip, inv_s_out=torch.tensor([1.0], device="cuda"))
    y2, yq2 = _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, skip=skip, inv_s_out=torch.tensor([1.0], device="cuda"))
    assert torch.equal(y.view(torch.int16), y2.view(torch.int16)) and torch.equal(yq.view(torch.uint8), yq2.view(torch.uint8))
    inplace = skip.clone()
    out, _ = _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, skip=inplace, out=inplace)
    assert out.data_ptr() == inplace.data_ptr() and torch.equal(inplace.view(torch.int16), y.view(torch.int16))
    big = torch.tensor([1e6], device="cuda")  # everything above 448e-6 saturates to 448, nothing becomes NaN
    _, ys = _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, skip=skip, inv_s_out=big)
    v, sat = ys.float(), y.float() > 1e-3
    assert not torch.isnan(v).any() and bool(sat.any()) and torch.equal(v[sat], torch.full_like(v[sat], 448.0))
    assert torch.equal(v[y.float() == 0], torch.zeros_like(v[y.float() == 0]))


def test_e4m3_k9_rejects_bad_arguments(operands):
    from chinesechesszero_b200 import _lib

    xq, wq, deq, bias, skip = operands
    inv = torch.tensor([1.0], device="cuda")
    with pytest.raises(_lib.CczError, match="no output"):
        _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, y=False)
    with pytest.raises(_lib.CczError, match="alias"):
        _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, inv_s_out=inv, out_q=xq)
    with pytest.raises(_lib.CczError, match="xq"):
        _lib.conv3x3_c256_e4m3(xq.float().to(torch.bfloat16).contiguous(memory_format=CL), wq, deq, bias)
    with pytest.raises(_lib.CczError, match="wq"):
        _lib.conv3x3_c256_e4m3(xq, wq.contiguous(), deq, bias)
    with pytest.raises(_lib.CczError, match="dequant"):
        _lib.conv3x3_c256_e4m3(xq, wq, deq.double(), bias)
    with pytest.raises(_lib.CczError, match="inv_s_out"):
        _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, inv_s_out=torch.tensor([1.0, 2.0], device="cuda"))
    with pytest.raises(_lib.CczError, match="out_q needs"):
        _lib.conv3x3_c256_e4m3(xq, wq, deq, bias, out_q=torch.empty_like(xq))
    # the C ABI checks on its own
    lib = _lib.load()
    s = _lib.stream_ptr()
    assert lib.ccz_conv3x3_c256_e4m3(None, wq.data_ptr(), deq.data_ptr(), bias.data_ptr(), None, None, xq.data_ptr() + 0, None, 4, None, s) != 0
    assert lib.ccz_conv3x3_c256_e4m3(xq.data_ptr() + 1, wq.data_ptr(), deq.data_ptr(), bias.data_ptr(), None, skip.data_ptr(), None, None, 4,
                                     None, s) != 0
    assert lib.ccz_conv3x3_c256_e4m3(xq.data_ptr(), wq.data_ptr(), deq.data_ptr(), bias.data_ptr(), None, skip.data_ptr(), skip.data_ptr(),
                                     inv.data_ptr(), 4, None, s) != 0


@pytest.fixture(scope="module")
def boards():
    from chinesechesszero_b200 import positions

    return positions.bench_positions(8192 + 4096, seed=3)


@pytest.fixture(scope="module")
def fp8_pair():
    """A 2-block 256-channel net (perturbed BatchNorm) with its fp8 evaluator calibrated on the default set."""
    from chinesechesszero_b200.net import BatchedEvaluator, Net
    from oracle import net_oracle

    torch.manual_seed(0)
    net = Net(resblocks_num=2).eval()
    net_oracle.perturb_(net.state_dict(), seed=1)
    net = net.cuda()
    return net, BatchedEvaluator(net, precision="fp8")


def test_stem_e4m3_copy_is_the_quantized_bf16_output(fp8_pair, boards):
    from chinesechesszero_b200 import _lib

    _, ev = fp8_pair
    b = boards[:777].contiguous()
    inv = ev._inv_sx[0:1]
    y_ref = _lib.stem_lookup(b, *ev.stem_lookup)
    y, yq = _lib.stem_lookup_e4m3(b, *ev.stem_lookup, inv)
    assert torch.equal(y.view(torch.int16), y_ref.view(torch.int16))
    assert torch.equal(yq.view(torch.uint8), _q(y_ref, inv).view(torch.uint8))
    count = torch.tensor([500], dtype=torch.int32, device="cuda")
    yc = torch.zeros_like(y)
    yqc = torch.zeros_like(yq)
    _lib.stem_lookup_e4m3(b, *ev.stem_lookup, inv, out=yc, out_q=yqc, count=count)
    assert torch.equal(yqc[:500].view(torch.uint8), yq[:500].view(torch.uint8))
    assert not yqc[500:].view(torch.uint8).any()
    with pytest.raises(_lib.CczError):
        _lib.stem_lookup_e4m3(b, *ev.stem_lookup, torch.tensor([1.0], dtype=torch.float64, device="cuda"))


@pytest.mark.parametrize("with_skip", [False, True])
def test_e4m3_k9_is_row_position_invariant(fp8_pair, boards, with_skip):
    """Boards permuted and embedded at other offsets, in batches of 1..300, 3793, 4096 and 8192 boards (tail-split rounds
    of every kind), and the device-count entry point, give every board the bits of the full 8192-board launch."""
    from chinesechesszero_b200 import _lib

    _, ev = fp8_pair
    x, xq = _lib.stem_lookup_e4m3(boards[:8192].contiguous(), *ev.stem_lookup, ev._inv_sx[0:1])
    skip = _lib.stem_lookup(boards[8192:].repeat(2, 1).contiguous(), *ev.stem_lookup) if with_skip else None
    wq, deq, b = ev.qblocks[0][0]
    inv = ev._inv_sy[0:1]
    full_y, full_q = _lib.conv3x3_c256_e4m3(xq, wq, deq, b, skip=skip, inv_s_out=inv)
    gen = torch.Generator(device="cpu").manual_seed(1 + with_skip)
    splits = set()
    for n in list(range(1, 301)) + [3793, 4096, 8192]:
        perm = torch.randperm(8192, generator=gen)[:n].cuda()
        xs = xq[perm].contiguous(memory_format=CL)
        ss = skip[perm].contiguous(memory_format=CL) if with_skip else None
        y, q = _lib.conv3x3_c256_e4m3(xs, wq, deq, b, skip=ss, inv_s_out=inv)
        assert torch.equal(y.view(torch.int16), full_y[perm].view(torch.int16)), f"n={n}"
        assert torch.equal(q.view(torch.uint8), full_q[perm].view(torch.uint8)), f"n={n}"
        splits.add(_lib.conv3x3_plan(n)["split_log2"])
    assert splits == {0, 1, 2}
    count = torch.tensor([3001], dtype=torch.int32, device="cuda")
    y, q = _lib.conv3x3_c256_e4m3(xq, wq, deq, b, skip=skip, inv_s_out=inv, count=count)
    assert torch.equal(y[:3001].view(torch.int16), full_y[:3001].view(torch.int16))
    assert torch.equal(q[:3001].view(torch.uint8), full_q[:3001].view(torch.uint8))


def _live_leaves(net, n_games=512):
    """Leaves of a live search whose games share their opening (many duplicates), as in test_leaf_dedup_gpu."""
    from chinesechesszero_b200 import _lib
    from chinesechesszero_b200.net import BatchedEvaluator
    from chinesechesszero_b200.search import LockstepSearch

    ev = BatchedEvaluator(net, dedup=False)
    s = LockstepSearch(n_games, nodes_per_game=8192)
    s.run(ev, 6)
    acts, _, counts = s.root_visits()
    g = torch.arange(n_games, device="cuda")
    s.advance(acts[g, g % counts.long()])
    s.run(ev, 6)
    _lib.mcts_select(s.arena, s.c_puct, s.leaf_boards, s.leaf_nodes)
    return s.leaf_boards.clone()


def test_fp8_evaluator_dedup_is_bitwise_equal_eager_and_under_graphs(fp8_pair):
    from chinesechesszero_b200.net import BatchedEvaluator

    net, on = fp8_pair
    leaves = _live_leaves(net)
    n_distinct = len({bytes(r[:91]) for r in leaves.cpu().numpy()})
    assert 8 < n_distinct < leaves.shape[0] // 4
    off = BatchedEvaluator(net, dedup=False, precision="fp8", calib_boards=on.calib_boards)
    lo, _, vo = off(None, leaves)
    ln, _, vn = on(None, leaves)
    assert torch.equal(lo, ln) and torch.equal(vo, vn)
    static = leaves.clone()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gl, _, gv = on(None, static)
    perm = torch.randperm(leaves.shape[0], device="cuda")
    static.copy_(leaves[perm])
    graph.replay()
    lo2, _, vo2 = off(None, leaves[perm].contiguous())
    assert torch.equal(gl, lo2) and torch.equal(gv, vo2)


def test_fp8_selfplay_ring_samples_identical_with_and_without_dedup(fp8_pair):
    """Eight resident moves with the bench's stagger (slots 0..23 moves into their games, max_game_moves 24)."""
    from chinesechesszero_b200.net import BatchedEvaluator
    from chinesechesszero_b200.selfplay import SelfPlayEngine

    net, ev_on = fp8_pair
    G, M = 384, 24
    out = []
    for dedup in (True, False):
        ev = BatchedEvaluator(net, dedup=dedup, precision="fp8", calib_boards=ev_on.calib_boards)
        eng = SelfPlayEngine(ev, n_games=G, n_playout=16, seed=4321, max_game_moves=M, resident_ring=8, nodes_per_game=16 * 41 * 8)
        eng._resident_state()["move_count"].copy_(torch.from_numpy(np.arange(G, dtype=np.int64) % M))
        for _ in range(8):
            eng.play_move_resident()
        eng.resident_backlog.append(eng.drain_resident())
        out.append(eng.resident_backlog)
    a, b = out
    assert len(a) == len(b)
    for da, db in zip(a, b):
        for k in da:
            assert np.array_equal(da[k].view(np.uint8), db[k].view(np.uint8)), k


# ---- accuracy against the fp32 reference Net ----------------------------------------------------------------------
# Bounds set from a B200 measurement (DESIGN.md §8, FP8 evaluator) of the sharpened golden nets on 518 positions outside
# the calibration set.  The value bound is relative to the bf16 evaluator's error on the same net: an untrained net's value
# input varies little between positions, so sharpening the value head to +-0.9 multiplies the tower's rounding error by a
# large gain, and both evaluators' absolute value errors scale with it (bf16 itself is off by up to 0.16 on seed0).  The
# policy bounds are absolute.
# Measured ratios fp8 / bf16 (board-record and planes paths, both nets): mean |d| 3.8-4.7x, max |d| over the 518 positions
# 3.7-7.3x (one position decides the max, so it varies more).
BOUND_VALUE_MEAN_VS_BF16 = 6.0
BOUND_VALUE_MAX_VS_BF16 = 10.0
BOUND_KL_MEAN = 0.02
BOUND_TOP1 = 0.95


def _sharpened(name):
    """The golden net `name` ("seed0" | "perturbed") with policy-FC and value-FC2 weights scaled so that the logits
    have std >= 2 and the values span about +-0.9 on opening and midgame positions."""
    from chinesechesszero_b200.net import Net
    from oracle import net_oracle

    torch.manual_seed(0)
    net = Net().eval()
    if name == "perturbed":
        net_oracle.perturb_(net.state_dict(), seed=1)
    return net.cuda()


def _eval_positions():
    from chinesechesszero_b200.net import calibration_boards

    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "net_reference.npz"))["records"]
    extra = calibration_boards(512, seed=7)  # another seed than the evaluator's calibration set
    return torch.cat([torch.from_numpy(gold).cuda(), extra]).contiguous()


@torch.no_grad()
def _fp32_forward(net, boards):
    from chinesechesszero_b200 import _lib

    _, _, _, planes = _lib.movegen_encode(boards)
    tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        logp, v = net(planes.float())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    return logp, v.view(-1)


@torch.no_grad()
def _sharpen_(net, boards):
    logp, _ = _fp32_forward(net, boards)
    logits = logp - logp.mean(1, keepdim=True)
    net.policy_fc.weight.mul_(2.5 / float(logits.std(1).mean()))
    net.policy_fc.bias.zero_()
    captured = {}
    hook = net.value_fc2.register_forward_hook(lambda m, i, o: captured.setdefault("z", o.detach().clone()))
    _fp32_forward(net, boards)
    hook.remove()
    z = captured["z"].view(-1) - net.value_fc2.bias  # value_fc2 without its bias
    lo, hi = float(z.min()), float(z.max())
    k = 2 * float(np.arctanh(0.9)) / (hi - lo)  # the positions' values span exactly [-0.9, 0.9]
    net.value_fc2.weight.mul_(k)
    net.value_fc2.bias.fill_(-k * (lo + hi) / 2)
    return k


def _metrics(ref_logp, ref_v, logits, v):
    logp = torch.log_softmax(logits.double(), 1)
    kl = (ref_logp.double().exp() * (ref_logp.double() - logp)).sum(1)
    return {"value_max": float((v.double() - ref_v.double()).abs().max()),
            "value_mean": float((v.double() - ref_v.double()).abs().mean()),
            "kl_mean": float(kl.mean()), "kl_max": float(kl.max()),
            "top1": float((logp.argmax(1) == ref_logp.argmax(1)).double().mean())}


def _within(m, m16):
    return (m["value_mean"] <= BOUND_VALUE_MEAN_VS_BF16 * m16["value_mean"] and m["value_max"] <= BOUND_VALUE_MAX_VS_BF16 * m16["value_max"]
            and m["kl_mean"] <= BOUND_KL_MEAN and m["top1"] >= BOUND_TOP1)


@pytest.mark.parametrize("name", ["seed0", "perturbed"])
def test_fp8_accuracy_against_fp32_reference(name, monkeypatch):
    from chinesechesszero_b200 import net as N

    boards = _eval_positions()
    net = _sharpened(name)
    value_gain = _sharpen_(net, boards)
    ref_logp, ref_v = _fp32_forward(net, boards)
    assert float((ref_logp - ref_logp.mean(1, keepdim=True)).std(1).mean()) >= 2.0
    assert float(ref_v.max()) > 0.85 and float(ref_v.min()) < -0.85
    ev8 = N.BatchedEvaluator(net, precision="fp8")
    ev16 = N.BatchedEvaluator(net)
    m8 = _metrics(ref_logp, ref_v, *ev8.forward(None, boards))
    m16 = _metrics(ref_logp, ref_v, *ev16.forward(None, boards))
    # the planes path (cuDNN stem + torch-side quantisation) agrees with the board-record path
    lp, vp = ev8.forward(_lib_planes(boards))
    mp = _metrics(ref_logp, ref_v, lp, vp)
    # negative control: activation scales 16x too small (clipping) must push the figures past the bounds
    monkeypatch.setattr(N, "activation_scale", lambda amax: amax.float().clamp_min(1e-30) / (448.0 * 16))
    bad = N.BatchedEvaluator(net, precision="fp8", calib_boards=ev8.calib_boards)
    mbad = _metrics(ref_logp, ref_v, *bad.forward(None, boards))
    report = {"net": name, "positions": int(boards.shape[0]), "value_fc2_gain": value_gain, "fp8": m8, "bf16": m16, "fp8_planes": mp,
              "control_clipped": mbad}
    print("FP8_ACCURACY " + json.dumps(report))
    out = os.environ.get("CCZ_FP8_ACCURACY_OUT")
    if out:
        with open(out, "a") as f:
            f.write(json.dumps(report) + "\n")
    assert _within(m8, m16), report
    assert _within(mp, m16), report
    assert not _within(mbad, m16), report


def _lib_planes(boards):
    from chinesechesszero_b200 import _lib

    return _lib.movegen_encode(boards)[3]


def test_fp8_refresh_keeps_addresses_and_captured_graph_follows(fp8_pair):
    """refresh() re-quantises and re-calibrates in place: every tensor keeps its address, and a graph captured before a
    weight update replays with the new weights and scales (equal to an eager search over a fresh evaluator)."""
    from chinesechesszero_b200.net import BatchedEvaluator, Net
    from chinesechesszero_b200.search import LockstepSearch
    from oracle import net_oracle

    calib = fp8_pair[1].calib_boards

    def root_q(s):
        a = s.arena
        return torch.stack([a.children(int(a.root[g]))["value"].view(torch.int32) for g in range(a.n_games)])

    torch.manual_seed(2)
    net = Net(resblocks_num=2).cuda().eval()
    ev = BatchedEvaluator(net, precision="fp8", calib_boards=calib)
    ptrs = {k: t.data_ptr() for k, t in ev._params.items()}
    scales = ev.fp8_scales["x"].clone(), ev.fp8_scales["y"].clone()
    s = LockstepSearch(n_games=8, nodes_per_game=8192)
    s.enable_graphs(ev)
    s.run(ev, 100)
    assert s._graphs.get(0) is not None
    old_q = root_q(s)
    net_oracle.perturb_(net.state_dict(), seed=5)
    with torch.no_grad():
        for rb in net.res_blocks:
            rb.conv1.weight.mul_(1.5)
    ev.refresh(net)
    assert {k: t.data_ptr() for k, t in ev._params.items()} == ptrs
    assert not torch.equal(ev.fp8_scales["y"], scales[1])
    torch.cuda.empty_cache()
    junk = [torch.randn(1 << 20, device="cuda") for _ in range(8)]
    s.reset()
    s.run(ev, 100)
    got = root_q(s)
    ref = LockstepSearch(n_games=8, nodes_per_game=8192)
    ref.run(BatchedEvaluator(net, precision="fp8", calib_boards=calib), 100)
    assert torch.equal(got, root_q(ref))
    assert not torch.equal(got, old_q)
    del junk


def test_fp8_selfplay_soak_keeps_the_pool_healthy():
    """1024 games x 100 playouts x 10 resident moves of the full 40-block net in fp8: no failed expansion, no dropped tree."""
    from chinesechesszero_b200.net import BatchedEvaluator, Net
    from chinesechesszero_b200.selfplay import SelfPlayEngine

    torch.manual_seed(0)
    net = Net().cuda().eval()
    ev = BatchedEvaluator(net, precision="fp8")
    eng = SelfPlayEngine(ev, n_games=1024, n_playout=100, seed=11, max_game_moves=24, resident_ring=12)
    eng._resident_state()["move_count"].copy_(torch.from_numpy(np.arange(1024, dtype=np.int64) % 24))
    for _ in range(10):
        eng.play_move_resident()
    st = eng.pool_events()
    assert st["expand_failed"] == 0 and st["trees_dropped"] == 0
