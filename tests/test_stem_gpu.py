"""K10 (csrc/ccz_stem.cuh): the stem convolution of search-time inputs evaluated from the board records as a
table lookup, against (a) a plain fp32 torch convolution of the planes K1 encodes for the same boards and
(b) the evaluator's generic stem; and the whole forward from boards against the forward from planes."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _boards(n=600):
    from tests.positions import edge_case_records, random_playout_positions

    # mid- and end-game positions of random playouts: both sides to move, captures, pieces on every edge
    recs = np.concatenate([random_playout_positions(8, 120, seed=3, every=1), edge_case_records()])
    rng = np.random.default_rng(0)
    recs = recs[rng.permutation(len(recs))[:n]]
    return torch.from_numpy(np.ascontiguousarray(recs)).cuda()


def test_stem_lookup_matches_fp32_conv_of_the_planes():
    from chinesechesszero_b200 import _lib
    from chinesechesszero_b200.net import Net, BatchedEvaluator
    from oracle import net_oracle

    torch.manual_seed(1)
    net = Net(resblocks_num=1)
    net_oracle.perturb_(net.state_dict(), seed=4)  # non-trivial BN statistics
    ev = BatchedEvaluator(net.cuda().eval(), conv_impl="k9")
    assert ev.stem_lookup is not None and not ev.needs_planes
    boards = _boards()
    assert int(boards[:, 90].sum()) not in (0, boards.shape[0])  # both turn values present
    _, _, _, planes = _lib.movegen_encode(boards)
    from tests.test_forward_stages_gpu import U_BF16, U_FP32, conv3x3_f64, elementwise_bound, gamma_f16, worst_ratio

    w, _, b32 = ev.stem
    p = planes.view(-1, 119, 10, 9)
    ref = torch.relu(conv3x3_f64(p, w) + b32.double().view(1, -1, 1, 1))
    y = _lib.stem_lookup(boards, *ev.stem_lookup)
    assert y.is_contiguous(memory_format=torch.channels_last)
    # same bf16 weights: per element, fp32 sums (table rows + bias_turn) and one bf16 rounding of the output
    bound = elementwise_bound(ref, conv3x3_f64(p.double().abs(), w.double().abs()), (U_FP32,),
                              b32.double().abs().view(1, -1, 1, 1), U_BF16, gamma_f16(119 * 9 + 1))
    assert worst_ratio(y, ref, bound) <= 1.0
    ref = ref.float()
    # and the generic (cuDNN) stem on the same planes agrees to one bf16 rounding
    x = planes.view(-1, 119, 10, 9).contiguous(memory_format=torch.channels_last)
    y2 = ev._conv_relu(x, ev.stem)
    assert (y.float() - y2.float()).abs().max().item() <= 2.0 ** -7 * ref.abs().max().item()


def test_forward_from_boards_equals_forward_from_planes():
    from chinesechesszero_b200 import _lib
    from chinesechesszero_b200.net import Net, BatchedEvaluator

    torch.manual_seed(2)
    ev = BatchedEvaluator(Net(resblocks_num=3).cuda().eval(), conv_impl="k9")
    boards = _boards(300)
    _, _, _, planes = _lib.movegen_encode(boards)
    lp, vp = ev.forward(planes)
    lb, vb = ev.forward(None, boards)
    assert (torch.softmax(lp, 1) - torch.softmax(lb, 1)).abs().max().item() < 2e-3
    assert (vp - vb).abs().max().item() < 5e-3
    # the evaluator protocol takes the boards route and never touches `planes`
    lc, kind, vc = ev(None, boards)
    assert kind == _lib.POLICY_LOGITS and torch.equal(lc, lb) and torch.equal(vc, vb)


def test_search_skips_plane_encoding_when_the_evaluator_reads_boards():
    from chinesechesszero_b200.net import Net, BatchedEvaluator
    from chinesechesszero_b200.search import LockstepSearch

    torch.manual_seed(3)
    ev = BatchedEvaluator(Net(resblocks_num=1).cuda().eval(), conv_impl="k9")
    s = LockstepSearch(n_games=8, node_cap=4096)
    s.planes.fill_(7.0)
    s.run(ev, 12)
    s.check_status()
    assert float(s.planes.min()) == 7.0  # K1 ran with planes = NULL
    _, visits, _ = s.root_visits()
    assert int(visits[0].sum()) == 11   # 12 playouts: the first expands the root, 11 visit its children
