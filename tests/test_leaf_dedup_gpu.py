"""Leaf deduplication (K12, csrc/ccz_dedup.cuh) and the device-count paths of K9 / K10 / K11 it feeds.

The evaluator forwards each distinct leaf position once and maps the results back to every game, so its
output must not depend on where a board sits in the batch: K9 must give every board the same bits whatever
the batch size, its row, and whether its tile lands in a tail-split (channel-sliced) round."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def acts():
    """Stem activations of 8192 distinct reachable positions, plus a second set as the skip input."""
    from chinesechesszero_b200 import _lib, positions
    from chinesechesszero_b200.net import BatchedEvaluator, Net

    torch.manual_seed(0)
    net = Net().eval()
    ev = BatchedEvaluator(net, "cuda")
    boards = positions.bench_positions(8192 + 4096, seed=3)
    x = _lib.stem_lookup(boards[:8192].contiguous(), *ev.stem_lookup)
    skip = _lib.stem_lookup(boards[8192:].repeat(2, 1).contiguous(), *ev.stem_lookup)
    w, _, b32 = ev.blocks[0][0]
    return x, skip, w, b32


def _invariance_sizes():
    return list(range(1, 301)) + [3793, 4096, 8192]


@pytest.mark.parametrize("with_skip", [False, True])
def test_k9_is_row_position_invariant(acts, with_skip):
    """Boards permuted and embedded at other offsets, in batches of 1..300, 3793, 4096 and 8192 boards (many of
    which end in tail-split rounds), come out bit-identical to the full 8192-board launch."""
    from chinesechesszero_b200 import _lib

    x, skip, w, b32 = acts
    full = _lib.conv3x3_c256(x, w, b32, skip if with_skip else None)
    gen = torch.Generator(device="cpu").manual_seed(1 + with_skip)
    splits = set()
    for n in _invariance_sizes():
        perm = torch.randperm(8192, generator=gen)[:n].cuda()
        xs = x[perm].contiguous(memory_format=torch.channels_last)
        ss = skip[perm].contiguous(memory_format=torch.channels_last) if with_skip else None
        y = _lib.conv3x3_c256(xs, w, b32, ss)
        assert torch.equal(y.view(torch.int16), full[perm].view(torch.int16)), f"n={n}"
        splits.add(_lib.conv3x3_plan(n)["split_log2"])
    assert splits == {0, 1, 2}


def _unique_ref(boards: np.ndarray):
    """NumPy reference of K12: rows in order of first occurrence of bytes 0..90."""
    first, rows = {}, np.empty(len(boards), dtype=np.int32)
    for g, rec in enumerate(boards):
        rows[g] = first.setdefault(rec[:91].tobytes(), len(first))
    reps = np.empty(len(first), dtype=np.int64)
    for g in range(len(boards) - 1, -1, -1):
        reps[rows[g]] = g
    return rows, reps, len(first)


def _run_unique(boards_np: np.ndarray):
    from chinesechesszero_b200 import _lib

    n = len(boards_np)
    boards = torch.from_numpy(boards_np).cuda()
    rows = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    uniq = torch.full((n, 96), 0xAB, dtype=torch.uint8, device="cuda")
    count = torch.zeros(1, dtype=torch.int32, device="cuda")
    total = torch.full((1,), 5, dtype=torch.int64, device="cuda")
    _lib.leaf_unique(boards, rows, uniq, count, total)
    u = int(count.item())
    assert int(total.item()) == 5 + u
    return rows.cpu().numpy(), uniq.cpu().numpy(), u


def _check_unique(boards_np: np.ndarray, expect_u=None):
    rows, uniq, u = _run_unique(boards_np)
    ref_rows, reps, ref_u = _unique_ref(boards_np)
    assert u == ref_u and (expect_u is None or u == expect_u)
    assert np.array_equal(rows, ref_rows)
    assert np.array_equal(uniq[:u], boards_np[reps])  # the whole record of the first occurrence
    assert (uniq[u:] == 0xAB).all()                    # rows >= U untouched
    return u


@pytest.fixture(scope="module")
def distinct_boards():
    from chinesechesszero_b200 import positions

    b = positions.bench_positions(12000, seed=7).cpu().numpy()  # perft leaves repeat positions (transpositions)
    _, first = np.unique(b[:, :91], axis=0, return_index=True)
    return b[np.sort(first)[:8192]]


@pytest.mark.parametrize("n", [1, 4096, 8192])
def test_leaf_unique_all_identical_and_all_distinct(distinct_boards, n):
    _check_unique(np.repeat(distinct_boards[3:4], n, axis=0), expect_u=1)
    _check_unique(distinct_boards[:n].copy(), expect_u=n)


@pytest.mark.parametrize("n", [1, 257, 4096, 8192, 16384])
def test_leaf_unique_random_duplicates_in_order_of_first_occurrence(distinct_boards, n):
    rng = np.random.default_rng(n)
    pick = rng.integers(0, max(1, n // 7), size=n)
    _check_unique(distinct_boards[pick])


def test_leaf_unique_identity_is_squares_and_side_to_move(distinct_boards):
    base = np.repeat(distinct_boards[10:11], 6, axis=0)
    base[1, 91:] ^= 0x5A          # clock / repetition bytes differ: same position
    base[2, 95] += 1
    base[3, 90] ^= 1              # side to move differs: another position
    base[4, 44] ^= 0x09           # one square differs
    base[5, 91:] = base[1, 91:]   # = row 0 again
    rows, _, u = _run_unique(base)
    assert u == 3 and rows.tolist() == [0, 0, 0, 1, 2, 0]


def test_count_entry_points_equal_the_plain_ones(acts, distinct_boards):
    """K10 / K9 over the first U boards of a capacity-G buffer equal the plain launches over U boards, bit for bit;
    K11 with a row map equals K11 over the gathered rows."""
    from chinesechesszero_b200 import _lib
    from chinesechesszero_b200.net import BatchedEvaluator, Net

    x, skip, w, b32 = acts
    ev = BatchedEvaluator(Net(resblocks_num=1).eval(), "cuda")
    boards = torch.from_numpy(distinct_boards[:4096]).cuda()
    for cap, u in [(4096, 1), (4096, 300), (4096, 3793), (8192, 8192), (8192, 4096), (4096, 0)]:
        count = torch.tensor([u], dtype=torch.int32, device="cuda")
        xs = x[:cap].contiguous(memory_format=torch.channels_last)
        for sk in (None, skip[:cap].contiguous(memory_format=torch.channels_last)):
            got = _lib.conv3x3_c256(xs, w, b32, sk, count=count)
            if u:
                ref = _lib.conv3x3_c256(xs[:u].contiguous(memory_format=torch.channels_last), w, b32,
                                        None if sk is None else sk[:u].contiguous(memory_format=torch.channels_last))
                assert torch.equal(got[:u].view(torch.int16), ref.view(torch.int16)), (cap, u)
        if cap <= 4096:
            out = torch.zeros((cap, 256, 10, 9), dtype=torch.bfloat16, device="cuda").contiguous(memory_format=torch.channels_last)
            _lib.stem_lookup(boards[:cap], *ev.stem_lookup, out=out, count=count)
            if u:
                ref = _lib.stem_lookup(boards[:u].contiguous(), *ev.stem_lookup)
                assert torch.equal(out[:u].view(torch.int16), ref.view(torch.int16))
            if u < cap:  # rows past the count are not written
                assert out[u:].abs().max().item() == 0
    g = 777
    h = torch.randn(g * 90, 32, device="cuda").to(torch.bfloat16)
    rows = torch.randint(0, g, (g,), dtype=torch.int32, device="cuda")
    a = torch.zeros((g, 2176), dtype=torch.bfloat16, device="cuda")
    b = torch.zeros_like(a)
    _lib.heads_pack(h, a, 1536, rows=rows)
    _lib.heads_pack(h.view(g, 90, 32)[rows.long()].reshape(g * 90, 32).contiguous(), b, 1536)
    assert torch.equal(a.view(torch.int16), b.view(torch.int16))


def _live_leaves(n_games=512):
    """A live search whose games share their opening: all start from the start position and play one of its first
    moves by game index, so the leaf batch holds many duplicates and a few dozen distinct positions."""
    from chinesechesszero_b200.net import BatchedEvaluator, Net
    from chinesechesszero_b200.search import LockstepSearch

    torch.manual_seed(0)
    net = Net(resblocks_num=2).cuda().eval()
    ev = BatchedEvaluator(net, dedup=False)
    s = LockstepSearch(n_games, nodes_per_game=8192)
    s.run(ev, 6)
    acts, _, counts = s.root_visits()
    g = torch.arange(n_games, device="cuda")
    s.advance(acts[g, g % counts.long()])
    s.run(ev, 6)
    return net, s


def test_evaluator_dedup_is_bitwise_equal_eager_and_under_graphs():
    from chinesechesszero_b200 import _lib
    from chinesechesszero_b200.net import BatchedEvaluator

    net, s = _live_leaves()
    _lib.mcts_select(s.arena, s.c_puct, s.leaf_boards, s.leaf_nodes)
    boards = s.leaf_boards.clone()
    n_distinct = len({bytes(r[:91]) for r in boards.cpu().numpy()})
    assert 8 < n_distinct < boards.shape[0] // 4
    off, on = BatchedEvaluator(net, dedup=False), BatchedEvaluator(net)
    lo, _, vo = off(None, boards)
    ln, _, vn = on(None, boards)
    assert torch.equal(lo, ln) and torch.equal(vo, vn)
    assert on.n_unique == n_distinct and off.n_unique == boards.shape[0] and on.n_evals == off.n_evals
    # graph replay on a batch with another duplicate pattern
    static = boards.clone()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gl, _, gv = on(None, static)
    perm = torch.randperm(boards.shape[0], device="cuda")
    static.copy_(boards[perm])
    graph.replay()
    lo2, _, vo2 = off(None, boards[perm].contiguous())
    assert torch.equal(gl, lo2) and torch.equal(gv, vo2)


def test_selfplay_ring_samples_identical_with_and_without_dedup():
    """Eight resident moves with the bench's stagger (slots 0..23 moves into their games, max_game_moves 24)."""
    from chinesechesszero_b200.net import BatchedEvaluator, Net
    from chinesechesszero_b200.selfplay import SelfPlayEngine

    torch.manual_seed(0)
    net = Net(resblocks_num=2).cuda().eval()
    G, M = 384, 24
    out = []
    for dedup in (True, False):
        ev = BatchedEvaluator(net, dedup=dedup)
        eng = SelfPlayEngine(ev, n_games=G, n_playout=16, seed=4321, max_game_moves=M, resident_ring=8,
                             nodes_per_game=16 * 41 * 8)
        eng._resident_state()["move_count"].copy_(torch.from_numpy(np.arange(G, dtype=np.int64) % M))
        for _ in range(8):
            eng.play_move_resident()
        eng.resident_backlog.append(eng.drain_resident())
        out.append((eng.resident_backlog, ev))
    (a, ev_on), (b, ev_off) = out
    assert len(a) == len(b)
    for da, db in zip(a, b):
        assert da.keys() == db.keys()
        for k in da:
            va, vb = da[k], db[k]
            if va.dtype == np.float64:
                va, vb = va.view(np.uint64), vb.view(np.uint64)
            assert np.array_equal(va, vb), k
    assert ev_on.n_unique < ev_off.n_unique
