"""A/B of leaf deduplication (K12, csrc/ccz_dedup.cuh) on the `value` arm of bench.py: 4096 games x 400 playouts, the
bench's stagger (slot g starts g % 24 moves into its game), max_game_moves 24, device-resident moves.

Two engines with the same seed play side by side, one evaluator with dedup and one without, alternating by move
(A B A B ...).  Reports ms per move of each mode, the unique fraction of the leaf batch per step (mean / min / max, and
per move), K9 per launch at U boards with TFLOP/s counted from U, the cost of K12 and of the K11 row map, whether the
ring samples of the two engines are identical, and the card's name and power limit.

    python scripts/bench_leaf_dedup.py [--games 4096] [--playouts 400] [--warmup 5] [--moves 10] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from chinesechesszero_b200 import _lib
from chinesechesszero_b200.net import BatchedEvaluator, Net
from chinesechesszero_b200.selfplay import SelfPlayEngine

K9_FLOP_PER_BOARD = 2 * 90 * 256 * 2304


class CountingEvaluator:
    """Records K12's count of every step in a device buffer (one 4-byte copy per step, no synchronisation)."""

    def __init__(self, ev, cap):
        self.ev, self.needs_planes = ev, ev.needs_planes
        self.counts = torch.zeros(cap, dtype=torch.int32, device="cuda")
        self.n = 0

    def __call__(self, planes, leaf_boards):
        out = self.ev(planes, leaf_boards)
        self.counts[self.n].copy_(self.ev._dedup_buffers(leaf_boards.shape[0])[2][0])
        self.n += 1
        return out


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--playouts", type=int, default=400)
    ap.add_argument("--max-game-moves", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--moves", type=int, default=10, help="timed moves per mode")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    G, P, M = a.games, a.playouts, a.max_game_moves
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    torch.manual_seed(0)
    net = Net().cuda().eval()
    ev_on, ev_off = BatchedEvaluator(net), BatchedEvaluator(net, dedup=False)
    counting = CountingEvaluator(ev_on, P * (a.warmup + a.moves))
    stagger = torch.from_numpy(np.arange(G, dtype=np.int64) % M)
    engines = {}
    for mode, ev in (("dedup", counting), ("plain", ev_off)):
        eng = SelfPlayEngine(ev, n_games=G, n_playout=P, seed=4321, max_game_moves=M, resident_ring=a.warmup + a.moves + 1)
        eng._resident_state()["move_count"].copy_(stagger)
        engines[mode] = eng
    ms = {"dedup": [], "plain": []}
    for i in range(a.warmup + a.moves):
        for mode, eng in engines.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            eng.play_move_resident()
            e1.record()
            torch.cuda.synchronize()
            if i >= a.warmup:
                ms[mode].append(e0.elapsed_time(e1))
    rings = {mode: eng.drain_resident() for mode, eng in engines.items()}  # the ring holds every move: nothing was backlogged
    same = all(np.array_equal(rings["dedup"][k].view(np.uint8), rings["plain"][k].view(np.uint8)) for k in rings["dedup"])
    frac = counting.counts[:counting.n].cpu().numpy().astype(np.float64) / G
    per_move = frac.reshape(-1, P).mean(1)
    timed_frac = frac[a.warmup * P:]

    # kernel costs on the last live leaf batch
    s = engines["dedup"].search
    _lib.mcts_select(s.arena, s.c_puct, s.leaf_boards, s.leaf_nodes)
    rows, uniq, count = ev_on._dedup_buffers(G)
    _lib.leaf_unique(s.leaf_boards, rows, uniq, count)
    U = int(count.item())
    k12_ms = timed(lambda: _lib.leaf_unique(s.leaf_boards, rows, uniq, count), 200)
    x = _lib.stem_lookup(uniq, *ev_on.stem_lookup, count=count)
    w, _, b32 = ev_on.blocks[0][0]
    k9_u_ms = timed(lambda: _lib.conv3x3_c256(x, w, b32, count=count), 50)
    k9_g_ms = timed(lambda: _lib.conv3x3_c256(x, w, b32), 50)
    h = torch.zeros((G * 90, 32), dtype=torch.bfloat16, device="cuda")
    ops = torch.zeros((G, ev_on._kp + ev_on._kv), dtype=torch.bfloat16, device="cuda")
    pack_rows_ms = timed(lambda: _lib.heads_pack(h, ops, ev_on._kp, rows=rows), 200)
    pack_ms = timed(lambda: _lib.heads_pack(h, ops, ev_on._kp), 200)
    res = {
        "gpu": smi.stdout.strip(), "games": G, "playouts": P, "max_game_moves": M, "warmup_moves": a.warmup,
        "timed_moves_per_mode": a.moves, "order": "dedup, plain alternating by move",
        "ms_per_move": {k: float(np.mean(v)) for k, v in ms.items()},
        "ms_per_move_each": ms,
        "speedup": float(np.mean(ms["plain"]) / np.mean(ms["dedup"])),
        "unique_frac_timed": {"mean": float(timed_frac.mean()), "min": float(timed_frac.min()), "max": float(timed_frac.max())},
        "unique_frac_per_move": [float(v) for v in per_move],
        "k9_at_U": {"U": U, "ms": k9_u_ms, "tflops": U * K9_FLOP_PER_BOARD / k9_u_ms / 1e9},
        "k9_at_G": {"G": G, "ms": k9_g_ms, "tflops": G * K9_FLOP_PER_BOARD / k9_g_ms / 1e9},
        "k12_ms": k12_ms, "k11_rows_ms": pack_rows_ms, "k11_ms": pack_ms,
        "ring_samples_identical": bool(same),
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
