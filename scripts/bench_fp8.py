"""A/B of the FP8 evaluator (BatchedEvaluator(precision="fp8"): e4m3 K9 / K10 tower) against the bf16 one, in one process.

  * K9 per launch, bf16 vs e4m3, at 4096 boards, plain and with skip, arms alternating; TFLOP/s counted from shapes.  Each
    arm cycles through 4 input sets (bf16: 4 x 189 MB, e4m3: 4 x 94 MB) so that the working set exceeds the 126 MB L2.
    SM clock and board power are sampled by nvidia-smi during each arm.
  * The forward pass of the 40-block net at 4096 distinct boards (dedup off), arms alternating.
  * play_move_resident ms/move with bench.py's `value` configuration (4096 games x 400 playouts, slot g starts g % 24 moves
    into its game, max_game_moves 24), the two engines alternating by move.
  * Accuracy of fp8 against bf16 on positions outside the calibration set (value |d|, KL, top-1 agreement) and the
    agreement of the most-visited root move of the two engines on the root positions they share.
  * The card's name and power limit, read in the same call.

    python scripts/bench_fp8.py [--games 4096] [--playouts 400] [--warmup 3] [--moves 6] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from bench import ClockSampler
from chinesechesszero_b200 import _lib
from chinesechesszero_b200.net import BatchedEvaluator, Net, calibration_boards
from chinesechesszero_b200.selfplay import SelfPlayEngine

K9_FLOP_PER_BOARD = 2 * 90 * 256 * 2304


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def sampled(fn, reps):
    s = ClockSampler(torch.cuda.current_device()).start()
    ms = timed(fn, reps)
    summary = s.stop()
    power = sorted(float(r[2]) for r in s.rows if len(r) > 2 and r[2].replace(".", "", 1).isdigit())
    summary["power_w_median"] = power[len(power) // 2] if power else None
    return ms, summary


def spread(v):
    v = np.asarray(v)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()), "n": int(v.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--playouts", type=int, default=400)
    ap.add_argument("--max-game-moves", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--moves", type=int, default=6, help="timed moves per arm")
    ap.add_argument("--k9-reps", type=int, default=200, help="K9 launches per timed window")
    ap.add_argument("--repeats", type=int, default=5, help="alternating windows per arm")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp8.py measures on the GPU; no CUDA device found")
    G, P, M = a.games, a.playouts, a.max_game_moves
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True)
    torch.manual_seed(0)
    net = Net().cuda().eval()
    ev16 = BatchedEvaluator(net, dedup=False)
    ev8 = BatchedEvaluator(net, precision="fp8", dedup=False)
    res = {"gpu": smi.stdout.strip(), "games": G, "playouts": P, "max_game_moves": M}

    # ---- K9 per launch --------------------------------------------------------------------------------------------
    from chinesechesszero_b200 import positions

    boards = positions.bench_positions(4 * 4096, seed=5)
    xs, xqs = [], []
    for i in range(4):
        x, xq = _lib.stem_lookup_e4m3(boards[i * 4096:(i + 1) * 4096].contiguous(), *ev8.stem_lookup, ev8._inv_sx[0:1])
        xs.append(x)
        xqs.append(xq)
    w16, _, b32 = ev16.blocks[0][1]
    wq, deq, _ = ev8.qblocks[0][1]
    inv = ev8._inv_sx[1:2]
    outs16 = [torch.empty_like(x) for x in xs]
    skips = [x.clone() for x in xs]
    yqs = [torch.empty_like(xq) for xq in xqs]
    n = 4096
    arms = {
        "bf16_plain": lambda i: _lib.conv3x3_c256(xs[i % 4], w16, b32, out=outs16[i % 4]),
        "e4m3_plain": lambda i: _lib.conv3x3_c256_e4m3(xqs[i % 4], wq, deq, b32, out=outs16[i % 4]),
        "bf16_skip": lambda i: _lib.conv3x3_c256(xs[i % 4], w16, b32, skip=skips[i % 4], out=outs16[i % 4]),
        "e4m3_skip": lambda i: _lib.conv3x3_c256_e4m3(xqs[i % 4], wq, deq, b32, skip=skips[i % 4], out=outs16[i % 4]),
        # what the fp8 tower runs: conv1 e4m3 -> e4m3 only; conv2 with skip -> bf16 + e4m3
        "e4m3_conv1_q_only": lambda i: _lib.conv3x3_c256_e4m3(xqs[i % 4], wq, deq, b32, y=False, out_q=yqs[i % 4], inv_s_out=inv),
        "e4m3_conv2_y_and_q": lambda i: _lib.conv3x3_c256_e4m3(xqs[i % 4], wq, deq, b32, skip=skips[i % 4], out=outs16[i % 4],
                                                               out_q=yqs[i % 4], inv_s_out=inv),
    }
    for fn in arms.values():  # warm-up: module load, attributes, occupancy query
        for i in range(8):
            fn(i)
    torch.cuda.synchronize()
    k9 = {k: [] for k in arms}
    clocks = {k: [] for k in arms}
    for _ in range(a.repeats):
        for k, fn in arms.items():
            ms, c = sampled(fn, a.k9_reps)
            k9[k].append(ms)
            clocks[k].append(c)
    res["k9_per_launch"] = {
        k: {"ms": spread(v), "tflops_at_median": n * K9_FLOP_PER_BOARD / float(np.median(v)) / 1e9,
            "sm_mhz": [c["sm_mhz"] for c in clocks[k]], "power_w": [c["power_w_median"] for c in clocks[k]],
            "throttle": sorted({r for c in clocks[k] for r in c["reasons"]})}
        for k, v in k9.items()}
    res["k9_speedup"] = {"plain": float(np.median(k9["bf16_plain"]) / np.median(k9["e4m3_plain"])),
                         "skip": float(np.median(k9["bf16_skip"]) / np.median(k9["e4m3_skip"]))}
    res["k9_note"] = "4096 boards per launch, 4 rotating input sets (working set > L2), arms alternating by window"
    del xs, xqs, outs16, skips, yqs

    # ---- forward ----------------------------------------------------------------------------------------------------
    fb = boards[:4096].contiguous()
    fwd = {"bf16": [], "fp8": []}
    for ev in (ev16, ev8):
        ev.forward(None, fb)
    for _ in range(a.repeats):
        for k, ev in (("bf16", ev16), ("fp8", ev8)):
            fwd[k].append(timed(lambda i, ev=ev: ev.forward(None, fb), 5))
    res["forward_ms_4096"] = {k: spread(v) for k, v in fwd.items()}
    res["forward_speedup"] = float(np.median(fwd["bf16"]) / np.median(fwd["fp8"]))

    # ---- accuracy fp8 vs bf16 on positions outside the calibration set ----------------------------------------------
    eb = calibration_boards(2048, seed=11)
    l16, v16 = ev16.forward(None, eb)
    l8, v8 = ev8.forward(None, eb)
    p16 = torch.log_softmax(l16.double(), 1)
    p8 = torch.log_softmax(l8.double(), 1)
    kl = (p16.exp() * (p16 - p8)).sum(1)
    res["accuracy_vs_bf16"] = {"positions": int(eb.shape[0]), "net": "Net() seed 0 (random init)",
                               "value_abs_diff_max": float((v8 - v16).abs().max()), "value_abs_diff_mean": float((v8 - v16).abs().mean()),
                               "kl_mean": float(kl.mean()), "kl_max": float(kl.max()),
                               "top1_agreement": float((p8.argmax(1) == p16.argmax(1)).double().mean())}
    del ev16, ev8
    torch.cuda.empty_cache()

    # ---- play_move_resident A/B ---------------------------------------------------------------------------------------
    stagger = torch.from_numpy(np.arange(G, dtype=np.int64) % M)
    engines = {}
    for k, prec in (("bf16", "bf16"), ("fp8", "fp8")):
        eng = SelfPlayEngine(BatchedEvaluator(net, precision=prec), n_games=G, n_playout=P, seed=4321, max_game_moves=M,
                             resident_ring=a.warmup + a.moves + 1)
        eng._resident_state()["move_count"].copy_(stagger)
        engines[k] = eng
    ms = {k: [] for k in engines}
    for i in range(a.warmup + a.moves):
        for k, eng in engines.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            eng.play_move_resident()
            e1.record()
            torch.cuda.synchronize()
            if i >= a.warmup:
                ms[k].append(e0.elapsed_time(e1))
    rings = {k: eng.drain_resident() for k, eng in engines.items()}
    rb16, rb8 = rings["bf16"], rings["fp8"]
    same_root = np.all(rb16["boards"].reshape(rb16["boards"].shape[0], G, -1) == rb8["boards"].reshape(rb8["boards"].shape[0], G, -1), axis=2)
    pick16 = rb16["pi"].reshape(same_root.shape[0], G, -1).argmax(2)
    pick8 = rb8["pi"].reshape(same_root.shape[0], G, -1).argmax(2)
    res["play_move_resident"] = {
        "ms_per_move": {k: spread(v) for k, v in ms.items()}, "ms_per_move_each": ms,
        "speedup": float(np.median(ms["bf16"]) / np.median(ms["fp8"])),
        "moves_per_s": {k: G / (float(np.median(v)) / 1e3) for k, v in ms.items()},
        "order": "bf16, fp8 alternating by move", "warmup_moves": a.warmup,
        "most_visited_root_move_agreement": {"shared_roots": int(same_root.sum()),
                                             "agreement": float((pick16 == pick8)[same_root].mean()) if same_root.any() else None},
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
