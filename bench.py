#!/usr/bin/env python
"""bench.py -- headline benchmark of the self-play hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W]            own arm (CUDA kernels + bf16 net)
  python bench.py ... --dump-outputs DIR                         also write the last timed move's samples as .npy
  python bench.py --impl reference [--steps K] [--warmup W]      reference arm (CPU port of collect.py)
  torchrun --nproc-per-node N ... bench.py --gpus N ...          one rank per GPU, games sharded

A *step* is one lockstep self-play move: n_playout (400) playouts in each of G (4096) concurrent
games per GPU -- select, movegen+encode, one bf16 net forward over the whole leaf batch, expand +
backup -- followed by move choice, tree re-rooting, terminal test and slot refill.
Prints ONE JSON line (see DESIGN.md "Measurement" for every key).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "self-play moves/sec at 400 playouts"  # the playout count in the string follows --playouts
UNIT = "moves/s"


def metric_name(playouts: int) -> str:
    return f"self-play moves/sec at {playouts} playouts"


def workload_name(games: int, playouts: int) -> str:
    tag = "configs[3] (per-GPU shard of the 8xB200 run)" if (games, playouts) == (8192, 800) else "configs[2]"
    return (f"{tag}: lockstep batched self-play, {games} concurrent games x {playouts} playouts per GPU, "
            "random-init 40x256 PolicyValueNet")


def ncu_traffic(kernel: str, units: int):
    """dram read+write bytes per launch from the committed ncu capture (profiles/ncu_traffic.json),
    scaled to `units`; None when no capture is recorded for the kernel."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)[kernel]
        return (t["dram_bytes_read"] + t["dram_bytes_write"]) * units / t["positions_per_launch"]
    except (OSError, KeyError, ValueError):
        return None


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--games", type=int, default=4096, help="concurrent games per GPU (configs[2]: 4096)")
    ap.add_argument("--playouts", type=int, default=400)
    ap.add_argument("--nodes-per-game", type=int, default=None,
                    help="average node budget per game of the shared MCTS page pool (default: 8 x 41 x playouts)")
    ap.add_argument("--max-game-moves", type=int, default=24,
                    help="self-play games are cut after this many moves and the slots start staggered, so that games "
                         "finish (and their replay is packed and written) at the steady-state rate inside the timed regions")
    ap.add_argument("--replay-dir", default=None, help="where the e2e arm writes data.h5 (default: a temporary directory)")
    ap.add_argument("--no-replay", action="store_true", help="e2e without replay packing / writing")
    ap.add_argument("--movegen-positions", type=int, default=1 << 20)
    ap.add_argument("--no-movegen", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the configs[4] train-step section")
    ap.add_argument("--graphs", action="store_true",
                    help="replay the lockstep step from CUDA graphs (the forward is then timed in a separate loop)")
    ap.add_argument("--cpu-moves", type=int, default=3, help="moves of the CPU-port sample (SURVEY 8d: the first 3 moves, ~16 s)")
    ap.add_argument("--conv-impl", default=None, choices=["k9", "k9_skip", "cudnn"],
                    help="tower convolution kernel (default: the evaluator's default, K9 = csrc/ccz_conv.cuh)")
    ap.add_argument("--conv-sample", type=int, default=8, help="bracket every K9 launch of every n-th forward with CUDA events")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the samples of the last timed move of the `value` arm as DIR/<name>.npy (float32 / "
                         "float64, rank 0, at most 64 MB: a fixed seeded subset of the games beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "own":
        ap.error("--dump-outputs needs --impl own")
    return args


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.thread = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return self
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir: str, sample: dict, limit: int = DUMP_LIMIT) -> None:
    """One move's per-game samples (SelfPlayEngine.drain_resident() keys, one row per game) as float32 / float64
    .npy files, so that two builds can be compared output for output.  ``game_index.npy`` names the games kept:
    all of them, or a fixed seeded subset when the files would exceed ``limit`` bytes."""
    import numpy as np

    arrays = {k: v.astype(np.float64 if v.dtype == np.float64 else np.float32) for k, v in sample.items()}
    n_games = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a[0].nbytes for a in arrays.values()) + 8  # + the float64 game index
    budget = limit - 128 * (len(arrays) + 1)  # an .npy header of these shapes is 128 bytes
    games = np.arange(n_games)
    if row_bytes * n_games > budget:
        games = np.sort(np.random.default_rng(0).choice(n_games, budget // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "game_index.npy"), games.astype(np.float64))
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a[games])


# ------------------------------------------------------------------------------------------------
def _reference_player(n_playout: int, cores: int):
    """(player, kind, what): the unmodified reference (oracle/_ref snapshot or /root/reference) when present,
    else the oracle port of the collect path."""
    from oracle import reference_arm

    if reference_arm.available():
        return (reference_arm.ReferenceSelfPlay(n_playout=n_playout, threads=cores), "reference",
                "UNMODIFIED reference modules (net.PolicyValueNet(use_gpu=False) CPU branch, mcts.MCTS_AI, the loop body of "
                "Game.start_self_play) with cchess replaced by the C-backed shim (favours the reference)")
    from oracle import collect_oracle

    return (collect_oracle.PortedSelfPlay(n_playout=n_playout, threads=cores), "port",
            "CPU port of collect.py -> game.py -> mcts.py -> net.py (shim board, flat search, fp32 batch-1 forward per playout)")


def cpu_baseline(n_moves: int, n_playout: int):
    """The reference's collect.py path on the host cores, bounded sample (SURVEY 8d: the first moves of one game)."""
    cores = os.cpu_count() or 1
    sp, kind, what = _reference_player(n_playout, cores)
    sp.policy_value_net.policy_value_fn(sp.game.board) if kind == "reference" else sp.policy_value_fn(sp.board)  # page in
    t0 = time.perf_counter()
    for _ in range(n_moves):
        sp.play_move()
    secs = time.perf_counter() - t0
    return {"value": n_moves / secs, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"first {n_moves} move(s) of one self-play game from the start position, {n_playout} playouts "
                      f"each, batch-1 fp32 forward per playout, {secs:.1f} s; {what}"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sp, kind, what = _reference_player(args.playouts, cores)
    for _ in range(args.warmup):
        sp.play_move()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sp.play_move()
    dt = time.perf_counter() - t0
    v = args.steps / dt
    sample = (f"{args.steps} consecutive move(s) of one self-play game after {args.warmup} warm-up move(s), {args.playouts} playouts "
              f"each, tree reuse, batch-1 fp32 forward per playout on {cores} host threads; {what}")
    print(json.dumps({
        "impl": "reference", "metric": metric_name(args.playouts), "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (random-init net, torch.manual_seed(0))",
        "config": {"workload": workload_name(args.games, args.playouts), "games_per_gpu": args.games, "n_playout": args.playouts,
                   "sample": "the reference plays its games one after the other (collect.py:138): each step is one move of ONE of the "
                             f"{args.games} games, {args.playouts} playouts; moves/s of one game = the reference's whole-job rate on this host"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------
def bench_movegen(torch, _lib, n_positions: int, peaks):
    """configs[1]: legal-move generation + plane encoding on ~1M perft-reachable positions."""
    from chinesechesszero_b200 import positions

    boards = positions.bench_positions(n_positions, seed=0)  # generated on the device by K1 + K2
    n = boards.shape[0]
    recs_host = boards[: min(n, 1 << 16)].cpu()
    ids = torch.empty((n, 128), dtype=torch.int16, device="cuda")
    counts = torch.empty((n,), dtype=torch.int16, device="cuda")
    flags = torch.empty((n,), dtype=torch.uint8, device="cuda")
    planes = torch.empty((n, 17, 7, 10, 9), dtype=torch.bfloat16, device="cuda")
    out = (ids, counts, flags, planes)
    for _ in range(3):
        _lib.movegen_encode(boards, out=out)
    times = []
    for _ in range(10):
        planes.view(torch.int16).fill_(-1)  # poison: 22 GB written, also flushes L2
        ids.fill_(-1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.movegen_encode(boards, out=out)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    mean_legal = float(counts.float().mean())
    bytes_per_pos = 21520 + 2 * mean_legal  # SURVEY.md §8(d)
    avg = sum(times) / len(times)
    gbs = n * bytes_per_pos / avg / 1e6
    # movegen only (planes = NULL)
    t2 = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.movegen_encode(boards, planes=False, out=(ids, counts, flags, None))
        e1.record()
        torch.cuda.synchronize()
        t2.append(e0.elapsed_time(e1))
    # end to end through the C ABI wrapper with HOST buffers (pinned), copies inside the timed region
    m = min(n, 1 << 16)
    h_boards = recs_host[:m].pin_memory()
    h_planes = torch.empty((m, 17, 7, 10, 9), dtype=torch.bfloat16).pin_memory()
    h_ids = torch.empty((m, 128), dtype=torch.int16).pin_memory()
    h_counts = torch.empty((m,), dtype=torch.int16).pin_memory()
    h_flags = torch.empty((m,), dtype=torch.uint8).pin_memory()
    sub = (ids[:m], counts[:m], flags[:m], planes[:m])
    e2e_t = []
    for it in range(4):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        d_boards = boards[:m]
        d_boards.copy_(h_boards, non_blocking=True)
        _lib.movegen_encode(d_boards, out=sub)
        h_ids.copy_(sub[0], non_blocking=True)
        h_counts.copy_(sub[1], non_blocking=True)
        h_flags.copy_(sub[2], non_blocking=True)
        h_planes.copy_(sub[3], non_blocking=True)
        torch.cuda.synchronize()
        if it:
            e2e_t.append(time.perf_counter() - t0)
    e2e_s = sum(e2e_t) / len(e2e_t)
    return {
        "workload": f"configs[1]: movegen + plane encode on {n} perft-3/4 positions from the start position",
        "metric": "movegen positions/sec", "value": n / avg * 1e3, "unit": "positions/s",
        "ms_per_launch": avg, "best_ms": min(times), "mean_legal_moves": mean_legal,
        "movegen_only_positions_per_s": n / (sum(t2) / len(t2)) * 1e3,
        "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": gbs / peaks["hbm_gbs"], "traffic": ncu_traffic("movegen_encode_kernel", n),
                     "algorithmic_bytes_per_launch": n * bytes_per_pos,
                     "bytes_per_position": bytes_per_pos, "peak_source": peaks["source"]},
        "e2e": {"value": m / e2e_s, "unit": "positions/s", "positions": m,
                "h2d_bytes_per_step": m * 96, "d2h_bytes_per_step": m * (21420 + 256 + 3)},
    }


def bench_train(torch, batch: int = 512, steps: int = 5):
    """configs[4]: the PolicyValueNet training step (train.py:130-267 semantics) in bf16, batch 512, on
    synthetic replay rows resident on the device."""
    from chinesechesszero_b200.train import TrainPipeline

    torch.manual_seed(0)
    pipe = TrainPipeline(batch_size=batch)
    g = torch.Generator(device="cuda").manual_seed(0)
    states = (torch.rand((batch, 17, 7, 10, 9), device="cuda", generator=g) > 0.95).float()
    pi = torch.rand((batch, 2086), device="cuda", generator=g) ** 8
    pi = pi / pi.sum(1, keepdim=True)
    z = torch.randint(-1, 2, (batch,), device="cuda", generator=g).float()
    for _ in range(2):
        pipe.train_step(states, pi, z)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = None
    for _ in range(steps):
        last = pipe.train_step(states, pi, z)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"workload": f"configs[4]: PolicyValueNet train step, bf16 autocast, channels_last weights, batch {batch} (old/new "
                        "policy eval, weight+optimizer backup, fwd/bwd, clip 5.0, Adam, KL)", "value": batch / ms * 1e3,
            "unit": "samples/s", "ms_per_step": ms, "loss": last["loss"], "kl": last["kl"]}


def run_own_arm(args):
    import numpy as np
    import torch

    from chinesechesszero_b200 import distributed as D

    rank, local_rank, world = D.shard_info()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    # NCCL writes its version banner to stdout when the first communicator is created; stdout must
    # carry exactly one JSON line, so fd 1 points at stderr while the group comes up
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        D.init("nccl", device=torch.device("cuda", local_rank))
        D.barrier()
        torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)

    from chinesechesszero_b200 import _lib
    from chinesechesszero_b200.net import FLOP_PER_POSITION, BatchedEvaluator, Net
    from chinesechesszero_b200.selfplay import SelfPlayEngine

    peaks = measured_peaks()
    torch.manual_seed(0)  # same random-init weights on every rank (net.py:120 default init)
    net = Net().cuda().eval()
    base_eval = BatchedEvaluator(net, conv_impl=args.conv_impl)
    G, P = args.games, args.playouts

    # per-phase device timing of the lockstep step: events around the forward and around our kernels
    class TimedEvaluator:
        def __init__(self):
            self.pairs = []
            self.conv = []  # (with_skip, start, end) of every K9 launch of the sampled forwards
            self.on = False
            self.needs_planes = base_eval.needs_planes  # False: the stem runs from the board records (K10)

        def __call__(self, planes, leaf_boards):
            if not self.on:
                return base_eval(planes, leaf_boards)
            sample = args.conv_sample > 0 and len(self.pairs) % args.conv_sample == 0
            base_eval.conv_events = self.conv if sample else None
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = base_eval(planes, leaf_boards)
            e1.record()
            base_eval.conv_events = None
            self.pairs.append((e0, e1))
            return out

    ev = base_eval if args.graphs else TimedEvaluator()
    M = max(2, args.max_game_moves)
    stagger = np.arange(G, dtype=np.int64) % M   # slot g behaves as if its current game were `stagger[g]` moves old

    def barrier():
        D.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        return D.max_over_ranks(ms, device="cuda")

    # =========== arm A: `e2e` -- the user-facing pipeline (CollectPipeline.collect_data) ===========
    # per move: search, visit counts / boards / flags read back to pinned host memory, host-side visit softmax + seeded
    # Dirichlet choice, chosen moves uploaded, re-root, terminal test, slot refill; every game that finishes is packed
    # by K8 (one upload, one launch, one read-back per chunk) and written to data.h5 (reference layout, gzip) by the
    # writer thread.  The timed region ends when the file is flushed.
    import shutil
    import tempfile

    from chinesechesszero_b200.collect import CollectPipeline

    tmp_dir = None
    replay_dir = args.replay_dir
    if replay_dir is None and not args.no_replay:
        replay_dir = tmp_dir = tempfile.mkdtemp(prefix=f"ccz_bench_rank{rank}_")
    pipe = CollectPipeline(n_games=G, n_playout=P, data_dir=replay_dir or tempfile.gettempdir(), states_mode="per_move",
                           seed=D.rank_seed(1234, rank), node_cap=args.nodes_per_game, max_game_moves=M, rank=rank, world=world,
                           write_h5=not args.no_replay, write_npy=False, evaluator=ev)
    pipe.load_model()
    eng = pipe.engine
    if args.graphs:
        eng.search.enable_graphs(ev)
    eng.move_count[:] = stagger
    e2e_warmup = min(args.warmup, 2)  # first-call costs only (the staggered slots are in steady state from move 1);
    for _ in range(e2e_warmup):       # the W warm-up moves of the contract precede the `value` region below
        pipe.collect_data()
    pipe.flush()
    barrier()
    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    h2d0, d2h0 = eng.h2d_bytes + pipe.packer.h2d_bytes, eng.d2h_bytes + pipe.packer.d2h_bytes
    games0 = pipe.iters
    w = pipe.writer
    wr0 = (w.games, w.samples, w.raw_bytes, w.busy_seconds) if w is not None else (0, 0, 0, 0.0)
    file0 = os.path.getsize(pipe.data_path) if (pipe.h5 is not None and os.path.exists(pipe.data_path)) else 0
    pack_launch0 = pipe.packer.launches
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    s0.record()
    for _ in range(args.steps):
        pipe.collect_data()
    pipe.flush()            # replay of every finished game compressed, written and indexed
    s1.record()
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    e2e_dev_ms = s0.elapsed_time(s1)
    e2e_value = world * G * args.steps / e2e_ms * 1e3
    h2d = (eng.h2d_bytes + pipe.packer.h2d_bytes - h2d0) / args.steps
    d2h = (eng.d2h_bytes + pipe.packer.d2h_bytes - d2h0) / args.steps
    pack_launches = pipe.packer.launches - pack_launch0
    replay_info = None
    if w is not None and pipe.h5 is not None:
        file1 = os.path.getsize(pipe.data_path)
        replay_info = {
            "games_written": w.games - wr0[0], "samples_written": w.samples - wr0[1],
            "rows_per_move": (w.samples - wr0[1]) / args.steps, "steady_state_rows_per_move": 2 * G,
            "note": "rows = samples + their mirrored twins; the first max_game_moves moves of a run write shorter games "
                    "(slots start staggered in mid-game), the steady state is 2 x games_per_gpu rows per move",
            "raw_mb_per_s": (w.raw_bytes - wr0[2]) / 1e6 / (e2e_ms / 1e3), "file_mb": (file1 - file0) / 1e6,
            "writer_busy_frac": (w.busy_seconds - wr0[3]) / (e2e_ms / 1e3),
            "format": "reference data.h5 layout (game_{k}/states f16 gzip, mcts_probs f64 gzip, winners f64, attr iters), per-rank shard",
            "k8_launches": pack_launches,
        }
    pool_e2e = eng.pool_events()
    games_finished = pipe.iters - games0
    pipe.close()
    if tmp_dir is not None:
        shutil.rmtree(tmp_dir, ignore_errors=True)
    del pipe, eng
    torch.cuda.empty_cache()

    # =========== arm B: `value` -- the same lockstep move with every input and output resident in HBM ===========
    # visit softmax, Dirichlet mix, sampling, re-root, terminal test and refill on the device, no host synchronisation;
    # the per-move samples go to a device ring that is drained to the host INSIDE the timed region.
    eng = SelfPlayEngine(ev, n_games=G, n_playout=P, nodes_per_game=args.nodes_per_game, seed=D.rank_seed(4321, rank),
                         use_graphs=args.graphs, max_game_moves=M, resident_ring=max(4, min(args.steps, 32)))
    eng._resident_state()["move_count"].copy_(torch.from_numpy(stagger))
    for _ in range(args.warmup):
        eng.play_move_resident()
    eng.resident_backlog.clear()
    eng.drain_resident()
    barrier()
    if not args.graphs:
        ev.on = True
    v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    v0.record()
    for _ in range(args.steps):
        eng.play_move_resident()
    eng.resident_backlog.append(eng.drain_resident())
    v1.record()
    barrier()
    if not args.graphs:
        ev.on = False
    clocks = sampler.stop() if sampler else None
    s0_s1_ms = v0.elapsed_time(v1)
    dev_ms = max_over_ranks(s0_s1_ms)
    value = world * G * args.steps / dev_ms * 1e3
    resident_samples = sum(int(d["boards"].shape[0]) for d in eng.resident_backlog) * G
    if args.dump_outputs and rank == 0:
        # a ring that filled with the last move was drained inside it, leaving the final drain empty
        last = next(d for d in reversed(eng.resident_backlog) if d["boards"].shape[0])
        dump_outputs(args.dump_outputs, {k: v[-1] for k, v in last.items()})
    pool_value = eng.pool_events()
    # K3 for `roofline.mcts`: 64 more playouts so that the trees are a few levels deep, then 50 launches in one event
    # bracket (select only reads the trees and writes the leaf scratch buffers)
    mcts_roof = None
    try:
        sr = eng.search
        sr.run(ev, 64, may_sync=False)
        for _ in range(5):
            _lib.mcts_select(sr.arena, sr.c_puct, sr.leaf_boards, sr.leaf_nodes)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(50):
            _lib.mcts_select(sr.arena, sr.c_puct, sr.leaf_boards, sr.leaf_nodes)
        a1.record()
        torch.cuda.synchronize()
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            k3_ncu = json.load(f).get("mcts_select_kernel", {})
        k3_bytes = (k3_ncu.get("dram_bytes_read", 0) + k3_ncu.get("dram_bytes_write", 0)) * G / k3_ncu.get("positions_per_launch", G)
        k3_gbs = k3_bytes / (k3_ncu["duration_us"] * 1e-6) / 1e9 if k3_ncu.get("duration_us") else None
        mcts_roof = {
            "kernel": "ccz::mcts_select_kernel<1> (K3: child runs staged in shared memory by TMA bulk copies, fp64 PUCT, warp-shuffle argmax)",
            "bound": "latency (two dependent loads per tree level over 4096 warps); HBM is the nominal roofline",
            "ms_per_launch_live": a0.elapsed_time(a1) / 50, "launches_timed": 50,
            "mean_live_nodes_per_game_live": float(sr.arena.n_nodes.float().mean()),
            "traffic": k3_bytes or None, "achieved": k3_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": None if k3_gbs is None else k3_gbs / peaks["hbm_gbs"], "ms_per_launch_ncu": k3_ncu.get("duration_us", 0) / 1e3,
            "issue_active_pct": k3_ncu.get("issue_active_pct"), "warps_active_pct": k3_ncu.get("warps_active_pct"),
            "note": "traffic, achieved GB/s and issue utilisation are those of the committed ncu capture (one launch on trees of "
                    "~23k nodes per game, profiles/r02_mcts_select_expand_ncu.csv); the live duration is on this run's shallower trees",
        }
    except Exception as e:  # noqa: BLE001 - an auxiliary figure must never cost the bench line
        mcts_roof = {"error": repr(e)}
    if args.graphs:
        # events cannot sit inside a captured graph: attribute the whole step to the forward, which
        # gives a lower bound on its throughput (its live share is 0.99 in the eager run)
        fwd_ms = [s0_s1_ms / (args.steps * P)]
        conv_ms = []
    else:
        fwd_ms = [a.elapsed_time(b) for a, b in ev.pairs]
        conv_ms = [(sk, a.elapsed_time(b)) for sk, a, b in ev.conv]
        ev.pairs, ev.conv = [], []
    fwd_avg = sum(fwd_ms) / len(fwd_ms)
    n_fwd = len(fwd_ms)

    if rank != 0:
        D.barrier()
        D.shutdown()
        return

    tflops = G * FLOP_PER_POSITION / fwd_avg / 1e9
    peak_tf = peaks["bf16_tflops_sustained"]
    step_share = None if args.graphs else fwd_avg * n_fwd / s0_s1_ms
    forward = {"kernel": f"bf16 Net.forward over the leaf batch (conv_impl={base_eval.conv_impl}: 3x3 tower on "
                         + ("K9 ccz::conv3x3_c256_kernel" if base_eval.conv_impl.startswith("k9") else "cuDNN")
                         + (", stem on K10 ccz::stem::stem_lookup_kernel from the board records" if not base_eval.needs_planes
                            else ", stem through cuDNN") + ", 1x1 heads + FC layers as cuBLAS GEMMs)",
               "achieved": tflops, "unit": "TFLOP/s", "frac": tflops / peak_tf, "flop_per_launch": G * FLOP_PER_POSITION,
               "ms_per_launch": fwd_avg, "launches_timed": n_fwd, "share_of_step": step_share}
    conv_flop = 2.0 * G * 90 * 256 * 2304  # one 3x3 256->256 convolution over G boards
    if not args.graphs and conv_ms:
        # dominant kernel = K9: mean duration of the launches bracketed inside the timed region
        k_avg = sum(t for _, t in conv_ms) / len(conv_ms)
        k_plain = [t for sk, t in conv_ms if not sk]
        k_skip = [t for sk, t in conv_ms if sk]
        per_fwd = len(conv_ms) / max(1, (n_fwd + args.conv_sample - 1) // args.conv_sample)
        roof = {"bound": "tensor", "achieved": conv_flop / k_avg / 1e9, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": conv_flop / k_avg / 1e9 / peak_tf, "traffic": ncu_traffic("conv3x3_c256_kernel", G),
                "kernel": "ccz::conv3x3_c256_kernel (K9: tcgen05 implicit GEMM, TMA im2col, bias+skip+ReLU epilogue)",
                "flop_per_launch": conv_flop, "ms_per_launch": k_avg, "launches_timed": len(conv_ms),
                "launches_per_forward": per_fwd,
                "ms_plain": sum(k_plain) / len(k_plain) if k_plain else None,
                "ms_with_skip": sum(k_skip) / len(k_skip) if k_skip else None,
                "share_of_step": k_avg * per_fwd * n_fwd / s0_s1_ms,
                "peak_source": peaks["source"] + " sustained", "forward": forward}
    else:
        roof = {"bound": "tensor", "achieved": tflops, "peak": peak_tf, "unit": "TFLOP/s", "frac": tflops / peak_tf,
                "traffic": None, "peak_source": peaks["source"] + " sustained", **{k: v for k, v in forward.items()
                                                                                   if k not in ("achieved", "unit", "frac")}}
    roof["mcts"] = mcts_roof
    k9_per_fwd = {"k9": 80, "k9_skip": 40}.get(base_eval.conv_impl, 0) + (0 if base_eval.needs_planes else 1)  # + K10
    line = {
        "metric": metric_name(P), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic (random-init net, torch.manual_seed(0); games from the start position)",
        "config": {
            "workload": workload_name(G, P),
            "games_per_gpu": G, "n_playout": P, "cuda_graphs": bool(args.graphs), "max_game_moves": M,
            "slots": "games are cut after max_game_moves and the slots start staggered: G / max_game_moves games finish (and are "
                     "replaced from the start position) with every move, the steady state of a long run",
            "resident_samples_drained_in_timed_region": resident_samples, "parallelism": f"games sharded x{world}, "
            "no collective on the hot path",
            "l2": "per-layer activations 4096x256x90 bf16 = 189 MB > 126 MB L2 (inputs larger than L2)",
            "step": "one lockstep move = n_playout x (select, movegen+encode, bf16 forward, expand+backup) + move "
                    "choice + re-root + terminal test + slot refill",
        },
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / args.steps, "games_finished": games_finished, "replay": replay_info,
                "api": "collect.CollectPipeline.collect_data() (the reference's collect.py entry point): SelfPlayEngine.play_move() "
                       "-- per-move visit counts / boards / flags read back to pinned host memory, host-side visit softmax + "
                       "seeded Dirichlet choice, chosen moves uploaded -- then K8 replay packing of the finished games and the "
                       "reference-layout data.h5 shard written by the writer thread, flushed inside the timed region"},
        # `value` region: per playout K3 select, K1 movegen, K4/K5 expand+backup, K10 stem, 80 x K9; per move the reserve
        # guard, K6 root read-out, K7a/K7b advance, K1 flags, reset
        "gpu_launches": args.steps * (P * (3 + k9_per_fwd) + 6),
        "pool": {"e2e": pool_e2e, "value": pool_value,
                 "note": "shared MCTS page pool (csrc/ccz_mcts.cuh): expand_failed / trees_dropped must be 0"},
        "roofline": roof,
        "e2e_warmup": e2e_warmup,
        "clocks": clocks,
        "evals_per_move": P,
    }
    del eng
    torch.cuda.empty_cache()
    # configs[1] / configs[4] / the CPU baseline ride along at N = 1 only (the scaling runs time self-play)
    if not args.no_movegen and world == 1:
        line["movegen"] = bench_movegen(torch, _lib, args.movegen_positions, peaks)
    if not args.no_train and world == 1:
        line["train"] = bench_train(torch)
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline(args.cpu_moves, P)
    print(json.dumps(line))
    D.barrier()
    D.shutdown()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_own_arm(args)


if __name__ == "__main__":
    main()
