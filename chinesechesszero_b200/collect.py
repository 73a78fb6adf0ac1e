"""Reference-shaped façade of ``collect.py`` (collect.py:26-198): the self-play data pipeline.

``CollectPipeline(init_model).run()`` keeps the reference's shape -- load the model (random init when
the file is missing, collect.py:49-56), play, preprocess + mirror (collect.py:64-131), append to the
replay store, bump the game counter -- but plays ``n_games`` games concurrently in lockstep on the
GPU (``selfplay.SelfPlayEngine``) and lets K8 do the densification.  Games are appended in the order
they finish; each finished game becomes one ``game_{k}`` unit exactly like one reference iteration.

Outputs (both in the reference's layouts):
  * ``<data_dir>/data.h5``  -- group ``game_{k}`` with ``states`` / ``mcts_probs`` (gzip) / ``winners`` and
    the root attribute ``iters`` (collect.py:146-167), written by ``h5lite`` (no h5py/libhdf5 here);
  * ``<data_dir>/states.npy, mcts.npy, winners.npy, meta.json`` -- what convert.py makes of that file and
    what the trainer reads (convert.py:85-99, train.py:95-100).
Multi-GPU: every rank writes its own ``<data_dir>/rank{r}/`` shard with disjoint ``game_{k}`` numbers
(``distributed.global_game_index``); ``merge_h5_shards`` folds them into one file.
"""
from __future__ import annotations

import argparse
import os

from . import distributed, h5lite, replay
from .net import PolicyValueNet
from .parameters import C_PUCT, DATA_DIR, MODEL_DIR, PLAYOUT
from .selfplay import SelfPlayEngine


class CollectPipeline:
    def __init__(self, init_model=None, n_games=4096, n_playout=PLAYOUT, c_puct=C_PUCT, data_dir=DATA_DIR,
                 states_mode="reference", seed=0, node_cap=None, max_game_moves=None, net_kwargs=None,
                 write_h5=True, write_npy=True, rank=0, world=1, gzip_level=4, h5_flush_every=None,
                 async_writer=True, evaluator=None, precision="bf16"):
        self.temp = 1.0
        self.n_playout = n_playout
        self.c_puct = c_puct
        self.init_model = init_model
        self.n_games = n_games
        self.episode_len = 0
        self.policy_value_net = None
        self.engine = None
        self._evaluator = evaluator  # a ready device evaluator instead of loading a model (benchmarks, tests)
        self.precision = precision  # of the evaluator built over the loaded model: "bf16" or "fp8" (BatchedEvaluator)
        self.rank, self.world = int(rank), int(world)
        self.data_dir = data_dir if self.world == 1 else os.path.join(data_dir, f"rank{self.rank}")
        self.data_path = os.path.join(self.data_dir, "data.h5")
        self.states_mode = states_mode
        self.seed = distributed.rank_seed(seed, self.rank)
        self.node_cap = node_cap
        self.max_game_moves = max_game_moves
        self.net_kwargs = net_kwargs or {}
        self.npy = replay.NpyReplayWriter(self.data_dir) if write_npy else None
        self.h5 = h5lite.H5ReplayWriter(self.data_path, gzip_level=gzip_level, flush_every=h5_flush_every) if write_h5 else None
        # collect.py:39-45: the game counter continues from the file.  One GPU: the ``iters`` attribute.  A shard of
        # a multi-GPU run holds every world-th game number, so its own count is the number of groups it links.
        if self.h5 is None:
            self.local_games = 0
        elif self.world == 1:
            self.local_games = self.h5.iters
        else:
            self.local_games = self.h5.n_groups
        self.iters = self.local_games
        self.packer = None
        # compression + file writes happen on a worker thread; ``async_writer=False`` keeps them inline
        self.writer = replay.AsyncReplayWriter(self.h5, self.npy) if async_writer else None

    def load_model(self):
        """collect.py:47-62: load once; fall back to random init when the model cannot be loaded."""
        if self.engine is None:
            if self._evaluator is not None:
                evaluator = self._evaluator
            else:
                model_path = self.init_model if self.init_model else os.path.join(MODEL_DIR, "current_policy.pkl")
                try:
                    self.policy_value_net = PolicyValueNet(model=model_path, **self.net_kwargs)
                except Exception:
                    self.policy_value_net = PolicyValueNet(**self.net_kwargs)
                evaluator = self.policy_value_net.evaluator(precision=self.precision)
            self.engine = SelfPlayEngine(evaluator, n_games=self.n_games, n_playout=self.n_playout,
                                         c_puct=self.c_puct, temp=self.temp, seed=self.seed,
                                         node_cap=self.node_cap, max_game_moves=self.max_game_moves)
            self.packer = replay.ReplayPacker(self.engine.device, self.states_mode)

    def collect_data(self, is_shown=False):
        """One lockstep move in every game slot; the games that finish with it are packed together
        (preprocess + flip, collect.py:141-142: one upload, one K8 launch, one read-back per chunk) and
        handed to the writer thread.  Returns the running game count (collect.py:176)."""
        self.load_model()
        finished = self.engine.play_move()
        if finished:
            for chunk in self.packer.pack(finished):
                n = len(chunk.spans)
                indices = None
                if self.world > 1:
                    indices = [distributed.global_game_index(self.local_games + i, self.rank, self.world) for i in range(n)]
                if self.writer is not None:
                    self.writer.submit(chunk, indices)
                else:
                    for k in range(n):
                        states, probs, winners = chunk.game_arrays(k)
                        if self.h5 is not None:
                            self.h5.add(states, probs, winners, index=None if indices is None else indices[k])
                        if self.npy is not None:
                            self.npy.add(states, probs, winners)
                    chunk.release()
                self.local_games += n
            self.episode_len = len(finished[-1])
            self.iters = self.local_games
        return self.iters

    def flush(self):
        """Everything collected so far is on disk and indexed (the trainer may open the files)."""
        if self.writer is not None:
            self.writer.drain()
        else:
            if self.h5 is not None:
                self.h5.flush()
            if self.npy is not None:
                self.npy.flush()

    def run(self, is_shown=False, max_games=None):
        first = self.iters
        try:
            while max_games is None or self.iters - first < max_games:
                self.collect_data(is_shown=is_shown)
        except KeyboardInterrupt:
            pass
        finally:
            self.close()
        return self.iters

    def pool_events(self) -> dict:
        """Counters of the MCTS page pool (``trees_dropped`` / ``expand_failed`` are 0 unless the pool could not grow)."""
        return self.engine.pool_events() if self.engine is not None else {}

    def close(self):
        if self.writer is not None:
            self.writer.close()
            self.writer = None
        if self.npy is not None:
            self.npy.close()
            self.npy = None
        if self.h5 is not None:
            self.h5.close()
            self.h5 = None


def merge_h5_shards(shard_paths, out_path, gzip_level=4):
    """Fold per-rank ``data.h5`` shards into one file numbered game_0.. in increasing shard index
    order (rank-interleaved, as ``global_game_index`` assigned them).  Every shard is opened once and the
    stored (deflated) datasets are copied as they are, so merging costs file I/O, not a second compression."""
    readers = [h5lite.H5Reader(p) for p in shard_paths]
    try:
        games = []
        for ri, r in enumerate(readers):
            for name in r.root_links():
                games.append((int(name.split("_")[1]), ri, name))
        games.sort()
        out = h5lite.H5ReplayWriter(out_path, gzip_level=gzip_level)
        for _, ri, name in games:
            out.add_raw(readers[ri].read_group_raw(name))
        n = out.iters
        out.close()
    finally:
        for r in readers:
            r.close()
    return n


if __name__ == "__main__":
    parser = argparse.ArgumentParser(description="collect Xiangqi self-play data on the GPU")
    parser.add_argument("--show", action="store_true", default=False)
    parser.add_argument("--model", type=str, default="current_policy.pkl")
    parser.add_argument("--games", type=int, default=4096)
    parser.add_argument("--max-games", type=int, default=None)
    args = parser.parse_args()
    rank, local_rank, world = distributed.shard_info()
    CollectPipeline(init_model=args.model, n_games=args.games, rank=rank, world=world).run(
        is_shown=args.show, max_games=args.max_games)
