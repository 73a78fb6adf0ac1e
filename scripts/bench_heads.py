"""A/B of the operand packing between the 1x1 heads and the FC layers: K11 (csrc/ccz_heads.cuh) vs the three torch
launches it replaces, as whole-forward time of the 40x256 evaluator at the lockstep batch size, alternating in one process."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from chinesechesszero_b200 import _lib
from chinesechesszero_b200.net import BatchedEvaluator, Net

G = int(os.environ.get("CCZ_G", "4096"))
torch.manual_seed(0)
ev = BatchedEvaluator(Net().cuda().eval(), dedup=False)  # G copies of one board: time G boards, not one
boards = _lib.boards_start(G)
res = {"k11": [], "torch": []}
for rnd in range(4):
    for name, flag in (("k11", True), ("torch", False)):
        ev.use_heads_pack = flag
        for _ in range(10):
            ev.forward(None, boards)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(40):
            ev.forward(None, boards)
        e1.record()
        torch.cuda.synchronize()
        res[name].append(e0.elapsed_time(e1) / 40)
ev.use_heads_pack = True
a = ev.forward(None, boards)
ev.use_heads_pack = False
b = ev.forward(None, boards)
print(json.dumps({"boards": G, "forward_ms_k11": res["k11"], "forward_ms_torch": res["torch"],
                  "identical_outputs": bool(torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]))}))
