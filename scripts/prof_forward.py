"""Two evaluator forwards at G leaves (ncu launch list: skip the first forward's launches)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from chinesechesszero_b200 import _lib
from chinesechesszero_b200.net import Net, BatchedEvaluator
G = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
torch.manual_seed(0)
ev = BatchedEvaluator(Net().cuda().eval(), dedup=False)  # G copies of one board: time G boards, not one
boards = torch.empty(G, 96, dtype=torch.uint8, device="cuda")
_lib.check(_lib.load().ccz_boards_start(boards.data_ptr(), G, _lib.stream_ptr()), "boards_start")
ids, counts, flags, planes = _lib.movegen_encode(boards)
for _ in range(2):
    logits, pk, v = ev(planes, boards)
torch.cuda.synchronize()
print("ok", float(v[0]))
