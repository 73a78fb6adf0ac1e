"""Short launch sequence for `ncu --set full`: K10 (stem lookup) and K9 (plain / with skip) at 4096 boards."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from chinesechesszero_b200 import _lib
from chinesechesszero_b200.net import Net, BatchedEvaluator

n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
torch.manual_seed(0)
ev = BatchedEvaluator(Net(resblocks_num=1).cuda().eval(), conv_impl="k9", dedup=False)
boards = torch.empty(n, 96, dtype=torch.uint8, device="cuda")
_lib.check(_lib.load().ccz_boards_start(boards.data_ptr(), n, _lib.stream_ptr()), "boards_start")
for _ in range(3):
    x = _lib.stem_lookup(boards, *ev.stem_lookup)
    (w1, _, b1), (w2, _, b2) = ev.blocks[0]
    y = _lib.conv3x3_c256(x, w1, b1)
    _lib.conv3x3_c256(y, w2, b2, skip=x, out=x)
torch.cuda.synchronize()
print("ok")
