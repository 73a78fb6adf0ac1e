"""Whole-forward time of the 40x256 evaluator per conv implementation (steady state, one GPU)."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from chinesechesszero_b200.net import Net, BatchedEvaluator, FLOP_PER_POSITION

G = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
impls = sys.argv[2:] or ["cudnn", "k9_skip", "k9"]
torch.manual_seed(0)
net = Net().cuda().eval()
from chinesechesszero_b200 import _lib
boards = torch.empty(G, 96, dtype=torch.uint8, device="cuda")
_lib.check(_lib.load().ccz_boards_start(boards.data_ptr(), G, _lib.stream_ptr()), "boards_start")
planes = _lib.movegen_encode(boards)[3]
USE_BOARDS = bool(os.environ.get("BOARDS"))
ref = None
for impl in impls:
    impl, _, chunk = impl.partition(":")
    ev = BatchedEvaluator(net, conv_impl=impl, chunk=int(chunk or 0), dedup=False)  # G copies of one board
    for _ in range(3):
        logits, v = ev.forward(planes, boards if USE_BOARDS else None)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    run = lambda: ev.forward(planes, boards if USE_BOARDS else None)
    if os.environ.get("GRAPH"):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            logits, v = ev.forward(planes, boards if USE_BOARDS else None)
        run = gr.replay
        for _ in range(10):
            run()
    e0.record()
    for _ in range(30):
        run()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 30
    p = torch.softmax(logits, 1)
    if ref is None:
        ref = (p, v)
    print(json.dumps({"conv_impl": impl, "chunk": ev.chunk, "batch": G, "ms": ms, "tflops": G * FLOP_PER_POSITION / ms / 1e9, "moves_per_s_at_400": 1e3 * G / (400 * ms),
                      "max_dp_vs_first": (p - ref[0]).abs().max().item(), "max_dv_vs_first": (v - ref[1]).abs().max().item()}), flush=True)
