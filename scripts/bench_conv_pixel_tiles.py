"""A/B of K9's tilings in one process: pixel tiles (variant 128, the bf16 default) against tiles of 256 consecutive
pixels (variant 2, the tiling before pixel tiles and still the e4m3 default), bf16 and e4m3, plain and with the skip
input.

Sizes: 4096 boards (the bench's games) and 3760 boards (about the bench's unique leaves per step, U, that
scripts/bench_leaf_dedup.py reports).  The two tilings alternate within every repeat, so clock and power drift hits both
alike; each sample is the mean over `--launches` back-to-back launches bracketed by CUDA events.  The activations are
larger than L2 (189 MB of bf16 input at 4096 boards).  Reports ms per launch (median, min, max over the repeats), the
new / old ratio of the medians, TFLOP/s counted as bench.py counts them (2 * 90 * 256 * 2304 per board, padding
included) and as the pixel tiles issue them (700 / 810 of that), the card's name and power limit.

    python scripts/bench_conv_pixel_tiles.py [--repeats 15] [--launches 100] [--out result.json]
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

FLOP_PER_BOARD = 2 * 90 * 256 * 2304
ISSUED = 700 / 810  # in-board (pixel, tap) pairs of a 10x9 board with pad 1
CL = torch.channels_last
VARIANTS = {"pixel": _lib.CONV_VARIANT_PIXEL, "consecutive": _lib.CONV_VARIANT_PAIR}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, launches):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 3760])
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_conv_pixel_tiles needs a CUDA device")

    torch.manual_seed(0)
    n_max = max(args.sizes)
    x = torch.randn(n_max, 256, 10, 9, device="cuda").relu().to(torch.bfloat16).contiguous(memory_format=CL)
    skip = torch.randn(n_max, 256, 10, 9, device="cuda").to(torch.bfloat16).contiguous(memory_format=CL)
    out = torch.empty_like(x, memory_format=CL)
    w = (torch.randn(256, 256, 3, 3, device="cuda") * 0.03).to(torch.bfloat16).contiguous(memory_format=CL)
    bias = torch.randn(256, device="cuda") * 0.1
    xq = (x.float() * 4).to(_lib.E4M3).contiguous(memory_format=CL)
    wq = (w.float() * 64).to(_lib.E4M3).contiguous(memory_format=CL)
    deq = torch.full((256,), 1 / 256, device="cuda")
    inv = torch.tensor([1.0], device="cuda")
    outq = torch.empty_like(xq, memory_format=CL)

    def case(dtype, n, with_skip, variant):
        sk = skip[:n] if with_skip else None
        if dtype == "bf16":
            return lambda: _lib.conv3x3_c256(x[:n], w, bias, sk, out=out[:n], variant=variant)
        return lambda: _lib.conv3x3_c256_e4m3(xq[:n], wq, deq, bias, skip=sk, out=out[:n], out_q=outq[:n], inv_s_out=inv,
                                              variant=variant)

    results = {"card": card(), "launches_per_sample": args.launches, "repeats": args.repeats, "cases": []}
    for dtype in ("bf16", "e4m3"):
        for n in args.sizes:
            for with_skip in (False, True):
                fns = {k: case(dtype, n, with_skip, v) for k, v in VARIANTS.items()}
                for fn in fns.values():
                    timed(fn, 10)
                ms = {k: [] for k in fns}
                for _ in range(args.repeats):
                    for k, fn in fns.items():
                        ms[k].append(timed(fn, args.launches))
                row = {"dtype": dtype, "boards": n, "skip": with_skip}
                for k, v in ms.items():
                    med = float(np.median(v))
                    row[k] = {"ms_median": round(med, 5), "ms_min": round(min(v), 5), "ms_max": round(max(v), 5),
                              "tflops_counted": round(FLOP_PER_BOARD * n / med / 1e9, 1)}
                row["pixel"]["tflops_issued"] = round(FLOP_PER_BOARD * ISSUED * n / row["pixel"]["ms_median"] / 1e9, 1)
                row["new_over_old"] = round(row["pixel"]["ms_median"] / row["consecutive"]["ms_median"], 4)
                results["cases"].append(row)
                print(json.dumps(row), flush=True)
    print(json.dumps({"card": results["card"]}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
