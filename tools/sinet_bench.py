"""Timing of the SI-Net (src/siNet.py:29-41) on 320x1224 images at batch B on one box: ms per SI-Net pass, then ms per
3x3 layer for all nine layers (by dilation) as the dispatch runs them, one JSON line each.  The first layer is timed
on an input with 6 live channels, as in the network.

    python tools/sinet_bench.py [--batch 32] [--reps 20] [--root DIR] [--label NAME]

--root times the package of another tree (for example a checkout of an earlier commit with its library built) with
this same script, so that two builds can be compared line for line on one box."""
import argparse
import json
import os
import sys

import torch

p = argparse.ArgumentParser()
p.add_argument("--batch", type=int, default=32)
p.add_argument("--reps", type=int, default=20)
p.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
p.add_argument("--label", default="")
args = p.parse_args()
ROOT = os.path.abspath(args.root)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from parity_utils import make_ae  # noqa: E402
from dsin_b200 import ops, siNet as sn, synth  # noqa: E402


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    B, H, W = args.batch, 320, 1224
    dev = torch.cuda.get_device_properties(0)
    common = {"label": args.label, "root": os.path.basename(ROOT), "gpu": dev.name, "batch": B, "hw": [H, W]}
    ae = make_ae(H, W, synth.make_weights(0, residual_gamma=0.25))
    a = torch.rand(B, H, W, 3, device="cuda") * 255
    b = torch.rand(B, H, W, 3, device="cuda") * 255
    ms = timed(lambda: ae._siNet.fused(a, b, terms=3), args.reps)
    print(json.dumps(dict(common, what="sinet_pass", ms=round(ms, 4), ms_per_pair=round(ms / B, 5))), flush=True)
    net = ae._siNet
    x = torch.randn(B, H, W, 32, device="cuda")
    x6 = x.clone()
    x6[..., 6:] = 0
    cur, cur6 = ops.f32_to_split(x), ops.f32_to_split(x6)
    total = 0.0
    for li, rate in enumerate(sn.SiNet.RATES):
        tcl = net._tc_first if li == 0 else net._tc[li - 1]
        inp = cur6 if li == 0 else cur
        ms = timed(lambda: ops.conv_tc(inp, tcl, terms=3), args.reps)
        total += ms
        print(json.dumps(dict(common, what="layer", layer=li + 1, dilation=rate, ms=round(ms, 4),
                              ms_per_pair=round(ms / B, 5))), flush=True)
    print(json.dumps(dict(common, what="nine_layers", ms=round(total, 4), ms_per_pair=round(total / B, 5))), flush=True)


if __name__ == "__main__":
    main()
