"""SI-Finder cost of the two matching modes (Pearson, and L2 + LAB = ae_config.use_L2andLAB) in one process.

    python tools/sif_l2_bench.py [--batches 8 32] [--reps 5] [--steps 4] [--warmup 3]

For each batch size: device-resident synthetic 320x1224 pairs (as bench.py --workload sif), both modes warmed up,
then `reps` rounds that alternate Pearson and L2, each round timing `steps` calls of match_images (prepare + match +
gather) with CUDA events; the match kernels alone are timed by the ops profiler (sif_match / sif_match_l2).  The
working set (~0.5 GB of fp16 operands per 8 pairs) exceeds L2, so every pass reads HBM.  One JSON line per batch
size: ms per pair (median over rounds, and the spread), algorithmic TFLOP/s at 849.6 GFLOP per pair, the L2 / Pearson
ratio, the exhaustive work-list size of each mode, the GPU name and its power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, W, PH, PW = 320, 1224, 20, 24
FLOP_PER_PAIR = 2.0 * (H - PH + 1) * (W - PW + 1) * (H // PH) * (W // PW) * (PH * PW * 3)  # 849.6e9


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["clocks_max_sm"] = [s.strip() for s in out.split(",")]
    except Exception as e:  # noqa: BLE001 -- the numbers are still valid, only unlabelled
        info["power_limit"] = "unknown (%s)" % e
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[8, 32])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("a CUDA device is required: this measures GPU time")
    from dsin_b200 import ops, synth
    from dsin_b200.siFinder import match_images
    info = gpu_info()
    mode = {"pearson": None, "l2": type("Cfg", (), {"use_L2andLAB": True})()}
    for B in args.batches:
        x, y = synth.make_batch(4, H, W, seed=77)
        reps = (B + 3) // 4
        xd = torch.tensor(np.concatenate([x] * reps)[:B]).cuda().permute(0, 2, 3, 1).contiguous()
        yd = torch.tensor(np.concatenate([y] * reps)[:B]).cuda().permute(0, 2, 3, 1).contiguous()
        for cfg in mode.values():
            for _ in range(args.warmup):
                match_images(xd, yd, yd, PH, PW, True, cfg)
        torch.cuda.synchronize()
        ms = {k: [] for k in mode}
        kern = {k: [] for k in mode}
        for _ in range(args.reps):
            for name, cfg in mode.items():
                ops.PROF.start()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    match_images(xd, yd, yd, PH, PW, True, cfg)
                e1.record()
                torch.cuda.synchronize()
                ops.PROF.stop()
                ms[name].append(e0.elapsed_time(e1) / (args.steps * B))
                kern[name].append(ops.PROF.summary()["sif_match_l2" if cfg else "sif_match"]["ms"] / (args.steps * B))
        # exhaustive work-list size of one call of each mode
        work_items = {}
        for name, cfg in mode.items():
            q, r, ps, ys = ops.sif_prepare(xd, yd, PH, PW, lab=cfg is not None)
            work = torch.empty(ops.sif_workspace_bytes(B, H, W, PH, PW, 1), dtype=torch.uint8, device="cuda")
            ops.sif_match(q, r, ps, ys, PH, PW, use_mask=True, method=1, l2=cfg is not None, work=work)
            work_items[name] = ops.sif_work_count(work, B, H, W, PH, PW)
        out = {"workload": "match_images 320x1224, prior on, synthetic pairs", "batch": B, "reps": args.reps,
               "steps_per_rep": args.steps, **info, "gflop_per_pair": FLOP_PER_PAIR / 1e9}
        for name in mode:
            med, kmed = float(np.median(ms[name])), float(np.median(kern[name]))
            out[name] = {"ms_per_pair": med, "ms_per_pair_min": float(min(ms[name])),
                         "ms_per_pair_max": float(max(ms[name])), "match_kernels_ms_per_pair": kmed,
                         "tflops_match_images": FLOP_PER_PAIR / (med * 1e-3) / 1e12,
                         "tflops_match_kernels": FLOP_PER_PAIR / (kmed * 1e-3) / 1e12,
                         "exhaustive_work_items": work_items[name]}
        out["ratio_l2_over_pearson"] = out["l2"]["ms_per_pair"] / out["pearson"]["ms_per_pair"]
        out["ratio_l2_over_pearson_match_kernels"] = (out["l2"]["match_kernels_ms_per_pair"]
                                                      / out["pearson"]["match_kernels_ms_per_pair"])
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
