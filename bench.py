#!/usr/bin/env python
"""bench.py -- DSIN inference hot path on B200 (one JSON line on stdout, rank 0).

  python bench.py --gpus N --steps K --warmup W            our CUDA path (libdsin_b200)
  python bench.py --impl reference ...                      the reference arithmetic on host cores
  python bench.py ... --dump-outputs DIR                    also write the last timed step's outputs to DIR/*.npy

A "step" is one AE.siNet_get_reconstructed-equivalent pass (AE(y), AE(x), bpp, SI-Finder, SI-Net;
/root/reference/src/AE.py:132-148) over one batch of synthetic 320x1224 pairs.

Default workload = BASELINE.json configs[4]: ONE global batch of 256 pairs per step, sharded over the N ranks with
dist.shard_range (256 / 128 / 64 / 32 pairs per GPU at N = 1 / 2 / 4 / 8: strong scaling) and processed in
micro-batches of 32 pairs -- at N = 1 this is north_star's "batch 32, 320x1224, 1xB200" operating point.
`--batch B` instead fixes B pairs per GPU per step (weak scaling); `--batch 8` is configs[1].
`value` = Mpixels/s with inputs resident in HBM; `e2e` = the same through the public numpy call on plain numpy
uint8 arrays (pageable -> pinned staging, H2D and D2H all inside the timed region).  N>1: one process per GPU
(torchrun), no data-path collective, one NCCL all-gather of per-rank metric partials; timing is the max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 320, 1224  # --hw HxW changes the geometry AND the metric / workload strings that name it
PH, PW = 20, 24
GFLOP_PER_PAIR_FULL = 1893.9  # SURVEY App. B / BASELINE.md section 4 (320x1224; scaled by area for other --hw)
GFLOP_PER_PAIR_DECODE = 1640.0  # decode-side region: AE(y) + decoder(x) + SI-Finder + SI-Net (SURVEY 8d)
GFLOP_PER_IMAGE_ENC_320x960 = 199.1  # configs[3]: encoder + quantiser + probclass (SURVEY App. B)
METRIC = "Mpixels/s decode (320x1224 pairs)"


def set_geometry(hw):
    global H, W, METRIC, GFLOP_PER_PAIR_FULL, GFLOP_PER_PAIR_DECODE
    h, w = (int(v) for v in hw.lower().split("x"))
    if (h, w) != (H, W):
        area = h * w / float(H * W)
        GFLOP_PER_PAIR_FULL *= area      # approximation off the BASELINE geometry (the SI-Finder term is not linear)
        GFLOP_PER_PAIR_DECODE *= area
        H, W = h, w
        METRIC = "Mpixels/s decode (%dx%d pairs; NOT the BASELINE geometry)" % (H, W)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def load_library():
    """libdsin_b200 as __graft_entry__.build() left it.  Nothing is compiled here: the tree may be read-only."""
    import __graft_entry__ as g
    if g._stale():
        sys.exit("bench.py: dsin_b200/libdsin_b200.so is missing or older than its sources; "
                 "run `python -c 'import __graft_entry__ as g; g.build()'` first")
    from dsin_b200 import _lib
    _lib.load()


DUMP_BYTES = 64 << 20


def dump_outputs(path, parts):
    """Writes what the last timed step returned, one dict of CUDA tensors per micro-batch, as path/<name>.npy:
    float64 outputs as float64, all others as float32 (the integer outputs are small enough to be exact).  Each output
    is concatenated over the micro-batches; one with more elements than its share of DUMP_BYTES is written as a
    sample of its flattened elements, at indices drawn with a fixed seed and kept in ascending order, so that two
    runs with the same arguments write the same elements."""
    import torch
    os.makedirs(path, exist_ok=True)
    names = sorted(parts[0])
    cap = DUMP_BYTES // (8 * len(names))  # elements per output, even if all are float64
    for name in names:
        t = torch.cat([p[name] for p in parts])
        if t.numel() > cap:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), cap, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        t = t.to(torch.float64 if t.dtype == torch.float64 else torch.float32)
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sust=p["bf16_tflops_sustained"], src="measured")
    except Exception:  # noqa: BLE001
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler(object):
    """SM clock and throttle reasons sampled DURING the timed region: NVML in-process every 10 ms (an nvidia-smi
    child needs longer to start than a short timed region lasts); nvidia-smi -lms as the fallback."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc, self.nvml, self.handle = gpu_index, [], None, None, None
        self.sm, self.mx, self.reasons, self._stop = [], None, set(), False
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:  # the CUDA ordinal is not the NVML index when CUDA_VISIBLE_DEVICES remaps devices
                uuid = "GPU-" + str(torch.cuda.get_device_properties(gpu_index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:  # noqa: BLE001
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:  # noqa: BLE001
            self.nvml = None

    def _poll(self):
        n = self.nvml
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                mask = int(get_reasons(self.handle))
                for name, bit in self.BITS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.01)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self._stop = True
            self.thread.join(timeout=1)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nme, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:  # noqa: BLE001
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def cpu_info():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return model, os.cpu_count() or 1


def oracle_seconds_per_pair(n_pairs=1, seed=0):
    """Times the CPU oracle (restated reference arithmetic, torch-CPU fp32, all host threads)."""
    import torch
    from dsin_b200 import synth
    from oracle import dsin_oracle as O
    # more threads than ~32 oversubscribe the small convs (measured on the B200 host: 128 threads are
    # 13x slower than 16-32, tools/oracle_thread_sweep.py)
    cores = min(32, os.cpu_count() or 1)
    torch.set_num_threads(cores)
    Wt = synth.make_weights(0, residual_gamma=0.25)
    x, y = synth.make_batch(n_pairs, H, W, seed=1000 + seed)
    t0 = time.perf_counter()
    O.reconstruct(x, y, Wt)
    return (time.perf_counter() - t0) / n_pairs, cores


def run_reference(args, rank):
    """--impl reference: TF1 cannot run here (SURVEY F2/F3), so the reference arm is the oracle's
    restatement of the same arithmetic on the host cores; each step = one 320x1224 pair."""
    if rank != 0:
        return
    model, cores = cpu_info()
    for i in range(1 if args.warmup >= 1 else 0):  # one warm-up pair is enough on CPU
        oracle_seconds_per_pair(1, seed=50 + i)
    times = []
    steps = args.steps
    for i in range(steps):
        s, cores = oracle_seconds_per_pair(1, seed=i)
        times.append(s)
    sec = float(np.mean(times))
    mpix = H * W * 1e-6 / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": mpix, "unit": "Mpixels/s", "n_gpus": args.gpus,
        "gpus_used": 0,
        "steps": steps, "warmup": 1, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "full inference (AE(y)+AE(x)+bpp+SI-Finder+SI-Net), 1 pair of 320x1224 per step; "
                               "restated reference arithmetic (torch-CPU fp32) -- TF 1.11 itself is not runnable",
                   "batch": 1, "H": H, "W": W},
        "cpu_baseline": {"value": mpix, "unit": "Mpixels/s", "cores": cores, "kind": "port",
                         "sample": "%d x 1 pair 320x1224, full inference; CPU: %s" % (steps, model)},
        "e2e": {"value": mpix, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def build_ae(device_index, residual_gamma=0.25, precision=None):
    from dsin_b200 import config_parser, synth
    from dsin_b200.AE import AE
    from dsin_b200.decoder_imgcomp import decoder
    from dsin_b200.encoder_imgcomp import encoder
    from dsin_b200.siFinder import siFinder
    from dsin_b200.siFull_img import SI_full_img
    from dsin_b200.siNet import siNet
    cfg = os.path.join(ROOT, "dsin_b200", "run_configs")
    ae_config, _ = config_parser.parse(os.path.join(cfg, "ae_run_configs"))
    pc_config, _ = config_parser.parse(os.path.join(cfg, "pc_run_configs"))
    Wt = synth.make_weights(0, residual_gamma=residual_gamma)
    ae_config.crop_size = (H, W)
    return AE(ae_config, pc_config, encoder, decoder, siFinder, SI_full_img, siNet, cfg, weights=Wt, precision=precision)


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    load_library()
    if world > 1:
        # NCCL writes its version / debug lines to the C-level stdout when NCCL_DEBUG is set in the environment:
        # point fd 1 at stderr while the communicator comes up, so that stdout carries the one JSON line only
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    from dsin_b200 import ops, precision, synth
    from dsin_b200.dist import gather_metrics, shard_range
    pk = peaks()
    ae = build_ae(local_rank, precision=args.precision)
    if getattr(args, "e2e_chunk", None):
        ae.e2e_chunk = args.e2e_chunk
    dev = torch.device("cuda", local_rank)

    # ---------------- which pairs this rank processes per step ----------------
    if args.batch is not None:     # weak scaling: B pairs per GPU per step (configs[1] = --batch 8)
        n_local, scaling, global_pairs = args.batch, "weak", args.batch * world
        workload = ("BASELINE configs[1]-style: full inference on batch %d of %dx%d pairs per GPU per step"
                    % (args.batch, H, W))
    else:                          # strong scaling: one global batch, contiguous shards (configs[4])
        lo, hi = shard_range(args.global_batch, rank, world)
        n_local, scaling, global_pairs = hi - lo, "strong", args.global_batch
        workload = ("BASELINE configs[4]: full inference on ONE global batch of %d %dx%d pairs per step, sharded "
                    "contiguously over %d GPU(s) (dist.shard_range), micro-batches of %d pairs"
                    % (args.global_batch, H, W, world, args.micro_batch))
    MB = min(args.micro_batch, n_local)
    micro = [MB] * (n_local // MB) + ([n_local % MB] if n_local % MB else [])

    # three distinct micro-batches of inputs per rank, rotated: with the activations of a micro-batch
    # (>= 2 x MB x 12.5 MB per trunk layer) far beyond the 126 MB L2
    NSETS = 3
    host_np, dev_sets = [], []
    for s in range(NSETS):
        x, y = synth.make_batch(MB, H, W, seed=1000 * (rank + 1) + 17 * s)
        # host inputs are plain numpy uint8 NCHW arrays, as the reference's DataProvider delivers them
        # (src/DataProvider.py:197-199)
        host_np.append((np.ascontiguousarray(x.astype(np.uint8)), np.ascontiguousarray(y.astype(np.uint8))))
        dev_sets.append((torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)))

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------- device-resident timing ----------------
    # The timed steps replay the CUDA graphs the public call uses (inputs already in HBM, copied device-to-device
    # into the captured input buffers): eager launching of ~230 kernels per micro-batch is host-bound when eight
    # ranks share a busy host.  The per-kernel breakdown comes from a profiled eager pass after the timed region.
    ae.reconstruct_device(dev_sets[0][0][:micro[0]], dev_sets[0][1][:micro[0]])  # packs the weights
    l0 = ops.launch_count()
    for j, m in enumerate(micro):
        ae.reconstruct_device(dev_sets[j % NSETS][0][:m], dev_sets[j % NSETS][1][:m])
    launches_per_step = ops.launch_count() - l0

    bits_parts = []
    last_step = []  # --dump-outputs: each micro-batch's outputs in the last timed step, less "dec" = [y_dec; x_dec]
    dump = args.dump_outputs is not None and rank == 0

    def step_graph(i, keep=False):
        for j, m in enumerate(micro):
            xd, yd = dev_sets[(i * len(micro) + j) % NSETS]
            out = ae.replay_device(xd[:m], yd[:m])
            if keep:
                bits_parts.append(out["bits_sum"].clone())  # graph outputs are static buffers
            if keep and dump and i == args.steps - 1:
                last_step.append({k: v.clone() for k, v in out.items() if torch.is_tensor(v) and k != "dec"})
        return out

    for i in range(args.warmup):
        step_graph(i)
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    torch.cuda.nvtx.range_push("timed")  # `ncu --nvtx --nvtx-include "timed/"` lists exactly the launches of this region
    for i in range(args.steps):
        step_graph(i, keep=True)
    torch.cuda.nvtx.range_pop()
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    launches = launches_per_step * args.steps
    clocks = sampler.stop() if rank == 0 else None
    if dump:
        dump_outputs(args.dump_outputs, last_step)
        del last_step[:]
    bits_total = float(sum(float(b.sum().item()) for b in bits_parts))
    npix_total = n_local * args.steps * H * W

    # profiled eager pass: CUDA events around every kernel call on the launching stream
    prof_mb = min(len(micro) * args.steps, 3)
    sync_all()
    ops.PROF.start()
    for j in range(prof_mb):
        ae.reconstruct_device(dev_sets[j % NSETS][0][:micro[0]], dev_sets[j % NSETS][1][:micro[0]])
    torch.cuda.synchronize()
    ops.PROF.stop()
    prof = ops.PROF.summary()
    prof_pairs = prof_mb * micro[0]

    # ---------------- decode-side region (SURVEY 8d): receiver only, qbar(x) and y given ----------------
    m0 = micro[0]
    qb_sets = [ae.reconstruct_device(dev_sets[s_][0][:m0], dev_sets[s_][1][:m0])["qbar"].clone() for s_ in range(NSETS)]
    qb_static, y_static = qb_sets[0].clone(), dev_sets[0][1][:m0].clone()
    for i in range(2):  # eager warm-up of the receiver path before capturing it
        ae.decode_side_device(qb_static, y_static)
    torch.cuda.synchronize()
    g_dec = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_dec, capture_error_mode="thread_local"):
        ae.decode_side_device(qb_static, y_static)
    dec_reps = max(1, min(len(micro) * args.steps, 8))

    def step_decode_side(i):
        qb_static.copy_(qb_sets[i % NSETS])
        y_static.copy_(dev_sets[i % NSETS][1][:m0])
        g_dec.replay()

    for i in range(2):
        step_decode_side(i)
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    d0.record()
    for i in range(dec_reps):
        step_decode_side(i)
    d1.record()
    sync_all()
    dec_ms_per_mb = d0.elapsed_time(d1) / dec_reps

    # ---------------- end-to-end timing (public numpy API, plain numpy uint8 arrays) ----------------
    def step_e2e(i):
        for j, m in enumerate(micro):
            xn, yn = host_np[(i * len(micro) + j) % NSETS]
            res = ae.siNet_get_reconstructed(xn[:m], yn[:m])
        return res

    for i in range(min(2, args.warmup)):
        step_e2e(i)
    sync_all()
    t0 = time.perf_counter()
    for i in range(args.steps):
        y_dec, y_syn, x_dec, x_with_si, bpp = step_e2e(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    h2d = 2 * n_local * 3 * H * W * 1  # uint8 images
    d2h = 4 * n_local * 3 * H * W * 4 + 8 * n_local

    # ---------------- quality metrics of the last micro-batch (outside the timed regions) ----------------
    m_last = micro[-1]
    xs_nhwc = ops.nchw_to_nhwc(dev_sets[((args.steps - 1) * len(micro) + len(micro) - 1) % NSETS][0][:m_last].contiguous())
    msssim_sum, msssim_n = 0.0, 0
    if not ae.AE_only:  # the final reconstruction the last end-to-end call returned
        rec_nhwc = ops.nchw_to_nhwc(torch.from_numpy(np.ascontiguousarray(x_with_si)).to(dev)).clamp(0, 255)
        msv = ops.msssim(xs_nhwc, rec_nhwc.contiguous(), form="standard")  # device fp64 MS-SSIM, per image
        msssim_sum, msssim_n = float(np.sum(msv)), int(msv.shape[0])

    # ---------------- reductions over ranks ----------------
    t = torch.tensor([ms, e2e_s * 1e3, dec_ms_per_mb], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    gm = gather_metrics(bits_total, float(npix_total), msssim_sum, msssim_n, device=dev)  # the only collective
    ms_max, e2e_ms_max, dec_ms_max = float(t[0]), float(t[1]), float(t[2])
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    pairs = global_pairs * args.steps
    value = pairs * H * W * 1e-6 / (ms_max * 1e-3)
    e2e_value = pairs * H * W * 1e-6 / (e2e_ms_max * 1e-3)
    dec_value = m0 * world * H * W * 1e-6 / (dec_ms_max * 1e-3)  # every rank runs the receiver micro-batch at once

    # ---------------- roofline of the dominant kernel ----------------
    tot_prof_ms = sum(x["ms"] for x in prof.values())
    top = max(prof.items(), key=lambda kv: kv[1]["ms"]) if prof else None
    kern = {}
    for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
        tf = (v["flops"] / (v["ms"] * 1e-3) / 1e12) if v["ms"] > 0 and v["flops"] else None
        kern[k] = {"ms_per_pair": v["ms"] / prof_pairs, "launches": v["launches"] / prof_mb,
                   "share": v["ms"] / tot_prof_ms, "tflops": tf,
                   "frac_of_bf16_sustained": (tf / pk["tf_sust"]) if tf else None}
    roof = None
    if top is not None:
        name, v = top
        ach = v["flops"] / (v["ms"] * 1e-3) / 1e12
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                ent = json.load(f).get(name, {})
            # the captures were taken at 8 pairs per launch; bytes scale with the pairs one launch processes
            if ent.get("bytes_per_launch"):
                traffic = ent["bytes_per_launch"] * micro[0] / float(ent.get("pairs_per_launch", 8))
        except Exception:  # noqa: BLE001
            pass
        mma_terms = 3 if name.startswith("tc3_") else 1
        roof = {"bound": "tensor", "kernel": name, "achieved": ach, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                "frac": ach / pk["tf_sust"], "traffic": traffic,
                "peak_source": pk["src"] + " bf16 dense sustained (fp16 shares the rate)",
                "mma_terms_per_product": mma_terms, "frac_counting_issued_mma_work": mma_terms * ach / pk["tf_sust"],
                "peak_of_this_precision_mode": pk["tf_sust"] / mma_terms,
                "frac_of_mode_peak": mma_terms * ach / pk["tf_sust"],
                "share_of_step": v["ms"] / tot_prof_ms,
                "avg_launch_ms": v["ms"] / v["launches"],
                "timing": "CUDA events around every launch of this kernel on the launching stream, eager pass of "
                          "%d micro-batch(es) of %d pairs right after the timed region (the timed steps replay CUDA "
                          "graphs)" % (prof_mb, micro[0])}
    whole = pairs / world * GFLOP_PER_PAIR_FULL / (ms_max * 1e-3) / 1e3  # TFLOP/s per GPU, algorithmic

    cpu = None
    if not args.no_cpu_baseline:
        sec, cores = oracle_seconds_per_pair(1)
        model, _ = cpu_info()
        cpu = {"value": H * W * 1e-6 / sec, "unit": "Mpixels/s", "cores": cores, "kind": "port",
               "sample": "1 pair %dx%d full inference, oracle torch-CPU fp32 (%.1f s); CPU: %s" % (H, W, sec, model)}

    line = {
        "metric": METRIC, "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": scaling,
        "vs_baseline": None, "dtype": precision.dtype_string(ae.precision), "data": "synthetic",
        "config": {"workload": workload + ", random-init KITTI_stereo_target_bpp0.02 shapes",
                   "global_batch_per_step": global_pairs, "pairs_per_gpu_per_step": n_local, "micro_batches": micro,
                   "H": H, "W": W, "patch": [PH, PW], "precision_policy": ae.precision.name,
                   "l2": "3 rotating input micro-batches; activations per micro-batch >> 126 MB L2",
                   "parallelism": "dp%d" % world,
                   "timed_region": "K x (replays of the three CUDA graphs per micro-batch), inputs copied device-to-device"},
        "e2e": {"value": e2e_value, "unit": "Mpixels/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms_max / args.steps,
                "inputs": "plain numpy uint8 arrays (pageable), staged through pinned buffers inside the timed call; one call per micro-batch, which the call itself runs as a pipeline of %d-pair chunks when it holds more (staging / H2D / kernels / D2H overlap)" % ae.e2e_chunk},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "regions": {
            "full": {"value": value, "unit": "Mpixels/s", "gflop_per_pair": GFLOP_PER_PAIR_FULL,
                     "what": "encode(x)+bpp + decode-side (the headline `value`)"},
            "decode_side": {"value": dec_value, "unit": "Mpixels/s",
                            "ms_per_micro_batch": dec_ms_max, "micro_batch": m0, "gflop_per_pair": GFLOP_PER_PAIR_DECODE,
                            "tflops_per_gpu": m0 * GFLOP_PER_PAIR_DECODE / (dec_ms_max * 1e-3) / 1e3,
                            "frac_of_bf16_sustained": m0 * GFLOP_PER_PAIR_DECODE / (dec_ms_max * 1e-3) / 1e3 / pk["tf_sust"],
                            "what": "receiver only: AE(y)->y_dec, decoder(qbar_x), SI-Finder, SI-Net"}},
        "whole_path_tflops_per_gpu": whole,
        "whole_path_frac_of_bf16_sustained": whole / pk["tf_sust"],
        "kernels": kern,
        "cpu_baseline": cpu,
        "bpp_aggregate": gm["bpp"], "msssim_mean_last_batch": gm["msssim"], "pairs_processed": pairs,
        "quality_note": "random-init weights: bpp / MS-SSIM are plumbing checks here, parity is in tests/",
    }
    print(json.dumps(line), flush=True)


def run_sif_only(args, rank, world, local_rank):
    """BASELINE configs[2]: SI-Finder (prepare + match + gather) in isolation on device-resident inputs."""
    import torch
    torch.cuda.set_device(local_rank)
    load_library()
    from dsin_b200 import ops, synth
    from dsin_b200.siFinder import match_images
    pk = peaks()
    B = args.batch
    dev = torch.device("cuda", local_rank)
    x, y = synth.make_batch(min(B, 4), H, W, seed=77)
    reps = (B + x.shape[0] - 1) // x.shape[0]
    xd = torch.tensor(np.concatenate([x] * reps)[:B]).to(dev).permute(0, 2, 3, 1).contiguous()
    yd = torch.tensor(np.concatenate([y] * reps)[:B]).to(dev).permute(0, 2, 3, 1).contiguous()
    for _ in range(args.warmup):
        match_images(xd, yd, yd, PH, PW, True)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ops.launch_count()
    ops.PROF.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        match_images(xd, yd, yd, PH, PW, True)
    e1.record()
    torch.cuda.synchronize()
    ops.PROF.stop()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    prof = ops.PROF.summary()
    flops = 2.0 * (H - PH + 1) * (W - PW + 1) * (H // PH) * (W // PW) * (PH * PW * 3) * B * args.steps
    ach = flops / (ms * 1e-3) / 1e12
    mm = prof.get("sif_match", {"ms": ms})
    ach_match = flops / (mm["ms"] * 1e-3) / 1e12
    if rank != 0:
        return
    print(json.dumps({
        "metric": METRIC + " -- SI-Finder only", "value": B * args.steps * H * W * 1e-6 / (ms * 1e-3),
        "unit": "Mpixels/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 coarse + f32/f64 exact rescoring",
        "data": "synthetic", "config": {"workload": "BASELINE configs[2]: SI-Finder prepare+match+gather in isolation, "
                                                    "batch %d of 320x1224" % B, "batch_per_gpu": B},
        "gpu_launches": int(ops.launch_count() - l0), "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "sif_match", "achieved": ach_match, "peak": pk["tf_sust"],
                     "unit": "TFLOP/s", "frac": ach_match / pk["tf_sust"], "traffic": None,
                     "peak_source": pk["src"] + " bf16 dense sustained", "whole_workload_tflops": ach},
    }), flush=True)


def run_enc_only(args, rank, world, local_rank):
    """BASELINE configs[3]: encoder + quantiser + probability model (the sender's rate path: symbols and bpp) on
    batch 64 of 320x960 crops, device-resident inputs; src/AE.py:50-53,85-87."""
    import torch
    torch.cuda.set_device(local_rank)
    load_library()
    if not args.hw:
        set_geometry("320x960")
    from dsin_b200 import ops, precision, synth
    pk = peaks()
    B = args.batch
    ae = build_ae(local_rank, precision=args.precision)
    pol = ae.precision
    dev = torch.device("cuda", local_rank)
    sets = []
    for s in range(3):  # three rotating batches (3 x 64 x 3.7 MB fp32 inputs, activations >> L2)
        x, _ = synth.make_batch(min(B, 8), H, W, seed=4000 + 31 * s)
        reps = (B + x.shape[0] - 1) // x.shape[0]
        sets.append(torch.from_numpy(np.concatenate([x] * reps)[:B]).to(dev))
    pad = ae.pc_imgcomp.auto_pad_value(ae.ae_imgcomp)

    def step(i):
        z = ae.ae_imgcomp.encode(sets[i % 3], terms=pol.enc_x)
        return ae.pc_imgcomp.bitcost(z.qbar, z.symbols, False, pad_value=pad, terms=pol.probclass)

    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ops.launch_count()
    ops.PROF.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        bc = step(i)
    e1.record()
    torch.cuda.synchronize()
    ops.PROF.stop()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    prof = ops.PROF.summary()
    if rank != 0:
        return
    gflop_img = GFLOP_PER_IMAGE_ENC_320x960 * (H * W) / (320.0 * 960.0)
    whole = B * args.steps * gflop_img / (ms * 1e-3) / 1e3
    name, v = max(prof.items(), key=lambda kv: kv[1]["ms"])
    ach = v["flops"] / (v["ms"] * 1e-3) / 1e12
    terms = 3 if name.startswith("tc3_") else 1
    tot = sum(x_["ms"] for x_ in prof.values())
    print(json.dumps({
        "metric": METRIC + " -- encoder + quantiser + probclass only", "value": B * args.steps * H * W * 1e-6 / (ms * 1e-3),
        "unit": "Mpixels/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": precision.dtype_string(pol),
        "data": "synthetic",
        "config": {"workload": "BASELINE configs[3]: encoder + quantiser + probclass bit cost, batch %d of %dx%d crops, "
                               "device-resident inputs, eager launches" % (B, H, W), "batch_per_gpu": B,
                   "precision_policy": pol.name, "l2": "3 rotating input batches; activations per step >> 126 MB L2"},
        "gpu_launches": int(ops.launch_count() - l0), "clocks": clocks,
        "bpp": float(bc._dsin_sum.sum().item()) / (B * H * W),
        "whole_path_tflops": whole, "whole_path_frac_of_bf16_sustained": whole / pk["tf_sust"],
        "roofline": {"bound": "tensor", "kernel": name, "achieved": ach, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                     "frac": ach / pk["tf_sust"], "traffic": None, "mma_terms_per_product": terms,
                     "frac_counting_issued_mma_work": terms * ach / pk["tf_sust"], "share_of_step": v["ms"] / tot,
                     "avg_launch_ms": v["ms"] / v["launches"], "peak_source": pk["src"] + " bf16 dense sustained"},
        "kernels": {k: {"ms_per_step": x_["ms"] / args.steps, "launches_per_step": x_["launches"] / args.steps,
                        "tflops": (x_["flops"] / (x_["ms"] * 1e-3) / 1e12) if x_["flops"] else None}
                    for k, x_ in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])},
    }), flush=True)


def run_codec(args, rank, world, local_rank):
    """SURVEY 8f N3: PC1 entropy coder (range coder driven by the probability model) on the symbols of one batch."""
    import torch
    torch.cuda.set_device(local_rank)
    load_library()
    from dsin_b200 import ops, synth
    B = args.batch
    ae = build_ae(local_rank)
    pc = ae.pc_imgcomp
    centers = ae.ae_imgcomp._centers
    x, y = synth.make_batch(B, H, W, seed=1000)
    out = ae.reconstruct_device(torch.tensor(x).cuda(), torch.tensor(y).cuda())
    sym, est_bits = out["symbols"], float(out["bits_sum"].sum())
    ns = args.streams
    for _ in range(args.warmup):
        b, sizes, _st = ops.pc_encode(sym, centers, pc._codec, ns)
        ops.pc_decode(b, sizes, tuple(sym.shape), centers, pc._codec)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ops.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    enc_ms = dec_ms = 0.0
    for _ in range(args.steps):
        ev[0].record()
        b, sizes, _st = ops.pc_encode(sym, centers, pc._codec, ns)
        ev[1].record()
        back = ops.pc_decode(b, sizes, tuple(sym.shape), centers, pc._codec)
        ev[2].record()
        torch.cuda.synchronize()
        enc_ms += ev[0].elapsed_time(ev[1])
        dec_ms += ev[1].elapsed_time(ev[2])
    clocks = sampler.stop()
    if rank != 0:
        return
    real_bits = 8 * int(sizes.sum())
    mpix = B * args.steps * H * W * 1e-6
    nsym = sym.numel()
    print(json.dumps({
        "metric": METRIC + " -- PC1 entropy coder only", "value": mpix / ((enc_ms + dec_ms) * 1e-3), "unit": "Mpixels/s",
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": (enc_ms + dec_ms) / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (fixed fmaf order) + u32 range coder",
        "data": "synthetic", "config": {"workload": "SURVEY 8f N3: encode + decode of the symbols of batch %d of 320x1224 "
                                                    "(32x40x153 symbols per image), %d streams per image" % (B, ns),
                                        "batch_per_gpu": B, "streams": ns},
        "encode_ms": enc_ms / args.steps, "decode_ms": dec_ms / args.steps,
        "encode_mpix_s": mpix / (enc_ms * 1e-3), "decode_mpix_s": mpix / (dec_ms * 1e-3),
        "symbols_per_s_decode": nsym * args.steps / (dec_ms * 1e-3),
        "gpu_launches": int(ops.launch_count() - l0), "clocks": clocks, "roundtrip_identical": bool(torch.equal(back, sym)),
        "payload_bits": real_bits, "estimated_bits": est_bits, "real_over_estimate": real_bits / est_bits,
        "bpp_real": real_bits / (B * H * W), "bpp_estimate": est_bits / (B * H * W),
        "roofline": {"bound": "latency", "note": "sequential dependence: 4 layers + range coder per wavefront step; "
                     "per step the fmaf chains read 8 B of shared memory per FMA (the measured limiter)",
                     "achieved": None, "peak": None, "unit": None, "frac": None, "traffic": None},
    }), flush=True)


def run_roundtrip(args, rank, world, local_rank):
    """Sender and receiver with real bitstreams through the public numpy API: compress(x) -> bytes;
    decompress(bytes, y) -> y_dec, y_syn, x_dec, x_with_si (host buffers on both sides)."""
    import torch
    torch.cuda.set_device(local_rank)
    load_library()
    from dsin_b200 import synth
    B = args.batch
    ae = build_ae(local_rank)
    x, y = synth.make_batch(B, H, W, seed=1000)
    x8, y8 = x.astype(np.uint8), y.astype(np.uint8)
    for _ in range(args.warmup):
        blobs = ae.compress(x8, nstreams=args.streams)
        ae.decompress(blobs, y8)
    torch.cuda.synchronize()
    t_enc = t_dec = 0.0
    for _ in range(args.steps):
        t0 = time.perf_counter()
        blobs = ae.compress(x8, nstreams=args.streams)
        t1 = time.perf_counter()
        y_dec, y_syn, x_dec, x_with_si = ae.decompress(blobs, y8)
        t2 = time.perf_counter()
        t_enc += t1 - t0
        t_dec += t2 - t1
    ref = ae.siNet_get_reconstructed(x8, y8)
    if rank != 0:
        return
    mpix = B * args.steps * H * W * 1e-6
    nbytes = sum(len(b) for b in blobs)
    print(json.dumps({
        "metric": METRIC + " -- sender/receiver with real bitstreams", "value": mpix / t_dec, "unit": "Mpixels/s",
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_dec / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": ae_dtype(), "data": "synthetic",
        "config": {"workload": "receiver: decompress(bitstreams, y) = PC1 decode + AE(y) + decoder(x) + SI-Finder + SI-Net, "
                               "batch %d of 320x1224, %d streams per image; sender timed beside it" % (B, args.streams),
                   "batch_per_gpu": B, "streams": args.streams},
        "sender_ms_per_step": t_enc / args.steps * 1e3, "sender_mpix_s": mpix / t_enc,
        "receiver_ms_per_step": t_dec / args.steps * 1e3, "receiver_mpix_s": mpix / t_dec,
        "bitstream_bytes_per_batch": nbytes, "bpp_real": 8.0 * nbytes / (B * H * W), "bpp_estimate": float(ref[4]),
        "max_abs_diff_x_with_si_vs_one_call": float(np.abs(np.array(x_with_si) - np.array(ref[3])).max()),
    }), flush=True)


def ae_dtype(policy=None):
    from dsin_b200 import precision
    return precision.dtype_string(policy)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=None,
                    help="pairs per GPU per step (weak scaling; 8 = BASELINE configs[1]); default: shard --global-batch")
    ap.add_argument("--global-batch", type=int, default=256, help="pairs per step over all GPUs (configs[4])")
    ap.add_argument("--micro-batch", type=int, default=32, help="pairs per device call")
    ap.add_argument("--precision", default=None, help="precision policy name (dsin_b200/precision.py); default: shipped")
    ap.add_argument("--hw", default=None, help="geometry HxW other than 320x1224 (the metric string then says so)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-chunk", type=int, default=None, help="AE.e2e_chunk for the end-to-end calls (default: the AE's)")
    ap.add_argument("--streams", type=int, default=8, help="range-coder streams per image (--workload codec)")
    ap.add_argument("--workload", default="full", choices=["full", "sif", "enc", "codec", "roundtrip"],
                    help="full = configs[4] / configs[1]; sif = configs[2] (SI-Finder in isolation, --batch 32); "
                         "enc = configs[3] (encoder + quantiser + probclass on 320x960 crops, --batch 64)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--workload full: after the timed steps, write what the last one returned (rank 0's pairs) "
                         "to DIR/<name>.npy, at most 64 MB in all; the copies of that step's outputs are timed with it")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "ours" or args.workload != "full"):
        ap.error("--dump-outputs writes the outputs of --impl ours --workload full")
    if args.hw:
        set_geometry(args.hw)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)
    if args.workload != "full" and args.batch is None:
        args.batch = {"sif": 32, "enc": 64}.get(args.workload, 8)
    if args.workload == "enc":
        run_enc_only(args, rank, world, local_rank)
        return
    if args.workload == "sif":
        run_sif_only(args, rank, world, local_rank)
        return
    if args.workload == "codec":
        run_codec(args, rank, world, local_rank)
        return
    if args.workload == "roundtrip":
        run_roundtrip(args, rank, world, local_rank)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
