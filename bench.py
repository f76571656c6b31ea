#!/usr/bin/env python
"""Benchmark of the hot path: images/sec of the full im_detect-equivalent (blob -> backbone -> RPN ->
proposals -> RoI head -> per-class NMS -> top-100 records) on synthetic COCO-shaped 600x800 inputs,
ResNet-101, 300 proposals, 81 classes  (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--net res101] [--no-cpu-baseline]
                    [--dump-outputs DIR]

ours       : this repo's sm_100a path.  `value` = device-resident input; `e2e` = through Network.detect() with
             pinned HOST input blob (H2D) and host read-back of the detection records (D2H) every step.
reference  : the reference's CPU implementation of the same path.  TensorFlow-1.x (the reference's only
             executor) is not installable offline, so this arm times the oracle port (oracle/: torch-CPU fp32
             convs + numpy/C box math) on all host cores -- labelled kind="port".
Under torchrun (N>1) every rank processes its own image per step (image-sharded, weak scaling) and the
detection records are all-gathered over NCCL each step; times are CUDA-event times, max over ranks.
"""
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
from tf_faster_rcnn_b200 import paths  # noqa: E402

paths.add_lib_path()

NETS = {
    # name: (num_classes, anchor scales, H, W, post_nms_top_n, label)
    "res101": (81, (4, 8, 16, 32), 600, 800, 300, "ResNet-101 COCO-shape 600x800 blob, A=12, 300 proposals, 81 classes"),
    "vgg16": (21, (8, 16, 32), 600, 800, 300, "VGG16 VOC-shape 600x800 blob, A=9, 300 proposals, 21 classes"),
    "mobile": (81, (4, 8, 16, 32), 600, 800, 300, "MobileNet-v1 1.0 COCO-shape 600x800 blob, A=12, 300 proposals, 81 classes"),
    "res152lg": (81, (2, 4, 8, 16, 32), 800, 1067, 1000, "ResNet-152 800x1067 blob, A=15, 1000 proposals, 81 classes"),
}


def make_config(label, net_name, batch, world, rec_bytes=None):
    """The `config` object of the JSON line: identical for both arms (the CPU arm times single images of the same workload)."""
    return {"workload": label, "net": net_name, "images_per_step_per_gpu": batch, "parallelism": "image-sharded dp%d" % world,
            "l2": "per-step working set (weight planes + activations of %d image(s), > 1 GB) exceeds the 126 MB L2; no explicit flush" % batch,
            "final_nms": "cpu_nms predicate (USE_GPU_NMS=False)", "rpn": "proposal_layer_tf semantics (USE_E2E_TF=True)",
            "collective": "one async all_gather_into_tensor of the record buffer per step" if world > 1 else "none"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clock, power and throttle reasons sampled while the timed region runs: NVML every 20 ms (the driver's 20-step runs last
    ~0.2 s), falling back to `nvidia-smi` every ~150 ms when the NVML binding is unavailable."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    MASKS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.source = index, [], False, "nvidia-smi"
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml, self.source = pynvml, "nvml"
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
        try:
            mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(h))
        except Exception:
            mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(h))
        try:
            power = n.nvmlDeviceGetPowerUsage(h) / 1000.0
        except Exception:
            power = float("nan")
        flags = ["Active" if mask & self.MASKS[nm] else "Not Active" for nm in self.NAMES]
        return [str(sm), str(self.max_mhz), str(power)] + flags

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self.rows.append(self._sample_nvml())
                    time.sleep(0.02)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        def num(v):
            try:
                return float(v)
            except ValueError:
                return None
        sm = [num(r[0]) for r in self.rows if r and num(r[0]) is not None]
        mx = [num(r[1]) for r in self.rows if len(r) > 1 and num(r[1]) is not None]
        pw = [num(r[2]) for r in self.rows if len(r) > 2 and num(r[2]) is not None and num(r[2]) == num(r[2])]
        reasons = set()
        for r in self.rows:
            for i, nm in enumerate(self.NAMES):
                if len(r) > 3 + i and r[3 + i].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(self.rows), "source": self.source}


def make_inputs(net_name, seed=3):
    from tf_faster_rcnn_b200 import synth
    C, scales, H, W, post, label = NETS[net_name]
    key = "res152" if net_name == "res152lg" else net_name
    weights = synth.make(key, C, 3 * len(scales), 3)      # replicas share the weights; each rank gets its own image
    blob = synth.synthetic_blob(H, W, seed)
    return key, C, scales, H, W, post, label, weights, blob


def cpu_reference_step(key, weights, blob, im_info, C, scales, post):
    """One image through the CPU port of the reference path (oracle): test_image + im_detect tail + test_net tail."""
    from oracle import pipeline as P
    o = P.opts(anchor_scales=scales, rpn_post_nms_top_n=post, use_gpu_nms=False)
    st = P.test_image(key, weights, blob, im_info, C, o)
    scores, boxes = P.im_detect_post(st["rois"], st["cls_prob"], st["bbox_pred"], float(im_info[2]), int(im_info[0]), int(im_info[1]))
    dets = P.test_net_post(scores, boxes, o)
    return sum(d.shape[0] for d in dets)


def all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is entitled to every core the process may run on."""
    import torch
    if os.environ.get("OMP_NUM_THREADS") and "FRCNN_CPU_THREADS" not in os.environ:
        # forced (torchrun sets 1): fall back to one thread per physical core (SMT siblings make oneDNN convs far slower:
        # 128 threads on the 64-core host measured 13x slower than 64)
        n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        torch.set_num_threads(max(1, n // 2 if n > 16 else n))
    elif "FRCNN_CPU_THREADS" in os.environ:
        torch.set_num_threads(int(os.environ["FRCNN_CPU_THREADS"]))
    return torch.get_num_threads()


def run_reference(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    all_host_threads()
    key, C, scales, H, W, post, label, weights, blob = make_inputs(args.net)
    im_info = np.array([H, W, 1.0], np.float32)
    cores = torch.get_num_threads()
    # one image is ~2.5-3 s of all host cores for ResNet-101: at most 2 warm-up images (thread pools, oneDNN primitive caches)
    warm = min(max(args.warmup, 1), 2) if args.steps > 1 else 1
    for _ in range(warm):
        cpu_reference_step(key, weights, blob, im_info, C, scales, post)
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_reference_step(key, weights, blob, im_info, C, scales, post)
    dt = time.perf_counter() - t0
    v = steps / dt
    line = {"impl": "reference", "metric": "images/sec", "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": steps,
            "steps_requested": args.steps, "warmup": warm, "ms_per_step": 1000 * dt / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(label, args.net, max(1, int(args.batch)), args.gpus),
            "impl_note": "TF1 unavailable offline: CPU port (oracle) of the reference path, torch-CPU fp32 convs; one image per timed step",
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port", "sample": "1 image of the bench workload per step"},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_ours(args):
    if args.precision == "f16x1":
        os.environ["FRCNN_CONV_IMPL"] = "f16x1"
    import torch
    import torch.distributed as dist
    from tf_faster_rcnn_b200 import _native, engine
    from model.config import cfg
    from nets.vgg16 import vgg16
    from nets.resnet_v1 import resnetv1
    from nets.mobilenet_v1 import mobilenetv1

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    _native.check(_native.lib().frcnn_check_device(local), "check_device")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    key, C, scales, H, W, post, label, weights, blob = make_inputs(args.net, seed=3 + rank)
    cfg.TEST.HAS_RPN = True
    cfg.TEST.RPN_POST_NMS_TOP_N = post
    cfg.USE_GPU_NMS = False        # the TF1-CPU reference semantics: final NMS = cpu_nms predicate
    net = vgg16() if key == "vgg16" else mobilenetv1() if key == "mobile" else resnetv1(int(key[3:]))
    net.create_architecture("TEST", C, tag="default", anchor_scales=scales, anchor_ratios=(0.5, 1, 2))
    net.load_weights(weights)
    im_info = np.array([H, W, 1.0], np.float32)
    B = max(1, int(args.batch))
    from tf_faster_rcnn_b200 import synth
    blobs = np.concatenate([blob] + [synth.synthetic_blob(H, W, 1000 + 17 * rank + b) for b in range(1, B)], axis=0)
    host_blob = torch.from_numpy(blobs).pin_memory()
    scales_b, origs_b = [1.0] * B, [(H, W)] * B
    if args.ncu or args.layers:
        net.use_cuda_graph = False
    plan = net.plan_for(H, W, B)
    plan.image.copy_(host_blob)
    if args.layers:
        # per-launch device times without the CPU launch overhead: each tape step is captured 8x into its own small graph
        fns = [(lbl, fn) for lbl, fn in plan.tape.steps] + [("detect_post", None)]
        plan.launch(post=True, detect=True)
        torch.cuda.synchronize()
        fns[-1] = ("detect_post", plan.post_steps[plan.slot])
        rows = []
        REP = 8
        for lbl, fn in fns:
            g = engine.LaunchGraph([fn] * REP)
            g.replay(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                g.replay()
            e1.record()
            torch.cuda.synchronize()
            rows.append((lbl, e0.elapsed_time(e1) * 1000 / (3 * REP)))
        tot = sum(t for _, t in rows)
        print("per-launch device times (us, warm, 8 back-to-back launches per graph replay), batch %d: total %.0f us = %.0f us per image over %d steps"
              % (B, tot, tot / B, len(rows)))
        groups = {}
        for lbl, t in rows:
            kind = lbl.split(":")[0]
            key_ = kind
            if kind == "conv":
                key_ = "conv:" + ("head" if "/block4/" in lbl or "cls_bbox" in lbl or "/fc" in lbl or "Conv2d_1[23]" in lbl else "rpn" if "/rpn" in lbl else "body")
            groups[key_] = groups.get(key_, 0) + t
        for k, v in sorted(groups.items(), key=lambda kv: -kv[1]):
            print("  %-16s %8.0f us  %5.1f%%" % (k, v, 100 * v / tot))
        fl = {}
        for cp, (lbl, _) in zip(plan.tape.conv_plans, [r for r in rows if r[0].startswith("conv:")]):
            fl[lbl] = cp
        for lbl, t in rows:
            extra = ""
            if lbl in fl:
                extra = "  %7.1f TFLOP/s" % (fl[lbl].flops / t / 1e6)
            print("    %-70s %8.1f%s" % (lbl, t, extra))
        return
    if args.ncu:
        plan.launch(post=True, detect=True)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        plan.launch(post=True, detect=True)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print("ncu pass done: %d tape steps + detect_post, batch %d" % (len(plan.tape.steps), B))
        return
    from tf_faster_rcnn_b200 import parallel
    plan.double_buffer = world > 1
    plan.launch(post=True, detect=True)                      # builds the record buffers
    torch.cuda.synchronize()
    rec_bytes = plan.rec.numel() * 4
    gather = parallel.RecordGather(plan.rec, world) if world > 1 else None
    step_no = [0]

    def step_resident():
        if gather is not None:
            gather.before_overwrite(plan.slot ^ 1)             # the gather of two steps ago has read the record buffer reused now
        plan.launch(post=True, detect=True)
        if gather is not None:                                # ONE asynchronous all-gather of the fixed-size records per step
            gather.issue(plan.slot, plan.rec)
        step_no[0] += 1

    pending = []
    host_blobs = [host_blob, host_blob.clone().pin_memory()]      # the application's two pinned input buffers (filled alternately)

    def step_e2e():
        """Public pipelined API: submit batch i (H2D of its pinned host blobs on the copy stream, graph replay, D2H of its records),
        then collect batch i-1 -- every step moves one batch in and one batch's records out; the copy of batch i overlaps the
        compute of batch i-1."""
        if gather is not None:
            gather.before_overwrite(plan.slot ^ 1)
        pending.append(net.submit_batch(host_blobs[step_no[0] & 1], scales_b, origs_b))
        if gather is not None:
            gather.issue(plan.slot, plan.rec)
        step_no[0] += 1
        if len(pending) > 1:
            return net.collect_batch(pending.pop(0))
        return None

    def drain_e2e():
        while pending:
            net.collect_batch(pending.pop(0))

    def barrier():
        torch.cuda.synchronize()
        if gather is not None:
            gather.before_overwrite(0); gather.before_overwrite(1)
            torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if gather is not None:                                # the last gathers are part of the job
            gather.before_overwrite(0); gather.before_overwrite(1)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms = timed(step_resident, args.steps)
    # what the timed path handed its caller in the last step: the per-image detection records, read back after the timing
    dumped = plan.records() if args.dump_outputs and rank == 0 else None
    # e2e through the public API
    for _ in range(3):
        step_e2e()
    drain_e2e()

    def e2e_steps_then_drain(state=[0]):
        step_e2e()
        state[0] += 1
        if state[0] == args.steps:                            # the last batch's records are read inside the timed region too
            drain_e2e()
    ms_e2e = timed(e2e_steps_then_drain, args.steps)
    # dominant kernel (tcgen05 conv/FC GEMM): time only its launches, on the launching stream (one graph of all of them)
    conv_steps = [fn for lbl, fn in plan.tape.steps if lbl.startswith("conv:")]
    cg = engine.LaunchGraph(conv_steps)

    def conv_only():
        cg.replay()
    for _ in range(3):
        conv_only()
    ms_conv = timed(conv_only, args.steps)
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    # the reference's own batch size beside the headline: the same image stream one image per graph replay (1 GPU only; untimed
    # by the contract -- reported so that both operating points come out of the same run)
    batch1 = None
    if world == 1 and B != 1 and not args.no_batch1:
        p1 = net.plan_for(H, W, 1)
        p1.image.copy_(host_blob[:1])
        for _ in range(3):
            p1.launch(post=True, detect=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n1 = args.steps
        e0.record()
        for _ in range(n1):
            p1.launch(post=True, detect=True)
        e1.record()
        torch.cuda.synchronize()
        ms1 = e0.elapsed_time(e1) / n1
        batch1 = {"value": 1000.0 / ms1, "unit": "images/s", "ms_per_image": ms1, "steps": n1,
                  "note": "device-resident, one image per graph replay (the reference's batch size)"}
    # context for the roofline: what the tensor cores of THIS board give a plain library GEMM right now (burst, 8192^3)
    lib_peaks = {}
    if rank == 0 and not args.no_lib_peaks:
        for nm, dt_, tf32 in (("fp16", torch.float16, False), ("tf32", torch.float32, True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            a_ = torch.randn(8192, 8192, device="cuda", dtype=dt_); b_ = torch.randn(8192, 8192, device="cuda", dtype=dt_)
            best = 0.0
            for i in range(6):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); torch.matmul(a_, b_); e1.record(); torch.cuda.synchronize()
                if i:
                    best = max(best, 2 * 8192.0 ** 3 / (e0.elapsed_time(e1) / 1e3) / 1e12)
            lib_peaks[nm + "_matmul_tflops_burst"] = best
            del a_, b_
        torch.backends.cuda.matmul.allow_tf32 = False
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk, pk_src = peaks()
    n_steps = args.steps
    value = world * B * n_steps / (ms / 1000.0)
    e2e_v = world * B * n_steps / (ms_e2e / 1000.0)
    conv_alg_flops = plan.tape.conv_flops
    conv_tflops = conv_alg_flops * n_steps / (ms_conv / 1000.0) / 1e12
    peak = pk.get("bf16_tflops_sustained", pk.get("bf16_tflops"))
    traffic, traffic_note = None, "no ncu capture of this net / batch committed"
    tp = os.path.join(ROOT, "profiles", "r02_conv_traffic.json")
    if os.path.exists(tp):                                    # tools/launch_list_summary.py over the committed ncu launch list of `bench.py --ncu`
        with open(tp) as f:
            tj = json.load(f).get("%s_b%d" % (args.net, B))
        if tj:
            traffic, traffic_note = tj["dram_bytes_per_conv_launch_avg"], tj["note"]
    # kernels of this repo launched per step: one per tape step (+1 reduce pass for conv plans with split tiles) + class_nms + cap_emit
    try:
        tails = sum(1 for cp in plan.tape.conv_plans if cp.info()["splits"] > 1)
    except Exception:
        tails = 0
    launches_per_step = len(plan.tape.steps) + tails + 2
    line = {
        "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": n_steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / n_steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("f16x3 (fp32-grade: fp16 hi/lo split of both operands, 3 tcgen05 kind::f16 MMAs per product, fp32 accumulate)"
                  if args.precision != "f16x1" else
                  "f16x1 THROUGHPUT MODE -- reduced precision (plain fp16 operands, fp32 accumulate), NOT the parity path and NOT the "
                  "headline: deviation from the oracle in profiles/r02_parity.md"),
        "data": "synthetic",
        "config": make_config(label, args.net, B, world, rec_bytes),
        "e2e": {"value": e2e_v, "unit": "images/s", "h2d_bytes_per_step": int(host_blob.numel() * 4 + B * 12), "d2h_bytes_per_step": int(rec_bytes),
                "ms_per_step": ms_e2e / n_steps, "api": "Network.submit_batch(pinned host blobs) / collect_batch() -> per-image detection records on the host, two batches in flight"},
        "gpu_launches": launches_per_step * n_steps,
        "batch1": batch1,
        "clocks": sampler.summary() if sampler else None,
        "roofline": {"bound": "tensor", "kernel": "conv_gemm_f16x3_kernel (all %d conv/FC launches of one step of %d image(s))" % (len(conv_steps), B),
                     "achieved": conv_tflops, "peak": peak, "unit": "TFLOP/s", "frac": conv_tflops / peak, "traffic": traffic,
                     "traffic_note": traffic_note,
                     "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (%s)" % pk_src,
                     "scheme_ceiling": {"tflops": peak / 3.0, "frac": conv_tflops / (peak / 3.0),
                                        "note": "the fp32-grade f16x3 scheme issues 3 fp16 MMAs per product: its own ceiling is peak/3"},
                     "library_gemm_now": lib_peaks,
                     "algorithmic_gflop_per_step": conv_alg_flops / 1e9, "conv_ms_per_step": ms_conv / n_steps,
                     "conv_share_of_step": (ms_conv / n_steps) / (ms / n_steps)},
    }
    if not args.no_cpu_baseline and world == 1:
        import torch as _t
        all_host_threads()
        t0 = time.perf_counter()
        cpu_reference_step(key, weights, blob, im_info, C, scales, post)      # warm-up (thread pools, oneDNN primitives)
        t1 = time.perf_counter()
        nrep = 2 if (t1 - t0) < 10 else 1
        t1 = time.perf_counter()
        for _ in range(nrep):
            cpu_reference_step(key, weights, blob, im_info, C, scales, post)
        dt = (time.perf_counter() - t1) / nrep
        line["cpu_baseline"] = {"value": 1.0 / dt, "unit": "images/s", "cores": _t.get_num_threads(), "kind": "port",
                                "sample": "%d image(s) of the same workload after 1 warm-up (an untuned CPU port, not TF1-Eigen)" % nrep}
    print(json.dumps(line))
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for b, dets in enumerate(dumped):                     # rows x1, y1, x2, y2, score, class of image b of the batch
            np.save(os.path.join(args.dump_outputs, "detections_%d.npy" % b), dets.astype(np.float32))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--net", default="res101", choices=sorted(NETS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batch1", action="store_true", help="skip the extra batch-1 measurement reported beside the headline")
    ap.add_argument("--no-lib-peaks", action="store_true", help="skip the two 8192^3 library matmuls timed for context after the run")
    ap.add_argument("--precision", default="fp32-grade", choices=["fp32-grade", "f16x1"],
                    help="f16x1 = the opt-in THROUGHPUT mode (plain fp16 operands, fp32 accumulate): NOT the parity path, its line says so")
    ap.add_argument("--batch", type=int, default=int(os.environ.get("FRCNN_BENCH_BATCH", "4")),
                    help="images per GPU per step (one graph replay); 1 = the reference's batch size")
    ap.add_argument("--layers", action="store_true", help="print a per-launch CUDA-event timing table of one image (eager, warm) and exit")
    ap.add_argument("--ncu", action="store_true", help="profiling aid: eager launches (no CUDA graph), one warm-up image, then ONE image "
                    "between cudaProfilerStart/Stop (run under `ncu --profile-from-start off`); prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the detection records of the last step (rank 0's images) as "
                         "DIR/detections_<image>.npy (float32 [n, 6]); the seeded inputs make runs comparable output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.layers or args.ncu):
        ap.error("--dump-outputs applies to the timed path of --impl ours only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
