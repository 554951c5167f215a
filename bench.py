#!/usr/bin/env python
"""bench.py — headline benchmark: images/sec of fai-detr-l-obj365 inference, bs=32/GPU, 640x640 (BASELINE.json).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...        # the reference's CPU path (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR     # also write what the last timed step computed as DIR/<name>.npy

A "step" = one pass of the hot path over one batch of 32 synthetic images: FAIDetr.forward (normalise -> ResNet50-vd ->
hybrid encoder -> 6-layer deformable decoder) + the fused DETR post-process kernel.
  value : whole-job images/s with inputs resident in HBM (CUDA-graph replay of the forward + post-process launch), in the PARITY-GREEN
          mode `fp32_tc` (fp32 storage, three fp16 tcgen05 products per conv/linear: meets north_star's 1e-3 / identical keep-set bars,
          tests/test_gpu_e2e.py, profiles/r02_error_budget.md).  The fp16 mode (one product; the reference's own CUDA numerics class, but
          outside the bars) is reported beside it as `fast_mode`.
  e2e   : same metric through the public API (FocoosModel.stream / infer_async) from PINNED HOST uint8 images, H2D and D2H inside
          the timed region, two batches in flight
Multi-GPU: inference = independent replicas, one process per GPU, no data-path collective ("replicas only"; weak scaling); the fine-tune
leg (BASELINE configs[4], `train_config5`) runs on every rank with the bucketed NCCL gradient all-reduce.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "images/sec fai-detr-l bs=32 640x640 inference"
GFLOP_PER_IMG_USEFUL = 139.05  # SURVEY.md §8(d): excludes the dead mask_features conv
IDEAL_US_PER_IMG_16BIT = 129.0  # SURVEY.md §8(d) sum-of-max roofline at 16-bit activations
IDEAL_US_PER_IMG_FP32 = 259.0   # SURVEY.md §8(d): fp32 activations + half-rate (tf32-class) MMA
DUMP_LIMIT_BYTES = 64 << 20


def ncu_traffic(kernel_substr: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, read from the committed ncu capture of THIS round
    (profiles/r02_ncu_dominant.csv, written by tools/ncu_extract.py from an `ncu --set full` report); None when no capture matches."""
    import csv
    path = os.path.join(ROOT, "profiles", "r02_ncu_dominant.csv")
    if not os.path.exists(path):
        return None, None
    with open(path) as f:
        for row in csv.DictReader(f):
            if kernel_substr in row.get("kernel", ""):
                return float(row["dram_bytes_read"]) + float(row["dram_bytes_write"]), os.path.relpath(path, ROOT)
    return None, None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"], "source": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback"}


def seeded_weights():
    from focoos_b200.utils.seeded_weights import seeded_state_dict

    with open(os.path.join(ROOT, "tests", "golden", "fai_detr_l_obj365_state_dict_manifest.json")) as f:
        man = json.load(f)
    return seeded_state_dict({k: torch.empty(v[0], dtype=getattr(torch, v[1])) for k, v in man.items()}, 0)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(path: str, arrays: dict) -> None:
    """Write each tensor as <path>/<name>.npy: floating point as float32, integers as float64 (exact).  Smallest first; an array that would
    take more than its share of what is left of DUMP_LIMIT_BYTES is replaced by a seeded sample of its flattened elements (the same
    positions for the same shape), so two builds run with the same arguments write files that compare element for element."""
    os.makedirs(path, exist_ok=True)
    left = DUMP_LIMIT_BYTES
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    for i, (name, t) in enumerate(items):
        a = t.detach().float().cpu().numpy() if t.is_floating_point() else t.detach().cpu().numpy().astype(np.float64)
        share = left // (len(items) - i)
        if a.nbytes > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a)
        left -= a.nbytes


def cpu_reference_run(batch: int, steps: int, warmup: int, sd, threads: int):
    """The reference's CPU path (oracle port of focoos' torch fp32 eval forward + post-process) on the host cores."""
    from oracle import detr_oracle as O
    from oracle.gen_golden import synth_images

    torch.set_num_threads(threads)
    imgs = synth_images(1, [(640, 640)] * batch)
    cfg = O.DetrOracleConfig()
    times = []
    with torch.no_grad():
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            x = O.detr_preprocess(imgs, (640, 640))
            s, b = O.detr_forward(sd, x, cfg)
            O.detr_postprocess(s, b, [(640, 640)] * batch, 0.5)
            if it >= warmup:
                times.append(time.perf_counter() - t0)
    return batch / float(np.mean(times)), float(np.mean(times)) * 1e3


def _graphed(step, use_graph):
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    if not use_graph:
        return step
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        step()
    return g.replay


def _throughput_ms(step, use_graph, steps):
    run = _graphed(step, use_graph)
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _latency(step, use_graph, warm=20, iters=100):
    run = _graphed(step, use_graph)
    for _ in range(warm):
        run()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return {"batch": 1, "p50_ms": ts[len(ts) // 2], "p90_ms": ts[int(len(ts) * 0.9)], "iters": iters, "warmup": warm, "what": "forward + on-device post-process of one 640x640 image, device-timed per iteration"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--precision", default="fp32_tc", choices=["fp16", "fp32", "fp32_tc"])
    ap.add_argument("--no-train-leg", action="store_true", help="skip the fine-tune leg (BASELINE configs[4])")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="skip the bs=1 latency, parity-mode and other-config legs")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the MaskFormer / BisenetFormer / fine-tune legs (separate processes)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (model logits / boxes and the "
                    "post-processed detections of rank 0) as DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    cores = os.cpu_count() or 1
    cpu_threads = min(cores, 32)  # torch CPU conv kernels stop scaling (and regress) beyond ~32 threads on this path
    config = {"workload": "fai-detr-l-obj365 bs=32/GPU 640x640 inference (BASELINE configs[1])", "per_gpu_batch": args.batch, "global_batch": args.batch * world,
              "weights": "seeded random (focoos_b200.utils.seeded_weights, seed 0)", "parallelism": f"replicas x{world}", "l2_policy": "inputs_larger_than_L2 (each step streams >2 GB of activations + 88 MB of weights through the 126 MB L2; 39 MB uint8 input batch)"}
    sd = seeded_weights()

    if args.impl == "reference":
        if rank != 0:
            return
        cb, csteps, cwarm = 2, max(5, min(args.steps, 8)), max(1, min(args.warmup, 2))
        v, ms = cpu_reference_run(cb, csteps, cwarm, sd, cpu_threads)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": csteps, "warmup": cwarm, "ms_per_step": ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": v, "unit": "images/s", "cores": cpu_threads, "host_cores": cores, "kind": "port", "sample": f"{csteps} timed passes of batch {cb} (reference is slower per image at larger CPU batches, BASELINE.md §3)"},
                "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return

    from focoos_b200 import DETRConfig, FocoosModel, ModelInfo, ops
    from focoos_b200.fai_detr import FAIDetr
    from oracle.gen_golden import synth_images  # input generator only (numpy); not a compute path

    from focoos_b200 import distributed as D

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    D.init_from_env("nccl", dev)  # replicas only: the group is used for the timing barrier / max-over-ranks, never for data
    import torch.distributed as dist
    model = FAIDetr(DETRConfig(), precision=args.precision)
    model.load_state_dict(sd, strict=True)
    fm = FocoosModel(model, ModelInfo(name="fai-detr-l-obj365", im_size=640))
    fm.model.to(dev)
    proc = fm.processor
    B = args.batch
    imgs_np = np.stack(synth_images(1 + rank, [(640, 640)] * B))  # [B,640,640,3] uint8
    host_u8 = torch.from_numpy(imgs_np).pin_memory()
    x_dev = host_u8.to(dev)  # uint8 [B,640,640,3] resident in HBM: the stem kernel reads it directly
    sizes = [(640, 640)] * B
    sizes_dev = torch.tensor(sizes, dtype=torch.int32, device=dev)

    def step_device():
        out = fm.model(x_dev)
        return out, ops.detr_postprocess(out.logits, out.boxes, sizes_dev, 300, 0.5)

    # ---- warm-up (also builds the engine), then capture forward+post-process in a CUDA graph
    l0 = ops.launch_count()
    step_device()
    torch.cuda.synchronize()
    launches_per_step = ops.launch_count() - l0
    graph = None
    if not args.no_graph:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                step_device()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            g_out = step_device()

    def run_step():
        if graph is not None:
            graph.replay()
            return g_out
        return step_device()

    for _ in range(max(args.warmup, 3)):
        run_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        e0.record()
        for _ in range(args.steps):
            last = run_step()
        e1.record()
        torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        out, (d_scores, d_labels, d_boxes, d_query, d_count) = last
        dump_outputs(args.dump_outputs, {"logits": out.logits, "boxes": out.boxes, "det_scores": d_scores, "det_labels": d_labels,
                                         "det_boxes": d_boxes, "det_query": d_query, "det_count": d_count})
    ms_total = D.max_over_ranks(e0.elapsed_time(e1), dev)  # device time, max over ranks
    D.synchronize()
    ms_step = ms_total / args.steps
    value = B * world / (ms_step / 1e3)

    # ---- e2e through the public API: pinned host uint8 -> H2D (copy stream) -> graph replay -> fused post-process -> packed D2H -> FocoosDetections,
    # two batches in flight (FocoosModel.stream / infer_async): every step still copies its own 39 MB input and reads its own result back
    def batches(n):
        for _ in range(n):
            yield host_u8

    for _ in fm.stream(batches(5), threshold=0.5):  # first call runs eagerly, the second captures the CUDA graph of model.forward
        pass
    torch.cuda.synchronize()
    # serving-style GC hygiene: everything allocated so far (model, packed weights, graph pools) moves to the permanent generation, so the cyclic
    # collector only ever walks the per-step detection objects (a full collection over the torch heap showed up as one ~50 ms step in 25)
    import gc
    gc.collect()
    gc.freeze()
    if world > 1:
        dist.barrier()
    e2e_steps = max(6, args.steps // 2)
    per_step = []
    t0 = time.perf_counter()
    ts = t0
    for dets in fm.stream(batches(e2e_steps), threshold=0.5):
        now = time.perf_counter()
        per_step.append((now - ts) * 1e3)
        ts = now
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    e2e_ms = D.max_over_ranks(e2e_ms, dev)
    per_step.sort()
    # the same API without pipelining (one blocking call per batch), for reference
    for _ in range(2):
        fm(host_u8, threshold=0.5, batched=True)
    t0 = time.perf_counter()
    nb = max(3, e2e_steps // 2)
    for _ in range(nb):
        dets = fm(host_u8, threshold=0.5, batched=True)
    blocking_ms = D.max_over_ranks((time.perf_counter() - t0) * 1e3 / nb, dev)
    e2e = {"value": B * world / (e2e_ms / 1e3), "unit": "images/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(host_u8.numel()),
           "d2h_bytes_per_step": B * (300 * 7 + 1) * 4, "p50_ms": per_step[len(per_step) // 2], "max_ms": per_step[-1], "steps": e2e_steps,
           "frac_of_value": (B * world / (e2e_ms / 1e3)) / value,
           "api": "FocoosModel.stream(pinned uint8 [B,H,W,3] batches), 2 in flight (infer_async: copy stream + staging buffers + pinned results)",
           "blocking_call": {"value": B * world / (blocking_ms / 1e3), "ms_per_step": blocking_ms, "api": "FocoosModel.__call__(pinned uint8 [B,H,W,3], batched=True)"}}
    fm._pipe = None
    fm._graphs.clear()
    torch.cuda.empty_cache()

    # ---- bs=1 latency (BASELINE.json metric, second half): p50/p90 of single-image forward+post-process, CUDA graph replay, device-timed
    lat = None
    fast = None
    if rank == 0 and not args.quick:
        x1, s1 = x_dev[:1].contiguous(), sizes_dev[:1].contiguous()

        def step1():
            o = fm.model(x1)
            return ops.detr_postprocess(o.logits, o.boxes, s1, 300, 0.5)

        lat = _latency(step1, not args.no_graph)
        # ---- the fp16 mode (one tcgen05 product per conv/linear) on the same workload: faster, outside the parity bars
        if args.precision == "fp32_tc":
            m2 = FAIDetr(DETRConfig(), precision="fp16")
            m2.load_state_dict(sd, strict=True)
            m2.to(dev)

            def step2():
                o = m2(x_dev)
                return ops.detr_postprocess(o.logits, o.boxes, sizes_dev, 300, 0.5)

            ms2 = _throughput_ms(step2, not args.no_graph, max(5, args.steps // 2))
            fast = {"precision": "fp16", "value": B / (ms2 / 1e3), "unit": "images/s", "ms_per_step": ms2, "n_gpus": 1,
                    "frac_of_ideal_16bit": (IDEAL_US_PER_IMG_16BIT * B / 1e3) / ms2,
                    "note": "fp16 storage, one product: the reference's own CUDA numerics class (fp16 autocast, focoos_model.py:604-609) but OUTSIDE north_star's bars (boxes 1.5e-3, "
                            "298-299/300 queries, ~70% identical integer boxes: profiles/r02_error_budget.md); not the headline"}
            del m2
            torch.cuda.empty_cache()

    # ---- roofline of the dominant kernel, timed alone on its heaviest layer shape: FPN 3x3 256->256 @80x80
    peaks = measured_peaks()
    roof = None
    if args.precision in ("fp16", "fp32_tc"):
        split = args.precision == "fp32_tc"
        wr32 = torch.randn((256, 3, 3, 256), device=dev) * 0.02
        br = torch.zeros(256, device=dev)
        if split:
            from focoos_b200.fai_detr import _split3_weights
            xr = ops.split_pair(torch.randn((B, 80, 80, 256), device=dev))
            wr = _split3_weights(wr32)
            yr = torch.empty((B, 80, 80, 256), device=dev, dtype=torch.float32)
            run_k = lambda: ops.conv2d(xr, wr, None, br, pad=1, act=ops.ACT_SILU, out=yr, algo=ops.ALGO_TCGEN05_SPLIT3)
        else:
            xr = torch.randn((B, 80, 80, 256), device=dev).half()
            wr = wr32.half()
            yr = torch.empty((B, 80, 80, 256), device=dev, dtype=torch.float16)
            run_k = lambda: ops.conv2d(xr, wr, None, br, pad=1, act=ops.ACT_SILU, out=yr)
        for _ in range(3):
            run_k()
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nrep = 20
        r0.record()
        for _ in range(nrep):
            run_k()
        r1.record()
        torch.cuda.synchronize()
        k_ms = r0.elapsed_time(r1) / nrep
        flops = 2.0 * B * 80 * 80 * 256 * 256 * 9
        ach = flops / (k_ms * 1e-3) / 1e12
        traffic, traffic_src = ncu_traffic("conv_tc_kernel")
        ideal_ms = (IDEAL_US_PER_IMG_FP32 if split else IDEAL_US_PER_IMG_16BIT) * B / 1e3
        roof = {"bound": "tensor", "kernel": "conv_tc_kernel on the 3x3 256->256 @80x80 conv (re-parameterised RepVGG block of the FPN CSPRepLayer; 3 launches/step at this shape, 16% of model FLOPs; "
                                             "conv_tc_kernel as a family = 97% of FLOPs)" + (", fp32-accurate as THREE fp16 tcgen05 products" if split else ""),
                "achieved": ach, "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": ach / peaks["tf_burst"], "peak_source": peaks["source"] + " burst bf16 (kernel timed alone)",
                "launch_ms": k_ms, "flops_per_launch": flops, "traffic": traffic, "traffic_source": traffic_src,
                "issued": {"tflops": ach * (3 if split else 1), "frac": ach * (3 if split else 1) / peaks["tf_burst"],
                           "note": "tensor-pipe work actually issued (3 products per algorithmic product in fp32_tc); `achieved`/`frac` count ALGORITHMIC flops only"},
                "model": {"useful_gflop_per_img": GFLOP_PER_IMG_USEFUL, "achieved_tflops_whole_step": GFLOP_PER_IMG_USEFUL * B / ms_step,
                          "ideal_ms_per_step": ideal_ms, "ideal_basis": "SURVEY 8(d) sum-of-max: " + ("fp32 activations + half-rate MMA (259 us/img)" if split else "16-bit activations (129 us/img)"),
                          "frac_of_ideal": ideal_ms / ms_step}}
        del xr, wr, yr
        torch.cuda.empty_cache()

    # ---- the other BASELINE.json inference configs (secondary numbers, each in its own process so that a failure there cannot touch the headline line):
    # configs[2] MaskFormer bs=16 800^2, configs[3] BisenetFormer bs=64 1024x512
    other = None
    if rank == 0 and world == 1 and not args.quick and not args.no_other_configs:
        other = {}
        root = os.path.dirname(os.path.abspath(__file__))
        for key, cmd in (("fai-mf-l-coco-ins bs=16 800x800 inference", ["tools/bench_mf.py"]), ("bisenetformer-l-ade bs=64 1024x512 inference", ["tools/bench_bisenet.py"])):
            try:
                env = dict(os.environ, FB200_TRACE="0")
                r = subprocess.run([sys.executable] + cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
                line = next(l for l in r.stdout.splitlines() if l.startswith("{"))
                d = json.loads(line)
                other[key] = {k: d[k] for k in ("images_per_s", "value", "ms_per_step", "unfused_images_per_s", "dtype", "phases_ms", "peak_mem_GB") if k in d}
                pl = next((l[len("PARITY_MODE "):] for l in r.stdout.splitlines() if l.startswith("PARITY_MODE {")), None)
                if pl:  # the same workload in the parity-green fp32_tc mode (tests/test_gpu_mf.py, tests/test_gpu_bisenet.py hold it to the fp32 bars)
                    pd_ = json.loads(pl)
                    other[key]["parity_mode"] = {k: pd_[k] for k in ("images_per_s", "ms_per_step", "unfused_images_per_s", "dtype", "precision", "error") if k in pd_}
            except Exception as e:  # noqa: BLE001
                other[key] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}

    # ---- BASELINE configs[4]: the fine-tune step with the data-parallel gradient all-reduce, on EVERY rank of this launch (so the driver's
    # 1/2/4/8-GPU runs each carry a DDP number; the headline line above is unaffected by a failure here)
    train = None
    if not args.quick and not args.no_train_leg:
        del fm, model
        torch.cuda.empty_cache()
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_train
            keys = ("value", "unit", "n_gpus", "ms_per_step", "steps", "warmup", "scaling", "dtype", "precision", "config", "kernel_launches_per_step", "phases_ms", "peak_mem_GB")
            # the reference's TrainerArgs.amp_enabled defaults to True (ports.py:1029): its iteration runs under torch.autocast(fp16) + GradScaler, so the config-5 number is
            # the "amp" precision (one fp16 tensor-core product, fp32 accumulation / storage); the fp32-accurate (three-product) step is reported next to it
            # several ranks: BatchNorm statistics over ALL ranks, like the reference (trainer/trainer.py:333-334 converts every BatchNorm to SyncBatchNorm whenever
            # world_size > 1); the step with per-rank statistics is reported next to it
            sync = world > 1
            t_amp = bench_train.run_leg(batch=16, size=640, steps=4, warmup=2, precision="amp", by_symbol=False, sync_bn=sync)
            train = {k: t_amp[k] for k in keys if k in t_amp}
            sub = ("value", "ms_per_step", "steps", "warmup", "dtype", "precision", "phases_ms", "peak_mem_GB")
            if sync:
                t_loc = bench_train.run_leg(batch=16, size=640, steps=2, warmup=1, precision="amp", by_symbol=False, sync_bn=False)
                train["local_batchnorm"] = {k: t_loc[k] for k in sub if k in t_loc}
            t_acc = bench_train.run_leg(batch=16, size=640, steps=2, warmup=1, precision="fp32_tc", by_symbol=False, sync_bn=sync)
            train["fp32_accurate"] = {k: t_acc[k] for k in sub if k in t_acc}
        except Exception as e:  # noqa: BLE001
            train = {"error": f"{type(e).__name__}: {str(e)[:300]}"}

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            cv, cms = cpu_reference_run(2, 6, 1, sd, cpu_threads)
            cpu = {"value": cv, "unit": "images/s", "cores": cpu_threads, "host_cores": cores, "kind": "port", "sample": "6 timed passes of batch 2 after 1 warm-up (oracle port of the reference's torch fp32 CPU forward + post-process)"}
        line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"fp16": "f16", "fp32": "f32", "fp32_tc": "f32 (storage and accumulation; every conv/linear product = 3 f16 tcgen05 products, error ~2^-21)"}[args.precision], "data": "synthetic",
                "parity": {"fp32_tc": "meets north_star: identical query sets and (class, int box) keep-sets, boxes/scores < 1e-3 (tests/test_gpu_e2e.py::test_fp32_tc_meets_the_parity_bars, profiles/r02_error_budget.md)",
                           "fp32": "meets north_star (CUDA-core fp32 mode)", "fp16": "outside north_star's bars (profiles/r02_error_budget.md)"}[args.precision],
                "config": config, "clocks": clk.summary(), "e2e": e2e, "gpu_launches": launches_per_step * args.steps, "launches_per_step": launches_per_step,
                "cuda_graph": graph is not None, "latency_bs1": lat, "fast_mode": fast, "other_configs": other, "train_config5": train, "roofline": roof, "cpu_baseline": cpu, "detections_img0": len(dets[0])}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
