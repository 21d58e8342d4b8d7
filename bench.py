#!/usr/bin/env python
"""bench.py — DGL training-step throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 5            # this repo's CUDA path
    python bench.py --impl reference --steps 2 --warmup 1     # CPU arm (oracle port, host cores)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A "step" is one DGL training step (reference main_dgl.py:93-158) on one synthetic batch of the
CREMA-D shape (spec 257x188, 3 frames of 3x224x224, 6 classes), ConcatFusion_DGL, fp32 master
weights, bf16 activations, fp32 accumulation.  Per-GPU batch is fixed (weak scaling).

Prints ONE JSON line (rank 0).  `value`: inputs already resident in HBM; `e2e`: the same step
through the public DGLStep.prefetch()/step()/read_stats() API with every step's pinned-host inputs
copied H2D (on a copy stream, overlapping the previous step) and the 7-float result read D2H inside
the timed region.  A second end-to-end leg takes the frames from a uint8 store resident in HBM and crops / resizes them
on the device (`e2e_device_pipeline`); at N > 1, where N host copies of 512 MB per step share one host, the faster of
the two legs is reported as `e2e` and the other next to it (`e2e_host_frames` / `e2e_device_pipeline`).  `roofline`: the dominant kernel class (implicit-GEMM convolutions),
algorithmic FLOPs / CUDA-event time measured in an instrumented pass after the timed region.
`cpu_baseline`: the CPU oracle port timed on this box's host cores on a bounded sample.

`--dump-outputs DIR` writes what the last step of the `value` region computed (rank 0) as float32 .npy files, so that
two builds can be compared output for output: the same arguments give the same inputs and initial weights.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "iccv2025-gdl_b200"))

METRIC = "DGL train samples/sec (CREMA-D shape)"
METRIC_OF = {"CREMAD": METRIC, "KineticSound": "DGL train samples/sec (Kinetics-Sounds shape)",
             "VGGSound": "DGL train samples/sec (VGGSound shape)"}
UNIT = "samples/s"
TRAIN_GFLOP_PER_SAMPLE = {"CREMAD": 42.57, "KineticSound": 50.56, "VGGSound": 50.56}  # BASELINE.md §3
DUMP_SAMPLE = 1 << 21  # elements of the ~22 M parameters / gradients that --dump-outputs writes (8 MB each)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return p["bf16_tflops_sustained"], p["hbm_gbs"], "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.f = gpu_index, None, None

    def start(self):
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.flush()
        self.f.seek(0)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                smax.append(float(c[2]))
            except ValueError:
                continue
            for nme, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def cpu_oracle_throughput(fusion, dataset, shape, batch, steps, warmup, threads=None):
    """The reference's algorithm on the host cores (oracle port; /root/reference cannot travel)."""
    import torch
    from oracle import dgl_oracle as O
    from oracle.synth import make_batch
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    sd = O.init_state(fusion, dataset, 0)
    mom = {}
    n = O.N_CLASSES[dataset]
    data = make_batch(batch, n, shape, seed=1)
    times = []
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        O.dgl_step(sd, mom, *data, fusion=fusion, alpha=4.0, lr=0.001)
        t1 = time.perf_counter()
        if s >= warmup:
            times.append(t1 - t0)
    sec = sum(times) / len(times)
    return batch / sec, sec, threads


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = a.cpu_batch
    v, sec, threads = cpu_oracle_throughput(a.fusion, a.dataset, a.dataset, batch, a.steps, a.warmup)
    sample = "%d timed steps of batch %d (CREMA-D shape, %s fusion) after %d warm-up" % (
        a.steps, batch, a.fusion, a.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a, batch, 1),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_cudnn_sidebar(a):
    """Side bar (VERDICT r1 #10, SURVEY.md §2.3): the SAME step through stock PyTorch on this B200 — the oracle
    restatement moved to cuda under torch.autocast(bfloat16), i.e. cuDNN 9 / cuBLAS sm_100 kernels — the only other
    Blackwell implementation of this path.  Context for the headline number, not a product path and not a baseline
    the driver computes ratios from: printed with "impl": "cudnn_sidebar"."""
    import torch
    from oracle import dgl_oracle as O
    from gdl_b200.shapes import HEAD_WIDTH, LABEL_MAX, make_batch
    if int(os.environ.get("RANK", "0")) != 0:
        return
    dev = torch.device("cuda", 0)
    torch.backends.cudnn.benchmark = True
    B = a.global_batch or a.batch
    out = {}
    for mode in ("bf16_autocast", "fp32_tf32"):
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = True
        # conv weights in channels_last so that cuDNN runs its NHWC tensor-core kernels without layout transposes
        sd = {k: (v.to(dev).contiguous(memory_format=torch.channels_last) if v.dim() == 4 else v.to(dev))
              for k, v in O.init_state(a.fusion, a.dataset, 0).items()}
        mom = {}
        data = [t.to(dev) for t in make_batch(B, HEAD_WIDTH[a.dataset], a.dataset, seed=1, label_max=LABEL_MAX[a.dataset])]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for s in range(max(a.warmup, 3) + a.steps):
            if s == max(a.warmup, 3):
                torch.cuda.synchronize()
                ev[0].record()
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(mode == "bf16_autocast")):
                O.dgl_step(sd, mom, *data, fusion=a.fusion, alpha=4.0, lr=0.001)
        ev[1].record()
        torch.cuda.synchronize()
        ms = ev[0].elapsed_time(ev[1]) / a.steps
        out[mode] = {"value": B / (ms / 1e3), "ms_per_step": ms}
        del sd, mom, data
        torch.cuda.empty_cache()
    best = out["bf16_autocast"]
    print(json.dumps({"impl": "cudnn_sidebar", "metric": METRIC_OF[a.dataset], "value": best["value"], "unit": UNIT,
                      "n_gpus": 1, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": best["ms_per_step"],
                      "higher_is_better": True, "dtype": "bf16 autocast (cuDNN/cuBLAS)", "data": "synthetic",
                      "config": workload_config(a, B, 1), "modes": out,
                      "note": "stock PyTorch %s: oracle restatement on cuda, autograd + cuDNN 9; includes its per-step "
                              "host syncs (float() of the losses / norm)" % torch.__version__}))


def workload_config(a, batch_per_gpu, n):
    head = {"concat": "ConcatFusion_DGL", "sum": "SumFusion_DGL", "film": "FiLM_DGL", "gated": "GatedFusion_DGL"}
    from gdl_b200.shapes import BATCH_SHAPES
    Fq, Tt, T, H, W = BATCH_SHAPES[a.dataset]
    mb = batch_per_gpu * (Fq * Tt + 3 * T * H * W) * 4 / 1e6
    return {"workload": "%s-shape DGL step, ResNet-18 audio+visual, %s, batch %d per GPU x %d GPU, "
                        "synthetic" % ("CREMA-D" if a.dataset == "CREMAD" else a.dataset,
                                       head.get(a.fusion, a.fusion), batch_per_gpu, n),
            "global_batch": batch_per_gpu * n, "parallelism": "dp%d" % n,
            "l2": ("per-step inputs (%.0f MB per GPU) and activations exceed the 126 MB L2; no flush needed" % mb)
                  if mb > 126 else ("per-step inputs are %.0f MB per GPU, the step's activations (%.1f GB) exceed the "
                                    "126 MB L2; no flush needed" % (mb, batch_per_gpu * 0.085))}


def run_gpu(a):
    import torch
    import torch.distributed as dist
    import gdl_b200
    from gdl_b200 import ops
    from gdl_b200.step import DGLStep
    from gdl_b200.shapes import BATCH_SHAPES as SHAPES, HEAD_WIDTH, LABEL_MAX, make_batch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    def say(msg):
        if os.environ.get("GDL_BENCH_VERBOSE"):
            sys.stderr.write("[rank %d %.1fs] %s\n" % (rank, time.perf_counter() - T0, msg))
            sys.stderr.flush()
    T0 = time.perf_counter()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
        pg = dist.group.WORLD
    n_cls = HEAD_WIDTH[a.dataset]
    Fq, Tt, T, H, W = SHAPES[a.dataset]
    if a.global_batch:
        if a.global_batch % world:
            raise SystemExit("--global-batch %d is not divisible by %d ranks" % (a.global_batch, world))
        B = a.global_batch // world      # strong scaling: the global batch is fixed, the per-GPU batch shrinks
    else:
        B = a.batch                      # weak scaling: the per-GPU batch is fixed
    args = argparse.Namespace(dataset=a.dataset, fusion_method=a.fusion, modality="full")
    gdl_b200.setup_seed(0)
    model = gdl_b200.AVClassifier_DGL(args)
    model.apply(gdl_b200.weight_init)
    model.to(dev).train()
    step = DGLStep(model, B, (Fq, Tt), (T, H, W), alpha=4.0, lr=0.001, world_size=world, process_group=pg,
                   use_graph=not a.no_graph)
    spec, image, label = make_batch(B, n_cls, a.dataset, seed=1 + rank, label_max=LABEL_MAX[a.dataset])
    spec_h, image_h, label_h = spec.pin_memory(), image.pin_memory(), label.pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in (spec_h, image_h, label_h))
    say("model + step built")
    step.load_inputs(spec_h, image_h, label_h)
    torch.cuda.synchronize()
    say("inputs loaded")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def host_prefetch():
        step.prefetch(spec_h, image_h, label_h)

    def timed(n_steps, e2e, prefetch=host_prefetch):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        if e2e:
            prefetch()                                       # batch 0: its copy is not overlapped
        for i in range(n_steps):
            if e2e:
                step.step()                                  # consumes the prefetched batch i
                if i + 1 < n_steps:
                    prefetch()                               # H2D of batch i+1 overlaps step i (copy stream)
                step.read_stats()          # D2H of the step's result (7 floats), syncs the step
            else:
                step.step()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        wall = (time.perf_counter() - t0) * 1e3
        t = torch.tensor([ms, wall], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t[0].item(), t[1].item()

    launches0 = ops.LAUNCHES
    for i in range(max(a.warmup, 3)):
        step.step()
        if os.environ.get("GDL_BENCH_VERBOSE"):
            torch.cuda.synchronize()
            say("warmup step %d done" % i)
    torch.cuda.synchronize()
    per_step_launches = None
    if a.no_graph:
        per_step_launches = (ops.LAUNCHES - launches0) // max(a.warmup, 3)
    else:
        # step 0 ran eagerly: its count is the per-step kernel count (graph replays launch the same kernels)
        per_step_launches = step.launches_per_step

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, wall_ms = timed(a.steps, e2e=False)
    say("timed region done")
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, step, model, torch)
    for _ in range(2):
        step.prefetch(spec_h, image_h, label_h)
        step.step()
    ms_e2e, _ = timed(a.steps, e2e=True)
    stats = step.read_stats()

    # Same end-to-end loop with the visual transform on the device (SURVEY.md §8f rank 2): decoded uint8 frames
    # resident in HBM, per step the host uploads the spectrograms, the labels and the crop boxes it drew
    # (24 bytes per frame); gdl_crop_resize_normalize produces the fp32 frames on the copy stream.
    dp = None
    if (H, W) == (224, 224) and not a.no_device_pipeline:
        from gdl_b200.datapipe import DeviceFrameStore, VisualPipeline, draw_frame_params
        fh, fw = (360, 480) if a.dataset == "CREMAD" else (256, 340)  # frame sizes of the datasets' jpg dumps
        n_store = 2 * B * T
        gen = torch.Generator(device=dev).manual_seed(7 + rank)
        store = DeviceFrameStore(torch.randint(0, 256, (n_store, fh, fw, 3), device=dev, dtype=torch.uint8,
                                               generator=gen))
        pipe = VisualPipeline(store, T, 224, max_frames=B * T)
        torch.manual_seed(11 + rank)
        rows = [draw_frame_params(f % n_store, fh, fw, "train") for f in range(B * T)]
        params_h = torch.tensor(rows, dtype=torch.int32).pin_memory()

        def device_prefetch():
            step.prefetch(spec_h, params_h, label_h, pipeline=pipe)
        for _ in range(2):
            device_prefetch()
            step.step()
        ms_dp, _ = timed(a.steps, e2e=True, prefetch=device_prefetch)
        dp = {"value": B * world * a.steps / (ms_dp / 1e3), "unit": UNIT,
              "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in (spec_h, params_h, label_h)),
              "d2h_bytes_per_step": 32, "ms_per_step": ms_dp / a.steps,
              "frame_store": "%d uint8 frames %dx%d resident in HBM (%.0f MB)" % (n_store, fh, fw,
                                                                                 n_store * fh * fw * 3 / 1e6),
              "note": "crop boxes / flips drawn on the host in the reference's RNG order; crop + Pillow-exact "
                      "bilinear resize + flip + normalise on the device (csrc/datapipe.cu)"}

    value = B * world * a.steps / (ms / 1e3)
    e2e_value = B * world * a.steps / (ms_e2e / 1e3)
    line = {"metric": METRIC_OF[a.dataset], "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps, "higher_is_better": True,
            "scaling": "strong" if a.global_batch else "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(a, B, world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 32,
                    "ms_per_step": ms_e2e / a.steps},
            "gpu_launches": per_step_launches * a.steps,
            "launches_per_step": per_step_launches,
            "clocks": clocks,
            "final_losses": {"Lf": stats[0], "La": stats[1], "Lv": stats[2]},
            "wall_ms_per_step": wall_ms / a.steps}
    line["e2e"]["path"] = "fp32 frames + spectrograms from pinned host memory (DGLStep.prefetch / step / read_stats)"
    if dp is not None:
        dp["path"] = "uint8 frame store in HBM, crop boxes + spectrograms from pinned host memory (prefetch(pipeline=))"
        if world > 1 and dp["value"] > line["e2e"]["value"]:
            # N > 1: N copies of 512 MB per step share one host (measured: the host-frames leg wins by 2 % at N = 2 and
            # loses by 11 % at N = 8), and the data-parallel entry point (main_dgl.py --audio_path synthetic_device,
            # SURVEY.md 8f rank 2) can keep the decoded frames on the GPUs: both legs are timed, the faster one is
            # reported as `e2e`, the other next to it
            line["e2e_host_frames"], line["e2e"] = line["e2e"], dp
        else:
            line["e2e_device_pipeline"] = dp

    if not a.no_roofline:
        # every rank runs the instrumented step (it contains the gradient all-reduce); rank 0 reports it
        roof, breakdown = roofline_pass(step, torch, ops, B)
        if rank == 0:
            line["roofline"], line["kernel_breakdown"] = roof, breakdown
    if world > 1:
        dist.barrier()
    if rank == 0:
        tf_peak, _, how = measured_peaks()
        gf = TRAIN_GFLOP_PER_SAMPLE[a.dataset]
        line["step_tensor_frac"] = {"achieved_tflops": value / world * gf / 1e3, "peak_tflops": tf_peak,
                                    "frac": value / world * gf / 1e3 / tf_peak, "peak_source": how,
                                    "gflop_per_sample": gf}
        if world == 1 and not a.no_cpu:
            v, sec, threads = cpu_oracle_throughput(a.fusion, a.dataset, a.dataset, a.cpu_batch, 2, 1)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": "2 timed steps of batch %d after 1 warm-up (oracle port, fp32, "
                                              "torch %s CPU)" % (a.cpu_batch, torch.__version__)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, step, model, torch):
    """What the step returns to its caller after its last run: the 7 statistics of read_stats(), the three logit sets,
    the updated parameters and their (clipped) gradients, and the BatchNorm running statistics.  Parameters and
    gradients are concatenated in arena order (head | audio | visual) and sampled at DUMP_SAMPLE fixed, seeded
    positions."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    params = torch.cat([p.detach().reshape(-1) for p in step.arena.params])
    grads = torch.cat([p.grad.reshape(-1) for p in step.arena.params])
    n = params.numel()
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:min(n, DUMP_SAMPLE)].sort().values
    idx = idx.to(params.device)
    bn = [t.reshape(-1) for m in model.modules() if isinstance(m, torch.nn.BatchNorm2d)
          for t in (m.running_mean, m.running_var)]
    out = {"stats": torch.tensor(step.read_stats()), "logits": step.logits, "params_sample": params[idx],
           "grads_sample": grads[idx], "bn_running_stats": torch.cat(bn)}
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def roofline_pass(step, torch, ops, B):
    """One instrumented eager step on a single stream: CUDA events around every op.  Returns the
    roofline object of the dominant kernel class and a per-class breakdown."""
    tf_peak, hbm_peak, how = measured_peaks()
    torch.cuda.synchronize()
    ops.TIMING = []
    saved = step.stream_a, step.stream_v, step.use_graph
    saved_ws = step.enc_a.wgrad_stream, step.enc_v.wgrad_stream
    cur = torch.cuda.current_stream()
    step.stream_a = step.stream_v = cur
    step.enc_a.wgrad_stream = step.enc_v.wgrad_stream = None  # everything serialised on one stream
    step.use_graph = False
    try:
        step.step()
        torch.cuda.synchronize()
        recs = ops.TIMING
    finally:
        ops.TIMING = None
        step.stream_a, step.stream_v, step.use_graph = saved
        step.enc_a.wgrad_stream, step.enc_v.wgrad_stream = saved_ws
    agg = {}
    dump = []
    for name, e0, e1, work in recs:
        ms = e0.elapsed_time(e1)
        dump.append((name, round(ms, 4), work))
        d = agg.setdefault(name, {"ms": 0.0, "launches": 0, "flops": 0.0, "bytes": 0.0})
        d["ms"] += ms
        d["launches"] += 1
        if work:
            d[work[0]] += work[1]
    if os.environ.get("GDL_DUMP_OPS"):
        json.dump(dump, open(os.environ["GDL_DUMP_OPS"], "w"))
    total = sum(d["ms"] for d in agg.values())
    breakdown = {}
    for name, d in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        e = {"ms": round(d["ms"], 3), "share": round(d["ms"] / total, 4), "ops": d["launches"]}
        if d["flops"]:
            e["tflops"] = round(d["flops"] / d["ms"] / 1e9, 1)
        if d["bytes"]:
            e["gbs"] = round(d["bytes"] / d["ms"] / 1e6, 1)
        breakdown[name] = e
    conv = [agg[k] for k in ("conv_fwd", "conv_dgrad", "conv_wgrad") if k in agg]
    flops = sum(d["flops"] for d in conv)
    ms = sum(d["ms"] for d in conv)
    nl = sum(d["launches"] for d in conv)
    ach = flops / ms / 1e9
    roof = {"bound": "tensor", "kernel": "conv_flat_kernel + conv_wgrad_flat_kernel + stem kernels (tcgen05 implicit GEMM; "
                                         "fwd+dgrad+wgrad aggregated over %d launches)" % nl,
            "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak, "traffic": None,
            "peak_source": how, "share_of_step": round(ms / total, 4),
            "avg_launch_ms": ms / nl, "flops_per_launch": flops / nl}
    # DRAM traffic per launch of the same kernels, from the committed ncu capture of this workload (ncu cannot run
    # inside a timed bench): bytes, averaged over the launches like `achieved`; null for other workloads.
    tpath = os.path.join(ROOT, "profiles", "r2_conv_traffic.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "r1_conv_traffic.json")
    if os.path.exists(tpath):
        t = json.load(open(tpath))
        crema = (step.F_, step.Tt, step.T) == (257, 188, 3)  # the capture is of the CREMA-D-shape workload
        if crema and t.get("batch") == B and abs(t.get("launches_per_step", 0) - nl) <= 2:
            roof["traffic"] = t["dram_bytes_per_launch"]
            roof["traffic_unit"] = "bytes of DRAM read+write per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)"
            roof["traffic_source"] = "profiles/%s: " % os.path.basename(tpath) + t["source"]
    return roof, breakdown


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="gdl_b200", choices=["gdl_b200", "reference", "cudnn_sidebar"])
    ap.add_argument("--batch", type=int, default=256, help="per-GPU batch (BASELINE configs[1]); weak scaling")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="fixed GLOBAL batch split over the ranks (strong scaling; BASELINE configs 3-4: 512 "
                         "KineticSound on 8 GPUs, 1024 VGGSound at 1/2/4/8)")
    ap.add_argument("--cpu-batch", type=int, default=64, help="CPU arm batch (BASELINE configs[0])")
    ap.add_argument("--fusion", default="concat")
    ap.add_argument("--dataset", default="CREMAD")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-device-pipeline", action="store_true", help="skip the e2e leg with the GPU visual transform")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, rank 0)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "gdl_b200":
        ap.error("--dump-outputs applies to --impl gdl_b200")
    if a.impl == "cudnn_sidebar":
        run_cudnn_sidebar(a)
    elif a.impl == "reference":
        a.warmup = min(a.warmup, 1)
        run_reference(a)
    else:
        run_gpu(a)


if __name__ == "__main__":
    main()
