#!/usr/bin/env python
"""bench.py - images/sec of the YOLO hot path (forward + decode + NMS) on synthetic 3x640x640 batches.

    python bench.py --gpus N --steps K --warmup W [--model v8n|v8s|v8x|...] [--batch B] [--gather comm|nccl]
    torchrun --nproc-per-node N bench.py --gpus N ...           (one rank per GPU)
    python bench.py --impl reference ...                         (the reference's CPU path, see below)
    python bench.py ... --dump-outputs DIR                       (also write the last timed step's outputs as DIR/*.npy)

One "step" = one pass of the hot path over one batch per GPU: yb_forward (tcgen05 fp16 network + DFL/box
decode) -> yb_nms (GPU NMS) [-> all-gather of the fixed-capacity detection payloads when N > 1: by default the
library's own peer-memory exchange (yb_comm_*, NVLink stores + flags, no NCCL kernel on the path), `--gather nccl`
for one packed ncclAllGather].  Workload at N=1 = BASELINE.json configs[1]: YOLOv8n detect, batch 32 x 3x640x640.

Printed JSON (one line, rank 0):
  value      images/s, device-timed (CUDA events, max over ranks), inputs resident in HBM; seeded-synthetic weights
             (a few hundred NMS survivors per image: the heavier post-processing case)
  real_weights  the same measurement with the reference's shipped Yolov8n checkpoint on a batch built from its five
             test images (v8n only; tests/golden fixtures)
  e2e        same metric through the host-buffer C-ABI calls yb_predict_u8_submit/_wait (pinned uint8 images in,
             detections out; H2D + D2H - and at N > 1 the detection gather - inside the timed region)
  roofline   the dominant kernel (conv_tc_kernel, the tcgen05 implicit-GEMM conv): algorithmic FLOPs and bytes of all
             its launches in one step / the time they take INSIDE the graph-replayed forward = event-timed forward
             minus the other kernels of the forward (stem / pool / upsample, each timed back to back with yb_time_op).
             kernel_ms_per_step <= forward_ms_per_step <= ms_per_step by construction.
  cpu_baseline  the oracle (PyTorch-CPU restatement of the reference's TorchSharp op sequence; the reference itself
             is C# and cannot run here) timed on this box's host cores
--impl reference times that same CPU path as the reference arm, all `batch` images per step, fp32.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# name -> (arch, size, task, GFLOP per image @640^2: 2*MACs of all convs, SURVEY.md section 8(d))
MODELS = {"v8n": ("v8", "n", "detect", 8.743), "v8s": ("v8", "s", "detect", 28.602), "v8x": ("v8", "x", "detect", 257.803),
          "v11n": ("v11", "n", "detect", 6.5), "v11s": ("v11", "s", "detect", 21.589),
          "v8n-seg": ("v8", "n", "segment", 12.6), "v8s-seg": ("v8", "s", "segment", 40.085)}
CONF, IOU, MAX_DET = 0.25, 0.45, 300
E2E_SLOTS = 3  # batches in flight through yb_predict_u8_submit/_wait
MASK_CAP = 32  # segment e2e: instance masks returned per image (byte planes of 640x640)
# compulsory bytes per image, fp16 input + fp32 prediction tensor (SURVEY.md section 8(d))
COMPULSORY_MB_IMG = {"detect": 3.87, "segment": 6.0}
# --dump-outputs: an output with more elements is written as a sample of this many; keeps a dump well under 64 MB
DUMP_SAMPLE = 1 << 20


def dump_outputs(out_dir, outputs):
    """Write each output of the last timed step as <out_dir>/<name>.npy, float32 (float64 for integer outputs).  An output
    of more than DUMP_SAMPLE elements becomes <name>_sample.npy: its values at DUMP_SAMPLE flat positions drawn with a
    fixed seed, in increasing order, so that two runs with the same arguments write files that compare element for element."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            t, name = t.reshape(-1)[idx.to(t.device)], name + "_sample"
        t = t.to(torch.float32 if t.is_floating_point() else torch.float64)
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tc_burst=1590.0, tc=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_run(model_key, batch, steps, warmup):
    """The reference's CPU path: un-fused conv->BN->SiLU graph + torchvision NMS via the oracle (PyTorch CPU = same
    libtorch operator family as TorchSharp), fp32, all `batch` images per step.  Thread count: the fastest of
    {16, 32, 64, all} on this host over one full step each (more threads than ~32 slow the small convs down on
    many-core boxes); reported as `cores`."""
    import torch
    from oracle import ops as oops
    from tests.util import oracle_model, synth_image
    arch, size, task, _ = MODELS[model_key]
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    m = oracle_model(arch, task, size)
    x = synth_image(batch, 640, 640)

    def step(inp):
        with torch.no_grad():
            inf = m(inp)[0]
        out, _ = oops.non_max_suppression(inf["boxes"], CONF, IOU, nc=80)
        if task == "segment":  # Segmenter.cs:54: masks of the kept detections
            for i, o in enumerate(out):
                if o.shape[0]:
                    oops.process_mask(inf["proto"][i], o[:, 6:], o[:, :4], (640, 640), upsample=True)

    best_t, best_n = None, ncpu
    for n in sorted({min(ncpu, c) for c in (16, 32, 64, ncpu)}):
        torch.set_num_threads(n)
        step(x[:4])
        t0 = time.perf_counter()
        step(x)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_t, best_n = dt, n
    torch.set_num_threads(best_n)
    for _ in range(warmup):
        step(x)
    t0 = time.perf_counter()
    for _ in range(steps):
        step(x)
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps * 1e3, best_n


def gpu_numa_cpus(device_index):
    """CPUs of the NUMA node the GPU hangs off, from sysfs (/sys/bus/pci/devices/<bdf>/local_cpulist), falling back to
    NVML's affinity mask."""
    import torch
    pr = torch.cuda.get_device_properties(device_index)
    bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
    try:
        txt = open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read().strip()
        cpus = []
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.extend(range(int(a), int(b) + 1))
            elif part:
                cpus.append(int(part))
        if cpus:
            return cpus, "sysfs local_cpulist"
    except OSError:
        pass
    import pynvml
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByPciBusId(f"0000{bdf}".encode()[-13:])
    ncpu = os.cpu_count()
    words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
    return [i for i in range(ncpu) if (int(words[i // 64]) >> (i % 64)) & 1], "NVML affinity"


def bind_to_gpu_numa(device_index):
    """Run this process - ALL its threads, so that pinned host allocations (first touch) land on the GPU's NUMA node -
    on the CPUs local to the GPU.  A pinned batch on the far socket copies at 17-25 GB/s instead of ~55 GB/s
    (tools/exp_h2d.py), which bounds the end-to-end number."""
    try:
        cpus, how = gpu_numa_cpus(device_index)
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return "not bound (no local cpus allowed)"
        n = 0
        for tid in os.listdir("/proc/self/task"):  # sched_setaffinity(0) only moves the calling thread
            try:
                os.sched_setaffinity(int(tid), allowed)
                n += 1
            except OSError:
                pass
        return f"{len(allowed)} GPU-local cpus ({how}), {n} threads bound"
    except Exception as e:  # best effort: the bench still runs, only the copy may be slower
        return f"not bound ({type(e).__name__}: {e})"


def synth_targets(B, seed):
    """SURVEY.md section 8(d): per image G in U{1..20} boxes, cls U{0..79}, cx,cy in U(0.1,0.9), w,h in U(0.05,0.5)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    rows = []
    for b in range(B):
        n = int(torch.randint(1, 21, (1,), generator=g))
        t = torch.empty(n, 6)
        t[:, 0] = b
        t[:, 1] = torch.randint(0, 80, (n,), generator=g).float()
        t[:, 2:4] = torch.rand(n, 2, generator=g) * 0.8 + 0.1
        t[:, 4:6] = torch.rand(n, 2, generator=g) * 0.45 + 0.05
        rows.append(t)
    return torch.cat(rows)


def train_main(args, rank, world, local_rank):
    """BASELINE configs[3]: YOLOv11s training step (train-mode forward with batch-statistics BatchNorm, v8DetectionLoss
    incl. the task-aligned assigner, backward through the whole graph, ONE NCCL all-reduce of the flat gradient buffer
    when N > 1, AdamW), batch 16 per GPU.  Dense convolutions (forward, dgrad, wgrad) run on the TF32 tcgen05 kernels
    (csrc/conv_tf32.cu; --train-kernels f32 times the fp32 CUDA-core parity kernels instead); depthwise convolutions,
    attention, BatchNorm / SiLU, the loss and AdamW are fp32 CUDA-core kernels of the library."""
    model = args.model if args.model.startswith("v11") else "v11s"
    arch, size, task, gflop_img = MODELS[model]
    B = args.batch if args.batch != 32 else 16
    config = {"workload": f"YOLO{model} detect training step (fwd + DFL/CIoU/BCE loss + bwd + AdamW), batch {B}x3x640x640 per GPU",
              "model": model, "batch_per_gpu": B, "global_batch": B * world, "imgsz": 640, "weights": "seeded synthetic",
              "parallelism": f"data-parallel x{world}" + (" + NCCL all-reduce of the flat gradient buffer" if world > 1 else "")}
    if args.impl == "reference":
        if rank != 0:
            return
        import torch
        from oracle import loss as oloss
        from tests.util import oracle_model, synth_image
        sb = 2  # bounded sample: the CPU step is ~2 s per image
        m = oracle_model(arch, task, size).train()
        opt = torch.optim.AdamW([p for k, p in m.named_parameters() if ".dfl." not in k], lr=1.19e-4, weight_decay=5e-4)
        crit = oloss.V8DetectionLoss(80)
        x, t = synth_image(sb, 640, 640), synth_targets(sb, 1)
        batch = {"batch_idx": t[:, 0], "cls": t[:, 1], "bboxes": t[:, 2:]}

        def step():
            _, preds = m(x)
            loss, _ = crit(preds, batch)
            opt.zero_grad()
            loss.sum().backward()
            opt.step()
        for _ in range(min(args.warmup, 1)):
            step()
        n = args.steps
        t0 = time.perf_counter()
        for _ in range(n):
            step()
        dt = (time.perf_counter() - t0) / n
        val = sb / dt
        print(json.dumps({"impl": "reference", "metric": f"train images/sec YOLO{model} 3x640x640", "value": round(val, 3),
                          "unit": "images/s", "n_gpus": args.gpus, "steps": n, "warmup": min(args.warmup, 1), "ms_per_step": round(dt * 1e3, 1),
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": config,
                          "cpu_baseline": {"value": round(val, 3), "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
                                           "sample": f"{sb} of {B} images per step, {n} steps (oracle autograd step on the host cores)"},
                          "e2e": {"value": round(val, 3), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    import torch
    import torch.distributed as dist
    from tests.util import oracle_model, synth_image
    from yolosharp_b200.train_v11 import KernelOpsV11, TrainStepV11
    assert torch.cuda.is_available(), "bench.py needs a B200"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    m = oracle_model(arch, task, size)
    tc = args.train_kernels == "tc"
    native = args.train_impl == "native" and tc
    if native:  # ONE C-ABI call per step (csrc/train_step.cu); the flat buffers are torch tensors of this process
        from yolosharp_b200.train_native import NativeTrainer
        st = NativeTrainer({k: v.detach().clone() for k, v in m.state_dict().items()}, "v11", size, 80, device=dev, max_batch=B)
    else:
        st = TrainStepV11({k: v.detach().clone() for k, v in m.state_dict().items()}, size, 80, device=dev, ops=KernelOpsV11(tensor_cores=tc))
    del m
    xs = [synth_image(B, 640, 640, seed=300 + rank * 4 + i).to(dev) for i in range(2)]
    ts = [synth_targets(B, 400 + rank * 4 + i) for i in range(2)]
    u8 = [synth_image(B, 640, 640, seed=300 + rank * 4 + i, dtype=torch.uint8).pin_memory() for i in range(2)]
    for i in range(args.warmup):
        st.step(xs[i & 1], ts[i & 1])
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank) if rank == 0 and not os.environ.get("YB_NO_SAMPLER") else None
    if world > 1:
        dist.barrier()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        _t0 = time.perf_counter()
        items = st.step(xs[i & 1], ts[i & 1])
        if os.environ.get("YB_STEP_TIMES"):
            torch.cuda.synchronize()
            print(f"step {i}: {(time.perf_counter() - _t0) * 1e3:.1f} ms", file=sys.stderr)
    e1.record()
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:  # the step hands its caller the loss items and leaves the updated weights
        dump_outputs(args.dump_outputs, {"loss_items": items, "weights": st.flat if native else st.P.flat})
    if world > 1:
        dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    clocks = sampler.stop() if sampler else None
    # e2e: pinned uint8 images -> device (scaled by 1/255 there), step, loss items back on the host.  The copy of step i+1's
    # images runs on a side stream into the other of two device slots while step i computes (what a prefetching loader
    # does); every step's copy is inside the timed region.
    n2 = max(2, args.steps)
    slots = [torch.empty((B, 3, 640, 640), dtype=torch.uint8, device=dev) for _ in range(2)]
    cs, cur = torch.cuda.Stream(dev), torch.cuda.current_stream(dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    free = [torch.cuda.Event() for _ in range(2)]

    def issue(i):
        with torch.cuda.stream(cs):
            cs.wait_event(free[i & 1])
            slots[i & 1].copy_(u8[i & 1], non_blocking=True)
            ready[i & 1].record(cs)

    def e2e_step(i, last):
        if not last:
            issue(i + 1)
        cur.wait_event(ready[i & 1])
        x = slots[i & 1] if native else slots[i & 1].float().mul_(1 / 255.0)
        items = st.step(x, ts[i & 1]).cpu()
        free[i & 1].record(cur)
        return items

    for e in free:
        e.record(cur)
    issue(0)
    e2e_step(0, False)  # untimed: first use of the slots and of the side stream
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(1, n2 + 1):
        host_items = e2e_step(i, i == n2)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        peaks = load_peaks()
        value = world * B * args.steps / (ms_total / 1e3)
        tflops = 3 * gflop_img * 1e9 * value / world / 1e12  # fwd + dgrad + wgrad ~ 3x the forward MACs
        print(json.dumps({"metric": f"train images/sec YOLO{model} 3x640x640", "value": round(value, 2), "unit": "images/s",
                          "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 2),
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "tf32" if tc else "f32",
                          "data": "synthetic", "config": dict(config, step="native (yb_train_step)" if native else "python graph walk"), "clocks": clocks,
                          "e2e": {"value": round(world * B * n2 / float(t.item()), 2), "unit": "images/s",
                                  "h2d_bytes_per_step": B * 3 * 640 * 640, "d2h_bytes_per_step": 12, "steps": n2,
                                  "api": ("yb_train_backward + yb_train_apply (one native graph walk per step; pinned uint8 images in, loss items out)"
                                          if native else "TrainStepV11.step over the C-ABI training kernels (pinned uint8 images in, loss items out)")},
                          "loss_items": [round(float(v), 4) for v in host_items],
                          "roofline": {"bound": "tensor", "achieved": round(tflops, 2), "peak": peaks["tc"], "unit": "TFLOP/s",
                                       "frac": round(tflops / peaks["tc"], 5), "traffic": None,
                                       "kernel": "tf_conv_kernel / tf_wgrad_kernel (TF32 tcgen05)" if tc else
                                                 "conv_generic / conv_backward_data / conv_backward_weight (fp32 CUDA cores)",
                                       "note": "whole-step figure: 3 x forward conv FLOPs / step time, against the sustained "
                                               "bf16 tensor peak (TF32 peaks at half of it); the step also holds the fp32 "
                                               "BatchNorm / SiLU / loss / AdamW kernels and the host-side launch chain"}}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="v8n", choices=sorted(MODELS))
    ap.add_argument("--batch", type=int, default=32, help="images per GPU per step")
    ap.add_argument("--gather", default="comm", choices=["comm", "nccl"], help="N > 1: detection exchange")
    ap.add_argument("--train-impl", default="native", choices=["native", "python"],
                    help="--mode train: the native step (csrc/train_step.cu) or the Python graph walk over the same kernels")
    ap.add_argument("--train-kernels", default="tc", choices=["tc", "f32"],
                    help="--mode train: dense convolutions on the TF32 tcgen05 kernels (default) or the fp32 parity kernels")
    ap.add_argument("--mode", default="infer", choices=["infer", "train"],
                    help="train: one YOLOv11s training step (fwd + v8DetectionLoss + bwd + all-reduce + AdamW), BASELINE configs[3]")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-real-weights", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (inputs are seeded, so two "
                         "builds run with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.mode == "train":
        return train_main(args, rank, world, local_rank)
    arch, size, task, gflop_img = MODELS[args.model]
    workload = (f"YOLO{args.model} {task} inference (forward+decode+NMS" + ("+masks" if task == "segment" else "") +
                f"), batch {args.batch}x3x640x640 per GPU")
    # identical in both arms (the driver compares it); arm-specific facts live outside `config`
    config = {"workload": workload, "model": args.model, "batch_per_gpu": args.batch, "global_batch": args.batch * world,
              "imgsz": 640, "conf": CONF, "iou": IOU, "max_det": MAX_DET, "weights": "seeded synthetic",
              "parallelism": f"batch-sharded x{world}"}

    if args.impl == "reference":
        if rank != 0:
            return
        val, ms, cores = cpu_reference_run(args.model, args.batch, args.steps, args.warmup)
        line = {"impl": "reference", "metric": f"images/sec YOLO{args.model} 3x640x640", "value": round(val, 2),
                "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": round(val, 2), "unit": "images/s", "cores": cores, "host_cpus": os.cpu_count(), "kind": "port",
                                 "sample": f"all {args.batch} images per step, {args.steps} steps, fp32; PyTorch-CPU "
                                           "restatement of the TorchSharp op sequence (the C# reference cannot run: no .NET)"},
                "e2e": {"value": round(val, 2), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    import yolosharp_b200 as y
    from yolosharp_b200 import dist as ydist
    from tests.util import oracle_model, synth_image
    assert torch.cuda.is_available(), "bench.py needs a B200 (no CPU fallback in the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    torch.cuda.init()
    host = {"affinity": bind_to_gpu_numa(local_rank), "omp_threads": torch.get_num_threads()}
    if world > 1:
        opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)
    B = args.batch
    seg = task == "segment"
    ROW = 6 + (32 if seg else 0)

    def make_engine(state_dict):
        eng = y.Engine(arch, size, task, 80, "f16", local_rank, B, 640, 640)
        eng.load_state_dict(state_dict)
        eng.finalize()
        return eng

    m = oracle_model(arch, task, size)  # seeded synthetic weights (weights only; the oracle net is not run here)
    eng = make_engine(m.state_dict())
    del m
    A, Cp = eng.anchors, eng.pred_channels
    gatherer = ydist.DetectionGather(B, MAX_DET, ROW, dev, mode=args.gather, slots=max(2, E2E_SLOTS)) if world > 1 else None

    def timed_run(eng, xs, steps, warmup, with_gather, snapshot=False):
        """Two-deep software pipeline: forward(i+1) runs on stream s_f while NMS (+ masks, + gather) of batch i runs on
        stream s_n, each with its own prediction / detection buffers - every step does all of its work inside the
        timed region.  Returns (ms_total over `steps`, mean detections per image, last pred buffer, forward-only ms per
        step, the last timed step's outputs if `snapshot` else None)."""
        s_f, s_n = torch.cuda.Stream(dev, priority=-1), torch.cuda.Stream(dev, priority=-1)
        preds = [torch.empty((B, Cp, A), dtype=torch.float32, device=dev) for _ in range(2)]
        protos = [torch.empty((B, 32, 160, 160), dtype=torch.float32, device=dev) for _ in range(2)] if seg else None
        mask_buf = [torch.empty((B, MAX_DET, 640, 640), dtype=torch.uint8, device=dev) for _ in range(2)] if seg else None
        if with_gather:
            detb = [gatherer.local_buffers(b) for b in range(2)]
        else:
            detb = [ydist.packed_detection_buffers(B, MAX_DET, ROW, dev) for _ in range(2)]
        keepb = [torch.empty((B, MAX_DET), dtype=torch.int32, device=dev) for _ in range(2)]
        ev_f = [torch.cuda.Event() for _ in range(2)]
        ev_n = [torch.cuda.Event() for _ in range(2)]

        def step(i):
            b = i & 1
            s_f.wait_event(ev_n[b])  # pred buffer b is free once NMS of step i-2 has consumed it
            eng.forward(xs[i % len(xs)], preds[b], protos[b] if seg else None, stream=s_f)
            ev_f[b].record(s_f)
            s_n.wait_event(ev_f[b])
            y.nms(preds[b], CONF, IOU, MAX_DET, 80, out=(detb[b][0], detb[b][1], keepb[b]), stream=s_n)
            if seg:  # instance masks of the kept detections (Ops.process_mask, upsample=true)
                y.masks(protos[b], detb[b][0], detb[b][1], 640, 640, stream=s_n, out=mask_buf[b])
            if with_gather:
                gatherer.gather(b, stream=s_n)
            ev_n[b].record(s_n)

        for i in range(max(warmup, 8)):  # >= 8 so every (input, buffer) pair has its CUDA graph captured
            step(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s_f)
        for i in range(steps):
            step(i)
        s_f.wait_stream(s_n)
        e1.record(s_f)
        torch.cuda.synchronize()
        last = None
        if snapshot:  # rows past an image's detection count hold stale data: they are not part of the result
            b = (steps - 1) & 1
            dets, counts = gatherer.gathered(b) if with_gather else detb[b][:2]  # all ranks' images when gathered
            rows = torch.arange(MAX_DET, device=dev)
            valid, local = rows < counts[:, None], rows < detb[b][1][:, None]
            last = {"pred": preds[b].clone(), "detections": torch.where(valid[..., None], dets, 0.0), "counts": counts.clone(),
                    "keep": torch.where(local, keepb[b], -1)}
            if seg:
                last["masks"] = mask_buf[b].masked_fill_(~local[:, :, None, None], 0)
        if world > 1:
            dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # forward alone (graph replay, same buffers): the time the roofline record is derived from
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(s_f)
        for i in range(steps):
            eng.forward(xs[i % len(xs)], preds[i & 1], protos[i & 1] if seg else None, stream=s_f)
        f1.record(s_f)
        torch.cuda.synchronize()
        return float(t.item()), float(detb[0][1].float().mean().item()), preds[0], f0.elapsed_time(f1) / steps, last

    xs = [synth_image(B, 640, 640, seed=100 + rank * 8 + i, dtype=torch.float16).to(dev) for i in range(4)]
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_total, mean_dets, pred, fwd_ms, last = timed_run(eng, xs, args.steps, args.warmup, world > 1,
                                                        snapshot=bool(args.dump_outputs) and rank == 0)
    clocks = sampler.stop() if sampler else None
    if last is not None:
        dump_outputs(args.dump_outputs, last)
        del last
    value = world * B * args.steps / (ms_total / 1e3)

    # ---- the same measurement on the reference's shipped checkpoint + its test images (v8n detect only) ----
    real = None
    if args.model == "v8n" and world == 1 and not args.no_real_weights:
        try:
            import numpy as np
            from tests.test_gpu_fp16_pinned import image_batch
            z = np.load(os.path.join(ROOT, "tests", "golden", "yolov8n_f16.npz"))
            eng_r = make_engine({k: torch.from_numpy(z[k]) for k in z.files})
            u8 = image_batch(B)
            xr = [torch.roll(u8, shifts=i, dims=0).to(dev) for i in range(4)]  # uint8 input: /255 fused into the stem
            ms_r, dets_r, _, fwd_r, _ = timed_run(eng_r, xr, max(10, args.steps // 2), args.warmup, False)
            real = {"value": round(B * max(10, args.steps // 2) / (ms_r / 1e3), 1), "unit": "images/s",
                    "weights": "reference Yolov8n.bin (tests/golden/yolov8n_f16.npz)",
                    "inputs": "32 x 640x640 uint8 built from the reference's 5 test images (pad 114, rolled copies)",
                    "forward_ms_per_step": round(fwd_r, 4), "mean_detections_per_image": round(dets_r, 2)}
            eng_r.close()
            del eng_r, xr
        except Exception as ex:  # fixtures missing: report why instead of failing the bench
            real = {"value": None, "error": f"{type(ex).__name__}: {ex}"}

    # ---- e2e: host uint8 images -> host detections through the pipelined C-ABI call pair
    #      yb_predict_u8_submit / yb_predict_u8_wait (two slots: H2D+forward+NMS[+gather]+D2H of step i+1 overlap step i) ----
    e2e_val, e2e_steps, d2h = None, 0, 0
    if not (seg and world > 1):
        NS = E2E_SLOTS
        torch.set_num_threads(1)  # the serving loop is ctypes calls only; idle intra-op workers cost it 15 % (profiles/r2_exp_e2e_matrix.txt)
        host["omp_threads_e2e"] = 1
        u8 = [synth_image(B, 640, 640, seed=200 + rank * 8 + i, dtype=torch.uint8).pin_memory() for i in range(NS)]
        GB = world * B if world > 1 else B
        dh = [torch.empty((GB, MAX_DET, ROW), dtype=torch.float32).pin_memory() for _ in range(NS)]
        ch = [torch.empty((GB,), dtype=torch.int32).pin_memory() for _ in range(NS)]
        d2h = GB * MAX_DET * ROW * 4 + GB * 4
        if seg:  # Segmenter.ImagePredict path: masks of the first MASK_CAP detections of every image come back as bytes
            mhost = [torch.empty((B, MASK_CAP, 640, 640), dtype=torch.uint8).pin_memory() for _ in range(NS)]
            d2h += B * MASK_CAP * 640 * 640
        e2e_steps = max(3 * NS, args.steps // 2)

        def submit(i):
            k = i % NS
            if world > 1:
                gatherer.predict_submit(eng, k, u8[k], dh[k], ch[k], CONF, IOU)
            elif seg:
                eng.predict_seg_u8_submit(k, u8[k], dh[k], ch[k], mhost[k], CONF, IOU, MAX_DET)
            else:
                eng.predict_u8_submit(k, u8[k], dh[k], ch[k], CONF, IOU, MAX_DET)

        def wait(slot):
            if world > 1:
                gatherer.predict_wait(eng, slot)
            else:
                eng.predict_u8_wait(slot)
        for i in range(3 * NS):
            submit(i)
            wait(i % NS)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            if i >= NS:
                wait(i % NS)  # results of step i-NS are in host memory
            submit(i)
        for k in range(NS):
            wait(k)
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_val = world * B * e2e_steps / float(t.item())

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel, from the graph-replayed forward ----
    peaks = load_peaks()
    prof = eng.profile(xs[0], pred)  # per-op algorithmic flops / bytes / kind (its eager times are NOT used)
    proto_dummy = torch.empty((B, 32, 160, 160), dtype=torch.float32, device=dev) if seg else None
    other_ms, others = 0.0, []
    for r in prof:
        if r["kind"] == 0 or r["kind"] == 6 and r["flops"] == 0 and r["ms"] < 0.004:
            continue
        if r["kind"] == 0:
            continue
        t_op = eng.time_op(r["index"], xs[0], pred, proto_dummy, reps=20)
        if r["kind"] == 6 and t_op < 0.003:  # fused decode placeholders launch nothing
            continue
        other_ms += t_op
        others.append({"name": r["name"], "ms": round(t_op, 4)})
    tc = [r for r in prof if r["kind"] == 0]
    tc_flops = sum(r["flops"] for r in tc)
    tc_bytes = sum(r["bytes"] for r in tc)
    tc_ms = max(fwd_ms - other_ms, 1e-6)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r2_conv_traffic.json")
    if os.path.exists(tpath):  # dram bytes of the same launches from an ncu capture (tools/ncu_traffic.py)
        tj = json.load(open(tpath))
        if tj.get("model") == args.model and tj.get("batch") == B:
            traffic = tj["dram_bytes_per_step"]
    t_tc = tc_flops / (peaks["tc"] * 1e12)
    t_hbm = tc_bytes / (peaks["hbm"] * 1e9)
    if t_hbm >= t_tc:
        ach = tc_bytes / (tc_ms / 1e3) / 1e9
        roof = {"bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm"], "unit": "GB/s",
                "frac": round(ach / peaks["hbm"], 4)}
    else:
        ach = tc_flops / (tc_ms / 1e3) / 1e12
        roof = {"bound": "tensor", "achieved": round(ach, 2), "peak": peaks["tc"], "unit": "TFLOP/s",
                "frac": round(ach / peaks["tc"], 4)}
    comp_mb = COMPULSORY_MB_IMG[task] * B
    roof.update({"traffic": traffic, "kernel": "conv_tc_kernel", "launches_per_step": len(tc),
                 "kernel_ms_per_step": round(tc_ms, 4), "forward_ms_per_step": round(fwd_ms, 4),
                 "other_kernels_ms_per_step": round(other_ms, 4), "other_kernels": others,
                 "share_of_step": round(tc_ms / (ms_total / args.steps), 3),
                 "how": "graph-replayed forward timed with CUDA events minus the non-conv kernels timed back to back "
                        "(yb_time_op); bytes = SURVEY 8(d) unfused layer bytes (in + out + residual + weights per launch)",
                 "algorithmic_gflop_per_step": round(tc_flops / 1e9, 2), "algorithmic_mb_per_step": round(tc_bytes / 1e6, 1),
                 "compulsory_mb_per_step": round(comp_mb, 1),
                 "traffic_over_compulsory": round(traffic / 1e6 / comp_mb, 2) if traffic else None,
                 "tensor_tflops": round(tc_flops / (tc_ms / 1e3) / 1e12, 2),
                 "tensor_frac_sustained": round(tc_flops / (tc_ms / 1e3) / 1e12 / peaks["tc"], 4),
                 "hbm_gbs": round(tc_bytes / (tc_ms / 1e3) / 1e9, 1), "peak_source": peaks["src"] + ", sustained TC",
                 "whole_net_tflops": round(gflop_img * 1e9 * value / world / 1e12, 2)})

    line = {"metric": f"images/sec YOLO{args.model} 3x640x640", "value": round(value, 1), "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": config, "clocks": clocks, "host": host,
            "timing": {"l2": "4 rotating input batches (>L2) and ~1 GB of activations rewritten per step",
                       "pipeline": "forward(i+1) overlaps NMS(i) on a second stream (double-buffered outputs)",
                       "gather": (gatherer.describe() if gatherer else None)},
            "e2e": {"value": round(e2e_val, 1) if e2e_val else None, "unit": "images/s", "h2d_bytes_per_step": B * 3 * 640 * 640,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "api": (f"yb_predict_seg_u8_submit/_wait, {E2E_SLOTS} slots (pinned host uint8 in; detections + {MASK_CAP} byte masks per image out)" if seg else
                            f"yb_predict_u8_submit/_wait, {E2E_SLOTS} slots (pinned host uint8 in, host detections out)") +
                           (", detections of all ranks gathered before the D2H copy" if world > 1 else "")},
            "gpu_launches": (eng.launches_per_forward() + 2 + (1 if seg else 0) + (3 if world > 1 else 0)) * args.steps,
            "launches_per_step": eng.launches_per_forward() + 2 + (1 if seg else 0) + (3 if world > 1 else 0),
            "mean_detections_per_image": round(mean_dets, 1), "roofline": roof}
    if real is not None:
        line["real_weights"] = real
    if world == 1 and not args.no_cpu_baseline:
        cb_b, cb_steps = 8, 10
        val, ms, cores = cpu_reference_run(args.model, cb_b, cb_steps, 3)
        line["cpu_baseline"] = {"value": round(val, 2), "unit": "images/s", "cores": cores, "host_cpus": os.cpu_count(), "kind": "port",
                                "sample": f"batch {cb_b} x {cb_steps} steps of the same workload (fp32, PyTorch-CPU oracle "
                                          "= restated TorchSharp op sequence; C# reference not runnable here)"}
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
