#!/usr/bin/env python
"""Benchmark of the HRNet-OCR-MScale hot path (BASELINE.json metric: 1024x2048 crops/sec, fwd+bwd).

  python bench.py --gpus N --steps K --warmup W            # B200 path (this repo), one rank per GPU under torchrun
  python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host CPU cores (oracle)

A step = one training iteration on one synthetic batch per GPU: zero_grad -> net(inputs) (fused fwd+bwd step through
the C ABI) -> loss.backward() (publish / all-reduce gradients) -> SGD step. Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# The SyncBN exchange spins inside kernels of two concurrent streams per GPU: give every stream its own hardware work
# queue (the default 8 connections can alias streams and turn a peer wait into a false cross-stream dependency).
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "semantic-segmentation_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

# Algorithmic work per 1024x2048 crop (SURVEY.md §8d / BASELINE.md §2, conv FLOPs = 2*MAC)
TFLOP_PER_CROP = {"ocrnet.HRNet_Mscale": 10.53, "ocrnet.HRNet": 7.77, "deepv3.DeepV3PlusW38": 34.95}
FWD_TFLOP_1X = 3.0546
# Launch-level roofline of one train step per 1024x2048 crop: sum over the step's launches of max(FLOPs / sustained bf16
# peak, bytes / HBM copy bandwidth), from the static trace of the real step program (tools/trace_step.py,
# profiles/r1_step_roofline_model.txt; peaks of MEASURED_PEAKS.json: 1386.7 TFLOP/s, 6572.9 GB/s)
# BatchNorm at --gpus N > 1: per-GPU statistics unless --syncbn. Every reference script trains with syncbn: true and the
# NVLink exchange is validated and measured at N = 2 (tests/test_gpu_multi.py, DESIGN.md 6) - but never at N = 4 / 8 (the
# round's GPU budget), so the driver's 1 -> 8 scaling runs use the configuration that is known to complete.
SYNCBN_DEFAULT = False
STEP_ROOFLINE_MS = {"ocrnet.HRNet_Mscale": 15.12, "ocrnet.HRNet": 11.34, "deepv3.DeepV3PlusW38": 30.8}
# the same model per kernel class (profiles/r2_step_roofline_model.txt): class -> (kernel-name fragments, roofline ms)
KERNEL_CLASSES = {
    "conv fwd+dgrad (tcgen05)": (("conv3x3_halo", "conv_igemm"), 2.960 + 2.954 + 0.135),
    "conv wgrad (tcgen05 + slab reduce)": (("wgrad_igemm", "wgrad_reduce"), 3.127),
    "batchnorm passes": (("bn_",), 2.405 + 1.672 + 1.225),
    "resample / fuse / accumulate": (("fuse_fwd", "upsample_adjoint", "masked_accum", "image_prep"), 0.359),
    "loss + OCR softmaxes": (("loss_fwd", "_bwd_kernel", "mid_fwd", "softmax", "spatial_", "count_valid", "colsum",
                              "cast_rows", "transpose_pad", "rmi_"), 0.19),
    "weights / gradients / optimizer": (("pack_weights", "grad_fold", "publish_grads", "sgd_step", "running_update"), 0.27 + 0.8),
}


def kernel_class_table(step_fn, ms_per_step):
    """One extra step under Kineto/CUPTI: per kernel class the launches, the summed kernel durations, their share of all
    kernel time, the union (wall-clock during which at least one kernel of the class runs) and the launch-level roofline
    time of the class. Durations come from the profiler run (a few % slower than the timed loop), shares are what matter."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step_fn()
        torch.cuda.synchronize()
    ev = []
    for e in prof.profiler.kineto_results.events():
        try:
            if "cuda" not in str(e.device_type()).lower():
                continue
            t0 = e.start_ns() if hasattr(e, "start_ns") else e.start_us() * 1000
            d = e.duration_ns() if hasattr(e, "duration_ns") else e.duration_us() * 1000
            ev.append((int(t0), int(t0 + d), e.name()))
        except Exception:
            continue
    if not ev:
        return None

    def union(iv):
        tot, a0, b0 = 0, None, None
        for a, b in sorted(iv):
            if b0 is None or a > b0:
                if b0 is not None:
                    tot += b0 - a0
                a0, b0 = a, b
            else:
                b0 = max(b0, b)
        return tot + ((b0 - a0) if b0 is not None else 0)

    total = sum(b - a for a, b, _ in ev)
    span = max(b for _, b, _ in ev) - min(a for a, _, _ in ev)
    out, used = {}, set()
    for cname, (keys, roof_ms) in KERNEL_CLASSES.items():
        idx = [i for i, (_, _, n) in enumerate(ev) if i not in used and any(k in n for k in keys)]
        used.update(idx)
        iv = [(ev[i][0], ev[i][1]) for i in idx]
        sm = sum(b - a for a, b in iv) / 1e6
        out[cname] = dict(launches=len(iv), sum_ms=round(sm, 3), share_of_kernel_time=round(sm * 1e6 / max(total, 1), 4),
                          union_ms=round(union(iv) / 1e6, 3), roofline_ms=round(roof_ms, 3),
                          roofline_frac=round(roof_ms / sm, 3) if sm > 0 else None)
    rest = [(a, b) for i, (a, b, _) in enumerate(ev) if i not in used]
    out["other (ATen fills, NCCL ...)"] = dict(launches=len(rest), sum_ms=round(sum(b - a for a, b in rest) / 1e6, 3))
    out["_step"] = dict(kernels=len(ev), span_ms=round(span / 1e6, 3), all_kernels_union_ms=round(union([(a, b) for a, b, _ in ev]) / 1e6, 3),
                        all_kernels_sum_ms=round(total / 1e6, 3), timed_ms_per_step=round(ms_per_step, 3))
    return out



def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of every measurement of this path (headline, end-to-end, recipe and other "
                         "configurations); the stock-PyTorch and CPU baselines time fixed short samples")
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--arch", default="ocrnet.HRNet_Mscale", choices=list(TFLOP_PER_CROP))
    ap.add_argument("--height", type=int, default=1024)
    ap.add_argument("--width", type=int, default=2048)
    ap.add_argument("--batch-per-gpu", type=int, default=1)
    ap.add_argument("--sup-wt", type=float, default=0.0)
    ap.add_argument("--criterion", default="ce", choices=["ce", "rmi"])
    ap.add_argument("--syncbn", dest="syncbn", action="store_true", default=None,
                    help="synchronise BatchNorm statistics across the GPUs through NVLink peer memory (syncbn: true in every "
                         "reference script); validated at N = 2")
    ap.add_argument("--no-syncbn", dest="syncbn", action="store_false", help="per-GPU BatchNorm statistics at N > 1 (default)")
    ap.add_argument("--torch-sgd", action="store_true", help="torch.optim.SGD instead of b200seg.optim.FusedSGD")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--torch-gpu-baseline", action="store_true",
                    help="time the reference algorithm through stock PyTorch (ATen / cuDNN, autocast bf16 and fp32) on "
                         "this GPU: the practical kernel to beat (BASELINE.md §3b step 5); adds `torch_gpu_baseline` and "
                         "`vs_torch_gpu` to the line. Default at --gpus 1; this flag forces it for N > 1 (rank 0)")
    ap.add_argument("--no-torch-gpu-baseline", action="store_true")
    ap.add_argument("--no-recipe", action="store_true", help="skip the second (RMI + supervised multi-scale) measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned to its caller as DIR/<name>.npy (float32): the loss, a "
                         "fixed seeded sample of the gradients and of the updated parameters, the BatchNorm running "
                         "statistics; the inputs depend on the arguments only, so two builds compare output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sust=p.get("bf16_tflops_sustained",
                                                                                     p["bf16_tflops"]), src="measured")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(smax) if smax else None,
                    reasons=sorted(reasons), samples=len(sm))


def usable_cores():
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 64))


def workload_name(args):
    """config.workload, identical for both arms (the driver pairs their lines)."""
    kind = "two-scale {0.5,1.0}" if args.arch in ("ocrnet.HRNet_Mscale", "mscale.HRNet") else "single-scale"
    return ("%s %s train step (zero_grad, fwd+bwd, SGD momentum + weight decay), %dx%d crops, "
            "%d crop/GPU, %s loss" % (args.arch, kind, args.height, args.width, args.batch_per_gpu, args.criterion.upper()))


DUMP_SAMPLE = 4 * 1024 * 1024      # elements of each sampled array: 16 MB in float32


def dump_outputs(out_dir, net, loss):
    """--dump-outputs: the loss of the last step, the gradients it published into param.grad and the parameters the
    optimizer left, both at the same DUMP_SAMPLE indices drawn from a fixed seed over the parameters in registration
    order, and every BatchNorm running mean / variance."""
    import numpy as np
    params = [p for _, p in net.named_parameters()]
    grads = torch.cat([p.grad.reshape(-1) for p in params])
    values = torch.cat([p.detach().reshape(-1) for p in params])
    g = torch.Generator().manual_seed(2024)
    idx = torch.randint(0, grads.numel(), (min(DUMP_SAMPLE, grads.numel()),), generator=g).sort().values
    idx = idx.to(grads.device)
    running = torch.cat([b.reshape(-1).float() for n, b in net.named_buffers() if "running_" in n])
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("loss", loss.detach().reshape(1)), ("grad_sample", grads[idx]), ("param_sample", values[idx]),
                    ("bn_running_stats", running)):
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def synth_batch(n, h, w, seed, device):
    g = torch.Generator().manual_seed(seed)
    images = torch.randn((n, 3, h, w), generator=g)
    gts = torch.randint(0, 19, (n, h, w), generator=g)
    gts[:, :8] = 255
    return images, gts


# ------------------------------------------------------------------------------------------------ reference (CPU) arm
def cpu_reference_step_time(arch, h, w, steps, warmup=1, budget_s=60.0, criterion="ce"):
    """The reference algorithm (oracle/seg_oracle.py, pinned to /root/reference by tests/golden) on the host cores:
    zero_grad -> two-scale fwd -> bwd -> SGD, fp32, PyTorch's default intra-op thread count (= the cores it can use).
    Returns (seconds per step at (h, w), timed steps); stops early once `budget_s` of wall clock is spent."""
    from oracle import seg_oracle as O
    # the cores this process may really use: affinity mask and cgroup CPU quota (a 64-thread pool on an 8-core quota
    # runs the oracle ~10x slower); also undoes torchrun's OMP_NUM_THREADS=1
    torch.set_num_threads(usable_cores())
    sd = O.synth_state_dict(arch, O.HRNET_W48, seed=0)
    params = [v.requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k]
    opt = torch.optim.SGD(params, lr=0.01, momentum=0.9, weight_decay=1e-4)
    images, gts = O.synth_batch(1, h, w, seed=1)
    crit = O.criterion_rmi if criterion == "rmi" else O.criterion_ce
    times = []
    t_start = time.perf_counter()
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad()
        ctx = O.Ctx(sd, training=True)
        if arch == "ocrnet.HRNet_Mscale":
            loss = O.mscale_two_scale(ctx, images, gts, criterion=crit)
        else:
            loss = O.ocrnet_forward(ctx, images, gts, criterion=crit)
        loss.backward()
        opt.step()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
        if times and time.perf_counter() - t_start > budget_s:
            break
    return sum(times) / len(times), len(times)


def torch_gpu_step_time(arch, h, w, autocast, criterion="ce", steps=4, warmup=2):
    """The reference algorithm (oracle restatement = the reference's own call sequence of F.conv2d / batch_norm /
    interpolate / softmax ...) through stock PyTorch on the current GPU: ATen + cuDNN kernels, NCHW, cudnn.benchmark as
    in train.py:330, optionally under torch.autocast(bf16) (the modern spelling of the reference's apex AMP O1).
    Baseline measurement only, rank 0, never on the product path. Returns milliseconds per step (CUDA events)."""
    from oracle import seg_oracle as O
    torch.backends.cudnn.benchmark = True
    sd = {k: v.cuda() for k, v in O.synth_state_dict(arch, O.HRNET_W48, seed=0).items()}
    params = [v.requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k]
    opt = torch.optim.SGD(params, lr=1e-3, momentum=0.9, weight_decay=1e-4)
    images, gts = O.synth_batch(1, h, w, seed=1)
    images, gts = images.cuda(), gts.cuda()
    crit = O.criterion_rmi if criterion == "rmi" else O.criterion_ce

    def step():
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            ctx = O.Ctx(sd, training=True)
            if arch == "ocrnet.HRNet_Mscale":
                loss = O.mscale_two_scale(ctx, images, gts, criterion=crit)
            else:
                loss = O.ocrnet_forward(ctx, images, gts, criterion=crit)
        loss.backward()
        opt.step()

    for _ in range(warmup):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # bounded sample: the full algorithm on a 128x256 crop (1/64 of the pixels); crops/s are rescaled by the pixel ratio
    # (cost is proportional to pixels: every layer is a convolution / pointwise op, SURVEY.md §8d)
    sh, sw = max(64, args.height // 8), max(128, args.width // 8)
    sec, timed = cpu_reference_step_time(args.arch, sh, sw, max(1, args.steps), warmup=1 if args.warmup else 0,
                                         budget_s=90.0, criterion=args.criterion)
    ratio = (sh * sw) / float(args.height * args.width)
    value = ratio / sec
    cores = torch.get_num_threads()
    line = dict(metric="1024x2048 crops/sec fwd+bwd HRNet-OCR-MScale", value=value, unit="crops/s", impl="reference",
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=1000.0 / value,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="fp32", data="synthetic",
                config=dict(workload=workload_name(args)),
                cpu_baseline=dict(value=value, unit="crops/s", cores=cores, kind="port",
                                  sample="%d timed step(s) of the full algorithm at %dx%d (1/%d of the pixels, 90 s "
                                         "budget), rescaled by the pixel ratio" % (timed, sh, sw, round(1 / ratio))),
                e2e=dict(value=value, unit="crops/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ B200 arm
def dominant_kernel_roofline(pk):
    """conv3x3_ocr (720->512 @256x512, the largest single kernel, SURVEY §2b K2) timed alone with CUDA events; L2 is
    flushed between iterations by writing a 256 MB buffer."""
    from b200seg import raw
    x = torch.randn((1, 256, 512, 720), device="cuda").to(torch.bfloat16)
    wt = torch.randn((512, 720, 3, 3), device="cuda") * 0.02
    bias = torch.zeros(512, device="cuda")
    w_f, _ = raw.pack_weight(wt, want_dgrad=False)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        raw.conv2d_fwd(x, w_f, bias, emit_stats=True)
    torch.cuda.synchronize()
    ms = []
    for _ in range(8):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        raw.conv2d_fwd(x, w_f, bias, emit_stats=True)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    t = ms[len(ms) // 2]
    flops = 2.0 * 256 * 512 * 720 * 512 * 9
    achieved = flops / (t * 1e-3) / 1e12
    # DRAM traffic of this launch from the committed `ncu --set full` capture (profiles/r1_ncu_full_prof_ocr.txt:
    # dram__bytes_read.sum 195.6 MB + dram__bytes_write.sum 100.6 MB); algorithmic bytes = in + out + weights in bf16
    algo_bytes = 2.0 * (256 * 512 * 720 + 256 * 512 * 512 + 512 * 720 * 9)
    return dict(bound="tensor", kernel="conv3x3_halo_kernel (conv3x3_ocr 720->512 3x3 @256x512, bf16, fp32 accum, "
                                       "BN statistics in the epilogue)",
                achieved=achieved, peak=pk["tf_burst"], unit="TFLOP/s", frac=achieved / pk["tf_burst"],
                peak_source=pk["src"] + " bf16_tflops (burst: kernel timed alone)", ms_per_launch=t,
                traffic=296.26e6, traffic_unit="bytes/launch (ncu dram read+write)",
                traffic_source="profiles/r1_ncu_full_prof_ocr.txt (one ncu --set full capture of this launch; not "
                               "re-measured in this run)", algorithmic_bytes=algo_bytes,
                note="the largest single launch (1.4 % of the step); whole-step figures: model_flops_utilisation, "
                     "step_roofline and kernel_classes")


def time_dominant_kernel_roofline(pk):
    """The kernel that takes the largest share of the step (profiles/r2_launch_summary_step_final.txt: conv3x3_halo_kernel<2>,
    21.6 % of the serialised kernel time, 851 launches) on its most expensive instance: the 48 -> 48 3x3 convolution of the
    high-resolution branch at 256x512 (64 forward launches + their data gradients per 1.0x pass). HBM-bound: algorithmic
    bytes = (in + out) x 2 B + weights = 25.2 MB per launch (SURVEY 8d per-conv figure). Timed alone with CUDA events on the
    launching stream, L2 flushed between iterations by writing a 256 MB buffer."""
    from b200seg import raw
    h, w, c = 256, 512, 48
    x = torch.randn((1, h, w, c), device="cuda").to(torch.bfloat16)
    wt = torch.randn((c, c, 3, 3), device="cuda") * 0.05
    w_f, _ = raw.pack_weight(wt, want_dgrad=False)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        raw.conv2d_fwd(x, w_f, None, emit_stats=True)
    torch.cuda.synchronize()
    ms = []
    for _ in range(12):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        raw.conv2d_fwd(x, w_f, None, emit_stats=True)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    t = ms[len(ms) // 2]
    algo_bytes = 2.0 * (2 * h * w * c + c * c * 9)
    achieved = algo_bytes / (t * 1e-3) / 1e9
    return dict(bound="hbm", kernel="conv3x3_halo_kernel<2> (48->48 3x3 @256x512 of the high-resolution HRNet branch, bf16, "
                                    "fp32 accumulate in TMEM, BN statistics in the epilogue)",
                achieved=achieved, peak=pk["hbm_gbs"], unit="GB/s", frac=achieved / pk["hbm_gbs"],
                peak_source=pk["src"] + " hbm_gbs (copy bandwidth)", ms_per_launch=t,
                traffic=12.70e6, traffic_unit="bytes/launch (ncu dram read+write)",
                traffic_source="profiles/r2_ncu_full_final.txt (ncu --set full of this launch: 12.70 MB read, the 12.6 MB "
                               "output stays in the 126 MB L2 at kernel end; not re-measured in this run)",
                algorithmic_bytes=algo_bytes,
                note="the kernel with the largest share of the step (21.6 % of the serialised kernel time); latency bound "
                     "with two resident CTAs per SM: tensor pipe ~11 %, DRAM ~7 % busy (DESIGN.md 7 gap 1). The largest "
                     "single launch is in roofline_largest_launch; whole-step figures: model_flops_utilisation, "
                     "step_roofline and kernel_classes")


def run_b200(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group(backend="nccl", init_method="env://")
    from b200seg.module import B200SegModule
    from b200seg import _lib

    torch.manual_seed(0)
    if args.syncbn is None:
        args.syncbn = SYNCBN_DEFAULT
    args.syncbn = bool(args.syncbn and world > 1)
    net = B200SegModule(args.arch, 19, criterion=args.criterion, supervised_mscale_wt=args.sup_wt,
                        use_cuda_graph=not args.no_graph, syncbn=args.syncbn).cuda().train()
    net._ddp_allreduce = world > 1
    # well-scaled weights (the reference's default N(0,1e-3) init underflows activations after a few BN-free paths)
    with torch.no_grad():
        for n_, p_ in net.named_parameters():
            if p_.dim() == 4 and n_.startswith("backbone"):
                fan_in = p_.shape[1] * p_.shape[2] * p_.shape[3]
                p_.normal_(0, (2.0 / fan_in) ** 0.5)
    if args.torch_sgd:
        opt = torch.optim.SGD(net.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4)
    else:
        from b200seg.optim import FusedSGD      # same update rule, one launch (SURVEY §8f row f3)
        opt = FusedSGD(net.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4)
    B, H, W = args.batch_per_gpu, args.height, args.width
    images_h, gts_h = synth_batch(B, H, W, 1 + rank, "cpu")
    images_h, gts_h = images_h.pin_memory(), gts_h.pin_memory()
    images_d, gts_d = images_h.cuda(), gts_h.cuda()

    def step(images, gts):
        opt.zero_grad(set_to_none=True)
        loss = net({"images": images, "gts": gts})
        loss.backward()
        opt.step()
        return loss

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    profile_mode = os.environ.get("B200SEG_PROFILE") == "1"     # ncu launch-list runs: 1 warm-up + 1 step, nothing else
    for _ in range(1 if profile_mode else max(args.warmup, 3)):
        step(images_d, gts_d)
    barrier()
    if profile_mode:
        torch.cuda.nvtx.range_push("timed_step")
        step(images_d, gts_d)
        torch.cuda.nvtx.range_pop()
        barrier()
        return
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- device-resident timing
    launches0 = _lib.KERNEL_LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        loss = step(images_d, gts_d)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, net, loss)
    if os.environ.get("B200SEG_TIME_ONLY") == "1":              # A/B runs of a switch: the device-timed figure only
        if rank == 0:
            print(json.dumps(dict(ms_per_step=ms / args.steps, steps=args.steps, time_only=True)))
        return
    # ---- end-to-end timing: pinned host inputs -> H2D every step, loss read back every step.
    # (a) pipelined read: the loss of step i is copied to pinned memory asynchronously and read on the host while step
    #     i+1 is already running (what a training loop that logs asynchronously does);
    # (b) blocking read: loss.item() right after every step (the reference's train.py:499-512 pattern) - this also
    #     exposes the launch latency of the ~4 900-node graph on an idle GPU every step.
    from b200seg.prefetch import DevicePrefetcher

    def host_batches(n):
        for _ in range(n):
            yield {"images": images_h, "gts": gts_h}      # pinned host tensors: every step's inputs cross PCIe again

    pin = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    evts = [torch.cuda.Event() for _ in range(2)]
    t_e0, t_e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    E2E_WARM = 2     # untimed iterations THROUGH the end-to-end path: the first one allocates the staging buffers (a
    #                  one-time ~200 ms cudaMalloc next to the step's 17 GB pools that used to land inside the timed region)
    prev = None
    loss_val = float("nan")
    dbg = os.environ.get("B200SEG_E2E_DEBUG") == "1"
    marks = []
    for i, batch in enumerate(DevicePrefetcher(host_batches(args.steps + E2E_WARM))):   # H2D of step i+1 under step i
        if i == E2E_WARM:
            barrier()
            t_e0.record()
        marks.append(time.perf_counter())
        loss = step(batch["images"], batch["gts"])
        slot = i % 2
        pin[slot].copy_(loss.detach().reshape(1), non_blocking=True)
        evts[slot].record()
        if prev is not None:
            evts[prev].synchronize()
            loss_val = float(pin[prev][0])
        prev = slot
    evts[prev].synchronize()
    loss_val = float(pin[prev][0])
    t_e1.record()
    barrier()
    ms_e2e = t_e0.elapsed_time(t_e1)
    if dbg and rank == 0:
        print("e2e-debug host ms between iterations:", [round((b - a) * 1e3, 1) for a, b in zip(marks, marks[1:])])
    b_e0, b_e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(args.steps + 1):
        if i == 1:                # one untimed iteration through this path as well
            barrier()
            b_e0.record()
        im = images_h.cuda(non_blocking=True)
        gt = gts_h.cuda(non_blocking=True)
        loss = step(im, gt)
        loss_val = loss.item()
    b_e1.record()
    barrier()
    ms_e2e_block = b_e0.elapsed_time(b_e1)
    clocks = sampler.stop() if rank == 0 else None
    # one extra (collective) step under the profiler on EVERY rank: a step contains the all-reduce / SyncBN exchanges
    try:
        classes = kernel_class_table(lambda: step(images_d, gts_d), ms / args.steps)
    except Exception as e:  # noqa
        classes = dict(error=repr(e))
    barrier()
    if dist is not None:
        t = torch.tensor([ms, ms_e2e, ms_e2e_block], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e, ms_e2e_block = float(t[0]), float(t[1]), float(t[2])
    if rank != 0:
        return
    crops = B * world * args.steps
    value = crops / (ms * 1e-3)
    e2e_value = crops / (ms_e2e * 1e-3)
    pk = peaks()
    largest = dominant_kernel_roofline(pk)
    try:
        roof = time_dominant_kernel_roofline(pk)
    except Exception as e:  # noqa  (never lose the bench line over the second measurement)
        roof = dict(largest, fallback_reason=repr(e))
    step_tflops = TFLOP_PER_CROP[args.arch] * (H * W) / (1024.0 * 2048.0) * B / (ms / args.steps * 1e-3) / 1e0
    kernels_per_step = getattr(net, "kernels_per_step", 0)
    line = dict(
        metric="1024x2048 crops/sec fwd+bwd HRNet-OCR-MScale", value=value, unit="crops/s", n_gpus=world,
        steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=ms / args.steps, higher_is_better=True,
        scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
        config=dict(workload=workload_name(args),
                    step="fused fwd+bwd through the C ABI inside one CUDA graph, gradient publish%s, %s" %
                         (" + one NCCL all-reduce over the flat gradient buffer" if world > 1 else "",
                          "torch.optim.SGD" if args.torch_sgd else "b200seg FusedSGD"),
                    batchnorm="SyncBN: per-layer statistics exchanged through NVLink peer memory (non-blocking post in the "
                              "finaliser, one-warp waiter kernels)" if (world > 1 and args.syncbn) else
                              "statistics local to each GPU" + (" (--no-syncbn)" if world > 1 else ""),
                    global_batch=B * world, parallelism="dp%d" % world, cuda_graph=not args.no_graph,
                    l2_policy="per-step working set (>4 GB of activations) far exceeds the 126 MB L2; the "
                              "single-kernel roofline run flushes L2 with a 256 MB write between iterations",
                    model_tflop_per_crop=TFLOP_PER_CROP[args.arch]),
        e2e=dict(value=e2e_value, unit="crops/s", ms_per_step=ms_e2e / args.steps,
                 h2d_bytes_per_step=int(images_h.numel() * 4 + gts_h.numel() * 8), d2h_bytes_per_step=4,
                 api="b200seg.prefetch.DevicePrefetcher(pinned host batches) -> net({'images','gts'}) -> loss.backward() -> "
                     "optimizer.step(); every step's inputs are copied host->device (copy stream, double buffer, "
                     "overlapping the previous step), the loss of every step is copied to pinned host memory and read while "
                     "the next step runs. Steady state of the pipeline after 2 untimed iterations through this path: the copy "
                     "of step i's inputs is issued while step i-1 runs, so the first timed step's inputs crossed PCIe just "
                     "before the region and the region contains steps-2 of the steps copies; blocking_read is the strict "
                     "variant (copy, step, loss.item() inside every timed iteration)",
                 blocking_read=dict(value=crops / (ms_e2e_block * 1e-3), ms_per_step=ms_e2e_block / args.steps,
                                    note="H2D copy of the step's inputs on the compute stream, the step, loss.item() - all "
                                         "inside every timed iteration (exposes the graph-launch latency on an idle GPU "
                                         "each step)")),
        gpu_launches=int(kernels_per_step * args.steps * 3),
        gpu_launches_note="%d b200seg kernels per step (inside one CUDA graph replay), three timed loops" % kernels_per_step,
        model_flops_utilisation=dict(achieved_tflops=step_tflops / 1.0, peak=pk["tf_sust"],
                                     frac=step_tflops / pk["tf_sust"], peak_source=pk["src"] + " sustained bf16"),
        step_roofline=dict(model_ms_per_step=STEP_ROOFLINE_MS[args.arch] * (H * W) / (1024.0 * 2048.0) * B,
                           frac=STEP_ROOFLINE_MS[args.arch] * (H * W) / (1024.0 * 2048.0) * B / (ms / args.steps),
                           what="sum over the step's launches of max(FLOPs/P, bytes/B), static trace of the step "
                                "program (profiles/r1_step_roofline_model.txt)"),
        roofline=roof, roofline_largest_launch=largest, kernel_classes=classes, clocks=clocks, last_loss=loss_val,
        max_memory_allocated_gb=round(torch.cuda.max_memory_allocated() / 2 ** 30, 2))
    if world == 1 and not args.no_recipe and args.criterion == "ce" and args.sup_wt == 0.0:
        # second reported number: the loss recipe of scripts/train_cityscapes.yml (rmi_loss: true,
        # supervised_mscale_loss_wt: 0.05) on the same crop
        try:
            del net, opt
            torch.cuda.empty_cache()
            net2 = B200SegModule(args.arch, 19, criterion="rmi", supervised_mscale_wt=0.05,
                                 use_cuda_graph=not args.no_graph).cuda().train()
            with torch.no_grad():
                for n_, p_ in net2.named_parameters():
                    if p_.dim() == 4 and n_.startswith("backbone"):
                        p_.normal_(0, (2.0 / (p_.shape[1] * p_.shape[2] * p_.shape[3])) ** 0.5)
            from b200seg.optim import FusedSGD as _SGD
            opt2 = _SGD(net2.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4)

            def step2():
                opt2.zero_grad(set_to_none=True)
                l2 = net2({"images": images_d, "gts": gts_d})
                l2.backward()
                opt2.step()
                return l2

            for _ in range(4):
                step2()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            r0.record()
            for _ in range(args.steps):
                l2 = step2()
            r1.record()
            torch.cuda.synchronize()
            ms2 = r0.elapsed_time(r1) / args.steps
            line["train_recipe_rmi_sup"] = dict(value=B * 1000.0 / ms2, unit="crops/s", ms_per_step=ms2, steps=args.steps,
                                                loss=float(l2), what="same step with criterion RMILoss and "
                                                "supervised_mscale_loss_wt 0.05 (scripts/train_cityscapes.yml:21-24)")
            del net2, opt2
        except Exception as e:  # noqa
            line["train_recipe_rmi_sup"] = dict(error=repr(e))
        net = opt = None
    if world == 1 and not args.no_recipe and args.criterion == "ce" and args.sup_wt == 0.0 and (H, W) == (1024, 2048):
        # the other single-GPU configurations of BASELINE.json, measured in the same run (bf16 arithmetic throughout)
        extra = {}
        try:   # cfg2: ocrnet.HRNet (single scale) 1024x2048, 2 crops per step
            torch.cuda.empty_cache()
            net3 = B200SegModule("ocrnet.HRNet", 19, criterion="ce", use_cuda_graph=not args.no_graph).cuda().train()
            from b200seg.optim import FusedSGD as _SGD3
            opt3 = _SGD3(net3.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4)
            im2, gt2 = synth_batch(2, H, W, 7, "cpu")
            im2, gt2 = im2.cuda(), gt2.cuda()
            for it in range(3 + args.steps):
                if it == 3:
                    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize()
                    c0.record()
                opt3.zero_grad(set_to_none=True)
                l3 = net3({"images": im2, "gts": gt2})
                l3.backward()
                opt3.step()
            c1.record()
            torch.cuda.synchronize()
            ms3 = c0.elapsed_time(c1) / args.steps
            extra["cfg2_ocrnet_HRNet_bs2_train"] = dict(
                value=2 * 1000.0 / ms3, unit="crops/s", ms_per_step=ms3, tflops=2 * 7.77 / (ms3 * 1e-3),
                what="ocrnet.HRNet single-scale train step, 2 x 1024x2048 crops per step, CE, bf16 storage / fp32 accumulate "
                     "(BASELINE cfg2 names fp16: this path has one precision policy, bf16)")
            del net3, opt3, im2, gt2
        except Exception as e:  # noqa
            extra["cfg2_ocrnet_HRNet_bs2_train"] = dict(error=repr(e))
        try:   # cfg5: 3-scale inference {0.5, 1.0, 2.0} of a 1024x2048 frame (the 2.0x pass runs at 2048x4096)
            torch.cuda.empty_cache()
            net4 = B200SegModule(args.arch, 19, n_scales=[0.5, 1.0, 2.0]).cuda().eval()
            from b200seg.evaltail import eval_minibatch
            with torch.no_grad():
                for it in range(2 + args.steps):
                    if it == 2:
                        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        torch.cuda.synchronize()
                        c0.record()
                    res = eval_minibatch(net4, images_d, gts_d, scales=(1.0,), do_flip=False)
                c1.record()
                torch.cuda.synchronize()
            ms4 = c0.elapsed_time(c1) / args.steps
            extra["cfg5_three_scale_inference"] = dict(
                value=1000.0 / ms4, unit="frames/s", ms_per_frame=ms4, tflops=16.04 / (ms4 * 1e-3),
                what="ocrnet.HRNet_Mscale nscale_forward {0.5,1.0,2.0} on a 1024x2048 frame + device-side argmax / "
                     "confusion matrix (evaltail.eval_minibatch), eager launches, BatchNorm from running statistics")
            del net4, res
        except Exception as e:  # noqa
            extra["cfg5_three_scale_inference"] = dict(error=repr(e))
        try:   # cfg4: deepv3.DeepV3PlusW38 (WideResNet-38 trunk, dilated ASPP) train step, 1 crop per GPU
            torch.cuda.empty_cache()
            net5 = B200SegModule("deepv3.DeepV3PlusW38", 19, criterion="ce", use_cuda_graph=not args.no_graph).cuda().train()
            from b200seg.optim import FusedSGD as _SGD5
            opt5 = _SGD5(net5.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4)
            for it in range(3 + args.steps):
                if it == 3:
                    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize()
                    c0.record()
                opt5.zero_grad(set_to_none=True)
                l5 = net5({"images": images_d, "gts": gts_d})
                l5.backward()
                opt5.step()
            c1.record()
            torch.cuda.synchronize()
            ms5 = c0.elapsed_time(c1) / args.steps
            extra["cfg4_deepv3_w38_train"] = dict(
                value=1000.0 / ms5, unit="crops/s", ms_per_step=ms5, tflops=34.95 / (ms5 * 1e-3), loss=float(l5),
                what="deepv3.DeepV3PlusW38 train step (WRN-38 trunk at output stride 8, dilations 2/4, ASPP 12/24/36, "
                     "decoder; Dropout2d of mod6/mod7 on), one 1024x2048 crop, CE, bf16 storage / fp32 accumulate, "
                     "34.95 TFLOP per crop (SURVEY 8d)")
            del net5, opt5
        except Exception as e:  # noqa
            extra["cfg4_deepv3_w38_train"] = dict(error=repr(e))
        line["other_configs"] = extra
        torch.cuda.empty_cache()
    if (args.torch_gpu_baseline or world == 1) and not args.no_torch_gpu_baseline:
        net = opt = None
        torch.cuda.empty_cache()
        tg = {}
        for name, ac in (("autocast_bf16", True), ("fp32_tf32_off", False)):
            try:
                ms_t = torch_gpu_step_time(args.arch, H, W, ac, args.criterion, steps=4 if ac else 2,
                                           warmup=2 if ac else 1)
                tg[name] = dict(ms_per_step=ms_t, value=B * 1000.0 / ms_t, unit="crops/s")
            except Exception as e:  # noqa
                tg[name] = dict(error=repr(e))
            torch.cuda.empty_cache()
        tg["what"] = ("the reference algorithm (oracle restatement = the reference's own call sequence) through stock "
                      "PyTorch eager: ATen/cuDNN, NCHW, cudnn.benchmark, torch.optim.SGD, %d crop, this GPU, "
                      "device-resident inputs; per-GPU figure" % B)
        line["torch_gpu_baseline"] = tg
        best = max((v["value"] for v in tg.values() if isinstance(v, dict) and "value" in v), default=None)
        if best:
            line["vs_torch_gpu"] = dict(value=(value / world) / best, e2e=(e2e_value / world) / best,
                                        note="per-GPU crops/s of this path / best stock-PyTorch figure above")
    if not args.no_cpu_baseline:
        try:
            sh, sw = 128, 256
            sec, timed = cpu_reference_step_time(args.arch, sh, sw, 1, warmup=1, budget_s=30.0, criterion=args.criterion)
            ratio = (sh * sw) / float(H * W)
            line["cpu_baseline"] = dict(value=ratio / sec, unit="crops/s", cores=torch.get_num_threads(), kind="port",
                                        sample="oracle (reference algorithm, fp32, host threads): 1 warm-up + %d timed "
                                               "train step at %dx%d, rescaled by the pixel ratio %.5f" %
                                               (timed, sh, sw, ratio))
        except Exception as e:  # noqa
            line["cpu_baseline"] = dict(value=None, error=repr(e))
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    try:
        run_b200(args)
    except Exception:
        # SyncBN post-mortem: which exchange every rank entered / completed last (pinned host record, p2p.py)
        import gc
        from b200seg.module import B200SegModule
        for obj in gc.get_objects():
            if isinstance(obj, B200SegModule) and getattr(obj, "_sync", None) is not None:
                print(obj._sync.describe_beacon(), file=sys.stderr, flush=True)
        raise


if __name__ == "__main__":
    main()
