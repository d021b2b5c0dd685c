#!/usr/bin/env python
"""bench.py -- headline benchmark of the fake-quantization hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--sweep] [--train] [--dump-outputs DIR]

A *step* is one pass of the fused uniform fake-quant forward+backward kernel
(qd_uniform_fwd_bwd, 'complicated' min/max backward) over one 64 Mi-float32
tensor with s=16 levels and bucket 256 -- the workload BASELINE.json's
north_star quotes its 70%-of-HBM-peak target on.  Algorithmic traffic is
16 bytes per element (read x, g; write q, gout; SURVEY.md section 8d).

Printed JSON line (rank 0):
  value      algorithmic GB/s, inputs resident in HBM, CUDA-event timed, all ranks aggregated
  e2e        same metric through the host-buffer C-ABI call (pinned host tensors in,
             host tensors out; H2D + kernel + D2H inside the timed region)
  roofline   achieved GB/s of the kernel vs the measured HBM copy peak
  cpu_baseline  the reference's op chain (oracle/torch_chain.py, a port: /root/reference
             is not on the GPU box) on the host cores, bounded sample
With N > 1 every rank runs an independent replica (the op does not shard:
DESIGN.md "Multi-GPU"), timing is the max over ranks.

--impl reference times the reference's CPU implementation of the path
(the op-chain port) on the host, same metric and unit.

--dump-outputs DIR writes what the last timed step returned to a caller, q and
the input gradient, as DIR/q.npy and DIR/grad_input.npy (float32).  Both are
the same fixed sample of DUMP_ROWS whole buckets (seeded, sorted bucket
indices), shape (DUMP_ROWS, BUCKET): 32 MB in all.  Inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_ELEMS = 1 << 26          # 64 Mi float32
LEVELS = 16
BUCKET = 256
BYTES_PER_ELEM = 16        # x, g read; q, gout written
MODE_NAME = "minmax"
DUMP_ROWS = 1 << 14        # buckets sampled by --dump-outputs: 4 Mi elements per array


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int, period=0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:                      # pragma: no cover - NVML missing
            self.err = str(e)

    def sample_once(self):
        """One synchronous sample (called while the timed region's work is queued on the GPU)."""
        if not self.ok:
            return
        nv = self.nv
        try:
            self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            try:
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            for bit, name in self._names().items():
                if mask & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _names(self):
        nv = self.nv
        return {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ----------------------------------------------------------------------------- CPU arm
def usable_cpus() -> int:
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:                                            # cgroup v2 quota, if any
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


_BEST_THREADS = None
TUNE_ELEMS = 1 << 22       # thread-count tuning sample: 4 Mi elements (16 MB per tensor, larger than any host L2)


def best_cpu_threads() -> int:
    """All the host threads the reference's torch ops can USE: torch's intra-op pool is tried at
    1, 2, 4, ... up to the usable CPU count on a 4 Mi-element sample (best of 3 per setting) and
    the fastest setting is kept -- on a container whose CPU quota is below the visible core
    count, more threads is slower."""
    global _BEST_THREADS
    if _BEST_THREADS is not None:
        return _BEST_THREADS
    import torch
    from oracle import torch_chain as T
    cap = usable_cpus()
    cands = sorted({c for c in (1, 2, 4, 8, 16, 32, 64, 128, cap) if c <= cap})
    x = torch.randn(TUNE_ELEMS) * 0.05
    g = torch.randn(TUNE_ELEMS)
    timing = {}
    for c in cands:
        torch.set_num_threads(c)
        best = float("inf")
        for _ in range(4):
            t0 = time.perf_counter()
            T.uniform_fwd(x, LEVELS, BUCKET)
            T.uniform_bwd_minmax(x, g, LEVELS, BUCKET)
            best = min(best, time.perf_counter() - t0)
        timing[c] = best
    _BEST_THREADS = min(timing, key=timing.get)
    torch.set_num_threads(_BEST_THREADS)
    return _BEST_THREADS


def cpu_port_throughput(n: int, repeats: int, warmup: int):
    """The reference's CPU path for one fwd+bwd over n elements (oracle/torch_chain.py, same torch
    ops, best thread count on this host).  Returns (GB/s at 16 B/elt from the MEAN pass time,
    mean seconds per pass, threads)."""
    import torch
    from oracle import torch_chain as T
    threads = best_cpu_threads()
    torch.set_num_threads(threads)
    g0 = torch.Generator().manual_seed(0)
    x = torch.randn(n, generator=g0) * 0.05
    g = torch.randn(n, generator=torch.Generator().manual_seed(1))
    total = 0.0
    for i in range(warmup + repeats):
        t0 = time.perf_counter()
        T.uniform_fwd(x, LEVELS, BUCKET)
        T.uniform_bwd_minmax(x, g, LEVELS, BUCKET)
        dt = time.perf_counter() - t0
        if i >= warmup:
            total += dt
    mean = total / repeats
    return n * BYTES_PER_ELEM / mean / 1e9, mean, threads


def run_reference_arm(args):
    """The reference's CPU implementation of the path on the FULL workload: every step is one
    forward + min/max backward op chain over all 64 Mi elements; `ms_per_step` is the measured
    mean over the K timed steps (nothing extrapolated)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.ref_elements or N_ELEMS
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    gbs, sec, threads = cpu_port_throughput(n, steps, warmup)
    sample = (f"full workload: all {n} elements per step, mean of {steps} timed steps after {warmup} warm-up; "
              f"thread count tuned on {TUNE_ELEMS} elements") if n == N_ELEMS else \
             f"REDUCED by --ref-elements: {n} of {N_ELEMS} elements per step (test hook, not a bench value)"
    cfg = workload_config(args.gpus)
    cfg["elements"] = n
    print(json.dumps({
        "impl": "reference", "metric": "fake_quant_fused_fwd_bwd_algorithmic_GBps", "value": round(gbs, 3), "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(sec * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": round(gbs, 3), "unit": "GB/s", "cores": threads, "kind": "port", "sample": sample,
                         "host_cpus_visible": os.cpu_count(), "host_cpus_usable": usable_cpus()},
        "e2e": {"value": round(gbs, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def workload_config(n_gpus):
    return {"workload": f"uniform fake-quant fused forward+backward ({MODE_NAME} backward), one {N_ELEMS}-float32 tensor per GPU, "
                        f"s={LEVELS}, bucket_size={BUCKET}, {BYTES_PER_ELEM} algorithmic bytes/element",
            "elements": N_ELEMS, "levels": LEVELS, "bucket_size": BUCKET, "backward": MODE_NAME,
            "parallelism": f"replicas x{n_gpus} (op does not shard)",
            "l2_policy": "inputs+outputs are 1 GiB per step, larger than the 126 MB L2; no flush needed"}


# ----------------------------------------------------------------------------- training legs
STUDENT_NAME = "ConvolForwardNet smallerModelSpec (22 tensors, 1,000,235 params), teacher teacherModelSpec"
WRN_NAME = "Wide_ResNet-16-22 student (60 tensors, 82,746,890 params), WRN-28-20 teacher"


def build_models(kind, dev):
    """Random-init student / teacher of BASELINE configs 2-4, built on `dev` (same seed on every rank)."""
    import torch
    from quantized_distillation_b200.cnn_models import conv_forward_model as cfm
    from quantized_distillation_b200.cnn_models.wide_resnet import Wide_ResNet
    torch.manual_seed(1234)
    with torch.device(dev):
        if kind in ("student", "diffquant"):
            spec = dict(cfm.smallerModelSpec)
            spec["spec_dropout_rates"] = []
            student = cfm.ConvolForwardNet(**spec, useBatchNorm=True, useAffineTransformInBatchNorm=True)
            teacher = cfm.ConvolForwardNet(**cfm.teacherModelSpec, useBatchNorm=True, useAffineTransformInBatchNorm=True).eval()
        else:
            student = Wide_ResNet(depth=16, widen_factor=22, dropout_rate=0.3, num_classes=10)
            teacher = Wide_ResNet(depth=28, widen_factor=20, dropout_rate=0.3, num_classes=10).eval()
    return student, teacher


def leg_settings(kind, world):
    if kind in ("student", "diffquant"):
        return dict(per_gpu_batch=25, bits=4, name=STUDENT_NAME,
                    kw=dict(initial_learning_rate=1e-3, weight_decayL2=2.2e-4))
    # reference: global batch 100, must divide by the GPU count (cifar10_wideResNet.py:49-51) -> 104 on 8 GPUs
    per = 100 // world if 100 % world == 0 else 13
    return dict(per_gpu_batch=per, bits=2, name=WRN_NAME,
                kw=dict(initial_learning_rate=0.1, weight_decayL2=5e-4, learning_rate_style="cifar100",
                        quantize_first_and_last_layer=False))


def run_train_leg(kind, world, rank, dev, steps, warmup, graph=False, flat=True, fused=False):
    """CIFAR10-shaped quantized distillation steps/s (BASELINE configs 2-4), synthetic data,
    random-init weights.  Every step copies its batch from pinned host memory and reads the
    loss back (print_every=1), so the number is end to end.  world > 1: FlatDataParallel (one
    NCCL all-reduce of the flat gradient per step, capturable) or stock DDP (flat=False)."""
    import torch
    from quantized_distillation_b200 import distributed as D
    from quantized_distillation_b200.cnn_models import conv_forward_model as cfm
    from quantized_distillation_b200.cnn_models import help_fun as hf

    st = leg_settings(kind, world)
    student, teacher = build_models(kind, dev)
    per_gpu_batch, bits = st["per_gpu_batch"], st["bits"]
    total = warmup + steps
    data = hf.synthetic_cifar_loader(total, per_gpu_batch, seed=100 + rank)
    ev = {}

    def hook(i, loss):
        if i == warmup:
            ev["t0"] = torch.cuda.Event(enable_timing=True)
            ev["t0"].record()
        if i == total:
            ev["t1"] = torch.cuda.Event(enable_timing=True)
            ev["t1"].record()

    info = {}
    if kind == "diffquant":
        info = cfm.optimize_quantization_points(student, data, data, initial_learning_rate=1e-5, epochs_to_train=1, print_every=1,
                                                numPointsPerTensor=4, bucket_size=256, use_distillation_loss=True,
                                                initialize_method="quantiles", verbose=False, evaluate=False, max_steps=total,
                                                step_hook=hook, cuda_graph_step=graph)[2]
        label = "differentiable quantization, 4 centroids per tensor, bucket 256 (BASELINE config 4)"
    else:
        model = D.wrap_data_parallel(student, dev, flat=flat)
        info = cfm.train_model_quantized(model, data, data, numBits=bits, bucket_size=256, use_distillation_loss=True,
                                         teacher_model=teacher, epochs_to_train=1, print_every=1, verbose=False, evaluate=False,
                                         max_steps=total, step_hook=hook, cuda_graph_step=graph, fused_optimizer_step=fused,
                                         **st["kw"])[1]
        label = f"{bits}-bit quantized distillation, bucket 256 (BASELINE config {2 if kind == 'student' else 3})"
    torch.cuda.synchronize(dev)
    ms = ev["t0"].elapsed_time(ev["t1"]) / steps
    ms = D.max_over_ranks(ms, dev)
    par = "single process" if world == 1 else ("FlatDataParallel: 1 NCCL all-reduce of the flat gradient per step" if flat
                                               else "stock DistributedDataParallel")
    out = {"config": f"{label}; {st['name']}; per-GPU batch {per_gpu_batch}, global batch {per_gpu_batch * world}, {par}, "
                     "synthetic CIFAR-shaped data, batch copied from pinned host memory and loss read back every step",
           "steps_per_s": round(1e3 / ms, 2), "ms_per_step": round(ms, 3), "images_per_s": round(per_gpu_batch * world * 1e3 / ms, 1),
           "steps": steps, "warmup": warmup, "n_gpus": world, "cuda_graph_step": bool(graph)}
    if fused:
        out["fused_optimizer_step"] = bool(info.get("fused_optimizer_step", False))
    if graph:
        out["captured"] = bool(info.get("cuda_graph_step", False))
    del student, teacher
    torch.cuda.empty_cache()
    return out


def reference_style_leg(kind, dev, steps, warmup, threads=None):
    """The SAME harness driven the way the reference drives it: per step, every selected
    parameter tensor goes through the reference's stock-torch op chain (oracle/torch_chain.py,
    bit-identical to the reference on the golden vectors) one tensor at a time, `p.data` is
    re-bound to the result and re-bound back after the backward pass
    (cnn_models/conv_forward_model.py:236-247, 286-302; :501-551 for the differentiable loop,
    pre-processed SearchSorted path incl. its per-step host numpy work).  dev = cuda: what the
    reference does on a GPU box (USE_CUDA=True).  dev = cpu: its CPU path, model included."""
    import torch
    from oracle import torch_chain as T
    from quantized_distillation_b200.cnn_models import conv_forward_model as cfm
    from quantized_distillation_b200.cnn_models import help_fun as hf
    import torch.optim as optim

    on_gpu = dev.type == "cuda"
    if not on_gpu:
        torch.set_num_threads(threads or best_cpu_threads())
    st = leg_settings(kind, 1)
    student, teacher = build_models(kind, dev)
    data = hf.synthetic_cifar_loader(warmup + steps, st["per_gpu_batch"], seed=100, pin=on_gpu)
    levels = 2 ** st["bits"]
    first_last = st["kw"].get("quantize_first_and_last_layer", True)

    if kind == "diffquant":
        teacher_net = student.eval()                                       # the unquantized network is the teacher (:497-498)
        import copy
        qmodel = copy.deepcopy(student)
        sel = cfm._selected_parameters(qmodel, True)
        pres = [T.PreprocessedCentroids(p.data, 256) for p in sel]          # one-time sort per tensor (:501-511)
        import numpy as np                                                 # percentile initialisation (help_functions.py:140-154)
        points = [torch.from_numpy(np.percentile(pre.sorted, np.linspace(0, 100, 4)).astype(np.float32)).to(dev)
                  .requires_grad_(True) for pre in pres]
        opt = optim.SGD(points, lr=1e-5, momentum=0.9, nesterov=True)
        qmodel.train()

        def step(batch):
            qmodel.zero_grad()
            opt.zero_grad()
            saved = []
            for p, pre, pts in zip(sel, pres, points):                     # :525-532
                q, idx = pre.forward(pts.data)
                p.data = q
                saved.append(idx)
            loss = hf.forward_and_backward(qmodel, batch, 1, 0, use_distillation_loss=True, teacher_model=teacher_net,
                                           return_tensor=True)
            for p, pre, pts, idx in zip(sel, pres, points, saved):          # :539-545
                pts.grad = T.nonuniform_bwd_points(p.grad.data, idx, pre.st, 4, 256)
            opt.step()
            for pts in points:                                              # :550-551
                pts.data = torch.sort(pts.data)[0]
            return loss
    else:
        model = student
        sel = cfm._selected_parameters(model, first_last)
        kw = st["kw"]
        opt = optim.SGD(model.parameters(), lr=kw["initial_learning_rate"], nesterov=True, momentum=0.9,
                        weight_decay=kw["weight_decayL2"])
        model.train()

        def step(batch):
            saved = [p.data for p in sel]                                   # state_dict() keeps the old storages alive (:286)
            for p in sel:                                                   # :236-247: one op chain per tensor
                p.data = T.uniform_fwd(p.data, levels, 256)[0]
            model.zero_grad()
            loss = hf.forward_and_backward(model, batch, 1, 0, use_distillation_loss=True, teacher_model=teacher,
                                           return_tensor=True)
            for p, w in zip(sel, saved):                                    # load_state_dict (:302)
                p.data = w
            opt.step()
            return loss

    def sync():
        if on_gpu:
            torch.cuda.synchronize(dev)

    t0 = None
    for i, batch in enumerate(data):
        if i == warmup:
            sync()
            t0 = time.perf_counter()
        float(step(batch).item())                                           # loss read back every step, like our leg
    sync()
    ms = (time.perf_counter() - t0) / steps * 1e3
    del student, teacher
    if on_gpu:
        torch.cuda.empty_cache()
    return {"steps_per_s": round(1e3 / ms, 3), "ms_per_step": round(ms, 3), "steps": steps, "warmup": warmup,
            "device": "cuda (stock torch op chain per tensor)" if on_gpu else f"cpu ({torch.get_num_threads()} threads, model included)"}


def train_legs(which, world, rank, dev, steps, with_cpu):
    """BASELINE configs 2/3/4: ours (eager and whole-step CUDA graph) and, at N=1, the
    reference-style harness timed in the same run."""
    import torch
    legs = {}
    for kind in which:
        wsteps = steps if kind != "wrn" else max(10, steps // 2)
        leg = {"eager": run_train_leg(kind, world, rank, dev, wsteps, 8, graph=False)}
        leg["cuda_graph_step"] = run_train_leg(kind, world, rank, dev, wsteps, 8, graph=True)
        cands = [leg["eager"], leg["cuda_graph_step"]]
        if kind != "diffquant":
            # restore + gradient fix-up + SGD + next step's quantization as one kernel (qd_plan_sgd_step), inside the graph
            leg["cuda_graph_fused_optimizer"] = run_train_leg(kind, world, rank, dev, wsteps, 8, graph=True, fused=True)
            cands.append(leg["cuda_graph_fused_optimizer"])
        best = max(cands, key=lambda r: r["steps_per_s"])
        leg["steps_per_s"], leg["images_per_s"], leg["ms_per_step"] = best["steps_per_s"], best["images_per_s"], best["ms_per_step"]
        # The model's convolutions are cuDNN's, in torch's default math mode: TF32 on the tensor cores
        # (torch.backends.cudnn.allow_tf32 = True) -- the mode the reference's own code gets under this torch, and the one
        # the reference-style baseline below runs in.  The quantization kernels are float32 throughout.  The same leg with
        # TF32 switched off (IEEE float32 convolutions, what the reference's 2018 stack computed) is reported next to it.
        leg["convolution_math"] = "torch default: TF32 (cudnn.allow_tf32=True); matmuls float32"
        tf32_was = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        try:
            strict = run_train_leg(kind, world, rank, dev, max(6, wsteps // 2), 5, graph=True, fused=kind != "diffquant")
        finally:
            torch.backends.cudnn.allow_tf32 = tf32_was
        leg["strict_fp32_convolutions"] = {k: strict[k] for k in ("steps_per_s", "ms_per_step", "images_per_s", "steps", "warmup",
                                                                  "cuda_graph_step", "captured")}
        if world == 1 and rank == 0:
            leg["reference_style_gpu"] = reference_style_leg(kind, dev, max(6, wsteps // 2), 3)
            leg["reference_style_steps_per_s"] = leg["reference_style_gpu"]["steps_per_s"]
            leg["speedup_vs_reference_style_gpu"] = round(leg["steps_per_s"] / leg["reference_style_gpu"]["steps_per_s"], 2)
            if with_cpu and kind != "wrn":
                leg["reference_style_cpu"] = reference_style_leg(kind, torch.device("cpu"), 3, 1)
            elif with_cpu:
                leg["reference_style_cpu"] = {"skipped": "WRN-16-22 + WRN-28-20 teacher at batch 100 on the host cores is minutes per step; "
                                                         "the per-step quantization alone is in cpu_reference_quantize_ms_per_step"}
                leg["cpu_reference_quantize_ms_per_step"] = round(cpu_model_quant_ms(WRN_SIZES(), 4, 256, repeats=1), 1)
        legs[kind] = leg
    return legs


def WRN_SIZES():
    from quantized_distillation_b200.cnn_models.wide_resnet import Wide_ResNet
    import torch
    with torch.device("meta"):
        m = Wide_ResNet(depth=16, widen_factor=22, dropout_rate=0.3, num_classes=10)
    return [p.numel() for p in m.parameters()][1:-1]


def cpu_model_quant_ms(sizes, levels, bucket, repeats=3):
    """The reference's per-step quantization loop on the host (conv_forward_model.py:236-247):
    one op chain per parameter tensor (oracle/torch_chain.py)."""
    import torch
    from oracle import torch_chain as T
    torch.set_num_threads(best_cpu_threads())
    params = [torch.randn(n) * 0.05 for n in sizes]
    best = float("inf")
    for _ in range(repeats + 1):
        t0 = time.perf_counter()
        T.quantize_model_step(params, levels, bucket)
        best = min(best, time.perf_counter() - t0)
    return best * 1e3


def dump_outputs(out_dir, q, gout):
    """The same seeded sample of DUMP_ROWS buckets of q and of the input gradient, as float32 .npy files."""
    import numpy as np
    import torch
    rows = np.sort(np.random.default_rng(0).choice(N_ELEMS // BUCKET, DUMP_ROWS, replace=False))
    sel = torch.from_numpy(rows).to(q.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("q", q), ("grad_input", gout)):
        np.save(os.path.join(out_dir, name + ".npy"), t.view(-1, BUCKET).index_select(0, sel).cpu().numpy())


# ----------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sweep", action="store_true", help="also print the per-size / per-op table (profiles/)")
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--train", default="auto", choices=["auto", "none", "student", "wrn", "diffquant", "all"],
                    help="CIFAR10-shaped quantized-distillation steps/s (BASELINE configs 2/3/4); auto = student at every N, "
                         "WRN-16-22 at N=1 and N=8, differentiable quantization at N=1")
    ap.add_argument("--train-steps", type=int, default=40)
    ap.add_argument("--ref-elements", type=int, default=0,
                    help="TEST HOOK for --impl reference: run the CPU arm on fewer elements (the line says so; not a bench value)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of the last timed step's outputs to DIR/*.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    # stdout carries ONE JSON line.  Libraries write there too (NCCL prints its version line to stdout when the box
    # sets NCCL_DEBUG=VERSION, and ignores NCCL_DEBUG_FILE at that level), so file descriptor 1 points at stderr for
    # the duration of the run and the line is written to the saved descriptor at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from quantized_distillation_b200 import _native as N

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the quantization ops have no CPU implementation")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # the captured training step holds an NCCL all-reduce: no watchdog thread may touch the CUDA API of
        # this process while a capture is open (the PyTorch CUDA-graphs note asks for the same setting)
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
        dist.init_process_group("nccl", device_id=dev)
    lib = N.lib()
    mode = N.BWD_MINMAX
    steps, warmup = args.steps, max(3, args.warmup)

    gen = torch.Generator(device=dev).manual_seed(rank)
    x = torch.randn(N_ELEMS, generator=gen, device=dev) * 0.05
    g = torch.randn(N_ELEMS, generator=gen, device=dev)
    q, gout = torch.empty_like(x), torch.empty_like(g)
    ws = N.workspace(N_ELEMS, BUCKET, dev)
    stream = torch.cuda.current_stream(dev)
    sp = N.stream_ptr(dev)

    def step():
        N.check(lib.qd_uniform_fwd_bwd(N.ptr(x), N.ptr(g), N.ptr(q), N.ptr(gout), N_ELEMS, BUCKET, LEVELS, mode, N.ptr(ws),
                                       ws.numel(), sp))

    for _ in range(warmup):
        step()
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(steps):
        step()
    ev1.record(stream)
    while not ev1.query():              # the K steps are queued: sample the clocks while they execute
        sampler.sample_once()
        time.sleep(0.002)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / steps
    per_gpu_gbs = N_ELEMS * BYTES_PER_ELEM / (ms_per_step * 1e-3) / 1e9
    value = per_gpu_gbs * world
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, q, gout)

    # ---- e2e: host buffers through the C ABI (H2D + kernel + D2H inside the timed region)
    # the pinned buffers are allocated and first touched on the CPUs of this GPU's NUMA node, so that N ranks
    # on one box do not all stage through the same socket's memory
    from quantized_distillation_b200 import distributed as D
    with D.numa_local(local_rank) as numa:
        hx = torch.empty(N_ELEMS, dtype=torch.float32).pin_memory()
        hx.copy_(x)
        hg = torch.empty(N_ELEMS, dtype=torch.float32).pin_memory()
        hg.copy_(g)
        hq = torch.empty(N_ELEMS, dtype=torch.float32).pin_memory()
        hgo = torch.empty(N_ELEMS, dtype=torch.float32).pin_memory()
        hq.zero_()
        hgo.zero_()
        torch.cuda.synchronize(dev)

    def e2e_step():
        N.check(lib.qd_uniform_fwd_bwd_host(N.ptr(hx), N.ptr(hg), N.ptr(hq), N.ptr(hgo), N_ELEMS, BUCKET, LEVELS, mode, local_rank))

    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_step()
    torch.cuda.synchronize(dev)
    e2e_s = (time.perf_counter() - t0) / args.e2e_steps
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    assert torch.equal(hq, q.cpu()), "e2e result differs from the resident-HBM result"
    e2e_gbs = N_ELEMS * BYTES_PER_ELEM / e2e_s / 1e9 * world

    # ---- the ceiling of the e2e leg on this box: the same four pinned buffers moved by plain cudaMemcpyAsync, both
    # directions at once, no kernel, every rank at the same time (so that at N > 1 it shows what the host side --
    # DRAM, PCIe switches -- gives N concurrent ranks); counted in the e2e leg's unit (16 algorithmic bytes per element)
    dx, dg = torch.empty_like(x), torch.empty_like(x)
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def copy_step():
        with torch.cuda.stream(s_in):
            dx.copy_(hx, non_blocking=True)
            dg.copy_(hg, non_blocking=True)
        with torch.cuda.stream(s_out):
            hq.copy_(q, non_blocking=True)
            hgo.copy_(gout, non_blocking=True)

    copy_step()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        copy_step()
    torch.cuda.synchronize(dev)
    copy_s = (time.perf_counter() - t0) / 4
    if world > 1:
        t = torch.tensor([copy_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        copy_s = float(t.item())
    copy_gbs = N_ELEMS * BYTES_PER_ELEM / copy_s / 1e9 * world
    del dx, dg

    peak, peak_src = load_peaks()
    out = {
        "metric": "fake_quant_fused_fwd_bwd_algorithmic_GBps", "value": round(value, 1), "unit": "GB/s",
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": round(ms_per_step, 5),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(world),
        "clocks": clocks,
        "e2e": {"value": round(e2e_gbs, 2), "unit": "GB/s", "h2d_bytes_per_step": 2 * N_ELEMS * 4 * world,
                "d2h_bytes_per_step": 2 * N_ELEMS * 4 * world, "ms_per_step": round(e2e_s * 1e3, 3), "steps": args.e2e_steps,
                "api": "qd_uniform_fwd_bwd_host (pinned host tensors in and out)", "pinned_buffers_numa": numa.applied,
                "copy_ceiling": {"value": round(copy_gbs, 2), "unit": "GB/s", "frac": round(e2e_gbs / copy_gbs, 4),
                                 "what": "the same pinned buffers moved by plain cudaMemcpyAsync, both directions at once, "
                                         "no kernel, all ranks concurrently, in the e2e leg's unit"}},
        "gpu_launches": steps,
        "roofline": {"bound": "hbm", "achieved": round(per_gpu_gbs, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(per_gpu_gbs / peak, 4), "frac_of_nominal_8000": round(per_gpu_gbs / 8000.0, 4),
                     "peak_source": peak_src, "traffic": None, "traffic_source": None,
                     "kernel": "qd::warp_rows_kernel<OP_UNIFORM, BWD_MINMAX, R=2, VEC>",
                     "algorithmic_bytes_per_launch": N_ELEMS * BYTES_PER_ELEM},
    }
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        try:
            with open(traffic_file) as f:
                tj = json.load(f)
            out["roofline"]["traffic"] = tj.get("uniform_fwd_bwd_minmax_64Mi_dram_bytes")
            out["roofline"]["traffic_source"] = ("profile constant, NOT measured in this run: dram__bytes_read.sum + "
                                                 "dram__bytes_write.sum of one `ncu --set full` launch, " + str(tj.get("source", "profiles/")))
        except Exception:
            pass

    if rank == 0 and world == 1 and not args.no_cpu:
        gbs, sec, threads = cpu_port_throughput(N_ELEMS, 3, 1)
        out["cpu_baseline"] = {"value": round(gbs, 3), "unit": "GB/s", "cores": threads, "kind": "port",
                               "sample": f"full workload ({N_ELEMS} elements), mean of 3 passes after 1 warm-up "
                                         f"({sec * 1e3:.0f} ms per pass), oracle/torch_chain.py (the reference's torch op "
                                         "chain; /root/reference is absent on the GPU box); thread count tuned over powers "
                                         f"of two up to the usable CPUs on {TUNE_ELEMS} elements",
                               "host_cpus_visible": os.cpu_count(), "host_cpus_usable": usable_cpus()}
    which = {"none": [], "student": ["student"], "wrn": ["wrn"], "diffquant": ["diffquant"], "all": ["student", "wrn", "diffquant"],
             "auto": ["student"] + (["wrn"] if world in (1, 8) else []) + (["diffquant"] if world == 1 else [])}[args.train]
    if world > 1:
        which = [k for k in which if k != "diffquant"]           # config 4 is a single-GPU configuration
    if which:
        out["train"] = train_legs(which, world, rank, dev, args.train_steps, with_cpu=not args.no_cpu)
    if args.sweep and rank == 0:
        from tools import sweep
        out["sweep_file"] = sweep.run(dev)
    if world > 1:
        dist.destroy_process_group()
    sys.stdout.flush()
    if rank == 0:
        os.write(real_stdout, (json.dumps(out) + "\n").encode())
    os.close(real_stdout)


if __name__ == "__main__":
    main()
