#!/usr/bin/env python
"""bench.py -- ResNet-50-DWT training-step throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload resnet|microbench] [--per-domain B] [--site-mode fused|modules]
                    [--dump-outputs DIR]

One "step" = one full training step of the ResNet-50-DWT harness model (harness/resnet50_dwt.py,
the reference topology with this repo's CUDA layers dropped in) on one synthetic Office-Home-shaped
batch: B source + B target + B target-aug images of 3x224x224 (B = 64 per domain -> 192 images per
GPU, SURVEY.md H4), forward, NLL(source) + 0.1 * MEC(target, target-aug), backward, SGD(momentum)
update.  N > 1: one process per GPU (torchrun), plain data parallel, gradients averaged by ONE NCCL
all-reduce of a flat 94.6 MB buffer per step (rank-local whitening statistics, nothing else exchanged).

Prints ONE JSON line on rank 0 (see the task contract): `value` = images/s with inputs resident in
HBM; `e2e` = images/s through the same public call with the step's images copied from pinned host
memory and the loss read back inside the timed region; `roofline` = the dominant hand-written
kernel family against the measured HBM peak; `cpu_baseline` = the CPU port of the reference
layers (oracle/torch_port.py, same harness model) timed on this box's host cores.

At N = 1 the line also carries
  `microbench`        BASELINE.json configs[1] (WTransform2d N=256 C=256 56x56 group_size=64, fwd+bwd: the TMA +
                      tcgen05 kernels) with its own roofline, per-kernel table, CPU baseline and reference-on-GPU time;
  `reference_on_gpu`  the reference's operator sequence (oracle/torch_port.py: stock ATen / cuBLAS / cuSOLVER / cuDNN
                      ops, eager, torch's default math modes) on the SAME B200 for configs[2] -- what a user of the
                      reference gets on this GPU today -- and the speed-up over it.

--impl reference: the reference's own CPU path (no GPU): the same step with the reference's
operator sequence on stock ATen CPU ops (oracle/torch_port.py), all host threads, a bounded sample.
--workload microbench: only BASELINE.json configs[1] (WTransform2d N=256 C=256 56x56 gs=64 fwd+bwd).
--dump-outputs DIR: after the K timed steps, DIR/{loss,logits,param_grads,params,buffers}.npy hold what the last
of them computed (dump_outputs()).  That step starts from the seeded checkpoint again (restored outside the timed
window), on the seeded batch: every run, whatever K and W, dumps one training step from the same inputs.
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
PLUGIN_DIR = os.path.join(ROOT, "dwt-domain-adaptation_b200")
for _p in (PLUGIN_DIR, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch                                     # noqa: E402
import torch.nn.functional as F                  # noqa: E402

LAMBDA_MEC = 0.1                                 # resnet50_dwt_mec_officehome.py:508
NUM_CLASSES = 65


def host_cores() -> int:
    """Usable host cores: min(affinity mask, cgroup CPU quota).  The GPU boxes expose 128 logical
    CPUs but cap the container at 16 by cgroup quota; oversubscribing the quota is ~10x slower."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "MEASURED_PEAKS.json"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        if os.environ.get("DWT_NO_CLOCK_SAMPLER"):          # diagnosis only: is the sampler perturbing the run?
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            # nvidia-smi's start-up (NVML init, driver queries) briefly stalls launches on the GPU it opens: let
            # it deliver its first sample before the timed region starts
            t_end = time.time() + 5.0
            while not self.rows and time.time() < t_end:
                time.sleep(0.02)
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------- model
DEFAULT_STEM = "s2d"     # harness option, same arithmetic (harness/resnet50_dwt.py _stem_s2d); --stem direct for the plain call


def build_model(layers, device, site_mode, seed=1, channels_last=False, stem_pad=0, stem_nchw=False, stem_s2d=False):
    from harness.resnet50_dwt import build_resnet50_dwt
    from harness.synth import synth_state_dict
    sd = {k: v.to(device) for k, v in synth_state_dict(seed=seed).items()}
    model = build_resnet50_dwt(sd, layers, site_mode=site_mode, channels_last=channels_last, stem_pad=stem_pad,
                               stem_nchw=stem_nchw, stem_s2d=stem_s2d).to(device)
    return model.train()


def make_optimizer(model):
    """SGD with the reference's two parameter groups (resnet50_dwt_mec_officehome.py:578-590)."""
    head = [p for n, p in model.named_parameters() if n.startswith("fc_out")]
    body = [p for n, p in model.named_parameters() if not n.startswith("fc_out")]
    return torch.optim.SGD([{"params": body, "lr": 1e-3}, {"params": head, "lr": 1e-2}], momentum=0.9,
                           weight_decay=5e-4)


class FlatGradAllReduce:
    """Plain data parallelism (SURVEY.md §8e): every parameter's .grad is a view into ONE flat fp32 buffer
    (94.6 MB for ResNet-50-DWT), averaged over the ranks by NCCL over NVLink (gloo in the CPU test).  Whitening / BN
    statistics are never exchanged: every rank normalises its own minibatch.

    gather="copy" (the default of bench.py, measured on 2 B200s: 31.48 vs 31.75 ms per step): autograd produces its own
    gradient tensors, ONE multi-tensor copy moves them into the flat buffer after backward, ONE all-reduce averages it, and
    .grad is re-pointed at the views for the optimizer -- instead of 161 small in-place accumulation kernels and a 94.6 MB
    memset per step.  gather="accumulate": .grad are the views themselves; then the buffer can also be cut into
    `segments` pieces that are all-reduced while backward is still running:

    The buffer is cut into `segments` contiguous pieces along the layer order and each piece is all-reduced as soon
    as backward has produced its last gradient (a post-accumulate hook per parameter counts them down): backward
    runs layer4 -> stem, so the big late-layer pieces (layer4 + fc = 60 MB, layer3 = 28 MB) travel while the earlier
    layers are still back-propagating and only the small stem / layer1 / layer2 piece (6 MB) is exposed at the end.
    The collectives are issued asynchronously on NCCL's own stream (async_op) and joined in reduce(); no Python runs
    at replay time -- the whole step, collectives and cross-stream edges included, is captured into the CUDA graph.
    Measured on 2 B200s the overlap buys nothing there (32.79 ms with 3 segments vs 32.71 ms with one collective: a
    60 MB all-reduce between two GPUs takes ~0.2 ms and its kernel competes with backward for SMs and HBM); it stays
    available (--grad-gather accumulate --grad-segments 3) for larger rank counts."""

    def __init__(self, model, world, segments=3, gather="accumulate"):
        import torch.distributed as dist
        self.world, self.dist, self.gather = world, dist, gather
        named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
        params = [p for _, p in named]
        self.params = params
        total = sum(p.numel() for p in params)
        self.flat = torch.zeros(total, dtype=torch.float32, device=params[0].device)
        off, offsets, self.views = 0, [], []
        for p in params:
            self.views.append(self.flat[off:off + p.numel()].as_strided(p.shape, p.stride()))   # same memory format as p
            offsets.append(off)
            off += p.numel()
        # gather = "accumulate": .grad IS the view, autograd adds into it (one small in-place add per parameter and a
        # memset per step); "copy": autograd produces its own gradient tensors, ONE multi-tensor copy moves them into the
        # flat buffer and .grad is re-pointed at the views for the optimizer; with segments > 1 the copy and the
        # collective of a segment are issued from the hook of its last gradient, overlapping the rest of backward
        if gather != "copy":
            for p, v in zip(params, self.views):
                p.grad = v
        # segment boundaries in layer order: [stem, layer1, layer2 | layer3 | layer4, fc_out] (fewer when asked)
        cuts = [0]
        if segments >= 3:
            cuts += [i for i, (n, _) in enumerate(named) if n.startswith("layer3.")][:1]
        if segments >= 2:
            cuts += [i for i, (n, _) in enumerate(named) if n.startswith("layer4.")][:1]
        cuts = sorted(set(cuts)) + [len(params)]
        self.ranges, self.seg_of = [], {}
        for k in range(len(cuts) - 1):
            a, b = cuts[k], cuts[k + 1]
            self.ranges.append((offsets[a], off if b == len(params) else offsets[b], b - a))
            for p in params[a:b]:
                self.seg_of[id(p)] = k
        self.seg_items = [(cuts[k], cuts[k + 1]) for k in range(len(cuts) - 1)]      # parameter index range of a segment
        self.pending = [r[2] for r in self.ranges]
        self.works = []
        self.launched = [False] * len(self.ranges)
        if world > 1:
            for p in params:                         # identical by construction (seeded); make it explicit
                dist.broadcast(p.data, 0)
            if len(self.ranges) > 1:
                for p in params:
                    p.register_post_accumulate_grad_hook(self._on_grad)

    def zero(self):
        self.pending = [r[2] for r in self.ranges]
        self.launched = [False] * len(self.ranges)
        self.works = []
        if self.gather == "copy":
            for p in self.params:
                p.grad = None
            return
        self.flat.zero_()

    def _on_grad(self, p):
        k = self.seg_of[id(p)]
        self.pending[k] -= 1
        if self.pending[k] == 0:
            self._launch(k)

    def _launch(self, k):
        a, b, _ = self.ranges[k]
        self.launched[k] = True
        if self.gather == "copy":                    # this segment's gradients -> its piece of the flat buffer
            i0, i1 = self.seg_items[k]
            torch._foreach_copy_(self.views[i0:i1], [p.grad for p in self.params[i0:i1]])
        seg = self.flat[a:b]
        if self.flat.is_cuda:
            self.works.append(self.dist.all_reduce(seg, op=self.dist.ReduceOp.AVG, async_op=True))
        else:
            self.works.append(self.dist.all_reduce(seg, op=self.dist.ReduceOp.SUM, async_op=True))

    def reduce(self):
        if self.gather == "copy" and (len(self.ranges) == 1 or self.world <= 1):
            torch._foreach_copy_(self.views, [p.grad for p in self.params])
            for p, v in zip(self.params, self.views):
                p.grad = v
        if self.world <= 1:
            return
        if len(self.ranges) == 1:                    # one collective after backward (round-1 behaviour)
            if self.flat.is_cuda:
                self.dist.all_reduce(self.flat, op=self.dist.ReduceOp.AVG)
            else:
                self.dist.all_reduce(self.flat, op=self.dist.ReduceOp.SUM)
                self.flat.div_(self.world)
            return
        for k in range(len(self.ranges) - 1, -1, -1):   # whatever backward did not complete (unused parameters), in a
            if not self.launched[k]:                     # fixed order on every rank
                self._launch(k)
        for w in self.works:
            w.wait()                                 # CUDA: the compute stream waits on NCCL's stream, the host does not
        if not self.flat.is_cuda:
            self.flat.div_(self.world)
        if self.gather == "copy":
            for p, v in zip(self.params, self.views):
                p.grad = v


def train_step(model, mec, opt, images, labels, sync=None, head=None):
    """-> (loss, logits).  head: dwt_b200.HeadLoss -- the same NLL + lambda*MEC as one fused launch (GPU arm)."""
    if sync is None:
        opt.zero_grad(set_to_none=True)
    else:
        sync.zero()
    logits = model(images)
    if head is not None:
        loss = head(logits, labels)
    else:
        src, tgt, aug = torch.split(logits, logits.shape[0] // 3, dim=0)
        loss = F.nll_loss(F.log_softmax(src, dim=1), labels) + LAMBDA_MEC * mec(tgt, aug)
    loss.backward()
    if sync is not None:
        sync.reduce()
    opt.step()
    return loss, logits


DUMP_SAMPLE = 1 << 21                            # elements kept of each flattened parameter-sized output


def dump_outputs(out_dir, model, loss, logits):
    """Write what one training step hands back to its caller as float32 .npy files: the loss and the logits whole;
    the parameter gradients, the updated parameters and the running statistics flattened in named_parameters /
    named_buffers order (logical NCHW order whatever the memory format), the first two as a fixed seeded sample of
    DUMP_SAMPLE of their 23.6 M elements -- the same elements in every run, so two builds compare output for output.
    Two runs of one build with the same arguments write bit-identical files (NVIDIA B200, 1000 W power limit)."""
    import numpy as np
    params = [p for _, p in model.named_parameters()]
    flat = {"param_grads": torch.cat([p.grad.reshape(-1) for p in params]),
            "params": torch.cat([p.detach().reshape(-1) for p in params]),
            "buffers": torch.cat([b.reshape(-1).float() for _, b in model.named_buffers()])}
    arrays = {"loss": loss.detach(), "logits": logits.detach()}
    for name, v in flat.items():
        if v.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(v.numel(), DUMP_SAMPLE, replace=False))
            v = v[torch.from_numpy(idx).to(v.device)]
        arrays[name] = v
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.float().cpu().numpy())


# ----------------------------------------------------------------------------------------- arms
def run_reference(args):
    """The reference's CPU path: harness model + CPU port of the reference layers, all host threads.
    Under torchrun only rank 0 works (one host, one set of cores): its images/s IS the whole-job figure of the
    CPU arm whatever --gpus says -- the host does not get faster when the GPU arm adds ranks."""
    import oracle.torch_port as port
    from harness.synth import synth_batch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    torch.set_num_threads(cores)
    dev = torch.device("cpu")
    if args.workload == "microbench":
        return run_reference_micro(args, port, cores)
    per_domain = args.cpu_per_domain
    model = build_model(port, dev, "modules")
    opt = make_optimizer(model)
    mec = port.MinEntropyConsensusLoss(NUM_CLASSES, dev)
    images, labels = synth_batch(seed=2, per_domain=per_domain)
    for _ in range(args.warmup):
        train_step(model, mec, opt, images, labels)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        train_step(model, mec, opt, images, labels)
    dt = (time.perf_counter() - t0) / args.steps
    val = 3 * per_domain / dt
    sample = (f"{args.steps} steps of {3 * per_domain} images (3x{per_domain}; the GPU arm steps 3x{args.per_domain} per rank), "
              "same model / loss / optimizer step")
    print(json.dumps({
        "impl": "reference", "metric": "ResNet-50-DWT images/sec fwd+bwd", "value": val, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, per_domain=args.per_domain),
        "implementation": {"site_mode": "modules (the reference's split -> 3 modules -> cat -> affine -> relu composition)",
                           "memory_format": "nchw", "launch": "eager, CPU",
                           "sample": f"each step is 3x{per_domain} images of the 3x{args.per_domain}-image workload step"},
        "whole_job": "one host: rank 0 alone runs; images/s of this host, independent of --gpus",
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_reference_micro(args, port, cores):
    """configs[1] on the host cores: the reference layer's operator sequence, N scaled down (the full N=256 tensor
    needs ~8 GB of autograd-saved copies and ~2 s per iteration; BASELINE.md §4 allows scaling N only)."""
    N, C, H, gs = args.micro_cpu_n, 256, 56, args.micro_gs
    torch.manual_seed(0)
    mix = torch.randn(C, C) / C ** 0.5 + torch.eye(C)
    x = (torch.einsum("dc,nchw->ndhw", mix, torch.randn(N, C, H, H)) + 2.0).contiguous().requires_grad_(True)
    dy = torch.randn(N, C, H, H)
    m = port.WTransform2d(C, gs).train()

    def step():
        torch.autograd.grad(m(x), x, dy)

    for _ in range(max(1, min(args.warmup, 2))):
        step()
    k = max(1, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(k):
        step()
    dt = (time.perf_counter() - t0) / k
    # the layer is linear in N: report the time scaled to the full-size tensor next to the measured one
    print(json.dumps({
        "impl": "reference", "metric": "WTransform2d fwd+bwd microbench", "value": 1.0 / (dt * args.micro_n / N),
        "unit": "iterations/s", "n_gpus": args.gpus, "steps": k, "warmup": args.warmup, "ms_per_step": dt * 1e3 * args.micro_n / N,
        "measured_ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"WTransform2d N={args.micro_n} C={C} H=W={H} group_size={gs} fwd+bwd",
                   "measured_at": f"N={N} (1/{args.micro_n // N} of the batch axis), time scaled by {args.micro_n // N}"},
        "cpu_baseline": {"value": 1.0 / (dt * args.micro_n / N), "unit": "iterations/s", "cores": torch.get_num_threads(),
                         "kind": "port", "sample": f"{k} iterations at N={N}, scaled x{args.micro_n // N} to N={args.micro_n}"},
        "e2e": {"value": 1.0 / (dt * args.micro_n / N), "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(args, per_domain):
    """The WORKLOAD both arms are quoted on (BASELINE.json configs[2] / [3] at --gpus N): identical in the GPU arm's line
    and in the reference arm's line.  How each arm runs it (layout, fused sites, CUDA graph, collective; the CPU arm's
    bounded sample) is in the line's `implementation` / `cpu_baseline.sample`, not here."""
    return {"workload": "ResNet-50-DWT synthetic Office-Home 224x224, train step = fwd + NLL + 0.1*MEC + bwd + SGD",
            "per_domain_batch": per_domain, "images_per_gpu": 3 * per_domain, "global_images": 3 * per_domain * args.gpus,
            "group_size": 4, "parallelism": f"dp{args.gpus}",
            "l2": "no explicit flush: per-step working set (activations) is tens of GB >> 126 MB L2"}


def implementation_note(args):
    seg = getattr(args, "grad_segments", 1)
    return {"site_mode": args.site_mode, "memory_format": args.memory_format,
            "block_input_gradients": ("summed inside the producing site's backward kernels (dwt_b200.fork_for_sum)"
                                      if getattr(args, "grad_fork", True) else "summed by autograd (aten::add)"),
            "stem": ("7x7/2 stem convolution evaluated as the 4x4/1 convolution of the 2x2 space-to-depth image (same arithmetic, "
                     "cuDNN tensor-core kernel)" if getattr(args, "stem", DEFAULT_STEM) == "s2d" else "7x7/2 convolution on the 3-channel image"),
            "launch": "CUDA-graph replay of the whole step" if args.cuda_graph else "eager",
            "grad_gather": getattr(args, "grad_gather", "accumulate"),
            "grad_sync": ("flat fp32 gradient buffer, one NCCL all-reduce (AVG) per step after backward" if seg == 1 else
                          f"flat fp32 gradient buffer, NCCL all-reduce (AVG) in {seg} segments issued as backward completes "
                          "them (layer4+fc, layer3, rest), overlapped with the remaining backward")}


def cpu_baseline(args, workload="resnet"):
    """Bounded CPU sample on rank 0: a few steps of the CPU port (configs[2] at a small per-domain batch, configs[1] at
    a fraction of N), in a subprocess that cannot see the GPU."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2" if workload == "resnet" else "3",
           "--warmup", "1", "--workload", workload, "--cpu-per-domain", str(args.cpu_per_domain),
           "--per-domain", str(args.per_domain), "--micro-n", str(args.micro_n), "--micro-cpu-n", str(args.micro_cpu_n),
           "--micro-gs", str(args.micro_gs)]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", RANK="0", WORLD_SIZE="1")
    for k in ("LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID"):
        env.pop(k, None)
    unit = "images/s" if workload == "resnet" else "iterations/s"
    try:
        out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600).stdout.strip().splitlines()
        return json.loads(out[-1])["cpu_baseline"]
    except Exception as e:                                   # the GPU number must not die with the CPU leg
        return {"value": None, "unit": unit, "cores": host_cores(), "kind": "port", "sample": f"failed: {e}"}


# ------------------------------------------------------------------------- reference on the same GPU
def reference_on_gpu_resnet(args, device):
    """configs[2] with the reference's operator sequence on this GPU (oracle/torch_port.py: x.mean / bmm /
    linalg.cholesky / inverse / grouped conv2d / F.batch_norm / split-cat-affine-relu composition, autograd backward),
    eager, NCHW, torch's default math modes (fp32 matmul, cuDNN TF32 convolutions -- the same convolutions as our
    arm).  /root/reference itself cannot travel to the GPU box; the port restates utils/whitening.py:37-61,
    utils/batch_norm.py:54-69, utils/consensus_loss.py:11-24 op for op (tests/test_oracle_vs_golden.py pins it)."""
    import oracle.torch_port as port
    from harness.synth import synth_batch
    B = args.per_domain
    model = build_model(port, device, "modules")
    opt = make_optimizer(model)
    mec = port.MinEntropyConsensusLoss(NUM_CLASSES, device)
    images, labels = synth_batch(seed=100, per_domain=B)
    images, labels = images.to(device), labels.to(device)

    def step():
        train_step(model, mec, opt, images, labels)

    for _ in range(3):
        step()
    k = max(3, min(args.steps, 10))
    ms = timed_loop(step, k, device, False)
    del model, opt
    return {"value": 3 * B * k / (ms / 1e3), "unit": "images/s", "ms_per_step": ms / k, "steps": k,
            "impl": "oracle/torch_port.py on cuda (stock ATen ops, eager, NCHW, matmul fp32, cuDNN TF32 convs)",
            "per_domain_batch": B}


def reference_on_gpu_micro(args, device):
    """configs[1] with the reference layer's operator sequence on this GPU (utils/whitening.py:41-59)."""
    import oracle.torch_port as port
    N, C, H, gs = args.micro_n, 256, 56, args.micro_gs
    torch.manual_seed(0)
    mix = torch.randn(C, C, device=device) / C ** 0.5 + torch.eye(C, device=device)
    x = (torch.einsum("dc,nchw->ndhw", mix, torch.randn(N, C, H, H, device=device)) + 2.0).contiguous().requires_grad_(True)
    dy = torch.randn(N, C, H, H, device=device)
    m = port.WTransform2d(C, gs).to(device).train()

    def step():
        torch.autograd.grad(m(x), x, dy)

    for _ in range(3):
        step()
    k = max(3, min(args.steps, 10))
    ms = timed_loop(step, k, device, False)
    return {"value": k / (ms / 1e3), "unit": "iterations/s", "ms_per_step": ms / k, "steps": k,
            "impl": "oracle/torch_port.py WTransform2d on cuda (mean, transposing copy, bmm, linalg.cholesky, inverse, "
                    "grouped conv2d; autograd backward), eager, fp32"}


def timed_loop(step_fn, steps, device, distributed, before_last=None):
    """Device time of `steps` calls of step_fn.  before_last (optional) runs between the last two steps, outside the
    timed window."""
    import torch.distributed as dist
    if distributed:
        dist.barrier()
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        if before_last is not None and i == steps - 1:
            p0.record()
            before_last()
            p1.record()
        step_fn()
    e1.record()
    torch.cuda.synchronize(device)
    ms = torch.tensor([e0.elapsed_time(e1) - (p0.elapsed_time(p1) if before_last is not None else 0.0)], device=device)
    if distributed:
        dist.barrier()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def finish(distributed, device):
    """Leave a multi-rank run without tearing NCCL down: destroying a process group whose collectives were
    captured into a live CUDA graph can dead-lock, and a benchmark that hangs after printing its line is worse
    than one that skips destructors."""
    sys.stdout.flush()
    sys.stderr.flush()
    if distributed:
        torch.cuda.synchronize(device)
        os._exit(0)


def run_ours(args):
    import torch.distributed as dist
    import dwt_b200
    from dwt_b200 import _native
    from harness.synth import synth_batch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    distributed = world > 1
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    if distributed:
        # NCCL prints its version banner on STDOUT at communicator creation; keep stdout for the JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
            torch.cuda.synchronize(device)
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    # cuDNN's heuristics choose the convolution algorithms from the shapes alone.  Autotuning (benchmark=True) chooses by
    # timing, so two runs could take different TF32 algorithms and compute different results: the training step turns
    # that rounding into several % of the gradients.  The fixed choice costs ~0.9 ms per step (29.7 vs 28.8 ms with
    # autotuning, NVIDIA B200 at 1000 W), most of it in the stem convolution.
    torch.backends.cudnn.benchmark = False
    _native.lib()                                           # fail loudly if the extension is missing

    if args.workload == "microbench":
        rec = run_microbench(args, device)
        if rank == 0:
            if args.cpu_baseline:
                rec["cpu_baseline"] = cpu_baseline(args, "microbench")
            rec["reference_on_gpu"] = reference_on_gpu_micro(args, device)
            rec["vs_reference_gpu"] = rec["value"] / rec["reference_on_gpu"]["value"]
            print(json.dumps(rec))
        return

    nhwc = args.memory_format == "nhwc"
    model = build_model(dwt_b200, device, args.site_mode, channels_last=nhwc, stem_pad=args.stem_pad, stem_nchw=args.stem_nchw,
                        stem_s2d=args.stem == "s2d")
    if not args.grad_fork:                                      # experiment: let autograd add the two gradients of a block input
        from harness.resnet50_dwt import Bottleneck
        for m in model.modules():
            if isinstance(m, Bottleneck):
                object.__setattr__(m, "_fork", None)
    net = model
    sync = FlatGradAllReduce(model, world, segments=args.grad_segments, gather=args.grad_gather) if distributed else None   # one GPU: plain .grad tensors
    opt = make_optimizer(model)
    # --dump-outputs: the last timed step starts again from the seeded checkpoint (weights and running statistics as
    # built, momentum buffers zero = a fresh SGD), so what it computes does not depend on the steps before it.  Training
    # on one fixed synthetic batch is chaotic -- a 1e-6 change of one weight reaches several % of the logits within
    # three steps -- so otherwise a cuDNN algorithm choice or a reordered sum decides what the dump holds.
    seeded = [t.detach().clone() for t in model.state_dict().values()] if args.dump_outputs else None

    def restore_seeded():
        torch._foreach_copy_(list(model.state_dict().values()), seeded)
        torch._foreach_zero_([s["momentum_buffer"] for s in opt.state.values()])

    mec = dwt_b200.MinEntropyConsensusLoss(NUM_CLASSES, device)
    head = dwt_b200.HeadLoss(NUM_CLASSES, LAMBDA_MEC)
    B = args.per_domain
    host_images, host_labels = synth_batch(seed=100 + rank, per_domain=B)
    if nhwc:
        host_images = host_images.contiguous(memory_format=torch.channels_last)
    host_images, host_labels = host_images.pin_memory(), host_labels.pin_memory()
    images, labels = host_images.to(device), host_labels.to(device)
    loss_host = torch.zeros((), dtype=torch.float32).pin_memory()
    last = {}                                               # (loss, logits) of the latest eager step, detached: a
                                                            # live autograd graph would break the CUDA-graph capture

    def step_resident():
        last["out"] = tuple(t.detach() for t in train_step(net, mec, opt, images, labels, sync, head))

    def step_e2e():
        im = host_images.to(device, non_blocking=True)
        lb = host_labels.to(device, non_blocking=True)
        loss, _ = train_step(net, mec, opt, im, lb, sync, head)
        loss_host.copy_(loss.detach(), non_blocking=True)
        torch.cuda.current_stream(device).synchronize()     # the user reads the loss every step

    for _ in range(args.warmup):
        step_resident()
    # Pass 1 (eager): every kernel launch of the library is bracketed by CUDA events -> per-kernel roofline.
    n0 = _native.launch_count()
    with ClockSampler(local) as clocks_eager:
        _native.profile_begin()
        ms_eager = timed_loop(step_resident, args.steps, device, distributed)
        prof_sites = _native.profile_end()
    prof = _native.by_family(prof_sites)
    launches = (_native.launch_count() - n0) // args.steps

    # Pass 2: the same step captured once into a CUDA graph and replayed (the step is ~1400 launches, the
    # host launch path is as long as the GPU work).  This is the reported `value`; identical kernels and work.
    graph, static_loss, static_logits = None, None, None
    if args.cuda_graph:
        try:
            side = torch.cuda.Stream(device)
            side.wait_stream(torch.cuda.current_stream(device))
            with torch.cuda.stream(side):
                for _ in range(3):
                    step_resident()
            torch.cuda.current_stream(device).wait_stream(side)
            torch.cuda.synchronize(device)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_loss, static_logits = train_step(net, mec, opt, images, labels, sync, head)
            torch.cuda.synchronize(device)
        except Exception as e:                      # capture is an optimisation, never a requirement
            graph = None
            sys.stderr.write(f"[bench] CUDA-graph capture unavailable ({type(e).__name__}: {e}); timing eagerly\n")
            torch.cuda.synchronize(device)

    if graph is not None:
        def step_timed():
            graph.replay()

        # e2e: the batch of step i+1 crosses PCIe (pinned host -> staging buffer, side stream) while the graph of
        # step i runs; each step still performs exactly one H2D of a full batch and one D2H of the loss.
        copy_stream = torch.cuda.Stream(device)
        stage_images, stage_labels = torch.empty_like(images), torch.empty_like(labels)
        with torch.cuda.stream(copy_stream):
            stage_images.copy_(host_images, non_blocking=True)
            stage_labels.copy_(host_labels, non_blocking=True)

        def step_e2e():
            cur = torch.cuda.current_stream(device)
            cur.wait_stream(copy_stream)                     # this step's batch has landed
            images.copy_(stage_images, non_blocking=True)    # device-to-device into the graph's static input
            labels.copy_(stage_labels, non_blocking=True)
            copy_stream.wait_stream(cur)                     # staging buffer is free again
            with torch.cuda.stream(copy_stream):
                stage_images.copy_(host_images, non_blocking=True)
                stage_labels.copy_(host_labels, non_blocking=True)
            graph.replay()
            loss_host.copy_(static_loss.detach(), non_blocking=True)
            cur.synchronize()                                # the user reads the loss every step
    else:
        step_timed = step_resident
    for _ in range(2):
        step_timed()
    with ClockSampler(local) as clocks:
        ms = timed_loop(step_timed, args.steps, device, distributed, before_last=restore_seeded if args.dump_outputs else None)
    if args.dump_outputs and rank == 0:                    # before the e2e passes below train the model further
        dump_outputs(args.dump_outputs, model, *((static_loss, static_logits) if graph is not None else last["out"]))
    for _ in range(2):
        step_e2e()
    ms_e2e = timed_loop(step_e2e, args.steps, device, distributed)

    # e2e from RESIZED UINT8 images (what the reference's loader workers hold before RandomCrop): B source + B target
    # images of 256x256x3 cross PCIe (4.6x fewer bytes than the three float views) and one dwt_augment_pair launch per
    # domain writes crop / flip / cv2-exact affine / normalise straight into the graph's static input (SURVEY §8f-4).
    e2e_u8 = None
    if graph is not None and not distributed:
        try:
            import numpy as np
            from dwt_b200 import PairedAugment, draw_params
            aug = PairedAugment(crop=224)
            rng = np.random.default_rng(1234)
            host_u8 = torch.randint(0, 256, (2 * B, 256, 256, 3), dtype=torch.uint8).pin_memory()
            host_par = [{k: v.pin_memory() for k, v in draw_params(B, 256, 224, rng).items()} for _ in range(2)]
            dev_u8 = torch.empty(host_u8.shape, dtype=torch.uint8, device=device)
            dev_par = [{k: torch.empty(v.shape, dtype=v.dtype, device=device) for k, v in hp.items()} for hp in host_par]
            fmt_cl = args.memory_format == "nhwc"

            def upload():
                dev_u8.copy_(host_u8, non_blocking=True)
                stage_labels.copy_(host_labels, non_blocking=True)
                for dp, hp in zip(dev_par, host_par):
                    for k in dp:
                        dp[k].copy_(hp[k], non_blocking=True)

            with torch.cuda.stream(copy_stream):
                upload()

            def step_u8():
                cur = torch.cuda.current_stream(device)
                cur.wait_stream(copy_stream)
                aug(dev_u8[:B], crop_plain=dev_par[0]["crop_plain"], out_plain=images[:B], want_aug=False,
                    channels_last=fmt_cl)                                                   # source view
                aug(dev_u8[B:], out_plain=images[B:2 * B], out_aug=images[2 * B:], channels_last=fmt_cl, **dev_par[1])
                labels.copy_(stage_labels, non_blocking=True)
                copy_stream.wait_stream(cur)
                with torch.cuda.stream(copy_stream):
                    upload()
                graph.replay()
                loss_host.copy_(static_loss.detach(), non_blocking=True)
                cur.synchronize()

            for _ in range(2):
                step_u8()
            ms_u8 = timed_loop(step_u8, args.steps, device, False)
            e2e_u8 = {"value": 3 * B * args.steps / (ms_u8 / 1e3), "unit": "images/s", "ms_per_step": ms_u8 / args.steps,
                      "h2d_bytes_per_step": host_u8.numel() + host_labels.numel() * 8 + sum(v.numel() * v.element_size() for hp in host_par for v in hp.values()),
                      "d2h_bytes_per_step": 4,
                      "input": "2B resized uint8 images 256x256x3; crop/flip/affine/normalise on the GPU (dwt_augment_pair)"}
        except Exception as e:                      # an extra measurement, never a requirement
            sys.stderr.write(f"[bench] uint8-input e2e skipped ({type(e).__name__}: {e})\n")

    per_gpu = 3 * B
    value = per_gpu * world * args.steps / (ms / 1e3)
    e2e = per_gpu * world * args.steps / (ms_e2e / 1e3)
    if rank != 0:
        finish(distributed, device)
        return
    peak, peak_src = measured_peaks()
    if args.sites_out:
        rows = [dict(zip(("kernel", "C", "HW", "GS", "D", "N"), k.split("|")), launches=v["launches"],
                     us_per_launch=1e3 * v["ms"] / v["launches"], gbs=v["bytes"] / max(v["ms"], 1e-9) / 1e6,
                     frac_of_peak=v["bytes"] / max(v["ms"], 1e-9) / 1e6 / peak, ms_per_step=v["ms"] / args.steps)
                for k, v in sorted(prof_sites.items(), key=lambda kv: -kv[1]["ms"])]
        os.makedirs(os.path.dirname(os.path.abspath(args.sites_out)), exist_ok=True)
        json.dump(rows, open(args.sites_out, "w"), indent=1)
    fams = {k: dict(v, gbs=(v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] > 0 else None),
                    us_per_launch=(1e3 * v["ms"] / v["launches"] if v["launches"] else None),
                    share_of_step=v["ms"] / ms_eager) for k, v in prof.items()}
    dom = max((k for k in fams if fams[k]["bytes"] > 0), key=lambda k: fams[k]["ms"], default=None)
    roof = None
    traffic_tab = {}
    for name in ("traffic_r02.json", "traffic_r01.json"):
        try:
            traffic_tab = json.load(open(os.path.join(ROOT, "profiles", name)))
            break
        except Exception:
            pass
    if dom is not None:
        f = fams[dom]
        ratio = traffic_tab.get("traffic_over_algorithmic", {}).get(dom)
        roof = {"bound": "hbm", "kernel": dom, "achieved": f["gbs"], "peak": peak, "unit": "GB/s",
                "frac": f["gbs"] / peak,
                # DRAM bytes per launch: this run's algorithmic bytes per launch x the traffic/algorithmic ratio of the
                # committed `ncu --set full` capture of the same kernel (never measured under the profiler here)
                "traffic": (ratio * f["bytes"] / f["launches"]) if ratio else None,
                "traffic_source": traffic_tab.get("source") if ratio else None, "peak_source": peak_src,
                "launches_timed": f["launches"], "avg_launch_us": f["us_per_launch"],
                "algorithmic_bytes_per_launch": f["bytes"] / f["launches"],
                "all_norm_kernels_share_of_step": sum(v["ms"] for v in fams.values()) / ms_eager,
                "timed_in": "eager pass of this run (launches bracketed by CUDA events; graph replay hides them)"}
        byte_fams = {k: v for k, v in fams.items() if v["bytes"] > 0 and k != "head_loss"}
        tot_b, tot_ms = sum(v["bytes"] for v in byte_fams.values()), sum(v["ms"] for v in fams.values() if v is not None)
        worst = min(byte_fams, key=lambda k: byte_fams[k]["gbs"])
        # every hand-written norm launch of the step, finalize launches included in the time: the path as a whole.
        # Algorithmic bytes over time can exceed the DRAM peak: the kernels sweep the tensor in the order that finds
        # the producer's last ~100 MB still in L2 (norm_cl.cu), and those bytes never reach HBM.
        roof["norm_path"] = {"achieved": tot_b / (tot_ms * 1e-3) / 1e9, "frac": tot_b / (tot_ms * 1e-3) / 1e9 / peak,
                             "algorithmic_gb_per_step": tot_b / args.steps / 1e9, "ms_per_step": tot_ms / args.steps,
                             "worst_family": worst, "worst_frac": byte_fams[worst]["gbs"] / peak}
    out = {
        "metric": "ResNet-50-DWT images/sec fwd+bwd", "value": value, "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, per_domain=B), "implementation": implementation_note(args),
        "e2e": {"value": e2e, "unit": "images/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": host_images.numel() * 4 + host_labels.numel() * 8, "d2h_bytes_per_step": 4},
        "gpu_launches": int(launches), "clocks": clocks.summary(), "roofline": roof, "kernels": fams,
        "e2e_uint8_input": e2e_u8,
        "cuda_graph": graph is not None, "eager_ms_per_step": ms_eager / args.steps,
        "conv_math": "cuDNN, TF32 allowed (torch default), algorithms chosen by cuDNN's heuristics (no autotuning) -- "
                     "convolutions are not part of the hot path",
    }
    if args.cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args)
    out["status_word"] = _native.status_all(device)            # 0: no kernel reported a failure during the run
    if not distributed and args.extras:
        # free the step's graph, model and activations before the two side measurements
        del graph, static_loss, static_logits, last, seeded, model, net, opt
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        try:
            ref = reference_on_gpu_resnet(args, device)
            ref["speedup_value"] = value / ref["value"]
            ref["speedup_e2e"] = e2e / ref["value"]
            out["reference_on_gpu"] = ref
        except Exception as e:
            out["reference_on_gpu"] = {"value": None, "error": f"{type(e).__name__}: {e}"}
        gc.collect()
        torch.cuda.empty_cache()
        try:
            mb = run_microbench(args, device)
            if args.cpu_baseline:
                mb["cpu_baseline"] = cpu_baseline(args, "microbench")
            mb["reference_on_gpu"] = reference_on_gpu_micro(args, device)
            mb["vs_reference_gpu"] = mb["value"] / mb["reference_on_gpu"]["value"]
            out["microbench"] = mb
        except Exception as e:
            out["microbench"] = {"value": None, "error": f"{type(e).__name__}: {e}"}
    print(json.dumps(out))
    finish(distributed, device)


def run_microbench(args, device):
    """BASELINE.json configs[1]: WTransform2d N=256 C=256 H=W=56 group_size=64, fwd+bwd -> record (dict)."""
    import dwt_b200
    from dwt_b200 import _native
    N, C, H, gs = args.micro_n, 256, 56, args.micro_gs
    torch.manual_seed(0)
    mix = torch.randn(C, C, device=device) / C ** 0.5 + torch.eye(C, device=device)
    # .contiguous(): einsum returns a permuted view, and a strided input would add a layout copy (and its backward) of
    # the 822 MB tensor to every step -- 0.5 ms that is not the layer's
    x = (torch.einsum("dc,nchw->ndhw", mix, torch.randn(N, C, H, H, device=device)) + 2.0).contiguous().requires_grad_(True)
    dy = torch.randn(N, C, H, H, device=device)
    m = dwt_b200.WTransform2d(C, gs).to(device).train()
    steps = max(args.steps, 20)                      # SURVEY §8d: >= 20 iterations after >= 5 warm-ups
    warm = max(args.warmup, 5)

    def step():
        y = m(x)
        torch.autograd.grad(y, x, dy)

    for _ in range(warm):
        step()
    graph = None
    if args.cuda_graph:                              # the launches as one graph: no host time between them
        side = torch.cuda.Stream(device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            step()
        torch.cuda.current_stream(device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            step()
        graph.replay()
    with ClockSampler(device.index) as clocks:
        _native.profile_begin()
        eager_ms = timed_loop(step, steps, device, False)
        prof = _native.by_family(_native.profile_end())
        ms = timed_loop(graph.replay, steps, device, False) if graph is not None else eager_ms
    peak, peak_src = measured_peaks()
    elems = N * C * H * H
    total_bytes = 32.0 * elems                       # 12 B/elem forward + 20 B/elem backward (SURVEY §8d)
    fams = {k: dict(v, gbs=(v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["bytes"] > 0 else None),
                    us_per_launch=1e3 * v["ms"] / v["launches"], frac=(v["bytes"] / (v["ms"] * 1e-3) / 1e9 / peak if v["bytes"] > 0 else None))
            for k, v in prof.items() if v["ms"] > 0}
    gbs = total_bytes * steps / (ms * 1e-3) / 1e9
    ratio, ratio_src = None, None
    for name in ("traffic_r02.json", "traffic_r01.json"):
        try:
            tab = json.load(open(os.path.join(ROOT, "profiles", name)))["tensor_core_path"]
            if gs >= 8:
                ratio, ratio_src = tab["traffic_over_algorithmic"]["fwd+bwd (all launches)"], tab["source"]
            break
        except Exception:
            pass
    tc = gs >= 8
    return {
        "metric": "WTransform2d fwd+bwd microbench", "value": steps / (ms * 1e-3), "unit": "iterations/s",
        "n_gpus": 1, "steps": steps, "warmup": warm, "ms_per_step": ms / steps,
        "eager_ms_per_step": eager_ms / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (tf32 tensor-core contraction with hi/lo split operands, split-tf32 apply, fp32 accumulate)" if tc else "f32",
        "data": "synthetic",
        "config": {"workload": f"WTransform2d N={N} C={C} H=W={H} group_size={gs} fwd+bwd",
                   "l2": f"tensor of {elems * 4 / 1e6:.0f} MB > 126 MB L2",
                   "launch": "cuda-graph replay" if graph is not None else "eager"},
        "roofline": {"bound": "hbm", "kernel": "fwd+bwd (all launches of the layer)", "achieved": gbs, "peak": peak, "unit": "GB/s",
                     "frac": gbs / peak, "traffic": ratio * total_bytes if ratio else None, "traffic_source": ratio_src,
                     "algorithmic_bytes_per_step": total_bytes, "peak_source": peak_src},
        "kernels": fams, "clocks": clocks.summary(), "gpu_launches": int(sum(v["launches"] for v in prof.values()) // steps),
        "status_word": _native.status_all(device),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=["resnet", "microbench"], default="resnet")
    ap.add_argument("--per-domain", type=int, default=64)
    ap.add_argument("--site-mode", choices=["fused", "modules"], default="fused")
    ap.add_argument("--memory-format", choices=["nchw", "nhwc"], default="nhwc",
                    help="activation layout of the GPU arm (nhwc = torch.channels_last end to end)")
    ap.add_argument("--cpu-per-domain", type=int, default=16,
                    help="per-domain batch of the CPU arm (a bounded sample of the GPU arm's 3x64-image step)")
    ap.add_argument("--micro-cpu-n", type=int, default=32, help="batch size of the CPU leg of the microbench (N scaled down)")
    ap.add_argument("--no-extras", dest="extras", action="store_false",
                    help="skip the microbench and reference-on-GPU sub-records of the default N=1 line")
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-cuda-graph", dest="cuda_graph", action="store_false",
                    help="time the eager step instead of a CUDA-graph replay of it")
    ap.add_argument("--sites-out", default="", help="write the per-site kernel table (JSON) here")
    ap.add_argument("--stem-pad", type=int, default=0, choices=[0, 4, 8],
                    help="zero-pad the 3-channel image (and the stem weight) to this many channels for cuDNN")
    ap.add_argument("--no-grad-fork", dest="grad_fork", action="store_false",
                    help="sum the two gradients of every block input with autograd's add instead of inside the site's backward kernels")
    ap.add_argument("--stem", default=DEFAULT_STEM, choices=["direct", "s2d"],
                    help="s2d: the 7x7/2 stem convolution as a 4x4/1 convolution of the 2x2 space-to-depth image (same arithmetic)")
    ap.add_argument("--stem-nchw", action="store_true", help="run only the 3-channel stem convolution in NCHW (experiment)")
    ap.add_argument("--grad-gather", choices=["accumulate", "copy"], default="copy",
                    help="how gradients reach the flat all-reduce buffer: autograd accumulates into views of it, or one "
                         "multi-tensor copy after backward")
    ap.add_argument("--grad-segments", type=int, default=1, choices=[1, 2, 3],
                    help="pieces the flat gradient buffer is all-reduced in (1 = one collective after backward)")
    ap.add_argument("--micro-n", type=int, default=256)
    ap.add_argument("--micro-gs", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last timed training step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "resnet"):
        ap.error("--dump-outputs writes the outputs of the ResNet-50-DWT training step: --impl ours --workload resnet")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
