#!/usr/bin/env python
"""bench.py -- images/sec of the ResNet-34 160x384 waypoint train step (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU under torchrun for N>1)
  python bench.py --impl reference --gpus N --steps K ...  the reference's CPU implementation of the same step
  python bench.py ... --dump-outputs DIR                   also writes what the last timed step computed (Workload.dump)

Workload (config.workload = "config2"): BASELINE.json configs[1] -- ImagePolicyModelSS('resnet34'), synthetic
batch 256/GPU, one full training step = student forward (train-mode BN) + phase-0 L1 waypoint loss against fixed
image-space targets + backward + Adam(lr=1e-4); data-parallel replicas all-reduce the gradient once per step.
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (which may be read-only)

GFLOP_PER_TRAIN_IMG = 28.034      # SURVEY.md 8(d): 3 x 9.441116 - 0.289014 (no dgrad for the stem)
DUMP_SAMPLE = 1 << 20             # parameters (and their gradients) written by --dump-outputs: 4 MB each in float32
METRIC = "images/sec (ResNet34 160x384 waypoint train step)"
# BASELINE.json configs -> workloads (SURVEY.md 8(d)); ALGORITHMIC conv GFLOP per training image
WORKLOADS = {
    "config2": dict(metric=METRIC, gflop=28.034, model="ImagePolicyModelSS resnet34 160x384",
                    step="student fwd+bwd+Adam, phase-0 L1 vs fixed targets"),
    # train_image_phase1.py:157-229: teacher forward (eval BN, no_grad) + student step with the phase-1 transform + L1 on all
    # four branches; under torchrun this is BASELINE's config 4 (data-parallel phase 1)
    "config3": dict(metric=METRIC, gflop=28.034 + 3.177972, model="ImagePolicyModelSS resnet34 160x384 + BirdViewPolicyModelSS resnet18 teacher",
                    step="teacher fwd (eval) + student fwd+bwd+Adam, phase-1 CoordConverter + L1 vs teacher, all branches"),
    # train_birdview.py:102-153: the privileged ResNet-18 agent's own train step
    "config5": dict(metric="images/sec (ResNet18 192x192 birdview waypoint train step)", gflop=9.129,
                    model="BirdViewPolicyModelSS resnet18 192x192x7", step="birdview fwd+bwd+Adam, L1 vs ground-truth waypoints"),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi sampled every 50 ms in a side process.  It is started before the warm-up (nvidia-smi needs a few hundred
    ms to come up) and only the samples stamped inside [mark(), stop()] -- the timed regions -- are reported."""
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines, self.windows = index, None, [], []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):             # a timed region starts
        self.windows.append([time.time(), None])

    def end(self):              # ... and ends
        if self.windows and self.windows[-1][1] is None:
            self.windows[-1][1] = time.time()

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.end()
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], None, [], set()
        for stamp, ln in self.lines:
            # a line is printed right after its sample is taken: keep those received inside the marked window
            if self.windows and not any(a <= stamp <= b + 0.02 for a, b in self.windows):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_min_mhz=(sm[0] if sm else None), sm_max_mhz=mx,
                    power_w_max=(max(power) if power else None), reasons=sorted(reasons), samples=len(sm),
                    window="device-resident timed loop + the two end-to-end timed loops")


def synthetic(B, seed, torch):
    """SURVEY 8(d) distributions: uint8-quantised RGB, Bernoulli(0.2) bird's-eye masks, speed U[0,10), command {1..4},
    image-space targets U[0,384)x[0,160), map-space waypoints U[0,192)."""
    g = torch.Generator().manual_seed(seed)
    rgb_u8 = torch.randint(0, 256, (B, 3, 160, 384), dtype=torch.uint8, generator=g)
    bev_u8 = (torch.rand(B, 7, 192, 192, generator=g) > 0.8).to(torch.uint8) * 255      # {0,255} masks -> ToTensor -> {0,1}
    speed = torch.rand(B, generator=g) * 10
    cmd = torch.randint(1, 5, (B,), generator=g).float()
    target = torch.rand(B, 5, 2, generator=g) * torch.tensor([384.0, 160.0])
    loc = torch.rand(B, 5, 2, generator=g) * 192
    return dict(rgb_u8=rgb_u8, bev_u8=bev_u8, speed=speed, cmd=cmd, target=target, location=loc)


def cpu_threads():
    """Threads for the CPU arm.  Measured on the 128-thread GPU host: torch/oneDNN on this B=8 step is ~20x SLOWER with
    128 intra-op threads (0.6 img/s) than with a few dozen, so the arm uses min(cores, LBC_CPU_THREADS or 32)."""
    n = os.cpu_count() or 1
    return max(1, min(n, int(os.environ.get("LBC_CPU_THREADS", "32"))))


def cpu_step_rate(torch, workload, B, warm, iters, threads=None):
    """The reference's CPU implementation of the workload's step (oracle port: torch CPU kernels + Adam), images/s."""
    import lbc_oracle as orc
    import learningbycheating_b200 as lbc
    if threads:
        torch.set_num_threads(threads)
    torch.manual_seed(0)
    student = orc.leafify(lbc.ImagePolicyModelSS("resnet34", all_branch=True).state_dict())
    teacher_mod = lbc.BirdViewPolicyModelSS("resnet18", all_branch=True)
    d = synthetic(B, 1, torch)
    rgb, bev = d["rgb_u8"].float() / 255, d["bev_u8"].float() / 255
    st = orc.new_adam_state()
    if workload == "config2":
        oh = orc.one_hot(d["cmd"])

        def step():
            for k in orc.param_keys(student):
                student[k].grad = None
            pred, _, newbuf = orc.policy_forward(student, rgb, d["speed"], oh, "resnet34", True, True)
            loss = orc.phase0_loss(pred, d["target"]).mean()
            loss.backward()
            st["step"] += 1
            with torch.no_grad():
                pk = [k for k in orc.param_keys(student) if student[k].grad is not None]
                for k in pk:
                    if k not in st["m"]:
                        st["m"][k] = torch.zeros_like(student[k])
                        st["v"][k] = torch.zeros_like(student[k])
                orc.adam_step({k: student[k] for k in pk}, {k: student[k].grad for k in pk}, st["m"], st["v"], st["step"])
                for k, v in newbuf.items():
                    student[k] = v
    elif workload == "config3":
        teacher = {k: v.clone() for k, v in teacher_mod.state_dict().items()}

        def step():
            orc.train_step(student, teacher, rgb, bev, d["speed"], d["cmd"], 1, adam_state=st)
    else:
        teacher = orc.leafify(teacher_mod.state_dict())

        def step():
            orc.birdview_train_step(teacher, bev, d["location"], d["speed"], d["cmd"], adam_state=st)

    for _ in range(warm):
        step()
    t0 = time.time()
    for _ in range(iters):
        step()
    dt = time.time() - t0
    return B * iters / dt, dt / iters


def mem_available_gb():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                return int(line.split()[1]) / 1e6
    except OSError:
        pass
    return 0.0


def run_reference(args):
    """The reference's own CPU implementation of the step (its only one: SURVEY.md 0 -- the repo ships no CUDA code) on the
    host cores: the oracle port of the workload.  Two samples, each `steps` timed iterations after `warmup` untimed ones: the
    reference's config-1 batch (8), and -- memory permitting -- the like-for-like batch of our arm (256, ~10 s per iteration
    on 32 threads); `value` is the like-for-like one when it ran."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    cores = cpu_threads()
    torch.set_num_threads(cores)
    rate8, sec8 = cpu_step_rate(torch, args.workload, 8, args.warmup, args.steps, cores)
    rate, sec, B = rate8, sec8, 8
    like = None
    if args.batch > 8 and mem_available_gb() > 120 and os.environ.get("LBC_CPU_LIKE_FOR_LIKE", "1") != "0":
        try:    # ~35 GB of autograd state at batch 256
            r, s_ = cpu_step_rate(torch, args.workload, args.batch, args.warmup, args.steps, cores)
            like = dict(value=r, batch_per_step=args.batch, sec_per_step=s_, timed_steps=args.steps)
            rate, sec, B = r, s_, args.batch
        except Exception as e:     # never let the optional sample take the arm down
            like = dict(error=str(e)[:200])
    sample = ("oracle port (torch CPU fp32) of the %s step, batch %d per step, %d of %d host threads (more threads are slower "
              "for this model)" % (args.workload, B, cores, os.cpu_count() or 1))
    out = dict(impl="reference", metric=wl["metric"], value=rate, unit="images/s", n_gpus=args.gpus, steps=args.steps,
               warmup=args.warmup, ms_per_step=sec * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
               dtype="f32", data="synthetic",
               config=dict(workload=args.workload, model=wl["model"], step=wl["step"], batch_per_step=B, batch_per_gpu=B,
                           global_batch=B),
               cpu_baseline=dict(value=rate, unit="images/s", cores=torch.get_num_threads(), kind="port", sample=sample,
                                 batch8=dict(value=rate8, sec_per_step=sec8, timed_steps=args.steps), like_for_like=like),
               e2e=dict(value=rate, unit="images/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(out))


class Workload:
    """One BASELINE config on one rank: device-resident step, and the same step fed from pinned host buffers."""

    def __init__(self, name, args, dev, rank, torch):
        import learningbycheating_b200 as lbc
        from learningbycheating_b200 import train_birdview as tb, train_image_phase0 as p0, train_image_phase1 as p1
        from learningbycheating_b200.distributed import DataParallel
        self.name, self.torch, self.dev, self.lbc = name, torch, dev, lbc
        B = args.batch
        torch.manual_seed(0)
        student = lbc.ImagePolicyModelSS("resnet34", all_branch=True, lbc_precision=args.precision)
        teacher = lbc.BirdViewPolicyModelSS("resnet18", all_branch=True, lbc_precision=args.precision)
        d = synthetic(B, 1 + rank, torch)
        self.host = d
        oh_h = lbc.one_hot(d["cmd"])
        if name == "config5":
            self.net = teacher.to(dev).train()
            self.teacher = None
            self.crit = tb.LocationLoss(choice="l1")
        else:
            self.net = student.to(dev).train()
            self.teacher = teacher.to(dev).eval() if name == "config3" else None
            self.crit = p0.LocationLoss(device=dev) if name == "config2" else p1.LocationLoss()
            self.conv = p1.CoordConverter(fixed_offset=4.0, device=dev) if name == "config3" else None
        self.opt = lbc.Adam(self.net.parameters(), lr=1e-4)
        self.dp = DataParallel(self.net, self.opt, overlap=args.overlap)
        # device-resident inputs (frames as the float tensors the reference's DataLoader hands over)
        self.rgb = (d["rgb_u8"].float() / 255).to(dev)
        self.bev = (d["bev_u8"].float() / 255).to(dev)
        self.speed, self.oh = d["speed"].to(dev), oh_h.to(dev)
        self.target, self.loc = d["target"].to(dev), d["location"].to(dev)
        # pinned host buffers of the end-to-end loop: frames as the data collector stores them (uint8, HWC for the camera,
        # data_collector.py:234-252; CHW masks for the bird's-eye view), ToTensor's /255 runs on the device
        self.pin = dict(rgb_u8=d["rgb_u8"].permute(0, 2, 3, 1).contiguous().pin_memory(), bev_u8=d["bev_u8"].pin_memory(),
                        rgb_f=(d["rgb_u8"].float() / 255).pin_memory(), bev_f=(d["bev_u8"].float() / 255).pin_memory(),
                        speed=d["speed"].pin_memory(), oh=oh_h.pin_memory(), target=d["target"].pin_memory(),
                        loc=d["location"].pin_memory())

    # ---- one optimizer step from device tensors (rgb / bev may be uint8 frames)
    def step_from(self, rgb, bev, speed, oh, target, loc):
        torch = self.torch
        if self.name == "config5":
            pred, preds = self.net(bev, speed, oh)
            loss = self.crit(pred, loc).mean()
            self.outputs = dict(pred=pred, preds=preds, loss=loss)
        elif self.name == "config3":
            with torch.no_grad():
                _, t_preds = self.teacher(bev, speed, oh)
            pred, preds = self.net(rgb, speed, oh)
            loss = self.crit(self.conv(preds), t_preds).mean()
            self.outputs = dict(pred=pred, preds=preds, teacher_preds=t_preds, loss=loss)
        else:
            pred, preds = self.net(rgb, speed, oh)
            loss = self.crit(pred, target).mean()
            self.outputs = dict(pred=pred, preds=preds, loss=loss)
        self.opt.zero_grad()
        self.dp.backward(loss)
        self.dp.step_after_backward()
        return loss

    def step(self):
        return self.step_from(self.rgb, self.bev, self.speed, self.oh, self.target, self.loc)

    def host_batch(self, u8):
        p = self.pin
        rgb = (p["rgb_u8"] if u8 else p["rgb_f"]) if self.name != "config5" else None
        bev = (p["bev_u8"] if u8 else p["bev_f"]) if self.name != "config2" else None
        return (rgb, bev, p["speed"], p["oh"], p["target"] if self.name == "config2" else None,
                p["loc"] if self.name == "config5" else None)

    def h2d_bytes(self, u8):
        return sum(t.numel() * t.element_size() for t in self.host_batch(u8) if t is not None)

    def dump(self, directory):
        """--dump-outputs: what the last step handed its caller, as DIR/<name>.npy in float32 -- the predictions and loss
        (outputs of step_from), the floating-point buffers (BatchNorm running statistics), and the parameters and gradients
        the step left behind, sampled at DUMP_SAMPLE positions of the flattened parameters() (seed 0: the same positions on
        every run; a parameter the loss does not reach has gradient zero).  About 8 MB, whatever the batch."""
        import numpy as np
        torch = self.torch
        params = list(self.net.parameters())
        flat_p = torch.cat([p.detach().reshape(-1) for p in params]).float()
        grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in params]
        flat_g = torch.cat([g.detach().reshape(-1) for g in grads]).float()
        idx = torch.randperm(flat_p.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
        idx = idx.to(flat_p.device)
        arrays = {k: v.detach().float() for k, v in self.outputs.items()}
        bufs = [b.detach().reshape(-1).float() for b in self.net.buffers() if b.dtype.is_floating_point]
        arrays.update(params_sample=flat_p[idx], grads_sample=flat_g[idx], buffers=torch.cat(bufs))
        os.makedirs(directory, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(directory, name + ".npy"), a.cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from learningbycheating_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (our arm) needs a B200; there is no CPU path"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = None
    if world > 1:
        # pin this rank to the CPUs next to its GPU before any pinned host buffer is allocated: pinned pages land on that
        # NUMA node, so the per-step host->device copies of the end-to-end loop do not cross the socket interconnect
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
            pynvml.nvmlDeviceSetCpuAffinity(h)
            numa = sorted(os.sched_getaffinity(0))
            numa = "%d cpus (%d..%d)" % (len(numa), numa[0], numa[-1])
        except Exception as e:      # affinity is an optimisation, never a requirement
            numa = "unavailable: %s" % str(e)[:80]
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    # kernel variants (lbc_b200.h: lbc_set_fast_kernels): bit 0 CTA-pair GEMMs, 1 row-of-taps weight gradient, 2 its CTA-pair
    # variant, (3 stem layout: the library default), 4 / 5 shared-row kernel for the 128- / 256-channel 3x3 convolutions
    pair = args.pair if args.pair >= 0 else int(os.environ.get("LBC_PAIR", "127") or 0)
    L.lbc_set_fast_kernels((0 if args.no_fast else 1) | (4 if pair & 1 else 8) | (16 if pair & 2 else 32) | (64 if pair & 4 else 128) |
                           (1024 if pair & 16 else 2048) | (4096 if pair & 32 else 8192) | (16384 if pair & 64 else 32768) |
                           (65536 if pair & 128 else 131072))
    B = args.batch
    # watchdog over the device phases (normally seconds): a run that makes no progress dumps every thread's Python stack and
    # exits non-zero instead of sitting in its caller's timeout without a word (seen once in ~100 runs, never reproduced)
    import faulthandler
    limit = float(os.environ.get("LBC_BENCH_WATCHDOG_S", "0") or 0) or (600.0 + 2.0 * (args.steps + args.warmup))
    done = threading.Event()

    def watchdog():
        if not done.wait(limit):
            sys.stderr.write("bench.py: device phase exceeded %.0f s -- stack of every thread follows\n" % limit)
            faulthandler.dump_traceback(file=sys.stderr, all_threads=True)
            sys.stderr.flush()
            os._exit(3)
    threading.Thread(target=watchdog, daemon=True).start()
    wl = WORKLOADS[args.workload]
    w = Workload(args.workload, args, dev, rank, torch)
    step = w.step

    step()                      # builds the native engines (allocations) outside every timed region
    w.dp.sync_initial_state()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()         # comes up during the warm-up; only samples after sampler.mark() are reported
    for _ in range(args.warmup):
        step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    if rank == 0:
        sampler.mark()
    n0 = L.lbc_kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        loss = step()
    e1.record()
    barrier()
    if rank == 0:
        sampler.end()
        if args.dump_outputs:       # before any later step overwrites the state the last timed step left
            w.dump(args.dump_outputs)
    ms = e0.elapsed_time(e1)
    launches = L.lbc_kernel_launch_count() - n0
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * B * args.steps / (ms / 1e3)

    # ---- end to end through the public API with HOST buffers (pinned): every step's inputs are copied host->device
    # inside the timed region (on the package's CudaPrefetcher side stream, overlapping the previous step's compute)
    # and the step's loss is read back device->host.
    from learningbycheating_b200.data import CudaPrefetcher
    e2e_steps = args.steps      # same K as the device-resident loop (pipeline fill/drain is inside the region)

    def host_batches(n, u8):
        for _ in range(n):
            yield w.host_batch(u8)

    prefetch = CudaPrefetcher(None, dev)   # one loader for the whole run: its two staging slots are allocated once

    def e2e_run(n, u8):
        # every step's loss is read back to the host; the read of step i is issued after step i+1 has been enqueued
        # (as a logging loop would do), so the device never drains waiting for the host
        last, pending = None, None
        prefetch.iterable = host_batches(n, u8)
        for batch in prefetch:
            l = w.step_from(*batch)
            if pending is not None:
                last = pending.item()  # device -> host read of the previous step's loss
            pending = l.detach()
        if pending is not None:
            last = pending.item()
        return last

    def e2e_measure(u8):
        e2e_run(3, u8)
        barrier()
        if rank == 0:
            sampler.mark()
        e0.record()
        e2e_run(e2e_steps, u8)
        e1.record()
        barrier()
        if rank == 0:
            sampler.end()
        tt = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return world * B * e2e_steps / (float(tt.item()) / 1e3)

    e2e_run(2, False)               # both variants warmed (pinned-host / side-stream allocator pools) before either is timed
    e2e_run(2, True)
    e2e_fp32 = e2e_measure(False)
    e2e_value = e2e_measure(True)
    clocks = sampler.stop() if rank == 0 else None
    h2d, h2d_fp32 = w.h2d_bytes(True), w.h2d_bytes(False)

    # ---- per-category device timing (CUDA events on the launching stream) for the roofline of the dominant kernel
    roof = None
    cats = {}
    nprof = 2
    if rank == 0:
        L.lbc_prof_reset()
        L.lbc_prof_enable(1)
    for _ in range(nprof):      # every rank steps (the step contains the gradient all-reduce); rank 0 records
        step()
    torch.cuda.synchronize()
    if rank == 0:
        import ctypes
        peaks = load_peaks()
        L.lbc_prof_enable(0)
        for cat in ("conv_fwd", "conv_dgrad", "conv_wgrad", "bn_fwd", "bn_bwd", "pool", "elementwise", "head", "pack"):
            msd, cnt, fl, by = ctypes.c_double(), ctypes.c_longlong(), ctypes.c_double(), ctypes.c_double()
            _lib.check(L.lbc_prof_get(cat.encode(), ctypes.byref(msd), ctypes.byref(cnt), ctypes.byref(fl), ctypes.byref(by)))
            cats[cat] = dict(ms_per_step=msd.value / nprof, launches_per_step=cnt.value / nprof,
                             gflop_per_step=fl.value / nprof / 1e9, gbytes_per_step=by.value / nprof / 1e9)
        L.lbc_prof_reset()
        conv_ms = sum(cats[c]["ms_per_step"] for c in ("conv_fwd", "conv_dgrad", "conv_wgrad"))
        conv_gf = sum(cats[c]["gflop_per_step"] for c in ("conv_fwd", "conv_dgrad", "conv_wgrad"))
        achieved = conv_gf / conv_ms if conv_ms > 0 else 0.0     # GFLOP/ms == TFLOP/s
        bn_ms = cats["bn_fwd"]["ms_per_step"] + cats["bn_bwd"]["ms_per_step"]
        bn_gb = cats["bn_fwd"]["gbytes_per_step"] + cats["bn_bwd"]["gbytes_per_step"]
        bn_gbs = bn_gb / bn_ms * 1e3 if bn_ms > 0 else 0.0
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "ncu_summary.json")
        if os.path.exists(tpath):       # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
            try:
                dk = json.load(open(tpath)).get("dominant_kernel")
                traffic, traffic_src = dk["dram_total"], dict(kernel=dk["kernel"], capture=dk["capture"],
                                                             algorithmic_bytes=dk["algorithmic_bytes"])
            except Exception:
                traffic = None
        split = args.precision == "fp32tc"
        roof = dict(bound="tensor", kernel="tcgen05 implicit-GEMM convolutions (fwd + dgrad + wgrad, all layers; CUDA-event "
                                           "brackets on the launching stream)" + (" -- split-precision mode: 3 MMAs per "
                                           "algorithmic product" if split else ""),
                    achieved=achieved, peak=peaks["tf_sust"], unit="TFLOP/s", frac=achieved / peaks["tf_sust"],
                    traffic=traffic, traffic_of=traffic_src, peak_source=peaks["source"] + " bf16_tflops_sustained (kernels timed inside a long step)",
                    hbm_kernels=dict(kernel="BatchNorm statistics/apply/backward kernels", achieved=bn_gbs, peak=peaks["hbm"],
                                     unit="GB/s", frac=bn_gbs / peaks["hbm"], bytes="algorithmic (DESIGN.md section 3)"),
                    per_category=cats)

    done.set()                  # device phases over: the CPU baseline below takes its own time
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = cpu_threads()
        rate, sec = cpu_step_rate(torch, args.workload, 8, 1, 4, cores)
        cpu_base = dict(value=rate, unit="images/s", cores=torch.get_num_threads(), kind="port",
                        sample="oracle port (torch CPU fp32) of the same step, batch 8, 4 timed iterations, %d of %d host threads"
                               % (cores, os.cpu_count() or 1))

    if rank == 0:
        out = dict(metric=wl["metric"], value=value, unit="images/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                   ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                   dtype={"bf16": "bf16", "fp32": "f32", "fp32tc": "f32 (split-precision tensor-core GEMMs)"}[args.precision],
                   data="synthetic",
                   config=dict(workload=args.workload, model=wl["model"], global_batch=world * B,
                               batch_per_gpu=B, parallelism="dp%d" % world, step=wl["step"],
                               l2="inputs+activations per step (>5 GB) far exceed the 126 MB L2; no explicit flush",
                               fast_kernels=not args.no_fast, cta_pair_gemm=bool(pair & 1), wgrad_row_of_taps=bool(pair & 2),
                               wgrad_cta_pair=bool(pair & 4), shared_row_conv=("layers 2-3" if pair & 32 else "layer 2" if pair & 16 else "off"), wgrad_nine_taps_c64=bool(pair & 64), layer1_on_pair_kernel=bool(pair & 128),
                               schedule=dict(wgrad_side_stream=int(os.environ.get("LBC_WGRAD_OVERLAP", "1")),
                                             pdl=int(os.environ.get("LBC_PDL", "1"))), cpu_affinity=numa, allreduce=("bucketed, overlapped with backward" if w.dp.overlap else "single, after backward") if world > 1 else "none"),
                   e2e=dict(value=e2e_value, unit="images/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=4, steps=e2e_steps,
                            frames="uint8 host frames (pinned), copied on the prefetch stream every step",
                            fp32_frames=dict(value=e2e_fp32, h2d_bytes_per_step=h2d_fp32)),
                   gpu_launches=int(launches), clocks=clocks, roofline=roof, cpu_baseline=cpu_base,
                   step_tflops=value * wl["gflop"] / 1e3, last_loss=float(loss.detach()))
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    # `kill -USR1 <pid>` (or `timeout -s USR1 ...`) dumps the Python stack of every thread: tells a device hang from a host one
    import faulthandler
    import signal
    faulthandler.register(signal.SIGUSR1, all_threads=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="images per GPU per step")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32", "fp32tc"])
    ap.add_argument("--no-fast", action="store_true", help="correctness-first kernels only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="config2", choices=sorted(WORKLOADS), help="BASELINE.json config (config3 under "
                    "torchrun = config4)")
    ap.add_argument("--overlap", action="store_true", help="bucketed all-reduce overlapped with backward instead of the "
                    "single all-reduce after backward (measured equal-to-slightly-slower on 2 GPUs: distributed.py)")
    ap.add_argument("--pair", type=int, default=-1, help="kernel variants: bit 0 = CTA-pair (cta_group::2) implicit-GEMM kernels, "
                                                         "bit 1 = row-of-taps weight gradient (default: LBC_PAIR)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to "
                    "DIR/<name>.npy (float32; inputs are seeded, so two builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of our arm's step; the reference arm has none to write")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
