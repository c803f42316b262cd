#!/usr/bin/env python
"""OSVOS hot-path benchmark (contract: the task statement; method: DESIGN.md section 6).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload infer480|train480|parent480]
                    [--dump-outputs DIR]

Default run (`--workload infer480`, what the driver launches), ONE JSON line on rank 0:

  headline   BASELINE.json configs[1]: forward of one 480x854 frame per step and GPU, device-resident (`value`) and end to
             end from pinned host memory (`e2e`).  Each is timed over exactly K steps between barrier + synchronize
             pairs, CUDA events on the launching stream, max over ranks.  K steps of a 0.7 ms frame are a short window:
             it takes a K of about 1500 to time a second.
  dp         BASELINE.json configs[3], the one multi-GPU path north_star names: parent training, batch 12 per GPU at
             480x854, 5-loss objective, FusedSGD, ONE NCCL allreduce(mean) of the 59.7 MB gradient bucket per step; run
             at every N including 1, with its own parity check (R ranks x 1 small frame against the oracle's
             nAveGrad = R accumulation, reference train_parent.py:163-172).
  parity     the CUDA forward against the CPU oracle on the benchmarked 480x854 frame: per-map max-rel logit error, mask
             flips (total / outside the |logit| < 1e-3 max band), IoU.
  roofline   dominant kernel class = the tcgen05 3x3 convolutions; per-launch CUDA events behind a parked GPU.
  gpu_reference   the UNMODIFIED reference modules (oracle/_ref) on the same B200 through cuDNN: TF32 default, strict
             fp32, channels_last + bf16 autocast - "the real kernel to beat" (SURVEY.md 8d).
  cpu_baseline    the same reference modules on the host cores (bounded sample).

`--impl reference` times the reference's own CPU path (oracle/_ref when present, else the oracle port).

`--dump-outputs DIR` writes what the timed path returned in its last step as DIR/<name>.npy (float32): the five logit
maps (infer480), the loss and the parameter gradients of that step (train480), the five losses and the updated
parameters (parent480).  Inputs and weights are seeded, so two builds run with the same arguments can be compared
output for output: the inference maps bit for bit; the training paths with a tolerance, as their gradient reductions are
not deterministic.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

# Only the result line may appear on stdout: libraries (NCCL prints its version banner there when NCCL_DEBUG=VERSION)
# are redirected to stderr for the lifetime of the process; emit() writes to the saved descriptor.
_RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line):
    _RESULT_OUT.write(json.dumps(line) + "\n")
    _RESULT_OUT.flush()


ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 480, 854
METRIC = "frames/sec at 480x854 fwd-only, batch 1 per GPU (OSVOS.forward -> 5 logit maps)"
MAX_DUMP_BYTES = 64 * 10**6    # --dump-outputs budget


def workload_label(workload):
    """The same string in the native and the reference arm."""
    return (f"{workload}: 1x3x{H}x{W} synthetic BGR frame per step (seeded, mean-subtracted 0..255), OSVOS VGG-16 trunk + 4 side "
            f"branches, seeded He-init weights")


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "tflops_burst": p["bf16_tflops"],
                "tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML polled in-process every ~5 ms (a timed window
    can be tens of ms, nvidia-smi's 100 ms loop never landed in it), nvidia-smi as the fallback."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, cuda_index):
        self.rows, self.stop_flag, self.thread, self.handle, self.nv, self.proc = [], False, None, None, None, None
        self.cuda_index = cuda_index
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            self.nv = pynvml
        except Exception:
            self.nv = None

    def _poll(self):
        nv, h = self.nv, self.handle
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    pw = None
                self.rows.append((sm, reasons, pw))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        self.rows, self.stop_flag = [], False
        if self.nv is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:                                                  # fallback: nvidia-smi loop
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.cuda_index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.smi_rows = []
            self.thread = threading.Thread(target=lambda: [self.smi_rows.append([v.strip() for v in l.split(",")])
                                                           for l in self.proc.stdout], daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.nv is not None:
            self.stop_flag = True
            if self.thread is not None:
                self.thread.join(timeout=1)
            sm = [r[0] for r in self.rows]
            pw = [r[2] for r in self.rows if r[2] is not None]
            mask = 0
            for r in self.rows:
                mask |= int(r[1])
            try:
                mx = self.nv.nvmlDeviceGetMaxClockInfo(self.handle, self.nv.NVML_CLOCK_SM)
            except Exception:
                mx = None
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                    "sm_max_mhz": mx, "power_w_max": max(pw) if pw else None, "samples": len(sm),
                    "reasons": [n for n, bit in self.REASONS if mask & bit], "how": "NVML polled in-process every 5 ms"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvml and nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for r in self.smi_rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        return {"sm_mhz": statistics.median([float(r[0]) for r in rows]) if rows else None,
                "sm_max_mhz": max([float(r[1]) for r in rows]) if rows else None,
                "power_w_max": max([float(r[2]) for r in rows if r[2].replace(".", "").isdigit()] or [0.0]),
                "samples": len(rows), "how": "nvidia-smi -lms 20",
                "reasons": [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]}


# ----------------------------------------------------------------------------------------------------------------
# CPU legs (reference arm, cpu_baseline): the reference's own modules from oracle/_ref, else the oracle port
# ----------------------------------------------------------------------------------------------------------------
def cpu_reference_fps(steps, warmup, workload):
    """The reference's CPU path (PyTorch fp32 / MKLDNN) on the host cores -> (fps, ms, cores, threads, kind)."""
    import torch
    from oracle import osvos_oracle as oc
    from oracle import ref_loader
    cores = os.cpu_count() or 1
    params = oc.he_params(seed=0)
    x, gt = oc.synthetic_frame(1, H, W, 1234)
    if ref_loader.available():
        kind = "reference"
        ref = ref_loader.load()
        net = ref_loader.build_reference(params, "cpu")

        def fwd():
            with torch.no_grad():
                return net(x)

        def fwd_bwd():
            net.zero_grad()
            outs = net(x)
            ref.layers.class_balanced_cross_entropy_loss(outs[-1], gt, size_average=False).backward()
    else:
        kind = "port"

        def fwd():
            with torch.no_grad():
                return oc.osvos_forward(params, x)

        def fwd_bwd():
            oc.forward_backward(params, x, gt, objective="online")
    one = fwd_bwd if workload == "train480" else fwd

    def probe(threads):
        torch.set_num_threads(threads)
        fwd()                                    # warm-up (thread pool, MKLDNN primitives)
        t0 = time.perf_counter()
        fwd()
        return time.perf_counter() - t0
    # "all the host threads it can use": torch's CPU conv slows down when oversubscribed on many-core hosts,
    # so the thread count is the fastest of {all cores, 64, 32, 16} on a one-frame probe.
    cands = sorted({c for c in (cores, 64, 32, 16) if c <= cores}, reverse=True)
    best = min(cands, key=probe)
    torch.set_num_threads(best)
    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = (time.perf_counter() - t0) / steps
    return 1.0 / dt, dt * 1e3, cores, torch.get_num_threads(), kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 60))          # bounded sample: ~0.45 s per frame on the host cores
    warmup = max(3, min(args.warmup, 20))        # same rule as the native arm (W >= 3)
    workload = "train480" if args.workload == "train480" else "infer480"
    fps, ms, cores, threads, kind = cpu_reference_fps(steps, warmup, workload)
    what = ("the unmodified reference modules (oracle/_ref: networks/vgg_osvos.py + layers/osvos_layers.py)"
            if kind == "reference" else "oracle port of the reference")
    line = {"impl": "reference", "metric": METRIC if workload == "infer480" else METRIC.replace("fwd-only", "fwd+bwd"),
            "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_label(workload)},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": kind,
                             "sample": f"{steps} steps of the full 480x854 frame after {warmup} warm-up: {what}, torch CPU "
                                       f"fp32 (MKLDNN) on {threads} threads of {cores} host cores"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ----------------------------------------------------------------------------------------------------------------
# timing helpers
# ----------------------------------------------------------------------------------------------------------------
class Timer:
    def __init__(self, dev, world):
        self.dev, self.world = dev, world

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        import torch
        import torch.distributed as dist
        t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def block(self, fn, k, after=None):
        """EXACTLY k steps between barrier + synchronize pairs; device time (CUDA events), max over ranks -> ms."""
        import torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            fn(i)
        if after is not None:
            after()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))

    def steps(self, fn, k, after=None):
        """Exactly k timed steps in one block -> (ms per step, info dict)."""
        ms = self.block(fn, k, after)
        return ms / k, {"timed_steps": k, "timed_ms_total": ms}


def dump_outputs(out_dir, arrays):
    """{name: tensor} -> out_dir/<name>.npy in float32."""
    import numpy as np
    host = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    assert total <= MAX_DUMP_BYTES, f"--dump-outputs: {total} bytes exceed {MAX_DUMP_BYTES}"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


# ----------------------------------------------------------------------------------------------------------------
# dp: parent training, batch 12 per GPU, gradient allreduce (BASELINE.json configs[3])
# ----------------------------------------------------------------------------------------------------------------
def dp_parity(rank, world, dev, precision):
    """R ranks x ONE small frame each, parent objective, allreduce(mean) of the bucket, against the single-process
    oracle with nAveGrad = R (reference train_parent.py:163-172).  -> dict on rank 0 (None elsewhere)."""
    import torch
    from oracle import osvos_oracle as oc
    from osvos_pytorch_b200 import parallel, training
    from osvos_pytorch_b200.networks.vgg_osvos import OSVOS
    h, w = 64, 96
    net = OSVOS(pretrained=0, verbose=False, precision=precision)
    net.load_state_dict(oc.he_params(seed=0), strict=False)
    net.to(dev).train()
    bucket = parallel.GradientBucket(parallel.trainable_parameters(net), dev)
    x, gt = oc.synthetic_frame(1, h, w, 500 + rank)
    outs = net(x.to(dev))
    losses = [training.class_balanced_cross_entropy_loss(o, gt.to(dev), size_average=False) for o in outs]
    (0.5 * sum(losses[:-1]) + losses[-1]).backward()
    bucket.allreduce_mean()
    torch.cuda.synchronize()
    if rank != 0:
        return None
    got = {n: p.grad.detach().cpu() for n, p in net.named_parameters() if not n.startswith("upscale")}
    params = oc.he_params(seed=0)
    acc = None
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    for r in range(world):
        xr, gr = oc.synthetic_frame(1, h, w, 500 + r)
        _, _, g = oc.forward_backward(params, xr, gr, objective="parent", side_weight=0.5, grad_scale=1.0 / world)
        acc = g if acc is None else {k: acc[k] + g[k] for k in g}
    errs = {k: float((got[k].double() - v.double()).norm() / v.double().norm()) for k, v in acc.items()}
    head = {k: e for k, e in errs.items() if k.startswith(("fuse", "score_dsn", "side_prep"))}
    trunk = {k: e for k, e in errs.items() if k not in head}
    tol_head, tol_trunk = 1e-3, 4e-2
    return {"frame": f"{world} ranks x 1x3x{h}x{w}", "oracle": f"single process, nAveGrad = {world} (train_parent.py:163-172)",
            "worst_rel_err": max(errs.values()), "worst_param": max(errs, key=errs.get),
            "worst_rel_err_side_fuse": max(head.values()), "worst_rel_err_trunk": max(trunk.values()),
            "tolerance": {"side_fuse": tol_head, "trunk": tol_trunk,
                          "note": "trunk bound = ReLU / argmax flips on a tiny map, tests/test_gpu_backward.py"},
            "ok": bool(max(head.values()) < tol_head and max(trunk.values()) < tol_trunk), "params_checked": len(errs)}


def run_dp(args, rank, world, local, dev, timer, steps, dump_dir=None):
    """-> the `dp` object (rank 0) : parent480, per-GPU batch `args.batch`, one allreduce(mean) + FusedSGD step per step.
    dump_dir: rank 0 writes the last timed step's losses and the parameters it updated there."""
    import torch
    import torch.distributed as dist
    from osvos_pytorch_b200 import ops, parallel, training
    from osvos_pytorch_b200.networks.vgg_osvos import OSVOS, he_init_
    parity = dp_parity(rank, world, dev, args.precision)
    net = he_init_(OSVOS(pretrained=0, verbose=False, precision=args.precision), seed=0)
    with torch.no_grad():               # keep the synthetic logits O(10), as train_online.py --synthetic does
        for mod in list(net.side_prep) + [net.fuse]:
            mod.weight.mul_(0.1)
    net = net.to(dev)
    parallel.broadcast_parameters(net, src=0)
    # one-launch SGD + grad zeroing + weight repack.  lr: He-init synthetic weights give O(1e5) summed losses whose
    # gradients make the reference's 1e-8 diverge within tens of steps; the arithmetic of a step does not depend on lr.
    opt = training.make_optimizer(net, "parent", lr=args.dp_lr, fused=True)
    bucket = parallel.GradientBucket(parallel.trainable_parameters(net), dev)
    bucket.time_collective = True
    batches = [training.synthetic_batch(args.batch, H, W, 1000 * rank + i, dev) for i in range(2)]
    loss_log = []

    def one(i):
        loss_log.append(training.parent_epoch(net, opt, bucket, [batches[i % 2]], 0, 240, 1))
    for i in range(3):
        one(i)
    torch.cuda.synchronize()
    l0 = ops.KERNEL_LAUNCHES[0]
    one(0)
    launches = ops.KERNEL_LAUNCHES[0] - l0
    bucket.collective_events.clear()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, info = timer.steps(one, steps)
    clocks = sampler.stop() if rank == 0 else None
    # the collective as it ran INSIDE the steps (device time between the events around it on this rank: payload +
    # waiting for the slowest rank), and alone, back to back (payload only)
    torch.cuda.synchronize()
    in_step = [a.elapsed_time(b) for a, b in bucket.collective_events]
    ar_in_step = timer.max_over_ranks(statistics.median(in_step)) if in_step else 0.0
    ar_alone = 0.0
    if world > 1:
        bucket.time_collective = False
        for _ in range(3):
            bucket.allreduce_mean()
        ar_alone = timer.block(lambda i: bucket.allreduce_mean(), 20) / 20
    # loss after the timed steps must be finite on every rank (a diverged / NaN replica would still "run")
    with torch.no_grad():
        net.eval()
        probe = net(batches[0]["image"][:1])[-1]
        finite = torch.tensor([float(torch.isfinite(probe).all())], device=dev)
        net.train()
    if world > 1:
        dist.all_reduce(finite, op=dist.ReduceOp.MIN)
    torch.cuda.synchronize()
    first, last = loss_log[0].tolist(), loss_log[-1].tolist()     # device tensors until here: no host sync per step
    if rank != 0:
        return None
    if dump_dir is not None:
        dump_outputs(dump_dir, {"losses": loss_log[-1], **{"param." + n: p for n, p in net.named_parameters()
                                                            if not n.startswith("upscale")}})
    fps = world * args.batch * 1000.0 / ms
    return {"workload": f"parent480 (BASELINE configs[3]): per-GPU batch {args.batch} x 3x{H}x{W} synthetic frames, global "
                        f"batch {world * args.batch}, 5-loss parent objective (train_parent.py:143-147), FusedSGD(lr {args.dp_lr:g}, "
                        f"mom .9, wd 2e-4), one optimizer step per step; He-init weights with the side branch scaled by 0.1",
            "parallelism": f"dp{world}: one ncclAllReduce(AVG) of the flat fp32 gradient bucket "
                           f"({bucket.numel * 4 / 1e6:.1f} MB) per step; weak scaling",
            "fps": fps, "fps_per_gpu": fps / world, "ms_per_step": ms, "steps": steps, **info,
            "allreduce_ms": ar_alone, "allreduce_share": ar_alone / ms if ms else None,
            "allreduce_in_step_ms": ar_in_step, "allreduce_in_step_share": ar_in_step / ms if ms else None,
            "allreduce_note": "allreduce_ms = the collective alone, back to back (payload cost); in_step = device time "
                              "between events around it inside the timed steps, max over ranks (payload + waiting for the "
                              "slowest rank = skew)",
            "nccl_ranks": world, "gpu_launches": int(launches), "outputs_finite_all_ranks": bool(float(finite) == 1.0),
            "optimizer_steps_run": len(loss_log), "losses_first_step": first, "losses_last_step": last,
            "losses_finite": bool(all(math.isfinite(v) for v in first + last)),
            "dtype": "bf16x3 (split-bf16 operands, fp32 accumulate)" if args.precision == "exact" else "bf16",
            "parity": parity, "clocks": clocks}


# ----------------------------------------------------------------------------------------------------------------
# parity of the benchmarked frame, gpu_reference
# ----------------------------------------------------------------------------------------------------------------
def forward_parity(net, dev):
    """CUDA forward vs the CPU oracle on the benchmarked 480x854 frame (north_star: logits within 1e-3 of max, masks equal)."""
    import torch
    from oracle import osvos_oracle as oc
    x, _ = oc.synthetic_frame(1, H, W, 1234)
    params = {k: v.detach().cpu() for k, v in net.state_dict().items() if not k.startswith("upscale")}
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    with torch.no_grad():
        ref = oc.osvos_forward(params, x)
        got = [o.cpu() for o in net(x.to(dev))]
    names = ["side1", "side2", "side3", "side4", "fused"]
    maps, flips_total, flips_outside = {}, 0, 0
    for n, g, r in zip(names, got, ref):
        scale = float(r.abs().max())
        diff = (g > 0) != (r > 0)
        outside = diff & (r.abs() > 1e-3 * scale)
        gi, ri = g > 0, r > 0
        union = float((gi | ri).sum())
        iou = float((gi & ri).sum()) / union if union > 0 else 1.0          # both masks empty: identical
        maps[n] = {"max_rel": float((g - r).abs().max()) / scale, "rms_rel": float((g - r).pow(2).mean().sqrt()) / scale,
                   "mask_flips": int(diff.sum()), "mask_flips_outside_band": int(outside.sum()), "iou": iou}
        flips_total += int(diff.sum())
        flips_outside += int(outside.sum())
    return {"frame": f"1x3x{H}x{W}, seed 1234, He-init weights (seed 0)", "oracle": "oracle/osvos_oracle.py (CPU fp32, pinned "
            "against the unmodified reference by tests/test_oracle.py)", "maps": maps,
            "worst_max_rel": max(m["max_rel"] for m in maps.values()), "tolerance_max_rel": 1e-3,
            "mask_flips_total": flips_total, "mask_flips_outside_band": flips_outside, "pixels_per_map": H * W,
            "band": "|reference logit| <= 1e-3 * max|reference logit| of the map (a flip inside it is below the logit tolerance)",
            "fused_iou": maps["fused"]["iou"],
            "ok": bool(max(m["max_rel"] for m in maps.values()) < 1e-3 and flips_outside == 0)}


def gpu_reference(dev):
    """The unmodified reference modules (oracle/_ref) on this GPU through PyTorch/cuDNN, same frame, fwd-only."""
    import torch
    from oracle import osvos_oracle as oc
    from oracle import ref_loader
    if not ref_loader.available():
        return {"unavailable": "oracle/_ref not built (bash oracle/make_ref.sh in the build container)"}
    params = oc.he_params(seed=0)
    x, _ = oc.synthetic_frame(1, H, W, 1234)
    with torch.no_grad():
        torch.set_num_threads(min(32, os.cpu_count() or 1))
        cpu = oc.osvos_forward(params, x)[-1]
    x = x.to(dev)
    out = {"what": "oracle/_ref networks/vgg_osvos.py OSVOS.forward on cuda (stock PyTorch eager + cuDNN), batch 1, "
                   "480x854, torch.no_grad, cudnn.benchmark=True, CUDA events over 60 iterations after 15 warm-up"}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        for mode in ("tf32_default", "fp32", "bf16_channels_last"):
            net = ref_loader.build_reference(params, dev).eval()
            torch.backends.cudnn.benchmark = True
            torch.backends.cudnn.allow_tf32 = mode != "fp32"
            torch.backends.cuda.matmul.allow_tf32 = mode != "fp32"
            xin = x
            if mode == "bf16_channels_last":
                net = net.to(memory_format=torch.channels_last)
                xin = x.contiguous(memory_format=torch.channels_last)

            def step():
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=(mode == "bf16_channels_last")):
                    return net(xin)
            for _ in range(15):
                o = step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(60):
                o = step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 60
            f = o[-1].float().cpu()
            out[mode] = {"fps": 1000.0 / ms, "ms": ms,
                         "fused_max_rel_vs_cpu_fp32": float((f - cpu).abs().max() / cpu.abs().max()),
                         "mask_flips_vs_cpu_fp32": int(((f > 0) != (cpu > 0)).sum())}
            del net
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = saved
    return out


def conv_traffic(precision, calls):
    """DRAM bytes per conv launch from the committed ncu capture matching this configuration, else None."""
    try:
        with open(os.path.join(ROOT, "profiles", "conv_dram_traffic.json")) as f:
            t = json.load(f)
        e = t.get(f"{precision}_{H}x{W}")
        if e and e.get("launches") == calls:
            return e["dram_bytes_per_step"] / calls, e.get("source")
    except Exception:
        pass
    return None, None


# ----------------------------------------------------------------------------------------------------------------
def run_parent_headline(args, rank, world, local, dev, timer):
    """--workload parent480: the dp object promoted to the headline line."""
    import torch.distributed as dist
    dp = run_dp(args, rank, world, local, dev, timer, max(1, args.steps), args.dump_outputs)
    if rank == 0:
        emit({"metric": "frames/sec at 480x854 fwd+bwd, parent training (5-loss objective, SGD step, DP allreduce)",
              "value": dp["fps"], "unit": "frames/s", "n_gpus": world, "steps": dp["steps"], "warmup": 3,
              "ms_per_step": dp["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
              "dtype": dp["dtype"], "data": "synthetic",
              "config": {"workload": dp["workload"], "parallelism": dp["parallelism"],
                         "l2": "per-step working set (>10 GB) exceeds L2", "timing": "CUDA events over K steps, max over ranks"},
              "allreduce_ms": dp["allreduce_ms"], "allreduce_share": dp["allreduce_share"], "dp": dp,
              "gpu_launches": dp["gpu_launches"], "clocks": dp["clocks"]})
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="infer480", choices=["infer480", "train480", "parent480"])
    ap.add_argument("--batch", type=int, default=12, help="parent480 / dp: frames per GPU per optimizer step")
    ap.add_argument("--precision", default="exact", choices=["exact", "fast"])
    ap.add_argument("--dp-steps", type=int, default=10, help="timed optimizer steps of the dp leg")
    ap.add_argument("--dp-lr", type=float, default=1e-10, help="learning rate of the dp leg (see run_dp)")
    ap.add_argument("--skip", default="", help="comma list of legs to skip: dp,parity,gpu_reference,cpu_baseline,roofline,e2e_extra")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager-train", action="store_true", help="train480: eager launches instead of the step graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned in its last step to "
                                                          "DIR/<name>.npy (float32)")
    args = ap.parse_args()
    skip = {s for s in args.skip.split(",") if s}
    if args.no_cpu_baseline:
        skip.add("cpu_baseline")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from oracle import osvos_oracle as oc           # checker legs + synthetic input generator only
    from osvos_pytorch_b200 import ops
    from osvos_pytorch_b200.layers.osvos_layers import class_balanced_cross_entropy_loss
    from osvos_pytorch_b200.networks.vgg_osvos import OSVOS, he_init_

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node == --gpus"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    timer = Timer(dev, world)
    steps, warmup = max(1, args.steps), max(3, args.warmup)
    if args.workload == "parent480":
        return run_parent_headline(args, rank, world, local, dev, timer)
    train = args.workload == "train480"

    net = he_init_(OSVOS(pretrained=0, verbose=False, precision=args.precision), seed=0).to(dev)
    net.train(train)
    n_in = 4                                          # rotate input frames (distinct seeds)
    frames = [oc.synthetic_frame(1, H, W, 1234 + i + 100 * rank) for i in range(n_in)]
    xs = [f[0].to(dev) for f in frames]
    gts = [f[1].to(dev) for f in frames]
    xs_host = [f[0].pin_memory() for f in frames]
    out_host = torch.empty((1, 1, H, W), dtype=torch.float32).pin_memory()
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    graphed = {"step": None}
    last = {}                                         # what the latest inference step returned

    def step(i, x=None):
        x = xs[i % n_in] if x is None else x
        if train:
            if args.eager_train:
                net.zero_grad(set_to_none=False)
                outs = net(x)
                loss = class_balanced_cross_entropy_loss(outs[-1], gts[i % n_in], size_average=False)
                loss.backward()
                return loss
            # fwd + online loss + bwd of the micro-batch as one replayed CUDA graph (osvos_pytorch_b200.training)
            sample = {"image": x, "gt": gts[i % n_in]}
            if graphed["step"] is None:
                from osvos_pytorch_b200.training import GraphedTrainStep
                graphed["step"] = GraphedTrainStep(
                    net, lambda outs, gt: class_balanced_cross_entropy_loss(outs[-1], gt, size_average=False), sample)
            return graphed["step"](sample)          # gradients accumulate, as between the reference's optimizer steps
        with torch.no_grad():
            last["outs"] = net(x)
        return last["outs"][-1]

    # kernels per step, counted on an eager pass (the timed inference steps replay a captured CUDA graph of
    # exactly these launches)
    graphs_on = net._engine.use_cuda_graph
    net._engine.use_cuda_graph = False
    eager_flag = args.eager_train
    args.eager_train = True                          # count launches on an eager pass
    step(0)
    l0 = ops.KERNEL_LAUNCHES[0]
    step(1)
    launches = ops.KERNEL_LAUNCHES[0] - l0
    args.eager_train = eager_flag
    net._engine.use_cuda_graph = graphs_on
    for i in range(warmup):
        step(i)
    # W steps are ~16 ms of work: not enough for the clocks / power state of an idle box to settle; keep stepping,
    # untimed, for half a second before the timed region.
    t_settle, i = time.perf_counter(), warmup
    while time.perf_counter() - t_settle < 0.5:
        for _ in range(20):
            step(i)
            i += 1
        torch.cuda.synchronize()
    # ---- device-resident throughput -------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, timed_info = timer.steps(step, steps)
    clocks = sampler.stop() if rank == 0 else None
    dump = None
    if args.dump_outputs is not None and rank == 0:
        if train:
            # the timed steps accumulate gradients: clear them and run the last timed step's frame once more
            net.zero_grad(set_to_none=False)
            dump = {"loss": step(steps - 1)}
            dump.update(("grad." + n, p.grad) for n, p in net.named_parameters() if p.grad is not None)
        else:
            dump = {f"out{k}": o for k, o in enumerate(last["outs"])}
        dump = {k: v.detach().cpu() for k, v in dump.items()}

    # ---- end to end: pinned host frame -> H2D -> OSVOS.forward -> D2H of the result ---
    def e2e_step(i):
        x = xs_host[i % n_in].to(dev, non_blocking=True)
        r = step(i, x)
        if train:
            loss_host.copy_(r.detach(), non_blocking=True)
        else:
            out_host.copy_(r, non_blocking=True)
    e2e_extra = {}
    if train:
        for i in range(3):
            e2e_step(i)
        ms_e2e, e2e_timed = timer.steps(e2e_step, steps)
    else:
        # the test-time loop of the reference (train_online.py:172-187) through the package's sequence pipeline:
        # every frame is copied H2D from pinned memory, run through OSVOS.forward, and its result copied D2H -
        # the three legs of consecutive frames overlap on separate streams (osvos_pytorch_b200/inference.py)
        from osvos_pytorch_b200.inference import SequenceSegmenter

        def sequence_timed(seg, k):
            for _ in seg(xs_host[i % n_in] for i in range(6)):      # warm-up, allocates the ring
                pass

            def run_all(_i):                                          # one timed "step" = the whole k-frame sequence
                for _ in seg(xs_host[j % n_in] for j in range(k)):
                    pass
            per_seq, info = timer.steps(run_all, 1, after=seg.join_current_stream)
            return per_seq / k, dict(info, timed_steps=k)
        ms_e2e, e2e_timed = sequence_timed(SequenceSegmenter(net, output="logits"), steps)
        if "e2e_extra" not in skip:
            for i in range(3):
                e2e_step(i)
            ms_serial, _ = timer.steps(e2e_step, steps)
            ms_png, _ = sequence_timed(SequenceSegmenter(net, output="bytescale"), steps)
            e2e_extra = {"serial_single_stream": {"value": world * 1000.0 / ms_serial, "ms_per_step": ms_serial},
                         "u8_png_payload": {"value": world * 1000.0 / ms_png, "ms_per_step": ms_png,
                                            "d2h_bytes_per_step": H * W,
                                            "note": "sigmoid + imsave bytescale on the device (ops.logits_to_u8)"}}

    # ---- roofline of the dominant kernel class (tcgen05 convs) ----------------------------------------------------
    # In forward_inference every kernel between the first conv and the tail IS a tcgen05 conv (stage-1 kernel, trunk, side
    # convs; the fold / pack kernels only run on the first pass), so ONE event pair - recorded just before the first conv
    # launch and just before the tail launch - brackets exactly the conv kernels of a pass, back to back, without the
    # per-launch event pairs that used to cost the stream a few us each (their sum exceeded the whole graphed step).
    conv_rec, eager_ms, parked = [], 0.0, True
    conv_spans = []
    reps = 0
    if rank == 0 and not train and "roofline" not in skip:
        rec = []
        span = {"a": None}
        origs = {n: getattr(ops, n) for n in ("conv3x3", "stage1_fused", "side_folded", "side_folded_multi", "conv_first",
                                              "tail_fwd")}

        def mark_first():
            if span["a"] is None:
                span["a"] = torch.cuda.Event(enable_timing=True)
                span["a"].record()

        def w_conv3x3(x, w_packed, bias, cout, *a, **k):
            mark_first()
            n_, hh, ww, ci = x.shape
            rec.append((2.0 * n_ * hh * ww * cout * 9 * ci, "side_conv_kernel" if cout == 16 else "conv3x3_halo_kernel"))
            return origs["conv3x3"](x, w_packed, bias, cout, *a, **k)

        def w_stage1(x, *a, **k):                 # conv1_1 + conv1_2 in one kernel: both layers' flops
            mark_first()
            n_, _, hh, ww = x.shape
            rec.append((2.0 * n_ * hh * ww * 64 * 9 * (3 + 64), "conv_stage1_fused_kernel"))
            return origs["stage1_fused"](x, *a, **k)

        def w_side(x, *a, **k):                   # algorithmic flops of the reference's side_prep (C -> 16), run folded (C -> 2)
            mark_first()
            n_, hh, ww, ci = x.shape
            rec.append((2.0 * n_ * hh * ww * 16 * 9 * ci, "side_conv_kernel"))
            return origs["side_folded"](x, *a, **k)

        def w_side_multi(xs, *a, **k):            # the four scales' folded side convs in one launch: all their flops
            mark_first()
            rec.append((sum(2.0 * x.shape[0] * x.shape[1] * x.shape[2] * 16 * 9 * x.shape[3] for x in xs),
                        f"side_conv_kernel ({len(xs)} scales in one launch)"))
            return origs["side_folded_multi"](xs, *a, **k)

        def w_first(x, *a, **k):                  # separate conv1_1 (training / fast mode): inside the span, flops counted
            mark_first()
            n_, _, hh, ww = x.shape
            rec.append((2.0 * n_ * hh * ww * 64 * 27, "conv_first_tc_kernel"))
            return origs["conv_first"](x, *a, **k)

        def w_tail(*a, **k):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            conv_spans.append((span["a"], e))
            span["a"] = None
            return origs["tail_fwd"](*a, **k)
        ops.conv3x3, ops.stage1_fused, ops.side_folded, ops.conv_first, ops.tail_fwd = w_conv3x3, w_stage1, w_side, w_first, w_tail
        ops.side_folded_multi = w_side_multi
        net._engine.use_cuda_graph = False          # the span events need the eager path
        reps = min(steps, 10)
        for i in range(3):                          # eager warm-up passes, not counted
            step(i)

        def instrumented(park_gpu):
            """`reps` eager passes.  An eager launch costs the host ~40 us (ctypes + tensor-map encodes), more than the short
            kernels take, so with the GPU idle the span would time the HOST.  park_gpu: a ~40 ms spin kernel is enqueued
            first and every launch of the passes queues up behind it; the GPU then runs them back to back."""
            torch.cuda.synchronize()
            rec.clear()
            conv_spans.clear()
            span["a"] = None
            if park_gpu:
                torch.cuda._sleep(int(0.04 * 1.9e9))
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record()
            for i in range(reps):
                step(i)
            p1.record()
            torch.cuda.synchronize()
            return p0.elapsed_time(p1) / reps       # the instrumented (eager) step
        try:
            eager_ms = instrumented(True)
        except Exception:                            # torch.cuda._sleep is a private helper: fall back to plain eager
            parked = False
            eager_ms = instrumented(False)
        for n, f in origs.items():
            setattr(ops, n, f)
        net._engine.use_cuda_graph = graphs_on
        conv_rec = list(rec)
        conv_span_ms = sum(a.elapsed_time(b) for a, b in conv_spans) / max(1, len(conv_spans))

    # ---- the north-star multi-GPU path (every N, 1 included) ------------------------------------------------------
    dp = None
    if not train and "dp" not in skip:
        dp = run_dp(args, rank, world, local, dev, timer, max(2, args.dp_steps))

    if world > 1:
        timer.barrier()
        dist.destroy_process_group()                 # everything below is rank-0-only work without collectives
    if rank != 0:
        return

    peaks = load_peaks()
    fps = world * 1000.0 / ms
    line = {
        "metric": METRIC if not train else METRIC.replace("fwd-only", "fwd+bwd (online objective)"),
        "value": fps, "unit": "frames/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16x3 (split-bf16 operands, fp32 accumulate)" if args.precision == "exact" else "bf16",
        "data": "synthetic",
        "config": {"workload": workload_label(args.workload), "precision": args.precision,
                   "parallelism": f"replicas x{world} for this headline (inference has no collective); the data-parallel "
                                  f"parent-training path is the `dp` object of this line",
                   "l2": "per-step activation traffic (~0.9 GB exact) exceeds the 126 MB L2; inputs rotate over 4 frames; no explicit flush",
                   "timing": "CUDA events on the launching stream, max over ranks; W warm-up steps + 0.5 s of untimed steps, "
                             "then exactly K timed steps (barrier + synchronize on both sides)",
                   "launch": ("captured CUDA graph of the step's kernels, replayed per step"
                              if ((graphs_on and not train) or (train and not args.eager_train)) else "eager launches")},
        "timed": timed_info,
        "e2e": {"value": world * 1000.0 / ms_e2e, "unit": "frames/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": 3 * H * W * 4, "d2h_bytes_per_step": (4 if train else H * W * 4),
                "timed": e2e_timed,
                "path": ("pinned host frame -> .to(cuda) -> fwd+loss+bwd -> D2H of the loss" if train else
                         "SequenceSegmenter: pinned host frame -> H2D -> OSVOS.forward (nn.Module API) -> D2H of the "
                         "fused logit map, legs of consecutive frames overlapped on 3 streams; the pipeline reads the fused "
                         "map out of the replayed graph's static output, so per frame it does ONE 1.6 MB device copy where the "
                         "device-resident `value` loop (net(x): five fresh maps) does one of 8.2 MB - with the PCIe legs "
                         "fully overlapped it can therefore come out level with or a fraction above `value`"), **e2e_extra},
        "gpu_launches": int(launches),
        "memcpy_per_step": (0 if train else 1),
        "gpu_launches_note": ("this repo's kernels per step (libosvos_b200.so), all inside one replayed CUDA graph; around the "
                              "replay the engine issues `memcpy_per_step` device-to-device copy through torch (the five maps out "
                              "into fresh caller-owned tensors; an input buffer that comes back is read in place by a graph "
                              "captured on it, so no input copy in steady state) - not counted as kernels"),
        "clocks": clocks,
    }
    if conv_rec:
        per = len(conv_rec) // reps
        conv_ms = conv_span_ms
        conv_flops = sum(f for f, _ in conv_rec) / reps
        kinds = {}
        for _, k in conv_rec:
            kinds[k] = kinds.get(k, 0) + 1
        kinds = {k: v // reps for k, v in kinds.items()}
        passes = 3 if args.precision == "exact" else 1
        ach = conv_flops / (conv_ms * 1e-3) / 1e12
        # upper bound from the headline itself: all conv flops over the WHOLE graphed step (as if nothing else ran in it)
        ach_floor_step = conv_flops / (ms * 1e-3) / 1e12
        traffic, tsrc = conv_traffic(args.precision, per)
        line["roofline"] = {
            "bound": "tensor",
            "kernel": "the step's tcgen05 implicit-GEMM 3x3 convolutions: " + " + ".join(f"{k} x{v}" for k, v in kinds.items())
                      + f" = {per} launches per step (every kernel of the step between the frame and the tail)",
            "achieved": ach, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s", "frac": ach / peaks["tflops_sustained"],
            "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernels timed inside the step)",
            "algorithmic_flops_per_step": conv_flops, "launches_per_step": per, "kernel_ms_per_step": conv_ms,
            "how": "ONE CUDA-event pair per pass spanning the conv launches (first conv launch -> tail launch), eager launches "
                   + ("queued behind a parked GPU (back-to-back kernel time)" if parked else "(host launch gaps included)"),
            "share_of_step": conv_ms / eager_ms, "instrumented_step_ms": eager_ms,
            "conv_flops_over_whole_graphed_step": {"achieved": ach_floor_step, "frac": ach_floor_step / peaks["tflops_sustained"],
                                                    "note": "all conv flops / the headline ms_per_step (tail and copies included)"},
            "tensor_pipe_passes": passes,
            # exact mode emulates fp32 operands with three bf16 passes (hi*hi + hi*lo + lo*hi): the tensor pipe EXECUTES
            # passes x the algorithmic flops; this is that figure over the peak
            "issued_mma_frac": ach * passes / peaks["tflops_sustained"],
            "traffic": traffic, "traffic_unit": "dram bytes per launch (average over the step's conv launches)",
            "traffic_source": tsrc}
    if dp is not None:
        line["dp"] = dp
    if not train and "parity" not in skip:
        line["parity"] = forward_parity(net, dev)
    if not train and "gpu_reference" not in skip:
        try:
            line["gpu_reference"] = gpu_reference(dev)
        except Exception as e:                       # a cuDNN hiccup must not cost the whole bench line
            line["gpu_reference"] = {"unavailable": f"{type(e).__name__}: {e}"}
    if "cpu_baseline" not in skip and world == 1:
        cfps, cms, cores, threads, kind = cpu_reference_fps(3, 1, args.workload)
        line["cpu_baseline"] = {"value": cfps, "unit": "frames/s", "cores": threads, "kind": kind,
                                "sample": f"3 steps of the same 480x854 frame after 1 warm-up; "
                                          f"{'unmodified reference modules (oracle/_ref)' if kind == 'reference' else 'oracle port'}"
                                          f" = the reference's torch CPU fp32 path on {threads} threads ({cores} host cores)"}
    if dump is not None:
        dump_outputs(args.dump_outputs, dump)
    emit(line)


if __name__ == "__main__":
    main()
