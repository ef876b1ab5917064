#!/usr/bin/env python
"""Benchmark of the distributed sigmoid (SigLIP) loss hot path (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 5                 # this repo's sm_100a path
    torchrun --nproc-per-node N ... bench.py --gpus N ...          # one rank per GPU (driver launches this)
    python bench.py --impl reference --gpus 1 --steps 20 --warmup 5  # the UNMODIFIED reference on the host cores
    python bench.py --batch 4096 --dim 768                         # another BASELINE.json config (configs[1])
    python bench.py --dump-outputs DIR                             # also write the last timed step's outputs (.npy)

Workload (BASELINE.json `metric`): per-rank batch B=16384, D=1024, bf16, W = --gpus text chunks per rank,
synthetic L2-normalised features (seed 1234 + rank), t' = log 10, b = -10. One "step" = one forward + backward of the
loss module (loss + dimg + dtxt + dt' + dbias). Prints ONE JSON line on rank 0.

Before anything is timed, every rank runs a PARITY pass on the real process group (B=2048, D=768): fused C-ABI call and
module surface against fp32 torch autograd of the reference's op sequence (distributed_sigmoid_loss.py:22-47) on the
same inputs, the text gradient all-reduced over the ranks; the max relative errors over all ranks are printed as
`parity` in the JSON line.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "image-text pairs/sec"
UNIT = "pairs/s"
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            p = json.load(f)
        return float(p["bf16_tflops_sustained"]), "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)"
    except Exception:
        return 1400.0, "B200_PROFILING.md fallback, sustained ~1.4 PFLOP/s (of fallback)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md) through NVML from a Python
    thread every ~5 ms (the C calls release the GIL)."""

    def __init__(self, gpu_index: int, period_s: float = 0.005):
        self.gpu_index = gpu_index
        self.period_s = period_s
        self.samples = []      # (sm_mhz, reasons_bitmask)
        self.max_mhz = None
        self._stop = threading.Event()
        self.thread = None
        self.nv = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                reasons = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((mhz, reasons))
            except Exception:
                pass
            time.sleep(self.period_s)

    def mark(self):
        """Index of the next sample: call at the start of the timed region."""
        return len(self.samples)

    def median_since(self, first: int):
        sel = sorted(s[0] for s in self.samples[first:])
        return sel[len(sel) // 2] if sel else None

    def stop(self, first: int = 0, last: int = None):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"], "samples": 0}
        self._stop.set()
        self.thread.join(timeout=1)
        sel = self.samples[first:last] or self.samples
        clocks = sorted(s[0] for s in sel)
        mask = 0
        for _, r in sel:
            mask |= r
        names = {"gpu_idle": 0x1, "applications_clocks_setting": 0x2, "sw_power_cap": 0x4, "hw_slowdown": 0x8,
                 "sync_boost": 0x10, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake_slowdown": 0x80, "display_clock_setting": 0x100}
        reasons = sorted(k for k, bit in names.items() if (mask & bit) and k != "gpu_idle")
        return {"sm_mhz": clocks[len(clocks) // 2] if clocks else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "reasons_mask": hex(mask), "samples": len(sel),
                "note": "sustained state by construction (warm-up until the step time is stable): a power-capped B200 "
                        "runs tensor work at 1.2-1.4 GHz; sw_power_cap is the expected reason"}


def _nvlink_counters(gpu_index: int):
    """Cumulative NVLink payload counters of one GPU in bytes (rx, tx), summed over its links, from NVML field values
    (NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX/TX, KiB units). None if the driver does not expose them."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        out = []
        for fid in (pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX, pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX):
            total, ok = 0, False
            try:       # scope UINT_MAX = all links
                v = pynvml.nvmlDeviceGetFieldValues(h, [(fid, 0xFFFFFFFF)])[0]
                if v.nvmlReturn == 0:
                    total, ok = int(v.value.ullVal), True
            except Exception:  # noqa: BLE001
                ok = False
            if not ok:
                for link in range(18):
                    try:
                        v = pynvml.nvmlDeviceGetFieldValues(h, [(fid, link)])[0]
                        if v.nvmlReturn == 0:
                            total += int(v.value.ullVal)
                            ok = True
                    except Exception:  # noqa: BLE001
                        break
            if not ok:
                return None
            out.append(total * 1024)
        return tuple(out)
    except Exception:  # noqa: BLE001
        return None


def _bind_to_gpu_numa_node(gpu_index: int):
    """Pin this process to the CPUs NVML reports as local to the GPU, so that pinned host memory is allocated on the
    GPU's NUMA node (host->device copies of the e2e path cross no socket link). Best effort."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return sorted(os.sched_getaffinity(0))[:1] + [len(os.sched_getaffinity(0))]
    except Exception:
        return None


def synth(rank: int, B: int, D: int):
    import torch

    g = torch.Generator().manual_seed(1234 + rank)
    img = torch.nn.functional.normalize(torch.randn(B, D, generator=g))
    txt = torch.nn.functional.normalize(torch.randn(B, D, generator=g))
    return img.to(torch.bfloat16), txt.to(torch.bfloat16)


DUMP_NAMES = ("loss", "dimg", "dtxt", "dt_prime", "dbias")
DUMP_GRAD_ELEMENTS = 7 << 20       # per gradient: two float32 samples of 28 MiB keep a dump under 64 MB


def dump_outputs(out_dir: str, outputs):
    """Writes one step's (loss, dimg, dtxt, dt', dbias) as <out_dir>/<name>.npy: float64 where the step returned
    float64, float32 otherwise. Gradients of more than DUMP_GRAD_ELEMENTS elements are cut to a fixed, seeded sample of
    rows (the same rows for both); grad_rows.npy lists the row indices."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    arrays = dict(zip(DUMP_NAMES, outputs))
    B, D = arrays["dimg"].shape
    rows = torch.arange(B)
    if B * D > DUMP_GRAD_ELEMENTS:
        rows = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:DUMP_GRAD_ELEMENTS // D].sort().values
    for name in ("dimg", "dtxt"):
        arrays[name] = arrays[name][rows.to(arrays[name].device)]
    arrays["grad_rows"] = rows
    for name, t in arrays.items():
        wide = t.dtype in (torch.float64, torch.int64)
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().to(torch.float64 if wide else torch.float32).numpy())


# ------------------------------------------------------------------------------------------------------
# Reference arm: the UNMODIFIED reference (baseline/_ref, placed by tools/fetch_ref.py) on the host cores
# ------------------------------------------------------------------------------------------------------
def _load_reference_module():
    """(DDPSigmoidLoss class of the unmodified reference, "reference") or (None, "port") when baseline/_ref is absent."""
    if os.path.exists(os.path.join(REF_DIR, "distributed_sigmoid_loss.py")):
        if REF_DIR not in sys.path:
            sys.path.insert(0, REF_DIR)
        import distributed_sigmoid_loss as ref_mod   # noqa: E402  (the reference's own file, byte-identical copy)

        return ref_mod.DDPSigmoidLoss, "reference"
    return None, "port"


def cpu_reference_times(B: int, D: int, steps: int, warmup: int):
    """Times `DDPSigmoidLoss(B).forward(img, txt)` + `.backward()` of the unmodified reference
    (distributed_sigmoid_loss.py:17-48) under a world_size-1 gloo group, fp32 on the bf16-rounded bench inputs, all
    host threads, FULL per-rank chunk (B x B logits). Falls back to the oracle's op-for-op port (kind "port") only if
    baseline/_ref is missing. Returns (seconds per step, threads, kind)."""
    import torch
    import torch.distributed as dist

    cls, kind = _load_reference_module()
    threads = torch.get_num_threads()
    img_b, txt_b = synth(0, B, D)
    img = img_b.float().requires_grad_(True)
    txt = txt_b.float().requires_grad_(True)
    times = []
    if cls is not None:
        if not dist.is_initialized():
            dist.init_process_group("gloo", store=dist.HashStore(), rank=0, world_size=1)
        mod = cls(B)
        params = [mod.t_prime, mod.bias]

        def step():
            for p in [img, txt] + params:
                p.grad = None
            loss = mod(img, txt)
            loss.backward()
            return float(loss.detach())
    else:
        from oracle.siglip_oracle import port_step

        tp = torch.tensor(math.log(10.0), dtype=torch.float64, requires_grad=True)
        bb = torch.tensor(-10.0, requires_grad=True)

        def step():
            for p in (img, txt, tp, bb):
                p.grad = None
            return float(port_step(img, [txt], tp, bb, 0).detach())
    loss = None
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        loss = step()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    if cls is not None and dist.is_initialized():
        dist.destroy_process_group()
    return sum(times) / len(times), threads, kind, loss


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    if "LOCAL_RANK" in os.environ:
        # under torchrun: the launcher exports OMP_NUM_THREADS=1 for its workers; the CPU arm is meant to use every
        # host thread, so rank 0 re-runs itself in a clean environment and relays the line
        env = {k: v for k, v in os.environ.items()
               if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "OMP_NUM_THREADS", "MASTER_ADDR", "MASTER_PORT",
                            "GROUP_RANK", "ROLE_RANK", "LOCAL_WORLD_SIZE", "ROLE_WORLD_SIZE", "GROUP_WORLD_SIZE",
                            "TORCHELASTIC_RUN_ID", "TORCHELASTIC_RESTART_COUNT", "TORCHELASTIC_MAX_RESTARTS")}
        out = subprocess.run([sys.executable, os.path.abspath(__file__)] + sys.argv[1:], env=env, capture_output=True,
                             text=True)
        sys.stderr.write(out.stderr[-2000:])
        sys.stdout.write(out.stdout)
        sys.stdout.flush()
        return out.returncode
    try:     # a parent bench process may have pinned itself to the GPU's NUMA node: the CPU arm uses every host core
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
    except OSError:
        pass
    B, D, W = args.batch, args.dim, args.gpus
    sec, threads, kind, loss = cpu_reference_times(B, D, max(1, args.steps), max(0, args.warmup))
    # One timed step = the reference's forward+backward over ONE full (B x B) chunk: exactly the whole job at N=1.
    # At N>1 the job is W ranks x W chunks of that unit on this one host (W x 8 GiB of B x B intermediates per rank do
    # not fit and per-chunk cost is linear in W, BASELINE.md §4): whole-job rate = W*B / (W*W * t_chunk), extrapolated.
    value = W * B / (W * W * sec)
    what = ("unmodified reference DDPSigmoidLoss.forward + .backward() (baseline/_ref/distributed_sigmoid_loss.py:8-48, "
            "world_size-1 gloo group)" if kind == "reference" else
            "oracle.port_step, the reference's op sequence (baseline/_ref missing: run tools/fetch_ref.py)")
    sample = (f"{what}; fp32 on the bf16-rounded bench inputs; every timed step scores the FULL {B} x {B} chunk of rank 0 "
              f"(D={D}): {sec:.3f} s per step on {threads} host threads")
    if W > 1:
        sample += (f"; N={W}: whole job = {W} ranks x {W} chunks of that unit on this host, rate extrapolated as "
                   f"W*B / (W^2 * t_chunk) (the measured per-step time is `ms_per_step`, the extrapolated full-job step is "
                   f"`extrapolated_job_step_ms`)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"SigLIP loss fwd+bwd, B={B}/rank D={D} W={W} chunks, reference implementation on CPU",
                   "global_batch": B * W, "batch_per_rank": B, "dim": D, "world": W},
        "loss": loss,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if W > 1:
        line["extrapolated_job_step_ms"] = W * W * sec * 1e3
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------------
# parity pass (before the timed region, on the real process group)
# ------------------------------------------------------------------------------------------------------
def _fp32_autograd(img, chunks, tp, bias, rank):
    """fp32 torch autograd of the reference's op sequence (distributed_sigmoid_loss.py:22-47) on the GPU: GEMM, scale,
    bias, labels (2*eye-1 on the own chunk, -1 elsewhere), logsigmoid, sum, / local batch. Returns loss, dimg, this
    rank's contribution to every chunk's text gradient, dt', dbias."""
    import torch

    dev = img.device
    a = img.detach().float().requires_grad_(True)
    cs = [c.detach().float().requires_grad_(True) for c in chunks]
    t = torch.tensor(float(tp), device=dev, requires_grad=True)
    b = torch.tensor(float(bias), device=dev, requires_grad=True)
    n = a.shape[0]
    total = torch.zeros((), device=dev)
    for c, txt in enumerate(cs):
        logits = a @ txt.T * t.exp() + b
        labels = (2 * torch.eye(n, device=dev) - 1) if c == rank else -torch.ones(n, device=dev)
        total = total + (-torch.nn.functional.logsigmoid(labels * logits)).sum()
    total = total / n
    total.backward()
    return float(total.detach()), a.grad, [c.grad for c in cs], float(t.grad), float(b.grad)


def parity_pass(rank, world, dev, cta_group, B=2048, D=768):
    import torch
    import torch.distributed as dist

    from distributed_sigmoid_loss_b200 import DDPSigmoidLoss

    tp, bias = math.log(10.0), -10.0
    img_h, txt_h = synth(100 + rank, B, D)
    img, txt = img_h.to(dev), txt_h.to(dev)
    chunks = [txt]
    if world > 1:
        chunks = [torch.empty_like(txt) for _ in range(world)]
        dist.all_gather(chunks, txt)
    r_loss, r_dimg, r_contrib, r_dtp, r_db = _fp32_autograd(img, chunks, tp, bias, rank)
    contrib = torch.stack(r_contrib)
    if world > 1:
        dist.all_reduce(contrib)             # text gradient = sum over the ranks' losses (all_gather's backward)
    r_dtxt = contrib[rank]

    def rel(a, b):
        return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))

    def srel(a, b):
        return abs(float(a) - b) / (abs(b) + 1e-300)

    mod = DDPSigmoidLoss(B, cta_group=cta_group).to(dev)
    eng = mod.engine_for(B, D, dev)
    tpt, bt = torch.tensor([tp], device=dev), torch.tensor([bias], device=dev)
    errs = {}
    for rep in range(2):                     # the second repetition exercises the step-to-step flag protocol
        loss, dimg, dtxt, dtp, db = eng.fwd_bwd(img, txt, tpt, bt)
        torch.cuda.synchronize()
        e = dict(loss=srel(loss, r_loss), dimg=rel(dimg, r_dimg), dtxt=rel(dtxt, r_dtxt), dt_prime=srel(dtp, r_dtp),
                 dbias=srel(db, r_db))
        for k, v in e.items():
            errs[k] = max(errs.get(k, 0.0), v)
    a, b = img.clone().requires_grad_(True), txt.clone().requires_grad_(True)
    lm = mod(a, b)
    lm.backward()
    torch.cuda.synchronize()
    merrs = dict(loss=srel(lm.detach(), r_loss), dimg=rel(a.grad.float(), r_dimg), dtxt=rel(b.grad.float(), r_dtxt),
                 dt_prime=srel(mod.t_prime.grad, r_dtp), dbias=srel(mod.bias.grad, r_db))
    # the module returns bf16 gradients for bf16 inputs (like autograd): they must be the round-to-nearest of the
    # fp32 gradients of the split path, i.e. only the 2^-9 rounding of the RESULT separates the two rows below
    keys = sorted(errs)
    t = torch.tensor([errs[k] for k in keys] + [merrs[k] for k in keys], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    vals = [float(x) for x in t]
    fused = dict(zip(keys, vals[:len(keys)]))
    module = dict(zip(keys, vals[len(keys):]))
    ok = all(v <= 1e-3 for v in fused.values()) and all(module[k] <= 1e-3 for k in ("loss", "dt_prime", "dbias")) \
        and module["dimg"] <= 4e-3 and module["dtxt"] <= 4e-3
    del mod, eng
    torch.cuda.empty_cache()
    return {"shape": [B, D], "world": world, "ranks_checked": world,
            "reference": "fp32 torch autograd of distributed_sigmoid_loss.py:22-47 on the same bf16 inputs; text gradient "
                         "all-reduced (SUM) over the real process group",
            "fused_fp32": fused, "module_bf16_grads": module, "tol": 1e-3,
            "tol_note": "fused_fp32 (C ABI, fp32 gradients): 1e-3 relative / relative-Frobenius; module rows: loss/dt'/db 1e-3, "
                        "dimg/dtxt are returned in bf16 like autograd (2^-9 rounding of the result): 4e-3",
            "max_over_ranks": True, "pass": bool(ok)}


# ------------------------------------------------------------------------------------------------------
# this repo's path
# ------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from distributed_sigmoid_loss_b200 import DDPSigmoidLoss, _capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = _bind_to_gpu_numa_node(local_rank)   # pinned host buffers next to the GPU's PCIe root (matters for e2e)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, D, W = args.batch, args.dim, world

    def allgather_floats(xs):
        t = torch.tensor(xs, device=dev, dtype=torch.float64)
        if world == 1:
            return [[float(v) for v in t]]
        out = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [[float(v) for v in o] for o in out]

    parity = None
    if not args.no_parity:
        parity = parity_pass(rank, world, dev, args.cta_group)

    img_h, txt_h = synth(rank, B, D)
    img = img_h.to(dev).requires_grad_(True)
    txt = txt_h.to(dev).requires_grad_(True)
    fused_step = {"auto": None, "fused": True, "split": False}[args.schedule]
    mod = DDPSigmoidLoss(B, cta_group=args.cta_group, fused_step=fused_step).to(dev)
    eng = mod.engine_for(B, D, dev)
    tpt = torch.tensor([math.log(10.0)], device=dev)
    bt = torch.tensor([-10.0], device=dev)
    img_d, txt_d = img.detach(), txt.detach()

    # every variant of a step returns what its caller receives: (loss, dimg, dtxt, dt', dbias)
    if args.api == "module":
        def step():
            img.grad = None
            txt.grad = None
            mod.t_prime.grad = None
            mod.bias.grad = None
            loss = mod(img, txt)
            loss.backward()
            return loss, img.grad, txt.grad, mod.t_prime.grad, mod.bias.grad
    elif args.api == "fused":   # the fused C-ABI entry siglip_fwd_bwd (BASELINE.json configs[1] "fused fwd+bwd"), bf16 gradients
        def step():
            return eng.fwd_bwd(img_d, txt_d, tpt, bt, torch.bfloat16)
    else:   # the same fused C-ABI step captured once into a CUDA graph and replayed (single rank only: the cross-rank
            # flag values of a multi-rank step are kernel parameters that advance every step)
        if world > 1:
            raise SystemExit("--api graph is a single-GPU measurement")
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            eng.fwd_bwd(img_d, txt_d, tpt, bt, torch.bfloat16)
            n_before = eng.launch_count
            with torch.cuda.graph(graph, stream=side):
                graph_out = eng.fwd_bwd(img_d, txt_d, tpt, bt, torch.bfloat16)
            graph_launches = eng.launch_count - n_before      # kernel nodes of the graph (2: loss + gradient kernel)
        torch.cuda.current_stream().wait_stream(side)

        def step():
            graph.replay()
            return graph_out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank, args.clock_period_ms * 1e-3)
    sampler.start()              # every rank samples its own GPU (NVML thread, 5 ms period)
    n_warm = max(args.warmup, 3)
    barrier()
    for _ in range(n_warm):
        step()
    barrier()

    def timed_batch(n):
        """n back-to-back steps; device time, max over ranks (identical on every rank: the loop below is collective)."""
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            step()
        b.record()
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # Sustained power state at every N. A B200 under tensor load drops from its burst clocks to the power-capped state
    # after ~50-100 ms (1.16 -> 1.33 ms per step at the headline shape; MEASURED_PEAKS.json: cuBLAS 1701.7 burst vs
    # 1432 sustained). The first steps after the requested warm-up are reported as "burst"; the warm-up then continues
    # in ~25 ms batches until (a) at least --sustain-ms of GPU time have passed AND (b) the step time of three
    # consecutive batches agrees within 1.5 % (the clocks have settled), at most 4 s.
    burst_ms = timed_batch(args.steps) / args.steps
    n_warm += args.steps
    warm_ms = burst_ms * args.steps
    hist = []
    nb = max(2, min(256, int(math.ceil(25.0 / max(burst_ms, 1e-3)))))
    while n_warm < 200000:
        t = timed_batch(nb)
        warm_ms += t
        n_warm += nb
        hist.append(t / nb)
        stable = len(hist) >= 3 and max(hist[-3:]) <= 1.015 * min(hist[-3:])
        if (warm_ms >= args.sustain_ms and stable) or warm_ms >= max(4000.0, args.sustain_ms):
            break
    barrier()
    launches0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # NVML queries take milliseconds: read the NVLink counters OUTSIDE the barrier-bracketed timed region (a late rank 0
    # would make every peer wait for its flags inside their kernels)
    nvl0 = _nvlink_counters(local_rank) if (rank == 0 and world > 1) else None
    barrier()
    first_sample = sampler.mark()
    e0.record()
    for _ in range(args.steps - 1):
        step()                  # outputs held until the next step returns would double its buffers (a cudaMalloc)
    outputs = step()
    e1.record()
    barrier()
    last_sample = sampler.mark()
    loss = outputs[0]
    # copies: later replays of the graph overwrite its output buffers
    dumped = [t.detach().clone() for t in outputs] if (args.dump_outputs and rank == 0) else None
    del outputs
    nvl1 = _nvlink_counters(local_rank) if (rank == 0 and world > 1) else None
    my_clock = sampler.median_since(first_sample)
    ms_mine = e0.elapsed_time(e1)
    ms_total = ms_mine
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t)
    ms_step = ms_total / args.steps
    launches = eng.launch_count - launches0
    if args.api == "graph":
        launches = graph_launches * args.steps                # replays launch the captured kernel nodes
    value = W * B / (ms_step * 1e-3)
    # Second timed region, right behind the first, same K steps: every loss / gradient launch bracketed by CUDA events on
    # the launch stream (the per-kernel durations of the roofline). Kept apart from the value above because an event
    # between two launches disables their programmatic dependent launch (set-up overlapping the previous tail).
    eng.set_option(_capi.SIGLIP_OPT_KERNEL_TIMING, 1)
    barrier()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for _ in range(args.steps):
        if args.api == "graph":       # events cannot sit inside a replay: the per-kernel times come from eager fused steps
            eng.fwd_bwd(img_d, txt_d, tpt, bt, torch.bfloat16)
        else:
            step()
    k1.record()
    barrier()
    ms_step_events = k0.elapsed_time(k1) / args.steps
    loss_ms, loss_n, grad_ms, grad_n = eng.kernel_times()
    eng.set_option(_capi.SIGLIP_OPT_KERNEL_TIMING, 0)
    per_rank = allgather_floats([ms_mine / args.steps, loss_ms / max(loss_n, 1), grad_ms / max(grad_n, 1),
                                 (loss_ms + grad_ms) / args.steps, my_clock if my_clock is not None else -1.0])

    # ---- N > 1: every GPU's OWN single-chunk step, all GPUs busy at the same time, no cross-rank dependency ------
    # (one-rank subgroups through the same public module): the spread between the GPUs of the box under identical load.
    # The coupled job cannot run faster than its slowest GPU, whatever the exchange costs.
    single = None
    if world > 1 and not args.no_scaling_diag:
        own_group = None
        for r in range(world):
            g = dist.new_group([r])
            if r == rank:
                own_group = g
        mod1 = DDPSigmoidLoss(B, group=own_group, cta_group=args.cta_group).to(dev)

        def step1():
            img.grad = None
            txt.grad = None
            mod1.t_prime.grad = None
            mod1.bias.grad = None
            mod1(img, txt).backward()

        def timed1(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                step1()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n
        for _ in range(3):
            step1()
        barrier()
        spent, n1 = 0.0, max(2, int(math.ceil(25.0 / max(burst_ms / W, 1e-3))))
        while spent < min(args.sustain_ms, 600.0):          # same wall time on every rank, nothing collective inside
            spent += timed1(n1) * n1
        barrier()
        t1 = timed1(args.steps * W)
        barrier()
        single = [r[0] for r in allgather_floats([t1])]
        del mod1
        torch.cuda.empty_cache()

    # ---- end to end: host buffers in, results out, through the C-ABI host entries ------------------------------
    # Every step copies ITS inputs host->device and its results device->host; with two staging sets the copies of step
    # n+1 overlap the kernels of step n (siglip_host_submit / siglip_host_wait). Two host input sets alternate.
    # Variant "scalars": loss/dt'/dbias come back, gradients stay on the device (what a training loop consumes there).
    # Variant "grads": the bf16 dimg/dtxt of every step also return to pinned host memory on a second copy stream.
    img_p = [img_h.pin_memory(), img_h.clone().pin_memory()]
    txt_p = [txt_h.pin_memory(), txt_h.clone().pin_memory()]
    gi_p = [torch.empty(B, D, dtype=torch.bfloat16).pin_memory() for _ in range(2)]
    gt_p = [torch.empty(B, D, dtype=torch.bfloat16).pin_memory() for _ in range(2)]
    tp0, b0 = math.log(10.0), -10.0

    def e2e_pipelined(n, grads=False):
        prev, res = None, None
        for i in range(n):
            if grads:
                t = eng.host_submit(img_p[i & 1], txt_p[i & 1], tp0, b0, gi_p[i & 1], gt_p[i & 1])
            else:
                t = eng.host_submit(img_p[i & 1], txt_p[i & 1], tp0, b0)
            if prev is not None:
                res = eng.host_wait(prev)
            prev = t
        return eng.host_wait(prev)

    def e2e_sync(n):
        for i in range(n):
            res = eng.fwd_bwd_host(img_p[i & 1], txt_p[i & 1], tp0, b0)
        return res

    def wall(fn, n, *a):
        barrier()
        t0 = time.perf_counter()
        res = fn(n, *a)
        barrier()
        dt = (time.perf_counter() - t0) / n
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t)
        return dt, res

    # Like `value`, the end-to-end numbers are taken in the SUSTAINED power state: each variant first runs for
    # ~--sustain-ms (a step count derived from the max-over-ranks step time, so every rank runs the same number of
    # collective steps), then K steps are timed back to back. The K steps measured right after a pause (what a 25 ms
    # timing loop would see: the GPU has recovered its boost clocks) are kept as `first_steps_ms_per_step`.
    n_sus = max(3, int(math.ceil(min(args.sustain_ms, 600.0) / max(ms_step, 1e-3))))
    e2e_sync(2)
    e2e_sync_s, _ = wall(e2e_sync, args.steps)
    e2e_pipelined(3)
    e2e_first_s, _ = wall(e2e_pipelined, args.steps)
    e2e_pipelined(n_sus)
    e2e_s, e2e_res = wall(e2e_pipelined, args.steps)
    e2e_pipelined(max(3, n_sus // 2), True)
    e2e_g_s, e2e_g_res = wall(e2e_pipelined, args.steps, True)
    e2e_value = W * B / e2e_s
    ws_bytes = eng.workspace_bytes

    clocks = sampler.stop(first_sample, last_sample)
    if rank == 0:
        peak, peak_src = _peaks()
        # dominant kernel: the gradient kernel (two of the three contractions): 4*B*B*D flops per launch
        flops_grad = 4.0 * B * B * D
        flops_loss = 2.0 * B * B * D
        grad_avg_ms = grad_ms / max(grad_n, 1)
        loss_avg_ms = loss_ms / max(loss_n, 1)
        achieved = flops_grad / (grad_avg_ms * 1e-3) / 1e12 if grad_n else None
        traffic, traffic_src = None, None
        prof = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(prof) and (B, D) == (16384, 1024):
            try:
                with open(prof) as f:
                    tj = json.load(f)
                traffic = tj.get("grad_kernel_dram_bytes_per_launch")
                traffic_src = tj.get("source", "profiles/roofline_traffic.json (one ncu --set full capture, not measured in this run)")
            except Exception:
                traffic = None

        def stats(col):
            v = sorted(r[col] for r in per_rank)
            return {"min": v[0], "median": v[len(v) // 2], "max": v[-1]}
        clocks["per_rank_sm_mhz"] = [r[4] for r in per_rank]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": W, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"SigLIP loss fused fwd+bwd, B={B}/rank D={D} bf16, W={W} text chunk(s)/rank"
                                   + (" (BASELINE.json headline shape; at N=1 the single-chunk case)"
                                      if (B, D) == (16384, 1024) else ""),
                       "global_batch": B * W, "batch_per_rank": B, "dim": D, "world": W,
                       "parallelism": f"dp{W}", "cta_group": args.cta_group,
                       "scaling_note": "weak scaling: B/rank fixed, each rank scores W = n_gpus text chunks, so per-rank work "
                                       "grows with N and pairs/s per GPU falls as 1/N at perfect scaling; compare "
                                       "tflops_per_gpu across N (FLOP-normalised efficiency = W*t(1)/t(W))",
                       "power_state": f"sustained: warm-up extended to {n_warm} steps ({warm_ms:.0f} ms of measured GPU time, "
                                      "until three consecutive ~25 ms batches agree within 1.5 %) before the timed steps, at every N",
                       "l2": "no explicit flush: each step streams >1 GiB (16-bit sigma operand) through the 126 MB L2"
                             if B >= 8192 else "no explicit flush: inputs + sigma operand of a step fit the 126 MB L2 at this "
                                               "shape (as they do in a training loop that calls the loss every step)",
                       "api": "DDPSigmoidLoss.forward + loss.backward() (torch autograd over the C ABI)"
                              if args.api == "module" else ("siglip_fwd_bwd (C ABI, one fused call, bf16 gradients)"
                                                            if args.api == "fused" else
                                                            "CUDA graph of one siglip_fwd_bwd step, replayed"),
                       "schedule": ("fused step: L0 L1 G1 ... G0, two sigma operands, cross-rank flags inside the kernels"
                                    if (fused_step or (fused_step is None and W > 1) or args.api != "module") else
                                    "split: W loss kernels in forward(), W gradient kernels in backward()")},
            "loss": float(loss.detach().reshape(-1)[0]),
            "parity": parity,
            "flops_per_step_per_rank": 6.0 * B * (W * B) * D,
            "tflops_per_gpu": 6.0 * B * (W * B) * D / (ms_step * 1e-3) / 1e12,
            "workspace_bytes": ws_bytes,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 2 * B * D * 2, "d2h_bytes_per_step": 12,
                    "ms_per_step": e2e_s * 1e3, "loss": e2e_res[0],
                    "api": "siglip_host_submit / siglip_host_wait (pinned host bf16 in, loss/dt'/dbias out per step, "
                           "gradients stay on device; two steps in flight: the copies of step n+1 overlap the kernels "
                           "of step n); host wall clock, sustained power state (the variant ran "
                           f"{n_sus} steps right before the {args.steps} timed ones)",
                    "first_steps_ms_per_step": e2e_first_s * 1e3,
                    "with_grads": {"value": W * B / e2e_g_s, "unit": UNIT, "ms_per_step": e2e_g_s * 1e3,
                                   "h2d_bytes_per_step": 2 * B * D * 2, "d2h_bytes_per_step": 2 * B * D * 2 + 12,
                                   "loss": e2e_g_res[0],
                                   "api": "same entries with gradient buffers: the bf16 dimg/dtxt of every step also return "
                                          "to pinned host memory on a second copy stream (overlapping the next step)"},
                    "sync_ms_per_step": e2e_sync_s * 1e3,
                    "sync_api": "siglip_fwd_bwd_host (copy, step, copy, wait: nothing overlapped)",
                    "cpu_affinity": numa},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "burst": {"value": W * B / (burst_ms * 1e-3), "unit": UNIT, "ms_per_step": burst_ms,
                      "tflops_per_gpu": 6.0 * B * (W * B) * D / (burst_ms * 1e-3) / 1e12,
                      "note": f"the {args.steps} steps right after the {max(args.warmup, 3)} warm-up steps, still at boost clocks "
                              "(shorter than ~50 ms only at small N); the headline value is the sustained one"},
            "roofline": {"bound": "tensor", "kernel": "siglip_gemm_kernel<cg,1> (dimg + dtxt contractions)",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": (achieved / peak) if achieved else None, "peak_source": peak_src,
                         "avg_launch_ms": grad_avg_ms, "launches_timed": grad_n,
                         "timed_in": f"a second region of {args.steps} steps right behind the value's region, every launch "
                                     f"bracketed by CUDA events on its stream: {ms_step_events:.4f} ms/step there on rank 0",
                         "ms_per_step_with_kernel_events": ms_step_events, "traffic": traffic,
                         "traffic_source": traffic_src,
                         "loss_kernel": {"achieved": flops_loss / (loss_avg_ms * 1e-3) / 1e12 if loss_n else None,
                                         "avg_launch_ms": loss_avg_ms, "launches_timed": loss_n}},
            "per_rank": {"ms_per_step": stats(0), "loss_kernel_ms_per_launch": stats(1),
                         "gradient_kernel_ms_per_launch": stats(2), "kernel_ms_per_step": stats(3),
                         "ms_per_step_by_rank": [r[0] for r in per_rank],
                         "kernel_ms_per_step_by_rank": [r[3] for r in per_rank],
                         "note": "CUDA events on each rank's launch stream over the timed steps; a rank's kernels include the "
                                 "time its auxiliary warps wait for peer flags"},
        }
        if single is not None:
            t1_0, t1_max = single[0], max(single)
            line["scaling_diag"] = {
                "single_chunk_ms_by_rank": single,
                "what": "every GPU's own W=1 step through the same module (one-rank subgroups), all GPUs loaded at the same "
                        "time, sustained state, no cross-rank dependency",
                "gpu_spread": t1_max / min(single) - 1.0,
                "efficiency_vs_rank0_single": W * t1_0 / ms_step,
                "efficiency_vs_slowest_gpu_single": W * t1_max / ms_step,
                "note": "FLOP-normalised weak-scaling efficiency W*t(1)/t(W). The coupled job is paced by its slowest GPU "
                        "(ranks wait for peer flags inside their kernels): against the slowest GPU's own single-chunk step "
                        "the remainder is what the exchange and the W>1 data flow cost"}
        if W > 1:
            # per step rank 0 pulls (W-1) bf16 text chunks and (W-1) fp32 dtxt contributions through the NVSwitch
            algo_rx = (W - 1) * (B * D * 2 + B * D * 4)
            nv = {"algorithmic_rx_bytes_per_step": algo_rx,
                  "algorithmic_rx_GBps": algo_rx / (ms_step * 1e-3) / 1e9, "peak_GBps_per_direction": 900.0,
                  "note": "all of it moved by ld.global from peer-mapped memory inside the loss / gradient kernels; "
                          "measured = NVML NVLink payload counters of GPU 0 over the timed region (includes the barrier)"}
            if nvl0 is not None and nvl1 is not None:
                nv["measured_rx_GBps"] = (nvl1[0] - nvl0[0]) / (ms_total * 1e-3) / 1e9
                nv["measured_tx_GBps"] = (nvl1[1] - nvl0[1]) / (ms_total * 1e-3) / 1e9
            else:
                nv["measured_rx_GBps"] = nv["measured_tx_GBps"] = None
            line["nvlink"] = nv
        if W == 1 and not args.no_cpu_baseline:
            # in a fresh process: this one is pinned to the GPU's NUMA node, the CPU baseline may use every host core
            try:
                env = dict(os.environ)
                for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
                    env.pop(k, None)
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--gpus", "1",
                                      "--steps", str(args.cpu_steps), "--warmup", "1", "--batch", str(B), "--dim", str(D)],
                                     capture_output=True, text=True, timeout=900, env=env).stdout
                ref = json.loads(out.strip().splitlines()[-1])
                line["cpu_baseline"] = ref["cpu_baseline"]
            except Exception as ex:  # noqa: BLE001
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": None, "kind": "reference",
                                        "sample": f"failed: {ex}"}
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if parity is not None and not parity["pass"]:
        return 3
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=16384)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--api", default="module", choices=["module", "fused", "graph"],
                    help="what one timed step calls: the nn.Module (forward + backward), the fused C-ABI entry, or a CUDA "
                         "graph of the fused C-ABI step (single GPU)")
    ap.add_argument("--schedule", default="auto", choices=["auto", "fused", "split"],
                    help="module schedule: auto = fused step (two sigma operands, in-kernel flags) on a multi-rank group and "
                         "split forward/backward on one rank; fused / split force one")
    ap.add_argument("--cta-group", type=int, default=int(os.environ.get("SIGLIP_CTA_GROUP", "2")))
    ap.add_argument("--cpu-steps", type=int, default=3, help="timed steps of the cpu_baseline leg inside the N=1 run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-scaling-diag", action="store_true")
    ap.add_argument("--clock-period-ms", type=float, default=5.0, help="NVML clock / throttle-reason sampling period")
    ap.add_argument("--sustain-ms", type=float, default=600.0,
                    help="minimum GPU time of the warm-up (power-capped sustained clocks at every N)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them returned on rank 0 (loss, dimg, dtxt, "
                         "dt_prime, dbias) as DIR/<name>.npy, at most 64 MB: larger gradients are cut to a seeded "
                         "sample of rows, listed in grad_rows.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's path, not of --impl reference")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
